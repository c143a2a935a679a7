"""Model selection without a GPU: the two references agree, the entry points are declared everywhere, the Python
layer's argument handling, and the library's checks and its failure without a device."""
import ctypes as C
import os

import numpy as np
import pytest

import redux_b200 as rb
import select_models_cases as smc
from test_capi_cpu import ROOT, _run_without_a_device

NAMES = ("redux_select_models", "redux_select_models_device", "redux_encode_batch_select")


@pytest.mark.parametrize("case", smc.CASES, ids=lambda c: c.name)
def test_walk_and_closed_form_agree(case):
    walk = smc.reference_costs(case, walk=True)
    closed = smc.reference_costs(case)
    assert (np.abs(walk - closed) <= smc.tolerance(closed)).all(), (case.name, np.abs(walk - closed).max())


def test_cases_cover_what_the_contract_names():
    """Widths 1, 3, 7, 8, 12, 16; split points at 0, inside, just below and above n; empty and symbol-less blocks;
    partial symbols; duplicate rows; K = 1 and K = 300; multi-CTA histograms; fresh and trained winners."""
    assert {c.params[0] for c in smc.CASES} >= {1, 3, 7, 8, 12, 16}
    assert {len(c.rows) for c in smc.CASES} >= {1, 300}
    kinds = set()
    for c in smc.CASES:
        s, f, _ = c.params
        F = (1 << f) - 1
        for b in c.blocks:
            n = len(b) * 8 // s
            kinds.add("empty" if not b else "no_symbol" if n == 0 else "partial" if len(b) * 8 % s else "whole")
            if n > 16384:
                kinds.add("multi_cta")
            for r in c.rows:
                room = F - int(r.astype(np.int64).sum())
                kinds.add("m0" if room == 0 else "m1" if room == 1 else "below_n" if room == n - 1 and n
                          else "above_n" if room == n + 1 else "other")
        tab = smc.table(c)
        if len({r.tobytes() for r in tab}) < len(tab):
            kinds.add("duplicate")
        if len(c.rows) > 1:
            win = smc.reference_costs(c).argmin(axis=1)
            kinds.update("fresh_wins" if (tab[w] == 1).all() else "trained_wins" for w in win)
    assert {"empty", "no_symbol", "partial", "multi_cta", "m0", "m1", "below_n", "above_n", "duplicate",
            "fresh_wins", "trained_wins"} <= kinds, kinds
    assert any(c.params[0] == 12 and any(len(b) == 1 for b in c.blocks) for c in smc.CASES)


def test_select_entry_points_are_declared():
    hdr = open(os.path.join(ROOT, "include", "redux_b200.h")).read()
    rs = open(os.path.join(ROOT, "bindings", "rust", "src", "lib.rs")).read()
    integ = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    for name in NAMES:
        assert "int %s(" % name in hdr and hasattr(rb.lib(), name)
        assert "fn %s(" % name in rs and "fn %s(" % name in integ
    assert "#define REDUX_KERNEL_KINDS    5" in hdr


def _no_context():
    ctx = rb.Context.__new__(rb.Context)
    ctx._h = C.c_void_p()
    return ctx


def test_python_arguments_are_checked_before_the_library():
    p = rb.Parameters(8, 14, 16)
    ctx = _no_context()
    data, off = np.zeros(8, np.uint8), np.array([0, 8], np.uint64)
    for call in (lambda m: ctx.select_models(data, off, m), lambda m: ctx.encode_batch_select(data, off, m),
                 lambda m: ctx.select_models_device(0, 0, 1, 8, m, 0)):
        with pytest.raises(rb.InvalidInput, match="no models"):
            call([])
        with pytest.raises(rb.InvalidInput, match="kinds"):
            call([rb.AdaptiveTreeModel(p), rb.AdaptiveLinearModel(p)])
        with pytest.raises(rb.InvalidInput, match="Parameters"):
            call([rb.AdaptiveTreeModel(p), rb.AdaptiveTreeModel(rb.Parameters(8, 30, 32))])


def test_select_calls_check_rows_and_fail_loudly_without_a_device():
    """No device: n_models 0 and a bad row are InvalidInput, an oversized table Unsupported, before a device is needed;
    valid calls return CUDA_ERROR rather than computing anything, and the Python methods raise CudaError."""
    _run_without_a_device("""
        import ctypes as C
        import numpy as np
        import pytest
        import redux_b200 as rb
        L = rb.lib()
        p = rb.Parameters(8, 14, 16)._c()
        data = np.zeros(16, dtype=np.uint8)
        off = np.array([0, 16], dtype=np.uint64)
        bm = np.full(1, 7, dtype=np.uint32)
        out = np.zeros(64, dtype=np.uint8)
        ooff = np.zeros(2, dtype=np.uint64)
        st = np.zeros(1, dtype=np.int32)
        good = np.ones((2, 257), dtype=np.uint32)
        zero = good.copy(); zero[1, 5] = 0
        over = good.copy(); over[0, 0] = (1 << 14)
        big_n = (256 << 20) // (258 * 4) + 1
        def calls(tab, n):
            t = tab.ctypes.data if tab is not None else None
            return (L.redux_select_models(None, C.byref(p), t, n, data.ctypes.data, off.ctypes.data, 1, bm.ctypes.data, None),
                    L.redux_select_models_device(None, 0, None, C.byref(p), t, n, data.ctypes.data, off.ctypes.data, 1, 16,
                                                 bm.ctypes.data, None),
                    L.redux_encode_batch_select(None, rb.MODEL_TREE, C.byref(p), t, n, data.ctypes.data, off.ctypes.data, 1,
                                                out.ctypes.data, out.size, ooff.ctypes.data, st.ctypes.data, bm.ctypes.data))
        assert calls(good, 2) == (rb.CUDA_ERROR,) * 3
        assert calls(good, 0) == (rb.INVALID_INPUT,) * 3
        assert calls(zero, 2) == (rb.INVALID_INPUT,) * 3
        assert calls(over, 2) == (rb.INVALID_INPUT,) * 3
        assert calls(np.zeros((big_n, 257), dtype=np.uint32), big_n) == (rb.UNSUPPORTED,) * 3   # size checked first
        assert (bm == 7).all()
        ctx = rb.Context.__new__(rb.Context)
        ctx._h = C.c_void_p()
        models = [rb.AdaptiveTreeModel(rb.Parameters(8, 14, 16))] * 2
        with pytest.raises(rb.CudaError):
            ctx.select_models(data, off, models)
        with pytest.raises(rb.CudaError):
            ctx.encode_batch_select(data, off, models)
    """)
