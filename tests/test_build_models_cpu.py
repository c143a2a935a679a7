"""Model building without a GPU: the entry points are declared everywhere, the ladder for every valid (s, f), the
library's argument checks before a device is needed, and its failure without one."""
import os

import numpy as np
import pytest

import build_models_cases as bmc
import redux_b200 as rb
from test_build_models_emu import emu_ladder, load_build_emu
from test_capi_cpu import ROOT, _run_without_a_device

NAMES = ("redux_build_models", "redux_build_models_device")


def test_build_entry_points_are_declared():
    hdr = open(os.path.join(ROOT, "include", "redux_b200.h")).read()
    rs = open(os.path.join(ROOT, "bindings", "rust", "src", "lib.rs")).read()
    integ = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    for name in NAMES:
        assert "int %s(" % name in hdr and hasattr(rb.lib(), name)
        assert "fn %s(" % name in rs and "fn %s(" % name in integ
    assert "#define REDUX_MAX_BUILD_SCRATCH_BYTES" in hdr
    assert hasattr(rb.Context, "build_models") and hasattr(rb.Context, "build_models_device")


def test_no_new_coder_kernels():
    assert len(rb.kernel_names()) == 37
    hdr = open(os.path.join(ROOT, "include", "redux_b200.h")).read()
    assert "#define REDUX_KERNEL_KINDS    5" in hdr


def test_ladder_of_every_valid_width_and_freq_bits():
    emu = load_build_emu()
    n = 0
    for s in range(1, 17):
        for f in range(s + 2, 32):
            T = emu_ladder(emu, s, f)
            assert T == bmc.ladder(s, f), (s, f)
            assert T[0] == (1 << f) - 1 and T[-1] >= 2 * ((1 << s) + 1)
            n += 1
    assert n > 200


def test_python_arguments_are_checked_before_the_library():
    p = rb.Parameters(8, 14, 16)
    ctx = rb.Context.__new__(rb.Context)
    ctx._h = None
    data, off = np.zeros(8, np.uint8), np.array([0, 4, 8], np.uint64)
    with pytest.raises(rb.InvalidInput, match="fresh"):
        ctx.build_models(data, off, rb.AdaptiveTreeModel(p).train([1, 2]), 2)
    with pytest.raises(rb.InvalidInput, match="init values"):
        ctx.build_models(data, off, rb.AdaptiveTreeModel(p), 2, init=[1])
    with pytest.raises(rb.InvalidInput, match="negative"):
        ctx.build_models(data, off, rb.AdaptiveTreeModel(p), 2, init=[1, -1])


def test_build_checks_come_first_and_fail_loudly_without_a_device():
    """No device: each argument check fires with its code before a device is needed, and valid calls return
    CUDA_ERROR in both forms rather than computing anything."""
    _run_without_a_device("""
        import ctypes as C
        import numpy as np
        import pytest
        import redux_b200 as rb
        L = rb.lib()
        data = np.zeros(64, dtype=np.uint8)
        off = np.array([0, 32, 64], dtype=np.uint64)
        tab = np.zeros((1 << 20, 258), dtype=np.uint32)
        bm = np.zeros(2, dtype=np.uint32)
        tot = np.zeros(4, dtype=np.float64)
        def calls(params, K, it, init=None, n=2):
            p = rb.Parameters(*params)._c()
            i = None if init is None else np.asarray(init, dtype=np.uint32)
            ip = None if i is None else i.ctypes.data
            return (L.redux_build_models(None, C.byref(p), K, it, ip, data.ctypes.data, off.ctypes.data, n,
                                         tab.ctypes.data, bm.ctypes.data, tot.ctypes.data),
                    L.redux_build_models_device(None, 0, None, C.byref(p), K, it, ip, data.ctypes.data,
                                                off.ctypes.data, n, 32, tab.ctypes.data, bm.ctypes.data,
                                                tot.ctypes.data))
        assert calls((8, 14, 16), 4, 2) == (rb.CUDA_ERROR,) * 2
        assert calls((8, 14, 16), 4, 2, [0, 4]) == (rb.CUDA_ERROR,) * 2
        assert calls((8, 14, 16), 0, 2) == (rb.INVALID_INPUT,) * 2
        assert calls((8, 14, 16), 4, 0) == (rb.INVALID_INPUT,) * 2
        assert calls((8, 14, 16), 4, 2, [0, 5]) == (rb.INVALID_INPUT,) * 2
        assert calls((8, 14, 16), 4, 2, n=0) == (rb.INVALID_INPUT,) * 2
        big_k = (256 << 20) // (258 * 4)
        assert calls((8, 14, 16), big_k, 1) == (rb.UNSUPPORTED,) * 2
        assert calls((8, 14, 16), big_k - 1, 1) == (rb.CUDA_ERROR,) * 2
        assert calls((17, 20, 24), 4, 2) == (rb.UNSUPPORTED,) * 2
        ctx = rb.Context.__new__(rb.Context)
        ctx._h = C.c_void_p()
        with pytest.raises(rb.CudaError):
            ctx.build_models(data, off, rb.AdaptiveTreeModel(rb.Parameters(8, 14, 16)), 4)
        used = rb.AdaptiveTreeModel(rb.Parameters(8, 14, 16))
        used.total_frequency(); used._state()          # a fresh model whose state is held as a row of ones
        with pytest.raises(rb.CudaError):               # reaches the library: it is still fresh
            ctx.build_models(data, off, used, 4)
    """)
