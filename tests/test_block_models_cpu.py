"""The per-block model calls without a GPU: what the Python layer checks before any call, the header's table cap, and
that the library fails loudly without a device."""
import os
import re

import numpy as np
import pytest

import redux_b200 as rb
from test_capi_cpu import ROOT, _run_without_a_device


def test_model_table_of_fresh_and_trained_models():
    p = rb.Parameters(8, 14, 16)
    fresh = rb.AdaptiveTreeModel(p)
    trained = rb.AdaptiveTreeModel(p).train([3, 3, 256])
    kind, pc, table = rb._model_table([fresh, trained, fresh])
    assert kind == rb.MODEL_TREE and (pc.symbol_bits, pc.freq_bits, pc.code_bits) == (8, 14, 16)
    assert table.dtype == np.uint32 and table.shape == (3, 257)
    assert (table[0] == 1).all() and (table[2] == 1).all()
    assert table[1, 3] == 3 and table[1, 256] == 2 and table[1].sum() == 260
    assert fresh.freq is None                        # a fresh model stays fresh


def test_mixed_kinds_or_parameters_are_refused():
    p = rb.Parameters(8, 14, 16)
    with pytest.raises(rb.InvalidInput):
        rb._model_table([])
    with pytest.raises(rb.InvalidInput, match="kinds"):
        rb._model_table([rb.AdaptiveTreeModel(p), rb.AdaptiveLinearModel(p)])
    with pytest.raises(rb.InvalidInput, match="Parameters"):
        rb._model_table([rb.AdaptiveTreeModel(p), rb.AdaptiveTreeModel(rb.Parameters(8, 14, 17))])


def test_start_tree_cap_is_in_the_header():
    hdr = open(os.path.join(ROOT, "include", "redux_b200.h")).read()
    m = re.search(r"#define REDUX_MAX_MODEL_TABLE_BYTES \(\(uint64_t\)(\d+) << (\d+)\)", hdr)
    assert m and int(m.group(1)) << int(m.group(2)) == 256 << 20
    for name in ("redux_encode_batch_models", "redux_decode_batch_models", "redux_encode_batch_device_models",
                 "redux_decode_batch_device_models"):
        assert name + "(" in hdr and hasattr(rb.lib(), name)


def test_block_model_calls_fail_loudly_without_a_device():
    """No device, no context (CUDA_ERROR); the new entry points given no context refuse it instead of coding."""
    _run_without_a_device("""
        import ctypes as C
        import numpy as np
        import pytest
        import redux_b200 as rb
        with pytest.raises(rb.CudaError):
            rb.Context()
        L = rb.lib()
        p = rb.Parameters(8, 14, 16)._c()
        table = np.ones(257, dtype=np.uint32)
        off = np.zeros(2, dtype=np.uint64)
        rc = L.redux_encode_batch_models(None, 1, C.byref(p), table.ctypes.data, 1, None, None, off.ctypes.data, 1,
                                         None, 0, off.ctypes.data, None)
        assert rc == rb.INVALID_INPUT
        rc = L.redux_decode_batch_models(None, 1, C.byref(p), table.ctypes.data, 1, None, None, off.ctypes.data, 1,
                                         None, off.ctypes.data, None, None, None)
        assert rc == rb.INVALID_INPUT
        for fn in (L.redux_encode_batch_device_models, L.redux_decode_batch_device_models):
            args = [None, 0, None, 1, C.byref(p), table.ctypes.data, 1, None] + [None] * (len(fn.argtypes) - 8)
            for k, t in enumerate(fn.argtypes):
                if t is C.c_uint64 and args[k] is None:
                    args[k] = 0
            assert fn(*args) == rb.INVALID_INPUT
    """)
