"""Model training and container version 2 without a GPU: argument handling of the Python layer, the header's
declarations, that the library fails loudly without a device, and that corrupt version 2 files are rejected before
anything is decoded."""
import io
import os
import struct

import numpy as np
import pytest

import redux_b200 as rb
import redux_b200.container as ct
from test_capi_cpu import ROOT, _run_without_a_device


def test_train_entry_points_are_declared():
    hdr = open(os.path.join(ROOT, "include", "redux_b200.h")).read()
    for name in ("redux_train_models", "redux_train_models_device"):
        assert "int %s(" % name in hdr and hasattr(rb.lib(), name)
    assert "#define REDUX_KERNEL_KINDS    5" in hdr
    rs = open(os.path.join(ROOT, "bindings", "rust", "src", "lib.rs")).read()
    assert "fn redux_train_models(" in rs and "fn redux_train_models_device(" in rs


def test_train_start_argument():
    p = rb.Parameters(8, 14, 16)
    fresh = rb.AdaptiveTreeModel(p)
    cls, params, pc, table, n_models, sm = rb._train_start(fresh, 5)
    assert cls is rb.AdaptiveTreeModel and params is p and table is None and n_models == 0 and sm is None
    trained = rb.AdaptiveLinearModel(p).train([7, 7, 9])
    cls, _, _, table, n_models, sm = rb._train_start(trained, 5)
    assert cls is rb.AdaptiveLinearModel and n_models == 1 and sm is None
    assert table.shape == (1, 257) and table[0, 7] == 3 and table.sum() == 260
    cls, _, _, table, n_models, sm = rb._train_start([fresh, rb.AdaptiveTreeModel(p).train([1])], 2)
    assert n_models == 2 and (sm == [0, 1]).all() and table[1, 1] == 2 and (table[0] == 1).all()
    assert fresh.freq is None
    with pytest.raises(rb.InvalidInput, match="3 start models for 2"):
        rb._train_start([fresh] * 3, 2)
    with pytest.raises(rb.InvalidInput, match="kinds"):
        rb._train_start([fresh, rb.AdaptiveLinearModel(p)], 2)
    with pytest.raises(rb.InvalidInput):
        rb._train_start([], 0)


def test_train_calls_fail_loudly_without_a_device():
    """No device: no context, and both entry points return CUDA_ERROR rather than computing anything."""
    _run_without_a_device("""
        import ctypes as C
        import numpy as np
        import pytest
        import redux_b200 as rb
        with pytest.raises(rb.CudaError):
            rb.Context()
        L = rb.lib()
        p = rb.Parameters(8, 14, 16)._c()
        data = np.zeros(16, dtype=np.uint8)
        off = np.array([0, 16], dtype=np.uint64)
        out = np.zeros(257, dtype=np.uint32)
        assert L.redux_train_models(None, C.byref(p), None, 0, None, data.ctypes.data, off.ctypes.data, 1,
                                    out.ctypes.data) == rb.CUDA_ERROR
        assert L.redux_train_models_device(None, 0, None, C.byref(p), None, 0, None, data.ctypes.data,
                                           off.ctypes.data, 1, 16, out.ctypes.data) == rb.CUDA_ERROR
        assert (out == 0).all()
    """)


# --------------------------------------------------------------------------- container version 2
P = (8, 14, 16)


def v2_file(table, blocks, idx, block_len=4, n_models=None, kind=rb.MODEL_TREE):
    """A version 2 file by hand: one segment of len(blocks) blocks with dummy streams."""
    table = np.asarray(table, dtype="<u4")
    out = ct.HEADER.pack(ct.MAGIC, 2, kind, *P, block_len)
    out += struct.pack("<I", table.shape[0] if n_models is None else n_models) + table.tobytes()
    n = len(blocks)
    out += struct.pack("<II", n, len(blocks[-1])) + np.asarray(idx, dtype="<u4").tobytes()
    out += np.array([len(b) for b in blocks], dtype="<u4").tobytes() + b"".join(blocks)
    return out + struct.pack("<II", 0, 0)


def test_v2_header_reads_the_model_table():
    table = np.ones((2, 257), dtype=np.uint32)
    table[1, 65] = 100
    ver, models, block_len = ct.read_header_any(io.BytesIO(v2_file(table, [b"xy"], [1])))
    assert ver == 2 and block_len == 4 and len(models) == 2
    assert all(type(m) is rb.AdaptiveTreeModel and (m.params.freq_bits, m.params.code_bits) == (14, 16) for m in models)
    assert (models[1].freq == table[1]).all() and models[1].total_frequency() == 257 + 99
    # version 1: one fresh model, and read_header keeps its v1-only contract
    buf = io.BytesIO()
    ct.write_header(buf, rb.AdaptiveLinearModel(rb.Parameters(*P)), 8)
    ver, models, block_len = ct.read_header_any(io.BytesIO(buf.getvalue()))
    assert ver == 1 and len(models) == 1 and models[0].freq is None and block_len == 8
    with pytest.raises(ct.ContainerError):
        ct.read_header(io.BytesIO(v2_file(table, [b"xy"], [1])))


@pytest.mark.parametrize("what", ["zero_entry", "over_fmax", "no_rows", "over_cap", "bad_index", "bad_version"])
def test_v2_corruptions_are_rejected_before_decoding(what):
    """Each of these raises ContainerError before a device is touched (the test runs without one)."""
    table = np.ones((2, 257), dtype=np.uint32)
    idx, n_models = [0, 1], None
    if what == "zero_entry":
        table[1, 3] = 0
    elif what == "over_fmax":
        table[0, 0] = (1 << 14) - 1 - 256 + 1                # total = freq_max + 1
    elif what == "no_rows":
        table, n_models = table[:0], 0
    elif what == "over_cap":
        n_models = (256 << 20) // (258 * 4) + 1
    elif what == "bad_index":
        idx = [0, 2]
    blob = v2_file(table, [b"abcd", b"ef"], idx, n_models=n_models)
    if what == "bad_version":
        blob = blob[:4] + b"\x03" + blob[5:]
    with pytest.raises(ct.ContainerError):
        ct.unpack(blob)


def test_truncated_v2_files_raise_eof():
    table = np.ones((3, 257), dtype=np.uint32)
    blob = v2_file(table, [b"abcd", b"ef"], [2, 0])
    for cut in (ct.HEADER.size + 2, ct.HEADER.size + 4 + 100, ct.HEADER.size + 4 + table.nbytes + 4,
                ct.HEADER.size + 4 + table.nbytes + 8 + 4):
        with pytest.raises(rb.Eof):
            ct.unpack(blob[:cut])


def test_pack_models_checks_block_model_first():
    """block_model too short for the data or naming a missing model: ContainerError before any device call (the
    test runs without one)."""
    models = [rb.AdaptiveTreeModel(rb.Parameters(*P)), rb.AdaptiveTreeModel(rb.Parameters(*P)).train([1, 2])]
    with pytest.raises(ct.ContainerError, match="3 blocks"):
        ct.pack_models(b"x" * 9, models, [0, 1], block_len=4)
    with pytest.raises(ct.ContainerError, match="outside"):
        ct.pack_models(b"x" * 9, models, [0, 1, 2], block_len=4)
    with pytest.raises(ct.ContainerError, match="outside"):
        ct.pack_models(b"x" * 9, models, [0, -1, 1], block_len=4)
    with pytest.raises(ct.ContainerError, match="byte-symbol"):
        ct.pack_models(b"x" * 9, [rb.AdaptiveTreeModel(rb.Parameters(12, 14, 16))], [0, 0, 0], block_len=4)
    with pytest.raises(rb.InvalidInput, match="kinds"):
        ct.pack_models(b"x" * 9, [models[0], rb.AdaptiveLinearModel(rb.Parameters(*P))], [0, 1, 0], block_len=4)
