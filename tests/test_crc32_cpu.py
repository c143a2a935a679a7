"""CRC-32 and container version 3 without a GPU: the entry points are declared everywhere, the library's argument
checks and its failure without a device, the version 3 header, and the writer's refusals before any device call."""
import io
import os
import struct

import numpy as np
import pytest

import redux_b200 as rb
from redux_b200 import container as ct
from test_capi_cpu import ROOT, _run_without_a_device

NAMES = ("redux_crc32_blocks", "redux_crc32_blocks_device", "redux_encode_batch_models_crc",
         "redux_encode_batch_select_crc", "redux_decode_batch_models_crc")


def test_crc_entry_points_are_declared():
    hdr = open(os.path.join(ROOT, "include", "redux_b200.h")).read()
    rs = open(os.path.join(ROOT, "bindings", "rust", "src", "lib.rs")).read()
    integ = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    for name in NAMES:
        assert "int %s(" % name in hdr and hasattr(rb.lib(), name)
        assert "fn %s(" % name in rs and "fn %s(" % name in integ
    assert "crc32fast::hash" in integ
    assert "#define REDUX_KERNEL_KINDS    5" in hdr
    # not a coder kernel: the library still names 37
    assert len(rb.kernel_names()) == 37 and not any("crc" in n for n in rb.kernel_names())


def test_crc_calls_check_arguments_and_fail_loudly_without_a_device():
    """No device: NULL buffers and offsets that decrease are InvalidInput before a device is needed; valid calls return
    CUDA_ERROR rather than computing anything, and the Python methods raise CudaError."""
    _run_without_a_device("""
        import ctypes as C
        import numpy as np
        import pytest
        import redux_b200 as rb
        L = rb.lib()
        p = rb.Parameters(8, 14, 16)._c()
        data = np.arange(32, dtype=np.uint8)
        good = np.array([0, 16, 32], dtype=np.uint64)
        down = np.array([0, 16, 8], dtype=np.uint64)
        row = np.ones(257, dtype=np.uint32)
        out = np.zeros(256, dtype=np.uint8)
        ooff = np.zeros(3, dtype=np.uint64)
        st = np.zeros(2, dtype=np.int32)
        bm = np.zeros(2, dtype=np.uint32)
        crc = np.full(2, 7, dtype=np.uint32)
        raw = np.zeros(64, dtype=np.uint8)
        rl, cons = np.zeros(2, dtype=np.uint64), np.zeros(2, dtype=np.uint64)
        def calls(off, c, lens=True):
            o = off.ctypes.data if off is not None else None
            cp = c.ctypes.data if c is not None else None
            return (L.redux_crc32_blocks(None, data.ctypes.data, o, 2, cp),
                    L.redux_crc32_blocks_device(None, 0, None, data.ctypes.data, o, None, 2, 16, cp),
                    L.redux_encode_batch_models_crc(None, rb.MODEL_TREE, C.byref(p), row.ctypes.data, 1, None,
                                                    data.ctypes.data, o, 2, out.ctypes.data, out.size,
                                                    ooff.ctypes.data, st.ctypes.data, cp),
                    L.redux_encode_batch_select_crc(None, rb.MODEL_TREE, C.byref(p), row.ctypes.data, 1,
                                                    data.ctypes.data, o, 2, out.ctypes.data, out.size,
                                                    ooff.ctypes.data, st.ctypes.data, bm.ctypes.data, cp),
                    L.redux_decode_batch_models_crc(None, rb.MODEL_TREE, C.byref(p), row.ctypes.data, 1, None,
                                                    data.ctypes.data, o, 2, raw.ctypes.data, o,
                                                    rl.ctypes.data if lens else None, cons.ctypes.data,
                                                    st.ctypes.data, cp))
        assert calls(good, crc) == (rb.CUDA_ERROR,) * 5
        assert calls(good, None) == (rb.INVALID_INPUT,) * 5
        assert calls(None, crc) == (rb.INVALID_INPUT,) * 5
        # offsets that decrease: the device form cannot see them (device memory)
        assert calls(down, crc) == (rb.INVALID_INPUT, rb.CUDA_ERROR) + (rb.INVALID_INPUT,) * 3
        assert calls(good, crc, lens=False)[4] == rb.INVALID_INPUT
        # NULL input with bytes to read
        assert L.redux_crc32_blocks(None, None, good.ctypes.data, 2, crc.ctypes.data) == rb.INVALID_INPUT
        assert L.redux_crc32_blocks_device(None, 0, None, None, good.ctypes.data, None, 2, 16,
                                           crc.ctypes.data) == rb.INVALID_INPUT
        # nothing to do still needs a device
        assert L.redux_crc32_blocks(None, None, None, 0, None) == rb.CUDA_ERROR
        assert (crc == 7).all()
        ctx = rb.Context.__new__(rb.Context)
        ctx._h = C.c_void_p()
        models = [rb.AdaptiveTreeModel(rb.Parameters(8, 14, 16))]
        for call in (lambda: ctx.crc32_blocks(data, good),
                     lambda: ctx.encode_batch_models_crc(data, good, models, None),
                     lambda: ctx.encode_batch_models_crc(data, good, models, None, check=False),
                     lambda: ctx.encode_batch_select_crc(data, good, models),
                     lambda: ctx.decode_batch_models_crc(data, good, good, models, None, check=False)):
            with pytest.raises(rb.CudaError):
                call()
    """)


def _v3(n_models=1, nsym=257, ver=3, table=None, s=8, f=14, c=16, kind=rb.MODEL_TREE, block_len=4096):
    head = ct.HEADER.pack(ct.MAGIC, ver, kind, s, f, c, block_len)
    if table is None:
        table = np.ones((n_models, nsym), dtype="<u4")
    return head + struct.pack("<I", n_models) + table.astype("<u4").tobytes()


def test_read_header_any_reads_version_3():
    trained = np.ones((2, 257), dtype=np.uint32)
    trained[1, :5] = 9
    ver, models, block_len = ct.read_header_any(io.BytesIO(_v3(2, table=trained)))
    assert ver == 3 and block_len == 4096 and len(models) == 2
    assert all(isinstance(m, rb.AdaptiveTreeModel) for m in models)
    assert (models[1].freq == trained[1]).all() and models[1].params.freq_bits == 14
    # read_header (version 1 only) still refuses it
    with pytest.raises(ct.ContainerError):
        ct.read_header(io.BytesIO(_v3()))


def test_read_header_any_rejects_bad_version_3_headers():
    zero = np.ones((1, 257), dtype=np.uint32)
    zero[0, 3] = 0
    over = np.ones((1, 257), dtype=np.uint32)
    over[0, 0] = 1 << 14
    for blob in (_v3(ver=4), _v3(block_len=0), _v3(kind=5), b"RDXC" + _v3()[4:], _v3(0), _v3(table=zero),
                 _v3(table=over), _v3((256 << 20) // (258 * 4) + 1, table=np.ones((1, 257)))):
        with pytest.raises(ct.ContainerError):
            ct.read_header_any(io.BytesIO(blob))
    with pytest.raises(rb.InvalidInput):
        ct.read_header_any(io.BytesIO(_v3(s=8, f=8, c=8)))          # Parameters::new rejects these
    for cut in (ct.HEADER.size + 2, len(_v3()) - 1):
        with pytest.raises(rb.Eof):
            ct.read_header_any(io.BytesIO(_v3()[:cut]))


class _NoDevice:
    """A context that fails the test if the writer asks it for anything."""

    def __getattr__(self, name):
        raise AssertionError("device call %s before the arguments were checked" % name)


def test_checksum_writers_refuse_before_any_device_call():
    p = rb.Parameters(8, 14, 16)
    trained = rb.AdaptiveTreeModel(p)
    trained.train(b"abc")
    data = bytes(range(200))
    nd = _NoDevice()
    with pytest.raises(ct.ContainerError, match="byte-symbol"):
        ct.pack(data, rb.AdaptiveTreeModel(rb.Parameters(4, 14, 16)), context=nd, checksum=True)
    with pytest.raises(ct.ContainerError, match="fresh"):
        ct.pack(data, trained, context=nd, checksum=True)
    with pytest.raises(ct.ContainerError, match="byte-symbol"):
        ct.pack_models(data, [rb.AdaptiveTreeModel(rb.Parameters(12, 20, 24))], [0], context=nd, checksum=True)
    with pytest.raises(ct.ContainerError, match="outside"):
        ct.pack_models(data, [p and rb.AdaptiveTreeModel(p)], [1], context=nd, checksum=True)
    with pytest.raises(ct.ContainerError, match="entries"):
        ct.pack_models(data, [rb.AdaptiveTreeModel(p)], [], block_len=100, context=nd, checksum=True)
    with pytest.raises(rb.InvalidInput, match="kinds"):
        ct.pack_auto(data, [rb.AdaptiveTreeModel(p), rb.AdaptiveLinearModel(p)], context=nd, checksum=True)
    big = [rb.AdaptiveTreeModel(p)] * ((256 << 20) // (258 * 4) + 1)
    with pytest.raises(ct.ContainerError, match="larger"):
        ct.pack_auto(data, big, context=nd, checksum=True)


def test_version_3_without_its_end_marker_is_refused_before_decoding():
    """A version 3 segment must be followed by another segment header or the end marker; the reader checks that before
    it decodes the segment (no device is touched here)."""
    blob = _v3() + struct.pack("<II", 1, 3) + struct.pack("<III", 0, 2, 0) + b"xy"
    with pytest.raises(ct.ContainerError, match="neither a segment nor the end marker"):
        ct.unpack(blob, context=_NoDevice())
