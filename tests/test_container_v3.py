"""Container version 3 (a CRC-32 per block) on a B200: `pytest -m gpu`.

pack / pack_models / pack_auto with checksum=True round trip, with ragged tails and several segments; each block's
stream is the one version 2 stores for the same input; a damaged CRC field is refused; and bit flips over the streams
of generator blocks never come back as wrong bytes: each either decodes to exactly the original block or fails the
version 3 reader's checks.
"""
import io
import struct
import zlib

import numpy as np
import pytest

import redux_b200 as rb
from redux_b200 import container as ct

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = rb.Context()
    yield c
    c.close()


def _data(n_bytes, seed):
    return rb.generate_blocks_host(0, (n_bytes + 4095) // 4096, 4096, seed)[:n_bytes].tobytes()


def _models(p):
    gen = rb.generate_blocks_host(0, 4, 4096, 11)
    a = rb.AdaptiveTreeModel(p)
    a.train(gen[4096:8192])
    return [rb.AdaptiveTreeModel(p), a]


def segments(blob):
    """[(model index, comp sizes, crcs or None, streams)] of every segment of a version 2 or 3 container."""
    f = io.BytesIO(blob)
    ver, models, block_len = ct.read_header_any(f)
    out = []
    while True:
        n, last = struct.unpack("<II", f.read(8))
        if n == 0:
            return ver, out
        idx = np.frombuffer(f.read(4 * n), "<u4")
        sizes = np.frombuffer(f.read(4 * n), "<u4")
        crc = np.frombuffer(f.read(4 * n), "<u4") if ver == 3 else None
        streams = [f.read(int(s)) for s in sizes]
        out.append((idx, sizes, crc, streams))


@pytest.mark.parametrize("n_bytes", [1, 4096 * 7, 4096 * 7 + 1234])
def test_round_trips_and_streams_equal_version_2(ctx, n_bytes):
    p = rb.Parameters(8, 14, 16)
    data = _data(n_bytes, n_bytes)
    models = _models(p)
    nb = (n_bytes + 4095) // 4096
    bm = np.arange(nb) % 2
    for write in (lambda cs: _pack_stream(ct.pack_stream, data, rb.AdaptiveTreeModel(p), cs),
                  lambda cs: _pack_stream(ct.pack_stream_models, data, models, cs, bm),
                  lambda cs: _pack_stream(ct.pack_stream_auto, data, models, cs)):
        v3, v2 = write(True), write(False)
        assert v3[4] == 3 and v2[4] in (1, 2)
        assert ct.unpack(v3, context=ctx) == data
        _, seg3 = segments(v3)
        seg2 = segments(v2)[1] if v2[4] == 2 else _v1_segments(v2)
        assert len(seg3) == len(seg2) == (nb + 2) // 3                  # three blocks per segment
        blocks = [data[i:i + 4096] for i in range(0, n_bytes, 4096)]
        k = 0
        for (i3, s3, c3, st3), (i2, s2, _, st2) in zip(seg3, seg2):
            assert st3 == st2 and (s3 == s2).all() and (i3 == i2).all()
            assert list(c3) == [zlib.crc32(b) for b in blocks[k:k + len(st3)]]
            k += len(st3)
    # the one-call writers
    assert ct.unpack(ct.pack(data, rb.AdaptiveTreeModel(p), block_len=4096, context=ctx, checksum=True), ctx) == data
    assert ct.unpack(ct.pack_models(data, models, bm, block_len=4096, context=ctx, checksum=True), ctx) == data
    assert ct.unpack(ct.pack_auto(data, models, block_len=4096, context=ctx, checksum=True), ctx) == data


def _pack_stream(fn, data, models, checksum, bm=None):
    out = io.BytesIO()
    args = (io.BytesIO(data), out, models) + ((bm,) if bm is not None else ())
    fn(*args, block_len=4096, batch_blocks=3, checksum=checksum)
    return out.getvalue()


def _v1_segments(blob):
    f = io.BytesIO(blob)
    ct.read_header(f)
    out = []
    while True:
        n, last = struct.unpack("<II", f.read(8))
        if n == 0:
            return out
        sizes = np.frombuffer(f.read(4 * n), "<u4")
        out.append((np.zeros(n, np.uint32), sizes, None, [f.read(int(s)) for s in sizes]))


def test_default_writes_are_unchanged(ctx):
    """Without checksum the writers give the versions they gave before: 1 from pack, 2 from the others."""
    p = rb.Parameters(8, 14, 16)
    data = _data(20000, 3)
    assert ct.pack(data, rb.AdaptiveTreeModel(p), block_len=4096, context=ctx)[4] == 1
    assert ct.pack_auto(data, _models(p), block_len=4096, context=ctx)[4] == 2


def test_damaged_crc_field_is_refused(ctx):
    p = rb.Parameters(8, 14, 16)
    data = _data(4096 * 5 + 7, 5)
    blob = bytearray(ct.pack(data, rb.AdaptiveTreeModel(p), block_len=4096, context=ctx, checksum=True))
    # header + u32 n_models + one row, then u32 n, u32 last, index[6], sizes[6], crc[6]
    crc_at = ct.HEADER.size + 4 + 257 * 4 + 8 + 2 * 4 * 6
    for block in (0, 5):
        bad = bytearray(blob)
        bad[crc_at + 4 * block + 1] ^= 0x10
        with pytest.raises(ct.ContainerError, match="segment 0, block %d: CRC-32" % block):
            ct.unpack(bytes(bad), context=ctx)
    assert ct.unpack(bytes(blob), context=ctx) == data


@pytest.mark.parametrize("params", [(8, 14, 16), (8, 30, 32)])
def test_bit_flips_never_return_wrong_bytes(ctx, params):
    """Every single-bit flip over the streams of four generator blocks (one per class), decoded as one batch through
    decode_batch_models_crc with slots of exactly the block's length: each variant either passes the version 3 reader's
    checks with exactly the original bytes, or fails them.  A few variants also go through unpack itself."""
    p = rb.Parameters(*params)
    model = rb.AdaptiveTreeModel(p)
    blocks = [rb.generate_blocks_host(i, 1, 1024, 17).tobytes() for i in range(4)]
    data = b"".join(blocks)
    blob = ct.pack(data, model, block_len=1024, context=ctx, checksum=True)
    _, [(idx, sizes, crcs, streams)] = segments(blob)
    variants, owner = [], []
    for b, s in enumerate(streams):
        for bit in range(8 * len(s)):
            v = bytearray(s)
            v[bit >> 3] ^= 1 << (bit & 7)
            variants.append(bytes(v))
            owner.append(b)
    owner = np.array(owner)
    n = len(variants)
    comp = np.frombuffer(b"".join(variants), dtype=np.uint8)
    coff = np.zeros(n + 1, dtype=np.uint64)
    coff[1:] = np.cumsum([len(v) for v in variants])
    roff = np.arange(n + 1, dtype=np.uint64) * np.uint64(1024)
    raw, raw_lens, used, status, crc = ctx.decode_batch_models_crc(comp, coff, roff, [model], None, check=False)
    stored = np.asarray(crcs, dtype=np.uint32)[owner]
    sizes_v = np.asarray(sizes, dtype=np.uint64)[owner]
    lens = np.full(n, 1024, dtype=np.uint64)
    passed = failed = 0
    for i in range(n):
        try:
            ct.check_segment(0, status[i:i + 1], raw_lens[i:i + 1], lens[i:i + 1], used[i:i + 1], sizes_v[i:i + 1],
                             crc[i:i + 1], stored[i:i + 1])
        except ct.ContainerError:
            failed += 1
            continue
        passed += 1
        assert raw[i * 1024:(i + 1) * 1024].tobytes() == blocks[owner[i]], i
    assert failed > 0.5 * n and passed + failed == n
    # the same through unpack: flips in the streams of a whole container
    body = len(blob) - 8 - sum(len(s) for s in streams)
    rng = np.random.default_rng(params[1])
    for bit in rng.choice(8 * sum(len(s) for s in streams), 24, replace=False):
        bad = bytearray(blob)
        bad[body + (bit >> 3)] ^= 1 << (bit & 7)
        try:
            out = ct.unpack(bytes(bad), context=ctx)
        except (ct.ContainerError, rb.Eof):
            continue
        assert out == data
