"""CRC-32 of every block on a B200: `pytest -m gpu`.

The cases of tests/crc32_cases.py (the host emulation runs the same ones in test_crc32_emu.py) through the host form
and the device form, with and without per-block lengths.  The fused calls return exactly what the calls without _crc
return, plus crc[i] == zlib.crc32 of input block i (encode) or of the bytes decoded into slot i (decode), also for
bad model indices, empty blocks, cut streams and full slots; through the pageable staging ring with small pieces; and
on two devices when the machine has them.
"""
import zlib

import numpy as np
import pytest

import crc32_cases as cc
import redux_b200 as rb

pytestmark = pytest.mark.gpu

P = rb.Parameters(8, 14, 16)


@pytest.fixture(scope="module")
def ctx():
    c = rb.Context()
    yield c
    c.close()


def _zlib(data, off, lens=None):
    n = off.size - 1
    ends = off[1:] if lens is None else off[:-1] + lens
    return np.array([zlib.crc32(data[int(off[i]):int(ends[i])].tobytes()) for i in range(n)], dtype=np.uint32)


@pytest.mark.parametrize("case", cc.CASES, ids=lambda c: c.name)
def test_host_form(ctx, case):
    data, off = cc.layout(case)
    assert (ctx.crc32_blocks(data, off) == cc.expected(case)).all()


@pytest.mark.parametrize("case", cc.CASES, ids=lambda c: c.name)
def test_device_form_with_and_without_lengths(ctx, case):
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    s = torch.cuda.current_stream().cuda_stream
    n = len(case.blocks)
    want = cc.expected(case)
    max_len = max(len(b) for b in case.blocks)
    for data, off, lens in (cc.layout(case) + (None,), cc.slots(case)):
        d_in = torch.from_numpy(data.copy()).to(dev)
        d_off = torch.from_numpy(off.astype(np.int64)).to(dev)
        d_lens = None if lens is None else torch.from_numpy(lens.astype(np.int64)).to(dev)
        d_crc = torch.full((n,), 7, dtype=torch.int32, device=dev)
        ctx.crc32_blocks_device(d_in, d_off, n, max_len, d_crc, d_lens=d_lens, device=dev.index, stream=s)
        torch.cuda.synchronize()
        assert (d_crc.cpu().numpy().view(np.uint32) == want).all()


def _models():
    """Three (8,14,16) tree models: fresh, trained on text-like bytes, trained on a run-heavy block."""
    gen = rb.generate_blocks_host(0, 4, 8192, 3)
    a, b = rb.AdaptiveTreeModel(P), rb.AdaptiveTreeModel(P)
    a.train(gen[8192:16384])
    b.train(gen[3 * 8192:])
    return [rb.AdaptiveTreeModel(P), a, b]


def _batch(n=300, seed=5):
    """Generator blocks of ragged lengths, empty blocks among them, back to back at unaligned offsets."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 9000, n)
    lens[::17] = 0
    lens[5] = 70000
    gen = rb.generate_blocks_host(0, n, 9000, seed)
    gen_big = rb.generate_blocks_host(7, 1, 70000, seed)
    blocks = [gen_big.tobytes() if i == 5 else gen[i * 9000:i * 9000 + int(lens[i])].tobytes() for i in range(n)]
    off = np.zeros(n + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(b) for b in blocks])
    return np.frombuffer(b"".join(blocks), dtype=np.uint8), off


def _check_encode_equal(base, fused):
    assert base[0].tobytes() == fused[0].tobytes()
    for x, y in zip(base[1:], fused[1:len(base)]):
        assert (x == y).all()


def test_fused_encode_forms(ctx):
    models = _models()
    data, off = _batch()
    n = off.size - 1
    bm = (np.arange(n) % 3).astype(np.uint32)
    bm[7] = 3                                                  # out of range: empty stream, still a CRC
    base = ctx.encode_batch_models(data, off, models, bm, check=False)
    fused = ctx.encode_batch_models_crc(data, off, models, bm, check=False)
    _check_encode_equal(base, fused)
    assert base[2][7] == rb.INVALID_INPUT and (np.delete(base[2], 7) == rb.OK).all()
    assert (fused[3] == _zlib(data, off)).all()
    with pytest.raises(rb.InvalidInput):
        ctx.encode_batch_models_crc(data, off, models, bm)
    base = ctx.encode_batch_select(data, off, models)
    fused = ctx.encode_batch_select_crc(data, off, models)
    _check_encode_equal(base, fused)
    assert len(set(base[3].tolist())) > 1                      # the choice is not trivial here
    assert (fused[4] == _zlib(data, off)).all()


def _streams(ctx, models, data, off, bm):
    comp, coff, st = ctx.encode_batch_models(data, off, models, bm)
    assert (st == 0).all()
    return comp, coff


def test_fused_decode(ctx):
    """Clean streams, streams cut short (EOF), a slot one byte short (OUT_CAPACITY), a bad model index, empty blocks;
    every output equals decode_batch_models', crc[i] is the CRC of what slot i holds."""
    models = _models()
    data, off = _batch(seed=9)
    n = off.size - 1
    bm = (np.arange(n) % 3).astype(np.uint32)
    comp, coff = _streams(ctx, models, data, off, bm)
    streams = [comp[int(coff[i]):int(coff[i + 1])].tobytes() for i in range(n)]
    lens = (off[1:] - off[:-1]).astype(np.int64)
    cut = [i for i in range(n) if lens[i] > 100][:6]
    for i in cut[:3]:
        streams[i] = streams[i][:len(streams[i]) // 2]         # EOF with a decoded prefix
    cap = lens.copy()
    for i in cut[3:]:
        cap[i] -= 1                                             # OUT_CAPACITY
    bad = bm.copy()
    bad[cut[0] + 1] = 9                                         # out of range
    c2 = np.frombuffer(b"".join(streams), dtype=np.uint8)
    co2 = np.zeros(n + 1, dtype=np.uint64)
    co2[1:] = np.cumsum([len(s) for s in streams])
    roff = np.zeros(n + 1, dtype=np.uint64)
    roff[1:] = np.cumsum(cap)
    for bmx in (bm, bad):
        raw_a = np.full(int(roff[-1]) + 1, 0xEE, dtype=np.uint8)
        raw_b = raw_a.copy()
        base = ctx.decode_batch_models(c2, co2, roff, models, bmx, raw=raw_a, check=False)
        fused = ctx.decode_batch_models_crc(c2, co2, roff, models, bmx, raw=raw_b, check=False)
        for x, y in zip(base[1:], fused[1:4]):
            assert (x == y).all()
        raw_lens = base[1]
        for i in range(n):
            a = base[0][int(roff[i]):int(roff[i]) + int(raw_lens[i])]
            assert a.tobytes() == fused[0][int(roff[i]):int(roff[i]) + int(raw_lens[i])].tobytes()
        assert (fused[4] == _zlib(fused[0], roff, raw_lens)).all()
        st = base[3]
        assert {rb.OK, rb.EOF, rb.OUT_CAPACITY} <= set(st.tolist())
        if bmx is bad:
            assert st[cut[0] + 1] == rb.INVALID_INPUT and fused[4][cut[0] + 1] == 0 and raw_lens[cut[0] + 1] == 0
    # slots exactly one byte short
    roff_short = np.zeros(n + 1, dtype=np.uint64)
    roff_short[1:] = np.cumsum(np.maximum(lens - 1, 0))
    base = ctx.decode_batch_models(comp, coff, roff_short, models, bm, check=False)
    fused = ctx.decode_batch_models_crc(comp, coff, roff_short, models, bm, check=False)
    for x, y in zip(base, fused[:4]):
        assert (x == y).all()
    assert (base[3][lens > 0] == rb.OUT_CAPACITY).all()
    assert (fused[4] == _zlib(fused[0], roff_short, base[1])).all()


def test_pageable_staging_with_small_pieces(ctx):
    """Pageable buffers through the library's pinned ring with 4 KiB pieces and two slots, so the ring wraps many
    times inside every chunk: the same CRCs, streams and bytes."""
    models = _models()
    data, off = _batch(n=600, seed=13)
    bm = (np.arange(off.size - 1) % 3).astype(np.uint32)
    want = _zlib(data, off)
    try:
        ctx.set_staging(True, min_bytes=4096, piece_bytes=4096, slots=2)
        enc = ctx.encode_batch_models_crc(data, off, models, bm)
        dec = ctx.decode_batch_models_crc(enc[0], enc[1], off, models, bm)
        sel = ctx.encode_batch_select_crc(data, off, models)
    finally:
        ctx.set_staging(True, min_bytes=8 << 20, piece_bytes=8 << 20, slots=4)
    plain = ctx.encode_batch_models(data, off, models, bm)
    assert enc[0].tobytes() == plain[0].tobytes() and (enc[3] == want).all()
    assert (dec[3] == 0).all() and dec[0][:int(off[-1])].tobytes() == data.tobytes() and (dec[4] == want).all()
    assert (sel[4] == want).all()


def test_two_devices(ctx):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    models = _models()
    data, off = _batch(seed=21)
    bm = (np.arange(off.size - 1) % 3).astype(np.uint32)
    want = _zlib(data, off)
    one = ctx.encode_batch_models_crc(data, off, models, bm)
    with rb.Context([0, 1]) as two:
        enc = two.encode_batch_models_crc(data, off, models, bm)
        dec = two.decode_batch_models_crc(enc[0], enc[1], off, models, bm)
        sel = two.encode_batch_select_crc(data, off, models)
        host = two.crc32_blocks(data, off)
    assert enc[0].tobytes() == one[0].tobytes() and (enc[3] == want).all()
    assert (dec[4] == want).all() and (sel[4] == want).all() and (host == want).all()
