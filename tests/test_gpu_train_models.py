"""Model training and container version 2 on a B200: `pytest -m gpu`.

The cases of tests/train_models_cases.py (the host emulation runs the same ones in test_train_models_emu.py) against
the reference's get_frequency; the host and device-resident forms against each other; the four generator classes
with samples long enough that many CTAs share one; every trained model coding its own block exactly as the oracle's
compress_trained; and the corpora packed into a version 2 container, walked by hand against the oracle.
"""
import ctypes as C
import io
import struct

import numpy as np
import pytest

import corpora_fixture as cf
import oracle_lib as o
import redux_b200 as rb
import redux_b200.container as ct
import train_models_cases as tmc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = rb.Context()
    yield c
    c.close()


def start_models(case):
    """One start model per sample, trained through Model.train (a fresh one left fresh)."""
    cls = rb.AdaptiveTreeModel if len(case.name) & 1 else rb.AdaptiveLinearModel
    made = []
    for seq in case.starts:
        m = cls(rb.Parameters(*case.params))
        if seq:
            m.train(seq)
        made.append(m)
    return made, [made[k] for k in case.sample_model]


def rows(models):
    return np.stack([m._state().copy() if m.freq is not None else np.ones(m.params.symbol_count, np.uint32)
                     for m in models])


@pytest.mark.parametrize("case", tmc.CASES, ids=lambda c: c.name)
def test_training_equals_reference(ctx, case):
    made, per_sample = start_models(case)
    before = [None if m.freq is None else m.freq.copy() for m in made]
    data, off = tmc.concat(case.samples)
    got = ctx.train_models(data, off, per_sample)
    assert len(got) == len(case.samples)
    assert all(type(g) is type(made[0]) and g.params is made[0].params for g in got)
    want = tmc.expected_rows(case)
    for i, g in enumerate(got):
        assert (g.freq == want[i]).all(), (case.name, i, np.flatnonzero(g.freq != want[i])[:8])
    for m, b in zip(made, before):                   # the start models are not modified
        assert (m.freq is None) if b is None else (m.freq == b).all()


@pytest.mark.parametrize("case", [c for c in tmc.CASES if c.name in ("s3_chunk0", "s8_chunk0", "s16_chunk0",
                                                                    "long_s13_chunk0", "freeze_s8_f12_chunk0")],
                         ids=lambda c: c.name)
def test_host_and_device_forms_agree(ctx, case):
    torch = pytest.importorskip("torch")
    made, per_sample = start_models(case)
    data, off = tmc.concat(case.samples)
    host = rows(ctx.train_models(data, off, per_sample))
    n, nsym = len(case.samples), (1 << case.params[0]) + 1
    d_in = torch.from_numpy(data).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    d_out = torch.full((n, nsym), 0xDEAD, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    ctx.train_models_device(d_in, d_off, n, max(len(x) for x in case.samples), d_out, per_sample, stream=stream)
    torch.cuda.synchronize()
    assert (d_out.cpu().numpy().view(np.uint32) == host).all()


def generator_samples(n, length, seed=0x5EED202610190000):
    data = rb.generate_blocks_host(0, n, length, seed)
    return data, np.arange(n + 1, dtype=np.uint64) * np.uint64(length)


@pytest.mark.parametrize("params", [(8, 30, 32), (8, 14, 16), (8, 22, 24)])
def test_generator_classes_and_long_samples(ctx, params):
    """All four generator classes (block index & 3), 320 KiB per sample: 20 CTAs per sample at (8,30,32), where
    nothing freezes early.  One shared start model, fresh and then trained."""
    n, length = 8, 320 << 10
    data, off = generator_samples(n, length)
    for start in (rb.AdaptiveTreeModel(rb.Parameters(*params)),
                  rb.AdaptiveTreeModel(rb.Parameters(*params)).train(data[:3000])):
        got = ctx.train_models(data, off, start)
        for i in range(n):
            want = rb.AdaptiveTreeModel(rb.Parameters(*params))
            if start.freq is not None:
                want.freq = start.freq.copy()
            want.train(data[i * length:(i + 1) * length])
            assert (got[i].freq == want.freq).all(), (params, i)


@pytest.mark.parametrize("params", [(8, 30, 32), (8, 14, 16), (8, 12, 18)])
def test_trained_models_code_their_blocks_as_the_oracle(ctx, params):
    """Train one model per block on the device, then encode every block from its own model: each stream is the
    oracle's compress_trained of the block with the block itself as the training sequence."""
    n, length = 8, 64 << 10
    data, off = generator_samples(n, length, seed=0x5EED202610190001)
    models = ctx.train_models(data, off, rb.AdaptiveLinearModel(rb.Parameters(*params)))
    comp, coff, status = ctx.encode_batch_models(data, off, models, np.arange(n))
    assert (status == 0).all()
    for i in range(n):
        block = data[i * length:(i + 1) * length]
        rc, want, _, _ = o.compress_trained(block, block, o.LINEAR, params)
        assert rc == 0 and comp[int(coff[i]):int(coff[i + 1])].tobytes() == want, (params, i)


def test_errors_before_launch(ctx):
    p = rb.Parameters(8, 14, 16)
    data, off = generator_samples(2, 64)
    bad = rb.AdaptiveTreeModel(p)
    bad.freq = np.ones(257, dtype=np.uint32)
    bad.freq[5] = 0
    with pytest.raises(rb.InvalidInput, match="model row 1"):
        ctx.train_models(data, off, [rb.AdaptiveTreeModel(p), bad])
    full = rb.AdaptiveTreeModel(p)
    full.freq = np.full(257, 64, dtype=np.uint32)      # total 16,448 > freq_max
    with pytest.raises(rb.InvalidInput, match="model row 0"):
        ctx.train_models(data, off, full)
    out = np.zeros((2, 257), dtype=np.uint32)
    table = np.ones((1, 257), dtype=np.uint32)
    sm = np.array([0, 1], dtype=np.uint32)
    pc = p._c()
    rc = rb.lib().redux_train_models(ctx._h, C.byref(pc), table.ctypes.data, 1, sm.ctypes.data, data.ctypes.data,
                                     off.ctypes.data, 2, out.ctypes.data)
    assert rc == rb.INVALID_INPUT and b"sample 1" in rb.lib().redux_ctx_last_error(ctx._h)
    with pytest.raises(rb.Unsupported):
        ctx.train_models(data, off, rb.AdaptiveTreeModel(rb.Parameters(17, 20, 24)))
    assert ctx.train_models(data[:0], np.zeros(1, dtype=np.uint64), rb.AdaptiveTreeModel(p)) == []


# --------------------------------------------------------------------------- container version 2
def test_container_v2_from_gpu_trained_models():
    """The corpora back to back in 64 KiB blocks; one model per file, trained on the device from the file's first
    64 KiB, plus a fresh model for every fifth block.  The container decodes to the input, and walked by hand, every
    block's stream is the oracle's compress_trained of that block with its model's training sequence."""
    params, L = (8, 22, 24), 65536
    files = cf.corpora()
    names = sorted(files)
    data = b"".join(files[k] for k in names)
    ctx = rb.Context()
    sample = [files[k][:L] for k in names]
    soff = np.zeros(len(names) + 1, dtype=np.uint64)
    np.cumsum([len(x) for x in sample], out=soff[1:])
    models = ctx.train_models(np.frombuffer(b"".join(sample), dtype=np.uint8), soff,
                              rb.AdaptiveTreeModel(rb.Parameters(*params)))
    models.append(rb.AdaptiveTreeModel(rb.Parameters(*params)))            # fresh, last row
    fresh = len(models) - 1
    starts = np.cumsum([0] + [len(files[k]) for k in names])
    n_blocks = (len(data) + L - 1) // L
    bm = [fresh if b % 5 == 4 else int(np.searchsorted(starts, b * L, side="right") - 1) for b in range(n_blocks)]
    out = io.BytesIO()
    ct.pack_stream_models(io.BytesIO(data), out, models, bm, block_len=L, batch_blocks=64, context=ctx)
    blob = out.getvalue()
    assert ct.unpack(blob, context=ctx) == data
    # walk the file
    ver, got_models, block_len = ct.read_header_any(io.BytesIO(blob))
    assert ver == 2 and block_len == L and len(got_models) == len(models)
    for g, m in zip(got_models, models):
        assert (g._state() == m._state()).all()
    pos, blk = ct.HEADER.size + 4 + 4 * len(models) * 257, 0
    while True:
        n, last = struct.unpack_from("<II", blob, pos)
        pos += 8
        if n == 0:
            break
        idx = np.frombuffer(blob, dtype="<u4", count=n, offset=pos)
        pos += 4 * n
        sizes = np.frombuffer(blob, dtype="<u4", count=n, offset=pos)
        pos += 4 * n
        for i in range(n):
            assert idx[i] == bm[blk]
            block = data[blk * L:(blk + 1) * L]
            train = sample[idx[i]] if idx[i] != fresh else b""
            rc, want, _, _ = o.compress_trained(block, np.frombuffer(train, dtype=np.uint8), o.TREE, params)
            assert rc == 0 and blob[pos:pos + int(sizes[i])] == want, blk
            pos += int(sizes[i])
            blk += 1
    assert blk == n_blocks and pos == len(blob)
    for cut in (10, ct.HEADER.size + 100, len(blob) // 2, len(blob) - 9):
        with pytest.raises((rb.Eof, ct.ContainerError)) as e:
            ct.unpack(blob[:cut], context=ctx)
        assert cut == 10 or e.type is rb.Eof
    ctx.close()
