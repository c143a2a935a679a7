"""Model selection on a B200: `pytest -m gpu`.

The cases of tests/select_models_cases.py (the host emulation runs the same ones in test_select_models_emu.py) against
the float64 references, in the host and the device-resident form; the fused encode against selection followed by
redux_encode_batch_models, on pinned, registered and pageable buffers and on two devices; chosen streams against the
oracle's compress_trained; and pack_auto of the corpora.
"""
import io
import struct

import numpy as np
import pytest

import corpora_fixture as cf
import oracle_lib as o
import redux_b200 as rb
import redux_b200.container as ct
import select_models_cases as smc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = rb.Context()
    yield c
    c.close()


def models_of(params, rows, cls=rb.AdaptiveTreeModel):
    out = []
    for r in rows:
        m = cls(rb.Parameters(*params))
        if not (np.asarray(r) == 1).all():
            m.freq = np.ascontiguousarray(r, dtype=np.uint32).copy()
        out.append(m)
    return out


def device_select(ctx, data, off, models, max_len):
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    n, k = off.size - 1, len(models)
    d_in = torch.from_numpy(np.concatenate([data, np.zeros(64, np.uint8)])).to(dev)
    d_off = torch.from_numpy(off.astype(np.int64)).to(dev)
    d_bm = torch.full((n,), -1, dtype=torch.int32, device=dev)
    d_cost = torch.zeros((n, k), dtype=torch.float64, device=dev)
    ctx.select_models_device(d_in, d_off, n, max_len, models, d_bm, d_cost, device=dev.index,
                             stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return d_bm.cpu().numpy().view(np.uint32), d_cost.cpu().numpy()


@pytest.mark.parametrize("case", smc.CASES, ids=lambda c: c.name)
def test_costs_and_choices_match_the_reference(ctx, case):
    """Host form, device form and a second host call: bit-identical costs and choices, within the tolerance of the
    reference; the choice is the reference argmin wherever the reference separates the best from the rest."""
    models = models_of(case.params, case.rows, rb.AdaptiveTreeModel if len(case.name) & 1 else rb.AdaptiveLinearModel)
    data, off = smc.concat(case.blocks)
    data = data[:int(off[-1])]
    choice, cost = ctx.select_models(data, off, models, costs=True)
    ref = smc.reference_costs(case)
    smc.check_choice(case, ref, cost, choice)
    again = ctx.select_models(data, off, models, costs=True)
    assert (again[0] == choice).all() and again[1].tobytes() == cost.tobytes()
    assert (ctx.select_models(data, off, models) == choice).all()
    d_choice, d_cost = device_select(ctx, data, off, models, max(len(b) for b in case.blocks))
    assert (d_choice == choice).all() and d_cost.tobytes() == cost.tobytes()


@pytest.mark.parametrize("case", smc.CASES, ids=lambda c: c.name)
def test_fused_encode_equals_select_then_encode(ctx, case):
    models = models_of(case.params, case.rows)
    data, off = smc.concat(case.blocks)
    data = data[:int(off[-1])]
    choice = ctx.select_models(data, off, models)
    comp, coff, status, bm = ctx.encode_batch_select(data, off, models)
    want = ctx.encode_batch_models(data, off, models, choice)
    assert (bm == choice).all() and (status == 0).all()
    assert comp.tobytes() == want[0].tobytes() and (coff == want[1]).all()
    raw, lens, _, st = ctx.decode_batch_models(comp, coff, off, models, bm)
    assert (st == 0).all()
    s = case.params[0]
    for i, b in enumerate(case.blocks):             # a trailing partial symbol is not coded (the reference's reader)
        if len(b) * 8 % s == 0:
            assert raw[int(off[i]):int(off[i]) + len(b)].tobytes() == b, (case.name, i)


def generator_batch(params, n, length, seed=0x5E1EC72026102200):
    """n generator blocks of `length` bytes and candidates: fresh plus one model per class trained on the device from
    a 64 KiB sample of that class."""
    ctx = rb.Context()
    data = rb.generate_blocks_host(0, n, length, seed)
    sample = rb.generate_blocks_host(1 << 20, 4, 65536, seed + 1)        # block index & 3 is the class
    soff = np.arange(5, dtype=np.uint64) * np.uint64(65536)
    models = [rb.AdaptiveTreeModel(rb.Parameters(*params))]
    models += ctx.train_models(sample, soff, rb.AdaptiveTreeModel(rb.Parameters(*params)))
    ctx.close()
    return data, np.arange(n + 1, dtype=np.uint64) * np.uint64(length), models


@pytest.mark.parametrize("params", [(8, 14, 16), (8, 30, 32)])
def test_fused_encode_on_pinned_registered_and_pageable_buffers(ctx, params):
    """Many chunks of the pipeline: the index and the streams equal select_models + encode_batch_models whether the
    caller's buffers are pinned, registered or pageable (staged through the library's ring)."""
    data, off, models = generator_batch(params, 3000, 4096)
    choice = ctx.select_models(data, off, models)
    assert len(set(choice.tolist())) > 1
    want = ctx.encode_batch_models(data, off, models, choice)
    cap = want[0].size + 4096
    # pinned
    hin, hout = rb.HostBuffer(data.size), rb.HostBuffer(cap)
    hin.array[:] = data
    got = ctx.encode_batch_select(hin.array, off, models, out=hout.array)
    assert (got[3] == choice).all() and got[0].tobytes() == want[0].tobytes() and (got[1] == want[1]).all()
    hin.close(); hout.close()
    # registered
    rin, rout = data.copy(), np.zeros(cap, dtype=np.uint8)
    rb.host_register(rin); rb.host_register(rout)
    try:
        got = ctx.encode_batch_select(rin, off, models, out=rout)
        assert (got[3] == choice).all() and got[0].tobytes() == want[0].tobytes() and (got[1] == want[1]).all()
    finally:
        rb.host_unregister(rin); rb.host_unregister(rout)
    # pageable, through the staging ring in small pieces
    try:
        ctx.set_staging(True, min_bytes=4096, piece_bytes=1 << 20, slots=2)
        got = ctx.encode_batch_select(data.copy(), off, models, out=np.zeros(cap, dtype=np.uint8))
    finally:
        ctx.set_staging(True, min_bytes=8 << 20, piece_bytes=8 << 20, slots=4)
    assert (got[3] == choice).all() and got[0].tobytes() == want[0].tobytes() and (got[1] == want[1]).all()
    # a sample of blocks against the oracle, from the chosen row
    for i in range(0, 3000, 97):
        r = models[choice[i]]._state()
        train = np.repeat(np.arange(r.size, dtype=np.uint64), r.astype(np.int64) - 1)
        rc, stream, _, _ = o.compress_trained(data[i * 4096:(i + 1) * 4096], train, o.TREE, params)
        assert rc == 0 and got[0][int(got[1][i]):int(got[1][i + 1])].tobytes() == stream, i
    raw, _, _, st = ctx.decode_batch_models(got[0], got[1], off, models, got[3])
    assert (st == 0).all() and raw[:data.size].tobytes() == data.tobytes()


def test_two_devices_give_the_same_choice_and_bytes(ctx):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    data, off, models = generator_batch((8, 14, 16), 1000, 4096)
    one = ctx.encode_batch_select(data, off, models)
    with rb.Context([0, 1]) as two:
        both = two.encode_batch_select(data, off, models)
    assert (one[3] == both[3]).all() and one[0].tobytes() == both[0].tobytes() and (one[1] == both[1]).all()


def test_pack_auto_of_the_corpora():
    """One model per file trained from its first 64 KiB plus a fresh one: pack_auto round-trips and stores the
    indices select_models gives."""
    params, L = (8, 14, 16), 65536
    files = cf.corpora()
    names = sorted(files)
    data = b"".join(files[k] for k in names)
    ctx = rb.Context()
    sample = [files[k][:L] for k in names]
    soff = np.zeros(len(names) + 1, dtype=np.uint64)
    np.cumsum([len(x) for x in sample], out=soff[1:])
    models = [rb.AdaptiveTreeModel(rb.Parameters(*params))]
    models += ctx.train_models(np.frombuffer(b"".join(sample), dtype=np.uint8), soff, models[0])
    blob = ct.pack_auto(data, models, block_len=L, context=ctx)
    assert ct.unpack(blob, context=ctx) == data
    n = (len(data) + L - 1) // L
    off = np.minimum(np.arange(n + 1, dtype=np.uint64) * np.uint64(L), np.uint64(len(data)))
    want = ctx.select_models(np.frombuffer(data, dtype=np.uint8), off, models)
    pos = ct.HEADER.size + 4 + 4 * len(models) * 257
    cnt, _ = struct.unpack_from("<II", blob, pos)
    assert cnt == n
    assert (np.frombuffer(blob, dtype="<u4", count=n, offset=pos + 8) == want).all()
    ctx.close()


def test_errors_before_launch(ctx):
    import torch
    p = rb.Parameters(8, 14, 16)
    data, off = np.zeros(64, np.uint8), np.array([0, 64], np.uint64)
    bad = rb.AdaptiveTreeModel(p)
    bad.freq = np.ones(257, dtype=np.uint32)
    bad.freq[5] = 0
    with pytest.raises(rb.InvalidInput, match="model row 1"):
        ctx.select_models(data, off, [rb.AdaptiveTreeModel(p), bad])
    with pytest.raises(rb.InvalidInput, match="model row 1"):
        ctx.encode_batch_select(data, off, [rb.AdaptiveTreeModel(p), bad])
    with pytest.raises(rb.Unsupported):
        ctx.select_models(data, off, [rb.AdaptiveTreeModel(rb.Parameters(17, 20, 24))])
    d = torch.zeros(64, dtype=torch.uint8, device="cuda")
    with pytest.raises(rb.Unsupported, match="2\\^31"):
        ctx.select_models_device(d, d, 1, 1 << 31, [rb.AdaptiveTreeModel(p)], d)
    assert ctx.select_models(data[:0], np.zeros(1, dtype=np.uint64), [rb.AdaptiveTreeModel(p)]).size == 0
