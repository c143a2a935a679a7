"""Learning start models on a B200: `pytest -m gpu`.

The rows of a round against the exact reference of tests/build_models_cases.py, the returned choice against
select_models on the returned table, determinism across calls and forms, chaining of rounds, and pack_learned /
pack_stream_learned round trips through the unchanged unpack, with sampled streams against the oracle.
"""
import io
import struct

import numpy as np
import pytest

import build_models_cases as bmc
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


def model_of(params, cls=rb.AdaptiveTreeModel):
    return cls(rb.Parameters(*params))


def concat(case):
    data, off = smc.concat(case.blocks)
    return data[:int(off[-1])], off


def table_of(models):
    return np.stack([m._state() for m in models])


@pytest.mark.parametrize("case", bmc.CASES, ids=lambda c: c.name)
def test_one_round_rows_equal_the_reference(ctx, case):
    """iterations=1: row k is row(aggregate(init), T_l*) bit for bit, and l* is within tolerance of the reference's
    best level; row 0 is fresh."""
    s, f, _ = case.params
    data, off = concat(case)
    models, bm, totals = ctx.build_models(data, off, model_of(case.params), case.K, 1, case.init)
    tab = table_of(models)
    assert tab.shape == (case.K + 1, (1 << s) + 1) and (tab[0] == 1).all()
    T = bmc.ladder(s, f)
    S, tol, cand = bmc.ladder_sums(case, case.init)
    for k in range(1, case.K + 1):
        lstar = T.index(int(tab[k].astype(np.int64).sum()))
        assert (tab[k] == cand[k - 1][lstar]).all(), (case.name, k, lstar)
        assert S[k - 1][lstar] <= S[k - 1].min() + 2 * tol[k - 1], (case.name, k, S[k - 1].tolist())
        if not (case.init == k).any():
            assert lstar == 0
    assert totals.shape == (1,)


def check_result(ctx, data, off, params, K, models, bm, totals):
    choice, cost = ctx.select_models(data, off, models, costs=True)
    assert (bm == choice).all()
    best = int(np.argmin(totals))
    chosen = cost[np.arange(choice.size), choice].sum()
    assert abs(totals[best] - chosen) <= 1e-9 * abs(chosen)
    _, fresh_cost = ctx.select_models(data, off, [model_of(params)], costs=True)
    fresh_total = fresh_cost.sum()
    assert (totals <= fresh_total * (1 + 1e-9)).all(), (totals.tolist(), fresh_total)
    assert all(totals[best] < t for t in totals[:best]) and all(totals[best] <= t for t in totals[best:])


@pytest.mark.parametrize("K,iterations", [(1, 1), (2, 3), (4, 5), (7, 2)])
def test_choice_equals_select_models_and_totals_hold(ctx, K, iterations):
    case = bmc.CASES[3]
    data, off = concat(case)
    models, bm, totals = ctx.build_models(data, off, model_of(case.params), K, iterations)
    assert totals.shape == (iterations,)
    check_result(ctx, data, off, case.params, K, models, bm, totals)


@pytest.mark.parametrize("case", bmc.CASES[:3], ids=lambda c: c.name)
def test_small_widths(ctx, case):
    data, off = concat(case)
    models, bm, totals = ctx.build_models(data, off, model_of(case.params, rb.AdaptiveLinearModel), case.K, 4,
                                          case.init)
    assert all(isinstance(m, rb.AdaptiveLinearModel) for m in models)
    check_result(ctx, data, off, case.params, case.K, models, bm, totals)


def test_rounds_chain(ctx):
    case = bmc.CASES[3]
    data, off = concat(case)
    m = model_of(case.params)
    _, _, two = ctx.build_models(data, off, m, case.K, 2, case.init)
    _, bm1, _ = ctx.build_models(data, off, m, case.K, 1, case.init)
    _, _, again = ctx.build_models(data, off, m, case.K, 1, bm1)
    assert two[1].tobytes() == again[0].tobytes()


def test_calls_and_forms_agree_bit_for_bit(ctx):
    import torch
    case = bmc.CASES[4]
    data, off = concat(case)
    m = model_of(case.params)
    K, it = case.K, 4
    one = ctx.build_models(data, off, m, K, it)
    two = ctx.build_models(data, off, m, K, it)
    assert (table_of(one[0]) == table_of(two[0])).all() and (one[1] == two[1]).all()
    assert one[2].tobytes() == two[2].tobytes()
    dev = torch.device("cuda", torch.cuda.current_device())
    d_in = torch.from_numpy(np.concatenate([data, np.zeros(64, np.uint8)])).to(dev)
    d_off = torch.from_numpy(off.astype(np.int64)).to(dev)
    d_tab = torch.zeros((K + 1, 257), dtype=torch.int32, device=dev)
    d_bm = torch.full((off.size - 1,), -1, dtype=torch.int32, device=dev)
    d_tot = torch.zeros(it, dtype=torch.float64, device=dev)
    ctx.build_models_device(d_in, d_off, off.size - 1, 4096 + 2, m, K, d_tab, d_bm, d_tot, iterations=it,
                            device=dev.index, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert (d_tab.cpu().numpy().view(np.uint32) == table_of(one[0])).all()
    assert (d_bm.cpu().numpy().view(np.uint32) == one[1]).all()
    assert d_tot.cpu().numpy().tobytes() == one[2].tobytes()


@pytest.mark.parametrize("params", [(8, 14, 16), (8, 30, 32)])
def test_generator_batches(ctx, params):
    case = bmc.generator_case(params, 512, 16384, 4)
    data, off = concat(case)
    models, bm, totals = ctx.build_models(data, off, model_of(params), 4, 6)
    check_result(ctx, data, off, params, 4, models, bm, totals)
    assert len(set(bm.tolist())) > 1


def test_argument_errors(ctx):
    p = (8, 14, 16)
    data, off = np.zeros(64, np.uint8), np.array([0, 32, 64], np.uint64)
    with pytest.raises(rb.InvalidInput, match="block 1"):
        ctx.build_models(data, off, model_of(p), 2, 1, [0, 3])
    trained = model_of(p).train([1, 2, 3])
    with pytest.raises(rb.InvalidInput):
        ctx.build_models(data, off, trained, 2)
    with pytest.raises(rb.InvalidInput):
        ctx.build_models(data, off, model_of(p), 0)


def _corpora():
    files = cf.corpora()
    return b"".join(files[k] for k in sorted(files))


@pytest.mark.parametrize("checksum", [False, True])
def test_pack_learned_round_trips(ctx, checksum):
    data = _corpora()
    L, K = 4096, 8
    blob = ct.pack_learned(data, model_of((8, 30, 32)), k=K, iterations=3, block_len=L, context=ctx,
                           checksum=checksum)
    assert blob[4] == (3 if checksum else 2)
    assert ct.unpack(blob, context=ctx) == data
    ver, models, _ = ct.read_header_any(io.BytesIO(blob))
    tab = table_of(models)
    assert tab.shape[0] == K + 1 and (tab[0] == 1).all()
    # streamed, several segments: the table is learned from the first segment only
    out = io.BytesIO()
    raw, size = ct.pack_stream_learned(io.BytesIO(data), out, model_of((8, 14, 16)), k=4, iterations=2, block_len=L,
                                       batch_blocks=64, context=ctx, checksum=checksum)
    blob = out.getvalue()
    assert raw == len(data) and size == len(blob) and ct.unpack(blob, context=ctx) == data
    _, models, _ = ct.read_header_any(io.BytesIO(blob))
    head = np.frombuffer(data[:64 * L], dtype=np.uint8)
    n0 = (head.size + L - 1) // L
    off0 = np.minimum(np.arange(n0 + 1, dtype=np.uint64) * np.uint64(L), np.uint64(head.size))
    want, _, _ = ctx.build_models(head, off0, model_of((8, 14, 16)), 4, 2)
    assert (table_of(models) == table_of(want)).all()
    # sampled streams of the first segment against the oracle, from the stored rows
    pos = ct.HEADER.size + 4 + 4 * len(models) * 257
    n, _ = struct.unpack_from("<II", blob, pos)
    idx = np.frombuffer(blob, dtype="<u4", count=n, offset=pos + 8)
    sizes = np.frombuffer(blob, dtype="<u4", count=n, offset=pos + 8 + 4 * n).astype(np.int64)
    start = pos + 8 + 8 * n + (4 * n if checksum else 0)
    coff = np.concatenate([[0], np.cumsum(sizes)]) + start
    for i in range(0, n, 7):
        r = models[int(idx[i])]._state()
        train = np.repeat(np.arange(r.size, dtype=np.uint64), r.astype(np.int64) - 1)
        rc, stream, _, _ = o.compress_trained(data[i * L:(i + 1) * L], train, o.TREE, (8, 14, 16))
        assert rc == 0 and blob[coff[i]:coff[i + 1]] == stream, i
