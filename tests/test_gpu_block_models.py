"""Blocks of one launch that start from different trained models, on a B200: `pytest -m gpu`.

The cases of tests/block_models_cases.py (the host emulation runs the same ones in test_block_models_emu.py): encode
through redux_encode_batch_models, decode through redux_decode_batch_device_models, each block against the oracle with
its own model, the decoder's error exits under mixed models, out-of-range row indices, and the kernels
redux_debug_launched_kernels reports.  Also: one model through the new calls equals the _ex calls byte for byte and
kernel for kernel; the host-buffer, pageable-staged and device-resident forms agree; two devices agree with one.
"""
import numpy as np
import pytest

import block_models_cases as bmc
import redux_b200 as rb

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = rb.Context()
    c.set_schedule(rb.SCHED_AUTO)
    yield c
    c.close()


def models_for(case):
    """The case's models as the Python API takes them: trained through Model.train, a fresh model left untouched."""
    cls = rb.AdaptiveTreeModel if len(case.name) & 1 else rb.AdaptiveLinearModel
    out = []
    for kind, t in zip(case.kinds, bmc.training(case)):
        m = cls(rb.Parameters(*case.params))
        if kind != "ones":
            m.train(t)
        out.append(m)
    return out


def _offsets(lens):
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(np.array(lens, dtype=np.uint64), out=off[1:])
    return off


class GpuBackend:
    """Encode through the host-buffer call, decode through the device-resident one (the bytes around the slots are
    device memory the test controls)."""

    def __init__(self, ctx, case):
        self.ctx, self.case = ctx, case
        self.models = models_for(case)
        ctx.launched_kernels(reset=True)

    def encode(self, blocks, table, bm):
        assert (rb._model_table(self.models)[2] == table).all()
        off = _offsets([len(b) for b in blocks])
        data = np.frombuffer(b"".join(blocks), dtype=np.uint8)
        out, out_off, status = self.ctx.encode_batch_models(data, off, self.models, bm, check=False)
        return [out[int(out_off[i]):int(out_off[i + 1])].tobytes() for i in range(len(blocks))], status

    def decode(self, comp, coff, raw, roff, max_len, table, bm):
        import torch
        n = coff.size - 1
        d_comp = torch.from_numpy(comp).cuda()
        d_coff = torch.from_numpy(coff.astype(np.int64)).cuda()
        d_raw = torch.from_numpy(raw).cuda()
        d_roff = torch.from_numpy(roff.astype(np.int64)).cuda()
        d_bm = torch.from_numpy(bm.astype(np.int32)).cuda()
        d_len = torch.full((n,), -1, dtype=torch.int64, device="cuda")
        d_cons = torch.full((n,), -1, dtype=torch.int64, device="cuda")
        d_st = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        self.ctx.decode_batch_device_models(d_comp, d_coff, n, max_len, d_raw, d_roff, d_len, d_cons, d_st, self.models,
                                            d_bm, device=torch.cuda.current_device(),
                                            stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        return d_raw.cpu().numpy(), d_len.cpu().numpy(), d_cons.cpu().numpy(), d_st.cpu().numpy()

    def kernels(self):
        return self.ctx.launched_kernels(reset=True)


@pytest.mark.parametrize("case", bmc.CASES, ids=lambda c: c.name)
def test_block_models_on_the_device(ctx, case):
    bmc.check_case(case, GpuBackend(ctx, case))


@pytest.mark.parametrize("case", [bmc.CASES[0], bmc.CASES[7], bmc.CASES[-2]], ids=lambda c: c.name)
def test_out_of_range_model_index_on_the_device(ctx, case):
    bmc.check_bad_index(case, GpuBackend(ctx, case))


def _case(name):
    return next(c for c in bmc.CASES if c.name == name)


def _batch(case):
    blocks = bmc.blocks_for(case)
    data = np.frombuffer(b"".join(blocks), dtype=np.uint8)
    bm = np.arange(len(blocks), dtype=np.uint32) % np.uint32(len(case.kinds))
    return blocks, data, _offsets([len(b) for b in blocks]), bm


@pytest.mark.parametrize("name", ["narrow_stg", "wide_u32_c32", "generic_c34"])
def test_one_model_equals_the_ex_calls(ctx, name):
    """n_models == 1 (block_model NULL) is the _ex call: same streams, same decoded bytes, same kernels."""
    case = _case(name)
    model = models_for(case)[-1]
    blocks, data, off, _ = _batch(case)
    ctx.launched_kernels(reset=True)
    a = ctx.encode_batch(data, off, model)
    ka = ctx.launched_kernels(reset=True)
    b = ctx.encode_batch_models(data, off, [model], None)
    kb = ctx.launched_kernels(reset=True)
    assert ka == kb == {case.enc}
    assert (a[1] == b[1]).all() and a[0].tobytes() == b[0].tobytes()
    da = ctx.decode_batch(a[0], a[1], off, model)
    ka = ctx.launched_kernels(reset=True)
    db = ctx.decode_batch_models(a[0], a[1], off, [model], None)
    kb = ctx.launched_kernels(reset=True)
    assert ka == kb == {case.dec}
    assert (da[0] == db[0]).all() and (da[1] == db[1]).all() and (da[2] == db[2]).all()


@pytest.mark.parametrize("name", ["wided_u32_c22", "generic_s4"])
def test_host_staged_and_device_forms_agree(ctx, name):
    """The host-buffer call with pageable buffers handed to the driver, the same through the library's pinned staging
    ring (several chunks, each with its slice of the index), and the device-resident call give the same streams and
    the same decoded blocks."""
    import torch
    case = _case(name)
    models = models_for(case)
    blocks, data, off, bm = _batch(case)
    try:
        ctx.set_staging(False)
        host = ctx.encode_batch_models(data, off, models, bm)
        host_dec = ctx.decode_batch_models(host[0], host[1], off, models, bm)
        ctx.set_staging(True, min_bytes=4096, piece_bytes=4096, slots=2)
        staged = ctx.encode_batch_models(data, off, models, bm)
        staged_dec = ctx.decode_batch_models(host[0], host[1], off, models, bm)
    finally:
        ctx.set_staging(True, min_bytes=8 << 20, piece_bytes=8 << 20, slots=4)
    assert host[0].tobytes() == staged[0].tobytes() and (host[1] == staged[1]).all()
    assert (host_dec[0] == staged_dec[0]).all() and (host_dec[3] == 0).all() and (staged_dec[3] == 0).all()
    # device-resident
    n = len(blocks)
    dev = torch.device("cuda", torch.cuda.current_device())
    s = torch.cuda.current_stream().cuda_stream
    d_in = torch.zeros(data.size + 64, dtype=torch.uint8, device=dev)
    d_in[:data.size] = torch.from_numpy(data.copy()).to(dev)
    d_off = torch.from_numpy(off.astype(np.int64)).to(dev)
    d_bm = torch.from_numpy(bm.astype(np.int32)).to(dev)
    cap = host[0].size + 64
    d_out = torch.zeros(cap, dtype=torch.uint8, device=dev)
    d_ooff = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    d_st = torch.full((n,), -1, dtype=torch.int32, device=dev)
    max_len = max(len(b) for b in blocks)
    ctx.encode_batch_device_models(d_in, d_off, n, max_len, d_out, cap, d_ooff, d_st, models, d_bm, device=dev.index,
                                   stream=s)
    torch.cuda.synchronize()
    assert (d_st.cpu().numpy() == 0).all()
    assert (d_ooff.cpu().numpy().astype(np.uint64) == host[1]).all()
    assert d_out[:host[0].size].cpu().numpy().tobytes() == host[0].tobytes()
    d_raw = torch.zeros(int(off[-1]) + 64, dtype=torch.uint8, device=dev)
    d_len = torch.zeros(n, dtype=torch.int64, device=dev)
    d_cons = torch.zeros(n, dtype=torch.int64, device=dev)
    ctx.decode_batch_device_models(d_out, d_ooff, n, max_len, d_raw, d_off, d_len, d_cons, d_st, models, d_bm,
                                   device=dev.index, stream=s)
    torch.cuda.synchronize()
    assert (d_st.cpu().numpy() == 0).all()
    assert (d_raw[:int(off[-1])].cpu().numpy() == host_dec[0][:int(off[-1])]).all()
    assert (d_len.cpu().numpy().astype(np.uint64) == host_dec[1]).all()


def test_two_devices_give_the_same_bytes(ctx):
    """Each device builds the model table and codes its shard with its own slice of the index."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    case = _case("wide_u32_c21")
    models = models_for(case)
    blocks, data, off, bm = _batch(case)
    one = ctx.encode_batch_models(data, off, models, bm)
    with rb.Context([0, 1]) as two:
        both = two.encode_batch_models(data, off, models, bm)
        dec = two.decode_batch_models(both[0], both[1], off, models, bm)
    assert one[0].tobytes() == both[0].tobytes() and (one[1] == both[1]).all()
    assert (dec[3] == 0).all() and dec[0][:int(off[-1])].tobytes() == data.tobytes()


def test_invalid_tables_are_refused_before_any_work(ctx):
    case = _case("narrow")
    models = models_for(case)
    blocks, data, off, bm = _batch(case)
    with pytest.raises(rb.InvalidInput, match="block_model"):
        ctx.encode_batch_models(data, off, models, None)
    with pytest.raises(rb.InvalidInput):
        ctx.encode_batch_models(data, off, [], bm)
    with pytest.raises(rb.InvalidInput, match="kinds"):
        ctx.encode_batch_models(data, off, [rb.AdaptiveTreeModel(rb.Parameters(8, 12, 18)),
                                            rb.AdaptiveLinearModel(rb.Parameters(8, 12, 18))], bm % 2)
    with pytest.raises(rb.InvalidInput, match="Parameters"):
        ctx.encode_batch_models(data, off, [rb.AdaptiveTreeModel(rb.Parameters(8, 12, 18)),
                                            rb.AdaptiveTreeModel(rb.Parameters(8, 12, 19))], bm % 2)
    bad = type(models[0])(rb.Parameters(8, 12, 18)).train([1, 2, 3])
    bad.freq[7] = 0
    with pytest.raises(rb.InvalidInput, match="model row 2: frequency below 1"):
        ctx.encode_batch_models(data, off, models[:2] + [bad], bm % 3)
    bad.freq[7] = 5000
    with pytest.raises(rb.InvalidInput, match="model row 2: total exceeds freq_max"):
        ctx.decode_batch_models(data, off, off, models[:2] + [bad], bm % 3)
