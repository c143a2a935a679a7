"""Every kernel the dispatcher can launch, against the oracle, on a B200: `pytest -m gpu`.

One row of tests/kernel_matrix_cases.py per (parameters, model, schedule, block shapes); each row encodes its blocks
(empty, 1 / 15 / 16 / 17 bytes, one-symbol runs, the row's long blocks), decodes them at exact capacity, then decodes
the decoder's error exits (cuts, garbage, trailing garbage, a slot one byte short, both at once) between good
neighbours in adjacent slots, and checks with redux_debug_launched_kernels that the kernels it names ran.  All rows
share one context and run in a fixed shuffled order, so that a launch depending on workspace, reciprocal-table or
shared-memory state left by the previous plan shows up as a mismatch.
"""
import random

import numpy as np
import pytest

import kernel_matrix_cases as km
import redux_b200 as rb

pytestmark = pytest.mark.gpu

SCHED = {"lane": rb.SCHED_LANE, "warp": rb.SCHED_WARP, "split": rb.SCHED_SPLIT}
ORDER = list(km.CASES)
random.Random(20261020).shuffle(ORDER)


@pytest.fixture(scope="module")
def ctx():
    c = rb.Context()
    yield c
    c.close()


class GpuBackend:
    """Encode through the host-buffer batch API, decode through the device-resident one (so that the bytes around
    the slots are device memory the test controls)."""

    def __init__(self, ctx, case):
        self.ctx = ctx
        model_cls = rb.AdaptiveTreeModel if len(case.name) & 1 else rb.AdaptiveLinearModel
        self.model = model_cls(rb.Parameters(*case.params))
        if case.train:
            self.model.train(km.train_for(case))
        ctx.set_schedule(SCHED[case.sched])
        ctx.launched_kernels(reset=True)

    def encode(self, blocks):
        lens = np.array([len(b) for b in blocks], dtype=np.uint64)
        off = np.zeros(len(blocks) + 1, dtype=np.uint64)
        np.cumsum(lens, out=off[1:])
        data = np.frombuffer(b"".join(blocks), dtype=np.uint8)
        out, out_off, status = self.ctx.encode_batch(data, off, self.model)
        assert (status == 0).all()
        return [out[int(out_off[i]):int(out_off[i + 1])].tobytes() for i in range(len(blocks))]

    def decode(self, comp, coff, raw, roff, max_len):
        import torch
        n = coff.size - 1
        d_comp = torch.from_numpy(comp).cuda()
        d_coff = torch.from_numpy(coff.astype(np.int64)).cuda()
        d_raw = torch.from_numpy(raw).cuda()
        d_roff = torch.from_numpy(roff.astype(np.int64)).cuda()
        d_len = torch.full((n,), -1, dtype=torch.int64, device="cuda")
        d_cons = torch.full((n,), -1, dtype=torch.int64, device="cuda")
        d_st = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        self.ctx.decode_batch_device(d_comp, d_coff, n, max_len, d_raw, d_roff, d_len, d_cons, d_st, self.model,
                                     device=torch.cuda.current_device(), stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        return d_raw.cpu().numpy(), d_len.cpu().numpy(), d_cons.cpu().numpy(), d_st.cpu().numpy()

    def kernels(self):
        return self.ctx.launched_kernels(reset=True)


@pytest.mark.parametrize("case", ORDER, ids=lambda c: c.name)
def test_kernel_matrix_row(ctx, case):
    km.check_row(case, GpuBackend(ctx, case))


def test_launched_kernels_hook(ctx):
    """The hook reads and resets the mask: a second read is empty, and a read without reset keeps it."""
    ctx.set_schedule(rb.SCHED_LANE)
    model = rb.AdaptiveTreeModel(rb.Parameters(8, 14, 16))
    data = np.frombuffer(b"kernel matrix", dtype=np.uint8)
    ctx.launched_kernels(reset=True)
    ctx.encode_batch(data, np.array([0, data.size], dtype=np.uint64), model)
    assert ctx.launched_kernels(reset=False) == {km.NARROW_STG[0]}
    assert ctx.launched_kernels(reset=True) == {km.NARROW_STG[0]}
    assert ctx.launched_kernels() == set()
