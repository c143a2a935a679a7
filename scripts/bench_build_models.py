"""Learning start models from the blocks on the device (redux_build_models): what it costs and what it buys.

  cost        device resident, 65,536 generator blocks of 64 KiB (4 GiB, larger than L2) at (8,14,16) and (8,30,32),
              K = 4, 16, 64, two starting memberships: contiguous ranges (the default; the generator's classes
              alternate block by block, so every cluster starts mixed and most empty after a round) and by class
              (init[b] = 1 + b mod K: every cluster holds blocks of one class and stays in use).
              Two independent timings of the same calls:
              - CUDA events around redux_build_models_device with 1, 2, ..., 8 rounds: round i costs t(i) - t(i - 1);
                the histogram pass is timed on its own with events around train_count_kernel over the same blocks
                (redux_train_models_device from a fresh (8,30,32) model counts every symbol with the same grid), so
                round 1 = t(1) - histogram pass (it also carries the call's few small uploads);
              - torch.profiler, in a pass of its own: the device time of every kernel and memset of one 8-round call,
                the histogram pass (train_count_kernel) apart and each round up to its build_total_kernel.
              Next to them redux_encode_batch_device_models of the same batch from the learned table and index.
  buys        the corpora in 4 KiB and 64 KiB blocks at both triples: container bytes (model table included) of pack
              (fresh only), pack_auto with fresh plus one model per file trained from the file's first 64 KiB (the
              by-file + select row of DESIGN.md 3.10), and pack_learned at K = 4, 16, 64 (8 rounds, no file
              boundaries); for each learned table the estimate (best round's total / 8) against the bytes of the
              streams encode_batch_select writes.
  convergence every round's total (iteration_cost_bits) of every run.

Prints one JSON line per measurement and, with --out FILE, writes all of them with the GPU's name, power limit and max
SM clock, read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import corpora_fixture as cf  # noqa: E402
import redux_b200 as rb  # noqa: E402
import redux_b200.container as ct  # noqa: E402

SEED = 0xB011D20261022001
REPS = 3


def timed(fn, reps=REPS):
    fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        fn()
    ev[1].record()
    ev[1].synchronize()
    return ev[0].elapsed_time(ev[1]) / reps


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def profiled_rounds(fn):
    """Device time (ms) of the histogram pass and of each round of one call, from a torch.profiler trace: kernels and
    memsets in stream order, the pass = train_count_kernel, a round ends with its build_total_kernel."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                 and ("kernel" in e.name or "Memset" in e.name)), key=lambda e: e.time_range.start)
    hist, rounds, cur = 0.0, [], 0.0
    for e in ev:
        ms = (e.time_range.end - e.time_range.start) / 1e3
        if "train_count_kernel" in e.name:
            hist += ms
        elif "Memset" in e.name and not rounds and cur == 0.0 and hist == 0.0:
            hist += ms                                       # the histogram rows' zeroing, before the pass
        else:
            cur += ms
            if "build_total_kernel" in e.name:
                rounds.append(cur)
                cur = 0.0
    return hist, rounds


def cost(ctx, params, n, length, emit):
    s = torch.cuda.current_stream().cuda_stream
    raw = torch.empty(n * length + 64, dtype=torch.uint8, device="cuda")
    ctx.generate_blocks_device(raw, 0, n, length, SEED, device=0, stream=s)
    off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * length
    bm = torch.zeros(n, dtype=torch.int32, device="cuda")
    cap = n * length + n * (length // 8) + (1 << 20)
    comp = torch.empty(cap, dtype=torch.uint8, device="cuda")
    coff = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    st = torch.zeros(n, dtype=torch.int32, device="cuda")
    fresh = rb.AdaptiveTreeModel(rb.Parameters(*params))
    # the histogram pass alone: train_count_kernel over every symbol of every block (no freeze below 2^30 - 1)
    counts = torch.empty((n, 257), dtype=torch.int32, device="cuda")
    every = rb.AdaptiveTreeModel(rb.Parameters(8, 30, 32))
    hist_ms = timed(lambda: ctx.train_models_device(raw, off, n, length, counts, every, device=0, stream=s))
    del counts
    for k in (4, 16, 64):
        tab = torch.zeros((k + 1, 257), dtype=torch.int32, device="cuda")
        tot = torch.zeros(8, dtype=torch.float64, device="cuda")
        for start, init in (("contiguous", None), ("by_class", 1 + np.arange(n, dtype=np.uint32) % k)):
            def build(it):
                ctx.build_models_device(raw, off, n, length, fresh, k, tab, bm, tot, iterations=it, init=init,
                                        device=0, stream=s)
            t = [timed(lambda: build(it)) for it in range(1, 9)]
            rounds = [t[0] - hist_ms] + [t[i] - t[i - 1] for i in range(1, 8)]
            p_hist, p_rounds = profiled_rounds(lambda: build(8))
            models = [fresh] + rb._trained_models(rb.AdaptiveTreeModel, fresh.params,
                                                  tab[1:].cpu().numpy().view(np.uint32))
            enc = timed(lambda: ctx.encode_batch_device_models(raw, off, n, length, comp, cap, coff, st, models, bm,
                                                               device=0, stream=s))
            assert (st.cpu().numpy() == 0).all()
            used = np.bincount(bm.cpu().numpy(), minlength=k + 1)
            emit({"what": "cost", "params": params, "blocks": n, "block_len": length, "K": k, "init": start,
                  "histogram_pass_ms": hist_ms, "build_ms_by_rounds": t, "round_ms": rounds,
                  "round1_over_encode": rounds[0] / enc, "profiled_histogram_ms": p_hist,
                  "profiled_round_ms": p_rounds, "profiled_round1_over_encode": p_rounds[0] / enc,
                  "encode_models_ms": enc, "rows_used": int((used > 0).sum()),
                  "stream_bytes": int(coff[-1].item()), "iteration_cost_bits": tot.cpu().numpy().tolist()})
    del raw, comp


def buys(ctx, params, block_len, emit):
    files = cf.corpora()
    names = sorted(files)
    blob = b"".join(files[k] for k in names)
    data = np.frombuffer(blob, dtype=np.uint8)
    fresh = rb.AdaptiveTreeModel(rb.Parameters(*params))
    sample = [files[k][:65536] for k in names]
    soff = np.zeros(len(names) + 1, dtype=np.uint64)
    np.cumsum([len(x) for x in sample], out=soff[1:])
    by_file = [fresh] + ctx.train_models(np.frombuffer(b"".join(sample), dtype=np.uint8), soff, fresh)
    row = {"what": "buys", "params": params, "block_len": block_len, "raw_bytes": int(data.size),
           "fresh_only": len(ct.pack(blob, fresh, block_len, context=ctx)),
           "by_file_select": len(ct.pack_auto(blob, by_file, block_len, context=ctx))}
    n = (data.size + block_len - 1) // block_len
    off = np.minimum(np.arange(n + 1, dtype=np.uint64) * np.uint64(block_len), np.uint64(data.size))
    for k in (4, 16, 64):
        packed = ct.pack_learned(blob, fresh, k=k, iterations=8, block_len=block_len, context=ctx)
        assert ct.unpack(packed, context=ctx) == blob
        models, _, totals = ctx.build_models(data, off, fresh, k, 8)
        comp, _, st, _ = ctx.encode_batch_select(data, off, models)
        assert (st == 0).all()
        row["learned_K%d" % k] = len(packed)
        row["learned_K%d_estimate_bytes" % k] = float(totals.min() / 8)
        row["learned_K%d_stream_bytes" % k] = int(comp.size)
        row["learned_K%d_iteration_cost_bits" % k] = totals.tolist()
    emit(row)


def main(out=None):
    ctx = rb.Context([0])
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    info = gpu_info()
    emit({"what": "gpu", "gpu": info})
    for params in ((8, 14, 16), (8, 30, 32)):
        cost(ctx, params, 65536, 65536, emit)
        torch.cuda.empty_cache()
    for params in ((8, 14, 16), (8, 30, 32)):
        for block_len in (4096, 65536):
            buys(ctx, params, block_len, emit)
    ctx.close()
    if out:
        with open(out, "w") as f:
            json.dump({"gpu": info, "results": lines}, f, indent=1)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    main(ap.parse_args().out)
