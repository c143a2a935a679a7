"""Choosing each block's start model on the device (redux_select_models): what it costs and what it buys.

  selection   device resident, 65,536 generator blocks of 64 KiB (4 GiB, larger than L2) and 16 blocks of 64 MiB, at
              (8,14,16) and (8,30,32); K = 1, 4, 16, 256 candidates (fresh plus models trained on the device from
              64 KiB generator samples of every class); CUDA events around redux_select_models_device, next to
              redux_encode_batch_device_models of the same batch with the chosen index
  end to end  from pinned host memory, (8,14,16), K = 16: encode_batch_select against select_models followed by
              encode_batch_models and against encode_batch_models with the index computed before the clock starts
  buys        the corpora in 4 KiB and 64 KiB blocks, candidates fresh plus one model per file trained from the file's
              first 64 KiB: total compressed bytes with the fresh model only, the by-file assignment, the estimate's
              choice and the exhaustive best (every model encoded, each block's smallest stream), sum(cost) / 8
              against the chosen streams' bytes, and the share of blocks whose choice is not the exhaustive best

Prints one JSON line per measurement and, with --out FILE, writes all of them with the GPU's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import corpora_fixture as cf  # noqa: E402
import redux_b200 as rb  # noqa: E402

SEED = 0x5E1EC72026102201
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


def wall(fn, reps=REPS):
    fn()
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t) / reps * 1e3


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def candidates(ctx, params, k):
    """Fresh plus k - 1 models trained on the device, each from one 64 KiB generator sample (classes in turn)."""
    models = [rb.AdaptiveTreeModel(rb.Parameters(*params))]
    if k > 1:
        sample = rb.generate_blocks_host(1 << 24, k - 1, 65536, SEED + 1)
        soff = np.arange(k, dtype=np.uint64) * np.uint64(65536)
        models += ctx.train_models(sample, soff, models[0])
    return models


def selection(ctx, params, n, length, emit):
    s = torch.cuda.current_stream().cuda_stream
    raw = torch.empty(n * length + 64, dtype=torch.uint8, device="cuda")
    ctx.generate_blocks_device(raw, 0, n, length, SEED, device=0, stream=s)
    off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * length
    bm = torch.zeros(n, dtype=torch.int32, device="cuda")
    cap = n * length + n * (length // 8) + (1 << 20)
    comp = torch.empty(cap, dtype=torch.uint8, device="cuda")
    coff = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    st = torch.zeros(n, dtype=torch.int32, device="cuda")
    for k in (1, 4, 16, 256):
        models = candidates(ctx, params, k)
        sel = timed(lambda: ctx.select_models_device(raw, off, n, length, models, bm, device=0, stream=s))
        enc = timed(lambda: ctx.encode_batch_device_models(raw, off, n, length, comp, cap, coff, st, models, bm,
                                                           device=0, stream=s))
        assert (st.cpu().numpy() == 0).all()
        used = np.bincount(bm.cpu().numpy(), minlength=k)
        emit({"what": "selection", "params": params, "blocks": n, "block_len": length, "K": k, "select_ms": sel,
              "encode_models_ms": enc, "select_over_encode": sel / enc, "models_used": int((used > 0).sum()),
              "select_GBps": n * length / sel / 1e6})
    del raw, comp


def end_to_end(ctx, params, emit):
    n, length, k = 16384, 65536, 16
    data = rb.HostBuffer(n * length)
    data.array[:] = rb.generate_blocks_host(0, n, length, SEED)
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(length)
    out = rb.HostBuffer(n * length + n * (length // 8) + (1 << 20))
    models = candidates(ctx, params, k)
    index = ctx.select_models(data.array, off, models)
    fused = wall(lambda: ctx.encode_batch_select(data.array, off, models, out=out.array))
    two = wall(lambda: ctx.encode_batch_models(data.array, off, models, ctx.select_models(data.array, off, models),
                                               out=out.array))
    given = wall(lambda: ctx.encode_batch_models(data.array, off, models, index, out=out.array))
    got = ctx.encode_batch_select(data.array, off, models, out=out.array)
    assert (got[3] == index).all()
    emit({"what": "end_to_end_pinned", "params": params, "blocks": n, "block_len": length, "K": k,
          "encode_batch_select_ms": fused, "select_then_encode_ms": two, "encode_given_index_ms": given,
          "GBps_fused": n * length / fused / 1e6})
    data.close(); out.close()


def buys(ctx, params, block_len, emit):
    files = cf.corpora()
    names = sorted(files)
    blob = b"".join(files[k] for k in names)
    data = np.frombuffer(blob, dtype=np.uint8)
    sample = [files[k][:65536] for k in names]
    soff = np.zeros(len(names) + 1, dtype=np.uint64)
    np.cumsum([len(x) for x in sample], out=soff[1:])
    fresh = rb.AdaptiveTreeModel(rb.Parameters(*params))
    models = [fresh] + ctx.train_models(np.frombuffer(b"".join(sample), dtype=np.uint8), soff, fresh)
    n = (data.size + block_len - 1) // block_len
    off = np.minimum(np.arange(n + 1, dtype=np.uint64) * np.uint64(block_len), np.uint64(data.size))
    starts = np.cumsum([0] + [len(files[k]) for k in names])
    by_file = (np.searchsorted(starts, off[:-1].astype(np.int64), side="right")).astype(np.uint32)   # row 1 + file
    sizes = np.zeros((len(models), n), dtype=np.int64)
    for m in range(len(models)):
        _, coff, st = ctx.encode_batch_models(data, off, models, np.full(n, m, dtype=np.uint32))
        assert (st == 0).all()
        sizes[m] = np.diff(coff.astype(np.int64))
    choice, cost = ctx.select_models(data, off, models, costs=True)
    chosen = sizes[choice, np.arange(n)]
    best = sizes.min(axis=0)
    emit({"what": "buys", "params": params, "block_len": block_len, "blocks": n, "K": len(models),
          "raw_bytes": int(data.size), "fresh_only": int(sizes[0].sum()),
          "by_file": int(sizes[by_file, np.arange(n)].sum()), "estimate_choice": int(chosen.sum()),
          "exhaustive_best": int(best.sum()),
          "sum_cost_bytes_of_choice": float(cost[np.arange(n), choice].sum() / 8),
          "share_not_exhaustive_best": float((chosen > best).mean())})


def main(out=None):
    ctx = rb.Context([0])
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    info = gpu_info()
    emit({"what": "gpu", "gpu": info})
    for params in ((8, 14, 16), (8, 30, 32)):
        selection(ctx, params, 65536, 65536, emit)
        selection(ctx, params, 16, 64 << 20, emit)
        torch.cuda.empty_cache()
    end_to_end(ctx, (8, 14, 16), emit)
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
