"""Training start models on the device (redux_train_models_device, DESIGN.md 3.9): how fast, and what it buys.

  bulk      65,536 generator samples of 64 KiB (4 GiB, larger than L2), device resident, CUDA events around each call,
            at (8,30,32) (every byte counted) and (8,14,16) (16,126 bytes per sample, then frozen): bytes counted per
            second next to the HBM peak DESIGN.md 3.5 measured (6,454.6 GB/s)
  classes   the same at (8,30,32) for each generator class alone (16,384 samples of one class: uniform, text-like,
            geometric, runs), which shows what the run aggregation and the per-warp sub-histograms leave of the
            contention the geometric and run classes cause
  sizes     the corpora (tests/golden/corpora) cut into 4 KiB and 64 KiB blocks, coded fresh and from a model per file
            trained on the device from the file's first 64 KiB: total compressed bytes
Every trained row of the bulk runs is checked against Model.train on a sample of rows.  Prints the result as JSON and,
with --out FILE, writes it to FILE with the GPU's name and power limit (profiles/r03_train_models.json)."""
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

SEED = 0x5EED202610180000
N, L = 65536, 65536
REPS = 5
HBM_PEAK_GBS = 6454.6


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


def check_rows(raw, out, params, rows):
    for i in rows:
        want = rb.AdaptiveTreeModel(rb.Parameters(*params)).train(raw[i].cpu().numpy())._state()
        assert (out[i].cpu().numpy().view(np.uint32) == want).all(), (params, i)


def main(out_path=None):
    ctx = rb.Context([0])
    s = torch.cuda.current_stream().cuda_stream
    res = {"gpu": gpu_info(), "hbm_peak_gbs_design_3_5": HBM_PEAK_GBS, "reps": REPS, "bulk": {}, "classes": {},
           "sizes": {}}
    print(res["gpu"], flush=True)
    raw = torch.empty(N * L, dtype=torch.uint8, device="cuda")
    ctx.generate_blocks_device(raw, 0, N, L, SEED, device=0, stream=s)
    off = torch.arange(N + 1, dtype=torch.int64, device="cuda") * L
    out = torch.empty((N, 257), dtype=torch.int32, device="cuda")
    rows = np.random.default_rng(7).integers(0, N, 16)
    for params in ((8, 30, 32), (8, 14, 16)):
        start = rb.AdaptiveTreeModel(rb.Parameters(*params))
        ms = timed(lambda: ctx.train_models_device(raw, off, N, L, out, start, stream=s))
        check_rows(raw.view(N, L), out, params, rows)
        per = min(L, (1 << params[1]) - 1 - 257)
        counted = N * per
        res["bulk"]["%d,%d,%d" % params] = {
            "samples": N, "sample_len": L, "bytes_counted_per_sample": per, "ms": round(ms, 3),
            "bytes_counted_gbs": round(counted / ms / 1e6, 1),
            "share_of_hbm_peak": round(counted / ms / 1e6 / HBM_PEAK_GBS, 3)}
        print(params, res["bulk"]["%d,%d,%d" % params], flush=True)
    names = ("uniform", "text", "geometric", "runs")
    m = N // 4
    moff = off[:m + 1].clone()
    mout = out[:m]
    start = rb.AdaptiveTreeModel(rb.Parameters(8, 30, 32))
    for k, name in enumerate(names):
        one = raw.view(N, L)[k::4].contiguous().view(-1)
        ms = timed(lambda: ctx.train_models_device(one, moff, m, L, mout, start, stream=s))
        check_rows(one.view(m, L), mout, (8, 30, 32), rows % m)
        res["classes"][name] = {"samples": m, "ms": round(ms, 3), "bytes_counted_gbs": round(m * L / ms / 1e6, 1)}
        print(name, res["classes"][name], flush=True)
        del one
    del raw, out
    torch.cuda.empty_cache()

    files = cf.corpora()
    names = sorted(files)
    for params in ((8, 14, 16), (8, 22, 24)):
        heads = [files[k][:65536] for k in names]
        hoff = np.zeros(len(names) + 1, dtype=np.uint64)
        np.cumsum([len(h) for h in heads], out=hoff[1:])
        fresh = rb.AdaptiveTreeModel(rb.Parameters(*params))
        models = ctx.train_models(np.frombuffer(b"".join(heads), dtype=np.uint8), hoff, fresh)
        for bl in (4096, 65536):
            data, bm, lens = [], [], []
            for fi, k in enumerate(names):
                d = files[k]
                for a in range(0, len(d), bl):
                    data.append(d[a:a + bl])
                    bm.append(fi)
            boff = np.zeros(len(data) + 1, dtype=np.uint64)
            np.cumsum([len(x) for x in data], out=boff[1:])
            arr = np.frombuffer(b"".join(data), dtype=np.uint8)
            _, c_fresh, st = ctx.encode_batch(arr, boff, fresh)
            assert (st == 0).all()
            _, c_tr, st = ctx.encode_batch_models(arr, boff, models, np.array(bm))
            assert (st == 0).all()
            key = "%d,%d,%d/%d" % (params + (bl,))
            res["sizes"][key] = {"blocks": len(data), "raw": int(boff[-1]), "fresh": int(c_fresh[-1]),
                                 "trained": int(c_tr[-1]), "trained_over_fresh": round(int(c_tr[-1]) / int(c_fresh[-1]), 4)}
            print(key, res["sizes"][key], flush=True)
    ctx.close()
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    main(ap.parse_args().out)
