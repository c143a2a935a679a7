"""A start model per block: what does one launch with K trained models cost against one model, and against K calls?

Device resident, 65,536 generator blocks of 64 KiB (4 GiB, larger than L2), CUDA events around each call, at
(8,14,16) and (8,30,32):
  single     one trained model through the _ex call (every block starts from it)
  models K   K trained models assigned to the blocks at random, one redux_*_batch_device_models call
  grouped K  the same blocks sorted by model (sorted before the clock starts) and coded by K _ex calls, one per model
  spread     half the lanes of every warp start fresh, half from a model 100 below freq_max: the lanes of a warp
             freeze at far-apart positions
Model k is trained on the first 4,000 bytes of generator block k.  Every configuration decodes to the input, and the
streams of the models calls equal the grouped calls' block for block.  Prints one JSON line per configuration and, with
--out FILE, writes all of them to FILE with the GPU's name and power limit (profiles/r03_block_models.json)."""
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
import oracle_lib as o  # noqa: E402
import redux_b200 as rb  # noqa: E402

SEED = 0x5EED202610180000
N, L = 65536, 65536
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


def main(out=None):
    ctx = rb.Context([0])
    s = torch.cuda.current_stream().cuda_stream
    dev = "cuda"
    raw = torch.empty(N * L, dtype=torch.uint8, device=dev)
    ctx.generate_blocks_device(raw, 0, N, L, SEED, device=0, stream=s)
    off = torch.arange(N + 1, dtype=torch.int64, device=dev) * L
    cap = N * L + N * (L // 8) + (1 << 20)
    comp = torch.empty(cap, dtype=torch.uint8, device=dev)
    coff = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    st = torch.zeros(N, dtype=torch.int32, device=dev)
    back = torch.empty(N * L, dtype=torch.uint8, device=dev)
    rl = torch.zeros(N, dtype=torch.int64, device=dev)
    cons = torch.zeros(N, dtype=torch.int64, device=dev)
    heads = raw.view(N, L)[:256, :4000].cpu().numpy()
    rng = np.random.default_rng(20261021)
    res = {"gpu": gpu_info(), "blocks": N, "block_len": L, "reps": REPS, "configs": {}}
    print(res["gpu"], flush=True)

    def run_models(params, models, bm, label):
        d_bm = torch.from_numpy(bm.astype(np.int32)).to(dev)
        ctx.launched_kernels(reset=True)
        te = timed(lambda: ctx.encode_batch_device_models(raw, off, N, L, comp, cap, coff, st, models, d_bm, 0, s))
        ke = ctx.launched_kernels(reset=True)
        assert int(st.abs().max()) == 0
        streams = comp[:int(coff[-1])].clone(), coff.clone()
        td = timed(lambda: ctx.decode_batch_device_models(streams[0], streams[1], N, L, back, off, rl, cons, st, models,
                                                          d_bm, 0, s))
        kd = ctx.launched_kernels(reset=True)
        assert int(st.abs().max()) == 0 and torch.equal(back, raw), label
        row = {"encode_ms": round(te, 2), "decode_ms": round(td, 2), "round_trip_GBps": round(N * L / (te + td) / 1e6, 2),
               "ratio": round(N * L / int(streams[1][-1]), 4), "kernels": sorted(ke | kd)}
        return row, streams

    def run_grouped(models, bm, label):
        """K _ex calls over the blocks sorted by model; returns the row and the streams in the original block order."""
        order = np.argsort(bm, kind="stable")
        bounds = np.searchsorted(bm[order], np.arange(len(models) + 1))
        sorted_raw = raw.view(N, L)[torch.from_numpy(order).to(dev)].reshape(-1)
        g_comp = torch.empty_like(comp)
        g_coff = [torch.zeros(int(bounds[g + 1] - bounds[g]) + 1, dtype=torch.int64, device=dev) for g in range(len(models))]
        g_base = [0] * (len(models) + 1)

        def enc():
            at = 0
            for g, m in enumerate(models):
                a, b = int(bounds[g]), int(bounds[g + 1])
                if a == b:
                    continue
                # each group's streams go to its own region of g_comp: L / 8 bytes of slack per block as `cap` has
                g_base[g] = at
                ctx.encode_batch_device(sorted_raw[a * L:b * L], off[:b - a + 1], b - a, L, g_comp[at:],
                                        cap - at, g_coff[g], st[a:b], m, 0, s)
                at += (b - a) * (L + L // 8)

        te = timed(enc)
        assert int(st.abs().max()) == 0
        sorted_back = torch.empty_like(raw)

        def dec():
            for g, m in enumerate(models):
                a, b = int(bounds[g]), int(bounds[g + 1])
                if a == b:
                    continue
                ctx.decode_batch_device(g_comp[g_base[g]:], g_coff[g], b - a, L, sorted_back[a * L:b * L], off[:b - a + 1],
                                        rl[a:b], cons[a:b], st[a:b], m, 0, s)

        td = timed(dec)
        torch.cuda.synchronize()
        assert int(st.abs().max()) == 0 and torch.equal(sorted_back, sorted_raw), label
        row = {"encode_ms": round(te, 2), "decode_ms": round(td, 2), "round_trip_GBps": round(N * L / (te + td) / 1e6, 2),
               "calls": int((bounds[1:] > bounds[:-1]).sum())}
        return row, (order, bounds, g_comp, g_coff, g_base)

    for params in ((8, 14, 16), (8, 30, 32)):
        fmax = (1 << params[1]) - 1
        models = []
        for k in range(256):
            m = rb.AdaptiveTreeModel(rb.Parameters(*params))
            models.append(m.train(heads[k]))
        # single model through the _ex call
        ctx.launched_kernels(reset=True)
        te = timed(lambda: ctx.encode_batch_device(raw, off, N, L, comp, cap, coff, st, models[0], 0, s))
        ke = ctx.launched_kernels(reset=True)
        single = comp[:int(coff[-1])].clone(), coff.clone()
        td = timed(lambda: ctx.decode_batch_device(single[0], single[1], N, L, back, off, rl, cons, st, models[0], 0, s))
        kd = ctx.launched_kernels(reset=True)
        assert int(st.abs().max()) == 0 and torch.equal(back, raw)
        i = 4097
        want = o.compress_trained(raw[i * L:(i + 1) * L].cpu().numpy(), heads[0], o.TREE, params)[1]
        assert single[0][int(single[1][i]):int(single[1][i + 1])].cpu().numpy().tobytes() == want
        row = {"encode_ms": round(te, 2), "decode_ms": round(td, 2), "round_trip_GBps": round(N * L / (te + td) / 1e6, 2),
               "ratio": round(N * L / int(single[1][-1]), 4), "kernels": sorted(ke | kd)}
        res["configs"]["%s single" % (params,)] = row
        print(params, "single", json.dumps(row), flush=True)
        for K in (4, 16, 256):
            bm = rng.integers(0, K, N).astype(np.uint32)
            row, streams = run_models(params, models[:K], bm, "models %d" % K)
            res["configs"]["%s models K=%d" % (params, K)] = row
            print(params, "models", K, json.dumps(row), flush=True)
            grow, (order, bounds, g_comp, g_coff, g_base) = run_grouped(models[:K], bm, "grouped %d" % K)
            res["configs"]["%s grouped K=%d" % (params, K)] = grow
            print(params, "grouped", K, json.dumps(grow), flush=True)
            # the same streams, block for block (sampled: 64 blocks)
            for i in rng.integers(0, N, 64):
                g = int(bm[i])
                j = int(np.nonzero(order[bounds[g]:bounds[g + 1]] == i)[0][0])
                a = g_comp[g_base[g] + int(g_coff[g][j]):g_base[g] + int(g_coff[g][j + 1])]
                b = streams[0][int(streams[1][i]):int(streams[1][i + 1])]
                assert torch.equal(a, b), (params, K, int(i))
            i = int(rng.integers(0, N))
            want = o.compress_trained(raw[i * L:(i + 1) * L].cpu().numpy(), heads[int(bm[i])], o.TREE, params)[1]
            assert streams[0][int(streams[1][i]):int(streams[1][i + 1])].cpu().numpy().tobytes() == want
            del streams, g_comp
            torch.cuda.empty_cache()
        # spread: lanes 0-15 of every warp fresh, lanes 16-31 from a model 100 below freq_max
        near = rb.AdaptiveTreeModel(rb.Parameters(*params))
        near.freq = np.full(257, (fmax - 100) // 257, dtype=np.uint32)
        near.freq[0] += (fmax - 100) - int(near.freq.sum())
        fresh = rb.AdaptiveTreeModel(rb.Parameters(*params))
        bm = ((np.arange(N) % 32) >= 16).astype(np.uint32)
        row, streams = run_models(params, [fresh, near], bm, "spread")
        res["configs"]["%s spread" % (params,)] = row
        print(params, "spread", json.dumps(row), flush=True)
        del streams
        torch.cuda.empty_cache()
    if out:
        with open(out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="write the results as JSON to this file")
    main(ap.parse_args().out)
