"""CRC-32 of every block on the device (redux_crc32_blocks, DESIGN.md 3.11): what the kernel reaches and what the
fused calls cost end to end.

  kernel      device resident, CUDA events around redux_crc32_blocks_device: 65,536 generator blocks of 64 KiB (4 GiB,
              larger than L2, so every pass reads HBM), 16 blocks of 64 MiB over the same bytes, and a ragged batch of
              0 .. 128 KiB blocks at unaligned offsets; GB/s and the share of the 6,454.6 GB/s measured HBM peak
  variants    the kernel's body in other shapes (scripts/crc32_variants.cu, compiled with nvcc into a temporary
              directory): replicas of the tables, threads per CTA, CTAs per SM, the next trip's vectors loaded before
              the current ones are folded; the same three batches, CUDA events, results checked against the library's,
              with each variant's registers, spills and resident CTAs per SM
  end to end  from pinned host memory, 16,384 generator blocks of 64 KiB at (8,14,16) with K = 16 models (fresh plus 15
              trained on the device): encode_batch_models, encode_batch_select and decode_batch_models against their
              _crc forms, run alternately in the same process, median and spread of each.  These calls synchronise
              the host and run on the library's own streams, so they are timed by the host's wall clock
              (time.perf_counter around each call), not by CUDA events; do not compare them with the kernel numbers
  host        zlib.crc32 on one core and on every core (zlib releases the GIL), for scale

Prints one JSON line per measurement and, with --out FILE, writes all of them with the GPU's name, power limit and
maximum SM clock, read in the same run."""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import redux_b200 as rb  # noqa: E402

SEED = 0xC3C32026102201
HBM_PEAK_GBS = 6454.6          # DESIGN.md 3.5, measured on this card type


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def events(fn, reps):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return out


def stats(ms, nbytes):
    ms = sorted(ms)
    med = float(np.median(ms))
    return {"median_ms": med, "min_ms": ms[0], "max_ms": ms[-1], "GBps": nbytes / med / 1e6,
            "share_of_hbm_peak": nbytes / med / 1e6 / HBM_PEAK_GBS}


def load_variants(tmp):
    """Compiles scripts/crc32_variants.cu into tmp; returns (library, {variant: ptxas registers and spills})."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    so = os.path.join(tmp, "crc32_variants.so")
    r = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                        "-Xptxas", "-v", "--expt-relaxed-constexpr", "-shared", "-o", so,
                        os.path.join(ROOT, "scripts", "crc32_variants.cu")], capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(r.stderr[-3000:])
    ptxas, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '.*crc_variant_(\d+)", line)
        if m:
            cur = int(m.group(1))
        elif cur is not None and "spill stores" in line:
            st, ld = re.findall(r"(\d+) bytes spill (?:stores|loads)", line)
            ptxas[cur] = {"spill_store_bytes": int(st), "spill_load_bytes": int(ld)}
        elif cur is not None and "Used" in line:
            ptxas[cur]["registers"] = int(re.search(r"Used (\d+) registers", line).group(1))
            cur = None
    L = C.CDLL(so)
    L.crc_variant_name.restype = C.c_char_p
    L.crc_variant_run.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p,
                                  C.c_int]
    assert L.crc_variant_setup() == 0
    return L, ptxas


def layouts(n, L):
    rng = np.random.default_rng(SEED & 0xFFFF)
    lens = rng.integers(0, 131072, 2 * n)
    lens = lens[np.cumsum(lens) < n * L - 4096][:n]
    starts = np.concatenate([[3], 3 + np.cumsum(lens)[:-1]])
    return {
        "65536x64KiB": (np.arange(n + 1, dtype=np.int64) * L, L),
        "16x64MiB": (np.arange(17, dtype=np.int64) * (64 << 20), 64 << 20),
        "ragged_0_128KiB_unaligned": (np.concatenate([starts, [starts[-1] + lens[-1]]]).astype(np.int64),
                                      int(lens.max())),
    }


def variant_runs(ctx, reps, d_in, n, L):
    """Every shape of scripts/crc32_variants.cu on the three batches; CRCs equal to the library's."""
    dev = d_in.device
    s = torch.cuda.current_stream().cuda_stream
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        V, ptxas = load_variants(tmp)
        for name, (off, max_len) in layouts(n, L).items():
            nb = off.size - 1
            d_off = torch.from_numpy(off).to(dev)
            want = torch.zeros(nb, dtype=torch.int32, device=dev)
            ctx.crc32_blocks_device(d_in, d_off, nb, max_len, want, stream=s)
            d_crc = torch.zeros(nb, dtype=torch.int32, device=dev)
            nbytes = int(off[-1] - off[0])
            for v in range(V.crc_variant_count()):
                vn = V.crc_variant_name(v).decode()

                def run():
                    assert V.crc_variant_run(v, d_in.data_ptr(), d_off.data_ptr(), nb, max_len, d_crc.data_ptr(), s,
                                             sms) == 0
                ms = events(run, reps)
                assert torch.equal(d_crc, want), (vn, name)
                r = res.setdefault(vn, {"ctas_per_sm": V.crc_variant_occupancy(v), **ptxas.get(v, {})})
                r[name] = stats(ms, nbytes)
                print(json.dumps({"variant": vn, "batch": name, **r[name]}), flush=True)
    return res


def kernel_runs(ctx, reps, variants):
    dev = torch.device("cuda", 0)
    s = torch.cuda.current_stream().cuda_stream
    n, L = 65536, 65536
    d_in = torch.empty(n * L + 64, dtype=torch.uint8, device=dev)
    ctx.generate_blocks_device(d_in, 0, n, L, SEED, stream=s)
    res = {}
    host = d_in[: 64 << 20].cpu().numpy()
    for name, (off, max_len) in layouts(n, L).items():
        nb = off.size - 1
        d_off = torch.from_numpy(off).to(dev)
        d_crc = torch.zeros(nb, dtype=torch.int32, device=dev)
        ms = events(lambda: ctx.crc32_blocks_device(d_in, d_off, nb, max_len, d_crc, stream=s), reps)
        nbytes = int(off[-1] - off[0])
        got = d_crc.cpu().numpy().view(np.uint32)
        # spot check against zlib over the first 64 MiB
        k = int(np.searchsorted(off, 64 << 20, side="right")) - 1
        want = [zlib.crc32(host[off[i]:off[i + 1]].tobytes()) for i in range(min(k, 64))]
        assert list(got[:len(want)]) == want, name
        res[name] = dict(stats(ms, nbytes), blocks=nb, bytes=nbytes, reps=reps)
        print(json.dumps({"kernel": name, **res[name]}), flush=True)
    var = variant_runs(ctx, reps, d_in, n, L) if variants else None
    del d_in
    torch.cuda.empty_cache()
    return res, var


def e2e_runs(ctx, pairs):
    p = rb.Parameters(8, 14, 16)
    n, L = 16384, 65536
    buf = rb.HostBuffer(n * L)
    buf.array[:] = rb.generate_blocks_host(0, n, L, SEED)
    data = buf.array
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(L)
    samples = rb.generate_blocks_host(10 ** 6, 15, L, SEED + 1)
    trained = ctx.train_models(samples, np.arange(16, dtype=np.uint64) * np.uint64(L), rb.AdaptiveTreeModel(p))
    models = [rb.AdaptiveTreeModel(p)] + trained
    bm = ctx.select_models(data, off, models)
    cap = int(n * (L + 64) * 2)
    out = rb.HostBuffer(cap)
    comp, coff, st = ctx.encode_batch_models(data, off, models, bm, out=out.array)
    comp = comp.copy()
    cbuf = rb.HostBuffer(comp.size)
    cbuf.array[:] = comp
    raw = rb.HostBuffer(n * L)
    calls = {
        "encode_batch_models": (lambda: ctx.encode_batch_models(data, off, models, bm, out=out.array),
                                lambda: ctx.encode_batch_models_crc(data, off, models, bm, out=out.array)),
        "encode_batch_select": (lambda: ctx.encode_batch_select(data, off, models, out=out.array),
                                lambda: ctx.encode_batch_select_crc(data, off, models, out=out.array)),
        "decode_batch_models": (lambda: ctx.decode_batch_models(cbuf.array, coff, off, models, bm, raw=raw.array),
                                lambda: ctx.decode_batch_models_crc(cbuf.array, coff, off, models, bm, raw=raw.array)),
    }
    res = {}
    for name, (base, fused) in calls.items():
        base()
        fused()
        tb, tf = [], []
        for _ in range(pairs):
            for fn, acc in ((base, tb), (fused, tf)):
                t = time.perf_counter()
                fn()
                acc.append((time.perf_counter() - t) * 1e3)
        mb, mf = float(np.median(tb)), float(np.median(tf))
        res[name] = {"base_ms": tb, "crc_ms": tf, "base_median_ms": mb, "crc_median_ms": mf,
                     "base_spread_ms": max(tb) - min(tb), "crc_spread_ms": max(tf) - min(tf),
                     "crc_over_base": mf / mb, "GBps_base": n * L / mb / 1e6, "GBps_crc": n * L / mf / 1e6}
        print(json.dumps({"e2e": name, **{k: v for k, v in res[name].items() if not k.endswith("_ms")},
                          "base_median_ms": mb, "crc_median_ms": mf}), flush=True)
    # the fused results equal the base ones on this batch
    e_base = ctx.encode_batch_models(data, off, models, bm)
    e_crc = ctx.encode_batch_models_crc(data, off, models, bm)
    assert e_base[0].tobytes() == e_crc[0].tobytes()
    assert (e_crc[3][:64] == [zlib.crc32(data[i * L:(i + 1) * L].tobytes()) for i in range(64)]).all()
    return res


def host_runs():
    nbytes = 256 << 20
    a = np.random.default_rng(1).integers(0, 256, nbytes, dtype=np.uint8).tobytes()
    zlib.crc32(a[:1 << 20])
    t = time.perf_counter()
    zlib.crc32(a)
    one = nbytes / (time.perf_counter() - t) / 1e9
    cores = os.cpu_count() or 1
    part = nbytes // cores
    views = [memoryview(a)[i * part:(i + 1) * part] for i in range(cores)]
    with ThreadPoolExecutor(cores) as ex:
        list(ex.map(zlib.crc32, views))
        t = time.perf_counter()
        list(ex.map(zlib.crc32, views))
        allc = part * cores / (time.perf_counter() - t) / 1e9
    r = {"one_core_GBps": one, "all_cores_GBps": allc, "cores": cores}
    print(json.dumps({"host_zlib": r}), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--pairs", type=int, default=5)
    ap.add_argument("--no-variants", action="store_true", help="skip the kernel shapes of scripts/crc32_variants.cu")
    a = ap.parse_args()
    rb.process_init()
    info = gpu_info()
    ctx = rb.Context()
    kernel, variants = kernel_runs(ctx, a.reps, not a.no_variants)
    res = {"gpu": info, "hbm_peak_GBps_measured": HBM_PEAK_GBS, "kernel": kernel, "kernel_variants": variants,
           "e2e_pinned": e2e_runs(ctx, a.pairs), "e2e_timer": "host wall clock (time.perf_counter) around each call",
           "host_zlib": host_runs(), "gpu_after": gpu_info()}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
