#!/usr/bin/env python3
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

  python bench.py [--gpus N --steps K --warmup W]            our CUDA path
  python bench.py --impl reference [...]                     the CPU arm (oracle port, all host threads)
  python bench.py --dump-outputs DIR [...]                   also write the timed path's outputs (see dump_outputs)

Workload (configs 3+4 of BASELINE.json): 65,536 independent 64 KiB blocks of mixed entropy
(DESIGN.md "generator"), AdaptiveTreeModel, Parameters(8,14,16) by default.  One STEP = encode the whole
batch, then decode the produced streams back (both directions of the hot path).  The metric is raw
(uncompressed) bytes per second of that round trip: MB/s = raw_bytes / (t_encode + t_decode) / 1e6.

  value    device-resident: inputs already in HBM, CUDA events around the K timed steps on the launching
           stream (kernels incl. size scan + compaction), max over ranks.  WEAK scaling under torchrun: every
           rank codes its own 65,536-block batch (distinct block indices), no collective on the data path.
  e2e      the same metric through the host-buffer C ABI (redux_encode_batch / redux_decode_batch) from
           pinned host memory: H2D of the raw bytes, kernels, D2H of the streams, then H2D of the streams,
           kernels, D2H of the decoded bytes -- all inside the timed region.  `copy_ceiling` beside it is the
           same byte counts moved by bare pinned copies on every rank at once (what the box allows).
  strong   (N > 1) ONE 65,536-block list cut into contiguous ranges over the N ranks (SURVEY.md 8(e)):
           total raw bytes / max-over-ranks time.
  ctx      (N > 1, rank 0) the library's own multi-device front end: one redux_ctx over all N GPUs, one call for
           the whole batch; parity against a single-device context and the oracle, and its end-to-end time.
  classes  encode / decode times of the other parameter classes (8,22,24) and (8,30,32) -- the latter is the
           only parameter set the reference's CLI uses (src/main.rs:108).
Rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from

SEED = 0x5EED202610180000
METRIC = "encode+decode round-trip throughput of raw input (bit-exact)"
UNIT = "MB/s"
NCU_TRAFFIC = ("r02_ncu_traffic.json", "r01_ncu_traffic.json")
ISSUE_PEAK = "r01_issue_peak.json"
DUMP_LIMIT = 64 * 10 ** 6           # bytes of .npy files --dump-outputs writes at most


def int_at_least(minimum):
    def parse(s):
        v = int(s)
        if v < minimum:
            raise argparse.ArgumentTypeError("must be >= %d" % minimum)
        return v
    return parse


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int_at_least(1), default=5, help="timed steps of the headline measurement")
    ap.add_argument("--warmup", type=int_at_least(0), default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--blocks", type=int, default=65536)
    ap.add_argument("--block-len", type=int, default=65536)
    ap.add_argument("--params", default="8,14,16")
    ap.add_argument("--model", default="tree", choices=["tree", "linear"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-classes", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-ctx", action="store_true")
    ap.add_argument("--no-host-memory-kinds", action="store_true", help="skip the pageable / registered e2e legs")
    ap.add_argument("--cpu-sample-blocks", type=int, default=0, help="0 = 32 blocks per host thread")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step computed "
                                                          "(rank 0's batch) as DIR/<name>.npy")
    return ap.parse_args()


def arith_dtype(params):
    """The integer type the coder arithmetic runs in: products fit u32 when code_bits + freq_bits <= 30
    (NARROW class), else u64 (DESIGN.md 3.3)."""
    return "u32" if params[1] + params[2] <= 30 else "u64"


_corpus = None


def text_corpus():
    """The corpus the text class (block index & 3 == 1) cuts its windows from: the concatenation, in sorted path
    order, of the Calgary and Canterbury corpora (BASELINE.md section 4, config 3) -- 6,040,451 bytes from the
    fixture tests/golden/corpora/corpora.tar.xz (byte-identical to the reference's resources/)."""
    global _corpus
    if _corpus is None:
        import numpy as np

        import corpora_fixture as cf
        files = cf.corpora()
        names = sorted(n for n in files if n.startswith(("calgary/", "canterbury/")))
        _corpus = np.frombuffer(b"".join(files[n] for n in names), dtype=np.uint8)
        assert _corpus.size == 6040451
    return _corpus


def workload_name(a, world=1):
    per = "%d x %d B mixed-entropy blocks (uniform / Calgary+Canterbury window / geometric / sparse), Adaptive%sModel, Parameters(%s)" % (
        a.blocks, a.block_len, a.model.capitalize(), a.params)
    return per if world == 1 else "%d ranks x (%s) = %d blocks" % (world, per, world * a.blocks)


def ncu_capture(a, kernel):
    """DRAM traffic and issue-slot utilisation of `kernel` from the committed ncu capture, if that capture
    was taken on exactly this per-GPU workload (they cannot be measured live: never time under a profiler)."""
    for name in NCU_TRAFFIC:
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            if d["workload"] == workload_name(a):
                return d["kernels"][kernel], d["source"]
        except Exception:
            continue
    return None, None


def issue_roofline(ncu, ncu_src, n_blocks, block_len, kernel_s):
    """The roofline that actually binds this path (north_star): warp-instruction issue.  achieved = warp
    instructions per symbol step (committed ncu capture of this workload) x symbol steps per launch / the
    kernel's live duration; peak = the issue rate measured on the box by scripts/issue_peak.cu."""
    if not ncu:
        return None
    steps = n_blocks / 32.0 * (block_len + 1)
    achieved = ncu["warp_inst_per_symbol_step"] * steps / kernel_s
    out = {"bound": "per-SM warp-instruction issue (4/clk/SM), the binding resource of this path",
           "achieved_warp_inst_per_s": round(achieved, -8), "issue_active_pct_of_peak": ncu["issue_active_pct"],
           "warp_inst_per_symbol_step": ncu["warp_inst_per_symbol_step"], "source": ncu_src}
    try:
        pk = json.load(open(os.path.join(ROOT, "profiles", ISSUE_PEAK)))
        peak = pk["issue_measured_warp_inst_per_s"]["alu_only"]
        out.update({"peak_warp_inst_per_s": peak, "frac": round(achieved / peak, 4),
                    "peak_source": "measured: profiles/%s (scripts/issue_peak.cu)" % ISSUE_PEAK})
    except Exception:
        pass
    return out


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------- CPU arm
# Only oracle/ is mapped here: the input comes from oracle/synth_blocks.c, the coder from oracle/redux_oracle.c.
def cpu_round_trip(a, n_sample, threads, first_block=0, keep_streams=False):
    """Encode + decode n_sample blocks with the oracle, one stream per thread.  Returns (seconds_enc, seconds_dec,
    raw_bytes, comp_bytes, streams) -- streams = the oracle's compressed bytes per block when keep_streams."""
    import numpy as np

    import oracle_lib as o
    kind = o.TREE if a.model == "tree" else o.LINEAR
    params = tuple(int(x) for x in a.params.split(","))
    L = a.block_len
    raw = o.generate_blocks(first_block, n_sample, L, SEED, corpus=text_corpus())
    off = np.arange(n_sample + 1, dtype=np.uint64) * np.uint64(L)
    t0 = time.perf_counter()
    rc, slots, slot_off, out_len, status = o.compress_batch(raw, off, kind, params, threads)
    t1 = time.perf_counter()
    assert rc == 0
    # decode straight from the slots (offsets = slot starts, lengths = out_len)
    comp_off = np.zeros(n_sample + 1, dtype=np.uint64)
    np.cumsum(out_len, out=comp_off[1:])
    streams = [slots[int(slot_off[i]):int(slot_off[i]) + int(out_len[i])] for i in range(n_sample)]
    comp = np.concatenate(streams)
    t2 = time.perf_counter()
    rc, back, raw_len, consumed, status = o.decompress_batch(comp, comp_off, off, kind, params, threads)
    t3 = time.perf_counter()
    assert rc == 0 and (back == raw).all()
    return t1 - t0, t3 - t2, int(raw.size), int(comp.size), (streams if keep_streams else None)


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_record(te, td, raw_bytes, threads, sample, build):
    v = raw_bytes / (te + td)
    return {"value": round(v / 1e6, 2), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
            "encode_MBps": round(raw_bytes / te / 1e6, 2), "decode_MBps": round(raw_bytes / td / 1e6, 2),
            "MiBps": round(v / 2 ** 20, 2), "per_thread_MBps": round(v / 1e6 / threads, 3),
            "encode_MiBps_per_thread": round(raw_bytes / te / 2 ** 20 / threads, 3),
            "decode_MiBps_per_thread": round(raw_bytes / td / 2 ** 20 / threads, 3),
            "build": build}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import oracle_lib as o
    build = o.use_native_build()
    threads = host_threads()
    n_sample = a.cpu_sample_blocks or min(a.blocks, 32 * threads)
    times = []
    for i in range(a.warmup + a.steps):
        te, td, raw_bytes, comp_bytes, _ = cpu_round_trip(a, n_sample, threads)
        if i >= a.warmup:
            times.append((te, td))
    te = sum(t[0] for t in times) / len(times)
    td = sum(t[1] for t in times) / len(times)
    value = raw_bytes / (te + td) / 1e6
    sample = "%d of %d blocks per step (%d B each), one stream per thread" % (n_sample, a.blocks, a.block_len)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": round((te + td) * 1e3, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "config": {"workload": workload_name(a), "sample": sample},
        "encode_MBps": round(raw_bytes / te / 1e6, 2), "decode_MBps": round(raw_bytes / td / 1e6, 2),
        "cpu_baseline": cpu_record(te, td, raw_bytes, threads, sample, build),
        "e2e": {"value": round(value, 2), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference crate is Rust (no toolchain in the image): this arm is the C oracle restatement; "
                "input from oracle/synth_blocks.c, the product library is not loaded",
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled every 10 ms during the timed region (NVML; nvidia-smi fallback)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index = index
        self.sm, self.reasons, self.mx = [], set(), None
        self.stop_flag = False
        self.th = None
        self.how = None

    def _nvml_loop(self, nv, h):
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                bits = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def _smi_loop(self):
        fields = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                  "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + fields,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                f = [x.strip() for x in line.split(",")]
                if len(f) >= 6:
                    try:
                        self.sm.append(float(f[0])); self.mx = float(f[1])
                    except ValueError:
                        continue
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(name)
        except Exception:
            pass

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            idx = self.index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except Exception:
                    pass
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.how = "nvml, 10 ms period"
            self.th = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
        except Exception:
            self.how = "nvidia-smi -lms 50"
            self.proc = None
            self.th = threading.Thread(target=self._smi_loop, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag = True
        if getattr(self, "proc", None):
            self.proc.terminate()
        if self.th:
            self.th.join(timeout=3)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons),
                "samples": len(sm), "how": self.how}


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPU cores next to its GPU (NVML's ideal affinity) BEFORE any pinned host
    buffer is allocated, so that the end-to-end copies of several ranks do not all cross to one NUMA node.
    Returns a short description for the JSON line; failure is harmless (the process stays unbound)."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        idx = index
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                idx = int(vis.split(",")[index])
            except Exception:
                pass
        h = nv.nvmlDeviceGetHandleByIndex(idx)
        before = len(os.sched_getaffinity(0))
        nv.nvmlDeviceSetCpuAffinity(h)
        return "cpu affinity %d -> %d cores (nvmlDeviceSetCpuAffinity)" % (before, len(os.sched_getaffinity(0)))
    except Exception as e:          # noqa: BLE001 -- best effort
        return "unbound (%s)" % type(e).__name__


# ------------------------------------------------------------------------------------- our arm
class DeviceBatch:
    """One device-resident batch: n blocks of L bytes starting at block index first_block, with everything the
    device API needs, and enc() / dec() on the current torch stream."""

    def __init__(self, rb, ctx, torch, local, n, L, first_block, params, model_name):
        self.n, self.L, self.local, self.ctx = n, L, local, ctx
        self.stream = torch.cuda.current_stream().cuda_stream
        self.model = (rb.AdaptiveTreeModel if model_name == "tree" else rb.AdaptiveLinearModel)(rb.Parameters(*params))
        self.raw = torch.empty(n * L, dtype=torch.uint8, device="cuda")
        ctx.generate_blocks_device(self.raw, first_block, n, L, SEED, device=local, stream=self.stream)
        self.in_off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * L
        self.cap = n * L + n * (L // 16) + 4096 * n // 64 + 65536      # > the ~1.006x worst case of uniform blocks
        self.comp = torch.empty(self.cap, dtype=torch.uint8, device="cuda")
        self.comp_off = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
        self.status = torch.zeros(n, dtype=torch.int32, device="cuda")
        self.back = torch.empty(n * L, dtype=torch.uint8, device="cuda")
        self.raw_lens = torch.zeros(n, dtype=torch.int64, device="cuda")
        self.consumed = torch.zeros(n, dtype=torch.int64, device="cuda")

    def enc(self):
        self.ctx.encode_batch_device(self.raw, self.in_off, self.n, self.L, self.comp, self.cap, self.comp_off,
                                     self.status, self.model, device=self.local, stream=self.stream)

    def dec(self):
        self.ctx.decode_batch_device(self.comp, self.comp_off, self.n, self.L, self.back, self.in_off, self.raw_lens,
                                     self.consumed, self.status, self.model, device=self.local, stream=self.stream)

    def check(self, torch):
        """Untimed whole-batch property check: every status OK, every block round-trips."""
        torch.cuda.synchronize()
        comp_bytes = int(self.comp_off[-1].item())
        assert comp_bytes <= self.cap and int(self.status.abs().max().item()) == 0
        assert torch.equal(self.back, self.raw), "round trip failed"
        return comp_bytes

    def timed(self, torch, steps, barrier):
        """K steps, CUDA events on the launching stream; returns (t_enc, t_dec) seconds per step."""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        t_enc = t_dec = 0.0
        barrier()
        for _ in range(steps):
            ev[0].record()
            self.enc()
            ev[1].record()
            self.dec()
            ev[2].record()
            ev[2].synchronize()
            t_enc += ev[0].elapsed_time(ev[1]) * 1e-3
            t_dec += ev[1].elapsed_time(ev[2]) * 1e-3
        barrier()
        return t_enc / steps, t_dec / steps


def dump_sample_size(rb, n, L, params):
    """How many blocks dump_outputs samples: as many as fit DUMP_LIMIT next to the per-block arrays, at the worst-case
    stream length, so that the count (and with it the sample) depends on the arguments only."""
    per_block = 8 * (4 * n + 1) + 4096                                  # float64 arrays over all blocks, npy headers
    per_sample = 4 * (L + rb.compress_bound(L, params[2], params[0])) + 16
    k = min(n, (DUMP_LIMIT - per_block) // per_sample)
    if k < 1:
        raise SystemExit("bench.py: --dump-outputs cannot fit %d blocks of %d B into %d bytes" % (n, L, DUMP_LIMIT))
    return k


def dump_outputs(out_dir, B, torch, k):
    """What the timed path's last step returned to its caller, as .npy files under out_dir (at most DUMP_LIMIT bytes):
      compressed_offsets, status, raw_lens, consumed   every block, float64 (exact below 2**53); status is the decoder's
      sample_blocks                                     k block indices drawn with SEED (same arguments, same sample)
      sample_compressed, sample_compressed_offsets      those blocks' streams (float32 per byte) and where each starts
      sample_decoded                                    those blocks' decoded bytes, float32 [k, block_len]
    Two builds run with the same arguments compute the same inputs, so their files compare value for value."""
    import numpy as np
    torch.cuda.synchronize()
    off = B.comp_off.cpu().numpy()
    idx = np.sort(np.random.default_rng(SEED).choice(B.n, size=k, replace=False))
    streams = [B.comp[int(off[i]):int(off[i + 1])] for i in idx]
    s_off = np.zeros(k + 1, dtype=np.float64)
    np.cumsum([s.numel() for s in streams], out=s_off[1:])
    decoded = B.back.view(B.n, B.L)[torch.as_tensor(idx, device=B.back.device)]
    arrays = {
        "compressed_offsets": off, "status": B.status.cpu().numpy(), "raw_lens": B.raw_lens.cpu().numpy(),
        "consumed": B.consumed.cpu().numpy(), "sample_blocks": idx, "sample_compressed_offsets": s_off,
        "sample_compressed": torch.cat(streams).cpu().numpy().astype(np.float32),
        "sample_decoded": decoded.cpu().numpy().astype(np.float32),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def copy_ceiling(torch, h_a, h_b, d_a, d_b, comp_bytes, barrier, steps=3):
    """The end-to-end step's byte counts moved by bare pinned copies, H2D and D2H concurrently on two streams:
    [raw up | streams down] then [streams up | raw down].  Every rank does it at once (barrier), so at N GPUs
    this is what the box's PCIe + host memory allow the e2e number to be."""
    up, down = torch.cuda.Stream(), torch.cuda.Stream()
    n = h_a.numel()

    def one():
        with torch.cuda.stream(up):
            d_a.copy_(h_a, non_blocking=True)
        with torch.cuda.stream(down):
            h_b[:comp_bytes].copy_(d_b[:comp_bytes], non_blocking=True)
        up.synchronize(); down.synchronize()
        with torch.cuda.stream(up):
            d_b[:comp_bytes].copy_(h_b[:comp_bytes], non_blocking=True)
        with torch.cuda.stream(down):
            h_a.copy_(d_a, non_blocking=True)
        up.synchronize(); down.synchronize()

    one()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    t = (time.perf_counter() - t0) / steps
    barrier()
    return t, n


def run_ours(a):
    import numpy as np
    import torch

    import redux_b200 as rb
    from redux_b200 import sharding
    queues = rb.process_init()      # before CUDA is initialised: 32 hardware queues for the e2e pipeline's streams

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(vals):
        return sharding.max_over_ranks(vals, dist, "cuda")

    def rank_sum(v):
        t = torch.tensor([float(v)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t)
        return float(t.item())

    params = tuple(int(x) for x in a.params.split(","))
    n, L = a.blocks, a.block_len
    ctx = rb.Context([local])
    ctx.set_text_corpus(text_corpus())
    first_block = sharding.weak_first_block(n, rank)      # weak scaling: distinct blocks per rank

    dump_k = dump_sample_size(rb, n, L, params) if a.dump_outputs else 0

    # ---- synthetic batch, resident in HBM
    B = DeviceBatch(rb, ctx, torch, local, n, L, first_block, params, a.model)
    for _ in range(a.warmup):
        B.enc()
        B.dec()

    # ---- timed region: K steps, device resident
    sampler = ClockSampler(local)
    ctx.timing_enable(True)
    ctx.timing_collect()
    launches0 = ctx.kernel_launches
    sampler.start()
    wall0 = time.perf_counter()
    t_e, t_d = B.timed(torch, a.steps, barrier)
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    launches = ctx.kernel_launches - launches0
    ktimes = ctx.timing_collect()
    ctx.timing_enable(False)

    comp_bytes = B.check(torch)

    # ---- parity of the timed steps' output: the first blocks' streams against the oracle's bytes (every rank, untimed).
    # With the CPU baseline on (rank 0, N = 1) the same oracle run is the baseline's sample.
    import oracle_lib as o
    threads = host_threads()
    want_cpu = rank == 0 and world == 1 and not a.no_cpu_baseline
    oracle_build = o.use_native_build() if want_cpu else "portable (-O3)"
    ns = (a.cpu_sample_blocks or min(n, 32 * threads)) if want_cpu else min(n, 64)
    te_cpu, td_cpu, rb_cpu, cb_cpu, want = cpu_round_trip(a, ns, threads, first_block, keep_streams=True)
    got_off = B.comp_off[:ns + 1].cpu().numpy()
    got = B.comp[:int(got_off[-1])].cpu().numpy()
    for i in range(ns):
        assert got[int(got_off[i]):int(got_off[i + 1])].tobytes() == want[i].tobytes(), \
            "block %d: GPU stream differs from the oracle's" % (first_block + i)
    parity_checked = int(rank_sum(ns))
    cpu = cpu_record(te_cpu, td_cpu, rb_cpu, threads,
                     "%d of %d blocks (%d B each), one stream per thread" % (ns, n, L), oracle_build) if want_cpu else None
    del want, got

    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, B, torch, dump_k)

    t_step, t_e, t_d = rank_max([t_e + t_d, t_e, t_d])
    raw_bytes = n * L
    value = world * raw_bytes / t_step / 1e6

    # ---- roofline of the dominant kernel (algorithmic bytes = raw + compressed + 16 B/block of metadata)
    peak, peak_src = peaks()
    alg_bytes = raw_bytes + comp_bytes + 16 * n
    kdur = {k: (v[0] / v[1] * 1e-3 if v[1] else None) for k, v in ktimes.items()}
    dom = "decode" if (kdur.get("decode") or 0) >= (kdur.get("encode") or 0) else "encode"
    achieved = alg_bytes / kdur[dom] / 1e9
    kname = dom + ("_lane_al_kernel" if params[2] <= 32 else "_lane_kernel")
    ncu, ncu_src = ncu_capture(a, kname)
    roofline = {"bound": "hbm", "kernel": kname, "achieved": round(achieved, 2), "peak": peak,
                "unit": "GB/s", "frac": round(achieved / peak, 5), "traffic": ncu["traffic"] if ncu else None,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                "kernel_ms": {k: (round(v * 1e3, 3) if v else None) for k, v in kdur.items()},
                "issue": issue_roofline(ncu, ncu_src, n, L, kdur[dom]),
                "note": "HBM is not the binding resource: a stream is a serial dependency chain, so the kernels "
                        "are bound by instruction issue / latency; frac is reported against HBM as the contract asks"}

    # ---- the other parameter classes on the same blocks (device resident; (8,30,32) is the reference CLI's)
    classes = None
    if not a.no_classes and a.params == "8,14,16":
        classes = {}
        for p in ("8,22,24", "8,30,32"):
            Bc = DeviceBatch(rb, ctx, torch, local, n, L, first_block, tuple(int(x) for x in p.split(",")), a.model)
            Bc.enc(); Bc.dec()
            cb = Bc.check(torch)
            ce, cd = Bc.timed(torch, max(2, min(a.steps, 3)), barrier)
            ce, cd = rank_max([ce, cd])
            classes[p] = {"encode_ms": round(ce * 1e3, 3), "decode_ms": round(cd * 1e3, 3),
                          "value": round(world * raw_bytes / (ce + cd) / 1e6, 2), "unit": UNIT,
                          "compressed_bytes": cb, "dtype": arith_dtype(tuple(int(x) for x in p.split(",")))}
            del Bc
            torch.cuda.empty_cache()

    # ---- strong scaling: ONE n-block list over the ranks by contiguous ranges (SURVEY.md 8(e))
    strong = None
    if world > 1 and not a.no_strong:
        s_first, s_count = sharding.shard_range(n, world, rank)
        Bs = DeviceBatch(rb, ctx, torch, local, s_count, L, s_first, params, a.model)
        for _ in range(2):
            Bs.enc(); Bs.dec()
        Bs.check(torch)
        se, sd = Bs.timed(torch, a.steps, barrier)
        s_step, se, sd = rank_max([se + sd, se, sd])
        strong = {"value": round(raw_bytes / s_step / 1e6, 2), "unit": UNIT, "ms_per_step": round(s_step * 1e3, 3),
                  "encode_ms": round(se * 1e3, 3), "decode_ms": round(sd * 1e3, 3), "blocks_per_gpu": s_count,
                  "total_blocks": n, "scaling": "strong",
                  "note": "a lane needs the same time for its block however few blocks are resident (serial chain per "
                          "stream), so the per-GPU time falls only from ~3.5 warps per scheduler contending for issue "
                          "slots to fewer; the limiting kernel is decode_lane_al_kernel's dependent chain"}
        del Bs
        torch.cuda.empty_cache()

    # ---- end to end through the host-buffer C ABI, pinned host memory
    e2e = None
    ctx_rec = None
    if not a.no_e2e:
        h_raw = torch.empty(n * L, dtype=torch.uint8, pin_memory=True)
        h_raw.copy_(B.raw)
        h_comp = torch.empty(B.cap, dtype=torch.uint8, pin_memory=True)
        h_back = torch.empty(n * L, dtype=torch.uint8, pin_memory=True)
        torch.cuda.synchronize()
        t_copy, _ = copy_ceiling(torch, h_back, h_comp, B.back, B.comp, comp_bytes, barrier)
        t_copy = rank_max([t_copy])[0]
        np_raw, np_comp, np_back = h_raw.numpy(), h_comp.numpy(), h_back.numpy()
        np_off = np.arange(n + 1, dtype=np.uint64) * np.uint64(L)
        model = B.model
        del B                                  # the host API stages in its own device buffers
        torch.cuda.empty_cache()

        def e2e_step(c, src, dst_comp, dst_back):
            out, out_off, st = c.encode_batch(src, np_off, model, out=dst_comp)
            c.decode_batch(dst_comp, out_off, np_off, model, raw=dst_back)
            return int(out_off[-1])

        def e2e_time(c, src, dst_comp, dst_back, k, sync_ranks=True):
            e2e_step(c, src, dst_comp, dst_back)
            if sync_ranks:
                barrier()
            t0 = time.perf_counter()
            for _ in range(k):
                cb = e2e_step(c, src, dst_comp, dst_back)
            torch.cuda.synchronize()
            t = (time.perf_counter() - t0) / k
            assert (dst_back == src).all()
            return t, cb

        ksteps = max(1, min(a.steps, 3))
        t_e2e, cb = e2e_time(ctx, np_raw, np_comp, np_back, ksteps)
        t_e2e = rank_max([t_e2e])[0]
        meta = 8 * (n + 1)
        ceiling = world * raw_bytes / t_copy / 1e6
        e2e = {"value": round(world * raw_bytes / t_e2e / 1e6, 2), "unit": UNIT,
               "h2d_bytes_per_step": raw_bytes + meta + cb + 2 * meta,
               "d2h_bytes_per_step": cb + meta + 4 * n + raw_bytes + 20 * n,
               "ms_per_step": round(t_e2e * 1e3, 2), "steps": ksteps, "timer": "host wall clock around the C-ABI calls",
               "host_memory": "pinned (cudaHostAlloc)", "cuda_device_max_connections": queues,
               "copy_ceiling": {"value": round(ceiling, 2), "unit": UNIT, "ms_per_step": round(t_copy * 1e3, 2),
                                "what": "bare pinned copies of the same bytes, up and down concurrently, all ranks at once"},
               "frac_of_copy_ceiling": round(world * raw_bytes / t_e2e / 1e6 / ceiling, 4)}

        # what a caller holding plain (pageable) buffers gets, and what page-locking them in place gives (N = 1)
        if world == 1 and not a.no_host_memory_kinds:
            p_raw = np.empty_like(np_raw); p_raw[:] = np_raw
            p_comp = np.empty_like(np_comp); p_back = np.empty_like(np_back)
            p_comp[:] = 0; p_back[:] = 0                  # touch: the pages must exist before they are timed
            tp, _ = e2e_time(ctx, p_raw, p_comp, p_back, 2, sync_ranks=False)
            e2e["pageable"] = {"value": round(raw_bytes / tp / 1e6, 2), "unit": UNIT, "ms_per_step": round(tp * 1e3, 2),
                               "host_memory": "pageable numpy buffers (what a Vec<u8> is), staged by the library through "
                                              "its pinned ring and host copy threads (redux_ctx_set_staging defaults)"}
            ctx.set_staging(False)
            td, _ = e2e_time(ctx, p_raw, p_comp, p_back, 1, sync_ranks=False)
            ctx.set_staging(True)
            e2e["pageable_driver_staged"] = {"value": round(raw_bytes / td / 1e6, 2), "unit": UNIT, "ms_per_step": round(td * 1e3, 2),
                                             "host_memory": "the same buffers handed to cudaMemcpyAsync as they are "
                                                            "(round-1 behaviour: the driver's synchronous staging)"}
            t0 = time.perf_counter()
            for arr in (p_raw, p_comp, p_back):
                rb.host_register(arr)
            t_reg = time.perf_counter() - t0
            tr_, _ = e2e_time(ctx, p_raw, p_comp, p_back, 1, sync_ranks=False)
            for arr in (p_raw, p_comp, p_back):
                rb.host_unregister(arr)
            e2e["registered"] = {"value": round(raw_bytes / tr_ / 1e6, 2), "unit": UNIT, "ms_per_step": round(tr_ * 1e3, 2),
                                 "host_memory": "the same buffers after redux_host_register",
                                 "register_ms_once": round(t_reg * 1e3, 1)}
            del p_raw, p_comp, p_back

        # ---- the library's own multi-device front end (SURVEY.md 8(e)): one context over all N GPUs, rank 0 drives,
        # the other ranks idle at the barrier.  Parity first (ragged batch, uneven shards), then the whole batch e2e.
        if world > 1 and not a.no_ctx:
            barrier()
            if rank == 0:
                ctx_rec = multi_device_ctx(rb, o, np, world, np_raw, np_off, np_comp, np_back, model, a, raw_bytes, threads)
            barrier()

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": round(t_step * 1e3, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": arith_dtype(params), "data": "synthetic",
            "config": {"workload": workload_name(a, world), "per_gpu_raw_bytes": raw_bytes,
                       "total_raw_bytes": world * raw_bytes, "total_blocks": world * n,
                       "compressed_bytes": comp_bytes, "ratio": round(raw_bytes / comp_bytes, 4),
                       "l2_policy": "inputs (4 GiB raw + streams) far exceed the 126 MB L2; no flush needed",
                       "parallelism": "blocks sharded by rank, no collective", "host_binding": numa},
            "encode_MBps": round(world * raw_bytes / t_e / 1e6, 2),
            "decode_MBps": round(world * raw_bytes / t_d / 1e6, 2),
            "parity_checked_blocks": parity_checked,
            "parity": "the streams of the first blocks of every rank's timed batch equal the CPU oracle's byte for "
                      "byte; the whole batch round-trips",
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "classes": classes, "strong": strong,
            "multi_device_ctx": ctx_rec, "multi_device_ctx_parity": (ctx_rec or {}).get("parity"),
            "gpu_launches": launches, "clocks": clocks, "wall_s_timed_region": round(wall, 3),
        }
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    ctx.close()
    return 0


def multi_device_ctx(rb, o, np, world, np_raw, np_off, np_comp, np_back, model, a, raw_bytes, threads):
    """One redux_ctx over `world` GPUs (contiguous block ranges per device inside the library, one host thread per
    device): bytes must equal a single-device context's and the oracle's; then the whole batch end to end."""
    n_par, Lp = 3001, 2500                                  # odd count: uneven shards; ragged: empty and short blocks
    rawp = o.generate_blocks(0, n_par, Lp, SEED)
    lens = np.full(n_par, Lp, dtype=np.uint64); lens[::7] = 0; lens[5::11] = 17
    off = np.zeros(n_par + 1, dtype=np.uint64); np.cumsum(lens, out=off[1:])
    data = np.concatenate([rawp[i * Lp:i * Lp + int(lens[i])] for i in range(n_par)])
    okind = o.TREE if a.model == "tree" else o.LINEAR
    params = tuple(int(x) for x in a.params.split(","))
    rec = {"devices": world, "parity_blocks": n_par}
    with rb.Context([0]) as one:
        ref_comp, ref_off, _ = one.encode_batch(data, off, model)
    with rb.Context(list(range(world))) as many:
        comp, coff, st = many.encode_batch(data, off, model)
        ok = comp.tobytes() == ref_comp.tobytes() and bool((coff == ref_off).all()) and bool((st == 0).all())
        back, rl, cons, st = many.decode_batch(comp, coff, off, model)
        ok = ok and bool((st == 0).all()) and bool((rl == lens).all()) and back[:int(off[-1])].tobytes() == data.tobytes()
        rc, slots, slot_off, out_len, status = o.compress_batch(data, off, okind, params, threads)
        ok = ok and rc == 0 and all(
            comp[int(coff[i]):int(coff[i + 1])].tobytes() == slots[int(slot_off[i]):int(slot_off[i]) + int(out_len[i])].tobytes()
            for i in range(n_par))
        rec["parity"] = bool(ok)
        # the whole batch through the one context, end to end from pinned memory (strong scaling of the library call)
        many.encode_batch(np_raw, np_off, model, out=np_comp)
        t0 = time.perf_counter()
        out, out_off, st = many.encode_batch(np_raw, np_off, model, out=np_comp)
        t1 = time.perf_counter()
        many.decode_batch(np_comp, out_off, np_off, model, raw=np_back)
        t2 = time.perf_counter()
        assert (np_back == np_raw).all()
        rec.update({"e2e_value": round(raw_bytes / (t2 - t0) / 1e6, 2), "unit": UNIT,
                    "encode_ms": round((t1 - t0) * 1e3, 2), "decode_ms": round((t2 - t1) * 1e3, 2),
                    "what": "ONE block list of %d blocks through one context over %d devices, host buffers" % (a.blocks, world)})
    return rec


def main():
    a = parse_args()
    if a.impl == "reference":
        return run_reference(a)
    return run_ours(a)


if __name__ == "__main__":
    sys.exit(main())
