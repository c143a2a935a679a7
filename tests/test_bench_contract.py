"""bench.py's JSON line against the driver's contract, checked on the committed record of the last GPU run
(profiles/r02_bench_default.json, profiles/r02_bench_reference_arm.json).  No GPU needed, except for the `-m gpu`
test of --dump-outputs."""
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASELINE = json.load(open(os.path.join(ROOT, "BASELINE.json")))


def _load(name):
    return json.load(open(os.path.join(ROOT, "profiles", name)))


def test_our_arm_line_has_every_contract_key():
    d = _load("r02_bench_default.json")
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert k in d, k
    assert d["unit"] == "MB/s" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and BASELINE["published"] == {}          # no published number to compare with
    assert d["data"] == "synthetic" and "workload" in d["config"] and "65536 x 65536" in d["config"]["workload"]
    assert d["warmup"] >= 3 and d["n_gpus"] == 1 and d["gpu_launches"] > 0
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3
    assert r["traffic"] is None or r["traffic"] >= r["algorithmic_bytes_per_launch"] * 0.9
    c = d["cpu_baseline"]
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in c, k
    assert c["kind"] in ("reference", "port") and c["cores"] >= 1
    e = d["e2e"]
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in e, k
    assert e["h2d_bytes_per_step"] > d["config"]["per_gpu_raw_bytes"] and e["value"] < d["value"]
    assert e["value"] > 50 * c["value"]                                      # the GPU path end to end vs the host cores
    # round 2: the line proves what it claims and carries the other classes, the copy ceiling and the host-memory kinds
    assert d["parity_checked_blocks"] >= 64
    assert set(d["classes"]) == {"8,22,24", "8,30,32"} and all(v["decode_ms"] > 0 for v in d["classes"].values())
    assert 0.5 < e["frac_of_copy_ceiling"] <= 1.0 and e["copy_ceiling"]["value"] >= e["value"]
    assert e["pageable"]["value"] < e["value"] and e["registered"]["value"] > 0.8 * e["value"]
    assert "Calgary+Canterbury" in d["config"]["workload"]
    k = d["clocks"]
    assert not set(k["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert k["sm_mhz"] and k["sm_mhz"] > 0.9 * k["sm_max_mhz"]


def test_reference_arm_line():
    d = _load("r02_bench_reference_arm.json")
    assert d["impl"] == "reference" and d["unit"] == "MB/s" and d["gpu_launches"] == 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    ours = _load("r02_bench_default.json")
    assert d["metric"] == ours["metric"] and d["config"]["workload"] == ours["config"]["workload"]


def test_reference_arm_runs_without_mapping_the_product_library():
    """The CPU arm generates its input with oracle/synth_blocks.c and codes with oracle/redux_oracle.c: after a
    run, /proc/self/maps of that process holds the oracle library and not libredux_b200.so."""
    import subprocess
    import sys
    code = (
        "import sys, io, json, contextlib\n"
        "sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0', '--cpu-sample-blocks', '8']\n"
        "sys.path.insert(0, %r)\n"
        "import bench\n"
        "buf = io.StringIO()\n"
        "with contextlib.redirect_stdout(buf):\n"
        "    bench.run_reference(bench.parse_args())\n"
        "maps = open('/proc/self/maps').read()\n"
        "d = json.loads(buf.getvalue())\n"
        "print(json.dumps({'oracle': 'libredux_oracle' in maps, 'product': 'libredux_b200' in maps, 'line': d}))\n"
    ) % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["oracle"] and not out["product"]
    line = out["line"]
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["cpu_baseline"]["per_thread_MBps"] > 0 and line["cpu_baseline"]["MiBps"] > 0


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_steps_computed(tmp_path):
    """--dump-outputs: float .npy files within the size limit, the same for the same workload whatever --steps and
    --warmup (0 included), every block decoded whole, and the sampled streams / decoded blocks equal to the oracle's
    streams / the generated input."""
    import subprocess
    import sys

    import numpy as np

    import bench
    import oracle_lib as o
    n, L = 256, 65536
    dumps = []
    for steps, warmup in ((1, 0), (2, 1)):
        d = tmp_path / ("s%d_w%d" % (steps, warmup))
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                            "--blocks", str(n), "--block-len", str(L), "--no-e2e", "--no-classes", "--no-cpu-baseline",
                            "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        assert sum(f.stat().st_size for f in d.iterdir()) <= bench.DUMP_LIMIT
        dumps.append({f.stem: np.load(f) for f in d.iterdir()})
    a, b = dumps
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert (a["status"] == 0).all() and (a["raw_lens"] == L).all()
    assert (a["consumed"] == np.diff(a["compressed_offsets"])).all()
    idx, s_off = a["sample_blocks"].astype(np.int64), a["sample_compressed_offsets"].astype(np.int64)
    assert 0 < idx.size < n and a["sample_decoded"].shape == (idx.size, L)
    raw = o.generate_blocks(0, n, L, bench.SEED, corpus=bench.text_corpus())
    for j, i in enumerate(idx):
        block = raw[i * L:(i + 1) * L]
        assert a["sample_compressed"][s_off[j]:s_off[j + 1]].astype(np.uint8).tobytes() == o.compress(block, o.TREE, (8, 14, 16))[1]
        assert (a["sample_decoded"][j].astype(np.uint8) == block).all()
