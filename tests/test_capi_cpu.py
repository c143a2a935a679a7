"""C-ABI library checks that need no GPU: it loads, exports every symbol include/redux_b200.h declares,
and its host-side arithmetic (Parameters, count reciprocals, closed-form renormalisation, generator)
agrees with the oracle / the reference's loop."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import oracle_lib as o
import redux_b200 as rb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "redux_b200.h")).read()
    names = sorted(set(re.findall(r"\b(redux_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 20
    L = rb.lib()
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing


def test_error_strings_match_reference_display():
    """src/lib.rs:66-73."""
    L = rb.lib()
    assert L.redux_error_string(rb.EOF) == b"Unexpected end of file"
    assert L.redux_error_string(rb.INVALID_INPUT) == b"Invalid data found while processing input"
    assert L.redux_error_string(rb.IO_ERROR).startswith(b"I/O error")


def test_parameters_new_matches_oracle_everywhere():
    """Same acceptance set and same derived constants as Parameters::new (src/model/mod.rs:63-81)."""
    for s in range(0, 14):
        for f in range(0, 36):
            for c in range(0, 66, 1):
                rc, p = o.params_new(s, f, c)
                try:
                    q = rb.Parameters(s, f, c)
                    ok = True
                except rb.InvalidInput:
                    ok = False
                assert ok == (rc == o.OK), (s, f, c)
                if ok:
                    for name, _ in o.Params._fields_:
                        assert getattr(q, name) == getattr(p, name), (s, f, c, name)


def test_params_supported_scope():
    L = rb.lib()
    mk = lambda s, f, c: C.byref(rb._ParamsC(s, f, c))
    assert L.redux_params_supported(mk(8, 14, 16)) == rb.OK
    assert L.redux_params_supported(mk(8, 30, 34)) == rb.OK
    assert L.redux_params_supported(mk(4, 10, 16)) == rb.OK          # generic path: any width up to 16
    assert L.redux_params_supported(mk(12, 14, 16)) == rb.OK
    assert L.redux_params_supported(mk(16, 18, 20)) == rb.OK
    assert L.redux_params_supported(mk(17, 19, 21)) == rb.UNSUPPORTED
    assert L.redux_params_supported(mk(8, 9, 16)) == rb.INVALID_INPUT


def test_compress_bound():
    assert rb.compress_bound(0, 16) == 2 and rb.compress_bound(0, 32) == 4
    assert rb.compress_bound(65536, 16) == (65537 * 16 + 7) // 8


def _magic(d, nbits, wide):
    m, sh = C.c_uint64(), C.c_uint32()
    assert rb.lib().redux_debug_magic(d, nbits, wide, C.byref(m), C.byref(sh)) == rb.OK
    return m.value, sh.value


@pytest.mark.parametrize("nbits,wide", [(22, 0), (26, 0), (30, 0), (34, 1), (46, 1), (54, 1), (62, 1)])
def test_count_reciprocal_is_exact(nbits, wide):
    """floor(n/d) == mulhi(n, magic) >> shift for every count d the coder can see and adversarial n."""
    rng = np.random.default_rng(nbits)
    L = rb.lib()
    fmax_bits = min(30, nbits - 12)
    ds = [257, 258, 259, 511, 512, 513, 1023, 1024, 1025, 4095, 4096, 16383, 65535, 65536, 65537,
          (1 << fmax_bits) - 1, (1 << fmax_bits) - 2]
    ds += [int(x) for x in rng.integers(257, 1 << fmax_bits, size=60)]
    top = (1 << nbits) - 1
    for d in ds:
        if d >= (1 << fmax_bits):
            continue
        m, sh = _magic(d, nbits, wide)
        assert m < (1 << (64 if wide else 32))
        ns = [0, 1, d - 1, d, d + 1, 2 * d - 1, 2 * d, top, top - 1, (top // d) * d, (top // d) * d - 1]
        ns += [int(x) for x in rng.integers(0, top, size=200, dtype=np.uint64)]
        ks = [int(x) for x in rng.integers(1, max(2, top // d), size=100, dtype=np.uint64)]
        ns += [k * d - 1 for k in ks] + [k * d for k in ks]
        for n in ns:
            n = int(n)
            if 0 <= n <= top:
                assert L.redux_debug_magic_divide(n, m, sh, wide) == n // d, (n, d, nbits)


def test_count_reciprocal_65_bit_is_exact_for_every_64_bit_numerator():
    """code_bits > 32: numerators reach 2^64 - 1 (code + freq <= 64), so the magic is 2^64 + m' and the product is
    formed without the carry.  Exact for counts up to freq_max (2^31 - 1) and adversarial 64-bit numerators."""
    rng = np.random.default_rng(65)
    L = rb.lib()
    top = (1 << 64) - 1
    ds = [257, 258, 511, 512, 513, 65535, 65536, 65537, (1 << 20) + 1, (1 << 31) - 1, (1 << 31) - 2, 1 << 30]
    ds += [int(x) for x in rng.integers(257, 1 << 31, size=80)]
    for d in ds:
        m, sh = _magic(d, 0, 2)
        assert m < (1 << 64) and sh >= 9
        ns = [0, 1, d - 1, d, d + 1, top, top - 1, (top // d) * d, (top // d) * d - 1, 1 << 63, (1 << 63) - 1]
        ns += [int(x) for x in rng.integers(0, top, size=200, dtype=np.uint64)]
        ks = [int(x) for x in rng.integers(1, top // d, size=100, dtype=np.uint64)]
        ns += [k * d - 1 for k in ks] + [k * d for k in ks]
        for n in ns:
            assert L.redux_debug_magic_divide(int(n), m, sh, 2) == int(n) // d, (n, d)


def test_count_reciprocal_double_is_exact_below_its_bound():
    """WIDE_D: floor(cum * range / d) as trunc(fma(n, 1/d, 2^-19)) for every total d < 349,525, cum <= d,
    range <= 2^32 -- exact multiples, their neighbours (the cases a rounding error could tip) and random products."""
    rng = np.random.default_rng(17)
    L = rb.lib()
    top = 349525
    ds = [257, 258, 511, 512, 513, 4095, 4096, 65535, 65536, 65537, 65793, (1 << 17) - 1, 1 << 17, (1 << 18) + 1, top - 1, top - 2, 98765]
    ds += [int(x) for x in rng.integers(257, top, size=150)]
    ranges = [1 << 32, (1 << 32) - 1, (1 << 31) + 1, 1 << 24, (1 << 30) + 2, 3, 2]
    for d in ds:
        m, sh = _magic(d, 0, 3)
        cums = [0, 1, d - 1, d, d // 2, d // 3] + [int(x) for x in rng.integers(0, d + 1, size=20)]
        for r in ranges + [int(x) for x in rng.integers(2, 1 << 32, size=20, dtype=np.uint64)]:
            for cum in cums:
                n = cum * r
                assert L.redux_debug_magic_divide(n, m, sh, 3) == n // d, (n, d)
        for k in [int(x) for x in rng.integers(1, 1 << 32, size=200, dtype=np.uint64)] + [(1 << 32) - 1, 1 << 32]:
            for n in (k * d, k * d - 1, k * d + 1):                      # multiples and their neighbours, quotients up to 2^32
                assert L.redux_debug_magic_divide(n, m, sh, 3) == n // d, (n, d)
    assert _bad_magic(top, 3)


def test_quotient_by_range_is_exact_for_64_bit_operands():
    """code_bits > 32 decoder: value = X / range (src/codec.rs:131) from a double estimate and one remainder check.
    Quotients up to 2^31 - 1 (a cumulative frequency), ranges from 2^31 to 2^62, X at exact multiples, just below and
    just above them (where a rounding error would tip the estimate), and at the top of the 64-bit range."""
    rng = np.random.default_rng(64)
    L = rb.lib()
    ranges = [(1 << 31) + 1, (1 << 33) - 1, 1 << 40, (1 << 47) + 12345, (1 << 53) - 1, (1 << 53) + 1, 1 << 60, (1 << 62) - 1, 1 << 62]
    ranges += [int(x) for x in rng.integers(1 << 31, 1 << 62, size=200, dtype=np.uint64)]
    for r in ranges:
        qmax = min((1 << 31) - 1, ((1 << 64) - 1) // r)
        qs = {0, 1, 2, qmax, qmax - 1, qmax // 2, qmax // 3} | {int(x) for x in rng.integers(0, qmax + 1, size=40)}
        for q in qs:
            if q < 0:
                continue
            for x in (q * r, q * r + 1, q * r + r - 1, q * r + r // 2):
                if x < (1 << 64):
                    assert L.redux_debug_div_by_range(x, r) == x // r, (x, r)
    for x in ((1 << 64) - 1, (1 << 64) - 2, (1 << 63) + 1):
        for r in ((1 << 62), (1 << 62) - 1, (1 << 61) + 7, (1 << 40) * 3):
            if x // r < (1 << 31):
                assert L.redux_debug_div_by_range(x, r) == x // r, (x, r)


def _bad_magic(d, wide):
    m, sh = C.c_uint64(), C.c_uint32()
    return rb.lib().redux_debug_magic(d, 0, wide, C.byref(m), C.byref(sh)) == rb.INVALID_INPUT


def test_count_reciprocal_exhaustive_small():
    """All numerators for a small class: nbits=18 over d in [257, 1023]."""
    for d in range(257, 1024, 7):
        m, sh = _magic(d, 18, 0)
        n = np.arange(0, 1 << 18, dtype=np.uint64)
        got = ((n * np.uint64(m)) >> np.uint64(32)) >> np.uint64(sh)
        assert (got == n // np.uint64(d)).all(), d


def _renorm_loop(low, high, c):
    """The reference's renormalisation loop, src/codec.rs:62-89 (bits ignored)."""
    q, half, q3, mx = 1 << (c - 2), 2 << (c - 2), 3 << (c - 2), (1 << c) - 1
    n1 = k = 0
    order = []
    while True:
        if high < half or low >= half:
            n1 += 1
            order.append("e12")
        elif low >= q and high < q3:
            k += 1
            low -= q
            high -= q
            order.append("e3")
        else:
            break
        high = ((high << 1) + 1) & mx
        low = (low << 1) & mx
    return n1, k, low, high, order


@pytest.mark.parametrize("c", [12, 16, 18, 24, 30, 32, 34, 44, 61])
def test_renorm_closed_form_equals_loop(c):
    """SURVEY.md A.6: the loop is n1 E1/E2 steps followed by k E3 steps, never interleaved.
    (A degenerate interval low == high is reachable in the coder and renormalises to the full range.)"""
    rng = np.random.default_rng(c)
    L = rb.lib()
    mx = (1 << c) - 1
    cases = [(0, mx), ((1 << (c - 1)) - 1, 1 << (c - 1)), (1 << (c - 2), (3 << (c - 2)) - 1),
             ((1 << (c - 1)) - 2, (1 << (c - 1)) + 1), (mx - 1, mx), (0, 1)]
    for _ in range(3000):
        a, b = sorted(int(x) for x in rng.integers(0, mx, size=2, dtype=np.uint64, endpoint=True))
        cases.append((a, b))
        w = int(rng.integers(1, c))          # narrow intervals: many common bits
        base = int(rng.integers(0, mx - (1 << w) + 1, dtype=np.uint64)) if mx > (1 << w) else 0
        a2 = base + int(rng.integers(0, 1 << w, dtype=np.uint64))
        b2 = base + int(rng.integers(0, 1 << w, dtype=np.uint64))
        cases.append((min(a2, b2), max(a2, b2)))
        mid = 1 << (c - 1)                   # straddling the middle: E3 runs
        d1 = int(rng.integers(1, 1 << w, dtype=np.uint64)) if w > 0 else 1
        d2 = int(rng.integers(0, 1 << w, dtype=np.uint64))
        if mid - d1 >= 0 and mid + d2 <= mx:
            cases.append((mid - d1, mid + d2))
    for low, high in cases:
        n1, k, nl, nh = C.c_uint32(), C.c_uint32(), C.c_uint64(), C.c_uint64()
        L.redux_debug_renorm(low, high, c, C.byref(n1), C.byref(k), C.byref(nl), C.byref(nh))
        if low == high:
            # the loop never terminates on paper for low == high only in the sense that every step is
            # E1/E2: after c steps the registers are (0, max); the reference stops there because the
            # interval is then the full range.
            assert (n1.value, k.value, nl.value, nh.value) == (c, 0, 0, mx)
            continue
        e = _renorm_loop(low, high, c)
        assert (n1.value, k.value, nl.value, nh.value) == e[:4], (low, high, c)
        assert e[4] == ["e12"] * e[0] + ["e3"] * e[1]


def test_generator_host_is_deterministic_and_mixed():
    a = rb.generate_blocks_host(0, 8, 4096, 0x5EED202610180000)
    b = rb.generate_blocks_host(0, 8, 4096, 0x5EED202610180000)
    assert (a == b).all()
    c = rb.generate_blocks_host(4, 4, 4096, 0x5EED202610180000)
    assert (a[4 * 4096:] == c).all(), "blocks depend on the absolute block index only"
    ent = []
    for i in range(4):
        blk = a[i * 4096:(i + 1) * 4096]
        p = np.bincount(blk, minlength=256) / blk.size
        p = p[p > 0]
        ent.append(float(-(p * np.log2(p)).sum()))
    assert ent[0] > 7.8 and 4.0 < ent[1] < 5.2 and 1.6 < ent[2] < 2.3 and ent[3] < 0.5, ent


def _run_without_a_device(body):
    """Run `body` in a fresh interpreter that sees no CUDA device (CUDA_VISIBLE_DEVICES=""), so that what the library
    does without a device is checked on every machine, one with GPUs included."""
    import subprocess
    import sys
    import textwrap
    code = "import sys\nsys.path.insert(0, %r)\n" % ROOT + textwrap.dedent(body)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]


def test_no_gpu_means_cuda_error_not_fallback():
    """The product path must fail loudly without a device (no CPU fallback)."""
    _run_without_a_device("""
        import io
        import pytest
        import redux_b200 as rb
        with pytest.raises(rb.CudaError):
            rb.Context()
        with pytest.raises(rb.CudaError):
            rb.compress(io.BytesIO(b"redux"), io.BytesIO(), rb.AdaptiveTreeModel(rb.Parameters(8, 14, 16)))
    """)


def test_product_package_does_not_touch_oracle():
    """Only tests/, smoke() and bench.py's CPU legs may use oracle/; the CPU emulation of the kernels
    (tests/host_emu, RDX_HOST_EMU) is test infrastructure too and never part of the shipped library."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "redux_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", "Makefile")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "redux_oracle" not in text and "oracle_lib" not in text, os.path.join(dirpath, f)
                assert "host_emu" not in text and "cuda_shim" not in text, os.path.join(dirpath, f)
    # the shared library itself exports no emulation entry point
    import subprocess
    syms = subprocess.run(["nm", "-D", "--defined-only", os.path.join(ROOT, "redux_b200", "libredux_b200.so")],
                          capture_output=True, text=True).stdout
    assert "emu_" not in syms and "oracle_" not in syms


def test_oracle_side_generator_equals_the_products_host_generator():
    """bench.py's CPU arm generates its input with oracle/synth_blocks.c so that it never maps the product
    library; the bytes must be the ones the product's generator (and therefore the GPU) produces."""
    import oracle_lib as o
    seed = 0x5EED202610180000
    for first, n, L in ((0, 64, 4096), (5, 9, 1001), (65530, 8, 65536), (3, 4, 7)):
        assert (o.generate_blocks(first, n, L, seed) == rb.generate_blocks_host(first, n, L, seed)).all()
    # with a corpus: the text class is a window of it, the other classes are unchanged
    corpus = np.frombuffer(bytes(range(256)) * 300, dtype=np.uint8)            # 76,800 bytes
    for first, n, L in ((0, 16, 4096), (1, 5, 65536), (1, 3, 76800)):
        a, b = o.generate_blocks(first, n, L, seed, corpus=corpus), rb.generate_blocks_host(first, n, L, seed, corpus=corpus)
        assert (a == b).all()
        plain = rb.generate_blocks_host(first, n, L, seed)
        for i in range(n):
            blk = a[i * L:(i + 1) * L]
            if (first + i) & 3 == 1:
                at = int(blk[0])
                assert (blk == corpus[at:at + L]).all()                       # a window: consecutive byte values
            else:
                assert (blk == plain[i * L:(i + 1) * L]).all()


def test_process_init_is_explicit_and_respects_the_applications_setting():
    """Loading the library must not touch the process environment (round 1 set CUDA_DEVICE_MAX_CONNECTIONS from a
    load-time constructor); redux_process_init() sets it to 32 only when the application has not set it."""
    import subprocess
    import sys
    code = (
        "import os, sys\n"
        "sys.path.insert(0, %r)\n"
        "import redux_b200 as rb\n"
        "rb.lib()\n"
        "before = os.environ.get('CUDA_DEVICE_MAX_CONNECTIONS')\n"
        "import ctypes\n"
        "libc = ctypes.CDLL(None); libc.getenv.restype = ctypes.c_char_p\n"
        "raw_before = libc.getenv(b'CUDA_DEVICE_MAX_CONNECTIONS')\n"
        "v = rb.process_init()\n"
        "raw_after = libc.getenv(b'CUDA_DEVICE_MAX_CONNECTIONS')\n"
        "print(repr((raw_before, v, raw_after)))\n"
    ) % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = {k: v for k, v in os.environ.items() if k != "CUDA_DEVICE_MAX_CONNECTIONS"}
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=120)
    assert out.returncode == 0, out.stderr[-1500:]
    assert eval(out.stdout.strip().splitlines()[-1]) == (None, 32, b"32")          # untouched by loading, set by the call
    env["CUDA_DEVICE_MAX_CONNECTIONS"] = "4"
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=120)
    assert eval(out.stdout.strip().splitlines()[-1]) == (b"4", 4, b"4")             # the application's setting wins


def test_pinned_memory_entry_points_fail_loudly_without_a_device():
    """No device: page-locking needs CUDA, and the entry points say so instead of handing out pageable memory."""
    _run_without_a_device("""
        import ctypes as C
        import numpy as np
        import redux_b200 as rb
        p = C.c_void_p()
        assert rb.lib().redux_host_alloc(4096, C.byref(p)) == rb.CUDA_ERROR and not p.value
        buf = np.zeros(4096, dtype=np.uint8)
        assert rb.lib().redux_host_register(buf.ctypes.data, buf.nbytes) == rb.CUDA_ERROR
        assert rb.lib().redux_host_alloc(0, C.byref(p)) == rb.OK          # nothing to allocate
    """)
