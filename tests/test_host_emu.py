"""The lane kernels' arithmetic, executed on the CPU, against the oracle (no GPU needed).

tests/host_emu/ compiles redux_b200/csrc/redux_lane_codec.cuh with g++ through a shim of the CUDA device
vocabulary and runs the kernels thread by thread (the lane mapping has no barriers or warp collectives, so
that is exactly what the GPU computes).  This is test infrastructure: it catches a wrong bit in a kernel
change before GPU minutes are spent; the shipped library has no CPU path and the `-m gpu` parity tests
remain the proof for the real device.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as o

HERE = os.path.dirname(os.path.abspath(__file__))
EMU_DIR = os.path.join(HERE, "host_emu")
EMU_SO = os.path.join(EMU_DIR, "_lane_emu.so")
CSRC = os.path.join(os.path.dirname(HERE), "redux_b200", "csrc")
SEED = 0x5EED202610180000


def _build():
    srcs = [os.path.join(EMU_DIR, "lane_emu.cpp"), os.path.join(EMU_DIR, "cuda_shim.h"),
            os.path.join(CSRC, "redux_lane_codec.cuh"), os.path.join(CSRC, "redux_lane_al.cuh"),
            os.path.join(CSRC, "redux_generic_codec.cuh"), os.path.join(CSRC, "redux_common.cuh")]
    if os.path.exists(EMU_SO) and all(os.path.getmtime(s) <= os.path.getmtime(EMU_SO) for s in srcs):
        return
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas",
                    "-o", EMU_SO, srcs[0]], check=True, cwd=EMU_DIR)


@pytest.fixture(scope="module")
def emu():
    return load_emu()


def load_emu():
    _build()
    L = C.CDLL(EMU_SO)
    u32, u64, vp, i32 = C.c_uint32, C.c_uint64, C.c_void_p, C.c_int
    L.emu_slot_stride.argtypes = [u32, u32, u64]
    L.emu_slot_stride.restype = u64
    L.emu_lane_plan.argtypes = [u32, u32, u64, u32, i32, vp]
    L.emu_lane_plan.restype = None
    L.emu_encode_lane.argtypes = [u32, u32, u64, i32, vp, vp, u64, vp, vp, vp]
    L.emu_decode_lane.argtypes = [u32, u32, u64, i32, vp, vp, u64, vp, vp, vp, vp, vp]
    L.emu_encode_lane_ex.argtypes = [u32, u32, u64, i32, vp, vp, vp, u64, vp, vp, vp]
    L.emu_decode_lane_ex.argtypes = [u32, u32, u64, i32, vp, vp, vp, u64, vp, vp, vp, vp, vp]
    L.emu_encode_generic.argtypes = [u32, u32, u32, vp, u32, vp, vp, u64, vp, u64, vp, vp]
    L.emu_decode_generic.argtypes = [u32, u32, u32, vp, u32, vp, vp, u64, vp, vp, vp, vp, vp]
    return L


def concat(blocks):
    lens = np.array([len(b) for b in blocks], dtype=np.uint64)
    off = np.zeros(len(blocks) + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    # pad: the kernels read whole aligned 16-byte chunks around a stream (alignment contract of the C ABI)
    data = np.zeros(int(off[-1]) + 64, dtype=np.uint8)
    data[:int(off[-1])] = np.frombuffer(b"".join(blocks), dtype=np.uint8)
    return data, off


def emu_encode(emu, blocks, f, c, wide=-1, freq=None):
    data, off = concat(blocks)
    n = len(blocks)
    max_len = max((len(b) for b in blocks), default=0)
    stride = emu.emu_slot_stride(f, c, max_len)
    slots = np.zeros(n * stride + 64, dtype=np.uint8)
    # 16-byte aligned base
    base = (-slots.ctypes.data) % 16
    sizes = np.zeros(n, dtype=np.uint32)
    status = np.full(n, -1, dtype=np.int32)
    fq = None if freq is None else np.ascontiguousarray(freq, dtype=np.uint32)
    emu.emu_encode_lane_ex(f, c, max_len, wide, None if fq is None else fq.ctypes.data, data.ctypes.data,
                           off.ctypes.data, n, slots.ctypes.data + base, sizes.ctypes.data, status.ctypes.data)
    assert (status == 0).all()
    return [slots[base + i * stride: base + i * stride + int(sizes[i])].tobytes() for i in range(n)]


def emu_decode(emu, streams, caps, f, c, wide=-1, freq=None):
    comp, coff = concat(streams)
    n = len(streams)
    roff = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(np.array(caps, dtype=np.uint64), out=roff[1:])
    raw = np.zeros(int(roff[-1]) + 64, dtype=np.uint8)
    raw_len = np.zeros(n, dtype=np.uint64)
    consumed = np.zeros(n, dtype=np.uint64)
    status = np.full(n, -1, dtype=np.int32)
    fq = None if freq is None else np.ascontiguousarray(freq, dtype=np.uint32)
    emu.emu_decode_lane_ex(f, c, max(caps, default=0), wide, None if fq is None else fq.ctypes.data, comp.ctypes.data,
                           coff.ctypes.data, n, raw.ctypes.data, roff.ctypes.data, raw_len.ctypes.data,
                           consumed.ctypes.data, status.ctypes.data)
    outs = [raw[int(roff[i]): int(roff[i]) + int(raw_len[i])].tobytes() for i in range(n)]
    return outs, raw_len, consumed, status


def make_blocks(rng, n, max_len):
    """Mixed entropy classes and ragged lengths (incl. empty and 1-byte blocks)."""
    blocks = []
    for i in range(n):
        L = [0, 1, 2, 3, 5, 15, 16, 17, 31, 33][i] if i < 10 else int(rng.integers(0, max_len + 1))
        k = i & 3
        if k == 0:
            b = rng.integers(0, 256, L, dtype=np.uint8)
        elif k == 1:
            b = rng.choice(np.frombuffer(b" etaoinshrdlu\n", dtype=np.uint8), L)
        elif k == 2:
            b = np.minimum(rng.geometric(0.5, L) - 1, 255).astype(np.uint8)
        else:
            b = np.where(rng.random(L) < 0.98, 0, rng.integers(0, 256, L)).astype(np.uint8)
        blocks.append(b.tobytes())
    return blocks


# (f, c): narrow incl. the frozen regime (f=10 freezes after 766 symbols), wide, c == 32, huge
PARAMS = [(10, 12), (10, 16), (14, 16), (12, 18), (16, 18), (22, 24), (20, 31), (30, 32), (24, 30), (30, 34), (20, 40),
          (10, 30), (12, 32), (10, 21),      # 64-bit-product classes that freeze early (tree-based frozen decoder)
          (10, 40), (10, 54)]                 # the same with code_bits > 32 (64-bit coder state)


@pytest.mark.parametrize("f,c", PARAMS)
def test_lane_kernels_equal_oracle(emu, f, c):
    rng = np.random.default_rng(1000 * f + c)
    blocks = make_blocks(rng, 40, 3000)
    blocks.append(bytes([255] * 2000))                    # symbol 255: the unstored node 256 path
    blocks.append(bytes(rng.integers(250, 256, 2500, dtype=np.uint8)))
    want = []
    for b in blocks:
        rc, out, ic, oc = o.compress(b, o.TREE, (8, f, c))
        assert rc == o.OK
        want.append(out)
    got = emu_encode(emu, blocks, f, c)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, "encode block %d (len %d) (8,%d,%d): %s vs %s" % (i, len(blocks[i]), f, c, g[:12].hex(), w[:12].hex())
    outs, raw_len, consumed, status = emu_decode(emu, want, [len(b) + 3 for b in blocks], f, c)
    assert (status == 0).all(), status
    for i, b in enumerate(blocks):
        assert outs[i] == b, "decode block %d (8,%d,%d)" % (i, f, c)
        assert int(consumed[i]) == len(want[i])


def test_wide_table_variant_and_long_frozen_block(emu):
    """u32 table entries (chosen when a block can make > 65,536 updates) and a block far past the freeze."""
    rng = np.random.default_rng(7)
    blocks = make_blocks(rng, 12, 9000) + [bytes(rng.integers(0, 4, 70000, dtype=np.uint8))]
    for f, c, wide in ((14, 16, 1), (22, 24, 1), (16, 18, -1), (17, 20, -1)):
        want = [o.compress(b, o.LINEAR, (8, f, c))[1] for b in blocks]
        assert emu_encode(emu, blocks, f, c, wide) == want
        outs, raw_len, consumed, status = emu_decode(emu, want, [len(b) for b in blocks], f, c, wide)
        assert (status == 0).all() and outs == blocks


def test_truncated_streams_and_full_sinks(emu):
    """Err(Eof) on a truncated stream leaves the decoded prefix (src/codec.rs:49-52 via get_bit);
    a full output slot reports OUT_CAPACITY; an exactly-full slot is fine."""
    rng = np.random.default_rng(11)
    f, c = 14, 16
    blocks = make_blocks(rng, 16, 1200)[4:]
    streams = [o.compress(b, o.TREE, (8, f, c))[1] for b in blocks]
    cut = [s[: max(0, len(s) - 1 - (i % 5))] for i, s in enumerate(streams)] + [b"", b"\xff"]
    caps = [len(b) + 8 for b in blocks] + [8, 8]
    outs, raw_len, consumed, status = emu_decode(emu, cut, caps, f, c)
    for i, s in enumerate(cut):
        rc, out, ic, oc = o.decompress(s, o.TREE, (8, f, c), out_cap=caps[i])
        assert int(status[i]) == rc, (i, int(status[i]), rc)
        assert outs[i] == out and int(consumed[i]) == ic, (i, len(outs[i]), len(out), int(consumed[i]), ic)
    # exact capacity: OK; one byte short: OUT_CAPACITY (6) with the prefix in place
    outs, raw_len, consumed, status = emu_decode(emu, streams, [len(b) for b in blocks], f, c)
    assert (status == 0).all() and outs == blocks
    nonempty = [(s, b) for s, b in zip(streams, blocks) if len(b)]
    outs, raw_len, consumed, status = emu_decode(emu, [s for s, _ in nonempty], [len(b) - 1 for _, b in nonempty], f, c)
    assert (status == 6).all()
    assert all(outs[i] == b[:-1] for i, (_, b) in enumerate(nonempty))


def test_bit_packer_pairs_equal_single_codes(emu):
    """BitSink2::put_pair (two symbols, one append) writes the bytes of two put_code calls: random code sequences with
    settled-bit counts 0..32, E3 runs that leave the pending count anywhere from 0 to beyond 32, so that both the
    merged path (nA + nB <= 32) and its in-order fallback are taken, at every accumulator phase."""
    emu.emu_put_pairs.argtypes = [C.c_void_p] * 3 + [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]
    emu.emu_put_pairs.restype = C.c_uint32
    rng = np.random.default_rng(2)
    fallback = merged = 0
    for trial in range(400):
        n = int(rng.integers(1, 60))
        wide = trial % 4 == 0                                  # every fourth trial: long codes and long pending runs
        n1 = rng.integers(0, 33 if wide else 12, n).astype(np.uint32)
        n1[rng.random(n) < 0.2] = 0
        k = np.where(rng.random(n) < 0.3, rng.integers(0, 40 if wide else 6, n), 0).astype(np.uint32)
        bits = np.array([int(rng.integers(0, 1 << int(x))) if x else 0 for x in n1], dtype=np.uint32)
        pend0 = int(rng.integers(0, 35)) if wide else int(rng.integers(0, 3))
        cap = 8 * (int(n1.sum()) + int(k.sum()) + pend0) // 8 + 64
        a = np.zeros(cap + 64, dtype=np.uint8); b = np.zeros(cap + 64, dtype=np.uint8)
        # 16-byte aligned slots, as the kernels' (word stores)
        oa = (-a.ctypes.data) % 16; ob = (-b.ctypes.data) % 16
        same = C.c_int(0)
        la = emu.emu_put_pairs(bits.ctypes.data, n1.ctypes.data, k.ctypes.data, n, pend0, a.ctypes.data + oa, b.ctypes.data + ob, C.byref(same))
        assert same.value == 1, (trial, n, la)
        # which path the pairs took (for the coverage assertion below)
        pend = pend0
        for i in range(0, n - 1, 2):
            na = int(n1[i]) + pend if n1[i] else 0
            pend1 = (0 if n1[i] else pend) + int(k[i])
            nb = int(n1[i + 1]) + pend1 if n1[i + 1] else 0
            pend = (0 if n1[i + 1] else pend1) + int(k[i + 1])
            if na + nb > 32: fallback += 1
            else: merged += 1
        # (an odd last code does not change pend's role here)
    assert fallback > 50 and merged > 1000, (fallback, merged)


def test_long_pending_runs(emu):
    """Inputs alternating around the interval midpoint keep the coder in E3 shifts (src/codec.rs:75-83; pending
    runs of ~10 bits here).  Runs far beyond 32 bits -- the packers' slow paths -- come from the adversarial
    `straddle*` golden vectors (tests/golden/make_golden.py), checked in test_kernels_equal_the_golden_vectors."""
    rng = np.random.default_rng(5)
    blocks = []
    for f, c in ((14, 16), (22, 24), (30, 32)):
        # search a few random two-symbol inputs for long runs is unreliable; use the structured input of the
        # golden generator instead: alternating 127/128 keeps the interval straddling the midpoint
        for L in (64, 500, 4000):
            blocks.append(bytes([127 + (i & 1) for i in range(L)]))
            blocks.append(bytes([128 - (i & 1) for i in range(L)]))
        want = [o.compress(b, o.TREE, (8, f, c))[1] for b in blocks]
        assert emu_encode(emu, blocks, f, c) == want
        outs, raw_len, consumed, status = emu_decode(emu, want, [len(b) for b in blocks], f, c)
        assert (status == 0).all() and outs == blocks


def _loop_step(c, low, high, cl, ch, count):
    """src/codec.rs:58-89 as written: narrow, then the E1/E2/E3 loop with put_bit (pending run starts at 0)."""
    half, q1, q3, mx = 2 << (c - 2), 1 << (c - 2), 3 << (c - 2), (1 << c) - 1
    rng = high - low + 1
    high = low + rng * ch // count - 1
    low = low + rng * cl // count
    out, pend, shifts = [], 0, 0
    while True:
        if high < half:
            out += [0] + [1] * pend; pend = 0
        elif low >= half:
            out += [1] + [0] * pend; pend = 0
        elif low >= q1 and high < q3:
            pend += 1; low -= q1; high -= q1
        else:
            break
        high = ((high << 1) + 1) & mx
        low = (low << 1) & mx
        shifts += 1
    v = 0
    for b in out:
        v = (v << 1) | b
    return low, high, shifts, v, len(out), pend


def test_al_step_closed_form_equals_loop(emu):
    """One coder step of the tuned kernels (left-aligned state, clamped shifts, FLO.SH counts) against the
    reference's renormalisation loop on random and adversarial states: collapsed intervals (low == high
    after narrowing, code_bits shifts), straddling states with long E3 runs, code_bits == 32."""
    emu.emu_step_al.argtypes = [C.c_uint32] * 7 + [C.POINTER(C.c_uint32)] * 2 + [C.POINTER(C.c_uint64)] + [C.POINTER(C.c_uint32)] * 2
    emu.emu_step_al.restype = C.c_uint32
    rng = np.random.default_rng(2026)
    for c, f in ((12, 10), (16, 14), (24, 22), (31, 20), (32, 30), (32, 12)):
        q1, half, mx = 1 << (c - 2), 2 << (c - 2), (1 << c) - 1
        fmax = (1 << f) - 1
        cases = []
        for i in range(3000):
            kind = i % 4
            if kind == 0:        # any legal state: low < half <= high or straddling quarters
                low = int(rng.integers(0, half)); high = int(rng.integers(half, mx + 1))
            elif kind == 1:      # narrowest legal range around the midpoint (long E3 runs)
                low = half - q1 // 2 - int(rng.integers(1, 3)); high = low + q1 + int(rng.integers(1, 4))
            elif kind == 2:      # tiny symbol widths: the narrowed interval collapses or nearly does
                low = int(rng.integers(0, q1)); high = low + q1 + 1 + int(rng.integers(0, 3))
            else:
                low = 0; high = mx
            high = min(high, mx)
            if high - low + 1 < q1 + 2:
                continue
            count = int(rng.integers(257, fmax + 1)) if kind != 2 else fmax
            cl = int(rng.integers(0, count)); ch = min(count, cl + (1 if kind == 2 else int(rng.integers(1, 40))))
            cases.append((low, high, cl, ch, count))
        collapsed = 0
        for low, high, cl, ch, count in cases:
            want = _loop_step(c, low, high, cl, ch, count)
            nl, nh, pa, nb = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
            bits = C.c_uint64()
            n = emu.emu_step_al(c, f, low, high, cl, ch, count, C.byref(nl), C.byref(nh), C.byref(bits), C.byref(nb), C.byref(pa))
            got = (nl.value, nh.value, n, bits.value, nb.value, pa.value)
            assert got == want, (c, f, low, high, cl, ch, count, got, want)
            collapsed += want[2] == c
        assert collapsed > 0 or f + 2 < c, "no collapsed interval exercised for (f,c)=(%d,%d)" % (f, c)


# ------------------------------------------------------------------ generic path
def gen_encode(emu, blocks, params, freq=None, n_threads=128):
    s, f, c = params
    data, off = concat(blocks)
    n = len(blocks)
    max_len = max((len(b) for b in blocks), default=0)
    bound = ((max_len * 8 // s + 1) * c + 7) // 8
    stride = ((bound + 15) & ~15) + 16
    slots = np.zeros(n * stride + 64, dtype=np.uint8)
    base = (-slots.ctypes.data) % 16
    sizes = np.zeros(n, dtype=np.uint32)
    status = np.full(n, -1, dtype=np.int32)
    fq = None if freq is None else np.ascontiguousarray(freq, dtype=np.uint32)
    emu.emu_encode_generic(s, f, c, None if fq is None else fq.ctypes.data, n_threads, data.ctypes.data,
                           off.ctypes.data, n, slots.ctypes.data + base, stride, sizes.ctypes.data, status.ctypes.data)
    assert (status == 0).all()
    return [slots[base + i * stride: base + i * stride + int(sizes[i])].tobytes() for i in range(n)]


def gen_decode(emu, streams, caps, params, freq=None, n_threads=128):
    s, f, c = params
    comp, coff = concat(streams)
    n = len(streams)
    roff = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(np.array(caps, dtype=np.uint64), out=roff[1:])
    raw = np.zeros(int(roff[-1]) + 64, dtype=np.uint8)
    raw_len = np.zeros(n, dtype=np.uint64)
    consumed = np.zeros(n, dtype=np.uint64)
    status = np.full(n, -1, dtype=np.int32)
    fq = None if freq is None else np.ascontiguousarray(freq, dtype=np.uint32)
    emu.emu_decode_generic(s, f, c, None if fq is None else fq.ctypes.data, n_threads, comp.ctypes.data,
                           coff.ctypes.data, n, raw.ctypes.data, roff.ctypes.data, raw_len.ctypes.data,
                           consumed.ctypes.data, status.ctypes.data)
    return [raw[int(roff[i]): int(roff[i]) + int(raw_len[i])].tobytes() for i in range(n)], raw_len, consumed, status


# the widths and (freq, code) pairs of the reference's model tests (src/model/tests.rs:95-251) + odd ones
GENERIC_PARAMS = [(4, 10, 16), (4, 14, 16), (4, 30, 32), (12, 14, 16), (12, 22, 24), (12, 30, 32),
                  (1, 3, 5), (3, 5, 7), (5, 8, 11), (7, 20, 40), (8, 14, 16), (16, 18, 20), (11, 31, 33)]


@pytest.mark.parametrize("params", GENERIC_PARAMS)
def test_generic_kernels_equal_oracle(emu, params):
    """Any symbol width: bytes equal compress(), decode equals decompress() -- including the reference's
    quirks for widths that do not divide 8 (trailing partial symbol dropped; decoder never flushes)."""
    rng = np.random.default_rng(sum(params))
    blocks = make_blocks(rng, 30, 600 if params[0] < 12 else 1500)
    blocks += [bytes(rng.integers(0, 256, 777, dtype=np.uint8)), bytes([0xFF] * 301)]
    want, back = [], []
    for b in blocks:
        rc, out, ic, oc = o.compress(b, o.TREE, params)
        assert rc == o.OK and ic == len(b)
        want.append(out)
        rc, dec, ic2, oc2 = o.decompress(out, o.LINEAR, params, out_cap=len(b) + 8)
        assert rc == o.OK and ic2 == len(out)
        back.append(dec)
    got = gen_encode(emu, blocks, params, n_threads=128)     # 32 blocks on 128 threads ...
    assert got == want
    got = gen_encode(emu, blocks[:20], params, n_threads=128)
    assert got == want[:20]
    outs, raw_len, consumed, status = gen_decode(emu, want, [len(b) + 8 for b in blocks], params)
    assert (status == 0).all()
    assert outs == back                                       # what decompress() writes (may lose trailing bits)
    assert [int(x) for x in consumed] == [len(w) for w in want]
    if 8 % params[0] == 0:
        assert back == blocks


def test_generic_threads_reuse_columns(emu):
    """More blocks than threads: a thread codes several blocks in turn and must reset its column."""
    rng = np.random.default_rng(3)
    params = (8, 14, 16)
    blocks = make_blocks(rng, 300, 300)
    want = [o.compress(b, o.TREE, params)[1] for b in blocks]
    assert gen_encode(emu, blocks, params, n_threads=128) == want
    outs, raw_len, consumed, status = gen_decode(emu, want, [len(b) for b in blocks], params, n_threads=128)
    assert (status == 0).all() and outs == blocks


@pytest.mark.parametrize("params", [(8, 14, 16), (8, 30, 32), (4, 10, 16), (12, 22, 24)])
def test_pretrained_models_equal_oracle(emu, params):
    """A model trained before compress()/decompress() got it (Model::get_frequency mutates,
    src/model/mod.rs:23-25): the device path starts every block from that frequency vector."""
    s, f, c = params
    rng = np.random.default_rng(s * 100 + f)
    nsym = (1 << s) + 1
    for n_train in (1, 50, 3000):
        train = rng.integers(0, min(nsym, 40), n_train)      # skewed; includes possibly freezing the model (f=10)
        freq = o.trained_frequencies(train, o.TREE, params)
        assert freq.sum() == min(nsym + n_train, (1 << f) - 1)
        blocks = make_blocks(rng, 12, 400)
        want = []
        for b in blocks:
            rc, out, ic, oc = o.compress_trained(b, train, o.LINEAR, params)
            assert rc == o.OK
            want.append(out)
        assert gen_encode(emu, blocks, params, freq=freq) == want
        outs, raw_len, consumed, status = gen_decode(emu, want, [len(b) + 4 for b in blocks], params, freq=freq)
        assert (status == 0).all()
        for i, w in enumerate(want):
            rc, dec, ic, oc = o.decompress_trained(w, train, o.TREE, params, out_cap=len(blocks[i]) + 4)
            assert rc == o.OK and outs[i] == dec and int(consumed[i]) == ic


def test_generic_truncated_and_full(emu):
    params = (12, 14, 16)
    rng = np.random.default_rng(9)
    blocks = [bytes(rng.integers(0, 256, n, dtype=np.uint8)) for n in (30, 31, 32, 33, 100, 3)]
    streams = [o.compress(b, o.TREE, params)[1] for b in blocks]
    cut = [s[:-1 - (i % 3)] for i, s in enumerate(streams)] + [b"", b"\x00"]
    caps = [len(b) + 8 for b in blocks] + [4, 4]
    outs, raw_len, consumed, status = gen_decode(emu, cut, caps, params)
    for i, s in enumerate(cut):
        rc, out, ic, oc = o.decompress(s, o.TREE, params, out_cap=caps[i])
        assert (int(status[i]), outs[i], int(consumed[i])) == (rc, out, ic), i
    # a slot one byte too small: the reference's writer fails (IoError) -> OUT_CAPACITY here, prefix in place
    outs, raw_len, consumed, status = gen_decode(emu, streams, [max(0, (len(b) * 8 // 12 * 12) // 8 - 1) for b in blocks], params)
    for i, s in enumerate(streams):
        cap = max(0, (len(blocks[i]) * 8 // 12 * 12) // 8 - 1)
        rc, out, ic, oc = o.decompress(s, o.TREE, params, out_cap=cap)
        assert rc == o.IO_ERROR and int(status[i]) == 6 and outs[i] == out, (i, rc, int(status[i]))


def test_wide_decoder_quotient_estimate_and_its_fallback(emu):
    """The wide-class decoder derives value = X / range from a float estimate while count <= 2^20 and
    falls back to the product-domain descent beyond: a 1.1 MB block crosses that boundary."""
    rng = np.random.default_rng(31)
    big = np.concatenate([rng.integers(0, 256, 400000, dtype=np.uint8),
                          rng.choice(np.frombuffer(b"acgt", dtype=np.uint8), 400000),
                          np.minimum(rng.geometric(0.3, 350000) - 1, 255).astype(np.uint8)]).tobytes()
    for f, c in ((22, 24), (30, 32)):
        rc, want, ic, oc = o.compress(big, o.TREE, (8, f, c))
        assert rc == o.OK
        assert emu_encode(emu, [big, b"abc"], f, c)[0] == want
        outs, raw_len, consumed, status = emu_decode(emu, [want], [len(big)], f, c)
        assert int(status[0]) == 0 and outs[0] == big and int(consumed[0]) == len(want)


def test_double_reciprocal_class_and_its_boundary(emu):
    """WIDE_D (totals below 349,525 for the whole launch: the two divisions by the total are one double-precision
    multiply-add each) against the oracle, on both sides of the bound: a block of 349,267 symbols keeps every total
    below it (257 + 349,267 = 349,524; 32-bit tables), one more symbol switches the launch to the 64-bit magics.  The
    quotient 2^32 (cum == total at full range, c = 32) and totals around 2^16 / 2^17 / 2^18 are all on this path."""
    rng = np.random.default_rng(349525)
    for L in (349267, 349268):
        blk = np.concatenate([rng.integers(0, 256, L // 3, dtype=np.uint8),
                              np.full(L // 3, 255, dtype=np.uint8),                    # symbol 255: cum_hi reaches cum(256)
                              np.minimum(rng.geometric(0.4, L - 2 * (L // 3)) - 1, 255).astype(np.uint8)]).tobytes()
        assert len(blk) == L
        for f, c in ((30, 32), (22, 24), (19, 21)):
            rc, want, ic, oc = o.compress(blk, o.TREE, (8, f, c))
            assert rc == o.OK
            assert emu_encode(emu, [blk, b"redux"], f, c)[0] == want, (L, f, c)
            outs, raw_len, consumed, status = emu_decode(emu, [want], [L + 1], f, c)
            assert int(status[0]) == 0 and outs[0] == blk and int(consumed[0]) == len(want), (L, f, c)


def test_kernels_equal_the_golden_vectors(emu):
    """Every committed golden vector (tests/golden/make_golden.py: an independent second reading of the
    reference, incl. odd symbol widths and models trained before the call) through the kernels that would
    code it on the device: tuned lane kernels for fresh byte models, generic kernels otherwise."""
    import json
    vecs = json.load(open(os.path.join(HERE, "golden", "kat_vectors.json")))
    assert len(vecs) >= 130
    for v in vecs:
        s, f, c = v["params"]
        data, want = bytes.fromhex(v["input"]), bytes.fromhex(v["compressed"])
        nbytes = (len(data) * 8 // s) * s // 8
        if s == 8 and (c <= 32 or "train" not in v):
            freq = None
            if "train" in v:     # trained byte model: the tuned lane kernels start from its tree
                freq = o.trained_frequencies(list(bytes.fromhex(v["train"])), o.TREE, (s, f, c))
            assert emu_encode(emu, [data], f, c, freq=freq) == [want], v["name"]
            outs, raw_len, consumed, status = emu_decode(emu, [want], [len(data)], f, c, freq=freq)
        else:
            freq = None
            if "train" in v:
                freq = o.trained_frequencies(list(bytes.fromhex(v["train"])), o.TREE, (s, f, c))
            assert gen_encode(emu, [data], (s, f, c), freq=freq) == [want], v["name"]
            outs, raw_len, consumed, status = gen_decode(emu, [want], [len(data)], (s, f, c), freq=freq)
        assert int(status[0]) == 0 and outs[0] == data[:nbytes] and int(consumed[0]) == len(want), v["name"]


@pytest.mark.parametrize("f,c", [(10, 12), (14, 16), (16, 18), (22, 24), (30, 32)])
def test_lane_kernels_from_a_trained_model(emu, f, c):
    """Byte symbols, code_bits <= 32, model trained before the call: the tuned lane kernels start from the
    trained tree (count_t = min(count0 + t, FMAX), cum(256) = total - freq(EOF)).  Training sets include the
    EOF symbol itself, a model trained all the way to the freeze, and totals that need u32 table entries."""
    rng = np.random.default_rng(100 * f + c)
    fmax = (1 << f) - 1
    trainings = [
        [int(x) for x in rng.integers(0, 40, 300)],
        [256] * 5 + [int(x) for x in rng.integers(0, 257, 200)],            # EOF trained: freq(EOF) = 6
        [int(x) for x in rng.integers(60, 70, min(fmax, 70000))],           # to the freeze (small f) / beyond u16 (large f)
    ]
    blocks = make_blocks(rng, 14, 2500) + [bytes([255] * 900), bytes(rng.integers(60, 70, 3000, dtype=np.uint8))]
    for train in trainings:
        freq = o.trained_frequencies(train, o.TREE, (8, f, c))
        want = []
        for b in blocks:
            rc, out, ic, oc = o.compress_trained(b, train, o.LINEAR, (8, f, c))
            assert rc == o.OK
            want.append(out)
        assert emu_encode(emu, blocks, f, c, freq=freq) == want, (f, c, len(train))
        outs, raw_len, consumed, status = emu_decode(emu, want, [len(b) + 2 for b in blocks], f, c, freq=freq)
        assert (status == 0).all() and outs == blocks
        assert [int(x) for x in consumed] == [len(w) for w in want]
        # truncated streams keep the reference's Eof behaviour
        cut = [w[:-1] for w in want]
        outs, raw_len, consumed, status = emu_decode(emu, cut, [len(b) + 2 for b in blocks], f, c, freq=freq)
        for i, sgm in enumerate(cut):
            rc, out, ic, oc = o.decompress_trained(sgm, train, o.TREE, (8, f, c), out_cap=len(blocks[i]) + 2)
            assert (int(status[i]), outs[i], int(consumed[i])) == (rc, out, ic), (i, f, c)
