"""The kernel matrix: one row per (parameters, model, schedule, block shapes) that selects a given coder kernel.

The device path chooses among 37 coder kernels (redux_b200/csrc/redux_capi.cu: pick_encoder / pick_decoder, the split
and generic launches) by arithmetic class, table entry width, FULL (u16 entries hold full tree values), code_bits ==
32, code_bits <= 16 (staged decoder window), lane / warp / split mapping, generic kernels, and whether the model was
trained.  Encode plans from the longest block, decode from the largest output slot.  Every row names the encode and
decode kernel it must reach (checked on the GPU by redux_debug_launched_kernels) and is chosen to reach the phase that
matters: adaptive, frozen, or both in one block.  Together the rows reach every kernel of the library.

Imported by test_gpu_kernel_matrix.py (GPU, every row), test_kernel_coverage.py (no GPU: completeness, the plan
behind each lane row, and the lane rows in the host emulation) -- plain data and helpers, no test in here.
"""
import zlib
from collections import namedtuple

import numpy as np

import oracle_lib as o

NSYM = 257                              # symbol_count of a byte model (EOF included)
WIDE_D_BOUND = 349525                   # kWideDMaxCount: totals below it divide by a double reciprocal
U16_MAX_UPDATES = 65536                 # fresh model: more updates than this need u32 table entries
FULL_MAX_UPDATES = 65535 - 256          # fresh model: up to this many updates the u16 entries hold full tree values


def tcap(f, count0=NSYM):
    """Model updates before the freeze: FMAX - count0 (2^f - 258 for a fresh model)."""
    return (1 << f) - 1 - count0


# the rows' thresholds, as computed
assert tcap(19) == 524030 and tcap(18) == 261886 and tcap(17) == 130814 and tcap(14) == 16126 and tcap(12) == 3838
assert WIDE_D_BOUND - NSYM == 349268    # a fresh block of 349,268 updates is the first one off WIDE_D

Case = namedtuple("Case", "name params train sched big enc dec caps")
# params: (symbol_bits, freq_bits, code_bits); train: symbols the model learns before the call (0 = fresh);
# sched: "lane" / "warp" / "split"; big: extra blocks (length, content) with content "mix" (mixed entropy) or a byte
# value (a run of one symbol); enc / dec: expected kernel names; caps: {slot capacity: decode kernel} -- the row's
# streams decoded again into slots of that capacity each


def C(name, params, enc, dec, big=(), train=0, sched="lane", caps=None):
    return Case(name, params, train, sched, tuple(big), enc, dec, caps or {})


def lane(tw, cls, full, c32, stg=False):
    args = "%s,%s,%s,%s" % (tw, cls, "full" if full else "!full", "c32" if c32 else "!c32")
    return "encode_lane_al<%s>" % args, "decode_lane_al<%s%s>" % (args, ",stg" if stg else "")


NARROW_STG = ("encode_lane_al<u16,Narrow,full,!c32>", "decode_lane_al<u16,Narrow,full,!c32,stg>")
NARROW = ("encode_lane_al<u16,Narrow,full,!c32>", "decode_lane_al<u16,Narrow,full,!c32>")
SPLIT_LENS = [(2047, "mix"), (2048, "mix"), (2049, "mix"), (3 * 2048, "mix")]   # split encoder model chunks: 2048

CASES = [
    # ---- tuned lane kernels, fresh models
    C("narrow_c16_frozen", (8, 14, 16), *NARROW_STG, big=[(tcap(14) + 4000, "mix")]),
    C("narrow_c18_frozen", (8, 12, 18), *NARROW, big=[(tcap(12) + 1, "mix"), (5000, "mix")]),
    C("wided_u16_full_c24", (8, 22, 24), *lane("u16", "WideD", True, False), big=[(FULL_MAX_UPDATES, "mix")]),
    C("wided_u16_full_c32", (8, 30, 32), *lane("u16", "WideD", True, True), big=[(FULL_MAX_UPDATES, "mix")]),
    C("wided_u16_c24", (8, 22, 24), *lane("u16", "WideD", False, False),
      big=[(FULL_MAX_UPDATES + 1, "mix"), (U16_MAX_UPDATES, 0x41)]),
    C("wided_u16_c32", (8, 30, 32), *lane("u16", "WideD", False, True), big=[(U16_MAX_UPDATES, "mix")],
      caps={65536: lane("u16", "WideD", False, True)[1], 70000: lane("u32", "WideD", True, True)[1],
            350000: lane("u32", "Wide", True, True)[1]}),
    C("wided_u32_c24", (8, 22, 24), *lane("u32", "WideD", True, False), big=[(U16_MAX_UPDATES + 1, "mix")]),
    C("wided_u32_frozen_c22", (8, 18, 22), *lane("u32", "WideD", True, False), big=[(270000, "mix")]),
    C("wided_u32_frozen_c32", (8, 17, 32), *lane("u32", "WideD", True, True), big=[(140000, "mix")]),
    C("wided_u32_last_c32", (8, 30, 32), *lane("u32", "WideD", True, True), big=[(WIDE_D_BOUND - NSYM - 1, "mix")]),
    C("wide_u32_first_c32", (8, 30, 32), *lane("u32", "Wide", True, True), big=[(WIDE_D_BOUND - NSYM, "mix")]),
    C("wide_u32_frozen_c21", (8, 19, 21), *lane("u32", "Wide", True, False), big=[(530000, "mix")]),
    C("wide_u32_frozen_c32", (8, 19, 32), *lane("u32", "Wide", True, True), big=[(tcap(19) + 5970, "mix")]),
    # ---- tuned lane kernels, trained models (count0 = 257 + training symbols)
    C("trained_narrow_c16", (8, 14, 16), *NARROW_STG, train=3000),
    C("trained_narrow_c18_frozen", (8, 12, 18), *NARROW, train=3000, big=[(2000, "mix")]),
    C("trained_wided_u16_c24", (8, 22, 24), *lane("u16", "WideD", True, False), train=3000),
    C("trained_wided_u32_c32", (8, 30, 32), *lane("u32", "WideD", True, True), train=65535 - NSYM + 1),
    C("trained_wide_u32_c22", (8, 20, 22), *lane("u32", "Wide", True, False), train=WIDE_D_BOUND - NSYM),
    # ---- code_bits > 32: encode/decode_lane_kernel<TW, kHuge>
    C("huge_u16_c40", (8, 20, 40), "encode_lane<u16,Huge>", "decode_lane<u16,Huge>", big=[(5000, "mix")]),
    C("huge_u16_one_path_c34", (8, 30, 34), "encode_lane<u16,Huge>", "decode_lane<u16,Huge>",
      big=[(U16_MAX_UPDATES, 0xFF), (U16_MAX_UPDATES, 0x00)]),
    C("huge_u32_frozen_c34", (8, 17, 34), "encode_lane<u32,Huge>", "decode_lane<u32,Huge>", big=[(140000, "mix")]),
    # ---- one stream per warp
    C("warp_narrow_frozen", (8, 12, 18), "encode_warp<Narrow>", "decode_warp_al<Narrow,!c32>", sched="warp",
      big=[(5000, "mix")]),
    C("warp_wide_c24", (8, 22, 24), "encode_warp<Wide>", "decode_warp_al<Wide,!c32>", sched="warp",
      big=[(U16_MAX_UPDATES, "mix")]),
    C("warp_wide_frozen_c21", (8, 19, 21), "encode_warp<Wide>", "decode_warp_al<Wide,!c32>", sched="warp",
      big=[(530000, "mix")]),
    C("warp_wide_frozen_c32", (8, 17, 32), "encode_warp<Wide>", "decode_warp_al<Wide,c32>", sched="warp",
      big=[(140000, "mix")]),
    C("warp_huge_frozen_c34", (8, 17, 34), "encode_warp<Huge>", "decode_warp<Huge>", sched="warp",
      big=[(140000, "mix")]),
    # ---- split encoder (decode side: the warp mapping); the last block of each row freezes inside a model chunk
    C("split_narrow_frozen", (8, 14, 16), "split_coder<Narrow,!c32>", "decode_warp_al<Narrow,!c32>", sched="split",
      big=SPLIT_LENS + [(20000, "mix")]),
    C("split_wide_c24", (8, 22, 24), "split_coder<Wide,!c32>", "decode_warp_al<Wide,!c32>", sched="split",
      big=SPLIT_LENS + [(U16_MAX_UPDATES, "mix")]),
    C("split_wide_frozen_c32", (8, 17, 32), "split_coder<Wide,c32>", "decode_warp_al<Wide,c32>", sched="split",
      big=SPLIT_LENS + [(140000, "mix")]),
    C("split_huge_takes_warp_c40", (8, 20, 40), "encode_warp<Huge>", "decode_warp<Huge>", sched="split",
      big=SPLIT_LENS),
    # ---- trained models always take the lane mapping
    C("trained_warp_takes_lane", (8, 22, 24), *lane("u16", "WideD", True, False), train=3000, sched="warp"),
    C("trained_split_takes_lane", (8, 14, 16), *NARROW_STG, train=3000, sched="split"),
    # ---- generic kernels (symbol_bits != 8, trained code_bits > 32): Fenwick columns in smem up to 7 bits
    C("generic_s4", (4, 14, 16), "encode_generic<smem>", "decode_generic<smem>"),
    C("generic_s7", (7, 20, 40), "encode_generic<smem>", "decode_generic<smem>"),
    C("generic_s9", (9, 22, 24), "encode_generic<global>", "decode_generic<global>"),
    C("generic_s16", (16, 18, 20), "encode_generic<global>", "decode_generic<global>"),
    C("generic_trained_c34", (8, 30, 34), "encode_generic<global>", "decode_generic<global>", train=3000,
      big=[(5000, "mix")]),
]


def expected_kernels():
    names = set()
    for case in CASES:
        names |= {case.enc, case.dec} | set(case.caps.values())
    return names


# ------------------------------------------------------------------ inputs and the oracle side
def rng_for(case):
    return np.random.default_rng(zlib.crc32(case.name.encode()))


def _mix(rng, n):
    """Uniform, text-like and geometric thirds: every phase of a long block sees varied symbols."""
    a, b = n // 3, n // 3
    return np.concatenate([rng.integers(0, 256, a, dtype=np.uint8),
                           rng.choice(np.frombuffer(b" etaoinshrdlu\n", dtype=np.uint8), b),
                           np.minimum(rng.geometric(0.3, n - a - b) - 1, 255).astype(np.uint8)]).tobytes()


def blocks_for(case):
    """Empty, 1-byte, 15/16/17-byte blocks, one-symbol runs (0x00 .. 0xFF: node 256 and single-path increments), a
    mixed 3000-byte block, then the row's own blocks."""
    rng = rng_for(case)
    blocks = [b""] + [rng.integers(0, 256, n, dtype=np.uint8).tobytes() for n in (1, 15, 16, 17)]
    blocks += [bytes([v]) * 300 for v in (0x00, 0x41, 0x7F, 0xFE, 0xFF)]
    blocks.append(_mix(rng, 3000))
    for n, what in case.big:
        blocks.append(_mix(rng, n) if what == "mix" else bytes([what]) * n)
    return blocks


def train_for(case):
    """The symbols the row's model learns before the call (EOF included), or None for a fresh model."""
    if not case.train:
        return None
    s = case.params[0]
    return np.random.default_rng(case.train).integers(0, (1 << s) + 1, case.train).astype(np.uint64)


def trained_freq(case):
    """Per-symbol frequencies after train_for(case) (Model::get_frequency, frozen at freq_max)."""
    s, f, _ = case.params
    train = train_for(case)
    fr = np.ones((1 << s) + 1, dtype=np.uint32)
    if train is not None:
        np.add.at(fr, train[:(1 << f) - 1 - fr.size].astype(np.int64), 1)
    return fr


def oracle_compress(case, block):
    train = train_for(case)
    if train is None:
        rc, out, ic, oc = o.compress(block, o.TREE, case.params)
    else:
        rc, out, ic, oc = o.compress_trained(block, train, o.TREE, case.params)
    assert rc == o.OK and ic == len(block)
    return out


def oracle_decompress(case, stream, cap):
    """(status, bytes, consumed) with the oracle's IO_ERROR (writer full) as the device's OUT_CAPACITY (6)."""
    train = train_for(case)
    if train is None:
        rc, out, ic, oc = o.decompress(stream, o.TREE, case.params, out_cap=cap)
    else:
        rc, out, ic, oc = o.decompress_trained(stream, train, o.TREE, case.params, out_cap=cap)
    return (6 if rc == o.IO_ERROR else rc), out, ic


def error_streams(case, blocks, streams):
    """(stream, capacity) pairs for the decoder's exits, on the longest stream and on the 0xFF run: cuts to 0, 1, 2, 3,
    half, len-3, len-2 and len-1 bytes (for rows that freeze, the last cuts end in the frozen phase), random garbage,
    trailing garbage, a slot one byte short (OUT_CAPACITY) and a cut stream in a slot one byte short (precedence)."""
    rng = rng_for(case)
    longest = max(range(len(blocks)), key=lambda i: len(blocks[i]))
    run_ff = blocks.index(bytes([0xFF]) * 300)
    out = []
    for i in (longest, run_ff):
        w, cap = streams[i], len(blocks[i])
        n_out = len(oracle_decompress(case, w, cap)[1])
        L = len(w)
        for cut in sorted({0, 1, 2, 3, L // 2, L - 3, L - 2, L - 1}):
            if 0 <= cut < L:
                out.append((w[:cut], cap))
        out.append((rng.integers(0, 256, min(L, 2048) + 1, dtype=np.uint8).tobytes(), cap))
        out.append((w + rng.integers(0, 256, 16, dtype=np.uint8).tobytes(), cap))
        out.append((w, n_out - 1))
        out.append((w[:L - 1], n_out - 1))
    return out


# ------------------------------------------------------------------ one row, on any backend
# A backend codes through one kernel implementation: encode(blocks) -> streams; decode(comp, coff, raw, roff, max_len)
# -> (raw, raw_lens, consumed, status) in place of the given buffers; kernels() -> names launched since the last call
# (None where the backend cannot tell).
LEAD = 3                 # first slot / stream offset: no slot or stream starts 4-byte aligned by accident
SENTINEL = 0xA5
GUARD = 64


def _aligned(n):
    buf = np.zeros(n + 16, dtype=np.uint8)
    a = (-buf.ctypes.data) % 16
    return buf[a:a + n]


def decode_items(backend, items, max_len=None):
    """Decodes (stream, capacity) pairs into adjacent slots with no slack behind LEAD bytes, on a SENTINEL-filled
    buffer with a GUARD tail; checks that nothing outside the slots changed.  Returns [(status, bytes, consumed)]."""
    n = len(items)
    coff = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum([len(s) for s, _ in items], out=coff[1:])
    coff += np.uint64(1)
    comp = _aligned(int(coff[-1]) + 64)
    comp[1:int(coff[-1])] = np.frombuffer(b"".join(s for s, _ in items), dtype=np.uint8)
    roff = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum([cap for _, cap in items], out=roff[1:])
    roff += np.uint64(LEAD)
    raw = _aligned(int(roff[-1]) + GUARD)
    raw[:] = SENTINEL
    max_len = max(cap for _, cap in items) if max_len is None else max_len
    raw, raw_lens, consumed, status = backend.decode(comp, coff, raw, roff, max_len)
    assert (raw[:LEAD] == SENTINEL).all(), "decoder wrote before the first slot"
    assert (raw[int(roff[-1]):] == SENTINEL).all(), "decoder wrote past the last slot"
    return [(int(status[i]), raw[int(roff[i]):int(roff[i]) + int(raw_lens[i])].tobytes(), int(consumed[i]))
            for i in range(n)]


def _check_kernels(backend, want, what):
    got = backend.kernels()
    assert got is None or got == {want}, "%s ran %s, expected %s" % (what, sorted(got), want)


def check_row(case, backend):
    blocks = blocks_for(case)
    want = [oracle_compress(case, b) for b in blocks]
    # 1. encode vs oracle
    got = backend.encode(blocks)
    _check_kernels(backend, case.enc, "encode")
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, "%s: block %d (len %d) encodes to %d bytes, oracle %d" % (case.name, i, len(blocks[i]), len(g), len(w))
    # 2. decode at exact capacity
    exact = [oracle_decompress(case, w, len(b)) for w, b in zip(want, blocks)]
    res = decode_items(backend, [(w, len(b)) for w, b in zip(want, blocks)])
    _check_kernels(backend, case.dec, "decode")
    for i, (r, e) in enumerate(zip(res, exact)):
        assert e[0] == 0 and e[2] == len(want[i]) and (case.params[0] != 8 or e[1] == blocks[i])
        assert r == e, "%s: block %d (len %d): status %d consumed %d vs %d" % (case.name, i, len(blocks[i]), r[0], r[2], e[2])
    # 3 + 4. the decoder's error exits, each between good neighbours whose slots start at offsets that are not
    # multiples of 4
    rng = rng_for(case)
    items, pos = [], LEAD
    for k, err in enumerate(error_streams(case, blocks, want)):
        n = (1 + k % 3 - pos) % 4 or 4                     # the error slot starts at 1, 2, 3 (mod 4) in turn
        filler = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        items += [(oracle_compress(case, filler), n), err]
        pos += n + err[1]
    filler = rng.integers(0, 256, 5, dtype=np.uint8).tobytes()
    items.append((oracle_compress(case, filler), 5))
    res = decode_items(backend, items, max_len=max(len(b) for b in blocks))
    _check_kernels(backend, case.dec, "decode of the error streams")
    for i, ((s, cap), r) in enumerate(zip(items, res)):
        e = oracle_decompress(case, s, cap)
        assert i % 2 == 1 or e[0] == 0, "filler %d must decode" % i
        assert r == e, "%s: item %d (%s, stream %d B, slot %d B): device (status %d, %d B, consumed %d) vs oracle " \
            "(status %d, %d B, consumed %d)" % (case.name, i, "error" if i % 2 else "good neighbour", len(s), cap,
                                                r[0], len(r[1]), r[2], e[0], len(e[1]), e[2])
    # the same streams decoded into slots whose capacity selects another kernel
    for cap, kernel in sorted(case.caps.items()):
        res = decode_items(backend, [(w, cap) for w in want])
        _check_kernels(backend, kernel, "decode into %d-byte slots" % cap)
        for i, r in enumerate(res):
            assert r == (0, blocks[i], len(want[i])), "%s: block %d into a %d-byte slot" % (case.name, i, cap)
