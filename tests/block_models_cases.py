"""Batches whose blocks start from different trained models (redux_encode_batch_models and friends).

Each case names parameters, the models of the call and the coder kernels the plan must select.  The models are given
by kind; every kind is trained by its own sequence of symbols, so the oracle codes block i with
compress_trained(block, training sequence of block i's model).  Block i starts from model i % len(models), so every warp
of a launch holds every model of its case.  Kinds:
  ones        a fresh model (every frequency 1)
  fmax        trained to exactly freq_max: tcap = 0, the block is frozen from its first symbol
  u32         total 70,000 > 65,535: the plan takes u32 table entries
  eof         a heavily trained EOF frequency
  mid         1,000 random symbols
  wided_last  total 349,524 - the longest block: the launch's largest total is one below the WIDE_D bound
  wide        total 349,625: past the WIDE_D bound, the plain WIDE class

Imported by test_block_models_emu.py (host emulation) and test_gpu_block_models.py (device) -- data and helpers only.
"""
import zlib
from collections import namedtuple

import numpy as np

import kernel_matrix_cases as km
import oracle_lib as o

INVALID_INPUT = 2
SENTINEL = 0xA5

Case = namedtuple("Case", "name params kinds enc dec")

CASES = [
    # tuned lane kernels (byte symbols, code_bits <= 32): one row per kernel a trained model can reach
    Case("narrow_stg", (8, 14, 16), ("ones", "fmax", "eof", "mid"), *km.NARROW_STG),
    Case("narrow", (8, 12, 18), ("ones", "fmax", "eof", "mid"), *km.NARROW),
    Case("wided_u16_c24", (8, 22, 24), ("ones", "eof", "mid"), *km.lane("u16", "WideD", True, False)),
    Case("wided_u16_c32", (8, 30, 32), ("ones", "eof", "mid"), *km.lane("u16", "WideD", True, True)),
    Case("wided_u32_c22", (8, 18, 22), ("ones", "fmax", "u32", "eof", "mid"), *km.lane("u32", "WideD", True, False)),
    Case("wided_u32_c32", (8, 17, 32), ("ones", "fmax", "u32", "eof", "mid"), *km.lane("u32", "WideD", True, True)),
    Case("wided_u32_last_c32", (8, 30, 32), ("ones", "u32", "eof", "wided_last"), *km.lane("u32", "WideD", True, True)),
    Case("wide_u32_c21", (8, 19, 21), ("ones", "fmax", "u32", "eof", "wided_last", "wide"),
         *km.lane("u32", "Wide", True, False)),
    Case("wide_u32_c32", (8, 30, 32), ("ones", "u32", "eof", "wided_last", "wide"), *km.lane("u32", "Wide", True, True)),
    # generic kernels: symbol_bits != 8, and trained models with code_bits > 32
    Case("generic_s4", (4, 14, 16), ("ones", "fmax", "eof", "mid"), "encode_generic<smem>", "decode_generic<smem>"),
    Case("generic_s12", (12, 16, 18), ("ones", "fmax", "eof", "mid"), "encode_generic<global>", "decode_generic<global>"),
    Case("generic_c34", (8, 30, 34), ("ones", "u32", "eof", "mid", "wide"), "encode_generic<global>",
         "decode_generic<global>"),
]


def is_generic(case):
    return case.enc.startswith("encode_generic")


def rng_for(case, what=""):
    return np.random.default_rng(zlib.crc32((case.name + what).encode()))


def _mix(rng, n):
    return km._mix(rng, n)


def blocks_for(case):
    """40 blocks: empty, short, runs of one symbol, mixed blocks of up to 3,000 bytes."""
    rng = rng_for(case, "blocks")
    blocks = [b""] + [rng.integers(0, 256, n, dtype=np.uint8).tobytes() for n in (1, 15, 16, 17)]
    blocks += [bytes([v]) * 300 for v in (0x00, 0x41, 0xFE, 0xFF)]
    blocks += [_mix(rng, int(n)) for n in rng.integers(20, 1500, 30)]
    blocks.append(_mix(rng, 3000))
    return blocks


def max_len(case):
    return max(len(b) for b in blocks_for(case))


def training(case):
    """The training sequence of every model of the case (EOF included among the symbols)."""
    s, f, _ = case.params
    nsym, fmax = (1 << s) + 1, (1 << f) - 1
    out = []
    for k, kind in enumerate(case.kinds):
        rng = rng_for(case, kind)
        n = {"ones": 0, "fmax": fmax - nsym, "u32": 70000 - nsym, "eof": 2500, "mid": 1000,
             "wided_last": km.WIDE_D_BOUND - 1 - max_len(case) - nsym, "wide": km.WIDE_D_BOUND + 100 - nsym}[kind]
        assert nsym + n <= fmax, (case.name, kind)
        t = rng.integers(0, nsym, n).astype(np.uint64)
        if kind == "eof":
            t[:2000] = nsym - 1
            rng.shuffle(t)
        out.append(t)
    return out


def freq_table(case):
    """uint32[n_models, symbol_count]: the frequencies each model has after its training (Model::get_frequency)."""
    s = case.params[0]
    nsym = (1 << s) + 1
    tab = np.ones((len(case.kinds), nsym), dtype=np.uint32)
    for m, t in enumerate(training(case)):
        np.add.at(tab[m], t.astype(np.int64), 1)
    return tab


def totals(case):
    return [int(r.sum()) for r in freq_table(case)]


def oracle_compress(case, train, block):
    rc, out, ic, _ = o.compress_trained(block, train, o.TREE, case.params)
    assert rc == o.OK and ic == len(block)
    return out


def oracle_decompress(case, train, stream, cap):
    """(status, bytes, consumed); the oracle's IO_ERROR (writer full) is the device's OUT_CAPACITY (6)."""
    rc, out, ic, _ = o.decompress_trained(stream, train, o.TREE, case.params, out_cap=cap)
    return (6 if rc == o.IO_ERROR else rc), out, ic


# ------------------------------------------------------------------ one case on any backend
# A backend codes through one implementation: encode(blocks, table, block_model) -> (streams, status);
# decode(comp, coff, raw, roff, max_len, table, block_model) -> (raw, raw_lens, consumed, status) in place of the given
# buffers; kernels() -> the names launched since the last call (None where the backend cannot tell).

def _aligned(n):
    return km._aligned(n)


def decode_items(backend, items, table, max_len=None):
    """(stream, capacity, row) triples into adjacent slots after km.LEAD bytes of a SENTINEL-filled buffer with a guard
    tail; checks that nothing outside the slots changed.  Returns [(status, bytes, consumed, slot bytes)]."""
    n = len(items)
    coff = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum([len(s) for s, _, _ in items], out=coff[1:])
    coff += np.uint64(1)
    comp = _aligned(int(coff[-1]) + 64)
    comp[1:int(coff[-1])] = np.frombuffer(b"".join(s for s, _, _ in items), dtype=np.uint8)
    roff = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum([cap for _, cap, _ in items], out=roff[1:])
    roff += np.uint64(km.LEAD)
    raw = _aligned(int(roff[-1]) + km.GUARD)
    raw[:] = SENTINEL
    bm = np.array([m for _, _, m in items], dtype=np.uint32)
    max_len = max(cap for _, cap, _ in items) if max_len is None else max_len
    raw, raw_lens, consumed, status = backend.decode(comp, coff, raw, roff, max_len, table, bm)
    assert (raw[:km.LEAD] == SENTINEL).all(), "decoder wrote before the first slot"
    assert (raw[int(roff[-1]):] == SENTINEL).all(), "decoder wrote past the last slot"
    return [(int(status[i]), raw[int(roff[i]):int(roff[i]) + int(raw_lens[i])].tobytes(), int(consumed[i]),
             raw[int(roff[i]):int(roff[i + 1])].tobytes()) for i in range(n)]


def _check_kernels(backend, want, what):
    got = backend.kernels()
    assert got is None or got == {want}, "%s ran %s, expected %s" % (what, sorted(got), want)


def check_case(case, backend):
    """Encode against the oracle block by block, decode at exact capacity, then the decoder's error exits (cut,
    garbage, trailing garbage, slot one byte short) of several models between good neighbours of other models."""
    blocks, train, table = blocks_for(case), training(case), freq_table(case)
    nm = len(case.kinds)
    bm = np.arange(len(blocks), dtype=np.uint32) % np.uint32(nm)
    want = [oracle_compress(case, train[bm[i]], b) for i, b in enumerate(blocks)]
    got, status = backend.encode(blocks, table, bm)
    _check_kernels(backend, case.enc, "encode")
    assert (status == 0).all(), status
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, "%s: block %d (len %d, model %s) encodes to %d bytes, oracle %d" % (
            case.name, i, len(blocks[i]), case.kinds[bm[i]], len(g), len(w))
    res = decode_items(backend, [(w, len(b), int(bm[i])) for i, (w, b) in enumerate(zip(want, blocks))], table)
    _check_kernels(backend, case.dec, "decode")
    for i, r in enumerate(res):
        exact = oracle_decompress(case, train[bm[i]], want[i], len(blocks[i]))
        assert exact[0] == 0 and exact[2] == len(want[i]) and (case.params[0] != 8 or exact[1] == blocks[i])
        assert r[:3] == exact, "%s: block %d (model %s): status %d consumed %d vs %d" % (
            case.name, i, case.kinds[bm[i]], r[0], r[2], exact[2])
    # error exits: the longest block and the 0xFF run under every model, each between good neighbours of the next model
    rng = rng_for(case, "errors")
    items, pos = [], km.LEAD
    longest = max(range(len(blocks)), key=lambda i: len(blocks[i]))
    run_ff = blocks.index(bytes([0xFF]) * 300)
    k = 0
    for m in range(nm):
        for i in (longest, run_ff):
            w = oracle_compress(case, train[m], blocks[i])
            cap, L = len(blocks[i]), len(w)
            n_out = len(oracle_decompress(case, train[m], w, cap)[1])
            errs = [(w[:cut], cap) for cut in sorted({0, 1, 2, L // 2, L - 1}) if 0 <= cut < L]
            errs += [(rng.integers(0, 256, min(L, 2048) + 1, dtype=np.uint8).tobytes(), cap),
                     (w + rng.integers(0, 256, 16, dtype=np.uint8).tobytes(), cap), (w, n_out - 1)]
            for s, c in errs:
                n = (1 + k % 3 - pos) % 4 or 4                     # the error slot starts at 1, 2, 3 (mod 4) in turn
                fm = (m + 1) % nm
                filler = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
                items += [(oracle_compress(case, train[fm], filler), n, fm), (s, c, m)]
                pos += n + c
                k += 1
    fm = 0
    items.append((oracle_compress(case, train[fm], b"tail!"), 5, fm))
    res = decode_items(backend, items, table, max_len=max(len(b) for b in blocks))
    _check_kernels(backend, case.dec, "decode of the error streams")
    for i, ((s, cap, m), r) in enumerate(zip(items, res)):
        e = oracle_decompress(case, train[m], s, cap)
        assert i % 2 == 1 or e[0] == 0, "filler %d must decode" % i
        assert r[:3] == e, "%s: item %d (%s, model %s, stream %d B, slot %d B): (status %d, %d B, consumed %d) vs " \
            "oracle (status %d, %d B, consumed %d)" % (case.name, i, "error" if i % 2 else "good neighbour",
                                                       case.kinds[m], len(s), cap, r[0], len(r[1]), r[2], e[0],
                                                       len(e[1]), e[2])


def check_bad_index(case, backend):
    """Blocks with row index n_models and 0xFFFFFFFF between good neighbours: INVALID_INPUT, an empty stream / nothing
    decoded (the slot keeps its bytes), the neighbours as the oracle codes them."""
    blocks, train, table = blocks_for(case), training(case), freq_table(case)
    nm = len(case.kinds)
    pick = [blocks[-1], blocks[6], blocks[-2], blocks[8], blocks[3]]
    bm = np.array([nm - 1, nm, 0, 0xFFFFFFFF, 1 % nm], dtype=np.uint32)
    good = [0, 2, 4]
    got, status = backend.encode(pick, table, bm)
    assert list(status) == [0, INVALID_INPUT, 0, INVALID_INPUT, 0], status
    assert got[1] == b"" and got[3] == b""
    want = {i: oracle_compress(case, train[bm[i]], pick[i]) for i in good}
    for i in good:
        assert got[i] == want[i], "%s: neighbour %d" % (case.name, i)
    # decode: the bad rows get a real stream (of model 0) and a slot the size of their block
    w0 = oracle_compress(case, train[0], pick[1]), oracle_compress(case, train[0], pick[3])
    items = [(want[0], len(pick[0]), int(bm[0])), (w0[0], len(pick[1]), int(bm[1])),
             (want[2], len(pick[2]), int(bm[2])), (w0[1], len(pick[3]), int(bm[3])), (want[4], len(pick[4]), int(bm[4]))]
    res = decode_items(backend, items, table)
    for i, r in enumerate(res):
        if i in good:
            assert r[:3] == oracle_decompress(case, train[bm[i]], want[i], len(pick[i])), "%s: neighbour %d" % (case.name, i)
        else:
            assert r[:3] == (INVALID_INPUT, b"", 0), r[:3]
            assert r[3] == bytes([SENTINEL]) * len(pick[i]), "the slot of a bad block was written"
