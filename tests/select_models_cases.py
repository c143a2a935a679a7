"""Cases and references of redux_select_models (each block's start model chosen by its ideal code length, DESIGN.md
3.10).

A case names parameters, candidate rows and blocks.  The cost of block x under row r is the ideal code length in bits of
what compress() codes from that start state: every data symbol, then EOF.  Two references give it in float64:

- walk_cost: position by position.  Where the model's training plus the block is short, this is the oracle's model
  (oracle_lib): trained to the row by get_frequency, then total_frequency() and get_frequency()'s hi - lo before each
  symbol's lookup.  Longer ones run the same counter in numpy.
- closed_cost: the closed form with scipy.special.gammaln.

Imported by test_select_models_emu.py (host emulation), test_select_models_cpu.py and test_gpu_select_models.py --
data and helpers only.
"""
import zlib
from collections import namedtuple

import numpy as np
from scipy.special import gammaln

import oracle_lib as o
from train_models_cases import sample_bytes

Case = namedtuple("Case", "name params chunk rows blocks")

ORACLE_WALK_MAX = 20000            # training + block symbols the oracle walks; longer walks run in numpy
REL_TOL, ABS_TOL = 1e-6, 0.05      # a cost within REL_TOL * cost + ABS_TOL bits of the reference


def symbols(data, s):
    """The symbols the reference's BitReader yields: s bits at a time, MSB-first, a trailing partial symbol dropped."""
    bits = np.unpackbits(np.frombuffer(bytes(data), dtype=np.uint8))
    n = bits.size // s
    if n == 0:
        return np.zeros(0, dtype=np.int64)
    w = bits[:n * s].reshape(n, s).astype(np.int64)
    return (w << np.arange(s - 1, -1, -1, dtype=np.int64)).sum(axis=1)


def _split(row, n, params):
    _, f, _ = params
    return min(n, (1 << f) - 1 - int(np.asarray(row, dtype=np.int64).sum()))


def closed_cost(row, syms, params):
    r = np.asarray(row, dtype=np.float64)
    T = r.sum()
    n = syms.size
    m = _split(row, n, params)
    h = np.bincount(syms[:m], minlength=r.size - 1).astype(np.float64)
    g = np.bincount(syms[m:], minlength=r.size - 1).astype(np.float64)
    rd = r[:-1]
    fr = rd + h
    Tp = T + m
    c = gammaln(T + m) - gammaln(T) - (gammaln(fr) - gammaln(rd)).sum()
    nz = g > 0
    c += (g[nz] * np.log(Tp / fr[nz])).sum() + np.log(Tp / r[-1])
    return float(c / np.log(2.0))


def _oracle_walk(row, syms, params):
    s, _, _ = params
    m = o.Model(o.TREE, *params)
    for x, cnt in enumerate(np.asarray(row, dtype=np.int64)):
        for _ in range(int(cnt) - 1):
            assert m.get_frequency(x)[0] == o.OK
    bits = 0.0
    for x in list(syms) + [(1 << s)]:
        total = m.total_frequency()
        rc, lo, hi = m.get_frequency(int(x))
        assert rc == o.OK
        bits += np.log2(total / (hi - lo))
    return float(bits)


def _numpy_walk(row, syms, params):
    r = np.asarray(row, dtype=np.int64)
    T = int(r.sum())
    n = syms.size
    m = _split(row, n, params)
    # before position t < m, symbol x has been seen #{u < t : x_u = x} times
    head = syms[:m]
    order = np.argsort(head, kind="stable")
    seen = np.empty(m, dtype=np.int64)
    if m:
        sh = head[order]
        starts = np.r_[0, np.flatnonzero(np.diff(sh)) + 1]
        run_id = np.repeat(np.arange(starts.size), np.diff(np.r_[starts, m]))
        seen[order] = np.arange(m) - starts[run_id]
    fr_head = r[head] + seen
    tot_head = T + np.arange(m, dtype=np.int64)
    f = r.copy()
    np.add.at(f, head, 1)
    Tp = T + m
    tail = syms[m:]
    bits = np.log2(tot_head / fr_head).sum() + np.log2(Tp / f[tail]).sum() + np.log2(Tp / r[-1])
    return float(bits)


def walk_cost(row, syms, params):
    trained = int(np.asarray(row, dtype=np.int64).sum()) - len(row)
    if trained + syms.size <= ORACLE_WALK_MAX:
        return _oracle_walk(row, syms, params)
    return _numpy_walk(row, syms, params)


def reference_costs(case, walk=False):
    """float64[n_blocks, n_models] reference costs in bits (closed form, or the walk)."""
    fn = walk_cost if walk else closed_cost
    s = case.params[0]
    return np.array([[fn(r, symbols(b, s), case.params) for r in case.rows] for b in case.blocks], dtype=np.float64)


def tolerance(ref):
    return REL_TOL * np.abs(ref) + ABS_TOL


def check_choice(case, ref, cost, choice):
    """Costs within tolerance; the choice's reference cost within twice the tolerance of the reference minimum; where
    the reference gap between best and second best exceeds twice the tolerance, the reference argmin."""
    err = np.abs(cost - ref)
    bad = np.argwhere(err > tolerance(ref))
    assert bad.size == 0, (case.name, bad[:4].tolist(), err.max())
    for i in range(ref.shape[0]):
        best = ref[i].min()
        assert ref[i, choice[i]] <= best + 2 * tolerance(best), (case.name, i, int(choice[i]), ref[i].tolist()[:8])
        srt = np.sort(ref[i])
        if srt.size == 1 or srt[1] - srt[0] > 2 * tolerance(srt[0]):
            assert choice[i] == int(np.argmin(ref[i])), (case.name, i, int(choice[i]), int(np.argmin(ref[i])))


def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


def row_with_total(rng, s, total, cls=1, eof=1):
    """A model's row: ones plus total - symbol_count counts drawn from the symbol distribution of a generator class."""
    nsym = (1 << s) + 1
    row = np.ones(nsym, dtype=np.int64)
    row[-1] = eof
    extra = total - int(row.sum())
    assert extra >= 0
    if extra:
        src = symbols(sample_bytes(rng, max(64, (4096 * s + 7) // 8), cls), s)
        p = np.bincount(src, minlength=nsym - 1).astype(np.float64) + 0.05
        row[:-1] += rng.multinomial(extra, p / p.sum())
    return row.astype(np.uint32)


def _width_case(s, f):
    """symbol_bits s: split points before (T = F), just inside (T = F - 1), and just below and above the reference
    block's symbol count; a fresh model; a duplicate row; empty, partial-symbol and longer blocks."""
    name = "s%d_f%d" % (s, f)
    rng = _rng(name)
    nsym, F = (1 << s) + 1, (1 << f) - 1
    n_ref = min(3000, (F - nsym) // 2)
    ref_len = (n_ref * s + 7) // 8
    n_ref = ref_len * 8 // s
    rows = [np.ones(nsym, dtype=np.uint32),
            row_with_total(rng, s, F, 1),
            row_with_total(rng, s, F - 1, 2),
            row_with_total(rng, s, F - (n_ref - 1), 1),
            row_with_total(rng, s, F - (n_ref + 1), 3, eof=3)]
    rows.append(rows[1].copy())                                   # duplicate: the tie goes to index 1
    one = (s + 7) // 8
    lens = [0, 1, one, ref_len, ref_len + 1, 2 * ref_len + 1, 3 * one + 1]
    blocks = [sample_bytes(rng, n, k % 4) for k, n in enumerate(lens)]
    blocks.append(sample_bytes(rng, ref_len, 1))                  # the class the trained rows come from
    return Case(name, (s, f, f + 2), 0, rows, blocks)


def _many_models_case(k):
    """k candidates at (8, 14, 16) with many distinct totals (more models than a CTA has threads when k = 300)."""
    name = "many_k%d" % k
    rng = _rng(name)
    s, f = 8, 14
    F = (1 << f) - 1
    rows = [np.ones(257, dtype=np.uint32)]
    for i in range(1, k):
        rows.append(rows[int(rng.integers(0, i))].copy() if i % 7 == 0 else
                    row_with_total(rng, s, int(rng.integers(300, F + 1)), i % 4))
    blocks = [sample_bytes(rng, int(n), j % 4) for j, n in enumerate([0, 1, 700, 5000, 9000, 17000])]
    return Case(name, (s, f, 16), 0, rows, blocks)


def _long_case(s, chunk):
    """Blocks long enough that the histogram pass spreads each over several CTAs; with an odd chunk the CTA boundaries
    fall inside bytes."""
    name = "long_s%d_chunk%d" % (s, chunk)
    rng = _rng(name)
    f = 30
    rows = [np.ones((1 << s) + 1, dtype=np.uint32), row_with_total(rng, s, 5000, 1), row_with_total(rng, s, 40000, 3)]
    lens = [60000 * s // 8, 50000 * s // 8 + 1]
    blocks = [sample_bytes(rng, n, k + 1) for k, n in enumerate(lens)]
    return Case(name, (s, f, 32), chunk, rows, blocks)


def _winner_case(f, c):
    """64 KiB blocks of each generator class, a fresh model and models trained from one 64 KiB sample of each class:
    trained models win their own class, the fresh model wins where none fits."""
    name = "winner_f%d" % f
    rng = _rng(name)
    F = (1 << f) - 1
    rows = [np.ones(257, dtype=np.uint32)]
    for cls in (1, 2, 3):
        syms = symbols(sample_bytes(rng, 65536, cls), 8)
        row = np.ones(257, dtype=np.int64)
        np.add.at(row, syms[:F - 257], 1)
        rows.append(row.astype(np.uint32))
    blocks = [sample_bytes(rng, 65536, cls) for cls in (0, 1, 2, 3)]
    return Case(name, (8, f, c), 0, rows, blocks)


CASES = ([_width_case(s, f) for s, f in ((1, 12), (3, 12), (7, 13), (8, 13), (12, 16), (16, 18))]
         + [_many_models_case(1), _many_models_case(300)]
         + [_long_case(3, 0), _long_case(8, 0), _long_case(3, 1001)]
         + [_winner_case(14, 16), _winner_case(30, 32)])


def table(case):
    return np.ascontiguousarray(np.stack(case.rows), dtype=np.uint32)


def concat(blocks):
    """Blocks back to back (+ 64 bytes of padding for the aligned 16-byte loads) and their offsets."""
    off = np.zeros(len(blocks) + 1, dtype=np.uint64)
    np.cumsum([len(x) for x in blocks], out=off[1:])
    data = np.zeros(int(off[-1]) + 64, dtype=np.uint8)
    data[:int(off[-1])] = np.frombuffer(b"".join(blocks), dtype=np.uint8)
    return data, off
