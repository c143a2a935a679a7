"""Cases of redux_train_models (training many start models from sample bytes, DESIGN.md 3.9).

A case names parameters, the symbol positions per CTA (`chunk`, 0 = the library's own), the start models as the
symbol sequences that train them (an empty one is a fresh model), the samples and the start model of each sample.  The
expected row of sample i is what the reference's model holds after get_frequency(sym) for every symbol of its start
sequence and then of the sample, the symbols being what the reference's BitReader yields from the sample's bytes.
The oracle (trained_frequencies, one call per symbol) gives it for short sequences, Model.train (vectorised, same
freeze rule) for long ones.

Imported by test_train_models_emu.py (host emulation) and test_gpu_train_models.py (device) -- data and helpers only.
"""
import ctypes as C
import zlib
from collections import namedtuple

import numpy as np

import oracle_lib as o

Case = namedtuple("Case", "name params chunk starts samples sample_model")

ORACLE_MAX_SYMBOLS = 12000          # longer sequences are checked with Model.train


def reference_symbols(data, s):
    """The symbols the reference's BitReader yields from `data` reading s bits at a time (src/bitio/mod.rs:94-108): a
    trailing partial symbol is dropped."""
    L = o.lib()
    a = o._as_u8(data)
    r = L.oracle_bitreader_new(a.ctypes.data, a.size)
    out, v = [], C.c_uint64()
    while L.oracle_bitreader_read_bits(r, s, C.byref(v)) == o.OK:
        out.append(v.value)
    L.oracle_bitreader_free(r)
    return out


def sample_bytes(rng, n, cls):
    """n bytes of one of the generator's four classes: uniform, text-like, geometric, runs."""
    if cls == 0:
        return rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    if cls == 1:
        return rng.choice(np.frombuffer(b"etaoin shrdlu cmfwyp,.\n", dtype=np.uint8), n).tobytes()
    if cls == 2:
        return np.minimum(rng.geometric(0.3, n) - 1, 255).astype(np.uint8).tobytes()
    runs = np.repeat(rng.integers(0, 256, n // 8 + 1, dtype=np.uint8), rng.integers(1, 64, n // 8 + 1))
    return runs[:n].tobytes() if runs.size >= n else (runs.tobytes() * (n // max(runs.size, 1) + 1))[:n]


def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


def _width_case(s, chunk):
    """symbol_bits s: ragged samples of up to ~2,000 symbols, empty ones and ones shorter than one symbol, from a fresh
    and a trained start."""
    name = "s%d_chunk%d" % (s, chunk)
    rng = _rng(name)
    one = (s + 7) // 8
    lens = [0, one - 1, one, one + 1, 2 * s, 257, int(rng.integers(1000 * s // 8 + 1, 2000 * s // 8 + 2))]
    samples = [sample_bytes(rng, n, k & 3) for k, n in enumerate(lens)]
    starts = [[], [int(x) for x in rng.integers(0, 1 << s, 40)]]
    return Case(name, (s, 30, 32), chunk, starts, samples, [k % 2 for k in range(len(samples))])


def _long_case(s, chunk):
    """Samples long enough that many CTAs share one; with an odd chunk, CTA boundaries fall inside bytes."""
    name = "long_s%d_chunk%d" % (s, chunk)
    rng = _rng(name)
    lens = [50000 * s // 8, 40000 * s // 8 + 1, 16384 * s // 8 + 3]
    samples = [sample_bytes(rng, n, k) for k, n in enumerate(lens)]
    return Case(name, (s, 30, 32), chunk, [[]], samples, [0] * len(samples))


def _freeze_case(s, f, c, chunk):
    """Samples whose limits lie below, at and above their symbol count, a start row already at freq_max (limit 0) and
    a mix of start rows in one call."""
    name = "freeze_s%d_f%d_chunk%d" % (s, f, chunk)
    rng = _rng(name)
    nsym, fmax = (1 << s) + 1, (1 << f) - 1
    room = fmax - nsym
    starts = [[], [int(x) for x in rng.integers(0, 1 << s, room)],          # fresh; trained to exactly freq_max
              [int(x) for x in rng.integers(0, 1 << s, room // 3)]]          # part-trained
    syms = [room - 100, room, room + 1, room + 500, room // 3, 2 * room // 3, 2 * room // 3 + 1]
    samples, model = [], []
    for k, n in enumerate(syms):
        for m in range(3):
            samples.append(sample_bytes(rng, (n * s + 7) // 8, (k + m) & 3))
            model.append(m)
    return Case(name, (s, f, c), chunk, starts, samples, model)


CASES = ([_width_case(s, 0) for s in range(1, 17)] + [_width_case(s, 97) for s in (1, 3, 5, 7, 8, 11, 13, 16)]
         + [_long_case(s, chunk) for s in (3, 8, 13) for chunk in (0, 1001)]
         + [_freeze_case(8, 12, 14, 0), _freeze_case(8, 12, 14, 97), _freeze_case(3, 11, 14, 101),
            _freeze_case(13, 16, 18, 0)])


def _state(params, seq):
    import redux_b200 as rb
    return rb.AdaptiveTreeModel(rb.Parameters(*params)).train(np.asarray(seq, dtype=np.int64))._state()


def start_table(case):
    """uint32[n_models, symbol_count]: the start rows of the case."""
    return np.stack([_state(case.params, seq) for seq in case.starts]).astype(np.uint32)


def expected_rows(case):
    """uint32[n_samples, symbol_count]: what the reference's model holds after each sample."""
    s = case.params[0]
    rows = []
    for smp, m in zip(case.samples, case.sample_model):
        seq = case.starts[m] + reference_symbols(smp, s)
        if len(seq) <= ORACLE_MAX_SYMBOLS:
            rows.append(o.trained_frequencies(seq, o.TREE, case.params))
        else:
            rows.append(_state(case.params, seq))
    return np.stack(rows).astype(np.uint32)


def concat(samples):
    """Samples back to back (+ 64 bytes of padding for the aligned 16-byte loads) and their offsets."""
    off = np.zeros(len(samples) + 1, dtype=np.uint64)
    np.cumsum([len(x) for x in samples], out=off[1:])
    data = np.zeros(int(off[-1]) + 64, dtype=np.uint8)
    data[:int(off[-1])] = np.frombuffer(b"".join(samples), dtype=np.uint8)
    return data, off
