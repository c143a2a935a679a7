"""Cases and references of redux_build_models (start models learned by clustering the blocks, DESIGN.md 3.12).

The aggregation, the ladder and the row rule are exact integer arithmetic here (Python ints for the 128-bit product);
the cost of a block under a row is select_models_cases' float64 closed form.

Imported by test_build_models_emu.py (host emulation), test_build_models_cpu.py and test_gpu_build_models.py -- data
and helpers only.
"""
import zlib
from collections import namedtuple

import numpy as np

import select_models_cases as smc
from train_models_cases import sample_bytes

Case = namedtuple("Case", "name params K blocks init")


def ladder(s, f, floor_mult=2):
    """T_l = F >> 2l while T_l >= floor_mult * nsym (the contract's floor is 2 nsym)."""
    F, nsym = (1 << f) - 1, (1 << s) + 1
    out = []
    while (F >> (2 * len(out))) >= floor_mult * nsym:
        out.append(F >> (2 * len(out)))
    return out


def histogram(block, s):
    """H_b: uint64[2^s], the block's symbols (MSB-first, a trailing partial symbol dropped)."""
    return np.bincount(smc.symbols(block, s), minlength=1 << s).astype(np.uint64)


def aggregate(hists, member, K):
    """G: K x 2^s Python ints, G[k-1] = sum of H_b over the blocks with member[b] == k."""
    bins = hists.shape[1] if len(hists) else 0
    G = [[0] * bins for _ in range(K)]
    for h, k in zip(hists, member):
        if k:
            row = G[int(k) - 1]
            for x in np.flatnonzero(h):
                row[x] += int(h[x])
    return G


def row(G, T, s):
    """row(G, T): uint32[nsym] with total exactly T."""
    nsym = (1 << s) + 1
    G = [int(g) for g in G]
    S = sum(G)
    if S == 0:
        G, S = [1] * (nsym - 1), nsym - 1
    D = T - nsym
    q = [D * g // S for g in G]
    r = [1 + v for v in q] + [1]
    xmax = max(range(nsym - 1), key=lambda x: (G[x], -x))
    r[xmax] += D - sum(q)
    out = np.array(r, dtype=np.uint64)
    assert int(out.sum()) == T and out.min() >= 1
    return out.astype(np.uint32)


def fresh(s):
    return np.ones((1 << s) + 1, dtype=np.uint32)


def ladder_sums(case, member):
    """S[k-1][l]: the reference (closed-form) cost of cluster k's blocks under row(G_k, T_l), and the candidates."""
    s, f, _ = case.params
    T = ladder(s, f)
    hists = np.stack([histogram(b, s) for b in case.blocks])
    G = aggregate(hists, member, case.K)
    cand = [[row(G[k], t, s) for t in T] for k in range(case.K)]
    syms = [smc.symbols(b, s) for b in case.blocks]
    S = np.zeros((case.K, len(T)))
    tol = np.zeros(case.K)
    for b, k in enumerate(member):
        if k:
            c = np.array([smc.closed_cost(cand[int(k) - 1][l], syms[b], case.params) for l in range(len(T))])
            S[int(k) - 1] += c
            tol[int(k) - 1] += float(smc.tolerance(c.min()))
    return S, tol, cand


def default_init(n, K):
    return np.array([1 + b * K // n for b in range(n)], dtype=np.uint32)


def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


def _small_case(s, f, K, n, length):
    """n blocks of the four generator classes at width s; init: contiguous ranges with one block set to fresh, so one
    cluster may be empty when K > n / 2."""
    name = "small_s%d_f%d_k%d" % (s, f, K)
    rng = _rng(name)
    blocks = [sample_bytes(rng, length + (i % 3), i % 4) for i in range(n)]
    init = default_init(n, K)
    init[0] = 0
    return Case(name, (s, f, f + 2), K, blocks, init)


def _empty_cluster_case():
    """K = 3 with nothing in cluster 2: its rows come from a histogram of ones."""
    name = "empty_cluster"
    rng = _rng(name)
    blocks = [sample_bytes(rng, 3000, c) for c in (1, 1, 3, 3)]
    return Case(name, (8, 14, 16), 3, blocks, np.array([1, 1, 3, 3], dtype=np.uint32))


def _one_bin_case():
    """A cluster of blocks holding one byte value: the whole remainder goes to that bin."""
    blocks = [bytes([7]) * 5000, bytes([7]) * 3000, bytes(range(256)) * 10]
    return Case("one_bin", (8, 14, 16), 2, blocks, np.array([1, 1, 2], dtype=np.uint32))


CASES = ([_small_case(s, f, K, n, L) for s, f, K, n, L in
          ((3, 12, 2, 6, 1500), (3, 20, 3, 6, 1500), (12, 16, 2, 5, 3000), (8, 14, 4, 16, 4096),
           (8, 30, 4, 16, 4096))]
         + [_empty_cluster_case(), _one_bin_case()])


def generator_case(params, n, length, K, seed=0xB011D2026102200):
    """n generator blocks (block index & 3 is the class) of `length` bytes, default init."""
    import redux_b200 as rb
    data = rb.generate_blocks_host(0, n, length, seed)
    blocks = [data[i * length:(i + 1) * length].tobytes() for i in range(n)]
    return Case("gen_%d_%d_%d" % params, params, K, blocks, None)
