"""Model building (redux_build.cuh) on the host emulation (tests/host_emu/build_emu.cpp) against the exact references
of build_models_cases.py.  No GPU needed; the device side is test_gpu_build_models.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import build_models_cases as bmc
import select_models_cases as smc
from test_host_emu import CSRC, EMU_DIR

BUILD_SO = os.path.join(EMU_DIR, "_build_emu.so")


def load_build_emu():
    srcs = [os.path.join(EMU_DIR, "build_emu.cpp"), os.path.join(EMU_DIR, "cuda_shim.h"),
            os.path.join(CSRC, "redux_build.cuh"), os.path.join(CSRC, "redux_select.cuh"),
            os.path.join(CSRC, "redux_train.cuh"), os.path.join(CSRC, "redux_common.cuh")]
    if not (os.path.exists(BUILD_SO) and all(os.path.getmtime(x) <= os.path.getmtime(BUILD_SO) for x in srcs)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas",
                        "-o", BUILD_SO, srcs[0]], check=True, cwd=EMU_DIR)
    L = C.CDLL(BUILD_SO)
    u32, u64, vp, i32 = C.c_uint32, C.c_uint64, C.c_void_p, C.c_int
    L.emu_build_ladder.argtypes = [u32, u32, vp, i32]
    L.emu_build_ladder.restype = u32
    L.emu_build_cluster.argtypes = [u32, u32, vp, vp, u64, vp]
    L.emu_build_cluster.restype = None
    L.emu_build_rows.argtypes = [u32, u32, u32, vp, vp, i32]
    L.emu_build_rows.restype = u32
    L.emu_build_round.argtypes = [u32, u32, u32, vp, vp, u64, u64, vp, vp, vp, vp, vp, i32]
    L.emu_build_round.restype = u32
    return L


@pytest.fixture(scope="module")
def emu():
    return load_build_emu()


def emu_ladder(emu, s, f, mutant=0):
    T = np.zeros(16, dtype=np.uint32)
    n = emu.emu_build_ladder(s, f, T.ctypes.data, mutant)
    return [int(t) for t in T[:n]]


def emu_rows(emu, s, f, G, mutant=0):
    """Candidate rows (K x L x nsym) of cluster sums G (K x 2^s, uint64)."""
    G = np.ascontiguousarray(G, dtype=np.uint64)
    K = G.shape[0]
    L = len(emu_ladder(emu, s, f, mutant))
    cand = np.zeros((K, L, (1 << s) + 1), dtype=np.uint32)
    assert emu.emu_build_rows(s, f, K, G.ctypes.data, cand.ctypes.data, mutant) == L
    return cand


# Cluster sums of the row cases: (kind, s, G row)
def _row_sums():
    rng = np.random.default_rng(0xB017)
    out = []
    for s in (1, 3, 8, 12, 16):
        bins = 1 << s
        ties = np.zeros(bins, np.uint64)
        ties[[bins // 2, bins - 1]] = 77                    # argmax tie: the lower bin gets the remainder
        ties[0] = 5
        one = np.zeros(bins, np.uint64)
        one[bins - 1] = 12345                               # one bin
        out += [("spread", s, rng.integers(0, 1000, bins).astype(np.uint64)), ("ties", s, ties), ("one", s, one),
                # sums past 2^32, products D G_x past 2^64 at large f
                ("big", s, rng.integers(1 << 40, 1 << 41, bins).astype(np.uint64)),
                ("empty", s, np.zeros(bins, np.uint64))]
    return out


# f = s + 2 (one ladder level) and large f
F_OF = {1: (3, 31), 3: (5, 12, 31), 8: (10, 14, 30), 12: (14, 16, 31), 16: (18, 31)}
ROW_CASES = [("%s_s%d_f%d" % (kind, s, f), s, f, G[None, :]) for kind, s, G in _row_sums() for f in F_OF[s]]
SF = ["s%d_f%d" % (s, f) for s in F_OF for f in F_OF[s]]


def row_cases():
    return ROW_CASES


def check_rows(emu, s, f, G, mutant=0):
    cand = emu_rows(emu, s, f, G, mutant)
    T = bmc.ladder(s, f)
    assert cand.shape[1] == len(T), "ladder length"
    for k in range(G.shape[0]):
        for li, t in enumerate(T):
            want = bmc.row([int(g) for g in G[k]], t, s)
            assert (cand[k, li] == want).all(), (k, li)


@pytest.mark.parametrize("name,s,f,G", list(row_cases()), ids=[c[0] for c in row_cases()])
def test_rows_equal_the_reference(emu, name, s, f, G):
    check_rows(emu, s, f, G)


def test_ladder_of_one_level_and_large_f():
    assert len(bmc.ladder(8, 10)) == 1 and len(bmc.ladder(8, 30)) == 7 + 4
    assert bmc.ladder(8, 14) == [16383, 4095, 1023]
    assert len(bmc.ladder(8, 22)) == 7 and bmc.ladder(8, 30)[-1] == 1023


def test_cluster_sums_equal_the_reference(emu):
    rng = np.random.default_rng(7)
    for s in (3, 8, 12):
        n, K = 300, 5
        hist = rng.integers(0, 1 << 31, (n, (1 << s) + 1), dtype=np.uint64).astype(np.uint32)
        hist[:, -1] = 0
        member = rng.integers(0, K + 1, n).astype(np.uint32)
        member[100:200] = 2                                       # long runs of one cluster
        G = np.zeros((K, 1 << s), dtype=np.uint64)
        emu.emu_build_cluster(s, K, hist.ctypes.data, member.ctypes.data, n, G.ctypes.data)
        want = bmc.aggregate(hist[:, :-1].astype(np.uint64), member, K)
        assert G.tolist() == want and max(max(r) for r in want) > 1 << 32


def emu_round(emu, case, member, mutant=0):
    s, f, _ = case.params
    data, off = smc.concat(case.blocks)
    n, K = len(case.blocks), case.K
    T = emu_ladder(emu, s, f, mutant)
    lcost = np.zeros((n, len(T)))
    level = np.zeros(K, dtype=np.uint32)
    table = np.ones((K + 1, (1 << s) + 1), dtype=np.uint32)
    meta = np.zeros(3 * (K + 1) + 2 * (len(T) + 1) + 1, dtype=np.uint32)
    member = np.ascontiguousarray(member, dtype=np.uint32)
    emu.emu_build_round(s, f, K, data.ctypes.data, off.ctypes.data, n, max(len(b) for b in case.blocks),
                        member.ctypes.data, lcost.ctypes.data, level.ctypes.data, table.ctypes.data,
                        meta.ctypes.data, mutant)
    return table, level, meta, T


def check_round(emu, case, mutant=0):
    """Every row equals the reference's candidate at the level chosen, and where the reference's best level beats the
    others by more than the tolerance of DESIGN.md 3.10, that level is chosen."""
    s, f, _ = case.params
    table, level, meta, T = emu_round(emu, case, case.init, mutant)
    S, tol, cand = bmc.ladder_sums(case, case.init)
    assert len(T) == S.shape[1], "ladder length"
    for k in range(case.K):
        assert (table[k + 1] == cand[k][level[k]]).all(), ("row", k)
        srt = np.sort(S[k])
        if srt.size == 1 or srt[1] - srt[0] > 2 * tol[k]:
            assert level[k] == int(np.argmin(S[k])), ("level", k, S[k].tolist())
    # the meta: {total, EOF} per row, the rows by split point, fresh last
    n_models, G = case.K + 1, len(T) + 1
    start = meta[:2 * n_models].reshape(n_models, 2)
    assert (start[:, 0] == table.astype(np.int64).sum(axis=1)).all() and (start[:, 1] == 1).all()
    order = meta[2 * n_models:3 * n_models]
    group = meta[3 * n_models:3 * n_models + G + 1]
    want = sorted(range(n_models), key=lambda k: -int(start[k, 0]))
    assert order.tolist() == want and group[0] == 0 and group[-1] == n_models


@pytest.mark.parametrize("case", bmc.CASES, ids=lambda c: c.name)
def test_round_equals_the_reference(emu, case):
    check_round(emu, case)


def _fails(fn):
    try:
        fn()
    except AssertionError:
        return True
    return False


# The cases each mutant must fail: the remainder in bin 0 fails wherever there is a remainder and the argmax is another
# bin (not for one bin, which takes all of D, nor the ones of an empty cluster, nor s = 1 where bin 0 is the larger); a 64-bit product fails where D G_x passes 2^64; an empty cluster not replaced by ones fails the empty
# ones; a ladder that stops at nsym has an extra level where F >> 2l falls in [nsym, 2 nsym).
KINDS = ("spread", "ties", "one", "big", "empty")
MUTANT_ROW_FAILS = {1: {"%s_%s" % (k, sf) for k in ("spread", "ties", "big") for sf in SF
                        if not (k != "ties" and sf.startswith("s1_"))},
                    2: {"big_s1_f31", "big_s3_f31", "big_s8_f30", "big_s12_f31", "big_s16_f31"},
                    3: {"empty_%s" % sf for sf in SF},
                    4: {"%s_%s" % (k, sf) for k in KINDS for sf in ("s3_f12", "s12_f31", "s16_f31")}}


@pytest.mark.parametrize("mutant", [1, 2, 3, 4])
def test_mutants_fail_named_cases(emu, mutant):
    failed = {name for name, s, f, G in row_cases() if _fails(lambda: check_rows(emu, s, f, G, mutant))}
    assert failed == MUTANT_ROW_FAILS[mutant]
    if mutant == 3:
        assert _fails(lambda: check_round(emu, bmc.CASES[5], mutant))     # empty_cluster
