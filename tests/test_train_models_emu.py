"""Model training (redux_train.cuh) on the host emulation (tests/host_emu/train_emu.cpp) against the reference's
get_frequency.  No GPU needed; the device side of the same cases is test_gpu_train_models.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as o
import train_models_cases as tmc
from test_host_emu import CSRC, EMU_DIR

TRAIN_SO = os.path.join(EMU_DIR, "_train_emu.so")


def load_train_emu():
    srcs = [os.path.join(EMU_DIR, "train_emu.cpp"), os.path.join(EMU_DIR, "cuda_shim.h"),
            os.path.join(CSRC, "redux_train.cuh"), os.path.join(CSRC, "redux_common.cuh")]
    if not (os.path.exists(TRAIN_SO) and all(os.path.getmtime(x) <= os.path.getmtime(TRAIN_SO) for x in srcs)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas",
                        "-o", TRAIN_SO, srcs[0]], check=True, cwd=EMU_DIR)
    L = C.CDLL(TRAIN_SO)
    u32, u64, vp = C.c_uint32, C.c_uint64, C.c_void_p
    L.emu_train_copies.argtypes = [u32]
    L.emu_train_copies.restype = u32
    L.emu_train.argtypes = [u32, u32, u32, vp, u32, vp, vp, vp, u64, u64, vp]
    L.emu_train.restype = None
    return L


@pytest.fixture(scope="module")
def emu():
    return load_train_emu()


def emu_train(emu, case, table, sample_model=None):
    s, f, _ = case.params
    data, off = tmc.concat(case.samples)
    n = len(case.samples)
    bm = np.ascontiguousarray(case.sample_model if sample_model is None else sample_model, dtype=np.uint32)
    table = np.ascontiguousarray(table, dtype=np.uint32)
    out = np.zeros((n, (1 << s) + 1), dtype=np.uint32)
    max_len = max(len(x) for x in case.samples)
    emu.emu_train(s, f, case.chunk, table.ctypes.data, table.shape[0], bm.ctypes.data, data.ctypes.data,
                  off.ctypes.data, n, max_len, out.ctypes.data)
    return out


@pytest.mark.parametrize("case", tmc.CASES, ids=lambda c: c.name)
def test_training_equals_reference(emu, case):
    want = tmc.expected_rows(case)
    got = emu_train(emu, case, tmc.start_table(case))
    for i in range(len(case.samples)):
        assert (got[i] == want[i]).all(), (case.name, i, np.flatnonzero(got[i] != want[i])[:8])


def test_cases_cover_what_the_semantics_name():
    """Every width, empty samples and samples shorter than one symbol, CTA boundaries inside a byte, a start row at
    freq_max, limits below, at and above the symbol count, and several start rows in one call."""
    assert {c.params[0] for c in tmc.CASES} == set(range(1, 17))
    lens = [(len(x) * 8, c.params[0]) for c in tmc.CASES for x in c.samples]
    assert any(b == 0 for b, _ in lens) and any(0 < b < s for b, s in lens)
    assert any(c.chunk and c.chunk * c.params[0] % 8 for c in tmc.CASES if c.params[0] in (3, 13))
    at_limit = 0
    for c in tmc.CASES:
        if not c.name.startswith("freeze"):
            continue
        s, f, _ = c.params
        room = (1 << f) - 1 - ((1 << s) + 1)
        assert len(c.starts[1]) == room and len(set(c.sample_model)) == 3
        nsyms = {len(x) * 8 // s for x in c.samples}
        assert min(nsyms) < room < max(nsyms)
        at_limit += room in nsyms
    assert at_limit >= 2


def test_linear_and_tree_models_train_alike():
    """The closed form is the same for both model kinds: the oracle's linear model ends where its tree model does."""
    case = tmc._freeze_case(3, 11, 14, 101)
    for smp, m in list(zip(case.samples, case.sample_model))[:6]:
        seq = case.starts[m] + tmc.reference_symbols(smp, 3)
        assert (o.trained_frequencies(seq, o.LINEAR, case.params) == o.trained_frequencies(seq, o.TREE, case.params)).all()


def test_copies_fit_shared_memory(emu):
    """One sub-histogram per warp while they fit in 64 KiB of shared memory, global counting past 14 bits."""
    for s in range(1, 17):
        k = emu.emu_train_copies(s)
        assert (k == 0) if s > 14 else (1 <= k <= 8 and k << s <= 16384), (s, k)
