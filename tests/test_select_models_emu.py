"""Model selection (redux_select.cuh) on the host emulation (tests/host_emu/select_emu.cpp) against the references of
select_models_cases.py.  No GPU needed; the device side of the same cases is test_gpu_select_models.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import select_models_cases as smc
from test_host_emu import CSRC, EMU_DIR

SELECT_SO = os.path.join(EMU_DIR, "_select_emu.so")


def load_select_emu():
    srcs = [os.path.join(EMU_DIR, "select_emu.cpp"), os.path.join(EMU_DIR, "cuda_shim.h"),
            os.path.join(CSRC, "redux_select.cuh"), os.path.join(CSRC, "redux_train.cuh"),
            os.path.join(CSRC, "redux_common.cuh")]
    if not (os.path.exists(SELECT_SO) and all(os.path.getmtime(x) <= os.path.getmtime(SELECT_SO) for x in srcs)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas",
                        "-o", SELECT_SO, srcs[0]], check=True, cwd=EMU_DIR)
    L = C.CDLL(SELECT_SO)
    u32, u64, vp = C.c_uint32, C.c_uint64, C.c_void_p
    L.emu_select.argtypes = [u32, u32, u32, vp, u32, vp, vp, u64, u64, vp, vp, C.c_int]
    L.emu_select.restype = None
    return L


@pytest.fixture(scope="module")
def emu():
    return load_select_emu()


def emu_select(emu, case, mutant=0):
    s, f, _ = case.params
    data, off = smc.concat(case.blocks)
    tab = smc.table(case)
    n = len(case.blocks)
    choice = np.zeros(n, dtype=np.uint32)
    cost = np.zeros((n, tab.shape[0]), dtype=np.float64)
    emu.emu_select(s, f, case.chunk, tab.ctypes.data, tab.shape[0], data.ctypes.data, off.ctypes.data, n,
                   max(len(b) for b in case.blocks), choice.ctypes.data, cost.ctypes.data, mutant)
    return choice, cost


@pytest.fixture(scope="module")
def refs():
    cache = {}

    def get(case):
        if case.name not in cache:
            cache[case.name] = smc.reference_costs(case)
        return cache[case.name]
    return get


@pytest.mark.parametrize("case", smc.CASES, ids=lambda c: c.name)
def test_selection_equals_reference(emu, refs, case):
    choice, cost = emu_select(emu, case)
    smc.check_choice(case, refs(case), cost, choice)


# The cases each mutant fails (DESIGN.md 3.10).  Ignoring the freeze (m = n always) fails every case with a model that
# freezes before the end of a block; at freq_bits 30 no model does.  Coding EOF against T instead of T' fails every case
# where log2(T'/T) exceeds the tolerance somewhere; in s16_f18 it stays below it.
WIDTH = ["s1_f12", "s3_f12", "s7_f13", "s8_f13", "s12_f16", "s16_f18"]
MUTANT_FAILS = {1: set(WIDTH + ["many_k1", "many_k300", "winner_f14"]),
                2: set(WIDTH[:-1] + ["many_k1", "many_k300", "long_s3_chunk0", "long_s8_chunk0", "long_s3_chunk1001",
                                     "winner_f14", "winner_f30"])}


@pytest.mark.parametrize("mutant", [1, 2])
def test_mutants_fail_named_cases(emu, refs, mutant):
    failed = set()
    for case in smc.CASES:
        choice, cost = emu_select(emu, case, mutant)
        try:
            smc.check_choice(case, refs(case), cost, choice)
        except AssertionError:
            failed.add(case.name)
    assert failed == MUTANT_FAILS[mutant]
