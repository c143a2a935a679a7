"""Blocks of one launch that start from different trained models, on the host emulation of the tuned lane kernels and
the generic kernels (tests/host_emu/block_models_emu.cpp), against the oracle block by block.  No GPU needed; the device
side of the same cases is test_gpu_block_models.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import block_models_cases as bmc
import kernel_matrix_cases as km
from test_host_emu import CSRC, EMU_DIR, concat, load_emu
from test_kernel_coverage import NARROW, WIDE, WIDE_D, lane_plan

MODELS_SO = os.path.join(EMU_DIR, "_block_models_emu.so")


def load_models_emu():
    srcs = [os.path.join(EMU_DIR, "block_models_emu.cpp"), os.path.join(EMU_DIR, "cuda_shim.h")] + [
        os.path.join(CSRC, h) for h in ("redux_lane_codec.cuh", "redux_lane_al.cuh", "redux_generic_codec.cuh",
                                        "redux_common.cuh")]
    if not (os.path.exists(MODELS_SO) and all(os.path.getmtime(x) <= os.path.getmtime(MODELS_SO) for x in srcs)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas",
                        "-o", MODELS_SO, srcs[0]], check=True, cwd=EMU_DIR)
    L = C.CDLL(MODELS_SO)
    u32, u64, vp, i32 = C.c_uint32, C.c_uint64, C.c_void_p, C.c_int
    L.emu_encode_lane_models.argtypes = [u32, u32, u64, i32, vp, u32, vp, vp, vp, u64, vp, vp, vp]
    L.emu_decode_lane_models.argtypes = [u32, u32, u64, i32, vp, u32, vp, vp, vp, u64, vp, vp, vp, vp, vp]
    L.emu_encode_generic_models.argtypes = [u32, u32, u32, vp, u32, vp, u32, vp, vp, u64, vp, u64, vp, vp]
    L.emu_decode_generic_models.argtypes = [u32, u32, u32, vp, u32, vp, u32, vp, vp, u64, vp, vp, vp, vp, vp]
    return L


class Emu:
    """The per-block model kernels (block_models_emu.cpp) and the front end's lane_plan (lane_emu.cpp)."""

    def __init__(self):
        self.models, self.lane = load_models_emu(), load_emu()


@pytest.fixture(scope="module")
def emu():
    return Emu()


class EmuBackend:
    """The kernels the front end would launch for the case, run thread by thread on the CPU."""

    def __init__(self, emu, case):
        self.emu, self.case = emu, case

    def encode(self, blocks, table, bm):
        s, f, c = self.case.params
        data, off = concat(blocks)
        n = len(blocks)
        max_len = max(len(b) for b in blocks)
        bound = ((max_len * 8 // s + 1) * c + 7) // 8
        stride = ((bound + 15) & ~15) + 16           # as lane_plan / make_plan size the slots
        slots = np.zeros(n * stride + 64, dtype=np.uint8)
        base = (-slots.ctypes.data) % 16
        sizes = np.full(n, 0xFFFFFFFF, dtype=np.uint32)
        status = np.full(n, -1, dtype=np.int32)
        table = np.ascontiguousarray(table, dtype=np.uint32)
        bm = np.ascontiguousarray(bm, dtype=np.uint32)
        args = (data.ctypes.data, off.ctypes.data, n, slots.ctypes.data + base)
        if bmc.is_generic(self.case):
            self.emu.models.emu_encode_generic_models(s, f, c, table.ctypes.data, table.shape[0], bm.ctypes.data, 128, *args,
                                               stride, sizes.ctypes.data, status.ctypes.data)
        else:
            assert self.emu.lane.emu_slot_stride(f, c, max_len) == stride
            self.emu.models.emu_encode_lane_models(f, c, max_len, -1, table.ctypes.data, table.shape[0], bm.ctypes.data, *args,
                                            sizes.ctypes.data, status.ctypes.data)
        return [slots[base + i * stride: base + i * stride + int(sizes[i])].tobytes() for i in range(n)], status

    def decode(self, comp, coff, raw, roff, max_len, table, bm):
        s, f, c = self.case.params
        n = coff.size - 1
        raw_len, consumed = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint64)
        status = np.full(n, -1, dtype=np.int32)
        table = np.ascontiguousarray(table, dtype=np.uint32)
        args = (comp.ctypes.data, coff.ctypes.data, n, raw.ctypes.data, roff.ctypes.data, raw_len.ctypes.data,
                consumed.ctypes.data, status.ctypes.data)
        if bmc.is_generic(self.case):
            self.emu.models.emu_decode_generic_models(s, f, c, table.ctypes.data, table.shape[0], bm.ctypes.data, 128, *args)
        else:
            self.emu.models.emu_decode_lane_models(f, c, max_len, -1, table.ctypes.data, table.shape[0], bm.ctypes.data, *args)
        return raw, raw_len, consumed, status

    def kernels(self):
        return None                    # test_case_plan_selects_its_kernel checks the selection


def plan_kernels(emu, case, max_len):
    """(encode, decode) kernels pick_encoder / pick_decoder choose for the plan of the case's largest start total."""
    _, f, c = case.params
    p = lane_plan(emu.lane, f, c, max_len, max(bmc.totals(case)), True)
    assert p["aligned"] and p["full_table"]
    if p["cls"] == NARROW:
        return km.NARROW_STG if c <= 16 else km.NARROW
    return km.lane("u32" if p["wide_table"] else "u16", {WIDE: "Wide", WIDE_D: "WideD"}[p["cls"]], True, c == 32)


LANE_CASES = [c for c in bmc.CASES if not bmc.is_generic(c)]


def test_cases_cover_every_trained_lane_kernel():
    """Every tuned lane kernel a trained model can reach (the trained and full-table rows of the kernel matrix) has a
    case here, and one case holds a fresh model, one trained to freq_max, one past 65,535, one with a heavily trained
    EOF and one a step below the WIDE_D bound in every warp."""
    reachable = {(c.enc, c.dec) for c in km.CASES if c.enc.startswith("encode_lane_al") and ",full," in c.enc}
    assert {(c.enc, c.dec) for c in LANE_CASES} == reachable
    assert any({"ones", "fmax", "u32", "eof", "wided_last"} <= set(c.kinds) for c in LANE_CASES)


@pytest.mark.parametrize("case", LANE_CASES, ids=lambda c: c.name)
def test_case_plan_selects_its_kernel(emu, case):
    """The plan from the case's largest start total selects the kernels the case names, and the models are what their
    kinds promise."""
    _, f, c = case.params
    tot = dict(zip(case.kinds, bmc.totals(case)))
    assert tot["ones"] == km.NSYM
    assert tot.get("fmax", (1 << f) - 1) == (1 << f) - 1
    assert tot.get("u32", 70000) == 70000 and tot.get("wide", km.WIDE_D_BOUND + 100) == km.WIDE_D_BOUND + 100
    if "wided_last" in tot:
        assert tot["wided_last"] + bmc.max_len(case) == km.WIDE_D_BOUND - 1
    assert plan_kernels(emu, case, bmc.max_len(case)) == (case.enc, case.dec)


@pytest.mark.parametrize("case", bmc.CASES, ids=lambda c: c.name)
def test_block_models_equal_oracle(emu, case):
    """Each block against compress_trained / decompress_trained with its own model's training, and the decoder's error
    exits under mixed models between good neighbours."""
    bmc.check_case(case, EmuBackend(emu, case))


@pytest.mark.parametrize("case", [bmc.CASES[0], bmc.CASES[7], bmc.CASES[-2]], ids=lambda c: c.name)
def test_out_of_range_model_index(emu, case):
    bmc.check_bad_index(case, EmuBackend(emu, case))


def test_plan_from_the_largest_total_serves_every_smaller_one(emu):
    """make_plan plans a launch for its largest start total.  Each choice lane_plan makes from that total -- u32
    entries, the WIDE_D class (a division valid below the bound), the reciprocal table's length -- must hold for every
    block that starts from a smaller total: swept over byte-symbol parameters with code_bits <= 32, block lengths and
    pairs of start totals around the thresholds."""
    checked = 0
    for f in range(10, 31, 2):
        fmax = (1 << f) - 1
        for c in (f + 2, 32) if f + 2 < 32 else (f + 2,):
            starts = sorted({t + d for t in (km.NSYM, 3000, 65535, km.WIDE_D_BOUND, fmax) for d in (-1, 0, 1)
                             if km.NSYM <= t + d <= fmax})
            for L in (0, 1, 1000, 65535, km.WIDE_D_BOUND - km.NSYM, 1 << 21):
                plans = {t: lane_plan(emu.lane, f, c, L, t, True) for t in starts}
                for lo in starts:
                    for hi in starts:
                        if lo > hi:
                            continue
                        a, b = plans[lo], plans[hi]
                        assert b["full_table"] and a["full_table"]
                        assert (a["cls"] == NARROW) == (b["cls"] == NARROW)
                        assert b["wide_table"] or not a["wide_table"], (f, c, L, lo, hi)
                        assert a["cls"] == WIDE_D or b["cls"] != WIDE_D, (f, c, L, lo, hi)
                        # highest reciprocal entry a block reads: count0 - 257 + min(len, tcap) (+ read-ahead)
                        assert lo + min(L, a["tcap"]) <= hi + min(L, b["tcap"])
                        assert a["tcap"] == fmax - lo
                        checked += 1
    assert checked > 1000
