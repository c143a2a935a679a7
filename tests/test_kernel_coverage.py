"""Every kernel the device path can launch has a row in the kernel matrix (tests/kernel_matrix_cases.py), and the lane
rows hold without a GPU: the plan behind each row selects the kernel the row names, and the tuned lane kernels, run
in the host emulation (tests/host_emu/), equal the oracle on each row's blocks and error streams.

The GPU side of the same table is tests/test_gpu_kernel_matrix.py, which also checks the kernel names through
redux_debug_launched_kernels.
"""
import ctypes as C

import numpy as np
import pytest

import kernel_matrix_cases as km
import redux_b200 as rb
from test_host_emu import emu_encode, load_emu

NARROW, WIDE, HUGE, WIDE_D = 0, 1, 2, 3          # ArithClass (redux_b200/csrc/redux_common.cuh)


@pytest.fixture(scope="module")
def emu():
    return load_emu()


def lane_plan(emu, f, c, max_len, count0=km.NSYM, pretrained=False):
    out = (C.c_uint32 * 5)()
    emu.emu_lane_plan(f, c, max_len, count0, 1 if pretrained else 0, out)
    return {"cls": out[0], "wide_table": bool(out[1]), "full_table": bool(out[2]), "aligned": bool(out[3]), "tcap": out[4]}


def lane_kernels(emu, case, max_len):
    """(encode, decode) kernel names pick_encoder / pick_decoder of redux_capi.cu choose for lane_plan's result."""
    _, f, c = case.params
    p = lane_plan(emu, f, c, max_len, int(km.trained_freq(case).sum()), case.train > 0)
    tw = "u32" if p["wide_table"] else "u16"
    if not p["aligned"]:
        return "encode_lane<%s,Huge>" % tw, "decode_lane<%s,Huge>" % tw
    if p["cls"] == NARROW:
        return km.NARROW_STG if c <= 16 else km.NARROW
    return km.lane(tw, {WIDE: "Wide", WIDE_D: "WideD"}[p["cls"]], p["full_table"], c == 32)


def is_lane_row(case):
    return case.enc.startswith("encode_lane")


def test_rows_reach_exactly_the_library_kernels():
    """The rows' kernels are exactly the kernels the library can launch: a kernel added without a row, or a row
    deleted that was the only one reaching its kernel, fails here."""
    names = rb.kernel_names()
    assert len(names) == len(set(names)) == 37
    expected = km.expected_kernels()
    assert expected == set(names), ("no row for %s" % sorted(set(names) - expected),
                                    "not a kernel: %s" % sorted(expected - set(names)))
    assert len({c.name for c in km.CASES}) == len(km.CASES)


def test_wide_class_plans_take_u32_entries(emu):
    """lane_plan keeps the plain WIDE class (64-bit magics) only when count0 + updates >= 349,525 > 65,535, which
    always takes u32 entries: the library has no u16 WIDE lane kernel, and lane_plan states the rule outright so
    that no threshold change can ask for one.  Swept over every byte-symbol (f, c) with c <= 32, block lengths at
    every threshold +-1 and fresh / trained start totals around 65,535 and 349,525.  NARROW plans are always u16
    entries with full values (the library has no other NARROW lane kernel)."""
    wide = 0
    for f in range(10, 31):
        fmax = (1 << f) - 1
        for c in range(f + 2, 33):
            lens = {0, 1, km.FULL_MAX_UPDATES, km.U16_MAX_UPDATES, km.WIDE_D_BOUND - km.NSYM, 1 << 20}
            lens |= {km.tcap(f), 65535 - km.NSYM}
            lens = {x + d for x in lens for d in (-1, 0, 1) if x + d >= 0}
            starts = [(km.NSYM, False), (km.NSYM, True)] + [(t + d, True) for t in (65535, km.WIDE_D_BOUND, fmax)
                                                             for d in (-1, 0, 1)]
            for count0, trained in starts:
                if count0 > fmax:
                    continue
                for L in sorted(lens | {km.tcap(f, count0) + d for d in (-1, 0, 1)}):
                    p = lane_plan(emu, f, c, L, count0, trained)
                    assert p["aligned"]
                    if p["cls"] == WIDE:
                        wide += 1
                        assert p["wide_table"], (f, c, L, count0, trained)
                    if p["cls"] == NARROW:
                        assert not p["wide_table"] and p["full_table"], (f, c, L, count0, trained)
    assert wide > 100


@pytest.mark.parametrize("case", [c for c in km.CASES if is_lane_row(c)], ids=lambda c: c.name)
def test_row_plan_selects_its_kernel(emu, case):
    """The front end's lane_plan at the row's longest block (and at each extra slot capacity) selects the kernels
    the row names, so moving a threshold in lane_plan shows up here before the GPU run."""
    blocks = km.blocks_for(case)
    assert lane_kernels(emu, case, max(len(b) for b in blocks)) == (case.enc, case.dec)
    for cap, kernel in case.caps.items():
        assert lane_kernels(emu, case, cap)[1] == kernel


class EmuBackend:
    """The lane kernels of redux_lane_codec.cuh / redux_lane_al.cuh run thread by thread on the CPU."""

    def __init__(self, emu, case):
        self.emu, self.case = emu, case
        self.freq = km.trained_freq(case) if case.train else None

    def encode(self, blocks):
        _, f, c = self.case.params
        return emu_encode(self.emu, blocks, f, c, freq=self.freq)

    def decode(self, comp, coff, raw, roff, max_len):
        _, f, c = self.case.params
        n = coff.size - 1
        raw_len, consumed = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint64)
        status = np.full(n, -1, dtype=np.int32)
        self.emu.emu_decode_lane_ex(f, c, max_len, -1, None if self.freq is None else self.freq.ctypes.data,
                                    comp.ctypes.data, coff.ctypes.data, n, raw.ctypes.data, roff.ctypes.data,
                                    raw_len.ctypes.data, consumed.ctypes.data, status.ctypes.data)
        return raw, raw_len, consumed, status

    def kernels(self):
        return None                    # test_row_plan_selects_its_kernel checks the selection


@pytest.mark.parametrize("case", [c for c in km.CASES if is_lane_row(c)], ids=lambda c: c.name)
def test_lane_row_in_host_emulation(emu, case):
    """Encode, exact-capacity decode, error exits and slot isolation of the row (km.check_row) on the emulated lane
    kernels: a wrong bit in one of them is caught here before GPU time is spent."""
    km.check_row(case, EmuBackend(emu, case))
