"""CRC-32 (redux_crc.cuh) on the host emulation (tests/host_emu/crc_emu.cpp) against zlib.crc32.  No GPU needed; the
device side of the same cases is test_gpu_crc32.py.  The emulation uses pieces of crc32_cases.EMU_PIECE bytes, so the
piece boundaries fall at odd places and every case longer than a few KiB spans several pieces."""
import ctypes as C
import os
import subprocess
import zlib

import numpy as np
import pytest

import crc32_cases as cc
from test_host_emu import CSRC, EMU_DIR

CRC_SO = os.path.join(EMU_DIR, "_crc_emu.so")


def load_crc_emu():
    srcs = [os.path.join(EMU_DIR, "crc_emu.cpp"), os.path.join(EMU_DIR, "cuda_shim.h"),
            os.path.join(CSRC, "redux_crc.cuh"), os.path.join(CSRC, "redux_common.cuh")]
    if not (os.path.exists(CRC_SO) and all(os.path.getmtime(x) <= os.path.getmtime(CRC_SO) for x in srcs)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas",
                        "-o", CRC_SO, srcs[0]], check=True, cwd=EMU_DIR)
    L = C.CDLL(CRC_SO)
    u32, u64, vp = C.c_uint32, C.c_uint64, C.c_void_p
    L.emu_crc32.argtypes = [vp, vp, vp, u64, u64, u32, vp, C.c_int, C.c_int]
    L.emu_crc32.restype = None
    return L


@pytest.fixture(scope="module")
def emu():
    return load_crc_emu()


def _padded(data):
    """The bytes in a buffer with 32 filler bytes on each side: the kernel's aligned loads may read up to 15 bytes
    beyond a block's first and last byte."""
    buf = np.full(data.size + 64, 0x77, dtype=np.uint8)
    buf[32:32 + data.size] = data
    return buf, buf[32:]


def emu_crc(emu, data, off, lens=None, piece=cc.EMU_PIECE, mutant=0, shape=0):
    buf, view = _padded(data)
    n = off.size - 1
    blk = lens if lens is not None else off[1:] - off[:-1]
    crc = np.zeros(max(n, 1), dtype=np.uint32)
    emu.emu_crc32(view.ctypes.data, off.ctypes.data, None if lens is None else lens.ctypes.data, n,
                  int(blk.max()) if n else 0, piece, crc.ctypes.data, mutant, shape)
    return crc[:n]


@pytest.mark.parametrize("case", cc.CASES, ids=lambda c: c.name)
def test_crc_equals_zlib(emu, case):
    data, off = cc.layout(case)
    assert (emu_crc(emu, data, off) == cc.expected(case)).all()


@pytest.mark.parametrize("case", cc.CASES, ids=lambda c: c.name)
def test_crc_with_lengths_equals_zlib(emu, case):
    data, off, lens = cc.slots(case)
    assert (emu_crc(emu, data, off, lens) == cc.expected(case)).all()


@pytest.mark.parametrize("shape", [1, 2, 3, 4])
@pytest.mark.parametrize("case", cc.CASES, ids=lambda c: c.name)
def test_other_kernel_shapes_equal_zlib(emu, case, shape):
    """The shapes scripts/bench_crc32.py times besides the library's: 16 replicas with the next vectors loaded ahead,
    8 replicas, one table with the next vectors loaded ahead, and two chains per lane (which needs segments of a
    multiple of 64 bytes: pieces of 2,048 bytes here)."""
    data, off = cc.layout(case)
    piece = 2048 if shape == 4 else cc.EMU_PIECE
    assert (emu_crc(emu, data, off, piece=piece, shape=shape) == cc.expected(case)).all()


@pytest.mark.parametrize("piece", [512, 1024, 4608, cc.LIB_PIECE])
def test_other_piece_lengths(emu, piece):
    case = next(c for c in cc.CASES if c.name == "random_ragged")
    data, off = cc.layout(case)
    assert (emu_crc(emu, data, off, piece=piece) == cc.expected(case)).all()


def test_cases_cover_what_the_contract_names():
    lens = {len(b) for c in cc.CASES for b in c.blocks}
    assert {0, 1, 2, 3, 15, 16, 17, 31, 4095, 4096, 4097} <= lens
    for p in (cc.EMU_PIECE, cc.LIB_PIECE):
        assert {p - 1, p, p + 1} <= lens
    assert max(lens) > 4 * cc.LIB_PIECE
    starts = set()
    for c in cc.CASES:
        _, off = cc.layout(c)
        starts |= {int(o) % 16 for o, b in zip(off[:-1], c.blocks) if 0 < len(b) < 8}
    assert starts == set(range(16))
    assert any(b == bytes(len(b)) and len(b) > 4096 for c in cc.CASES for b in c.blocks)
    assert any(b == b"\xff" * len(b) and len(b) > 4096 for c in cc.CASES for b in c.blocks)


# The cases each mutant fails.  Pieces XORed without their shift, and the initial value applied per piece, fail
# exactly the cases with a block of more than one piece; the tail mask one byte too long fails every case with a block
# whose end is not 16-byte aligned (the filler or the next block's first byte is never zero here).
MULTI_PIECE = {"lengths", "lengths_lead3", "empty_between", "constant", "generator", "random_ragged",
               "emu_piece_edges", "lib_piece_edges", "many_pieces"}
MUTANT_FAILS = {1: MULTI_PIECE, 2: MULTI_PIECE,
                3: MULTI_PIECE | {"starts_mod16", "starts_mod16_short"}}


def test_multi_piece_cases_are_the_ones_named():
    def pieces(start, n):
        e = start + n
        vs, ep = (start if n >= 4 else e - 4) // 16 * 16, (e + 15) // 16 * 16
        return -(-(ep - vs) // cc.EMU_PIECE) if n else 0
    multi = set()
    for c in cc.CASES:
        _, off = cc.layout(c)
        if any(pieces(int(o), len(b)) > 1 for o, b in zip(off[:-1], c.blocks)):
            multi.add(c.name)
    assert multi == MULTI_PIECE


@pytest.mark.parametrize("mutant", [1, 2, 3])
def test_mutants_fail_named_cases(emu, mutant):
    failed = set()
    for case in cc.CASES:
        data, off = cc.layout(case)
        if not (emu_crc(emu, data, off, mutant=mutant) == cc.expected(case)).all():
            failed.add(case.name)
    assert failed == MUTANT_FAILS[mutant]


def test_zlib_agrees_with_the_definition():
    """CRC-32/ISO-HDLC bit by bit: reflected 0xEDB88320, initial value and final XOR 0xFFFFFFFF."""
    def crc(data):
        c = 0xFFFFFFFF
        for b in data:
            c ^= b
            for _ in range(8):
                c = (c >> 1) ^ (0xEDB88320 if c & 1 else 0)
        return c ^ 0xFFFFFFFF
    for b in (b"", b"a", b"123456789", bytes(range(256))):
        assert crc(b) == zlib.crc32(b)
    assert zlib.crc32(b"123456789") == 0xCBF43926
