"""CRC-32 cases shared by the emulation (test_crc32_emu.py) and the device tests (test_gpu_crc32.py), with
zlib.crc32 as the reference.  A case is a list of blocks laid out back to back after `lead` bytes of filler; its
expected CRCs are zlib.crc32 of each block."""
import zlib
from dataclasses import dataclass, field

import numpy as np

import redux_b200 as rb

LIB_PIECE = 65536          # kCrcPiece (redux_crc.cuh): bytes per warp item in the library
EMU_PIECE = 1536           # the emulation's piece: 3 x 512 bytes, so piece boundaries fall at odd places


@dataclass
class Case:
    name: str
    blocks: list
    lead: int = 0
    tags: set = field(default_factory=set)


def _rand(rng, n):
    return rng.integers(0, 256, n, dtype=np.uint8).tobytes()


def _around(p):
    return [p - 31, p - 17, p - 16, p - 1, p, p + 1, p + 15, p + 16, 2 * p - 1, 2 * p + 1]


def _build():
    rng = np.random.default_rng(20261022)
    gen = rb.generate_blocks_host(0, 8, 4096, 7)                       # two blocks of each generator class
    cases = [
        Case("lengths", [_rand(rng, n) for n in (0, 1, 2, 3, 15, 16, 17, 31, 4095, 4096, 4097)], tags={"lengths"}),
        Case("lengths_lead3", [_rand(rng, n) for n in (1, 2, 3, 4, 5, 15, 16, 17, 31, 4095, 4096, 4097)], lead=3),
        # block i starts at 17 * i (all 16 residues), and short blocks of odd lengths at every residue too
        Case("starts_mod16", [_rand(rng, 17) for _ in range(17)], tags={"starts"}),
        Case("starts_mod16_short", [_rand(rng, n) for n in [1] * 16 + [3] * 16 + [5] * 16 + [2] * 8], lead=1,
             tags={"starts"}),
        Case("empty_between", [b"", _rand(rng, 100), b"", b"", _rand(rng, 4097), b"", _rand(rng, 3), b""], lead=9,
             tags={"empty"}),
        Case("all_empty", [b""] * 5, tags={"empty"}),
        Case("constant", [bytes(1000), b"\xff" * 1000, bytes(70001), b"\xff" * 70001, bytes(5), b"\xff" * 3],
             lead=7, tags={"constant"}),
        Case("generator", [gen[i * 4096:(i + 1) * 4096].tobytes() for i in range(8)], lead=2, tags={"generator"}),
        Case("random_ragged", [_rand(rng, int(n)) for n in rng.integers(0, 20000, 40)], lead=11, tags={"random"}),
        Case("emu_piece_edges", [_rand(rng, n) for n in _around(EMU_PIECE)], lead=4, tags={"piece"}),
        Case("lib_piece_edges", [_rand(rng, n) for n in _around(LIB_PIECE)], lead=13, tags={"piece"}),
        Case("many_pieces", [_rand(rng, (1 << 20) + 7), _rand(rng, 5), _rand(rng, (4 << 20) + 7)], lead=5,
             tags={"many"}),
    ]
    return cases


CASES = _build()


def layout(case):
    """(data uint8, offsets uint64[n+1]) of the blocks back to back after case.lead filler bytes."""
    lens = [len(b) for b in case.blocks]
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    off[0] = case.lead
    off[1:] = case.lead + np.cumsum(np.array(lens, dtype=np.uint64))
    data = np.frombuffer(b"\xa5" * case.lead + b"".join(case.blocks), dtype=np.uint8)
    return data, off


def slots(case, spare=13):
    """(data, slot offsets uint64[n+1], lens uint64[n]): each block at the start of a slot `spare` bytes longer, the
    rest of the slot filler, as a device-resident decode leaves slots and their lengths."""
    parts, off, lens = [b"\x5a" * case.lead], [case.lead], []
    for b in case.blocks:
        parts.append(b + b"\xc3" * spare)
        off.append(off[-1] + len(b) + spare)
        lens.append(len(b))
    return (np.frombuffer(b"".join(parts), dtype=np.uint8), np.array(off, dtype=np.uint64),
            np.array(lens, dtype=np.uint64))


def expected(case):
    return np.array([zlib.crc32(b) for b in case.blocks], dtype=np.uint32)
