// crc_emu.cpp -- TEST INFRASTRUCTURE: crc32_blocks_kernel of redux_b200/csrc/redux_crc.cuh runs on the CPU.
// The table phases run thread by thread, each for all threads before the next, as the kernel's barriers order them;
// then every item's 32 lanes run one after another, their shifted values are XORed as the warp's shuffles XOR them,
// and lane 0's term is XORed into the block's word.  Built by tests/test_crc32_emu.py with g++; compared there
// against zlib.crc32.  Not part of the product.
#include "cuda_shim.h"

#include <vector>

thread_local EmuIdx threadIdx, blockIdx, blockDim, gridDim;

#include "../../redux_b200/csrc/redux_crc.cuh"

using namespace rdx;

namespace {

// The kernel of shape <R replicas, prefetch PF> item by item; mutant as emu_crc32.
template <uint32_t R, bool PF, bool DUAL = false>
void emu_run(const CrcJob &j, int mutant)
{
    std::vector<uint32_t> tab(1024 * R);
    for (uint32_t t = 0; t < 256; ++t) crc_fill_entries<R>(tab.data(), t, 256);
    for (uint32_t t = 0; t < 256; ++t) crc_fill_replicas<R>(tab.data(), t, 256);
    for (uint64_t it = 0; it < j.n_items; ++it) {
        CrcPiece pc;
        if (!crc_piece(j, it, &pc)) continue;
        if (mutant == 2 && pc.q) {
            // the piece starts a block of its own: the initial value's pattern over its first four bytes
            const uintptr_t first = pc.ep - (pc.q + 1) * j.piece;
            if (first > pc.a) { pc.a = first; pc.ps = first; pc.pat = 0xFFFFFFFFu; }
        }
        if (mutant == 3) pc.e += 1;
        uint32_t r = 0;
        for (uint32_t lane = 0; lane < 32; ++lane)
            r ^= crc_mulmod(crc_lane_shift(j.piece >> 5, lane),
                            crc_lane<R, PF, DUAL>(pc, j.piece, tab.data() + lane % R, lane));
        if (mutant == 3) pc.e -= 1;
        uint32_t term;
        if (mutant == 1) {
            CrcPiece p0 = pc;
            p0.q = 0;
            term = crc_piece_term(p0, j.piece, r) ^ (pc.q ? 0xFFFFFFFFu : 0u);
        } else {
            term = crc_piece_term(pc, j.piece, r);
            if (mutant == 2 && pc.q) term ^= 0xFFFFFFFFu;
        }
        j.crc[pc.block] ^= term;
    }
}

}  // namespace

extern "C" {

// What redux_crc32_blocks_device enqueues (crc_enqueue in redux_capi.cu) with `piece` bytes per item (0: the
// library's kCrcPiece).  lens: NULL, or the length of each block at in + in_off[i].  shape 0: the library's (CrcLib);
// 1: 16 replicas with prefetch; 2: 8 replicas; 3: one table with prefetch; 4: two chains per lane (the other shapes
// bench_crc32.py times).
// mutant 0: the kernel as it is; 1: pieces XORed without their shift x^(8 q piece); 2: the initial value and final
// XOR applied per piece instead of per block (each piece coded as if it started a block of its own); 3: the tail mask
// one byte too long (the byte after the block read as part of it).
void emu_crc32(const uint8_t *in, const uint64_t *in_off, const uint64_t *lens, uint64_t n_blocks,
               uint64_t max_block_len, uint32_t piece, uint32_t *crc, int mutant, int shape)
{
    CrcJob j;
    j.in = in; j.in_off = in_off; j.lens = lens; j.crc = crc; j.n_blocks = n_blocks;
    j.piece = piece ? piece : kCrcPiece;
    j.n_items = n_blocks * ((max_block_len + 30 + j.piece - 1) / j.piece);
    for (uint64_t i = 0; i < n_blocks; ++i) crc[i] = 0;
    if (!max_block_len) return;
    switch (shape) {
    case 0: emu_run<CrcLib::kReplicas, CrcLib::kPrefetch>(j, mutant); break;
    case 1: emu_run<16, true>(j, mutant); break;
    case 2: emu_run<8, false>(j, mutant); break;
    case 3: emu_run<1, true>(j, mutant); break;
    default: emu_run<32, false, true>(j, mutant); break;
    }
}

}  // extern "C"
