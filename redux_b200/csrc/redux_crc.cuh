// redux_crc.cuh -- CRC-32 of every block of a ragged batch (redux_crc32_blocks, DESIGN.md 3.11).
//
// The checksum is CRC-32/ISO-HDLC, the CRC of zlib.crc32 and crc32fast::hash: reflected polynomial 0xEDB88320,
// initial value and final XOR 0xFFFFFFFF.  Words below are in the reflected representation: bit 31 is the
// coefficient of x^0, and multiplying by x is a right shift with a conditional XOR of the polynomial.
//
// Algebra.  raw(M) is the register after M from a zero register (no initial value, no final XOR).  It is linear:
//     raw(A || B) = raw(A) * x^(8|B|) ^ raw(B)        (products mod P)
// and leading zero bytes do not change it.  The initial value is four message bytes: with n >= 4, complementing
// the first four bytes (XOR 0xFF each) adds 0xFFFFFFFF * x^(8n) to raw(M), exactly what the initial value adds.
// A block of n < 4 bytes gets the four bytes kCrcShortPattern[n] XORed over [e - 4, e) instead, the bytes before
// the block taken as zeros; they add the same term.  So crc32(M) = raw(M with the pattern) ^ 0xFFFFFFFF.
//
// Split.  A block's padded message runs over whole 16-byte vectors [vs, ep): vs is the vector of the pattern's
// first byte, ep = the block's end rounded up to 16.  Bytes outside the block read as zeros (those before it are
// leading zeros; the t = ep - e < 16 after it are undone at the end by kCrcUnshift[t] = x^(-8t)).  Pieces of
// `piece` bytes are counted back from ep: piece q is [ep - (q+1) * piece, ep - q * piece), so its shift to the end is
// x^(8 q piece) whatever the block's length, and a block of n bytes has ceil((ep - vs) / piece) pieces.  A warp codes
// one piece; lane l the l-th of its 32 segments of piece/32 bytes, whose shift to the end of the piece is the
// per-lane constant x^(8 * seg * (31 - l)).  The warp XORs the shifted lane values, lane 0 applies the piece's shift
// and, for piece 0, x^(-8t) and the final XOR, and merges the result into the block's word with atomicXor.  XOR is
// order-free, so the word is the same whatever order the pieces land in.
//
// Work split.  Item i of the grid is (block i % n_blocks, piece i / n_blocks): every block's piece 0 comes first, so
// the pieces that exist are spread over all warps and the items past a block's last piece, which return at once,
// gather at the end.  An empty block has no pieces; its word stays 0 = crc32 of no bytes.
//
// Tables.  Slice-by-4: T_k[v] = raw(byte v followed by k zero bytes), k = 0..3.  32 lanes looking up data-dependent
// entries of one table collide on shared-memory banks; every entry is stored R times, entry e of lane l at word
// e * R + l % R (DESIGN.md 3.2 does the same for the Fenwick tables), so with R = 32 a lane only ever reads its own
// bank.  CTAs are persistent over the items; CrcLib below is the shape the library launches.
//
// The phases are separate functions so that the CPU emulation of the tests under tests/ can run them lane by lane.
#pragma once
#include "redux_common.cuh"

namespace rdx {

// How a CTA runs the kernel: R replicas of the tables (lane l reads replica l % R: 32 / R lanes share a bank's worth
// of entries, so a lookup costs up to 32 / R wavefronts), THREADS threads, MINB CTAs per SM (the register budget
// follows: 65,536 / (THREADS x MINB) per thread), PF: each lane's next four vectors are loaded before the current
// four are folded, and DUAL: a lane folds the two halves of its segment as two independent register chains,
// interleaved, and joins them with one shift by the half's length.  scripts/bench_crc32.py times the shapes against
// each other (DESIGN.md 3.11); CrcLib is the one the library launches.
template <uint32_t R, uint32_t THREADS, uint32_t MINB, bool PF, bool DUAL = false>
struct CrcShape {
    static constexpr uint32_t kReplicas = R, kThreads = THREADS, kMinBlocks = MINB;
    static constexpr bool kPrefetch = PF, kDual = DUAL;
    static constexpr size_t kSmemBytes = (size_t)4 * 256 * R * sizeof(uint32_t);
};
using CrcLib = CrcShape<32, 1024, 1, true>;     // the fastest shape on every batch of DESIGN.md 3.11

constexpr uint32_t kCrcThreads = CrcLib::kThreads;
constexpr size_t kCrcSmemBytes = CrcLib::kSmemBytes;
constexpr uint32_t kCrcPiece = 65536;                   // bytes per warp item (the library's choice; CrcJob::piece)
constexpr uint32_t kCrcPoly = 0xEDB88320u;
constexpr uint32_t kCrcOne = 0x80000000u;               // x^0

#if defined(RDX_HOST_EMU)
#define RDX_CRC_TABLE static const
#else
#define RDX_CRC_TABLE __device__ const
#endif

// x^(2^k) mod P, k = 0..31 (x^(2^32) = x, so the table repeats with period 32)
RDX_CRC_TABLE uint32_t kCrcX2n[32] = {
    0x40000000, 0x20000000, 0x08000000, 0x00800000, 0x00008000, 0xedb88320, 0xb1e6b092, 0xa06a2517,
    0xed627dae, 0x88d14467, 0xd7bbfe6a, 0xec447f11, 0x8e7ea170, 0x6427800e, 0x4d47bae0, 0x09fe548f,
    0x83852d0f, 0x30362f1a, 0x7b5a9cc3, 0x31fec169, 0x9fec022a, 0x6c8dedc4, 0x15d6874d, 0x5fde7a4e,
    0xbad90e37, 0x2e4e5eef, 0x4eaba214, 0xa8a472c0, 0x429a969e, 0x148d302a, 0xc40ba6d0, 0xc4e22c3c};
// x^(-8t) mod P, t = 0..15: undoes the t zero bytes between a block's end and the next 16-byte boundary
RDX_CRC_TABLE uint32_t kCrcUnshift[16] = {
    0x80000000, 0x6567cb95, 0xd7125358, 0x1f81b6e1, 0x5b358fd3, 0xeb21cebf, 0x2ff880c5, 0x97fc423c,
    0x2e9bb40b, 0x2fb98a7d, 0xd6f6fa3c, 0x2059d4a0, 0x36511375, 0x525983aa, 0x31619cb3, 0x0f125cae};
// the four bytes (little-endian) whose raw CRC is 0xFFFFFFFF * x^(8n): the initial value of a block of n bytes,
// n = 0..4 (from n = 4 on it is 0xFFFFFFFF, XORed over the block's first four bytes)
RDX_CRC_TABLE uint32_t kCrcShortPattern[5] = {0x9226f562, 0xa32e2681, 0x9a1c9d90, 0xf0958fd9, 0xffffffff};

struct CrcJob {
    const uint8_t *in;
    const uint64_t *in_off;      // block i starts at in + in_off[i]
    const uint64_t *lens;        // NULL: block i ends at in + in_off[i+1]; else it has lens[i] bytes
    uint32_t *crc;               // n_blocks words, zero before the launch
    uint64_t n_blocks;
    uint64_t n_items;            // n_blocks x pieces of the longest block
    uint32_t piece;              // bytes per item, a multiple of 32 x 16
};

// a * b mod P
RDX_HD uint32_t crc_mulmod(uint32_t a, uint32_t b)
{
    uint32_t p = 0;
    for (int i = 0; i < 32; ++i) {
        p ^= b & (uint32_t)((int32_t)a >> 31);
        a <<= 1;
        b = (b >> 1) ^ (kCrcPoly & (uint32_t)((int32_t)(b << 31) >> 31));
    }
    return p;
}

// x^(n * 2^k) mod P: square-and-multiply over the bits of n
__device__ __forceinline__ uint32_t crc_x2n(uint64_t n, uint32_t k)
{
    uint32_t p = kCrcOne;
    for (; n; n >>= 1, ++k)
        if (n & 1) p = crc_mulmod(kCrcX2n[k & 31], p);
    return p;
}

// T_k[v] for entry i = k * 256 + v, bit by bit
RDX_HD uint32_t crc_table_entry(uint32_t i)
{
    uint32_t c = i & 255;
    for (uint32_t b = 0; b < 8 * ((i >> 8) + 1); ++b) c = (c >> 1) ^ (kCrcPoly & (0u - (c & 1)));
    return c;
}

// Phase 1: the 1,024 entries into replica 0 of their rows.  Phase 2: the other R - 1 replicas.
template <uint32_t R>
__device__ __forceinline__ void crc_fill_entries(uint32_t *tab, uint32_t tid, uint32_t threads)
{
    for (uint32_t i = tid; i < 1024; i += threads) tab[i * R] = crc_table_entry(i);
}
template <uint32_t R>
__device__ __forceinline__ void crc_fill_replicas(uint32_t *tab, uint32_t tid, uint32_t threads)
{
    for (uint32_t w = tid; w < 1024 * R; w += threads)
        if (w % R) tab[w] = tab[w - w % R];
}

// Lane l's segment shift to the end of its piece: x^(8 * seg * (31 - l)).
__device__ __forceinline__ uint32_t crc_lane_shift(uint32_t seg, uint32_t lane)
{
    return crc_x2n((uint64_t)seg * (31 - lane), 3);
}

// One 4-byte word through the slice-by-4 tables; `tab` is the lane's replica (table base + lane % R).
template <uint32_t R>
__device__ __forceinline__ uint32_t crc_word(const uint32_t *tab, uint32_t c, uint32_t w)
{
    c ^= w;
    return tab[(768 + (c & 255)) * R] ^ tab[(512 + ((c >> 8) & 255)) * R] ^ tab[(256 + ((c >> 16) & 255)) * R] ^
           tab[(c >> 24) * R];
}

template <uint32_t R>
__device__ __forceinline__ uint32_t crc_vec(const uint32_t *tab, uint32_t c, const uint4 &v)
{
    c = crc_word<R>(tab, c, v.x);
    c = crc_word<R>(tab, c, v.y);
    c = crc_word<R>(tab, c, v.z);
    return crc_word<R>(tab, c, v.w);
}

__device__ __forceinline__ uint4 crc_load(uintptr_t p)
{
    return __ldg(reinterpret_cast<const uint4 *>(p));
}

// The piece an item names.  False when the block has no such piece (uniform over the warp).
struct CrcPiece {
    uint64_t block, q;
    uintptr_t a, e;              // the block's bytes [a, e)
    uintptr_t ps;                // the initial-value pattern is XORed over [ps, ps + 4)
    uint32_t pat;
    uintptr_t vs, ep;            // the padded message [vs, ep), 16-byte aligned
};

__device__ __forceinline__ bool crc_piece(const CrcJob &j, uint64_t item, CrcPiece *pc)
{
    pc->block = item % j.n_blocks;
    pc->q = item / j.n_blocks;
    const uint64_t b = j.in_off[pc->block];
    const uint64_t n = j.lens ? j.lens[pc->block] : j.in_off[pc->block + 1] - b;
    if (n == 0) return false;
    pc->a = (uintptr_t)(j.in + b);
    pc->e = pc->a + n;
    pc->ps = n >= 4 ? pc->a : pc->e - 4;
    pc->pat = kCrcShortPattern[n >= 4 ? 4 : n];
    pc->vs = pc->ps & ~(uintptr_t)15;
    pc->ep = (pc->e + 15) & ~(uintptr_t)15;
    return pc->q * j.piece < pc->ep - pc->vs;
}

// A vector at the block's edges: loaded bytes inside [a, e), zeros outside, the pattern XORed over [ps, ps + 4).
__device__ __forceinline__ uint4 crc_edge(const CrcPiece &pc, uintptr_t p)
{
    uint4 v = make_uint4(0, 0, 0, 0);
    if (p + 16 > pc.a && p < pc.e) v = __ldg(reinterpret_cast<const uint4 *>(p));
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (uint32_t k = 0; k < 16; ++k) {
        const uintptr_t pos = p + k;
        uint32_t m = (pos >= pc.a && pos < pc.e) ? 0xFFu : 0u;
        uint32_t x = pos - pc.ps < 4 ? (pc.pat >> (8 * (uint32_t)(pos - pc.ps))) & 0xFF : 0u;
        w[k >> 2] = (w[k >> 2] & ~(0xFFu << (8 * (k & 3)))) |
                    ((((w[k >> 2] >> (8 * (k & 3))) & m) ^ x) << (8 * (k & 3)));
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// raw CRC of lane `lane`'s segment of the piece: [s1 - seg, s1) within the padded message, s1 = ep - q * piece -
// (31 - lane) * seg.  Vectors that hold no edge are loaded four at a time (PF: the next four before the current four
// are folded; DUAL: a whole edge-free segment, seg a multiple of 64, as two interleaved chains).
template <uint32_t R, bool PF, bool DUAL = false>
__device__ __forceinline__ uint32_t crc_lane(const CrcPiece &pc, uint32_t piece, const uint32_t *tab, uint32_t lane)
{
    const uint32_t seg = piece >> 5;
    const uint64_t back = pc.q * piece + (uint64_t)(31 - lane) * seg;    // bytes between the segment's end and ep
    if (back >= pc.ep - pc.vs) return 0;
    const uintptr_t s1 = pc.ep - back;
    uintptr_t p = s1 - (s1 - pc.vs < seg ? s1 - pc.vs : seg);
    const uintptr_t fast_lo = (pc.a + 4 + 15) & ~(uintptr_t)15;       // vectors in [fast_lo, fast_hi) have no edge
    const uintptr_t fast_hi = pc.e & ~(uintptr_t)15;
    const uintptr_t hi = s1 < fast_hi ? s1 : fast_hi;
    uint32_t c = 0;
    if (DUAL && seg % 64 == 0 && s1 - p == seg && p >= fast_lo && s1 <= fast_hi) {
        const uint32_t half = seg >> 1;
        uint32_t cb = 0;
        for (const uintptr_t mid = p + half; p < mid; p += 32) {
            const uint4 a0 = crc_load(p), a1 = crc_load(p + 16), b0 = crc_load(p + half), b1 = crc_load(p + half + 16);
            c = crc_vec<R>(tab, c, a0);
            cb = crc_vec<R>(tab, cb, b0);
            c = crc_vec<R>(tab, c, a1);
            cb = crc_vec<R>(tab, cb, b1);
        }
        return crc_mulmod(crc_x2n(half, 3), c) ^ cb;
    }
    for (; p < s1 && p < fast_lo; p += 16) c = crc_vec<R>(tab, c, crc_edge(pc, p));
    if (PF && p + 64 <= hi) {
        uint4 v0 = crc_load(p), v1 = crc_load(p + 16), v2 = crc_load(p + 32), v3 = crc_load(p + 48);
        for (; p + 128 <= hi; p += 64) {
            const uint4 n0 = crc_load(p + 64), n1 = crc_load(p + 80), n2 = crc_load(p + 96), n3 = crc_load(p + 112);
            c = crc_vec<R>(tab, c, v0);
            c = crc_vec<R>(tab, c, v1);
            c = crc_vec<R>(tab, c, v2);
            c = crc_vec<R>(tab, c, v3);
            v0 = n0; v1 = n1; v2 = n2; v3 = n3;
        }
        c = crc_vec<R>(tab, c, v0);
        c = crc_vec<R>(tab, c, v1);
        c = crc_vec<R>(tab, c, v2);
        c = crc_vec<R>(tab, c, v3);
        p += 64;
    }
    for (; p + 64 <= hi; p += 64) {
        const uint4 v0 = crc_load(p), v1 = crc_load(p + 16), v2 = crc_load(p + 32), v3 = crc_load(p + 48);
        c = crc_vec<R>(tab, c, v0);
        c = crc_vec<R>(tab, c, v1);
        c = crc_vec<R>(tab, c, v2);
        c = crc_vec<R>(tab, c, v3);
    }
    for (; p < hi; p += 16) c = crc_vec<R>(tab, c, crc_load(p));
    for (; p < s1; p += 16) c = crc_vec<R>(tab, c, crc_edge(pc, p));
    return c;
}

// Lane 0, after the warp's XOR of the shifted lane values r: the piece's term of the block's CRC.
__device__ __forceinline__ uint32_t crc_piece_term(const CrcPiece &pc, uint32_t piece, uint32_t r)
{
    if (pc.q) r = crc_mulmod(crc_x2n(pc.q * piece, 3), r);
    const uint32_t t = (uint32_t)(pc.ep - pc.e);
    if (t) r = crc_mulmod(kCrcUnshift[t], r);
    return pc.q ? r : r ^ 0xFFFFFFFFu;
}

#if !defined(RDX_HOST_EMU)
// The kernel body for shape S; tab: S::kSmemBytes of shared memory.
template <class S>
__device__ __forceinline__ void crc32_blocks_run(const CrcJob &j, uint32_t *tab)
{
    crc_fill_entries<S::kReplicas>(tab, threadIdx.x, S::kThreads);
    __syncthreads();
    crc_fill_replicas<S::kReplicas>(tab, threadIdx.x, S::kThreads);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t shift = crc_lane_shift(j.piece >> 5, lane);
    const uint64_t warps = (uint64_t)gridDim.x * (S::kThreads / 32);
    for (uint64_t it = (uint64_t)blockIdx.x * (S::kThreads / 32) + (threadIdx.x >> 5); it < j.n_items; it += warps) {
        CrcPiece pc;
        if (!crc_piece(j, it, &pc)) continue;
        const uint32_t raw = crc_lane<S::kReplicas, S::kPrefetch, S::kDual>(pc, j.piece, tab + lane % S::kReplicas,
                                                                              lane);
        uint32_t r = crc_mulmod(shift, raw);
#pragma unroll
        for (int o = 16; o; o >>= 1) r ^= __shfl_xor_sync(0xFFFFFFFFu, r, o);
        if (lane == 0) atomicXor(&j.crc[pc.block], crc_piece_term(pc, j.piece, r));
    }
}

__global__ void __launch_bounds__(CrcLib::kThreads, CrcLib::kMinBlocks) crc32_blocks_kernel(CrcJob j)
{
    extern __shared__ uint32_t crc_tab[];
    crc32_blocks_run<CrcLib>(j, crc_tab);
}
#endif

}  // namespace rdx
