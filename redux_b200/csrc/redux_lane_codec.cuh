// redux_lane_codec.cuh -- throughput mapping: ONE STREAM PER LANE, 32 independent streams per warp.
//
// The pieces every lane kernel shares (jobs, arithmetic class traits, table layout, bit and byte I/O) and the lane
// kernels of the HUGE class (code_bits > 32: 64-bit coder state).  The tuned lane kernels for code_bits <= 32 are in
// redux_lane_al.cuh.  What the reference does per stream on one CPU thread (src/codec.rs:55-176 over
// src/model/adaptive_tree.rs) runs here in every lane of every warp:
//   * the stream's Fenwick table lives in shared memory, LANE-INTERLEAVED so that lane l only ever
//     touches bank l: whatever nodes the 32 data-dependent walks visit, an access is one wavefront.
//     32-bit tables: node i of lane l is word i*32 + l.  16-bit tables: the word (i>>1)*32 + l holds
//     node i (even, low half) and node i+1 (odd, high half) of lane l;
//   * the table stores INCREMENTS only.  The reference initialises tree[i] = lowbit(i)
//     (adaptive_tree.rs:43-45) and a Fenwick prefix path decomposes i into its set bits, so
//     cum(i) = i + sum(increments on the path).  Node 256 (every data symbol's update ends there,
//     adaptive_tree.rs:86-89) equals the number of updates so far and node 257 (EOF) is constant 1:
//     neither is stored.  256 x u16 per stream = 512 B -> 14 warps (448 streams) per SM, which is
//     what lets 65,536 blocks be resident on 148 SMs in ONE wave (443 streams per SM);
//   * the encoder loads one node per tree level for the range query and the update together
//     (LaneTable2::query, redux_lane_al.cuh); the decoder descends four ways per round on 32-bit residuals
//     of the quotient value = X / range and increments the nodes where it turns left (LaneDecoder::run);
//   * count_t = min(257 + t, FMAX) depends on the position only (SURVEY.md A.5), so the two divisions
//     by count (src/codec.rs:59-60) are multiplications by a per-position 65-bit magic shared by all
//     streams, and the loop splits into an adaptive phase (t < FMAX-257) and a frozen phase (no updates,
//     constant reciprocal; the encoder rewrites its table as the cumulative array);
//   * renormalisation (src/codec.rs:62-89 / :140-158) is the closed form of redux_common.cuh;
//   * bits are packed into a 64-bit register and leave as whole big-endian 32-bit words
//     (MSB-first bytes, src/bitio/mod.rs:148-198) into the stream's private output slot; raw bytes
//     arrive as 16-byte vector loads prefetched one chunk ahead.
// No __syncthreads, no warp collectives: lanes are fully independent and may be ragged.
#pragma once
#include "redux_common.cuh"

namespace rdx {

constexpr int kLaneWarpsPerCta = 7;                 // 7 warps x 16 KiB tables; 2 CTAs per SM
constexpr int kLaneThreads = kLaneWarpsPerCta * 32;
constexpr int kTabNodes = 256;                      // nodes 0..255 (node 0 stays 0: the "absent" node)
// After the last warp's table: one 4-byte STAGING SLOT per thread (redux_lane_al.cuh, StageSlot).  The same bytes
// serve as the padded row the tuned kernels' unconditional load of the update path's "node 256" falls into
// (never stored).  2 x (7 x 16 KiB + 896 B + 1 KiB reserved per CTA) = 233,216 B of the SM's 233,472: two CTAs
// per SM, and not a byte to spare for a second slot.
// Before the slots: one ZERO ROW (128 B).  The frozen narrow decoder (redux_lane_al.cuh) reads entry 256 of its
// cumulative array as "the word after the table": for warps 0..5 that is row 0 of the next warp's table, whose low
// halfword is node 0 / C[0] = 0 in every phase, for the last warp it is this row.  With it the two CTAs fill the
// SM's 233,472 bytes exactly.
constexpr int kTabZeroRowBytes = 128;
constexpr int kTabPadBytes = kTabZeroRowBytes + kLaneThreads * 4;

struct LaneEncJob {
    const uint8_t *in;          // raw bytes
    const uint64_t *in_off;     // [n_blocks+1]
    uint64_t n_blocks;
    uint8_t *slots;             // n_blocks * slot_stride bytes, 16-byte aligned
    uint64_t slot_stride;
    uint32_t *sizes;            // [n_blocks] compressed bytes
    int32_t *status;            // [n_blocks]
    const void *magic;          // Magic32/Magic64 [magic_len], entry tt <-> count 257+tt
    uint32_t f, c;
    uint32_t tcap;              // FMAX - NSYM: number of model updates before the freeze
    uint32_t one;               // 1 << (32 - c) for c <= 32 (redux_lane_al.cuh), else 0
    // pre-trained start state (tuned kernels only): NULL / 257 / 1 for a fresh model
    const uint32_t *init_tree;  // tree[0..255] of the start model (adaptive_tree.rs layout), or NULL
    uint32_t count0;            // its total frequency; `magic` entry t <-> count0 + t, tcap = FMAX - count0
    uint32_t eof_freq;          // frequency of the EOF symbol: cum(256) = total - eof_freq
    // reciprocal of the frozen total FMAX (= magic[tcap]) as launch constants: the frozen loops read it from the
    // constant bank, so no in-loop instruction depends on a global load's scoreboard (tuned kernels only)
    uint64_t gf_m; uint32_t gf_sh;
};

struct LaneDecJob {
    const uint8_t *comp;
    const uint64_t *comp_off;   // [n_blocks+1]
    uint64_t n_blocks;
    uint8_t *raw;
    const uint64_t *raw_off;    // [n_blocks+1] slot offsets (capacities)
    uint64_t *raw_len;          // [n_blocks]
    uint64_t *consumed;         // [n_blocks]
    int32_t *status;
    const void *magic;
    uint32_t f, c;
    uint32_t tcap;
    uint32_t one;               // as in LaneEncJob
    const uint32_t *init_tree;  // as in LaneEncJob
    uint32_t count0, eof_freq;
    uint64_t gf_m; uint32_t gf_sh;   // as in LaneEncJob
};

// ------------------------------------------------------------------ arithmetic class traits
template <int CLS> struct Cls;
template <> struct Cls<kNarrow> {
    using S = uint32_t; using P = uint32_t; using M = Magic32;
    static __device__ __forceinline__ P mulr(uint32_t v, S rm1) { return v * rm1 + v; }   // v * range
    static __device__ __forceinline__ P mul_add(uint32_t v, S rm1, P acc) { return v * (rm1 + 1u) + acc; }
    static __device__ __forceinline__ P divc(P n, const M &g, uint32_t) { return div_magic32(n, g); }
    static __device__ __forceinline__ M ldm(const M *p) {
        uint2 v = __ldg(reinterpret_cast<const uint2 *>(p)); M g; g.m = v.x; g.sh = v.y; return g;
    }
    static __device__ __forceinline__ M mk(uint64_t m, uint32_t sh) { M g; g.m = (uint32_t)m; g.sh = sh; return g; }
};
template <> struct Cls<kWide> {
    using S = uint32_t; using P = uint64_t; using M = Magic64;
    static __device__ __forceinline__ P mulr(uint32_t v, S rm1) { return (uint64_t)v * rm1 + v; }
    static __device__ __forceinline__ P mul_add(uint32_t v, S rm1, P acc) { return (uint64_t)v * rm1 + (acc + v); }
    static __device__ __forceinline__ P divc(P n, const M &g, uint32_t) { return div_magic64(n, g); }
    static __device__ __forceinline__ M ldm(const M *p) {
        uint4 v = __ldg(reinterpret_cast<const uint4 *>(p));
        M g; g.m = ((uint64_t)v.y << 32) | v.x; g.sh = v.z; g.pad = 0; return g;
    }
    static __device__ __forceinline__ M mk(uint64_t m, uint32_t sh) { M g; g.m = m; g.sh = sh; g.pad = 0; return g; }
};
template <> struct Cls<kWideD> {
    using S = uint32_t; using P = uint64_t; using M = MagicD;
    static __device__ __forceinline__ P mulr(uint32_t v, S rm1) { return (uint64_t)v * rm1 + v; }
    static __device__ __forceinline__ P mul_add(uint32_t v, S rm1, P acc) { return (uint64_t)v * rm1 + (acc + v); }
    static __device__ __forceinline__ P divc(P n, const M &g, uint32_t) { return div_magicd(n, g); }
    static __device__ __forceinline__ M ldm(const M *p) { M g; g.r = __ldg(reinterpret_cast<const double *>(p)); return g; }
    static __device__ __forceinline__ M mk(uint64_t bits, uint32_t) {
        M g;
#if defined(__CUDA_ARCH__)
        g.r = __longlong_as_double((long long)bits);
#else
        union { double d; uint64_t u; } cv; cv.u = bits; g.r = cv.d;
#endif
        return g;
    }
};
template <> struct Cls<kHuge> {
    using S = uint64_t; using P = uint64_t; using M = Magic64;
    static __device__ __forceinline__ P mulr(uint32_t v, S rm1) { return (uint64_t)v * rm1 + v; }
    static __device__ __forceinline__ P mul_add(uint32_t v, S rm1, P acc) { return (uint64_t)v * (rm1 + 1u) + acc; }
    static __device__ __forceinline__ P divc(P n, const M &g, uint32_t) { return div_magic65(n, g); }
    static __device__ __forceinline__ M ldm(const M *p) {
        uint4 v = __ldg(reinterpret_cast<const uint4 *>(p));
        M g; g.m = ((uint64_t)v.y << 32) | v.x; g.sh = v.z; g.pad = 0; return g;
    }
    static __device__ __forceinline__ M mk(uint64_t m, uint32_t sh) { M g; g.m = m; g.sh = sh; g.pad = 0; return g; }
};

// ------------------------------------------------------------------ Fenwick increments in smem
// Indices below are in units of TW from the lane's base pointer.  A node row is 32 entries apart
// ("<< 5"); in the 16-bit layout an odd node n shares the word of even node n-1, i.e. sits at
// (n-1)*32 + 1 = n*32 - 31.
template <typename TW>
struct LaneTable {
    static constexpr int kOddAdj = (sizeof(TW) == 2) ? -31 : 0;
    static constexpr int kLaneMul = (sizeof(TW) == 2) ? 2 : 1;
    TW *t;   // table base of the warp + lane * kLaneMul

    __device__ __forceinline__ void init(void *smem, uint32_t warp, uint32_t lane) {
        t = reinterpret_cast<TW *>(smem) + (size_t)warp * kTabNodes * 32 + lane * kLaneMul;
    }
    __device__ __forceinline__ void clear() {
        // every word of the lane's column: 256 (u32) or 128 (u16 pairs) 32-bit words
        uint32_t *w = reinterpret_cast<uint32_t *>(t);
        constexpr int kWords = kTabNodes * (int)sizeof(TW) / 4;
#pragma unroll 8
        for (int i = 0; i < kWords; ++i) w[i * 32] = 0;
    }

    // index (in TW units from t) of node n, either parity
    static __device__ __forceinline__ int node_index(uint32_t n) { return (int)(n << 5) + ((n & 1u) ? kOddAdj : 0); }
};

// ------------------------------------------------------------------ bit packer (encoder output)
struct BitSink {
    uint64_t acc;      // newest bit at bit 0
    uint32_t nb;       // valid bits in acc, < 32 between calls
    uint32_t *w;       // next output word (slot is 16-byte aligned)
    uint32_t *w0;

    __device__ __forceinline__ void init(uint8_t *slot) { acc = 0; nb = 0; w = w0 = (uint32_t *)slot; }
    // append the low n (0..32) bits of v (v < 2^n)
    __device__ __forceinline__ void put(uint32_t v, uint32_t n) {
        acc = (acc << n) | v;
        nb += n;
        if (nb >= 32) {
            nb -= 32;
            *w++ = __byte_perm((uint32_t)(acc >> nb), 0, 0x0123);   // first bit -> MSB of first byte
        }
    }
    // x = n1 >= 1 code bits (MSB first); the first is followed by `pend` copies of its inverse
    // (put_bit, src/codec.rs:39-46).  With b = first bit: [b][pend x !b][rest] as one number is
    // x + 2^(n1+pend-1) - 2^(n1-1) for either value of b.
    __device__ __forceinline__ void put_code(uint64_t x, uint32_t n1, uint32_t pend) {
        const uint32_t n = n1 + pend;
        if (n <= 32) {
            put((uint32_t)x + (1u << (n - 1)) - (1u << (n1 - 1)), n);
        } else {
            const uint32_t b = (uint32_t)(x >> (n1 - 1)) & 1u;
            put(b, 1);
            while (pend > 0) {
                const uint32_t m = pend < 32 ? pend : 32;
                put(b ? 0u : (0xFFFFFFFFu >> (32 - m)), m);
                pend -= m;
            }
            uint32_t r = n1 - 1;                               // remaining bits of x
            if (r > 32) { put((uint32_t)(x >> 32) & (0xFFFFFFFFu >> (64 - r)), r - 32); r = 32; }
            if (r) put((uint32_t)x & (0xFFFFFFFFu >> (32 - r)), r);
        }
    }
    // flush_bits (src/bitio/mod.rs:183-198): left-align, zero-pad. Returns the byte count.
    __device__ __forceinline__ uint32_t finish() {
        const uint32_t bytes = (uint32_t)(w - w0) * 4 + (nb + 7) / 8;
        if (nb) *w = __byte_perm((uint32_t)(acc << (32 - nb)), 0, 0x0123);
        return bytes;
    }
};

// ------------------------------------------------------------------ byte source (encoder input)
// 16-byte aligned vector loads, one chunk prefetched ahead; bytes are shifted out of a word register.
struct ByteSource {
    const uint4 *p;         // next chunk to prefetch
    const uint4 *last;      // last chunk that may be read
    uint4 nxt;              // prefetched chunk
    uint32_t w, x, y, z;    // current word (already shifted) and the following words of the chunk
    uint32_t pos;           // byte position (chunk-relative phase in the low 4 bits)

    __device__ __forceinline__ void init(const uint8_t *src, uint32_t len) {
        const uintptr_t a = (uintptr_t)src;
        const uint4 *c0 = reinterpret_cast<const uint4 *>(a & ~(uintptr_t)15);
        pos = (uint32_t)(a & 15);
        last = reinterpret_cast<const uint4 *>((a + (len ? len - 1 : 0)) & ~(uintptr_t)15);
        uint4 q = make_uint4(0, 0, 0, 0);
        nxt = q;
        if (len) {
            q = __ldg(c0);
            nxt = __ldg(c0 < last ? c0 + 1 : last);
        }                                   // len == 0: next() is never called, nothing is loaded
        p = c0 + 2;
        const uint32_t ws = pos >> 2;
        w = ws == 0 ? q.x : ws == 1 ? q.y : ws == 2 ? q.z : q.w;
        x = ws == 0 ? q.y : ws == 1 ? q.z : q.w;
        y = ws == 0 ? q.z : q.w;
        z = q.w;
        w >>= 8 * (pos & 3);
    }
    __device__ __forceinline__ uint32_t next() {
        const uint32_t sym = w & 0xFFu;
        w >>= 8;
        ++pos;
        if ((pos & 3) == 0) {
            if ((pos & 15) == 0) {
                w = nxt.x; x = nxt.y; y = nxt.z; z = nxt.w;
                nxt = __ldg(p <= last ? p : last);   // past the end: re-read the last chunk, never consumed
                ++p;
            } else {
                w = x; x = y; y = z;
            }
        }
        return sym;
    }
};

// One coding step of the encoder (src/codec.rs:55-89): narrow the interval to [cl, ch) / count,
// renormalise in closed form, emit the settled bits.  Returns the number of shifts.
template <int CLS>
__device__ __forceinline__ uint32_t encode_step(typename Cls<CLS>::S &low, typename Cls<CLS>::S &high,
                                                uint32_t &pend, BitSink &sink, uint32_t cl, uint32_t ch,
                                                uint32_t count, const typename Cls<CLS>::M &g, uint32_t c)
{
    using C = Cls<CLS>;
    using S = typename C::S;
    using P = typename C::P;
    const S rm1 = high - low;                                      // range - 1  (:58)
    const P nh = C::mulr(ch, rm1), nl = C::mulr(cl, rm1);
    const S h2 = low + (S)C::divc(nh, g, count) - 1;               // :59
    const S l2 = low + (S)C::divc(nl, g, count);                   // :60
    const Renorm<S> r = renorm<S>(l2, h2, c);                      // :62-89
    if (r.n1) {
        sink.put_code((uint64_t)(l2 >> (c - r.n1)), r.n1, pend);
        pend = r.k;
    } else {
        pend += r.k;
    }
    low = r.low; high = r.high;
    return r.n1 + r.k;
}

template <typename TW, bool FULL> struct LaneTable2;       // redux_lane_al.cuh: one-walk query + update

// ------------------------------------------------------------------ encoder
// The library launches these kernels (encoder and decoder) with CLS = kHuge only; code_bits <= 32 runs the tuned
// kernels of redux_lane_al.cuh.  The bodies use nothing but the class traits, so CLS stays a parameter.
template <typename TW, int CLS>
__global__ void __launch_bounds__(kLaneThreads, 2)
encode_lane_kernel(const LaneEncJob job)
{
    using C = Cls<CLS>;
    using S = typename C::S;
    using M = typename C::M;
    extern __shared__ uint4 smem_u4[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t blk = (uint64_t)blockIdx.x * kLaneThreads + threadIdx.x;
    if (blk >= job.n_blocks) return;

    LaneTable2<TW, false> tab;                             // increments only, as LaneTable
    tab.init(smem_u4, warp, lane);
    tab.clear();

    const uint64_t off = job.in_off[blk];
    const uint32_t len = (uint32_t)(job.in_off[blk + 1] - off);
    const uint32_t c = job.c;
    const S maxv = (S)((c == sizeof(S) * 8) ? ~(S)0 : ((((S)1) << c) - 1));
    const M *magic = reinterpret_cast<const M *>(job.magic);
    const uint32_t tcap = job.tcap;

    ByteSource src;
    src.init(job.in + off, len);
    BitSink sink;
    sink.init(job.slots + blk * job.slot_stride);
    S low = 0, high = maxv;
    uint32_t pend = 0;

    // adaptive phase: the model still learns, count grows by one per symbol
    const uint32_t n_adapt = len < tcap ? len : tcap;
    uint32_t t = 0;
    M gn = C::ldm(magic);                                  // reciprocal of position t, loaded one ahead
    for (; t < n_adapt; ++t) {
        const M g = gn;
        gn = C::ldm(magic + t + 1);
        const uint32_t sym = src.next();
        uint32_t cl, ch;
        tab.template query<true>(sym, t, cl, ch);          // cum(256) - 256 = the number of updates so far
        encode_step<CLS>(low, high, pend, sink, cl, ch, kNsym + t, g, c);
    }
    // frozen phase (adaptive_tree.rs:84): total == FMAX, table and reciprocal are constant
    const uint32_t tt = n_adapt;                          // updates done = min(len, tcap)
    const M gf = gn;                                      // = magic[tt]
    const uint32_t countf = kNsym + tt;
    if (t < len) {
        tab.freeze_to_cumulative();
        // The lookup does not depend on the coder state (SURVEY.md A.7): fetch + look up symbol t+1 before
        // coding symbol t, so the shared-memory latency overlaps the range update of the previous symbol.
        uint32_t cl, ch;
        tab.query_frozen(src.next(), countf - 1u, cl, ch);   // cum(256) = total - 1
        for (; t + 1 < len; ++t) {
            const uint32_t cl_cur = cl, ch_cur = ch;
            tab.query_frozen(src.next(), countf - 1u, cl, ch);   // cum(256) = total - 1
            encode_step<CLS>(low, high, pend, sink, cl_cur, ch_cur, countf, gf, c);
        }
        encode_step<CLS>(low, high, pend, sink, cl, ch, countf, gf, c);
        ++t;
    }
    // EOF symbol: cum(256) = total - 1 (EOF's own frequency never grows), then the tail of
    // src/codec.rs:91-99: the remaining `extra` MSBs of low, then flush.
    const uint32_t shifts = encode_step<CLS>(low, high, pend, sink, countf - 1, countf, countf, gf, c);
    const uint32_t extra = c - shifts;
    if (extra) sink.put_code((uint64_t)(low >> (c - extra)), extra, pend);
    job.sizes[blk] = sink.finish();
    job.status[blk] = 0;
}

// ------------------------------------------------------------------ bit source (decoder input)
// Aligned 32-bit words, byte-swapped into a 64-bit bit buffer.  The word after the one being
// consumed is always already in flight (`nxt`), so a refill never waits on memory.
struct BitSource {
    uint64_t bb;            // bit buffer, valid bits are the low `bn`
    uint32_t bn;
    uint32_t nxt;           // prefetched next word, still in memory byte order (swapped when consumed,
                            // so that nothing depends on the load until the next refill)
    const uint32_t *w;      // word after nxt
    const uint32_t *wlast;  // last word that may be read
    uint32_t left;          // stream bits not yet consumed (streams are < 2^29 bytes here)
    uint32_t total;

    static __device__ __forceinline__ uint32_t swap(uint32_t x) { return __byte_perm(x, 0, 0x0123); }
    __device__ __forceinline__ void init(const uint8_t *src, uint32_t len) {
        const uintptr_t a = (uintptr_t)src;
        const uint32_t mis = (uint32_t)(a & 3);
        w = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
        wlast = w + ((mis + len + 3) >> 2) - 1;
        total = left = len * 8;
        bb = 0; bn = 0; nxt = 0;
        if (len) {
            bb = swap(__ldg(w)); bn = 32 - 8 * mis;
            nxt = __ldg(w + 1 <= wlast ? w + 1 : wlast);
        } else {
            wlast = w;                      // never dereferenced: has() fails before any take()
        }
        w += 2;
    }
    __device__ __forceinline__ bool has(uint32_t n) const { return n <= left; }
    __device__ __forceinline__ uint32_t used() const { return total - left; }
    // next n (0..32) bits, MSB first (src/bitio/mod.rs:78-120); caller checked has(n)
    __device__ __forceinline__ uint32_t take(uint32_t n) {
        if (bn < n) {
            bb = (bb << 32) | swap(nxt);
            bn += 32;
            nxt = __ldg(w <= wlast ? w : wlast);   // past the end: re-read the last word, never consumed
            ++w;
        }
        bn -= n;
        left -= n;
        const uint32_t mask = n ? (0xFFFFFFFFu >> (32 - n)) : 0u;
        return (uint32_t)(bb >> bn) & mask;
    }
    __device__ __forceinline__ uint64_t take64(uint32_t n) {   // n <= 64
        if (n <= 32) return take(n);
        uint64_t hi = take(n - 32);
        return (hi << 32) | take(32);
    }
};

// ------------------------------------------------------------------ byte sink (decoder output)
// Decoded symbols leave as aligned 32-bit words; the (possibly unaligned) head and tail of a
// block's slot are written byte-wise so neighbouring blocks are never touched.
struct ByteSink {
    uintptr_t dst, pw;      // slot start, current (aligned) word
    uint32_t wacc, sh;
    __device__ __forceinline__ void init(uint8_t *d) {
        dst = (uintptr_t)d; pw = dst & ~(uintptr_t)3; wacc = 0; sh = 8 * (uint32_t)(dst & 3);
    }
    __device__ __forceinline__ void store_bytes(uintptr_t from, uintptr_t to) const {
        for (uintptr_t p = from; p < to; ++p)
            *reinterpret_cast<uint8_t *>(p) = (uint8_t)(wacc >> (8 * (p & 3)));
    }
    __device__ __forceinline__ void put(uint32_t sym) {
        wacc |= sym << sh;
        sh += 8;
        if (sh == 32) {
            if (pw >= dst) *reinterpret_cast<uint32_t *>(pw) = wacc;
            else store_bytes(dst, pw + 4);
            pw += 4; wacc = 0; sh = 0;
        }
    }
    __device__ __forceinline__ void finish() const {
        if (sh) store_bytes(pw > dst ? pw : dst, pw + (sh >> 3));
    }
    // word-at-a-time interface (tuned decoder): valid once the position is word aligned, which also means the
    // slot's unaligned head is behind us
    __device__ __forceinline__ bool word_aligned() const { return sh == 0; }
    __device__ __forceinline__ void put_word(uint32_t wv) { *reinterpret_cast<uint32_t *>(pw) = wv; pw += 4; }
    __device__ __forceinline__ void partial(uint32_t wv, uint32_t nbytes) { wacc = wv; sh = 8 * nbytes; }   // finish() stores them
};

// ------------------------------------------------------------------ decoder
template <typename TW, int CLS>
struct LaneDecoder {
    using C = Cls<CLS>;
    using S = typename C::S;
    using P = typename C::P;
    using M = typename C::M;
    LaneTable<TW> tab;
    BitSource src;
    ByteSink out;
    S low, high, value, maxv;
    uint32_t c, t, cap;
    int32_t st;          // 0 running, -1 EOF symbol decoded (success), >0 error code

    // Decodes symbols while t < t_end.  ADAPT: the model still learns (count = 257 + t, one reciprocal
    // per position); otherwise the table is frozen at `count`.
    template <bool ADAPT>
    __device__ __forceinline__ void run(uint32_t t_end, const M *magic, uint32_t count_frozen, const M &g_frozen) {
        const S body = maxv >> 1, half = body + 1;
        M gn = ADAPT ? C::ldm(magic + t) : g_frozen;          // reciprocal of position t, loaded one ahead
        while (t < t_end) {
            const uint32_t count = ADAPT ? kNsym + t : count_frozen;
            const M g = gn;
            if (ADAPT) gn = C::ldm(magic + t + 1);
            // src/codec.rs:129-131 without the division: find i with cum(i)*range <= X < cum(i+1)*range,
            // X = (value-low+1)*count - 1.
            const S rm1 = high - low;
            const P X = C::mulr(count, (S)(value - low)) - 1;
            // step m = 256: node 256 = count-1 (adaptive_tree.rs:119-127 with the unstored node)
            const bool is_eof = X >= C::mulr(count - 1, rm1);
            // Quotient first, as the 64-bit-product class of redux_lane_al.cuh: the reference's
            // value = X / range (src/codec.rs:131) from a double estimate made exact by one remainder check
            // (div_by_range64), then the 4-ary descent on plain 32-bit values in the residual domain --
            // R = v - lo, N = v - hi < 0, each round's three sign bits move the position, unsigned min / max
            // pick the new bounds -- with the model update on the left turns.  Four dependent table round trips
            // of 32-bit adds instead of eight of 64-bit multiply-adds and 64-bit comparisons.  A step that ends
            // the stream afterwards (EOF symbol, bits ran out, sink full) leaves a table nobody reads again.
            const uint32_t v = div_by_range64((uint64_t)X, (uint64_t)rm1 + 1u);
            uint32_t R = v, N = v - (count - 1u);                 // node 256 = count - 1
            uint32_t I = 0;                                       // i * 32
#pragma unroll
            for (int m = 128; m >= 2; m >>= 2) {
                const int h = m >> 1;
                const int oddadj = (h == 1) ? LaneTable<TW>::kOddAdj : 0;      // nodes i+1, i+3 are odd
                const uint32_t ia = I + (uint32_t)(m << 5), ib = (uint32_t)((int)I + (h << 5) + oddadj),
                               ic = (uint32_t)((int)I + ((m + h) << 5) + oddadj);
                const uint32_t ar = tab.t[ia], br = tab.t[ib], cr = tab.t[ic];
                const uint32_t da = R - ((uint32_t)m + ar), db = R - ((uint32_t)h + br), dc = da - ((uint32_t)h + cr);
                const uint32_t ma = (uint32_t)((int32_t)da >> 31), mb = (uint32_t)((int32_t)db >> 31), mc = (uint32_t)((int32_t)dc >> 31);
                if (ADAPT) {                                      // + 1 where the descent turns left (node c: only after a right turn)
                    tab.t[ia] = (TW)(ar - ma);
                    tab.t[ib] = (TW)(br - mb);
                    tab.t[ic] = (TW)(cr - mc + ma);
                }
                const uint32_t r1 = da < dc ? da : dc, r2 = R < db ? R : db;
                const uint32_t n1 = da > dc ? da : dc, n2 = N > db ? N : db;
                R = r1 < r2 ? r1 : r2;
                N = n1 > n2 ? n1 : n2;
                I += (3u + ma + mb + mc) * (uint32_t)(h << 5);
            }
            const P plo = C::mulr(v - R, rm1), phi = C::mulr(v - N, rm1);
            if (is_eof) {                                         // src/codec.rs:136-138: no renorm, no reads
                st = -1;
                return;
            }
            const uint32_t sym = I >> 5;
            // src/codec.rs:133-134
            high = low + (S)C::divc(phi, g, count) - 1;
            low = low + (S)C::divc(plo, g, count);
            // src/codec.rs:140-158 in closed form
            const Renorm<S> r = renorm<S>(low, high, c);
            const uint32_t n = r.n1 + r.k;
            if (!src.has(n)) { st = 1; src.left = 0; return; }    // Err(Eof) inside get_bit
            if (t >= cap) { src.left -= n; st = 6; return; }      // sink full (the symbol's bits were read)
            const S chunk = (S)src.take64(n);
            S v1 = (r.n1 >= sizeof(S) * 8) ? (S)0 : (S)((value << r.n1) & maxv);
            v1 |= (S)(chunk >> r.k);
            value = (v1 & half) | ((S)(v1 << r.k) & body) | (chunk & (S)((((S)1) << r.k) - 1));
            low = r.low; high = r.high;
            out.put(sym);
            ++t;
        }
    }
};

template <typename TW, int CLS>
__global__ void __launch_bounds__(kLaneThreads, 2)
decode_lane_kernel(const LaneDecJob job)
{
    using D = LaneDecoder<TW, CLS>;
    using S = typename D::S;
    using M = typename D::M;
    extern __shared__ uint4 smem_u4[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t blk = (uint64_t)blockIdx.x * kLaneThreads + threadIdx.x;
    if (blk >= job.n_blocks) return;

    D d;
    d.tab.init(smem_u4, warp, lane);
    d.tab.clear();

    const uint64_t coff = job.comp_off[blk];
    const uint64_t clen = job.comp_off[blk + 1] - coff;
    const uint64_t roff = job.raw_off[blk];
    const uint64_t cap64 = job.raw_off[blk + 1] - roff;
    if (clen >= (1ull << 29)) {                 // 32-bit bit counters; such a stream is not lane work
        job.raw_len[blk] = 0; job.consumed[blk] = 0; job.status[blk] = 5;
        return;
    }
    d.c = job.c;
    d.maxv = (S)((d.c == sizeof(S) * 8) ? ~(S)0 : ((((S)1) << d.c) - 1));
    d.cap = cap64 > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)cap64;
    d.src.init(job.comp + coff, (uint32_t)clen);
    d.out.init(job.raw + roff);
    d.st = 0; d.t = 0;
    d.low = 0; d.high = d.maxv; d.value = 0;
    const M *magic = reinterpret_cast<const M *>(job.magic);
    const uint32_t tcap = job.tcap;

    // src/codec.rs:124-127: prime code_bits bits
    if (!d.src.has(d.c)) { d.st = 1; d.src.left = 0; }
    else d.value = (S)d.src.take64(d.c);

    const M g0 = D::C::ldm(magic);
    if (d.st == 0) d.template run<true>(tcap, magic, 0, g0);
    if (d.st == 0) {
        const M gf = D::C::ldm(magic + tcap);
        d.template run<false>(0xFFFFFFFFu, magic, kNsym + tcap, gf);
    }
    d.out.finish();
    job.raw_len[blk] = d.t;
    job.consumed[blk] = (d.src.used() + 7) >> 3;
    job.status[blk] = d.st < 0 ? 0 : d.st;
}

}  // namespace rdx
