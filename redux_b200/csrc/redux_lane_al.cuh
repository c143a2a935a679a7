// redux_lane_al.cuh -- the tuned lane kernels for code_bits <= 32 (32-bit coder state): one stream per
// lane exactly as in redux_lane_codec.cuh (same table layout, same jobs, same bytes), with the
// instruction count per symbol cut where profiles/r01_final_* showed the issue slots going:
//   * LEFT-ALIGNED coder state.  low/high (src/codec.rs:11-24) live in the top c bits of a 32-bit
//     register (high's spare low bits are ones, low's zeros).  The closed-form renormalisation of
//     src/codec.rs:62-89 then needs no code_bits arithmetic at all: n1 = clz(low ^ high) and the total
//     n1 + k = clz((low ^ high) & ~((low & ~high) << 1)) are one FLO.SH each, side by side (renorm_counts;
//     bfind.shiftamt; neither operand can be zero because of the spare bits), the settled bits are the top
//     n1 bits of low (one funnel shift) and high refills with ones through a funnel shift;
//   * the decoder's code value (src/codec.rs:124-158) is a 32-bit WINDOW into the compressed stream whose
//     top c bits are the value and whose low bits are look-ahead; E1/E2 shifts are a funnel shift that
//     pulls the following stream bits in, E3 shifts keep the MSB and drop the bits below it -- 4
//     instructions instead of extracting n bits and merging them;
//   * branch-free pending-bit emission (put_bit, src/codec.rs:39-46) and a word-indexed packer that takes
//     two symbols per append (BitSink2::put_pair);
//   * the adaptive encoder loads ONE Fenwick node per tree level, which serves the range query where the
//     symbol's bit is set and the update where it is clear (adaptive_tree.rs:63-92; LaneTable2::query);
//   * the decoder descends four ways per round on the sign bits of residuals -- no predicates -- and, once the
//     model is frozen, on the absolute boundaries of the cumulative array (LaneDecoderAl::step);
//   * FULL tables (whenever the entry type can hold them): nodes store the reference's actual tree
//     values (adaptive_tree.rs:43-45 initialises tree[i] = lowbit(i)) instead of increments, so neither
//     the query nor the decoder's descent adds the implicit lowbit terms back.
// Bit-exactness against the oracle is checked on the CPU by the emulation tests under tests/ (these kernels
// compiled with g++ through a shim) and on the device by tests/test_gpu_parity.py.
#pragma once
#include "redux_common.cuh"
#include "redux_lane_codec.cuh"

namespace rdx {

// Pins a launch constant in a register.  ptxas re-reads kernel parameters from the constant bank at every use (one
// LDCU per use and per symbol step in the encoder's loops); adding a zero it cannot know to be zero -- the top bit
// of a block offset loaded from memory -- makes the value a computed one that lives in a register.
__device__ __forceinline__ uint32_t pinned(uint32_t x, uint64_t loaded_offset) { return x + (uint32_t)(loaded_offset >> 63); }
__device__ __forceinline__ uint64_t pinned(uint64_t x, uint64_t loaded_offset) { return x + (loaded_offset >> 63); }

// count-leading-zeros of a NON-ZERO word as one instruction (FLO.U32.SH)
__device__ __forceinline__ uint32_t clz_nz(uint32_t x) {
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("bfind.shiftamt.u32 %0, %1;" : "=r"(r) : "r"(x));
    return r;
#else
    return (uint32_t)__builtin_clz(x);
#endif
}

// clz that may see zero as one instruction: FLO.SH answers 0xFFFFFFFF for 0, which every CLAMPED shift
// below treats like 32
__device__ __forceinline__ uint32_t clz_sh(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return clz_nz(x);
#else
    return x ? (uint32_t)__builtin_clz(x) : 0xFFFFFFFFu;
#endif
}
// x << n and "the top n bits of x" with n up to 32 (and beyond: clamped), one SHF each
__device__ __forceinline__ uint32_t shl_c(uint32_t x, uint32_t n) { return __funnelshift_lc(0u, x, n); }
__device__ __forceinline__ uint32_t top_bits(uint32_t x, uint32_t n) { return __funnelshift_lc(x, 0u, n); }
// leading bits low and high share (E1/E2 count).  C32: code_bits == 32 leaves no spare low bits, so the
// XOR can be zero (interval collapsed to one value) and the count must come out as exactly 32.
template <bool C32>
__device__ __forceinline__ uint32_t common_prefix(uint32_t x) { return C32 ? (uint32_t)clz32(x) : clz_nz(x); }

__device__ __forceinline__ uint32_t umin32(uint32_t a, uint32_t b) { return a < b ? a : b; }
__device__ __forceinline__ uint32_t umax32(uint32_t a, uint32_t b) { return a > b ? a : b; }

// Keeps the descent's position in ONE register chain: without it the compiler re-associates the position into
// two induction chains, one scaled for the table addresses and one for the symbol (two more instructions a round).
__device__ __forceinline__ void pin_chain(uint32_t &x) {
#if defined(__CUDA_ARCH__)
    asm volatile("" : "+r"(x));
#else
    (void)x;
#endif
}

// Shift counts of one symbol's renormalisation (src/codec.rs:62-89) from the left-aligned l2 = low', nh2 = ~high':
// n1 = E1/E2 shifts = length of the common prefix of low' and high', n = n1 + the E3 shifts.  After the common
// prefix low' has a 0 and high' a 1; the E3 shifts are the run of positions after that one where low' has 1 and
// high' has 0, i.e. the run of ones of d = l2 & nh2 that starts at position n1 + 1 (d is zero up to position n1).
// Shifted up by one that run continues the common prefix seamlessly: (equal bits) | (d << 1) has exactly n leading
// ones -- position n1 + k is inside or right behind the run, where the bits differ and d << 1 has its first zero.
// So n needs ONE count-leading-zeros on the chain (round 1 counted n1, shifted by it and counted again: two FLOs
// of 18 cycles each in series on every symbol of every stream); n1 is counted beside it, off the low/high chain.
// The operand of the second count can only be zero when low' == high' in all 32 bits (C32).
template <bool C32>
__device__ __forceinline__ void renorm_counts(uint32_t l2, uint32_t nh2, uint32_t &n1, uint32_t &n)
{
    const uint32_t differ = ~(l2 ^ nh2);                           // low' ^ high'
    n1 = common_prefix<C32>(differ);
    n = common_prefix<C32>(differ & ~((l2 & nh2) << 1));
}

// ------------------------------------------------------------------ Fenwick table, v2 access paths
// Same lane-interleaved storage as LaneTable<TW>.  FULL: node i holds the reference's tree[i]
// (lowbit(i) + increments); otherwise increments only (u16 entries that must survive 65,536 updates).
template <typename TW, bool FULL>
struct LaneTable2 : LaneTable<TW> {
    using B = LaneTable<TW>;
    using B::t;
    // The lane's column as (CTA's shared-memory base, byte offset of the column in it).  The offset is
    // warp * slab + lane * 4: bits 7 and up of the slab-relative part are zero, exactly where the row of a node goes
    // (a row = 32 lanes x 4 bytes), so `row bits | column offset` needs no addition and the shared-memory base
    // stays in the instruction's uniform operand.
    uint8_t *smem0;
    uint32_t col;
    __device__ __forceinline__ void init(void *smem, uint32_t warp, uint32_t lane) {
        B::init(smem, warp, lane);
        smem0 = reinterpret_cast<uint8_t *>(smem);
        col = warp * (uint32_t)(kTabNodes * 32 * sizeof(TW)) + lane * 4u;
#if defined(__CUDA_ARCH__)
        // opaque: knowing that the bits are disjoint the compiler turns the OR back into an addition and folds the
        // shared-memory base into it -- two instructions per access again
        asm volatile("" : "+r"(col));
#endif
    }

    // init_tree != NULL: start from a model the caller trained (FULL tables only); tree[0..255] as u32
    __device__ __forceinline__ void reset(const uint32_t *init_tree = nullptr) {
        uint32_t *w = reinterpret_cast<uint32_t *>(t);
        constexpr int kWords = kTabNodes * (int)sizeof(TW) / 4;
        if (FULL && init_tree) {
            if (sizeof(TW) == 2) {
#pragma unroll 4
                for (int m = 0; m < kWords; ++m) w[m * 32] = __ldg(init_tree + 2 * m) | (__ldg(init_tree + 2 * m + 1) << 16);
            } else {
#pragma unroll 4
                for (int i = 0; i < kWords; ++i) w[i * 32] = __ldg(init_tree + i);
            }
        } else if (!FULL) {
#pragma unroll 8
            for (int i = 0; i < kWords; ++i) w[i * 32] = 0;
        } else if (sizeof(TW) == 2) {
            // word m = nodes (2m, 2m+1): lowbit(2m) = 2*lowbit(m) (node 0 stays 0), lowbit(2m+1) = 1
#pragma unroll 8
            for (int m = 0; m < kWords; ++m) w[m * 32] = (uint32_t)(2 * (m & -m)) | (1u << 16);
        } else {
#pragma unroll 8
            for (int i = 0; i < kWords; ++i) w[i * 32] = (uint32_t)(i & -i);
        }
    }

    // Byte-addressed access for the decoder's descent.  A position is the shared-window byte address of a node of
    // this lane's column (host emulation: the byte offset from the column's start), so a table load is
    // [position + constant] with nothing to add per access -- the descent's position chain carries the address
    // itself.
    static constexpr int kNodeBytes = 32 * (int)sizeof(TW);               // table index (i << 5) in bytes: i * kNodeBytes
    __device__ __forceinline__ uint32_t pos0() const {
#if defined(__CUDA_ARCH__)
        return (uint32_t)__cvta_generic_to_shared(t);
#else
        return 0u;
#endif
    }
    __device__ __forceinline__ uint32_t ld_at(uint32_t a) const {
#if defined(__CUDA_ARCH__)
        uint32_t v;                                           // a 32-bit destination of a 16-bit load is zero-extended
        if (sizeof(TW) == 2) asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
        else asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
        return v;
#else
        return *reinterpret_cast<const TW *>(reinterpret_cast<const uint8_t *>(t) + a);
#endif
    }
    __device__ __forceinline__ void st_at(uint32_t a, uint32_t v) {
#if defined(__CUDA_ARCH__)
        // a 32-bit source of a 16-bit store is truncated: no conversion instruction
        if (sizeof(TW) == 2) asm volatile("st.shared.u16 [%0], %1;" :: "r"(a), "r"(v) : "memory");
        else asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory");
#else
        *reinterpret_cast<TW *>(reinterpret_cast<uint8_t *>(t) + a) = (TW)v;
#endif
    }

    // (cum(s), cum(s+1)) of adaptive_tree.rs:63-80 and, when UPDATE, update(s+1) of :83-92, sharing the
    // node addresses.  `cum256` = cum(256) = total - frequency of EOF (the unstored node 256; for a fresh model
    // 256 + the number of updates so far); with increments-only tables (!FULL) the caller passes it minus 256.
    // One node per tree level serves the range query AND the update.  The descent to s (adaptive_tree.rs:119-127)
    // stands, at level k = 7..0, on node n_k = (s & (0xFF << (k+1))) + 2^k.  Where bit k of s is set it turns right:
    // n_k = s & (0xFF << k) is a node of the prefix path of s (get_frequency_range, :63-80).  Where the bit is clear
    // it turns left: n_k = (s | (2^k - 1)) + 1 is a node of the update path of s + 1 (:83-92).  cum(s + 1) walks the
    // same nodes with the bits of s + 1: above the lowest clear bit k* of s the bits (and nodes) agree, bit k* is set
    // and its node (s + 1) & (0xFF << k*) is n_k* again, the bits below are clear.  So eight loads -- round 1 loaded
    // sixteen, a query node and an update node per level, of which one was masked off -- give both sums and the
    // values to increment; with u16 entries both sums accumulate in one register (low half cum(s), high half
    // cum(s+1): neither can carry, a cumulative value is at most 65,535 here).
    template <bool UPDATE>
    __device__ __forceinline__ void query(uint32_t s, uint32_t cum256, uint32_t &cl, uint32_t &ch) {
        const uint32_t z = s | ((s + 1u) << 16);               // bits of s and of s + 1, 16 apart
        TW *a[8];
        uint32_t v[8];
        // byte offset of node n_k in the CTA's shared memory: (row of the even node below it | column) + a constant
        constexpr uint32_t NB = 32u * (uint32_t)sizeof(TW);    // bytes from node i to node i + 1
        const uint32_t SB = s * NB;
        a[0] = reinterpret_cast<TW *>(smem0 + (((SB & (0xFEu * NB)) | col) + (sizeof(TW) == 2 ? 2u : NB)));   // the odd node of s's pair
#pragma unroll
        for (int k = 1; k < 8; ++k)
            a[k] = reinterpret_cast<TW *>(smem0 + (((SB & (((0xFFu << (k + 1)) & 0xFFu) * NB)) | col) + (NB << k)));
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = *a[k];
        uint32_t lo, hi;
        if (sizeof(TW) == 2) {
            uint32_t acc = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) acc += v[k] * ((z >> k) & 0x00010001u);
            lo = acc & 0xFFFFu; hi = acc >> 16;
        } else {                                               // (predicated adds for u16 too: measured +30 instructions)
            lo = 0; hi = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                if (z & (1u << k)) lo += v[k];
                if (z & (0x10000u << k)) hi += v[k];
            }
        }
        cl = lo + (FULL ? 0u : s);
        ch = (s == 255u ? cum256 : hi) + (FULL ? 0u : s + 1u);
        if (UPDATE) {
            // all loads before all stores: the nodes are distinct, which the compiler cannot know
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (!(s & (1u << k))) *a[k] = (TW)(v[k] + 1u);
        }
    }

    // update(s+1) alone (decoder: the search already produced the range)
    __device__ __forceinline__ void update(uint32_t s) {
        const uint32_t S = s << 5;
        const uint32_t q = ~s & 255u;
        const uint32_t levels = q ^ __funnelshift_rc(0x80000000u, 0u, clz_sh(q));
        TW *p0 = t + B::node_index((s + 1u) & 255u);
        TW *a[8];
        uint32_t u[8];
        const uint32_t u0 = *p0;
#pragma unroll
        for (int k = 1; k < 8; ++k) {
            a[k] = t + (S & (0x1FE0u << k)) + (32 << k);
            u[k] = *a[k];                                      // unconditional, see query<>
        }
        if (q) *p0 = (TW)(u0 + 1u);
#pragma unroll
        for (int k = 1; k < 8; ++k)
            if (levels & (1u << (k - 1))) *a[k] = (TW)(u[k] + 1u);
    }

    // Frozen model (adaptive_tree.rs:84): rewrite the tree in place as the cumulative array of
    // AdaptiveLinearModel (adaptive_linear.rs:26-28): C[i] = cum(i) (FULL) or cum(i) - i.  Descending i
    // only reads nodes <= i, which are still tree nodes.
    __device__ __forceinline__ void freeze_to_cumulative() {
        for (uint32_t i = 255; i >= 1; --i) {
            uint32_t sum = 0;
            for (uint32_t x = i; x; x &= x - 1) sum += t[B::node_index(x)];
            t[B::node_index(i)] = (TW)sum;
        }
    }
    __device__ __forceinline__ void query_frozen(uint32_t s, uint32_t cum256, uint32_t &cl, uint32_t &ch) const {
        uint32_t lo, hi;
        if (sizeof(TW) == 2) {
            // C[s] sits at byte (s >> 1) * 128 + (s & 1) * 2 of the lane's column; C[s+1] two bytes further for an
            // even s, in the next word row (126 bytes further) for an odd one.  For s = 255 that is the padded row
            // after the table: loaded, never used.
            // (row of the pair | column) + the halfword, from the CTA's shared-memory base (see `col`)
            const uint32_t odd = s & 1u;
            const uint8_t *pb = smem0 + ((((s << 6) & 0x3F80u) | col) + (odd << 1));
            lo = *reinterpret_cast<const uint16_t *>(pb);
            hi = *reinterpret_cast<const uint16_t *>(pb + odd * 124u + 2u);
        } else {
            lo = t[s << 5];
            hi = t[((s + 1) & 255u) << 5];
        }
        cl = lo + (FULL ? 0u : s);
        ch = (s == 255u) ? cum256 : hi + (FULL ? 0u : s + 1u);
    }
};

// ------------------------------------------------------------------ bit packer, word-indexed
struct BitSink2 {
    uint64_t acc;      // newest bit at bit 0
    uint32_t nb;       // valid bits in acc, < 32 between calls
    uint32_t wi;       // next output word
    uint32_t *w0;      // slot (16-byte aligned)

    __device__ __forceinline__ void init(uint8_t *slot) { acc = 0; nb = 0; wi = 0; w0 = (uint32_t *)slot; }
    __device__ __forceinline__ void put(uint32_t v, uint32_t n) {          // n <= 32, v < 2^n
        acc = (acc << n) | v;
        nb += n;
        if (nb >= 32) {
            nb -= 32;
            w0[wi++] = __byte_perm((uint32_t)(acc >> nb), 0, 0x0123);      // first bit -> MSB of first byte
        }
    }
    // put_bit semantics (src/codec.rs:39-46) for one symbol: `bits` = the n1 settled bits (MSB first),
    // the first followed by `pend` copies of its inverse; k = this symbol's E3 shifts.  Returns the new
    // pending count.  [b][pend x !b][rest] as one number is bits + 2^(n1+pend-1) - 2^(n1-1) for either b;
    // with n1 == 0 nothing is emitted and the pending run grows.
    __device__ __forceinline__ uint32_t put_code(uint32_t bits, uint32_t n1, uint32_t pend, uint32_t k) {
        const bool emit = n1 != 0;
        const uint32_t n = emit ? n1 + pend : 0u;
        if (__builtin_expect(n > 32, 0)) {                                  // rare: long E3 run
            const uint32_t b = (bits >> (n1 - 1)) & 1u;
            put(b, 1);
            while (pend > 0) {
                const uint32_t m = pend < 32 ? pend : 32;
                put(b ? 0u : (0xFFFFFFFFu >> (32 - m)), m);
                pend -= m;
            }
            if (n1 > 1) put(bits & (0xFFFFFFFFu >> (33 - n1)), n1 - 1);
        } else {
            // 2^(x-1) with x = 0 -> 0: clamped funnel shift of (1:0)
            put(bits + __funnelshift_lc(0u, 1u, n - 1u) - __funnelshift_lc(0u, 1u, n1 - 1u), n);
        }
        return (emit ? 0u : pend) + k;
    }
    // Two symbols' codes through ONE append.  Symbol A emits nA = n1A + pend bits (or none), symbol B nB bits after
    // it; while nA + nB <= 32 -- nearly always: a symbol settles about as many bits as its information content -- they
    // are one number, (VA << nB) | VB, and the accumulator shift, the word-boundary test and the predicated store
    // sequence run once for the pair instead of once per symbol.  Otherwise (a long pending run, two very rare symbols
    // in a row) the two codes take the one-symbol path in order.  Returns the new pending count.
    struct Code { uint32_t bits, n1, k; };
    __device__ __forceinline__ uint32_t put_pair(const Code &A, const Code &B, uint32_t pend) {
        const bool ea = A.n1 != 0;
        const uint32_t na = ea ? A.n1 + pend : 0u;
        const uint32_t pend1 = (ea ? 0u : pend) + A.k;
        const bool eb = B.n1 != 0;
        const uint32_t nb2 = eb ? B.n1 + pend1 : 0u;
        if (__builtin_expect(na + nb2 > 32, 0)) {
            (void)put_code(A.bits, A.n1, pend, A.k);
            return put_code(B.bits, B.n1, pend1, B.k);
        }
        const uint32_t va = A.bits + __funnelshift_lc(0u, 1u, na - 1u) - __funnelshift_lc(0u, 1u, A.n1 - 1u);
        const uint32_t vb = B.bits + __funnelshift_lc(0u, 1u, nb2 - 1u) - __funnelshift_lc(0u, 1u, B.n1 - 1u);
        put(shl_c(va, nb2) | vb, na + nb2);
        return (eb ? 0u : pend1) + B.k;
    }
    __device__ __forceinline__ uint32_t finish() {                          // flush_bits (src/bitio/mod.rs:183-198)
        const uint32_t bytes = wi * 4 + (nb + 7) / 8;
        if (nb) w0[wi] = __byte_perm((uint32_t)(acc << (32 - nb)), 0, 0x0123);
        return bytes;
    }
};

// ------------------------------------------------------------------ staging slot (global -> shared, asynchronous)
// Every stream's next input word travels through a private 4-byte shared-memory slot filled by cp.async
// (LDGSTS) instead of through a register filled by LDG.  Why: ptxas puts every in-loop LDG on ONE scoreboard,
// and a scoreboard is a counter -- waiting for the oldest load waits for the youngest too.  Lanes refill at
// different symbols, so in round 1 some lane's one-step-old load was always outstanding when another lane
// consumed its own, older word: 10-16 % of both coders' time sat on that scoreboard
// (profiles/r01_final5_ncu_full_summary.md; the SASS with its wait masks: scripts/sass_ctl.py).  cp.async groups
// are waited for with a DEPTH (cp.async.wait_group N leaves the N youngest groups in flight), which is
// exactly the partial wait the register path cannot express, and the in-loop code no longer contains a
// single LDG whose scoreboard an unrelated instruction could be made to wait on.
struct StageSlot {
#if defined(__CUDA_ARCH__)
    uint32_t sa;                                            // shared-window address of this thread's slot
    __device__ __forceinline__ void init(void *slot) { sa = (uint32_t)__cvta_generic_to_shared(slot); }
    __device__ __forceinline__ void request(const uint32_t *g) const {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(sa), "l"(g));
    }
    __device__ __forceinline__ uint32_t read() const {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(sa));
        return v;
    }
    static __device__ __forceinline__ void commit() { asm volatile("cp.async.commit_group;"); }
    template <int KEEP> static __device__ __forceinline__ void wait() { asm volatile("cp.async.wait_group %0;" :: "n"(KEEP)); }
#else
    uint32_t val;                                           // host emulation: the copy completes at once
    void init(void *) { val = 0; }
    void request(const uint32_t *g) { val = *g; }
    uint32_t read() const { return val; }
    static void commit() {}
    template <int KEEP> static void wait() {}
#endif
};

// this thread's slot: the CTA's slots follow its kLaneWarpsPerCta tables (kTabPadBytes)
template <typename TW>
__device__ __forceinline__ void *lane_stage_slot(void *smem) {
    return reinterpret_cast<uint8_t *>(smem) + (size_t)kLaneWarpsPerCta * kTabNodes * 32 * sizeof(TW) + kTabZeroRowBytes + threadIdx.x * 4;
}

// ------------------------------------------------------------------ byte source (encoder input), v3
// Aligned 32-bit words: `cur` holds the word at the position (already shifted), the word after it is in the
// staging slot or on its way there.  Every lane consumes exactly one word per four symbols, so the main
// loop's refill -- wait for the slot, read it, request the next word -- comes once per word and always finds
// a copy that was issued four symbol steps (> 1,000 cycles) earlier.
struct ByteSource3 {
    const uint32_t *base;   // 4-byte aligned start of the stream's first word
    uint32_t wi, wlast;     // next word to request / last word that may be read
    uint32_t cur;
    uint32_t pos;           // byte position (word-relative phase in the low 2 bits)
    StageSlot slot;

    __device__ __forceinline__ void request() {
        slot.request(base + (wi < wlast ? wi : wlast));     // past the end: re-read, never consumed
        ++wi;
    }
    __device__ __forceinline__ void init(const uint8_t *src, uint32_t len, void *slot_mem) {
        const uintptr_t a = (uintptr_t)src;
        base = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
        pos = (uint32_t)(a & 3);
        wlast = len ? (pos + len - 1) >> 2 : 0;
        wi = 1;
        cur = 0;
        slot.init(slot_mem);
        if (len) {                          // len == 0: next() is never called, nothing is loaded
            cur = __ldg(base) >> (8 * pos);
            request();
            StageSlot::commit();
        }
    }
    __device__ __forceinline__ void refill() {              // pos just reached a word boundary
        StageSlot::wait<0>();
        cur = slot.read();
        request();
        StageSlot::commit();
    }
    __device__ __forceinline__ uint32_t next() {
        const uint32_t sym = cur & 0xFFu;
        cur >>= 8;
        ++pos;
        if ((pos & 3) == 0) refill();
        return sym;
    }
    // the next four symbols at once (byte j = symbol j); only when the position is word aligned
    __device__ __forceinline__ bool word_aligned() const { return (pos & 3) == 0; }
    __device__ __forceinline__ uint32_t take_word() {
        const uint32_t v = cur;
        pos += 4;
        refill();
        return v;
    }
};

// One coding step on left-aligned state (src/codec.rs:55-89).  L: low << sh, H: (high << sh) | ones.
// Returns the number of shifts.
template <int CLS, bool C32>
__device__ __forceinline__ uint32_t encode_step_al(uint32_t &L, uint32_t &H, uint32_t &pend, BitSink2 &sink,
                                                   uint32_t cl, uint32_t ch, uint32_t count,
                                                   const typename Cls<CLS>::M &g, uint32_t sh, uint32_t one)
{
    using C = Cls<CLS>;
    using P = typename C::P;
    const uint32_t rm1 = (H - L) >> sh;                            // range - 1  (:58)
    const P nh = C::mulr(ch, rm1), nl = C::mulr(cl, rm1);
    // `one` == 1 << sh, handed in as an opaque value so that quotient * one + L stays a single IMAD
    const uint32_t nh2 = ~((uint32_t)C::divc(nh, g, count) * one + (L - 1u));   // ~high' (:59)
    const uint32_t l2 = (uint32_t)C::divc(nl, g, count) * one + L;              // low'   (:60)
    uint32_t n1, n;                                                // E1/E2 shifts (:63-74), all shifts (<= c)
    renorm_counts<C32>(l2, nh2, n1, n);
    const uint32_t k = n - n1;                                     // E3 shifts (:75-83)
    pend = sink.put_code(top_bits(l2, n1), n1, pend, k);
    L = shl_c(l2, n) & 0x7FFFFFFFu;                                // :87-88 after the E3 subtraction
    H = ~shl_c(nh2, n) | 0x80000000u;                              // high refills with ones
    return n;
}

// The same step with the emission left to the caller (BitSink2::put_pair): returns the settled bits and the two counts.
template <int CLS, bool C32>
__device__ __forceinline__ BitSink2::Code encode_core_al(uint32_t &L, uint32_t &H, uint32_t cl, uint32_t ch, uint32_t count,
                                                         const typename Cls<CLS>::M &g, uint32_t sh, uint32_t one)
{
    using C = Cls<CLS>;
    using P = typename C::P;
    const uint32_t rm1 = (H - L) >> sh;
    const P nh = C::mulr(ch, rm1), nl = C::mulr(cl, rm1);
    const uint32_t nh2 = ~((uint32_t)C::divc(nh, g, count) * one + (L - 1u));
    const uint32_t l2 = (uint32_t)C::divc(nl, g, count) * one + L;
    uint32_t n1, n;
    renorm_counts<C32>(l2, nh2, n1, n);
    BitSink2::Code cd;
    cd.bits = top_bits(l2, n1); cd.n1 = n1; cd.k = n - n1;
    L = shl_c(l2, n) & 0x7FFFFFFFu;
    H = ~shl_c(nh2, n) | 0x80000000u;
    return cd;
}

// ------------------------------------------------------------------ encoder
template <typename TW, int CLS, bool FULL, bool C32>
__global__ void __launch_bounds__(kLaneThreads, 2)
encode_lane_al_kernel(const LaneEncJob job)
{
    using C = Cls<CLS>;
    using M = typename C::M;
    extern __shared__ uint4 smem_u4[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t blk = (uint64_t)blockIdx.x * kLaneThreads + threadIdx.x;
    if (blk >= job.n_blocks) return;

    LaneTable2<TW, FULL> tab;
    tab.init(smem_u4, warp, lane);
    tab.reset(job.init_tree);

    const uint64_t off = job.in_off[blk];
    const uint32_t len = (uint32_t)(job.in_off[blk + 1] - off);
    const uint32_t c = job.c, sh = 32 - c;
    const uint32_t one = pinned(job.one, off);
    const uint32_t count0 = job.count0, eof_freq = job.eof_freq;   // 257 and 1 for a fresh model
    const M *magic = reinterpret_cast<const M *>(job.magic);
    const uint32_t tcap = job.tcap;

    ByteSource3 src;
    src.init(job.in + off, len, lane_stage_slot<TW>(smem_u4));
    BitSink2 sink;
    sink.init(job.slots + blk * job.slot_stride);
    uint32_t L = 0, H = 0xFFFFFFFFu;                       // low = 0, high = code_max (src/codec.rs:30-31)
    uint32_t pend = 0;

    // Both phases walk the input word by word once the position is word aligned: the four symbols of a word
    // are extracted with constant byte selectors, the per-symbol position bookkeeping disappears, and the
    // reciprocals of the adaptive phase arrive four positions ahead of their use.
    // adaptive phase: the model still learns, count grows by one per symbol
    const uint32_t n_adapt = len < tcap ? len : tcap;
    uint32_t t = 0;
    M gn = C::ldm(magic);                                  // reciprocal of position t, loaded one ahead
    auto adapt_coded = [&](uint32_t sym, const M &g) {
        uint32_t cl, ch;
        // cum(256) = total - freq(EOF); increments-only tables (fresh models only) keep the 256 implicit
        tab.template query<true>(sym, count0 + t - eof_freq - (FULL ? 0u : 256u), cl, ch);
        encode_step_al<CLS, C32>(L, H, pend, sink, cl, ch, count0 + t, g, sh, one);
        ++t;
    };
    auto adapt_core = [&](uint32_t sym, const M &g) {
        uint32_t cl, ch;
        tab.template query<true>(sym, count0 + t - eof_freq - (FULL ? 0u : 256u), cl, ch);
        const BitSink2::Code cd = encode_core_al<CLS, C32>(L, H, cl, ch, count0 + t, g, sh, one);
        ++t;
        return cd;
    };
    auto adapt_step = [&](uint32_t sym) {
        const M g = gn;
        gn = C::ldm(magic + t + 1);
        adapt_coded(sym, g);
    };
    while (t < n_adapt && !src.word_aligned()) adapt_step(src.next());
    if (t + 4 <= n_adapt) {
        M g0 = gn, g1 = C::ldm(magic + t + 1), g2 = C::ldm(magic + t + 2), g3 = C::ldm(magic + t + 3);
        while (t + 4 <= n_adapt) {
            const M m0 = C::ldm(magic + t + 4), m1 = C::ldm(magic + t + 5), m2 = C::ldm(magic + t + 6), m3 = C::ldm(magic + t + 7);
            const uint32_t wv = src.take_word();
            // the four symbols of a word go to the bit packer as two pairs (BitSink2::put_pair)
            const BitSink2::Code c0 = adapt_core(__byte_perm(wv, 0, 0x4440), g0), c1 = adapt_core(__byte_perm(wv, 0, 0x4441), g1);
            pend = sink.put_pair(c0, c1, pend);
            const BitSink2::Code c2 = adapt_core(__byte_perm(wv, 0, 0x4442), g2), c3 = adapt_core(__byte_perm(wv, 0, 0x4443), g3);
            pend = sink.put_pair(c2, c3, pend);
            g0 = m0; g1 = m1; g2 = m2; g3 = m3;
        }
        gn = g0;
    }
    while (t < n_adapt) adapt_step(src.next());
    // frozen phase (adaptive_tree.rs:84): total == FMAX, table and reciprocal are constant
    // reciprocal of FMAX: launch constants (no global load in the frozen loop)
    const M gfz = C::mk(pinned(job.gf_m, off), pinned(job.gf_sh, off));
    const uint32_t countf = count0 + n_adapt;
    const uint32_t cum256f = countf - eof_freq;
    if (t < len) {
        tab.freeze_to_cumulative();
        // the lookup does not depend on the coder state (SURVEY.md A.7): look symbol t+1 up before coding
        // symbol t, so the shared-memory latency overlaps the range update
        uint32_t cl, ch;
        tab.query_frozen(src.next(), cum256f, cl, ch);
        ++t;                                               // t = symbols looked up so far
        auto frozen_step = [&](uint32_t sym) {             // codes the symbol looked up before, looks `sym` up
            const uint32_t cl_cur = cl, ch_cur = ch;
            tab.query_frozen(sym, cum256f, cl, ch);
            encode_step_al<CLS, C32>(L, H, pend, sink, cl_cur, ch_cur, countf, gfz, sh, one);
            ++t;
        };
        auto frozen_core = [&](uint32_t sym) {             // the same, emission left to put_pair
            const uint32_t cl_cur = cl, ch_cur = ch;
            tab.query_frozen(sym, cum256f, cl, ch);
            const BitSink2::Code cd = encode_core_al<CLS, C32>(L, H, cl_cur, ch_cur, countf, gfz, sh, one);
            ++t;
            return cd;
        };
        while (t < len && !src.word_aligned()) frozen_step(src.next());
        while (t + 4 <= len) {
            const uint32_t wv = src.take_word();
            const BitSink2::Code c0 = frozen_core(__byte_perm(wv, 0, 0x4440)), c1 = frozen_core(__byte_perm(wv, 0, 0x4441));
            pend = sink.put_pair(c0, c1, pend);
            const BitSink2::Code c2 = frozen_core(__byte_perm(wv, 0, 0x4442)), c3 = frozen_core(__byte_perm(wv, 0, 0x4443));
            pend = sink.put_pair(c2, c3, pend);
        }
        while (t < len) frozen_step(src.next());
        encode_step_al<CLS, C32>(L, H, pend, sink, cl, ch, countf, gfz, sh, one);
    }
    const M gf = n_adapt == tcap ? gfz : gn;               // reciprocal of the final total
    // EOF symbol: [cum(256), total), then the tail of src/codec.rs:91-99: the remaining `extra` MSBs of
    // low, the first of them carrying the pending run, then flush
    const uint32_t shifts = encode_step_al<CLS, C32>(L, H, pend, sink, cum256f, countf, countf, gf, sh, one);
    const uint32_t extra = c - shifts;
    sink.put_code(top_bits(L, extra), extra, pend, 0);
    job.sizes[blk] = sink.finish();
    job.status[blk] = 0;
    StageSlot::wait<0>();                                  // nothing of this thread may still be in flight at exit
}

// ------------------------------------------------------------------ bit window (decoder input)
// w0:w1:w2 are three consecutive big-endian stream words; the window = the 32 stream bits starting at bit `pos` of
// w0.  The word after w2 is in the staging slot (StageSlot) or on its way there: a refill shifts the words, reads the
// slot and requests the following word.
// A step that consumes at most 16 bits (code_bits <= 16, the decoder's STG flag) lets the refill run every SECOND
// step: after a refill pos < 32, two steps add at most 32, so one word always suffices, the first step of a pair
// reads its window from w0:w1 (pos < 32) and the second from w0:w1 or w1:w2 (pos < 48).  That halves the refill
// code issued per symbol (13 instructions, all predicated: some lane of the warp refills almost every step) and the
// cp.async bookkeeping (commit + wait + the three padding LDS ptxas puts before every LDGSTS), and every wait finds a
// copy that was requested a whole pair of steps (> 1,000 cycles) earlier -- nothing younger exists.  Wider classes
// refill after every step (their steps are twice as long).
struct BitWindow {
    uint32_t w0, w1, w2, pos;
    const uint32_t *base;
    uint32_t idx, last;     // next word to request / last word that may be read
    StageSlot slot;

    static __device__ __forceinline__ uint32_t swap(uint32_t x) { return __byte_perm(x, 0, 0x0123); }
    __device__ __forceinline__ uint32_t word_at(uint32_t i) const { return __ldg(base + (i < last ? i : last)); }
    __device__ __forceinline__ void request() {
        slot.request(base + (idx < last ? idx : last));                    // past the end: re-read, never used
        ++idx;
    }
    // len >= 1.  Returns the first 32 bits of the stream and leaves the window right after them.
    __device__ __forceinline__ uint32_t init(const uint8_t *src, uint32_t len, void *slot_mem) {
        const uintptr_t a = (uintptr_t)src;
        const uint32_t mis = (uint32_t)(a & 3);
        base = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
        last = ((mis + len + 3) >> 2) - 1;
        pos = 8 * mis;
        slot.init(slot_mem);
        w0 = swap(word_at(0)); w1 = swap(word_at(1));
        const uint32_t first = win();
        w0 = w1; w1 = swap(word_at(2)); w2 = swap(word_at(3));
        idx = 4;
        request();
        StageSlot::commit();
        return first;
    }
    // pos < 32 (after every refill point)
    __device__ __forceinline__ uint32_t win() const { return __funnelshift_l(w1, w0, pos); }
    // pos < 64 (second step of a pair); the funnel shift takes its count modulo 32
    __device__ __forceinline__ uint32_t win2() const {
        const bool up = pos >= 32;
        return __funnelshift_l(up ? w2 : w1, up ? w1 : w0, pos);
    }
    __device__ __forceinline__ void skip(uint32_t n) { pos += n; }          // first step of a pair: n <= 16, no refill
    __device__ __forceinline__ void advance(uint32_t n) {                   // refill point; pos + n < 64
        StageSlot::wait<0>();
        pos += n;
        if (pos >= 32) { pos -= 32; w0 = w1; w1 = w2; w2 = swap(slot.read()); request(); }
        StageSlot::commit();
    }
};

// Register-only variant (the word after w1 in `nxt`, loaded one refill ahead) for the warp mapping
// (redux_warp_codec.cuh), where the window is warp-uniform: one refill cadence, nothing to decouple.
struct BitWindowReg {
    uint32_t w0, w1, nxt, pos;
    const uint32_t *base;
    uint32_t idx, last;     // next word to prefetch / last word that may be read

    static __device__ __forceinline__ uint32_t swap(uint32_t x) { return __byte_perm(x, 0, 0x0123); }
    __device__ __forceinline__ uint32_t ld() {
        const uint32_t v = __ldg(base + (idx < last ? idx : last));        // past the end: re-read, never used
        ++idx;
        return v;
    }
    __device__ __forceinline__ uint32_t init(const uint8_t *src, uint32_t len) {
        const uintptr_t a = (uintptr_t)src;
        const uint32_t mis = (uint32_t)(a & 3);
        base = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
        last = ((mis + len + 3) >> 2) - 1;
        idx = 0;
        pos = 8 * mis;
        w0 = swap(ld()); w1 = swap(ld()); nxt = ld();
        const uint32_t first = win();
        w0 = w1; w1 = swap(nxt); nxt = ld();
        return first;
    }
    __device__ __forceinline__ uint32_t win() const { return __funnelshift_l(w1, w0, pos); }
    __device__ __forceinline__ void advance(uint32_t n) {                   // n <= 32
        pos += n;
        if (pos >= 32) { pos -= 32; w0 = w1; w1 = swap(nxt); nxt = ld(); }
    }
};

// 1 / x to 1 ulp (MUFU.RCP); x is a range in [2, 2^32], far from the denormal and overflow cases __fdividef guards
__device__ __forceinline__ float rcp_approx(float x) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return 1.0f / x;
#endif
}

// Largest total frequency for which the float estimate of value = X / range is within one of the quotient.
constexpr uint32_t kQuotientMaxCount = 1u << 20;

// ------------------------------------------------------------------ byte sink (decoder output), phase-free
// Decoded symbols leave as aligned 32-bit words whatever the byte phase of the stream's slot: the bytes not yet
// stored sit in the TOP c8 bits of `top` (oldest lowest), four new symbols wv complete the word
// (wv << c8) | (top >> (32 - c8)) -- one funnel shift -- and leave their own top c8 bits pending.  Every lane runs
// the same instructions whether its slot starts at byte phase 0, 1, 2 or 3.  That matters: round 1 walked to a
// word boundary symbol by symbol first, the lanes of a warp left that head loop after 0..3 steps, and because the
// decoder's loops are left by early returns the compiler's convergence barriers never brought them back together:
// a warp whose 32 slots had four different phases ran the whole stream four times over (measured 4.0x,
// scripts/bench_alignment.py; any ragged batch, e.g. the corpus files one stream each, is such a warp).
// The slot's first word also holds up to three bytes of the neighbouring slot, which must not be written: that one
// word is stored to a private scratch location instead and its own bytes follow byte-wise at the end.
struct ByteSinkF {
    uint32_t *w0;        // the slot's first (aligned) word
    uint32_t *pw;        // aligned word holding the next pending byte
    uint32_t *wp;        // where the next word store goes: pw, or the scratch word while the first word is open
    uint32_t top, c8;    // pending bytes: the top c8 bits of `top`
    uint32_t ph;         // byte phase of the slot inside its first word

    __device__ __forceinline__ void init(uint8_t *d, uint32_t *scratch) {
        const uintptr_t a = (uintptr_t)d;
        w0 = pw = reinterpret_cast<uint32_t *>(a & ~(uintptr_t)3);
        ph = (uint32_t)(a & 3);
        c8 = 8 * ph;                      // the neighbour's bytes in the first word count as pending (never stored)
        top = 0;
        wp = ph ? scratch : pw;
    }
    __device__ __forceinline__ void store_word(uint32_t word) {
#if defined(__CUDA_ARCH__)
        asm volatile("st.global.u32 [%0], %1;" :: "l"(wp), "r"(word) : "memory");    // both targets are global memory
#else
        *wp = word;
#endif
        ++pw;
        wp = pw;
    }
    // four symbols (byte j = symbol j)
    __device__ __forceinline__ void put4(uint32_t wv) {
        store_word(__funnelshift_l(top, wv, c8));
        top = wv;
    }
    // one symbol (the steps after the last whole group of four of a phase)
    __device__ __forceinline__ void put(uint32_t sym) {
        top = (top >> 8) | (sym << 24);
        c8 += 8;
        if (c8 == 32) { store_word(top); c8 = 0; }
    }
    __device__ __forceinline__ void partial(uint32_t wv, uint32_t nbytes) {       // the first nbytes symbols of wv
        for (uint32_t j = 0; j < nbytes; ++j) put((wv >> (8 * j)) & 0xFFu);
    }
    // the bytes no word store carried: the pending ones, and our part of the slot's first word
    __device__ __forceinline__ void finish(const uint32_t *scratch) const {
        const bool head_open = pw == w0;                                           // no word was ever completed
        uint8_t *b = reinterpret_cast<uint8_t *>(pw);
        const uint32_t c = c8 >> 3;
        for (uint32_t i = head_open ? ph : 0u; i < c; ++i)
            b[i] = (uint8_t)(top >> (32 - c8 + 8 * i));
        if (!head_open && ph) {
            const uint32_t headw = *scratch;                                       // this thread's own earlier store
            uint8_t *h = reinterpret_cast<uint8_t *>(w0);
            for (uint32_t j = ph; j < 4; ++j) h[j] = (uint8_t)(headw >> (8 * j));
        }
    }
};

// ------------------------------------------------------------------ decoder
// STG: a step never consumes more than 16 bits (code_bits <= 16): pairs of steps share one refill point (BitWindow).
template <typename TW, int CLS, bool FULL, bool C32, bool STG>
struct LaneDecoderAl {
    using C = Cls<CLS>;
    using P = typename C::P;
    using M = typename C::M;
    // narrow class: once the model is frozen the table is the cumulative array (searched with absolute boundaries)
    static constexpr bool kFrozenCum = CLS == kNarrow && FULL && sizeof(TW) == 2;
    LaneTable2<TW, FULL> tab;
    BitWindow bw;
    ByteSinkF out;
    uint32_t L, H, V;    // left-aligned low / high (src/codec.rs:11-24) and the code-value window
    uint32_t sh, one, t, left;   // one == 1 << sh, opaque to the compiler (keeps q * one + L an IMAD)
    uint32_t count0, eof_freq;   // start total / frequency of EOF (257 / 1 for a fresh model)
    uint32_t top_a, top_b, top_c;   // nodes 128, 64, 192 (the first descent round) live in registers
    int32_t st;          // 0 running, -1 EOF symbol decoded (success), >0 error code

    // One symbol (src/codec.rs:123-161).  Returns false when the stream ends here -- EOF symbol decoded
    // (st = -1), bits ran out (st = 1) or, when PEEK, a data symbol with nowhere to go (st = 6) -- and true
    // with the symbol in `sym_out` and every state register advanced otherwise.
    // The model update (adaptive_tree.rs:83-92) needs no walk of its own: the nodes of update(s+1) are exactly
    // the nodes at which the descent to s turned LEFT (each covers s from above; the last one is the unstored
    // node 256), and the descent has just loaded their values -- so each left turn stores value + 1.  After a
    // step that returns false the stream is finished, so what such a step stored no longer matters.
    // MODE: 0 = refill after the step (window at pos < 32); 1 / 2 = first / second step of a pair that refills once
    // (STG only, see BitWindow).
    template <bool ADAPT, bool PEEK, int MODE = 0>
    __device__ __forceinline__ bool step(uint32_t &sym_out, const M &g, uint32_t count_frozen) {
        constexpr bool UPD = ADAPT && !PEEK;
        const uint32_t count = ADAPT ? count0 + t : count_frozen;
        // src/codec.rs:129-131 without the division: find i with cum(i)*range <= X < cum(i+1)*range,
        // X = (value-low+1)*count - 1
        const uint32_t rm1 = (H - L) >> sh;
        const P X = C::mulr(count, (V - L) >> sh) - 1;
        P plo = 0, phi = 0;
        uint32_t I = 0;                                       // i * 32: the descent's position, in table entries
        bool is_eof;                                          // value >= cum(256) = count - freq(EOF): the EOF symbol
        if (kFrozenCum && !ADAPT) {
            // Frozen model, narrow class: the table has been rewritten as the cumulative array C[i] = cum(i) of
            // AdaptiveLinearModel (adaptive_linear.rs:26-28; freeze_to_cumulative) and get_symbol (:61-70) is a 4-ary
            // search on ABSOLUTE boundaries: the residuals X - C[.] * range of a round's three boundaries do not
            // depend on each other or on earlier rounds, their sign bits move the position, and nothing else is
            // tracked until the last round, which fetches its whole group of five entries and takes the symbol's two
            // boundaries from their residuals (the tree descent had to carry the lower and the upper product through
            // every round: four min / max operations per round).  Entry i sits where tree node i sat: halfword
            // i & 1 of the lane's word i >> 1.
            const uint32_t nrange = ~rm1;                     // -(range)
            const uint32_t Xr = (uint32_t)X;
            const uint32_t N0 = Xr - (uint32_t)C::mulr(count - eof_freq, rm1);       // X - cum(256) * range
            is_eof = (int32_t)N0 >= 0;
            uint32_t J = tab.pos0();                          // data-dependent part of the position (a byte address)
            int kb = 0;                                       // constant part, folded into the loads' offsets
#pragma unroll
            for (int h = 64; h >= 4; h >>= 2) {               // entries i + h, i + 2h, i + 3h (even: 64 bytes per entry)
                const bool cached = h == 64;
                const uint32_t vb = cached ? top_b : tab.ld_at(J + (uint32_t)(kb + h * 64));
                const uint32_t va = cached ? top_a : tab.ld_at(J + (uint32_t)(kb + 2 * h * 64));
                const uint32_t vc = cached ? top_c : tab.ld_at(J + (uint32_t)(kb + 3 * h * 64));
                // -1: the boundary lies above X.  The search stands at the far end i + 3h and moves back
                const uint32_t ma = (uint32_t)((int32_t)(va * nrange + Xr) >> 31), mb = (uint32_t)((int32_t)(vb * nrange + Xr) >> 31),
                               mc = (uint32_t)((int32_t)(vc * nrange + Xr) >> 31);
                J += (ma + mb + mc) * (uint32_t)(h * 64);
                pin_chain(J);
                kb += 3 * h * 64;
            }
            // last round: the whole group C[i .. i+4] (i is a multiple of four: bytes +0, +2, +128, +130, +256 of entry
            // i) in ONE round trip.  Its residuals are ordered, d0 >= d1 >= ... >= d4, with d0 >= 0; the symbol's lower
            // boundary is the one with the smallest non-negative residual (the unsigned minimum), its upper boundary
            // the one with the largest negative residual (the unsigned maximum -- N0 = X - cum(256) * range, negative
            // for every data symbol, stands in for C[256], which the table does not hold: "entry 256" reads a zero,
            // see kTabZeroRowBytes, whose residual X is non-negative and so never the maximum).
            const uint32_t e0 = tab.ld_at(J + (uint32_t)kb), e1 = tab.ld_at(J + (uint32_t)(kb + 2)), e2 = tab.ld_at(J + (uint32_t)(kb + 128)),
                           e3 = tab.ld_at(J + (uint32_t)(kb + 130)), e4 = tab.ld_at(J + (uint32_t)(kb + 256));
            const uint32_t d0 = e0 * nrange + Xr, d1 = e1 * nrange + Xr, d2 = e2 * nrange + Xr, d3 = e3 * nrange + Xr, d4 = e4 * nrange + Xr;
            const uint32_t R = umin32(umin32(d0, d1), umin32(d2, d3));
            const uint32_t N = umax32(umax32(N0, d1), umax32(umax32(d2, d3), d4));
            // s = i + the number of boundaries C[i+1 .. i+3] at or below X
            const uint32_t cnt = 3u + (uint32_t)((int32_t)d1 >> 31) + (uint32_t)((int32_t)d2 >> 31) + (uint32_t)((int32_t)d3 >> 31);
            I = (((J - tab.pos0() + (uint32_t)kb) >> 6) + cnt) << 5;      // entry i sits at byte (i >> 1) * 128
            plo = Xr - R;
            phi = Xr - N;
        } else
        if (CLS == kNarrow) {
            // 4-ary descent in the RESIDUAL domain, without a single predicate.  R = X - (largest boundary known to
            // be <= X) and N = X - (smallest boundary known to be > X, two's complement: negative).  A round forms the
            // residuals of its three boundaries cum(i+h) <= cum(i+m) <= cum(i+m+h) (products < 2^30, so every residual
            // fits a signed word); each sign bit is one comparison, their sum is how far the descent moves
            // (0, h, m or m+h nodes), the new R is the smallest non-negative residual = the UNSIGNED minimum of all of
            // them, the new N the largest negative one = the unsigned maximum.  Round 2's form -- compare, select the
            // second boundary, compare, select the index -- paid two predicate latencies (13 cycles each) per round on
            // the chain; here a round is IMAD, SHF, IADD3, IMAD between two table loads.
            const uint32_t nrange = ~rm1;                     // -(range): range = rm1 + 1
            uint32_t R = (uint32_t)X;
            uint32_t N = (uint32_t)X - (uint32_t)C::mulr(count - eof_freq, rm1);   // node 256
            is_eof = (int32_t)N >= 0;
            uint32_t J = tab.pos0();
            int kc = 0;
#pragma unroll
            for (int m = 128; m >= 2; m >>= 2) {
                const int h = m >> 1;
                const int oddadj = (h == 1) ? LaneTable<TW>::kOddAdj : 0;      // nodes i+1, i+3 are odd
                const bool cached = m == 128;
                // position = J + kc entries: J (a byte address, LaneTable2::pos0) collects the data-dependent steps --
                // each round moves back from its far end i + m + h by up to three half-steps -- and kc the constants,
                // which fold into the loads' immediate offsets
                constexpr int EB = (int)sizeof(TW);                            // bytes per table entry
                const uint32_t ia = J + (uint32_t)((kc + (m << 5)) * EB), ib = J + (uint32_t)((kc + (h << 5) + oddadj) * EB),
                               ic = J + (uint32_t)((kc + ((m + h) << 5) + oddadj) * EB);
                const uint32_t ar = cached ? top_a : tab.ld_at(ia);
                const uint32_t br = cached ? top_b : tab.ld_at(ib);
                const uint32_t cr = cached ? top_c : tab.ld_at(ic);
                const uint32_t da = ((FULL ? 0u : (uint32_t)m) + ar) * nrange + R;
                const uint32_t db = ((FULL ? 0u : (uint32_t)h) + br) * nrange + R;
                const uint32_t dc = ((FULL ? 0u : (uint32_t)h) + cr) * nrange + da;
                // -1: the boundary lies above X, the descent turns left there
                const uint32_t ma = (uint32_t)((int32_t)da >> 31), mb = (uint32_t)((int32_t)db >> 31), mc = (uint32_t)((int32_t)dc >> 31);
                if (UPD) {
                    // a left turn = the node covers the symbol from above = it is on the symbol's update path
                    // (node c only when the first level went right: ma = -1 implies mc = -1, so that is mc - ma);
                    // stored unconditionally: value + 0 or + 1
                    if (cached) { top_a -= ma; top_b -= mb; top_c -= mc - ma; }
                    else {
                        tab.st_at(ia, ar - ma);
                        tab.st_at(ib, br - mb);
                        tab.st_at(ic, cr - mc + ma);
                    }
                }
                R = umin32(umin32(R, db), umin32(da, dc));
                N = umax32(umax32(N, db), umax32(da, dc));
                J += (ma + mb + mc) * (uint32_t)((h << 5) * EB);
                pin_chain(J);
                kc += 3 * (h << 5);
            }
            I = (J - tab.pos0() + (uint32_t)kc * (uint32_t)sizeof(TW)) / (uint32_t)sizeof(TW);
            plo = (uint32_t)X - R;
            phi = (uint32_t)X - N;
        } else
        if (CLS == kWide && count > kQuotientMaxCount) {          // (WIDE_D: totals stay below 2^17)
            // 64-bit products, very long streams: the plain product-domain descent
            phi = C::mulr(count - eof_freq, rm1);
            is_eof = X >= phi;
#pragma unroll
            for (int m = 128; m >= 2; m >>= 1) {              // even nodes i + m
                // nodes 128, 64 and 192 are the register copies (the shared-memory ones are stale while ADAPT runs)
                const bool low_half = I == 0;                 // m == 64: node 64 or node 192
                const uint32_t tr = m == 128 ? top_a : m == 64 ? (low_half ? top_b : top_c) : (uint32_t)tab.t[I + (uint32_t)(m << 5)];
                const P pr = C::mul_add((FULL ? 0u : (uint32_t)m) + tr, rm1, plo);
                const bool right = X >= pr;
                if (UPD && !right) {
                    if (m == 128) top_a += 1u;
                    else if (m == 64) { if (low_half) top_b += 1u; else top_c += 1u; }
                    else tab.t[I + (uint32_t)(m << 5)] = (TW)(tr + 1u);
                }
                if (right) { I += (uint32_t)(m << 5); plo = pr; } else { phi = pr; }
            }
            {                                                 // m = 1: odd node i + 1
                const uint32_t tr = tab.t[(int)I + 32 + LaneTable<TW>::kOddAdj];
                const P pr = C::mul_add((FULL ? 0u : 1u) + tr, rm1, plo);
                const bool right = X >= pr;
                if (UPD && !right) tab.t[(int)I + 32 + LaneTable<TW>::kOddAdj] = (TW)(tr + 1u);
                if (right) { I += 32u; plo = pr; } else { phi = pr; }
            }
        } else {
            // 64-bit products: get the reference's value = X / range (src/codec.rs:131) FIRST -- a float
            // estimate made exact by one remainder check -- and search in the 32-bit value domain, two
            // tree levels per round like the narrow class.  The quotient is < count <= 2^20, so the relative
            // errors 2^-24 (X) + 2 x 2^-24 (range) + 2^-23 (MUFU.RCP) + 2^-24 (product) keep the estimate within
            // 0.375 of X / range; biased down by 0.4 its truncation is the quotient or one less (never more, never
            // negative beyond -0.775, which truncates to 0), so ONE one-sided check finishes it.
            uint32_t v = (uint32_t)fmaf(__ull2float_rn((unsigned long long)X), rcp_approx((float)rm1 + 1.0f), -0.4f);
            if (X - C::mulr(v, rm1) > (P)rm1) v += 1u;         // remainder >= range: the estimate was one too low
            // the residual-domain 4-ary descent of the narrow class on plain values: R = v - lo, N = v - hi < 0
            uint32_t R = v, N = v - (count - eof_freq);
            is_eof = (int32_t)N >= 0;                         // the quotient is in hand: no product for node 256
            uint32_t J = tab.pos0();
            int kc = 0;
#pragma unroll
            for (int m = 128; m >= 2; m >>= 2) {
                const int h = m >> 1;
                const int oddadj = (h == 1) ? LaneTable<TW>::kOddAdj : 0;
                const bool cached = m == 128;
                constexpr int EB = (int)sizeof(TW);                            // bytes per table entry
                const uint32_t ia = J + (uint32_t)((kc + (m << 5)) * EB), ib = J + (uint32_t)((kc + (h << 5) + oddadj) * EB),
                               ic = J + (uint32_t)((kc + ((m + h) << 5) + oddadj) * EB);
                const uint32_t ar = cached ? top_a : tab.ld_at(ia);
                const uint32_t br = cached ? top_b : tab.ld_at(ib);
                const uint32_t cr = cached ? top_c : tab.ld_at(ic);
                const uint32_t da = R - ((FULL ? 0u : (uint32_t)m) + ar);
                const uint32_t db = R - ((FULL ? 0u : (uint32_t)h) + br);
                const uint32_t dc = da - ((FULL ? 0u : (uint32_t)h) + cr);
                const uint32_t ma = (uint32_t)((int32_t)da >> 31), mb = (uint32_t)((int32_t)db >> 31), mc = (uint32_t)((int32_t)dc >> 31);
                if (UPD) {
                    if (cached) { top_a -= ma; top_b -= mb; top_c -= mc - ma; }
                    else {
                        tab.st_at(ia, ar - ma);
                        tab.st_at(ib, br - mb);
                        tab.st_at(ic, cr - mc + ma);
                    }
                }
                R = umin32(umin32(R, db), umin32(da, dc));
                N = umax32(umax32(N, db), umax32(da, dc));
                J += (ma + mb + mc) * (uint32_t)((h << 5) * EB);
                pin_chain(J);
                kc += 3 * (h << 5);
            }
            I = (J - tab.pos0() + (uint32_t)kc * (uint32_t)sizeof(TW)) / (uint32_t)sizeof(TW);
            const uint32_t lo = v - R, hi = v - N;
            plo = C::mulr(lo, rm1);
            phi = C::mulr(hi, rm1);
        }
        const uint32_t sym = I >> 5;
        // src/codec.rs:133-134 (for the EOF symbol the descent's products are meaningless but harmless: the step
        // leaves through the single exit below before anything is stored or consumed)
        const uint32_t nh2 = ~((uint32_t)C::divc(phi, g, count) * one + (L - 1u));
        const uint32_t l2 = (uint32_t)C::divc(plo, g, count) * one + L;
        // src/codec.rs:140-158 in closed form
        uint32_t n1, n;
        renorm_counts<C32>(l2, nh2, n1, n);
        const uint32_t k = n - n1;
        // ONE exit per step: the EOF symbol (src/codec.rs:136-138: no renorm, no reads), bits running out inside
        // get_bit (:49-52: Err(Eof)) or, when PEEK, a data symbol with nowhere to go
        if ((int)PEEK | (int)is_eof | (int)(n > left)) {            // bitwise: one condition, one branch
            if (is_eof) st = -1;
            else if (n > left) { st = 1; left = 0; }
            else { st = 6; left -= n; }       // the reference read this symbol's bits before its write failed
            return false;
        }
        left -= n;
        // E1/E2: shift the window, pulling the next stream bits in; E3: keep the MSB, drop k bits below it
        const uint32_t win = MODE == 2 ? bw.win2() : bw.win();
        const uint32_t A = __funnelshift_lc(win, V, n1);
        const uint32_t Bv = __funnelshift_lc(shl_c(win, n1), A, k);
        V = (A & 0x80000000u) | (Bv & 0x7FFFFFFFu);
        if (MODE == 1) bw.skip(n); else bw.advance(n);
        L = shl_c(l2, n) & 0x7FFFFFFFu;
        H = ~shl_c(nh2, n) | 0x80000000u;
        sym_out = sym;
        ++t;
        return true;
    }

    // Decodes symbols while t < t_end.  ADAPT: the model still learns (count = count0 + t, one reciprocal per
    // position, loaded four positions ahead in the main loop); otherwise the table is frozen at `count_frozen`.
    // PEEK: the output slot is full -- decode one more symbol only to tell a complete stream (EOF next) from
    // Err(Eof) and from OUT_CAPACITY.
    // The loop runs four symbols per round from the first symbol on (ByteSinkF takes them at any byte phase): their
    // bytes go to constant positions of one word and the per-symbol sink and loop bookkeeping disappears.
    template <bool ADAPT, bool PEEK>
    __device__ __forceinline__ void run(uint32_t t_end, const M *magic, uint32_t count_frozen, const M &g_frozen) {
        // the three nodes of the first descent round (128, 64, 192) live in registers: one shared-memory round
        // trip off every symbol's chain; the adaptive phase counts into them and writes them back at the end
        top_a = tab.t[128 << 5]; top_b = tab.t[64 << 5]; top_c = tab.t[192 << 5];
        uint32_t sym = 0;
        if (PEEK) {
            if (t < t_end) (void)step<ADAPT, true>(sym, ADAPT ? C::ldm(magic + t) : g_frozen, count_frozen);
            return;
        }
        // reciprocals of positions t .. t+3, each loaded four positions ahead (the table is padded: reading past the
        // last position a short stream uses is harmless)
        M g0 = ADAPT ? C::ldm(magic + t) : g_frozen, g1 = g0, g2 = g0, g3 = g0;
        if (ADAPT) { g1 = C::ldm(magic + t + 1); g2 = C::ldm(magic + t + 2); g3 = C::ldm(magic + t + 3); }
        while (t + 4 <= t_end) {
            M m0 = g0, m1 = g1, m2 = g2, m3 = g3;
            if (ADAPT) {
                m0 = C::ldm(magic + t + 4); m1 = C::ldm(magic + t + 5); m2 = C::ldm(magic + t + 6); m3 = C::ldm(magic + t + 7);
            }
            constexpr int M1 = STG ? 1 : 0, M2 = STG ? 2 : 0;     // pairs of steps share one refill point
            // a step that ends the stream (st != 0 from then on) leaves through `break`: both loops and the code
            // after them converge in one place, so the exits need one convergence scope, not two
            uint32_t wv;
            if (!step<ADAPT, false, M1>(sym, g0, count_frozen)) break;
            wv = sym;
            if (!step<ADAPT, false, M2>(sym, g1, count_frozen)) { out.partial(wv, 1); break; }
            wv |= sym << 8;
            if (!step<ADAPT, false, M1>(sym, g2, count_frozen)) { out.partial(wv, 2); break; }
            wv |= sym << 16;
            if (!step<ADAPT, false, M2>(sym, g3, count_frozen)) { out.partial(wv, 3); break; }
            out.put4(wv | (sym << 24));
            if (ADAPT) { g0 = m0; g1 = m1; g2 = m2; g3 = m3; }
        }
        M gn = g0;
        while (st == 0 && t < t_end) {
            const M g = gn;
            if (ADAPT) gn = C::ldm(magic + t + 1);
            if (!step<ADAPT, false>(sym, g, count_frozen)) break;
            out.put(sym);
        }
        if (ADAPT) { tab.t[128 << 5] = (TW)top_a; tab.t[64 << 5] = (TW)top_b; tab.t[192 << 5] = (TW)top_c; }
    }
};

template <typename TW, int CLS, bool FULL, bool C32, bool STG>
__global__ void __launch_bounds__(kLaneThreads, 2)
decode_lane_al_kernel(const LaneDecJob job)
{
    using D = LaneDecoderAl<TW, CLS, FULL, C32, STG>;
    using M = typename D::M;
    extern __shared__ uint4 smem_u4[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t blk = (uint64_t)blockIdx.x * kLaneThreads + threadIdx.x;
    D d;
    d.tab.init(smem_u4, warp, lane);
    if (D::kFrozenCum) {
        // "Entry 256" of a frozen cumulative array is read as the halfword after the table: node 0 / C[0] of the same
        // lane of the NEXT warp, or the zero row after the last warp's table (kTabZeroRowBytes).  It must read zero
        // whatever that thread is doing -- also when it has no block at all, or has not started yet -- so every
        // thread of the CTA clears it here, before the first one can get that far.
        reinterpret_cast<uint32_t *>(d.tab.t)[0] = 0u;
        if (warp == kLaneWarpsPerCta - 1)
            reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(smem_u4) + (size_t)kLaneWarpsPerCta * kTabNodes * 32 * sizeof(TW))[lane] = 0u;
        __syncthreads();
    }
    if (blk >= job.n_blocks) return;
    d.tab.reset(job.init_tree);

    const uint64_t coff = job.comp_off[blk];
    const uint64_t clen = job.comp_off[blk + 1] - coff;
    const uint64_t roff = job.raw_off[blk];
    const uint64_t cap64 = job.raw_off[blk + 1] - roff;
    if (clen >= (1ull << 29)) {                 // 32-bit bit counters; such a stream is not lane work
        job.raw_len[blk] = 0; job.consumed[blk] = 0; job.status[blk] = 5;
        return;
    }
    const uint32_t c = job.c;
    const uint32_t cap = cap64 > 0xFFFFFFFEull ? 0xFFFFFFFEu : (uint32_t)cap64;
    const uint32_t total_bits = (uint32_t)clen * 8;
    d.sh = 32 - c; d.one = job.one; d.count0 = job.count0; d.eof_freq = job.eof_freq;
    uint32_t *scratch = reinterpret_cast<uint32_t *>(job.consumed + blk);   // this thread's own word until the end
    d.out.init(job.raw + roff, scratch);
    d.st = 0; d.t = 0;
    d.L = 0; d.H = 0xFFFFFFFFu; d.V = 0; d.left = 0;
    const M *magic = reinterpret_cast<const M *>(job.magic);
    const uint32_t tcap = job.tcap;

    // src/codec.rs:124-127: prime code_bits bits (Err(Eof) if the stream is shorter)
    if (total_bits < c) {
        d.st = 1;
    } else {
        d.V = d.bw.init(job.comp + coff, (uint32_t)clen, lane_stage_slot<TW>(smem_u4));
        d.left = total_bits - c;
    }
    // The two phases are entered unconditionally (a stream that already failed gets an empty range of positions): a
    // divergent `if` around them would be one more convergence scope every symbol step's exit has to break out of.
    const M g0 = D::C::ldm(magic);
    const uint32_t e1 = d.st != 0 ? 0u : (tcap < cap ? tcap : cap);
    d.template run<true, false>(e1, magic, 0, g0);
    if (d.st == 0 && d.t == cap && cap < tcap) d.template run<true, true>(d.t + 1, magic, 0, g0);
    const M gf = D::C::mk(job.gf_m, job.gf_sh);               // reciprocal of FMAX: launch constants, no global load
    if (D::kFrozenCum && d.st == 0) d.tab.freeze_to_cumulative();   // a frozen step will run (at least the peek)
    d.template run<false, false>(d.st != 0 ? d.t : cap, magic, d.count0 + tcap, gf);
    if (d.st == 0) d.template run<false, true>(d.t + 1, magic, d.count0 + tcap, gf);
    d.out.finish(scratch);
    job.raw_len[blk] = d.t;
    job.consumed[blk] = (total_bits - d.left + 7) >> 3;
    job.status[blk] = d.st < 0 ? 0 : d.st;
    StageSlot::wait<0>();                                  // nothing of this thread may still be in flight at exit
}

}  // namespace rdx
