// redux_warp_codec.cuh -- latency mapping: ONE STREAM PER WARP, the 32 lanes cooperate on each symbol.
//
// For batches too small to fill the machine with one stream per lane (BASELINE.json configs 1, 2, 5: a
// file or a handful of 1 MiB blocks per stream) the only lever is the latency of one symbol.  Here the
// frequency model is the reference's LINEAR layout -- the plain cumulative array of
// AdaptiveLinearModel (src/model/adaptive_linear.rs:21-70) -- spread over the warp's REGISTERS:
//   lane l holds inc[l + 32 j], j = 0..7, where cum(i) = i + inc[i] (increments only, as in the lane
//   kernel; cum(256) = 256 + number of updates is implied, cum(257) = total).
//   * lookup (adaptive_linear.rs:51-59): cum(s), cum(s+1) are two register selects (the row j = i >> 5
//     is warp-uniform) + two shuffles;
//   * update (adaptive_linear.rs:33-39: "freq[i] += 1 for i > symbol") is 8 predicated adds executed by
//     all 32 lanes at once instead of a 257-step loop -- with the same freeze rule;
//   * search (adaptive_linear.rs:61-70: first i with value < freq[i+1]) is 8 compares per lane and one
//     warp add-reduction: the symbol is the number of boundaries cum(i), 1 <= i <= 255, that are <= value.
//     Done in the product domain (cum(i)*range <= X) so the decoder's division by range disappears
//     exactly as in the lane kernel.
// The coder state (low/high/pending, bit buffers) is warp-uniform: every lane computes it, lane 0 stores.
// Output is bit-identical to the lane kernel and to the oracle (tests/test_gpu_parity.py runs both).
#pragma once
#include "redux_common.cuh"
#include "redux_lane_codec.cuh"
#include "redux_lane_al.cuh"

namespace rdx {

constexpr int kWarpCtaWarps = 4;                       // small CTAs: spread few streams over many SMs
constexpr int kWarpCtaThreads = kWarpCtaWarps * 32;
constexpr uint32_t kFullMask = 0xFFFFFFFFu;

struct WarpTable {
    uint32_t r[8];          // inc[lane + 32 j]
    uint32_t lane;

    __device__ __forceinline__ void init(uint32_t l) {
        lane = l;
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = 0;
    }
    // inc[i] for a warp-uniform i in 0..255
    __device__ __forceinline__ uint32_t get(uint32_t i) const {
        // depth-3 select tree on the (warp-uniform) row bits instead of a 7-deep chain
        const bool b0 = i & 32u, b1 = i & 64u, b2 = i & 128u;
        const uint32_t a0 = b0 ? r[1] : r[0], a1 = b0 ? r[3] : r[2], a2 = b0 ? r[5] : r[4], a3 = b0 ? r[7] : r[6];
        const uint32_t c0 = b1 ? a1 : a0, c1 = b1 ? a3 : a2;
        return __shfl_sync(kFullMask, b2 ? c1 : c0, (int)(i & 31));
    }
    // (cum(s), cum(s+1)) of a data symbol; `updates` = inc[256]
    __device__ __forceinline__ void query(uint32_t s, uint32_t updates, uint32_t &cl, uint32_t &ch) const {
        cl = s + get(s);
        const uint32_t hi = get((s + 1) & 255u);
        ch = s + 1 + (s == 255u ? updates : hi);
    }
    // every cumulative entry above the symbol grows by one (only while the model is not frozen)
    __device__ __forceinline__ void update(uint32_t s, bool adapt = true) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] += (adapt && lane + 32u * j > s) ? 1u : 0u;
    }
};

// 128 raw bytes per warp load: lane l holds word l of the current 128-byte line.
struct WarpByteSource {
    const uint32_t *base;    // aligned
    uint32_t last_word;      // index of the last word that may be read
    uint32_t cw, nw;         // this lane's word of the current / next line
    uint32_t g;              // byte position relative to base
    uint32_t lane;

    __device__ __forceinline__ uint32_t ld(uint32_t word) const {
        return __ldg(base + (word <= last_word ? word : last_word));
    }
    __device__ __forceinline__ void init(const uint8_t *src, uint32_t len, uint32_t l) {
        const uintptr_t a = (uintptr_t)src;
        base = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);     // never reads below the stream's word
        g = (uint32_t)(a & 3);
        lane = l;
        last_word = len ? (g + len - 1) >> 2 : 0;
        cw = nw = 0;
        if (len) { cw = ld(lane); nw = ld(32 + lane); }
    }
    __device__ __forceinline__ uint32_t next() {
        const uint32_t w = __shfl_sync(kFullMask, cw, (int)((g >> 2) & 31));
        const uint32_t sym = (w >> (8 * (g & 3))) & 0xFFu;
        ++g;
        if ((g & 127) == 0) { cw = nw; nw = ld(((g >> 7) + 1) * 32 + lane); }
        return sym;
    }
};

// Bit packer whose stores are issued by one lane only (state is warp-uniform).
struct WarpBitSink : BitSink {
    bool en;
    __device__ __forceinline__ void put(uint32_t v, uint32_t n) {
        acc = (acc << n) | v;
        nb += n;
        if (nb >= 32) {
            nb -= 32;
            if (en) *w = __byte_perm((uint32_t)(acc >> nb), 0, 0x0123);
            ++w;
        }
    }
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
            uint32_t r = n1 - 1;
            if (r > 32) { put((uint32_t)(x >> 32) & (0xFFFFFFFFu >> (64 - r)), r - 32); r = 32; }
            if (r) put((uint32_t)x & (0xFFFFFFFFu >> (32 - r)), r);
        }
    }
    __device__ __forceinline__ uint32_t finish() {
        const uint32_t bytes = (uint32_t)(w - w0) * 4 + (nb + 7) / 8;
        if (nb && en) *w = __byte_perm((uint32_t)(acc << (32 - nb)), 0, 0x0123);
        return bytes;
    }
};

template <int CLS>
__device__ __forceinline__ uint32_t warp_encode_step(typename Cls<CLS>::S &low, typename Cls<CLS>::S &high,
                                                     uint32_t &pend, WarpBitSink &sink, uint32_t cl, uint32_t ch,
                                                     uint32_t count, const typename Cls<CLS>::M &g, uint32_t c)
{
    using C = Cls<CLS>;
    using S = typename C::S;
    using P = typename C::P;
    const S rm1 = high - low;
    const P nh = C::mulr(ch, rm1), nl = C::mulr(cl, rm1);
    const S h2 = low + (S)C::divc(nh, g, count) - 1;               // src/codec.rs:59
    const S l2 = low + (S)C::divc(nl, g, count);                   // src/codec.rs:60
    const Renorm<S> r = renorm<S>(l2, h2, c);                      // src/codec.rs:62-89
    if (r.n1) {
        sink.put_code((uint64_t)(l2 >> (c - r.n1)), r.n1, pend);
        pend = r.k;
    } else {
        pend += r.k;
    }
    low = r.low; high = r.high;
    return r.n1 + r.k;
}

template <int CLS>
__global__ void __launch_bounds__(kWarpCtaThreads)
encode_warp_kernel(const LaneEncJob job)
{
    using C = Cls<CLS>;
    using S = typename C::S;
    using M = typename C::M;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t blk = (uint64_t)blockIdx.x * kWarpCtaWarps + (threadIdx.x >> 5);
    if (blk >= job.n_blocks) return;                               // warp-uniform

    WarpTable tab;
    tab.init(lane);
    const uint64_t off = job.in_off[blk];
    const uint32_t len = (uint32_t)(job.in_off[blk + 1] - off);
    const uint32_t c = job.c;
    const S maxv = (S)((c == sizeof(S) * 8) ? ~(S)0 : ((((S)1) << c) - 1));
    const M *magic = reinterpret_cast<const M *>(job.magic);
    const uint32_t tcap = job.tcap;

    WarpByteSource src;
    src.init(job.in + off, len, lane);
    WarpBitSink sink;
    sink.init(job.slots + blk * job.slot_stride);
    sink.en = lane == 0;
    S low = 0, high = maxv;
    uint32_t pend = 0;

    const uint32_t n_adapt = len < tcap ? len : tcap;
    uint32_t t = 0;
    M gn = C::ldm(magic);
    for (; t < n_adapt; ++t) {                                     // adaptive phase
        const M g = gn;
        gn = C::ldm(magic + t + 1);
        const uint32_t sym = src.next();
        uint32_t cl, ch;
        tab.query(sym, t, cl, ch);
        tab.update(sym);
        warp_encode_step<CLS>(low, high, pend, sink, cl, ch, kNsym + t, g, c);
    }
    const uint32_t tt = n_adapt;
    const M gf = gn;
    const uint32_t countf = kNsym + tt;
    for (; t < len; ++t) {                                         // frozen phase
        const uint32_t sym = src.next();
        uint32_t cl, ch;
        tab.query(sym, tt, cl, ch);
        warp_encode_step<CLS>(low, high, pend, sink, cl, ch, countf, gf, c);
    }
    // (Running the model half one symbol ahead of the coder -- legal by SURVEY.md A.7 -- was measured
    // SLOWER here: 4.0 vs 4.7 MB/s on one 768 KB stream; a single in-order warp gains nothing from it.)
    const uint32_t shifts = warp_encode_step<CLS>(low, high, pend, sink, countf - 1, countf, countf, gf, c);
    const uint32_t extra = c - shifts;                             // src/codec.rs:91-99
    if (extra) sink.put_code((uint64_t)(low >> (c - extra)), extra, pend);
    const uint32_t bytes = sink.finish();
    if (lane == 0) { job.sizes[blk] = bytes; job.status[blk] = 0; }
}

// ------------------------------------------------------------------ decoder
struct WarpByteSink : ByteSink {
    bool en;
    __device__ __forceinline__ void put(uint32_t sym) {
        wacc |= sym << sh;
        sh += 8;
        if (sh == 32) {
            if (en) {
                if (pw >= dst) *reinterpret_cast<uint32_t *>(pw) = wacc;
                else store_bytes(dst, pw + 4);
            }
            pw += 4; wacc = 0; sh = 0;
        }
    }
    __device__ __forceinline__ void finish() const {
        if (sh && en) store_bytes(pw > dst ? pw : dst, pw + (sh >> 3));
    }
};

template <int CLS>
struct WarpDecoder {
    using C = Cls<CLS>;
    using S = typename C::S;
    using P = typename C::P;
    using M = typename C::M;
    WarpTable tab;
    BitSource src;          // warp-uniform: every lane reads the same words (one broadcast transaction)
    WarpByteSink out;
    S low, high, value, maxv;
    uint32_t c, t, cap;
    int32_t st;

    template <bool ADAPT>
    __device__ __forceinline__ void run(uint32_t t_end, const M *magic, uint32_t count_frozen, const M &g_frozen) {
        const S body = maxv >> 1, half = body + 1;
        M gn = ADAPT ? C::ldm(magic + t) : g_frozen;
        while (t < t_end) {
            const uint32_t count = ADAPT ? kNsym + t : count_frozen;
            const M g = gn;
            if (ADAPT) gn = C::ldm(magic + t + 1);
            const S rm1 = high - low;
            const P X = C::mulr(count, (S)(value - low)) - 1;      // (value-low+1)*count - 1
            const uint32_t updates = count - kNsym;
            if (X >= C::mulr(count - 1, rm1)) { st = -1; return; } // EOF symbol (src/codec.rs:136-138)
            // number of boundaries cum(i), i = 1..255, with cum(i)*range <= X
            uint32_t cnt = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uint32_t i = tab.lane + 32u * j;
                const P p = C::mulr(i + tab.r[j], rm1);
                cnt += (i != 0u && p <= X) ? 1u : 0u;
            }
            const uint32_t sym = __reduce_add_sync(kFullMask, cnt);
            uint32_t cl, ch;
            tab.query(sym, updates, cl, ch);
            high = low + (S)C::divc(C::mulr(ch, rm1), g, count) - 1;    // src/codec.rs:133
            low = low + (S)C::divc(C::mulr(cl, rm1), g, count);         // src/codec.rs:134
            if (ADAPT) tab.update(sym);
            const Renorm<S> r = renorm<S>(low, high, c);                // src/codec.rs:140-158
            const uint32_t n = r.n1 + r.k;
            if (!src.has(n)) { st = 1; src.left = 0; return; }
            if (t >= cap) { src.left -= n; st = 6; return; }           // sink full (the symbol's bits were read)
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

template <int CLS>
__global__ void __launch_bounds__(kWarpCtaThreads)
decode_warp_kernel(const LaneDecJob job)
{
    using D = WarpDecoder<CLS>;
    using S = typename D::S;
    using M = typename D::M;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t blk = (uint64_t)blockIdx.x * kWarpCtaWarps + (threadIdx.x >> 5);
    if (blk >= job.n_blocks) return;

    D d;
    d.tab.init(lane);
    const uint64_t coff = job.comp_off[blk];
    const uint64_t clen = job.comp_off[blk + 1] - coff;
    const uint64_t roff = job.raw_off[blk];
    const uint64_t cap64 = job.raw_off[blk + 1] - roff;
    if (clen >= (1ull << 29)) {
        if (lane == 0) { job.raw_len[blk] = 0; job.consumed[blk] = 0; job.status[blk] = 5; }
        return;
    }
    d.c = job.c;
    d.maxv = (S)((d.c == sizeof(S) * 8) ? ~(S)0 : ((((S)1) << d.c) - 1));
    d.cap = cap64 > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)cap64;
    d.src.init(job.comp + coff, (uint32_t)clen);
    d.out.init(job.raw + roff);
    d.out.en = lane == 0;
    d.st = 0; d.t = 0;
    d.low = 0; d.high = d.maxv; d.value = 0;
    const M *magic = reinterpret_cast<const M *>(job.magic);
    const uint32_t tcap = job.tcap;

    if (!d.src.has(d.c)) { d.st = 1; d.src.left = 0; }
    else d.value = (S)d.src.take64(d.c);

    const M g0 = D::C::ldm(magic);
    if (d.st == 0) d.template run<true>(tcap, magic, 0, g0);
    if (d.st == 0) {
        const M gf = D::C::ldm(magic + tcap);
        d.template run<false>(0xFFFFFFFFu, magic, kNsym + tcap, gf);
    }
    d.out.finish();
    if (lane == 0) {
        job.raw_len[blk] = d.t;
        job.consumed[blk] = (d.src.used() + 7) >> 3;
        job.status[blk] = d.st < 0 ? 0 : d.st;
    }
}

// ------------------------------------------------------------------ decoder, code_bits <= 32 (tuned)
// Same mapping (one stream per warp, cumulative array of AdaptiveLinearModel in registers, coder state
// warp-uniform) with the coder of redux_lane_al.cuh -- left-aligned low/high, the code value as a bit
// window, FLO.SH renormalisation -- and a search that is off the multiplier:
//   * value = ((pending-low+1)*count - 1) / range (src/codec.rs:131) comes from a float estimate made
//     exact by one remainder check (the quotient is < count <= 2^20; beyond that an exact 64-bit division);
//   * every lane compares its 8 cumulative entries with the value (get_symbol, adaptive_linear.rs:61-70);
//     cum_lo is the warp maximum of the entries <= value, cum_hi the warp minimum of the entries > value
//     (bounded by cum(256) = count - 1): two redux.sync the narrowing waits for, while the symbol itself
//     (a third one, the count of entries <= value) is only needed by the model update and the output.
template <int CLS, bool C32>
__global__ void __launch_bounds__(kWarpCtaThreads)
decode_warp_al_kernel(const LaneDecJob job)
{
    using C = Cls<CLS>;
    using P = typename C::P;
    using M = typename C::M;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t blk = (uint64_t)blockIdx.x * kWarpCtaWarps + (threadIdx.x >> 5);
    if (blk >= job.n_blocks) return;                               // warp-uniform

    const uint64_t coff = job.comp_off[blk];
    const uint64_t clen = job.comp_off[blk + 1] - coff;
    const uint64_t roff = job.raw_off[blk];
    const uint64_t cap64 = job.raw_off[blk + 1] - roff;
    if (clen >= (1ull << 29)) {
        if (lane == 0) { job.raw_len[blk] = 0; job.consumed[blk] = 0; job.status[blk] = 5; }
        return;
    }
    const uint32_t c = job.c, sh = 32 - c, one = job.one, tcap = job.tcap;
    const uint32_t cap = cap64 > 0xFFFFFFFEull ? 0xFFFFFFFEu : (uint32_t)cap64;
    const uint32_t total_bits = (uint32_t)clen * 8;
    const M *magic = reinterpret_cast<const M *>(job.magic);

    uint32_t cum[8];                                               // cum(lane + 32 j); a fresh model: cum(i) = i
#pragma unroll
    for (int j = 0; j < 8; ++j) cum[j] = lane + 32u * j;
    BitWindowReg bw;
    WarpByteSink out;
    out.init(job.raw + roff);
    out.en = lane == 0;
    uint32_t L = 0, H = 0xFFFFFFFFu, V = 0, left = 0, t = 0;
    int32_t st = 0;
    if (total_bits < c) {                                          // src/codec.rs:124-127
        st = 1;
    } else {
        V = bw.init(job.comp + coff, (uint32_t)clen);
        left = total_bits - c;
    }
    M gn = C::ldm(magic);
    while (st == 0) {
        const uint32_t tt = t < tcap ? t : tcap;                   // updates so far
        const uint32_t count = kNsym + tt;
        const M g = gn;
        gn = C::ldm(magic + (t + 1 < tcap ? t + 1 : tcap));
        const uint32_t rm1 = (H - L) >> sh;
        const P X = C::mulr(count, (V - L) >> sh) - 1;
        // value = X / range
        uint32_t v;
        if (count <= kQuotientMaxCount) {
            v = (uint32_t)__fdividef(CLS == kNarrow ? __uint2float_rn((uint32_t)X) : __ull2float_rn((unsigned long long)X),
                                     (float)rm1 + 1.0f);
            const P pv = C::mulr(v, rm1);
            if (pv > X) v -= 1u;
            else if (X - pv > (P)rm1) v += 1u;
        } else {
            v = (uint32_t)((unsigned long long)X / ((unsigned long long)rm1 + 1ull));
        }
        if (v >= count - 1) { st = -1; break; }                    // EOF symbol (src/codec.rs:136-138)
        uint32_t below = 0, lo = 0, hi = count - 1;                // entries <= value; their max; min of the rest
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const bool le = cum[j] <= v;
            below += le ? 1u : 0u;
            lo = max(lo, le ? cum[j] : 0u);
            hi = min(hi, le ? 0xFFFFFFFFu : cum[j]);
        }
        const uint32_t cl = __reduce_max_sync(kFullMask, lo);
        const uint32_t ch = __reduce_min_sync(kFullMask, hi);
        const uint32_t sym = __reduce_add_sync(kFullMask, below) - 1u;     // cum(0) = 0 always counts
        // src/codec.rs:133-134 and :140-158 in closed form
        const uint32_t nh2 = ~((uint32_t)C::divc(C::mulr(ch, rm1), g, count) * one + (L - 1u));
        const uint32_t l2 = (uint32_t)C::divc(C::mulr(cl, rm1), g, count) * one + L;
        uint32_t n1, n;
        renorm_counts<C32>(l2, nh2, n1, n);
        const uint32_t k = n - n1;
        if (n > left) { st = 1; left = 0; break; }                 // Err(Eof) inside get_bit (:49-52)
        if (t >= cap) { st = 6; left -= n; break; }                // sink full (the symbol's bits were read)
        left -= n;
        const uint32_t win = bw.win();
        const uint32_t A = __funnelshift_lc(win, V, n1);
        const uint32_t Bv = __funnelshift_lc(shl_c(win, n1), A, k);
        V = (A & 0x80000000u) | (Bv & 0x7FFFFFFFu);
        bw.advance(n);
        L = shl_c(l2, n) & 0x7FFFFFFFu;
        H = ~shl_c(nh2, n) | 0x80000000u;
        if (t < tcap) {                                            // adaptive_linear.rs:33-39, frozen at freq_max
#pragma unroll
            for (int j = 0; j < 8; ++j) cum[j] += (lane + 32u * j > sym) ? 1u : 0u;
        }
        out.put(sym);
        ++t;
    }
    out.finish();
    if (lane == 0) {
        job.raw_len[blk] = t;
        job.consumed[blk] = (total_bits - left + 7) >> 3;
        job.status[blk] = st < 0 ? 0 : st;
    }
}

}  // namespace rdx
