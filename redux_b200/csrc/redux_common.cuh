// redux_common.cuh -- shared host/device arithmetic of the B200 coder.
//
// Everything here is written from the algorithm's definition (SURVEY.md Appendix A), not from the
// reference's code shape: the reference renormalises bit by bit and divides by the running total
// (src/codec.rs:58-89); the device path uses the closed forms below, and tests/ prove them equal
// to the loop on the oracle.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define RDX_HD __host__ __device__ __forceinline__
#else
#define RDX_HD inline
#endif

namespace rdx {

constexpr int kSymbolBits = 8;          // device path scope: byte symbols (SURVEY.md A.9)
constexpr uint32_t kEof = 256;          // Parameters::symbol_eof   (src/model/mod.rs:69)
constexpr uint32_t kNsym = 257;         // Parameters::symbol_count (src/model/mod.rs:70)

// Arithmetic class of a (freq_bits, code_bits) pair.
//   NARROW: code+freq <= 30 -> every product fits 32 bits, 32-bit magic division.
//   WIDE  : code <= 32      -> 32-bit coder state, 64-bit products, 64-bit magic division.
//   HUGE  : code  > 32      -> 64-bit coder state, products < 2^64 (code+freq <= 64), hardware-less
//                              64-bit division (rare parameter corner; correctness only).
//   WIDE_D: WIDE whose totals stay below 349,525 for the whole launch (e.g. any 64 KiB block of a fresh model): the
//           two divisions by the total become one double-precision multiply-add each (lane_plan decides).
enum ArithClass { kNarrow = 0, kWide = 1, kHuge = 2, kWideD = 3 };

RDX_HD int arith_class(uint32_t f, uint32_t c) {
    return (c + f <= 30) ? kNarrow : (c <= 32 ? kWide : kHuge);
}

// Parameters::new validation (src/model/mod.rs:64), identical rejection rule.
RDX_HD bool params_valid(uint64_t s, uint64_t f, uint64_t c) {
    return !(s < 1 || f < s + 2 || c < f + 2 || 64 < c + f);
}

// ---------------------------------------------------------------------------------------------
// count reciprocal.  The coder divides by count_t = min(NSYM + t, FMAX) (SURVEY.md A.5): a pure
// function of the symbol position t, identical for every stream.  floor(n / d) for n < 2^nbits is
// computed as mulhi(n, magic) >> shift with
//     l = ceil(log2 d),  S = max(W, nbits + l),  magic = floor(2^S / d) + 1,  shift = S - W
// (W = 32 or 64).  Exact because e = magic*d - 2^S lies in [1, d] <= 2^l <= 2^(S-nbits), so the
// error term n*e/(d*2^S) < 1/d never carries the quotient over an integer.
// magic < 2^W needs nbits + 1 <= W - 1, i.e. nbits <= 30 (W=32) / nbits <= 62 (W=64).
// ---------------------------------------------------------------------------------------------
struct Magic32 { uint32_t m; uint32_t sh; };
struct Magic64 { uint64_t m; uint32_t sh; uint32_t pad; };

RDX_HD uint32_t ceil_log2_u64(uint64_t d) {
    uint32_t l = 0;
    while (l < 64 && ((uint64_t)1 << l) < d) ++l;
    return l;
}

// Long division of 2^S by d (d < 2^32, S <= 126) -> floor(2^S/d) truncated to 64 bits.
// Only called with quotients that fit (see above).  Bit-serial restoring division: runs once per
// table entry at set-up time, never on the coding path.
RDX_HD uint64_t pow2_div(uint32_t S, uint64_t d) {
    uint64_t q = 0, r = 0;
    // dividend = 1 followed by S zero bits; feed bits MSB first
    for (int i = (int)S; i >= 0; --i) {
        r = (r << 1) | (i == (int)S ? 1u : 0u);
        q <<= 1;
        if (r >= d) { r -= d; q |= 1; }
    }
    return q;
}

RDX_HD Magic32 make_magic32(uint32_t d, uint32_t nbits) {
    uint32_t l = ceil_log2_u64(d);
    uint32_t S = nbits + l; if (S < 32) S = 32;
    Magic32 r; r.m = (uint32_t)(pow2_div(S, d) + 1); r.sh = S - 32;
    return r;
}
RDX_HD Magic64 make_magic64(uint64_t d, uint32_t nbits) {
    uint32_t l = ceil_log2_u64(d);
    uint32_t S = nbits + l; if (S < 64) S = 64;
    Magic64 r; r.m = pow2_div(S, d) + 1; r.sh = S - 64; r.pad = 0;
    return r;
}

RDX_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
RDX_HD uint64_t mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}
RDX_HD uint32_t div_magic32(uint32_t n, Magic32 g) { return mulhi32(n, g.m) >> g.sh; }
RDX_HD uint64_t div_magic64(uint64_t n, Magic64 g) { return mulhi64(n, g.m) >> g.sh; }

// code_bits > 32: numerators reach 2^64 (code + freq <= 64, src/model/mod.rs:64), one bit more than a 64-bit magic can
// serve.  The 65-bit magic 2^64 + m' of p = 64 + l, l = ceil(log2 d), divides EVERY 64-bit numerator exactly
// (e = (2^64 + m') d - 2^p lies in [1, d] and n e < 2^64 2^l = 2^p); its product with n is formed without the carry:
// t = mulhi(n, m') <= n, (n + t) / 2 = ((n - t) >> 1) + t, then the remaining l - 1 bits of the shift (l >= 9 here:
// d >= 257).  Two of these replace the two 64-bit hardware-less divisions per symbol the HUGE class used to pay.
RDX_HD Magic64 make_magic65(uint64_t d) {
    const uint32_t l = ceil_log2_u64(d);
    Magic64 r; r.m = pow2_div(64 + l, d) + 1; r.sh = l; r.pad = 0;     // pow2_div truncates to 64 bits: drops the 2^64
    return r;
}
RDX_HD uint64_t div_magic65(uint64_t n, Magic64 g) {
    const uint64_t t = mulhi64(n, g.m);
    return (((n - t) >> 1) + t) >> (g.sh - 1);
}

// WIDE_D: floor(n / d) for n = cum * range (cum <= d, range <= 2^32) as trunc(fma(n, r, 2^-19)) with r = the double
// nearest to 1/d, valid for every total d < 349,525 (= 2^19 / 1.5).  n < 2^51 and d are exact doubles;
// |n r - n/d| <= (n/d) 2^-53 <= 2^-21 and the rounding of the fused result (magnitude <= 2^32) adds at most another
// 2^-21, so the computed value lies within E = 2^-20 of n/d + 2^-19.  If d divides n the result is >= k + 2^-19 - E > k;
// otherwise n/d is at least 1/d below the next integer and 2^-19 + E = 1.5 x 2^-19 < 1/d keeps the result below it:
// the truncation is the exact quotient, no correction step.
// (The conversion goes through 64 bits: the quotient reaches 2^32 when cum == d and range == 2^32.)
// floor(X / range) for the code_bits > 32 decoder: X < count * range < 2^64, so the quotient is below count <= 2^31.
// The double quotient carries three roundings of 2^-53 relative each (two conversions, one IEEE division): it lies
// within 2^31 * 3 * 2^-53 < 2^-20 of X / range.  Biased down by 2^-18 its truncation is the quotient or one less
// (never more), which ONE remainder check settles; v * range <= X then, so the product cannot overflow.
RDX_HD uint32_t div_by_range64(uint64_t X, uint64_t range) {
#if defined(__CUDA_ARCH__)
    const double q = __ull2double_rn(X) / __ull2double_rn(range) - 0x1p-18;
#else
    const double q = (double)X / (double)range - 0x1p-18;
#endif
    uint32_t v = q > 0.0 ? (uint32_t)q : 0u;
    if (X - (uint64_t)v * range >= range) ++v;
    return v;
}

struct MagicD { double r; };
constexpr uint32_t kWideDMaxCount = 349525;                   // totals must stay BELOW this
RDX_HD MagicD make_magicd(uint32_t d) { MagicD g; g.r = 1.0 / (double)d; return g; }
RDX_HD uint64_t div_magicd(uint64_t n, MagicD g) {
#if defined(__CUDA_ARCH__)
    return __double2ull_rz(fma(__ull2double_rn(n), g.r, 0x1p-19));
#else
    return (uint64_t)__builtin_fma((double)n, g.r, 0x1p-19);
#endif
}

RDX_HD int clz32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __clz((int)x);
#else
    return x ? __builtin_clz(x) : 32;
#endif
}
RDX_HD int clz64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __clzll((long long)x);
#else
    return x ? __builtin_clzll(x) : 64;
#endif
}

// ---------------------------------------------------------------------------------------------
// Renormalisation closed form (SURVEY.md A.6).  Given the narrowed interval [low, high] in a c-bit
// register: n1 = number of leading bits low and high share (the E1/E2 shifts of src/codec.rs:63-74,
// each emitting that bit), then k = length of the run, starting just below the MSB, where low has 1
// and high has 0 (the E3 shifts of :75-83).  E1/E2 can never follow an E3 inside one symbol, so
// the whole loop is (n1, k).  T = uint32_t (c <= 32) or uint64_t (c <= 61).
// ---------------------------------------------------------------------------------------------
template <typename T> struct Renorm { T low, high; uint32_t n1, k; };

// Shifts that give 0 once the amount reaches the register width (the degenerate low == high case
// shifts a 32-bit register by 32).
RDX_HD uint32_t shl_sat(uint32_t x, uint32_t n) { return (uint32_t)((uint64_t)x << n); }              // n <= 63
RDX_HD uint64_t shl_sat(uint64_t x, uint32_t n) { return n >= 64 ? 0 : x << n; }
RDX_HD uint32_t ones_sat(uint32_t, uint32_t n) { return (uint32_t)(((uint64_t)1 << n) - 1); }          // n <= 63
RDX_HD uint64_t ones_sat(uint64_t, uint32_t n) { return n >= 64 ? ~(uint64_t)0 : (((uint64_t)1 << n) - 1); }

template <typename T>
RDX_HD Renorm<T> renorm(T low, T high, uint32_t c) {
    constexpr int W = sizeof(T) * 8;
    const T maxv = (c == (uint32_t)W) ? ~(T)0 : ((((T)1) << c) - 1);
    const T body = maxv >> 1;                                 // bits below the MSB
    const T half = body + 1;
    const T x = low ^ high;
    const int lz = (W == 32) ? clz32((uint32_t)x) : clz64((uint64_t)x);
    const uint32_t n1 = (uint32_t)lz - (uint32_t)(W - c);     // x == 0 -> lz == W -> n1 == c
    // E3 run: after the n1 shifts, positions c-2 downwards with low=1, high=0.  Shifting (low & ~high)
    // left by n1 + (W+1-c) puts position c-2 of the shifted registers at bit W-1 and drops everything above.
    const T z = shl_sat((T)(low & ~high), n1 + (uint32_t)(W + 1 - c));
    const T nz = ~z;                                          // low (W+1-c) >= 1 bits are ones: clz <= c-1
    const uint32_t k = (uint32_t)((W == 32) ? clz32((uint32_t)nz) : clz64((uint64_t)nz));
    const uint32_t n = n1 + k;                                // total shifts, <= c
    Renorm<T> r;
    r.n1 = n1; r.k = k;
    // both stages at once: shift by n, high refills with ones; MSB of low is 0, of high is 1 (src/codec.rs:87-88
    // after the E3 subtraction of :77-78)
    r.low = shl_sat(low, n) & body;
    r.high = ((shl_sat(high, n) | ones_sat((T)0, n)) & body) | half;
    return r;
}

// Shape of one lane-kernel launch derived from (freq_bits, code_bits) and the longest block: arithmetic
// class, number of model updates before the freeze (FMAX - NSYM, adaptive_tree.rs:84), table entry width,
// reciprocal-table length and the per-block worst-case output slot ((len+1) symbols x code_bits bits,
// SURVEY.md A.4).  Shared by the host front end (redux_capi.cu) and the test harness.
struct LanePlan {
    int cls; uint32_t f, c, tcap; bool wide_table; uint32_t magic_len; uint64_t slot_stride;
    bool aligned;     // c <= 32 (32-bit coder state): the tuned kernels of redux_lane_al.cuh
    bool full_table;  // table entries can hold the reference's tree values (lowbit + increments)
    uint64_t gf_m; uint32_t gf_sh;   // reciprocal of the frozen total FMAX (classes with a reciprocal table)
};
// count0 = total frequency of the start model: symbol_count for a fresh one, larger for a model the caller
// trained before the call (then the table must hold full tree values: pretrained = true).
RDX_HD LanePlan lane_plan(uint32_t f, uint32_t c, uint64_t max_block_len, uint32_t count0 = kNsym,
                          bool pretrained = false) {
    LanePlan pl;
    pl.f = f; pl.c = c;
    pl.cls = arith_class(f, c);
    const uint64_t fmax = ((uint64_t)1 << f) - 1;
    pl.tcap = (uint32_t)(fmax - count0);                       // f <= 31 -> fits
    const uint64_t updates = max_block_len < pl.tcap ? max_block_len : pl.tcap;
    // u16 entries suffice while increments (fresh) / cumulative values (trained) fit
    pl.wide_table = pretrained ? (uint64_t)count0 + updates > 65535 : updates > 65536;
    // counts 257 .. count0 + updates, + the read-ahead of the word-wise loops (up to 7 positions past the end)
    pl.magic_len = (uint32_t)(count0 - kNsym + updates) + 8;
    const uint64_t bound = ((max_block_len + 1) * (uint64_t)c + 7) / 8;
    pl.slot_stride = ((bound + 15) & ~(uint64_t)15) + 16;
    pl.aligned = pl.cls != kHuge;
    pl.full_table = pretrained || pl.wide_table || updates + 256 <= 65535;   // cum(i) <= 256 + updates must fit u16
    // every total of the launch below the bound: the double-reciprocal division (see MagicD)
    if (pl.cls == kWide && (uint64_t)count0 + updates < kWideDMaxCount) pl.cls = kWideD;
    // plain WIDE: totals reach kWideDMaxCount > 65,535, so the table takes u32 entries with full values (the
    // conditions above already say so; stated here so that no threshold change can pair WIDE with u16 entries)
    if (pl.cls == kWide) pl.wide_table = pl.full_table = true;
    pl.gf_m = 0; pl.gf_sh = 0;
    if (pl.cls == kNarrow)    { const Magic32 g = make_magic32((uint32_t)fmax, f + c); pl.gf_m = g.m; pl.gf_sh = g.sh; }
    else if (pl.cls == kWide) { const Magic64 g = make_magic64(fmax, f + c); pl.gf_m = g.m; pl.gf_sh = g.sh; }
    else if (pl.cls == kWideD && fmax < kWideDMaxCount) {      // the frozen phase can only be reached with fmax below the bound
        const MagicD g = make_magicd((uint32_t)fmax);
        union { double d; uint64_t u; } cv; cv.d = g.r; pl.gf_m = cv.u;
    }
    return pl;
}

// ---------------------------------------------------------------------------------------------
// Synthetic mixed-entropy blocks (BASELINE.json configs 3-4).  Counter-based splitmix64 so that the
// GPU can fill any 8-byte group independently: draw(block, w) = mix(seed + block*K + (w+1)*GAMMA).
// class = block & 3:
//   0 uniform bytes                                   H ~ 8.0  bit/byte
//   1 text: a block-sized window of a corpus the caller supplies (bench.py: Calgary + Canterbury, H ~ 4.5-5),
//     or, without one, a 256-entry Zipf table over 55 symbols  H ~ 4.5
//   2 geometric: ctz of a 16-bit field                H ~ 2.0
//   3 sparse: 0x00 with p = 63/64, else a random byte H ~ 0.24
// (the reference's corpora cannot travel to the GPU box, so class 1 is a table-driven stand-in for
// the "corpus window" class of SURVEY.md 8(d); order-0 statistics are what an order-0 coder sees.)
// ---------------------------------------------------------------------------------------------
RDX_HD uint64_t splitmix_mix(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
RDX_HD uint64_t gen_draw(uint64_t seed, uint64_t block, uint64_t w) {
    return splitmix_mix(seed + block * 0xD1342543DE82EF95ull + (w + 1) * 0x9E3779B97F4A7C15ull);
}
// text-like table: rank r owns max(1, 60/(r+1)) of the 256 slots (integer Zipf law; the slots run
// out at rank 54, order-0 entropy 4.53 bit/byte -- calgary/book1 measures 4.527).
RDX_HD uint8_t text_symbol(uint32_t u8v) {
    const char *alphabet = " etaoinshrdlucmfwypvbgk,.\n-'\";ETAOINSHRDLUCMFWYPVBGKjxqz0123456";
    uint32_t acc = 0;
    for (uint32_t r = 0; r < 64; ++r) {
        uint32_t n = 60 / (r + 1); if (n < 1) n = 1;
        acc += n;
        if (u8v < acc) return (uint8_t)alphabet[r];
    }
    return (uint8_t)alphabet[63];
}
// Text class with a corpus (BASELINE.md section 4, config 3: "64 KiB window of the concatenation of calgary +
// canterbury at offset next() % (L - 65536)"): the block is corpus[off, off + block_len), off drawn once per block.
RDX_HD uint64_t text_window_offset(uint64_t seed, uint64_t block, uint64_t corpus_len, uint64_t block_len) {
    return gen_draw(seed, block, ~(uint64_t)0 - 1) % (corpus_len - block_len + 1);
}
// 8 output bytes for 64-bit group w of `block`.  corpus == NULL (or shorter than a block): the table-driven
// stand-in for the text class.
RDX_HD uint64_t gen_group(uint64_t seed, uint64_t block, uint64_t w, const uint8_t *text_lut,
                          const uint8_t *corpus = nullptr, uint64_t corpus_len = 0, uint64_t block_len = 0) {
    uint64_t r = gen_draw(seed, block, w);
    uint32_t cls = (uint32_t)(block & 3);
    if (cls == 0) return r;
    uint64_t out = 0;
    if (cls == 1 && corpus && corpus_len >= block_len && block_len) {
        const uint64_t at = text_window_offset(seed, block, corpus_len, block_len) + 8 * w;
        for (int j = 0; j < 8; ++j) out |= (uint64_t)(at + j < corpus_len ? corpus[at + j] : 0) << (8 * j);
        return out;
    }
    if (cls == 1) {
        for (int j = 0; j < 8; ++j) out |= (uint64_t)text_lut[(r >> (8 * j)) & 255] << (8 * j);
        return out;
    }
    uint64_t r2 = splitmix_mix(r ^ 0xA5A5A5A5A5A5A5A5ull);
    for (int j = 0; j < 8; ++j) {
        uint32_t u = (uint32_t)(((j < 4 ? r : r2) >> (16 * (j & 3))) & 0xFFFF);
        uint32_t b;
        if (cls == 2) { uint32_t v = u | 0x8000u; b = 0; while (!(v & 1)) { v >>= 1; ++b; } }
        else          { b = (u < 0xFC00u) ? 0u : (u & 0xFFu); }
        out |= (uint64_t)b << (8 * j);
    }
    return out;
}

}  // namespace rdx
