// redux_train.cuh -- trains many start models from sample bytes (redux_train_models, DESIGN.md 3.9).
//
// The reference trains a model by calling Model::get_frequency(sym) (src/model/mod.rs:23-25) for every symbol its
// BitReader yields (symbol_bits at a time, MSB-first, a trailing partial symbol dropped: src/bitio/mod.rs:94-108).
// Each call adds one to the symbol's frequency until the total reaches freq_max, and no sample symbol is EOF, so
// the trained vector has a closed form:
//     out = start row + histogram of the first min(n_sym, freq_max - total(start row)) symbols,
//     n_sym = floor(8 * len / symbol_bits).
// The same for both model kinds.  Counts are integers, so the atomics below give the exact result in any order.
//
//   train_init_kernel    copies each sample's start row into its output row
//   train_count_kernel   one CTA per (sample, chunk of symbol positions below the sample's limit): counts the
//                        chunk's symbols and adds the counts to the output row
//
// A chunk is a range of symbol POSITIONS; symbol k is read at bit k * symbol_bits, so a width that does not divide
// 8 never has a symbol split between two CTAs or two threads.  Counting:
//   - symbol_bits <= 14: sub-histograms in shared memory (one per warp while they fit in 64 KiB), flushed into the
//     output row with one global atomic per non-zero bin;
//   - symbol_bits 15 and 16: straight into the output row in global memory;
//   - every thread adds a RUN of equal consecutive symbols with one atomic, so the run and geometric classes of the
//     generator, which send most symbols to one bin, do not queue 32 lanes on one shared-memory address per symbol.
// The phases are separate functions so that the CPU emulation of the tests under tests/ can run them thread by
// thread, phase by phase, as the barriers order them.
#pragma once
#include "redux_common.cuh"

namespace rdx {

constexpr uint32_t kTrainThreads = 256;
constexpr uint32_t kTrainChunk = 16384;            // symbol positions per CTA (the library's choice; TrainJob::chunk)
constexpr uint32_t kTrainSmemWords = 16384;        // shared-memory histogram words per CTA (64 KiB)
constexpr uint32_t kTrainMaxSmemSymbolBits = 14;   // wider alphabets count in global memory

struct TrainJob {
    const uint8_t *in;
    const uint64_t *in_off;      // sample i = in[in_off[i] .. in_off[i+1])
    const uint32_t *table;       // start rows, nsym entries each
    const uint2 *sample;         // per sample: {start row, freq_max - total(start row)}
    uint32_t *out;               // n_samples x nsym
    uint64_t n_samples;
    uint64_t n_ctas;             // n_samples * chunks
    uint32_t s, nsym;
    uint32_t chunk;              // symbol positions per CTA
    uint32_t chunks;             // CTAs per sample
    uint32_t copies;             // sub-histograms in shared memory; 0: count in global memory
};

// Sub-histograms of 2^s bins in shared memory: one per warp while they fit, 0 for symbol_bits > 14.
RDX_HD uint32_t train_copies(uint32_t s)
{
    if (s > kTrainMaxSmemSymbolBits) return 0;
    const uint32_t fit = kTrainSmemWords >> s;
    return fit < kTrainThreads / 32 ? fit : kTrainThreads / 32;
}

// The positions one CTA counts: [lo, hi) of sample `sample`, hi <= the sample's limit.  False if there are none.
struct TrainRange {
    uint64_t sample;
    uint32_t lo, hi;
    const uint8_t *base;
    uint32_t *row;               // the sample's output row
};

__device__ __forceinline__ bool train_range(const TrainJob &j, uint64_t cta, TrainRange *r)
{
    r->sample = cta / j.chunks;
    const uint64_t b = j.in_off[r->sample], e = j.in_off[r->sample + 1];
    const uint64_t n_sym = (e - b) * 8 / j.s;
    const uint64_t limit = n_sym < j.sample[r->sample].y ? n_sym : (uint64_t)j.sample[r->sample].y;   // < 2^31
    const uint64_t lo = (cta % j.chunks) * j.chunk;
    if (lo >= limit) return false;
    r->lo = (uint32_t)lo;
    r->hi = (uint32_t)(lo + j.chunk < limit ? lo + j.chunk : limit);
    r->base = j.in + b;
    r->row = j.out + r->sample * j.nsym;
    return true;
}

__device__ __forceinline__ void train_zero(const TrainJob &j, uint32_t *hist, uint32_t tid)
{
    const uint32_t words = j.copies << j.s;
    for (uint32_t i = tid; i < words; i += kTrainThreads) hist[i] = 0;
}

// Adds `n` to bin `sym`: this warp's sub-histogram, or the output row.
__device__ __forceinline__ void train_add(const TrainJob &j, const TrainRange &r, uint32_t *hist, uint32_t tid,
                                          uint32_t sym, uint32_t n)
{
    if (j.copies) atomicAdd(&hist[((tid >> 5) % j.copies << j.s) + sym], n);
    else atomicAdd(&r.row[sym], n);
}

// Symbol at position k: bits [k*s, k*s + s) MSB-first.  Reads only the bytes those bits occupy (all below the
// sample's length, since k < n_sym).
__device__ __forceinline__ uint32_t train_symbol(const uint8_t *base, uint32_t s, uint64_t k)
{
    const uint64_t bit = k * s;
    const uint32_t sh = (uint32_t)(bit & 7);
    const uint8_t *p = base + (bit >> 3);
    const uint32_t nb = (sh + s + 7) >> 3;                  // 1 .. 3 bytes
    uint32_t w = (uint32_t)p[0] << 16;
    if (nb > 1) w |= (uint32_t)p[1] << 8;
    if (nb > 2) w |= (uint32_t)p[2];
    return (w >> (24 - sh - s)) & ((1u << s) - 1);
}

__device__ __forceinline__ void train_count(const TrainJob &j, const TrainRange &r, uint32_t *hist, uint32_t tid)
{
    uint32_t cur = 0, run = 0;
    if (j.s == 8) {
        // byte symbols: aligned 16-byte loads over the chunk's bytes (alignment contract of the _device calls),
        // bytes outside [lo, hi) masked off
        const uintptr_t a = (uintptr_t)(r.base + r.lo), e = (uintptr_t)(r.base + r.hi);
        const uintptr_t va = a & ~(uintptr_t)15;
        const uint32_t n_vec = (uint32_t)((e - va + 15) >> 4);
        for (uint32_t v = tid; v < n_vec; v += kTrainThreads) {
            const uintptr_t p = va + 16 * (uintptr_t)v;
            const uint4 q = *reinterpret_cast<const uint4 *>(p);
            const uint32_t k0 = p < a ? (uint32_t)(a - p) : 0u;
            const uint32_t k1 = p + 16 > e ? (uint32_t)(e - p) : 16u;
#pragma unroll
            for (uint32_t k = 0; k < 16; ++k) {
                if (k < k0 || k >= k1) continue;
                const uint32_t word = k < 4 ? q.x : k < 8 ? q.y : k < 12 ? q.z : q.w;
                const uint32_t sym = (word >> (8 * (k & 3))) & 0xFF;
                if (sym == cur) { ++run; continue; }
                if (run) train_add(j, r, hist, tid, cur, run);
                cur = sym; run = 1;
            }
        }
    } else {
        // other widths: each thread a run of consecutive positions
        const uint32_t per = (j.chunk + kTrainThreads - 1) / kTrainThreads;
        const uint32_t k0 = r.lo + tid * per;
        const uint32_t k1 = k0 + per < r.hi ? k0 + per : r.hi;
        for (uint32_t k = k0; k < k1; ++k) {
            const uint32_t sym = train_symbol(r.base, j.s, k);
            if (sym == cur) { ++run; continue; }
            if (run) train_add(j, r, hist, tid, cur, run);
            cur = sym; run = 1;
        }
    }
    if (run) train_add(j, r, hist, tid, cur, run);
}

__device__ __forceinline__ void train_flush(const TrainJob &j, const TrainRange &r, const uint32_t *hist, uint32_t tid)
{
    if (!j.copies) return;
    const uint32_t bins = 1u << j.s;
    for (uint32_t b = tid; b < bins; b += kTrainThreads) {
        uint32_t n = 0;
        for (uint32_t c = 0; c < j.copies; ++c) n += hist[(c << j.s) + b];
        if (n) atomicAdd(&r.row[b], n);
    }
}

#if !defined(RDX_HOST_EMU)
__global__ void __launch_bounds__(kTrainThreads) train_init_kernel(TrainJob j)
{
    for (uint64_t i = blockIdx.x; i < j.n_samples; i += gridDim.x) {
        const uint32_t *src = j.table + (uint64_t)j.sample[i].x * j.nsym;
        uint32_t *dst = j.out + i * j.nsym;
        for (uint32_t b = threadIdx.x; b < j.nsym; b += kTrainThreads) dst[b] = src[b];
    }
}

__global__ void __launch_bounds__(kTrainThreads) train_count_kernel(TrainJob j)
{
    extern __shared__ uint32_t train_hist[];
    for (uint64_t cta = blockIdx.x; cta < j.n_ctas; cta += gridDim.x) {
        TrainRange r;
        if (!train_range(j, cta, &r)) continue;             // uniform over the CTA
        train_zero(j, train_hist, threadIdx.x);
        __syncthreads();
        train_count(j, r, train_hist, threadIdx.x);
        __syncthreads();
        train_flush(j, r, train_hist, threadIdx.x);
        __syncthreads();                                     // before the next chunk zeroes the histogram
    }
}
#endif

}  // namespace rdx
