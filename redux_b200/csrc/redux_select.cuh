// redux_select.cuh -- picks each block's start model by its estimated compressed size (redux_select_models,
// DESIGN.md 3.10).
//
// The reference model is a counter: +1 per coded symbol until the total reaches freq_max, then frozen.  So the ideal
// code length of a block under start row r (total T, EOF entry r_EOF) depends only on the block's histograms.  With
// n = floor(8 len / s) symbols, F = freq_max, m = min(n, F - T) adaptive symbols, h the histogram of the first m
// symbols, g = H - h the histogram of the rest and f = r + h the frozen row (total T' = T + m), in natural logs:
//     cost ln2 = [lnG(T+m) - lnG(T)] - sum_x [lnG(r_x+h_x) - lnG(r_x)] + sum_x g_x ln(T'/f_x) + ln(T'/r_EOF)
// (lnG = log-gamma): the data symbols in order, then EOF against the frozen total.
//
//   train_count_kernel   (redux_train.cuh) the full histogram H of every block into a scratch row
//   select_cost_kernel   one CTA per block: the cost of every candidate and the argmin
//
// The host sorts the candidates by split point F - T (ascending) and groups equal split points.  A CTA walks the
// groups in that order.  A group whose split point lies inside the block (0 < m < n) first advances a running
// histogram h of the block's prefix up to m; a group at m = 0 uses h = 0 and one at m = n uses h = H, so neither reads
// the block's bytes again.  Each warp evaluates whole models: lane l sums the bins l, l + 32, ... of the non-zero bins
// of H, lane 0 adds the 32 partial sums in lane order and the per-model terms.  Every cost is so computed in one fixed
// order whichever warp computes it, and the argmin (lowest index among equal costs) does not depend on the order in
// which the warps' candidates are combined: the choice is deterministic.
//
// The running histogram lives in shared memory for symbol_bits <= 14 and in a per-block scratch row of global memory
// above.  The phases are separate functions so that the CPU emulation under tests/ can run them thread by thread, as
// the barriers order them.
#pragma once
#include "redux_train.cuh"

namespace rdx {

constexpr uint32_t kSelectThreads = 256;
constexpr uint32_t kSelectWarps = kSelectThreads / 32;
constexpr uint32_t kSelectMaxSmemSymbolBits = 14;            // wider alphabets keep the running histogram in global memory
constexpr double kSelectInvLn2 = 1.4426950408889634;         // 1 / ln 2

struct SelectJob {
    const uint8_t *in;
    const uint64_t *in_off;      // block i = in[in_off[i] .. in_off[i+1])
    const uint32_t *rows;        // n_models candidate rows, nsym entries each (EOF last)
    const uint2 *start;          // per model: {total, EOF entry}
    const uint32_t *order;       // model indices, split point freq_max - total ascending
    const uint32_t *group;       // n_groups + 1: order[group[g] .. group[g+1]) share split point split[g]
    const uint32_t *split;       // n_groups distinct split points, ascending
    const uint32_t *hist;        // n_blocks x nsym: the full histogram of every block
    uint32_t *run;               // n_blocks x 2^s running histograms (symbol_bits > 14), else unused
    uint32_t *block_model;       // n_blocks: the choice
    double *cost;                // n_blocks x n_models costs in bits, or NULL
    double *best_cost = nullptr; // n_blocks: the chosen model's cost in bits, or NULL (redux_build_models)
    uint64_t n_blocks;
    uint32_t n_models, n_groups, s, nsym;
};

// Per-CTA view of one block.
struct SelectBlock {
    const uint8_t *base;
    uint32_t n;                  // symbols (< 2^31)
    const uint32_t *H;           // full histogram
    uint32_t *h;                 // running prefix histogram (shared or global)
    bool prefix;                 // some split point lies inside the block: h is needed
};

struct SelectBest { double c; uint32_t k; };

struct SelectShared {
    double part[kSelectThreads];               // per-lane partial sums of the model each warp evaluates
    SelectBest best[kSelectWarps];
};

__device__ __forceinline__ SelectBlock select_block(const SelectJob &j, uint64_t blk, uint32_t *smem_run)
{
    SelectBlock b;
    const uint64_t s0 = j.in_off[blk], s1 = j.in_off[blk + 1];
    b.base = j.in + s0;
    b.n = (uint32_t)((s1 - s0) * 8 / j.s);
    b.H = j.hist + blk * j.nsym;
    b.h = j.s <= kSelectMaxSmemSymbolBits ? smem_run : j.run + (blk << j.s);
    b.prefix = false;
    for (uint32_t g = 0; g < j.n_groups; ++g)
        if (j.split[g] > 0 && j.split[g] < b.n) { b.prefix = true; break; }
    return b;
}

__device__ __forceinline__ void select_zero(const SelectJob &j, const SelectBlock &b, uint32_t tid)
{
    const uint32_t bins = 1u << j.s;
    for (uint32_t x = tid; x < bins; x += kSelectThreads) b.h[x] = 0;
}

// Adds the symbols at positions [a, e) to the running histogram: each thread a run of consecutive positions, equal
// neighbours added with one atomic.
__device__ __forceinline__ void select_advance(const SelectJob &j, const SelectBlock &b, uint32_t a, uint32_t e,
                                               uint32_t tid)
{
    const uint32_t per = (e - a + kSelectThreads - 1) / kSelectThreads;
    const uint32_t k0 = a + tid * per;
    const uint32_t k1 = k0 + per < e ? k0 + per : e;
    uint32_t cur = 0, run = 0;
    for (uint32_t k = k0; k < k1; ++k) {
        const uint32_t sym = train_symbol(b.base, j.s, k);
        if (sym == cur) { ++run; continue; }
        if (run) atomicAdd(&b.h[cur], run);
        cur = sym; run = 1;
    }
    if (run) atomicAdd(&b.h[cur], run);
}

// Lane `lane`'s share of the per-bin terms of model k with m adaptive symbols (natural logs):
//     - [lnG(r_x + h_x) - lnG(r_x)] + g_x ln(T' / f_x)   over the bins x = lane, lane + 32, ... with H_x > 0
__device__ __forceinline__ double select_partial(const SelectJob &j, const SelectBlock &b, uint32_t k, uint32_t m,
                                                 uint32_t lane)
{
    const uint32_t *r = j.rows + (uint64_t)k * j.nsym;
    const double tp = (double)j.start[k].x + (double)m;
    double acc = 0.0;
    for (uint32_t x = lane; x < j.nsym - 1; x += 32) {
        const uint32_t hx = b.H[x];
        if (!hx) continue;
        const uint32_t h = m == 0 ? 0u : m == b.n ? hx : b.h[x];
        const uint32_t g = hx - h;
        const double rx = (double)r[x], fx = rx + (double)h;
        if (h) acc -= lgamma(fx) - lgamma(rx);
        if (g) acc += (double)g * log(tp / fx);
    }
    return acc;
}

// Lane 0: the cost in bits of model k from its warp's 32 partial sums (in lane order) and the per-model terms
//     lnG(T+m) - lnG(T) + ln(T' / r_EOF).
__device__ __forceinline__ double select_bits(const SelectJob &j, uint32_t k, uint32_t m, const double *part)
{
    double acc = 0.0;
    for (uint32_t l = 0; l < 32; ++l) acc += part[l];
    const double t = (double)j.start[k].x, tp = t + (double)m;
    if (m) acc += lgamma(tp) - lgamma(t);
    acc += log(tp / (double)j.start[k].y);
    return acc * kSelectInvLn2;
}

// Lane 0: select_bits of model k, written to the cost row when asked, and kept if it beats the warp's best so far
// (lowest index among equal costs).
__device__ __forceinline__ void select_finish(const SelectJob &j, const SelectBlock &b, uint64_t blk, uint32_t k,
                                              uint32_t m, const double *part, SelectBest *best)
{
    (void)b;
    const double c = select_bits(j, k, m, part);
    if (j.cost) j.cost[blk * j.n_models + k] = c;
    if (c < best->c || (c == best->c && k < best->k)) { best->c = c; best->k = k; }
}

// Thread 0: the block's choice from the warps' bests.
__device__ __forceinline__ void select_choose(const SelectJob &j, uint64_t blk, const SelectBest *best)
{
    SelectBest w = best[0];
    for (uint32_t i = 1; i < kSelectWarps; ++i)
        if (best[i].c < w.c || (best[i].c == w.c && best[i].k < w.k)) w = best[i];
    j.block_model[blk] = w.k;
    if (j.best_cost) j.best_cost[blk] = w.c;
}

// The adaptive symbols of group g in a block of n symbols.
__device__ __forceinline__ uint32_t select_m(const SelectJob &j, const SelectBlock &b, uint32_t g)
{
    return j.split[g] < b.n ? j.split[g] : b.n;
}

#if !defined(RDX_HOST_EMU)
__global__ void __launch_bounds__(kSelectThreads) select_cost_kernel(SelectJob j)
{
    extern __shared__ uint32_t select_run[];
    __shared__ SelectShared sh;
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (uint64_t blk = blockIdx.x; blk < j.n_blocks; blk += gridDim.x) {
        const SelectBlock b = select_block(j, blk, select_run);
        if (b.prefix) select_zero(j, b, tid);
        SelectBest best = {__longlong_as_double(0x7FF0000000000000ll), 0xFFFFFFFFu};
        uint32_t pos = 0;
        for (uint32_t g = 0; g < j.n_groups; ++g) {
            const uint32_t m = select_m(j, b, g);
            if (m > pos && m < b.n) {            // uniform over the CTA
                __syncthreads();                  // h is zeroed, and the previous split point's models are done
                select_advance(j, b, pos, m, tid);
                __syncthreads();
                pos = m;
            }
            for (uint32_t q = j.group[g] + warp; q < j.group[g + 1]; q += kSelectWarps) {
                sh.part[tid] = select_partial(j, b, j.order[q], m, lane);
                __syncwarp();
                if (lane == 0) select_finish(j, b, blk, j.order[q], m, sh.part + warp * 32, &best);
                __syncwarp();
            }
        }
        if (lane == 0) sh.best[warp] = best;
        __syncthreads();
        if (tid == 0) select_choose(j, blk, sh.best);
        __syncthreads();                          // before the next block reuses h and the bests
    }
}
#endif

}  // namespace rdx
