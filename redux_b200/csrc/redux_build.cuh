// redux_build.cuh -- learns a table of start models from the blocks themselves (redux_build_models, DESIGN.md 3.12).
//
// Lloyd-style clustering of the blocks by their ideal code length (redux_select.cuh).  Membership M[b] is a table
// index: 0 = fresh, k in 1..K = cluster k.  One iteration, starting from M:
//   1. G_k = sum of the full histograms H_b of the blocks in cluster k (u64, exact);
//   2. candidate rows C_{k,l} = row(G_k, T_l) for every ladder level l, T_l = F >> 2l while T_l >= 2 nsym;
//   3. S_{k,l} = sum over the members of cluster k of their cost under C_{k,l}; l*_k = argmin (lowest l on a tie);
//   4. Table = [fresh, C_{1,l*_1}, ..., C_{K,l*_K}], and A = what select_cost_kernel chooses for Table;
//   5. M = A for the next iteration.
// The row rule: r_x = 1 + floor(D G_x / S) with D = T - nsym, S = sum G (G = ones when S = 0), the remainder
// D - sum floor(...) added to the bin with the largest G_x (lowest x on a tie), r_EOF = 1: total exactly T.
//
//   train_count_kernel        (redux_train.cuh) H of every block, once per call
//   build_cluster_kernel      G from H and M: a CTA walks a run of blocks, one thread per bin, and adds a bin's sum
//                             to G with one u64 atomic whenever the cluster changes (integers: exact in any order)
//   build_row_kernel          one CTA per (k, l): C_{k,l} and its {total, EOF}
//   build_ladder_kernel       one CTA per block: the cost of its own cluster's L candidates (select_partial /
//                             select_bits of redux_select.cuh, the prefix histogram walked once for all levels)
//   build_choice_kernel       one CTA per cluster: S_{k,l} in a fixed order, l*, and row k of Table
//   build_meta_kernel         one thread: select_cost_kernel's {total, EOF} | order | group | split of Table
//   select_cost_kernel        (redux_select.cuh) A and every block's chosen cost
//   build_total_kernel        one CTA: the iteration's total in a fixed order; keeps Table and A if it is the best
//
// Every sum of doubles runs in an order fixed by the block and thread indices, so the result does not depend on
// scheduling.  The phases are separate functions so that the CPU emulation under tests/ can run them thread by thread.
#pragma once
#include "redux_select.cuh"

namespace rdx {

constexpr uint32_t kBuildThreads = 256;
constexpr uint32_t kBuildMaxLevels = 16;          // s = 1, f = 31 has 15
constexpr uint32_t kBuildClusterRun = 64;         // blocks per CTA of build_cluster_kernel
constexpr uint32_t kBuildTotalThreads = 1024;

// The ladder of row totals: T_l = F >> 2l while T_l >= 2 nsym.  Returns L (>= 1, since f >= s + 2).
RDX_HD uint32_t build_ladder(uint32_t s, uint32_t f, uint32_t *T)
{
    const uint64_t F = ((uint64_t)1 << f) - 1, nsym = ((uint64_t)1 << s) + 1;
    uint32_t L = 0;
    while (L < kBuildMaxLevels && (F >> (2 * L)) >= 2 * nsym) { T[L] = (uint32_t)(F >> (2 * L)); ++L; }
    return L;
}

struct BuildJob {
    const uint32_t *hist;        // n_blocks x nsym full histograms
    const uint32_t *member;      // n_blocks: M
    unsigned long long *G;       // K x 2^s cluster sums
    uint32_t *cand;              // K x L candidate rows (cluster k - 1, level l at (k - 1) L + l), nsym entries each
    uint2 *cand_start;           // K x L: {total, EOF}
    const double *lcost;         // n_blocks x L ladder costs
    uint32_t *table;             // (K + 1) x nsym: Table of the iteration
    uint32_t *meta;              // select_cost_kernel's meta of Table (SelectSetup layout, L + 1 groups)
    uint32_t *level;             // K: l*_k
    uint64_t n_blocks;
    uint32_t K, L, s, nsym, fmax;
    uint32_t T[kBuildMaxLevels];
};

// ---- cluster sums
// Thread `tid` adds bin x = tid, tid + kBuildThreads, ... of blocks [b0, b1) to G, one atomic per run of blocks of the
// same cluster.
__device__ __forceinline__ void build_cluster(const BuildJob &j, uint64_t b0, uint64_t b1, uint32_t tid)
{
    const uint32_t bins = 1u << j.s;
    for (uint32_t x = tid; x < bins; x += kBuildThreads) {
        uint32_t cur = 0;
        unsigned long long acc = 0;
        for (uint64_t b = b0; b < b1; ++b) {
            const uint32_t k = j.member[b];
            if (k != cur) {
                if (cur && acc) atomicAdd(&j.G[((uint64_t)(cur - 1) << j.s) + x], acc);
                cur = k; acc = 0;
            }
            if (k) acc += j.hist[b * j.nsym + x];
        }
        if (cur && acc) atomicAdd(&j.G[((uint64_t)(cur - 1) << j.s) + x], acc);
    }
}

// ---- candidate rows
struct BuildRowPart { unsigned long long sum, gmax; uint32_t xmax; };

// G_x of cluster k (0-based), the ones of an empty cluster when S == 0.
__device__ __forceinline__ unsigned long long build_g(const BuildJob &j, uint32_t k, uint32_t x, bool empty)
{
    return empty ? 1ull : j.G[((uint64_t)k << j.s) + x];
}

// Phase 1, thread tid: its share of S and of the argmax (largest G_x, lowest x).
__device__ __forceinline__ BuildRowPart build_row_scan(const BuildJob &j, uint32_t k, uint32_t tid)
{
    BuildRowPart p = {0ull, 0ull, 0xFFFFFFFFu};
    for (uint32_t x = tid; x < j.nsym - 1; x += kBuildThreads) {
        const unsigned long long g = build_g(j, k, x, false);
        p.sum += g;
        if (p.xmax == 0xFFFFFFFFu || g > p.gmax) { p.gmax = g; p.xmax = x; }   // x ascends: ties keep the lowest
    }
    return p;
}

// Thread 0, between the phases: S and the argmax from the threads' parts (exact in any order).  The argmax of an
// empty cluster is bin 0 (all ones).
__device__ __forceinline__ BuildRowPart build_row_combine(const BuildRowPart *part, uint32_t n)
{
    BuildRowPart r = part[0];
    for (uint32_t t = 1; t < n; ++t) {
        r.sum += part[t].sum;
        if (part[t].xmax != 0xFFFFFFFFu &&
            (r.xmax == 0xFFFFFFFFu || part[t].gmax > r.gmax || (part[t].gmax == r.gmax && part[t].xmax < r.xmax))) {
            r.gmax = part[t].gmax; r.xmax = part[t].xmax;
        }
    }
    if (r.sum == 0) r.xmax = 0;
    return r;
}

// Phase 2, thread tid: r_x = 1 + floor(D G_x / S) (128-bit product) for its bins of row (k, l); returns the sum of its
// floors.
__device__ __forceinline__ unsigned long long build_row_write(const BuildJob &j, uint32_t k, uint32_t l,
                                                              unsigned long long S, uint32_t tid)
{
    const bool empty = S == 0;
    const unsigned long long sum = empty ? (1ull << j.s) : S;
    const unsigned long long D = j.T[l] - j.nsym;
    uint32_t *row = j.cand + ((uint64_t)k * j.L + l) * j.nsym;
    unsigned long long q = 0;
    for (uint32_t x = tid; x < j.nsym - 1; x += kBuildThreads) {
        const unsigned __int128 p = (unsigned __int128)D * build_g(j, k, x, empty);
        const unsigned long long fx = (unsigned long long)(p / sum);
        row[x] = 1u + (uint32_t)fx;
        q += fx;
    }
    return q;
}

// Thread 0, after phase 2: the remainder to the argmax bin, EOF = 1, and the row's {total, EOF}.
__device__ __forceinline__ void build_row_finish(const BuildJob &j, uint32_t k, uint32_t l, uint32_t xmax,
                                                 const unsigned long long *q, uint32_t n)
{
    unsigned long long sum = 0;
    for (uint32_t t = 0; t < n; ++t) sum += q[t];
    uint32_t *row = j.cand + ((uint64_t)k * j.L + l) * j.nsym;
    row[xmax] += (uint32_t)((j.T[l] - j.nsym) - sum);
    row[j.nsym - 1] = 1;
    j.cand_start[(uint64_t)k * j.L + l] = make_uint2(j.T[l], 1u);
}

// ---- ladder costs
// The selection's view of the candidates: rows = cand, start = cand_start, split[l] = F - T_l (ascending), L groups.
struct BuildLadderJob {
    SelectJob sel;
    const uint32_t *member;
    double *lcost;               // n_blocks x L
    uint32_t L;
};

// ---- ladder choice
// Thread tid's share of S_{k,l}: blocks b = tid, tid + kBuildThreads, ... in cluster k (1-based).
__device__ __forceinline__ double build_choice_part(const BuildJob &j, uint32_t k, uint32_t l, uint32_t tid)
{
    double acc = 0.0;
    for (uint64_t b = tid; b < j.n_blocks; b += kBuildThreads)
        if (j.member[b] == k) acc += j.lcost[b * j.L + l];
    return acc;
}

// Thread 0: S_{k,l} from the threads' parts in thread order.
__device__ __forceinline__ double build_choice_sum(const double *part, uint32_t n)
{
    double s = 0.0;
    for (uint32_t t = 0; t < n; ++t) s += part[t];
    return s;
}

// Thread tid: row k (1-based) of Table is candidate (k, l*).
__device__ __forceinline__ void build_choice_copy(const BuildJob &j, uint32_t k, uint32_t l, uint32_t tid)
{
    const uint32_t *src = j.cand + ((uint64_t)(k - 1) * j.L + l) * j.nsym;
    uint32_t *dst = j.table + (uint64_t)k * j.nsym;
    for (uint32_t x = tid; x < j.nsym; x += kBuildThreads) dst[x] = src[x];
}

// One thread: the meta of Table as select_setup lays it out, {total, EOF} per model | order | group | split, with
// the L + 1 possible split points as groups (empty ones included: they change no cost and no choice).  Totals T_l
// fall with l and fresh's nsym is the smallest, so "split point ascending, stable" is a counting sort by level with
// fresh last.
__device__ __forceinline__ void build_meta(const BuildJob &j)
{
    const uint32_t n_models = j.K + 1, G = j.L + 1;
    uint2 *start = reinterpret_cast<uint2 *>(j.meta);
    uint32_t *order = j.meta + 2 * n_models, *group = order + n_models, *split = group + G + 1;
    start[0] = make_uint2(j.nsym, 1u);
    for (uint32_t g = 0; g <= G; ++g) group[g] = 0;
    for (uint32_t k = 1; k <= j.K; ++k) {
        start[k] = make_uint2(j.T[j.level[k - 1]], 1u);
        ++group[j.level[k - 1] + 1];
    }
    group[G] = 1;                                                    // fresh
    for (uint32_t g = 0; g < G; ++g) group[g + 1] += group[g];
    for (uint32_t l = 0; l < j.L; ++l) split[l] = j.fmax - j.T[l];
    split[j.L] = j.fmax - j.nsym;
    // scatter: group[g] is used as the next free slot, then restored
    for (uint32_t k = 1; k <= j.K; ++k) order[group[j.level[k - 1]]++] = k;
    order[group[j.L]++] = 0;
    for (uint32_t g = G; g > 0; --g) group[g] = group[g - 1];
    group[0] = 0;
}

// ---- the iteration's total, and the best table so far
struct BuildTotalJob {
    const double *best_cost;     // n_blocks: each block's chosen cost (select_cost_kernel)
    double *totals;              // iterations
    const uint32_t *table, *choice;
    uint32_t *out_table, *out_choice;    // NULL: not kept
    uint64_t n_blocks, table_words;
    uint32_t it;
};

__device__ __forceinline__ double build_total_part(const BuildTotalJob &j, uint32_t tid)
{
    double acc = 0.0;
    for (uint64_t b = tid; b < j.n_blocks; b += kBuildTotalThreads) acc += j.best_cost[b];
    return acc;
}

// Thread 0: the total from the threads' parts in thread order; true if it beats every earlier iteration.
__device__ __forceinline__ bool build_total_finish(const BuildTotalJob &j, const double *part)
{
    double t = 0.0;
    for (uint32_t i = 0; i < kBuildTotalThreads; ++i) t += part[i];
    j.totals[j.it] = t;
    for (uint32_t i = 0; i < j.it; ++i)
        if (!(t < j.totals[i])) return false;
    return true;
}

__device__ __forceinline__ void build_total_keep(const BuildTotalJob &j, uint32_t tid)
{
    if (j.out_table)
        for (uint64_t i = tid; i < j.table_words; i += kBuildTotalThreads) j.out_table[i] = j.table[i];
    if (j.out_choice)
        for (uint64_t i = tid; i < j.n_blocks; i += kBuildTotalThreads) j.out_choice[i] = j.choice[i];
}

#if !defined(RDX_HOST_EMU)
__global__ void __launch_bounds__(kBuildThreads) build_cluster_kernel(BuildJob j)
{
    const uint64_t b0 = (uint64_t)blockIdx.x * kBuildClusterRun;
    const uint64_t b1 = b0 + kBuildClusterRun < j.n_blocks ? b0 + kBuildClusterRun : j.n_blocks;
    build_cluster(j, b0, b1, threadIdx.x);
}

__global__ void __launch_bounds__(kBuildThreads) build_row_kernel(BuildJob j)
{
    __shared__ BuildRowPart part[kBuildThreads];
    __shared__ unsigned long long q[kBuildThreads];
    __shared__ BuildRowPart all;
    const uint32_t k = blockIdx.x / j.L, l = blockIdx.x % j.L, tid = threadIdx.x;
    part[tid] = build_row_scan(j, k, tid);
    __syncthreads();
    if (tid == 0) all = build_row_combine(part, kBuildThreads);
    __syncthreads();
    q[tid] = build_row_write(j, k, l, all.sum, tid);
    __syncthreads();
    if (tid == 0) build_row_finish(j, k, l, all.xmax, q, kBuildThreads);
}

// select_cost_kernel's walk with one model per group: the candidates of the block's own cluster, level by level.
__global__ void __launch_bounds__(kSelectThreads) build_ladder_kernel(BuildLadderJob lj)
{
    extern __shared__ uint32_t build_run[];
    __shared__ double part[kSelectThreads];
    const SelectJob &j = lj.sel;
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (uint64_t blk = blockIdx.x; blk < j.n_blocks; blk += gridDim.x) {
        const uint32_t c = lj.member[blk];
        if (c == 0) continue;                                        // uniform over the CTA
        const SelectBlock b = select_block(j, blk, build_run);
        if (b.prefix) select_zero(j, b, tid);
        uint32_t pos = 0;
        for (uint32_t l = 0; l < lj.L; ++l) {
            const uint32_t m = select_m(j, b, l);
            if (m > pos && m < b.n) {
                __syncthreads();
                select_advance(j, b, pos, m, tid);
                __syncthreads();
                pos = m;
            }
            if (warp == l % kSelectWarps) {
                const uint32_t k = (c - 1) * lj.L + l;
                part[tid] = select_partial(j, b, k, m, lane);
                __syncwarp();
                if (lane == 0) lj.lcost[blk * lj.L + l] = select_bits(j, k, m, part + warp * 32);
                __syncwarp();
            }
        }
        __syncthreads();                                             // before the next block reuses h
    }
}

__global__ void __launch_bounds__(kBuildThreads) build_choice_kernel(BuildJob j)
{
    __shared__ double part[kBuildThreads];
    __shared__ double best;
    __shared__ uint32_t lbest;
    const uint32_t k = blockIdx.x + 1, tid = threadIdx.x;
    for (uint32_t l = 0; l < j.L; ++l) {
        part[tid] = build_choice_part(j, k, l, tid);
        __syncthreads();
        if (tid == 0) {
            const double s = build_choice_sum(part, kBuildThreads);
            if (l == 0 || s < best) { best = s; lbest = l; }
        }
        __syncthreads();
    }
    if (tid == 0) j.level[k - 1] = lbest;
    build_choice_copy(j, k, lbest, tid);
}

__global__ void build_meta_kernel(BuildJob j)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) build_meta(j);
}

__global__ void __launch_bounds__(kBuildTotalThreads) build_total_kernel(BuildTotalJob j)
{
    __shared__ double part[kBuildTotalThreads];
    __shared__ bool keep;
    part[threadIdx.x] = build_total_part(j, threadIdx.x);
    __syncthreads();
    if (threadIdx.x == 0) keep = build_total_finish(j, part);
    __syncthreads();
    if (keep) build_total_keep(j, threadIdx.x);
}
#endif

}  // namespace rdx
