// build_emu.cpp -- TEST INFRASTRUCTURE: the model-building kernels of redux_b200/csrc/redux_build.cuh run on the CPU.
// Each kernel runs CTA by CTA, each phase for all threads before the next, as the kernels' barriers order them.  Built
// by tests/test_build_models_emu.py with g++; compared there against the references of tests/build_models_cases.py.
// Not part of the product.
#include "cuda_shim.h"

#include <algorithm>
#include <vector>

thread_local EmuIdx threadIdx, blockIdx, blockDim, gridDim;

// the threads of a CTA run one after another, so an atomic add is a plain add
static inline uint32_t atomicAdd(uint32_t *p, uint32_t v)
{
    const uint32_t old = *p;
    *p = old + v;
    return old;
}
static inline unsigned long long atomicAdd(unsigned long long *p, unsigned long long v)
{
    const unsigned long long old = *p;
    *p = old + v;
    return old;
}

#include "../../redux_b200/csrc/redux_build.cuh"

using namespace rdx;

// Mutants: 1 the remainder put in bin 0; 2 a 64-bit product D G_x; 3 an empty cluster not replaced by ones (every
// floor 0, the remainder to bin 0); 4 the ladder stopping at nsym instead of 2 nsym.
enum { kRemainderBin0 = 1, kProduct64 = 2, kEmptyNotOnes = 3, kLadderNsym = 4 };

static uint32_t ladder(uint32_t s, uint32_t f, uint32_t *T, int mutant)
{
    if (mutant != kLadderNsym) return build_ladder(s, f, T);
    const uint64_t F = ((uint64_t)1 << f) - 1, nsym = ((uint64_t)1 << s) + 1;
    uint32_t L = 0;
    while (L < kBuildMaxLevels && (F >> (2 * L)) >= nsym) { T[L] = (uint32_t)(F >> (2 * L)); ++L; }
    return L;
}

// build_row_kernel for every (k, l) of a job whose G, cand and cand_start are set.
static void run_rows(const BuildJob &j, int mutant)
{
    std::vector<BuildRowPart> part(kBuildThreads);
    std::vector<unsigned long long> q(kBuildThreads);
    for (uint32_t k = 0; k < j.K; ++k)
        for (uint32_t l = 0; l < j.L; ++l) {
            for (uint32_t t = 0; t < kBuildThreads; ++t) part[t] = build_row_scan(j, k, t);
            BuildRowPart all = build_row_combine(part.data(), kBuildThreads);
            if (mutant == kRemainderBin0) all.xmax = 0;
            for (uint32_t t = 0; t < kBuildThreads; ++t) q[t] = build_row_write(j, k, l, all.sum, t);
            if (mutant == kProduct64 || (mutant == kEmptyNotOnes && all.sum == 0)) {
                uint32_t *row = j.cand + ((uint64_t)k * j.L + l) * j.nsym;
                std::fill(q.begin(), q.end(), 0ull);
                const bool empty = all.sum == 0;
                for (uint32_t x = 0; x < j.nsym - 1; ++x) {
                    const unsigned long long g = build_g(j, k, x, empty);
                    const unsigned long long fx = mutant == kEmptyNotOnes ? 0ull
                        : (unsigned long long)(j.T[l] - j.nsym) * g / (empty ? 1ull << j.s : all.sum);
                    row[x] = 1u + (uint32_t)fx;
                    q[0] += fx;
                }
            }
            build_row_finish(j, k, l, all.xmax, q.data(), kBuildThreads);
        }
}

extern "C" {

uint32_t emu_build_ladder(uint32_t s, uint32_t f, uint32_t *T, int mutant) { return ladder(s, f, T, mutant); }

// build_cluster_kernel: G (K x 2^s) from hist (n x nsym) and member (n).
void emu_build_cluster(uint32_t s, uint32_t K, const uint32_t *hist, const uint32_t *member, uint64_t n,
                       unsigned long long *G)
{
    BuildJob j{};
    j.hist = hist; j.member = member; j.G = G; j.n_blocks = n; j.K = K; j.s = s; j.nsym = (1u << s) + 1;
    std::fill(G, G + ((uint64_t)K << s), 0ull);
    for (uint64_t b0 = 0; b0 < n; b0 += kBuildClusterRun)
        for (uint32_t t = 0; t < kBuildThreads; ++t) build_cluster(j, b0, std::min<uint64_t>(b0 + kBuildClusterRun, n), t);
}

// build_row_kernel: cand (K x L x nsym) from G (K x 2^s).  Returns L.
uint32_t emu_build_rows(uint32_t s, uint32_t f, uint32_t K, const unsigned long long *G, uint32_t *cand, int mutant)
{
    BuildJob j{};
    j.K = K; j.s = s; j.nsym = (1u << s) + 1;
    j.L = ladder(s, f, j.T, mutant);
    std::vector<unsigned long long> g(G, G + ((uint64_t)K << s));
    std::vector<uint2> cs((size_t)K * j.L);
    j.G = g.data(); j.cand = cand; j.cand_start = cs.data();
    run_rows(j, mutant);
    return j.L;
}

// One round up to the table, as build_enqueue runs it: the histogram pass (train_count's phases), cluster sums, rows,
// build_ladder_kernel (lcost: n x L), build_choice_kernel (level: K, table: (K+1) x nsym, row 0 left as given) and
// build_meta_kernel (meta).  Returns L.
uint32_t emu_build_round(uint32_t s, uint32_t f, uint32_t K, const uint8_t *in, const uint64_t *in_off, uint64_t n,
                         uint64_t max_block_len, const uint32_t *member, double *lcost, uint32_t *level,
                         uint32_t *table, uint32_t *meta, int mutant)
{
    const uint32_t nsym = (1u << s) + 1;
    // histogram pass
    std::vector<uint32_t> hist(n * nsym, 0);
    std::vector<uint2> sample(n, make_uint2(0u, 0x7FFFFFFFu));
    TrainJob tj;
    tj.in = in; tj.in_off = in_off; tj.table = nullptr; tj.sample = sample.data(); tj.out = hist.data();
    tj.n_samples = n; tj.s = s; tj.nsym = nsym; tj.chunk = kTrainChunk;
    const uint64_t max_n = max_block_len * 8 / s;
    tj.chunks = (uint32_t)std::max<uint64_t>((max_n + kTrainChunk - 1) / kTrainChunk, 1);
    tj.n_ctas = max_n ? n * tj.chunks : 0;
    tj.copies = train_copies(s);
    std::vector<uint32_t> thist(((size_t)tj.copies << s) + 1);
    for (uint64_t cta = 0; cta < tj.n_ctas; ++cta) {
        TrainRange r;
        if (!train_range(tj, cta, &r)) continue;
        for (uint32_t t = 0; t < kTrainThreads; ++t) train_zero(tj, thist.data(), t);
        for (uint32_t t = 0; t < kTrainThreads; ++t) train_count(tj, r, thist.data(), t);
        for (uint32_t t = 0; t < kTrainThreads; ++t) train_flush(tj, r, thist.data(), t);
    }
    BuildJob j{};
    j.hist = hist.data(); j.member = member; j.n_blocks = n; j.K = K; j.s = s; j.nsym = nsym;
    j.fmax = (uint32_t)(((uint64_t)1 << f) - 1);
    j.L = ladder(s, f, j.T, mutant);
    std::vector<unsigned long long> G((uint64_t)K << s);
    std::vector<uint32_t> cand((size_t)K * j.L * nsym);
    std::vector<uint2> cs((size_t)K * j.L);
    j.G = G.data(); j.cand = cand.data(); j.cand_start = cs.data();
    for (uint64_t b0 = 0; b0 < n; b0 += kBuildClusterRun)
        for (uint32_t t = 0; t < kBuildThreads; ++t) build_cluster(j, b0, std::min<uint64_t>(b0 + kBuildClusterRun, n), t);
    run_rows(j, mutant);
    // build_ladder_kernel
    std::vector<uint32_t> split(j.L);
    for (uint32_t l = 0; l < j.L; ++l) split[l] = j.fmax - j.T[l];
    std::vector<uint32_t> run(s > kSelectMaxSmemSymbolBits ? n << s : 0);
    std::vector<uint32_t> smem_run((size_t)1 << std::min(s, kSelectMaxSmemSymbolBits));
    BuildLadderJob lj;
    lj.sel.in = in; lj.sel.in_off = in_off; lj.sel.rows = cand.data(); lj.sel.start = cs.data();
    lj.sel.split = split.data(); lj.sel.hist = hist.data(); lj.sel.run = run.data(); lj.sel.n_blocks = n;
    lj.sel.n_models = K * j.L; lj.sel.n_groups = j.L; lj.sel.s = s; lj.sel.nsym = nsym;
    lj.member = member; lj.lcost = lcost; lj.L = j.L;
    double part[kSelectThreads];
    for (uint64_t blk = 0; blk < n; ++blk) {
        const uint32_t c = member[blk];
        if (!c) continue;
        const SelectBlock b = select_block(lj.sel, blk, smem_run.data());
        if (b.prefix) for (uint32_t t = 0; t < kSelectThreads; ++t) select_zero(lj.sel, b, t);
        uint32_t pos = 0;
        for (uint32_t l = 0; l < j.L; ++l) {
            const uint32_t m = select_m(lj.sel, b, l);
            if (m > pos && m < b.n) {
                for (uint32_t t = 0; t < kSelectThreads; ++t) select_advance(lj.sel, b, pos, m, t);
                pos = m;
            }
            const uint32_t k = (c - 1) * j.L + l;
            for (uint32_t lane = 0; lane < 32; ++lane) part[lane] = select_partial(lj.sel, b, k, m, lane);
            lcost[blk * j.L + l] = select_bits(lj.sel, k, m, part);
        }
    }
    // build_choice_kernel, build_meta_kernel
    j.lcost = lcost; j.table = table; j.level = level; j.meta = meta;
    double cpart[kBuildThreads];
    for (uint32_t k = 1; k <= K; ++k) {
        double best = 0.0;
        uint32_t lbest = 0;
        for (uint32_t l = 0; l < j.L; ++l) {
            for (uint32_t t = 0; t < kBuildThreads; ++t) cpart[t] = build_choice_part(j, k, l, t);
            const double sum = build_choice_sum(cpart, kBuildThreads);
            if (l == 0 || sum < best) { best = sum; lbest = l; }
        }
        level[k - 1] = lbest;
        for (uint32_t t = 0; t < kBuildThreads; ++t) build_choice_copy(j, k, lbest, t);
    }
    build_meta(j);
    return j.L;
}

}  // extern "C"
