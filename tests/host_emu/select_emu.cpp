// select_emu.cpp -- TEST INFRASTRUCTURE: the model-selection kernels of redux_b200/csrc/redux_select.cuh run on the CPU.
// The histogram pass runs train_count_kernel's phases as train_emu.cpp does; select_cost_kernel runs block by block,
// each phase (zero, advance, the lanes' partial sums, lane 0's finish, the choice) for all threads before the next, as
// the kernel's barriers order them.  Built by tests/test_select_models_emu.py with g++; compared there against the
// references of tests/select_models_cases.py.  Not part of the product.
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

#include "../../redux_b200/csrc/redux_select.cuh"

using namespace rdx;

extern "C" {

// What redux_select_models enqueues (select_setup / select_enqueue in redux_capi.cu) for rows already checked, with
// `chunk` symbol positions per histogram CTA (0: the library's kTrainChunk).  mutant 0: the kernels as they are;
// 1: every model coded adaptively to the end of the block (no freeze); 2: EOF coded against the start total T
// instead of the frozen total T' (costs adjusted after the kernel's finish, the choice taken again from them).
void emu_select(uint32_t s, uint32_t f, uint32_t chunk, const uint32_t *rows, uint32_t n_models, const uint8_t *in,
                const uint64_t *in_off, uint64_t n_blocks, uint64_t max_block_len, uint32_t *block_model, double *cost,
                int mutant)
{
    const uint32_t nsym = (1u << s) + 1, fmax = (uint32_t)(((uint64_t)1 << f) - 1);
    std::vector<uint2> start(n_models);
    for (uint32_t k = 0; k < n_models; ++k) {
        uint64_t t = 0;
        for (uint32_t b = 0; b < nsym; ++b) t += rows[(uint64_t)k * nsym + b];
        start[k] = make_uint2((uint32_t)t, rows[(uint64_t)k * nsym + nsym - 1]);
    }
    std::vector<uint32_t> order(n_models), group, split;
    for (uint32_t k = 0; k < n_models; ++k) order[k] = k;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return start[a].x > start[b].x; });
    for (uint32_t q = 0; q < n_models; ++q) {
        const uint32_t room = mutant == 1 ? 0xFFFFFFFFu : fmax - start[order[q]].x;
        if (split.empty() || split.back() != room) { group.push_back(q); split.push_back(room); }
    }
    group.push_back(n_models);

    // histogram pass
    std::vector<uint32_t> hist(n_blocks * nsym, 0);
    std::vector<uint2> sample(n_blocks, make_uint2(0u, 0x7FFFFFFFu));
    TrainJob tj;
    tj.in = in; tj.in_off = in_off; tj.table = nullptr; tj.sample = sample.data(); tj.out = hist.data();
    tj.n_samples = n_blocks; tj.s = s; tj.nsym = nsym;
    tj.chunk = chunk ? chunk : kTrainChunk;
    const uint64_t max_n = max_block_len * 8 / s;
    tj.chunks = (uint32_t)((max_n + tj.chunk - 1) / tj.chunk);
    if (tj.chunks == 0) tj.chunks = 1;
    tj.n_ctas = max_n ? n_blocks * tj.chunks : 0;
    tj.copies = train_copies(s);
    std::vector<uint32_t> thist(((size_t)tj.copies << s) + 1);
    for (uint64_t cta = 0; cta < tj.n_ctas; ++cta) {
        TrainRange r;
        if (!train_range(tj, cta, &r)) continue;
        for (uint32_t t = 0; t < kTrainThreads; ++t) train_zero(tj, thist.data(), t);
        for (uint32_t t = 0; t < kTrainThreads; ++t) train_count(tj, r, thist.data(), t);
        for (uint32_t t = 0; t < kTrainThreads; ++t) train_flush(tj, r, thist.data(), t);
    }

    // select_cost_kernel
    std::vector<uint32_t> run(s > kSelectMaxSmemSymbolBits ? n_blocks << s : 0);
    std::vector<uint32_t> smem_run((size_t)1 << std::min(s, kSelectMaxSmemSymbolBits));
    std::vector<double> cost_rows(n_blocks * n_models);
    SelectJob j;
    j.in = in; j.in_off = in_off; j.rows = rows; j.start = start.data(); j.order = order.data();
    j.group = group.data(); j.split = split.data(); j.hist = hist.data(); j.run = run.data();
    j.block_model = block_model; j.cost = cost_rows.data(); j.n_blocks = n_blocks;
    j.n_models = n_models; j.n_groups = (uint32_t)split.size(); j.s = s; j.nsym = nsym;
    SelectShared sh;
    for (uint64_t blk = 0; blk < n_blocks; ++blk) {
        const SelectBlock b = select_block(j, blk, smem_run.data());
        if (b.prefix) for (uint32_t t = 0; t < kSelectThreads; ++t) select_zero(j, b, t);
        SelectBest best[kSelectWarps];
        for (auto &w : best) { w.c = INFINITY; w.k = 0xFFFFFFFFu; }
        uint32_t pos = 0;
        for (uint32_t g = 0; g < j.n_groups; ++g) {
            const uint32_t m = select_m(j, b, g);
            if (m > pos && m < b.n) {
                for (uint32_t t = 0; t < kSelectThreads; ++t) select_advance(j, b, pos, m, t);
                pos = m;
            }
            for (uint32_t w = 0; w < kSelectWarps; ++w)
                for (uint32_t q = j.group[g] + w; q < j.group[g + 1]; q += kSelectWarps) {
                    for (uint32_t lane = 0; lane < 32; ++lane)
                        sh.part[w * 32 + lane] = select_partial(j, b, j.order[q], m, lane);
                    select_finish(j, b, blk, j.order[q], m, sh.part + w * 32, &best[w]);
                }
        }
        for (uint32_t w = 0; w < kSelectWarps; ++w) sh.best[w] = best[w];
        select_choose(j, blk, sh.best);
        if (mutant == 2) {
            double bc = INFINITY;
            for (uint32_t k = 0; k < n_models; ++k) {
                const uint32_t m = std::min<uint32_t>(b.n, fmax - start[k].x);
                double &c = cost_rows[blk * n_models + k];
                c += (log((double)start[k].x) - log((double)start[k].x + m)) * kSelectInvLn2;
                if (c < bc) { bc = c; block_model[blk] = k; }
            }
        }
    }
    if (cost) std::copy(cost_rows.begin(), cost_rows.end(), cost);
}

}  // extern "C"
