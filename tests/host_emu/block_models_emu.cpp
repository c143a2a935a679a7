// block_models_emu.cpp -- TEST INFRASTRUCTURE: the tuned lane kernels and the generic kernels with a start model per
// block (BlockModels), run on the CPU thread by thread through tests/host_emu/cuda_shim.h as lane_emu.cpp runs them.
// Built by tests/test_block_models_emu.py with g++; compared there against the oracle.  Not part of the product.
#include "cuda_shim.h"

#include <algorithm>
#include <vector>

thread_local EmuIdx threadIdx, blockIdx, blockDim, gridDim;

#include "../../redux_b200/csrc/redux_lane_codec.cuh"
#include "../../redux_b200/csrc/redux_lane_al.cuh"
#include "../../redux_b200/csrc/redux_generic_codec.cuh"

namespace rdx {
// dynamic shared memory of one CTA: 7 warps x 256 nodes x 32 lanes x 4 B
uint4 smem_u4[(kLaneWarpsPerCta * kTabNodes * 32 * 4 + kTabPadBytes) / 16];
// dynamic shared memory of the generic kernels: Fenwick columns of alphabets up to kGenericSmemSymbolBits
uint32_t gen_cols[((1u << kGenericSmemSymbolBits) + 2) * kGenericThreads];
}

using namespace rdx;

namespace {

std::vector<uint8_t> build_magic(const LanePlan &pl)
{
    std::vector<uint8_t> buf;
    const uint32_t nbits = pl.f + pl.c;
    if (pl.cls == kHuge) {
        buf.resize(sizeof(Magic64) * pl.magic_len);
        Magic64 *m = reinterpret_cast<Magic64 *>(buf.data());
        for (uint32_t i = 0; i < pl.magic_len; ++i) m[i] = make_magic65(kNsym + i);
        return buf;
    }
    if (pl.cls == kWideD) {
        buf.resize(sizeof(MagicD) * pl.magic_len);
        MagicD *m = reinterpret_cast<MagicD *>(buf.data());
        for (uint32_t i = 0; i < pl.magic_len; ++i) m[i] = make_magicd(kNsym + i);
        return buf;
    }
    if (pl.cls == kNarrow) {
        buf.resize(sizeof(Magic32) * pl.magic_len);
        Magic32 *m = reinterpret_cast<Magic32 *>(buf.data());
        for (uint32_t i = 0; i < pl.magic_len; ++i) m[i] = make_magic32(kNsym + i, nbits);
    } else {
        buf.resize(sizeof(Magic64) * pl.magic_len);
        Magic64 *m = reinterpret_cast<Magic64 *>(buf.data());
        for (uint32_t i = 0; i < pl.magic_len; ++i) m[i] = make_magic64(kNsym + i, nbits);
    }
    return buf;
}

template <typename K, typename J>
void run_grid(K kernel, const J &job, uint64_t n_blocks)
{
    const uint32_t grid = (uint32_t)((n_blocks + kLaneThreads - 1) / kLaneThreads);
    blockDim.x = kLaneThreads; blockDim.y = blockDim.z = 1;
    gridDim.x = grid; gridDim.y = gridDim.z = 1;
    for (uint32_t b = 0; b < grid; ++b)
        for (uint32_t t = 0; t < (uint32_t)kLaneThreads; ++t) {
            blockIdx.x = b; threadIdx.x = t;
            kernel(job);
        }
}

}  // namespace

namespace {
// The start models of a call as prepare_models of redux_capi.cu puts them on the device: the trees of every row
// (build_tree_kernel, one launch), {total, EOF frequency} of every row.  freqs == NULL: a fresh model (the tuned lane
// kernels then get no models at all; the generic kernels one row of ones).
struct ModelTable {
    std::vector<uint32_t> trees;
    std::vector<uint2> start;
    bool on = false;
    BlockModels bm(const uint32_t *block_model) const {
        BlockModels b{};
        b.trees = trees.data(); b.start = start.data(); b.block_model = block_model; b.n_models = (uint32_t)start.size();
        return b;
    }
    uint32_t max_total() const { uint32_t m = 0; for (const uint2 &x : start) m = std::max(m, x.x); return m; }
    uint32_t min_total() const { uint32_t m = 0xFFFFFFFFu; for (const uint2 &x : start) m = std::min(m, x.x); return m; }
};
ModelTable model_table(uint32_t nsym, const uint32_t *freqs, uint32_t n_models)
{
    ModelTable t;
    t.on = freqs != nullptr;
    if (!freqs) n_models = 1;
    const uint64_t nodes = (uint64_t)n_models * (nsym + 1);
    t.trees.assign(nodes, 0);
    blockDim.x = 256; gridDim.x = (uint32_t)((nodes + 255) / 256);
    for (uint32_t b = 0; b < gridDim.x; ++b)
        for (uint32_t th = 0; th < 256; ++th) { blockIdx.x = b; threadIdx.x = th; build_tree_kernel(freqs, nsym, t.trees.data(), n_models); }
    for (uint32_t m = 0; m < n_models; ++m) {
        uint32_t total = 0;
        for (uint32_t i = 0; i < nsym; ++i) total += freqs ? freqs[(size_t)m * nsym + i] : 1u;
        t.start.push_back(make_uint2(total, freqs ? freqs[(size_t)m * nsym + nsym - 1] : 1u));
    }
    return t;
}
// the plan of a launch whose blocks start from the models of `mt`: planned for the largest start total (make_plan)
LanePlan models_plan(uint32_t f, uint32_t c, uint64_t max_block_len, int force_wide_table, const ModelTable &mt)
{
    LanePlan pl = lane_plan(f, c, max_block_len, mt.on ? mt.max_total() : kNsym, mt.on);
    if (force_wide_table >= 0) { pl.wide_table = force_wide_table != 0; if (pl.wide_table) pl.full_table = true; }
    return pl;
}
}  // namespace

// force_wide_table: -1 = as the front end would choose, 0 = u16 entries, 1 = u32 entries.  freqs: n_models rows of 257
// frequencies, block i starts from row block_model[i] (NULL: row 0); freqs == NULL: every block starts fresh.
extern "C" int emu_encode_lane_models(uint32_t f, uint32_t c, uint64_t max_block_len, int force_wide_table,
                                      const uint32_t *freqs, uint32_t n_models, const uint32_t *block_model,
                                      const uint8_t *in, const uint64_t *in_off, uint64_t n_blocks,
                                      uint8_t *slots, uint32_t *sizes, int32_t *status)
{
    const ModelTable mt = model_table(kNsym, freqs, n_models);
    const LanePlan pl = models_plan(f, c, max_block_len, force_wide_table, mt);
    std::vector<uint8_t> magic = build_magic(pl);
    LaneEncJob job;
    job.in = in; job.in_off = in_off; job.n_blocks = n_blocks;
    job.slots = slots; job.slot_stride = pl.slot_stride; job.sizes = sizes; job.status = status;
    job.magic = magic.empty() ? nullptr : magic.data(); job.f = pl.f; job.c = pl.c;
    job.one = pl.c <= 32 ? 1u << (32 - pl.c) : 0u;
    job.tcap = (uint32_t)(((uint64_t)1 << pl.f) - 1 - kNsym);      // of the job's own (fresh) start model
    job.init_tree = nullptr; job.count0 = kNsym; job.eof_freq = 1;
    job.models = mt.on ? mt.bm(block_model) : BlockModels{};
    job.gf_m = pl.gf_m; job.gf_sh = pl.gf_sh;
#define RUN_AL(TW, FULL) \
    (pl.cls == kWideD && pl.c == 32 ? run_grid(encode_lane_al_kernel<TW, kWideD, FULL, true>, job, n_blocks) : \
     pl.cls == kWideD  ? run_grid(encode_lane_al_kernel<TW, kWideD, FULL, false>, job, n_blocks) : \
     pl.cls == kNarrow ? run_grid(encode_lane_al_kernel<TW, kNarrow, FULL, false>, job, n_blocks) : \
     pl.c == 32        ? run_grid(encode_lane_al_kernel<TW, kWide, FULL, true>, job, n_blocks) : \
                         run_grid(encode_lane_al_kernel<TW, kWide, FULL, false>, job, n_blocks))
    if (!pl.aligned && pl.wide_table) run_grid(encode_lane_kernel<uint32_t, kHuge>, job, n_blocks);
    else if (!pl.aligned) run_grid(encode_lane_kernel<uint16_t, kHuge>, job, n_blocks);
    else if (pl.wide_table) RUN_AL(uint32_t, true);
    else if (pl.full_table) RUN_AL(uint16_t, true);
    else RUN_AL(uint16_t, false);
#undef RUN_AL
    return 0;
}

extern "C" int emu_decode_lane_models(uint32_t f, uint32_t c, uint64_t max_block_len, int force_wide_table,
                                      const uint32_t *freqs, uint32_t n_models, const uint32_t *block_model,
                                      const uint8_t *comp, const uint64_t *comp_off, uint64_t n_blocks,
                                      uint8_t *raw, const uint64_t *raw_off, uint64_t *raw_len,
                                      uint64_t *consumed, int32_t *status)
{
    const ModelTable mt = model_table(kNsym, freqs, n_models);
    const LanePlan pl = models_plan(f, c, max_block_len, force_wide_table, mt);
    std::vector<uint8_t> magic = build_magic(pl);
    LaneDecJob job;
    job.comp = comp; job.comp_off = comp_off; job.n_blocks = n_blocks;
    job.raw = raw; job.raw_off = raw_off; job.raw_len = raw_len; job.consumed = consumed;
    job.status = status; job.magic = magic.empty() ? nullptr : magic.data(); job.f = pl.f; job.c = pl.c;
    job.one = pl.c <= 32 ? 1u << (32 - pl.c) : 0u;
    job.tcap = (uint32_t)(((uint64_t)1 << pl.f) - 1 - kNsym);      // of the job's own (fresh) start model
    job.init_tree = nullptr; job.count0 = kNsym; job.eof_freq = 1;
    job.models = mt.on ? mt.bm(block_model) : BlockModels{};
    job.gf_m = pl.gf_m; job.gf_sh = pl.gf_sh;
#define RUN_AL(TW, FULL) \
    (pl.cls == kWideD && pl.c == 32 ? run_grid(decode_lane_al_kernel<TW, kWideD, FULL, true, false>, job, n_blocks) : \
     pl.cls == kWideD  ? run_grid(decode_lane_al_kernel<TW, kWideD, FULL, false, false>, job, n_blocks) : \
     pl.cls == kNarrow && pl.c <= 16 ? run_grid(decode_lane_al_kernel<TW, kNarrow, FULL, false, true>, job, n_blocks) : \
     pl.cls == kNarrow ? run_grid(decode_lane_al_kernel<TW, kNarrow, FULL, false, false>, job, n_blocks) : \
     pl.c == 32        ? run_grid(decode_lane_al_kernel<TW, kWide, FULL, true, false>, job, n_blocks) : \
                         run_grid(decode_lane_al_kernel<TW, kWide, FULL, false, false>, job, n_blocks))
    if (!pl.aligned && pl.wide_table) run_grid(decode_lane_kernel<uint32_t, kHuge>, job, n_blocks);
    else if (!pl.aligned) run_grid(decode_lane_kernel<uint16_t, kHuge>, job, n_blocks);
    else if (pl.wide_table) RUN_AL(uint32_t, true);
    else if (pl.full_table) RUN_AL(uint16_t, true);
    else RUN_AL(uint16_t, false);
#undef RUN_AL
    return 0;
}


// ------------------------------------------------------------------ generic path (any symbol width, pre-trained models)
namespace {
struct GenericSetup { ModelTable mt; std::vector<uint32_t> tabs; std::vector<Magic64> magic; GenericJob job; };

void generic_setup(GenericSetup &g, uint32_t s, uint32_t f, uint32_t c, const uint32_t *freqs, uint32_t n_models,
                   const uint32_t *block_model, uint32_t n_threads, uint64_t max_bytes)
{
    const uint32_t nsym = (1u << s) + 1;
    g.mt = model_table(nsym, freqs, n_models);
    g.tabs.assign((size_t)(nsym + 1) * n_threads, 0xDEADBEEFu);
    g.job = GenericJob{};
    g.job.tabs = g.tabs.data(); g.job.init_tree = g.mt.trees.data();
    g.job.models = g.mt.on ? g.mt.bm(block_model) : BlockModels{};
    g.job.s = s; g.job.f = f; g.job.c = c; g.job.n_threads = n_threads;
    // reciprocals of every total a block can reach (as prepare_models of redux_capi.cu sizes them)
    const uint64_t lo = g.mt.min_total(), hi = g.mt.max_total();
    const uint64_t fmax = ((uint64_t)1 << f) - 1, syms = max_bytes * 8 / s + 1;
    const uint64_t top = fmax < hi + syms ? fmax : hi + syms;
    g.magic.resize((size_t)(top - lo + 2));
    for (size_t i = 0; i < g.magic.size(); ++i) g.magic[i] = make_magic65(lo + i);
    g.job.magic = g.magic.data(); g.job.magic_len = (uint32_t)g.magic.size(); g.job.init_total = (uint32_t)lo;
}

template <typename K>
void run_generic(K kernel, const GenericJob &job)
{
    blockDim.x = kGenericThreads; gridDim.x = job.n_threads / kGenericThreads;
    for (uint32_t b = 0; b < gridDim.x; ++b)
        for (uint32_t t = 0; t < (uint32_t)kGenericThreads; ++t) { blockIdx.x = b; threadIdx.x = t; kernel(job); }
}
}  // namespace

// n_threads: multiple of 128; fewer threads than blocks makes threads code several blocks in turn.  freqs / n_models /
// block_model as for emu_encode_lane_models (rows of symbol_count frequencies).
extern "C" int emu_encode_generic_models(uint32_t s, uint32_t f, uint32_t c, const uint32_t *freqs, uint32_t n_models,
                                         const uint32_t *block_model, uint32_t n_threads,
                                         const uint8_t *in, const uint64_t *in_off, uint64_t n_blocks,
                                         uint8_t *slots, uint64_t slot_stride, uint32_t *sizes, int32_t *status)
{
    GenericSetup g;
    uint64_t max_bytes = 0;
    for (uint64_t i = 0; i < n_blocks; ++i) max_bytes = std::max<uint64_t>(max_bytes, in_off[i + 1] - in_off[i]);
    generic_setup(g, s, f, c, freqs, n_models, block_model, n_threads, max_bytes);
    g.job.in = in; g.job.in_off = in_off; g.job.n_blocks = n_blocks;
    g.job.slots = slots; g.job.slot_stride = slot_stride; g.job.sizes = sizes; g.job.status = status;
    run_generic(encode_generic_kernel, g.job);
    return 0;
}


extern "C" int emu_decode_generic_models(uint32_t s, uint32_t f, uint32_t c, const uint32_t *freqs, uint32_t n_models,
                                         const uint32_t *block_model, uint32_t n_threads,
                                         const uint8_t *comp, const uint64_t *comp_off, uint64_t n_blocks,
                                         uint8_t *raw, const uint64_t *raw_off, uint64_t *raw_len, uint64_t *consumed,
                                         int32_t *status)
{
    GenericSetup g;
    uint64_t max_bytes = 0;
    for (uint64_t i = 0; i < n_blocks; ++i) max_bytes = std::max<uint64_t>(max_bytes, raw_off[i + 1] - raw_off[i]);
    generic_setup(g, s, f, c, freqs, n_models, block_model, n_threads, max_bytes);
    g.job.in = comp; g.job.in_off = comp_off; g.job.n_blocks = n_blocks;
    g.job.raw = raw; g.job.raw_off = raw_off; g.job.raw_len = raw_len; g.job.consumed = consumed; g.job.status = status;
    run_generic(decode_generic_kernel, g.job);
    return 0;
}

