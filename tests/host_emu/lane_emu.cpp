// lane_emu.cpp -- TEST INFRASTRUCTURE: runs the lane kernels of redux_b200/csrc/redux_lane_codec.cuh on
// the CPU, thread by thread, through tests/host_emu/cuda_shim.h (see there for why that is exact).
// Built by tests/test_host_emu.py with g++; compared there against the oracle.  Not part of the product.
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
}

namespace rdx {
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

extern "C" uint64_t emu_slot_stride(uint32_t f, uint32_t c, uint64_t max_block_len)
{
    return lane_plan(f, c, max_block_len).slot_stride;
}

// The front end's lane_plan (the same header): out = {cls, wide_table, full_table, aligned, tcap}.
extern "C" void emu_lane_plan(uint32_t f, uint32_t c, uint64_t max_block_len, uint32_t count0, int pretrained, uint32_t *out)
{
    const LanePlan pl = lane_plan(f, c, max_block_len, count0, pretrained != 0);
    out[0] = (uint32_t)pl.cls; out[1] = pl.wide_table; out[2] = pl.full_table; out[3] = pl.aligned; out[4] = pl.tcap;
}

// force_wide_table: -1 = as the front end would choose, 0 = u16 entries, 1 = u32 entries
namespace {
// start state of a trained byte model for the tuned lane kernels: tree[0..257], total, EOF frequency
struct LaneStart { std::vector<uint32_t> tree; uint32_t count0 = kNsym, eof_freq = 1; bool on = false; };
LaneStart lane_start(const uint32_t *freq)
{
    LaneStart st;
    if (!freq) return st;
    st.on = true;
    st.tree.assign(kNsym + 1, 0);
    blockDim.x = 256; gridDim.x = 2;
    for (uint32_t b = 0; b < 2; ++b)
        for (uint32_t t = 0; t < 256; ++t) { blockIdx.x = b; threadIdx.x = t; build_tree_kernel(freq, kNsym, st.tree.data()); }
    st.count0 = 0;
    for (uint32_t i = 0; i < kNsym; ++i) st.count0 += freq[i];
    st.eof_freq = freq[kEof];
    return st;
}
const void *shift_magic(const LanePlan &pl, const std::vector<uint8_t> &magic, uint32_t count0)
{
    if (magic.empty()) return nullptr;
    return magic.data() + (size_t)(count0 - kNsym) * (pl.cls == kNarrow ? sizeof(Magic32) : pl.cls == kWideD ? sizeof(MagicD) : sizeof(Magic64));
}
}  // namespace

extern "C" int emu_encode_lane_ex(uint32_t f, uint32_t c, uint64_t max_block_len, int force_wide_table, const uint32_t *freq,
                                  const uint8_t *in, const uint64_t *in_off, uint64_t n_blocks,
                                  uint8_t *slots, uint32_t *sizes, int32_t *status)
{
    const LaneStart st0 = lane_start(freq);
    LanePlan pl = lane_plan(f, c, max_block_len, st0.count0, st0.on);
    if (force_wide_table >= 0) { pl.wide_table = force_wide_table != 0; if (pl.wide_table) pl.full_table = true; }
    std::vector<uint8_t> magic = build_magic(pl);
    LaneEncJob job;
    job.in = in; job.in_off = in_off; job.n_blocks = n_blocks;
    job.slots = slots; job.slot_stride = pl.slot_stride; job.sizes = sizes; job.status = status;
    job.magic = shift_magic(pl, magic, st0.count0); job.f = pl.f; job.c = pl.c; job.tcap = pl.tcap;
    job.one = pl.c <= 32 ? 1u << (32 - pl.c) : 0u;
    job.init_tree = st0.on ? st0.tree.data() : nullptr; job.count0 = st0.count0; job.eof_freq = st0.eof_freq;
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

extern "C" int emu_encode_lane(uint32_t f, uint32_t c, uint64_t max_block_len, int force_wide_table,
                               const uint8_t *in, const uint64_t *in_off, uint64_t n_blocks,
                               uint8_t *slots, uint32_t *sizes, int32_t *status)
{
    return emu_encode_lane_ex(f, c, max_block_len, force_wide_table, nullptr, in, in_off, n_blocks, slots, sizes, status);
}

extern "C" int emu_decode_lane_ex(uint32_t f, uint32_t c, uint64_t max_block_len, int force_wide_table, const uint32_t *freq,
                                  const uint8_t *comp, const uint64_t *comp_off, uint64_t n_blocks,
                                  uint8_t *raw, const uint64_t *raw_off, uint64_t *raw_len,
                                  uint64_t *consumed, int32_t *status)
{
    const LaneStart st0 = lane_start(freq);
    LanePlan pl = lane_plan(f, c, max_block_len, st0.count0, st0.on);
    if (force_wide_table >= 0) { pl.wide_table = force_wide_table != 0; if (pl.wide_table) pl.full_table = true; }
    std::vector<uint8_t> magic = build_magic(pl);
    LaneDecJob job;
    job.comp = comp; job.comp_off = comp_off; job.n_blocks = n_blocks;
    job.raw = raw; job.raw_off = raw_off; job.raw_len = raw_len; job.consumed = consumed;
    job.status = status; job.magic = shift_magic(pl, magic, st0.count0); job.f = pl.f; job.c = pl.c; job.tcap = pl.tcap;
    job.one = pl.c <= 32 ? 1u << (32 - pl.c) : 0u;
    job.init_tree = st0.on ? st0.tree.data() : nullptr; job.count0 = st0.count0; job.eof_freq = st0.eof_freq;
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

extern "C" int emu_decode_lane(uint32_t f, uint32_t c, uint64_t max_block_len, int force_wide_table,
                               const uint8_t *comp, const uint64_t *comp_off, uint64_t n_blocks,
                               uint8_t *raw, const uint64_t *raw_off, uint64_t *raw_len,
                               uint64_t *consumed, int32_t *status)
{
    return emu_decode_lane_ex(f, c, max_block_len, force_wide_table, nullptr, comp, comp_off, n_blocks, raw, raw_off,
                              raw_len, consumed, status);
}

// One coder step of the tuned kernels on an arbitrary (low, high) state, for the closed-form-vs-loop test.
// Returns the shift count; *bits / *nbits = what the step appended to an empty packer (pending run 0 before).
extern "C" uint32_t emu_step_al(uint32_t c, uint32_t f, uint32_t low, uint32_t high, uint32_t cl, uint32_t ch,
                                uint32_t count, uint32_t *new_low, uint32_t *new_high, uint64_t *bits,
                                uint32_t *nbits, uint32_t *pend_after)
{
    alignas(16) uint8_t slot[64] = {0};
    BitSink2 sink;
    sink.init(slot);
    const uint32_t sh = 32 - c, one = 1u << sh;
    uint32_t L = low << sh, H = (high << sh) | (one - 1u), pend = 0, n;
    const Magic64 g = make_magic64(count, f + c);
    if (c == 32) n = encode_step_al<kWide, true>(L, H, pend, sink, cl, ch, count, g, sh, one);
    else         n = encode_step_al<kWide, false>(L, H, pend, sink, cl, ch, count, g, sh, one);
    *new_low = L >> sh; *new_high = H >> sh;
    // whole words already stored + the accumulator remainder
    uint64_t v = 0;
    for (uint32_t i = 0; i < sink.wi; ++i) v = (v << 32) | __byte_perm(sink.w0[i], 0, 0x0123);
    v = (v << sink.nb) | (sink.acc & ((sink.nb ? (1ull << sink.nb) : 1ull) - 1));
    *bits = v; *nbits = sink.wi * 32 + sink.nb; *pend_after = pend;
    return n;
}

// The bit packer's pair path against its one-symbol path: a sequence of n codes (bits[i], n1[i], k[i]) from pending
// count pend0, appended pairwise by put_pair (an odd last one by put_code) into out_pair and one by one by put_code into
// out_single.  Returns the byte count of out_pair; *same = 1 when the bytes, lengths and final pending counts agree.
extern "C" uint32_t emu_put_pairs(const uint32_t *bits, const uint32_t *n1, const uint32_t *k, uint32_t n, uint32_t pend0,
                                  uint8_t *out_pair, uint8_t *out_single, int *same)
{
    BitSink2 a, b;
    a.init(out_pair); b.init(out_single);
    uint32_t pa = pend0, pb = pend0;
    for (uint32_t i = 0; i + 1 < n; i += 2) {
        BitSink2::Code A{bits[i], n1[i], k[i]}, B{bits[i + 1], n1[i + 1], k[i + 1]};
        pa = a.put_pair(A, B, pa);
    }
    if (n & 1) pa = a.put_code(bits[n - 1], n1[n - 1], pa, k[n - 1]);
    for (uint32_t i = 0; i < n; ++i) pb = b.put_code(bits[i], n1[i], pb, k[i]);
    const uint32_t la = a.finish(), lb = b.finish();
    *same = la == lb && pa == pb && memcmp(out_pair, out_single, la) == 0;
    return la;
}

// ------------------------------------------------------------------ generic path (any symbol width, pre-trained models)
namespace {
struct GenericSetup { std::vector<uint32_t> init, tabs; std::vector<Magic64> magic; GenericJob job; };

void generic_setup(GenericSetup &g, uint32_t s, uint32_t f, uint32_t c, const uint32_t *freq, uint32_t n_threads,
                   uint64_t max_bytes)
{
    const uint32_t nsym = (1u << s) + 1;
    g.init.assign(nsym + 1, 0);
    blockDim.x = 256; gridDim.x = (nsym + 1 + 255) / 256;
    for (uint32_t b = 0; b < gridDim.x; ++b)
        for (uint32_t t = 0; t < 256; ++t) { blockIdx.x = b; threadIdx.x = t; build_tree_kernel(freq, nsym, g.init.data()); }
    uint64_t total = 0;
    for (uint32_t i = 0; i < nsym; ++i) total += freq ? freq[i] : 1u;
    g.tabs.assign((size_t)(nsym + 1) * n_threads, 0xDEADBEEFu);
    g.job = GenericJob{};
    g.job.tabs = g.tabs.data(); g.job.init_tree = g.init.data(); g.job.init_total = (uint32_t)total;
    g.job.s = s; g.job.f = f; g.job.c = c; g.job.n_threads = n_threads;
    // reciprocals of every total a block can reach (as prepare_generic of redux_capi.cu sizes them)
    const uint64_t fmax = ((uint64_t)1 << f) - 1, syms = max_bytes * 8 / s + 1;
    const uint64_t top = fmax < total + syms ? fmax : total + syms;
    g.magic.resize((size_t)(top - total + 2));
    for (size_t i = 0; i < g.magic.size(); ++i) g.magic[i] = make_magic65(total + i);
    g.job.magic = g.magic.data(); g.job.magic_len = (uint32_t)g.magic.size();
}

template <typename K>
void run_generic(K kernel, const GenericJob &job)
{
    blockDim.x = kGenericThreads; gridDim.x = job.n_threads / kGenericThreads;
    for (uint32_t b = 0; b < gridDim.x; ++b)
        for (uint32_t t = 0; t < (uint32_t)kGenericThreads; ++t) { blockIdx.x = b; threadIdx.x = t; kernel(job); }
}
}  // namespace

// n_threads: multiple of 128; fewer threads than blocks makes threads code several blocks in turn
extern "C" int emu_encode_generic(uint32_t s, uint32_t f, uint32_t c, const uint32_t *freq, uint32_t n_threads,
                                  const uint8_t *in, const uint64_t *in_off, uint64_t n_blocks,
                                  uint8_t *slots, uint64_t slot_stride, uint32_t *sizes, int32_t *status)
{
    GenericSetup g;
    uint64_t max_bytes = 0;
    for (uint64_t i = 0; i < n_blocks; ++i) max_bytes = std::max<uint64_t>(max_bytes, in_off[i + 1] - in_off[i]);
    generic_setup(g, s, f, c, freq, n_threads, max_bytes);
    g.job.in = in; g.job.in_off = in_off; g.job.n_blocks = n_blocks;
    g.job.slots = slots; g.job.slot_stride = slot_stride; g.job.sizes = sizes; g.job.status = status;
    run_generic(encode_generic_kernel, g.job);
    return 0;
}

extern "C" int emu_decode_generic(uint32_t s, uint32_t f, uint32_t c, const uint32_t *freq, uint32_t n_threads,
                                  const uint8_t *comp, const uint64_t *comp_off, uint64_t n_blocks,
                                  uint8_t *raw, const uint64_t *raw_off, uint64_t *raw_len, uint64_t *consumed,
                                  int32_t *status)
{
    GenericSetup g;
    uint64_t max_bytes = 0;
    for (uint64_t i = 0; i < n_blocks; ++i) max_bytes = std::max<uint64_t>(max_bytes, raw_off[i + 1] - raw_off[i]);
    generic_setup(g, s, f, c, freq, n_threads, max_bytes);
    g.job.in = comp; g.job.in_off = comp_off; g.job.n_blocks = n_blocks;
    g.job.raw = raw; g.job.raw_off = raw_off; g.job.raw_len = raw_len; g.job.consumed = consumed; g.job.status = status;
    run_generic(decode_generic_kernel, g.job);
    return 0;
}
