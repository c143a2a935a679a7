// redux_capi.cu -- C ABI (include/redux_b200.h) + the block-batching host front end.
//
// Replaces, for in-memory streams, redux::compress / redux::decompress (src/lib.rs:102-120) and
// the constructors that feed them (src/model/mod.rs:63, adaptive_linear.rs:21, adaptive_tree.rs:36).
// There is deliberately no CPU path in this file: without a CUDA device every computing entry
// point returns REDUX_CUDA_ERROR.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <atomic>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/redux_b200.h"
#include "redux_batch_kernels.cuh"
#include "redux_common.cuh"
#include "redux_lane_codec.cuh"
#include "redux_lane_al.cuh"
#include "redux_generic_codec.cuh"
#include "redux_warp_codec.cuh"
#include "redux_split_encoder.cuh"

using namespace rdx;

// The pipelined host-buffer API keeps ~18 streams busy per device.  CUDA multiplexes streams onto
// CUDA_DEVICE_MAX_CONNECTIONS hardware queues (default 8); streams that share a queue serialise in
// submission order, which measured as three chunks of sixteen stalling ~30 ms behind unrelated copies
// (profiles/r01_e2e_pipeline.md).  The variable is read when the process creates its first CUDA context, and
// it is process-wide, so the library does NOT touch it on its own (round 1 did, from a load-time constructor:
// a hidden side effect on the embedding application).  redux_process_init() is the explicit, optional form.
extern "C" int redux_process_init(void)
{
    const char *cur = std::getenv("CUDA_DEVICE_MAX_CONNECTIONS");
    if (cur) return std::atoi(cur);                       // the application's own setting wins
    setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
    return 32;
}

namespace {

// Every coder kernel the dispatcher can launch, each listed once: its KernelId (redux_debug_launched_kernels), its
// name, and for the lane and warp kernels the instantiation and (lane kernels) the table entry type that sizes its
// dynamic shared memory.  Enum, names, shared-memory limits and the launch switches below are generated from these
// lists.  Lane kernels: <table entry type, class, full tree values, code_bits == 32[, staged window refill]>; NARROW
// (c + f <= 30) implies at most 16,126 updates, so u16 entries with full values; plain WIDE (totals reach 349,525)
// always takes u32 entries (lane_plan).
#define RDX_LANE_ENCODERS(X) \
    X(kEncNarrow,          "encode_lane_al<u16,Narrow,full,!c32>",     (encode_lane_al_kernel<uint16_t, kNarrow, true, false>), uint16_t)        \
    X(kEncWideU32,         "encode_lane_al<u32,Wide,full,!c32>",       (encode_lane_al_kernel<uint32_t, kWide, true, false>), uint32_t)          \
    X(kEncWideU32C32,      "encode_lane_al<u32,Wide,full,c32>",        (encode_lane_al_kernel<uint32_t, kWide, true, true>), uint32_t)           \
    X(kEncWideDU32,        "encode_lane_al<u32,WideD,full,!c32>",      (encode_lane_al_kernel<uint32_t, kWideD, true, false>), uint32_t)         \
    X(kEncWideDU16Full,    "encode_lane_al<u16,WideD,full,!c32>",      (encode_lane_al_kernel<uint16_t, kWideD, true, false>), uint16_t)         \
    X(kEncWideDU16,        "encode_lane_al<u16,WideD,!full,!c32>",     (encode_lane_al_kernel<uint16_t, kWideD, false, false>), uint16_t)        \
    X(kEncWideDU32C32,     "encode_lane_al<u32,WideD,full,c32>",       (encode_lane_al_kernel<uint32_t, kWideD, true, true>), uint32_t)          \
    X(kEncWideDU16FullC32, "encode_lane_al<u16,WideD,full,c32>",       (encode_lane_al_kernel<uint16_t, kWideD, true, true>), uint16_t)          \
    X(kEncWideDU16C32,     "encode_lane_al<u16,WideD,!full,c32>",      (encode_lane_al_kernel<uint16_t, kWideD, false, true>), uint16_t)         \
    X(kEncHugeU16,         "encode_lane<u16,Huge>",                    (encode_lane_kernel<uint16_t, kHuge>), uint16_t)                                  \
    X(kEncHugeU32,         "encode_lane<u32,Huge>",                    (encode_lane_kernel<uint32_t, kHuge>), uint32_t)
// The narrow decoder comes twice: code_bits <= 16 runs the STAGED window refill (redux_lane_al.cuh, BitWindow).
#define RDX_LANE_DECODERS(X) \
    X(kDecNarrowStg,       "decode_lane_al<u16,Narrow,full,!c32,stg>", (decode_lane_al_kernel<uint16_t, kNarrow, true, false, true>), uint16_t)   \
    X(kDecNarrow,          "decode_lane_al<u16,Narrow,full,!c32>",     (decode_lane_al_kernel<uint16_t, kNarrow, true, false, false>), uint16_t)  \
    X(kDecWideU32,         "decode_lane_al<u32,Wide,full,!c32>",       (decode_lane_al_kernel<uint32_t, kWide, true, false, false>), uint32_t)    \
    X(kDecWideU32C32,      "decode_lane_al<u32,Wide,full,c32>",        (decode_lane_al_kernel<uint32_t, kWide, true, true, false>), uint32_t)     \
    X(kDecWideDU32,        "decode_lane_al<u32,WideD,full,!c32>",      (decode_lane_al_kernel<uint32_t, kWideD, true, false, false>), uint32_t)   \
    X(kDecWideDU16Full,    "decode_lane_al<u16,WideD,full,!c32>",      (decode_lane_al_kernel<uint16_t, kWideD, true, false, false>), uint16_t)   \
    X(kDecWideDU16,        "decode_lane_al<u16,WideD,!full,!c32>",     (decode_lane_al_kernel<uint16_t, kWideD, false, false, false>), uint16_t)  \
    X(kDecWideDU32C32,     "decode_lane_al<u32,WideD,full,c32>",       (decode_lane_al_kernel<uint32_t, kWideD, true, true, false>), uint32_t)    \
    X(kDecWideDU16FullC32, "decode_lane_al<u16,WideD,full,c32>",       (decode_lane_al_kernel<uint16_t, kWideD, true, true, false>), uint16_t)    \
    X(kDecWideDU16C32,     "decode_lane_al<u16,WideD,!full,c32>",      (decode_lane_al_kernel<uint16_t, kWideD, false, true, false>), uint16_t)   \
    X(kDecHugeU16,         "decode_lane<u16,Huge>",                    (decode_lane_kernel<uint16_t, kHuge>), uint16_t)                                  \
    X(kDecHugeU32,         "decode_lane<u32,Huge>",                    (decode_lane_kernel<uint32_t, kHuge>), uint32_t)
#define RDX_WARP_ENCODERS(X) \
    X(kEncWarpNarrow,      "encode_warp<Narrow>",                      encode_warp_kernel<kNarrow>)                  \
    X(kEncWarpWide,        "encode_warp<Wide>",                        encode_warp_kernel<kWide>)                    \
    X(kEncWarpHuge,        "encode_warp<Huge>",                        encode_warp_kernel<kHuge>)
#define RDX_WARP_DECODERS(X) \
    X(kDecWarpNarrow,      "decode_warp_al<Narrow,!c32>",              (decode_warp_al_kernel<kNarrow, false>))      \
    X(kDecWarpWide,        "decode_warp_al<Wide,!c32>",                (decode_warp_al_kernel<kWide, false>))        \
    X(kDecWarpWideC32,     "decode_warp_al<Wide,c32>",                 (decode_warp_al_kernel<kWide, true>))         \
    X(kDecWarpHuge,        "decode_warp<Huge>",                        decode_warp_kernel<kHuge>)
// Launched by hand (their launch shapes differ): the split coder and the generic kernels, whose Fenwick columns are in
// shared memory (symbol_bits <= kGenericSmemSymbolBits) or in global memory.
#define RDX_OTHER_KERNELS(X) \
    X(kSplitNarrow,        "split_coder<Narrow,!c32>")                   \
    X(kSplitWide,          "split_coder<Wide,!c32>")                     \
    X(kSplitWideC32,       "split_coder<Wide,c32>")                      \
    X(kEncGenericSmem,     "encode_generic<smem>")                       \
    X(kEncGenericGlobal,   "encode_generic<global>")                     \
    X(kDecGenericSmem,     "decode_generic<smem>")                       \
    X(kDecGenericGlobal,   "decode_generic<global>")
#define RDX_ALL_KERNELS(X) \
    RDX_LANE_ENCODERS(X) RDX_LANE_DECODERS(X) RDX_WARP_ENCODERS(X) RDX_WARP_DECODERS(X) RDX_OTHER_KERNELS(X)
#define RDX_KERNEL_ENUM(id, ...) id,
enum KernelId : int { RDX_ALL_KERNELS(RDX_KERNEL_ENUM) kKernelIdCount };
#undef RDX_KERNEL_ENUM
static_assert(kKernelIdCount <= 64, "the launched-kernel mask is 64 bits wide");

struct MagicEntry { int cls; uint32_t nbits; uint32_t len; void *ptr; };

// Grow-only device buffer.
struct DevBuf {
    void *p = nullptr; size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaError_t e = cudaFree(p); p = nullptr; cap = 0; if (e != cudaSuccess) return e; }
        size_t want = bytes + (bytes >> 3);          // 12.5% headroom against regrowth
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { (void)cudaGetLastError(); e = cudaMalloc(&p, bytes); want = bytes; }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// Grow-only pinned host buffer (small bookkeeping arrays of the pipelined host API).
struct HostBuf {
    void *p = nullptr; size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        cudaError_t e = cudaHostAlloc(&p, bytes + (bytes >> 2), cudaHostAllocDefault);
        if (e == cudaSuccess) cap = bytes + (bytes >> 2);
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

constexpr int kPipeStreams = 16;          // one compute stream per chunk in flight (host-buffer API)

// ------------------------------------------------------------------ pageable host memory: library-side staging
// The crate's callers hold plain Vec<u8>s (src/lib.rs:102-120 streams through io::Read / io::Write;
// INTEGRATION.md lands that in pageable memory).  cudaMemcpyAsync on pageable memory is staged by the driver through
// one bounce buffer on the CALLING thread, synchronously: the chunk pipeline of the host-buffer API collapses into
// copy, compute, copy one after the other (measured 3.4 GB/s end to end against 21.7 GB/s from pinned buffers,
// profiles/r02_bench_default.json).  When a caller's buffer is neither pinned nor registered the library therefore
// stages it itself: a few host threads copy piece after piece between the caller's memory and a small ring of
// pinned slots, and the asynchronous copies run between the ring and the device, so host copies, PCIe transfers in
// both directions and the kernels overlap as they do from pinned buffers.
class CopyPool {
    struct Task { uint8_t *dst; const uint8_t *src; size_t n; int *left; };
    std::vector<std::thread> workers;
    std::deque<Task> q;
    std::mutex m;
    std::condition_variable cv_work, cv_done;
    bool stop = false;

    void run() {
        std::unique_lock<std::mutex> l(m);
        for (;;) {
            cv_work.wait(l, [&] { return stop || !q.empty(); });
            if (q.empty()) return;                          // stop requested and nothing left
            Task t = q.front(); q.pop_front();
            l.unlock();
            std::memcpy(t.dst, t.src, t.n);
            l.lock();
            if (--*t.left == 0) cv_done.notify_all();
        }
    }
public:
    explicit CopyPool(int n_workers) { for (int i = 0; i < n_workers; ++i) workers.emplace_back([this] { run(); }); }
    ~CopyPool() {
        { std::lock_guard<std::mutex> l(m); stop = true; }
        cv_work.notify_all();
        for (auto &t : workers) t.join();
    }
    // memcpy cut into one slice per thread (the caller copies a slice itself); returns when all of it has landed.
    // Safe to call from several threads at once.
    void copy(void *dst_, const void *src_, size_t n) {
        uint8_t *dst = (uint8_t *)dst_; const uint8_t *src = (const uint8_t *)src_;
        constexpr size_t kMinSlice = 256 << 10;
        size_t parts = std::min<size_t>(workers.size() + 1, (n + kMinSlice - 1) / kMinSlice);
        if (parts <= 1) { std::memcpy(dst, src, n); return; }
        const size_t per = ((n + parts - 1) / parts + 63) & ~(size_t)63;
        int left = 0;
        {
            std::lock_guard<std::mutex> l(m);
            for (size_t a = per; a < n; a += per) { q.push_back({dst + a, src + a, std::min(per, n - a), &left}); ++left; }
        }
        cv_work.notify_all();
        std::memcpy(dst, src, std::min(per, n));
        std::unique_lock<std::mutex> l(m);
        cv_done.wait(l, [&] { return left == 0; });
    }
};

// Ring of pinned slots between the caller's pageable memory and one copy stream; a slot's event says when the
// asynchronous copy that used it last has finished.
struct StageRing {
    uint8_t *buf = nullptr; size_t piece = 0; int n = 0;
    std::vector<cudaEvent_t> ev;
    std::vector<char> recorded;
    cudaError_t ensure(size_t piece_bytes, int slots) {
        if (buf && piece == piece_bytes && n == slots) return cudaSuccess;
        release();
        cudaError_t e = cudaHostAlloc((void **)&buf, piece_bytes * (size_t)slots, cudaHostAllocDefault);
        if (e != cudaSuccess) { buf = nullptr; return e; }
        piece = piece_bytes; n = slots;
        ev.assign((size_t)slots, nullptr); recorded.assign((size_t)slots, 0);
        for (auto &x : ev) if ((e = cudaEventCreateWithFlags(&x, cudaEventDisableTiming)) != cudaSuccess) return e;
        return cudaSuccess;
    }
    void release() {
        for (auto x : ev) if (x) cudaEventDestroy(x);
        ev.clear(); recorded.clear();
        if (buf) cudaFreeHost(buf);
        buf = nullptr; piece = 0; n = 0;
    }
    uint8_t *slot(int i) const { return buf + (size_t)i * piece; }
};

// How the host-buffer calls treat pageable memory (redux_ctx_set_staging).
struct StagingConfig {
    int enable = 1;                       // 0: hand pageable pointers to cudaMemcpyAsync as they are
    size_t min_bytes = (size_t)8 << 20;   // smaller transfers are not worth a ring and a feeder thread
    size_t piece_bytes = (size_t)8 << 20;
    int slots = 4;
    int threads = 0;                      // copy threads; 0 = chosen from the host's core count
};

struct DeviceState {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t pipe[kPipeStreams] = {};
    cudaStream_t copy = nullptr;          // device-to-host stream of the encode pipeline
    cudaStream_t h2d = nullptr;           // host-to-device stream: input copies never queue behind kernels
    HostBuf pin_off, pin_status, pin_aux0, pin_aux1;
    DevBuf slots, sizes, flag;                 // encoder workspace
    DevBuf st_in, st_off, st_out, st_ooff, st_status, st_aux0, st_aux1, st_roff;   // host-API staging
    DevBuf split_hist, split_pairs;            // split encoder: chunk histograms, per-position ranges
    DevBuf gen_tabs, gen_init, gen_freq, gen_magic;   // generic path: Fenwick columns, start tree, uploaded frequencies, reciprocals
    uint8_t *text_lut = nullptr;
    DevBuf corpus; uint64_t corpus_len = 0;    // text-class corpus of the synthetic generator (redux_ctx_set_text_corpus)
    std::vector<MagicEntry> magics;
    bool smem_set = false;
    // The device-resident entry points share ONE workspace per device (slots, sizes, generic-path columns ...).
    // Calls may arrive on different streams, so each call first makes its stream wait for the previous call's
    // last kernel (ws_busy) and records it again when it is enqueued: at most one device call in flight per
    // device, asynchronous to the host all the same.
    cudaEvent_t ws_busy = nullptr;
    bool ws_recorded = false;
    // pinned rings of the pageable-memory path (pointers: DeviceState is copied into per-thread views)
    StageRing *ring_up = nullptr, *ring_down = nullptr;
};

}  // namespace

struct TimedSpan { cudaEvent_t a, b; int kind; int device; };

struct redux_ctx {
    std::vector<DeviceState> devs;
    int sched = REDUX_SCHED_AUTO;
    std::string last_error;
    uint64_t launches = 0;
    bool timing = false;                  // bracket every kernel with CUDA events (bench.py)
    const uint32_t *model_freq = nullptr;  // pre-trained start state of the running *_ex call (host pointer)
    std::vector<TimedSpan> spans;
    StagingConfig staging;
    CopyPool *pool = nullptr;              // created by the first call that meets pageable memory
    // bit k: kernel KernelId k was launched since the last reset (redux_debug_launched_kernels).  Atomic: the
    // per-device workers of a multi-device call OR their bits in from their own threads.
    std::atomic<uint64_t> kernels_launched{0};
    void note_kernel(int id) { kernels_launched.fetch_or((uint64_t)1 << id, std::memory_order_relaxed); }
};

namespace {

int fail(redux_ctx *ctx, int code, const char *what, cudaError_t e = cudaSuccess)
{
    if (ctx) {
        char buf[512];
        if (e != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
        else snprintf(buf, sizeof buf, "%s", what);
        ctx->last_error = buf;
    }
    return code;
}

#define CU_TRY(ctx, expr)                                                             \
    do { cudaError_t e__ = (expr);                                                    \
         if (e__ != cudaSuccess) { (void)cudaGetLastError();                          \
             return fail((ctx), REDUX_CUDA_ERROR, #expr, e__); } } while (0)

DeviceState *find_dev(redux_ctx *ctx, int device)
{
    for (auto &d : ctx->devs) if (d.device == device) return &d;
    return nullptr;
}

template <typename K>
cudaError_t allow_smem(K kernel, size_t bytes)
{
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// Dynamic shared memory of a lane kernel: one table of TW entries per warp + the pad (redux_lane_codec.cuh)
template <typename TW>
constexpr size_t lane_smem() { return (size_t)kLaneWarpsPerCta * kTabNodes * 32 * sizeof(TW) + kTabPadBytes; }

cudaError_t configure_kernels()
{
    cudaError_t e;
#define RDX_CFG(id, name, kernel, TW) if ((e = allow_smem(kernel, lane_smem<TW>())) != cudaSuccess) return e;
    RDX_LANE_ENCODERS(RDX_CFG) RDX_LANE_DECODERS(RDX_CFG)
#undef RDX_CFG
    // generic kernels: Fenwick columns of alphabets up to 7 bits in shared memory (66 KB per CTA at 7 bits)
    if ((e = allow_smem(encode_generic_kernel, generic_smem_bytes(kGenericSmemSymbolBits))) != cudaSuccess) return e;
    return allow_smem(decode_generic_kernel, generic_smem_bytes(kGenericSmemSymbolBits));
}

// Shape of one launch derived from the parameters and the longest block.
struct Plan {
    int cls; uint32_t f, c, tcap; bool wide_table; uint32_t magic_len; uint64_t slot_stride;
    bool aligned = false, full_table = false;   // see LanePlan
    uint64_t gf_m = 0; uint32_t gf_sh = 0;      // see LanePlan
    int lane_cls = kNarrow;                     // class of the tuned lane kernels (kWideD where the plan allows it)
    uint64_t gf_m_wide = 0; uint32_t gf_sh_wide = 0;   // frozen reciprocal of the plain WIDE class (warp / split paths)
    // generic path (redux_generic_codec.cuh): symbol_bits != 8 or a pre-trained model
    bool generic = false; uint32_t s = 8, gen_threads = 0, gen_total = 0;
    // byte symbols, code_bits <= 32, model trained before the call: the tuned lane kernels start from its tree
    bool pretrained = false; uint32_t count0 = kNsym, eof_freq = 1;
    uint32_t *gen_tabs = nullptr; const uint32_t *gen_init = nullptr;
    const Magic64 *gen_magic = nullptr; uint32_t gen_magic_len = 0;
    bool warp = false;      // one stream per warp (latency mapping) instead of one per lane
    bool split = false;     // encode only: parallel model phase + one-warp coder chain (redux_split_encoder.cuh)
    uint64_t max_len = 0;   // longest block of the launch
};

// REDUX_SCHED_AUTO, encode: up to this many streams the split encoder (parallel model phase + one coder warp per
// stream) beats 32 streams per warp (profiles/r02_small_batches_corpora.json, profiles/r02_underfilled.json: 512
// blocks of 64 KiB encode in 7.1 ms split vs 7.6 ms lane, 9.7 vs 12.2 ms at (8,30,32); 2,048 blocks 19.6 vs 8.3 ms).  The plain warp encoder never
// wins (29 corpus files: 31 MB/s against 62 lane and 86 split), so AUTO falls back to the lane mapping, not to it.
constexpr uint64_t kWarpAutoMaxBlocks = 512;

// One stream per warp, encode and decode: only when the caller asks for it (REDUX_SCHED_WARP / REDUX_SCHED_SPLIT; the
// split schedule decodes with the warp mapping).  REDUX_SCHED_AUTO decodes with the lane mapping: since the decoder's
// output sink is phase-free (round 2) a lane decodes every class faster than a cooperating warp at every batch size
// measured, ragged corpus batches included (profiles/r02_small_batches_corpora.json: 29 files 28.6 vs 20.0 MB/s,
// 12 x 1 MiB 51.3 vs 35.9 MB/s at (8,14,16); 15.2 vs 13.6 and 27.3 vs 24.3 MB/s at (8,30,32); one stream 4.9 vs 3.4 /
// 2.6 vs 2.3 MB/s).
bool choose_warp(const redux_ctx *ctx)
{
    return ctx->sched == REDUX_SCHED_WARP || ctx->sched == REDUX_SCHED_SPLIT;
}

// The split encoder needs 8 bytes of workspace per input position; beyond 2 GB the warp mapping is used.
constexpr uint64_t kSplitMaxPairBytes = (uint64_t)2 << 30;
bool choose_split(const redux_ctx *ctx, uint64_t n_blocks, int cls, uint64_t max_len)
{
    if (ctx->sched == REDUX_SCHED_LANE || ctx->sched == REDUX_SCHED_WARP) return false;
    if (ctx->sched == REDUX_SCHED_AUTO && n_blocks > kWarpAutoMaxBlocks) return false;
    if (cls == kHuge || max_len == 0) return false;
    const uint64_t stride = (max_len + 31) & ~(uint64_t)31;
    return n_blocks * stride * sizeof(uint2) <= kSplitMaxPairBytes;
}

int make_plan(redux_ctx *ctx, const redux_params_t *p, uint64_t max_block_len, Plan *pl)
{
    if (!p) return fail(ctx, REDUX_INVALID_INPUT, "params is NULL");
    if (!params_valid(p->symbol_bits, p->freq_bits, p->code_bits))
        return fail(ctx, REDUX_INVALID_INPUT, "Parameters::new rejects these parameters");
    if (p->symbol_bits > kGenericMaxSymbolBits)
        return fail(ctx, REDUX_UNSUPPORTED, "device path implements symbol_bits <= 16");
    if (max_block_len > 0xFFFFFFF0ull)
        return fail(ctx, REDUX_UNSUPPORTED, "blocks longer than 2^32-16 bytes are not supported");
    pl->s = p->symbol_bits;
    pl->max_len = max_block_len;
    const bool huge = arith_class(p->freq_bits, p->code_bits) == kHuge;
    pl->generic = p->symbol_bits != (uint32_t)kSymbolBits || (ctx->model_freq != nullptr && huge);
    uint64_t total0 = ((uint64_t)1 << p->symbol_bits) + 1;
    if (ctx->model_freq) {
        // the observable state of a trained reference model: every symbol at least once, total <= freq_max
        // (it starts at symbol_count and stops growing at freq_max, adaptive_tree.rs:84)
        const uint64_t nsym = total0, fmax = ((uint64_t)1 << p->freq_bits) - 1;
        total0 = 0;
        for (uint64_t i = 0; i < nsym; ++i) {
            if (ctx->model_freq[i] < 1) return fail(ctx, REDUX_INVALID_INPUT, "model frequency below 1");
            total0 += ctx->model_freq[i];
        }
        if (total0 > fmax) return fail(ctx, REDUX_INVALID_INPUT, "model total exceeds freq_max");
    }
    pl->gen_total = (uint32_t)total0;
    if (pl->generic) {
        // worst case: every coded symbol (floor(8 len / s) data symbols + EOF) emits code_bits bits
        pl->f = p->freq_bits; pl->c = p->code_bits; pl->cls = kHuge; pl->tcap = 0; pl->wide_table = true;
        pl->magic_len = 0;
        const uint64_t bound = redux_compress_bound_ex(max_block_len, p->symbol_bits, p->code_bits);
        pl->slot_stride = ((bound + 15) & ~(uint64_t)15) + 16;
        return REDUX_OK;
    }
    // (trained) tuned lane kernels: count_t = min(count0 + t, FMAX), full tree values in the table
    pl->pretrained = ctx->model_freq != nullptr;
    pl->count0 = (uint32_t)total0; pl->eof_freq = ctx->model_freq ? ctx->model_freq[kEof] : 1u;
    const LanePlan lp = lane_plan(p->freq_bits, p->code_bits, max_block_len, pl->count0, pl->pretrained);
    pl->lane_cls = lp.cls;
    pl->f = lp.f; pl->c = lp.c; pl->cls = lp.cls == kWideD ? (int)kWide : lp.cls; pl->tcap = lp.tcap; pl->wide_table = lp.wide_table;
    pl->magic_len = lp.magic_len; pl->slot_stride = lp.slot_stride;
    pl->aligned = lp.aligned; pl->full_table = lp.full_table;
    pl->gf_m = lp.gf_m; pl->gf_sh = lp.gf_sh;
    return REDUX_OK;
}

// The reciprocal table the launch will read: the tuned lane kernels of the WIDE_D class divide by double
// reciprocals, everything else on the same parameters (warp mapping, split encoder) by the 64-bit magics.
int magic_class(const Plan &pl) { return (pl.lane_cls == kWideD && !pl.warp && !pl.split) ? (int)kWideD : pl.cls; }
size_t magic_entry_size(int mcls) { return mcls == kNarrow ? sizeof(Magic32) : mcls == kWideD ? sizeof(MagicD) : sizeof(Magic64); }

int get_magic(redux_ctx *ctx, DeviceState *d, cudaStream_t stream, const Plan &pl, const void **out)
{
    *out = nullptr;
    if (pl.generic) return REDUX_OK;
    const int mcls = magic_class(pl);
    // HUGE and WIDE_D: one table serves every numerator width
    const uint32_t nbits = (mcls == kHuge || mcls == kWideD) ? 0u : pl.f + pl.c;
    for (auto &m : d->magics)
        if (m.cls == mcls && m.nbits == nbits && m.len >= pl.magic_len) { *out = m.ptr; return REDUX_OK; }
    const size_t esz = magic_entry_size(mcls);
    // + 64: split_coder_kernel prefetches whole rounds of 32 positions and may index up to 63 entries past the
    // last position it uses (values never consumed, but the reads must stay inside the allocation)
    const uint32_t len = std::max<uint32_t>(pl.magic_len, 1024) + 64;
    void *ptr = nullptr;
    CU_TRY(ctx, cudaMalloc(&ptr, esz * len));
    const uint32_t threads = 256, grid = (len + threads - 1) / threads;
    if (mcls == kNarrow)     build_magic_kernel<Magic32><<<grid, threads, 0, stream>>>((Magic32 *)ptr, len, nbits);
    else if (mcls == kWideD) build_magic_kernel<MagicD><<<grid, threads, 0, stream>>>((MagicD *)ptr, len, nbits);
    else                     build_magic_kernel<Magic64><<<grid, threads, 0, stream>>>((Magic64 *)ptr, len, nbits);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    // the table must be visible to work on any stream of this device
    CU_TRY(ctx, cudaStreamSynchronize(stream));
    d->magics.push_back({mcls, nbits, len, ptr});
    *out = ptr;
    return REDUX_OK;
}

// Generic path set-up: uploads the start frequencies (if any), builds the start tree on the device and
// sizes the per-thread Fenwick columns.  At most ~2 GB of columns; a thread codes several blocks in turn.
int prepare_generic(redux_ctx *ctx, DeviceState *d, cudaStream_t stream, const redux_params_t *p, uint64_t n_blocks, Plan *pl)
{
    if (!pl->generic && !pl->pretrained) return REDUX_OK;
    const uint32_t nsym = (1u << p->symbol_bits) + 1;
    const uint32_t *d_freq = nullptr;
    if (ctx->model_freq) {                                   // validated by make_plan
        CU_TRY(ctx, d->gen_freq.reserve(nsym * sizeof(uint32_t)));
        CU_TRY(ctx, cudaMemcpyAsync(d->gen_freq.p, ctx->model_freq, nsym * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
        d_freq = (const uint32_t *)d->gen_freq.p;
    }
    CU_TRY(ctx, d->gen_init.reserve((nsym + 1) * sizeof(uint32_t)));
    build_tree_kernel<<<(nsym + 1 + 255) / 256, 256, 0, stream>>>(d_freq, nsym, (uint32_t *)d->gen_init.p);
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    pl->gen_init = (const uint32_t *)d->gen_init.p;
    if (!pl->generic) {                                      // tuned lane kernels: only the start tree is needed
        CU_TRY(ctx, cudaStreamSynchronize(stream));
        return REDUX_OK;
    }
    // reciprocals of every total a block of this call can reach: init_total .. min(freq_max, init_total + symbols)
    {
        const uint64_t fmax = ((uint64_t)1 << p->freq_bits) - 1;
        const uint64_t syms = pl->max_len * 8 / p->symbol_bits + 1;                     // data symbols + EOF
        const uint64_t top = std::min<uint64_t>(fmax, (uint64_t)pl->gen_total + syms);
        const uint32_t len = (uint32_t)(top - pl->gen_total + 2);
        CU_TRY(ctx, d->gen_magic.reserve((size_t)len * sizeof(Magic64)));
        build_magic_kernel<Magic64><<<(len + 255) / 256, 256, 0, stream>>>((Magic64 *)d->gen_magic.p, len, 0u, pl->gen_total);
        ctx->launches++;
        CU_TRY(ctx, cudaGetLastError());
        pl->gen_magic = (const Magic64 *)d->gen_magic.p; pl->gen_magic_len = len;
    }
    const uint64_t col_bytes = (uint64_t)(nsym + 1) * sizeof(uint32_t);
    uint64_t threads = std::min<uint64_t>((n_blocks + kGenericThreads - 1) / kGenericThreads * kGenericThreads,
                                          (uint64_t)148 * 16 * kGenericThreads);
    const uint64_t budget = (uint64_t)2 << 30;
    if (threads * col_bytes > budget) threads = std::max<uint64_t>(budget / col_bytes / kGenericThreads, 1) * kGenericThreads;
    CU_TRY(ctx, d->gen_tabs.reserve(threads * col_bytes));
    // the start tree must be complete before kernels on other streams read it; the upload buffer is reused
    CU_TRY(ctx, cudaStreamSynchronize(stream));
    pl->gen_threads = (uint32_t)threads;
    pl->gen_tabs = (uint32_t *)d->gen_tabs.p;
    return REDUX_OK;
}

// Reciprocal table as the kernels index it: entry t <-> count0 + t (the table itself starts at count 257).
const void *lane_magic(const Plan &pl, const void *magic)
{
    if (!magic || !pl.pretrained) return magic;
    const size_t esz = magic_entry_size(magic_class(pl));
    return (const uint8_t *)magic + (size_t)(pl.count0 - kNsym) * esz;
}

GenericJob generic_job(const Plan &pl)
{
    GenericJob g{};
    g.tabs = pl.gen_tabs; g.init_tree = pl.gen_init; g.init_total = pl.gen_total;
    g.s = pl.s; g.f = pl.f; g.c = pl.c; g.n_threads = pl.gen_threads;
    g.magic = pl.gen_magic; g.magic_len = pl.gen_magic_len;
    return g;
}

// The fields LaneEncJob and LaneDecJob take from the plan.
template <typename J>
void set_plan_fields(J &job, const Plan &pl, const void *magic)
{
    job.magic = lane_magic(pl, magic); job.f = pl.f; job.c = pl.c; job.tcap = pl.tcap;
    job.one = pl.c <= 32 ? 1u << (32 - pl.c) : 0u;
    job.init_tree = pl.pretrained ? pl.gen_init : nullptr; job.count0 = pl.count0; job.eof_freq = pl.eof_freq;
    job.gf_m = pl.gf_m; job.gf_sh = pl.gf_sh;
}

// The lane or warp coder kernel a plan runs (the split and generic kernels are launched on their own).
KernelId pick_encoder(const Plan &pl)
{
    const bool c32 = pl.c == 32;
    if (pl.warp) return pl.cls == kNarrow ? kEncWarpNarrow : pl.cls == kWide ? kEncWarpWide : kEncWarpHuge;
    if (!pl.aligned) return pl.wide_table ? kEncHugeU32 : kEncHugeU16;
    if (pl.lane_cls == kNarrow) return kEncNarrow;
    if (pl.lane_cls == kWide) return c32 ? kEncWideU32C32 : kEncWideU32;
    if (pl.wide_table) return c32 ? kEncWideDU32C32 : kEncWideDU32;
    if (pl.full_table) return c32 ? kEncWideDU16FullC32 : kEncWideDU16Full;
    return c32 ? kEncWideDU16C32 : kEncWideDU16;
}
KernelId pick_decoder(const Plan &pl)
{
    const bool c32 = pl.c == 32;
    if (pl.warp) return pl.cls == kNarrow ? kDecWarpNarrow : pl.cls == kHuge ? kDecWarpHuge : c32 ? kDecWarpWideC32 : kDecWarpWide;
    if (!pl.aligned) return pl.wide_table ? kDecHugeU32 : kDecHugeU16;
    if (pl.lane_cls == kNarrow) return pl.c <= 16 ? kDecNarrowStg : kDecNarrow;
    if (pl.lane_cls == kWide) return c32 ? kDecWideU32C32 : kDecWideU32;
    if (pl.wide_table) return c32 ? kDecWideDU32C32 : kDecWideDU32;
    if (pl.full_table) return c32 ? kDecWideDU16FullC32 : kDecWideDU16Full;
    return c32 ? kDecWideDU16C32 : kDecWideDU16;
}

// Starts lane or warp kernel `id` on job.n_blocks streams; false if `id` is not one of them.
#define RDX_LAUNCH_LANE(id, name, kernel, TW) case id: kernel<<<lane_grid, kLaneThreads, lane_smem<TW>(), s>>>(job); return true;
#define RDX_LAUNCH_WARP(id, name, kernel) case id: kernel<<<warp_grid, kWarpCtaThreads, 0, s>>>(job); return true;
bool launch_coder(KernelId id, const LaneEncJob &job, cudaStream_t s)
{
    const uint32_t lane_grid = (uint32_t)((job.n_blocks + kLaneThreads - 1) / kLaneThreads);
    const uint32_t warp_grid = (uint32_t)((job.n_blocks + kWarpCtaWarps - 1) / kWarpCtaWarps);
    switch (id) {
    RDX_LANE_ENCODERS(RDX_LAUNCH_LANE)
    RDX_WARP_ENCODERS(RDX_LAUNCH_WARP)
    default: return false;
    }
}
bool launch_coder(KernelId id, const LaneDecJob &job, cudaStream_t s)
{
    const uint32_t lane_grid = (uint32_t)((job.n_blocks + kLaneThreads - 1) / kLaneThreads);
    const uint32_t warp_grid = (uint32_t)((job.n_blocks + kWarpCtaWarps - 1) / kWarpCtaWarps);
    switch (id) {
    RDX_LANE_DECODERS(RDX_LAUNCH_LANE)
    RDX_WARP_DECODERS(RDX_LAUNCH_WARP)
    default: return false;
    }
}
#undef RDX_LAUNCH_LANE
#undef RDX_LAUNCH_WARP

// Split encoder: model phase over all chunks of all streams, then one coder warp per stream (its KernelId in *kid).
int launch_encode_split(redux_ctx *ctx, DeviceState *d, const Plan &pl, const LaneEncJob &job, cudaStream_t s, KernelId *kid)
{
    if (!d) return fail(ctx, REDUX_INVALID_INPUT, "device is not part of this context");
    SplitJob sj;
    sj.in = job.in; sj.in_off = job.in_off; sj.n_blocks = job.n_blocks;
    sj.chunks_per_stream = (uint32_t)((pl.max_len + kSplitChunk - 1) / kSplitChunk);
    sj.pair_stride = (pl.max_len + 31) & ~(uint64_t)31;
    sj.tcap = pl.tcap;
    const uint64_t chunks = job.n_blocks * sj.chunks_per_stream;
    CU_TRY(ctx, d->split_hist.reserve(chunks * 256 * sizeof(uint32_t)));
    CU_TRY(ctx, d->split_pairs.reserve(job.n_blocks * sj.pair_stride * sizeof(uint2)));
    sj.hist = (uint32_t *)d->split_hist.p; sj.pairs = (uint2 *)d->split_pairs.p;
    split_hist_kernel<<<(uint32_t)chunks, 256, 0, s>>>(sj);
    split_scan_kernel<<<(uint32_t)job.n_blocks, 256, 0, s>>>(sj);
    split_model_kernel<<<(uint32_t)((chunks + kSplitModelWarps - 1) / kSplitModelWarps), kSplitModelWarps * 32, 0, s>>>(sj);
    const uint32_t grid = (uint32_t)job.n_blocks;
    if (pl.cls == kNarrow)   { split_coder_kernel<kNarrow, false><<<grid, 32, 0, s>>>(job, sj); *kid = kSplitNarrow; }
    else if (pl.c == 32)     { split_coder_kernel<kWide, true><<<grid, 32, 0, s>>>(job, sj);    *kid = kSplitWideC32; }
    else                     { split_coder_kernel<kWide, false><<<grid, 32, 0, s>>>(job, sj);   *kid = kSplitWide; }
    ctx->launches += 3;      // + the one counted by the caller
    return REDUX_OK;
}

int check_kind(redux_ctx *ctx, int kind)
{
    if (kind != REDUX_MODEL_LINEAR && kind != REDUX_MODEL_TREE)
        return fail(ctx, REDUX_INVALID_INPUT, "unknown model kind");
    return REDUX_OK;
}

// RAII device switch
struct DeviceGuard {
    int prev = -1; bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; (void)cudaGetLastError(); }
        if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// Brackets one kernel launch with events on the launching stream when ctx->timing is on.
struct KernelTimer {
    redux_ctx *ctx; cudaStream_t s; TimedSpan span; bool on;
    KernelTimer(redux_ctx *c, int device, cudaStream_t st, int kind) : ctx(c), s(st), on(c->timing) {
        if (!on) return;
        span.kind = kind; span.device = device;
        if (cudaEventCreate(&span.a) != cudaSuccess || cudaEventCreate(&span.b) != cudaSuccess) { on = false; return; }
        cudaEventRecord(span.a, s);
    }
    ~KernelTimer() { if (on) { cudaEventRecord(span.b, s); ctx->spans.push_back(span); } }
};

// One device call in flight per device (see DeviceState::ws_busy).
cudaError_t ws_acquire(DeviceState *d, cudaStream_t s)
{
    return d->ws_recorded ? cudaStreamWaitEvent(s, d->ws_busy, 0) : cudaSuccess;
}
cudaError_t ws_release(DeviceState *d, cudaStream_t s)
{
    cudaError_t e = cudaEventRecord(d->ws_busy, s);
    if (e == cudaSuccess) d->ws_recorded = true;
    return e;
}

}  // namespace

// =============================================================================== host arithmetic

extern "C" int redux_parameters_new(uint32_t s, uint32_t f, uint32_t c, redux_parameters_t *o)
{
    if (!params_valid(s, f, c)) return REDUX_INVALID_INPUT;        // src/model/mod.rs:64-65
    if (o) {
        o->symbol_bits = s; o->symbol_eof = (uint64_t)1 << s; o->symbol_count = ((uint64_t)1 << s) + 1;
        o->freq_bits = f;   o->freq_max = ((uint64_t)1 << f) - 1;
        o->code_bits = c;   o->code_min = 0;
        o->code_one_fourth = (uint64_t)1 << (c - 2);
        o->code_half = (uint64_t)2 << (c - 2);
        o->code_three_fourths = (uint64_t)3 << (c - 2);
        o->code_max = ((uint64_t)1 << c) - 1;
    }
    return REDUX_OK;
}

extern "C" int redux_params_supported(const redux_params_t *p)
{
    if (!p || !params_valid(p->symbol_bits, p->freq_bits, p->code_bits)) return REDUX_INVALID_INPUT;
    return p->symbol_bits <= kGenericMaxSymbolBits ? REDUX_OK : REDUX_UNSUPPORTED;
}

extern "C" const char *redux_error_string(int code)
{
    switch (code) {
    case REDUX_OK: return "OK";
    case REDUX_EOF: return "Unexpected end of file";                          // src/lib.rs:69
    case REDUX_INVALID_INPUT: return "Invalid data found while processing input";  // src/lib.rs:70
    case REDUX_IO_ERROR: return "I/O error";                                  // src/lib.rs:71
    case REDUX_CUDA_ERROR: return "CUDA error";
    case REDUX_UNSUPPORTED: return "Parameters not supported by the device path";
    case REDUX_OUT_CAPACITY: return "Output buffer too small";
    default: return "Unknown error";
    }
}

extern "C" uint64_t redux_compress_bound(uint64_t in_len, uint32_t code_bits)
{
    return ((in_len + 1) * (uint64_t)code_bits + 7) / 8;
}

extern "C" uint64_t redux_compress_bound_ex(uint64_t in_len, uint32_t symbol_bits, uint32_t code_bits)
{
    if (symbol_bits == 0) return 0;
    return ((in_len * 8 / symbol_bits + 1) * (uint64_t)code_bits + 7) / 8;
}

extern "C" int redux_debug_magic(uint64_t d, uint32_t nbits, int wide, uint64_t *magic, uint32_t *shift)
{
    if (d < 1 || d >> 32) return REDUX_INVALID_INPUT;
    if (wide == 2) { if (d < 2) return REDUX_INVALID_INPUT; Magic64 g = make_magic65(d); *magic = g.m; *shift = g.sh; return REDUX_OK; }
    if (wide == 3) {
        if (d >= kWideDMaxCount) return REDUX_INVALID_INPUT;
        union { double f; uint64_t u; } cv; cv.f = make_magicd((uint32_t)d).r; *magic = cv.u; *shift = 0; return REDUX_OK;
    }
    if (wide) { if (nbits > 62) return REDUX_INVALID_INPUT; Magic64 g = make_magic64(d, nbits); *magic = g.m; *shift = g.sh; }
    else      { if (nbits > 30) return REDUX_INVALID_INPUT; Magic32 g = make_magic32((uint32_t)d, nbits); *magic = g.m; *shift = g.sh; }
    return REDUX_OK;
}

extern "C" uint32_t redux_debug_div_by_range(uint64_t x, uint64_t range) { return div_by_range64(x, range); }

extern "C" uint64_t redux_debug_magic_divide(uint64_t n, uint64_t magic, uint32_t shift, int wide)
{
    if (wide == 2) { Magic64 g{magic, shift, 0}; return div_magic65(n, g); }
    if (wide == 3) { union { double f; uint64_t u; } cv; cv.u = magic; MagicD g; g.r = cv.f; return div_magicd(n, g); }
    if (wide) { Magic64 g{magic, shift, 0}; return div_magic64(n, g); }
    Magic32 g{(uint32_t)magic, shift};
    return div_magic32((uint32_t)n, g);
}

extern "C" void redux_debug_renorm(uint64_t low, uint64_t high, uint32_t c, uint32_t *n1, uint32_t *k,
                                   uint64_t *nl, uint64_t *nh)
{
    if (c <= 32) { Renorm<uint32_t> r = renorm<uint32_t>((uint32_t)low, (uint32_t)high, c); *n1 = r.n1; *k = r.k; *nl = r.low; *nh = r.high; }
    else         { Renorm<uint64_t> r = renorm<uint64_t>(low, high, c); *n1 = r.n1; *k = r.k; *nl = r.low; *nh = r.high; }
}

extern "C" void redux_debug_shard(uint64_t n_blocks, uint32_t n_devices, uint32_t g, uint64_t *first, uint64_t *count)
{
    // the partition rule of the host front end (make_shards below)
    const uint64_t a = n_blocks * g / n_devices, b = n_blocks * (g + 1) / n_devices;
    *first = a; *count = b - a;
}

// Resident CTAs per SM of the headline kernels (u16 tables).  The shared-memory budget is exact to the byte
// (redux_lane_codec.cuh, kTabPadBytes): anything but 2 means a change pushed a kernel over it and halved the
// number of resident streams.  Needs a device.
extern "C" int redux_debug_lane_occupancy(int *enc_ctas_per_sm, int *dec_ctas_per_sm)
{
    if (!enc_ctas_per_sm || !dec_ctas_per_sm) return REDUX_INVALID_INPUT;
    if (configure_kernels() != cudaSuccess) { (void)cudaGetLastError(); return REDUX_CUDA_ERROR; }
    const size_t s16 = (size_t)kLaneWarpsPerCta * kTabNodes * 32 * 2 + kTabPadBytes;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(enc_ctas_per_sm, encode_lane_al_kernel<uint16_t, kNarrow, true, false>,
                                                      kLaneThreads, s16) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(dec_ctas_per_sm, decode_lane_al_kernel<uint16_t, kNarrow, true, false, true>,
                                                      kLaneThreads, s16) != cudaSuccess) {
        (void)cudaGetLastError();
        return REDUX_CUDA_ERROR;
    }
    return REDUX_OK;
}

extern "C" const char *redux_debug_kernel_name(int id)
{
#define RDX_KERNEL_NAME(id, name, ...) name,
    static const char *const names[] = { RDX_ALL_KERNELS(RDX_KERNEL_NAME) };
#undef RDX_KERNEL_NAME
    return id >= 0 && id < kKernelIdCount ? names[id] : nullptr;
}

extern "C" int redux_debug_launched_kernels(redux_ctx_t *ctx, uint64_t *mask, int reset)
{
    if (!ctx || !mask) return REDUX_INVALID_INPUT;
    *mask = reset ? ctx->kernels_launched.exchange(0) : ctx->kernels_launched.load();
    return REDUX_OK;
}

extern "C" void redux_generate_blocks_host(uint8_t *out, uint64_t first_block, uint64_t n_blocks,
                                           uint64_t block_len, uint64_t seed)
{
    redux_generate_blocks_host_ex(out, first_block, n_blocks, block_len, seed, nullptr, 0);
}

extern "C" void redux_generate_blocks_host_ex(uint8_t *out, uint64_t first_block, uint64_t n_blocks,
                                              uint64_t block_len, uint64_t seed, const uint8_t *corpus, uint64_t corpus_len)
{
    uint8_t lut[256];
    for (uint32_t u = 0; u < 256; ++u) lut[u] = text_symbol(u);
    const uint64_t groups = (block_len + 7) >> 3;
    for (uint64_t b = 0; b < n_blocks; ++b)
        for (uint64_t w = 0; w < groups; ++w) {
            uint64_t v = gen_group(seed, first_block + b, w, lut, corpus, corpus_len, block_len);
            for (uint64_t j = 0; j < 8 && w * 8 + j < block_len; ++j)
                out[b * block_len + w * 8 + j] = (uint8_t)(v >> (8 * j));
        }
}

// =================================================================================== host memory
// The host-buffer API copies straight from / to the caller's pointers.  From pinned (page-locked) memory the
// copies are asynchronous and the chunk pipeline overlaps them with the kernels; from pageable memory CUDA stages
// every copy through its own bounce buffer and the calls degrade to roughly the speed of a host memcpy.
extern "C" int redux_host_alloc(size_t bytes, void **out)
{
    if (!out) return REDUX_INVALID_INPUT;
    *out = nullptr;
    if (bytes == 0) return REDUX_OK;
    if (cudaHostAlloc(out, bytes, cudaHostAllocPortable) != cudaSuccess) { (void)cudaGetLastError(); *out = nullptr; return REDUX_CUDA_ERROR; }
    return REDUX_OK;
}
extern "C" int redux_host_free(void *p)
{
    if (!p) return REDUX_OK;
    if (cudaFreeHost(p) != cudaSuccess) { (void)cudaGetLastError(); return REDUX_CUDA_ERROR; }
    return REDUX_OK;
}
extern "C" int redux_host_register(void *p, size_t bytes)
{
    if (!p || bytes == 0) return REDUX_INVALID_INPUT;
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) { (void)cudaGetLastError(); return REDUX_CUDA_ERROR; }
    return REDUX_OK;
}
extern "C" int redux_host_unregister(void *p)
{
    if (!p) return REDUX_INVALID_INPUT;
    if (cudaHostUnregister(p) != cudaSuccess) { (void)cudaGetLastError(); return REDUX_CUDA_ERROR; }
    return REDUX_OK;
}

// ======================================================================================= context

extern "C" int redux_ctx_create(const int *devices, int n_devices, redux_ctx_t **out)
{
    if (!out) return REDUX_INVALID_INPUT;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) { (void)cudaGetLastError(); return REDUX_CUDA_ERROR; }
    redux_ctx *ctx = new redux_ctx();
    std::vector<int> devs;
    if (!devices || n_devices <= 0) {
        int cur = 0;
        if (cudaGetDevice(&cur) != cudaSuccess) { delete ctx; return REDUX_CUDA_ERROR; }
        devs.push_back(cur);
    } else {
        devs.assign(devices, devices + n_devices);
    }
    uint8_t lut[256];
    for (uint32_t u = 0; u < 256; ++u) lut[u] = text_symbol(u);
    for (int dev : devs) {
        if (dev < 0 || dev >= count) { redux_ctx_destroy(ctx); return REDUX_INVALID_INPUT; }
        DeviceGuard g(dev);
        DeviceState d;
        d.device = dev;
        cudaDeviceProp prop;
        if (!g.ok || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) { redux_ctx_destroy(ctx); return REDUX_CUDA_ERROR; }
        if (prop.major < 10) { redux_ctx_destroy(ctx); return REDUX_CUDA_ERROR; }   // sm_100a binary only
        bool streams_ok = cudaEventCreateWithFlags(&d.ws_busy, cudaEventDisableTiming) == cudaSuccess &&
                          cudaStreamCreateWithFlags(&d.copy, cudaStreamNonBlocking) == cudaSuccess &&
                          cudaStreamCreateWithFlags(&d.h2d, cudaStreamNonBlocking) == cudaSuccess;
        for (int i = 0; i < kPipeStreams && streams_ok; ++i)
            streams_ok = cudaStreamCreateWithFlags(&d.pipe[i], cudaStreamNonBlocking) == cudaSuccess;
        if (!streams_ok || cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking) != cudaSuccess ||
            configure_kernels() != cudaSuccess ||
            cudaMalloc((void **)&d.text_lut, 256) != cudaSuccess ||
            cudaMemcpy(d.text_lut, lut, 256, cudaMemcpyHostToDevice) != cudaSuccess) {
            (void)cudaGetLastError();
            ctx->devs.push_back(d);
            redux_ctx_destroy(ctx);
            return REDUX_CUDA_ERROR;
        }
        ctx->devs.push_back(d);
    }
    *out = ctx;
    return REDUX_OK;
}

extern "C" void redux_ctx_destroy(redux_ctx_t *ctx)
{
    if (!ctx) return;
    for (auto &d : ctx->devs) {
        DeviceGuard g(d.device);
        cudaDeviceSynchronize();
        if (d.ws_busy) cudaEventDestroy(d.ws_busy);
        if (d.stream) cudaStreamDestroy(d.stream);
        if (d.copy) cudaStreamDestroy(d.copy);
        if (d.h2d) cudaStreamDestroy(d.h2d);
        for (int i = 0; i < kPipeStreams; ++i) if (d.pipe[i]) cudaStreamDestroy(d.pipe[i]);
        for (HostBuf *b : {&d.pin_off, &d.pin_status, &d.pin_aux0, &d.pin_aux1}) b->release();
        for (DevBuf *b : {&d.slots, &d.sizes, &d.flag, &d.st_in, &d.st_off, &d.st_out, &d.st_ooff,
                          &d.st_status, &d.st_aux0, &d.st_aux1, &d.st_roff, &d.corpus, &d.gen_magic, &d.gen_tabs, &d.gen_init, &d.gen_freq, &d.split_hist, &d.split_pairs}) b->release();
        for (auto &m : d.magics) cudaFree(m.ptr);
        if (d.text_lut) cudaFree(d.text_lut);
        for (StageRing *r : {d.ring_up, d.ring_down}) if (r) { r->release(); delete r; }
    }
    delete ctx->pool;
    delete ctx;
}

extern "C" int redux_ctx_device_count(const redux_ctx_t *ctx) { return ctx ? (int)ctx->devs.size() : 0; }
extern "C" const char *redux_ctx_last_error(const redux_ctx_t *ctx) { return ctx ? ctx->last_error.c_str() : ""; }
extern "C" uint64_t redux_ctx_kernel_launches(const redux_ctx_t *ctx) { return ctx ? ctx->launches : 0; }

extern "C" int redux_ctx_timing_enable(redux_ctx_t *ctx, int on)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    ctx->timing = on != 0;
    return REDUX_OK;
}

extern "C" int redux_ctx_timing_collect(redux_ctx_t *ctx, double *ms, uint64_t *counts)
{
    if (!ctx || !ms || !counts) return REDUX_INVALID_INPUT;
    for (int k = 0; k < REDUX_KERNEL_KINDS; ++k) { ms[k] = 0; counts[k] = 0; }
    int rc = REDUX_OK;
    for (auto &sp : ctx->spans) {
        DeviceGuard g(sp.device);
        float t = 0;
        if (cudaEventSynchronize(sp.b) == cudaSuccess && cudaEventElapsedTime(&t, sp.a, sp.b) == cudaSuccess) {
            ms[sp.kind] += t; counts[sp.kind] += 1;
        } else { (void)cudaGetLastError(); rc = REDUX_CUDA_ERROR; }
        cudaEventDestroy(sp.a); cudaEventDestroy(sp.b);
    }
    ctx->spans.clear();
    return rc;
}

extern "C" int redux_ctx_set_text_corpus(redux_ctx_t *ctx, const uint8_t *corpus, uint64_t corpus_len)
{
    if (!ctx || (!corpus && corpus_len)) return REDUX_INVALID_INPUT;
    for (auto &d : ctx->devs) {
        DeviceGuard g(d.device);
        d.corpus_len = 0;
        if (!corpus_len) continue;
        CU_TRY(ctx, d.corpus.reserve(corpus_len));
        CU_TRY(ctx, cudaMemcpy(d.corpus.p, corpus, corpus_len, cudaMemcpyHostToDevice));
        d.corpus_len = corpus_len;
    }
    return REDUX_OK;
}

extern "C" int redux_ctx_set_schedule(redux_ctx_t *ctx, int sched)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    if (sched == REDUX_SCHED_AUTO || sched == REDUX_SCHED_LANE || sched == REDUX_SCHED_WARP || sched == REDUX_SCHED_SPLIT) { ctx->sched = sched; return REDUX_OK; }
    return fail(ctx, REDUX_INVALID_INPUT, "unknown schedule");
}

extern "C" int redux_ctx_set_staging(redux_ctx_t *ctx, int enable, size_t min_bytes, size_t piece_bytes, int slots, int threads)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    if (slots < 0 || threads < 0 || slots > 64 || threads > 256) return fail(ctx, REDUX_INVALID_INPUT, "staging: slots / threads out of range");
    if (piece_bytes && (piece_bytes < 4096 || piece_bytes > ((size_t)1 << 30))) return fail(ctx, REDUX_INVALID_INPUT, "staging: piece_bytes out of range");
    ctx->staging.enable = enable != 0;
    if (min_bytes) ctx->staging.min_bytes = min_bytes;
    if (piece_bytes) ctx->staging.piece_bytes = (piece_bytes + 63) & ~(size_t)63;
    if (slots) ctx->staging.slots = std::max(2, slots);
    if (threads && threads != ctx->staging.threads) {
        ctx->staging.threads = threads;
        delete ctx->pool;                     // no call is running: the next one recreates it
        ctx->pool = nullptr;
    }
    return REDUX_OK;
}

extern "C" int redux_ctx_synchronize(redux_ctx_t *ctx, int device, void *stream)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    DeviceState *d = find_dev(ctx, device);
    if (!d) return fail(ctx, REDUX_INVALID_INPUT, "device is not part of this context");
    DeviceGuard g(device);
    CU_TRY(ctx, cudaStreamSynchronize((cudaStream_t)stream));
    return REDUX_OK;
}

// ============================================================================ device-resident API
namespace {

// Enqueues encode + size scan + compaction for n_blocks blocks on stream s.  Workspace slices are given
// explicitly so that several chunks of one batch can be in flight on different streams.
int encode_launch(redux_ctx *ctx, int device, cudaStream_t s, const Plan &pl, const void *magic,
                  const uint8_t *d_in, const uint64_t *d_in_off, uint64_t n_blocks,
                  uint8_t *d_out, uint64_t out_capacity, uint64_t *d_out_off, int32_t *d_status,
                  uint8_t *slots, uint32_t *sizes, int32_t *flag)
{
    LaneEncJob job;
    job.in = d_in; job.in_off = d_in_off; job.n_blocks = n_blocks;
    job.slots = slots; job.slot_stride = pl.slot_stride;
    job.sizes = sizes; job.status = d_status;
    set_plan_fields(job, pl, magic);
    {
        KernelTimer kt(ctx, device, s, REDUX_KERNEL_ENCODE);
        KernelId kid;
        if (pl.generic) {
            GenericJob g = generic_job(pl);
            g.in = d_in; g.in_off = d_in_off; g.n_blocks = n_blocks;
            g.slots = slots; g.slot_stride = pl.slot_stride; g.sizes = sizes; g.status = d_status;
            encode_generic_kernel<<<pl.gen_threads / kGenericThreads, kGenericThreads, generic_smem_bytes(pl.s), s>>>(g);
            kid = pl.s <= kGenericSmemSymbolBits ? kEncGenericSmem : kEncGenericGlobal;
        }
        else if (pl.split) {
            DeviceState *d = find_dev(ctx, device);
            int rc = launch_encode_split(ctx, d, pl, job, s, &kid);
            if (rc) return rc;
        }
        else {
            kid = pick_encoder(pl);
            if (!launch_coder(kid, job, s)) return fail(ctx, REDUX_CUDA_ERROR, "no encoder for the plan");
        }
        ctx->note_kernel(kid);
    }
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    {
        KernelTimer kt(ctx, device, s, REDUX_KERNEL_SCAN);
        scan_sizes_kernel<<<1, kScanThreads, 0, s>>>(sizes, n_blocks, d_out_off, out_capacity, flag);
    }
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    const uint32_t cgrid = (uint32_t)std::min<uint64_t>(n_blocks, 148 * 16);
    {
        KernelTimer kt(ctx, device, s, REDUX_KERNEL_COMPACT);
        compact_kernel<<<cgrid, kCompactThreads, 0, s>>>(slots, pl.slot_stride, sizes, d_out_off, n_blocks,
                                                         d_out, out_capacity, d_status);
    }
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    return REDUX_OK;
}

int decode_launch(redux_ctx *ctx, int device, cudaStream_t s, const Plan &pl, const void *magic,
                  const uint8_t *d_comp, const uint64_t *d_comp_off, uint64_t n_blocks,
                  uint8_t *d_raw, const uint64_t *d_raw_off, uint64_t *d_raw_lens, uint64_t *d_consumed,
                  int32_t *d_status)
{
    LaneDecJob job;
    job.comp = d_comp; job.comp_off = d_comp_off; job.n_blocks = n_blocks;
    job.raw = d_raw; job.raw_off = d_raw_off; job.raw_len = d_raw_lens; job.consumed = d_consumed;
    job.status = d_status;
    set_plan_fields(job, pl, magic);
    {
        KernelTimer kt(ctx, device, s, REDUX_KERNEL_DECODE);
        KernelId kid;
        if (pl.generic) {
            GenericJob g = generic_job(pl);
            g.in = d_comp; g.in_off = d_comp_off; g.n_blocks = n_blocks;
            g.raw = d_raw; g.raw_off = d_raw_off; g.raw_len = d_raw_lens; g.consumed = d_consumed; g.status = d_status;
            decode_generic_kernel<<<pl.gen_threads / kGenericThreads, kGenericThreads, generic_smem_bytes(pl.s), s>>>(g);
            kid = pl.s <= kGenericSmemSymbolBits ? kDecGenericSmem : kDecGenericGlobal;
        }
        else {
            kid = pick_decoder(pl);
            if (!launch_coder(kid, job, s)) return fail(ctx, REDUX_CUDA_ERROR, "no decoder for the plan");
        }
        ctx->note_kernel(kid);
    }
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    return REDUX_OK;
}

}  // namespace

extern "C" int redux_encode_batch_device(redux_ctx_t *ctx, int device, void *stream_, int model_kind,
                                         const redux_params_t *params, const uint8_t *d_in,
                                         const uint64_t *d_in_offsets, uint64_t n_blocks,
                                         uint64_t max_block_len, uint8_t *d_out, uint64_t out_capacity,
                                         uint64_t *d_out_offsets, int32_t *d_status)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    int rc;
    if ((rc = check_kind(ctx, model_kind))) return rc;
    Plan pl;
    if ((rc = make_plan(ctx, params, max_block_len, &pl))) return rc;
    pl.warp = !pl.generic && !pl.pretrained && choose_warp(ctx);
    pl.split = !pl.generic && !pl.pretrained && choose_split(ctx, n_blocks, pl.cls, max_block_len);
    DeviceState *d = find_dev(ctx, device);
    if (!d) return fail(ctx, REDUX_INVALID_INPUT, "device is not part of this context");
    if (!d_in_offsets || !d_out_offsets || !d_status || (!d_out && out_capacity))
        return fail(ctx, REDUX_INVALID_INPUT, "NULL buffer");
    DeviceGuard g(device);
    cudaStream_t s = (cudaStream_t)stream_;   // NULL = the default stream, as in CUDA
    if (n_blocks == 0) { CU_TRY(ctx, cudaMemsetAsync(d_out_offsets, 0, sizeof(uint64_t), s)); return REDUX_OK; }
    if (n_blocks > 0x7FFFFFFFull * 32) return fail(ctx, REDUX_UNSUPPORTED, "too many blocks in one launch");

    CU_TRY(ctx, ws_acquire(d, s));              // the previous device call may still be using the workspace
    const void *magic = nullptr;
    if ((rc = get_magic(ctx, d, s, pl, &magic))) return rc;
    if ((rc = prepare_generic(ctx, d, s, params, n_blocks, &pl))) return rc;
    CU_TRY(ctx, d->slots.reserve(n_blocks * pl.slot_stride));
    CU_TRY(ctx, d->sizes.reserve(n_blocks * sizeof(uint32_t)));
    CU_TRY(ctx, d->flag.reserve(sizeof(int32_t)));
    rc = encode_launch(ctx, device, s, pl, magic, d_in, d_in_offsets, n_blocks, d_out, out_capacity,
                       d_out_offsets, d_status, (uint8_t *)d->slots.p, (uint32_t *)d->sizes.p,
                       (int32_t *)d->flag.p);
    CU_TRY(ctx, ws_release(d, s));
    return rc;
}

extern "C" int redux_decode_batch_device(redux_ctx_t *ctx, int device, void *stream_, int model_kind,
                                         const redux_params_t *params, const uint8_t *d_comp,
                                         const uint64_t *d_comp_offsets, uint64_t n_blocks,
                                         uint64_t max_block_len, uint8_t *d_raw,
                                         const uint64_t *d_raw_offsets, uint64_t *d_raw_lens,
                                         uint64_t *d_consumed, int32_t *d_status)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    int rc;
    if ((rc = check_kind(ctx, model_kind))) return rc;
    Plan pl;
    if ((rc = make_plan(ctx, params, max_block_len, &pl))) return rc;
    pl.warp = !pl.generic && !pl.pretrained && choose_warp(ctx);
    DeviceState *d = find_dev(ctx, device);
    if (!d) return fail(ctx, REDUX_INVALID_INPUT, "device is not part of this context");
    if (n_blocks == 0) return REDUX_OK;
    if (!d_comp_offsets || !d_raw_offsets || !d_raw_lens || !d_consumed || !d_status)
        return fail(ctx, REDUX_INVALID_INPUT, "NULL buffer");
    DeviceGuard g(device);
    cudaStream_t s = (cudaStream_t)stream_;   // NULL = the default stream, as in CUDA
    CU_TRY(ctx, ws_acquire(d, s));
    const void *magic = nullptr;
    if ((rc = get_magic(ctx, d, s, pl, &magic))) return rc;
    if ((rc = prepare_generic(ctx, d, s, params, n_blocks, &pl))) return rc;
    rc = decode_launch(ctx, device, s, pl, magic, d_comp, d_comp_offsets, n_blocks, d_raw, d_raw_offsets,
                       d_raw_lens, d_consumed, d_status);
    CU_TRY(ctx, ws_release(d, s));
    return rc;
}

extern "C" int redux_generate_blocks_device(redux_ctx_t *ctx, int device, void *stream_, uint8_t *d_out,
                                            uint64_t first_block, uint64_t n_blocks, uint64_t block_len,
                                            uint64_t seed)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    DeviceState *d = find_dev(ctx, device);
    if (!d) return fail(ctx, REDUX_INVALID_INPUT, "device is not part of this context");
    if (n_blocks == 0 || block_len == 0) return REDUX_OK;
    DeviceGuard g(device);
    cudaStream_t s = (cudaStream_t)stream_;   // NULL = the default stream, as in CUDA
    {
        KernelTimer kt(ctx, device, s, REDUX_KERNEL_GENERATE);
        generate_kernel<<<148 * 8, 256, 0, s>>>(d_out, first_block, n_blocks, block_len, seed, d->text_lut,
                                                (const uint8_t *)d->corpus.p, d->corpus_len);
    }
    ctx->launches++;
    CU_TRY(ctx, cudaGetLastError());
    return REDUX_OK;
}

// ================================================================================ host-buffer API
// End-to-end path.  A device's shard is cut into chunks of blocks; chunk k runs
//     H2D(raw bytes, on the shared h2d stream) -> encode -> scan -> compact -> D2H(offsets, status)
// on its own compute stream
// so the copy engines and the SMs overlap (the coder kernels are latency-bound per lane: a chunk takes
// about as long as the whole batch, so many chunks must be in flight together).  The host then walks the
// chunks in order and streams each chunk's compacted bytes to its final place in the caller's buffer.
namespace {

struct Shard { uint64_t first, count; };

// REDUX_TRACE=1: host-side timeline of the pipelined host-buffer calls on stderr (tuning aid).
struct Trace {
    bool on; std::chrono::steady_clock::time_point t0;
    Trace() : on(std::getenv("REDUX_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void mark(const char *what, long k = -1) const {
        if (!on) return;
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (k >= 0) fprintf(stderr, "[redux trace] %8.2f ms  %s %ld\n", ms, what, k);
        else fprintf(stderr, "[redux trace] %8.2f ms  %s\n", ms, what);
    }
};

std::vector<Shard> make_shards(uint64_t n_blocks, size_t n_dev)
{
    // contiguous block-index ranges, SURVEY.md 8(e); same rule as redux_debug_shard
    std::vector<Shard> s(n_dev);
    for (size_t g = 0; g < n_dev; ++g) {
        uint64_t a = n_blocks * g / n_dev, b = n_blocks * (g + 1) / n_dev;
        s[g] = {a, b - a};
    }
    return s;
}

// tuning knobs (environment, read once): number of chunks per shard and of compute streams they rotate over
int env_int(const char *name, int dflt, int lo, int hi)
{
    const char *v = std::getenv(name);
    if (!v) return dflt;
    int x = std::atoi(v);
    return x < lo ? lo : (x > hi ? hi : x);
}
int pipe_chunks()  { static int v = env_int("REDUX_PIPE_CHUNKS", 20, 1, 256); return v; }
int pipe_streams() { static int v = env_int("REDUX_PIPE_STREAMS", kPipeStreams, 1, kPipeStreams); return v; }

// Cuts a shard into chunks of whole CTAs.  A lane needs the same ~10-25 ms for its block however few
// blocks are in flight, so what a chunk's size controls is only WHEN its copy-in ends and its copy-out
// can start.  ramp < 0: small chunks FIRST (decode: the device-to-host link is the bottleneck, so the
// first decoded bytes must be ready as early as possible); ramp > 0: small chunks LAST (encode: the
// host-to-device link is the bottleneck, so as little as possible may remain after the last byte lands).
std::vector<Shard> make_chunks(uint64_t count, int ramp)
{
    const uint64_t cta = kLaneThreads;
    const uint64_t ctas = (count + cta - 1) / cta;
    std::vector<uint64_t> sizes;                                  // in CTAs
    const uint64_t want = (uint64_t)pipe_chunks();
    static const int ramp_on = env_int("REDUX_PIPE_RAMP", 1, 0, 1);
    if (ramp != 0 && ramp_on && ctas >= 128) {
        static const uint64_t steps[] = {4, 4, 8, 12, 16};
        uint64_t used = 0;
        for (uint64_t st : steps) { sizes.push_back(st); used += st; }
        const uint64_t rest = ctas - used;
        const uint64_t nrest = want > 5 ? want - 5 : 1;
        const uint64_t per = (rest + nrest - 1) / nrest;
        for (uint64_t a = 0; a < rest; a += per) sizes.push_back(std::min(per, rest - a));
        if (ramp > 0) std::reverse(sizes.begin(), sizes.end());
    } else {
        uint64_t per = std::max<uint64_t>((ctas + want - 1) / want, 8);   // at least 8 CTAs each
        for (uint64_t a = 0; a < ctas; a += per) sizes.push_back(std::min(per, ctas - a));
    }
    std::vector<Shard> c;
    uint64_t first = 0;
    for (uint64_t sz : sizes) {
        const uint64_t n = std::min(sz * cta, count - first);
        if (n) c.push_back({first, n});
        first += n;
    }
    return c;
}

struct EventSet {
    std::vector<cudaEvent_t> ev;
    cudaError_t create(size_t n) {
        ev.assign(n, nullptr);
        for (auto &e : ev) { cudaError_t r = cudaEventCreateWithFlags(&e, cudaEventDisableTiming); if (r != cudaSuccess) return r; }
        return cudaSuccess;
    }
    ~EventSet() { for (auto e : ev) if (e) cudaEventDestroy(e); }
};

// Runs fn(view, device_state, g) for every shard: inline for one device, one host thread per device
// otherwise.  Each worker gets a private view of the context (own error string / launch counter) so the
// workers never share mutable state; the views are merged afterwards.
template <typename F>
void for_each_device(redux_ctx *ctx, size_t nd, std::vector<int> &rcs, F fn)
{
    if (nd == 1) { rcs[0] = fn(ctx, &ctx->devs[0], (size_t)0); return; }
    std::vector<std::thread> th;
    std::vector<std::string> errs(nd);
    std::vector<uint64_t> launches(nd, 0);
    std::vector<std::vector<TimedSpan>> spans(nd);
    for (size_t g = 0; g < nd; ++g) th.emplace_back([&, g] {
        redux_ctx view; view.sched = ctx->sched; view.timing = ctx->timing; view.model_freq = ctx->model_freq;
        view.staging = ctx->staging; view.pool = ctx->pool;
        view.devs.push_back(ctx->devs[g]);
        rcs[g] = fn(&view, &view.devs[0], g);
        ctx->kernels_launched.fetch_or(view.kernels_launched.load(std::memory_order_relaxed), std::memory_order_relaxed);
        ctx->devs[g] = view.devs[0];          // workspaces may have grown
        view.devs.clear(); view.pool = nullptr;
        errs[g] = view.last_error; launches[g] = view.launches; spans[g] = view.spans;
    });
    for (auto &t : th) t.join();
    for (size_t g = 0; g < nd; ++g) {
        ctx->launches += launches[g];
        ctx->spans.insert(ctx->spans.end(), spans[g].begin(), spans[g].end());
        if (rcs[g]) ctx->last_error = errs[g];
    }
}

// Waits for everything this device still has in flight (used on error paths before buffers are reused).
void drain(DeviceState *d)
{
    cudaStreamSynchronize(d->h2d);
    for (int i = 0; i < kPipeStreams; ++i) cudaStreamSynchronize(d->pipe[i]);
    cudaStreamSynchronize(d->copy);
}

// ---- pageable caller memory (see CopyPool)
// true when `p` is host memory CUDA does not know (neither cudaHostAlloc'ed nor registered) and the transfer is big
// enough to be worth staging
bool needs_staging(const redux_ctx *ctx, const void *p, uint64_t bytes)
{
    if (!ctx->staging.enable || !p || bytes < ctx->staging.min_bytes) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeUnregistered;
}

// creates the copy threads on first use (called before the per-device workers start)
void ensure_pool(redux_ctx *ctx)
{
    if (ctx->pool) return;
    int n = ctx->staging.threads;
    if (n <= 0) {
        // measured on a 16-core host (profiles/r02_staging.json): 1 thread 6.2, 4: 11.4, 8: 14.1, 12: 16.1 GB/s end to
        // end (pinned buffers: 19.7); the feeder and the drainer copy too
        const int hw = (int)std::thread::hardware_concurrency();
        n = std::max(1, std::min(16, hw * 3 / 4));
    }
    ctx->pool = new CopyPool(n);
}

cudaError_t ensure_ring(const redux_ctx *ctx, StageRing **ring)
{
    if (!*ring) *ring = new StageRing();
    return (*ring)->ensure(ctx->staging.piece_bytes, std::max(2, ctx->staging.slots));
}

// Host -> device through the ring: blocks the calling (feeder) thread for the host copies only.
cudaError_t staged_h2d(StageRing *ring, CopyPool *pool, cudaStream_t stream, uint8_t *dst_dev, const uint8_t *src,
                       uint64_t n, int *next_slot, const std::atomic<bool> *stop)
{
    for (uint64_t a = 0; a < n; a += ring->piece) {
        if (stop && stop->load(std::memory_order_relaxed)) return cudaSuccess;
        const size_t len = (size_t)std::min<uint64_t>(ring->piece, n - a);
        const int i = *next_slot;
        *next_slot = (i + 1) % ring->n;
        cudaError_t e;
        if (ring->recorded[i] && (e = cudaEventSynchronize(ring->ev[i])) != cudaSuccess) return e;
        pool->copy(ring->slot(i), src + a, len);
        if ((e = cudaMemcpyAsync(dst_dev + a, ring->slot(i), len, cudaMemcpyHostToDevice, stream)) != cudaSuccess) return e;
        if ((e = cudaEventRecord(ring->ev[i], stream)) != cudaSuccess) return e;
        ring->recorded[i] = 1;
    }
    return cudaSuccess;
}

// Device -> host through the ring, driven by the drainer thread: push() enqueues the asynchronous copies of one
// range piece by piece and, when the ring is full, first retires the oldest piece (waits for it, copies it to the
// caller's memory); flush() retires everything.
struct DownStager {
    StageRing *ring; CopyPool *pool; cudaStream_t stream;
    struct Pending { int slot; uint8_t *dst; size_t n; };
    std::deque<Pending> fifo;
    int next = 0;
    cudaError_t retire_one() {
        const Pending p = fifo.front(); fifo.pop_front();
        cudaError_t e = cudaEventSynchronize(ring->ev[p.slot]);
        if (e != cudaSuccess) return e;
        pool->copy(p.dst, ring->slot(p.slot), p.n);
        return cudaSuccess;
    }
    cudaError_t push(uint8_t *dst_host, const uint8_t *src_dev, uint64_t n) {
        for (uint64_t a = 0; a < n; a += ring->piece) {
            cudaError_t e;
            if ((int)fifo.size() == ring->n && (e = retire_one()) != cudaSuccess) return e;
            const size_t len = (size_t)std::min<uint64_t>(ring->piece, n - a);
            const int i = next; next = (next + 1) % ring->n;
            if ((e = cudaMemcpyAsync(ring->slot(i), src_dev + a, len, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
            if ((e = cudaEventRecord(ring->ev[i], stream)) != cudaSuccess) return e;
            ring->recorded[i] = 1;
            fifo.push_back({i, dst_host + a, len});
        }
        return cudaSuccess;
    }
    // retires finished pieces while `gate` (an event the caller is about to wait for) is still pending
    cudaError_t retire_while_pending(cudaEvent_t gate) {
        while (!fifo.empty() && cudaEventQuery(gate) == cudaErrorNotReady) {
            cudaError_t e = retire_one();
            if (e != cudaSuccess) return e;
        }
        (void)cudaGetLastError();                           // cudaErrorNotReady is not an error
        return cudaSuccess;
    }
    cudaError_t flush() {
        while (!fifo.empty()) { cudaError_t e = retire_one(); if (e != cudaSuccess) return e; }
        return cudaSuccess;
    }
};

// Hand-off between the thread that enqueues the chunks (and feeds the staged input) and the thread that drains
// their results: chunk k may be waited for once `enqueued > k`.
struct ChunkProgress {
    std::mutex m; std::condition_variable cv;
    size_t enqueued = 0; bool done = false;
    std::atomic<bool> stop{false};                          // the drainer failed: stop feeding
    void advance() { { std::lock_guard<std::mutex> l(m); ++enqueued; } cv.notify_all(); }
    void finish() { { std::lock_guard<std::mutex> l(m); done = true; } cv.notify_all(); }
    bool wait_for(size_t k) {                               // false: the feeder ended before chunk k
        std::unique_lock<std::mutex> l(m);
        cv.wait(l, [&] { return enqueued > k || done; });
        return enqueued > k;
    }
};

// Cross-shard hand-off of redux_encode_batch on several devices.  The streams of the whole batch lie back to
// back in the caller's buffer, so shard g's bytes start where the shards below it end: every worker publishes
// its total as soon as its last chunk is coded, waits for the totals below it, and then copies its own bytes
// out -- no worker waits for a shard ABOVE it, shard 0 streams chunk by chunk from the start.
struct ShardSync {
    std::mutex m;
    std::condition_variable cv;
    std::vector<int64_t> total;           // -1: not known yet
    bool aborted = false;
    explicit ShardSync(size_t n) : total(n, -1) {}
    void publish(size_t g, uint64_t t) { { std::lock_guard<std::mutex> l(m); total[g] = (int64_t)t; } cv.notify_all(); }
    void abort() { { std::lock_guard<std::mutex> l(m); aborted = true; } cv.notify_all(); }
    // base offset of shard g; false when another shard failed
    bool base_of(size_t g, uint64_t *base) {
        std::unique_lock<std::mutex> l(m);
        cv.wait(l, [&] {
            if (aborted) return true;
            for (size_t i = 0; i < g; ++i) if (total[i] < 0) return false;
            return true;
        });
        if (aborted) return false;
        uint64_t b = 0;
        for (size_t i = 0; i < g; ++i) b += (uint64_t)total[i];
        *base = b;
        return true;
    }
};

// One device's shard of redux_encode_batch: shard g of the hand-off `sync` (nullptr: the only shard).
// Shard 0 knows its base (0) from the start and copies the compacted bytes of chunk k to out + (bytes of the
// chunks before it) as soon as the chunk is done; a higher shard keeps its bytes on the device (st_out, chunk k
// at chunk_base[k]) until the shards below it have published their totals.
struct EncShardOut {
    std::vector<uint64_t> local_off;     // [count+1] shard-local offsets of the back-to-back streams
    std::vector<uint64_t> chunk_base;    // device offset of chunk k inside st_out
    std::vector<uint64_t> chunk_total;   // compacted bytes of chunk k
    std::vector<Shard> chunks;
    uint64_t total = 0;
};

int encode_shard(redux_ctx *ctx, DeviceState *d, const redux_params_t *p, const uint8_t *in,
                 const uint64_t *in_off, Shard sh, uint8_t *out, uint64_t out_cap,
                 int32_t *status, EncShardOut *res, ShardSync *sync, size_t g_index)
{
    const bool streaming = !sync || g_index == 0;          // the shard's base is known up front
    Trace tr;
    DeviceGuard g(d->device);
    const uint64_t base = in_off[sh.first], bytes = in_off[sh.first + sh.count] - base;
    uint64_t max_len = 0;
    std::vector<uint64_t> rel(sh.count + 1);
    for (uint64_t i = 0; i <= sh.count; ++i) {
        rel[i] = in_off[sh.first + i] - base;
        if (i) { if (rel[i] < rel[i - 1]) return fail(ctx, REDUX_INVALID_INPUT, "offsets not monotonic");
                 max_len = std::max(max_len, rel[i] - rel[i - 1]); }
    }
    Plan pl;
    int rc = make_plan(ctx, p, max_len, &pl);
    if (rc) return rc;
    pl.warp = !pl.generic && !pl.pretrained && choose_warp(ctx);
    pl.split = !pl.generic && !pl.pretrained && choose_split(ctx, sh.count, pl.cls, max_len);
    // chunks of the generic path would share the Fenwick columns (and split chunks the range workspace): one chunk
    res->chunks = (pl.generic || pl.split) ? std::vector<Shard>{{0, sh.count}} : make_chunks(sh.count, +1);
    const size_t nc = res->chunks.size();
    res->chunk_base.assign(nc, 0); res->chunk_total.assign(nc, 0);
    res->local_off.assign(sh.count + 1, 0);
    std::vector<uint64_t> chunk_cap(nc);
    uint64_t dcap = 0;
    for (size_t k = 0; k < nc; ++k) {
        uint64_t w = 0;
        for (uint64_t i = 0; i < res->chunks[k].count; ++i) {
            const uint64_t b = res->chunks[k].first + i;
            w += redux_compress_bound_ex(rel[b + 1] - rel[b], pl.s, pl.c);
        }
        chunk_cap[k] = w;
        res->chunk_base[k] = dcap;
        dcap += (w + 15) & ~(uint64_t)15;
    }
    CU_TRY(ctx, d->st_in.reserve(bytes + 32));
    CU_TRY(ctx, d->st_off.reserve((sh.count + 1) * sizeof(uint64_t)));
    CU_TRY(ctx, d->st_out.reserve(dcap + 32));
    CU_TRY(ctx, d->st_ooff.reserve((sh.count + nc) * sizeof(uint64_t)));
    CU_TRY(ctx, d->st_status.reserve(sh.count * sizeof(int32_t)));
    CU_TRY(ctx, d->slots.reserve(sh.count * pl.slot_stride));
    CU_TRY(ctx, d->sizes.reserve(sh.count * sizeof(uint32_t)));
    CU_TRY(ctx, d->flag.reserve(nc * sizeof(int32_t)));
    CU_TRY(ctx, d->pin_off.reserve((sh.count + nc) * sizeof(uint64_t)));
    CU_TRY(ctx, d->pin_status.reserve(sh.count * sizeof(int32_t)));
    const void *magic = nullptr;
    if ((rc = get_magic(ctx, d, d->h2d, pl, &magic))) return rc;
    if ((rc = prepare_generic(ctx, d, d->h2d, p, sh.count, &pl))) return rc;
    EventSet evs;                       // [0, nc): chunk done; [nc, 2nc): chunk input on the device
    CU_TRY(ctx, evs.create(2 * nc));
    // pageable caller memory goes through the pinned rings (CopyPool); then the enqueue loop below runs on a feeder
    // thread of its own, because it blocks on host copies while the results of earlier chunks are being drained
    const bool stage_in = needs_staging(ctx, in, bytes), stage_out = needs_staging(ctx, out, std::min(out_cap, dcap));
    const bool staged = stage_in || stage_out;
    if (stage_in) CU_TRY(ctx, ensure_ring(ctx, &d->ring_up));
    if (stage_out) CU_TRY(ctx, ensure_ring(ctx, &d->ring_down));
    CU_TRY(ctx, cudaMemcpyAsync(d->st_off.p, rel.data(), rel.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, d->h2d));

    uint8_t *d_in = (uint8_t *)d->st_in.p, *d_out = (uint8_t *)d->st_out.p;
    uint64_t *d_off = (uint64_t *)d->st_off.p, *d_ooff = (uint64_t *)d->st_ooff.p;
    int32_t *d_status = (int32_t *)d->st_status.p;
    uint64_t *h_ooff = (uint64_t *)d->pin_off.p;
    int32_t *h_status = (int32_t *)d->pin_status.p;
    ChunkProgress prog;
    // While the feeder runs it is the only thread that touches ctx (error text, launch counter, timing spans).
    auto enqueue_all = [&]() -> int {
        int up_slot = 0;
        for (size_t k = 0; k < nc && !prog.stop.load(std::memory_order_relaxed); ++k) {
            const Shard c = res->chunks[k];
            cudaStream_t s = d->pipe[k % pipe_streams()];
            int rc2 = REDUX_OK;
            cudaError_t e = cudaSuccess;
            const uint64_t b0 = rel[c.first], b1 = rel[c.first + c.count];
            if (b1 > b0) e = stage_in ? staged_h2d(d->ring_up, ctx->pool, d->h2d, d_in + b0, in + base + b0, b1 - b0, &up_slot, &prog.stop)
                                      : cudaMemcpyAsync(d_in + b0, in + base + b0, b1 - b0, cudaMemcpyHostToDevice, d->h2d);
            if (e == cudaSuccess) e = cudaEventRecord(evs.ev[nc + k], d->h2d);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(s, evs.ev[nc + k], 0);
            if (e == cudaSuccess)
                rc2 = encode_launch(ctx, d->device, s, pl, magic, d_in, d_off + c.first, c.count,
                                    d_out + res->chunk_base[k], chunk_cap[k], d_ooff + c.first + k,
                                    d_status + c.first, (uint8_t *)d->slots.p + c.first * pl.slot_stride,
                                    (uint32_t *)d->sizes.p + c.first, (int32_t *)d->flag.p + k);
            if (e == cudaSuccess && rc2 == REDUX_OK)
                e = cudaMemcpyAsync(h_ooff + c.first + k, d_ooff + c.first + k, (c.count + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess && rc2 == REDUX_OK)
                e = cudaMemcpyAsync(h_status + c.first, d_status + c.first, c.count * sizeof(int32_t), cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess && rc2 == REDUX_OK) e = cudaEventRecord(evs.ev[k], s);
            if (rc2 != REDUX_OK) return rc2;
            if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(ctx, REDUX_CUDA_ERROR, "encode pipeline enqueue", e); }
            prog.advance();
        }
        return REDUX_OK;
    };
    int feeder_rc = REDUX_OK;
    std::thread feeder;
    if (staged) {
        feeder = std::thread([&] { DeviceGuard fg(d->device); feeder_rc = enqueue_all(); prog.finish(); });
    } else {
        feeder_rc = enqueue_all();
        prog.finish();
        if (feeder_rc != REDUX_OK) { drain(d); return feeder_rc; }
        tr.mark("encode: all chunks enqueued");
    }
    // in order: offsets of chunk k become shard-local offsets; its bytes go out while later chunks run
    DownStager down{d->ring_down, ctx->pool, d->copy, {}, 0};
    uint64_t pos = 0;
    // copies the prefix of chunk k that fits the caller's buffer to out + at
    auto place = [&](size_t k, uint64_t at) -> cudaError_t {
        uint64_t nbytes = res->chunk_total[k];
        if (at >= out_cap) return cudaSuccess;
        if (at + nbytes > out_cap) nbytes = out_cap - at;
        if (!nbytes) return cudaSuccess;
        if (stage_out) return down.push(out + at, d_out + res->chunk_base[k], nbytes);
        return cudaMemcpyAsync(out + at, d_out + res->chunk_base[k], nbytes, cudaMemcpyDeviceToHost, d->copy);
    };
    cudaError_t derr = cudaSuccess;                         // first error of this (draining) thread
    const char *dwhat = "encode pipeline";
    bool other_failed = false;
    size_t k_done = 0;
    for (; k_done < nc; ++k_done) {
        const size_t k = k_done;
        const Shard c = res->chunks[k];
        if (!prog.wait_for(k)) break;                       // the feeder gave up: its code is the call's
        if (stage_out && (derr = down.retire_while_pending(evs.ev[k])) != cudaSuccess) break;
        if ((derr = cudaEventSynchronize(evs.ev[k])) != cudaSuccess) break;
        tr.mark("encode: chunk done", (long)k);
        const uint64_t *lo = h_ooff + c.first + k;
        for (uint64_t i = 0; i <= c.count; ++i) res->local_off[c.first + i] = pos + lo[i];
        std::memcpy(status + c.first, h_status + c.first, c.count * sizeof(int32_t));
        res->chunk_total[k] = lo[c.count];
        if (streaming && (derr = place(k, pos)) != cudaSuccess) { dwhat = "encode pipeline D2H"; break; }
        pos += lo[c.count];
    }
    if (k_done == nc) {
        res->total = pos;
        if (sync) sync->publish(g_index, pos);
        if (!streaming) {
            uint64_t at = 0;
            if (!sync->base_of(g_index, &at)) other_failed = true;      // another shard failed: its code is the call's
            else {
                tr.mark("encode: base known");
                for (size_t k = 0; k < nc && derr == cudaSuccess; ++k) {
                    if ((derr = place(k, at)) != cudaSuccess) dwhat = "encode pipeline D2H";
                    at += res->chunk_total[k];
                }
            }
        }
        if (derr == cudaSuccess && !other_failed) {
            derr = stage_out ? down.flush() : cudaStreamSynchronize(d->copy);
            if (derr != cudaSuccess) dwhat = "encode pipeline D2H";
        }
    }
    if (feeder.joinable()) {
        if (derr != cudaSuccess || other_failed) prog.stop.store(true);
        feeder.join();
    }
    if (feeder_rc != REDUX_OK) { drain(d); return feeder_rc; }
    if (other_failed) { drain(d); return REDUX_OK; }
    if (derr != cudaSuccess) { drain(d); (void)cudaGetLastError(); return fail(ctx, REDUX_CUDA_ERROR, dwhat, derr); }
    tr.mark("encode: last D2H done");
    return REDUX_OK;
}

}  // namespace

extern "C" int redux_encode_batch(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                                  const uint8_t *in, const uint64_t *in_offsets, uint64_t n_blocks,
                                  uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    int rc;
    if ((rc = check_kind(ctx, model_kind))) return rc;
    Plan probe;
    if ((rc = make_plan(ctx, params, 0, &probe))) return rc;
    if (!in_offsets || !out_offsets || (n_blocks && !status)) return fail(ctx, REDUX_INVALID_INPUT, "NULL buffer");
    out_offsets[0] = 0;
    if (n_blocks == 0) return REDUX_OK;

    if (needs_staging(ctx, in, in_offsets[n_blocks] - in_offsets[0]) || needs_staging(ctx, out, out_capacity)) ensure_pool(ctx);
    const size_t nd = std::min<uint64_t>(ctx->devs.size(), n_blocks);
    std::vector<Shard> shards = make_shards(n_blocks, nd);
    std::vector<EncShardOut> res(nd);
    std::vector<int> rcs(nd, REDUX_OK);
    ShardSync sync(nd);
    for_each_device(ctx, nd, rcs, [&](redux_ctx *view, DeviceState *d, size_t g) {
        const int r = encode_shard(view, d, params, in, in_offsets, shards[g], out, out_capacity,
                                   status + shards[g].first, &res[g], nd > 1 ? &sync : nullptr, g);
        if (r != REDUX_OK) sync.abort();
        return r;
    });
    for (size_t g = 0; g < nd; ++g) if (rcs[g]) return rcs[g];

    // global offsets (the bytes are already in place: every shard copied its own)
    uint64_t base = 0;
    for (size_t g = 0; g < nd; ++g) {
        for (uint64_t i = 0; i <= shards[g].count; ++i) out_offsets[shards[g].first + i] = base + res[g].local_off[i];
        base += res[g].total;
    }
    if (base > out_capacity) {
        for (uint64_t i = 0; i < n_blocks; ++i)
            if (out_offsets[i + 1] > out_capacity) status[i] = REDUX_OUT_CAPACITY;
        return fail(ctx, REDUX_OUT_CAPACITY, "output buffer too small for the compressed batch");
    }
    for (uint64_t i = 0; i < n_blocks; ++i) if (status[i]) return status[i];
    return REDUX_OK;
}

namespace {

// One device's shard of redux_decode_batch: chunk k runs
//     H2D(compressed bytes) -> decode -> D2H(decoded slots) -> D2H(lengths, consumed, status)
// (H2D on the shared h2d stream, the rest on the chunk's own stream); nothing depends on another chunk or shard.
int decode_shard(redux_ctx *ctx, DeviceState *d, const redux_params_t *p, const uint8_t *comp,
                 const uint64_t *comp_off, Shard sh, uint8_t *raw, const uint64_t *raw_off,
                 uint64_t *raw_lens, uint64_t *consumed, int32_t *status)
{
    Trace tr;
    DeviceGuard g(d->device);
    const uint64_t cbase = comp_off[sh.first], cbytes = comp_off[sh.first + sh.count] - cbase;
    const uint64_t rbase = raw_off[sh.first], rbytes = raw_off[sh.first + sh.count] - rbase;
    std::vector<uint64_t> rel(2 * (sh.count + 1));            // [crel | rrel]
    uint64_t *crel = rel.data(), *rrel = rel.data() + sh.count + 1;
    uint64_t max_len = 0;
    for (uint64_t i = 0; i <= sh.count; ++i) {
        crel[i] = comp_off[sh.first + i] - cbase;
        rrel[i] = raw_off[sh.first + i] - rbase;
        if (i) {
            if (crel[i] < crel[i - 1] || rrel[i] < rrel[i - 1]) return fail(ctx, REDUX_INVALID_INPUT, "offsets not monotonic");
            max_len = std::max(max_len, rrel[i] - rrel[i - 1]);
        }
    }
    Plan pl;
    int rc = make_plan(ctx, p, max_len, &pl);
    if (rc) return rc;
    pl.warp = !pl.generic && !pl.pretrained && choose_warp(ctx);
    const std::vector<Shard> chunks = pl.generic ? std::vector<Shard>{{0, sh.count}} : make_chunks(sh.count, -1);
    const size_t nc = chunks.size();
    CU_TRY(ctx, d->st_in.reserve(cbytes + 32));
    CU_TRY(ctx, d->st_off.reserve(rel.size() * sizeof(uint64_t)));
    CU_TRY(ctx, d->st_out.reserve(rbytes + 32));
    CU_TRY(ctx, d->st_aux0.reserve(sh.count * sizeof(uint64_t)));
    CU_TRY(ctx, d->st_aux1.reserve(sh.count * sizeof(uint64_t)));
    CU_TRY(ctx, d->st_status.reserve(sh.count * sizeof(int32_t)));
    CU_TRY(ctx, d->pin_aux0.reserve(sh.count * sizeof(uint64_t)));
    CU_TRY(ctx, d->pin_aux1.reserve(sh.count * sizeof(uint64_t)));
    CU_TRY(ctx, d->pin_status.reserve(sh.count * sizeof(int32_t)));
    const void *magic = nullptr;
    if ((rc = get_magic(ctx, d, d->pipe[0], pl, &magic))) return rc;
    if ((rc = prepare_generic(ctx, d, d->pipe[0], p, sh.count, &pl))) return rc;
    EventSet evs;                       // [0, nc): chunk input on the device; [nc, 2nc): chunk decoded
    CU_TRY(ctx, evs.create(2 * nc));
    // pageable caller memory: see encode_shard
    const bool stage_in = needs_staging(ctx, comp, cbytes), stage_out = needs_staging(ctx, raw, rbytes);
    const bool staged = stage_in || stage_out;
    if (stage_in) CU_TRY(ctx, ensure_ring(ctx, &d->ring_up));
    if (stage_out) CU_TRY(ctx, ensure_ring(ctx, &d->ring_down));
    CU_TRY(ctx, cudaMemcpyAsync(d->st_off.p, rel.data(), rel.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, d->h2d));
    uint8_t *d_comp = (uint8_t *)d->st_in.p, *d_raw = (uint8_t *)d->st_out.p;
    uint64_t *d_coff = (uint64_t *)d->st_off.p, *d_roff = d_coff + sh.count + 1;
    uint64_t *d_len = (uint64_t *)d->st_aux0.p, *d_cons = (uint64_t *)d->st_aux1.p;
    int32_t *d_status = (int32_t *)d->st_status.p;
    uint64_t *h_len = (uint64_t *)d->pin_aux0.p, *h_cons = (uint64_t *)d->pin_aux1.p;
    int32_t *h_status = (int32_t *)d->pin_status.p;
    ChunkProgress prog;
    auto enqueue_all = [&]() -> int {
        int up_slot = 0;
        for (size_t k = 0; k < nc && !prog.stop.load(std::memory_order_relaxed); ++k) {
            const Shard c = chunks[k];
            cudaStream_t s = d->pipe[k % pipe_streams()];
            int rc2 = REDUX_OK;
            cudaError_t e = cudaSuccess;
            const uint64_t c0 = crel[c.first], c1 = crel[c.first + c.count];
            const uint64_t r0 = rrel[c.first], r1 = rrel[c.first + c.count];
            if (c1 > c0) e = stage_in ? staged_h2d(d->ring_up, ctx->pool, d->h2d, d_comp + c0, comp + cbase + c0, c1 - c0, &up_slot, &prog.stop)
                                      : cudaMemcpyAsync(d_comp + c0, comp + cbase + c0, c1 - c0, cudaMemcpyHostToDevice, d->h2d);
            if (e == cudaSuccess) e = cudaEventRecord(evs.ev[k], d->h2d);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(s, evs.ev[k], 0);
            if (e == cudaSuccess)
                rc2 = decode_launch(ctx, d->device, s, pl, magic, d_comp, d_coff + c.first, c.count, d_raw,
                                    d_roff + c.first, d_len + c.first, d_cons + c.first, d_status + c.first);
            // the whole slot range of the chunk goes back; bytes beyond raw_lens[i] inside a slot are unspecified
            // (into pageable memory: by the drainer below, through the ring)
            if (e == cudaSuccess && rc2 == REDUX_OK && stage_out) e = cudaEventRecord(evs.ev[nc + k], s);
            if (e == cudaSuccess && rc2 == REDUX_OK && !stage_out && r1 > r0)
                e = cudaMemcpyAsync(raw + rbase + r0, d_raw + r0, r1 - r0, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess && rc2 == REDUX_OK)
                e = cudaMemcpyAsync(h_len + c.first, d_len + c.first, c.count * sizeof(uint64_t), cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess && rc2 == REDUX_OK)
                e = cudaMemcpyAsync(h_cons + c.first, d_cons + c.first, c.count * sizeof(uint64_t), cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess && rc2 == REDUX_OK)
                e = cudaMemcpyAsync(h_status + c.first, d_status + c.first, c.count * sizeof(int32_t), cudaMemcpyDeviceToHost, s);
            if (rc2 != REDUX_OK) return rc2;
            if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(ctx, REDUX_CUDA_ERROR, "decode pipeline enqueue", e); }
            prog.advance();
        }
        return REDUX_OK;
    };
    int feeder_rc = REDUX_OK;
    std::thread feeder;
    if (staged) {
        feeder = std::thread([&] { DeviceGuard fg(d->device); feeder_rc = enqueue_all(); prog.finish(); });
    } else {
        feeder_rc = enqueue_all();
        prog.finish();
    }
    cudaError_t derr = cudaSuccess;
    if (stage_out) {
        // chunk k's decoded slots leave on the copy stream once its kernel is done, piece by piece through the ring
        DownStager down{d->ring_down, ctx->pool, d->copy, {}, 0};
        for (size_t k = 0; k < nc && derr == cudaSuccess; ++k) {
            if (!prog.wait_for(k)) break;
            const Shard c = chunks[k];
            const uint64_t r0 = rrel[c.first], r1 = rrel[c.first + c.count];
            if ((derr = cudaStreamWaitEvent(d->copy, evs.ev[nc + k], 0)) != cudaSuccess) break;
            if (r1 > r0) derr = down.push(raw + rbase + r0, d_raw + r0, r1 - r0);
        }
        if (derr == cudaSuccess) derr = down.flush();
    }
    if (feeder.joinable()) {
        if (derr != cudaSuccess) prog.stop.store(true);
        feeder.join();
    }
    if (feeder_rc != REDUX_OK) { drain(d); return feeder_rc; }
    if (derr != cudaSuccess) { drain(d); (void)cudaGetLastError(); return fail(ctx, REDUX_CUDA_ERROR, "decode pipeline D2H", derr); }
    tr.mark("decode: all chunks enqueued");
    for (int i = 0; i < kPipeStreams; ++i) { CU_TRY(ctx, cudaStreamSynchronize(d->pipe[i])); tr.mark("decode: stream drained", i); }
    std::memcpy(raw_lens + sh.first, h_len, sh.count * sizeof(uint64_t));
    std::memcpy(consumed + sh.first, h_cons, sh.count * sizeof(uint64_t));
    std::memcpy(status + sh.first, h_status, sh.count * sizeof(int32_t));
    return REDUX_OK;
}

}  // namespace

extern "C" int redux_decode_batch(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                                  const uint8_t *comp, const uint64_t *comp_offsets, uint64_t n_blocks,
                                  uint8_t *raw, const uint64_t *raw_offsets, uint64_t *raw_lens,
                                  uint64_t *consumed, int32_t *status)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    int rc;
    if ((rc = check_kind(ctx, model_kind))) return rc;
    Plan probe;
    if ((rc = make_plan(ctx, params, 0, &probe))) return rc;
    if (n_blocks == 0) return REDUX_OK;
    if (!comp_offsets || !raw_offsets || !raw_lens || !consumed || !status)
        return fail(ctx, REDUX_INVALID_INPUT, "NULL buffer");
    if (needs_staging(ctx, comp, comp_offsets[n_blocks] - comp_offsets[0]) ||
        needs_staging(ctx, raw, raw_offsets[n_blocks] - raw_offsets[0])) ensure_pool(ctx);
    const size_t nd = std::min<uint64_t>(ctx->devs.size(), n_blocks);
    std::vector<Shard> shards = make_shards(n_blocks, nd);
    std::vector<int> rcs(nd, REDUX_OK);
    for_each_device(ctx, nd, rcs, [&](redux_ctx *view, DeviceState *d, size_t g) {
        return decode_shard(view, d, params, comp, comp_offsets, shards[g], raw, raw_offsets,
                            raw_lens, consumed, status);
    });
    for (size_t g = 0; g < nd; ++g) if (rcs[g]) return rcs[g];
    for (uint64_t i = 0; i < n_blocks; ++i) if (status[i]) return status[i];
    return REDUX_OK;
}

// ================================================================================== single stream

extern "C" int redux_compress(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                              const uint8_t *in, uint64_t in_len, uint8_t *out, uint64_t out_capacity,
                              uint64_t *in_count, uint64_t *out_count)
{
    if (in_count) *in_count = 0;
    if (out_count) *out_count = 0;
    uint64_t in_off[2] = {0, in_len}, out_off[2] = {0, 0};
    int32_t st = 0;
    int rc = redux_encode_batch(ctx, model_kind, params, in, in_off, 1, out, out_capacity, out_off, &st);
    if (rc == REDUX_OK || rc == REDUX_OUT_CAPACITY) {
        if (in_count) *in_count = in_len;                 // BitReader::get_count (src/lib.rs:108)
        if (out_count) *out_count = out_off[1];           // BitWriter::get_count
    }
    return rc;
}

extern "C" int redux_decompress(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                                const uint8_t *in, uint64_t in_len, uint8_t *out, uint64_t out_capacity,
                                uint64_t *in_count, uint64_t *out_count)
{
    if (in_count) *in_count = 0;
    if (out_count) *out_count = 0;
    uint64_t comp_off[2] = {0, in_len}, raw_off[2] = {0, out_capacity}, raw_len = 0, consumed = 0;
    int32_t st = 0;
    int rc = redux_decode_batch(ctx, model_kind, params, in, comp_off, 1, out, raw_off, &raw_len, &consumed, &st);
    if (rc == REDUX_OK || rc == REDUX_EOF || rc == REDUX_OUT_CAPACITY) {
        if (in_count) *in_count = consumed;
        if (out_count) *out_count = raw_len;
    }
    return rc;
}

// ================================================================== pre-trained models (8(f) rank 4)

extern "C" int redux_encode_batch_ex(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                                     const uint32_t *model_freq, const uint8_t *in, const uint64_t *in_offsets,
                                     uint64_t n_blocks, uint8_t *out, uint64_t out_capacity,
                                     uint64_t *out_offsets, int32_t *status)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    ctx->model_freq = model_freq;
    const int rc = redux_encode_batch(ctx, model_kind, params, in, in_offsets, n_blocks, out, out_capacity,
                                      out_offsets, status);
    ctx->model_freq = nullptr;
    return rc;
}

extern "C" int redux_decode_batch_ex(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                                     const uint32_t *model_freq, const uint8_t *comp, const uint64_t *comp_offsets,
                                     uint64_t n_blocks, uint8_t *raw, const uint64_t *raw_offsets,
                                     uint64_t *raw_lens, uint64_t *consumed, int32_t *status)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    ctx->model_freq = model_freq;
    const int rc = redux_decode_batch(ctx, model_kind, params, comp, comp_offsets, n_blocks, raw, raw_offsets,
                                      raw_lens, consumed, status);
    ctx->model_freq = nullptr;
    return rc;
}

extern "C" int redux_encode_batch_device_ex(redux_ctx_t *ctx, int device, void *stream, int model_kind,
                                            const redux_params_t *params, const uint32_t *model_freq,
                                            const uint8_t *d_in, const uint64_t *d_in_offsets, uint64_t n_blocks,
                                            uint64_t max_block_len, uint8_t *d_out, uint64_t out_capacity,
                                            uint64_t *d_out_offsets, int32_t *d_status)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    ctx->model_freq = model_freq;               // HOST pointer; uploaded and turned into the start tree on `stream`
    const int rc = redux_encode_batch_device(ctx, device, stream, model_kind, params, d_in, d_in_offsets, n_blocks,
                                             max_block_len, d_out, out_capacity, d_out_offsets, d_status);
    ctx->model_freq = nullptr;
    return rc;
}

extern "C" int redux_decode_batch_device_ex(redux_ctx_t *ctx, int device, void *stream, int model_kind,
                                            const redux_params_t *params, const uint32_t *model_freq,
                                            const uint8_t *d_comp, const uint64_t *d_comp_offsets, uint64_t n_blocks,
                                            uint64_t max_block_len, uint8_t *d_raw, const uint64_t *d_raw_offsets,
                                            uint64_t *d_raw_lens, uint64_t *d_consumed, int32_t *d_status)
{
    if (!ctx) return REDUX_INVALID_INPUT;
    ctx->model_freq = model_freq;
    const int rc = redux_decode_batch_device(ctx, device, stream, model_kind, params, d_comp, d_comp_offsets, n_blocks,
                                             max_block_len, d_raw, d_raw_offsets, d_raw_lens, d_consumed, d_status);
    ctx->model_freq = nullptr;
    return rc;
}
