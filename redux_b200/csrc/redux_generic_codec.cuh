// redux_generic_codec.cuh -- the rest of the Parameters space (SURVEY.md 8(f) rank 4).
//
// The tuned kernels (redux_lane_al.cuh) cover byte symbols with code_bits <= 32, fresh or pre-trained.
// Everything else the reference accepts runs here, still one stream per lane and still bit-exact:
//   * any symbol_bits 1..16 (Parameters::new allows any width, src/model/mod.rs:63-81; the reference's
//     model tests run 4 and 12, src/model/tests.rs:95-251).  Symbols are read MSB-first across byte
//     boundaries exactly like BitReader::read_bits (src/bitio/mod.rs:78-120): a trailing partial symbol
//     is consumed and dropped (it becomes EOF, src/codec.rs:106-110), and the decoder writes symbols with
//     BitWriter::write_bits but never flushes (src/codec.rs:164-176), so trailing bits that do not fill
//     a byte are lost -- both quirks of the reference are reproduced, not repaired;
//   * any code_bits (64-bit coder state; products stay below 2^64 because code_bits + freq_bits <= 64,
//     src/model/mod.rs:64; the divisions by the total use the 65-bit magic of redux_common.cuh);
//   * with those, a model that was TRAINED before compress()/decompress() received it (trained byte models
//     with code_bits <= 32 run on the tuned kernels): the reference takes a
//     Box<Model> (src/lib.rs:102) whose get_frequency() has possibly been called already
//     (src/model/mod.rs:23-25); its state is exactly the per-symbol frequency vector, handed over here
//     as the Fenwick tree built from it.
// The frequency table is the reference's tree itself (adaptive_tree.rs:34-136: u32 nodes, index 0 unused,
// nodes 1..symbol_count), one column per thread: [node][thread], so that the 32 data-dependent walks of a
// warp touch 32 different banks / one coalesced row.  Alphabets of up to 7 bits (130 nodes, 66 KB per CTA)
// keep their columns in SHARED memory; wider ones in GLOBAL memory (L2-latency bound), where a thread codes
// blocks tid, tid + T, ... with the same column.  This is the completeness path: no reciprocal tables, loops
// as the reference writes them.
#pragma once
#include "redux_common.cuh"
#include "redux_lane_codec.cuh"

namespace rdx {

constexpr uint32_t kGenericMaxSymbolBits = 16;
constexpr int kGenericThreads = 128;
constexpr uint32_t kGenericSmemSymbolBits = 7;      // up to this width the Fenwick columns live in shared memory
// dynamic shared memory of the generic kernels: [nsym + 1][kGenericThreads] u32, or nothing
RDX_HD size_t generic_smem_bytes(uint32_t s) {
    return s <= kGenericSmemSymbolBits ? ((size_t)(1u << s) + 2) * kGenericThreads * sizeof(uint32_t) : 0;
}

struct GenericJob {
    const uint8_t *in;          // encode: raw bytes / decode: compressed bytes
    const uint64_t *in_off;     // [n_blocks+1]
    uint64_t n_blocks;
    // encode output
    uint8_t *slots; uint64_t slot_stride; uint32_t *sizes;
    // decode output
    uint8_t *raw; const uint64_t *raw_off; uint64_t *raw_len; uint64_t *consumed;
    int32_t *status;
    uint32_t *tabs;             // [nsym + 1][n_threads] Fenwick columns
    const uint32_t *init_tree;  // [nsym + 1] tree every block starts from (fresh: tree[i] = lowbit(i))
    uint32_t init_total;        // its total frequency; with `models`: the smallest start total of the call
    BlockModels models;         // a start model per block: block i starts from its row instead of init_tree
    uint32_t s, f, c;
    uint32_t n_threads;
    // 65-bit reciprocals (redux_common.cuh, make_magic65) of the totals init_total .. init_total + magic_len - 1: a
    // block's total is a function of its start total and its position, so the two divisions by it
    // (src/codec.rs:59-60 / :133-134) are two multiplications; the decoder's division by the range (:131) stays a
    // division
    const Magic64 *magic; uint32_t magic_len;
};

// reciprocal of the total `count` (magic_base <= count < magic_base + magic_len by construction of the table)
__device__ __forceinline__ Magic64 generic_magic(const GenericJob &job, uint32_t count) {
    uint32_t i = count - job.init_total;
    if (i >= job.magic_len) i = job.magic_len - 1;      // only if the caller's max_block_len understated a block: stay in bounds
    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(job.magic + i));
    Magic64 g; g.m = ((uint64_t)v.y << 32) | v.x; g.sh = v.z; g.pad = 0;
    return g;
}

// Row of block blk (0 without a table), or false when its index is out of range.
__device__ __forceinline__ bool generic_row(const GenericJob &job, uint64_t blk, uint32_t &m) {
    m = 0;
    return !job.models.start || block_row(job.models, blk, m);
}

// The reference's AdaptiveTreeModel over one column of `tabs`.
struct GenericTree {
    uint32_t *t; uint32_t stride;       // node i at t[i * stride]
    uint32_t nsym, eof, total, fmax;

    // start from row m of the call's models (generic_row checked it), or from init_tree without a table
    __device__ __forceinline__ void reset(const GenericJob &job, uint32_t tid, uint32_t *smem_cols, uint32_t m) {
        if (job.s <= kGenericSmemSymbolBits) { t = smem_cols + threadIdx.x; stride = kGenericThreads; }
        else                                 { t = job.tabs + tid; stride = job.n_threads; }
        eof = 1u << job.s; nsym = eof + 1;
        fmax = (uint32_t)(((uint64_t)1 << job.f) - 1);
        total = job.models.start ? job.models.start[m].x : job.init_total;
        const uint32_t *init = job.models.start ? job.models.trees + (size_t)m * (nsym + 1) : job.init_tree;
        for (uint32_t i = 0; i <= nsym; ++i) t[(size_t)i * stride] = init[i];
    }
    // get_frequency_single (adaptive_tree.rs:51-59)
    __device__ __forceinline__ uint32_t prefix(uint32_t i) const {
        uint32_t sum = 0;
        for (; i > 0; i &= i - 1) sum += t[(size_t)i * stride];
        return sum;
    }
    // update (adaptive_tree.rs:83-92): frozen once total == freq_max
    __device__ __forceinline__ void update(uint32_t sym) {
        if (total >= fmax) return;
        for (uint32_t i = sym + 1; i <= nsym; i += i & (0u - i)) t[(size_t)i * stride] += 1;
        total += 1;
    }
    // get_symbol's descent (adaptive_tree.rs:115-127)
    __device__ __forceinline__ uint32_t find(uint64_t value) const {
        uint32_t i = 0;
        for (uint32_t m = eof; m > 0 && i < eof; m >>= 1) {
            const uint32_t tv = t[(size_t)(i + m) * stride];
            if (value >= tv) { i += m; value -= tv; }
        }
        return i;
    }
};

// BitWriter::write_bits over a byte slot of arbitrary alignment, WITHOUT the final flush_bits
// (decompress_stream never calls it, src/codec.rs:164-176).
struct SymbolSink {
    uint8_t *dst; uint64_t cap, written; uint32_t acc, nb; bool full;
    __device__ __forceinline__ void init(uint8_t *d, uint64_t c) { dst = d; cap = c; written = 0; acc = 0; nb = 0; full = false; }
    __device__ __forceinline__ void put(uint32_t sym, uint32_t bits) {      // bits <= 16, nb <= 7 before
        acc = (acc << bits) | sym;
        nb += bits;
        while (nb >= 8) {
            if (written == cap) { full = true; return; }                     // the byte has nowhere to go
            nb -= 8;
            dst[written++] = (uint8_t)(acc >> nb);
        }
    }
};

__global__ void __launch_bounds__(kGenericThreads)
encode_generic_kernel(const GenericJob job)
{
    extern __shared__ uint32_t gen_cols[];
    const uint32_t tid = blockIdx.x * kGenericThreads + threadIdx.x;
    if (tid >= job.n_threads) return;
    const uint32_t c = job.c, s = job.s;
    const uint64_t maxv = (c == 64) ? ~(uint64_t)0 : ((((uint64_t)1) << c) - 1);
    GenericTree tree;
    for (uint64_t blk = tid; blk < job.n_blocks; blk += job.n_threads) {
        uint32_t m;
        if (!generic_row(job, blk, m)) { job.sizes[blk] = 0; job.status[blk] = kStatusInvalidInput; continue; }
        const uint64_t off = job.in_off[blk];
        const uint64_t len = job.in_off[blk + 1] - off;
        if (len >= (1ull << 29)) { job.sizes[blk] = 0; job.status[blk] = 5; continue; }
        tree.reset(job, tid, gen_cols, m);
        BitSource src;                                       // read_bits(symbol_bits) over the raw bytes
        src.init(job.in + off, (uint32_t)len);
        BitSink sink;
        sink.init(job.slots + blk * job.slot_stride);
        uint64_t low = 0, high = maxv;
        uint32_t pend = 0;
        for (;;) {
            // src/codec.rs:106-110: Err(Eof) -- also on a trailing partial symbol -- codes symbol_eof
            const bool data = src.has(s);
            const uint32_t sym = data ? src.take(s) : tree.eof;
            const uint64_t count = tree.total;               // read before the lookup mutates it (:56-57)
            const uint64_t cl = tree.prefix(sym), ch = tree.prefix(sym + 1);
            tree.update(sym);
            const uint64_t range = high - low + 1;           // :58 (2^64 cannot occur: c <= 61)
            const Magic64 g = generic_magic(job, (uint32_t)count);
            const uint64_t h2 = low + div_magic65(range * ch, g) - 1;
            const uint64_t l2 = low + div_magic65(range * cl, g);
            const Renorm<uint64_t> r = renorm<uint64_t>(l2, h2, c);
            if (r.n1) { sink.put_code(l2 >> (c - r.n1), r.n1, pend); pend = r.k; }
            else pend += r.k;
            low = r.low; high = r.high;
            if (!data) {                                     // :91-99
                const uint32_t extra = c - (r.n1 + r.k);
                if (extra) sink.put_code(low >> (c - extra), extra, pend);
                break;
            }
        }
        job.sizes[blk] = sink.finish();
        job.status[blk] = 0;
    }
}

__global__ void __launch_bounds__(kGenericThreads)
decode_generic_kernel(const GenericJob job)
{
    extern __shared__ uint32_t gen_cols[];
    const uint32_t tid = blockIdx.x * kGenericThreads + threadIdx.x;
    if (tid >= job.n_threads) return;
    const uint32_t c = job.c, s = job.s;
    const uint64_t maxv = (c == 64) ? ~(uint64_t)0 : ((((uint64_t)1) << c) - 1);
    const uint64_t body = maxv >> 1, half = body + 1;
    GenericTree tree;
    for (uint64_t blk = tid; blk < job.n_blocks; blk += job.n_threads) {
        uint32_t m;
        if (!generic_row(job, blk, m)) {
            job.raw_len[blk] = 0; job.consumed[blk] = 0; job.status[blk] = kStatusInvalidInput;
            continue;
        }
        const uint64_t coff = job.in_off[blk];
        const uint64_t clen = job.in_off[blk + 1] - coff;
        const uint64_t roff = job.raw_off[blk];
        if (clen >= (1ull << 29)) { job.raw_len[blk] = 0; job.consumed[blk] = 0; job.status[blk] = 5; continue; }
        tree.reset(job, tid, gen_cols, m);
        BitSource src;
        src.init(job.in + coff, (uint32_t)clen);
        SymbolSink out;
        out.init(job.raw + roff, job.raw_off[blk + 1] - roff);
        uint64_t low = 0, high = maxv, value = 0;
        int32_t st = 0;
        if (!src.has(c)) { st = 1; src.left = 0; }            // src/codec.rs:124-127
        else value = src.take64(c);
        while (st == 0) {
            const uint64_t range = high - low + 1;
            const uint64_t count = tree.total;
            const uint64_t v = ((value - low + 1) * count - 1) / range;       // :131
            const uint32_t sym = tree.find(v);
            const uint64_t cl = tree.prefix(sym), ch = tree.prefix(sym + 1);
            if (v >= ch) { st = 2; break; }                   // get_symbol's InvalidInput (unreachable, kept)
            tree.update(sym);
            const Magic64 g = generic_magic(job, (uint32_t)count);
            high = low + div_magic65(range * ch, g) - 1;      // :133-134
            low = low + div_magic65(range * cl, g);
            if (sym == tree.eof) break;                       // :136-138
            const Renorm<uint64_t> r = renorm<uint64_t>(low, high, c);
            const uint32_t n = r.n1 + r.k;
            if (!src.has(n)) { st = 1; src.left = 0; break; } // Err(Eof) inside get_bit
            const uint64_t chunk = src.take64(n);
            uint64_t v1 = (r.n1 >= 64) ? 0 : ((value << r.n1) & maxv);
            v1 |= chunk >> r.k;
            value = (v1 & half) | ((v1 << r.k) & body) | (chunk & ((((uint64_t)1) << r.k) - 1));
            low = r.low; high = r.high;
            out.put(sym, s);                                  // write_bits(symbol, symbol_bits) (:171)
            if (out.full) { st = 6; break; }
        }
        job.raw_len[blk] = out.written;
        job.consumed[blk] = (src.used() + 7) >> 3;
        job.status[blk] = st;
    }
}

// Fenwick trees of n_models frequency vectors freq[m * nsym ..][0..nsym) (adaptive_tree.rs layout: node i covers the
// lowbit(i) symbols ending at symbol i-1) into tree[m * (nsym + 1) ..], nsym + 1 entries each; freq == NULL: one fresh
// model (every frequency 1).  The totals are summed by the host.  One thread per node; tiny, runs once per call.
__global__ void build_tree_kernel(const uint32_t *freq, uint32_t nsym, uint32_t *tree, uint32_t n_models = 1)
{
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= (uint64_t)n_models * (nsym + 1)) return;
    const uint32_t m = (uint32_t)(k / (nsym + 1)), i = (uint32_t)(k % (nsym + 1));
    const uint32_t *fm = freq ? freq + (size_t)m * nsym : nullptr;
    uint32_t sum = 0;
    if (i > 0) {
        const uint32_t lb = i & (0u - i);
        for (uint32_t j = i - lb; j < i; ++j) sum += fm ? fm[j] : 1u;
    }
    tree[k] = sum;
}

}  // namespace rdx
