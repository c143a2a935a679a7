/*
 * redux_b200.h -- C ABI of the B200-native batched adaptive arithmetic coder.
 *
 * Drop-in boundary for ONE path of peterbudai/redux: redux::compress / redux::decompress
 * (src/lib.rs:102-120) over AdaptiveLinearModel / AdaptiveTreeModel
 * (src/model/adaptive_linear.rs:21, src/model/adaptive_tree.rs:36) built from
 * Parameters::new(symbol_bits, freq_bits, code_bits) (src/model/mod.rs:63-81), producing the
 * reference's headerless MSB-first bitstream (src/bitio/mod.rs:148-198) byte for byte.
 *
 * Plain pointers and sizes only; no torch / C++ types.  The library is a CUDA (sm_100a) product:
 * there is NO CPU fallback.  Every entry point that computes returns REDUX_CUDA_ERROR when no
 * usable device exists.  INTEGRATION.md shows the Rust `extern "C"` stub that binds these.
 */
#ifndef REDUX_B200_H
#define REDUX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- error codes: 0-3 mirror redux::Error (src/lib.rs:57-64); 4-6 are new to the device path */
#define REDUX_OK             0
#define REDUX_EOF            1  /* Error::Eof: compressed stream ended early (src/bitio/mod.rs:106-108) */
#define REDUX_INVALID_INPUT  2  /* Error::InvalidInput (src/model/mod.rs:64-65, src/bitio/mod.rs:79,149) */
#define REDUX_IO_ERROR       3  /* Error::IoError */
#define REDUX_CUDA_ERROR     4  /* CUDA runtime failure / no device; see redux_ctx_last_error() */
#define REDUX_UNSUPPORTED    5  /* valid Parameters the device path does not implement (symbol_bits > 16) */
#define REDUX_OUT_CAPACITY   6  /* an output buffer was too small (the streaming analogue is IoError) */

/* ---- model kinds: which reference constructor the caller would have used */
#define REDUX_MODEL_LINEAR 0    /* AdaptiveLinearModel::new (src/model/adaptive_linear.rs:21-30) */
#define REDUX_MODEL_TREE   1    /* AdaptiveTreeModel::new   (src/model/adaptive_tree.rs:36-48)   */

/* ---- stream-to-thread mapping (new; the reference is single-threaded) */
#define REDUX_SCHED_AUTO 0      /* choose by batch shape: encode = SPLIT below 512 streams, else LANE; decode = LANE */
#define REDUX_SCHED_LANE 1      /* one stream per lane, 32 streams per warp: throughput mapping */
#define REDUX_SCHED_WARP 2      /* one stream per warp, lanes cooperate per symbol: latency mapping */
#define REDUX_SCHED_SPLIT 3     /* encode: model phase parallel over the positions of a stream, then one coder warp
                                   per stream (few long streams); decode: as REDUX_SCHED_WARP */

/* Parameters::new arguments (src/model/mod.rs:63). */
typedef struct redux_params {
    uint32_t symbol_bits;
    uint32_t freq_bits;
    uint32_t code_bits;
} redux_params_t;

/* struct Parameters (src/model/mod.rs:33-59), all derived fields. */
typedef struct redux_parameters {
    uint64_t symbol_bits, symbol_eof, symbol_count;
    uint64_t freq_bits, freq_max;
    uint64_t code_bits, code_min, code_one_fourth, code_half, code_three_fourths, code_max;
} redux_parameters_t;

typedef struct redux_ctx redux_ctx_t;

/* Parameters::new (src/model/mod.rs:63-81): REDUX_OK or REDUX_INVALID_INPUT, same rejection rule.
 * `out` may be NULL (validation only). Pure host arithmetic, no device needed. */
int redux_parameters_new(uint32_t symbol_bits, uint32_t freq_bits, uint32_t code_bits,
                         redux_parameters_t *out);

/* REDUX_OK if the device path implements these parameters, REDUX_INVALID_INPUT if Parameters::new
 * rejects them, REDUX_UNSUPPORTED otherwise. */
int redux_params_supported(const redux_params_t *params);

/* Display strings of redux::Error (src/lib.rs:66-73) for codes 1-3; own text for 0 and 4-6. */
const char *redux_error_string(int code);

/* Upper bound of one compressed stream: (in_len+1 symbols) * code_bits bits, rounded up to bytes
 * (each coded symbol, EOF included, emits at most code_bits bits). */
uint64_t redux_compress_bound(uint64_t in_len, uint32_t code_bits);
/* The same for any symbol width: floor(8*in_len / symbol_bits) data symbols (a trailing partial symbol is
 * dropped by the reference's reader, src/bitio/mod.rs:94-108 + src/codec.rs:106-110) plus EOF. */
uint64_t redux_compress_bound_ex(uint64_t in_len, uint32_t symbol_bits, uint32_t code_bits);

/* ---- process-wide set-up (optional).  The host-buffer API pipelines ~18 CUDA streams per device; CUDA maps streams
 * onto CUDA_DEVICE_MAX_CONNECTIONS hardware queues (default 8), and streams that share a queue serialise.
 * redux_process_init() sets that variable to 32 unless the application already set it, and returns the value in
 * force.  It only has an effect BEFORE the process creates its first CUDA context, it changes the environment of
 * the whole process, and nothing in this library calls it implicitly: an application that manages the variable
 * itself simply does not call it (the end-to-end calls then run ~20 % slower, the results are identical). */
int redux_process_init(void);

/* ---- host memory for the host-buffer API.  redux_encode_batch / redux_decode_batch copy straight from / to the
 * caller's pointers (the reference streams through &mut io::Read / io::Write, src/lib.rs:102-109; a binding lands
 * that in a byte buffer, INTEGRATION.md 3).  Page-locked buffers make those copies asynchronous so the chunk
 * pipeline overlaps them with the kernels.  Pageable buffers (a plain Vec<u8>) work too: the library stages them
 * itself through a small ring of pinned slots filled / emptied by a few host copy threads (redux_ctx_set_staging),
 * so the pipeline stays asynchronous at the speed the host can memcpy (bench.py reports pinned, registered, staged
 * and driver-staged numbers).  redux_host_alloc returns page-locked memory usable with every device;
 * redux_host_register page-locks an existing allocation (e.g. a long-lived Vec<u8>) in place -- pinning costs
 * ~0.1 ms per MiB, so do it once. */
int redux_host_alloc(size_t bytes, void **out);
int redux_host_free(void *p);
int redux_host_register(void *p, size_t bytes);
int redux_host_unregister(void *p);

/* ---- context: owns per-device streams and workspaces. Not thread-safe (one caller at a time).
 * devices == NULL or n_devices <= 0: use the current device only. */
int  redux_ctx_create(const int *devices, int n_devices, redux_ctx_t **ctx);
void redux_ctx_destroy(redux_ctx_t *ctx);
int  redux_ctx_device_count(const redux_ctx_t *ctx);
const char *redux_ctx_last_error(const redux_ctx_t *ctx);
/* REDUX_SCHED_*; default AUTO. */
int  redux_ctx_set_schedule(redux_ctx_t *ctx, int sched);
/* How redux_encode_batch / redux_decode_batch treat caller buffers that are neither page-locked nor registered.
 * enable != 0 (default): transfers of at least min_bytes go through `slots` pinned slots of piece_bytes each per
 * device and direction, copied by `threads` host threads (0 = chosen from the core count) created on first use and
 * joined by redux_ctx_destroy; enable == 0: such pointers are handed to cudaMemcpyAsync as they are (the driver's own
 * synchronous staging).  A zero size / count keeps the current value.  Defaults: 8 MiB, 8 MiB, 4 slots.  Results
 * are identical either way.  Call it between batch calls, not during one. */
int  redux_ctx_set_staging(redux_ctx_t *ctx, int enable, size_t min_bytes, size_t piece_bytes, int slots, int threads);
/* Number of kernels this context has launched so far (for bench.py's gpu_launches). */
uint64_t redux_ctx_kernel_launches(const redux_ctx_t *ctx);

/* Per-kernel device timing (measurement aid): when enabled, every kernel launch is bracketed by CUDA
 * events on the stream it is launched on. redux_ctx_timing_collect() waits for the recorded launches,
 * adds their durations per kernel kind into ms[REDUX_KERNEL_KINDS] / counts[REDUX_KERNEL_KINDS] and
 * forgets them. */
#define REDUX_KERNEL_ENCODE   0
#define REDUX_KERNEL_SCAN     1
#define REDUX_KERNEL_COMPACT  2
#define REDUX_KERNEL_DECODE   3
#define REDUX_KERNEL_GENERATE 4
#define REDUX_KERNEL_KINDS    5
int redux_ctx_timing_enable(redux_ctx_t *ctx, int on);
int redux_ctx_timing_collect(redux_ctx_t *ctx, double *ms, uint64_t *counts);

/* ---- single stream: the literal replacement of redux::compress / redux::decompress
 * (src/lib.rs:102-109 / :113-120) for in-memory streams. *in_count / *out_count are the returned
 * tuple (bytes read from input, bytes written to output). A fresh model is built per call, as the
 * reference consumes its Box<Model>. Host pointers. */
int redux_compress(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                   const uint8_t *in, uint64_t in_len, uint8_t *out, uint64_t out_capacity,
                   uint64_t *in_count, uint64_t *out_count);
int redux_decompress(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                     const uint8_t *in, uint64_t in_len, uint8_t *out, uint64_t out_capacity,
                     uint64_t *in_count, uint64_t *out_count);

/* ---- batch, host buffers (the end-to-end path: H2D + kernels + D2H inside the call).
 * Block i is an independent reference stream: compress() of in[in_offsets[i] .. in_offsets[i+1]).
 * Blocks are sharded over the context's devices by contiguous index ranges (no collective).
 *
 * encode: out receives the streams back to back; out_offsets[n_blocks+1] receives their byte
 *   offsets (out_offsets[i+1]-out_offsets[i] = second element of compress()'s tuple); status[i] is
 *   the per-block code. Returns the first non-OK code (REDUX_OUT_CAPACITY if out is too small). */
int redux_encode_batch(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                       const uint8_t *in, const uint64_t *in_offsets, uint64_t n_blocks,
                       uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status);

/* decode: stream i = comp[comp_offsets[i] .. comp_offsets[i+1]); its symbols go to
 *   raw[raw_offsets[i] ..) with capacity raw_offsets[i+1]-raw_offsets[i]; raw_lens[i] = bytes written
 *   (second tuple element of decompress()), consumed[i] = compressed bytes read (first element).
 *   A truncated stream gives status REDUX_EOF with the bytes decoded so far left in place; bytes beyond
 *   raw_lens[i] inside slot i are unspecified.  A full slot gives REDUX_OUT_CAPACITY (unless the stream ends or is
 *   cut first); consumed[i] then includes the bits of the symbol that found no room, as the reference's reader. */
int redux_decode_batch(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                       const uint8_t *comp, const uint64_t *comp_offsets, uint64_t n_blocks,
                       uint8_t *raw, const uint64_t *raw_offsets, uint64_t *raw_lens,
                       uint64_t *consumed, int32_t *status);

/* ---- pre-trained models.  The reference's compress()/decompress() take a Box<Model> (src/lib.rs:102,113)
 * that the caller may have trained already through Model::get_frequency (src/model/mod.rs:23-25); the
 * observable state of either model kind is its per-symbol frequency vector.  model_freq[symbol_count]
 * (symbol_count = 2^symbol_bits + 1, EOF last; every entry >= 1, sum <= freq_max, else
 * REDUX_INVALID_INPUT) is that vector; NULL = a fresh model.  Every block of the batch starts from it.
 * Byte-symbol models with code_bits <= 32 run on the same tuned kernels as fresh models (same speed).
 * Otherwise identical to redux_encode_batch / redux_decode_batch. */
int redux_encode_batch_ex(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                          const uint32_t *model_freq,
                          const uint8_t *in, const uint64_t *in_offsets, uint64_t n_blocks,
                          uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status);
int redux_decode_batch_ex(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                          const uint32_t *model_freq,
                          const uint8_t *comp, const uint64_t *comp_offsets, uint64_t n_blocks,
                          uint8_t *raw, const uint64_t *raw_offsets, uint64_t *raw_lens,
                          uint64_t *consumed, int32_t *status);

/* ---- a start model per block.  A batch of compress() calls that each get their own Box<Model>, trained or fresh,
 * is one call: model_freqs holds n_models frequency vectors of symbol_count entries back to back (host memory; each row
 * validated like model_freq above, an invalid row gives REDUX_INVALID_INPUT and redux_ctx_last_error names it; a fresh
 * model is a row of ones), and block i starts from row block_model[i].  block_model == NULL is allowed only when
 * n_models == 1 (every block uses row 0); n_models == 0 is REDUX_INVALID_INPUT.  A block whose row index is >= n_models
 * gets status REDUX_INVALID_INPUT and an empty stream / empty output; the other blocks are unaffected.  The start trees
 * take n_models x (symbol_count + 1) x 4 bytes of device memory; a table larger than REDUX_MAX_MODEL_TABLE_BYTES
 * returns REDUX_UNSUPPORTED.  One model kind and one set of parameters per call.  Blocks of one launch that start from
 * different totals freeze at different positions, which can cost time (DESIGN.md 3.8).  The _ex calls are the
 * n_models == 1 case.  Otherwise identical to redux_encode_batch / redux_decode_batch. */
#define REDUX_MAX_MODEL_TABLE_BYTES ((uint64_t)256 << 20)
int redux_encode_batch_models(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                              const uint32_t *model_freqs, uint32_t n_models, const uint32_t *block_model,
                              const uint8_t *in, const uint64_t *in_offsets, uint64_t n_blocks,
                              uint8_t *out, uint64_t out_capacity, uint64_t *out_offsets, int32_t *status);
int redux_decode_batch_models(redux_ctx_t *ctx, int model_kind, const redux_params_t *params,
                              const uint32_t *model_freqs, uint32_t n_models, const uint32_t *block_model,
                              const uint8_t *comp, const uint64_t *comp_offsets, uint64_t n_blocks,
                              uint8_t *raw, const uint64_t *raw_offsets, uint64_t *raw_lens,
                              uint64_t *consumed, int32_t *status);

/* ---- training start models on the device.  Sample i (in[in_offsets[i] .. in_offsets[i+1])) trains a copy of start
 * row sample_model[i] exactly as the reference's Model::get_frequency(sym) (src/model/mod.rs:23-25) would for every
 * symbol its BitReader yields from the sample (symbol_bits at a time, MSB-first, a trailing partial symbol dropped:
 * src/bitio/mod.rs:94-108): the start row plus the histogram of the first min(n_sym, freq_max - total(row)) symbols,
 * n_sym = floor(8 * len / symbol_bits).  The EOF entry never changes.  Both model kinds train to the same vector, so
 * there is no model_kind argument.  out_freqs receives n_samples rows of symbol_count entries.
 * model_freqs / n_models / sample_model follow redux_encode_batch_models (host memory in both forms; each row checked
 * the same way, and an invalid row or an index >= n_models gives REDUX_INVALID_INPUT before anything launches, named
 * by redux_ctx_last_error); model_freqs == NULL with n_models == 0 starts every sample from a fresh model.
 * symbol_bits > 16 gives REDUX_UNSUPPORTED; n_samples == 0 does nothing.  The host form runs on the context's first
 * device and returns when out_freqs is written.  Without a device both return REDUX_CUDA_ERROR. */
int redux_train_models(redux_ctx_t *ctx, const redux_params_t *params,
                       const uint32_t *model_freqs, uint32_t n_models, const uint32_t *sample_model,
                       const uint8_t *in, const uint64_t *in_offsets, uint64_t n_samples,
                       uint32_t *out_freqs);
/* The same on device-resident buffers (d_in under the alignment contract below, d_in_offsets[n_samples+1],
 * d_out_freqs[n_samples x symbol_count]; model_freqs and sample_model stay HOST pointers, copied during the call),
 * enqueued on `stream` like the other _device calls.  max_sample_len: an upper bound of every sample's length. */
int redux_train_models_device(redux_ctx_t *ctx, int device, void *stream, const redux_params_t *params,
                              const uint32_t *model_freqs, uint32_t n_models, const uint32_t *sample_model,
                              const uint8_t *d_in, const uint64_t *d_in_offsets, uint64_t n_samples,
                              uint64_t max_sample_len, uint32_t *d_out_freqs);

/* ---- batch, device-resident buffers (kernel-only timing; all pointers are device memory on
 * `device`, which must be one of the context's devices; work is enqueued on `stream` (a
 * cudaStream_t; NULL = the CUDA default stream) and is asynchronous to the host).
 * A device has ONE workspace: a call enqueued on another stream of the same device first waits (on the device,
 * cudaStreamWaitEvent) for the previous call's kernels, so calls never overlap on one device whatever streams
 * they use.  Growing a workspace for a larger batch synchronises the device once.
 * max_block_len: an upper bound of every block's raw length (sizes the per-block output slots).
 * Alignment contract: the kernels read d_in / d_comp with aligned vector loads (at most 16 bytes), so the
 * bytes from the enclosing 16-byte boundaries of the first and last byte of each stream must be readable
 * (true for any cudaMalloc / torch allocation: granularity >= 256 B); values outside a stream are ignored.
 * total_in_bytes = in_offsets[n_blocks] as known by the host. */
int redux_encode_batch_device(redux_ctx_t *ctx, int device, void *stream, int model_kind,
                              const redux_params_t *params,
                              const uint8_t *d_in, const uint64_t *d_in_offsets, uint64_t n_blocks,
                              uint64_t max_block_len,
                              uint8_t *d_out, uint64_t out_capacity, uint64_t *d_out_offsets,
                              int32_t *d_status);
int redux_decode_batch_device(redux_ctx_t *ctx, int device, void *stream, int model_kind,
                              const redux_params_t *params,
                              const uint8_t *d_comp, const uint64_t *d_comp_offsets, uint64_t n_blocks,
                              uint64_t max_block_len,
                              uint8_t *d_raw, const uint64_t *d_raw_offsets, uint64_t *d_raw_lens,
                              uint64_t *d_consumed, int32_t *d_status);
/* The same with a pre-trained start model (see redux_encode_batch_ex; model_freq is a HOST pointer, copied during
 * the call). */
int redux_encode_batch_device_ex(redux_ctx_t *ctx, int device, void *stream, int model_kind,
                                 const redux_params_t *params, const uint32_t *model_freq,
                                 const uint8_t *d_in, const uint64_t *d_in_offsets, uint64_t n_blocks,
                                 uint64_t max_block_len,
                                 uint8_t *d_out, uint64_t out_capacity, uint64_t *d_out_offsets,
                                 int32_t *d_status);
int redux_decode_batch_device_ex(redux_ctx_t *ctx, int device, void *stream, int model_kind,
                                 const redux_params_t *params, const uint32_t *model_freq,
                                 const uint8_t *d_comp, const uint64_t *d_comp_offsets, uint64_t n_blocks,
                                 uint64_t max_block_len,
                                 uint8_t *d_raw, const uint64_t *d_raw_offsets, uint64_t *d_raw_lens,
                                 uint64_t *d_consumed, int32_t *d_status);
/* The same with a start model per block (see redux_encode_batch_models): model_freqs is a HOST pointer, copied during
 * the call; d_block_model is a DEVICE pointer [n_blocks] (NULL only when n_models == 1), read by the kernels. */
int redux_encode_batch_device_models(redux_ctx_t *ctx, int device, void *stream, int model_kind,
                                     const redux_params_t *params, const uint32_t *model_freqs, uint32_t n_models,
                                     const uint32_t *d_block_model,
                                     const uint8_t *d_in, const uint64_t *d_in_offsets, uint64_t n_blocks,
                                     uint64_t max_block_len,
                                     uint8_t *d_out, uint64_t out_capacity, uint64_t *d_out_offsets,
                                     int32_t *d_status);
int redux_decode_batch_device_models(redux_ctx_t *ctx, int device, void *stream, int model_kind,
                                     const redux_params_t *params, const uint32_t *model_freqs, uint32_t n_models,
                                     const uint32_t *d_block_model,
                                     const uint8_t *d_comp, const uint64_t *d_comp_offsets, uint64_t n_blocks,
                                     uint64_t max_block_len,
                                     uint8_t *d_raw, const uint64_t *d_raw_offsets, uint64_t *d_raw_lens,
                                     uint64_t *d_consumed, int32_t *d_status);
/* Waits for the work enqueued on `stream` of `device`. */
int redux_ctx_synchronize(redux_ctx_t *ctx, int device, void *stream);

/* ---- synthetic workload (BASELINE.json configs 3-4; DESIGN.md "generator"): fills
 * d_out[i*block_len .. (i+1)*block_len) for block indices first_block+i, i < n_blocks, with the
 * mixed-entropy classes (block index & 3: uniform / text-like / geometric / runs), splitmix64 seeded
 * by seed + block index. Deterministic; redux_generate_blocks_host produces the same bytes on the
 * CPU (used by the tests to prove the two agree). */
int redux_generate_blocks_device(redux_ctx_t *ctx, int device, void *stream, uint8_t *d_out,
                                 uint64_t first_block, uint64_t n_blocks, uint64_t block_len,
                                 uint64_t seed);
void redux_generate_blocks_host(uint8_t *out, uint64_t first_block, uint64_t n_blocks,
                                uint64_t block_len, uint64_t seed);
/* Text class from a corpus (BASELINE.md section 4, config 3): with a corpus of at least block_len bytes, blocks of
 * class 1 are block_len-byte windows of it at a per-block pseudo-random offset instead of the table-driven stand-in.
 * redux_ctx_set_text_corpus uploads it to every device of the context for redux_generate_blocks_device (NULL, 0
 * clears it); redux_generate_blocks_host_ex is the CPU twin. */
int redux_ctx_set_text_corpus(redux_ctx_t *ctx, const uint8_t *corpus, uint64_t corpus_len);
void redux_generate_blocks_host_ex(uint8_t *out, uint64_t first_block, uint64_t n_blocks,
                                   uint64_t block_len, uint64_t seed, const uint8_t *corpus, uint64_t corpus_len);

/* ---- debug / self-test hooks (host arithmetic only; used by the CPU tests)
 * Exact-division magic for divisor d and numerators < 2^nbits (DESIGN.md "count reciprocal"):
 * floor(n/d) == mulhi(n, magic) >> shift. wide=0: 32-bit mulhi, wide=1: 64-bit mulhi, wide=2: the 65-bit magic of the
 * code_bits > 32 class (nbits ignored: exact for every 64-bit numerator; divide = (((n - t) >> 1) + t) >> (shift - 1),
 * t = mulhi64(n, magic)); wide=3: the double reciprocal of the WIDE_D class (magic = the bits of 1.0/d, d < 2^17;
 * exact for n = cum * range < 2^49 with cum <= d). */
int redux_debug_magic(uint64_t d, uint32_t nbits, int wide, uint64_t *magic, uint32_t *shift);
uint64_t redux_debug_magic_divide(uint64_t n, uint64_t magic, uint32_t shift, int wide);
/* floor(x / range) as the code_bits > 32 decoder computes it (double estimate + one remainder check); exact whenever
 * the quotient is below 2^31 (it is a cumulative frequency: < freq_max). */
uint32_t redux_debug_div_by_range(uint64_t x, uint64_t range);
/* Closed-form renormalisation (SURVEY.md A.6) of one (low, high) pair: returns n1 (E1/E2 shifts) in
 * *n1 and k (E3 shifts) in *k and the renormalised pair. */
void redux_debug_renorm(uint64_t low, uint64_t high, uint32_t code_bits,
                        uint32_t *n1, uint32_t *k, uint64_t *new_low, uint64_t *new_high);

/* Resident CTAs per SM of the tuned encoder / decoder with 16-bit tables (must be 2; needs a device). */
int redux_debug_lane_occupancy(int *enc_ctas_per_sm, int *dec_ctas_per_sm);

/* Which coder kernels the context has launched: bit k of *mask is set when the kernel instantiation with ID k ran
 * since the last reset (reset != 0 clears the mask after reading it).  Lets tests check which of the 37 kernels a
 * parameter set, block length, capacity, model and schedule actually selects.  Costs one host-side atomic OR per
 * coder launch. */
int redux_debug_launched_kernels(redux_ctx_t *ctx, uint64_t *mask, int reset);
/* Name of kernel ID id, e.g. "decode_lane_al<u32,WideD,full,c32>"; NULL past the last ID.  Needs no device. */
const char *redux_debug_kernel_name(int id);

/* The host front end's partition rule: device g of n_devices codes blocks [first, first+count). */
void redux_debug_shard(uint64_t n_blocks, uint32_t n_devices, uint32_t g, uint64_t *first, uint64_t *count);

#ifdef __cplusplus
}
#endif
#endif /* REDUX_B200_H */
