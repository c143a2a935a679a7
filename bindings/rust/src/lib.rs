//! UNCOMPILED: written against `include/redux_b200.h`; the build image has no Rust toolchain, so this file has
//! never been through `rustc`.  It mirrors the C ABI one to one and adds the two safe wrappers a maintainer of
//! `peterbudai/redux` would call from `redux::compress` / `redux::decompress` (src/lib.rs:102-120).
//! The tested bindings of this repository are the Python ctypes one (`redux_b200/__init__.py`) and the plain-C
//! consumer of `tests/test_c_abi_from_c.py`.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct redux_params_t { pub symbol_bits: u32, pub freq_bits: u32, pub code_bits: u32 }

#[repr(C)]
pub struct redux_ctx_t { _private: [u8; 0] }

pub const REDUX_OK: c_int = 0;
pub const REDUX_EOF: c_int = 1;            // Error::Eof          (src/lib.rs:59)
pub const REDUX_INVALID_INPUT: c_int = 2;  // Error::InvalidInput (src/lib.rs:61)
pub const REDUX_IO_ERROR: c_int = 3;       // Error::IoError      (src/lib.rs:63)
pub const REDUX_CUDA_ERROR: c_int = 4;
pub const REDUX_UNSUPPORTED: c_int = 5;
pub const REDUX_OUT_CAPACITY: c_int = 6;
pub const REDUX_MODEL_LINEAR: c_int = 0;   // AdaptiveLinearModel::new (src/model/adaptive_linear.rs:21)
pub const REDUX_MODEL_TREE: c_int = 1;     // AdaptiveTreeModel::new   (src/model/adaptive_tree.rs:36)
pub const REDUX_SCHED_AUTO: c_int = 0;
pub const REDUX_SCHED_LANE: c_int = 1;
pub const REDUX_SCHED_WARP: c_int = 2;
pub const REDUX_SCHED_SPLIT: c_int = 3;

extern "C" {
    pub fn redux_parameters_new(symbol_bits: u32, freq_bits: u32, code_bits: u32, out: *mut c_void) -> c_int;
    pub fn redux_params_supported(p: *const redux_params_t) -> c_int;
    pub fn redux_error_string(code: c_int) -> *const c_char;
    pub fn redux_compress_bound(in_len: u64, code_bits: u32) -> u64;
    pub fn redux_compress_bound_ex(in_len: u64, symbol_bits: u32, code_bits: u32) -> u64;
    pub fn redux_process_init() -> c_int;
    pub fn redux_host_alloc(bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn redux_host_free(p: *mut c_void) -> c_int;
    pub fn redux_host_register(p: *mut c_void, bytes: usize) -> c_int;
    pub fn redux_host_unregister(p: *mut c_void) -> c_int;
    pub fn redux_ctx_create(devices: *const c_int, n_devices: c_int, ctx: *mut *mut redux_ctx_t) -> c_int;
    pub fn redux_ctx_destroy(ctx: *mut redux_ctx_t);
    pub fn redux_ctx_device_count(ctx: *const redux_ctx_t) -> c_int;
    pub fn redux_ctx_last_error(ctx: *const redux_ctx_t) -> *const c_char;
    pub fn redux_ctx_set_schedule(ctx: *mut redux_ctx_t, sched: c_int) -> c_int;
    /// pageable caller buffers: staged through the library's pinned ring and copy threads (default) or left to the driver
    pub fn redux_ctx_set_staging(ctx: *mut redux_ctx_t, enable: c_int, min_bytes: usize, piece_bytes: usize, slots: c_int, threads: c_int) -> c_int;
    pub fn redux_compress(ctx: *mut redux_ctx_t, model_kind: c_int, p: *const redux_params_t,
                          input: *const u8, in_len: u64, out: *mut u8, out_cap: u64,
                          in_count: *mut u64, out_count: *mut u64) -> c_int;
    pub fn redux_decompress(ctx: *mut redux_ctx_t, model_kind: c_int, p: *const redux_params_t,
                            input: *const u8, in_len: u64, out: *mut u8, out_cap: u64,
                            in_count: *mut u64, out_count: *mut u64) -> c_int;
    pub fn redux_encode_batch(ctx: *mut redux_ctx_t, model_kind: c_int, p: *const redux_params_t,
                              input: *const u8, in_offsets: *const u64, n_blocks: u64,
                              out: *mut u8, out_cap: u64, out_offsets: *mut u64, status: *mut i32) -> c_int;
    pub fn redux_decode_batch(ctx: *mut redux_ctx_t, model_kind: c_int, p: *const redux_params_t,
                              comp: *const u8, comp_offsets: *const u64, n_blocks: u64,
                              raw: *mut u8, raw_offsets: *const u64, raw_lens: *mut u64,
                              consumed: *mut u64, status: *mut i32) -> c_int;
    pub fn redux_encode_batch_ex(ctx: *mut redux_ctx_t, model_kind: c_int, p: *const redux_params_t,
                                 model_freq: *const u32, input: *const u8, in_offsets: *const u64, n_blocks: u64,
                                 out: *mut u8, out_cap: u64, out_offsets: *mut u64, status: *mut i32) -> c_int;
    pub fn redux_decode_batch_ex(ctx: *mut redux_ctx_t, model_kind: c_int, p: *const redux_params_t,
                                 model_freq: *const u32, comp: *const u8, comp_offsets: *const u64, n_blocks: u64,
                                 raw: *mut u8, raw_offsets: *const u64, raw_lens: *mut u64,
                                 consumed: *mut u64, status: *mut i32) -> c_int;
    pub fn redux_encode_batch_models(ctx: *mut redux_ctx_t, model_kind: c_int, p: *const redux_params_t,
                                     model_freqs: *const u32, n_models: u32, block_model: *const u32,
                                     input: *const u8, in_offsets: *const u64, n_blocks: u64,
                                     out: *mut u8, out_cap: u64, out_offsets: *mut u64, status: *mut i32) -> c_int;
    pub fn redux_decode_batch_models(ctx: *mut redux_ctx_t, model_kind: c_int, p: *const redux_params_t,
                                     model_freqs: *const u32, n_models: u32, block_model: *const u32,
                                     comp: *const u8, comp_offsets: *const u64, n_blocks: u64,
                                     raw: *mut u8, raw_offsets: *const u64, raw_lens: *mut u64,
                                     consumed: *mut u64, status: *mut i32) -> c_int;
    pub fn redux_encode_batch_device(ctx: *mut redux_ctx_t, device: c_int, stream: *mut c_void, model_kind: c_int,
                                     p: *const redux_params_t, d_in: *const u8, d_in_offsets: *const u64,
                                     n_blocks: u64, max_block_len: u64, d_out: *mut u8, out_cap: u64,
                                     d_out_offsets: *mut u64, d_status: *mut i32) -> c_int;
    pub fn redux_decode_batch_device(ctx: *mut redux_ctx_t, device: c_int, stream: *mut c_void, model_kind: c_int,
                                     p: *const redux_params_t, d_comp: *const u8, d_comp_offsets: *const u64,
                                     n_blocks: u64, max_block_len: u64, d_raw: *mut u8, d_raw_offsets: *const u64,
                                     d_raw_lens: *mut u64, d_consumed: *mut u64, d_status: *mut i32) -> c_int;
    pub fn redux_encode_batch_device_models(ctx: *mut redux_ctx_t, device: c_int, stream: *mut c_void, model_kind: c_int,
                                            p: *const redux_params_t, model_freqs: *const u32, n_models: u32,
                                            d_block_model: *const u32, d_in: *const u8, d_in_offsets: *const u64,
                                            n_blocks: u64, max_block_len: u64, d_out: *mut u8, out_cap: u64,
                                            d_out_offsets: *mut u64, d_status: *mut i32) -> c_int;
    pub fn redux_decode_batch_device_models(ctx: *mut redux_ctx_t, device: c_int, stream: *mut c_void, model_kind: c_int,
                                            p: *const redux_params_t, model_freqs: *const u32, n_models: u32,
                                            d_block_model: *const u32, d_comp: *const u8, d_comp_offsets: *const u64,
                                            n_blocks: u64, max_block_len: u64, d_raw: *mut u8, d_raw_offsets: *const u64,
                                            d_raw_lens: *mut u64, d_consumed: *mut u64, d_status: *mut i32) -> c_int;
    // one trained frequency row per sample (n_samples x symbol_count); model_freqs / sample_model are host memory
    pub fn redux_train_models(ctx: *mut redux_ctx_t, p: *const redux_params_t, model_freqs: *const u32, n_models: u32,
                              sample_model: *const u32, input: *const u8, in_offsets: *const u64, n_samples: u64,
                              out_freqs: *mut u32) -> c_int;
    pub fn redux_train_models_device(ctx: *mut redux_ctx_t, device: c_int, stream: *mut c_void, p: *const redux_params_t,
                                     model_freqs: *const u32, n_models: u32, sample_model: *const u32,
                                     d_in: *const u8, d_in_offsets: *const u64, n_samples: u64, max_sample_len: u64,
                                     d_out_freqs: *mut u32) -> c_int;
    pub fn redux_ctx_synchronize(ctx: *mut redux_ctx_t, device: c_int, stream: *mut c_void) -> c_int;
}

/// Owns a `redux_ctx_t` (streams and workspaces of the selected GPUs). Not `Sync`: one caller at a time.
pub struct Context { raw: *mut redux_ctx_t }

impl Context {
    /// `devices` empty = the current device.
    pub fn new(devices: &[i32]) -> Result<Context, c_int> {
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { redux_ctx_create(if devices.is_empty() { std::ptr::null() } else { devices.as_ptr() },
                                            devices.len() as c_int, &mut raw) };
        if rc == REDUX_OK { Ok(Context { raw }) } else { Err(rc) }
    }

    /// Block `i` of the result is byte for byte what `redux::compress` writes for `blocks[i]` alone.
    /// `model_freq`: `None` = fresh model, else the trained model's per-symbol frequencies.
    pub fn compress_blocks(&mut self, blocks: &[&[u8]], model_kind: c_int, p: redux_params_t,
                           model_freq: Option<&[u32]>) -> Result<Vec<Vec<u8>>, c_int> {
        let mut input = Vec::new();
        let mut off = vec![0u64];
        for b in blocks { input.extend_from_slice(b); off.push(input.len() as u64); }
        let cap: u64 = blocks.iter().map(|b| unsafe { redux_compress_bound_ex(b.len() as u64, p.symbol_bits, p.code_bits) }).sum();
        let mut out = vec![0u8; cap as usize];
        let mut out_off = vec![0u64; blocks.len() + 1];
        let mut status = vec![0i32; blocks.len().max(1)];
        let fq = model_freq.map_or(std::ptr::null(), |f| f.as_ptr());
        let rc = unsafe { redux_encode_batch_ex(self.raw, model_kind, &p, fq, input.as_ptr(), off.as_ptr(), blocks.len() as u64,
                                                out.as_mut_ptr(), cap, out_off.as_mut_ptr(), status.as_mut_ptr()) };
        if rc != REDUX_OK { return Err(rc); }
        Ok((0..blocks.len()).map(|i| out[out_off[i] as usize..out_off[i + 1] as usize].to_vec()).collect())
    }

    /// Mirror of `compress_blocks`; `max_len[i]` bounds the decoded size of stream `i`.
    pub fn decompress_blocks(&mut self, streams: &[&[u8]], max_len: &[usize], model_kind: c_int, p: redux_params_t,
                             model_freq: Option<&[u32]>) -> Result<Vec<Vec<u8>>, c_int> {
        let mut comp = Vec::new();
        let mut coff = vec![0u64];
        for s in streams { comp.extend_from_slice(s); coff.push(comp.len() as u64); }
        let mut roff = vec![0u64];
        for m in max_len { let last = *roff.last().unwrap(); roff.push(last + *m as u64); }
        let mut raw = vec![0u8; *roff.last().unwrap() as usize];
        let (mut lens, mut cons) = (vec![0u64; streams.len().max(1)], vec![0u64; streams.len().max(1)]);
        let mut status = vec![0i32; streams.len().max(1)];
        let fq = model_freq.map_or(std::ptr::null(), |f| f.as_ptr());
        let rc = unsafe { redux_decode_batch_ex(self.raw, model_kind, &p, fq, comp.as_ptr(), coff.as_ptr(), streams.len() as u64,
                                                raw.as_mut_ptr(), roff.as_ptr(), lens.as_mut_ptr(), cons.as_mut_ptr(),
                                                status.as_mut_ptr()) };
        if rc != REDUX_OK { return Err(rc); }
        Ok((0..streams.len()).map(|i| raw[roff[i] as usize..(roff[i] + lens[i]) as usize].to_vec()).collect())
    }
}

impl Drop for Context {
    fn drop(&mut self) { unsafe { redux_ctx_destroy(self.raw) } }
}
