"""redux_b200 -- host-side mirror of the reference's public interface for ONE path:
``redux::compress`` / ``redux::decompress`` (src/lib.rs:102-120) over ``AdaptiveLinearModel`` /
``AdaptiveTreeModel`` built from ``Parameters::new(symbol_bits, freq_bits, code_bits)``
(src/model/mod.rs:63-81), plus the new block-batching front end.

Everything computes inside ``libredux_b200.so`` (hand-written sm_100a CUDA behind the C ABI of
``include/redux_b200.h``).  There is no CPU fallback: importing works anywhere, but any call that
codes data raises ``CudaError`` without a B200, and a missing shared library raises ImportError.

The reference's toolchain (Rust) is absent from the build image, so this mirror is Python over
ctypes; INTEGRATION.md holds the Rust ``extern "C"`` binding a maintainer would add instead.
"""
import ctypes as C
import os
import subprocess

import numpy as np

__all__ = [
    "Parameters", "AdaptiveLinearModel", "AdaptiveTreeModel", "Model", "compress", "decompress",
    "Context", "ReduxError", "Eof", "InvalidInput", "IoError", "CudaError", "Unsupported", "OutCapacity",
    "compress_bound", "kernel_names", "build", "lib", "process_init", "HostBuffer", "host_register", "host_unregister",
]

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libredux_b200.so")

OK, EOF, INVALID_INPUT, IO_ERROR, CUDA_ERROR, UNSUPPORTED, OUT_CAPACITY = range(7)
MODEL_LINEAR, MODEL_TREE = 0, 1
SCHED_AUTO, SCHED_LANE, SCHED_WARP, SCHED_SPLIT = 0, 1, 2, 3


# --------------------------------------------------------------------------- errors (src/lib.rs:57-84)
class ReduxError(Exception):
    code = -1


class Eof(ReduxError):
    """Error::Eof -- the input stream has ended (unexpectedly)."""
    code = EOF


class InvalidInput(ReduxError):
    """Error::InvalidInput."""
    code = INVALID_INPUT


class IoError(ReduxError):
    """Error::IoError."""
    code = IO_ERROR


class CudaError(ReduxError):
    code = CUDA_ERROR


class Unsupported(ReduxError):
    code = UNSUPPORTED


class OutCapacity(ReduxError):
    code = OUT_CAPACITY


_ERRORS = {e.code: e for e in (Eof, InvalidInput, IoError, CudaError, Unsupported, OutCapacity)}


class _ParamsC(C.Structure):
    _fields_ = [("symbol_bits", C.c_uint32), ("freq_bits", C.c_uint32), ("code_bits", C.c_uint32)]


class _ParametersC(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "symbol_bits", "symbol_eof", "symbol_count", "freq_bits", "freq_max", "code_bits",
        "code_min", "code_one_fourth", "code_half", "code_three_fourths", "code_max")]


def build(verbose=False):
    """Compile redux_b200/libredux_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc")], capture_output=not verbose, text=True)
    if r.returncode != 0:
        raise RuntimeError("building libredux_b200.so failed:\n%s\n%s" % (r.stdout, r.stderr))
    return _SO


_lib = None


def lib():
    """The loaded C-ABI library. Raises ImportError when the CUDA extension was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise ImportError("redux_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)" % _SO)
    L = C.CDLL(_SO)
    u32, u64, vp, i32 = C.c_uint32, C.c_uint64, C.c_void_p, C.c_int
    pp = C.POINTER(_ParamsC)
    L.redux_parameters_new.argtypes = [u32, u32, u32, C.POINTER(_ParametersC)]
    L.redux_params_supported.argtypes = [pp]
    L.redux_error_string.argtypes = [i32]
    L.redux_error_string.restype = C.c_char_p
    L.redux_compress_bound.argtypes = [u64, u32]
    L.redux_compress_bound.restype = u64
    L.redux_compress_bound_ex.argtypes = [u64, u32, u32]
    L.redux_compress_bound_ex.restype = u64
    L.redux_ctx_create.argtypes = [C.POINTER(C.c_int), i32, C.POINTER(vp)]
    L.redux_ctx_destroy.argtypes = [vp]
    L.redux_ctx_destroy.restype = None
    L.redux_ctx_device_count.argtypes = [vp]
    L.redux_ctx_last_error.argtypes = [vp]
    L.redux_ctx_last_error.restype = C.c_char_p
    L.redux_ctx_set_schedule.argtypes = [vp, i32]
    L.redux_ctx_set_staging.argtypes = [vp, i32, C.c_size_t, C.c_size_t, i32, i32]
    L.redux_ctx_kernel_launches.argtypes = [vp]
    L.redux_ctx_kernel_launches.restype = u64
    L.redux_ctx_synchronize.argtypes = [vp, i32, vp]
    L.redux_ctx_timing_enable.argtypes = [vp, i32]
    L.redux_ctx_timing_collect.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(u64)]
    for name in ("redux_compress", "redux_decompress"):
        getattr(L, name).argtypes = [vp, i32, pp, vp, u64, vp, u64, C.POINTER(u64), C.POINTER(u64)]
    L.redux_encode_batch.argtypes = [vp, i32, pp, vp, vp, u64, vp, u64, vp, vp]
    L.redux_decode_batch.argtypes = [vp, i32, pp, vp, vp, u64, vp, vp, vp, vp, vp]
    L.redux_encode_batch_ex.argtypes = [vp, i32, pp, vp, vp, vp, u64, vp, u64, vp, vp]
    L.redux_decode_batch_ex.argtypes = [vp, i32, pp, vp, vp, vp, u64, vp, vp, vp, vp, vp]
    L.redux_encode_batch_device.argtypes = [vp, i32, vp, i32, pp, vp, vp, u64, u64, vp, u64, vp, vp]
    L.redux_decode_batch_device.argtypes = [vp, i32, vp, i32, pp, vp, vp, u64, u64, vp, vp, vp, vp, vp]
    L.redux_generate_blocks_device.argtypes = [vp, i32, vp, vp, u64, u64, u64, u64]
    L.redux_generate_blocks_host.argtypes = [vp, u64, u64, u64, u64]
    L.redux_generate_blocks_host.restype = None
    L.redux_generate_blocks_host_ex.argtypes = [vp, u64, u64, u64, u64, vp, u64]
    L.redux_generate_blocks_host_ex.restype = None
    L.redux_ctx_set_text_corpus.argtypes = [vp, vp, u64]
    L.redux_debug_magic.argtypes = [u64, u32, i32, C.POINTER(u64), C.POINTER(u32)]
    L.redux_debug_magic_divide.argtypes = [u64, u64, u32, i32]
    L.redux_debug_magic_divide.restype = u64
    L.redux_debug_div_by_range.argtypes = [u64, u64]
    L.redux_debug_div_by_range.restype = u32
    L.redux_debug_renorm.argtypes = [u64, u64, u32, C.POINTER(u32), C.POINTER(u32), C.POINTER(u64), C.POINTER(u64)]
    L.redux_debug_renorm.restype = None
    L.redux_debug_shard.argtypes = [u64, u32, u32, C.POINTER(u64), C.POINTER(u64)]
    L.redux_debug_shard.restype = None
    L.redux_debug_lane_occupancy.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.redux_debug_launched_kernels.argtypes = [vp, C.POINTER(u64), i32]
    L.redux_debug_kernel_name.argtypes = [i32]
    L.redux_debug_kernel_name.restype = C.c_char_p
    L.redux_process_init.argtypes = []
    L.redux_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.redux_host_free.argtypes = [vp]
    L.redux_host_register.argtypes = [vp, C.c_size_t]
    L.redux_host_unregister.argtypes = [vp]
    L.redux_encode_batch_device_ex.argtypes = [vp, i32, vp, i32, pp, vp, vp, vp, u64, u64, vp, u64, vp, vp]
    L.redux_decode_batch_device_ex.argtypes = [vp, i32, vp, i32, pp, vp, vp, vp, u64, u64, vp, vp, vp, vp, vp]
    L.redux_encode_batch_models.argtypes = [vp, i32, pp, vp, u32, vp, vp, vp, u64, vp, u64, vp, vp]
    L.redux_decode_batch_models.argtypes = [vp, i32, pp, vp, u32, vp, vp, vp, u64, vp, vp, vp, vp, vp]
    L.redux_encode_batch_device_models.argtypes = [vp, i32, vp, i32, pp, vp, u32, vp, vp, vp, u64, u64, vp, u64, vp, vp]
    L.redux_decode_batch_device_models.argtypes = [vp, i32, vp, i32, pp, vp, u32, vp, vp, vp, u64, u64, vp, vp, vp, vp, vp]
    L.redux_train_models.argtypes = [vp, pp, vp, u32, vp, vp, vp, u64, vp]
    L.redux_train_models_device.argtypes = [vp, i32, vp, pp, vp, u32, vp, vp, vp, u64, u64, vp]
    _lib = L
    return L


def _raise(code, ctx=None):
    if code == OK:
        return
    msg = lib().redux_error_string(code).decode()
    if ctx is not None and ctx._h:
        detail = lib().redux_ctx_last_error(ctx._h).decode()
        if detail:
            msg = "%s (%s)" % (msg, detail)
    raise _ERRORS.get(code, ReduxError)(msg)


def process_init():
    """Optional, before CUDA is initialised in this process: ask for 32 hardware queues unless the application
    set CUDA_DEVICE_MAX_CONNECTIONS itself (include/redux_b200.h).  Returns the value in force."""
    return int(lib().redux_process_init())


class HostBuffer:
    """Page-locked host memory from redux_host_alloc as a numpy uint8 array (`.array`); freed by close()."""

    def __init__(self, nbytes):
        self._p = C.c_void_p()
        _raise(lib().redux_host_alloc(nbytes, C.byref(self._p)))
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self._p.value)) if nbytes else np.zeros(0, np.uint8)

    def close(self):
        if self._p:
            self.array = None
            lib().redux_host_free(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def host_register(array):
    """Page-lock an existing numpy buffer in place (redux_host_register); pair with host_unregister."""
    _raise(lib().redux_host_register(array.ctypes.data, array.nbytes))


def host_unregister(array):
    _raise(lib().redux_host_unregister(array.ctypes.data))


def kernel_names():
    """Names of every coder kernel instantiation the library can launch, in ID order (needs no device)."""
    names = []
    while True:
        n = lib().redux_debug_kernel_name(len(names))
        if n is None:
            return names
        names.append(n.decode())


def compress_bound(in_len, code_bits, symbol_bits=8):
    return int(lib().redux_compress_bound_ex(in_len, symbol_bits, code_bits))


# --------------------------------------------------------------------------- Parameters / models
class Parameters:
    """``Parameters::new(symbol, frequency, code)`` (src/model/mod.rs:63-81): same fields, same
    rejection rule (raises ``InvalidInput``)."""

    def __init__(self, symbol_bits, freq_bits, code_bits):
        out = _ParametersC()
        rc = lib().redux_parameters_new(symbol_bits, freq_bits, code_bits, C.byref(out))
        if rc != OK:
            raise InvalidInput(lib().redux_error_string(rc).decode())
        for name, _ in _ParametersC._fields_:
            setattr(self, name, int(getattr(out, name)))

    @classmethod
    def new(cls, symbol, frequency, code):
        return cls(symbol, frequency, code)

    def _c(self):
        return _ParamsC(self.symbol_bits, self.freq_bits, self.code_bits)

    def __repr__(self):
        return "Parameters(%d, %d, %d)" % (self.symbol_bits, self.freq_bits, self.code_bits)


class Model:
    """An adaptive model handed to compress()/decompress(); consumed by the call like the reference's
    ``Box<Model>`` (src/lib.rs:102).  Fresh unless the caller trained it first: like the reference's trait
    object it can be trained through ``get_frequency(symbol)``, which looks the symbol up AND counts it
    (src/model/mod.rs:23-25); the coder then starts every stream from that state.  The state is plain
    bookkeeping (one counter per symbol) kept on the host; all coding happens on the device."""
    kind = None

    def __init__(self, parameters):
        if not isinstance(parameters, Parameters):
            parameters = Parameters(*parameters)
        self.params = parameters
        self.freq = None            # None = fresh (every symbol once); else uint32[symbol_count]

    def parameters(self):
        return self.params

    @classmethod
    def new(cls, parameters):
        return cls(parameters)

    def _state(self):
        if self.freq is None:
            self.freq = np.ones(self.params.symbol_count, dtype=np.uint32)
        return self.freq

    def total_frequency(self):
        """Model::total_frequency (adaptive_tree.rs:100-103 / adaptive_linear.rs:47-49)."""
        return int(self.params.symbol_count if self.freq is None else self.freq.sum())

    def get_frequency(self, symbol):
        """Model::get_frequency (adaptive_tree.rs:105-113 / adaptive_linear.rs:51-59): the symbol's
        cumulative range BEFORE the update, then the update -- frozen once the total reaches freq_max."""
        if symbol > self.params.symbol_eof:
            raise InvalidInput("Invalid data found while processing input")
        fr = self._state()
        lo = int(fr[:symbol].sum())
        hi = lo + int(fr[symbol])
        if int(fr.sum()) < self.params.freq_max:
            fr[symbol] += 1
        return lo, hi

    def train(self, symbols):
        """get_frequency() for every symbol of an iterable (vectorised; same freeze rule)."""
        fr = self._state()
        room = self.params.freq_max - int(fr.sum())
        sy = np.asarray(list(symbols) if not isinstance(symbols, np.ndarray) else symbols, dtype=np.int64)
        if sy.size and (sy.min() < 0 or sy.max() > self.params.symbol_eof):
            raise InvalidInput("Invalid data found while processing input")
        sy = sy[:max(room, 0)]
        np.add.at(fr, sy, 1)
        return self

    def _freq_ptr(self):
        if self.freq is None:
            return None
        self.freq = np.ascontiguousarray(self.freq, dtype=np.uint32)
        return self.freq.ctypes.data


class AdaptiveLinearModel(Model):
    """AdaptiveLinearModel::new (src/model/adaptive_linear.rs:21-30)."""
    kind = MODEL_LINEAR


class AdaptiveTreeModel(Model):
    """AdaptiveTreeModel::new (src/model/adaptive_tree.rs:36-48)."""
    kind = MODEL_TREE


def _model_table(models):
    """(kind, C parameters, uint32[n_models, symbol_count] frequency table) of a sequence of models: one model kind and
    one Parameters for all of them (InvalidInput otherwise); a fresh model is a row of ones."""
    models = list(models)
    if not models:
        raise InvalidInput("no models")
    kind, p = models[0].kind, models[0].params
    key = (p.symbol_bits, p.freq_bits, p.code_bits)
    for m in models:
        if m.kind != kind:
            raise InvalidInput("models of different kinds in one call")
        if (m.params.symbol_bits, m.params.freq_bits, m.params.code_bits) != key:
            raise InvalidInput("models with different Parameters in one call")
    table = np.ones((len(models), p.symbol_count), dtype=np.uint32)
    for i, m in enumerate(models):
        if m.freq is not None:
            table[i] = m.freq
    return kind, p._c(), table


def _block_model(block_model):
    return None if block_model is None else np.ascontiguousarray(block_model, dtype=np.uint32)


def _train_start(start, n):
    """(class, Parameters, C parameters, start table or None, n_models, sample_model or None) of the `start` argument of
    train_models: one model for every sample (None table when it is fresh), or a list of n models, sample i starting
    from start[i]."""
    if isinstance(start, Model):
        p = start.params
        if start.freq is None:
            return type(start), p, p._c(), None, 0, None
        return type(start), p, p._c(), np.ascontiguousarray(start.freq, dtype=np.uint32)[None, :], 1, None
    start = list(start)
    if len(start) != n:
        raise InvalidInput("train_models: %d start models for %d samples" % (len(start), n))
    if n == 0:
        raise InvalidInput("train_models: an empty list of start models names no Parameters")
    _, pc, table = _model_table(start)
    return type(start[0]), start[0].params, pc, table, n, np.arange(n, dtype=np.uint32)


def _trained_models(cls, params, rows):
    out = []
    for r in rows:
        m = cls(params)
        m.freq = r.copy()
        out.append(m)
    return out


def _ptr(x):
    """Host numpy array or device tensor -> raw address."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    return int(x)


# --------------------------------------------------------------------------- context + batch API
class Context:
    """Owns the per-device streams and workspaces (``redux_ctx_t``)."""

    def __init__(self, devices=None):
        self._h = C.c_void_p()
        if devices is None:
            rc = lib().redux_ctx_create(None, 0, C.byref(self._h))
        else:
            arr = (C.c_int * len(devices))(*devices)
            rc = lib().redux_ctx_create(arr, len(devices), C.byref(self._h))
        if rc != OK:
            self._h = C.c_void_p()
            _raise(rc)

    def close(self):
        if self._h:
            lib().redux_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def device_count(self):
        return lib().redux_ctx_device_count(self._h)

    @property
    def kernel_launches(self):
        return int(lib().redux_ctx_kernel_launches(self._h))

    def launched_kernels(self, reset=True):
        """Names of the coder kernels launched since the last reset (see kernel_names())."""
        mask = C.c_uint64()
        _raise(lib().redux_debug_launched_kernels(self._h, C.byref(mask), 1 if reset else 0), self)
        return {n for i, n in enumerate(kernel_names()) if mask.value >> i & 1}

    def set_schedule(self, sched):
        _raise(lib().redux_ctx_set_schedule(self._h, sched), self)

    def set_staging(self, enable=True, min_bytes=0, piece_bytes=0, slots=0, threads=0):
        """How pageable (not page-locked) caller buffers are moved: through the library's pinned ring and copy
        threads (default), or handed to the driver as they are.  Zero keeps a value."""
        _raise(lib().redux_ctx_set_staging(self._h, 1 if enable else 0, min_bytes, piece_bytes, slots, threads), self)

    def timing_enable(self, on=True):
        _raise(lib().redux_ctx_timing_enable(self._h, 1 if on else 0), self)

    def timing_collect(self):
        """{kernel kind: (total ms, launches)} for the launches recorded since the last collect."""
        ms = (C.c_double * 5)()
        cnt = (C.c_uint64 * 5)()
        _raise(lib().redux_ctx_timing_collect(self._h, ms, cnt), self)
        names = ("encode", "scan", "compact", "decode", "generate")
        return {n: (float(ms[i]), int(cnt[i])) for i, n in enumerate(names)}

    def synchronize(self, device=0, stream=None):
        _raise(lib().redux_ctx_synchronize(self._h, device, stream), self)

    # ---- single stream (host memory)
    def compress(self, data, model, out_capacity=None):
        """bytes -> (compressed bytes, (in_count, out_count)); redux::compress (src/lib.rs:102-109)."""
        a = np.frombuffer(bytes(data), dtype=np.uint8)
        cap = out_capacity if out_capacity is not None else compress_bound(a.size, model.params.code_bits,
                                                                           model.params.symbol_bits)
        out = np.empty(max(cap, 1), dtype=np.uint8)
        pc = model.params._c()
        if model.freq is not None:
            off = np.array([0, a.size], dtype=np.uint64)
            out_off = np.zeros(2, dtype=np.uint64)
            st = np.zeros(1, dtype=np.int32)
            rc = lib().redux_encode_batch_ex(self._h, model.kind, C.byref(pc), model._freq_ptr(),
                                             a.ctypes.data if a.size else None, _ptr(off), 1, out.ctypes.data, cap,
                                             _ptr(out_off), _ptr(st))
            _raise(rc, self)
            return out[:int(out_off[1])].tobytes(), (a.size, int(out_off[1]))
        ic, oc = C.c_uint64(), C.c_uint64()
        rc = lib().redux_compress(self._h, model.kind, C.byref(pc), a.ctypes.data if a.size else None, a.size,
                                  out.ctypes.data, cap, C.byref(ic), C.byref(oc))
        _raise(rc, self)
        return out[:oc.value].tobytes(), (ic.value, oc.value)

    def decompress(self, data, model, out_capacity):
        """bytes -> (raw bytes, (in_count, out_count)); redux::decompress (src/lib.rs:113-120)."""
        a = np.frombuffer(bytes(data), dtype=np.uint8)
        out = np.empty(max(out_capacity, 1), dtype=np.uint8)
        pc = model.params._c()
        if model.freq is not None:
            coff = np.array([0, a.size], dtype=np.uint64)
            roff = np.array([0, out_capacity], dtype=np.uint64)
            rl, cons = np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64)
            st = np.zeros(1, dtype=np.int32)
            rc = lib().redux_decode_batch_ex(self._h, model.kind, C.byref(pc), model._freq_ptr(),
                                             a.ctypes.data if a.size else None, _ptr(coff), 1, out.ctypes.data,
                                             _ptr(roff), _ptr(rl), _ptr(cons), _ptr(st))
            icv, ocv = int(cons[0]), int(rl[0])
        else:
            ic, oc = C.c_uint64(), C.c_uint64()
            rc = lib().redux_decompress(self._h, model.kind, C.byref(pc), a.ctypes.data if a.size else None, a.size,
                                        out.ctypes.data, out_capacity, C.byref(ic), C.byref(oc))
            icv, ocv = ic.value, oc.value
        if rc not in (OK,):
            err = _ERRORS.get(rc, ReduxError)(lib().redux_error_string(rc).decode())
            err.partial = out[:ocv].tobytes()
            err.counts = (icv, ocv)
            raise err
        return out[:ocv].tobytes(), (icv, ocv)

    # ---- batch, host buffers
    def encode_batch(self, data, offsets, model, out=None, check=True):
        """data: uint8 array; offsets: uint64[n+1]. Returns (out uint8 array view, out_offsets, status)."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = offsets.size - 1
        if out is None:
            lens = offsets[1:] - offsets[:-1]
            nsym = lens * np.uint64(8) // np.uint64(model.params.symbol_bits) + np.uint64(1)
            cap = int((nsym * np.uint64(model.params.code_bits) + np.uint64(7)).sum() // 8) + 8 * n
            out = np.empty(max(cap, 1), dtype=np.uint8)
        out_off = np.zeros(n + 1, dtype=np.uint64)
        status = np.zeros(max(n, 1), dtype=np.int32)
        pc = model.params._c()
        rc = lib().redux_encode_batch_ex(self._h, model.kind, C.byref(pc), model._freq_ptr(), _ptr(data),
                                         _ptr(offsets), n, _ptr(out), out.size, _ptr(out_off), _ptr(status))
        if check:
            _raise(rc, self)
        return out[:int(out_off[n])], out_off, status[:n]

    def decode_batch(self, comp, comp_offsets, raw_offsets, model, raw=None, check=True):
        """Returns (raw uint8 array, raw_lens, consumed, status)."""
        comp = np.ascontiguousarray(comp, dtype=np.uint8)
        comp_offsets = np.ascontiguousarray(comp_offsets, dtype=np.uint64)
        raw_offsets = np.ascontiguousarray(raw_offsets, dtype=np.uint64)
        n = comp_offsets.size - 1
        if raw is None:
            raw = np.zeros(max(int(raw_offsets[-1]), 1), dtype=np.uint8)
        raw_lens = np.zeros(max(n, 1), dtype=np.uint64)
        consumed = np.zeros(max(n, 1), dtype=np.uint64)
        status = np.zeros(max(n, 1), dtype=np.int32)
        pc = model.params._c()
        rc = lib().redux_decode_batch_ex(self._h, model.kind, C.byref(pc), model._freq_ptr(), _ptr(comp),
                                         _ptr(comp_offsets), n, _ptr(raw), _ptr(raw_offsets), _ptr(raw_lens),
                                         _ptr(consumed), _ptr(status))
        if check:
            _raise(rc, self)
        return raw, raw_lens[:n], consumed[:n], status[:n]

    def encode_batch_models(self, data, offsets, models, block_model, out=None, check=True):
        """encode_batch with a start model per block: block i starts from models[block_model[i]] (block_model None:
        only with one model).  models: AdaptiveLinearModel / AdaptiveTreeModel of one kind and one Parameters, fresh or
        trained.  A block whose index is out of range gets status InvalidInput and an empty stream.  Returns
        (out uint8 array view, out_offsets, status)."""
        kind, pc, table = _model_table(models)
        bm = _block_model(block_model)
        data = np.ascontiguousarray(data, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = offsets.size - 1
        if out is None:
            lens = offsets[1:] - offsets[:-1]
            nsym = lens * np.uint64(8) // np.uint64(pc.symbol_bits) + np.uint64(1)
            cap = int((nsym * np.uint64(pc.code_bits) + np.uint64(7)).sum() // 8) + 8 * n
            out = np.empty(max(cap, 1), dtype=np.uint8)
        out_off = np.zeros(n + 1, dtype=np.uint64)
        status = np.zeros(max(n, 1), dtype=np.int32)
        rc = lib().redux_encode_batch_models(self._h, kind, C.byref(pc), _ptr(table), table.shape[0], _ptr(bm),
                                             _ptr(data), _ptr(offsets), n, _ptr(out), out.size, _ptr(out_off),
                                             _ptr(status))
        if check:
            _raise(rc, self)
        return out[:int(out_off[n])], out_off, status[:n]

    def decode_batch_models(self, comp, comp_offsets, raw_offsets, models, block_model, raw=None, check=True):
        """decode_batch with a start model per block (see encode_batch_models).  Returns (raw uint8 array, raw_lens,
        consumed, status)."""
        kind, pc, table = _model_table(models)
        bm = _block_model(block_model)
        comp = np.ascontiguousarray(comp, dtype=np.uint8)
        comp_offsets = np.ascontiguousarray(comp_offsets, dtype=np.uint64)
        raw_offsets = np.ascontiguousarray(raw_offsets, dtype=np.uint64)
        n = comp_offsets.size - 1
        if raw is None:
            raw = np.zeros(max(int(raw_offsets[-1]), 1), dtype=np.uint8)
        raw_lens = np.zeros(max(n, 1), dtype=np.uint64)
        consumed = np.zeros(max(n, 1), dtype=np.uint64)
        status = np.zeros(max(n, 1), dtype=np.int32)
        rc = lib().redux_decode_batch_models(self._h, kind, C.byref(pc), _ptr(table), table.shape[0], _ptr(bm),
                                             _ptr(comp), _ptr(comp_offsets), n, _ptr(raw), _ptr(raw_offsets),
                                             _ptr(raw_lens), _ptr(consumed), _ptr(status))
        if check:
            _raise(rc, self)
        return raw, raw_lens[:n], consumed[:n], status[:n]

    # ---- training start models on the device (redux_train_models, DESIGN.md 3.9)
    def train_models(self, data, offsets, start):
        """One new model per sample: sample i = data[offsets[i]:offsets[i+1]] trains a copy of its start model exactly
        as get_frequency() of every symbol the reference's reader yields from it would.  start: one model (fresh or
        trained) for every sample, or a list of n models, sample i starting from start[i].  The models passed in are
        not modified.  Returns a list of n models of start's kind and Parameters."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = offsets.size - 1
        cls, params, pc, table, n_models, sm = _train_start(start, n)
        out = np.zeros((max(n, 1), params.symbol_count), dtype=np.uint32)
        _raise(lib().redux_train_models(self._h, C.byref(pc), _ptr(table), n_models, _ptr(sm),
                                        _ptr(data) if data.size else None, _ptr(offsets), n, _ptr(out)), self)
        return _trained_models(cls, params, out[:n])

    def train_models_device(self, d_in, d_in_offsets, n_samples, max_sample_len, d_out_freqs, start, device=0,
                            stream=None):
        """train_models on device-resident buffers: d_out_freqs (uint32, n_samples x symbol_count) receives the rows.
        Asynchronous on `stream`; `start` as in train_models (host models)."""
        _, _, pc, table, n_models, sm = _train_start(start, n_samples)
        _raise(lib().redux_train_models_device(self._h, device, stream, C.byref(pc), _ptr(table), n_models, _ptr(sm),
                                               _ptr(d_in), _ptr(d_in_offsets), n_samples, max_sample_len,
                                               _ptr(d_out_freqs)), self)

    # ---- batch, device-resident (tensors or raw device addresses); asynchronous on `stream`
    def encode_batch_device(self, d_in, d_in_offsets, n_blocks, max_block_len, d_out, out_capacity,
                            d_out_offsets, d_status, model, device=0, stream=None):
        pc = model.params._c()
        _raise(lib().redux_encode_batch_device_ex(self._h, device, stream, model.kind, C.byref(pc), model._freq_ptr(),
                                                  _ptr(d_in), _ptr(d_in_offsets), n_blocks, max_block_len, _ptr(d_out),
                                                  out_capacity, _ptr(d_out_offsets), _ptr(d_status)), self)

    def decode_batch_device(self, d_comp, d_comp_offsets, n_blocks, max_block_len, d_raw, d_raw_offsets,
                            d_raw_lens, d_consumed, d_status, model, device=0, stream=None):
        pc = model.params._c()
        _raise(lib().redux_decode_batch_device_ex(self._h, device, stream, model.kind, C.byref(pc), model._freq_ptr(),
                                                  _ptr(d_comp), _ptr(d_comp_offsets), n_blocks, max_block_len,
                                                  _ptr(d_raw), _ptr(d_raw_offsets), _ptr(d_raw_lens), _ptr(d_consumed),
                                                  _ptr(d_status)), self)

    def encode_batch_device_models(self, d_in, d_in_offsets, n_blocks, max_block_len, d_out, out_capacity,
                                   d_out_offsets, d_status, models, d_block_model, device=0, stream=None):
        """encode_batch_device with a start model per block: d_block_model is a device uint32 tensor (or address) of
        n_blocks row indices, None only with one model."""
        kind, pc, table = _model_table(models)
        _raise(lib().redux_encode_batch_device_models(self._h, device, stream, kind, C.byref(pc), _ptr(table),
                                                      table.shape[0], _ptr(d_block_model), _ptr(d_in), _ptr(d_in_offsets),
                                                      n_blocks, max_block_len, _ptr(d_out), out_capacity,
                                                      _ptr(d_out_offsets), _ptr(d_status)), self)

    def decode_batch_device_models(self, d_comp, d_comp_offsets, n_blocks, max_block_len, d_raw, d_raw_offsets,
                                   d_raw_lens, d_consumed, d_status, models, d_block_model, device=0, stream=None):
        kind, pc, table = _model_table(models)
        _raise(lib().redux_decode_batch_device_models(self._h, device, stream, kind, C.byref(pc), _ptr(table),
                                                      table.shape[0], _ptr(d_block_model), _ptr(d_comp),
                                                      _ptr(d_comp_offsets), n_blocks, max_block_len, _ptr(d_raw),
                                                      _ptr(d_raw_offsets), _ptr(d_raw_lens), _ptr(d_consumed),
                                                      _ptr(d_status)), self)

    def set_text_corpus(self, corpus):
        """bytes / uint8 array (or None): the corpus the synthetic generator cuts its text-class blocks from."""
        if corpus is None:
            _raise(lib().redux_ctx_set_text_corpus(self._h, None, 0), self)
            return
        a = np.frombuffer(bytes(corpus), dtype=np.uint8) if not isinstance(corpus, np.ndarray) else np.ascontiguousarray(corpus, dtype=np.uint8)
        _raise(lib().redux_ctx_set_text_corpus(self._h, a.ctypes.data, a.size), self)

    def generate_blocks_device(self, d_out, first_block, n_blocks, block_len, seed, device=0, stream=None):
        _raise(lib().redux_generate_blocks_device(self._h, device, stream, _ptr(d_out), first_block, n_blocks,
                                                  block_len, seed), self)


def generate_blocks_host(first_block, n_blocks, block_len, seed, corpus=None):
    out = np.empty(n_blocks * block_len, dtype=np.uint8)
    if corpus is None:
        lib().redux_generate_blocks_host(out.ctypes.data, first_block, n_blocks, block_len, seed)
    else:
        a = np.frombuffer(bytes(corpus), dtype=np.uint8) if not isinstance(corpus, np.ndarray) else np.ascontiguousarray(corpus, dtype=np.uint8)
        lib().redux_generate_blocks_host_ex(out.ctypes.data, first_block, n_blocks, block_len, seed, a.ctypes.data, a.size)
    return out


_default_ctx = None


def _ctx():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context()
    return _default_ctx


# --------------------------------------------------------------------------- the drop-in pair
def compress(istream, ostream, model, context=None):
    """``redux::compress(istream, ostream, model) -> (u64, u64)`` (src/lib.rs:102-109).
    istream: object with ``read()`` (std::io::Read); ostream: object with ``write()`` (std::io::Write).
    Returns (bytes read from istream, bytes written to ostream). Raises the Error variants."""
    data = istream.read()
    out, counts = (context or _ctx()).compress(data, model)
    ostream.write(out)
    return counts


def decompress(istream, ostream, model, context=None, max_output=None):
    """``redux::decompress(istream, ostream, model) -> (u64, u64)`` (src/lib.rs:113-120).
    The stream is headerless, so the decoded length is unknown up front: the output slot starts at
    ``max_output`` (default 8x the input + 64 KiB) and is doubled while the device reports it full."""
    data = istream.read()
    ctx = context or _ctx()
    cap = max_output if max_output is not None else 8 * len(data) + 65536
    while True:
        try:
            out, counts = ctx.decompress(data, model, cap)
            break
        except OutCapacity:
            if max_output is not None:
                raise
            cap *= 4
        except Eof as e:
            ostream.write(getattr(e, "partial", b""))   # streaming semantics: decoded prefix stays written
            raise
    ostream.write(out)
    return counts
