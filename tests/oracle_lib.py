"""ctypes binding of the CPU oracle (oracle/libredux_oracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package (redux_b200/) never imports it.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(_HERE), "oracle")
_SO_PORTABLE = os.path.join(ORACLE_DIR, "libredux_oracle.so")
_SO = _SO_PORTABLE

OK, EOF, INVALID_INPUT, IO_ERROR = 0, 1, 2, 3
LINEAR, TREE = 0, 1


class Params(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "symbol_bits", "symbol_eof", "symbol_count", "freq_bits", "freq_max", "code_bits",
        "code_min", "code_one_fourth", "code_half", "code_three_fourths", "code_max")]


def build(force=False):
    srcs = [os.path.join(ORACLE_DIR, f) for f in ("redux_oracle.c", "synth_blocks.c", "redux_oracle.h")]
    if force or not os.path.exists(_SO_PORTABLE) or any(
            os.path.exists(src) and os.path.getmtime(src) > os.path.getmtime(_SO_PORTABLE) for src in srcs):
        subprocess.run(["make", "-C", ORACLE_DIR, "-s"], check=True)
    return _SO_PORTABLE


_lib = None
_flavour = "portable (-O3)"


def use_native_build():
    """bench.py's CPU arm: rebuild the oracle with -O3 -march=native ON THIS HOST and load that build (must be
    called before the first lib()).  The build goes to a temporary directory (removed at exit), so that the
    benchmark runs from a read-only tree.  Falls back to the portable build when there is no compiler.  Returns
    a description for the JSON line."""
    global _SO, _flavour
    if _lib is not None:
        return _flavour
    try:
        tmp = tempfile.mkdtemp(prefix="redux_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        native = os.path.join(tmp, "libredux_oracle_native.so")
        r = subprocess.run(["make", "-C", ORACLE_DIR, "-s", "NATIVE=" + native, "native"],
                           capture_output=True, text=True, timeout=120)
        if r.returncode == 0 and os.path.exists(native):
            _SO = native
            _flavour = "-O3 -march=native, built on this host"
    except Exception:
        pass
    return _flavour


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if _SO == _SO_PORTABLE:
        build()
    L = C.CDLL(_SO)
    L.oracle_generate_blocks.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64]
    L.oracle_generate_blocks.restype = None
    L.oracle_generate_blocks_ex.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64]
    L.oracle_generate_blocks_ex.restype = None
    u64, p8, pu64 = C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)
    L.oracle_params_new.argtypes = [u64, u64, u64, C.POINTER(Params)]
    L.oracle_params_new.restype = C.c_int
    L.oracle_model_new.argtypes = [C.c_int, C.POINTER(Params)]
    L.oracle_model_new.restype = C.c_void_p
    L.oracle_model_free.argtypes = [C.c_void_p]
    L.oracle_model_total_frequency.argtypes = [C.c_void_p]
    L.oracle_model_total_frequency.restype = u64
    L.oracle_model_get_frequency.argtypes = [C.c_void_p, u64, pu64, pu64]
    L.oracle_model_get_symbol.argtypes = [C.c_void_p, u64, pu64, pu64, pu64]
    L.oracle_model_get_freq_table.argtypes = [C.c_void_p, C.c_void_p]
    L.oracle_bitwriter_new.argtypes = [p8, C.c_size_t]
    L.oracle_bitwriter_new.restype = C.c_void_p
    L.oracle_bitwriter_free.argtypes = [C.c_void_p]
    L.oracle_bitwriter_write_bits.argtypes = [C.c_void_p, u64, u64]
    L.oracle_bitwriter_flush_bits.argtypes = [C.c_void_p]
    L.oracle_bitwriter_get_count.argtypes = [C.c_void_p]
    L.oracle_bitwriter_get_count.restype = u64
    L.oracle_bitreader_new.argtypes = [p8, C.c_size_t]
    L.oracle_bitreader_new.restype = C.c_void_p
    L.oracle_bitreader_free.argtypes = [C.c_void_p]
    L.oracle_bitreader_read_bits.argtypes = [C.c_void_p, u64, pu64]
    L.oracle_bitreader_get_count.argtypes = [C.c_void_p]
    L.oracle_bitreader_get_count.restype = u64
    for name in ("oracle_compress", "oracle_decompress"):
        fn = getattr(L, name)
        fn.argtypes = [C.c_int, u64, u64, u64, p8, C.c_size_t, p8, C.c_size_t, pu64, pu64]
        fn.restype = C.c_int
    for name in ("oracle_compress_trained", "oracle_decompress_trained"):
        fn = getattr(L, name)
        fn.argtypes = [C.c_int, u64, u64, u64, p8, C.c_size_t, p8, C.c_size_t, p8, C.c_size_t, pu64, pu64]
        fn.restype = C.c_int
    L.oracle_compress_bound.argtypes = [C.c_size_t, u64, u64]
    L.oracle_compress_bound.restype = C.c_size_t
    L.oracle_compress_batch.argtypes = [C.c_int, u64, u64, u64, p8, p8, u64, p8, p8, p8, p8, C.c_int]
    L.oracle_compress_batch.restype = C.c_int
    L.oracle_decompress_batch.argtypes = [C.c_int, u64, u64, u64, p8, p8, u64, p8, p8, p8, p8, p8, C.c_int]
    L.oracle_decompress_batch.restype = C.c_int
    _lib = L
    return L


def params_new(s, f, c):
    p = Params()
    rc = lib().oracle_params_new(s, f, c, C.byref(p))
    return rc, p


def compress_bound(n, s=8, c=32):
    return lib().oracle_compress_bound(n, s, c)


def _as_u8(data):
    a = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    return np.ascontiguousarray(a, dtype=np.uint8)


def compress(data, kind=TREE, params=(8, 30, 32), out_cap=None):
    """redux::compress over memory. Returns (status, out_bytes, in_count, out_count)."""
    a = _as_u8(data)
    s, f, c = params
    cap = out_cap if out_cap is not None else max(16, (a.size + 1) * 8 + 16)
    out = np.zeros(cap, dtype=np.uint8)
    ic, oc = C.c_uint64(0), C.c_uint64(0)
    rc = lib().oracle_compress(kind, s, f, c, a.ctypes.data, a.size, out.ctypes.data, cap,
                               C.byref(ic), C.byref(oc))
    return rc, out[:oc.value].tobytes(), ic.value, oc.value


def decompress(data, kind=TREE, params=(8, 30, 32), out_cap=None):
    """redux::decompress over memory. Returns (status, out_bytes, in_count, out_count)."""
    a = _as_u8(data)
    s, f, c = params
    cap = out_cap if out_cap is not None else max(64, a.size * 64 + 1024)
    out = np.zeros(cap, dtype=np.uint8)
    ic, oc = C.c_uint64(0), C.c_uint64(0)
    rc = lib().oracle_decompress(kind, s, f, c, a.ctypes.data, a.size, out.ctypes.data, cap,
                                 C.byref(ic), C.byref(oc))
    return rc, out[:oc.value].tobytes(), ic.value, oc.value


def _trained(fn, data, train, kind, params, cap):
    a = _as_u8(data)
    tr = np.ascontiguousarray(train, dtype=np.uint64)
    s, f, c = params
    out = np.zeros(cap, dtype=np.uint8)
    ic, oc = C.c_uint64(0), C.c_uint64(0)
    rc = fn(kind, s, f, c, tr.ctypes.data, tr.size, a.ctypes.data, a.size, out.ctypes.data, cap, C.byref(ic), C.byref(oc))
    return rc, out[:oc.value].tobytes(), ic.value, oc.value


def compress_trained(data, train, kind=TREE, params=(8, 30, 32), out_cap=None):
    """compress() with a model the caller trained by calling get_frequency(sym) for sym in `train` first."""
    s, f, c = params
    cap = out_cap if out_cap is not None else max(16, (len(data) * 8 // s + 1) * 8 + 16)
    return _trained(lib().oracle_compress_trained, data, train, kind, params, cap)


def decompress_trained(data, train, kind=TREE, params=(8, 30, 32), out_cap=None):
    cap = out_cap if out_cap is not None else max(64, len(data) * 64 + 1024)
    return _trained(lib().oracle_decompress_trained, data, train, kind, params, cap)


def trained_frequencies(train, kind=TREE, params=(8, 30, 32)):
    """Per-symbol frequency vector of a model after get_frequency(sym) for sym in `train` (uint32[symbol_count])."""
    m = Model(kind, *params)
    for t in train:
        rc, lo, hi = m.get_frequency(int(t))
        assert rc == OK
    tab = m.get_freq_table()
    return (tab[:, 1] - tab[:, 0]).astype(np.uint32)


def generate_blocks(first_block, n_blocks, block_len, seed, corpus=None):
    """The synthetic mixed-entropy blocks of the benchmark, from the oracle side (oracle/synth_blocks.c); corpus =
    the bytes the text class cuts its windows from (None: the table-driven stand-in)."""
    out = np.empty(n_blocks * block_len, dtype=np.uint8)
    if corpus is None:
        lib().oracle_generate_blocks(out.ctypes.data, first_block, n_blocks, block_len, seed)
    else:
        a = np.frombuffer(bytes(corpus), dtype=np.uint8) if not isinstance(corpus, np.ndarray) else np.ascontiguousarray(corpus, dtype=np.uint8)
        lib().oracle_generate_blocks_ex(out.ctypes.data, first_block, n_blocks, block_len, seed, a.ctypes.data, a.size)
    return out


def compress_batch(inp, in_off, kind=TREE, params=(8, 30, 32), threads=1):
    """One stream per block, `threads` host threads. inp: uint8 array, in_off: uint64[n+1].
    Returns (rc, out uint8 array of slots, slot_off uint64[n+1], out_len uint64[n], status int32[n])."""
    s, f, c = params
    inp = np.ascontiguousarray(inp, dtype=np.uint8)
    in_off = np.ascontiguousarray(in_off, dtype=np.uint64)
    n = in_off.size - 1
    lens = (in_off[1:] - in_off[:-1]).astype(np.uint64)
    caps = ((lens + 1) * np.uint64(c) + np.uint64(7)) // np.uint64(8)
    slot_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(caps, out=slot_off[1:])
    out = np.empty(int(slot_off[-1]), dtype=np.uint8)
    out_len = np.zeros(n, dtype=np.uint64)
    status = np.zeros(n, dtype=np.int32)
    rc = lib().oracle_compress_batch(kind, s, f, c, inp.ctypes.data, in_off.ctypes.data, n,
                                     out.ctypes.data, slot_off.ctypes.data, out_len.ctypes.data,
                                     status.ctypes.data, threads)
    return rc, out, slot_off, out_len, status


def decompress_batch(comp, comp_off, raw_off, kind=TREE, params=(8, 30, 32), threads=1):
    """Decode blocks comp[comp_off[i]:comp_off[i+1]] into slots raw_off. Returns
    (rc, raw uint8 array, raw_len, consumed, status)."""
    s, f, c = params
    comp = np.ascontiguousarray(comp, dtype=np.uint8)
    comp_off = np.ascontiguousarray(comp_off, dtype=np.uint64)
    raw_off = np.ascontiguousarray(raw_off, dtype=np.uint64)
    n = comp_off.size - 1
    raw = np.empty(int(raw_off[-1]), dtype=np.uint8)
    raw_len = np.zeros(n, dtype=np.uint64)
    consumed = np.zeros(n, dtype=np.uint64)
    status = np.zeros(n, dtype=np.int32)
    rc = lib().oracle_decompress_batch(kind, s, f, c, comp.ctypes.data, comp_off.ctypes.data, n,
                                       raw.ctypes.data, raw_off.ctypes.data, raw_len.ctypes.data,
                                       consumed.ctypes.data, status.ctypes.data, threads)
    return rc, raw, raw_len, consumed, status


class Model:
    """Model trait object (src/model/mod.rs:17-29) over the oracle."""

    def __init__(self, kind, s, f, c):
        rc, p = params_new(s, f, c)
        assert rc == OK
        self.params = p
        self._m = lib().oracle_model_new(kind, C.byref(p))

    def __del__(self):
        if getattr(self, "_m", None):
            lib().oracle_model_free(self._m)
            self._m = None

    def total_frequency(self):
        return lib().oracle_model_total_frequency(self._m)

    def get_frequency(self, symbol):
        lo, hi = C.c_uint64(), C.c_uint64()
        rc = lib().oracle_model_get_frequency(self._m, symbol, C.byref(lo), C.byref(hi))
        return rc, lo.value, hi.value

    def get_symbol(self, value):
        s, lo, hi = C.c_uint64(), C.c_uint64(), C.c_uint64()
        rc = lib().oracle_model_get_symbol(self._m, value, C.byref(s), C.byref(lo), C.byref(hi))
        return rc, s.value, lo.value, hi.value

    def get_freq_table(self):
        out = np.zeros(2 * self.params.symbol_count, dtype=np.uint64)
        lib().oracle_model_get_freq_table(self._m, out.ctypes.data)
        return out.reshape(-1, 2)
