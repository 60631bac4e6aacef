"""ctypes wrapper over oracle/c/liblc_oracle.so — the plain-C restatement of the reference's CPU path.

TEST / BENCH INFRASTRUCTURE ONLY (see oracle/liquid_oracle.py): used by tests to cross-check the C port against the
Python oracle, and by bench.py as the timed CPU baseline. Never imported by liquid_cache_b200.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pyarrow as pa

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c")
_LIB = None


def _load_fresh_build() -> C.CDLL:
    """gcc -O3 -march=native on the machine that will time it, into a temporary directory: the tree may be read-only."""
    with tempfile.TemporaryDirectory() as d:
        so = os.path.join(d, "liblc_oracle.so")
        subprocess.run(["make", "-C", _HERE, "-B", f"OUT={so}"], check=True, stdout=subprocess.DEVNULL)
        return C.CDLL(so)


def lib(rebuild: bool = False) -> C.CDLL:
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "liblc_oracle.so")
        l = _load_fresh_build() if rebuild or not os.path.exists(so) else C.CDLL(so)
        vp, u32, u64, i64 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int64
        l.lco_int_encode.restype = vp
        l.lco_int_encode.argtypes = [vp, vp, u32, C.c_int, C.c_int]
        l.lco_int_free.argtypes = [vp]
        l.lco_int_filter.restype = u32
        l.lco_int_filter.argtypes = [vp, vp, vp, vp, C.POINTER(u32)]
        l.lco_int_eval.restype = u32
        l.lco_int_eval.argtypes = [vp, vp, C.c_int, i64, u64, vp, vp, C.POINTER(u32)]
        l.lco_fsst_train.restype = vp
        l.lco_fsst_train.argtypes = [vp, vp, u32]
        l.lco_fsst_free.argtypes = [vp]
        l.lco_str_encode.restype = vp
        l.lco_str_encode.argtypes = [vp, vp, vp, u32, vp, C.c_int]
        l.lco_str_free.argtypes = [vp]
        l.lco_str_bytes.restype = u64
        l.lco_str_bytes.argtypes = [vp]
        l.lco_str_like.restype = u32
        l.lco_str_like.argtypes = [vp, vp, vp, u32, C.c_int, vp, vp, C.POINTER(u32)]
        l.lco_str_eq.restype = u32
        l.lco_str_eq.argtypes = [vp, vp, vp, u32, C.c_int, vp, vp, C.POINTER(u32)]
        l.lco_str_filter.restype = u32
        l.lco_str_filter.argtypes = [vp, vp, vp, vp, vp, C.POINTER(u32), C.POINTER(u64)]
        l.lco_and_then.argtypes = [vp, u64, vp, u64, vp]
        l.lco_scan.restype = u64
        l.lco_scan.argtypes = [vp, u32, C.c_int, vp, u32, C.c_int, i64, C.c_int, i64, u32, C.POINTER(u64)]
        l.lco_scan_serial.restype = u64
        l.lco_scan_serial.argtypes = [vp, u32, C.c_int, vp, u32, C.c_int, i64, C.c_int, i64, C.POINTER(u64)]
        l.lco_pool_create.restype = vp
        l.lco_pool_create.argtypes = [u32]
        l.lco_pool_destroy.argtypes = [vp]
        l.lco_pool_set_second.argtypes = [vp, vp, C.c_int, i64]
        l.lco_pool_scan.restype = u64
        l.lco_pool_scan.argtypes = [vp, vp, u32, C.c_int, vp, u32, C.c_int, i64, C.c_int, i64, u32, C.POINTER(u64)]
        _LIB = l
    return _LIB


def _validity_bytes(arr: pa.Array):
    if arr.null_count == 0:
        return None
    v = np.asarray(arr.is_valid().to_numpy(zero_copy_only=False), dtype=bool)
    return np.packbits(v, bitorder="little")


def _sel_bytes(sel):
    if sel is None:
        return None
    m = np.asarray(sel.to_numpy(zero_copy_only=False) if isinstance(sel, pa.Array) else sel, dtype=bool)
    b = np.packbits(m, bitorder="little")
    return np.concatenate([b, np.zeros(16, np.uint8)])


def _mask_array(mask: np.ndarray, valid: np.ndarray, k: int, nulls: int) -> pa.Array:
    vals = np.unpackbits(mask, bitorder="little")[:k].astype(bool)
    if nulls == 0:
        return pa.array(vals, type=pa.bool_())
    ok = np.unpackbits(valid, bitorder="little")[:k].astype(bool)
    return pa.array(vals, type=pa.bool_(), mask=~ok)


class CIntArray:
    def __init__(self, arr: pa.Array):
        from .liquid_oracle import _int_storage

        np_dt, bits = _int_storage(arr.type)
        self.arrow_type, self.np_dt, self.n = arr.type, np_dt, len(arr)
        plain = arr.cast(pa.from_numpy_dtype(np_dt)) if not pa.types.is_integer(arr.type) else arr
        vals = np.ascontiguousarray(plain.fill_null(0).to_numpy(zero_copy_only=False).astype(np_dt))
        valid = _validity_bytes(arr)
        self._keep = (vals, valid)
        self.ptr = lib().lco_int_encode(vals.ctypes.data, valid.ctypes.data if valid is not None else None, self.n, bits,
                                        1 if np_dt.kind == "i" else 0)

    def __del__(self):
        try:
            lib().lco_int_free(self.ptr)
        except Exception:
            pass

    def filter(self, sel) -> pa.Array:
        s = _sel_bytes(sel)
        out = np.zeros(max(self.n, 1), dtype=self.np_dt)
        valid = np.zeros(self.n // 8 + 16, dtype=np.uint8)
        nulls = C.c_uint32(0)
        k = lib().lco_int_filter(self.ptr, s.ctypes.data if s is not None else None, out.ctypes.data, valid.ctypes.data,
                                 C.byref(nulls))
        mask = None if nulls.value == 0 else ~np.unpackbits(valid, bitorder="little")[:k].astype(bool)
        plain = pa.array(out[:k], mask=mask)
        return plain.cast(self.arrow_type) if plain.type != self.arrow_type else plain

    def eval(self, op: str, literal: int, sel) -> pa.Array:
        s = _sel_bytes(sel)
        opi = {"=": 0, "!=": 1, "<": 2, "<=": 3, ">": 4, ">=": 5}[op]
        mask = np.zeros(self.n // 8 + 16, dtype=np.uint8)
        valid = np.zeros(self.n // 8 + 16, dtype=np.uint8)
        nulls = C.c_uint32(0)
        k = lib().lco_int_eval(self.ptr, s.ctypes.data if s is not None else None, opi, literal if literal < 2**63 else 0,
                               literal & (2**64 - 1), mask.ctypes.data, valid.ctypes.data, C.byref(nulls))
        return _mask_array(mask, valid, k, nulls.value)


class CFsst:
    def __init__(self, arr: pa.Array):
        off, data = _utf8_buffers(arr)
        self._keep = (off, data)
        self.ptr = lib().lco_fsst_train(data.ctypes.data, off.ctypes.data, len(arr))

    def __del__(self):
        try:
            lib().lco_fsst_free(self.ptr)
        except Exception:
            pass


def _utf8_buffers(arr: pa.Array):
    arr = arr.cast(pa.string()) if arr.type != pa.string() else arr
    bufs = arr.buffers()
    off = np.frombuffer(bufs[1], dtype=np.int32, count=len(arr) + 1 + arr.offset)[arr.offset:].copy()
    data = np.frombuffer(bufs[2], dtype=np.uint8).copy() if bufs[2] is not None and bufs[2].size else np.zeros(8, np.uint8)
    data = np.concatenate([data, np.zeros(16, np.uint8)])
    return off, data


class CStrArray:
    def __init__(self, arr: pa.Array, fsst: CFsst, build_fingerprints: bool = False):
        off, data = _utf8_buffers(arr)
        valid = _validity_bytes(arr)
        self.n, self.fsst = len(arr), fsst
        self.ptr = lib().lco_str_encode(off.ctypes.data, data.ctypes.data, valid.ctypes.data if valid is not None else None,
                                        self.n, fsst.ptr, 1 if build_fingerprints else 0)

    def __del__(self):
        try:
            lib().lco_str_free(self.ptr)
        except Exception:
            pass

    def nbytes(self) -> int:
        return int(lib().lco_str_bytes(self.ptr))

    def _run(self, fn, sel, needle: bytes, negate: bool) -> pa.Array:
        s = _sel_bytes(sel)
        mask = np.zeros(self.n // 8 + 16, dtype=np.uint8)
        valid = np.zeros(self.n // 8 + 16, dtype=np.uint8)
        nulls = C.c_uint32(0)
        k = fn(self.ptr, s.ctypes.data if s is not None else None, needle, len(needle), 1 if negate else 0,
               mask.ctypes.data, valid.ctypes.data, C.byref(nulls))
        return _mask_array(mask, valid, k, nulls.value)

    def like(self, inner: bytes, sel=None, negate=False) -> pa.Array:
        return self._run(lib().lco_str_like, sel, inner, negate)

    def eq(self, needle: bytes, sel=None, negate=False) -> pa.Array:
        return self._run(lib().lco_str_eq, sel, needle, negate)

    def filter(self, sel=None) -> pa.Array:
        s = _sel_bytes(sel)
        off = np.zeros(self.n + 1, dtype=np.int32)
        valid = np.zeros(self.n // 8 + 16, dtype=np.uint8)
        nulls, nbytes = C.c_uint32(0), C.c_uint64(0)
        k = lib().lco_str_filter(self.ptr, s.ctypes.data if s is not None else None, off.ctypes.data, None, valid.ctypes.data,
                                 C.byref(nulls), C.byref(nbytes))
        data = np.zeros(int(nbytes.value) + 16, dtype=np.uint8)
        k = lib().lco_str_filter(self.ptr, s.ctypes.data if s is not None else None, off.ctypes.data, data.ctypes.data,
                                 valid.ctypes.data, C.byref(nulls), C.byref(nbytes))
        vb = None
        if nulls.value:
            vb = pa.py_buffer(valid[: (k + 7) // 8].copy())
        return pa.Array.from_buffers(pa.string(), k, [vb, pa.py_buffer(off[: k + 1].copy()),
                                                      pa.py_buffer(data[: int(nbytes.value)].copy())], null_count=nulls.value)


def and_then(left: np.ndarray, right: np.ndarray) -> np.ndarray:
    lb = np.concatenate([np.packbits(left, bitorder="little"), np.zeros(16, np.uint8)])
    rb = np.concatenate([np.packbits(right, bitorder="little"), np.zeros(24, np.uint8)])
    out = np.zeros(len(lb) + 8, dtype=np.uint8)
    lib().lco_and_then(lb.ctypes.data, len(left), rb.ctypes.data, len(right), out.ctypes.data)
    return np.unpackbits(out, bitorder="little")[: len(left)].astype(bool)


def scan(entries: list, kind: int, needle: bytes = b"", op1: int = 0, lit1: int = 0, op2: int = 0, lit2: int = 0,
         nthreads: int = 1):
    """Threaded scan driver over encoded entries (CStrArray / CIntArray). Returns (matched rows, rows scanned)."""
    ptrs = (C.c_void_p * len(entries))(*[e.ptr for e in entries])
    rows = C.c_uint64(0)
    matched = lib().lco_scan(ptrs, len(entries), kind, needle, len(needle), op1, lit1, op2, lit2, nthreads, C.byref(rows))
    return int(matched), int(rows.value)


class ScanPool:
    """Persistent worker threads for the timed CPU arm (created once, outside every timed region), standing in for the
    reference's tokio partition tasks. `bind(entries)` fixes the entry list so that a pass is one C call with no Python
    work inside the clock."""

    def __init__(self, nthreads: int):
        self.nthreads = max(1, int(nthreads))
        self.ptr = lib().lco_pool_create(self.nthreads)
        self._ptrs = None
        self._n = 0

    def bind(self, entries: list) -> "ScanPool":
        self._keep = entries
        self._n = len(entries)
        self._ptrs = (C.c_void_p * self._n)(*[e.ptr for e in entries])
        return self

    def bind_second(self, entries2: list, op3: int, lit3: int) -> "ScanPool":
        """kind 4: the second column of every batch (same order as the bound list) and the conjunct on it."""
        assert len(entries2) == self._n
        self._keep2 = entries2
        self._ptrs2 = (C.c_void_p * self._n)(*[e.ptr for e in entries2])
        lib().lco_pool_set_second(self.ptr, self._ptrs2, op3, lit3)
        return self

    def scan(self, kind: int, needle: bytes = b"", op1: int = 0, lit1: int = 0, op2: int = 0, lit2: int = 0, grain: int = 4):
        rows = C.c_uint64(0)
        matched = lib().lco_pool_scan(self.ptr, self._ptrs, self._n, kind, needle, len(needle), op1, lit1, op2, lit2, grain,
                                      C.byref(rows))
        return int(matched), int(rows.value)

    def scan_serial(self, kind: int, needle: bytes = b"", op1: int = 0, lit1: int = 0, op2: int = 0, lit2: int = 0,
                    first: int = 0, count=None):
        """The same pass on the calling thread over entries [first, first+count) — the single-thread figure."""
        count = self._n - first if count is None else min(count, self._n - first)
        sub = (C.c_void_p * count)(*[self._ptrs[first + i] for i in range(count)])
        rows = C.c_uint64(0)
        matched = lib().lco_scan_serial(sub, count, kind, needle, len(needle), op1, lit1, op2, lit2, C.byref(rows))
        return int(matched), int(rows.value)

    def close(self):
        if self.ptr:
            lib().lco_pool_destroy(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
