"""grab_b200 -- B200-native scan engine behind grab's match loop.

This package is a thin ctypes face over ``libgscan.so`` (C ABI: ``include/gscan.h``), used by the
tests and ``bench.py``.  The product is the library; there is NO Python or CPU implementation of
the scan -- importing works without a GPU, but opening a context raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GSCAN_LIB") or os.path.join(_HERE, "libgscan.so")  # GSCAN_LIB: tuning variants

MODE_ALL, MODE_FIRST, MODE_LINE = 0, 1, 2
LITERAL, STRICT_REF = 1, 2
UNIT_DEVICE = 1
UNIT_FD = 2  # ptr carries an open descriptor, the window is [base_off, base_off + len) of it (pread by the engine)
ENGINE_FIXED, ENGINE_RUN, ENGINE_NONE, ENGINE_VM = 1, 2, 3, 4
KERNEL_NONE, KERNEL_PAIR, KERNEL_TRIPLE, KERNEL_BALANCED, KERNEL_HASH, KERNEL_RUN = 0, 1, 2, 3, 4, 5


class GscanError(RuntimeError):
    pass


class Unit(ctypes.Structure):
    _fields_ = [("ptr", ctypes.c_void_p), ("len", ctypes.c_uint64), ("base_off", ctypes.c_uint64),
                ("file_id", ctypes.c_uint32), ("flags", ctypes.c_uint32)]


class Match(ctypes.Structure):
    _fields_ = [("start", ctypes.c_uint64), ("file_id", ctypes.c_uint32), ("match_len", ctypes.c_uint32)]


MATCH_DTYPE = np.dtype([("start", "<u8"), ("file_id", "<u4"), ("match_len", "<u4")])
UNIT_DTYPE = np.dtype([("ptr", "<u8"), ("len", "<u8"), ("base_off", "<u8"), ("file_id", "<u4"), ("flags", "<u4")])


class PatternInfo(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("minlen", "maxlen", "captures", "engine", "n_sequences",
                                              "n_filter_tests", "filter_anchor", "filter_delta", "scan_kernel", "scan_variant")]


class Stats(ctypes.Structure):
    _fields_ = [("bytes_scanned", ctypes.c_uint64), ("n_candidates", ctypes.c_uint64), ("n_matches", ctypes.c_uint64),
                ("n_units", ctypes.c_uint32), ("n_tiles", ctypes.c_uint32), ("scan_launches", ctypes.c_uint32),
                ("total_launches", ctypes.c_uint32), ("scan_kernel_ms", ctypes.c_float), ("resolve_ms", ctypes.c_float),
                ("h2d_ms", ctypes.c_float), ("total_ms", ctypes.c_float), ("vm_limit_hit", ctypes.c_uint32), ("reserved", ctypes.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


# every symbol include/gscan.h declares, with its prototype
_PROTOS = {
    "gscan_compile": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.POINTER(ctypes.c_void_p)]),
    "gscan_free_pattern": (None, [ctypes.c_void_p]),
    "gscan_minlen": (ctypes.c_int, [ctypes.c_void_p]),
    "gscan_pattern_get_info": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(PatternInfo)]),
    "gscan_last_error": (ctypes.c_char_p, []),
    "gscan_open": (ctypes.c_void_p, [ctypes.c_int]),
    "gscan_close": (None, [ctypes.c_void_p]),
    "gscan_why": (ctypes.c_char_p, [ctypes.c_void_p]),
    "gscan_scan_batch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32,
                                        ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_size_t)]),
    "gscan_free_matches": (None, [ctypes.c_void_p, ctypes.c_void_p]),
    "gscan_scan_batch_async": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32]),
    "gscan_scan_wait": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_size_t)]),
    "gscan_batch_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_void_p)]),
    "gscan_batch_scan": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32,
                                        ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_size_t)]),
    "gscan_batch_free": (None, [ctypes.c_void_p, ctypes.c_void_p]),
    "gscan_last_stats": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(Stats)]),
    "gscan_last_device_matches": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_size_t)]),
    "gscan_host_alloc": (ctypes.c_void_p, [ctypes.c_size_t]),
    "gscan_host_free": (None, [ctypes.c_void_p]),
    "gscan_device_alloc": (ctypes.c_void_p, [ctypes.c_void_p, ctypes.c_size_t]),
    "gscan_device_free": (None, [ctypes.c_void_p, ctypes.c_void_p]),
    "gscan_memcpy_d2h": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t]),
    "gscan_memcpy_h2d": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t]),
    "gscan_synth_corpus": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64,
                                          ctypes.c_uint64, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_uint32]),
    "gscan_read_probe": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.POINTER(ctypes.c_float),
                                        ctypes.POINTER(ctypes.c_uint64)]),
    "gscan_tma_probe": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_float)]),
    "gscan_abi_version": (ctypes.c_int, []),
}

_lib = None


def lib():
    """Loads libgscan.so (built by __graft_entry__.build() / make -C grab_b200/csrc).  No fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GscanError("libgscan.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                             "the scan has no CPU fallback")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class Pattern:
    """FileGrep::prepare (reference grab.cc:101-123): compile + minimum length."""

    def __init__(self, pattern, literal=False, strict_ref=False):
        if isinstance(pattern, str):
            pattern = pattern.encode("latin-1")
        h = ctypes.c_void_p()
        flags = (LITERAL if literal else 0) | (STRICT_REF if strict_ref else 0)
        if lib().gscan_compile(pattern, len(pattern), flags, ctypes.byref(h)) != 0:
            raise GscanError(lib().gscan_last_error().decode())
        self._h = h

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.gscan_free_pattern(self._h)
            self._h = None

    @property
    def minlen(self):
        return lib().gscan_minlen(self._h)

    @property
    def info(self):
        i = PatternInfo()
        lib().gscan_pattern_get_info(self._h, ctypes.byref(i))
        return {n: getattr(i, n) for n, _ in i._fields_}


class Batch:
    def __init__(self, ctx, handle, keepalive):
        self.ctx, self._h, self._keep = ctx, handle, keepalive

    def free(self):
        if self._h:
            lib().gscan_batch_free(self.ctx._h, self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """One per host thread and GPU, like a FileGrep object (reference main.cc:195-199)."""

    def __init__(self, device=0):
        self._h = lib().gscan_open(device)
        if not self._h:
            raise GscanError(lib().gscan_last_error().decode())
        self.device = device

    def close(self):
        if self._h:
            lib().gscan_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def why(self):
        return lib().gscan_why(self._h).decode()

    def _check(self, rc):
        if rc != 0:
            raise GscanError(self.why())

    # ---- unit tables -------------------------------------------------------------------
    @staticmethod
    def units_from_buffers(bufs, file_ids=None, base_offs=None):
        """bufs: list of bytes / numpy uint8 arrays (host).  Returns (unit array, keepalive)."""
        arr = np.zeros(len(bufs), dtype=UNIT_DTYPE)
        keep = []
        for i, b in enumerate(bufs):
            a = np.frombuffer(b, dtype=np.uint8) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b, dtype=np.uint8)
            keep.append(a)
            arr[i]["ptr"] = a.ctypes.data if a.size else 0
            arr[i]["len"] = a.size
            arr[i]["base_off"] = base_offs[i] if base_offs is not None else 0
            arr[i]["file_id"] = file_ids[i] if file_ids is not None else i
        return arr, keep

    @staticmethod
    def fd_units(windows, file_ids=None):
        """windows: list of (descriptor, file offset, length): descriptor windows (GSCAN_UNIT_FD), read by the engine's
        staging threads with pread() -- the descriptors stay the caller's and must stay open until the scan returns."""
        arr = np.zeros(len(windows), dtype=UNIT_DTYPE)
        for i, (fd, off, n) in enumerate(windows):
            arr[i]["ptr"] = fd
            arr[i]["len"] = n
            arr[i]["base_off"] = off
            arr[i]["file_id"] = file_ids[i] if file_ids is not None else i
            arr[i]["flags"] = UNIT_FD
        return arr

    @staticmethod
    def device_units(dptr, n_files, file_len, stride=None, first_file_id=0):
        stride = file_len if stride is None else stride
        arr = np.zeros(n_files, dtype=UNIT_DTYPE)
        arr["ptr"] = dptr + np.arange(n_files, dtype=np.uint64) * np.uint64(stride)
        arr["len"] = file_len
        arr["file_id"] = first_file_id + np.arange(n_files, dtype=np.uint32)
        arr["flags"] = UNIT_DEVICE
        return arr

    def _take(self, out, n, copy=True):
        """The records of a scan as a numpy array.  copy=False: a view of the context's pinned result buffer, valid until
        the next scan on this context with copy=False (or close()) -- no per-record work on the host."""
        if not copy and getattr(self, "_lent", None):
            lib().gscan_free_matches(self._h, self._lent)
            self._lent = None
        if n.value == 0:
            return np.zeros(0, dtype=MATCH_DTYPE)
        buf = (ctypes.c_char * (n.value * MATCH_DTYPE.itemsize)).from_address(out.value)
        res = np.frombuffer(buf, dtype=MATCH_DTYPE)
        if not copy:
            self._lent = out
            return res
        res = res.copy()
        lib().gscan_free_matches(self._h, out)
        return res

    # ---- scanning ----------------------------------------------------------------------
    def scan_units(self, pattern, units, mode=MODE_ALL, copy=True):
        """gscan_scan_batch over a UNIT_DTYPE array."""
        units = np.ascontiguousarray(units, dtype=UNIT_DTYPE)
        out, n = ctypes.c_void_p(), ctypes.c_size_t()
        self._check(lib().gscan_scan_batch(self._h, pattern._h, units.ctypes.data, len(units), mode,
                                           ctypes.byref(out), ctypes.byref(n)))
        return self._take(out, n, copy)

    def scan_units_async(self, pattern, units, mode=MODE_ALL):
        """gscan_scan_batch_async: returns at once; `wait()` of the returned handle delivers the records.  The unit table and
        the buffers are kept alive by the handle."""
        units = np.ascontiguousarray(units, dtype=UNIT_DTYPE)
        self._check(lib().gscan_scan_batch_async(self._h, pattern._h, units.ctypes.data, len(units), mode))
        ctx = self

        class Job:
            def __init__(self):
                self.keep = (units, pattern)

            def wait(self):
                out, n = ctypes.c_void_p(), ctypes.c_size_t()
                ctx._check(lib().gscan_scan_wait(ctx._h, ctypes.byref(out), ctypes.byref(n)))
                self.keep = None
                return ctx._take(out, n)
        return Job()

    def scan(self, pattern, bufs, mode=MODE_ALL, file_ids=None, base_offs=None):
        units, keep = self.units_from_buffers(bufs, file_ids, base_offs)
        res = self.scan_units(pattern, units, mode)
        del keep
        return res

    def batch_create(self, units, keepalive=None):
        units = np.ascontiguousarray(units, dtype=UNIT_DTYPE)
        h = ctypes.c_void_p()
        self._check(lib().gscan_batch_create(self._h, units.ctypes.data, len(units), ctypes.byref(h)))
        return Batch(self, h, keepalive)

    def batch_scan(self, pattern, batch, mode=MODE_ALL, copy=True):
        out, n = ctypes.c_void_p(), ctypes.c_size_t()
        self._check(lib().gscan_batch_scan(self._h, pattern._h, batch._h, mode, ctypes.byref(out), ctypes.byref(n)))
        return self._take(out, n, copy)

    def last_device_matches(self):
        """(device pointer, count) of the last scan's records in HBM (valid until the next scan on this context)."""
        p, n = ctypes.c_void_p(), ctypes.c_size_t()
        self._check(lib().gscan_last_device_matches(self._h, ctypes.byref(p), ctypes.byref(n)))
        return (p.value or 0), n.value

    def stats(self):
        s = Stats()
        lib().gscan_last_stats(self._h, ctypes.byref(s))
        return s.as_dict()

    # ---- utilities ---------------------------------------------------------------------
    def device_alloc(self, nbytes):
        p = lib().gscan_device_alloc(self._h, nbytes)
        if not p:
            raise GscanError(self.why())
        return p

    def device_free(self, dptr):
        lib().gscan_device_free(self._h, dptr)

    def d2h(self, dptr, nbytes):
        out = np.empty(nbytes, dtype=np.uint8)
        self._check(lib().gscan_memcpy_d2h(self._h, out.ctypes.data, dptr, nbytes))
        return out

    def h2d(self, dptr, arr):
        arr = np.ascontiguousarray(arr, dtype=np.uint8)
        self._check(lib().gscan_memcpy_h2d(self._h, dptr, arr.ctypes.data, arr.size))

    def synth_corpus(self, dptr, seed, first_file_id, n_files, file_len, stride=None, needle=None, needle_every=0):
        stride = file_len if stride is None else stride
        self._check(lib().gscan_synth_corpus(self._h, dptr, seed, first_file_id, n_files, file_len, stride,
                                             needle, len(needle) if needle else 0, needle_every))

    def tma_probe(self, batch, geom=0):
        ms = ctypes.c_float()
        self._check(lib().gscan_tma_probe(self._h, batch._h, geom, ctypes.byref(ms)))
        return ms.value

    def read_probe(self, dptr, nbytes):
        ms, cs = ctypes.c_float(), ctypes.c_uint64()
        self._check(lib().gscan_read_probe(self._h, dptr, nbytes, ctypes.byref(ms), ctypes.byref(cs)))
        return ms.value, cs.value
