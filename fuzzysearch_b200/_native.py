"""ctypes binding of libfuzzb200.so (C-ABI declared in include/fuzzb200.h).

There is no Python or CPU fallback: if the shared library is missing or no CUDA device is usable
the calls raise (``NativeLibraryMissing`` / ``CudaError``).
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfuzzb200.so")

FZB_OK = 0
FZB_E_INVALID = -1
FZB_E_CUDA = -2
FZB_E_UNSUPPORTED = -3
FZB_E_NGRAM_ZERO = -4
FZB_MAX_PATTERN = 255
FZB_SEG_SHORT_BYTES = 4096    # segments up to this length are searched one warp each; longer ones one by one
FZB_SEG_MAX_COUNT = 1 << 23   # segments per fzb_search_segments call (the segment number's bits in a raw record)

RAW, FINAL = 0, 1
F_NO_FINAL, F_FORCE_DENSE, F_FORCE_LP, F_FORCE_NGRAMS, F_TINY_LIST, F_GLOBAL, F_FORCE_SAMPLED = 1, 2, 4, 8, 16, 32, 64

ROUTE_NAMES = {8: "segments", 7: "batch", 0: "exact", 1: "ngrams/sampled-filter", 2: "ngrams/dense-filter", 3: "lp",
               4: "hamming", 5: "generic-ngrams", 6: "generic-lp"}


class NativeLibraryMissing(ImportError):
    pass


class CudaError(RuntimeError):
    pass


class UnsupportedError(NotImplementedError):
    pass


class Stats(ctypes.Structure):
    _fields_ = [("gpu_ms", ctypes.c_double), ("filter_ms", ctypes.c_double),
                ("bytes_scanned", ctypes.c_uint64), ("n_candidates", ctypes.c_uint64),
                ("n_launches", ctypes.c_uint32), ("route", ctypes.c_uint32)]


# every symbol include/fuzzb200.h declares: name -> (restype, argtypes)
_vp, _u8p = ctypes.c_void_p, ctypes.c_void_p
_u32, _u64, _i32, _i64 = ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int, ctypes.c_int64
_vpp = ctypes.POINTER(ctypes.c_void_p)
SYMBOLS = {
    "fzb_version": (_i32, []),
    "fzb_device_count": (_i32, []),
    "fzb_last_error": (ctypes.c_char_p, []),
    "fzb_haystack_create": (_i32, [_u8p, _u64, _i32, _vpp]),
    "fzb_haystack_create_shard": (_i32, [_u8p, _u64, _u64, _u64, _u64, _u64, _i32, _vpp]),
    "fzb_haystack_adopt_device": (_i32, [_vp, _u64, _u64, _u64, _u64, _u64, _i32, _vpp]),
    "fzb_haystack_alloc": (_i32, [_u64, _u64, _u64, _u64, _u64, _i32, _vpp, _vpp]),
    "fzb_haystack_fill_synthetic": (_i32, [_vp, _u8p, _u32, _u64]),
    "fzb_synth_host": (None, [_u8p, _u64, _u64, _u8p, _u32, _u64]),
    "fzb_haystack_write": (_i32, [_vp, _u64, _u8p, _u64]),
    "fzb_haystack_read": (_i32, [_vp, _u64, _u8p, _u64]),
    "fzb_nccl_set_library": (None, [ctypes.c_char_p]),
    "fzb_nccl_unique_id": (_i32, [_vp]),
    "fzb_haystack_comm_init": (_i32, [_vp, _vp, _i32, _i32]),
    "fzb_comm_init_local": (_i32, [_vp, _i32]),
    "fzb_haystack_p2p_enabled": (_i32, [_vp]),
    "fzb_p2p_export": (_i32, [_vp, _i32, _i32, _vp]),
    "fzb_p2p_connect": (_i32, [_vp, _vp]),
    "fzb_p2p_disable": (None, [_vp]),
    "fzb_haystack_upload": (_i32, [_vp, _u8p, _u64]),
    "fzb_haystack_upload_symbols": (_i32, [_vp, _vp, _u64, _u32, _vp, _u32]),
    "fzb_host_alloc": (_vp, [_u64]),
    "fzb_host_free": (None, [_vp]),
    "fzb_timer_start": (_i32, [_vp]),
    "fzb_timer_stop": (_i32, [_vp, ctypes.POINTER(ctypes.c_double)]),
    "fzb_haystack_len": (_u64, [_vp]),
    "fzb_haystack_destroy": (None, [_vp]),
    "fzb_search_levenshtein": (_i32, [_vp, _u8p, _u32, _u32, _u32, _vpp]),
    "fzb_search_hamming": (_i32, [_vp, _u8p, _u32, _u32, _u32, _vpp]),
    "fzb_search_generic": (_i32, [_vp, _u8p, _u32, _u32, _u32, _u32, _u32, _u32, _vpp]),
    "fzb_search_exact": (_i32, [_vp, _u8p, _u32, _u32, _vpp]),
    "fzb_search_segments": (_i32, [_vp, _u8p, _u32, _vp, _u64, _u32, _u32, _u32, _u32, _u32, _vpp]),
    "fzb_result_segment_counts": (_i32, [_vp, _i32, _vp]),
    "fzb_search_exact_window": (_i32, [_vp, _u8p, _u32, _u64, _u64, _u32, _vpp]),
    "fzb_search_levenshtein_batch": (_i32, [_vp, _u8p, _vp, _vp, _u32, _u32, _vpp, ctypes.POINTER(Stats)]),
    "fzb_find_near_matches": (_i32, [_u8p, _u32, _u8p, _u64, _u32, _u32, _u32, _u32, _i32, _vpp]),
    "fzb_has_near_match": (_i32, [_vp, _u8p, _u32, _u32, _u32, _u32, _u32, ctypes.POINTER(ctypes.c_int)]),
    "fzb_release_workspace": (None, []),
    "fzb_result_count": (_u64, [_vp, _i32]),
    "fzb_result_copy": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "fzb_result_hulls": (_i32, [_vp, _vp, _vp]),
    "fzb_result_group_rows": (_i64, [_vp, _vp, _u64]),
    "fzb_merge_groups": (_i64, [_vp, _u64, _vp, _vp, _vp]),
    "fzb_consolidate_groups": (_i64, [_vp, _vp, _vp, _u64, _vp]),
    "fzb_result_stats": (_i32, [_vp, ctypes.POINTER(Stats)]),
    "fzb_result_destroy": (None, [_vp]),
    "fzb_consolidate": (_i64, [_vp, _vp, _vp, _u64, _vp, _vp, _vp]),
    "fzb_debug_counters": (_i32, [_vp, _vp]),
    "fzb_debug_expand": (_i32, [_u8p, _vp, _u8p, _vp, _vp, _vp, _u32, _i32, _vp]),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C fuzzysearch_b200/csrc`). fuzzysearch_b200 has no CPU fallback."
                % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            f = getattr(l, name)
            f.restype = res
            f.argtypes = args
        _lib = l
    return _lib


def device_count():
    return int(lib().fzb_device_count())


def last_error():
    return lib().fzb_last_error().decode("utf-8", "replace")


def check(rc):
    if rc == FZB_OK:
        return
    msg = last_error()
    if rc in (FZB_E_INVALID, FZB_E_NGRAM_ZERO):
        raise ValueError(msg)
    if rc == FZB_E_UNSUPPORTED:
        raise UnsupportedError(msg)
    raise CudaError(msg)


def as_u8(buf):
    """bytes-like -> contiguous numpy uint8 view (zero-copy where possible)."""
    if isinstance(buf, np.ndarray):
        if buf.dtype != np.uint8:
            raise TypeError("numpy sequences must have dtype uint8")
        return np.ascontiguousarray(buf).reshape(-1)
    try:
        mv = memoryview(buf)
    except TypeError:
        raise TypeError("only contiguous sequences of single-byte values are supported")
    if mv.itemsize != 1 or not mv.contiguous:
        raise TypeError("only contiguous sequences of single-byte values are supported")
    return np.frombuffer(mv, dtype=np.uint8)


def ptr(arr):
    return ctypes.c_void_p(arr.ctypes.data if arr.size else 0)


class Result(object):
    """Owns an fzb_result*; exposes the raw and final lists as numpy arrays."""

    def __init__(self, handle):
        self._h = handle

    def close(self):
        if self._h:
            lib().fzb_result_destroy(self._h)
            self._h = None

    __del__ = close

    def count(self, which=FINAL):
        return int(lib().fzb_result_count(self._h, which))

    def arrays(self, which=FINAL, anchors=False):
        n = self.count(which)
        start = np.empty(n, dtype=np.int64)
        end = np.empty(n, dtype=np.int64)
        dist = np.empty(n, dtype=np.int32)
        if anchors:
            ng = np.empty(n, dtype=np.int32)
            ix = np.empty(n, dtype=np.int64)
            check(lib().fzb_result_copy(self._h, which, ptr(start), ptr(end), ptr(dist), ptr(ng), ptr(ix)))
            return start, end, dist, ng, ix
        check(lib().fzb_result_copy(self._h, which, ptr(start), ptr(end), ptr(dist), None, None))
        return start, end, dist

    def group_rows(self, out=None):
        """FINAL list as int64 rows (start, end, dist, hull_start, hull_end): what a shard
        contributes to the multi-GPU merge (fzb_merge_groups).  With `out` (int64 [cap,5], C
        contiguous) the rows are written there and the TOTAL count is returned."""
        if out is not None:
            cnt = lib().fzb_result_group_rows(self._h, ptr(out), out.shape[0])
            if cnt < 0:
                check(int(cnt))
            return int(cnt)
        n = self.count(FINAL)
        rows = np.empty((max(n, 1), 5), dtype=np.int64)
        cnt = lib().fzb_result_group_rows(self._h, ptr(rows), n)
        if cnt < 0:
            check(int(cnt))
        return rows[:n]

    def segment_counts(self, which=FINAL):
        """fzb_search_segments results: the length of each segment's `which` list (uint64 array)."""
        n = int(self._nseg)
        out = np.empty(n, dtype=np.uint64)
        check(lib().fzb_result_segment_counts(self._h, which, ptr(out)))
        return out

    def triples(self, which=FINAL):
        s, e, d = self.arrays(which)
        return list(zip(s.tolist(), e.tolist(), d.tolist()))

    def stats(self):
        st = Stats()
        check(lib().fzb_result_stats(self._h, ctypes.byref(st)))
        return {"gpu_ms": st.gpu_ms, "filter_ms": st.filter_ms, "bytes_scanned": st.bytes_scanned,
                "n_candidates": st.n_candidates, "n_launches": st.n_launches,
                "route": ROUTE_NAMES.get(st.route, str(st.route))}


class Haystack(object):
    """Owns an fzb_haystack*: a device-resident sequence (or one shard of a global sequence)."""

    def __init__(self, handle, dev_ptr=None):
        self._h = handle
        self.dev_ptr = dev_ptr

    @classmethod
    def from_host(cls, data, device=0, buf_lo=0, global_len=None, own_lo=None, own_hi=None):
        a = as_u8(data)
        n = a.size
        if global_len is None:
            global_len, own_lo, own_hi = n, 0, n
        h = ctypes.c_void_p()
        check(lib().fzb_haystack_create_shard(ptr(a), n, buf_lo, global_len, own_lo, own_hi, device,
                                              ctypes.byref(h)))
        return cls(h)

    @classmethod
    def alloc(cls, buf_len, device=0, buf_lo=0, global_len=None, own_lo=None, own_hi=None):
        if global_len is None:
            global_len, own_lo, own_hi = buf_len, 0, buf_len
        h = ctypes.c_void_p()
        dp = ctypes.c_void_p()
        check(lib().fzb_haystack_alloc(buf_len, buf_lo, global_len, own_lo, own_hi, device,
                                       ctypes.byref(h), ctypes.byref(dp)))
        return cls(h, dp.value)

    @classmethod
    def adopt(cls, dev_ptr, buf_len, device=0, buf_lo=0, global_len=None, own_lo=None, own_hi=None):
        if global_len is None:
            global_len, own_lo, own_hi = buf_len, 0, buf_len
        h = ctypes.c_void_p()
        check(lib().fzb_haystack_adopt_device(ctypes.c_void_p(dev_ptr), buf_len, buf_lo, global_len,
                                              own_lo, own_hi, device, ctypes.byref(h)))
        return cls(h, dev_ptr)

    def close(self):
        if self._h:
            lib().fzb_haystack_destroy(self._h)
            self._h = None

    __del__ = close

    def __len__(self):
        return int(lib().fzb_haystack_len(self._h))

    def comm_init(self, unique_id, rank, world_size):
        """Collective: bind this shard handle to an NCCL communicator (FZB_F_GLOBAL searches)."""
        _prefer_bundled_nccl()
        buf = (ctypes.c_uint8 * 128).from_buffer_copy(bytes(unique_id))
        check(lib().fzb_haystack_comm_init(self._h, buf, rank, world_size))

    def p2p_export(self, rank, world_size):
        """-> this rank's 64-byte CUDA IPC handle (NCCL-free world, step 1)."""
        buf = (ctypes.c_uint8 * 64)()
        check(lib().fzb_p2p_export(self._h, rank, world_size, buf))
        return bytes(buf)

    def p2p_connect(self, handles):
        """handles: the rank-major concatenation of every rank's handle (step 2)."""
        buf = (ctypes.c_uint8 * len(handles)).from_buffer_copy(bytes(handles))
        check(lib().fzb_p2p_connect(self._h, buf))

    def p2p_disable(self):
        lib().fzb_p2p_disable(self._h)

    def p2p_enabled(self):
        return bool(lib().fzb_haystack_p2p_enabled(self._h))

    def upload(self, data):
        a = as_u8(data)
        check(lib().fzb_haystack_upload(self._h, ptr(a), a.size))

    def upload_symbols(self, units, alphabet):
        """units: numpy uint16 / uint32 code units; alphabet: the pattern's distinct symbols, ascending.
        The device reduces every unit to one byte: 1 + its rank in `alphabet`, 0 if absent."""
        units = np.ascontiguousarray(units)
        if units.dtype not in (np.uint16, np.uint32):
            raise TypeError("code units must be uint16 or uint32")
        alpha = np.ascontiguousarray(alphabet, dtype=np.uint32)
        check(lib().fzb_haystack_upload_symbols(self._h, ptr(units), units.size, units.dtype.itemsize, ptr(alpha),
                                                alpha.size))

    def debug_counters(self):
        out = np.zeros(32, dtype=np.uint32)
        check(lib().fzb_debug_counters(self._h, ptr(out)))
        return out.tolist()

    def timer_start(self):
        check(lib().fzb_timer_start(self._h))

    def timer_stop(self):
        ms = ctypes.c_double()
        check(lib().fzb_timer_stop(self._h, ctypes.byref(ms)))
        return ms.value

    def fill_synthetic(self, alphabet, seed):
        a = as_u8(alphabet)
        check(lib().fzb_haystack_fill_synthetic(self._h, ptr(a), a.size, seed))

    def write(self, offset, data):
        a = as_u8(data)
        check(lib().fzb_haystack_write(self._h, offset, ptr(a), a.size))

    def read(self, offset, n):
        out = np.empty(n, dtype=np.uint8)
        check(lib().fzb_haystack_read(self._h, offset, ptr(out), n))
        return out.tobytes()

    def _pat(self, pattern):
        p = as_u8(pattern)
        return p, ptr(p), p.size

    def search_levenshtein(self, pattern, k, flags=0):
        p, pp, m = self._pat(pattern)
        r = ctypes.c_void_p()
        check(lib().fzb_search_levenshtein(self._h, pp, m, k, flags, ctypes.byref(r)))
        return Result(r)

    def search_hamming(self, pattern, k, flags=0):
        p, pp, m = self._pat(pattern)
        r = ctypes.c_void_p()
        check(lib().fzb_search_hamming(self._h, pp, m, k, flags, ctypes.byref(r)))
        return Result(r)

    def search_generic(self, pattern, max_subs, max_ins, max_dels, max_l, flags=0):
        p, pp, m = self._pat(pattern)
        r = ctypes.c_void_p()
        check(lib().fzb_search_generic(self._h, pp, m, max_subs, max_ins, max_dels, max_l, flags,
                                       ctypes.byref(r)))
        return Result(r)

    def search_levenshtein_batch(self, patterns, ks, flags=0):
        """-> (list of Result, one per pattern; summed stats dict)."""
        pats = [as_u8(p) for p in patterns]
        blob = np.concatenate(pats) if pats else np.zeros(0, np.uint8)
        offsets = np.zeros(len(pats) + 1, dtype=np.uint32)
        offsets[1:] = np.cumsum([p.size for p in pats])
        ks = np.ascontiguousarray(ks, dtype=np.uint32)
        out = (ctypes.c_void_p * max(len(pats), 1))()
        st = Stats()
        check(lib().fzb_search_levenshtein_batch(self._h, ptr(blob), ptr(offsets), ptr(ks), len(pats), flags, out,
                                                 ctypes.byref(st)))
        results = [Result(ctypes.c_void_p(out[i])) for i in range(len(pats))]
        return results, {"gpu_ms": st.gpu_ms, "filter_ms": st.filter_ms, "bytes_scanned": st.bytes_scanned,
                         "n_candidates": st.n_candidates, "n_launches": st.n_launches, "route": "batch"}

    def search_segments(self, pattern, offsets, max_subs, max_ins, max_dels, max_l, flags=0):
        """One pattern over the segments [offsets[i], offsets[i+1]) of this sequence, each searched as a whole sequence
        (normalised limits, as for has_near_match).  -> Result with segment-major lists; .segment_counts(which)."""
        p, pp, m = self._pat(pattern)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        if offsets.ndim != 1 or offsets.size < 1:
            raise ValueError("offsets must hold count + 1 entries")
        r = ctypes.c_void_p()
        check(lib().fzb_search_segments(self._h, pp, m, ptr(offsets), offsets.size - 1, max_subs, max_ins, max_dels,
                                        max_l, flags, ctypes.byref(r)))
        res = Result(r)
        res._nseg = offsets.size - 1
        return res

    def has_near_match(self, pattern, max_subs, max_ins, max_dels, max_l):
        """True iff the search would return at least one match; stops at the first chunk that holds one."""
        p, pp, m = self._pat(pattern)
        found = ctypes.c_int(0)
        check(lib().fzb_has_near_match(self._h, pp, m, max_subs, max_ins, max_dels, max_l, ctypes.byref(found)))
        return bool(found.value)

    def search_exact(self, pattern, flags=0, start=None, end=None):
        """All occurrences; with start / end: those wholly inside [start, end) (only that window is scanned)."""
        p, pp, m = self._pat(pattern)
        r = ctypes.c_void_p()
        if start is None and end is None:
            check(lib().fzb_search_exact(self._h, pp, m, flags, ctypes.byref(r)))
        else:
            n = len(self)
            start = 0 if start is None else max(0, min(int(start), n))
            end = n if end is None else max(0, min(int(end), n))
            check(lib().fzb_search_exact_window(self._h, pp, m, start, end, flags, ctypes.byref(r)))
        return Result(r)


def comm_init_local(haystacks):
    """Bind Haystack objects (one process, one or several GPUs) into a world of shards: haystacks[r] = rank r."""
    arr = (ctypes.c_void_p * len(haystacks))(*[h._h for h in haystacks])
    check(lib().fzb_comm_init_local(arr, len(haystacks)))


class PinnedBuffer(object):
    """Page-locked host memory exposed as a numpy uint8 array (``.array``)."""

    def __init__(self, n):
        self._p = lib().fzb_host_alloc(n)
        if not self._p:
            raise CudaError(last_error())
        self.array = np.ctypeslib.as_array(ctypes.cast(self._p, ctypes.POINTER(ctypes.c_uint8)), shape=(n,))

    def close(self):
        if self._p:
            self.array = None
            lib().fzb_host_free(self._p)
            self._p = None

    __del__ = close


_nccl_path_set = False


def _prefer_bundled_nccl():
    """If the PyTorch wheel's NCCL is installed, make the library load THAT libnccl.so.2: the SONAME
    is shared process-wide, and torch (imported before or after) needs its own, newer build."""
    global _nccl_path_set
    if _nccl_path_set:
        return
    _nccl_path_set = True
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        if spec and spec.submodule_search_locations:
            path = os.path.join(list(spec.submodule_search_locations)[0], "lib", "libnccl.so.2")
            if os.path.exists(path):
                lib().fzb_nccl_set_library(path.encode())
    except Exception:  # noqa: BLE001 -- fall back to the default search path
        pass


def nccl_unique_id():
    _prefer_bundled_nccl()
    buf = (ctypes.c_uint8 * 128)()
    check(lib().fzb_nccl_unique_id(buf))
    return bytes(buf)


def synth_host(global_offset, n, alphabet, seed):
    a = as_u8(alphabet)
    out = np.empty(n, dtype=np.uint8)
    lib().fzb_synth_host(ptr(out), global_offset, n, ptr(a), a.size, seed)
    return out


def find_near_matches_host(pattern, haystack, max_subs, max_ins, max_dels, max_l, device=0):
    """One-shot C-ABI call with host buffers (upload + search + consolidate)."""
    p = as_u8(pattern)
    a = as_u8(haystack)
    r = ctypes.c_void_p()
    check(lib().fzb_find_near_matches(ptr(p), p.size, ptr(a), a.size, max_subs, max_ins, max_dels, max_l,
                                      device, ctypes.byref(r)))
    return Result(r)


def debug_expand(cases, device=0):
    """Test hook: cases = [(sub, seq, max_l, variant)], variant 0 auto / 1 short / 2 long ->
    int32 array [n, 8] (see fzb_debug_expand in include/fuzzb200.h)."""
    n = len(cases)
    # (one spare byte each: a batch made of empty sequences only must still hand the library a non-NULL pointer)
    subs = np.frombuffer(b"".join(bytes(c[0]) for c in cases) + b"\0", dtype=np.uint8)
    seqs = np.frombuffer(b"".join(bytes(c[1]) for c in cases) + b"\0", dtype=np.uint8)
    so = np.zeros(n + 1, dtype=np.uint32)
    qo = np.zeros(n + 1, dtype=np.uint32)
    so[1:] = np.cumsum([len(c[0]) for c in cases])
    qo[1:] = np.cumsum([len(c[1]) for c in cases])
    ks = np.ascontiguousarray([c[2] for c in cases], dtype=np.int32)
    vs = np.ascontiguousarray([c[3] for c in cases], dtype=np.int32)
    out = np.zeros((max(n, 1), 8), dtype=np.int32)
    check(lib().fzb_debug_expand(ptr(subs), ptr(so), ptr(seqs), ptr(qo), ptr(ks), ptr(vs), n, device, ptr(out)))
    return out[:n]


def consolidate_groups(start, end, dist):
    """-> int64 rows (start, end, dist, hull_start, hull_end), one per group of overlapping matches."""
    start = np.ascontiguousarray(start, dtype=np.int64)
    end = np.ascontiguousarray(end, dtype=np.int64)
    dist = np.ascontiguousarray(dist, dtype=np.int32)
    rows = np.empty((max(start.size, 1), 5), dtype=np.int64)
    cnt = lib().fzb_consolidate_groups(ptr(start), ptr(end), ptr(dist), start.size, ptr(rows))
    if cnt < 0:
        check(int(cnt))
    return rows[:cnt]


def merge_groups(rows, as_arrays=False):
    """fzb_merge_groups: rows[n,5] (start,end,dist,hull_start,hull_end) -> global final triples
    (list of tuples, or the three numpy arrays with as_arrays=True)."""
    rows = np.ascontiguousarray(rows, dtype=np.int64).reshape(-1, 5)
    n = rows.shape[0]
    os_, oe, od = np.empty(n, np.int64), np.empty(n, np.int64), np.empty(n, np.int32)
    cnt = lib().fzb_merge_groups(ptr(rows), n, ptr(os_), ptr(oe), ptr(od))
    if cnt < 0:
        check(int(cnt))
    if as_arrays:
        return os_[:cnt], oe[:cnt], od[:cnt]
    return list(zip(os_[:cnt].tolist(), oe[:cnt].tolist(), od[:cnt].tolist()))


def consolidate(start, end, dist):
    start = np.ascontiguousarray(start, dtype=np.int64)
    end = np.ascontiguousarray(end, dtype=np.int64)
    dist = np.ascontiguousarray(dist, dtype=np.int32)
    n = start.size
    os_, oe, od = np.empty(n, np.int64), np.empty(n, np.int64), np.empty(n, np.int32)
    cnt = lib().fzb_consolidate(ptr(start), ptr(end), ptr(dist), n, ptr(os_), ptr(oe), ptr(od))
    if cnt < 0:
        check(int(cnt))
    return os_[:cnt], oe[:cnt], od[:cnt]
