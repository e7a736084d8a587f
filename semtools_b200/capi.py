"""ctypes binding of include/semtools_b200.h -- one Python callable per C entry
point, same names, same argument meaning.  Raises StbError on any negative
status; never substitutes a CPU computation."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("STB_LIB_PATH") or os.path.join(_HERE, "lib", "libsemtools_b200.so")

STB_DIM = 256
STB_OK, STB_ERR_ARG, STB_ERR_CUDA, STB_ERR_NOMEM = 0, -1, -2, -3
STB_ERR_RANGE, STB_ERR_CAPACITY, STB_ERR_STATE = -4, -5, -6
STB_MODE_SEARCH_DOCUMENTS, STB_MODE_STORE_QUERY = 0, 1

# every symbol include/semtools_b200.h declares (tests check the .so exports all)
SYMBOLS = [
    "stb_version", "stb_last_error", "stb_device_count", "stb_ctx_create", "stb_ctx_destroy",
    "stb_ctx_sync", "stb_ctx_stream", "stb_table_load", "stb_table_destroy", "stb_corpus_create",
    "stb_corpus_destroy", "stb_corpus_append", "stb_corpus_append_dev", "stb_corpus_clear",
    "stb_corpus_rows", "stb_corpus_data_dev", "stb_corpus_read", "stb_embed", "stb_embed_dev",
    "stb_embed_status", "stb_search",
    "stb_search_topk_dev", "stb_corpus_prepare", "stb_corpus_tier_stats", "stb_corpus_prepare_batch", "stb_search_batch", "stb_search_batch_dev",
    "stb_xchg_create", "stb_xchg_destroy", "stb_xchg_local_handle",
    "stb_xchg_connect", "stb_xchg_connect_local", "stb_search_topk_xchg", "stb_search_xchg", "stb_search_many", "stb_xchg_create_batch", "stb_search_batch_xchg_dev", "stb_ivfpq_build",
    "stb_ivfpq_destroy", "stb_ivfpq_stats", "stb_ivfpq_search", "stb_ivfpq_search_dev", "stb_hits_merge_dev", "stb_hits_merge_batch_dev", "stb_hits_merge", "stb_fnv1a64", "stb_line_id", "stb_line_ids",
    "stb_ctx_counters", "stb_debug_ticket_check", "stb_debug_scan_front", "stb_debug_timestamps", "stb_debug_batch_gemm", "stb_debug_batch_params",
]


class StbHit(C.Structure):
    _fields_ = [("distance", C.c_double), ("row", C.c_uint64)]


HIT_DTYPE = np.dtype([("distance", np.float64), ("row", np.uint64)])


class StbError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"stb status {status}: {message}")
        self.status = status


_lib = None
vp = C.c_void_p
u64, u32, i32, f64 = C.c_uint64, C.c_uint32, C.c_int, C.c_double


def lib() -> C.CDLL:
    """Load libsemtools_b200.so; fails loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(scripts/build_lib.sh).  semtools_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    L.stb_version.restype = i32
    L.stb_last_error.restype = C.c_char_p
    L.stb_device_count.restype = i32
    L.stb_ctx_create.argtypes = [i32, vp, C.POINTER(vp)]
    L.stb_ctx_destroy.argtypes = [vp]
    L.stb_ctx_sync.argtypes = [vp]
    L.stb_ctx_stream.argtypes = [vp]
    L.stb_ctx_stream.restype = vp
    L.stb_table_load.argtypes = [vp, vp, u64, u32, vp, u64, vp, u64, i32, C.POINTER(vp)]
    L.stb_table_destroy.argtypes = [vp]
    L.stb_corpus_create.argtypes = [vp, u32, u64, u64, C.POINTER(vp)]
    L.stb_corpus_destroy.argtypes = [vp]
    L.stb_corpus_append.argtypes = [vp, vp, u64]
    L.stb_corpus_append_dev.argtypes = [vp, vp, u64]
    L.stb_corpus_clear.argtypes = [vp]
    L.stb_corpus_rows.argtypes = [vp, C.POINTER(u64)]
    L.stb_corpus_data_dev.argtypes = [vp, C.POINTER(vp)]
    L.stb_corpus_read.argtypes = [vp, u64, u64, vp]
    L.stb_embed.argtypes = [vp, vp, vp, vp, u64, vp, vp]
    L.stb_embed_dev.argtypes = [vp, vp, vp, vp, u64, vp]
    L.stb_embed_status.argtypes = [vp]
    L.stb_search.argtypes = [vp, vp, vp, u32, i32, f64, i32, vp, u32, vp, u64, C.POINTER(u64)]
    L.stb_search_topk_dev.argtypes = [vp, vp, vp, u32, vp, vp]
    L.stb_corpus_prepare_batch.argtypes = [vp]
    L.stb_corpus_prepare.argtypes = [vp, i32]
    L.stb_corpus_tier_stats.argtypes = [vp, vp, vp, vp]
    L.stb_search_batch.argtypes = [vp, vp, vp, u32, u32, vp, vp]
    L.stb_search_batch_dev.argtypes = [vp, vp, vp, u32, u32, vp, vp]
    L.stb_xchg_create.argtypes = [vp, u32, u32, u32, C.POINTER(vp)]
    L.stb_xchg_destroy.argtypes = [vp]
    L.stb_xchg_local_handle.argtypes = [vp, vp]
    L.stb_xchg_connect.argtypes = [vp, vp]
    L.stb_xchg_connect_local.argtypes = [vp, C.POINTER(vp)]
    L.stb_search_topk_xchg.argtypes = [vp, vp, vp, u32, vp, vp, vp]
    L.stb_search_xchg.argtypes = [vp, vp, vp, u32, vp, vp, C.POINTER(u32), C.POINTER(i32)]
    L.stb_search_many.argtypes = [vp, vp, vp, u32, u32, vp, vp, vp, vp]
    L.stb_xchg_create_batch.argtypes = [vp, u32, u32, u32, u32, C.POINTER(vp)]
    L.stb_search_batch_xchg_dev.argtypes = [vp, vp, vp, u32, u32, vp, vp, vp]
    L.stb_ivfpq_build.argtypes = [vp, vp, u32, u32, u32, C.POINTER(vp)]
    L.stb_ivfpq_destroy.argtypes = [vp]
    L.stb_ivfpq_stats.argtypes = [vp, C.POINTER(u64), C.POINTER(u32), C.POINTER(u32), C.POINTER(u64)]
    L.stb_ivfpq_search.argtypes = [vp, vp, u32, u32, u32, vp, C.POINTER(u32), C.POINTER(u64)]
    L.stb_ivfpq_search_dev.argtypes = [vp, vp, u32, u32, u32, vp, vp]
    L.stb_hits_merge_dev.argtypes = [vp, vp, u32, u32, u32, vp]
    L.stb_hits_merge_batch_dev.argtypes = [vp, vp, u32, u32, u32, u32, vp]
    L.stb_hits_merge.argtypes = [vp, vp, u32, u32, u32, vp, C.POINTER(u32)]
    L.stb_fnv1a64.argtypes = [C.c_char_p, u64]
    L.stb_fnv1a64.restype = u64
    L.stb_line_id.argtypes = [C.c_char_p, u64, C.c_int32]
    L.stb_line_ids.argtypes = [vp, vp, u32, vp, u64, vp]
    L.stb_line_id.restype = u64
    L.stb_ctx_counters.argtypes = [vp, C.POINTER(u64), C.POINTER(u64)]
    L.stb_debug_timestamps.argtypes = [vp, i32, vp]
    L.stb_debug_ticket_check.argtypes = [vp, C.POINTER(u64), C.POINTER(u64)]
    L.stb_debug_scan_front.argtypes = [vp, i32, C.POINTER(u64)]
    L.stb_debug_batch_gemm.argtypes = [vp, vp, u32, vp, u64, vp, vp]
    L.stb_debug_batch_params.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_double)]
    for name in SYMBOLS:
        fn = getattr(L, name)
        if fn.restype is C.c_int and name not in ("stb_version", "stb_device_count"):
            fn.restype = i32
    _lib = L
    return L


def _check(rc: int, allow_capacity: bool = False) -> int:
    if rc < 0 and not (allow_capacity and rc == STB_ERR_CAPACITY):
        raise StbError(rc, lib().stb_last_error().decode("utf-8", "replace"))
    return rc


def _np_ptr(a):
    return None if a is None else a.ctypes.data_as(vp)


def device_count() -> int:
    return int(lib().stb_device_count())


def batch_params():
    """(shadow_is_f16, eps) of this build's K2 path (stb_debug_batch_params; host-only)."""
    f16, eps = C.c_int(0), C.c_double(0.0)
    _check(lib().stb_debug_batch_params(C.byref(f16), C.byref(eps)))
    return bool(f16.value), float(eps.value)


def fnv1a64(data: bytes) -> int:
    """fnv1a_hash / DocMeta::id (reference src/workspace/store.rs:651-661, :75-80)."""
    return int(lib().stb_fnv1a64(data, len(data)))


def line_id(path: str, line_number: int) -> int:
    """LineEmbedding::id (reference src/workspace/store.rs:82-89)."""
    b = path.encode("utf-8")
    return int(lib().stb_line_id(b, len(b), line_number))


def line_ids(paths, rows) -> np.ndarray:
    """stb_line_ids: LineEmbedding ids of all rows ((path index, line_number) int32 pairs) in one
    native call (a store with millions of rows used to make one ctypes call per row)."""
    rows = np.ascontiguousarray(rows, dtype=np.int32).reshape(-1, 2)
    enc = [p.encode("utf-8") for p in paths]
    offs = np.zeros(len(enc) + 1, dtype=np.uint64)
    if enc:
        offs[1:] = np.cumsum([len(b) for b in enc])
    blob = np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8)
    out = np.zeros(len(rows), dtype=np.uint64)
    _check(lib().stb_line_ids(_np_ptr(blob), _np_ptr(offs), len(enc), _np_ptr(rows), len(rows), _np_ptr(out)))
    return out


class Context:
    """stb_ctx: one CUDA device + stream.  `stream` is an optional raw cudaStream_t."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self._h = vp()
        _check(lib().stb_ctx_create(device, vp(stream) if stream else None, C.byref(self._h)))
        self.device = device

    def close(self):
        if getattr(self, "_h", None) is not None and self._h and _lib is not None:
            _lib.stb_ctx_destroy(self._h)
            self._h = None

    __del__ = close

    def sync(self):
        _check(lib().stb_ctx_sync(self._h))

    @property
    def stream(self) -> int:
        return int(lib().stb_ctx_stream(self._h) or 0)

    def counters(self):
        a, b = u64(0), u64(0)
        _check(lib().stb_ctx_counters(self._h, C.byref(a), C.byref(b)))
        return {"kernel_launches": int(a.value), "fallback_searches": int(b.value)}

    def ticket_check(self):
        """stb_debug_ticket_check: (device counter, host-booked value); raises StbError on a mismatch."""
        a, b = u64(0), u64(0)
        _check(lib().stb_debug_ticket_check(self._h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def scan_front(self, value: int | None = None) -> int:
        """stb_debug_scan_front: sets K1's scan front to `value` (a virtual row) if given; returns it."""
        v = u64(0 if value is None else value)
        _check(lib().stb_debug_scan_front(self._h, 0 if value is None else 1, C.byref(v)))
        return int(v.value)

    # -- K4 ------------------------------------------------------------------
    def hits_merge(self, lists: np.ndarray, top_k: int) -> np.ndarray:
        """lists: (n_lists, per_list) array of HIT_DTYPE; returns the merged top_k."""
        lists = np.ascontiguousarray(lists, dtype=HIT_DTYPE)
        n_lists, per_list = lists.shape
        out = np.zeros(max(top_k, 1), dtype=HIT_DTYPE)
        n = u32(0)
        _check(lib().stb_hits_merge(self._h, _np_ptr(lists), n_lists, per_list, top_k, _np_ptr(out),
                                    C.byref(n)))
        return out[: n.value]

    def hits_merge_batch_dev(self, lists_dev: int, n_lists: int, nq: int, per_list: int, top_k: int, out_dev: int):
        """lists_dev [n_lists][nq][per_list] -> out_dev [nq][top_k] (sharded K2)."""
        _check(lib().stb_hits_merge_batch_dev(self._h, vp(lists_dev), n_lists, nq, per_list, top_k, vp(out_dev)))

    def hits_merge_dev(self, lists_dev: int, n_lists: int, per_list: int, top_k: int, out_dev: int):
        _check(lib().stb_hits_merge_dev(self._h, vp(lists_dev), n_lists, per_list, top_k, vp(out_dev)))


class Table:
    """stb_table: the StaticModel tensors resident in HBM."""

    def __init__(self, ctx: Context, E, weights=None, mapping=None, normalize=True):
        E = np.ascontiguousarray(E, dtype=np.float32)
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float32)
        m = None if mapping is None else np.ascontiguousarray(mapping, dtype=np.uint32)
        self.ctx = ctx
        self._h = vp()
        _check(lib().stb_table_load(ctx._h, _np_ptr(E), E.shape[0], E.shape[1], _np_ptr(w),
                                    0 if w is None else w.size, _np_ptr(m), 0 if m is None else m.size,
                                    int(normalize), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h and _lib is not None:
            _lib.stb_table_destroy(self._h)
            self._h = None

    __del__ = close


class Corpus:
    """stb_corpus: contiguous N x 256 f32 line-vector matrix in HBM."""

    def __init__(self, ctx: Context, capacity_rows: int = 1024, row_base: int = 0):
        self.ctx = ctx
        self.row_base = row_base
        self._h = vp()
        _check(lib().stb_corpus_create(ctx._h, STB_DIM, capacity_rows, row_base, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h and _lib is not None:
            _lib.stb_corpus_destroy(self._h)
            self._h = None

    __del__ = close

    def append(self, rows: np.ndarray):
        rows = np.ascontiguousarray(rows, dtype=np.float32)
        if rows.size == 0:
            return
        if rows.ndim != 2 or rows.shape[1] != STB_DIM:
            raise StbError(STB_ERR_ARG, f"rows must be (n,{STB_DIM}) f32")
        _check(lib().stb_corpus_append(self._h, _np_ptr(rows), rows.shape[0]))

    def append_dev(self, rows_dev: int, n: int):
        _check(lib().stb_corpus_append_dev(self._h, vp(rows_dev), n))

    def clear(self):
        _check(lib().stb_corpus_clear(self._h))

    def __len__(self) -> int:
        n = u64(0)
        _check(lib().stb_corpus_rows(self._h, C.byref(n)))
        return int(n.value)

    @property
    def data_dev(self) -> int:
        p = vp()
        _check(lib().stb_corpus_data_dev(self._h, C.byref(p)))
        return int(p.value or 0)

    def read(self, first: int = 0, n: int | None = None) -> np.ndarray:
        n = len(self) - first if n is None else n
        out = np.empty((n, STB_DIM), dtype=np.float32)
        _check(lib().stb_corpus_read(self._h, first, n, _np_ptr(out)))
        return out

    # -- K1 + K4 -------------------------------------------------------------
    def search(self, q, top_k: int = 3, max_distance: float | None = None,
               mode: int = STB_MODE_SEARCH_DOCUMENTS, row_ranges=None, cap: int | None = None):
        """stb_search.  Returns a HIT_DTYPE array ordered by (distance,row)."""
        q = np.ascontiguousarray(q, dtype=np.float32)
        if q.size != STB_DIM:
            raise StbError(STB_ERR_ARG, f"query must have {STB_DIM} floats")
        rr, n_rr = None, 0
        if row_ranges is not None:
            rr = np.ascontiguousarray(row_ranges, dtype=np.uint64).reshape(-1, 2)
            n_rr = rr.shape[0]
            if n_rr == 0:
                rr = np.zeros((1, 2), dtype=np.uint64)   # non-null pointer, zero ranges
        if cap is None:
            cap = max(top_k, 1) if (max_distance is None or mode == STB_MODE_STORE_QUERY) else max(top_k, 4096)
        while True:
            out = np.zeros(max(cap, 1), dtype=HIT_DTYPE)
            n = u64(0)
            rc = _check(lib().stb_search(self.ctx._h, self._h, _np_ptr(q), top_k,
                                         int(max_distance is not None), float(max_distance or 0.0), mode,
                                         _np_ptr(rr), n_rr, _np_ptr(out), cap, C.byref(n)), allow_capacity=True)
            if rc == STB_ERR_CAPACITY:
                cap = int(n.value)
                continue
            return out[: int(n.value)]

    def search_many(self, queries, top_k: int = 10, xchg=None):
        """stb_search_many: nq independent single queries, one synchronisation.  Returns a list of
        HIT_DTYPE arrays (x is None) or (list, complete flags) for the sharded form."""
        queries = np.ascontiguousarray(queries, dtype=np.float32)
        if queries.ndim != 2 or queries.shape[1] != STB_DIM:
            raise StbError(STB_ERR_ARG, f"queries must be (nq,{STB_DIM}) f32")
        nq = queries.shape[0]
        out = np.zeros((nq, max(top_k, 1)), dtype=HIT_DTYPE)
        cnt = np.zeros(max(nq, 1), dtype=np.uint32)
        ok = np.ones(max(nq, 1), dtype=np.uint8)
        _check(lib().stb_search_many(self.ctx._h, self._h, _np_ptr(queries), nq, top_k, xchg._h if xchg is not None else None,
                                     _np_ptr(out), _np_ptr(cnt), _np_ptr(ok)))
        res = [out[i, : cnt[i]] for i in range(nq)]
        return res if xchg is None else (res, ok[:nq].astype(bool))

    # -- K2 -----------------------------------------------------------------
    def prepare(self, what: int = 3):
        """stb_corpus_prepare: build the reduced-width candidate copies now
        (STB_PREPARE_Q8 = 1, STB_PREPARE_H16 = 2)."""
        _check(lib().stb_corpus_prepare(self._h, what))

    def tier_stats(self):
        """stb_corpus_tier_stats -> {"f32"|"h16"|"q8": {"tries", "proven", "built_rows"}}."""
        tries, proven = np.zeros(3, np.uint32), np.zeros(3, np.uint32)
        built = np.zeros(3, np.uint64)
        _check(lib().stb_corpus_tier_stats(self._h, _np_ptr(tries), _np_ptr(proven), _np_ptr(built)))
        return {name: {"tries": int(tries[i]), "proven": int(proven[i]), "built_rows": int(built[i])}
                for i, name in enumerate(("f32", "h16", "q8"))}

    def prepare_batch(self):
        """stb_corpus_prepare_batch: build the bf16 tensor-core shadow now."""
        _check(lib().stb_corpus_prepare_batch(self._h))

    def search_batch(self, queries, top_k: int = 10):
        """stb_search_batch.  Returns a list of HIT_DTYPE arrays, one per query."""
        queries = np.ascontiguousarray(queries, dtype=np.float32)
        if queries.ndim != 2 or queries.shape[1] != STB_DIM:
            raise StbError(STB_ERR_ARG, f"queries must be (nq,{STB_DIM}) f32")
        nq = queries.shape[0]
        out = np.zeros((nq, max(top_k, 1)), dtype=HIT_DTYPE)
        cnt = np.zeros(max(nq, 1), dtype=np.uint32)
        _check(lib().stb_search_batch(self.ctx._h, self._h, _np_ptr(queries), nq, top_k, _np_ptr(out), _np_ptr(cnt)))
        return [out[i, : cnt[i]] for i in range(nq)]

    def search_batch_dev(self, q_dev: int, nq: int, top_k: int, out_hits_dev: int, out_status_dev: int):
        """stb_search_batch_dev: asynchronous, everything stays in HBM."""
        _check(lib().stb_search_batch_dev(self.ctx._h, self._h, vp(q_dev), nq, top_k, vp(out_hits_dev),
                                          vp(out_status_dev)))

    def search_topk_dev(self, q_dev: int, top_k: int, out_hits_dev: int, out_status_dev: int):
        """stb_search_topk_dev: asynchronous, everything stays in HBM."""
        _check(lib().stb_search_topk_dev(self.ctx._h, self._h, vp(q_dev), top_k, vp(out_hits_dev),
                                         vp(out_status_dev)))


class IvfPq:
    """stb_ivfpq: approximate IVF-PQ index over a corpus (K5; self-specified, see header)."""

    def __init__(self, corpus: "Corpus", nlist: int = 4096, train_rows: int = 262144, iters: int = 8):
        self.corpus = corpus
        self._h = vp()
        _check(lib().stb_ivfpq_build(corpus.ctx._h, corpus._h, nlist, train_rows, iters, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h and _lib is not None:
            _lib.stb_ivfpq_destroy(self._h)
            self._h = None

    __del__ = close

    def stats(self):
        rows, nbytes, nlist, mx = u64(0), u64(0), u32(0), u32(0)
        _check(lib().stb_ivfpq_stats(self._h, C.byref(rows), C.byref(nlist), C.byref(mx), C.byref(nbytes)))
        return {"rows": int(rows.value), "nlist": int(nlist.value), "max_list": int(mx.value),
                "index_bytes": int(nbytes.value)}

    def search(self, q, nprobe: int = 64, top_k: int = 10, rerank: int = 256):
        q = np.ascontiguousarray(q, dtype=np.float32)
        out = np.zeros(max(top_k, 1), dtype=HIT_DTYPE)
        n, scanned = u32(0), u64(0)
        _check(lib().stb_ivfpq_search(self._h, _np_ptr(q), nprobe, top_k, rerank, _np_ptr(out), C.byref(n),
                                      C.byref(scanned)))
        return out[: n.value], int(scanned.value)


    def search_dev(self, q_dev: int, nprobe: int, top_k: int, rerank: int, out_hits_dev: int, out_status_dev: int):
        """stb_ivfpq_search_dev: asynchronous, everything stays in HBM."""
        _check(lib().stb_ivfpq_search_dev(self._h, vp(q_dev), nprobe, top_k, rerank, vp(out_hits_dev), vp(out_status_dev)))


class Exchange:
    """stb_xchg: peer-memory exchange buffers for the fused multi-GPU search."""
    HANDLE_BYTES = 64

    def __init__(self, ctx: Context, world: int, rank: int, max_k: int, max_nq: int = 0):
        """max_nq > 0 also allocates the batch area for the sharded K2 exchange (stb_xchg_create_batch)."""
        self.ctx, self.world, self.rank, self.max_k, self.max_nq = ctx, world, rank, max_k, max_nq
        self._h = vp()
        if max_nq:
            _check(lib().stb_xchg_create_batch(ctx._h, world, rank, max_k, max_nq, C.byref(self._h)))
        else:
            _check(lib().stb_xchg_create(ctx._h, world, rank, max_k, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h and _lib is not None:
            _lib.stb_xchg_destroy(self._h)
            self._h = None

    __del__ = close

    def local_handle(self) -> bytes:
        buf = (C.c_uint8 * self.HANDLE_BYTES)()
        _check(lib().stb_xchg_local_handle(self._h, buf))
        return bytes(buf)

    def connect(self, handles: list):
        """handles[r] = rank r's 64-byte IPC handle (other processes)."""
        blob = b"".join(handles)
        assert len(blob) == self.world * self.HANDLE_BYTES
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        _check(lib().stb_xchg_connect(self._h, buf))

    def connect_local(self, peers: list):
        """peers[r] = the Exchange of rank r living in this process."""
        arr = (vp * self.world)(*[p._h for p in peers])
        _check(lib().stb_xchg_connect_local(self._h, arr))

    def search(self, corpus: "Corpus", q, top_k: int):
        """stb_search_xchg: host query in, merged global hits out; returns (hits, complete)."""
        q = np.ascontiguousarray(q, dtype=np.float32)
        out = np.zeros(max(top_k, 1), dtype=HIT_DTYPE)
        n, ok = u32(0), i32(0)
        _check(lib().stb_search_xchg(self.ctx._h, corpus._h, _np_ptr(q), top_k, self._h, _np_ptr(out), C.byref(n),
                                     C.byref(ok)))
        return out[: n.value], bool(ok.value)

    def search_batch_dev(self, corpus: "Corpus", q_dev: int, nq: int, top_k: int, out_hits_dev: int, out_status_dev: int):
        """stb_search_batch_xchg_dev: K2 on the local shard + fused NVLink exchange + per-query merge."""
        _check(lib().stb_search_batch_xchg_dev(self.ctx._h, corpus._h, vp(q_dev), nq, top_k, self._h, vp(out_hits_dev),
                                               vp(out_status_dev)))

    def search_topk(self, corpus: "Corpus", q_dev: int, top_k: int, out_hits_dev: int, out_status_dev: int):
        """stb_search_topk_xchg: one kernel = scan + NVLink exchange + global merge."""
        _check(lib().stb_search_topk_xchg(self.ctx._h, corpus._h, vp(q_dev), top_k, self._h, vp(out_hits_dev),
                                          vp(out_status_dev)))


def embed_dev(ctx: Context, table: Table, offsets_dev: int, ids_dev: int, n_lines: int, out_dev: int):
    """stb_embed_dev: asynchronous, CSR and output already in HBM."""
    _check(lib().stb_embed_dev(ctx._h, table._h, vp(offsets_dev), vp(ids_dev), n_lines, vp(out_dev)))


def embed_status(ctx: Context):
    """stb_embed_status: sync + raise StbError(STB_ERR_RANGE) if a token was out of range."""
    _check(lib().stb_embed_status(ctx._h))


def embed(ctx: Context, table: Table, offsets, ids, out: bool = True, append_to: Corpus | None = None):
    """stb_embed (K3).  offsets: (n_lines+1,) u64 CSR; ids: u32 token ids."""
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    ids = np.ascontiguousarray(ids, dtype=np.uint32)
    n_lines = offsets.size - 1
    res = np.empty((n_lines, STB_DIM), dtype=np.float32) if out else None
    if ids.size == 0:
        ids = np.zeros(1, dtype=np.uint32)
    _check(lib().stb_embed(ctx._h, table._h, _np_ptr(offsets), _np_ptr(ids), n_lines, _np_ptr(res),
                           append_to._h if append_to is not None else None))
    return res
