"""ctypes view of libmmq_host.so: the product's .hits loader and hit-class
builder (mmseq_b200/csrc/hits_loader.cpp), replacing src/hitsio.cpp:250-447 and
src/mmseq.cpp:395-441 of the reference."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmmq_host.so")

LAYOUT_COLLAPSED = 0
LAYOUT_PER_FRAGMENT = 1
LAYOUT_PER_FRAGMENT_SORTED = 2
LAYOUT_PER_FRAGMENT_BY_LENGTH = 3
LAYOUT_IDENTITY_COLUMNS = 16
LAYOUT_HEADER_ORDER_COLUMNS = 32

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not built: run `make hostlib`")
        L = C.CDLL(LIB_PATH)
        vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
        L.mmqh_load.restype = vp
        L.mmqh_load.argtypes = [C.c_char_p, i32, C.c_char_p, i32]
        L.mmqh_from_records.restype = vp
        L.mmqh_from_records.argtypes = [i64, vp, i64, vp, vp, vp, i32, C.c_char_p, i32]
        L.mmqh_write_trace_gz.restype = i32
        L.mmqh_write_trace_gz.argtypes = [C.c_char_p, C.c_char_p, i64, vp, vp, i32]
        L.mmqh_gz_huffman.restype = i64
        L.mmqh_gz_huffman.argtypes = [vp, i64, vp]
        L.mmqh_fmt_g6.restype = i64
        L.mmqh_fmt_g6.argtypes = [vp, i64, vp]
        L.mmqh_inflate_parallel.restype = i64
        L.mmqh_inflate_parallel.argtypes = [vp, i64, i32, vp, i64]
        L.mmqh_free.restype = None
        L.mmqh_free.argtypes = [vp]
        L.mmqh_dim.restype = i64
        L.mmqh_dim.argtypes = [vp, i32]
        for nm in ["row_ptr", "col", "k", "w", "set_ptr", "set_col", "set_k", "col2hdr", "hdr2col", "doublehits", "efflen", "truelen", "gene_of",
                   "gene_ptr", "gene_members", "ident_ptr", "ident_members"]:
            f = getattr(L, "mmqh_" + nm)
            f.restype = vp
            f.argtypes = [vp]
        L.mmqh_name.restype = C.c_char_p
        L.mmqh_name.argtypes = [vp, i64]
        L.mmqh_gene_name.restype = C.c_char_p
        L.mmqh_gene_name.argtypes = [vp, i64]
        L.mmqh_scaled_len.restype = i32
        L.mmqh_scaled_len.argtypes = [vp, vp]
        _lib = L
    return _lib


def _arr(ptr, n, dtype):
    if not ptr or n == 0:
        return None if not ptr else np.zeros(0, dtype)
    ct = {np.int64: C.c_int64, np.int32: C.c_int32, np.float32: C.c_float, np.float64: C.c_double}[dtype]
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), shape=(n,)).copy()


class Hits:
    """Header tables + hit-class CSR of one hits file (or of in-memory records)."""

    def __init__(self, handle, with_names=True):
        L = lib()
        d = lambda w: int(L.mmqh_dim(handle, w))
        self.T, self.G, self.I, self.N, self.n, self.m, self.nnz, self.n_classes, self.schema = [d(i) for i in range(9)]
        self.row_ptr = _arr(L.mmqh_row_ptr(handle), self.m + 1, np.int64)
        self.col = _arr(L.mmqh_col(handle), self.nnz, np.int32)
        self.k = _arr(L.mmqh_k(handle), self.m, np.int32)
        self.w = _arr(L.mmqh_w(handle), self.nnz, np.float32)
        # per-fragment layouts: the distinct sets behind the rows, as a LAYOUT_COLLAPSED load returns
        # them in row_ptr / col / k (None in the collapsed layout)
        self.set_ptr = _arr(L.mmqh_set_ptr(handle), self.n_classes + 1, np.int64)
        self.set_col = _arr(L.mmqh_set_col(handle), d(9), np.int32)
        self.set_k = _arr(L.mmqh_set_k(handle), self.n_classes, np.int32)
        # weighted per-fragment layouts: first record (0-based) whose weights are all zero, or -1
        self.first_zero_weight_record = d(10)
        self.col2hdr = _arr(L.mmqh_col2hdr(handle), self.n, np.int32)
        self.hdr2col = _arr(L.mmqh_hdr2col(handle), self.T, np.int32)
        self.doublehits = _arr(L.mmqh_doublehits(handle), self.n, np.int32)
        self.efflen = _arr(L.mmqh_efflen(handle), self.T, np.float64)
        self.truelen = _arr(L.mmqh_truelen(handle), self.T, np.int32) if with_names else None
        self.len = np.zeros(self.n)
        if L.mmqh_scaled_len(handle, self.len.ctypes.data_as(C.c_void_p)):
            raise RuntimeError("Error: transcript has a length of zero.")
        if with_names:
            self.names = [L.mmqh_name(handle, t).decode() for t in range(self.T)]
            self.gene_names = [L.mmqh_gene_name(handle, g).decode() for g in range(self.G)]
            self.gene_of = _arr(L.mmqh_gene_of(handle), self.T, np.int32)
            self.gene_ptr = _arr(L.mmqh_gene_ptr(handle), self.G + 1, np.int64)
            self.gene_members = _arr(L.mmqh_gene_members(handle), int(self.gene_ptr[-1]), np.int32)
            self.ident_ptr = _arr(L.mmqh_ident_ptr(handle), self.I + 1, np.int64)
            self.ident_members = _arr(L.mmqh_ident_members(handle), int(self.ident_ptr[-1]), np.int32)
        L.mmqh_free(handle)


def write_trace_gz(path, ids, trace, keep=None):
    """trace_writer.h (the host program's *.trace_gibbs.gz writer): trace[feature, slot]."""
    tr = np.ascontiguousarray(trace, np.float64)
    kp = None if keep is None else np.ascontiguousarray(keep, np.uint8)
    rc = lib().mmqh_write_trace_gz(os.fsencode(path), "\n".join(ids).encode(), len(ids), None if kp is None else kp.ctypes.data_as(C.c_void_p),
                                   tr.ctypes.data_as(C.c_void_p), tr.shape[1])
    if rc:
        raise RuntimeError(f"cannot write {path}")


def gz_huffman(data):
    """huff_gz.h (the trace files' compressor): one gzip member holding `data`."""
    buf = np.frombuffer(bytes(data), np.uint8) if len(data) else np.zeros(0, np.uint8)
    out = np.empty(len(buf) + 1024, np.uint8)
    n = lib().mmqh_gz_huffman(buf.ctypes.data_as(C.c_void_p) if len(buf) else None, len(buf), out.ctypes.data_as(C.c_void_p))
    return out[:n].tobytes()


def fmt_g6(values):
    """fmt_g6.h (the host program's "%g" for trace files) on an array; list of strings."""
    v = np.ascontiguousarray(values, np.float64)
    out = np.empty(40 * len(v) + 8, np.uint8)
    n = lib().mmqh_fmt_g6(v.ctypes.data_as(C.c_void_p), len(v), out.ctypes.data_as(C.c_void_p))
    return out[:n].tobytes().decode().split()


def inflate_parallel(data, threads, cap):
    """inflate_par.h (the loader's multi-threaded inflate) on a zlib stream; None when it refuses the stream."""
    buf = np.frombuffer(data, np.uint8)
    out = np.empty(cap, np.uint8)
    n = lib().mmqh_inflate_parallel(buf.ctypes.data_as(C.c_void_p), len(buf), threads, out.ctypes.data_as(C.c_void_p), cap)
    if n == -1:
        return None
    assert n >= 0, "output buffer too small"
    return out[:n].tobytes()


def load_hits(path, layout=LAYOUT_COLLAPSED):
    err = C.create_string_buffer(512)
    h = lib().mmqh_load(os.fsencode(path), layout, err, 512)
    if not h:
        raise RuntimeError(err.value.decode())
    return Hits(h)


def from_records(T, efflen, frag_ptr, frag_tid, frag_w=None, layout=LAYOUT_COLLAPSED):
    efflen = np.ascontiguousarray(efflen, np.float64)
    frag_ptr = np.ascontiguousarray(frag_ptr, np.int64)
    frag_tid = np.ascontiguousarray(frag_tid, np.int32)
    fw = None if frag_w is None else np.ascontiguousarray(frag_w, np.float32)
    err = C.create_string_buffer(512)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    h = lib().mmqh_from_records(T, p(efflen), len(frag_ptr) - 1, p(frag_ptr), p(frag_tid), p(fw), layout, err, 512)
    if not h:
        raise RuntimeError(err.value.decode())
    return Hits(h, with_names=False)


def sort_classes_by_cost(h):
    """A device order of collapsed classes other than the loader's: by kind of draw (singleton, k == 1,
    categorical draws up to MMQ_CAT_K = 8192, binomial chain), then size, then count — what suits the
    general kernel (the class plan of mmq_create orders a shard itself).  Returns (row_ptr, col, k,
    class_id) where class_id[i] is the canonical (first-appearance) index to hand to
    mmq_problem.class_id; tests and bench.py use it to exercise explicit class ids."""
    d = np.diff(h.row_ptr)
    kind = np.where(d == 1, 0, np.where(h.k == 1, 1, np.where(h.k <= 8192, 2, 3)))
    order = np.lexsort((h.k, d, kind))
    dd = d[order]
    rp = np.concatenate([[0], np.cumsum(dd)]).astype(np.int64)
    starts = h.row_ptr[:-1][order]
    idx = np.repeat(starts - rp[:-1], dd) + np.arange(int(rp[-1]))
    return rp, h.col[idx], h.k[order], order.astype(np.int64)
