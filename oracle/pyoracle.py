"""ctypes bindings for the CPU checker (oracle/libvs_oracle.so) and, when present, the
unmodified reference builds under oracle/_ref/ (oracle/Makefile).

TEST / BASELINE INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs; never by sqlite_vector_b200/.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")

# enums: /root/reference/src/distance-cpu.h:36-58
F32, F16, BF16, U8, I8 = 1, 2, 3, 4, 5
L2, L2SQ, COS, DOT, L1 = 1, 2, 3, 4, 5
Q_AUTO, Q_U8, Q_S8 = 0, 1, 2
TYPE_NAMES = {F32: "f32", F16: "f16", BF16: "bf16", U8: "u8", I8: "i8"}
METRIC_NAMES = {L2: "l2", L2SQ: "l2sq", COS: "cos", DOT: "dot", L1: "l1"}
ELEM_SIZE = {F32: 4, F16: 2, BF16: 2, U8: 1, I8: 1}
NP_STORAGE = {F32: np.float32, F16: np.uint16, BF16: np.uint16, U8: np.uint8, I8: np.int8}

_vp, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t


def build(ref: bool = True) -> None:
    """Compile the checker (and the reference, when /root/reference exists) via oracle/Makefile."""
    target = ["all"] if ref else ["oracle"]
    subprocess.run(["make", "-C", HERE, "-s"] + target, check=True)


def _ptr(a):
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


class Oracle:
    """The restatement in oracle/vs_oracle.c."""

    def __init__(self, path: str | None = None):
        path = path or os.path.join(HERE, "libvs_oracle.so")
        if not os.path.exists(path):
            build(ref=False)
        self.lib = L = C.CDLL(path)
        L.vso_distance.restype = _f
        L.vso_distance.argtypes = [_i, _i, _vp, _vp, _i, _i]
        L.vso_clamp_tiny.restype = _f
        L.vso_clamp_tiny.argtypes = [_f]
        L.vso_quantize.restype = None
        L.vso_quantize.argtypes = [_i, _vp, _vp, _f, _f, _i, _i]
        L.vso_quant_params.restype = _i
        L.vso_quant_params.argtypes = [_i, _vp, _i64, _i, _i, _vp, _vp, _vp]
        L.vso_scan_topk.restype = _i
        L.vso_scan_topk.argtypes = [_i, _i, _vp, _vp, _i64, _i, _sz, _sz, _vp, _i, _i, _i, _vp, _vp, _vp]
        L.vso_topk_from_distances.restype = _i
        L.vso_topk_from_distances.argtypes = [_vp, _vp, _i64, _i, _i, _vp, _vp]
        L.vso_distances_all.restype = None
        L.vso_distances_all.argtypes = [_i, _i, _vp, _vp, _i64, _i, _sz, _sz, _i, _vp]
        L.vso_build_quant_buffer.restype = None
        L.vso_build_quant_buffer.argtypes = [_i, _vp, _vp, _i64, _i, _f, _f, _i, _vp]
        L.vso_f32_to_f16.restype = C.c_uint16
        L.vso_f32_to_f16.argtypes = [_f]
        L.vso_f32_to_bf16.restype = C.c_uint16
        L.vso_f32_to_bf16.argtypes = [_f]
        L.vso_f16_to_f32.restype = _f
        L.vso_f16_to_f32.argtypes = [C.c_uint16]

    def distance(self, metric, vtype, a, b, int_exact=False) -> float:
        n = a.size
        return float(self.lib.vso_distance(metric, vtype, _ptr(a), _ptr(b), n, int(int_exact)))

    def quantize(self, vtype, v, offset, scale, qtype) -> np.ndarray:
        out = np.zeros(v.size, dtype=np.uint8 if qtype == Q_U8 else np.int8)
        self.lib.vso_quantize(vtype, _ptr(v), _ptr(out), float(offset), float(scale), v.size, qtype)
        return out

    def quant_params(self, vtype, vectors, qtype_in=Q_AUTO):
        n, dim = vectors.shape
        s, o, q = C.c_float(), C.c_float(), C.c_int()
        self.lib.vso_quant_params(vtype, _ptr(vectors), n, dim, qtype_in, C.byref(s), C.byref(o), C.byref(q))
        return s.value, o.value, q.value

    def build_quant_buffer(self, vtype, vectors, rowids, offset, scale, qtype) -> np.ndarray:
        n, dim = vectors.shape
        out = np.zeros(n * (8 + dim), dtype=np.uint8)
        rid = None if rowids is None else np.ascontiguousarray(rowids, dtype=np.int64)
        self.lib.vso_build_quant_buffer(vtype, _ptr(vectors), _ptr(rid), n, dim, float(offset), float(scale), qtype, _ptr(out))
        return out

    def scan_topk(self, metric, vtype, query, data, n, dim, stride, vec_off, rowids, k, start_max_index=0, int_exact=False):
        ids = np.zeros(max(k, 1), dtype=np.int64)
        dist = np.zeros(max(k, 1), dtype=np.float64)
        rid = None if rowids is None else np.ascontiguousarray(rowids, dtype=np.int64)
        cnt = self.lib.vso_scan_topk(metric, vtype, _ptr(query), _ptr(data), n, dim, stride, vec_off, _ptr(rid), k,
                                     start_max_index, int(int_exact), _ptr(ids), _ptr(dist), None)
        return ids[:cnt].copy(), dist[:cnt].copy()

    def scan_dense(self, metric, vtype, query, vectors, rowids, k, **kw):
        """vFullScanRun arithmetic over a dense [n, dim] column."""
        n, dim = vectors.shape
        return self.scan_topk(metric, vtype, query, vectors.view(np.uint8).reshape(-1), n, dim,
                              dim * ELEM_SIZE[vtype], 0, rowids, k, **kw)

    def scan_quant_buffer(self, metric, qtype, qquery, buf, n, dim, k, **kw):
        """vQuantRunMemory over the preload buffer n x [int64 rowid | dim bytes]."""
        vt = U8 if qtype == Q_U8 else I8
        return self.scan_topk(metric, vt, qquery, buf, n, dim, 8 + dim, 8, None, k, **kw)

    def topk_from_distances(self, dist, ids, k, start_max_index=0):
        dist = np.ascontiguousarray(dist, dtype=np.float32)
        idsa = None if ids is None else np.ascontiguousarray(ids, dtype=np.int64)
        oi = np.zeros(max(k, 1), dtype=np.int64)
        od = np.zeros(max(k, 1), dtype=np.float64)
        cnt = self.lib.vso_topk_from_distances(_ptr(dist), _ptr(idsa), dist.size, k, start_max_index, _ptr(oi), _ptr(od))
        return oi[:cnt].copy(), od[:cnt].copy()

    def distances_all(self, metric, vtype, query, vectors, int_exact=False) -> np.ndarray:
        n, dim = vectors.shape
        out = np.zeros(n, dtype=np.float32)
        self.lib.vso_distances_all(metric, vtype, _ptr(query), _ptr(vectors.view(np.uint8).reshape(-1)), n, dim,
                                   dim * ELEM_SIZE[vtype], 0, int(int_exact), _ptr(out))
        return out

    def f32_to_f16(self, x: np.ndarray) -> np.ndarray:
        return np.array([self.lib.vso_f32_to_f16(float(v)) for v in np.asarray(x, dtype=np.float32).ravel()],
                        dtype=np.uint16).reshape(np.shape(x))

    def f32_to_bf16(self, x: np.ndarray) -> np.ndarray:
        return np.array([self.lib.vso_f32_to_bf16(float(v)) for v in np.asarray(x, dtype=np.float32).ravel()],
                        dtype=np.uint16).reshape(np.shape(x))


class RefHarness:
    """oracle/_ref/libref_{cpu,avx2}.so — the reference's own functions (oracle/ref_harness.c)."""

    def __init__(self, variant: str = "cpu"):
        path = os.path.join(REF_DIR, f"libref_{variant}.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.variant = variant
        self.lib = L = C.CDLL(path)  # RTLD_LOCAL + -Bsymbolic: both variants can coexist in one process
        L.refh_backend.restype = C.c_char_p
        L.refh_backend.argtypes = [_i]
        L.refh_distance.restype = _f
        L.refh_distance.argtypes = [_i, _i, _vp, _vp, _i]
        L.refh_clamp_tiny.restype = _f
        L.refh_clamp_tiny.argtypes = [_f]
        L.refh_quantize.restype = None
        L.refh_quantize.argtypes = [_i, _vp, _vp, _f, _f, _i, _i]
        L.refh_f32_to_f16.restype = C.c_uint16
        L.refh_f32_to_f16.argtypes = [_f]
        L.refh_f32_to_bf16.restype = C.c_uint16
        L.refh_f32_to_bf16.argtypes = [_f]
        L.refh_f16_to_f32.restype = _f
        L.refh_f16_to_f32.argtypes = [C.c_uint16]
        L.refh_quant_scan.restype = _i
        L.refh_quant_scan.argtypes = [_vp, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp]
        L.refh_flat_scan.restype = _i
        L.refh_flat_scan.argtypes = [_i, _i, _vp, _vp, _i64, _i, _sz, _sz, _vp, _i, _i, _vp, _vp]
        L.refh_time_queries.restype = C.c_double
        L.refh_time_queries.argtypes = [_vp, _i64, _i, _sz, _sz, _i, _i, _i, _i, _i, _vp, _sz, _i, _i, _vp]
        self.backend = L.refh_backend(0).decode()

    def distance(self, metric, vtype, a, b) -> float:
        return float(self.lib.refh_distance(metric, vtype, _ptr(a), _ptr(b), a.size))

    def quantize(self, vtype, v, offset, scale, qtype) -> np.ndarray:
        out = np.zeros(v.size, dtype=np.uint8 if qtype == Q_U8 else np.int8)
        self.lib.refh_quantize(vtype, _ptr(v), _ptr(out), float(offset), float(scale), v.size, qtype)
        return out

    def scan_quant_buffer(self, metric, qtype, qquery, buf, n, dim, k, start_max_index=0):
        ids = np.zeros(max(k, 1), dtype=np.int64)
        dist = np.zeros(max(k, 1), dtype=np.float64)
        cnt = self.lib.refh_quant_scan(_ptr(buf), n, dim, qtype, metric, k, _ptr(qquery), start_max_index, _ptr(ids), _ptr(dist), None)
        return ids[:cnt].copy(), dist[:cnt].copy()

    def scan_dense(self, metric, vtype, query, vectors, rowids, k, start_max_index=0):
        n, dim = vectors.shape
        ids = np.zeros(max(k, 1), dtype=np.int64)
        dist = np.zeros(max(k, 1), dtype=np.float64)
        rid = np.ascontiguousarray(rowids, dtype=np.int64)
        cnt = self.lib.refh_flat_scan(metric, vtype, _ptr(query), _ptr(vectors.view(np.uint8).reshape(-1)), n, dim,
                                      dim * ELEM_SIZE[vtype], 0, _ptr(rid), k, start_max_index, _ptr(ids), _ptr(dist))
        return ids[:cnt].copy(), dist[:cnt].copy()

    def time_queries(self, data, n, dim, stride, vec_off, metric, vtype, quant, qtype, k, queries, threads, reps) -> float:
        q = np.ascontiguousarray(queries)
        qbytes = q.nbytes // (threads * reps)
        cs = C.c_int64()
        return float(self.lib.refh_time_queries(_ptr(data), n, dim, stride, vec_off, metric, vtype, int(quant), qtype, k,
                                                _ptr(q.view(np.uint8).reshape(-1)), qbytes, threads, reps, C.byref(cs)))


# ---------------------------------------------------------------- deterministic inputs (SURVEY §8d)
def gen_f32(n: int, dim: int, seed: int) -> np.ndarray:
    return np.random.Generator(np.random.PCG64(seed)).standard_normal((n, dim), dtype=np.float32)


def f32_to_bf16_np(x: np.ndarray) -> np.ndarray:
    """RNE bit trick of src/distance-cpu.h:103-108, vectorised."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    return ((u + np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1))) >> np.uint32(16)).astype(np.uint16)


def f32_to_f16_np(x: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(x, dtype=np.float32).astype(np.float16).view(np.uint16)


def convert(x_f32: np.ndarray, vtype: int, *, scale_u8: bool = True) -> np.ndarray:
    """Derive the column in `vtype` storage from an f32 matrix the way SURVEY §8(d) prescribes."""
    if vtype == F32:
        return np.ascontiguousarray(x_f32, dtype=np.float32)
    if vtype == F16:
        return f32_to_f16_np(x_f32)
    if vtype == BF16:
        return f32_to_bf16_np(x_f32)
    if vtype == I8:
        return np.clip(np.rint(x_f32 * 24.0), -128, 127).astype(np.int8)
    if vtype == U8:
        return np.clip(np.rint(np.abs(x_f32) * 48.0), 0, 255).astype(np.uint8)
    raise ValueError(vtype)
