"""Pins oracle/vs_oracle.c against the UNMODIFIED reference (oracle/_ref, built by oracle/Makefile).

The reference's answers to these calls are recorded once from that build (tests/refgolden.py), so the
comparison runs on machines without the reference sources.
"""
import numpy as np
import pytest

from oracle import pyoracle as po

TYPES = [po.F32, po.F16, po.BF16, po.U8, po.I8]
METRICS = [po.L2, po.L2SQ, po.COS, po.DOT, po.L1]


def _same(a, b):
    a, b = np.float32(a), np.float32(b)
    return (np.isnan(a) and np.isnan(b)) or a.view(np.uint32) == b.view(np.uint32)


def test_backends(ref_cpu, ref_avx2):
    assert ref_cpu.backend == "CPU"      # stock flags never enable AVX2 (SURVEY trap 1)
    assert ref_avx2.backend == "AVX2"


@pytest.mark.parametrize("vtype", TYPES)
@pytest.mark.parametrize("metric", METRICS)
def test_distance_bit_exact(oracle, ref_cpu, vtype, metric):
    rng = np.random.Generator(np.random.PCG64(100 * vtype + metric))
    for dim in (1, 3, 4, 7, 16, 33, 128, 384, 771):
        x = po.convert(rng.standard_normal((6, dim), dtype=np.float32), vtype)
        for i in range(0, 6, 2):
            got = oracle.distance(metric, vtype, x[i], x[i + 1])
            want = ref_cpu.distance(metric, vtype, x[i], x[i + 1])
            assert _same(got, want), (vtype, metric, dim, got, want)
        assert _same(oracle.distance(metric, vtype, x[0], x[0]), ref_cpu.distance(metric, vtype, x[0], x[0]))


@pytest.mark.parametrize("vtype", [po.F16, po.BF16, po.F32])
@pytest.mark.parametrize("metric", METRICS)
def test_distance_special_values(oracle, ref_cpu, vtype, metric):
    specials = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 1.0, -2.5, 65504.0, 1e-8, 3.0], dtype=np.float32)
    rng = np.random.Generator(np.random.PCG64(7))
    for trial in range(200):
        dim = int(rng.integers(1, 12))
        a = rng.choice(specials, dim).astype(np.float32)
        b = rng.choice(specials, dim).astype(np.float32)
        if trial % 3 == 0:  # mostly finite with one odd lane
            a = rng.standard_normal(dim).astype(np.float32); b = rng.standard_normal(dim).astype(np.float32)
            a[rng.integers(dim)] = rng.choice(specials)
        xa, xb = po.convert(a, vtype), po.convert(b, vtype)
        got, want = oracle.distance(metric, vtype, xa, xb), ref_cpu.distance(metric, vtype, xa, xb)
        assert _same(got, want), (vtype, metric, a, b, got, want)


@pytest.mark.parametrize("vtype", [po.U8, po.I8])
@pytest.mark.parametrize("metric", METRICS)
def test_int_exact_matches_avx2(oracle, ref_avx2, vtype, metric):
    """int_exact=1 is the int32-accumulating AVX2 behaviour (src/distance-avx2.c:586-950)."""
    rng = np.random.Generator(np.random.PCG64(5))
    for dim in (16, 384, 1536, 4096):
        lo, hi = (0, 256) if vtype == po.U8 else (-128, 128)
        x = rng.integers(lo, hi, (4, dim)).astype(po.NP_STORAGE[vtype])
        for i in (0, 2):
            assert _same(oracle.distance(metric, vtype, x[i], x[i + 1], int_exact=True),
                         ref_avx2.distance(metric, vtype, x[i], x[i + 1])), (vtype, metric, dim)


def test_conversions(oracle, ref_cpu):
    rng = np.random.Generator(np.random.PCG64(3))
    vals = np.concatenate([rng.standard_normal(2000).astype(np.float32) * np.float32(10.0) ** rng.integers(-9, 6, 2000).astype(np.float32),
                           np.array([0, -0.0, np.inf, -np.inf, np.nan, 65504, 65519.99, 65520, 6e-8, 5.96e-8, 2.98e-8, 2.99e-8, 6.1e-5, 1e-45], dtype=np.float32)])
    for v in vals:
        v = float(v)
        assert oracle.lib.vso_f32_to_f16(v) == ref_cpu.lib.refh_f32_to_f16(v), v
        assert oracle.lib.vso_f32_to_bf16(v) == ref_cpu.lib.refh_f32_to_bf16(v), v
    for h in range(0, 65536, 7):
        assert _same(oracle.lib.vso_f16_to_f32(h), ref_cpu.lib.refh_f16_to_f32(h)), h
    x = rng.standard_normal(500).astype(np.float32)
    assert np.array_equal(po.f32_to_f16_np(x), oracle.f32_to_f16(x))
    assert np.array_equal(po.f32_to_bf16_np(x), oracle.f32_to_bf16(x))


@pytest.mark.parametrize("vtype", TYPES)
@pytest.mark.parametrize("qtype", [po.Q_U8, po.Q_S8])
def test_quantize_bytes(oracle, ref_cpu, vtype, qtype):
    rng = np.random.Generator(np.random.PCG64(11 + vtype))
    for dim in (1, 5, 384):
        x = po.convert(rng.standard_normal((3, dim), dtype=np.float32) * 3, vtype)
        scale, offset, _ = oracle.quant_params(vtype, x, qtype)
        for r in range(3):
            assert np.array_equal(oracle.quantize(vtype, x[r], offset, scale, qtype).view(np.uint8),
                                  ref_cpu.quantize(vtype, x[r], offset, scale, qtype).view(np.uint8))


@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("qtype", [po.Q_U8, po.Q_S8])
def test_quant_scan_topk_exact(oracle, ref_cpu, metric, qtype):
    """vQuantRunMemory + vFullScanSortSlots, including tie handling (small value range => many ties)."""
    rng = np.random.Generator(np.random.PCG64(metric * 10 + qtype))
    for (n, dim, k, spread) in [(500, 16, 20, 3), (3000, 32, 20, 40), (64, 8, 100, 2), (1000, 4, 7, 1), (2000, 384, 33, 60)]:
        lo, hi = (0, 2 * spread) if qtype == po.Q_U8 else (-spread, spread)
        vec = rng.integers(lo, hi + 1, (n, dim)).astype(np.uint8 if qtype == po.Q_U8 else np.int8)
        rowids = (np.arange(n, dtype=np.int64) * 3 + 5)
        buf = np.zeros((n, 8 + dim), dtype=np.uint8)
        buf[:, :8] = rowids.view(np.uint8).reshape(n, 8)
        buf[:, 8:] = vec.view(np.uint8)
        buf = buf.reshape(-1)
        q = rng.integers(lo, hi + 1, dim).astype(vec.dtype)
        for smi in (0, min(3, k - 1)):
            ids_o, d_o = oracle.scan_quant_buffer(metric, qtype, q, buf, n, dim, k, start_max_index=smi)
            ids_r, d_r = ref_cpu.scan_quant_buffer(metric, qtype, q, buf, n, dim, k, start_max_index=smi)
            assert np.array_equal(ids_o, ids_r) and np.array_equal(d_o, d_r), (n, dim, k)


@pytest.mark.parametrize("vtype", TYPES)
def test_dense_scan_topk_exact(oracle, ref_cpu, vtype):
    rng = np.random.Generator(np.random.PCG64(77 + vtype))
    x = po.convert(rng.standard_normal((800, 24), dtype=np.float32), vtype)
    rowids = np.arange(1, 801, dtype=np.int64)
    q = x[17].copy()
    for metric in METRICS:
        ids_o, d_o = oracle.scan_dense(metric, vtype, q, x, rowids, 20)
        ids_r, d_r = ref_cpu.scan_dense(metric, vtype, q, x, rowids, 20)
        assert np.array_equal(ids_o, ids_r) and np.array_equal(d_o, d_r), (vtype, metric)
