"""Property tests that pin the oracle to the UNMODIFIED reference build (oracle/_ref) on drawn inputs: distances for every
(type, metric) pair with special values mixed in, and the k-slot top-k (ties, start_max_index, k > n).  CPU only.  Each test
draws 400 examples from a fixed seed, so the inputs are the same on every run and in any test order; the reference's answers
to them are recorded by tests/refgolden.py."""
import numpy as np

from oracle import pyoracle as po

TYPES = [po.F32, po.F16, po.BF16, po.U8, po.I8]
METRICS = [po.L2, po.L2SQ, po.COS, po.DOT, po.L1]
SPECIALS = [np.nan, np.inf, -np.inf, 0.0, -0.0, 65504.0, -65504.0, 1e-8, 3.0e38, -3.0e38, 5.96e-8]
EXAMPLES = 400


def _same(a, b):
    a, b = np.float32(a), np.float32(b)
    return (np.isnan(a) and np.isnan(b)) or a.view(np.uint32) == b.view(np.uint32)


def _draws(stream, **params):
    """EXAMPLES parameter sets: an integer range (lo, hi) gives lo or hi one time in eight each, else a uniform draw (the ends
    are where the slot logic and the vector tails break); a list gives one of its items"""
    rng = np.random.Generator(np.random.PCG64(stream))
    for _ in range(EXAMPLES):
        ex = {}
        for name, p in params.items():
            if isinstance(p, tuple):
                u = rng.random()
                ex[name] = p[0] if u < 0.125 else p[1] if u < 0.25 else int(rng.integers(p[0], p[1] + 1))
            else:
                ex[name] = p[int(rng.integers(len(p)))]
        yield ex


def test_distance_matches_reference(oracle, ref_cpu):
    for ex in _draws(1, seed=(0, 2**32 - 1), dim=(1, 70), vtype=TYPES, metric=METRICS, nspecial=(0, 4), scale=[1e-3, 1.0, 50.0, 3000.0]):
        _distance_case(oracle, ref_cpu, **ex)


def _distance_case(oracle, ref_cpu, seed, dim, vtype, metric, nspecial, scale):
    rng = np.random.Generator(np.random.PCG64(seed))
    a = (rng.standard_normal(dim) * scale).astype(np.float32)
    b = (rng.standard_normal(dim) * scale).astype(np.float32)
    if vtype in (po.F32, po.F16, po.BF16):
        for _ in range(nspecial):
            (a if rng.integers(2) else b)[rng.integers(dim)] = rng.choice(SPECIALS)
    xa, xb = po.convert(a, vtype), po.convert(b, vtype)
    got, want = oracle.distance(metric, vtype, xa, xb), ref_cpu.distance(metric, vtype, xa, xb)
    assert _same(got, want), (vtype, metric, dim, a, b, got, want)


def test_quant_scan_topk_matches_reference(oracle, ref_cpu):
    """vQuantRunMemory + vFullScanSortSlots on tie-heavy data, any start_max_index below k"""
    for ex in _draws(2, seed=(0, 2**32 - 1), n=(1, 400), dim=(1, 24), k=(1, 40), spread=(1, 6), qtype=[po.Q_U8, po.Q_S8], metric=METRICS,
                     smi=(0, 39)):
        _quant_scan_case(oracle, ref_cpu, **ex)


def _quant_scan_case(oracle, ref_cpu, seed, n, dim, k, spread, qtype, metric, smi):
    rng = np.random.Generator(np.random.PCG64(seed))
    lo, hi = (0, 2 * spread) if qtype == po.Q_U8 else (-spread, spread)
    vec = rng.integers(lo, hi + 1, (n, dim)).astype(np.uint8 if qtype == po.Q_U8 else np.int8)
    rowids = rng.permutation(n).astype(np.int64) * 7 - 3
    buf = np.zeros((n, 8 + dim), dtype=np.uint8)
    buf[:, :8] = rowids.view(np.uint8).reshape(n, 8)
    buf[:, 8:] = vec.view(np.uint8)
    q = rng.integers(lo, hi + 1, dim).astype(vec.dtype)
    smi = smi % k
    ids_o, d_o = oracle.scan_quant_buffer(metric, qtype, q, buf.reshape(-1), n, dim, k, start_max_index=smi)
    ids_r, d_r = ref_cpu.scan_quant_buffer(metric, qtype, q, buf.reshape(-1), n, dim, k, start_max_index=smi)
    assert np.array_equal(ids_o, ids_r) and np.array_equal(d_o, d_r), (n, dim, k, smi, qtype, metric)


def test_dense_scan_topk_matches_reference(oracle, ref_cpu):
    for ex in _draws(3, seed=(0, 2**32 - 1), n=(1, 300), dim=(1, 20), k=(1, 30), vtype=TYPES, metric=METRICS):
        _dense_scan_case(oracle, ref_cpu, **ex)


def _dense_scan_case(oracle, ref_cpu, seed, n, dim, k, vtype, metric):
    rng = np.random.Generator(np.random.PCG64(seed))
    x = po.convert(np.round(rng.standard_normal((n, dim)) * 2).astype(np.float32), vtype)       # coarse values: many equal distances
    rowids = np.arange(1, n + 1, dtype=np.int64)
    q = x[rng.integers(n)].copy()
    ids_o, d_o = oracle.scan_dense(metric, vtype, q, x, rowids, k)
    ids_r, d_r = ref_cpu.scan_dense(metric, vtype, q, x, rowids, k)
    assert np.array_equal(ids_o, ids_r) and np.array_equal(d_o, d_r), (vtype, metric, n, dim, k)
