"""Recorded answers of the unmodified reference, so that every comparison with it also runs where it cannot be built.

Each call a test makes on the reference (a RefHarness function on flat buffers, or a SQL script through its loadable
extension) is keyed by a digest of the function and all of its inputs.  `python tests/golden/make_golden.py --record` runs
the tests that use the reference against the live build in oracle/_ref/ and stores every answer in
tests/golden/reference_calls.npz and tests/golden/reference_sql.json.gz; otherwise the tests are answered from those files.
A call without a recorded answer is an error: the test or its inputs changed, and the recording has to be made again
where the reference can be built."""
import gzip
import hashlib
import json
import os

import numpy as np

from oracle import pyoracle as po

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CALLS = os.path.join(G, "reference_calls.npz")
SQL = os.path.join(G, "reference_sql.json.gz")

RECORDING = False            # set by make_golden.py --record: answer from the live build and keep every answer
_recorded_calls = {}         # "variant.function" -> {digest: tuple of 1-D arrays}
_recorded_sql = {}           # hex digest -> results of the script
_stored_calls = None
_stored_sql = None


def _digest(name, args) -> int:
    h = hashlib.blake2b(name.encode(), digest_size=8)
    for a in args:
        if isinstance(a, np.ndarray):
            a = np.ascontiguousarray(a)
            h.update(f"|{a.dtype.str}{a.shape}|".encode())
            h.update(a.tobytes())
        elif isinstance(a, (bool, int, np.integer)):
            h.update(f"|i{int(a)}".encode())
        elif isinstance(a, (float, np.floating)):
            h.update(f"|f{float(a)!r}".encode())
        else:
            h.update(f"|{a!r}".encode())
    return int.from_bytes(h.digest(), "little")


def _missing(what):
    return LookupError(f"no recorded reference answer for {what}; record again with tests/golden/make_golden.py --record")


def _answer(name, key):
    global _stored_calls
    if _stored_calls is None:
        with np.load(CALLS) as z:
            _stored_calls = {f: z[f] for f in z.files}
    keys = _stored_calls.get(f"{name}.keys")
    i = -1 if keys is None else int(np.searchsorted(keys, np.uint64(key)))
    if i < 0 or i >= keys.size or int(keys[i]) != key:
        raise _missing(name)
    out, c = [], 0
    while f"{name}.v{c}" in _stored_calls:
        off = _stored_calls[f"{name}.off{c}"]
        out.append(_stored_calls[f"{name}.v{c}"][off[i]:off[i + 1]])
        c += 1
    return tuple(out)


def _f32(x):
    return (np.array([x], dtype=np.float32),)


def _u16(x):
    return (np.array([x], dtype=np.uint16),)


def _f32_bits(f) -> int:
    return int(np.array(f, dtype=np.float32).view(np.uint32))


class _Lib:
    """the scalar conversion entry points tests call on RefHarness.lib; keyed by the bits of their one argument (which the
    C signature narrows to float / uint16), not by a digest: thousands of them are recorded"""

    def __init__(self, ref):
        self._ref = ref

    def refh_f32_to_f16(self, f):
        return self._ref._call("f32_to_f16", None, lambda h: h.lib.refh_f32_to_f16(f), _u16, lambda t: int(t[0][0]), key=_f32_bits(f))

    def refh_f32_to_bf16(self, f):
        return self._ref._call("f32_to_bf16", None, lambda h: h.lib.refh_f32_to_bf16(f), _u16, lambda t: int(t[0][0]), key=_f32_bits(f))

    def refh_f16_to_f32(self, h16):
        return self._ref._call("f16_to_f32", None, lambda h: h.lib.refh_f16_to_f32(h16), _f32, lambda t: float(t[0][0]), key=int(h16) & 0xFFFF)


class Reference:
    """pyoracle.RefHarness with the calls the tests make, answered from the recording (while recording: by the live build)."""

    def __init__(self, variant: str = "cpu"):
        self.variant = variant
        self._live = po.RefHarness(variant) if RECORDING else None
        self.lib = _Lib(self)
        self.backend = self._call("backend", (), lambda h: h.backend, lambda s: (np.frombuffer(s.encode(), np.uint8),),
                                  lambda t: t[0].tobytes().decode())

    def _call(self, name, args, live, encode, decode, key=None):
        name = f"{self.variant}.{name}"
        if key is None:
            key = _digest(name, args)
        if RECORDING:
            res = live(self._live)
            _recorded_calls.setdefault(name, {})[key] = tuple(np.ascontiguousarray(a).reshape(-1) for a in encode(res))
            return res
        return decode(_answer(name, key))

    def distance(self, metric, vtype, a, b) -> float:
        return self._call("distance", (metric, vtype, a, b), lambda h: h.distance(metric, vtype, a, b), _f32, lambda t: float(t[0][0]))

    def quantize(self, vtype, v, offset, scale, qtype) -> np.ndarray:
        dtype = np.uint8 if qtype == po.Q_U8 else np.int8
        return self._call("quantize", (vtype, v, offset, scale, qtype), lambda h: h.quantize(vtype, v, offset, scale, qtype),
                          lambda q: (q.view(np.uint8),), lambda t: t[0].view(dtype).copy())

    def scan_quant_buffer(self, metric, qtype, qquery, buf, n, dim, k, start_max_index=0):
        return self._call("scan_quant_buffer", (metric, qtype, qquery, buf, n, dim, k, start_max_index),
                          lambda h: h.scan_quant_buffer(metric, qtype, qquery, buf, n, dim, k, start_max_index=start_max_index),
                          lambda r: r, lambda t: (t[0].copy(), t[1].copy()))

    def scan_dense(self, metric, vtype, query, vectors, rowids, k, start_max_index=0):
        return self._call("scan_dense", (metric, vtype, query, vectors, np.asarray(rowids, dtype=np.int64), k, start_max_index),
                          lambda h: h.scan_dense(metric, vtype, query, vectors, rowids, k, start_max_index=start_max_index),
                          lambda r: r, lambda t: (t[0].copy(), t[1].copy()))


def run_reference_sql(statements):
    """tests.sqlrun.run_sql on the stock build of the reference extension (oracle/_ref/cpu/vector.so)"""
    global _stored_sql
    key = f"{_digest('sql', (json.dumps(statements),)):016x}"
    if RECORDING:
        from tests.sqlrun import REF_CPU, run_sql
        _recorded_sql[key] = res = run_sql(REF_CPU, statements)
        return res
    if _stored_sql is None:
        with gzip.open(SQL, "rt") as f:
            _stored_sql = json.load(f)
    if key not in _stored_sql:
        raise _missing("this SQL script")
    return _stored_sql[key]


def save():
    """write what a recording run collected (replacing the previous recording)"""
    out = {}
    for name, rows in sorted(_recorded_calls.items()):
        keys = np.array(sorted(rows), dtype=np.uint64)
        out[f"{name}.keys"] = keys
        for c in range(len(rows[int(keys[0])])):
            parts = [rows[int(k)][c] for k in keys]
            out[f"{name}.off{c}"] = np.cumsum([0] + [p.size for p in parts]).astype(np.int64)
            out[f"{name}.v{c}"] = np.concatenate(parts)
    np.savez_compressed(CALLS, **out)
    with gzip.GzipFile(SQL, "wb", mtime=0) as f:
        f.write(json.dumps(dict(sorted(_recorded_sql.items())), separators=(",", ":")).encode())
