"""The extension's SQL surface vs the reference: encoders, options, error strings, quantization bytes and
metadata (CPU, no scans) and the scans themselves through SQL (GPU).  Golden outputs come from the unmodified
reference extension (tests/golden/make_golden.py --sql)."""
import json
import os

import pytest

from tests import sql_cases
from tests.refgolden import run_reference_sql
from tests.sqlrun import OURS, ROOT, run_sql

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# statements where we deliberately differ from the reference (see DESIGN.md "deviations")
SURFACE_DEVIATIONS = {
    "SELECT vector_init('w2', 'e', 'type=INT8,dimension=4')",   # reference reports an empty NOMEM error (inverted ternary, sqlite-vector.c:1086)
}


def _stmt(s):
    return s if isinstance(s, str) else s[0]


def test_surface_matches_reference_golden():
    script = sql_cases.surface_script()
    ours = run_sql(OURS, script)
    want = json.load(open(os.path.join(G, "sql_surface.json")))
    assert len(ours) == len(want)
    for s, a, b in zip(script, ours, want):
        if _stmt(s) in SURFACE_DEVIATIONS:
            assert "error" in a and "error" in b
            continue
        assert a == b, (_stmt(s), a, b)


def test_surface_matches_live_reference():
    script = sql_cases.surface_script()
    ours, ref = run_sql(OURS, script), run_reference_sql(script)
    for s, a, b in zip(script, ours, ref):
        if _stmt(s) not in SURFACE_DEVIATIONS:
            assert a == b, (_stmt(s), a, b)


def test_version_and_backend_strings():
    r = run_sql(OURS, ["SELECT vector_version()", "SELECT vector_backend()"])
    assert r[0]["rows"][0][0].startswith("0.9.23")
    assert "CUDA sm_100a" in r[1]["rows"][0][0]


def test_scan_without_gpu_fails_loudly():
    import sqlite_vector_b200 as vs
    if vs.load_engine().device_count() > 0:
        pytest.skip("a GPU is present")
    r = run_sql(OURS, ["CREATE TABLE t (id INTEGER PRIMARY KEY, e BLOB)", "SELECT vector_init('t','e','type=INT8,dimension=4')",
                       "INSERT INTO t VALUES (1, x'01020304')", "SELECT * FROM vector_full_scan('t','e',x'01020304',1)"])
    assert "no CUDA device" in r[3]["error"]


def test_api_slot_positions_against_sqlite_header():
    """sqlite_abi.h hard-codes positions inside sqlite3_api_routines; verify them against the positions a compiler gave every
    member of a real sqlite3ext.h, offsetof(sqlite3_api_routines, member) / sizeof(void *) (tests/golden/make_golden.py --abi)."""
    import re
    abi = open(os.path.join(ROOT, "sqlite_vector_b200", "csrc", "sqlite_abi.h")).read()
    slots = [(n, int(i)) for n, i in re.findall(r"VSQ_(\w+) = (\d+)", abi) if n != "API_SLOTS_USED"]
    want = json.load(open(os.path.join(G, "sqlite3_api_slots.json")))
    assert [(n, want.get(n)) for n, _ in slots] == slots
    assert len(slots) > 40


def test_bad_argument_types_give_errors_not_crashes():
    """the reference segfaults on a non-INTEGER k (its error path formats argc with %s, sqlite-vector.c:1754); we report it"""
    r = run_sql(OURS, ["CREATE TABLE t (id INTEGER PRIMARY KEY, e BLOB)", "SELECT vector_init('t','e','type=INT8,dimension=4')",
                       "SELECT * FROM vector_full_scan('t','e',x'01020304','x')", "SELECT * FROM vector_full_scan('t',2,x'01020304',1)",
                       "SELECT * FROM vector_quantize_scan('t','e',1.5,1)", "SELECT * FROM vector_full_scan('t','e',x'0102',1)"])
    assert r[2]["error"] == "vector_full_scan: argument 4 must be of type INTEGER (got TEXT)."
    assert r[3]["error"] == "vector_full_scan: argument 2 must be of type TEXT (got INTEGER)."
    assert r[4]["error"] == "vector_quantize_scan: argument 3 must be of type TEXT or BLOB (got REAL)."
    assert "input vector has 2 bytes, expected 4" in r[5]["error"] or "no CUDA device" in r[5]["error"]


@pytest.mark.gpu
def test_scans_through_sql_match_reference_golden():
    script = sql_cases.scan_script()
    ours = run_sql(OURS, script)
    want = json.load(open(os.path.join(G, "sql_scan.json")))
    assert len(ours) == len(want)
    n_checked = 0
    for s, a, b in zip(script, ours, want):
        st = _stmt(s)
        if "error" in b or "error" in a:
            assert ("error" in a) == ("error" in b), (st, a, b)
            if "argument" in b.get("error", "") or "Quantization table" in b.get("error", "") or "JSON" in b.get("error", ""):
                assert a["error"] == b["error"], st
            continue
        ra, rb = a["rows"], b["rows"]
        assert len(ra) == len(rb), (st, ra[:3], rb[:3])
        for x, y in zip(ra, rb):
            for u, v in zip(x, y):
                if isinstance(v, float) and isinstance(u, float):
                    assert abs(u - v) <= 1e-5 * max(abs(v), 1.0), (st, x, y)
                else:
                    assert u == v, (st, x, y)
        n_checked += 1
    assert n_checked > 40


# ---- batched table-valued functions (an addition; the reference has one vector per call)
def _batch_setup(n=300, dim=8, vtype="INT8"):
    import numpy as np
    rng = np.random.Generator(np.random.PCG64(5))
    x = rng.integers(-20, 21, (n, dim)).astype(np.int8)
    s = ["CREATE TABLE t (id INTEGER PRIMARY KEY, e BLOB)", f"SELECT vector_init('t','e','type={vtype},dimension={dim}')"]
    for i in range(n):
        s.append(["INSERT INTO t(id, e) VALUES (?, ?)", [3 * i + 2, {"hex": x[i].tobytes().hex()}]])
    return x, s


def test_batch_tvf_argument_errors():
    x, s = _batch_setup(5)
    s += ["SELECT * FROM vector_full_scan_batch('t','e',x'0102030405060708')",
          "SELECT * FROM vector_full_scan_batch('t','e',1.5,3)",
          "SELECT * FROM vector_full_scan_batch('t','e',x'01020304',3)",
          "SELECT * FROM vector_full_scan_batch('nope','e',x'0102030405060708',3)",
          "SELECT * FROM vector_quantize_scan_batch('t','e','[1,2,3]',3)",
          "SELECT * FROM vector_quantize_scan_batch('t','e',x'0102030405060708','k')",
          "SELECT * FROM vector_quantize_scan_batch('t','e',x'0102030405060708',2)"]
    r = run_sql(OURS, s)[-7:]
    assert "error" in r[0]                                                    # 3 arguments: SQLite itself refuses the missing hidden column
    assert r[1]["error"] == "vector_full_scan_batch: argument 3 must be of type TEXT or BLOB (got REAL)."
    assert r[2]["error"] == "vector_full_scan_batch: input has 4 bytes, expected a positive multiple of 8 (dimension 8)."
    assert r[3]["error"] == "vector_full_scan_batch: unable to retrieve context."
    assert r[4]["error"] == "vector_quantize_scan_batch: input has 3 bytes, expected a positive multiple of 8 (dimension 8)."
    assert r[5]["error"] == "vector_quantize_scan_batch: argument 4 must be of type INTEGER (got TEXT)."
    assert r[6]["error"].startswith("Quantization table not found")


@pytest.mark.gpu
def test_batch_tvf_equals_single_query_functions():
    import numpy as np
    x, s = _batch_setup(300)
    rng = np.random.Generator(np.random.PCG64(6))
    q = rng.integers(-20, 21, (20, 8)).astype(np.int8)          # 20 queries >= 16: the batch entry point of the engine
    allq = {"hex": q.tobytes().hex()}
    k = 7
    s.append(["SELECT query, id, distance FROM vector_full_scan_batch('t','e',?,?)", [allq, k]])
    for b in range(20):
        s.append(["SELECT id, distance FROM vector_full_scan('t','e',?,?)", [{"hex": q[b].tobytes().hex()}, k]])
    s.append("SELECT vector_quantize('t','e')")
    s.append(["SELECT query, id, distance FROM vector_quantize_scan_batch('t','e',?,?)", [allq, k]])
    for b in range(20):
        s.append(["SELECT id, distance FROM vector_quantize_scan('t','e',?,?)", [{"hex": q[b].tobytes().hex()}, k]])
    jq = "[" + ",".join(str(int(v)) for v in q[:2].reshape(-1)) + "]"
    s.append([f"SELECT query, id, distance FROM vector_full_scan_batch('t','e','{jq}',3)", []])
    s.append(["SELECT count(*) FROM vector_full_scan_batch('t','e',?,0)", [allq]])
    r = run_sql(OURS, s)
    base = len(s) - (2 * 21 + 3)
    for off in (base, base + 22):                                            # full scan block, then (after vector_quantize) the quantized block
        batch = r[off]["rows"]
        assert len(batch) == 20 * k, r[off]
        for b in range(20):
            single = r[off + 1 + b]["rows"]
            assert [row[1:] for row in batch if row[0] == b] == single, (off, b)
    js = r[-2]["rows"]
    assert [row[2] for row in js if row[0] == 1] == [row[1] for row in r[base + 2]["rows"][:3]]     # k=3 vs the head of k=7: same distances
    assert r[-1]["rows"] == [[0]]


@pytest.mark.gpu
def test_config1_through_sql_matches_reference_golden():
    """BASELINE config 1 at its stated size: vector_full_scan L2 f32 dim=384 n=100k k=20 through SQL, against the output of the
    unmodified reference extension (tests/golden/make_golden.py --c1): rowids exact, distances within 1e-5 relative; the
    int8 quantize + preload + vector_quantize_scan leg on the same table: bit-exact."""
    from tests.sqlrun import run_c1
    want = json.load(open(os.path.join(G, "sql_c1.json")))
    got = run_c1(OURS)
    assert got["quantized_rows"] == want["quantized_rows"] == 100000
    for b, (a, w) in enumerate(zip(got["full"], want["full"])):
        assert [r[0] for r in a] == [r[0] for r in w], ("full", b)
        assert all(abs(x[1] - y[1]) <= 1e-5 * abs(y[1]) for x, y in zip(a, w)), ("full", b)
    for b, (a, w) in enumerate(zip(got["quant"], want["quant"])):
        assert a == w, ("quant", b)


@pytest.mark.gpu
def test_k_sequence_and_transactions_through_sql():
    """(1) ADVICE r1 high: k=100 then k=10 then k=33 on one connection; (2) ADVICE r1 medium: a scan inside a transaction
    sees the uncommitted row, a scan after ROLLBACK / ROLLBACK TO must not; (3) vector_quantize nests inside a caller's
    transaction (savepoint) and its lazily staged chunks do not survive a ROLLBACK."""
    import numpy as np

    from oracle import pyoracle as po
    rng = np.random.Generator(np.random.PCG64(11))
    n, dim = 3000, 16
    x = rng.integers(-40, 41, (n, dim)).astype(np.int8)
    ids = np.arange(n, dtype=np.int64) * 2 + 1
    q = rng.integers(-40, 41, dim).astype(np.int8)
    qb = {"hex": q.tobytes().hex()}
    s = ["CREATE TABLE t (id INTEGER PRIMARY KEY, e BLOB)", "CREATE TABLE other (v)", f"SELECT vector_init('t','e','type=INT8,dimension={dim}')"]
    s += [["INSERT INTO t(id, e) VALUES (?, ?)", [int(ids[i]), {"hex": x[i].tobytes().hex()}]] for i in range(n)]
    mark = len(s)
    s += [["SELECT id, distance FROM vector_full_scan('t','e',?,100)", [qb]],        # 0
          ["SELECT id, distance FROM vector_full_scan('t','e',?,10)", [qb]],         # 1
          ["SELECT id, distance FROM vector_full_scan('t','e',?,33)", [qb]],         # 2
          "BEGIN",                                                                   # 3
          ["INSERT INTO t(id, e) VALUES (100001, ?)", [qb]],                         # 4  distance 0 to the query
          ["SELECT id, distance FROM vector_full_scan('t','e',?,3)", [qb]],          # 5  sees it
          "ROLLBACK",                                                                # 6
          ["SELECT id, distance FROM vector_full_scan('t','e',?,3)", [qb]],          # 7  must not
          "BEGIN", "SAVEPOINT sp",                                                   # 8 9
          ["INSERT INTO t(id, e) VALUES (100002, ?)", [qb]],                         # 10
          ["SELECT id, distance FROM vector_full_scan('t','e',?,3)", [qb]],          # 11 sees it
          "ROLLBACK TO sp",                                                          # 12
          ["SELECT id, distance FROM vector_full_scan('t','e',?,3)", [qb]],          # 13 must not
          "INSERT INTO other VALUES (1)",                                            # 14 unrelated write
          ["SELECT id, distance FROM vector_full_scan('t','e',?,3)", [qb]],          # 15
          "COMMIT",                                                                  # 16
          "BEGIN", "SELECT vector_quantize('t','e')",                                # 17 18 nests (reference: fails + rolls the caller back)
          ["SELECT id, distance FROM vector_quantize_scan('t','e',?,5)", [qb]],      # 19 lazily staged inside the transaction
          "ROLLBACK",                                                                # 20 shadow table gone again
          ["SELECT id, distance FROM vector_quantize_scan('t','e',?,5)", [qb]],      # 21 error: not quantized
          "SELECT vector_quantize('t','e','qtype=BOGUS')",                           # 22 error, transaction state intact
          "SELECT vector_quantize('t','e')",                                         # 23
          ["SELECT id, distance FROM vector_quantize_scan('t','e',?,5)", [qb]],      # 24
          ]
    r = run_sql(OURS, s)[mark:]
    orc = po.Oracle()

    def want(k, xs=x, rid=ids):
        a, d = orc.scan_dense(po.L2, po.I8, q, xs, rid, k)
        return [[int(i), float(v)] for i, v in zip(a, d)]
    assert r[0]["rows"] == want(100) and r[1]["rows"] == want(10) and r[2]["rows"] == want(33)
    assert r[5]["rows"][0] == [100001, 0.0]
    assert r[7]["rows"] == want(3), "rolled-back row served from the device copy"
    assert r[11]["rows"][0] == [100002, 0.0]
    assert r[13]["rows"] == want(3) and r[15]["rows"] == want(3)
    assert r[18] == {"rows": [[n]]}, r[18]
    assert len(r[19]["rows"]) == 5
    assert "Quantization table not found" in r[21].get("error", ""), r[21]
    assert "Invalid quantization type" in r[22].get("error", "")
    assert r[23] == {"rows": [[n]]} and r[24]["rows"] == r[19]["rows"]


@pytest.mark.gpu
def test_vector_quantize_on_the_gpu_matches_reference_golden():
    """f2: with a device present vector_quantize runs its min / max and quantization loops as kernels (vsb_quantizer_*): the
    shadow-table bytes, chunk boundaries and stored parameters must equal the reference's golden output exactly, the kernels
    must actually have run, and the host loops (VSB_QUANTIZE_HOST=1) must give the same bytes."""
    script = sql_cases.surface_script()
    want = json.load(open(os.path.join(G, "sql_surface.json")))
    gpu = run_sql(OURS, script, want_launches=True)
    host = run_sql(OURS, script, env={"VSB_QUANTIZE_HOST": "1"}, want_launches=True)
    assert gpu[-1]["kernel_launches"] > host[-1]["kernel_launches"], "vector_quantize did not launch its kernels"
    for s, a, h, b in zip(script, gpu[:-1], host[:-1], want):
        if _stmt(s) in SURFACE_DEVIATIONS:
            continue
        assert a == b, (_stmt(s), a, b)
        assert h == b, (_stmt(s), h, b)
