"""Generate tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref, built by oracle/Makefile
from the reference tree):

    make -C oracle REF=<reference tree> && python tests/golden/make_golden.py
    python tests/golden/make_golden.py --record          # reference answers replayed by tests/refgolden.py
    python tests/golden/make_golden.py --abi <dir of sqlite3ext.h>

Everything written is produced by reference code: distances by dispatch_distance_table (stock "CPU"
build = distance-cpu.c), quantized bytes by quantize_*, top-k by vQuantRunMemory / the vFullScanRun
arithmetic + vFullScanSortSlots.  Inputs are stored beside the outputs so the fixtures are self-contained.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
TYPES = [po.F32, po.F16, po.BF16, po.U8, po.I8]
METRICS = [po.L2, po.L2SQ, po.COS, po.DOT, po.L1]


def main():
    ref = po.RefHarness("cpu")
    avx = po.RefHarness("avx2")
    assert ref.backend == "CPU" and avx.backend == "AVX2"
    rng = np.random.Generator(np.random.PCG64(20260922))

    # 1. distances: 5 types x 5 metrics x dims, 24 row pairs each
    dist = {}
    for vt in TYPES:
        for dim in (5, 128, 384):
            x = po.convert(rng.standard_normal((25, dim), dtype=np.float32), vt)
            dist[f"x_{vt}_{dim}"] = x
            for m in METRICS:
                dist[f"d_{vt}_{dim}_{m}"] = np.array([ref.distance(m, vt, x[0], x[i]) for i in range(25)], dtype=np.float32)
                if vt in (po.U8, po.I8):
                    dist[f"davx2_{vt}_{dim}_{m}"] = np.array([avx.distance(m, vt, x[0], x[i]) for i in range(25)], dtype=np.float32)
    # special values (f16 / bf16 / f32)
    sp = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 1.0, -2.5, 65504.0, 3.0, 0.5], dtype=np.float32)
    for vt in (po.F32, po.F16, po.BF16):
        a = po.convert(rng.choice(sp, (40, 6)).astype(np.float32), vt)
        b = po.convert(rng.choice(sp, (40, 6)).astype(np.float32), vt)
        dist[f"spa_{vt}"], dist[f"spb_{vt}"] = a, b
        for m in METRICS:
            dist[f"spd_{vt}_{m}"] = np.array([ref.distance(m, vt, a[i], b[i]) for i in range(40)], dtype=np.float32)
    np.savez_compressed(os.path.join(OUT, "distances.npz"), **dist)

    # 2. quantizer bytes
    qz = {}
    for vt in TYPES:
        x = po.convert(rng.standard_normal((8, 48), dtype=np.float32) * 2.5, vt)
        qz[f"x_{vt}"] = x
        for qt in (po.Q_U8, po.Q_S8):
            scale, offset = (37.5, -2.0) if qt == po.Q_U8 else (31.0, 0.0)
            qz[f"q_{vt}_{qt}"] = np.stack([ref.quantize(vt, x[r], offset, scale, qt).view(np.uint8) for r in range(8)])
            qz[f"p_{vt}_{qt}"] = np.array([scale, offset], dtype=np.float32)
    np.savez_compressed(os.path.join(OUT, "quantize.npz"), **qz)

    # 3. top-k with heavy ties (quantized preload buffer) and fp dense scans
    tk = {}
    case = 0
    for qt in (po.Q_U8, po.Q_S8):
        for (n, dim, k, spread) in [(600, 16, 20, 3), (2500, 32, 20, 30), (50, 8, 100, 2), (900, 4, 7, 1)]:
            lo, hi = (0, 2 * spread) if qt == po.Q_U8 else (-spread, spread)
            vec = rng.integers(lo, hi + 1, (n, dim)).astype(np.uint8 if qt == po.Q_U8 else np.int8)
            rowids = np.arange(n, dtype=np.int64) * 2 + 11
            q = rng.integers(lo, hi + 1, dim).astype(vec.dtype)
            buf = np.zeros((n, 8 + dim), dtype=np.uint8)
            buf[:, :8] = rowids.view(np.uint8).reshape(n, 8)
            buf[:, 8:] = vec.view(np.uint8)
            tk[f"c{case}_meta"] = np.array([qt, n, dim, k], dtype=np.int64)
            tk[f"c{case}_vec"], tk[f"c{case}_rowids"], tk[f"c{case}_q"] = vec, rowids, q
            for m in METRICS:
                ids, d = ref.scan_quant_buffer(m, qt, q, buf.reshape(-1), n, dim, k)
                tk[f"c{case}_ids_{m}"], tk[f"c{case}_dist_{m}"] = ids, d
            case += 1
    tk["ncases"] = np.array([case])
    for vt in (po.F32, po.F16, po.BF16):
        x = po.convert(rng.standard_normal((700, 24), dtype=np.float32), vt)
        q = po.convert(rng.standard_normal((1, 24), dtype=np.float32), vt)[0]
        rowids = np.arange(1, 701, dtype=np.int64)
        tk[f"fp{vt}_x"], tk[f"fp{vt}_q"] = x, q
        for m in METRICS:
            ids, d = ref.scan_dense(m, vt, q, x, rowids, 20)
            tk[f"fp{vt}_ids_{m}"], tk[f"fp{vt}_dist_{m}"] = ids, d
    np.savez_compressed(os.path.join(OUT, "topk.npz"), **tk)
    for f in ("distances.npz", "quantize.npz", "topk.npz"):
        print(f, os.path.getsize(os.path.join(OUT, f)), "bytes")


if __name__ == "__main__" and not {"--sql", "--c1", "--record", "--abi"} & set(sys.argv):
    main()


def sql_golden():
    """SQL-level outputs of the unmodified reference extension (stock build, backend 'CPU')."""
    import json
    from tests import sql_cases
    from tests.sqlrun import REF_CPU, run_sql
    for name, script in (("sql_surface.json", sql_cases.surface_script()), ("sql_scan.json", sql_cases.scan_script())):
        res = run_sql(REF_CPU, script)
        with open(os.path.join(OUT, name), "w") as f:
            json.dump(res, f)
        print(name, os.path.getsize(os.path.join(OUT, name)), "bytes,", sum("error" in r for r in res), "error results")


if __name__ == "__main__" and "--sql" in sys.argv:
    sql_golden()


def c1_golden():
    """BASELINE config 1 (vector_full_scan L2 f32 dim=384 n=100k k=20) through SQL on the unmodified reference (stock build)"""
    import json
    from tests.sqlrun import REF_CPU, run_c1
    res = run_c1(REF_CPU)
    keep = {"full": res["full"], "quant": res["quant"], "quantized_rows": res["quantized_rows"],
            "config": {"n": 100000, "dim": 384, "k": 20, "nq": 3, "metric": "L2", "rowids": "3*i+1", "seeds": [1234, 4321]}}
    with open(os.path.join(OUT, "sql_c1.json"), "w") as f:
        json.dump(keep, f)
    print("sql_c1.json", os.path.getsize(os.path.join(OUT, "sql_c1.json")), "bytes; reference ms per full scan", res["ms_full"], "quant", res["ms_quant"])


if __name__ == "__main__" and "--c1" in sys.argv:
    c1_golden()


RECORDED_TESTS = ["tests/test_oracle_vs_reference.py", "tests/test_oracle_fuzz.py", "tests/test_sql_fuzz.py",
                  "tests/test_sql_surface.py::test_surface_matches_live_reference"]


def record():
    """run the tests that compare with the reference against its live build, and store every answer it gave them"""
    import pytest
    from tests import refgolden
    refgolden.RECORDING = True
    rc = pytest.main(["-q", "-p", "no:cacheprovider", "-m", "not gpu"] + [os.path.join(ROOT, t) for t in RECORDED_TESTS])
    if rc != 0:
        raise SystemExit(f"pytest exited with {rc}: nothing recorded")
    refgolden.save()
    for f in (refgolden.CALLS, refgolden.SQL):
        print(os.path.relpath(f, ROOT), os.path.getsize(f), "bytes")


if __name__ == "__main__" and "--record" in sys.argv:
    record()


def abi_slots(hdr_dir):
    """slot of every sqlite3_api_routines member, as the compiler lays the struct out: offsetof / sizeof(void *)"""
    import json
    import subprocess
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from gen_sqlite_abi import members
    names = members(os.path.join(hdr_dir, "sqlite3ext.h"))
    lines = "\n".join(f'    printf("%s %zu\\n", "{n}", offsetof(sqlite3_api_routines, {n}) / sizeof(void *));' for n in names)
    src = "#include <stddef.h>\n#include <stdio.h>\n#include \"sqlite3ext.h\"\nint main(void) {\n" + lines + "\n    return 0;\n}\n"
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "slots.c"), "w") as f:
            f.write(src)
        subprocess.run(["gcc", "-I", hdr_dir, "-o", os.path.join(tmp, "slots"), os.path.join(tmp, "slots.c")], check=True)
        out = subprocess.run([os.path.join(tmp, "slots")], capture_output=True, text=True, check=True).stdout
    slots = {n: int(i) for n, i in (ln.split() for ln in out.splitlines())}
    with open(os.path.join(OUT, "sqlite3_api_slots.json"), "w") as f:
        json.dump(slots, f, indent=0)
    print("sqlite3_api_slots.json:", len(slots), "members")


if __name__ == "__main__" and "--abi" in sys.argv:
    abi_slots(sys.argv[sys.argv.index("--abi") + 1])
