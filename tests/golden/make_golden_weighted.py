#!/usr/bin/env python
"""Golden vectors for the weighted CSR, cheapest_path_length and iterativelength2, produced by the UNMODIFIED
reference (oracle/_ref/duckdb).  Run in the build container only:

    python tests/golden/make_golden_weighted.py                     # every case
    python tests/golden/make_golden_weighted.py neg_i64 special_f64 # only these

Name the cases you add or change: a rewritten .npz differs in its zip timestamps even when its arrays do not.

Writes tests/golden/refw_<name>.npz: the inputs (n, edge rows with a BIGINT or DOUBLE weight, pairs) and what the
reference returned:
    w_type                csr_get_w_type(0)                               (csr_get_w_type.cpp)
    csr_v, csr_e, csr_w   get_csr_v(0) / get_csr_e(0) / get_csr_w(0)      (pgq_scan.cpp:84-141); the order of a vertex's
                          edges is the order in which DuckDB's join handed them to create_csr_edge -- compare per vertex
    cost, cost_valid      cheapest_path_length(0, n, src, dst)            (cheapest_path_length.cpp)
    length2, length2_valid  iterativelength2(0, n, src, dst)              (iterativelength2.cpp)
The weighted CSR is built by one statement (the 8-argument create_csr_edge overloads, csr_creation.cpp:227-235)
and queried by the next ones of the same CLI session, the way test/sql/scalar/get_csr_w_type.test does.
threads = 1: deterministic single-thread edge order.  All pairs have non-NULL sources (a NULL source shifts the
lanes of the reference's batch, cheapest_path_length.cpp:18-25 vs 88-93 -- see DESIGN.md section 7)."""
import csv
import io
import os
import subprocess
import sys
import tempfile

import numpy as np
import pyarrow as pa
import pyarrow.parquet as pq

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from duckpgq_extension_b200 import datagen  # noqa: E402

DUCKDB = os.path.join(ROOT, "oracle", "_ref", "duckdb")

BUILD = """
SELECT count(CREATE_CSR_EDGE(0, (SELECT count(a.id) FROM v a),
         CAST((SELECT sum(CREATE_CSR_VERTEX(0, (SELECT count(a.id) FROM v a), sub.dense_id, sub.cnt))
               FROM (SELECT a.rowid AS dense_id, count(k.src) AS cnt FROM v a LEFT JOIN e k ON k.src = a.id
                     GROUP BY a.rowid) sub) AS BIGINT),
         (SELECT count(*) FROM e k JOIN v a ON a.id = k.src JOIN v c ON c.id = k.dst),
         a.rowid, c.rowid, k.rowid, k.w))
  FROM e k JOIN v a ON a.id = k.src JOIN v c ON c.id = k.dst;
"""
PLAIN_CTE = """
WITH cte1 AS (
  SELECT CREATE_CSR_EDGE(1, (SELECT count(a.id) FROM v a),
         CAST((SELECT sum(CREATE_CSR_VERTEX(1, (SELECT count(a.id) FROM v a), sub.dense_id, sub.cnt))
               FROM (SELECT a.rowid AS dense_id, count(k.src) AS cnt FROM v a LEFT JOIN e k ON k.src = a.id
                     GROUP BY a.rowid) sub) AS BIGINT),
         (SELECT count(*) FROM e k JOIN v a ON a.id = k.src JOIN v c ON c.id = k.dst),
         a.rowid, c.rowid, k.rowid) AS temp
  FROM e k JOIN v a ON a.id = k.src JOIN v c ON c.id = k.dst)
"""


def run_sql(sql: str) -> str:
    out = subprocess.run([DUCKDB, "-csv", "-noheader"], input=sql, capture_output=True, text=True)
    if out.returncode != 0 or "Error" in out.stderr:
        raise RuntimeError(out.stderr + out.stdout)
    return out.stdout


def save(name, n, src, dst, w, psrc, pdst, pdst_valid=None):
    src, dst, psrc, pdst = (np.asarray(x, dtype=np.int64) for x in (src, dst, psrc, pdst))
    w = np.asarray(w)
    is_f = w.dtype.kind == "f"
    P = len(psrc)
    with tempfile.TemporaryDirectory() as td:
        pq.write_table(pa.table({"id": np.arange(n, dtype=np.int64)}), f"{td}/v.parquet")
        pq.write_table(pa.table({"src": src, "dst": dst, "w": w.astype(np.float64 if is_f else np.int64)}), f"{td}/e.parquet")
        pdm = pa.array(pdst, mask=None if pdst_valid is None else ~pdst_valid.astype(bool))
        pq.write_table(pa.table({"i": np.arange(P, dtype=np.int64), "src": psrc, "dst": pdm}), f"{td}/p.parquet")
        sql = f"""
SET threads TO 1;
CREATE TABLE v AS SELECT * FROM read_parquet('{td}/v.parquet');
CREATE TABLE e AS SELECT * FROM read_parquet('{td}/e.parquet');
CREATE TABLE p AS SELECT * FROM read_parquet('{td}/p.parquet');
{BUILD}
.print ---T
SELECT csr_get_w_type(0);
.print ---V
SELECT csrv FROM get_csr_v(0);
.print ---E
SELECT csre FROM get_csr_e(0);
.print ---W
SELECT csrw FROM get_csr_w(0);
.print ---C
SELECT p.i, cheapest_path_length(0, (SELECT count(*) FROM v), p.src, p.dst) FROM p ORDER BY p.i;
.print ---L
{PLAIN_CTE} SELECT p.i, iterativelength2(1, (SELECT count(*) FROM v), p.src, p.dst) + __x.temp
  FROM p, (SELECT count(cte1.temp) * 0 AS temp FROM cte1) __x ORDER BY p.i;
"""
        txt = run_sql(sql)
    w_type = int(txt.split("---T\n")[1].split("---V\n")[0].strip())
    csr_v = np.array([int(x) for x in txt.split("---V\n")[1].split("---E\n")[0].split()], dtype=np.int64)
    csr_e = np.array([int(x) for x in txt.split("---E\n")[1].split("---W\n")[0].split()], dtype=np.int64)
    wpart = txt.split("---W\n")[1].split("---C\n")[0].split()
    cpart = txt.split("---C\n")[1].split("---L\n")[0]
    lpart = txt.split("---L\n")[1]
    csr_w = np.array([float(x) if is_f else int(x) for x in wpart], dtype=np.float64 if is_f else np.int64)
    cost = np.zeros(P, dtype=np.float64 if is_f else np.int64)
    cvalid = np.zeros(P, dtype=np.uint8)
    for r in csv.reader(io.StringIO(cpart)):
        if r[1] not in ("", "NULL"):
            cost[int(r[0])] = float(r[1]) if is_f else int(r[1])
            cvalid[int(r[0])] = 1
    l2 = np.full(P, -1, dtype=np.int64)
    l2v = np.zeros(P, dtype=np.uint8)
    for r in csv.reader(io.StringIO(lpart)):
        if r[1] not in ("", "NULL"):
            l2[int(r[0])] = int(r[1])
            l2v[int(r[0])] = 1
    out = os.path.join(HERE, f"refw_{name}.npz")
    np.savez_compressed(out, n=np.int64(n), src=src.astype(np.int32), dst=dst.astype(np.int32), w=w,
                        psrc=psrc.astype(np.int32), pdst=pdst.astype(np.int32),
                        pdst_valid=(np.ones(P, np.uint8) if pdst_valid is None else pdst_valid.astype(np.uint8)),
                        w_type=np.int64(w_type), csr_v=csr_v.astype(np.int32), csr_e=csr_e.astype(np.int32), csr_w=csr_w, cost=cost, cost_valid=cvalid, length2=l2.astype(np.int32),
                        length2_valid=l2v)
    print(f"{name}: n={n} m={len(src)} pairs={P} w_type={w_type} reachable={int(cvalid.sum())} -> {os.path.getsize(out)} bytes")


# weights of special_f64 that may sit on any edge: none of them lowers a cycle's cost.  -NaN is one of them:
# DuckDB keeps a NaN's sign (signbit(csrw) over get_csr_w is true for a -NaN weight, which prints as -nan).  The
# text output drops NaN payloads, so both NaNs are the canonical quiet ones.
SPECIAL_ANYWHERE = (np.inf, 1e308) + tuple(np.array([0x7FF8000000000000, 0xFFF8000000000000], np.uint64).view(np.float64))


def margin_weights(rng, n, src, dst, scale, f64):
    """forward edges (src < dst) get a weight in [-scale, scale], every backward or self edge n*scale+1 or more.
    A cycle has at least one backward edge, so every cycle costs more than zero: the reference (and the device)
    would relax a negative cycle forever."""
    lo = n * scale + 1
    if f64:
        return np.where(src < dst, rng.uniform(-scale, scale, len(src)), lo + rng.random(len(src)) * lo)
    return np.where(src < dst, rng.integers(-scale, scale + 1, len(src)), rng.integers(lo, 2 * lo, len(src)))


def unreached_part(rng, n, m, frac=0.35):
    """A multigraph whose part U (a random `frac` of the vertices) has no in-edge from outside it, so a source
    outside U reaches no vertex of U, plus one forward edge out of every U vertex but the last id (`extra`, to be
    weighted negative).  The reference relaxes every vertex in every sweep, also one still at max/2: a target in
    U then has the cost max/2 + (negative)."""
    in_u = rng.random(n) < frac
    src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
    into_u = ~in_u[src] & in_u[dst]
    src, dst = np.where(into_u, dst, src), np.where(into_u, src, dst)
    u = np.flatnonzero(in_u & (np.arange(n) < n - 1))
    extra = np.concatenate([np.zeros(m, bool), np.ones(len(u), bool)])
    return np.concatenate([src, u]), np.concatenate([dst, rng.integers(u + 1, n)]), in_u, extra


def neg_i64():
    rng = np.random.default_rng(101)
    n = 400
    src, dst, in_u, extra = unreached_part(rng, n, 2400)
    w = margin_weights(rng, n, src, dst, 1000, False)
    w[extra] = -rng.integers(1, 1001, extra.sum())
    ps = rng.choice(np.flatnonzero(~in_u), 300)
    pd = np.where(rng.random(300) < 0.4, rng.choice(np.flatnonzero(in_u), 300), rng.integers(0, n, 300))
    save("neg_i64", n, src, dst, w, ps, pd)


def neg_f64():
    # max/2 + (a weight of about 1) rounds back to max/2: a DOUBLE cost leaves the sentinel through a weight of
    # about -1e308 (max/2 - 1e308 = -1.0115e307).  Four more vertices without out-edges are the heads of such
    # edges out of U; the first two are reached from outside U as well, so -1e308 makes a reached target cheaper.
    rng = np.random.default_rng(102)
    n = 400
    src, dst, in_u, extra = unreached_part(rng, n, 2400)
    w = margin_weights(rng, n, src, dst, 1000, True)
    w[extra] = -rng.uniform(1, 1000, extra.sum())
    sinks = np.arange(n, n + 4)
    src = np.concatenate([src, rng.choice(np.flatnonzero(in_u), 4), rng.choice(np.flatnonzero(~in_u), 2)])
    dst = np.concatenate([dst, sinks, sinks[:2]])
    w = np.concatenate([w, -1e308 * (1 + 0.5 * rng.random(4)), rng.uniform(0, 1000, 2)])
    in_u = np.concatenate([in_u, [False, False, True, True]])
    ps = rng.choice(np.flatnonzero(~in_u), 300)
    pd = np.where(rng.random(300) < 0.4, rng.choice(np.flatnonzero(in_u), 300), rng.integers(0, n + 4, 300))
    pd[::15] = rng.choice(sinks, len(pd[::15]))
    save("neg_f64", n + 4, src, dst, w, ps, pd)


def special_f64():
    # +-inf, NaN, subnormals, +-0.0, 1e308 (sums overflow to inf), 1e16 next to weights of about 1 (the rounded
    # sum depends on the path).  Whatever could lower a cycle's cost (-inf, 0.0, -0.0, the subnormals) sits on
    # forward edges only; -inf only on edges into vertices without out-edges, or every cost would be -inf.
    rng = np.random.default_rng(103)
    n = 300
    src, dst = datagen.random_graph(n, 2400, seed=103)
    sinks = np.arange(n - 20, n)
    src, dst = src[src < n - 20], dst[src < n - 20]
    m = len(src)
    w = margin_weights(rng, n, src, dst, 1, True)
    fwd = np.flatnonzero(src < dst)
    for x in SPECIAL_ANYWHERE:
        w[rng.choice(m, m // 50, replace=False)] = x
    for x in (5e-324, 2.2250738585072009e-308, -5e-324, 0.0, -0.0, 1.0):
        w[rng.choice(fwd, m // 50, replace=False)] = x
    w[rng.choice(np.flatnonzero(np.isin(dst, sinks[:10])), 3, replace=False)] = -np.inf
    big = np.isin(dst, sinks[10:]) & ~np.isnan(w)
    w[big] = 1e16 + rng.uniform(-3, 3, big.sum())
    ps, pd = rng.integers(0, n, 300), rng.integers(0, n, 300)
    pd[::6] = rng.choice(sinks, len(pd[::6]))
    save("special_f64", n, src, dst, w, ps, pd)


def sentinel_i64():
    # max/2 = INT64_MAX/2.  From source 0, 1 costs max/2 - 1 (a cost), 2 max/2 (NULL: the sentinel itself), 3
    # max/2 + 1 (NULL: never stored); 5 / 6 / 7 the same over two edges; 9 / 10 / 11 the same from vertex 8, which
    # no source reaches (max/2 + -1, + 0, + 1).  Vertex 8 is no row's source: a source is relaxed for every lane.
    # Every sum stays inside int64 (max/2 + (max/2 + 1) = INT64_MAX).
    s = np.iinfo(np.int64).max // 2
    h = (s + 1) // 2
    w = np.array([s - 1, s, s + 1, h, s - 1 - h, s - h, s + 1 - h, -1, 0, 1], dtype=np.int64)
    src = [0, 0, 0, 0, 4, 4, 4, 8, 8, 8]
    dst = [1, 2, 3, 4, 5, 6, 7, 9, 10, 11]
    save("sentinel_i64", 12, src, dst, w, np.repeat([0, 4, 11], 12), np.tile(np.arange(12), 3))


def first_four():
    rng = np.random.default_rng(77)
    # the 6-vertex example of the raw-UDF form, parallel edges with different weights
    yield "tiny_i64", (6, [0, 1, 0, 2, 4, 0], [1, 2, 2, 3, 5, 1], np.array([5, 7, 20, 1, 2, 3]), [0, 0, 0, 4, 3, 1],
                       [2, 3, 5, 5, 0, 1])
    # random multigraph, integer weights, 700 pairs (batches 256 + 256 + 128 + 32 + 16 + 8 + 4).  No NULL targets:
    # the reference indexes dists[] with the value under the NULL (cheapest_path_length.cpp:95-96) and aborts
    n = 300
    src, dst = datagen.random_graph(n, 1500, seed=5)
    ps, pd = rng.integers(0, n, 700), rng.integers(0, n, 700)
    yield "rand300_i64", (n, src, dst, rng.integers(1, 100, len(src)), ps, pd)
    # double weights (sums depend on the path order -> the bit-exactness claim), R-MAT shape
    n, src, dst = datagen.rmat_edges(9, edge_factor=6)
    ps, pd = datagen.hashed_pairs(400, n)
    yield "rmat9_f64", (n, src, dst, rng.random(len(src)) * 10.0 + 0.001, ps, pd)
    # a chain with shortcuts: many relaxation sweeps
    n = 150
    src = np.concatenate([np.arange(0, 149), rng.integers(0, 150, 40)])
    dst = np.concatenate([np.arange(1, 150), rng.integers(0, 150, 40)])
    yield "chain150_f64", (n, src, dst, rng.random(len(src)) + 0.5, rng.integers(0, n, 200), rng.integers(0, n, 200))


# the first four share one random stream: they are made in order, and only the named ones are saved
FIRST_FOUR = ("tiny_i64", "rand300_i64", "rmat9_f64", "chain150_f64")
CASES = {"neg_i64": neg_i64, "neg_f64": neg_f64, "special_f64": special_f64, "sentinel_i64": sentinel_i64}


def main(names):
    unknown = set(names) - set(FIRST_FOUR) - set(CASES)
    if unknown:
        raise SystemExit(f"unknown case(s) {sorted(unknown)}; known: {list(FIRST_FOUR) + list(CASES)}")
    names = names or list(FIRST_FOUR) + list(CASES)
    if set(names) & set(FIRST_FOUR):
        for name, args in first_four():
            if name in names:
                save(name, *args)
    for name in names:
        if name in CASES:
            CASES[name]()


if __name__ == "__main__":
    main(sys.argv[1:])
