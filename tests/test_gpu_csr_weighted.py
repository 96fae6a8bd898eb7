"""The CSR-construction and weighted-path side of the C ABI: chunked / concurrent create_csr_edge feeding,
the BIGINT / DOUBLE weight overloads, cheapest_path_length -- against outputs of the reference binary
(tests/golden/refw_*.npz, made by tests/golden/make_golden_weighted.py) and the CPU restatement."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import GOLDEN
from duckpgq_extension_b200 import datagen, pgq
from oracle import pgq_oracle as orc

pytestmark = pytest.mark.gpu

WEIGHTED = sorted(f[5:-4] for f in os.listdir(GOLDEN) if f.startswith("refw_") and f.endswith(".npz"))


def load_weighted(name):
    z = np.load(os.path.join(GOLDEN, f"refw_{name}.npz"))
    g = {k: z[k] for k in z.files}
    for k in ("src", "dst", "psrc", "pdst", "length2"):
        g[k] = g[k].astype(np.int64)
    g["n"] = int(g["n"])
    return g


def build_chunked(ctx, n, src, dst, eid, weight=None, chunk=2048):
    """create_csr_vertex + create_csr_edge, DataChunk by DataChunk, as DuckDB would feed them."""
    csr = pgq.DeviceCSR.create(ctx, n)
    cnt = np.bincount(src, minlength=n).astype(np.int64)
    ids = np.arange(n, dtype=np.int64)
    total = 0
    for o in range(0, n, chunk):
        total += csr.add_vertex_counts(ids[o:o + chunk], cnt[o:o + chunk])
    m = len(src)
    assert total == m
    for o in range(0, m, chunk):
        csr.add_edges(m, m, src[o:o + chunk], dst[o:o + chunk], eid[o:o + chunk], None if weight is None else weight[o:o + chunk])
    csr.finalize()
    return csr


def per_vertex_sorted(v, e, w, n):
    """(edge, weight) pairs of every vertex in a canonical order: the order inside a vertex is the arrival order
    of the rows at create_csr_edge, which for the reference binary is DuckDB's join output order.  Weights as
    bits (int64 view), so that NaNs compare and -0.0 differs from 0.0."""
    row = np.repeat(np.arange(n), np.diff(np.asarray(v[:n + 1], dtype=np.int64)))
    wb = np.ascontiguousarray(w).view(np.int64)
    order = np.lexsort((wb, e, row))
    return np.asarray(e)[order], wb[order]


@pytest.mark.parametrize("name", WEIGHTED)
def test_weighted_csr_and_cheapest_path_golden(gpu_ctx, name):
    """get_csr_w / csr_get_w_type / cheapest_path_length / iterativelength2 of the reference binary."""
    g = load_weighted(name)
    n, src, dst, w = g["n"], g["src"], g["dst"], g["w"]
    eid = np.arange(len(src), dtype=np.int64)
    csr = build_chunked(gpu_ctx, n, src, dst, eid, w, chunk=97)
    assert csr.weight_type() == int(g["w_type"])
    got_w = csr.download_weights()
    dv, de, _ = csr.download()
    assert got_w.dtype == g["csr_w"].dtype and dv.tolist() == g["csr_v"].tolist()
    for a, b in zip(per_vertex_sorted(dv, de, got_w, n), per_vertex_sorted(g["csr_v"], g["csr_e"].astype(np.int64), g["csr_w"], n)):
        assert np.array_equal(a, b)  # bit-exact, doubles too
    cost, valid, st = csr.cheapest_path_length(g["psrc"], g["pdst"])
    assert np.array_equal(valid, g["cost_valid"])
    assert np.array_equal(cost[valid == 1].view(np.int64), g["cost"][valid == 1].view(np.int64))  # bits, also for DOUBLE sums
    # the restatement agrees with the reference binary as well (pins oracle/pgq_oracle.c's Bellman-Ford)
    v, e, ids, ow = orc.csr_build_weighted(n, src, dst, w)
    assert np.array_equal(ow.view(np.int64), got_w.view(np.int64)) and np.array_equal(e, de)  # device build == single-thread restatement, position by position, bits
    ocost, ovalid = orc.cheapest_path_length(n, v, e, ow, g["psrc"], g["pdst"])
    assert np.array_equal(ovalid, g["cost_valid"]) and np.array_equal(ocost[ovalid == 1].view(np.int64), g["cost"][ovalid == 1].view(np.int64))
    # iterativelength2 is served by the same searches as iterativelength
    out, ov, _ = csr.iterativelength(g["psrc"], g["pdst"])
    assert np.array_equal(ov, g["length2_valid"]) and np.array_equal(out, g["length2"])
    csr.free()


def test_cheapest_path_nulls_and_batches(gpu_ctx):
    """NULL sources / targets are NULL results (the reference mis-aligns / aborts there, DESIGN.md section 7); more
    rows than one 256-lane batch; parallel edges: the cheaper one counts."""
    rng = np.random.default_rng(3)
    n = 500
    src, dst = datagen.random_graph(n, 3000, seed=13)
    w = rng.integers(1, 50, len(src))
    v, e, ids, ow = orc.csr_build_weighted(n, src, dst, w)
    csr = build_chunked(gpu_ctx, n, src, dst, np.arange(len(src), dtype=np.int64), w)
    p = 1000
    ps, pd = rng.integers(0, n, p), rng.integers(0, n, p)
    sv = (rng.random(p) > 0.1).astype(np.uint8)
    dv = (rng.random(p) > 0.1).astype(np.uint8)
    cost, valid, st = csr.cheapest_path_length(ps, pd, sv, dv)
    ocost, ovalid = orc.cheapest_path_length(n, v, e, ow, ps, pd, sv, dv)
    assert np.array_equal(valid, ovalid) and np.array_equal(cost[valid == 1], ocost[ovalid == 1])
    assert not valid[(sv == 0) | (dv == 0)].any() and st["batches"] >= 4
    with pytest.raises(pgq.PgqError):  # no weights -> "Need to initialize CSR before doing cheapest path"
        plain = pgq.DeviceCSR.build(gpu_ctx, n, src, dst)
        try:
            plain.cheapest_path_length(ps, pd)
        finally:
            plain.free()
    csr.free()


def test_udf_mirror_weighted(gpu_ctx):
    """create_csr_edge's weight overload + cheapest_path_length through the Python mirror of the UDFs."""
    st = pgq.DuckPGQState(gpu_ctx)
    src = np.array([0, 1, 0, 2, 4, 0]); dst = np.array([1, 2, 2, 3, 5, 1]); w = np.array([5, 7, 20, 1, 2, 3])
    total = int(pgq.create_csr_vertex(st, 0, 6, np.arange(6), np.bincount(src, minlength=6)).sum())
    r = pgq.create_csr_edge(st, 0, 6, total, len(src), src, dst, np.arange(6), w)
    assert r.tolist() == w.tolist()  # (int32) weight, csr_creation.cpp:167
    cost, valid = pgq.cheapest_path_length(st, 0, 6, [0, 0, 0, 4, 3, 1], [2, 3, 5, 5, 0, 1])
    assert cost[valid == 1].tolist() == [10, 11, 2, 0] and valid.tolist() == [1, 1, 0, 1, 0, 1]
    st.query_end()
    assert 0 not in st.csr_list


def test_chunked_build_one_thread_is_the_reference_order(gpu_ctx):
    """>= 64 chunks fed by ONE thread in ticket order = the reference's single-thread CSR, bit for bit."""
    n, src, dst = datagen.rmat_edges(13)  # 131 072 edges = 128 chunks of 1024
    eid = np.random.default_rng(1).permutation(len(src)).astype(np.int64)
    v, e, ids = orc.csr_build(n, src, dst, eid)
    csr = build_chunked(gpu_ctx, n, src, dst, eid, chunk=1024)
    dv, de, dids = csr.download()
    assert np.array_equal(dv, v) and np.array_equal(de, e) and np.array_equal(dids, ids)
    csr.free()


def test_chunked_build_from_eight_threads(gpu_ctx):
    """create_csr_edge is ALWAYS called concurrently by DuckDB's worker threads (csr_creation.cpp:134 hands out
    atomic tickets): 8 threads x 64 chunks.  The offsets equal the reference's; every vertex's adjacency is a
    permutation of the reference's (edge, edge id) pairs; chunks keep their internal order."""
    n, src, dst = datagen.rmat_edges(14, edge_factor=8)  # 131 072 edges
    m = len(src)
    eid = np.arange(m, dtype=np.int64) * 5 + 3
    v, e, ids = orc.csr_build(n, src, dst, eid)
    csr = pgq.DeviceCSR.create(gpu_ctx, n)
    cnt = np.bincount(src, minlength=n).astype(np.int64)
    assert csr.add_vertex_counts(np.arange(n, dtype=np.int64), cnt) == m
    chunk = m // (8 * 64)
    chunks = [(o, min(m, o + chunk)) for o in range(0, m, chunk)]
    assert len(chunks) >= 8 * 64

    def feed(t):
        for lo, hi in chunks[t::8]:
            csr.add_edges(m, m, src[lo:hi], dst[lo:hi], eid[lo:hi])

    with ThreadPoolExecutor(max_workers=8) as pool:
        list(pool.map(feed, range(8)))
    csr.finalize()
    dv, de, dids = csr.download()
    assert np.array_equal(dv, v)
    key_ref = np.lexsort((ids, e, np.repeat(np.arange(n), np.diff(v[:n + 1]))))
    key_dev = np.lexsort((dids, de, np.repeat(np.arange(n), np.diff(dv[:n + 1]))))
    assert np.array_equal(e[key_ref], de[key_dev]) and np.array_equal(ids[key_ref], dids[key_dev])
    # searches over it give the reference's answers (hop counts do not depend on the adjacency order)
    ps, pd = datagen.hashed_pairs(500, n)
    exp, expv, _ = orc.iterativelength(n, v, e, ps, pd, None, 512)
    out, valid, _ = csr.iterativelength(ps, pd)
    assert np.array_equal(out, exp) and np.array_equal(valid, expv)
    csr.free()


def test_rowid_out_of_range_is_reported_at_finalize(gpu_ctx):
    csr = pgq.DeviceCSR.create(gpu_ctx, 4)
    csr.add_vertex_counts([0, 1, 2, 3], [1, 1, 0, 0])
    csr.add_edges(2, 2, [0, 1], [1, 7], [0, 1])  # asynchronous staging: accepted here ...
    with pytest.raises(pgq.InvalidInputException):
        csr.finalize()                           # ... reported here
    csr.free()


def test_csr_buffers_are_recycled(gpu_ctx):
    """DuckPGQ rebuilds a CSR of the same shape for every query: the second build takes its device buffers
    from the context's cache (same addresses are not observable through the ABI, equal results and a
    non-growing footprint are)."""
    n, src, dst = datagen.rmat_edges(12)
    ps, pd = datagen.hashed_pairs(300, n)
    base = None
    for _ in range(4):
        csr = pgq.DeviceCSR.build(gpu_ctx, n, src, dst)
        out, valid, _ = csr.iterativelength(ps, pd)
        if base is None:
            base = (out.copy(), valid.copy())
        assert np.array_equal(out, base[0]) and np.array_equal(valid, base[1])
        csr.free()
