"""Pins the CPU restatement (oracle/pgq_oracle.c) to the reference: (1) outputs of the reference
binary itself (tests/golden/ref_*.npz, made by tests/golden/make_golden.py with oracle/_ref/duckdb),
(2) known-answer vectors transcribed from the reference's own sqllogictests."""
import glob
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_names, load_golden
from oracle import pgq_oracle as orc


@pytest.mark.parametrize("name", golden_names())
def test_csr_build_matches_reference(name):
    g = load_golden(name)
    v, e, ids = orc.csr_build(g["n"], g["src"], g["dst"])
    assert v.tolist() == g["csr_v"].tolist()          # get_csr_v(0): n+2 entries
    assert e.tolist() == g["csr_e"].tolist()          # get_csr_e(0): single-thread arrival order
    assert sorted(ids.tolist()) == list(range(len(g["src"])))


@pytest.mark.parametrize("name", golden_names())
@pytest.mark.parametrize("lanes", [512, 64])
def test_iterativelength_matches_reference(name, lanes):
    g = load_golden(name)
    out, valid, st = orc.iterativelength(g["n"], g["csr_v"], g["csr_e"], g["psrc"], g["pdst"], g["psrc_valid"], lanes)
    assert valid.tolist() == g["length_valid"].tolist()
    assert out.tolist() == g["length"].tolist()
    assert st.batches >= 1 or len(g["psrc"]) == 0


@pytest.mark.parametrize("name", [n for n in golden_names() if load_golden(n)["has_paths"]])
def test_shortestpath_matches_reference(name):
    g = load_golden(name)
    _, _, ids = orc.csr_build(g["n"], g["src"], g["dst"])
    paths, _ = orc.shortestpath(g["n"], g["csr_v"], g["csr_e"], ids, g["psrc"], g["pdst"], g["psrc_valid"], 512)
    assert paths == g["paths"]


def test_kat_getpgschema_csr():
    # test/sql/scalar/getpgschema.test:20,86-106
    k = json.load(open(os.path.join(GOLDEN, "kat_reference_tests.json")))["getpgschema_csr"]
    v, e, _ = orc.csr_build(k["n"], k["src"], k["dst"])
    assert e.tolist() == k["get_csr_e"]
    assert v.tolist() == k["get_csr_v"]


def test_kat_shortest_path_test():
    # test/sql/path_finding/shortest_path.test:59-82 (all reachable pairs, {1,3})
    k = json.load(open(os.path.join(GOLDEN, "kat_reference_tests.json")))["shortest_path_any_shortest_1_3"]
    v, e, ids = orc.csr_build(k["n"], k["src"], k["dst"])
    ps = [r["src"] for r in k["rows"]]
    pd = [r["dst"] for r in k["rows"]]
    paths, _ = orc.shortestpath(k["n"], v, e, ids, ps, pd)
    lens, valid, _ = orc.iterativelength(k["n"], v, e, ps, pd)
    for r, path, ln, ok in zip(k["rows"], paths, lens, valid):
        assert ok and ln == r["path_length"]
        assert path == r["element_id"]


def test_kat_complex_matching_snb():
    # test/sql/path_finding/complex_matching.test:329-360: a.id = 16 (rowid 16), {1,3}, 26 element_id lists
    k = json.load(open(os.path.join(GOLDEN, "kat_reference_tests.json")))["complex_matching_snb_from_16"]
    g = load_golden("snb0003_allpairs")
    _, _, ids = orc.csr_build(g["n"], g["src"], g["dst"])
    n = g["n"]
    ps = np.full(n, k["src_rowid"], dtype=np.int64)
    pd = np.arange(n, dtype=np.int64)
    paths, _ = orc.shortestpath(n, g["csr_v"], g["csr_e"], ids, ps, pd)
    lens, valid, _ = orc.iterativelength(n, g["csr_v"], g["csr_e"], ps, pd)
    got = sorted(p for p, ln, ok in zip(paths, lens, valid) if ok and 1 <= ln <= 3)
    assert got == sorted(k["element_ids"])


def test_kat_shortest_path_raw_udf():
    # test/sql/path_finding/shortest_path.test:96-128: shortestpath() / iterativelength() called directly
    k = json.load(open(os.path.join(GOLDEN, "kat_reference_tests.json")))["shortest_path_raw_udf_from_daniel"]
    v, e, ids = orc.csr_build(k["n"], k["src"], k["dst"])
    pd = np.arange(k["n"], dtype=np.int64)
    ps = np.full(k["n"], k["src_rowid"], dtype=np.int64)
    paths, _ = orc.shortestpath(k["n"], v, e, ids, ps, pd)
    lens, valid, _ = orc.iterativelength(k["n"], v, e, ps, pd)
    got = {int(b): p for b, p, ln, ok in zip(pd, paths, lens, valid) if ok and k["lower"] <= ln <= k["upper"]}
    assert got == {r["dst"]: r["path"] for r in k["rows"]}


def test_kat_complex_matching_segments():
    # test/sql/path_finding/complex_matching.test:55-72: the {1,3} segment inside a longer pattern
    k = json.load(open(os.path.join(GOLDEN, "kat_reference_tests.json")))["complex_matching_snb_segments_from_9"]
    g = load_golden("snb0003_allpairs")
    _, _, ids = orc.csr_build(g["n"], g["src"], g["dst"])
    pd = np.array([seg[-1] for seg in k["segments"]], dtype=np.int64)
    ps = np.full(len(pd), k["src_rowid"], dtype=np.int64)
    paths, _ = orc.shortestpath(g["n"], g["csr_v"], g["csr_e"], ids, ps, pd)
    assert paths == k["segments"]


def test_kat_undirected_all_pairs():
    # test/sql/path_finding/undirected_paths.test:97-123: the undirected CSR is edges + reversed edges,
    # de-duplicated per (src, dst) (compressed_sparse_row.cpp:164-172); lower bound 0 -> src == dst gives 0
    k = json.load(open(os.path.join(GOLDEN, "kat_reference_tests.json")))["undirected_all_pairs_lengths"]
    both = sorted(set(zip(k["src"] + k["dst"], k["dst"] + k["src"])))
    v, e, _ = orc.csr_build(k["n"], [a for a, _ in both], [b for _, b in both])
    n = k["n"]
    ps = np.repeat(np.arange(n, dtype=np.int64), n)
    pd = np.tile(np.arange(n, dtype=np.int64), n)
    lens, valid, _ = orc.iterativelength(n, v, e, ps, pd)
    assert valid.all()
    assert lens.reshape(n, n).tolist() == k["path_length"]


def test_snb_c1_summary():
    # SURVEY.md section 6 / BASELINE.md: all 2500 Person pairs -> 375 reachable, sum 658, max 4
    g = load_golden("snb0003_allpairs")
    out, valid, st = orc.iterativelength(g["n"], g["csr_v"], g["csr_e"], g["psrc"], g["pdst"])
    assert int(valid.sum()) == 375 and int(out[valid == 1].sum()) == 658 and int(out.max()) == 4
    assert st.batches == 5  # 2450 searches (src == dst rows take no lane) in blocks of 512


def test_constraint_exception():
    # test/sql/path_finding/non-unique-vertices.test:40-81: sum(cnt) != count(*) -> ConstraintException
    with pytest.raises(orc.ConstraintError) as ei:
        orc.csr_build_stepwise(3, [0, 1, 2], [1, 1, 0], 3, [0, 1, 1], [1, 2, 0], [0, 1, 2])
    assert "Non-existent/non-unique vertices detected" in str(ei.value)


def test_work_counter_definition():
    # W = sum over levels of the out-degrees of the frontier vertices (SURVEY.md section 8d), including the
    # level that finds nothing new and the re-entry of a source that lies on a cycle.
    v, e, _ = orc.csr_build(3, [0, 1, 2], [1, 2, 0])  # 3-cycle
    out, valid, st = orc.iterativelength(3, v, e, [0], [2])
    assert out.tolist() == [2] and st.levels == 2 and st.edges_traversed == 2
    out, valid, st = orc.iterativelength(4, np.array([0, 1, 2, 3, 3, 3]), e, [0], [3])  # unreachable
    assert valid.tolist() == [0] and st.levels == 4 and st.edges_traversed == 4  # 0,1,2, then 0 again


# ---- the restatement's extensions, pinned to the reference binary as well ------------------------------------
WEIGHTED = sorted(f[5:-4] for f in os.listdir(GOLDEN) if f.startswith("refw_") and f.endswith(".npz"))


def per_vertex_sorted(v, e, w, n):
    """(edge, weight) pairs of every vertex in a canonical order: the order inside a vertex is the arrival order
    of the rows at create_csr_edge, which for the reference binary is DuckDB's join output order.  Weights as
    bits (int64 view), so that NaNs compare and -0.0 differs from 0.0."""
    row = np.repeat(np.arange(n), np.diff(np.asarray(v[:n + 1], dtype=np.int64)))
    wb = np.ascontiguousarray(w).view(np.int64)
    order = np.lexsort((wb, e, row))
    return np.asarray(e)[order], wb[order]


@pytest.mark.parametrize("name", WEIGHTED)
def test_weighted_csr_cheapest_path_and_iterativelength2_golden(name):
    """tests/golden/refw_*.npz = outputs of oracle/_ref/duckdb (make_golden_weighted.py): get_csr_w,
    cheapest_path_length (BIGINT and DOUBLE: exact equality) and iterativelength2."""
    z = np.load(os.path.join(GOLDEN, f"refw_{name}.npz"))
    n, src, dst, w = int(z["n"]), z["src"].astype(np.int64), z["dst"].astype(np.int64), z["w"]
    ps, pd = z["psrc"].astype(np.int64), z["pdst"].astype(np.int64)
    v, e, ids, ow = orc.csr_build_weighted(n, src, dst, w)
    assert ow.dtype == z["csr_w"].dtype and v.tolist() == z["csr_v"].tolist()
    for a, b in zip(per_vertex_sorted(v, e, ow, n), per_vertex_sorted(z["csr_v"], z["csr_e"].astype(np.int64), z["csr_w"], n)):
        assert np.array_equal(a, b)  # weights bit-exact, doubles too
    cost, valid = orc.cheapest_path_length(n, v, e, ow, ps, pd)
    assert np.array_equal(valid, z["cost_valid"]) and np.array_equal(cost[valid == 1].view(np.int64), z["cost"][valid == 1].view(np.int64))
    out, ov, _ = orc.iterativelength2(n, v, e, ps, pd)
    assert np.array_equal(ov, z["length2_valid"]) and np.array_equal(out, z["length2"].astype(np.int64))
    out1, ov1, _ = orc.iterativelength(n, v, e, ps, pd)  # the two formulations answer alike
    assert np.array_equal(out, out1) and np.array_equal(ov, ov1)


@pytest.mark.parametrize("name", ["rmat10", "rand40_nulls", "chain200", "snb0003_allpairs"])
def test_extended_batch_compositions_keep_the_answers(name):
    """orc_iterativelength_ex: with no flag it IS orc_iterativelength (results and counters); the degree
    shortcut, one lane per distinct source and the OpenMP level loop never change an answer, and the OpenMP
    loop never changes a counter."""
    g = load_golden(name)
    n, v, e, ps, pd, sv = g["n"], g["csr_v"], g["csr_e"], g["psrc"], g["pdst"], g["psrc_valid"]
    for lanes in (64, 512):
        base, bvalid, bst = orc.iterativelength(n, v, e, ps, pd, sv, lanes)
        assert base.tolist() == g["length"].tolist()
        out, valid, st, used = orc.iterativelength_ex(n, v, e, ps, pd, sv, lanes)
        assert np.array_equal(out, base) and np.array_equal(valid, bvalid) and st == bst
        out, valid, st, _ = orc.iterativelength_ex(n, v, e, ps, pd, sv, lanes, omp=True)
        assert np.array_equal(out, base) and np.array_equal(valid, bvalid) and st == bst
        for prune, dedup in ((True, False), (False, True), (True, True)):
            out, valid, st, used = orc.iterativelength_ex(n, v, e, ps, pd, sv, lanes, prune=prune, dedup=dedup)
            assert np.array_equal(out, base) and np.array_equal(valid, bvalid), (prune, dedup)
            out2, _, st2, used2 = orc.iterativelength_ex(n, v, e, ps, pd, sv, lanes, prune=prune, dedup=dedup, omp=True)
            assert np.array_equal(out2, base) and st2 == st and used2 == used
            assert st.edges_traversed <= bst.edges_traversed or dedup  # (fewer, wider lanes can regroup the batches)


def test_one_lane_per_distinct_source_definition():
    # 3 sources x 4 destinations in join order; lanes numbered by first appearance: 2 -> 0, 0 -> 1, 1 -> 2
    v, e, _ = orc.csr_build(5, [0, 1, 2, 3], [1, 2, 3, 4])  # a chain
    ps = np.array([2, 0, 2, 1, 0, 1, 2, 0, 1, 2, 0, 1])
    pd = np.array([3, 1, 4, 2, 4, 0, 2, 0, 4, 0, 3, 1])
    out, valid, st, used = orc.iterativelength_ex(5, v, e, ps, pd, None, 64, dedup=True)
    ref, refv, rst = orc.iterativelength(5, v, e, ps, pd, None, 64)
    assert np.array_equal(out, ref) and np.array_equal(valid, refv)
    assert used == 3 and st.batches == 1 and rst.batches == 1
    # W: the three lanes' frontiers are {2,0,1} -> {3,1,2} -> {4,2,3} -> {3,4} -> {4}: out-degrees 3+3+2+1+0
    # (W counts frontier VERTICES, so 12 lanes sharing these frontiers inside one batch cost the same 9 ...
    assert st.edges_traversed == 9 and rst.edges_traversed == 9
    # ... and the saving shows up as soon as the rows no longer fit one batch: 130 rows, 18 of them src == dst = 2 batches vs 1)
    ps2, pd2 = np.tile(ps, 11)[:130], np.tile(pd, 11)[:130]
    _, _, st2, used2 = orc.iterativelength_ex(5, v, e, ps2, pd2, None, 64, dedup=True)
    _, _, rst2 = orc.iterativelength(5, v, e, ps2, pd2, None, 64)
    assert used2 == 3 and st2.batches == 1 and rst2.batches == 2 and rst2.edges_traversed == 2 * st2.edges_traversed


# ---- SURVEY section 8f NEXT-4: the checkers of the reference's other CSR consumers, pinned to the reference binary
# (tests/golden/make_golden_next4.py); nothing on the device computes these yet.
NEXT4 = sorted(glob.glob(os.path.join(GOLDEN, "refn4_*.npz")))


@pytest.mark.parametrize("path", NEXT4, ids=[os.path.basename(p)[6:-4] for p in NEXT4])
def test_next4_restatements_match_reference(path):
    g = np.load(path)
    n = int(g["n"])
    v, e = g["csr_v"].astype(np.int64), g["csr_e"].astype(np.int64)
    assert len(v) == n + 2  # CSR::vsize = n + 2 (csr_creation.cpp:30)
    ids = np.arange(n)
    lcc, lv = orc.local_clustering_coefficient(n, v, e, ids)
    assert lv.all() and np.array_equal(lcc.view(np.uint32), g["lcc"].view(np.uint32))  # FLOAT, bit for bit
    wcc, wv = orc.weakly_connected_component(n, v, e, ids)
    assert wv.all() and np.array_equal(wcc, g["wcc"])  # the reference's component LABELS, not just the partition
    pr, pv, iters = orc.pagerank(n, v, e, ids)
    assert pv.all() and np.array_equal(pr, g["pagerank"]) and iters > 0  # DOUBLE, bit for bit (same summation order)


def test_next4_edge_cases():
    v, e, _ = orc.csr_build(4, [0, 1], [1, 0])
    lcc, lv = orc.local_clustering_coefficient(4, v, e, [0, 3, 2], [1, 1, 0])
    assert lcc.tolist() == [0.0, 0.0, 0.0] and lv.tolist() == [1, 1, 0]  # degree < 2 -> 0; NULL source -> NULL
    wcc, wv = orc.weakly_connected_component(4, v, e, [0, 1, 2, 3, 4, 7, -1])
    assert wcc[:5].tolist() == [1, 1, 2, 3, 4] and wv.tolist() == [1, 1, 1, 1, 1, 0, 0]  # root(0) hangs under root(1)
    pr, pv, _ = orc.pagerank(4, v, e, [0, 1, 2, 5, 6], [1, 1, 1, 1, 1])
    assert pv.tolist() == [1, 1, 1, 1, 0] and pr[0] == pr[1] and pr[2] == pr[3]  # ids < vsize = n + 2 are answered
