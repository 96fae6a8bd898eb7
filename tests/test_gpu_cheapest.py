"""cheapest_path_length (pgq_cheapest.cu) against the CPU restatement of the reference's batched Bellman-Ford
(oracle/pgq_oracle.c), at the edges where a parallel relaxation can part from a sequential one: negative weights
out of vertices no source reaches, infinities and NaNs, costs next to the "unreachable" sentinel max/2, row counts
around the lane width, lane counts picked from the vertex count, hubs, and a weighted CSR fed by many threads.
Every comparison is exact: the valid masks, and the cost bits (doubles viewed as int64, so -0.0 / +0.0 and the
infinities count).

Graphs with negative weights use a margin construction: an edge u -> v with u < v ("forward") gets a weight in
[-scale, scale], every other edge (backward or self) at least n * scale + 1.  A cycle has at least one backward
edge, so every cycle costs more than zero and the relaxation ends.  The oracle always runs first: were a graph to
hold a cycle that keeps lowering a cost in rounded arithmetic, the CPU would spin, not the GPU."""
import itertools
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from duckpgq_extension_b200 import datagen, pgq
from oracle import pgq_oracle as orc
from test_gpu_csr_weighted import build_chunked

pytestmark = pytest.mark.gpu

SENT_I64 = np.iinfo(np.int64).max // 2   # the reference's "unreachable": INT64_MAX / 2
SENT_F64 = np.finfo(np.float64).max / 2  # DBL_MAX / 2


def f64_bits(*bits):
    return np.array(bits, dtype=np.uint64).view(np.float64)


POS_NAN, NEG_NAN, NEG_NAN_PAYLOAD = f64_bits(0x7FF8000000000000, 0xFFF8000000000000, 0xFFF0000000000123)


def margin_weights(rng, n, src, dst, dtype, scale):
    """forward (src < dst) weights in [-scale, scale], backward and self edges in [n*scale+1, 2*n*scale+1]"""
    lo = n * scale + 1
    if np.dtype(dtype).kind == "f":
        fwd = rng.uniform(-scale, scale, len(src))
        back = lo + rng.random(len(src)) * lo
    else:
        fwd = rng.integers(-scale, scale + 1, len(src))
        back = rng.integers(lo, 2 * lo, len(src))
    return np.where(src < dst, fwd, back).astype(dtype)


def weighted_csr(ctx, n, src, dst, w, chunk=4096):
    """device CSR (create_csr_edge chunks, one thread) + the oracle's CSR of the same rows"""
    src, dst = np.asarray(src, np.int64), np.asarray(dst, np.int64)
    csr = build_chunked(ctx, n, src, dst, np.arange(len(src), dtype=np.int64), w, chunk=chunk)
    v, e, _, ow = orc.csr_build_weighted(n, src, dst, w)
    return csr, v, e, ow


def assert_same(cost, valid, ocost, ovalid):
    bad = np.flatnonzero(valid != ovalid)
    assert bad.size == 0, f"valid differs at rows {bad[:8].tolist()}: device {valid[bad[:8]].tolist()}, " \
                          f"oracle {ovalid[bad[:8]].tolist()}, device cost {cost[bad[:8]].tolist()}"
    m = valid == 1
    a, b = cost[m].view(np.int64), ocost[m].view(np.int64)
    bad = np.flatnonzero(a != b)
    assert bad.size == 0, f"{bad.size} costs differ, e.g. device {cost[m][bad[:8]].tolist()} oracle {ocost[m][bad[:8]].tolist()}"


def check(csr, n, v, e, ow, ps, pd, sv=None, dv=None):
    ocost, ovalid = orc.cheapest_path_length(n, v, e, ow, ps, pd, sv, dv)
    cost, valid, st = csr.cheapest_path_length(ps, pd, sv, dv)
    assert_same(cost, valid, ocost, ovalid)
    return cost, valid, st


# ---- 1. negative weights out of vertices no source reaches --------------------------------------------------------

def unreached_part_graph(rng, n, m, dtype, scale, frac=0.35):
    """A multigraph with a part U (a random `frac` of the vertices) that has no in-edge from outside U, so no source
    outside U reaches it; every U vertex but the last id has a negative out-edge (to anywhere above it)."""
    in_u = rng.random(n) < frac
    src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
    into_u = ~in_u[src] & in_u[dst]
    src, dst = np.where(into_u, dst, src), np.where(into_u, src, dst)  # R -> U edges turned round: U -> R
    u = np.flatnonzero(in_u & (np.arange(n) < n - 1))
    usrc, udst = u, rng.integers(u + 1, n)
    w = margin_weights(rng, n, src, dst, dtype, scale)
    uw = -(rng.integers(1, scale + 1, len(u)) if np.dtype(dtype).kind == "i" else rng.uniform(0.01, 1, len(u)) * scale)
    src, dst, w = np.concatenate([src, usrc]), np.concatenate([dst, udst]), np.concatenate([w, uw.astype(dtype)])
    assert not (~in_u[src] & in_u[dst]).any() and in_u.mean() >= 0.3
    return src, dst, w, in_u


@pytest.mark.parametrize("dtype", [np.int64, np.float64])
def test_negative_weights_out_of_unreached_vertices(gpu_ctx, dtype):
    """The reference relaxes every vertex in every sweep, also one still at max/2: a target no source reaches gets
    max/2 + (negative) -- a valid cost -- and with DOUBLE weights of about -1e308 even reached targets get
    cheaper.  5 000 vertices, 40 000 edges, 700 rows (three batches)."""
    rng = np.random.default_rng(11 if dtype is np.int64 else 12)
    n = 5000
    src, dst, w, in_u = unreached_part_graph(rng, n, 40000 - 1800, dtype, 1000)
    sinks = np.arange(n, n + 6)
    if dtype is np.float64:
        # max/2 + w(small) rounds back to max/2: DOUBLE costs leave the sentinel through weights of about -1e308
        # (max/2 - 1e308 = -1.0115e307).  Six more vertices without out-edges, each at the head of such an edge
        # out of U; the first three are also reached from outside U.
        tails = rng.choice(np.flatnonzero(in_u), 6)
        heads = rng.choice(np.flatnonzero(~in_u), 3)
        src = np.concatenate([src, tails, heads])
        dst = np.concatenate([dst, sinks, sinks[:3]])
        w = np.concatenate([w, -1e308 * (1 + 0.5 * rng.random(6)), rng.uniform(0, 1000, 3)])
        n += 6
        in_u = np.concatenate([in_u, [False] * 3 + [True] * 3])
    csr, v, e, ow = weighted_csr(gpu_ctx, n, src, dst, w)
    p = 700
    ps = rng.choice(np.flatnonzero(~in_u), p)
    pd = np.where(rng.random(p) < 0.4, rng.choice(np.flatnonzero(in_u), p), rng.integers(0, n, p))
    if dtype is np.float64:
        pd[::20] = rng.choice(sinks, len(pd[::20]))
    cost, valid, st = check(csr, n, v, e, ow, ps, pd)
    assert st["lanes"] == 256 and st["batches"] == 3
    # the cases exist: targets in U (which no source reaches) with a cost ...
    assert valid[in_u[pd]].sum() > (50 if dtype is np.int64 else 5)
    if dtype is np.float64:  # ... and reached targets that max/2 - 1e308 makes cheaper
        assert (valid[np.isin(pd, sinks[:3])] == 1).all() and (cost[np.isin(pd, sinks[:3])] < -1e306).all()
    csr.free()


# ---- 2. infinities, NaNs, subnormals, signed zeros, overflow -------------------------------------------------------

def test_special_doubles(gpu_ctx):
    """+-inf, +NaN, -NaN (two bit patterns: the C ABI takes any double), subnormals, +-0.0, 1e308 (sums overflow
    to inf) and 1e16 next to weights of about 1 (rounded sums depend on the path), ~1 % each.  A NaN never
    lowers a cost (NaN < x is false); max/2 + (-inf) = -inf is a cost."""
    rng = np.random.default_rng(21)
    n = 2000
    src, dst = datagen.random_graph(n, 16000, seed=21)
    sinks = np.arange(n - 20, n)  # no out-edges: a -inf into them goes no further
    src, dst = src[src < n - 20], dst[src < n - 20]
    m = len(src)
    w = margin_weights(rng, n, src, dst, np.float64, 1)
    fwd = np.flatnonzero(src < dst)
    anywhere = [np.inf, POS_NAN, NEG_NAN, NEG_NAN_PAYLOAD, 1e308]  # none of these lowers a cycle's cost
    forward_only = [5e-324, 2.2250738585072009e-308, -5e-324, 0.0, -0.0, 1e16, 3e16]
    for x in anywhere:
        w[rng.choice(m, m // 100, replace=False)] = x
    for x in forward_only:
        w[rng.choice(fwd, m // 100, replace=False)] = x
    w[rng.choice(np.flatnonzero(np.isin(dst, sinks[:10])), 5, replace=False)] = -np.inf
    big = np.isin(dst, sinks[10:]) & ~np.isnan(w)  # reached through 1e16 only: 1e16 + (a sum of about 1s), rounded
    w[big] = 1e16 + rng.uniform(-3, 3, big.sum())
    assert np.signbit(w[np.isnan(w)]).any()
    csr, v, e, ow = weighted_csr(gpu_ctx, n, src, dst, w, chunk=1000)
    assert np.array_equal(csr.download_weights().view(np.int64), ow.view(np.int64))  # NaN payloads and signs kept
    ps, pd = rng.integers(0, n, 600), rng.integers(0, n, 600)
    pd[::10] = rng.choice(sinks, 60)
    cost, valid, _ = check(csr, n, v, e, ow, ps, pd)
    c = cost[valid == 1]
    assert not np.isnan(c).any() and np.isinf(c).any() and (np.abs(c[np.isfinite(c)]) > 1e15).any()
    # every source at the head of a NaN edge: its own NaN must not reach the neighbour
    k = np.flatnonzero(np.isnan(w) & (src != dst))[:256]
    check(csr, n, v, e, ow, src[k], dst[k])
    csr.free()


# ---- 3. costs just below, at and above the sentinel ----------------------------------------------------------------

@pytest.mark.parametrize("dtype", [np.int64, np.float64])
def test_sentinel_crossing(gpu_ctx, dtype):
    """A cost of max/2 is "unreachable" (NULL), one above is never stored (NULL), one below is a cost -- whether
    it comes from a source or from a vertex still at max/2 with a negative out-edge (8 -> 9).  Vertex 8 is no
    row's source in the first call: a source is relaxed for all lanes of its batch."""
    if dtype is np.int64:
        s = SENT_I64
        below, at, above, half = s - 1, s, s + 1, (s + 1) // 2
        w = [below, at, above, half, below - half, at - half, above - half, -1, 0, 1]
    else:
        s = SENT_F64
        below, at, above, half = np.nextafter(s, 0), s, np.nextafter(s, np.inf), s / 2
        w = [below, at, above, half, np.nextafter(half, 0), half, np.nextafter(half, np.inf), below - s, -0.0, 0.0]
    src = [0, 0, 0, 0, 4, 4, 4, 8, 8, 8]
    dst = [1, 2, 3, 4, 5, 6, 7, 9, 10, 11]
    n = 12
    csr, v, e, ow = weighted_csr(gpu_ctx, n, src, dst, np.array(w, dtype=dtype))
    cost, valid, _ = check(csr, n, v, e, ow, np.repeat([0, 11], n), np.tile(np.arange(n), 2))
    got = {t: (cost[t].item() if valid[t] else None) for t in range(n)}  # rows of source 0
    assert got[1] == below and got[2] is None and got[3] is None
    assert got[6] is None and got[9] == below and got[10] is None and got[11] is None
    check(csr, n, v, e, ow, np.repeat([8, 4], n), np.tile(np.arange(n), 2))
    csr.free()


# ---- 4. row counts around the lane width ---------------------------------------------------------------------------

@pytest.mark.parametrize("p", [1, 31, 32, 33, 255, 256, 257, 513])
def test_rows_around_the_lane_width(gpu_ctx, p):
    """lanes = rows rounded up to 32, at most 256; more rows take more batches.  The first batch's source (0, the
    head of a chain) reaches every chain vertex, later batches' source (699, no out-edges) only itself: a
    distance or dirty array carried over from the first batch shows up as costs where there are none."""
    rng = np.random.default_rng(40 + p)
    n = 700
    rs, rd = datagen.random_graph(n, 2500, seed=p)
    keep = rs != n - 1
    src = np.concatenate([np.arange(599), rs[keep]])
    dst = np.concatenate([np.arange(1, 600), rd[keep]])
    lanes = min(256, (p + 31) // 32 * 32)
    ps = np.where(np.arange(p) < lanes, 0, n - 1)
    pd = rng.integers(0, n, p)
    pd[-1] = n - 1
    for w in (rng.integers(0, 100, len(src)), margin_weights(rng, n, src, dst, np.float64, 10)):
        csr, v, e, ow = weighted_csr(gpu_ctx, n, src, dst, w)
        cost, valid, st = check(csr, n, v, e, ow, ps, pd)
        assert st["lanes"] == lanes and st["batches"] == -(-p // lanes)
        later = np.arange(p) >= lanes
        assert not valid[later & (pd != n - 1)].any()
        csr.free()


# ---- 5. lanes picked from the vertex count -------------------------------------------------------------------------

@pytest.mark.parametrize("n,lanes", [(1 << 20, 256), ((1 << 20) + 1, 128), ((1 << 21) + 1, 64), ((1 << 22) + 1, 32)])
def test_lanes_from_the_vertex_count(gpu_ctx, n, lanes):
    """The distance array (n x lanes x 8 bytes) may take 2 GiB: at n = 2^20 256 lanes fit exactly, one vertex
    more halves them.  ~256 k edges spread over the whole id range plus an ascending chain of 3 000 vertices that
    ends at the last id; the oracle runs 64 rows at a time (n x 64 x 8 bytes of host memory)."""
    rng = np.random.default_rng(n)
    chain = np.unique(np.concatenate([rng.integers(0, n, 3000), [n - 1]]))
    rs, rd = rng.integers(0, n, 256_000), rng.integers(0, n, 256_000)
    src, dst = np.concatenate([chain[:-1], rs]), np.concatenate([chain[1:], rd])
    w = rng.integers(0, 1000, len(src))
    csr, v, e, ow = weighted_csr(gpu_ctx, n, src, dst, w, chunk=65536)
    p = 256
    ps = np.concatenate([rng.choice(chain[:100], 3 * p // 4), rs[: p // 4]])
    pd = np.where(rng.random(p) < 0.7, rng.choice(chain, p), rng.integers(0, n, p))
    pd[:8] = n - 1
    parts = [orc.cheapest_path_length(n, v, e, ow, ps[o:o + 64], pd[o:o + 64]) for o in range(0, p, 64)]
    ocost, ovalid = np.concatenate([c for c, _ in parts]), np.concatenate([x for _, x in parts])
    cost, valid, st = csr.cheapest_path_length(ps, pd)
    assert_same(cost, valid, ocost, ovalid)
    assert st["lanes"] == lanes and st["batches"] == p // lanes
    assert valid.sum() > p // 3
    csr.free()


# ---- 6. a hub, parallel edges, an in-star ---------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", [np.int64, np.float64])
def test_hub_parallel_edges_and_in_star(gpu_ctx, dtype):
    """Vertex 0 has 2^18 distinct out-neighbours and 1 000 parallel edges to one target (the cheapest counts);
    2^17 of the neighbours point at one sink, so one sweep has as many warps atomicMin the same slot."""
    rng = np.random.default_rng(60)
    leaves = np.arange(1, (1 << 18) + 1)
    sink, target = (1 << 18) + 1, (1 << 18) + 2
    n = target + 1
    star = leaves[: 1 << 17]
    src = np.concatenate([np.zeros(len(leaves), np.int64), star, np.zeros(1000, np.int64)])
    dst = np.concatenate([leaves, np.full(len(star), sink), np.full(1000, target)])
    if dtype is np.int64:
        w = rng.integers(1000, 1 << 40, len(src))
    else:
        w = rng.uniform(1.0, 1e6, len(src))
    w = w.astype(dtype)
    csr, v, e, ow = weighted_csr(gpu_ctx, n, src, dst, w, chunk=2048)
    p = 64
    ps = np.zeros(p, np.int64)
    ps[32:] = rng.choice(star, 32)
    pd = np.where(np.arange(p) % 3 == 0, sink, np.where(np.arange(p) % 3 == 1, target, rng.choice(leaves, p)))
    cost, valid, _ = check(csr, n, v, e, ow, ps, pd)
    hub_sink = np.min(w[: len(star)] + w[len(leaves):len(leaves) + len(star)])  # the same IEEE sums as the relaxation
    assert cost[0] == hub_sink and valid[0] == 1
    assert cost[1] == w[-1000:].min() and valid[1] == 1
    csr.free()


# ---- 7. a weighted CSR fed from 8 threads -----------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", [np.int64, np.float64])
def test_weighted_chunked_build_from_eight_threads(gpu_ctx, dtype):
    """8 threads x 64 create_csr_edge chunks with weights, in whatever ticket order: every vertex's (neighbour,
    edge id, weight) multiset is the reference's, so a weight stays with its edge; the costs over that CSR are
    the reference's (the fixed point does not depend on the order of a vertex's edges)."""
    rng = np.random.default_rng(70)
    n, src, dst = datagen.rmat_edges(14, edge_factor=8)
    m = len(src)
    eid = np.arange(m, dtype=np.int64) * 5 + 3
    w = margin_weights(rng, n, src, dst, dtype, 100)
    v, e, ids, ow = orc.csr_build_weighted(n, src, dst, w, eid)
    csr = pgq.DeviceCSR.create(gpu_ctx, n)
    assert csr.add_vertex_counts(np.arange(n, dtype=np.int64), np.bincount(src, minlength=n)) == m
    chunk = m // (8 * 64)
    chunks = [(o, min(m, o + chunk)) for o in range(0, m, chunk)]
    assert len(chunks) >= 8 * 64

    def feed(t):
        for lo, hi in chunks[t::8]:
            csr.add_edges(m, m, src[lo:hi], dst[lo:hi], eid[lo:hi], w[lo:hi])

    with ThreadPoolExecutor(max_workers=8) as pool:
        list(pool.map(feed, range(8)))
    csr.finalize()
    dv, de, dids = csr.download()
    dw = csr.download_weights()
    assert np.array_equal(dv, v) and dw.dtype == ow.dtype
    rows = np.repeat(np.arange(n), np.diff(v[:n + 1]))
    key_ref = np.lexsort((ow.view(np.int64), ids, e, rows))
    key_dev = np.lexsort((dw.view(np.int64), dids, de, rows))
    assert np.array_equal(e[key_ref], de[key_dev]) and np.array_equal(ids[key_ref], dids[key_dev])
    assert np.array_equal(ow[key_ref].view(np.int64), dw[key_dev].view(np.int64))
    ps, pd = datagen.hashed_pairs(300, n)
    check(csr, n, v, e, ow, ps, pd)
    csr.free()


# ---- 8. concurrent calls on one CSR -------------------------------------------------------------------------------------

def test_concurrent_cheapest_and_iterativelength(gpu_ctx):
    """8 threads call cheapest_path_length and iterativelength in turn on one weighted CSR, with row counts that
    reserve the shared workspace slots at different sizes: every answer is the reference's, and a call repeated
    gives the same bits."""
    rng = np.random.default_rng(80)
    n = 3000
    src, dst = datagen.random_graph(n, 20000, seed=80)
    w = margin_weights(rng, n, src, dst, np.float64, 50)
    csr, v, e, ow = weighted_csr(gpu_ctx, n, src, dst, w)
    P = 700
    ps, pd = rng.integers(0, n, P), rng.integers(0, n, P)
    ocost, ovalid = orc.cheapest_path_length(n, v, e, ow, ps, pd)
    olen, olv, _ = orc.iterativelength(n, v, e, ps, pd, None, 512)
    sizes = [700, 33, 300, 1, 513]

    def work(t):
        for i in range(6):
            k = sizes[(t + i) % len(sizes)]
            if (t + i) % 2:
                a = csr.cheapest_path_length(ps[:k], pd[:k])
                b = csr.cheapest_path_length(ps[:k], pd[:k])
                assert_same(a[0], a[1], ocost[:k], ovalid[:k])
                assert np.array_equal(a[0].view(np.int64), b[0].view(np.int64)) and np.array_equal(a[1], b[1])
            else:
                out, ov, _ = csr.iterativelength(ps[:k], pd[:k])
                assert np.array_equal(out, olen[:k]) and np.array_equal(ov, olv[:k])

    with ThreadPoolExecutor(max_workers=8) as pool:
        list(pool.map(work, range(8)))
    csr.free()


# ---- 9. errors ----------------------------------------------------------------------------------------------------------

def test_ids_out_of_range_and_empty_input(gpu_ctx):
    """A source or target outside [0, n) is an InvalidInputException; under a NULL mask the same ids are NULL rows;
    no rows give no rows; the CSR answers correctly after an error."""
    rng = np.random.default_rng(90)
    n = 50
    src, dst = datagen.random_graph(n, 300, seed=90)
    w = margin_weights(rng, n, src, dst, np.int64, 5)
    csr, v, e, ow = weighted_csr(gpu_ctx, n, src, dst, w)
    ps, pd = rng.integers(0, n, 40), rng.integers(0, n, 40)
    for bad, col in itertools.product([-1, n, 1 << 40], ["src", "dst"]):
        s, d = ps.copy(), pd.copy()
        (s if col == "src" else d)[17] = bad
        with pytest.raises(pgq.InvalidInputException):
            csr.cheapest_path_length(s, d)
        mask = np.ones(40, np.uint8)
        mask[17] = 0
        sv, dv = (mask, None) if col == "src" else (None, mask)
        _, valid, _ = check(csr, n, v, e, ow, s, d, sv, dv)
        assert valid[17] == 0
    cost, valid, st = csr.cheapest_path_length(np.zeros(0, np.int64), np.zeros(0, np.int64))
    assert cost.shape == (0,) and valid.shape == (0,) and st["batches"] == 0
    check(csr, n, v, e, ow, ps, pd)
    csr.free()
