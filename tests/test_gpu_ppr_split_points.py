"""Batched personalized PageRank and its per-seed top-K where their kernels split the work.

The step kernel of ppr_core.cuh runs persistent CTAs over merge-path tiles of kBT * kBIPT items, and rows that stay
open at a tile end are finished by ppr_fixup_kernel, 256 tiles per block.  The top-K of ppr_topk.cu scans its tie
counts in passes of kSel * kTiePer blocks of kTieChunk nodes, so a second pass (and the count carried into it) only
exists past (kSel * kTiePer)^2 = 2^24 nodes.  Tests at small sizes never reach these splits.

- Geometry (no GPU): the constants are read from the sources; numpy mirrors of diagonal_search_global and
  dev::order_key are checked against a plain merge-path walk and against the float order.
- Graph T: a chosen in-degree sequence whose partition holds a row ending on a tile's last item, a row starting on a
  tile's first item, two rows covering 3 or more whole tiles (one open across tiles 255 and 256, the first two fix-up
  blocks), a tile without non-zeros, a partial last tile and more than 8 tiles per SM.  Every batch column is within
  L1 1e-6 of orc_personalized, and every top-K row is the top of its dense column bit for bit.
- Graph S: 2^24 + 4099 nodes, seeds without edges and one ring of all other nodes, so each row's top is known from
  the construction; the ties that fill it lie on both sides of node 2^24.
- Non-finite ranks: pagerank_top_k_device orders +-NaN, +-Inf, +-0 and subnormals by dev::order_key (then id), and
  so does the batch top-K on a graph whose ranks mix NaN and finite values."""
import functools
import os
import re
import time

import numpy as np
import pytest

from test_gpu_pagerank_batch import _columns, _device_graph
from test_gpu_pagerank_personalized import _sass_summary, graph, orc_personalized
from test_gpu_ppr_topk import _assert_row

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gpu-spmv_b200", "csrc")
LIBDIR = os.path.join(ROOT, "gpu-spmv_b200", "lib")
D = 0.85
B200_SMS = 148


# ---------------------------------------------------------------------------------------------- geometry ----
def _constant(source, name):
    text = open(os.path.join(CSRC, source)).read()
    m = re.search(rf"\bconstexpr\s+int\s+{name}\s*=\s*(\d+)\s*;", text)
    assert m, f"constexpr int {name} not found in {source}"
    return int(m.group(1))


@functools.lru_cache(maxsize=None)
def _geometry():
    g = {"kBT": _constant("ppr_core.cuh", "kBT"), "kBIPT": _constant("ppr_core.cuh", "kBIPT"),
         "kSel": _constant("ppr_topk.cu", "kSel"), "kTiePer": _constant("ppr_topk.cu", "kTiePer")}
    g["tile"] = g["kBT"] * g["kBIPT"]            # merge items per step tile
    g["tie_chunk"] = g["kSel"] * g["kTiePer"]    # nodes per tie-count block
    g["tie_pass"] = g["kSel"] * g["kTiePer"]     # tie blocks per pass of ppr_topk_tie_scan_kernel
    return g


def _tile_coords(rp, tile):
    """numpy mirror of diagonal_search_global (merge_rows.cuh) at the diagonals ppr_partition_kernel searches:
    min(t * tile, rows + nnz) for t = 0 .. num_tiles.  Returns (num_tiles + 1, 2) int64 (row, nz)."""
    rp = np.asarray(rp, np.int64)
    rows, nnz = rp.size - 1, int(rp[-1])
    total = rows + nnz
    num_tiles = -(-total // tile)
    diag = np.minimum(np.arange(num_tiles + 1, dtype=np.int64) * tile, total)
    lo = np.maximum(diag - nnz, 0)
    hi = np.minimum(diag, rows)
    while True:
        live = lo < hi
        if not live.any():
            break
        mid = lo + ((hi - lo) >> 1)
        go_right = live & (rp[np.minimum(mid + 1, rows)] <= diag - mid - 1)
        lo = np.where(go_right, mid + 1, lo)
        hi = np.where(live & ~go_right, mid, hi)
    return np.stack([lo, diag - lo], axis=1)


def _walk_coords(rp, tile):
    """The same coordinates from a plain walk of the merge path: a row's non-zeros, then its end item."""
    rows, nnz = len(rp) - 1, int(rp[-1])
    total = rows + nnz
    out, r, z = [], 0, 0
    for d in range(total + 1):
        if d % tile == 0 or d == total:
            out.append((r, z))
        if d == total:
            break
        if z < rp[r + 1]:
            z += 1
        else:
            r += 1
    return np.array(out, np.int64)


def _order_key(x):
    """numpy mirror of dev::order_key: the fp32 bits as a sign-magnitude number, -0 = +0, NaN placed by its sign."""
    x = np.asarray(x, np.float32)
    u = x.view(np.uint32).copy()
    u[x == 0] = 0
    return np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)


def _key_order(x, k):
    """The first k indices by (order key descending, index ascending)."""
    key = _order_key(x).astype(np.int64)
    return np.lexsort((np.arange(key.size), -key))[:k]


def _f32(bits):
    return np.array(bits, np.uint32).view(np.float32)


def test_constants_are_read_from_the_sources():
    g = _geometry()
    assert all(g[k] > 0 for k in ("kBT", "kBIPT", "kSel", "kTiePer")), g
    with pytest.raises(AssertionError):
        _constant("ppr_core.cuh", "kNoSuchConstant")


@pytest.mark.parametrize("tile", ["kernel", 7])
def test_tile_mirror_matches_a_merge_path_walk(tile):
    tile = _geometry()["tile"] if tile == "kernel" else tile
    rng = np.random.default_rng(3)
    cases = [[0], [5], [3 * tile + 2], [0, 0, 0], [tile - 1, 0, 0, 1]]
    for j in range(12):
        n = int(rng.integers(1, 3000))
        deg = rng.poisson(rng.uniform(0.2, 6.0), n)
        deg[rng.random(n) < 0.2] = 0  # empty rows, also in runs
        if j % 3 == 0:
            deg[rng.integers(0, n)] = int(rng.integers(tile, 4 * tile))  # a row over several tiles
        if j % 4 == 1:
            s = int(rng.integers(0, n))
            deg[s:s + 2 * tile] = 0
        cases.append(list(deg))
    for deg in cases:
        rp = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64)
        got, want = _tile_coords(rp, tile), _walk_coords(rp, tile)
        assert np.array_equal(got, want), (len(deg), int(rp[-1]))


def test_order_key_mirror():
    k = _order_key(_f32([0x00000000, 0x80000000]))
    assert k[0] == k[1] == 0x80000000  # -0 and +0
    inf, ninf, pnan, nnan = _order_key(np.array([np.inf, -np.inf], np.float32)).tolist() + \
        _order_key(_f32([0x7FC00000, 0xFFC00000])).tolist()
    assert pnan > inf and nnan < ninf
    assert _order_key(_f32([0x7FC00001]))[0] > pnan and _order_key(_f32([0xFFC00001]))[0] < nnan
    rng = np.random.default_rng(4)
    x = np.concatenate([rng.standard_normal(5000) * 10.0 ** rng.integers(-40, 38, 5000),
                        _f32(rng.integers(1, 0x00800000, 500)), -_f32(rng.integers(1, 0x00800000, 500)),
                        [np.inf, -np.inf, np.finfo(np.float32).max, -np.finfo(np.float32).max]]).astype(np.float32)
    x = np.unique(x[x != 0])
    keys = _order_key(x)
    assert (np.diff(keys.astype(np.int64)) > 0).all()  # strictly increasing with the float order


# --------------------------------------------------------------------- graph T: tiles and fix-up blocks ----
@functools.lru_cache(maxsize=None)
def _graph_t():
    """Row = destination, value 1/outdeg(src).  Nodes with id % 10 == 3 are never a source (dangling); rows of
    in-degree 0 have no in-edges.  The in-degree sequence is placed, in increasing item order, so that the
    partition has the features _tile_features checks.  Returns (n, rp, ci, va, hub rows)."""
    tile = _geometry()["tile"]
    rng = np.random.default_rng(2024)
    n = 300_007
    deg = rng.poisson(5.0, n).astype(np.int64)
    hub = 5 * tile  # at least 3 whole tiles wherever it starts

    def starts():  # merge item of each row's first non-zero (its end item when empty)
        return np.cumsum(deg) - deg + np.arange(n)

    def end_on_tile_end(t):  # the row before the item lengthened to end on tile t's last item
        e = np.cumsum(deg) + np.arange(n)
        r = int(np.searchsorted(e, (t + 1) * tile - 1, "left")) - 1
        deg[r] += (t + 1) * tile - 1 - e[r]

    hub1 = int(np.searchsorted(starts(), 40 * tile + 300))
    deg[hub1] = hub
    end_on_tile_end(79)
    e0 = int(np.searchsorted(starts(), 150 * tile + 77))
    deg[e0:e0 + 3000] = 0  # more than 2 tiles of empty rows
    hub2 = int(np.searchsorted(starts(), 254 * tile + 600))  # open at the ends of tiles 254 .. 258
    deg[hub2] = hub
    end_on_tile_end(600)
    if (n + deg.sum()) % tile == 0:
        deg[n - 1] += 1
    rp = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    pool = np.flatnonzero(np.arange(n) % 10 != 3)
    src = rng.choice(pool, int(rp[-1]))
    row = np.repeat(np.arange(n), deg)
    src = src[np.lexsort((src, row))]
    outdeg = np.bincount(src, minlength=n)
    return n, rp, src.astype(np.int32), (1.0 / outdeg[src]).astype(np.float32), (hub1, hub2)


def _tile_features(rp, tile):
    c = _tile_coords(rp, tile)
    rp = np.asarray(rp, np.int64)
    rows, num_tiles = rp.size - 1, c.shape[0] - 1
    cx, cy = c[:, 0], c[:, 1]
    t = np.arange(num_tiles)
    f = {"num_tiles": num_tiles}
    # (a) a non-empty row whose end item is the last item of a tile (not the last tile)
    f["a"] = t[(t < num_tiles - 1) & (cx[1:] > cx[:-1]) & (cy[1:] == rp[cx[1:]]) & (cx[1:] >= 1) &
               (rp[cx[1:]] > rp[np.maximum(cx[1:] - 1, 0)]) & (cy[1:] > cy[:-1])]
    # (b) a non-empty row whose first non-zero is the first item of a tile
    f["b"] = t[(t >= 1) & (cx[:-1] < rows) & (cy[:-1] == rp[cx[:-1]]) & (rp[np.minimum(cx[:-1] + 1, rows)] > cy[:-1])]
    # rows open at a tile end: what ppr_step_kernel stores in carry_row (has_open)
    open_start = np.where(cx[1:] > cx[:-1], rp[cx[1:]], np.where(cx[:-1] < rows, rp[cx[:-1]], cy[1:]))
    carry = np.where((cx[1:] < rows) & (cy[1:] > np.maximum(open_start, cy[:-1])), cx[1:], -1)
    f["carry"] = carry
    # (c) rows covering whole tiles: tiles inside one row's non-zeros
    inside = cx[:-1][(cx[1:] == cx[:-1]) & (cy[1:] > cy[:-1])]
    rows_, counts = np.unique(inside, return_counts=True)
    f["c"] = dict(zip(rows_.tolist(), counts.tolist()))
    # (d) a full tile without non-zeros
    f["d"] = t[(t < num_tiles - 1) & (cy[1:] == cy[:-1])]
    f["e"] = (rows + int(rp[-1])) % tile
    return f


def test_graph_t_partition_has_every_split():
    tile = _geometry()["tile"]
    n, rp, ci, va, (hub1, hub2) = _graph_t()
    f = _tile_features(rp, tile)
    assert n % 2 == 1
    assert f["a"].size, "no row ends on a tile's last item"
    assert f["b"].size, "no row starts on a tile's first item"
    assert f["c"].get(hub1, 0) >= 3 and f["c"].get(hub2, 0) >= 3, (f["c"], hub1, hub2)
    assert f["carry"][255] == f["carry"][256] == hub2, "the hub run does not cross fix-up blocks 0 and 1"
    assert f["d"].size, "no tile without non-zeros"
    assert f["e"] != 0, "the last tile is full"
    assert f["num_tiles"] > 8 * B200_SMS, f["num_tiles"]
    assert (np.diff(rp) == 0).any() and (np.bincount(ci, minlength=n) == 0).any()  # no in-edges; dangling


def _graph_t_columns(n, rp, ci, va, hubs):
    """One-hot seeds on the hub rows around seven _columns vectors: k = 1 is the hub open across fix-up blocks,
    k = 9 puts the other hub alone in the second chunk."""
    hub1, hub2 = hubs
    one = np.zeros((2, n), np.float32)
    one[0, hub2] = 1.0
    one[1, hub1] = 1.0
    return np.concatenate([one[:1], _columns(n, rp, ci, va, 7, seed=17), one[1:]])


@pytest.mark.gpu
def test_graph_t_columns_and_rows_match_the_oracle(sp, cuda):
    ss = _sass_summary()
    assert {"ppr::ppr_partition_kernel", "ppr::ppr_step_kernel", "ppr::ppr_fixup_kernel"} <= \
        ss.shipped_kernels(os.path.join(LIBDIR, "libspmv_b200_ppr.so"))
    n, rp, ci, va, hubs = _graph_t()
    G = _device_graph(sp, cuda, n, rp, ci, va)
    pool = _graph_t_columns(n, rp, ci, va, hubs)
    tol, cap = 1e-7, 500
    cfg = sp.make_pagerank_config(D, tol, cap)
    at, own = {}, {}
    worst, t0 = 0.0, time.perf_counter()
    for k in (1, 8, 9):
        V = pool[:k]
        ranks, iters, res, conv, _ = sp.pagerank_personalized_batch(G.ptr, V, cfg)
        dense = ranks.cpu().numpy()
        for c in range(k):
            key = (c, int(iters[c]))
            if key not in at:
                at[key] = orc_personalized(n, rp, ci, va, V[c], tol=tol, max_it=cap, fixed_it=int(iters[c]))[0]
            err = float(np.abs(dense[:, c].astype(np.float64) - at[key]).sum())
            worst = max(worst, err)
            assert err <= 1e-6, f"k={k} column {c}: L1 {err:.3e} to the restatement after {iters[c]} iterations"
            if c not in own:
                own[c] = orc_personalized(n, rp, ci, va, V[c], tol=tol, max_it=cap)[1::3]
            assert abs(int(iters[c]) - own[c][0]) <= 1 and bool(conv[c]) == own[c][1], (k, c, iters[c], own[c])
        for top in (1, 37, 1024):
            ids, vals = (t.cpu().numpy() for t in sp.pagerank_personalized_batch_top_k(G.ptr, V, top, cfg)[:2])
            for c in range(k):
                _assert_row(ids[c], vals[c], dense[:, c], top, f"graph T k={k} top={top} row {c}")
    print(f"graph T: n={n}, worst L1 {worst:.3e}, {time.perf_counter() - t0:.1f} s")


# ---------------------------------------------------------------------- graph S: ties past 2^24 nodes ----
@functools.lru_cache(maxsize=None)
def _graph_s():
    """Seed nodes have no edges; every other node is on one directed ring (values 1.0), so all ring ranks are
    bit-equal and each seed's rank depends on its weight alone.  n = one tie-scan pass of nodes + kTieChunk + 3,
    i.e. 2^24 + 4099 nodes in 4098 tie blocks.  Returns (n, rp, ci, va, ring, columns): each column is
    (heavy ids, weight-1 ids), all sorted, heavy ones of weight 2."""
    g = _geometry()
    chunk, pass_nodes = g["tie_chunk"], g["tie_pass"] * g["tie_chunk"]
    n = pass_nodes + chunk + 3
    rng = np.random.default_rng(31)
    hi = pass_nodes + 1 + rng.permutation(n - pass_nodes - 1)  # nodes past pass_nodes
    fixed_lo = np.array([chunk - 1, chunk, pass_nodes - 1])
    lo = rng.choice(pass_nodes, 2000, replace=False)
    lo = lo[~np.isin(lo, fixed_lo)][:1000]
    a_w1 = np.concatenate([fixed_lo, lo[:597], [pass_nodes], hi[:899]])  # 600 below pass_nodes, 900 at or above
    a_heavy = np.concatenate([lo[597:602], hi[2100:2105]])
    b_heavy = np.concatenate([lo[602:607], hi[2105:2110]])
    b_w1 = np.concatenate([lo[607:917], hi[2110:2300]])
    c_w1 = hi[900:2100]
    cols = [(np.sort(a_heavy), np.sort(a_w1)), (np.sort(b_heavy), np.sort(b_w1)), (np.array([], np.int64), np.sort(c_w1))]
    seeds = np.concatenate([x for col in cols for x in col])
    assert np.unique(seeds).size == seeds.size
    is_seed = np.zeros(n, bool)
    is_seed[seeds] = True
    ring = np.flatnonzero(~is_seed)
    deg = (~is_seed).astype(np.int64)
    rp = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    ci = np.roll(ring, 1).astype(np.int32)  # row ring[j] gets the edge from ring[j - 1]
    return n, rp, ci, np.ones(ring.size, np.float32), ring, cols


def _graph_s_expected(ring, cols, top):
    """Each row from the construction: heavy seeds by id, then weight-1 seeds by id, then ring nodes by id."""
    return [np.concatenate([h, w, ring[:max(0, top - h.size - w.size)]])[:top].astype(np.int32) for h, w in cols]


@pytest.mark.gpu
def test_graph_s_rows_past_two_to_the_24(sp, cuda):
    import scipy.sparse as S
    ss = _sass_summary()
    assert "ppr::ppr_topk_tie_scan_kernel" in ss.shipped_kernels(os.path.join(LIBDIR, "libspmv_b200_ppr_topk.so"))
    g = _geometry()
    n, rp, ci, va, ring, cols = _graph_s()
    blocks = -(-n // g["tie_chunk"])
    assert blocks > g["tie_pass"] and n - 1 < 2 ** 31, blocks  # a second pass of the tie scan
    top = 1024
    data, indices, indptr = [], [], [0]
    for h, w in cols:
        idx = np.concatenate([h, w])
        order = np.argsort(idx)
        indices.append(idx[order])
        data.append(np.concatenate([np.full(h.size, 2.0), np.ones(w.size)])[order])
        indptr.append(indptr[-1] + idx.size)
    V = S.csr_matrix((np.concatenate(data).astype(np.float32), np.concatenate(indices), indptr), shape=(len(cols), n))
    G = _device_graph(sp, cuda, n, rp, ci, va)
    cfg = sp.make_pagerank_config(D, 0.0, 30)
    t0 = time.perf_counter()
    ranks, iters, res, conv, _ = sp.pagerank_personalized_batch(G.ptr, V, cfg)
    ids, vals, it2, _, conv2, _ = sp.pagerank_personalized_batch_top_k(G.ptr, V, top, cfg)
    t_gpu = time.perf_counter() - t0
    assert (iters == 30).all() and not conv.any() and np.array_equal(it2, iters) and not conv2.any()
    dense = ranks.cpu().numpy()
    ids, vals = ids.cpu().numpy(), vals.cpu().numpy()
    expected = _graph_s_expected(ring, cols, top)
    t_orc, worst = 0.0, 0.0
    for c, ((h, w), want) in enumerate(zip(cols, expected)):
        col = dense[:, c]
        # the construction: heavy > weight 1 > ring > the other columns' seeds (0), each group one value
        groups = [h, w, ring]
        vals_of = [np.unique(col[x].view(np.uint32)) for x in groups if x.size]
        assert all(v.size == 1 for v in vals_of), f"column {c}: a group holds several values"
        levels = [float(v.view(np.float32)[0]) for v in vals_of]
        assert levels == sorted(levels, reverse=True) and len(set(levels)) == len(levels) and levels[-1] > 0, levels
        assert np.array_equal(ids[c], want), f"column {c}: ids differ at {np.flatnonzero(ids[c] != want)[:8]}"
        assert np.array_equal(vals[c].view(np.uint32), col[want].view(np.uint32)), f"column {c}: values"
        d_ids, d_vals = sp.pagerank_top_k_device(ranks[:, c].contiguous(), top)
        assert np.array_equal(d_ids, want) and np.array_equal(d_vals.view(np.uint32), col[want].view(np.uint32)), c
        v = np.zeros(n, np.float32)
        v[h], v[w] = 2.0, 1.0
        t1 = time.perf_counter()
        o, o_it, _, _, o_conv = orc_personalized(n, rp, ci, va, v, tol=0.0, max_it=30)
        t_orc += time.perf_counter() - t1
        assert o_it == 30 and not o_conv
        err = float(np.abs(col.astype(np.float64) - o).sum())
        worst = max(worst, err)
        assert err <= 1e-6, f"column {c}: L1 {err:.3e} to the restatement"
    print(f"graph S: n={n}, worst L1 {worst:.3e}, batch + top-K {t_gpu:.1f} s, oracle {t_orc:.1f} s")


# -------------------------------------------------------------------------------------- non-finite ranks ----
def _non_finite_vector(kind, n=20_000, seed=6):
    """Ranks holding +-NaN (several payloads), +-Inf, +-0, subnormals and finite values, with equal values on both
    sides of the 4096-element chunk boundaries.  "high": the k = 17 threshold is among NaNs and the k = 1000 one
    among equal finite values; "low": most values are negative, so k = 17 and k = 1000 end among +-0."""
    rng = np.random.default_rng(seed)
    x = np.empty(n, np.float32)
    free = rng.permutation(n)
    edges = [e + d for e in range(4096, n, 4096) for d in (-2, -1, 0, 1)]
    free = np.concatenate([edges, free[~np.isin(free, edges)]])
    at = 0

    def put(vals):
        nonlocal at
        vals = np.asarray(vals, np.float32)
        x[free[at:at + vals.size]] = vals
        at += vals.size

    sub = lambda m: _f32(rng.integers(1, 0x00800000, m))  # noqa: E731  positive subnormals
    if kind == "high":
        put(np.full(30, 0.5, np.float32))                 # the chunk boundaries first, then scattered
        put(_f32([0x7FC00000] * 20 + [0x7FC00123] * 5 + [0x7FFFFFFF] * 3 + [0xFFC00000] * 10 + [0xFFC01234] * 2))
        put([np.inf] * 6 + [-np.inf] * 6)
        put(rng.uniform(0.6, 1e30, 900))
        put(np.full(70, 0.5, np.float32))
        put(np.where(rng.random(2000) < 0.5, 0.0, -0.0))
        put(sub(500))
        put(-sub(500))
        put(rng.uniform(-1e3, 0.49, n - at))
    else:
        put(np.where(rng.random(40) < 0.5, 0.0, -0.0))    # +-0 at the boundaries
        put(sub(10))
        put([np.float32(1e-30)] * 3 + [np.float32(2.5e-38)] * 2)
        put(np.where(rng.random(3000) < 0.5, 0.0, -0.0))
        put(_f32([0xFFC00000] * 20 + [0xFFFFFFFF] * 4))
        put([-np.inf] * 8)
        put(-sub(1000))
        put(-rng.uniform(1e-20, 1e30, n - at))
    assert at == n
    return x


def test_non_finite_vectors_hit_the_intended_ties():
    for kind in ("high", "low"):
        x = _non_finite_vector(kind)
        key = _order_key(x)
        for k in (17, 1000):
            o = _key_order(x, k + 1)
            thr = key[o[k - 1]]
            tied = np.flatnonzero(key == thr)
            assert tied.size > 1 and key[o[k]] == thr, (kind, k)  # the k-th and (k+1)-th are equal
            taken = o[:k][key[o[:k]] == thr] // 4096
            assert k == 17 and kind == "low" or taken.min() < taken.max(), (kind, k)  # taken ties in several chunks
        if kind == "high":
            assert np.isnan(x[_key_order(x, 17)]).all()
        else:
            t = x[_key_order(x, 1000)[20:]]
            assert (t == 0).all() and np.signbit(t).any() and (~np.signbit(t)).any()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["high", "low"])
def test_device_top_k_orders_non_finite_ranks_by_key(sp, cuda, kind):
    import torch
    x = _non_finite_vector(kind)
    d = torch.as_tensor(x).to(cuda)
    for k in (1, 17, 1000):
        ids, vals = sp.pagerank_top_k_device(d, k)
        want = _key_order(x, k)
        assert np.array_equal(ids, want), f"{kind} k={k}: ids differ at {np.flatnonzero(ids != want)[:8]}"
        assert np.array_equal(vals.view(np.uint32), x[want].view(np.uint32)), f"{kind} k={k}: values"


def _nan_graph():
    """A graph whose ranks mix NaN and finite values: one NaN edge weight feeds a sink region (60 nodes, every one
    with out-edges inside the region only, none dangling), so the region turns NaN while the rest, and the dangling
    mass, stay finite."""
    rng = np.random.default_rng(8)
    n, m = 3001, 60
    main, region = n - m, np.arange(n - m, n)
    edges = [(i, int(j)) for i in range(main) if i % 13 for j in rng.integers(0, main, 3)]
    edges += [(int(region[j]), int(region[(j + 1) % m])) for j in range(m)]
    edges += [(int(a), int(b)) for a in region for b in rng.choice(region, 2)]
    edges.append((5, int(region[0])))
    rp, ci, va = graph(n, edges)
    row = int(region[0])
    j = rp[row] + int(np.flatnonzero(ci[rp[row]:rp[row + 1]] == 5)[0])
    va[j] = np.nan
    return n, rp, ci, va, region


@pytest.mark.gpu
def test_batch_top_k_with_nan_ranks(sp, cuda):
    n, rp, ci, va, region = _nan_graph()
    G = _device_graph(sp, cuda, n, rp, ci, va)
    V = _columns(n, rp, ci, va, 9, seed=11)
    cfg = sp.make_pagerank_config(D, 1e-6, 30)
    ranks = sp.pagerank_personalized_batch(G.ptr, V, cfg)[0]
    dense = ranks.cpu().numpy()
    nan = np.isnan(dense)
    assert nan[region].all() and not nan[:region[0]].any(), "the ranks do not mix NaN and finite values as built"
    for top in (1, 37, 1024):
        ids, vals = (t.cpu().numpy() for t in sp.pagerank_personalized_batch_top_k(G.ptr, V, top, cfg)[:2])
        for c in range(V.shape[0]):
            col = dense[:, c]
            want = _key_order(col, top)
            what = f"NaN graph top={top} row {c}"
            assert np.array_equal(ids[c], want), f"{what}: ids differ at {np.flatnonzero(ids[c] != want)[:8]}"
            assert np.array_equal(vals[c].view(np.uint32), col[want].view(np.uint32)), what
            d_ids, d_vals = sp.pagerank_top_k_device(ranks[:, c].contiguous(), top)
            assert np.array_equal(d_ids, want) and np.array_equal(d_vals.view(np.uint32), col[want].view(np.uint32)), what
