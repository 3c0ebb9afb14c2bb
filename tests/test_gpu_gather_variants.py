"""Katz, cuGraph-semantics PageRank (uniform, personalised, weighted) and in-tree PageRank under every gather
configuration, on graphs shaped to reach the boundaries of the layout (tests/_boundary_graphs.py).

The gather phase runs the same SELL and heavy-segment kernels for all three algorithms; which instantiation runs, which
cache hints it uses and how slices are dealt to warps are build-time knobs (graph_build.cu build_graph).  None of them
may change a bit of any result.  Every result is also checked against the oracles (oracle/*.c) and, for fixed iteration
counts, against a high-precision restatement within a rounding bound derived from the graph.

The CPU tests (no marker) check that the graphs reach their boundaries in the layout model, that the bounds are tight
enough to mean something (<= 1e-11), and that the high-precision restatements agree with both oracles."""
import math

import numpy as np
import pytest

import _boundary_graphs as B
from _checkers import Oracle
from test_cugraph_oracle import oracle_cugraph_pagerank
from test_katz_oracle import oracle_katz

GRAPHS = B.all_graphs()
GRAPH_IDS = [g.name for g in GRAPHS]
FIXED_K = (1, 2, 20)
REL_TOL = 1e-9

# every knob build_graph reads for the gather (cleared before each handle, then set per variant)
KNOBS = ["MGB200_IDX_FLAGS", "MGB200_FORCE_MULTI_PATH", "MGB200_L1_HOT_K", "MGB200_L2_HOT_MB", "MGB200_SMEM_TABLE_KB",
         "MGB200_SELL_MODE", "MGB200_SELL_WORK_ITEMS", "MGB200_SLICE_COST", "MGB200_SELL_KERNEL", "MGB200_SELL_ITEMS",
         "MGB200_OVERLAP_EPILOGUE", "MGB200_BUILD_CHUNK_EDGES", "MGB200_MULTI_AWARE", "MGB200_LABELLING",
         "MGB200_HEAVY_MIN_DEGREE", "MGB200_SEGMENT_EDGES"]

VARIANTS = {
    "default": {},
    "idx_flags": {"MGB200_IDX_FLAGS": "1"},
    "force_multi_path": {"MGB200_IDX_FLAGS": "0", "MGB200_FORCE_MULTI_PATH": "1"},
    "no_l1_hints": {"MGB200_L1_HOT_K": "-1"},
    "no_l2_hot_flags": {"MGB200_L2_HOT_MB": "0", "MGB200_IDX_FLAGS": "1"},
    "smem_table_1": {"MGB200_SMEM_TABLE_KB": "1"},
    "smem_table_64": {"MGB200_SMEM_TABLE_KB": "64"},
    "smem_table_200": {"MGB200_SMEM_TABLE_KB": "200"},
    "tickets_1": {"MGB200_SELL_MODE": "0", "MGB200_SELL_WORK_ITEMS": "1"},
    "tickets_37": {"MGB200_SELL_MODE": "0", "MGB200_SELL_WORK_ITEMS": "37"},
    "tickets_100000": {"MGB200_SELL_MODE": "0", "MGB200_SELL_WORK_ITEMS": "100000"},
    "static_1": {"MGB200_SELL_MODE": "1", "MGB200_SELL_WORK_ITEMS": "1"},
    "static_5": {"MGB200_SELL_MODE": "1", "MGB200_SELL_WORK_ITEMS": "5"},
    "slice_cost_0": {"MGB200_SLICE_COST": "0"},
    "stream_1": {"MGB200_SELL_KERNEL": "stream", "MGB200_SELL_ITEMS": "1"},
    "stream_7": {"MGB200_SELL_KERNEL": "stream", "MGB200_SELL_ITEMS": "7"},
    "no_overlap_epilogue": {"MGB200_OVERLAP_EPILOGUE": "0"},  # launch_iteration only: in-tree PageRank
}
IN_TREE_ONLY = {"no_overlap_epilogue"}

LAYOUT_FIELDS = ["heavy_rows", "heavy_edges", "heavy_segments", "sell_rows", "sell_slices", "sell_entries", "zero_rows",
                 "local_edges"]


def katz_params(g):
    """(alpha, eps) with gamma > 0 -- alpha^2 * max out-degree < 1 -- whose exact walk counts stay below 2^52 for every
    iteration the oracle runs, the precondition for bit-exact Katz; the first candidate that qualifies."""
    deg_max = int(g.outdeg.max())
    for scale, eps in [(0.5, 1e-2), (0.3, 1e-2), (0.2, 1e-1), (0.1, 1e-1)]:
        alpha = scale / math.sqrt(deg_max + 1.0)
        rc, _, it = oracle_katz(g.n, g.f, g.t, alpha, eps, guard=2000)
        if rc == 0 and max(B.walk_counts(g.n, g.f, g.t, it)) < 2 ** 52:
            return alpha, eps
    raise AssertionError(f"{g.name}: no Katz parameters keep the walk counts below 2^52")


def katz_negative_gamma(g):
    """alpha = 0.2 (the reference default) gives gamma < 0 once alpha^2 * max out-degree > 1."""
    return 0.2 * 0.2 * int(g.outdeg.max()) > 1.0


# ---- CPU: the graphs reach their boundaries, the bounds mean something, the references agree ------------------------

@pytest.mark.parametrize("g", GRAPHS, ids=GRAPH_IDS)
def test_graphs_reach_their_layout_boundaries(g):
    lay = B.layout(g.indeg, g.H, g.S)
    d = np.sort(g.indeg)[::-1]
    heavy, sell = d[d >= g.H], d[(d >= 1) & (d < g.H)]
    widths = B.slice_widths(g.indeg, g.H)
    want = g.intended
    assert lay["local_edges"] == len(g.f) and lay["heavy_rows"] + lay["sell_rows"] + lay["zero_rows"] == g.n
    if "heavy_rows" in want:
        assert (lay["heavy_rows"] > 0) == want["heavy_rows"] and (lay["sell_rows"] > 0) == want["sell_rows"]
    for deg in want.get("heavy_degrees", []):
        assert deg in heavy, deg
    if "heavy_degrees" in want:
        present = set(heavy.tolist())
        assert {g.H, g.H + 1} <= present
        for k in (1, 2):  # segment boundaries k*S - 1, k*S, k*S + 1 wherever they are heavy
            assert {x for x in (k * g.S - 1, k * g.S, k * g.S + 1) if x >= g.H} <= present
        assert {255, 256, 257} <= present  # the heavy kernel's unrolled step (256 edges) against its tail loop
        assert max(heavy) == B.hub_in_degree(g.S) or B.hub_in_degree(g.S) < g.H
        assert want["sell_degree"] in sell
        assert set(range(1, 18)) <= set(widths.tolist())  # both sides of 8 and 16 (SELL_UNROLL)
        runs = np.diff(np.flatnonzero(np.concatenate([[True], widths > 2, [True]]))) - 1
        assert runs.max() >= want["narrow_slices"]  # a run of > 40 narrow slices
        items = B.work_items(widths, 1)
        assert items[0][1] - items[0][0] > 32  # one work item crosses its 32-slice block of slice ends
        assert lay["sell_rows"] % B.SLICE_ROWS != 0  # the last slice is partly filled
        assert lay["zero_rows"] > 0
    if want.get("n_sell_mod") is not None:
        assert lay["sell_rows"] % B.SLICE_ROWS == want["n_sell_mod"]
    if want.get("odd_n"):
        assert g.n % 2 == 1 and g.n <= 1024 // 8  # SMEM_TABLE_KB=1 holds 128 labels: the table covers every label
    assert lay["sell_entries"] == B.SLICE_ROWS * int(widths.sum())


def test_every_boundary_is_reached_by_some_graph():
    mods = {B.layout(g.indeg, g.H, g.S)["sell_rows"] % 32 for g in GRAPHS if g.intended.get("heavy_degrees")}
    assert {1, 31} <= mods
    assert any(B.layout(g.indeg, g.H, g.S)["sell_rows"] == 0 for g in GRAPHS)
    assert any(B.layout(g.indeg, g.H, g.S)["heavy_rows"] == 0 for g in GRAPHS)
    assert any(g.n == 1 for g in GRAPHS)
    assert {g.S for g in GRAPHS} >= {1, 31, 32, 256, 257}
    assert any(katz_negative_gamma(g) for g in GRAPHS)


@pytest.mark.parametrize("g", GRAPHS, ids=GRAPH_IDS)
def test_rounding_bounds_are_tight(g):
    for k in FIXED_K:
        assert B.pagerank_bound(g, k) <= 1e-11
        for weighted in (False, True):
            for pers in (False, True):
                assert B.cugraph_bound(g, k, weighted, pers) <= 1e-11


@pytest.mark.parametrize("g", GRAPHS, ids=GRAPH_IDS)
def test_high_precision_reference_agrees_with_the_oracles(g):
    oracle = Oracle()
    for k in FIXED_K:
        # (stop_epsilon=0 still stops early once no rank moves at all: n == 1)
        ref, it = oracle.pagerank(g.n, g.f, g.t, max_iterations=k, stop_epsilon=0.0)
        assert B.max_rel_err(ref, B.hp_pagerank(g.n, g.f, g.t, it)) < 1e-13, k
        for weights in (None, g.w):
            for seeds in (None, g.seeds):
                ref, it, _ = oracle_cugraph_pagerank(g.n, g.f, g.t, weights=weights, personalization=seeds,
                                                     epsilon=0.0, max_iterations=k)
                hp = B.hp_cugraph_pagerank(g.n, g.f, g.t, k, weights=weights, seeds=seeds)
                assert it == k and B.max_rel_err(ref, hp) < 1e-13, (k, weights is None, seeds is None)


@pytest.mark.parametrize("g", GRAPHS, ids=GRAPH_IDS)
def test_katz_walk_counts_stay_exact(g):
    alpha, eps = katz_params(g)
    assert alpha * alpha * int(g.outdeg.max()) < 1.0


# ---- GPU: the configuration matrix --------------------------------------------------------------------------------

_oracles = {}   # (graph, what, args) -> oracle / reference results
_defaults = {}  # graph -> results under the default gather configuration


def cached(key, fn):
    if key not in _oracles:
        _oracles[key] = fn()
    return _oracles[key]


def set_env(monkeypatch, g, extra):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("MGB200_HEAVY_MIN_DEGREE", str(g.H))
    monkeypatch.setenv("MGB200_SEGMENT_EDGES", str(g.S))  # unset, it would be sized from the heavy edge count
    for k, v in extra.items():
        monkeypatch.setenv(k, v)


def cugraph_runs(g, handle, weighted):
    from memgraph_b200 import personalized as P
    out = {}
    for pers in (False, True):
        seeds = g.seeds if pers else (None, None)
        for k in FIXED_K:
            out[(pers, k)] = P.cugraph_pagerank(handle, *seeds, max_iterations=k, stop_epsilon=0.0)
        out[(pers, "default")] = P.cugraph_pagerank(handle, *seeds)
    return out


def run_variant(g, env, monkeypatch, in_tree_only=False):
    """Every algorithm on fresh handles built under `env`: {name: result}."""
    import memgraph_b200 as mg
    from memgraph_b200 import katz, personalized as P
    set_env(monkeypatch, g, env)
    res = {}
    with mg.PageRankGraph.from_arrays(g.n, g.f, g.t) as h:
        res["info"] = dict(h.info)
        for k in FIXED_K:
            res[("pr", k)] = h.run(max_iterations=k, stop_epsilon=0.0)
        res[("pr", "default")] = h.run()
        if in_tree_only:
            return res
        res["katz+"] = katz.set_katz(h, *katz_params(g))
        if katz_negative_gamma(g):
            res["katz-"] = katz.set_katz(h, 0.2, 1e-2)
        res["cugraph"] = cugraph_runs(g, h, False)
    with P.weighted_graph(g.n, g.f, g.t, g.w) as h:
        res["winfo"] = dict(h.info)
        res["weighted"] = cugraph_runs(g, h, True)
    return res


def check_against_oracles(g, res):
    lay = B.layout(g.indeg, g.H, g.S)
    for key in ("info", "winfo"):
        if key in res:
            assert {f: res[key][f] for f in LAYOUT_FIELDS} == lay, key
    oracle = Oracle()
    for k in FIXED_K + ("default",):
        kw = dict(max_iterations=k, stop_epsilon=0.0) if k != "default" else {}
        ref, it = cached((g.name, "pr", k), lambda: oracle.pagerank(g.n, g.f, g.t, **kw))
        ranks, st = res[("pr", k)]
        assert st.iterations == it, k
        assert B.max_rel_err(ranks, ref) < REL_TOL, k
        if k != "default":
            hp = cached((g.name, "hp_pr", k), lambda: B.hp_pagerank(g.n, g.f, g.t, it))
            err = B.max_rel_err(ranks, hp)
            assert err <= B.pagerank_bound(g, it), (k, err)
            note_worst("pagerank", k, err, B.pagerank_bound(g, it))
    if "katz+" not in res:
        return
    alpha, eps = katz_params(g)
    for key, (a, e) in (("katz+", (alpha, eps)), ("katz-", (0.2, 1e-2))):
        if key not in res:
            continue
        rc, ref, it = cached((g.name, key), lambda: oracle_katz(g.n, g.f, g.t, a, e))
        got, st = res[key]
        assert rc == 0 and st["iterations"] == it and np.array_equal(got, ref), key
        assert (st["gamma"] > 0) == (key == "katz+")
    for what, weighted in (("cugraph", False), ("weighted", True)):
        for (pers, k), (got, st) in res[what].items():
            w = g.w if weighted else None
            seeds = g.seeds if pers else None
            kw = dict(max_iterations=k, epsilon=0.0) if k != "default" else {}
            ref, it, conv = cached((g.name, what, pers, k),
                                   lambda: oracle_cugraph_pagerank(g.n, g.f, g.t, weights=w, personalization=seeds, **kw))
            assert st["iterations"] == it and bool(st["converged"]) == conv, (what, pers, k)
            assert B.max_rel_err(got, ref) < REL_TOL, (what, pers, k)
            if k != "default":
                hp = cached((g.name, "hp", what, pers, k),
                            lambda: B.hp_cugraph_pagerank(g.n, g.f, g.t, k, weights=w, seeds=seeds))
                bound = B.cugraph_bound(g, k, weighted, pers)
                err = B.max_rel_err(got, hp)
                assert err <= bound, (what, pers, k, err, bound)
                note_worst(what, k, err, bound)


_worst = {}  # (algorithm, k) -> (error / bound, error, bound) of the closest call, printed at the end of the module


def note_worst(what, k, err, bound):
    if err / bound >= _worst.get((what, k), (-1.0,))[0]:
        _worst[(what, k)] = (err / bound, err, bound)


def assert_same_bits(a, b, where):
    for key in a:
        if key in ("info", "winfo") or key not in b:
            continue
        x, y = a[key], b[key]
        if isinstance(x, dict):  # cuGraph runs
            for kk in x:
                assert np.array_equal(x[kk][0], y[kk][0]), (where, key, kk)
                assert x[kk][1]["iterations"] == y[kk][1]["iterations"], (where, key, kk)
        else:
            assert np.array_equal(x[0], y[0]), (where, key)


def defaults(g, monkeypatch):
    if g.name not in _defaults:
        res = run_variant(g, {}, monkeypatch)
        check_against_oracles(g, res)
        _defaults[g.name] = res
    return _defaults[g.name]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS), ids=list(VARIANTS))
@pytest.mark.parametrize("g", GRAPHS, ids=GRAPH_IDS)
def test_gather_variant(g, variant, monkeypatch):
    """Layout = the CPU model; every algorithm bit-identical to the default configuration of the same (H, S); in-tree
    PageRank and cuGraph PageRank within 1e-9 of their oracles with the same iteration counts (and converged flags) and
    within the rounding bound of the high-precision reference; Katz np.array_equal to its oracle."""
    base = defaults(g, monkeypatch)
    if variant == "default":
        return
    res = run_variant(g, VARIANTS[variant], monkeypatch, in_tree_only=variant in IN_TREE_ONLY)
    check_against_oracles(g, res)
    assert_same_bits(base, res, variant)


@pytest.mark.gpu
@pytest.mark.parametrize("g", GRAPHS, ids=GRAPH_IDS)
def test_weighted_ranks_are_reproducible_across_handles_and_build_chunking(g, monkeypatch):
    from memgraph_b200 import personalized as P
    base = defaults(g, monkeypatch)["weighted"]
    for env in ({}, {"MGB200_BUILD_CHUNK_EDGES": "7777"}, {"MGB200_BUILD_CHUNK_EDGES": "7777", "MGB200_IDX_FLAGS": "1"}):
        set_env(monkeypatch, g, env)
        with P.weighted_graph(g.n, g.f, g.t, g.w) as h:
            again = cugraph_runs(g, h, True)
        for key in base:
            assert np.array_equal(base[key][0], again[key][0]), (env, key)


@pytest.mark.gpu
def test_out_weight_sums_follow_input_order(monkeypatch):
    """A hub whose out-edge weights are, in input order, 2^53 and then 2^20 edges of weight 1.0.  Summed left to right
    every 1.0 is a tie that rounds back to 2^53, so out_w = 2^53 exactly; any other order reaches up to 2^53 + 2^20, a
    relative error of 1.2e-10 in everything the hub contributes.  The weight-2^53 edge sits late in the edge list,
    behind a long run of other edges, so that an order-free accumulation is very likely to add 1.0 edges first.

    Nearly all of the hub's mass goes to one target, which gets 85 % of its rank from the hub.  Every row has at most a
    few hundred in-edges (the hub 200), so the different summation order inside the rows leaves about 1e-14 between
    device and oracle -- far below the 1e-12 asserted and the 1e-10 an out-weight sum in another order would cause."""
    from memgraph_b200 import personalized as P
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    rng = np.random.default_rng(21)
    n, hub, target = 1 << 16, 0, 1
    feeders = np.arange(2, 202)                     # out-degree 1, all into the hub: the hub carries a large rank
    filler = 600_000                                # among the other vertices, hub and target untouched
    f = np.concatenate([feeders, rng.integers(202, n, filler), [hub], np.full(1 << 20, hub)])
    t = np.concatenate([np.full(len(feeders), hub), rng.integers(2, n, filler), [target], rng.integers(2, n, 1 << 20)])
    w = np.concatenate([np.ones(len(feeders) + filler), [2.0 ** 53], np.ones(1 << 20)])
    left_to_right = 2.0 ** 53
    for _ in range(4):
        left_to_right += 1.0
    assert left_to_right == 2.0 ** 53 and math.fsum([2.0 ** 53] + [1.0] * 4) == 2.0 ** 53 + 4
    with P.weighted_graph(n, f, t, w) as h:
        got, st = P.cugraph_pagerank(h, max_iterations=10, stop_epsilon=0.0)
    ref, it, _ = oracle_cugraph_pagerank(n, f, t, weights=w, epsilon=0.0, max_iterations=10)
    assert st["iterations"] == it == 10
    hub_targets = np.unique(t[len(feeders) + filler:])
    err = float(np.max(np.abs(got[hub_targets] - ref[hub_targets]) / ref[hub_targets]))
    assert err < 1e-12, err


@pytest.mark.gpu
def test_report_worst_error_against_bound():
    """Runs last in this module: prints the largest observed error / bound per algorithm (all already asserted <= 1)."""
    for key in sorted(_worst, key=str):
        ratio, err, bound = _worst[key]
        print(f"closest to its bound {key}: error {err:.3e}, bound {bound:.3e} (ratio {ratio:.3e})")
    assert all(v[0] <= 1.0 for v in _worst.values())
