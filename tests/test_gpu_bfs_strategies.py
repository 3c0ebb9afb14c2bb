"""The breadth-first expansion (memgraph_b200/csrc/bfs.cu) under every traversal strategy, on graphs shaped to reach its
segment, bitmap and direction boundaries (tests/_bfs_graphs.py).

MGB200_BFS_STRATEGY pins the per-level choice between top-down and bottom-up, so each graph runs every path whatever
its size.  Distances must equal the oracle (oracle/bfs_oracle.c) exactly, and every statistic but traverse_ms must equal
the CPU model of mgb200_bfs_run: bench.py derives its roofline bytes from edges_inspected, reached and levels, and
reports kernel_launches.

The CPU tests (no marker) check that the graphs reach their boundaries, that the model's distances equal the oracle's
under every strategy and bounds set, that the model takes the auto switch where the graphs were built to make it switch,
and that it reproduces what tests/test_gpu_bfs.py asserts at RMAT scale-20."""
import ctypes
import random

import numpy as np
import pytest

import _bfs_graphs as B
from _checkers import BfsOracle, oracle_rmat_edges

GRAPHS = B.all_graphs()
GRAPH_IDS = [g.name for g in GRAPHS]
STAT_FIELDS = ("levels", "top_down_levels", "bottom_up_levels", "reached", "edges_inspected", "kernel_launches")
ENV = "MGB200_BFS_STRATEGY"

_models, _oracle = {}, {}


def model(g):
    if g.name not in _models:
        _models[g.name] = B.Model(g.n, g.f, g.t)
    return _models[g.name]


def oracle(g, source, direction, lower, upper):
    key = (g.name, source, direction, lower, upper)
    if key not in _oracle:
        _oracle[key] = BfsOracle().distances(g.n, g.f, g.t, source, direction, lower, upper)
    return _oracle[key]


def deepest(g, source, direction):
    return int(model(g).trace(source, direction)[0].max())


# ---- CPU: the graphs reach their boundaries, the model agrees with the oracle ------------------------------------------

def sorted_out(g, u):
    return np.sort(g.t[g.f == u]).astype(np.int64)


@pytest.mark.parametrize("g", GRAPHS, ids=GRAPH_IDS)
def test_graphs_reach_their_boundaries(g):
    want = g.intended
    assert all(0 <= s < g.n for s in g.sources)
    if "hub_degrees" in want:
        half = want["half"]
        for h, d in zip(want["hubs"], want["hub_degrees"]):
            targets = sorted_out(g, h)
            assert len(targets) == d and len(np.unique(targets)) == d, h
            assert g.degree(h + half, B.IN) == d  # the mirror
        assert max(-(-d // B.SEG_EDGES) for d in want["hub_degrees"]) > 32
        out = sorted_out(g, want["repeat_hub"])
        at = np.flatnonzero(out == want["repeat_target"])
        assert len(at) == B.REPEAT_HUB["repeats"] and at[0] < 1023 and at[-1] > 2048  # across both segment edges
        assert np.all(np.diff(at) == 1) and len(np.unique(out)) == len(out) - len(at) + 1
    if "hub_positions" in want:
        level1 = sorted_out(g, 0)
        assert level1.tolist() == want["level1"] and len(level1) <= B.SEG_EDGES  # one work item: queue in this order
        degs = np.array([g.degree(v, B.OUT) for v in level1])
        hubs = np.flatnonzero(degs)
        assert {int(p): int(degs[p]) for p in hubs} == want["hub_positions"]
        runs = np.diff(np.concatenate([[-1], hubs, [len(level1)]])) - 1
        assert runs[0] >= 100 and runs[-1] >= 100 and max(runs[1:-1]) >= 100 and 0 in runs[1:-1]
        assert g.degree(want["half"], B.IN) == len(level1)
    if "junctions" in want:
        for u, (a, b) in zip(g.sources, want["junctions"]):
            assert (g.degree(u, B.OUT), g.degree(u, B.IN)) == (a, b + 1)  # b fresh in-neighbours and the witness
            nbrs = np.concatenate([g.t[g.f == u], g.f[g.t == u]]).astype(np.int64)
            nbrs = nbrs[nbrs != u + 1 + a + b]  # the witness
            assert len(np.unique(nbrs)) == a + b and all(g.degree(v, B.BOTH) == 1 for v in nbrs)
        assert {a % B.SEG_EDGES for a, _ in want["junctions"]} >= {0, 1, B.SEG_EDGES - 1}
        assert any(a + b > a > 0 and a % B.SEG_EDGES == 0 for a, b in want["junctions"])  # the junction on a segment edge
    if "frontier" in want and g.n > 2:
        assert sorted_out(g, want["source"]).tolist() == want["frontier"]
        assert set(want["frontier"]) == {v for v in (0, 31, 32, 63, 64, g.n - 1) if v < g.n}
        for p in want["frontier"]:
            child = sorted_out(g, p)
            assert len(child) == 1 and g.degree(int(child[0]), B.IN) == 1
    if "switch_sources" in want:
        assert 1000 <= g.n <= 10000
    if "path_levels" in want:
        assert deepest(g, 0, B.OUT) >= want["path_levels"] >= 3000
    if want.get("m0"):
        assert g.m == 0
    if "isolated" in want:
        assert g.degree(want["isolated"], B.BOTH) == 0
        assert g.degree(want["self_loop_only"], B.BOTH) == 2 and sorted_out(g, want["self_loop_only"]).tolist() == [1]
        pairs = list(zip(g.f.tolist(), g.t.tolist()))
        assert all(pairs.count(e) >= 2 for e in want["duplicates"])
        assert g.degree(want["no_out"], B.OUT) == 0 < g.degree(want["no_out"], B.IN)


def test_every_boundary_is_reached_by_some_graph():
    ns = {g.n for g in GRAPHS}
    assert {1, 2, 31, 32, 33, 63, 64, 65, 1025, 4097} <= ns
    assert any(g.m == 0 for g in GRAPHS) and any(g.n == 1 and g.m == 1 for g in GRAPHS)


@pytest.mark.parametrize("g", GRAPHS, ids=GRAPH_IDS)
def test_model_distances_equal_the_oracle(g):
    m = model(g)
    for source in g.sources:
        for direction in (B.OUT, B.IN, B.BOTH):
            for strategy in B.STRATEGIES:
                for lower, upper in B.bounds_sets(deepest(g, source, direction)):
                    dist, st = m.run(source, direction, lower, upper, strategy)
                    assert np.array_equal(dist, oracle(g, source, direction, lower, upper)), (
                        source, direction, strategy, lower, upper)
                    assert st["reached"] >= int((dist > 0).sum())


def test_model_switches_top_down_bottom_up_top_down_on_auto_switch():
    g = next(g for g in GRAPHS if g.name == "auto_switch")
    m = model(g)
    for direction, source in g.intended["switch_sources"].items():
        _, st = m.run(source, direction)
        depth, levels = m.trace(source, direction)
        assert B.strategy_sequence(levels, st).startswith("TBT"), direction
        if direction != B.BOTH:  # pinned to the exact boundary of the switch
            assert levels[1]["m_f"] == levels[1]["m_u"] // B.SWITCH_DIVISOR + 1 and levels[1]["nf"] > 1024
            assert levels[2]["m_f"] == levels[2]["m_u"] // B.SWITCH_DIVISOR and levels[2]["nf"] > 1024


def test_model_reproduces_the_rmat_scale20_facts():
    """tests/test_gpu_bfs.py asserts these of the device at RMAT scale-20, direction OUT, source 0."""
    scale = 20
    n, m = 1 << scale, 16 << scale
    f, t = oracle_rmat_edges(scale, m)
    md = B.Model(n, f, t)
    dist, st = md.run(0, B.OUT)
    assert np.array_equal(dist, BfsOracle().distances(n, f, t, 0, B.OUT))
    assert st["bottom_up_levels"] >= 1 and st["top_down_levels"] >= 1
    assert st["reached"] == int((dist > 0).sum())
    assert st["edges_inspected"] < m


# ---- GPU -----------------------------------------------------------------------------------------------------------------

_handles = {}


@pytest.fixture(scope="module")
def bfs():
    from memgraph_b200 import bfs
    yield bfs
    for h in _handles.values():
        h.close()
    _handles.clear()


def handle(bfs, g):
    if g.name not in _handles:
        _handles[g.name] = bfs.BfsGraph(g.n, g.f, g.t)
    return _handles[g.name]


def set_strategy(monkeypatch, strategy):
    if strategy == "auto":
        monkeypatch.delenv(ENV, raising=False)  # the default path, as bench.py runs it
    else:
        monkeypatch.setenv(ENV, strategy)


def run(h, source, direction, lower=1, upper=B.INT64_MAX):
    dist, st = h.distances(source, direction, lower, upper)
    return dist.astype(np.int64), {k: st[k] for k in STAT_FIELDS}


@pytest.mark.gpu
@pytest.mark.parametrize("strategy", B.STRATEGIES)
@pytest.mark.parametrize("direction", list(B.DIRECTIONS), ids=list(B.DIRECTIONS))
@pytest.mark.parametrize("g", GRAPHS, ids=GRAPH_IDS)
def test_boundary_graph(bfs, g, direction, strategy, monkeypatch):
    d = B.DIRECTIONS[direction]
    h = handle(bfs, g)
    set_strategy(monkeypatch, strategy)
    for source in g.sources:
        for lower, upper in B.bounds_sets(deepest(g, source, d)):
            dist, st = run(h, source, d, lower, upper)
            where = (source, lower, upper)
            assert np.array_equal(dist, oracle(g, source, d, lower, upper)), where
            assert st == model(g).run(source, d, lower, upper, strategy)[1], where


def sm_count():
    from memgraph_b200 import _native as N
    sms = ctypes.c_int(0)
    assert N.lib().mgb200_device_info(0, None, 0, ctypes.byref(sms), None) == 0
    return sms.value


_rmat = {}


def rmat_model(scale):
    if scale not in _rmat:
        n, m = 1 << scale, 16 << scale
        f, t = oracle_rmat_edges(scale, m)
        _rmat[scale] = (n, f, t, B.Model(n, f, t))
    return _rmat[scale]


@pytest.mark.gpu
@pytest.mark.parametrize("scale,strategy", [(21, "bottom_up"), (20, "top_down"), (20, "auto")])
@pytest.mark.parametrize("direction", list(B.DIRECTIONS), ids=list(B.DIRECTIONS))
def test_rmat_grid_stride_loops(bfs, scale, strategy, direction, monkeypatch):
    """Scale-21 has more vertices than the bottom-up grid has threads, and a scale-20 level has more top-down work
    items than the top-down grid has warps: both grid-stride loops go round more than once."""
    d = B.DIRECTIONS[direction]
    n, f, t, md = rmat_model(scale)
    sms = sm_count()
    set_strategy(monkeypatch, strategy)
    with bfs.BfsGraph(n, f, t) as h:
        for source in (0, n // 3, n - 1):
            _, levels = md.trace(source, d, strategy)
            if strategy == "bottom_up":
                assert (n + 31) // 32 * 32 > B.BOTTOM_UP_THREADS_PER_SM * sms
            if strategy == "top_down" and source == 0:
                assert max(r["segments"] for r in levels) > B.TOP_DOWN_WARPS_PER_SM * sms
            dist, st = run(h, source, d)
            assert np.array_equal(dist, BfsOracle().distances(n, f, t, source, d)), source
            assert st == md.run(source, d, strategy=strategy)[1], source


def state_calls():
    """the shuffled call sequence of test_state_does_not_carry_between_runs"""
    calls = []
    for g in GRAPHS:
        if g.name in ("hub_segments", "auto_switch"):
            k = {s: max(deepest(g, s, d) for d in range(3)) for s in g.sources}
            for s in g.sources[:3]:
                for d in range(3):
                    for strategy in B.STRATEGIES + ("auto_explicit",):
                        for lower, upper in ((1, B.INT64_MAX), (2, 3), (k[s], k[s]), (1, 0)):
                            calls.append((g.name, s, d, strategy, lower, upper))
    random.Random(7).shuffle(calls)
    assert len(calls) > 100
    return calls


@pytest.mark.gpu
def test_state_does_not_carry_between_runs(bfs, monkeypatch):
    """One handle per graph runs the calls in shuffled order; each result must equal a fresh handle's."""
    by_name = {g.name: g for g in GRAPHS}
    calls = state_calls()
    reused = {name: bfs.BfsGraph(by_name[name].n, by_name[name].f, by_name[name].t) for name in {c[0] for c in calls}}
    try:
        for i, (name, s, d, strategy, lower, upper) in enumerate(calls):
            g = by_name[name]
            if strategy == "auto_explicit":
                monkeypatch.setenv(ENV, "auto")
            else:
                set_strategy(monkeypatch, strategy)
            got = run(reused[name], s, d, lower, upper)
            if i % 4 == 0:  # a fresh handle for every fourth call, the model and the oracle for all
                with bfs.BfsGraph(g.n, g.f, g.t) as fresh:
                    again = run(fresh, s, d, lower, upper)
                assert np.array_equal(got[0], again[0]) and got[1] == again[1], (i, name, s, d, strategy)
            assert np.array_equal(got[0], oracle(g, s, d, lower, upper)), (i, name, s, d, strategy)
            model_strategy = "auto" if strategy == "auto_explicit" else strategy
            assert got[1] == model(g).run(s, d, lower, upper, model_strategy)[1], (i, name, s, d, strategy)
    finally:
        for h in reused.values():
            h.close()


@pytest.mark.gpu
def test_benchmark_input_path(bfs, monkeypatch):
    """bench.py --workload bfs: the scale-24 RMAT stream generated on the device, a handle from
    mgb200_bfs_graph_create_device, the first of bench's seeded sources.  Bit-identical to the create_host handle of the
    same edges and equal to the oracle; once more with the distances written to device memory."""
    import memgraph_b200 as mg
    from memgraph_b200 import _native as N
    monkeypatch.delenv(ENV, raising=False)
    lib = N.lib()
    scale, seed = 24, 42
    n, m = 1 << scale, 16 << scale
    ptrs = []

    def dev(nbytes):
        p = N.vp()
        assert lib.mgb200_device_malloc(0, nbytes, ctypes.byref(p)) == 0
        ptrs.append(p)
        return p

    try:
        d_from, d_to = dev(4 * m), dev(4 * m)
        mg.rmat_edges_device(scale, m, d_from, d_to, seed=seed, device=0)
        on_device = bfs.BfsGraph.from_device(n, m, d_from, d_to)
        f, t = mg.rmat_edges_host(scale, m, seed=seed)
        back = np.empty(m, dtype=np.uint32)
        assert lib.mgb200_copy_to_host(0, back.ctypes.data, d_from, 4 * m) == 0
        assert np.array_equal(back, f)
        assert lib.mgb200_copy_to_host(0, back.ctypes.data, d_to, 4 * m) == 0
        assert np.array_equal(back, t)
        del back
        on_host = bfs.BfsGraph(n, f, t)
        rng = np.random.default_rng(seed)
        sources = [0] + [int(x) for x in rng.integers(0, n, size=8)][:2]  # bench.py run_bfs_arm, same seed
        with on_device, on_host:
            for s in sources:
                dist, st = run(on_device, s, B.OUT)
                dist_h, st_h = run(on_host, s, B.OUT)
                assert np.array_equal(dist, dist_h) and st == st_h, s
                assert np.array_equal(dist, BfsOracle().distances(n, f, t, s, B.OUT)), s
            d_dist = dev(4 * n)
            stats = N.BfsStats()
            assert lib.mgb200_bfs_run(on_device._h, sources[1], B.OUT, 1, B.INT64_MAX, d_dist, 1,
                                      ctypes.byref(stats)) == 0
            got = np.empty(n, dtype=np.int32)
            assert lib.mgb200_copy_to_host(0, got.ctypes.data, d_dist, 4 * n) == 0
            dist_h, st_h = run(on_host, sources[1], B.OUT)
            assert np.array_equal(got.astype(np.int64), dist_h)
            assert {k: getattr(stats, k) for k in STAT_FIELDS} == st_h
    finally:
        for p in ptrs:
            lib.mgb200_device_free(0, p)


@pytest.mark.gpu
def test_errors(bfs, monkeypatch):
    from memgraph_b200 import _native as N
    from memgraph_b200.pagerank import MgB200Error
    lib = N.lib()
    monkeypatch.delenv(ENV, raising=False)
    # an endpoint equal to n: refused, and no handle comes back
    n = 10
    f, t = np.array([0, 3, n], dtype=np.uint32), np.array([1, 4, 2], dtype=np.uint32)
    ptrs = []
    try:
        for a in (f, t):
            p = N.vp()
            assert lib.mgb200_device_malloc(0, a.nbytes, ctypes.byref(p)) == 0
            ptrs.append(p)
            assert lib.mgb200_copy_to_device(0, p, a.ctypes.data, a.nbytes) == 0
        h = N.vp(0x1234)
        assert lib.mgb200_bfs_graph_create_device(0, n, len(f), ptrs[0], ptrs[1], ctypes.byref(h)) == N.ERR_INVALID_ARGUMENT
        assert h.value is None
        assert "edge endpoint out of range" in lib.mgb200_last_error().decode()
        with pytest.raises(MgB200Error, match="edge endpoint out of range"):
            bfs.BfsGraph.from_device(n, len(f), ptrs[0], ptrs[1])
    finally:
        for p in ptrs:
            lib.mgb200_device_free(0, p)
    with bfs.BfsGraph(n, [0, 3], [1, 4]) as g:
        for source in (n, n + 5, 2 ** 63):
            with pytest.raises(MgB200Error, match="source vertex out of range"):
                g.distances(source)
        for direction in (-1, 3):
            with pytest.raises(MgB200Error, match="invalid argument"):
                g.distances(0, direction)
        for value in ("sideways", "", "TOP_DOWN", "top-down", "auto "):
            monkeypatch.setenv(ENV, value)
            with pytest.raises(MgB200Error, match=f"unknown MGB200_BFS_STRATEGY '{value}'"):
                g.distances(0)
        monkeypatch.setenv(ENV, "alternate")
        assert g.distances(0)[0].tolist() == [-1, 1] + [-1] * (n - 2)
    with bfs.BfsGraph(0, [], []) as empty:
        with pytest.raises(MgB200Error, match="source vertex out of range"):
            empty.distances(0)
