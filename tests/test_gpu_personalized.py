"""-m gpu: cuGraph-semantics PageRank (uniform / personalised teleport, include/mgb200_personalized.h) against
oracle/cugraph_pagerank_oracle.c, which is pinned on the reference's own cuGraph e2e fixtures (test_cugraph_oracle.py).
Tolerance 1e-9 relative (1e-12 absolute floor for exact zeros) and EQUAL iteration counts; the fixtures themselves are
also run through the device path."""
import numpy as np
import pytest

from test_cugraph_oracle import FIXTURES, fixture_arrays, oracle_cugraph_pagerank

pytestmark = pytest.mark.gpu


def gpu(n, f, t, pers=None, **kw):
    from memgraph_b200 import personalized as P
    pv, pw = (pers if pers is not None else (None, None))
    return P.cugraph_pagerank_from_edges(n, np.asarray(f, dtype=np.uint64), np.asarray(t, dtype=np.uint64),
                                         personalization_vertices=pv, personalization_values=pw, **kw)


def close(got, ref):
    return float(np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1e-3))) < 1e-9


@pytest.mark.parametrize("fx", [f for f in FIXTURES if f["nodes"]], ids=lambda f: f["name"])
def test_reference_e2e_fixtures_on_the_device(fx):
    dense, f, t, pers = fixture_arrays(fx)
    ranks, st = gpu(len(dense), f, t, pers)
    ref, it, conv = oracle_cugraph_pagerank(len(dense), f, t, personalization=pers)
    assert st["iterations"] == it and bool(st["converged"]) == conv
    assert close(ranks, ref)
    for gid, want in fx["expected"]:
        digits = len(str(want).split(".")[1]) if "." in str(want) else 0
        assert abs(ranks[dense[gid]] - want) < max(1.5 * 10.0 ** -digits, 2e-5)


@pytest.mark.parametrize("seed", range(4))
def test_random_graphs_uniform_and_personalised(seed, monkeypatch):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(200, 5000))
    m = int(n * rng.integers(2, 9))
    f, t = rng.integers(0, n, m), rng.integers(0, n, m)
    monkeypatch.setenv("MGB200_HEAVY_MIN_DEGREE", "16")  # heavy rows take part
    for pers in [None, (rng.integers(0, n, 5), rng.uniform(0.1, 2.0, 5)), (np.array([7, 7, 3]), np.array([1.0, 2.0, 0.5]))]:
        for kw in [dict(), dict(max_iterations=7, stop_epsilon=0.0), dict(damping_factor=0.5, stop_epsilon=1e-12, max_iterations=300)]:
            got, st = gpu(n, f, t, pers, **kw)
            ref, it, conv = oracle_cugraph_pagerank(n, f, t, personalization=pers,
                                                    alpha=kw.get("damping_factor", 0.85), epsilon=kw.get("stop_epsilon", 1e-5),
                                                    max_iterations=kw.get("max_iterations", 100))
            assert st["iterations"] == it and bool(st["converged"]) == conv, (seed, kw)
            assert close(got, ref), (seed, kw)
            assert abs(got.sum() - 1.0) < 1e-9  # dangling mass is redistributed: the vector stays stochastic


def test_rmat_scale18_all_row_classes_and_errors():
    import memgraph_b200 as mg
    from memgraph_b200 import personalized as P
    scale = 18
    n, m = 1 << scale, 16 << scale
    f, t = mg.rmat_edges_host(scale, m)
    seeds = (np.array([0, 12345, 99999]), np.array([0.2, 0.5, 0.3]))
    with mg.PageRankGraph.from_arrays(n, f, t) as g:
        assert g.info["heavy_rows"] > 0 and g.info["sell_rows"] > 0 and g.info["zero_rows"] > 0
        got, st = P.cugraph_pagerank(g, *seeds, max_iterations=30, stop_epsilon=1e-9)
        plain, st2 = P.cugraph_pagerank(g, max_iterations=20, stop_epsilon=0.0)
        again, _ = P.cugraph_pagerank(g, max_iterations=20, stop_epsilon=0.0)
        assert np.array_equal(plain, again)  # fixed reduction trees: bit-reproducible
        # the in-tree PageRank still works on the same handle afterwards
        ranks, _ = g.run(max_iterations=5, stop_epsilon=0.0)
        assert abs(ranks.sum() - 1.0) < 1e-12
        with pytest.raises(mg.MgB200Error):
            P.cugraph_pagerank(g, [n + 5], [1.0])
        with pytest.raises(mg.MgB200Error):
            P.cugraph_pagerank(g, [1, 2], [0.0, 0.0])
    ref, it, conv = oracle_cugraph_pagerank(n, f, t, personalization=seeds, epsilon=1e-9, max_iterations=30)
    assert st["iterations"] == it and close(got, ref)
    ref2, it2, _ = oracle_cugraph_pagerank(n, f, t, epsilon=0.0, max_iterations=20)
    assert st2["iterations"] == it2 == 20 and close(plain, ref2)


@pytest.mark.parametrize("seed", range(3))
def test_edge_weights(seed, monkeypatch):
    """weight_property path: one non-negative FP64 weight per edge (mgb200_graph_create_host_weighted_u32); every gathered
    value is multiplied by its weight, contributions are divided by the out-WEIGHT sums.  Zero weights are legal (a vertex
    whose out-edges all weigh 0 is dangling).  Tolerance: the out-weight sums equal the oracle's bit for bit (both add
    in input edge order), but the device sums every row in source-label order, the oracle in edge order."""
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(300, 4000))
    m = int(n * rng.integers(3, 10))
    f, t = rng.integers(0, n, m), rng.integers(0, n, m)
    w = rng.uniform(0.0, 5.0, m)
    w[rng.integers(0, m, m // 20)] = 0.0
    w[f == f[0]] = 0.0  # a vertex whose out-edges all weigh 0: dangling, contributes nothing along them
    monkeypatch.setenv("MGB200_HEAVY_MIN_DEGREE", "16")
    for pers in [None, (rng.integers(0, n, 4), rng.uniform(0.1, 1.0, 4))]:
        got, st = gpu(n, f, t, pers, weights=w, stop_epsilon=1e-10, max_iterations=200)
        ref, it, conv = oracle_cugraph_pagerank(n, f, t, weights=w, personalization=pers, epsilon=1e-10, max_iterations=200)
        assert st["iterations"] == it and bool(st["converged"]) == conv
        assert close(got, ref)
    # a constant weight cancels: identical to the unweighted handle up to rounding
    a, _ = gpu(n, f, t, None, weights=np.full(m, 2.5), max_iterations=15, stop_epsilon=0.0)
    b, _ = gpu(n, f, t, None, max_iterations=15, stop_epsilon=0.0)
    assert float(np.max(np.abs(a - b) / b)) < 1e-12


def test_weighted_handle_keeps_the_in_tree_algorithms_unweighted():
    import memgraph_b200 as mg
    from memgraph_b200 import personalized as P
    from _checkers import Oracle
    rng = np.random.default_rng(8)
    n, m = 2000, 15000
    f, t = rng.integers(0, n, m), rng.integers(0, n, m)
    with P.weighted_graph(n, f, t, rng.uniform(0.5, 2.0, m)) as g:
        ranks, st = g.run(max_iterations=20, stop_epsilon=0.0)
    ref, it = Oracle().pagerank(n, f, t, max_iterations=20, stop_epsilon=0.0)
    assert st.iterations == it and float(np.max(np.abs(ranks - ref) / ref)) < 1e-9
    with pytest.raises(mg.MgB200Error):
        P.weighted_graph(n, f, t, -np.ones(m))
