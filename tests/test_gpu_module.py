"""-m gpu: the B200 drop-in module, loaded and called the way Memgraph does (through the fake mgp
host), against the oracle, the committed e2e fixtures and the committed rows of the reference's own
module loaded through the very same host."""
import json
import os
import threading

import numpy as np
import pytest

import _fakehost as fh
from _checkers import Oracle
from test_module_host import (MODULE_ARGS, module_rows_digests, oracle_through_module_semantics, run_e2e_fixture,
                              scattered_graph)

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
REL_TOL = 1e-9  # north_star: 1e-6 relative


@pytest.fixture(scope="module")
def oracle():
    return Oracle()


@pytest.fixture(scope="module")
def module():
    m = fh.Module(fh.MODULE_SO)
    yield m
    assert m.close() == 0


def rel_err(a, b):
    return float(np.max(np.abs(a - b) / b)) if len(b) else 0.0


def test_e2e_fixtures(module):
    """mage/tests/e2e/pagerank_test/{test_chain,test_empty,test_influential_node,test_influential_node_transfer}."""
    spec = json.load(open(os.path.join(GOLDEN, "pagerank_e2e_cases.json")))
    for case in spec["cases"]:
        rows = run_e2e_fixture(module, case)
        assert len(rows) == len(case["output"]), case["name"]
        for (node, rank), exp in zip(rows, case["output"]):
            assert node == exp["node"] and abs(rank - exp["rank"]) < spec["tolerance_abs"], case["name"]


@pytest.mark.parametrize("args", [(), (20, 0.85, 0.0, 8), (1000,), (0,), (50, 0.5)])
def test_config1_graph_through_the_module(module, oracle, args):
    n, m = 10_000, 50_000
    gids, src, dst = scattered_graph(n, m, seed=42)
    before = fh.live_objects()
    with fh.Graph(gids, src, dst) as g:
        nodes, ranks = module.call(g, *args)
    assert fh.live_objects() == before
    names = ["max_iterations", "damping_factor", "stop_epsilon", "num_of_threads"]
    kw = dict(zip(names, args))
    order, exp, _ = oracle_through_module_semantics(oracle, gids, src, dst, **kw)
    assert np.array_equal(nodes, order)  # one row per vertex, vertex-iteration (ascending gid) order
    assert rel_err(ranks, exp) < REL_TOL


def test_same_rows_as_the_reference_module(module, oracle):
    """The reference module's rows on this graph are committed as digests (golden/pagerank_reference_module.json); the
    oracle reproduces them bit for bit, so the B200 module is compared with the reference's rows through it."""
    ref = json.load(open(os.path.join(GOLDEN, "pagerank_reference_module.json")))["same_rows"]
    assert [c["args"] for c in ref] == [[], [20, 0.85, 0.0, 4], [7, 0.3, 0.0, 1]]
    gids, src, dst = scattered_graph(3000, 20000, seed=7)
    with fh.Graph(gids, src, dst) as g:
        for case in ref:
            args = case["args"]
            n2, r2, _ = oracle_through_module_semantics(oracle, gids, src, dst, **dict(zip(MODULE_ARGS, args)))
            assert module_rows_digests(oracle, gids, src, dst, args) == case
            n1, r1 = module.call(g, *args)
            assert np.array_equal(n1, n2)
            assert rel_err(r1, r2) < REL_TOL


def test_isolated_vertices_and_self_loops(module, oracle):
    gids = np.array([3, 14, 15, 92, 65], dtype=np.int64)
    src = np.array([3, 3, 14, 14, 92], dtype=np.int64)
    dst = np.array([14, 14, 14, 3, 3], dtype=np.int64)  # multi-edge, self-loop; 15 and 65 isolated
    with fh.Graph(gids, src, dst) as g:
        nodes, ranks = module.call(g, 20, 0.85, 0.0, 1)
    order, exp, _ = oracle_through_module_semantics(oracle, gids, src, dst, max_iterations=20, stop_epsilon=0.0)
    assert np.array_equal(nodes, order) and rel_err(ranks, exp) < REL_TOL


def test_vanished_vertex_analytical_vs_transactional(module):
    gids = np.arange(1, 9, dtype=np.int64)
    src, dst = gids[:-1], gids[1:]
    with fh.Graph(gids, src, dst, transactional=False) as g:
        g.hide_vertex(8)  # FindVertex fails at emission time: analytical mode skips the row
        nodes, ranks = module.call(g)
        assert 8 not in nodes and len(nodes) == len(gids) - 1
    with fh.Graph(gids, src, dst, transactional=True) as g:
        g.hide_vertex(8)
        with pytest.raises(fh.ProcedureError, match=r"^pagerank\.get: Invalid ID!$"):
            module.call(g)


def test_concurrent_calls_from_several_sessions(module, oracle):
    """tests/e2e/concurrent_query_modules: the same procedure runs concurrently from several queries."""
    graphs = [scattered_graph(2000 + 100 * i, 15000, seed=100 + i) for i in range(6)]
    results = [None] * len(graphs)

    def work(i):
        gids, src, dst = graphs[i]
        with fh.Graph(gids, src, dst) as g:
            results[i] = module.call(g, 30, 0.85, 0.0, 1)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(graphs))]
    [t.start() for t in threads]
    [t.join() for t in threads]
    for i, (gids, src, dst) in enumerate(graphs):
        order, exp, _ = oracle_through_module_semantics(oracle, gids, src, dst, max_iterations=30, stop_epsilon=0.0)
        assert np.array_equal(results[i][0], order) and rel_err(results[i][1], exp) < REL_TOL


def test_abort_between_iteration_batches(module):
    n = 50_000
    gids = np.arange(n, dtype=np.int64)
    rng = np.random.default_rng(1)
    src, dst = rng.integers(0, n, 400_000), rng.integers(0, n, 400_000)
    with fh.Graph(gids, src, dst) as g:
        module.call(g, 5, 0.85, 0.0, 1)
        assert g.abort_polls() > 0
