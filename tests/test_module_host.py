"""No-GPU tests of the drop-in boundary: what the REFERENCE's own pagerank module returned through the
fake mgp host (BASELINE config #1, committed under golden/) pins the oracle's module semantics, then
the B200 module is checked for everything that does not need a device: exports, registered
signature, argument validation, error texts, loud failure without a GPU, no leaked host objects."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

import _fakehost as fh
from _checkers import Oracle, sha256_of

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODULE_ARGS = ["max_iterations", "damping_factor", "stop_epsilon", "num_of_threads"]

EXPECTED_SIGNATURE = ("get(max_iterations = 100 :: INTEGER, damping_factor = 0.84999999999999998 :: FLOAT, "
                      "stop_epsilon = 1.0000000000000001e-05 :: FLOAT, num_of_threads = 1 :: INTEGER) :: "
                      "(node :: NODE, rank :: FLOAT)")


@pytest.fixture(scope="module")
def oracle():
    return Oracle()


@pytest.fixture(scope="module")
def ref_module():
    """What the reference's pagerank.so (oracle/_ref/pagerank_reference.so) did when loaded and called through this
    host: tests/golden/pagerank_reference_module.json, written by make_golden.py."""
    return json.load(open(os.path.join(GOLDEN, "pagerank_reference_module.json")))


@pytest.fixture(scope="module")
def b200_module():
    m = fh.Module(fh.MODULE_SO)
    yield m
    assert m.close() == 0


def scattered_graph(n, m, seed):
    """Non-contiguous, unsorted gids, like a real database hands out."""
    rng = np.random.default_rng(seed)
    gids = rng.choice(np.arange(10 * n + 7, dtype=np.int64), size=n, replace=False)
    s = rng.integers(0, n, size=m)
    t = rng.integers(0, n, size=m)
    return gids, gids[s], gids[t]


def oracle_through_module_semantics(oracle, gids, src, dst, **kw):
    """What pagerank.get must return: dense ids in ascending-gid visit order, one row per vertex."""
    order = np.sort(gids)
    frm, to = oracle.map_gids(order, src, dst)
    # the module sees each vertex's out-edges grouped by source in visit order
    perm = np.argsort(frm, kind="stable")
    ranks, it = oracle.pagerank(len(order), frm[perm], to[perm], **kw)
    return order, ranks, it


# ---- the reference's own module through this host (config #1), pinning the oracle's module semantics --------

def test_reference_module_signature(ref_module):
    assert ref_module["signature"] == EXPECTED_SIGNATURE


def module_rows_digests(oracle, gids, src, dst, args):
    """(nodes, ranks) the oracle says pagerank.get(*args) returns, as the digests the golden file stores."""
    order, exp, _ = oracle_through_module_semantics(oracle, gids, src, dst, **dict(zip(MODULE_ARGS, args)))
    return {"args": list(args), "nodes_sha256": sha256_of(order, np.int64), "ranks_sha256": sha256_of(exp)}


def test_config1_reference_module_erdos_renyi_10k_50k(ref_module, oracle):
    """BASELINE config #1: 10k-node / 50k-edge Erdos-Renyi graph through the reference algorithm and
    the C-ABI module loader, no GPU.  Default args and (20, 0.85, 0.0, 8).  Same algorithm, same order
    of operations, so the reference module's rows and the oracle's agree bit for bit."""
    gids, src, dst = scattered_graph(10_000, 50_000, seed=42)
    assert [c["args"] for c in ref_module["config1"]] == [[], [20, 0.85, 0.0, 8]]
    for case in ref_module["config1"]:
        assert module_rows_digests(oracle, gids, src, dst, case["args"]) == case


def e2e_fixture_graph(case):
    """(gid_of, gids, src, dst) of an e2e fixture: gids follow creation order."""
    ids = sorted({v for e in case["edges_by_node_id"] for v in e})
    gid_of = {node_id: 1000 + 3 * i for i, node_id in enumerate(ids)}
    src = [gid_of[a] for a, _ in case["edges_by_node_id"]]
    dst = [gid_of[b] for _, b in case["edges_by_node_id"]]
    return gid_of, list(gid_of.values()), src, dst


def e2e_fixture_rows(gid_of, nodes, ranks):
    id_of = {v: k for k, v in gid_of.items()}
    return sorted([id_of[int(gid)], float(r)] for gid, r in zip(nodes, ranks))  # ORDER BY node ASC


def run_e2e_fixture(module, case):
    gid_of, gids, src, dst = e2e_fixture_graph(case)
    with fh.Graph(gids, src, dst) as g:
        nodes, ranks = module.call(g, *case["call_args"])
    return e2e_fixture_rows(gid_of, nodes, ranks)


def test_reference_module_e2e_fixtures(ref_module, oracle):
    """mage/tests/e2e/pagerank_test/*: expected rows at abs 1e-3 (test_module.py:21,76); the oracle
    returns exactly the reference module's rows."""
    spec = json.load(open(os.path.join(GOLDEN, "pagerank_e2e_cases.json")))
    assert {c["name"] for c in spec["cases"]} == {"test_chain", "test_empty", "test_influential_node",
                                                  "test_influential_node_transfer"} == set(ref_module["e2e"])
    for case in spec["cases"]:
        rows = ref_module["e2e"][case["name"]]
        gid_of, gids, src, dst = e2e_fixture_graph(case)
        order, ranks, _ = oracle_through_module_semantics(oracle, gids, src, dst,
                                                          **dict(zip(MODULE_ARGS, case["call_args"])))
        assert e2e_fixture_rows(gid_of, order, ranks) == rows, case["name"]
        assert len(rows) == len(case["output"])
        for (node, rank), exp in zip(rows, case["output"]):
            assert node == exp["node"] and abs(rank - exp["rank"]) < spec["tolerance_abs"], case["name"]


def test_reference_module_unit_vectors_through_host(ref_module, oracle):
    spec = json.load(open(os.path.join(GOLDEN, "pagerank_unit_vectors.json")))
    through_host = {c["case"]: c for c in ref_module["unit_vectors"]}
    for i, case in enumerate(spec["cases"]):
        if case["m"] != len(case["edges"]):
            assert i not in through_host
            continue
        gids = np.arange(case["n"], dtype=np.int64) * 5 + 11
        e = np.array(case["edges"], dtype=np.int64).reshape(-1, 2)
        nodes, ranks = np.array(through_host[i]["nodes"], dtype=np.int64), np.array(through_host[i]["ranks"])
        order, exp_oracle, _ = oracle_through_module_semantics(oracle, gids, gids[e[:, 0]] if len(e) else [],
                                                               gids[e[:, 1]] if len(e) else [])
        assert np.array_equal(order, nodes) and np.array_equal(exp_oracle, ranks)
        assert np.array_equal(nodes, gids)
        exp = np.array(case["expected"])
        if len(exp):
            err = np.abs(ranks - exp)
            assert err.max() < 1e-3 and err.mean() < 1e-3


def test_host_argument_validation(ref_module, b200_module):
    """The host rejects malformed calls before the procedure runs; the thread-count error is the
    reference module's text under the calling module's name."""
    with fh.Graph([1, 2], [1], [2]) as g:
        with pytest.raises(fh.ProcedureError, match="must be of type FLOAT"):
            b200_module.call(g, 10, 1)  # integer literal for damping_factor is rejected (cypher_types.hpp:95,104)
        with pytest.raises(fh.ProcedureError, match="requires between 0 and 4 arguments"):
            b200_module.call(g, 10, 0.85, 1e-5, 1, 7)
        with pytest.raises(fh.ProcedureError) as err:
            b200_module.call(g, 10, 0.85, 1e-5, 0)
    reference_text = ref_module["zero_threads_error"]
    assert reference_text == "pagerank_reference.get: Number of threads can't be zero (0)!"
    assert str(err.value) == "pagerank.get: " + reference_text.split(": ", 1)[1]


# ---- the B200 module: everything that needs no device -------------------------------------------------------

def test_b200_module_exports_and_imports(ref_module):
    out = subprocess.run(["nm", "-D", "--defined-only", fh.MODULE_SO], capture_output=True, text=True, check=True).stdout
    assert " T mgp_init_module" in out and " T mgp_shutdown_module" in out
    und = subprocess.run(["nm", "-D", "--undefined-only", fh.MODULE_SO], capture_output=True, text=True, check=True).stdout
    imported = sorted(line.split()[-1] for line in und.splitlines() if " mgp_" in line)
    strong = sorted(line.split()[-1] for line in und.splitlines() if " U mgp_" in line)
    # exactly the reference module's 30 imports are strong; the optional extras are weak
    reference_imports = sorted("""mgp_list_at mgp_value_get_int mgp_value_get_double mgp_value_make_int
        mgp_value_make_double mgp_value_make_vertex mgp_value_destroy mgp_type_int mgp_type_float mgp_type_node
        mgp_module_add_read_procedure mgp_proc_add_opt_arg mgp_proc_add_result mgp_graph_approximate_vertex_count
        mgp_graph_approximate_edge_count mgp_graph_iter_vertices mgp_vertices_iterator_get mgp_vertices_iterator_next
        mgp_vertices_iterator_destroy mgp_vertex_iter_out_edges mgp_edges_iterator_get mgp_edges_iterator_next
        mgp_edges_iterator_destroy mgp_edge_get_to mgp_vertex_get_id mgp_graph_get_vertex_by_id
        mgp_graph_is_transactional mgp_result_new_record mgp_result_record_insert mgp_result_set_error_msg""".split())
    assert strong == reference_imports
    assert set(imported) - set(strong) <= {"mgp_must_abort", "mgp_result_reserve", "mgp_log"}
    # nothing CUDA-related is left undefined: the runtime is linked statically (dlopen RTLD_NOW | RTLD_LOCAL)
    assert "cuda" not in und.lower() and "nccl" not in und.lower()
    assert ref_module["imports"] == reference_imports


def test_b200_module_signature_is_the_reference_signature(b200_module, ref_module):
    assert b200_module.signature() == EXPECTED_SIGNATURE == ref_module["signature"]


def test_b200_module_error_paths_without_device(b200_module):
    before = fh.live_objects()
    with fh.Graph([5, 9, 2], [5, 9], [9, 2]) as g:
        # num_of_threads == 0: the reference's text, produced before any device work
        with pytest.raises(fh.ProcedureError, match=r"^pagerank\.get: Number of threads can't be zero \(0\)!$"):
            b200_module.call(g, 100, 0.85, 1e-5, 0)
        with pytest.raises(fh.ProcedureError, match="must be of type FLOAT"):
            b200_module.call(g, 10, 1)
        import conftest
        if not conftest.HAVE_GPU:
            # no CPU fallback: a call that needs the device fails loudly through the procedure's error message
            with pytest.raises(fh.ProcedureError, match=r"^pagerank\.get: CUDA error"):
                b200_module.call(g)
    # empty graph: zero rows, no device needed (test_empty fixture)
    with fh.Graph([], [], []) as g:
        nodes, ranks = b200_module.call(g)
        assert len(nodes) == 0 and len(ranks) == 0
        with pytest.raises(fh.ProcedureError, match="Number of threads can't be zero"):
            b200_module.call(g, 100, 0.85, 1e-5, 0)
    assert fh.live_objects() == before  # iterators / values released on the error paths too


def test_b200_module_polls_must_abort_during_ingest(b200_module):
    n = 10_000
    gids = np.arange(n, dtype=np.int64)
    with fh.Graph(gids, gids[:-1], gids[1:]) as g:
        g.set_abort(True)
        with pytest.raises(fh.ProcedureError, match="aborted"):
            b200_module.call(g)
        assert g.abort_polls() >= 1


MGP_ENUMS = {"MGP_ERROR_": "mgp_error", "MGP_LOG_LEVEL_": "mgp_log_level", "MGP_VALUE_TYPE_": "mgp_value_type"}


def mgp_abi_probe(header, include_dir, workdir):
    """Compiles and runs a probe that prints, for every function and enumerator include/mgp_abi.h declares, the
    function's mangled C++ type (return and parameter types, typeid) and the enumerator's value, plus the layout of
    mgp_vertex_id, all as seen through `header`.  Returns {name: value}."""
    text = open(os.path.join(REPO, "include", "mgp_abi.h")).read()
    text = text[text.index("#else"):]  # the restated declarations, not the branch that includes the reference header
    functions = sorted(set(re.findall(r"\b(mgp_\w+)\(", text)))
    enumerators = sorted(set(re.findall(r"\b(MGP_(?:ERROR|LOG_LEVEL|VALUE_TYPE)_\w+)", text)))
    lines = [f'printf("%s %s\\n", "{f}", typeid({f}).name());' for f in functions]
    for e in enumerators:
        enum = next(v for k, v in MGP_ENUMS.items() if e.startswith(k))
        lines.append(f'printf("%s %d\\n", "{e}", (int){enum}::{e});')
    lines.append('printf("sizeof(mgp_vertex_id) %zu\\n", sizeof(mgp_vertex_id));')
    lines.append('printf("offsetof(mgp_vertex_id,as_int) %zu\\n", offsetof(mgp_vertex_id, as_int));')
    probe = os.path.join(workdir, "mgp_abi_probe.cpp")
    with open(probe, "w") as f:
        f.write("#include <cstddef>\n#include <cstdio>\n#include <typeinfo>\n#include \"%s\"\nint main() {\n%s\n}\n"
                % (header, "\n".join(lines)))
    exe = os.path.join(workdir, "mgp_abi_probe")
    subprocess.run(["g++", "-std=c++20", "-I", include_dir, probe, "-o", exe], check=True)
    out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    return dict(line.split(" ", 1) for line in out.splitlines())


def test_mgp_abi_matches_the_reference_header(tmp_path):
    """include/mgp_abi.h restates a slice of the reference's include/mg_procedure.h.  Every prototype, enumerator and
    the vertex-id layout it declares, probed through mgp_abi.h, equals what the same probe printed through the
    reference header (tests/golden/mgp_abi_reference.json, written by make_golden.py), so every call the modules
    make has the real prototype."""
    ref = json.load(open(os.path.join(GOLDEN, "mgp_abi_reference.json")))["probe"]
    ours = mgp_abi_probe("mgp_abi.h", os.path.join(REPO, "include"), str(tmp_path))
    assert ours == ref
    assert [ours[k] for k in ("MGP_ERROR_NO_ERROR", "MGP_ERROR_OUT_OF_RANGE", "MGP_ERROR_NOT_YET_IMPLEMENTED",
                              "MGP_LOG_LEVEL_CRITICAL", "sizeof(mgp_vertex_id)", "offsetof(mgp_vertex_id,as_int)")] == \
        ["0", "4", "13", "5", "8", "0"]
