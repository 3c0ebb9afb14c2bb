#!/usr/bin/env python3
"""Regenerates the golden fixtures in this directory from the reference checkout.

Runs only where /root/reference exists (the build container); the GPU box uses the committed
JSON files.  Sources:

* ``pagerank_unit_vectors.json``  <- mage/cpp/pagerank_module/pagerank_test.cpp:35-65
  (12 ``PageRankGraph(n, m, {edges})`` known-answer cases, expected ranks to 9 digits,
  default arguments, tolerance mg_test_utils.hpp:25,107-112 = 1e-3 on max AND on mean error).
* ``pagerank_e2e_cases.json``     <- mage/tests/e2e/pagerank_test/<case>/{input.cyp,test.yml}
  (Cypher set-up + expected ``node, rank`` rows, pytest.approx(abs=1e-3), test_module.py:21,76).
* ``pagerank_ref_outputs.json``   <- outputs of the reference algorithm itself (oracle/_ref,
  built by oracle/Makefile) on small seeded graphs at several argument settings, 17 digits,
  so the GPU box -- which has no /root/reference -- can still compare against the real thing.
* ``pagerank_ref_threads.json``, ``katz_ref_outputs.json``, ``pagerank_reference_module.json``,
  ``mgp_abi_reference.json``      <- what the reference's own binaries under oracle/_ref and its
  include/mg_procedure.h give on the inputs the tests generate, so a checkout without them still
  compares against the reference.  Vectors too large to keep whole are stored as the SHA-256 of
  their little-endian bytes, which keeps the comparisons bit-exact.
"""
import ctypes
import json
import os
import re
import sys

import numpy as np
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("MG_REFERENCE", "/root/reference")


def unit_vectors():
    text = open(os.path.join(REF, "mage/cpp/pagerank_module/pagerank_test.cpp")).read()
    body = text[text.index("testing::Values(") :]
    cases = []
    # every case: PageRankGraph(<n>, <m>, {<edges>}) ... std::vector<double>{<expected>}
    pat = re.compile(
        r"PageRankGraph\(\s*(\d+)\s*,\s*(\d+)\s*,\s*\{(.*?)\}\s*\)\s*,\s*std::vector<double>\s*\{\{?(.*?)\}?\}\s*\)",
        re.S,
    )
    for m in pat.finditer(body):
        n, m_arg, edges_txt, exp_txt = m.groups()
        edges = [[int(a), int(b)] for a, b in re.findall(r"\{\s*(\d+)\s*,\s*(\d+)\s*\}", edges_txt)]
        expected = [float(x) for x in re.findall(r"[0-9]+\.[0-9]+", exp_txt)]
        cases.append({"n": int(n), "m": int(m_arg), "edges": edges, "expected": expected})
    assert len(cases) == 12, len(cases)
    return {
        "source": "mage/cpp/pagerank_module/pagerank_test.cpp:35-65",
        "args": {"max_iterations": 100, "damping_factor": 0.85, "stop_epsilon": 1e-5, "num_of_threads": 1},
        "tolerance_abs": 1e-3,
        "cases": cases,
    }


def e2e_cases():
    base = os.path.join(REF, "mage/tests/e2e/pagerank_test")
    out = []
    for name in sorted(os.listdir(base)):
        if name.startswith("test_cugraph"):
            continue  # cuGraph siblings: different module, informative only
        d = os.path.join(base, name)
        cyp = open(os.path.join(d, "input.cyp")).read()
        spec = yaml.safe_load(open(os.path.join(d, "test.yml")))
        edges = [[int(a), int(b)] for a, b in re.findall(
            r"MERGE \(a:Node \{id: (\d+)\}\) MERGE \(b:Node \{id: (\d+)\}\) CREATE \(a\)-\[:RELATION\]->\(b\)", cyp)]
        call = re.search(r"pagerank\.get\((.*?)\)", spec["query"]).group(1).strip()
        args = [int(call)] if call else []
        out.append({"name": name, "edges_by_node_id": edges, "call_args": args, "output": spec["output"]})
    return {"source": "mage/tests/e2e/pagerank_test/*", "tolerance_abs": 1e-3, "cases": out}


def ref_outputs():
    lib = ctypes.CDLL(os.path.join(REPO, "oracle/_ref/libpagerank_ref.so"))
    lib.ref_graph_create.restype = ctypes.c_void_p
    lib.ref_graph_create.argtypes = [ctypes.c_uint64] * 3 + [ctypes.c_void_p] * 2 + [ctypes.c_char_p, ctypes.c_size_t]
    lib.ref_pagerank.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_double, ctypes.c_double, ctypes.c_uint32,
                                 ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t]
    lib.ref_graph_destroy.argtypes = [ctypes.c_void_p]
    cases = []
    rng = np.random.default_rng(20260921)
    settings = [(100, 0.85, 1e-5, 1), (20, 0.85, 0.0, 1), (7, 0.5, 0.0, 1), (0, 0.85, 1e-5, 1), (1000, 0.85, 1e-9, 1)]
    for n, m in [(1, 0), (3, 0), (17, 40), (64, 64), (200, 1500), (1000, 3000)]:
        frm = rng.integers(0, n, size=m, dtype=np.uint64)
        to = rng.integers(0, n, size=m, dtype=np.uint64)
        err = ctypes.create_string_buffer(256)
        g = lib.ref_graph_create(n, m, m, frm.ctypes.data, to.ctypes.data, err, 256)
        assert g, err.value
        for (it, d, eps, t) in settings:
            out = np.zeros(n, dtype=np.float64)
            rc = lib.ref_pagerank(g, it, d, eps, t, out.ctypes.data, err, 256)
            assert rc == 0, err.value
            cases.append({"n": n, "from": frm.tolist(), "to": to.tolist(),
                          "args": {"max_iterations": it, "damping_factor": d, "stop_epsilon": eps, "num_of_threads": t},
                          "ranks": [repr(float(x)) for x in out]})
        lib.ref_graph_destroy(g)
    return {"source": "oracle/_ref/libpagerank_ref.so = reference algorithm/pagerank.cpp compiled in place "
                      "(g++ -std=c++20 -O2, no -funsafe-math-optimizations)", "cases": cases}


def bfs_unit_graph():
    """tests/unit/bfs_common.hpp: the 6-vertex graph kEdges (:46-54) and the expected distances of its own
    oracle -- Floyd-Warshall over the direction-adjusted edge list (:58-110), then the bounds filter
    (:452-462: lower -1 -> 0, upper -1 -> vertex count; a == b is never reported)."""
    text = open(os.path.join(REF, "tests/unit/bfs_common.hpp")).read()
    block = text[text.index("kEdges = {"):]
    block = block[:block.index("};")]
    edges = [[int(a), int(b)] for a, b in re.findall(r"\{(\d+),\s*(\d+),\s*\"[ab]\"\}", block)]
    n = int(re.search(r"kVertexCount = (\d+)", text).group(1))
    assert len(edges) == 9 and n == 6

    def floyd_warshall(pairs):
        inf = 10**9
        d = [[inf] * n for _ in range(n)]
        for a, b in pairs:
            d[a][b] = 1
        for i in range(n):
            d[i][i] = 0
        for k in range(n):
            for i in range(n):
                for j in range(n):
                    if d[i][k] < inf and d[k][j] < inf:
                        d[i][j] = min(d[i][j], d[i][k] + d[k][j])
        return [[-1 if x >= inf else x for x in row] for row in d]

    cases = []
    for name, pairs in [("OUT", edges), ("IN", [[b, a] for a, b in edges]),
                        ("BOTH", edges + [[b, a] for a, b in edges])]:
        full = floyd_warshall(pairs)
        for lower, upper in [(-1, -1), (1, 1), (1, 2), (2, 2), (2, 3), (3, 6), (1, 6)]:
            lo = 0 if lower == -1 else lower
            hi = n if upper == -1 else upper
            dist = [[(full[a][b] if a != b and full[a][b] != -1 and lo <= full[a][b] <= hi else -1) for b in range(n)]
                    for a in range(n)]
            cases.append({"direction": name, "lower": lower, "upper": upper, "dist": dist})
    return {"source": "tests/unit/bfs_common.hpp:42-110,423-470", "n": n, "edges": edges, "cases": cases}


TESTS = os.path.dirname(HERE)


def ref_threads():
    """The reference algorithm (oracle/_ref/libpagerank_ref.so) on test_oracle.thread_cases, as float64 digests."""
    sys.path.insert(0, TESTS)
    from _checkers import OracleError, Reference, sha256_of
    from test_oracle import THREAD_COUNTS, thread_cases
    ref = Reference()
    cases = [{"threads": threads, "n": n, "m": m, "args": kw,
              "sha256": sha256_of(ref.pagerank(n, frm, to, num_of_threads=threads, **kw))}
             for threads in THREAD_COUNTS for n, m, frm, to, kw in thread_cases(threads)]
    try:
        ref.pagerank(2, [0], [1], num_of_threads=0)
        raise AssertionError("the reference accepted num_of_threads = 0")
    except OracleError as ex:
        zero_threads_error = str(ex)
    nan = bool(np.all(np.isnan(ref.pagerank(3, [0, 1], [1, 2], damping_factor=1.0, max_iterations=50))))
    return {"source": "oracle/_ref/libpagerank_ref.so = reference algorithm/pagerank.cpp compiled in place; ranks as "
                      "SHA-256 of their little-endian float64 bytes",
            "cases": cases, "edge_cases": {"zero_threads_error": zero_threads_error, "damping_1_all_nan": nan}}


def katz_ref():
    """The reference's katz.cpp (oracle/_ref/libkatz_ref.so) on test_katz_oracle.katz_cases that separate within the
    oracle's guard (the reference would spin on the others), as float64 digests."""
    sys.path.insert(0, TESTS)
    from _checkers import sha256_of
    from test_katz_oracle import katz_cases, oracle_katz, ref_katz
    cases = []
    for n, m, f, t, alpha, eps in katz_cases():
        if oracle_katz(n, f, t, alpha, eps, guard=2000)[0] == 0:
            cases.append({"n": n, "m": m, "alpha": alpha, "eps": eps, "sha256": sha256_of(ref_katz(n, f, t, alpha, eps))})
    return {"source": "oracle/_ref/libkatz_ref.so = reference katz_centrality_module/algorithm/katz.cpp compiled in "
                      "place; centralities as SHA-256 of their little-endian float64 bytes", "cases": cases}


def reference_module():
    """The reference's pagerank.so (oracle/_ref/pagerank_reference.so) loaded and called through the fake mgp host
    on the inputs of test_module_host.py and test_gpu_module.py."""
    import subprocess
    sys.path.insert(0, TESTS)
    import _fakehost as fh
    from _checkers import sha256_of
    from test_module_host import e2e_fixture_graph, e2e_fixture_rows, scattered_graph
    out = {"source": "oracle/_ref/pagerank_reference.so = reference mage/cpp/pagerank_module compiled in place, "
                     "called through tests/mgp_fake_host.cpp; large outputs as SHA-256 of their little-endian bytes"}
    und = subprocess.run(["nm", "-D", "--undefined-only", fh.REF_MODULE_SO], capture_output=True, text=True,
                         check=True).stdout
    out["imports"] = sorted(line.split()[-1] for line in und.splitlines() if " U mgp_" in line)
    with fh.Module(fh.REF_MODULE_SO) as module:
        out["signature"] = module.signature()
        with fh.Graph([1, 2], [1], [2]) as g:
            try:
                module.call(g, 10, 0.85, 1e-5, 0)
                raise AssertionError("the reference module accepted num_of_threads = 0")
            except fh.ProcedureError as ex:
                out["zero_threads_error"] = str(ex)

        def digests(graph, args_list):
            gids, src, dst = graph
            rows = []
            with fh.Graph(gids, src, dst) as g:
                for args in args_list:
                    nodes, ranks = module.call(g, *args)
                    rows.append({"args": list(args), "nodes_sha256": sha256_of(nodes, np.int64),
                                 "ranks_sha256": sha256_of(ranks)})
            return rows

        out["config1"] = digests(scattered_graph(10_000, 50_000, seed=42), [(), (20, 0.85, 0.0, 8)])
        out["same_rows"] = digests(scattered_graph(3000, 20000, seed=7), [(), (20, 0.85, 0.0, 4), (7, 0.3, 0.0, 1)])
        out["e2e"] = {}
        for case in e2e_cases()["cases"]:
            gid_of, gids, src, dst = e2e_fixture_graph(case)
            with fh.Graph(gids, src, dst) as g:
                out["e2e"][case["name"]] = e2e_fixture_rows(gid_of, *module.call(g, *case["call_args"]))
        out["unit_vectors"] = []
        for i, case in enumerate(unit_vectors()["cases"]):
            if case["m"] != len(case["edges"]):
                continue
            gids = np.arange(case["n"], dtype=np.int64) * 5 + 11
            e = np.array(case["edges"], dtype=np.int64).reshape(-1, 2)
            with fh.Graph(gids, gids[e[:, 0]] if len(e) else [], gids[e[:, 1]] if len(e) else []) as g:
                nodes, ranks = module.call(g)
            out["unit_vectors"].append({"case": i, "nodes": nodes.tolist(), "ranks": ranks.tolist()})
    return out


def mgp_abi_reference():
    """test_module_host.mgp_abi_probe through the reference's include/mg_procedure.h."""
    import tempfile
    sys.path.insert(0, TESTS)
    from test_module_host import mgp_abi_probe
    with tempfile.TemporaryDirectory() as tmp:
        probe = mgp_abi_probe("mg_procedure.h", os.path.join(REF, "include"), tmp)
    return {"source": "include/mg_procedure.h: typeid(function).name() of every function include/mgp_abi.h declares, "
                      "the value of every enumerator it declares, and the layout of mgp_vertex_id", "probe": probe}


def main():
    if not os.path.isdir(REF):
        sys.exit("reference checkout not present; golden fixtures are committed, nothing to do")
    for name, fn in [("pagerank_unit_vectors.json", unit_vectors), ("pagerank_e2e_cases.json", e2e_cases),
                     ("pagerank_ref_outputs.json", ref_outputs), ("bfs_unit_graph.json", bfs_unit_graph),
                     ("pagerank_ref_threads.json", ref_threads), ("katz_ref_outputs.json", katz_ref),
                     ("pagerank_reference_module.json", reference_module), ("mgp_abi_reference.json", mgp_abi_reference)]:
        with open(os.path.join(HERE, name), "w") as f:
            json.dump(fn(), f, indent=None if "ref_outputs" in name else 1, separators=(",", ":") if "ref_outputs" in name else None)
            f.write("\n")
        print("wrote", name)


if __name__ == "__main__":
    main()
