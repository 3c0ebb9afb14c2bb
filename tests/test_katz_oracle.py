"""Groundwork for the next path (Katz centrality, SURVEY 8f-1): oracle/katz_oracle.cpp pinned bit-exact against the
reference's own katz.cpp compiled in place (oracle/_ref/libkatz_ref.so), whose outputs are committed under golden/."""
import ctypes
import json
import os

import numpy as np

from _checkers import ORACLE_SO, build_checkers, sha256_of

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KATZ_REF_SO = os.path.join(REPO, "oracle", "_ref", "libkatz_ref.so")


def oracle_katz(n, f, t, alpha=0.2, eps=1e-2, guard=10000):
    if not os.path.exists(ORACLE_SO):
        build_checkers()
    L = ctypes.CDLL(ORACLE_SO)
    if not hasattr(L, "oracle_katz"):
        build_checkers()
        L = ctypes.CDLL(ORACLE_SO)
    L.oracle_katz.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double,
                              ctypes.c_double, ctypes.c_uint64, ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64)]
    f = np.ascontiguousarray(f, dtype=np.uint64)
    t = np.ascontiguousarray(t, dtype=np.uint64)
    out = np.zeros(n)
    it = ctypes.c_uint64(0)
    rc = L.oracle_katz(n, len(f), f.ctypes.data, t.ctypes.data, alpha, eps, guard, out.ctypes.data, ctypes.byref(it))
    return rc, out, it.value


def ref_katz(n, f, t, alpha=0.2, eps=1e-2):
    L = ctypes.CDLL(KATZ_REF_SO)
    L.ref_katz.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double,
                           ctypes.c_double, ctypes.c_void_p]
    f = np.ascontiguousarray(f, dtype=np.uint64)
    t = np.ascontiguousarray(t, dtype=np.uint64)
    out = np.full(n, np.nan)
    assert L.ref_katz(n, len(f), f.ctypes.data, t.ctypes.data, alpha, eps, out.ctypes.data) == 0
    return out


def test_closed_form_on_a_chain():
    # 0 -> 1 -> 2: omega_1 = [0, 1, 1], omega_2 = [0, 0, 1], omega_3 = 0; c = alpha * omega_1 + alpha^2 * omega_2 + ...
    rc, c, it = oracle_katz(3, [0, 1], [1, 2], alpha=0.2, eps=1e-2)
    assert rc == 0 and it >= 2
    assert np.allclose(c, [0.0, 0.2, 0.2 + 0.04], atol=1e-15)
    rc, c, it = oracle_katz(4, [], [])
    assert rc == 0 and it == 0 and not c.any()


def katz_cases():
    """The seeded graphs compared with the reference: yields (n, m, f, t, alpha, eps)."""
    rng = np.random.default_rng(17)
    for n, m in [(6, 9), (20, 40), (100, 250), (400, 1200), (1500, 3000)]:
        for alpha, eps in [(0.2, 1e-2), (0.05, 1e-3), (0.1, 1e-2)]:
            f, t = rng.integers(0, n, m), rng.integers(0, n, m)
            yield n, m, f, t, alpha, eps


def test_bit_exact_vs_the_reference_katz():
    """The reference's centralities (tests/golden/katz_ref_outputs.json, written by make_golden.py from the reference's
    own katz.cpp) are stored as the SHA-256 of their float64 bytes, so equality stays bit-exact."""
    spec = json.load(open(os.path.join(GOLDEN, "katz_ref_outputs.json")))
    expected = {(c["n"], c["m"], c["alpha"], c["eps"]): c["sha256"] for c in spec["cases"]}
    checked = set()
    for n, m, f, t, alpha, eps in katz_cases():
        rc, c, it = oracle_katz(n, f, t, alpha, eps, guard=2000)
        if rc != 0:
            continue  # does not separate within the guard (alpha^2 * deg_max >= 1): the reference would spin too
        assert sha256_of(c) == expected[(n, m, alpha, eps)], (n, m, alpha, eps, it)
        checked.add((n, m, alpha, eps))
    assert checked == set(expected) and len(checked) >= 8
