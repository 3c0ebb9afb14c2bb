"""ctypes front-ends for the CHECKERS (oracle/): the plain-C restatement and, when oracle/Makefile
built it from a reference checkout, the reference's own algorithm.  Only tests/, tests/golden/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(REPO, "oracle", "_build", "libpagerank_oracle.so")
REF_SO = os.path.join(REPO, "oracle", "_ref", "libpagerank_ref.so")
REF_MODULE_SO = os.path.join(REPO, "oracle", "_ref", "pagerank_reference.so")


def build_checkers():
    """(Re)build oracle/_build (always) and oracle/_ref (only where the reference checkout exists)."""
    subprocess.run(["make", "-s", "-C", os.path.join(REPO, "oracle"), "all"], check=True)


def ensure_checkers_fresh():
    """Rebuild the plain-C/C++ restatements when a source under oracle/ is newer than the library.  Called once at
    session start (conftest.py), BEFORE anything dlopen()s the library: a stale copy that is already loaded stays
    loaded, so rebuilding later in the session cannot add a missing symbol."""
    import glob
    srcs = glob.glob(os.path.join(REPO, "oracle", "*.c")) + glob.glob(os.path.join(REPO, "oracle", "*.cpp"))
    if not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < max(os.path.getmtime(f) for f in srcs):
        subprocess.run(["make", "-s", "-C", os.path.join(REPO, "oracle"), "oracle"], check=True)


class OracleError(RuntimeError):
    pass


def oracle_rmat_edges(scale, count=None, seed=42, a=0.57, b=0.19, c=0.19, first=0, threads=None):
    """oracle/rmat_oracle.c: the benchmark's RMAT edge stream as uint64 (from, to) WITHOUT the product library."""
    if not os.path.exists(ORACLE_SO):
        build_checkers()
    L = ctypes.CDLL(ORACLE_SO)
    L.oracle_rmat_edges.argtypes = [ctypes.c_uint32, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_double,
                                    ctypes.c_double, ctypes.c_double, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p]
    count = (16 << scale) if count is None else count
    frm = np.empty(count, dtype=np.uint64)
    to = np.empty(count, dtype=np.uint64)
    rc = L.oracle_rmat_edges(scale, first, count, seed, a, b, c, threads or min(os.cpu_count() or 1, 32),
                             frm.ctypes.data, to.ctypes.data)
    if rc:
        raise OracleError(f"oracle_rmat_edges failed: {rc}")
    return frm, to


def _u64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint64))


def sha256_of(a, dtype=np.float64):
    """Hex SHA-256 of the array's little-endian bytes: how golden files store vectors too large to keep whole while
    still pinning them bit for bit."""
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.dtype(dtype).newbyteorder("<")).tobytes()).hexdigest()


class Oracle:
    """oracle/pagerank_oracle.c"""

    def __init__(self):
        if not os.path.exists(ORACLE_SO):
            build_checkers()
        L = ctypes.CDLL(ORACLE_SO)
        L.oracle_error_string.restype = ctypes.c_char_p
        L.oracle_error_string.argtypes = [ctypes.c_int]
        L.oracle_graph_create.argtypes = [ctypes.c_uint64] * 3 + [ctypes.c_void_p] * 2 + [ctypes.POINTER(ctypes.c_void_p)]
        L.oracle_graph_destroy.argtypes = [ctypes.c_void_p]
        L.oracle_pagerank.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_double, ctypes.c_double,
                                      ctypes.c_uint32, ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64)]
        L.oracle_map_gids.argtypes = [ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64] + [ctypes.c_void_p] * 4
        self.L = L

    def graph(self, n, frm, to, m=None):
        frm, to = _u64(frm), _u64(to)
        h = ctypes.c_void_p()
        rc = self.L.oracle_graph_create(n, len(frm) if m is None else m, len(frm), frm.ctypes.data, to.ctypes.data,
                                        ctypes.byref(h))
        if rc:
            raise OracleError(self.L.oracle_error_string(rc).decode())
        return h

    def run(self, h, n, max_iterations=100, damping_factor=0.85, stop_epsilon=1e-5, num_of_threads=1):
        out = np.zeros(n, dtype=np.float64)
        it = ctypes.c_uint64(0)
        rc = self.L.oracle_pagerank(h, max_iterations & (2**64 - 1), damping_factor, stop_epsilon,
                                    num_of_threads & 0xFFFFFFFF, out.ctypes.data, ctypes.byref(it))
        if rc:
            raise OracleError(self.L.oracle_error_string(rc).decode())
        return out, it.value

    def free(self, h):
        self.L.oracle_graph_destroy(h)

    def pagerank(self, n, frm, to, m=None, **kw):
        h = self.graph(n, frm, to, m)
        try:
            return self.run(h, n, **kw)
        finally:
            self.free(h)

    def map_gids(self, visited, src_gid, dst_gid):
        visited = np.ascontiguousarray(visited, dtype=np.int64)
        s = np.ascontiguousarray(src_gid, dtype=np.int64)
        d = np.ascontiguousarray(dst_gid, dtype=np.int64)
        f = np.zeros(len(s), dtype=np.uint64)
        t = np.zeros(len(s), dtype=np.uint64)
        rc = self.L.oracle_map_gids(len(visited), visited.ctypes.data, len(s), s.ctypes.data, d.ctypes.data,
                                    f.ctypes.data, t.ctypes.data)
        if rc:
            raise OracleError(self.L.oracle_error_string(rc).decode())
        return f, t


def pull_oracle_pagerank(n, frm, to, max_iterations=100, damping_factor=0.85, stop_epsilon=1e-5, threads=None):
    """oracle/pagerank_pull_oracle.c: the multi-threaded pull-form checker for graphs too big for Oracle (validated
    against it in tests/test_oracle.py).  Returns (ranks, iterations)."""
    if not os.path.exists(ORACLE_SO):
        build_checkers()
    L = ctypes.CDLL(ORACLE_SO)
    L.oracle_pull_pagerank.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                       ctypes.c_double, ctypes.c_double, ctypes.c_uint32, ctypes.c_void_p,
                                       ctypes.POINTER(ctypes.c_uint64)]
    frm, to = _u64(frm), _u64(to)
    out = np.zeros(n, dtype=np.float64)
    it = ctypes.c_uint64(0)
    rc = L.oracle_pull_pagerank(n, len(frm), frm.ctypes.data, to.ctypes.data, max_iterations & (2**64 - 1), damping_factor,
                                stop_epsilon, threads or min(os.cpu_count() or 1, 128), out.ctypes.data, ctypes.byref(it))
    if rc:
        raise OracleError(f"oracle_pull_pagerank failed: {rc}")
    return out, it.value


class Reference:
    """oracle/_ref/libpagerank_ref.so -- the reference's own pagerank.cpp behind oracle/ref_shim.cpp."""

    @staticmethod
    def available():
        return os.path.exists(REF_SO)

    def __init__(self):
        L = ctypes.CDLL(REF_SO)
        L.ref_graph_create.restype = ctypes.c_void_p
        L.ref_graph_create.argtypes = [ctypes.c_uint64] * 3 + [ctypes.c_void_p] * 2 + [ctypes.c_char_p, ctypes.c_size_t]
        L.ref_pagerank.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_double, ctypes.c_double,
                                   ctypes.c_uint32, ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t]
        L.ref_graph_destroy.argtypes = [ctypes.c_void_p]
        self.L = L

    def graph(self, n, frm, to, m=None):
        frm, to = _u64(frm), _u64(to)
        err = ctypes.create_string_buffer(256)
        h = self.L.ref_graph_create(n, len(frm) if m is None else m, len(frm), frm.ctypes.data, to.ctypes.data, err, 256)
        if not h:
            raise OracleError(err.value.decode())
        return h

    def run(self, h, n, max_iterations=100, damping_factor=0.85, stop_epsilon=1e-5, num_of_threads=1):
        out = np.zeros(n, dtype=np.float64)
        err = ctypes.create_string_buffer(256)
        rc = self.L.ref_pagerank(h, max_iterations & (2**64 - 1), damping_factor, stop_epsilon,
                                 num_of_threads & 0xFFFFFFFF, out.ctypes.data, err, 256)
        if rc:
            raise OracleError(err.value.decode())
        return out

    def free(self, h):
        self.L.ref_graph_destroy(h)

    def pagerank(self, n, frm, to, m=None, **kw):
        h = self.graph(n, frm, to, m)
        try:
            return self.run(h, n, **kw)
        finally:
            self.free(h)


class BfsOracle:
    """oracle/bfs_oracle.c (same shared object as the PageRank oracle)."""
    OUT, IN, BOTH = 0, 1, 2

    def __init__(self):
        if not os.path.exists(ORACLE_SO):
            build_checkers()
        L = ctypes.CDLL(ORACLE_SO)
        if not hasattr(L, "oracle_bfs"):
            build_checkers()
            L = ctypes.CDLL(ORACLE_SO)
        L.oracle_bfs.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                 ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p]
        self.L = L

    def distances(self, n, frm, to, source, direction=0, lower=1, upper=2**63 - 1):
        frm, to = _u64(frm), _u64(to)
        out = np.empty(n, dtype=np.int64)
        rc = self.L.oracle_bfs(n, len(frm), frm.ctypes.data, to.ctypes.data, source, direction, lower, upper,
                               out.ctypes.data)
        if rc:
            raise OracleError(f"oracle_bfs failed: {rc}")
        return out
