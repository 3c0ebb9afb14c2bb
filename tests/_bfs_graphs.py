"""CPU side of tests/test_gpu_bfs_strategies.py: graphs shaped to reach the boundaries of the breadth-first expansion
(memgraph_b200/csrc/bfs.cu) and a numpy restatement of mgb200_bfs_run that predicts its distances and every field of
mgb200_bfs_stats except traverse_ms.

Distances do not depend on the order of work, and neither do the statistics: a top-down level inspects the whole forward
degree of its frontier; a bottom-up level has every unvisited vertex scan its sorted reverse adjacency up to its first
parent in the frontier, and nothing else writes that vertex's depth during the level.  The switch between the two is
integer arithmetic on host-side counters."""
from dataclasses import dataclass, field

import numpy as np

OUT, IN, BOTH = 0, 1, 2
DIRECTIONS = {"OUT": OUT, "IN": IN, "BOTH": BOTH}
STRATEGIES = ("auto", "top_down", "bottom_up", "alternate")  # MGB200_BFS_STRATEGY
INT64_MIN, INT64_MAX = -2 ** 63, 2 ** 63 - 1
INT_MAX = 2 ** 31 - 1

SEG_EDGES = 1024              # kSegEdges: edges per top-down work item (one warp)
SWITCH_DIVISOR = 14           # bottom-up when m_f > m_u / 14 ...
SWITCH_MIN_FRONTIER = 1024    # ... and the frontier holds more than 1024 vertices
TOP_DOWN_WARPS_PER_SM = 64    # top_down_kernel: 8 blocks of 8 warps per SM, a grid-stride loop over the work items
BOTTOM_UP_THREADS_PER_SM = 32 * 256  # bottom_up_kernel: at most 32 blocks of 256 threads per SM, grid-stride over n


# ---- graphs ------------------------------------------------------------------------------------------------------------

@dataclass
class Graph:
    name: str
    n: int
    f: np.ndarray              # uint64 sources, input edge order
    t: np.ndarray              # uint64 targets
    sources: list              # the sources the GPU tests run from
    intended: dict = field(default_factory=dict)  # what the graph was built to reach

    @property
    def m(self):
        return len(self.f)

    def degree(self, v, direction):
        """forward degree of v in `direction` (BOTH: out-degree + in-degree)"""
        out = int(np.count_nonzero(self.f == v))
        inn = int(np.count_nonzero(self.t == v))
        return (out, inn, out + inn)[direction]


def _graph(name, n, edges, sources, seed, **intended):
    """Shuffled input order: the device sorts every row, so the order of the edge list must not matter."""
    e = np.asarray(edges, dtype=np.uint64).reshape(-1, 2)
    e = e[np.random.default_rng(seed).permutation(len(e))]
    return Graph(name, n, np.ascontiguousarray(e[:, 0]), np.ascontiguousarray(e[:, 1]), list(sources), intended)


def _mirror(n, edges):
    """The graph plus a reversed copy on ids n..2n-1: IN from v + n walks exactly what OUT from v walks, so the shapes
    aimed at the forward (out) adjacency are reached in both directions."""
    e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    return 2 * n, np.concatenate([e, e[:, ::-1] + n])


HUB_DEGREES = (1, 31, 32, 33, 1023, 1024, 1025, 2047, 2048, 2049, 32 * SEG_EDGES + 1)
REPEAT_HUB = dict(before=1000, repeats=1100, after=200)  # one target repeated across both edges of segment 1


def hub_segments():
    """Hubs whose out-degree is each of HUB_DEGREES, with distinct targets (32 * 1024 + 1 is 33 segments), plus one hub
    whose sorted out-list is 1000 distinct targets, then one target repeated 1100 times (positions 1000..2099, across
    the segment edges at 1024 and 2048), then 200 more: three warps race on that target's depth and exactly one CAS
    may win.  Every hub target has one out-edge into a pool of 500 vertices, each pool vertex one out-edge to a hub,
    so the traversal goes on past level 1.  Mirrored for IN."""
    rng = np.random.default_rng(101)
    hubs = list(range(len(HUB_DEGREES) + 1))
    nxt = len(hubs)
    edges, leaves = [], []
    for h, d in zip(hubs, HUB_DEGREES):
        edges += [(h, nxt + k) for k in range(d)]
        leaves += range(nxt, nxt + d)
        nxt += d
    rep = hubs[-1]
    b, r, a = REPEAT_HUB["before"], REPEAT_HUB["repeats"], REPEAT_HUB["after"]
    ids = list(range(nxt, nxt + b + 1 + a))  # ascending: the repeated one is the (b+1)-th
    nxt += len(ids)
    edges += [(rep, v) for v in ids[:b]] + [(rep, ids[b])] * r + [(rep, v) for v in ids[b + 1:]]
    leaves += ids
    pool = np.arange(nxt, nxt + 500)
    nxt += 500
    edges += [(v, int(p)) for v, p in zip(leaves, rng.choice(pool, len(leaves)))]
    edges += [(int(p), int(h)) for p, h in zip(pool, rng.choice(hubs, len(pool)))]
    n, e = _mirror(nxt, edges)
    sources = [0, 4, 6, 9, 10, rep, 10 + nxt, 6 + nxt]  # degrees 1, 1023, 1025, 2049, 32769, the repeat hub; mirrored
    return _graph("hub_segments", n, e, sources, 102, hub_degrees=list(HUB_DEGREES), hubs=hubs, repeat_hub=rep,
                  repeat_target=ids[b], half=nxt)


ZERO_RUN_HUBS = {300: 1, 500: 1024, 700: 1025, 701: 2049}  # position in the level-1 queue -> forward degree


def zero_runs():
    """The source's out-list is 1000 vertices; at the positions of ZERO_RUN_HUBS sit hubs of out-degree 1, 1024, 1025
    and 2049, every other one has out-degree 0.  At <= 1024 edges the source is one top-down work item, so one warp
    pushes the level-1 queue in adjacency order: runs of zero-degree vertices come before, between and after the hubs,
    and seg_scan holds long runs of equal entries that the binary search must step over.  Mirrored for IN."""
    width = 1000
    edges = [(0, 1 + k) for k in range(width)]
    nxt = 1 + width
    for pos, d in ZERO_RUN_HUBS.items():
        edges += [(1 + pos, nxt + k) for k in range(d)]
        nxt += d
    n, e = _mirror(nxt, edges)
    return _graph("zero_runs", n, e, [0, nxt, 1 + 500], 103, level1=list(range(1, 1 + width)),
                  hub_positions=dict(ZERO_RUN_HUBS), half=nxt)


JUNCTIONS = ((0, 5), (1, 1030), (1023, 2), (1024, 3), (1025, 1024), (2047, 1), (2048, 1))  # (out-degree, fresh in-nbrs)


def both_junction():
    """For BOTH the forward adjacency of u is its out-list followed by its in-list, so the out/in junction sits at
    position a = out-degree: 0, 1, 1023, 1024, 1025, 2047 and 2048 -- the start, the second slot, the last slot of a
    segment, a segment edge and one past it.  Every neighbour is a fresh vertex whose only edge is the one to u: it is
    reachable through its own position and nothing else.  Each junction vertex also has a witness w, with three
    in-edges from fresh vertices and one out-edge to u (so u's in-list is b fresh vertices and w): bottom-up from u
    under BOTH, w scans its in-list and then finds u in its out-list."""
    edges, sources, nxt = [], [], 0
    for a, b in JUNCTIONS:
        u = nxt
        sources.append(u)
        edges += [(u, u + 1 + k) for k in range(a)] + [(u + 1 + a + k, u) for k in range(b)]
        w = u + 1 + a + b
        edges += [(w + 1 + k, w) for k in range(3)] + [(w, u)]
        nxt = w + 4
    return _graph("both_junction", nxt, edges, sources, 104, junctions=list(JUNCTIONS))


BITMAP_N = (1, 2, 31, 32, 33, 63, 64, 65, 1025, 4097)


def bitmap_edges(n):
    """A source whose out-neighbours are ids 0, 31, 32, 63, 64 and n-1 (those below n): bit 0 and bit 31 of a word,
    both sides of every word edge, the last partial word, and n-1 next to the n_round tail lanes.  Each of them has one
    private child, found bottom-up only if its parent's own bit is read."""
    frontier = sorted({v for v in (0, 31, 32, 63, 64, n - 1) if 0 <= v < n})
    if n <= 2:  # no room for a separate source: n = 1 is a self-loop, n = 2 a two-cycle
        edges = [(0, 0)] if n == 1 else [(0, 1), (1, 0)]
        return _graph(f"bitmap_n{n}", n, edges, list(range(n)), 105, frontier=frontier)
    free = [v for v in range(n) if v not in frontier]
    source, children = free[0], free[1:]
    edges = [(source, v) for v in frontier]
    edges += [(p, c) for p, c in zip(frontier, children)]
    return _graph(f"bitmap_n{n}", n, edges, [source, 0, n - 1], 105, frontier=frontier, source=source)


def auto_switch():
    """Three components and a filler, sized so that the auto heuristic goes top-down, bottom-up, top-down in every
    direction, with the switch pinned to its exact boundary for OUT and IN.

    A (OUT from a, IN from its mirror a'): a -> 1100 L1 vertices, whose 2 out-edges each reach all of 1500 L2
    vertices; X out-edges go from L2 vertices into 300 L3 vertices.  Level 1 has m_f = 2200 = m_u // 14 + 1 (bottom-up,
    one edge above the boundary) and level 2 has nf = 1500 > 1024 with m_f = X = m_u // 14 (top-down, exactly on it).
    C (BOTH from c): c -> 1100 L1 vertices, each with 4 out-edges into 600 L2 vertices: level 1 goes bottom-up, level 2
    (at most 600 <= 1024 vertices) top-down.  The filler is a separate random component that sets m."""
    p, q, r2, r3, pc, qc, rc = 1100, 2, 1500, 300, 1100, 4, 600
    rng = np.random.default_rng(106)
    # m - p == 14 * (p * q - 1)  =>  level 1 of A: m_u // 14 == p * q - 1 < m_f
    m_total = 14 * (p * q - 1) + p
    x = (m_total - p - p * q) // 14  # level 2 of A: m_f == m_u // 14
    a, l1, l2, l3 = 0, np.arange(1, 1 + p), np.arange(1 + p, 1 + p + r2), np.arange(1 + p + r2, 1 + p + r2 + r3)
    half = 1 + p + r2 + r3
    ea = [(a, int(v)) for v in l1]
    ea += [(int(u), int(l2[(q * i + j) % r2])) for i, u in enumerate(l1) for j in range(q)]  # every L2 vertex reached
    ea += [(int(u), int(v)) for u, v in zip(rng.choice(l2, x), rng.choice(l3, x))]
    n_a, ea = _mirror(half, ea)
    c = n_a
    c1, c2 = np.arange(c + 1, c + 1 + pc), np.arange(c + 1 + pc, c + 1 + pc + rc)
    ec = [(c, int(v)) for v in c1] + [(int(u), int(v)) for u in c1 for v in rng.choice(c2, qc, replace=False)]
    filler0, filler_n = c + 1 + pc + rc, 800
    filler_m = m_total - len(ea) - len(ec)
    assert filler_m > 0
    ef = np.stack([rng.integers(filler0, filler0 + filler_n, filler_m),
                   rng.integers(filler0, filler0 + filler_n, filler_m)], axis=1)
    edges = np.concatenate([ea, np.asarray(ec), ef])
    switch_sources = {OUT: a, IN: a + half, BOTH: c}
    return _graph("auto_switch", filler0 + filler_n, edges, [a, a + half, c], 107, switch_sources=switch_sources,
                  pinned_levels={1: "bottom_up", 2: "top_down"})


DEEP_LEVELS = 3000


def deep_path():
    """A path 0 -> 1 -> ... -> 3000 with side branches: every 7th path vertex has a leaf, every 21st a two-step
    branch, and every 100th an edge back to the start of its hundred.  3000 levels of expansion; the bounds cut it."""
    L = DEEP_LEVELS
    edges = [(i, i + 1) for i in range(L)]
    nxt = L + 1
    for i in range(0, L, 7):
        edges.append((i, nxt))
        nxt += 1
    for i in range(3, L, 21):
        edges += [(i, nxt), (nxt, nxt + 1)]
        nxt += 2
    edges += [(i, i - 99) for i in range(100, L, 100)]
    return _graph("deep_path", nxt, edges, [0, L // 2, L], 108, path_levels=L)


def degenerate():
    """m = 0; n = 1 with a self-loop; and a graph with an isolated vertex (0), a vertex whose only edge is a self-loop
    (1), duplicate edges (2 -> 3 three times, 3 -> 4 twice), and a vertex with in-edges but no out-edges (5): empty for
    OUT, not for IN."""
    return [
        _graph("no_edges", 5, [], [0, 4], 109, m0=True),
        _graph("single_self_loop", 1, [(0, 0)], [0], 110),
        _graph("isolated_loops_duplicates", 8,
               [(1, 1), (2, 3), (2, 3), (2, 3), (3, 4), (3, 4), (4, 2), (6, 5), (7, 5), (7, 5), (6, 7), (4, 6)],
               [0, 1, 2, 5], 111, isolated=0, self_loop_only=1, duplicates=[(2, 3), (3, 4)], no_out=5),
    ]


def all_graphs():
    return [hub_segments(), zero_runs(), both_junction()] + [bitmap_edges(n) for n in BITMAP_N] + [
        auto_switch(), deep_path()] + degenerate()


def bounds_sets(k):
    """(lower, upper) pairs for a traversal whose deepest level is k."""
    return [(1, INT64_MAX), (0, 5), (INT64_MIN, 2), (2, 3), (1, 1), (k, k), (k + 1, INT64_MAX), (1, 2 ** 40),
            (1, 0), (1, -1), (4, 3)]


# ---- the model of mgb200_bfs_run ---------------------------------------------------------------------------------------

class Csr:
    """One side of the device graph: rows sorted by (row, neighbour), duplicates kept (bfs.cu build_side)."""

    def __init__(self, n, row, col):
        key = np.sort((np.asarray(row, dtype=np.uint64) << np.uint64(32)) | np.asarray(col, dtype=np.uint64))
        self.adj = (key & np.uint64(0xFFFFFFFF)).astype(np.uint32)
        self.deg = np.bincount((key >> np.uint64(32)).astype(np.int64), minlength=n).astype(np.int64)
        self.ptr = np.concatenate([[0], np.cumsum(self.deg)]).astype(np.int64)

    def rows(self, vertices):
        """the adjacency entries of `vertices`, concatenated"""
        starts, lens = self.ptr[vertices], self.deg[vertices]
        total = int(lens.sum())
        if total == 0:
            return np.empty(0, dtype=np.uint32)
        offsets = np.repeat(starts - (np.cumsum(lens) - lens), lens) + np.arange(total)
        return self.adj[offsets]


class Model:
    """The device graph of (n, f, t) as the model sees it."""

    def __init__(self, n, f, t):
        self.n, self.m = n, len(f)
        self.out = Csr(n, f, t)
        self.inn = Csr(n, t, f)
        self._traces = {}

    def sides(self, direction):
        """(forward lists, reverse lists), each in concatenation order (bfs.cu mgb200_bfs_run: Adj a then b)"""
        return {OUT: ([self.out], [self.inn]), IN: ([self.inn], [self.out]),
                BOTH: ([self.out, self.inn], [self.inn, self.out])}[direction]

    def trace(self, source, direction, strategy="auto"):
        """The unbounded traversal: final depths and one record per expansion, the last one finding nothing."""
        key = (source, direction, strategy)
        if key not in self._traces:
            self._traces[key] = self._trace(source, direction, strategy)
        return self._traces[key]

    def _trace(self, source, direction, strategy):
        n = self.n
        forward, reverse = self.sides(direction)
        m_dir = 2 * self.m if direction == BOTH else self.m
        depth = np.full(n, -1, dtype=np.int64)
        depth[source] = 0
        frontier = np.array([source], dtype=np.int64)
        explored, level, levels = 0, 0, []
        while len(frontier) and level < INT_MAX - 1:
            nf = len(frontier)
            deg = sum(c.deg[frontier] for c in forward)
            m_f = int(deg.sum())
            m_u = m_dir - explored if m_dir > explored else 0
            explored += m_f
            if strategy == "auto":
                bottom_up = m_f > m_u // SWITCH_DIVISOR and nf > SWITCH_MIN_FRONTIER
            elif strategy in ("top_down", "bottom_up"):
                bottom_up = strategy == "bottom_up"
            elif strategy == "alternate":
                bottom_up = level % 2 == 1
            else:
                raise ValueError(strategy)
            if bottom_up:
                nxt, inspected = _bottom_up(reverse, depth, frontier)
            else:
                nxt, inspected = _top_down(forward, depth, frontier), m_f
            depth[nxt] = level + 1
            levels.append(dict(bottom_up=bottom_up, nf=nf, m_f=m_f, m_u=m_u, found=len(nxt), inspected=inspected,
                               segments=int(((deg + SEG_EDGES - 1) // SEG_EDGES).sum())))
            frontier = nxt
            if len(nxt):
                level += 1
        return depth, levels

    def run(self, source, direction, lower=1, upper=INT64_MAX, strategy="auto"):
        """(dist int64[n], stats) as mgb200_bfs_run returns them, traverse_ms left out."""
        depth, levels = self.trace(source, direction, strategy)
        return predict(self.n, source, depth, levels, lower, upper)


def _top_down(forward, depth, frontier):
    """The unvisited vertices among the frontier's forward neighbours (each once, whatever its multiplicity)."""
    nb = np.concatenate([c.rows(frontier) for c in forward]).astype(np.int64)
    return np.unique(nb[depth[nb] == -1])


def _bottom_up(reverse, depth, frontier):
    """Every unvisited vertex reads its reverse lists in order up to and including its first frontier parent."""
    n = len(depth)
    in_frontier = np.zeros(n, dtype=bool)
    in_frontier[frontier] = True
    searching = depth == -1
    read = np.zeros(n, dtype=np.int64)
    for c in reverse:
        hits = np.flatnonzero(in_frontier[c.adj])
        rows = np.searchsorted(c.ptr, hits, side="right") - 1
        first = np.ones(len(rows), dtype=bool)
        first[1:] = rows[1:] != rows[:-1]
        rows, hits = rows[first], hits[first]
        keep = searching[rows]
        rows, hits = rows[keep], hits[keep]
        read[searching] += c.deg[searching]                 # no parent in this list: the whole list
        read[rows] += hits - c.ptr[rows] + 1 - c.deg[rows]  # a parent: up to it
        searching[rows] = False
    found = (depth == -1) & ~searching
    return np.flatnonzero(found), int(read.sum())


def predict(n, source, depth, levels, lower, upper):
    """mgb200_bfs_run's level loop over a recorded unbounded traversal: a stop at upper_bound is not followed by another
    expansion; a run that is not stopped ends with an expansion that finds nothing, counted as a level of its
    strategy.  Launches: init, then per level the frontier scan plus 3 (bottom-up) or 2 (top-down, the CUB scan
    counted), then finalize."""
    st = dict(levels=0, top_down_levels=0, bottom_up_levels=0, reached=0, edges_inspected=0, kernel_launches=1)
    level, i = 0, 0
    nf = 1
    if not (upper < 1 or lower > upper):
        while nf > 0 and level < upper and level < INT_MAX - 1:
            rec = levels[i]
            i += 1
            st["bottom_up_levels" if rec["bottom_up"] else "top_down_levels"] += 1
            st["kernel_launches"] += 1 + (3 if rec["bottom_up"] else 2)
            st["edges_inspected"] += rec["inspected"]
            nf = rec["found"]
            st["reached"] += nf
            if nf > 0:
                level += 1
    st["levels"] = level
    st["kernel_launches"] += 1 if n > 0 else 0
    ids = np.arange(n)
    dist = np.where((ids != source) & (depth > 0) & (depth >= lower) & (depth <= upper), depth, -1)
    return dist, st


def strategy_sequence(levels, stats):
    """'T' / 'B' per expansion the run performed"""
    k = stats["top_down_levels"] + stats["bottom_up_levels"]
    return "".join("B" if r["bottom_up"] else "T" for r in levels[:k])
