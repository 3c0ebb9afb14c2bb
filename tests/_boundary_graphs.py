"""CPU side of tests/test_gpu_gather_variants.py: graphs shaped to reach the boundaries of the gather layout, a model of
the layout build_graph reports for them (graph_build.cu), and high-precision restatements of the PageRank recurrences
(oracle/pagerank_oracle.c, oracle/cugraph_pagerank_oracle.c) with the rounding bounds the device results must meet."""
import math
from dataclasses import dataclass, field

import numpy as np

SLICE_ROWS = 32        # kSliceRows: rows per SELL slice
SELL_UNROLL = 8        # MGB_SELL_UNROLL: columns per batch of the SELL walk
HEAVY_UNROLL = 8       # kUnroll of heavy_segments_kernel: 32 * 8 = 256 edges per unrolled step
SELL_ONLY_H = 1 << 30  # a heavy minimum degree no row reaches
U = 2.0 ** -53         # unit roundoff of FP64


@dataclass
class Graph:
    name: str
    n: int
    f: np.ndarray  # uint64 sources, input edge order
    t: np.ndarray  # uint64 targets
    H: int         # MGB200_HEAVY_MIN_DEGREE
    S: int         # MGB200_SEGMENT_EDGES
    w: np.ndarray = None                          # weights of the weighted variant
    seeds: tuple = None                           # (vertices, values) of the personalised runs, one duplicate
    intended: dict = field(default_factory=dict)  # boundaries the graph was built to reach

    @property
    def indeg(self):
        return np.bincount(self.t.astype(np.int64), minlength=self.n)

    @property
    def outdeg(self):
        return np.bincount(self.f.astype(np.int64), minlength=self.n)


def _finish(name, n, f, t, H, S, rng, intended):
    """Shuffled edge order, weights (some 0, and one source whose out-edges all weigh 0), seeds with a duplicate."""
    order = rng.permutation(len(f))
    f, t = np.asarray(f, dtype=np.uint64)[order], np.asarray(t, dtype=np.uint64)[order]
    w = rng.uniform(0.0, 5.0, len(f))
    w[rng.random(len(f)) < 0.05] = 0.0
    outdeg = np.bincount(f.astype(np.int64), minlength=n)
    several = np.flatnonzero(outdeg >= 2)
    if len(several):
        w[f == several[len(several) // 2]] = 0.0
    a, b = int(rng.integers(0, n)), int(rng.integers(0, n))
    seeds = (np.array([a, b, a], dtype=np.uint64), np.array([1.0, 2.0, 0.5]))
    return Graph(name, n, f, t, H, S, w, seeds, intended)


def hub_in_degree(S):
    """About 10 S; for the largest segment sizes 8 S + 1, which keeps the in-tree bound at 20 iterations under 1e-11."""
    return 10 * S if 10 * S <= 2100 else 8 * S + 1


def boundary_graph(H, S, seed, n_sell_mod=None):
    """Every vertex gets a chosen in-degree; each in-edge's source is drawn at random from all vertices except a few
    sinks (self-loops and multi-edges allowed), then 300 of those sources become one hub with a large out-degree.

    Heavy rows: H, H+1; S-1, S, S+1, 2S-1, 2S, 2S+1 (segment boundaries); 255, 256, 257 (the heavy kernel's unrolled
    step of 32 x 8 edges against its tail loop); about 10 S.  Only the degrees >= H are heavy, so some of these are
    absent for small S.  SELL rows: one of degree H-1 and 32 rows at every width 1..17 (both sides of every multiple of
    the SELL walk's 8-column batch), a run of more than 40 slices of widths 1 and 2 (a work item longer than 32 slices
    reloads its slice ends), and enough extra degree-1 rows to make n_sell % 32 == n_sell_mod (a partly filled last
    slice).  Plus zero in-degree rows."""
    assert H >= 18, "the SELL widths 1..17 must stay below H"
    rng = np.random.default_rng(seed)
    heavy_targets = [H, H + 1, S - 1, S, S + 1, 2 * S - 1, 2 * S, 2 * S + 1, 255, 256, 257, hub_in_degree(S)]
    heavy = sorted({d for d in heavy_targets if d >= H})
    sell = [H - 1] + [wd for wd in range(1, 18) for _ in range(SLICE_ROWS)] + [2] * (20 * SLICE_ROWS) + [1] * (
        22 * SLICE_ROWS)
    if n_sell_mod is not None:
        sell += [1] * ((n_sell_mod - len(sell)) % SLICE_ROWS)
    zero = 40
    degs = np.array(heavy + sell + [0] * zero, dtype=np.int64)
    n = len(degs)
    vid = rng.permutation(n)  # vertex id of each in-degree slot
    sinks = rng.choice(n, 12, replace=False)
    allowed = np.setdiff1d(np.arange(n), sinks)
    t = np.repeat(vid, degs)
    f = rng.choice(allowed, len(t))
    hub = int(allowed[rng.integers(0, len(allowed))])
    f[rng.choice(len(f), 300, replace=False)] = hub  # the in-degrees stay as designed
    intended = dict(heavy_degrees=[d for d in heavy], sell_degree=H - 1, widths=list(range(1, 18)), narrow_slices=41,
                    n_sell_mod=n_sell_mod, zero_rows=True, heavy_rows=True, sell_rows=True)
    return _finish(f"boundary_H{H}_S{S}", n, f, t, H, S, rng, intended)


def random_graph(name, n, m, H, S, seed, intended):
    rng = np.random.default_rng(seed)
    f, t = rng.integers(0, n, m), rng.integers(0, n, m)
    return _finish(name, n, f, t, H, S, rng, intended)


def all_graphs():
    gs = [boundary_graph(24, 1, 11), boundary_graph(24, 31, 12, n_sell_mod=1), boundary_graph(24, 32, 13, n_sell_mod=31),
          boundary_graph(24, 256, 14), boundary_graph(24, 257, 15)]
    gs.append(random_graph("heavy_only", 600, 4000, 1, 32, 16, dict(heavy_rows=True, sell_rows=False)))
    gs.append(random_graph("sell_only", 1500, 9000, SELL_ONLY_H, 256, 17, dict(heavy_rows=False, sell_rows=True)))
    one = _finish("single_self_loop", 1, [0], [0], 24, 1, np.random.default_rng(18), dict(heavy_rows=False, sell_rows=True))
    gs.append(one)
    # 127 labels: SMEM_TABLE_KB=1 and 64 both give a table of 126 (rounded down to an even count), label 126 is read
    # from global memory
    gs.append(random_graph("odd_n_table", 127, 900, 24, 31, 19, dict(odd_n=True)))
    return gs


# ---- the layout build_graph reports ----------------------------------------------------------------------------------

def layout(indeg, H, S):
    """GraphInfo fields predicted from the in-degrees: rows sorted by in-degree descending; degree >= H heavy, 1..H-1
    SELL (slices of 32 rows, width = degree of the slice's first row), 0 zero rows."""
    d = np.sort(np.asarray(indeg, dtype=np.int64))[::-1]
    heavy = d[d >= H]
    sell = d[(d >= 1) & (d < H)]
    widths = sell[::SLICE_ROWS]
    return dict(heavy_rows=len(heavy), heavy_edges=int(heavy.sum()), heavy_segments=int(((heavy + S - 1) // S).sum()),
                sell_rows=len(sell), sell_slices=len(widths), sell_entries=SLICE_ROWS * int(widths.sum()),
                zero_rows=int((d == 0).sum()), local_edges=int(d.sum()))


def slice_widths(indeg, H):
    d = np.sort(np.asarray(indeg, dtype=np.int64))[::-1]
    return d[(d >= 1) & (d < H)][::SLICE_ROWS]


def work_items(widths, n_items, slice_cost=8):
    """Slice ranges of the SELL work items (sell_items_kernel): item i starts at the first slice s whose cost
    colbase[s] + slice_cost * s reaches i / n_items of the total; n_items is capped at the slice count."""
    widths = np.asarray(widths, dtype=np.int64)
    ns = len(widths)
    n_items = min(ns, n_items)
    colbase = np.concatenate([[0], np.cumsum(widths)])
    cost = colbase + slice_cost * np.arange(ns + 1)
    total = int(colbase[-1]) + slice_cost * ns
    begin = [int(np.searchsorted(cost, (total * i) // n_items, side="left")) for i in range(n_items)] + [ns]
    return [(begin[i], begin[i + 1]) for i in range(n_items)]


# ---- high-precision restatements ---------------------------------------------------------------------------------------

EXTENDED = np.finfo(np.longdouble).nmant >= 63  # x86 80-bit or wider; else exactly rounded sums with math.fsum


def _segment_sum(vals, idx, n):
    """sum of vals[e] into slot idx[e]: in long double, or exactly rounded per slot (math.fsum)."""
    if EXTENDED:
        out = np.zeros(n, dtype=np.longdouble)
        np.add.at(out, idx, vals)
        return out
    out = np.zeros(n)
    order = np.argsort(idx, kind="stable")
    bounds = np.searchsorted(idx[order], np.arange(n + 1))
    for v in range(n):
        out[v] = math.fsum(vals[order[bounds[v]:bounds[v + 1]]])
    return out


def _total(vals):
    return vals.sum(dtype=np.longdouble) if EXTENDED else math.fsum(vals)


def _ld(x):
    return np.asarray(x, dtype=np.longdouble if EXTENDED else np.float64)


def hp_pagerank(n, f, t, iterations, damping=0.85):
    """oracle/pagerank_oracle.c for a fixed iteration count, normalised like its last step."""
    f, t = np.asarray(f, dtype=np.int64), np.asarray(t, dtype=np.int64)
    outdeg = _ld(np.bincount(f, minlength=n))
    d = _ld(damping)
    rank = np.full(n, _ld(1) / _ld(n))
    for _ in range(iterations):
        rank = (_ld(1) - d) / _ld(n) + d * _segment_sum(rank[f] / outdeg[f], t, n)
    return rank / _total(rank)


def hp_cugraph_pagerank(n, f, t, iterations, weights=None, seeds=None, alpha=0.85):
    """oracle/cugraph_pagerank_oracle.c for a fixed iteration count: out-weight sums, dangling mass, teleport p."""
    f, t = np.asarray(f, dtype=np.int64), np.asarray(t, dtype=np.int64)
    w = _ld(np.ones(len(f)) if weights is None else weights)
    out_w = _segment_sum(w, f, n)
    if seeds is None:
        p = np.full(n, _ld(1) / _ld(n))
    else:
        vals = _ld(seeds[1])
        p = _segment_sum(vals / _total(vals), np.asarray(seeds[0], dtype=np.int64), n)
    a = _ld(alpha)
    dangling = out_w == 0
    live = ~dangling[f]
    pr = np.full(n, _ld(1) / _ld(n))
    for _ in range(iterations):
        spread = a * _total(pr[dangling]) + (_ld(1) - a)
        gathered = _segment_sum(w[live] * (pr[f[live]] / out_w[f[live]]), t[live], n)
        pr = a * gathered + spread * p
    return pr


# ---- rounding bounds --------------------------------------------------------------------------------------------------

def pagerank_bound(g, k):
    """In-tree PageRank after k iterations: every row is a sum of at most D_in positive terms, in any order, and the
    final normalisation divides by a sum of n positive terms: 2 k (D_in + ceil(log2 n) + 8) 2^-53."""
    return 2 * k * (int(g.indeg.max()) + math.ceil(math.log2(g.n)) + 8) * U


def cugraph_bound(g, k, weighted=False, personalised=False):
    """cuGraph-semantics PageRank after k iterations.  Every quantity is a sum of non-negative terms, so an iterate whose
    entries carry relative errors <= E yields, computed exactly, entries with relative errors <= E; each iteration
    then adds, to first order and in units of 2^-53, per row v:
        contribution pr[u] / out_w[u]                1, plus the out-weight sum's own error: D_out - 1 on a weighted
                                                     handle (a sum of D_out non-negative weights), 0 otherwise
                                                     (integer out-degrees are exact)
        weight * contribution                        1 (weighted only)
        the row's sum of at most D_in terms          D_in - 1, in any order (SELL padding adds exact zeros)
        alpha * gathered                             1
        dangling mass: sum over n_dang sinks         n_dang - 1, then alpha * dangling, 1 - alpha, their sum: 3
        teleport p[v]                                uniform 1/n: 1; personalised: sum of the values, quotient, and
                                                     duplicate seeds added up: <= 2 n_pers
        spread * p[v], and the final sum            2
    plus 1 for the initial 1/n.  So per iteration delta <= (D_in + D_out [weighted] + n_dang + 2 n_pers + 10) 2^-53,
    and after k iterations (1 + delta)^k - 1 <= 1.01 k delta while k delta <= 1e-11; the factor also covers the
    reference's own long-double rounding (2^-11 of the same terms)."""
    ow = np.bincount(g.f.astype(np.int64), weights=g.w if weighted else None, minlength=g.n)
    n_dang = int((ow == 0).sum())
    d_out = int(g.outdeg.max()) if weighted else 0
    n_pers = len(g.seeds[0]) if personalised else 0
    return 1.01 * k * (int(g.indeg.max()) + d_out + n_dang + 2 * n_pers + 10) * U


def max_rel_err(got, ref):
    """max |got - ref| / |ref| over ref != 0; where ref == 0 the result must be exactly 0 (else inf)."""
    got, ref = np.asarray(got, dtype=np.longdouble), np.asarray(ref, dtype=np.longdouble)
    zero = ref == 0
    if np.any(got[zero] != 0):
        return math.inf
    if not np.any(~zero):
        return 0.0
    return float(np.max(np.abs(got[~zero] - ref[~zero]) / np.abs(ref[~zero])))


def walk_counts(n, f, t, iterations):
    """Exact walk counts omega_i = A^T omega_{i-1}, omega_0 = 1 (Python integers), for i = 1..iterations."""
    f, t = np.asarray(f, dtype=np.int64), np.asarray(t, dtype=np.int64)
    omega = np.ones(n, dtype=object)
    out = []
    for _ in range(iterations):
        nxt = np.zeros(n, dtype=object)
        np.add.at(nxt, t, omega[f])
        omega = nxt
        out.append(max(omega) if n else 0)
    return out
