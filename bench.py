#!/usr/bin/env python3
"""bench.py -- PageRank edges/s on synthetic RMAT (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--scale S] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one complete hot-path pass: ParallelIterativePageRank semantics with
(max_iterations=20, damping=0.85, stop_epsilon=0.0) over the device-resident graph, i.e. 20 power
iterations + the final normalise (SURVEY 8d timed region; graph generation, CSR build and ingest are
reported separately).  value = E * iterations * steps / device time (CUDA events on the launching
stream, max over ranks).  e2e = the same metric through the public C-ABI call with a HOST output
buffer (params from host memory in, double[N] ranks copied device->host inside the timed region).

--impl reference times the reference's own algorithm (oracle/_ref, compiled from
/root/reference by oracle/Makefile; the plain-C port in oracle/ when that is absent) on the box's
host cores, all threads, on a bounded sample of the same workload (RMAT of a smaller scale).

N > 1: launched by torchrun, one rank per GPU; every rank builds its vertex partition of the same
RMAT graph and the partitions exchange contributions over NVLink peer memory inside the kernels
(torch.distributed is used only to swap IPC handles and to take the max of the timings).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)

ITERATIONS = 20
DAMPING = 0.85
EDGE_FACTOR = 16
SEED = 42
ALGO_BYTES_PER_EDGE = 12  # 4 B column index + 8 B gathered FP64 contribution      (SURVEY 8d)
ALGO_BYTES_PER_ROW = 24   # 4 B row offset + 4 B out-degree + 8 B old + 8 B new rank (SURVEY 8d)
REAL_STDOUT = 1
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def log(*a):
    print(*a, file=sys.stderr, flush=True)


DUMP_SAMPLE = 1 << 21  # elements kept of an output larger than DUMP_SAMPLE * 16 B (32 MiB)


def dump_output(directory, name, values):
    """--dump-outputs: writes what the last timed step returned as DIR/<name>.npy in float64, so that two builds run
    with the same arguments (same seeded inputs) can be compared output for output.  An output larger than 32 MiB is
    reduced to a fixed, seeded sample of DUMP_SAMPLE elements, whose positions go to DIR/<name>_index.npy (float64)."""
    os.makedirs(directory, exist_ok=True)
    values = np.asarray(values, dtype=np.float64)
    if values.nbytes > 16 * DUMP_SAMPLE:
        index = np.sort(np.random.default_rng(SEED).choice(len(values), DUMP_SAMPLE, replace=False))
        np.save(os.path.join(directory, name + "_index.npy"), index.astype(np.float64))
        values = values[index]
    np.save(os.path.join(directory, name + ".npy"), values)
    log(f"dumped {name} ({len(values)} values) to {directory}")


# ---- clocks sampling (nvidia-smi during the timed region) ---------------------------------------------

class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- peaks ----------------------------------------------------------------------------------------------

def hbm_peak():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        v = float(json.load(open(p))["hbm_gbs"])
        return v, "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


KERNEL_SOURCES = ("memgraph_b200/csrc/pagerank_kernels.cu", "memgraph_b200/csrc/core.hpp", "memgraph_b200/csrc/graph_build.cu")


def kernel_source_sha():
    import hashlib
    h = hashlib.sha256()
    for rel in KERNEL_SOURCES:
        h.update(open(os.path.join(REPO, rel), "rb").read())
    return h.hexdigest()


def ncu_traffic(world):
    """Per-launch DRAM bytes (read + write) of the dominant kernel from the committed `ncu --set full` capture of a
    partition of `world` (profiles/ncu_traffic.json, written by scripts/make_ncu_traffic.py from the .ncu-rep).  The file is
    stamped with a hash of the kernel sources it was captured from; a stale capture reads as null, not as a number."""
    try:
        d = json.load(open(os.path.join(REPO, "profiles", "ncu_traffic.json")))
        if d.get("kernel_source_sha256") != kernel_source_sha():
            return None
        return d["sell_rows_kernel_dram_bytes_per_launch"].get(str(world))
    except Exception:
        return None


# ---- reference arm / cpu baseline -------------------------------------------------------------------------

REF_THREAD_CANDIDATES = (1, 2, 4, 8, 16, 32, 64)


def _ref_impl():
    """(impl, kind): the reference's own pagerank.cpp compiled in place (oracle/_ref) or, where that is absent,
    the plain-C port.  Neither imports the product package: the RMAT input comes from oracle/rmat_oracle.c."""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from _checkers import Oracle, Reference  # noqa: E402  (bench.py's reference leg may execute oracle/)
    if Reference.available():
        return Reference(), "reference"
    return Oracle(), "port"


def cpu_reference_run(scale, steps, warmup, threads=None, sweep=True):
    """Times the reference's ParallelIterativePageRank (only that call, like the GPU side) on the benchmark's RMAT
    graph of `scale`.  The reference's thread count is a tunable with an interior optimum (every iteration merges one
    full-length vector per thread on the main thread, pagerank.cpp:104-112, so more threads eventually lose): with
    `sweep` one call per candidate T is timed first and the timed steps run at the best T.  Returns a dict."""
    impl, kind = _ref_impl()
    from _checkers import oracle_rmat_edges  # noqa: E402
    hw = os.cpu_count() or 1
    n, m = 1 << scale, EDGE_FACTOR << scale
    s, t = oracle_rmat_edges(scale, m, seed=SEED)
    t0 = time.perf_counter()
    g = impl.graph(n, s, t)
    build_s = time.perf_counter() - t0
    del s, t

    def call(T):
        t1 = time.perf_counter()
        impl.run(g, n, max_iterations=ITERATIONS, damping_factor=DAMPING, stop_epsilon=0.0, num_of_threads=T)
        return time.perf_counter() - t1

    sweep_s = {}
    if kind != "reference":
        threads = 1  # the C port walks the thread blocks sequentially
    elif threads is None:
        cands = sorted({c for c in REF_THREAD_CANDIDATES if c <= hw} | {hw}) if sweep else [min(8, hw)]
        for T in cands:
            sweep_s[T] = call(T)
            if T > 1 and sweep_s[T] > 2.5 * min(sweep_s.values()):
                break  # past the optimum and getting worse: larger T only adds serial merge work
        threads = min(sweep_s, key=sweep_s.get)
    for _ in range(warmup):
        call(threads)
    times = [call(threads) for _ in range(steps)]
    dt = float(sum(times))
    impl.free(g)
    eps = lambda sec: m * ITERATIONS / sec
    return {"value": m * ITERATIONS * steps / dt, "unit": "edges/s", "cores": threads, "kind": kind,
            "threads": threads, "host_threads_available": hw, "scale": scale, "best_of": len(sweep_s) or 1,
            "thread_sweep_edges_per_s": {str(k): eps(v) for k, v in sweep_s.items()},
            "value_1_thread": eps(sweep_s[1]) if 1 in sweep_s else None,
            "sample": f"RMAT scale-{scale} EF{EDGE_FACTOR} (N={n}, E={m}), {ITERATIONS} iterations, stop_epsilon=0, "
                      f"{steps} timed call(s) of ParallelIterativePageRank at its best thread count T={threads} "
                      f"(swept {sorted(sweep_s)} of {hw} host threads); graph ctor {build_s:.1f}s excluded",
            "ms_per_step": dt / steps * 1e3, "build_s": build_s}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # Bounded sample.  Same generator, same parameters, same call as the B200 arm; only the RMAT scale is bounded so
    # that ctor + thread sweep + (steps + warmup) calls stay within MGB200_REF_BUDGET_S (default 240 s).  Cost model
    # from a scale-20 probe at its best T: the call and the ctor grow ~2.4x per scale once the rank vectors leave the caches.
    budget = float(os.environ.get("MGB200_REF_BUDGET_S", "240"))
    calls = max(1, args.steps) + max(0, args.warmup)
    cap = min(args.cpu_scale, args.scale)
    probe_scale = min(20, cap)
    probe = cpu_reference_run(probe_scale, 1, 0)
    per_call, ctor = probe["ms_per_step"] / 1e3, probe["build_s"]
    scale = probe_scale
    est = lambda pc, ct: ct + pc * (calls + 6)  # 6 ~ the thread sweep
    while scale < cap and est(per_call * 2.4, ctor * 2.4) <= budget:
        scale += 1
        per_call *= 2.4
        ctor *= 2.4
    log(f"reference arm: probe scale-{probe_scale} {probe['ms_per_step']:.0f} ms/call at T={probe['threads']} -> "
        f"sample scale-{scale} (~{per_call:.1f} s/call x {calls} calls + ctor ~{ctor:.0f} s, budget {budget:.0f} s)")
    res = cpu_reference_run(scale, max(1, args.steps), max(0, args.warmup))
    line = {
        "impl": "reference", "metric": "pagerank_edges_per_second", "value": res["value"], "unit": "edges/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"PageRank RMAT scale-{args.scale} EF16, {ITERATIONS} iterations, d={DAMPING}, "
                               f"stop_epsilon=0, seed {SEED} (reference arm: bounded sample = the same generator at "
                               f"RMAT scale-{scale}, capped by --cpu-scale {args.cpu_scale} and a {budget:.0f} s budget)",
                   "sample_scale": scale, "threads": res["threads"]},
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "threads", "scale", "best_of",
                                             "host_threads_available", "value_1_thread", "thread_sweep_edges_per_s")},
        "e2e": {"value": res["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ---- B200 arm ------------------------------------------------------------------------------------------------

def dev_alloc(N, lib, device, nbytes):
    p = N.vp()
    rc = lib.mgb200_device_malloc(device, nbytes, ctypes.byref(p))
    if rc:
        raise RuntimeError(lib.mgb200_last_error().decode())
    return p


def measure_e2e_call(args, mg, N, lib, device, scale, n, m, host_out):
    import torch
    from memgraph_b200.pagerank import _check
    out = {}
    # the box's pinned H2D rate, for scale: 1 GiB, best of 3
    pin = torch.empty(1 << 28, dtype=torch.int32, pin_memory=True)
    dst = torch.empty(1 << 28, dtype=torch.int32, device=f"cuda:{device}")
    best = 1e9
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dst.copy_(pin, non_blocking=True)
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    out["pcie_pinned_h2d_gbs"] = (1 << 30) / best / 1e9
    del pin, dst
    # host COO of the benchmark graph: generated on the device (same bytes as the timed graph), copied back
    d_from = dev_alloc(N, lib, device, 4 * m)
    d_to = dev_alloc(N, lib, device, 4 * m)
    mg.rmat_edges_device(scale, m, d_from, d_to, seed=SEED, device=device)
    f32 = np.empty(m, dtype=np.uint32)
    t32 = np.empty(m, dtype=np.uint32)
    _check(lib.mgb200_copy_to_host(device, f32.ctypes.data, d_from, 4 * m))
    _check(lib.mgb200_copy_to_host(device, t32.ctypes.data, d_to, 4 * m))
    lib.mgb200_device_free(device, d_from)
    lib.mgb200_device_free(device, d_to)

    def one_shot(create, f, t, label, bytes_per_edge):
        res = None
        for _ in range(2):  # first call allocates the process-wide pinned staging
            h = N.vp()
            t0 = time.perf_counter()
            _check(create(device, n, m, f.ctypes.data, t.ctypes.data, 0, 1, ctypes.byref(h)))
            t1 = time.perf_counter()
            info = N.GraphInfo()
            _check(lib.mgb200_graph_get_info(h, ctypes.byref(info)))
            p, _cb = make_params_e2e()
            st = N.RunStatsC()
            _check(lib.mgb200_pagerank_run(h, ctypes.byref(p), host_out.ctypes.data, ctypes.byref(st)))
            t2 = time.perf_counter()
            lib.mgb200_graph_destroy(h)
            t3 = time.perf_counter()
            res = {"seconds": t3 - t0, "edges_per_s": m * ITERATIONS / (t3 - t0), "create_s": t1 - t0,
                   "upload_ms": info.upload_ms, "device_build_ms": info.build_ms, "run_s": t2 - t1, "destroy_s": t3 - t2,
                   "h2d_bytes": 8 * m, "h2d_gbs_during_upload": 8 * m / (info.upload_ms * 1e-3) / 1e9,
                   "host_bytes_read_per_edge": bytes_per_edge, "d2h_bytes": 8 * n, "rank_sum_check": float(host_out[:n].sum())}
        out[label] = res

    from memgraph_b200.pagerank import make_params
    make_params_e2e = lambda: make_params(ITERATIONS, DAMPING, 0.0)
    one_shot(lib.mgb200_graph_create_host_u32, f32, t32, "one_shot_u32", 8)
    f64 = f32.astype(np.uint64)
    t64 = t32.astype(np.uint64)
    del f32, t32
    one_shot(lib.mgb200_graph_create_host, f64, t64, "one_shot_u64", 16)
    del f64, t64
    out["h2d_fraction_of_pinned_rate"] = {k: out[k]["h2d_gbs_during_upload"] / out["pcie_pinned_h2d_gbs"]
                                          for k in ("one_shot_u32", "one_shot_u64")}
    # the drop-in module through the mgp ABI (fake host = tests' restatement of the engine side)
    try:
        sys.path.insert(0, os.path.join(REPO, "tests"))
        import _fakehost as fh
        ms = min(scale, int(os.environ.get("MGB200_MODULE_E2E_SCALE", "20")))
        mn, mm = 1 << ms, EDGE_FACTOR << ms
        f, t = mg.rmat_edges_host(ms, mm, seed=SEED)
        gids = np.arange(mn, dtype=np.int64)
        with fh.Module(fh.MODULE_SO) as module, fh.Graph(gids, f.astype(np.int64), t.astype(np.int64)) as g:
            module.call(g, ITERATIONS, DAMPING, 0.0, 1)
            t0 = time.perf_counter()
            nodes, ranks = module.call(g, ITERATIONS, DAMPING, 0.0, 1)
            dt = time.perf_counter() - t0
            os.environ["MGB200_GRAPH_CACHE"] = "1"
            module.call(g, ITERATIONS, DAMPING, 0.0, 1)
            t0 = time.perf_counter()
            module.call(g, ITERATIONS, DAMPING, 0.0, 1)
            dtc = time.perf_counter() - t0
            os.environ.pop("MGB200_GRAPH_CACHE", None)
        out["module_through_mgp_abi"] = {"scale": ms, "seconds": dt, "edges_per_s": mm * ITERATIONS / dt, "rows": int(len(nodes)),
                                         "seconds_with_graph_cache_hit": dtc, "rank_sum_check": float(np.sum(ranks)),
                                         "note": "CALL pagerank.get(20, 0.85, 0.0, 1) through libmgp_fake_host.so: pull "
                                                 "(3 ABI calls per edge), upload, build, iterate, emit (5 ABI calls per row)"}
    except Exception as ex:  # pragma: no cover
        out["module_through_mgp_abi"] = {"unavailable": repr(ex)}
    return out


CLASS_NAMES = ["zero_rows", "sell_rows", "sell_epilogue_push", "heavy_segments", "heavy_finish", "iter_end_barrier"]


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else (NCCL banners, torchrun chatter from
    libraries writing to fd 1) was diverted to stderr by main()."""
    os.write(REAL_STDOUT, (json.dumps(line) + "\n").encode())


def run_b200_arm(args):
    import memgraph_b200 as mg
    from memgraph_b200 import _native as N
    from memgraph_b200.pagerank import make_params, _check, _stats
    lib = N.lib()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            log(f"bench.py: --gpus {args.gpus} needs torchrun (WORLD_SIZE={world}); running rank 0 only is invalid")
            return 2
    device = local_rank
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(device)
        dist.init_process_group("nccl", device_id=torch.device("cuda", device))

    scale = args.scale
    n, m = 1 << scale, EDGE_FACTOR << scale
    t0 = time.perf_counter()
    # profiling aid (--quick only): MGB200_LONE_WORLD=P runs partition 0 of P on ONE GPU without peers -- the per-GPU
    # kernels of an N=P run, under ncu if wanted; ranks are meaningless, timings are not
    lone = int(os.environ.get("MGB200_LONE_WORLD", "0")) if (args.quick and world == 1) else 0
    if lone > 1:
        os.environ["MGB200_LONE_PARTITION"] = "1"
    # every rank builds its partition straight from the generator, a chunk of edges at a time (no device ever holds the
    # whole edge list: graph size scales with the GPU count)
    g = mg.PageRankGraph.from_rmat(scale, m, seed=SEED, device=device, part_rank=rank,
                                   part_world=lone if lone > 1 else world)
    build_wall_s = time.perf_counter() - t0
    gen_s = 0.0
    info = g.info
    log(f"[rank {rank}] RMAT scale-{scale}: generate + build {build_wall_s:.2f}s (device {info['build_ms']:.0f} ms), "
        f"rows {info['local_rows']} edges {info['local_edges']} heavy_rows {info['heavy_rows']} "
        f"heavy_edges {info['heavy_edges']} segs {info['heavy_segments']} sell_rows {info['sell_rows']} "
        f"sell_entries {info['sell_entries']} zero_rows {info['zero_rows']} resident {info['resident_bytes']/2**30:.2f} GiB "
        f"build peak {info['build_peak_bytes']/2**30:.2f} GiB")

    if world > 1:
        import torch
        handle = ctypes.create_string_buffer(N.IPC_HANDLE_BYTES)
        _check(lib.mgb200_graph_export_window(g.handle, handle))
        handles = [None] * world
        dist.all_gather_object(handles, handle.raw)
        arr = (N.vp * world)()
        keep = []
        for q in range(world):
            if q != rank:
                buf = ctypes.create_string_buffer(handles[q], N.IPC_HANDLE_BYTES)
                keep.append(buf)
                arr[q] = ctypes.cast(buf, N.vp)
        _check(lib.mgb200_graph_connect_peers(g.handle, arr, None))
        dist.barrier()

    local_rows = info["local_rows"]
    d_out = dev_alloc(N, lib, device, 8 * max(n if world == 1 else local_rows, 1))

    def step_device(timed_kernel=False):
        p, _cb = make_params(ITERATIONS, DAMPING, 0.0, on_device=True, time_spmv_kernel=timed_kernel)
        st = N.RunStatsC()
        if world == 1 and lone <= 1:
            _check(lib.mgb200_pagerank_run(g.handle, ctypes.byref(p), d_out, ctypes.byref(st)))
        else:
            _check(lib.mgb200_pagerank_run_partition(g.handle, ctypes.byref(p), d_out, None, ctypes.byref(st)))
        return _stats(st)

    for _ in range(max(args.warmup, 3)):
        step_device()
    if dist is not None:
        dist.barrier()
    sampler = ClockSampler(device)
    if rank == 0:
        sampler.start()
    step_ms, launches, kernel_ms, kernel_launches, iters = [], 0, 0.0, 0, 0
    class_ms = np.zeros(6)
    for _ in range(args.steps):
        if dist is not None:
            dist.barrier()
        st = step_device(timed_kernel=True)
        step_ms.append(st.iterate_ms)
        launches += st.kernel_launches
        kernel_ms += st.kernel_ms
        kernel_launches += st.kernel_timed_launches
        class_ms += np.array(st.class_ms)
        iters = st.iterations
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:  # single GPU (checked in main): d_out holds the ranks of the last timed step
        ranks = np.empty(n, dtype=np.float64)
        _check(lib.mgb200_copy_to_host(device, ranks.ctypes.data, d_out, 8 * n))
        dump_output(args.dump_outputs, "ranks", ranks)
        del ranks
    total_ms = float(sum(step_ms))
    if dist is not None:
        import torch
        tm = torch.tensor([total_ms], dtype=torch.float64, device=f"cuda:{device}")
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        total_ms = float(tm.item())
        ln = torch.tensor([launches], dtype=torch.int64, device=f"cuda:{device}")
        dist.all_reduce(ln, op=dist.ReduceOp.SUM)
        launches = int(ln.item())
    assert iters == ITERATIONS, f"executed {iters} iterations, expected {ITERATIONS}"
    value = m * ITERATIONS * args.steps / (total_ms * 1e-3)

    if args.quick:
        if rank == 0:
            emit({"quick": True, "scale": scale, "n_gpus": world, "ms_per_iteration": total_ms / args.steps / ITERATIONS,
                  "edges_per_s": value, "sell_kernel_ms": kernel_ms / max(kernel_launches, 1),
                  "class_ms_per_iteration": {k: round(float(v) / (args.steps * ITERATIONS), 4)
                                             for k, v in zip(CLASS_NAMES, class_ms)},
                  "build_wall_s": build_wall_s, "resident_gib": info["resident_bytes"] / 2**30,
                  "build_peak_gib": info["build_peak_bytes"] / 2**30, "local_edges": info["local_edges"],
                  "tag": os.environ.get("MGB200_TAG", "")})
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return 0
    # e2e: the public call with a HOST output buffer (D2H of the ranks inside the timed region)
    e2e = None
    if world == 1:
        pinned = None
        try:
            import torch  # plumbing: pinned host memory for the output buffer
            pinned = torch.empty(n, dtype=torch.float64, pin_memory=True).numpy()
        except Exception as ex:  # pragma: no cover
            log("pinned allocation failed, using pageable host memory:", ex)
        host_out = pinned if pinned is not None else np.empty(n, dtype=np.float64)
        g.run(ITERATIONS, DAMPING, 0.0, out=host_out)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            _, st = g.run(ITERATIONS, DAMPING, 0.0, out=host_out)
        e2e_dt = time.perf_counter() - t0
        e2e = {"value": m * ITERATIONS * args.steps / e2e_dt, "unit": "edges/s",
               "h2d_bytes_per_step": ctypes.sizeof(N.RunParams), "d2h_bytes_per_step": 8 * n,
               "api": "mgb200_pagerank_run(graph, params, host_rank_out) == ParallelIterativePageRank(graph, ...) -> "
                      "std::vector<double>", "rank_sum_check": float(host_out[:n].sum())}
    else:
        # partitioned: each rank copies its slice of the ranks to host memory inside the timed call
        try:
            import torch  # plumbing: pinned host memory for the result slices
            host_out = torch.empty(max(local_rows, 1), dtype=torch.float64, pin_memory=True).numpy()
            host_vtx = torch.empty(max(local_rows, 1), dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)
        except Exception as ex:  # pragma: no cover
            log("pinned allocation failed, using pageable host memory:", ex)
            host_out = np.empty(max(local_rows, 1), dtype=np.float64)
            host_vtx = np.empty(max(local_rows, 1), dtype=np.uint32)
        p, _cb = make_params(ITERATIONS, DAMPING, 0.0)
        _check(lib.mgb200_pagerank_run_partition(g.handle, ctypes.byref(p), host_out.ctypes.data,
                                                 host_vtx.ctypes.data, ctypes.byref(N.RunStatsC())))  # untimed first call
        st = N.RunStatsC()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            _check(lib.mgb200_pagerank_run_partition(g.handle, ctypes.byref(p), host_out.ctypes.data,
                                                     host_vtx.ctypes.data, ctypes.byref(st)))
        import torch
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=f"cuda:{device}")
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        sm = torch.tensor([float(host_out[:local_rows].sum())], dtype=torch.float64, device=f"cuda:{device}")
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        e2e = {"value": m * ITERATIONS * args.steps / float(dt.item()), "unit": "edges/s",
               "h2d_bytes_per_step": ctypes.sizeof(N.RunParams) * world, "d2h_bytes_per_step": 12 * n,
               "api": "mgb200_pagerank_run_partition(graph, params, host_rank_out, host_vertex_out) on every rank",
               "rank_sum_check": float(sm.item())}

    # e2e_call: what ONE `CALL pagerank.get()` pays beyond the iteration -- host COO in, host ranks out, graph built inside
    # the call (SURVEY 8f-3).  (a) the one-shot C-ABI entry points at the benchmark scale, uint64 pairs as in the
    # reference's EdgePair and uint32 dense ids as the module holds them; (b) the drop-in module through the mgp ABI
    # (tests' fake host; ABI-bound: 3 calls per edge, 5 per emitted row) on a smaller graph.
    e2e_call = None
    host_gib = os.sysconf("SC_PHYS_PAGES") * os.sysconf("SC_PAGE_SIZE") / 2**30
    if world == 1 and not args.no_e2e_call and lone <= 1 and host_gib < 40 * m / 2**30 + 16:
        log(f"e2e_call skipped: {host_gib:.0f} GiB of host memory is not enough for the host COO copies of scale-{scale}")
    elif world == 1 and not args.no_e2e_call and lone <= 1:
        try:
            e2e_call = measure_e2e_call(args, mg, N, lib, device, scale, n, m, host_out)
        except Exception as ex:  # pragma: no cover
            log("e2e_call failed:", repr(ex))

    # N > 1: rank parity against the single-GPU result on the same graph, outside the timed region.  Every rank drops
    # its (vertex, rank) slice into a full-length vector (disjoint slices, summed over NVLink), rank 0 rebuilds the
    # WHOLE graph as one partition on its own GPU, runs the same call and compares all N ranks.
    parity = None
    if world > 1 and not args.no_parity and scale <= 27:  # the single-GPU reference build must fit one device
        import torch
        dev = torch.device("cuda", device)
        full = torch.zeros(n, dtype=torch.float64, device=dev)
        idx = torch.from_numpy(host_vtx[:local_rows].astype(np.int64)).to(dev)
        full[idx] = torch.from_numpy(host_out[:local_rows]).to(dev)
        owned = torch.zeros(n, dtype=torch.int32, device=dev)
        owned[idx] = 1
        dist.all_reduce(full)
        dist.all_reduce(owned)
        if rank == 0:
            t0 = time.perf_counter()
            g1 = mg.PageRankGraph.from_rmat(scale, m, seed=SEED, device=device)
            single = torch.empty(n, dtype=torch.float64, device=dev)
            p1, _cb1 = make_params(ITERATIONS, DAMPING, 0.0, on_device=True)
            st1 = N.RunStatsC()
            _check(lib.mgb200_pagerank_run(g1.handle, ctypes.byref(p1), single.data_ptr(), ctypes.byref(st1)))
            g1.close()
            rel = ((full - single).abs() / single).max()
            parity = {"max_rel_vs_n1": float(rel.item()), "vertices_checked": n,
                      "every_vertex_owned_once": bool((owned == 1).all().item()),
                      "iterations_n1": int(st1.iterations), "iterations_partitioned": int(iters),
                      "how": "rank 0 rebuilt the whole graph as ONE partition on its GPU after the timed region and "
                             "compared all ranks of the partitioned run with it", "seconds": time.perf_counter() - t0}
            del single
        del full, owned, idx
        dist.barrier()

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    peak, peak_src = hbm_peak()
    sell_edges = info["local_edges"] - info["heavy_edges"]
    roofline = None
    if kernel_launches:
        per_launch_bytes = ALGO_BYTES_PER_EDGE * sell_edges + ALGO_BYTES_PER_ROW * info["sell_rows"]
        avg_ms = kernel_ms / kernel_launches
        achieved = per_launch_bytes / (avg_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "sell_rows_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "peak_source": peak_src,
                    "traffic": ncu_traffic(world),
                    "algorithmic_bytes_per_launch": per_launch_bytes, "avg_launch_ms": avg_ms,
                    "timed_launches": kernel_launches,
                    "units_per_launch": {"edges": sell_edges, "rows": info["sell_rows"]},
                    "whole_iteration": {
                        "algorithmic_bytes": ALGO_BYTES_PER_EDGE * m + ALGO_BYTES_PER_ROW * n,
                        "achieved": (ALGO_BYTES_PER_EDGE * m + ALGO_BYTES_PER_ROW * n) * ITERATIONS * args.steps
                        / (total_ms * 1e-3) / 1e9 / world,
                        "frac": (ALGO_BYTES_PER_EDGE * m + ALGO_BYTES_PER_ROW * n) * ITERATIONS * args.steps
                        / (total_ms * 1e-3) / 1e9 / world / peak,
                        "note": "12E+24N per iteration over the whole timed region (all kernels, per GPU)"}}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            r = cpu_reference_run(min(args.cpu_scale, 22), 1, 0)
            cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "threads", "scale", "best_of",
                                     "host_threads_available", "value_1_thread", "thread_sweep_edges_per_s")}
        except Exception as ex:
            log("cpu_baseline failed:", ex)

    line = {
        "metric": "pagerank_edges_per_second", "value": value, "unit": "edges/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"PageRank RMAT scale-{scale} EF16 (N={n}, E={m}), {ITERATIONS} iterations, d={DAMPING}, "
                               f"stop_epsilon=0, seed {SEED}", "parallelism": f"vertex-partition x{world}",
                   "l2": "inputs larger than L2 (index stream %.1f GB/iteration)" % (4 * m / 1e9),
                   "graph_build_wall_s": build_wall_s, "graph_build_ms": info["build_ms"], "build_peak_gib": info["build_peak_bytes"] / 2**30,
                   "heavy_rows": info["heavy_rows"], "heavy_edges": info["heavy_edges"], "sell_rows": info["sell_rows"],
                   "sell_entries": info["sell_entries"], "zero_rows": info["zero_rows"]},
        "ms_per_iteration": total_ms / args.steps / ITERATIONS,
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "e2e_call": e2e_call, "parity": parity, "gpu_launches": launches, "clocks": clocks,
        "kernel_ms_per_iteration": {k: float(v) / (args.steps * ITERATIONS) for k, v in zip(CLASS_NAMES, class_ms)},
    }
    emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_bfs_arm(args):
    """Next path (BASELINE config #5): BFS expand on RMAT scale-24, 1 GPU.  value = input edges / traversal
    time (Graph500-style TEPS) over K seeded sources."""
    import memgraph_b200 as mg
    from memgraph_b200 import _native as N
    from memgraph_b200 import bfs as B
    lib = N.lib()
    scale = args.scale if args.scale != 26 else 24
    n, m = 1 << scale, EDGE_FACTOR << scale
    d_from = dev_alloc(N, lib, 0, 4 * m)
    d_to = dev_alloc(N, lib, 0, 4 * m)
    mg.rmat_edges_device(scale, m, d_from, d_to, seed=SEED, device=0)
    t0 = time.perf_counter()
    g = B.BfsGraph.from_device(n, m, d_from, d_to)
    build_s = time.perf_counter() - t0
    lib.mgb200_device_free(0, d_from)
    lib.mgb200_device_free(0, d_to)
    rng = np.random.default_rng(SEED)
    sources = [0] + [int(x) for x in rng.integers(0, n, size=max(args.steps + args.warmup, 1))]
    for s in sources[:max(args.warmup, 3)]:
        g.distances(s)
    ms, reached, inspected, level_counts, launches = [], [], [], [], 0
    t0 = time.perf_counter()
    for s in sources[:args.steps]:
        dist, st = g.distances(s)
        ms.append(st["traverse_ms"]); reached.append(st["reached"]); inspected.append(st["edges_inspected"])
        level_counts.append(st["levels"])
        launches += st["kernel_launches"]
    e2e_dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_output(args.dump_outputs, "distances", dist)
    total = float(sum(ms))
    # Roofline (HBM-bound integer work).  Algorithmic bytes of one direction-optimising traversal (DESIGN.md 7):
    #   4 B per inspected adjacency entry + 12 B per reached vertex (8 B row offsets, 4 B distance written)
    #   + 2 * N/8 B per level (frontier bitmap written, then read by the next level)
    algo = [4 * i + 12 * r + 2 * (n // 8) * l for i, r, l in zip(inspected, reached, level_counts)]
    peak, peak_src = hbm_peak()
    achieved = float(sum(algo)) / (total * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "bfs traversal (all level kernels of one source)", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src, "traffic": None,
                "algorithmic_bytes_per_launch": float(np.mean(algo)),
                "formula": "4*edges_inspected + 12*reached + 2*(N/8)*levels per traversal",
                "note": "a traversal that inspects 4 % of the adjacency is latency-bound by its ~7 dependent levels, "
                        "not by bytes; the fraction is reported for completeness"}
    cpu = None
    if not args.no_cpu_baseline:
        try:
            sys.path.insert(0, os.path.join(REPO, "tests"))
            from _checkers import BfsOracle, oracle_rmat_edges  # bench.py's cpu_baseline leg may execute oracle/
            cs = min(scale, 22)
            cn, cm = 1 << cs, EDGE_FACTOR << cs
            f, t = oracle_rmat_edges(cs, cm, seed=SEED)
            t0 = time.perf_counter()
            BfsOracle().distances(cn, f, t, 0)
            dt = time.perf_counter() - t0
            cpu = {"value": cm / dt, "unit": "edges/s", "cores": 1, "kind": "port",
                   "sample": f"oracle/bfs_oracle.c (restatement of the cursor in src/query/plan/operator.cpp:2692-2912; the "
                             f"engine cannot be built here), RMAT scale-{cs}, source 0, one traversal incl. adjacency build"}
        except Exception as ex:
            log("cpu_baseline failed:", ex)
    emit({"metric": "bfs_input_edges_per_second", "value": m * args.steps / (total * 1e-3), "unit": "edges/s",
          "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total / args.steps,
          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
          "config": {"workload": f"BFS expand (direction OUT, default bounds) RMAT scale-{scale} EF16 (N={n}, E={m}), "
                                 f"{args.steps} seeded sources", "graph_build_s": build_s,
                     "reached_per_source": reached, "edges_inspected_per_source": inspected, "levels_per_source": level_counts},
          "roofline": roofline, "cpu_baseline": cpu,
          "e2e": {"value": m * args.steps / e2e_dt, "unit": "edges/s", "h2d_bytes_per_step": 32,
                  "d2h_bytes_per_step": 4 * n, "api": "mgb200_bfs_run(graph, source, ..., host_dist_out)"},
          "gpu_launches": launches})
    return 0


def run_katz_arm(args):
    """Next path (SURVEY 8f-1): static Katz centrality, katz_alg::SetKatz, on RMAT scale-22 (1 GPU).  A step is one
    SetKatz call on the device-resident graph; value = E * iterations / loop time (CUDA events)."""
    import memgraph_b200 as mg
    from memgraph_b200 import _native as N
    from memgraph_b200 import katz as K
    lib = N.lib()
    scale = args.scale if args.scale != 26 else 22
    n, m = 1 << scale, EDGE_FACTOR << scale
    d_from = dev_alloc(N, lib, 0, 4 * m)
    d_to = dev_alloc(N, lib, 0, 4 * m)
    mg.rmat_edges_device(scale, m, d_from, d_to, seed=SEED, device=0)
    g = mg.PageRankGraph.from_device(n, m, d_from, d_to)
    lib.mgb200_device_free(0, d_from)
    lib.mgb200_device_free(0, d_to)
    # alpha: the module's default 0.2 makes gamma negative on a skewed graph (alpha^2 deg_max > 1) and the reference stops
    # after ONE iteration; the benchmark uses the largest "real" problem, alpha = 0.9 / sqrt(deg_max + 1), epsilon = 1e-3
    try:
        _, st0 = K.set_katz(g, 0.2, 1e-2, 1)
    except K.NotConverged as ex:
        st0 = ex.stats
    deg_max = st0["max_out_degree"]
    alpha, eps = 0.9 / float(np.sqrt(deg_max + 1.0)), 1e-3
    for _ in range(max(args.warmup, 3)):
        K.set_katz(g, alpha, eps)
    ms, iters, launches = [], 0, 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cent, st = K.set_katz(g, alpha, eps)
        ms.append(st["iterate_ms"]); iters = st["iterations"]; launches += st["kernel_launches"]
    e2e_dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_output(args.dump_outputs, "centrality", cent)
    total = float(sum(ms))
    info = g.info
    g.close()
    # per iteration: the gather phase (12 B per edge like PageRank) + per vertex: omega written 8, c read+written 16, ur
    # written 8, row offset 4 = 36 B, + the separation test reading c, ur once and writing/reading one sort key = 24 B
    algo_iter = 12 * m + 60 * n
    peak, peak_src = hbm_peak()
    achieved = algo_iter * iters * args.steps / (total * 1e-3) / 1e9
    cpu = None
    if not args.no_cpu_baseline:
        try:
            sys.path.insert(0, os.path.join(REPO, "tests"))
            from _checkers import oracle_rmat_edges
            from test_katz_oracle import oracle_katz, ref_katz, KATZ_REF_SO
            cs = min(scale, 20)
            cn, cm = 1 << cs, EDGE_FACTOR << cs
            f, t = oracle_rmat_edges(cs, cm, seed=SEED)
            dmax = int(np.bincount(f.astype(np.int64), minlength=cn).max())
            ca = 0.9 / float(np.sqrt(dmax + 1.0))
            rc, _c, cit = oracle_katz(cn, f, t, ca, eps)
            kind = "reference" if os.path.exists(KATZ_REF_SO) else "port"
            t0 = time.perf_counter()
            if kind == "reference":
                ref_katz(cn, f, t, ca, eps)
            else:
                oracle_katz(cn, f, t, ca, eps)
            dt = time.perf_counter() - t0
            cpu = {"value": cm * cit / dt, "unit": "edges/s", "cores": 1, "kind": kind,
                   "sample": f"katz_alg::SetKatz on RMAT scale-{cs}, alpha {ca:.4g}, epsilon {eps}, {cit} iterations, graph "
                             f"ingest included (the reference builds its adjacency inside the call)"}
        except Exception as ex:
            log("cpu_baseline failed:", ex)
    emit({"metric": "katz_edges_per_second", "value": m * iters * args.steps / (total * 1e-3), "unit": "edges/s", "n_gpus": 1,
          "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total / args.steps, "higher_is_better": True,
          "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
          "config": {"workload": f"Katz centrality (SetKatz) RMAT scale-{scale} EF16 (N={n}, E={m}), alpha {alpha:.5g} "
                                 f"(= 0.9/sqrt(deg_max+1), deg_max {deg_max}), epsilon {eps}, {iters} iterations to separation",
                     "heavy_rows": info["heavy_rows"], "sell_rows": info["sell_rows"], "zero_rows": info["zero_rows"]},
          "ms_per_iteration": total / args.steps / max(iters, 1),
          "roofline": {"bound": "hbm", "kernel": "whole Katz iteration (gather kernels + epilogue + separation test)",
                       "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                       "traffic": None, "algorithmic_bytes_per_launch": algo_iter, "formula": "12*E + 60*N per iteration"},
          "cpu_baseline": cpu,
          "e2e": {"value": m * iters * args.steps / e2e_dt, "unit": "edges/s", "h2d_bytes_per_step": 24,
                  "d2h_bytes_per_step": 8 * n, "api": "mgb200_katz_run(graph, alpha, epsilon, 0, host_centrality_out)"},
          "gpu_launches": launches})
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=int, default=int(os.environ.get("MGB200_BENCH_SCALE", "26")))
    ap.add_argument("--cpu-scale", type=int, default=int(os.environ.get("MGB200_CPU_SCALE", "24")),
                    help="RMAT scale of the bounded CPU sample (reference arm / cpu_baseline)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e-call", action="store_true", help="skip the one-shot host-COO-in / host-ranks-out measurement")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the comparison with the single-GPU result")
    ap.add_argument("--workload", default="pagerank", choices=["pagerank", "bfs", "katz"],
                    help="pagerank (the BASELINE metric, default), bfs (config #5) or katz (SURVEY 8f-1)")
    ap.add_argument("--quick", action="store_true", help="sweep mode: device-resident timing only, compact JSON")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the output of the last one as DIR/<name>.npy (float64; a fixed "
                         "seeded sample of outputs over 32 MiB); single-GPU B200 path only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.gpus != 1 or args.impl != "b200"):
        ap.error("--dump-outputs needs --gpus 1 and --impl b200")
    global REAL_STDOUT
    sys.stdout.flush()
    REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # anything a library prints to stdout lands on stderr; emit() writes the JSON line
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.workload == "bfs":
        return run_bfs_arm(args)
    if args.workload == "katz":
        return run_katz_arm(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
