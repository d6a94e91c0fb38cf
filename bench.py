#!/usr/bin/env python
"""bench.py -- the headline benchmark of BASELINE.json on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (config.workload): BASELINE.json configs[1] -- R-MAT scale-22, average degree 16, FP32 values,
`A.mxv(u, semiring=FP32.PLUS_TIMES)` (SpMV), the configuration the metric "SpMV GEdge/s" is quoted on.  A "step" is
one SpMV over the whole graph.  With N > 1 the matrix is 1-D row-block partitioned (equal blocks of the pseudo-randomly
relabelled vertex ids: equal rows and equal work), one process per GPU; a step is the local GrB_mxv followed by the library's own all-gather of
the output slices over NVLink peer memory (csrc/dist.cu: push kernel + flag wait, no NCCL call on the data path), so
every rank ends the step holding the full result vector (strong scaling: the graph is fixed as N grows).  The
replicated result of the LAST timed step is checked on rank 0 against the CPU port (presence bit-exact) and an fp64
reference (<= 1e-6 relative) at every N.

value      whole-job GEdge/s, inputs resident in HBM, CUDA events on the library's stream, max over ranks.
e2e        the same call made the way a user of the reference makes it -- Matrix.mxv of the host-side mirror of the
           reference's interface -> libb200grb.so -- with u coming from pinned host memory and w (values + presence)
           going back to pinned host memory inside the timed region.
roofline   algorithmic bytes of one local SpMV / device time of one step of the SAME timed loop; the dominant kernel's
           share of the step comes from the committed ncu launch list (profiles/).
The line also carries SpGEMM (configs[3]) with its own roofline and CPU baseline, BFS (configs[2]) and SSSP (configs[4]
shape), each with a full-size parity flag; with N > 1 they run in their distributed forms (row panels / all-gather /
all-reduce).

--impl reference times the CPU side: SuiteSparse:GraphBLAS is not installable offline, so the reference arm is the
OpenMP port in oracle/grb_fast.c (kind "port") on the host cores this process may use (cgroup quota honoured).
"""
import argparse
import ctypes
import importlib.util
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "SpMV GEdge/s (R-MAT s22 d16 PLUS_TIMES_FP32 mxv)"
UNIT = "GEdge/s"
GENERATOR = "Graph500 R-MAT a,b,c,d=.57,.19,.19,.05 ef16 seed 1, dedup"


# ------------------------------------------------------------------ inputs
def _generators():
    """pygraphblas_b200/generators.py loaded BY PATH: the reference arm must not dlopen the CUDA library."""
    spec = importlib.util.spec_from_file_location("_b200grb_generators", os.path.join(ROOT, "pygraphblas_b200", "generators.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def cached_graph(scale, edgefactor=16, seed=1):
    """R-MAT CSR (n, indptr, indices), cached under /tmp so both arms / all ranks share one build."""
    base = f"/tmp/b200grb_rmat_s{scale}_e{edgefactor}_seed{seed}"
    if os.path.exists(base + ".done"):
        return 1 << scale, np.load(base + "_indptr.npy"), np.load(base + "_indices.npy")
    n, indptr, indices = _generators().rmat_csr(scale, edgefactor, seed)
    try:
        np.save(base + "_indptr.npy", indptr)
        np.save(base + "_indices.npy", indices)
        open(base + ".done", "w").close()
    except OSError:
        pass
    return n, indptr, indices


def spmv_inputs(nnz, n):
    rng = np.random.default_rng(2)
    vals = (rng.random(nnz, dtype=np.float32) + np.float32(0.5)).astype(np.float32)    # U[0.5, 1.5)
    u = rng.random(n, dtype=np.float32)                                                # U[0, 1)
    return vals, u


def workload_config(scale, n, nnz):
    """The SAME dict in both arms (the driver compares them)."""
    return {"workload": f"R-MAT scale-{scale} avg-deg-16 FP32 SpMV PLUS_TIMES (BASELINE.json configs[1])",
            "n": int(n), "nnz": int(nnz), "generator": GENERATOR,
            "l2": "inputs (A: %.0f MB) exceed the 126 MB L2; no explicit flush" % (nnz * 8 / 1e6)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def profile_json(name):
    try:
        with open(os.path.join(ROOT, "profiles", name)) as f:
            return json.load(f)
    except Exception:
        return {}


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag, self.thread, self.ok = [], set(), False, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max = None

    def _run(self):
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((clk, util))
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.ok:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max, "reasons": [], "samples": 0}
        loaded = [c for c, u in self.samples if u > 0] or [c for c, _ in self.samples]
        return {"sm_mhz": float(np.median(loaded)), "sm_max_mhz": self.max, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------ CPU port (reference arm / cpu_baseline)
_BUDGET = None


def host_cpu_budget():
    """(threads this process may usefully run, description): the scheduler affinity capped by the cgroup CPU quota
    (a 1-GPU lease is often a slice of the host: 128 'visible' CPUs behind a quota of 16).  Read once, BEFORE the
    OpenMP runtime of the port is loaded: with OMP_PROC_BIND it pins the calling thread, which would shrink the mask."""
    global _BUDGET
    if _BUDGET is not None:
        return _BUDGET
    aff = len(os.sched_getaffinity(0))
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:             # cgroup v2: "<quota|max> <period>"
            q, p = f.read().split()
            if q != "max":
                quota = float(q) / float(p)
    except Exception:
        try:                                                   # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    eff = aff if quota is None else max(1, min(aff, int(np.ceil(quota))))
    _BUDGET = (eff, {"affinity_cpus": aff, "cgroup_cpu_quota": quota})
    return _BUDGET


def oracle_lib():
    host_cpu_budget()
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    from oracle import oracle as orc
    L = orc.lib()
    L.fast_num_threads.restype = ctypes.c_int
    L.fast_spmv_plan_f32.restype = ctypes.c_void_p
    L.fast_bfs_step.restype = ctypes.c_int64
    return L


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


DUMP_BYTES = 64_000_000


def dump_outputs(dirname, x, present):
    """--dump-outputs DIR: the result vector w of the last timed step, as a caller of mxv receives it, in DIR/<name>.npy:
    w_values (float32, 0 where w has no entry) and w_present (float32, 1 where it has one).  Above DUMP_BYTES in all, a
    fixed seeded sample of the rows is written instead, with their ids in w_rows (float64)."""
    out = {"w_values": np.where(present != 0, x, 0).astype(np.float32), "w_present": (present != 0).astype(np.float32)}
    if 8 * len(x) > DUMP_BYTES - 4096:
        rows = np.sort(np.random.default_rng(0).choice(len(x), size=(DUMP_BYTES - 4096) // 16, replace=False))
        out = {k: v[rows] for k, v in out.items()}
        out["w_rows"] = rows.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def cpu_spmv(n, indptr, indices, vals, u, min_seconds, max_reps):
    """The OpenMP port in its best measured configuration; returns (threads_used, budget, times, w, presence)."""
    L = oracle_lib()
    w = np.zeros(n, np.float32)
    pres = np.zeros(n, np.uint8)
    args = (ctypes.c_int64(n), P(indptr), P(indices), P(vals), P(u), P(w), P(pres))
    budget, info = host_cpu_budget()
    # the baseline gets its best configuration, chosen by measurement (best of three passes each): the CPU budget and
    # fractions of it (on SMT hosts fewer threads than logical CPUs are often faster for this gather-bound loop) x two
    # variants of the port -- dynamic row chunks, or nnz-balanced per-thread partitions first-touched by their thread
    best = None
    for nt in sorted({budget, max(1, 3 * budget // 4), max(1, budget // 2), max(1, budget // 4)}, reverse=True):
        L.fast_set_threads(ctypes.c_int(nt))
        plan = ctypes.c_void_p(L.fast_spmv_plan_f32(ctypes.c_int64(n), P(indptr), P(indices), P(vals), ctypes.c_int(nt)))
        for variant in ("rows", "plan"):
            run = (lambda: L.fast_spmv_plus_times_f32(*args)) if variant == "rows" else (lambda: L.fast_spmv_plan_run_f32(plan, P(u), P(w), P(pres)))
            run()                                  # warm-up / page-in
            dt = None
            for _ in range(3):
                t0 = time.perf_counter()
                run()
                d = time.perf_counter() - t0
                dt = d if dt is None or d < dt else dt
            if best is None or dt < best[0]:
                best = (dt, nt, variant)
        L.fast_spmv_plan_free_f32(plan)
    L.fast_set_threads(ctypes.c_int(best[1]))
    plan = ctypes.c_void_p(L.fast_spmv_plan_f32(ctypes.c_int64(n), P(indptr), P(indices), P(vals), ctypes.c_int(best[1]))) if best[2] == "plan" else None
    run = (lambda: L.fast_spmv_plan_run_f32(plan, P(u), P(w), P(pres))) if plan else (lambda: L.fast_spmv_plus_times_f32(*args))
    times = []
    t_all = time.perf_counter()
    while len(times) < max_reps and (time.perf_counter() - t_all < min_seconds or len(times) < 3):
        t0 = time.perf_counter()
        run()
        times.append(time.perf_counter() - t0)
    if plan:
        L.fast_spmv_plan_free_f32(plan)
    info = dict(info, threads_used=int(best[1]), variant=best[2])
    return int(best[1]), info, times, w, pres


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, indptr, indices = cached_graph(args.scale)
    nnz = len(indices)
    vals, u = spmv_inputs(nnz, n)
    cpu_spmv(n, indptr, indices, vals, u, 0.0, max(args.warmup, 1))
    threads, info, times, w, pres = cpu_spmv(n, indptr, indices, vals, u, float("inf"), args.steps)      # exactly K timed passes
    times = times[:args.steps]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, w, pres)
    ms = 1e3 * float(np.median(times))
    value = nnz / (ms * 1e-3) / 1e9
    sample = f"{len(times)} full SpMV passes over the scale-{args.scale} graph ({nnz} edges each), median"
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
           "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": workload_config(args.scale, n, nnz),
           "note": "CPU OpenMP port of the reference path (SuiteSparse:GraphBLAS is not installable offline)",
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "host": info},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU fallback (use --impl reference for the CPU port)")
    os.environ.setdefault("B200GRB_DEVICE", str(local))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import pygraphblas_b200 as gb
    from pygraphblas_b200 import Matrix, Vector, FP32
    from pygraphblas_b200.distributed import Comm
    lib, ffi = gb.lib, gb.ffi
    sp_ = ffi.new("void**")
    lib.B200_get_stream(sp_)
    stream = torch.cuda.ExternalStream(int(ffi.cast("uintptr_t", sp_[0])), device=torch.device("cuda", local))
    ctx = {"torch": torch, "dist": dist, "gb": gb, "stream": stream, "world": world, "rank": rank, "args": args}

    # ---- graph (rank 0 builds the cache first, the others read it)
    if world > 1 and rank != 0:
        dist.barrier()
    n, indptr, indices = cached_graph(args.scale)
    if world > 1 and rank == 0:
        dist.barrier()
    nnz = len(indices)
    vals, u_host = spmv_inputs(nnz, n)
    if world == 1:
        r0, lrows, lnnz, ncols_l, newid = 0, n, nnz, n, None
        A = Matrix.from_csr(indptr, indices, vals, n, n, FP32)
        u = Vector.from_numpy(u_host)
    else:
        # 1-D row blocks of P A P' for a fixed pseudo-random relabelling P of the vertices: R-MAT puts its hubs at low ids, so
        # contiguous blocks of the ORIGINAL ids are either row-balanced or nnz-balanced, never both; blocks of the relabelled
        # ids have equal length (equal slices on the links) AND equal work.  Results are mapped back (x[newid]) for the check.
        from pygraphblas_b200.distributed import local_block_scattered, to_scattered
        newid, lb, lptr, lidx, lval = local_block_scattered(indptr, indices, vals, world, rank)
        r0, lrows, lnnz, ncols_l = rank * lb, lb, len(lidx), world * lb
        A = Matrix.from_csr(lptr, lidx, lval, lrows, ncols_l, FP32)
        u = Vector.from_numpy(to_scattered(u_host, newid, ncols_l))
    w = Vector.sparse(FP32, lrows)
    sr = FP32.PLUS_TIMES
    comm = Comm(ncols_l, FP32, rank, world) if world > 1 else None
    ctx["comm"] = comm

    def step():
        A.mxv(u, semiring=sr, out=w)
        if comm is not None:
            comm.allgather(w, r0)

    def sync_all():
        lib.B200_device_synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    sampler = ClockSampler(local)
    for _ in range(max(args.warmup, 3)):
        step()
    sync_all()
    sampler.start()
    launches0 = lib.B200_kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(args.steps):
        step()
    e1.record(stream)
    sync_all()
    launches = lib.B200_kernel_launches() - launches0
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs:
        # read back before the loops below run the same mxv again
        x_last, p_last = comm.allgather(w, r0).to_numpy() if comm is not None else w.to_numpy()
        if rank == 0:
            dump_outputs(args.dump_outputs, x_last if newid is None else x_last[newid], p_last if newid is None else p_last[newid])
    local_ms = ms_total / args.steps
    if world > 1:
        # the exchange's share of a step: a second pass of the same loop with events around each local SpMV (kept out of the
        # timed pass: at 8 GPUs a step is ~100 us and two event records per step are host time it cannot hide)
        ks = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for k in range(args.steps):
            ks[k][0].record(stream)
            A.mxv(u, semiring=sr, out=w)
            ks[k][1].record(stream)
            comm.allgather(w, r0)
        sync_all()
        local_ms = float(np.mean([a.elapsed_time(b) for a, b in ks]))
    # keep the device busy a little longer so that the clock sampler sees the kernels under load
    t_end = time.perf_counter() + 1.0
    while time.perf_counter() < t_end:
        for _ in range(20):
            A.mxv(u, semiring=sr, out=w)
        lib.B200_device_synchronize()
    clocks = sampler.stop()
    if world > 1:
        t = torch.tensor([ms_total, local_ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, local_ms = float(t[0].item()), float(t[1].item())
    ms = ms_total / args.steps
    value = nnz / (ms * 1e-3) / 1e9

    # ---- roofline of the dominant kernel from the SAME timed loop
    alg_bytes = lnnz * 8 + (lrows + 1) * 4 + ncols_l * 4 + lrows * 5
    peak, peak_src = measured_peaks()
    prof = profile_json("spmv_traffic.json")
    share = float(prof.get("dominant_kernel_share_of_step", 1.0))      # from the committed ncu launch list of this command
    kernel_ms = local_ms * share
    roofline = {"bound": "hbm", "kernel": prof.get("kernel", "spmv_run_hot2_kernel<float,float,PLUS,TIMES>"),
                "achieved": alg_bytes / (kernel_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": alg_bytes / (kernel_ms * 1e-3) / 1e9 / peak,
                "traffic": prof.get("dram_bytes_per_launch") if world == 1 else None,
                "algorithmic_bytes": int(alg_bytes), "kernel_ms": kernel_ms, "kernel_share_of_step": share,
                "step_ms_local_spmv": local_ms, "step_frac": alg_bytes / (local_ms * 1e-3) / 1e9 / peak,
                "how": "algorithmic bytes of the local SpMV / (CUDA-event time of the local SpMV in the timed loop x the dominant kernel's share of "
                       "that step in the committed ncu launch list, profiles/); step_frac charges the whole step (prep + kernel + fix-up) instead",
                "peak_source": peak_src}

    if args.quick:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "ms_per_step": ms, "roofline": roofline,
                              "gpu_launches": int(launches), "clocks": clocks, "quick": True}), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    config = workload_config(args.scale, n, nnz)
    config["parallelism"] = ("single GPU" if world == 1 else
                             f"1-D row blocks x{world} of the pseudo-randomly relabelled graph (equal rows and equal work per block); per step: local GrB_mxv + the library's all-gather of the output slices "
                             "(peer push over NVLink + flag wait, csrc/dist.cu; no NCCL on the data path)")
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
           "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": config, "roofline": roofline, "gpu_launches": int(launches), "clocks": clocks}
    if world > 1:
        out["exchange"] = {"ms_per_step": max(ms - local_ms, 0.0), "local_spmv_ms": local_ms, "split_from": "a second pass of the same loop with per-step events",
                           "bytes_pushed_per_rank": int(lrows * 5 * (world - 1)), "what": "push kernel (128-bit NVLink stores into every peer) + flag wait"}

    # ---- the result every rank now holds, checked on rank 0: presence bit-exact vs the CPU port, values vs fp64
    if comm is not None:
        x_rep, p_rep = comm.allgather(w, r0).to_numpy()
        x_rep, p_rep = x_rep[newid], p_rep[newid]              # back to the original vertex ids
    else:
        x_rep, p_rep = w.to_numpy()
    if rank == 0:
        import scipy.sparse as sp
        ref64 = sp.csr_matrix((vals.astype(np.float64), indices, indptr), shape=(n, n)) @ u_host.astype(np.float64)
        nonempty = np.diff(indptr) > 0
        rel = np.abs(x_rep[nonempty].astype(np.float64) - ref64[nonempty]) / np.abs(ref64[nonempty])
        out["max_rel_err_vs_fp64"] = float(rel.max())
        out["parity_tolerance"] = 1e-6
        pattern_ok = bool(np.array_equal(p_rep != 0, nonempty))
        out["parity_full_size"] = bool(pattern_ok and rel.max() <= 1e-6)
        out["parity_what"] = ("replicated result of the last timed step on rank 0: presence bit pattern == non-empty rows (and == the CPU port's), "
                              "values <= 1e-6 relative vs an fp64 scipy reference (N = 1 also: presence == the CPU port's, values within 2e-5 of its fp32 row-order sums)")

    # ---- end to end with host buffers through the mirror of the reference's API (the call a pygraphblas user makes)
    out["e2e"] = bench_e2e(ctx, A, ncols_l, lrows, nnz, u_host if world == 1 else u.to_numpy()[0], x_rep if world == 1 else None)

    if rank == 0 and world == 1:
        # ---- CPU baseline on the same workload (bounded sample)
        threads, info, times, w_cpu, p_cpu = cpu_spmv(n, indptr, indices, vals, u_host, args.cpu_seconds, 200)
        cpu_ms = 1e3 * float(np.median(times))
        out["cpu_baseline"] = {"value": nnz / (cpu_ms * 1e-3) / 1e9, "unit": UNIT, "cores": threads, "kind": "port", "host": info,
                               "sample": f"{len(times)} full SpMV passes over the same scale-{args.scale} graph (median), oracle/grb_fast.c OpenMP port"}
        ref64 = None
        port_rel = np.abs(x_rep[p_cpu != 0].astype(np.float64) - w_cpu[p_cpu != 0]) / np.abs(w_cpu[p_cpu != 0])
        out["max_rel_diff_vs_cpu_port"] = float(port_rel.max())      # the port sums in fp32 row order: it is the less accurate of the two
        out["parity_full_size"] = bool(out["parity_full_size"] and np.array_equal(p_rep, p_cpu) and port_rel.max() <= 2e-5)
    extras = []
    if not args.no_extras:
        if world == 1:
            extras = [("spgemm", bench_spgemm), ("spgemm_unmasked", bench_spgemm_unmasked), ("spgemm_unmasked_streamed", bench_spgemm_unmasked_streamed),
                      ("bfs", bench_bfs), ("sssp", bench_sssp)]
        else:
            extras = [("spgemm", bench_spgemm_panels), ("bfs", bench_bfs_dist), ("sssp", bench_sssp_dist)]
    for key, fn in extras:
        # the other configured workloads (BASELINE.json configs[3], [2], [4]); a failure there must not lose the headline line
        try:
            res = fn(ctx, n, indptr, indices)
        except Exception as e:                      # reported, not hidden
            res = {"error": f"{type(e).__name__}: {e}"[:300]}
        if rank == 0:
            out[key] = res
    if rank == 0:
        print(json.dumps(out), flush=True)
    if comm is not None:
        comm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bench_e2e(ctx, A_mirror, n, lrows, nnz, u_host, x_dev):
    """One step = u (pinned host) -> HBM, Matrix.mxv, w values + presence -> pinned host; A stays resident in HBM as it
    stays in the reference's process memory.  The mxv is the mirror's Matrix.mxv (the reference's matrix.py:2586-2726);
    the bulk dense import/export entry points stand in for the per-element setElement loop the reference would otherwise use."""
    torch, gb, args, world, rank = ctx["torch"], ctx["gb"], ctx["args"], ctx["world"], ctx["rank"]
    lib, ffi = gb.lib, gb.ffi
    from pygraphblas_b200 import Vector, FP32
    NB = 3                                                   # three steps in flight: step i+1's import, step i's kernels and step i-1's export overlap
    u_pin = [torch.empty(n, dtype=torch.float32).pin_memory().numpy() for _ in range(NB)]
    w_pin = [torch.empty(lrows, dtype=torch.float32).pin_memory().numpy() for _ in range(NB)]
    p_pin = [torch.empty(lrows, dtype=torch.uint8).pin_memory().numpy() for _ in range(NB)]
    for b in range(NB):
        u_pin[b][:] = u_host
    ue = [Vector.from_numpy(u_pin[b]) for b in range(NB)]
    we = [Vector.sparse(FP32, lrows) for _ in range(NB)]
    through = "pygraphblas_b200.Matrix.mxv (host-side mirror of the reference's method)"
    mxv = lambda b: A_mirror.mxv(ue[b], semiring=FP32.PLUS_TIMES, out=we[b])
    up = [ffi.cast("void*", x.ctypes.data) for x in u_pin]
    wp = [ffi.cast("void*", x.ctypes.data) for x in w_pin]
    pp = [ffi.cast("uint8_t*", x.ctypes.data) for x in p_pin]

    def serial_step():
        assert lib.B200_Vector_set_dense(ue[0]._vector[0], up[0], ffi.NULL, 0) == 0
        mxv(0)
        assert lib.B200_Vector_export_dense(we[0]._vector[0], wp[0], pp[0], 0) == 0          # returns with the data in host memory

    def pipelined_step(i):
        b = i % NB
        # where = 2: pinned host memory on the library's copy streams (GraphBLAS non-blocking mode): the import of THIS step runs
        # under the previous step's kernels, the export of this step under the next step's; every step still moves its own input
        # host -> HBM and its own result HBM -> host
        assert lib.B200_Vector_set_dense(ue[b]._vector[0], up[b], ffi.NULL, 2) == 0
        mxv(b)
        assert lib.B200_Vector_export_dense(we[b]._vector[0], wp[b], pp[b], 2) == 0
        if i >= 2:
            assert lib.GrB_Vector_wait(we[(i - 2) % NB]._vector) == 0                          # step i-2's result is now in host memory (its buffers are next)

    def timed(fn, steps):
        lib.B200_device_synchronize(); torch.cuda.synchronize()
        if world > 1:
            ctx["dist"].barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            fn(i)
        lib.B200_device_synchronize(); torch.cuda.synchronize()
        s_ = (time.perf_counter() - t0) / steps
        if world > 1:
            t = torch.tensor([s_], device="cuda")
            ctx["dist"].all_reduce(t, op=ctx["dist"].ReduceOp.MAX)
            s_ = float(t.item())
        return s_

    for i in range(3):
        serial_step()
    serial_s = timed(lambda i: serial_step(), args.steps)
    w_serial, p_serial = w_pin[0].copy(), p_pin[0].copy()
    for i in range(6):
        pipelined_step(i)
    e2e_s = timed(pipelined_step, args.steps)
    res = {"value": nnz / e2e_s / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(n * 4 * world), "d2h_bytes_per_step": int(sum_rows(ctx, lrows) * 5),
           "ms_per_step": e2e_s * 1e3, "through": through,
           "what": "per step: u (pinned host) -> HBM, Matrix.mxv, w values + presence -> pinned host; A resident in HBM; steps are independent requests, "
                   "triple-buffered so that step i+1's import and step i-1's export overlap step i's kernels (copy streams, where = 2)",
           "serial": {"value": nnz / serial_s / 1e9, "ms_per_step": serial_s * 1e3, "what": "the same step with blocking copies, one step at a time (latency-bound)"}}
    same = all(np.array_equal(w_pin[b][p_pin[b] != 0], w_serial[p_serial != 0]) and np.array_equal(p_pin[b], p_serial) for b in range(NB))
    res["pipelined_equals_serial"] = bool(same)
    if not same:                                     # reported, not hidden: which buffers differ, where and by how much
        diag = []
        for b in range(NB):
            dp = np.flatnonzero(p_pin[b] != p_serial)
            both = (p_pin[b] != 0) & (p_serial != 0)
            dv = np.flatnonzero(both & (w_pin[b] != w_serial))
            rel = np.abs(w_pin[b][dv].astype(np.float64) - w_serial[dv]) / np.maximum(np.abs(w_serial[dv].astype(np.float64)), 1e-30) if len(dv) else np.zeros(0)
            diag.append({"buffer": b, "presence_diffs": int(len(dp)), "value_diffs": int(len(dv)), "first_value_diffs": [int(x) for x in dv[:4]],
                         "max_rel_diff": float(rel.max()) if len(dv) else 0.0,
                         "zeros_where_serial_nonzero": int(np.count_nonzero(both & (w_pin[b] == 0) & (w_serial != 0)))})
        res["mismatch"] = diag
    if x_dev is not None:
        res["matches_device_result"] = bool(same and np.array_equal(w_serial[p_serial != 0], x_dev[p_serial != 0]))
    return res


def sum_rows(ctx, lrows):
    if ctx["world"] == 1:
        return lrows
    t = ctx["torch"].tensor([lrows], device="cuda")
    ctx["dist"].all_reduce(t)
    return int(t.item())


# ------------------------------------------------------------------ configs[3]: masked SpGEMM (triangle kernel)
def lower_triangle(scale):
    import scipy.sparse as sp
    n, indptr, indices = cached_graph(scale)
    S = sp.csr_matrix((np.ones(len(indices), np.int8), indices, indptr), shape=(n, n))
    Ls = sp.tril(S + S.T, -1).tocsr()
    Ls.sort_indices()
    return n, Ls.indptr.astype(np.int64), Ls.indices.astype(np.uint32)


def spgemm_alg_bytes(nnzA, flops, nnz_out, nrows, nnzM, bA, bB, bC):
    """SURVEY.md section 8(d), Gustavson model."""
    return nnzA * (4 + bA) + nnzA * 8 + flops * (4 + bB) + nnz_out * (4 + bC) + (nrows + 1) * 8 + nnzM * 4


def bench_spgemm(ctx, *_):
    """BASELINE.json configs[3]: scale-20 triangle-counting kernel C<L> = L (+.pair) L, 1 GPU."""
    torch, gb, args, stream = ctx["torch"], ctx["gb"], ctx["args"], ctx["stream"]
    from pygraphblas_b200 import Matrix, INT64, descriptor
    lib = gb.lib
    scale = args.spgemm_scale
    n, lp, lj = lower_triangle(scale)
    nnzL = len(lj)
    L = Matrix.from_csr(lp, lj, np.ones(nnzL, np.int64), n, n, INT64)
    C = None
    for _ in range(2):
        C = L.mxm(L, mask=L, semiring=INT64.PLUS_PAIR, desc=descriptor.S)
    lib.B200_device_synchronize()
    reps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = lib.B200_kernel_launches()
    e0.record(stream)
    for _ in range(reps):
        C = None
        C = L.mxm(L, mask=L, semiring=INT64.PLUS_PAIR, desc=descriptor.S)
    e1.record(stream)
    lib.B200_device_synchronize()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    flops, nout = gb.ffi.new("uint64_t*"), gb.ffi.new("uint64_t*")
    lib.B200_last_mxm_stats(flops, nout)
    Cp, Cj, Cx = C.to_csr()
    tri = int(Cx.sum())
    alg = spgemm_alg_bytes(nnzL, int(flops[0]), int(nout[0]), n, nnzL, 0, 0, 8)
    peak, _ = measured_peaks()
    prof = profile_json("spgemm_traffic.json")
    res = {"workload": f"R-MAT scale-{scale}: L = tril(A+A',-1), C<L> = L (+.pair) L, INT64 (BASELINE.json configs[3])",
           "value": int(nout[0]) / (ms * 1e-3) / 1e6, "unit": "Mnnz-out/s", "ms": ms, "nnz_L": nnzL, "products": int(flops[0]),
           "nnz_out": int(nout[0]), "triangles": tri, "gproducts_per_s": int(flops[0]) / (ms * 1e-3) / 1e9,
           "gpu_launches_per_call": int((lib.B200_kernel_launches() - l0) / reps),
           "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": alg / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes": int(alg), "traffic": prof.get("dram_bytes_per_call"),
                        "note": "pattern-only operands (b_A = b_B = 0), INT64 output; the flops x 4 B term is served by the L2 (operands fit), so DRAM traffic is far below it"}}
    # CPU port, one pass; parity on the FULL result: pattern and every value
    Lc = oracle_lib()
    budget, info = host_cpu_budget()
    Lc.fast_set_threads(ctypes.c_int(budget))
    cval = np.zeros(nnzL, np.int64)
    chas = np.zeros(nnzL, np.uint8)
    t0 = time.perf_counter()
    Lc.fast_masked_saxpy_plus_pair_i64(ctypes.c_int64(n), ctypes.c_int64(n), P(lp), P(lj), P(lp), P(lj), P(lp), P(lj), P(cval), P(chas))
    cpu_s = time.perf_counter() - t0
    res["cpu_baseline"] = {"value": int(chas.sum()) / cpu_s / 1e6, "unit": "Mnnz-out/s", "cores": budget, "kind": "port", "host": info,
                           "sample": "1 pass of the same masked SpGEMM (oracle/grb_fast.c masked Gustavson, OpenMP)"}
    keep = chas != 0
    rows = np.repeat(np.arange(n), np.diff(lp))
    ref_ptr = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(rows[keep], minlength=n), out=ref_ptr[1:])
    res["parity_full_size"] = bool(np.array_equal(Cp, ref_ptr) and np.array_equal(Cj, lj[keep]) and np.array_equal(Cx, cval[keep]))
    res["parity_what"] = "row pointers, column ids and every value of C against the CPU port"
    return res


def bench_spgemm_unmasked(ctx, *_):
    """Secondary of configs[3]: unmasked A.mxm(A, FP32.PLUS_SECOND) (the product configs[3] names, without the triangle mask)
    at the scale --spgemm-unmasked-scale; CPU baseline on a bounded sample of rows; parity on that sample (pattern + values)."""
    torch, gb, args, stream = ctx["torch"], ctx["gb"], ctx["args"], ctx["stream"]
    from pygraphblas_b200 import Matrix, FP32
    import scipy.sparse as sp
    lib = gb.lib
    scale = args.spgemm_unmasked_scale
    n, indptr, indices = cached_graph(scale)
    nnz = len(indices)
    rng = np.random.default_rng(5)
    vals = (rng.integers(1, 5, nnz) / 4.0).astype(np.float32)            # quarter-valued: sums are exact in fp32
    A = Matrix.from_csr(indptr, indices, vals, n, n, FP32)
    C = None
    times = []
    for rep in range(5):              # the first calls grow the memory pool to two result sets (old C is freed after the new one exists)
        C = None                      # the previous result goes back to the pool BEFORE the call: its 3.7 GB block is reused, not re-mapped
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        C = A.mxm(A, semiring=FP32.PLUS_SECOND)
        e1.record(stream)
        lib.B200_device_synchronize(); torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = float(np.median(times[2:]))
    flops, nout = gb.ffi.new("uint64_t*"), gb.ffi.new("uint64_t*")
    lib.B200_last_mxm_stats(flops, nout)
    alg = spgemm_alg_bytes(nnz, int(flops[0]), int(nout[0]), n, 0, 0, 4, 4)
    peak, _ = measured_peaks()
    res = {"workload": f"R-MAT scale-{scale}: C = A (+.second) A, FP32, unmasked (BASELINE.json configs[3] product without the mask)",
           "value": int(nout[0]) / (ms * 1e-3) / 1e6, "unit": "Mnnz-out/s", "ms": ms, "nnz_A": nnz, "products": int(flops[0]), "nnz_out": int(nout[0]),
           "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak,
                        "algorithmic_bytes": int(alg), "traffic": None}}
    # bounded CPU sample: the first rows that hold ~1/64 of the products (scipy, single thread: a third-party number for PLUS_TIMES-shaped work)
    S = sp.csr_matrix((vals, indices, indptr), shape=(n, n))
    rows = max(64, n // 256)
    Ssub = S[:rows]
    ones_like = sp.csr_matrix((np.ones(nnz, np.float32), indices, indptr), shape=(n, n))[:rows]
    t0 = time.perf_counter()
    R = (ones_like @ S).tocsr()                      # PLUS_SECOND: sum over k of B(k,j) = pattern(A) * B
    cpu_s = time.perf_counter() - t0
    R.sort_indices()
    Cp, Cj, Cx = C.to_csr()
    k1 = int(Cp[rows])
    res["cpu_baseline"] = {"value": R.nnz / cpu_s / 1e6, "unit": "Mnnz-out/s", "cores": 1, "kind": "port",
                           "sample": f"rows [0, {rows}) of the same product ({R.nnz} output entries) with scipy.sparse csr_matmat, 1 thread"}
    res["parity_full_size"] = bool(np.array_equal(Cp[:rows + 1], R.indptr) and np.array_equal(Cj[:k1], R.indices) and np.array_equal(Cx[:k1], R.data))
    res["parity_what"] = f"pattern and values of the first {rows} rows against scipy (exact: quarter-valued inputs)"
    del Ssub
    return res


def streamed_plan(n, indptr, indices, vals, cap):
    """Row panels of the streamed unmasked product: greedy cuts so that a panel holds at most `cap` products (at least one row),
    the total number of products, and the closed form of the sum of all values of C = A (+.second) A:
    sum_i sum_{k in A(i,:)} rowsum_A(k)  (fp64; exact for quarter-valued entries)."""
    rowlen = np.diff(indptr)
    rows = np.repeat(np.arange(n), rowlen)
    fl = np.bincount(rows, weights=rowlen[indices].astype(np.float64), minlength=n)          # products of row i
    cum = np.concatenate(([0.0], np.cumsum(fl)))
    cuts = [0]
    while cuts[-1] < n:
        r0 = cuts[-1]
        r1 = int(np.searchsorted(cum, cum[r0] + cap, side="right")) - 1
        cuts.append(min(n, max(r1, r0 + 1)))
    rowsum = np.bincount(rows, weights=np.asarray(vals, np.float64), minlength=n)
    return cuts, int(cum[-1]), float(rowsum[indices].sum())


def streamed_sample(n, indptr):
    """A strided sample of rows (R-MAT hubs sit at low ids: the stride mixes heavy and light rows): the row ids, the sample's
    row pointer and the positions of its entries in the parent CSR."""
    S = np.arange(min(7, n - 1), n, max(1, n // 1024))
    sp_ptr = np.concatenate(([0], np.cumsum(np.diff(indptr)[S]))).astype(np.int64)
    take = np.concatenate([np.arange(indptr[r], indptr[r + 1]) for r in S]).astype(np.int64)
    return S, sp_ptr, take


def bench_spgemm_unmasked_streamed(ctx, *_):
    """configs[3]'s product WITHOUT the mask at configs[3]'s own scale: A (+.second) A on R-MAT scale 20 makes ~2e10 products and
    ~9e9 output entries -- 72 GB as CSR and more entries than 32-bit offsets address -- so it is STREAMED as row panels
    C_g = A_g (+.second) A (A_g = a block of rows of A, blocks cut by products): each panel is formed by GrB_mxm (symbolic ->
    numeric), reduced on the device to (nvals, sum of values) and dropped before the next one.  Parity: the sum of all values of
    C against its closed form sum_i sum_{k in A(i,:)} rowsum_A(k) (exact: quarter-valued inputs, fp64 reductions), and pattern +
    values of a strided sample of rows against scipy."""
    torch, gb, args, stream = ctx["torch"], ctx["gb"], ctx["args"], ctx["stream"]
    from pygraphblas_b200 import Matrix, FP32
    import scipy.sparse as sp
    lib = gb.lib
    scale = args.spgemm_streamed_scale
    n, indptr, indices = cached_graph(scale)
    nnz = len(indices)
    rng = np.random.default_rng(5)
    vals = (rng.integers(1, 5, nnz) / 4.0).astype(np.float32)
    cap = float(args.spgemm_streamed_cap)
    cuts, total_products, expect = streamed_plan(n, indptr, indices, vals, cap)
    A = Matrix.from_csr(indptr, indices, vals, n, n, FP32)
    panels = []
    for g in range(len(cuts) - 1):
        r0, r1 = cuts[g], cuts[g + 1]
        k0, k1 = int(indptr[r0]), int(indptr[r1])
        panels.append(Matrix.from_csr((indptr[r0:r1 + 1] - k0).astype(np.int64), indices[k0:k1], vals[k0:k1], r1 - r0, n, FP32))

    def sweep():
        nv, total, prods = 0, 0.0, 0
        flops, nout = gb.ffi.new("uint64_t*"), gb.ffi.new("uint64_t*")
        for Ag in panels:
            C = Ag.mxm(A, semiring=FP32.PLUS_SECOND)
            lib.B200_last_mxm_stats(flops, nout)
            nv += int(C.nvals); prods += int(flops[0])
            total += float(C.reduce_float())                  # FP64 PLUS monoid: exact for these values
            C = None                                          # the panel goes back to the pool before the next one is formed
        return nv, total, prods

    sweep()                                                   # grows the memory pool to the largest panel
    lib.B200_device_synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    nout, total, prods = sweep()
    e1.record(stream)
    lib.B200_device_synchronize(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    alg = spgemm_alg_bytes(nnz, prods, nout, n, 0, 0, 4, 4)
    peak, _ = measured_peaks()
    res = {"workload": f"R-MAT scale-{scale}: C = A (+.second) A, FP32, unmasked, streamed as {len(panels)} row panels of <= {cap:.3g} products "
                       "(BASELINE.json configs[3] product without the mask, at configs[3]'s scale)",
           "value": nout / (ms * 1e-3) / 1e6, "unit": "Mnnz-out/s", "ms": ms, "panels": len(panels), "nnz_A": nnz, "products": prods, "nnz_out": nout,
           "gproducts_per_s": prods / (ms * 1e-3) / 1e9, "csr_bytes_of_C": int(nout) * 8,
           "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak,
                        "algorithmic_bytes": int(alg), "traffic": None},
           "timed": "per panel: GrB_mxm (flops, bins, symbolic, scan, numeric), nvals, GrB_Matrix_reduce_FP64; the panels' results are dropped, not kept"}
    # a strided sample of rows (hubs sit at low ids: the stride mixes heavy and light rows) against scipy, single thread
    S, sp_ptr, take = streamed_sample(n, indptr)
    As = Matrix.from_csr(sp_ptr, indices[take], vals[take], len(S), n, FP32)
    Cs = As.mxm(A, semiring=FP32.PLUS_SECOND)
    Cp, Cj, Cx = Cs.to_csr()
    full = sp.csr_matrix((vals, indices, indptr), shape=(n, n))
    ones_s = sp.csr_matrix((np.ones(len(take), np.float32), indices[take], sp_ptr), shape=(len(S), n))
    t0 = time.perf_counter()
    R = (ones_s @ full).tocsr()
    cpu_s = time.perf_counter() - t0
    R.sort_indices()
    res["cpu_baseline"] = {"value": R.nnz / cpu_s / 1e6, "unit": "Mnnz-out/s", "cores": 1, "kind": "port",
                           "sample": f"{len(S)} rows (every {max(1, n // 1024)}th) of the same product ({R.nnz} output entries) with scipy.sparse csr_matmat, 1 thread"}
    sample_ok = bool(np.array_equal(Cp, R.indptr) and np.array_equal(Cj, R.indices) and np.array_equal(Cx, R.data))
    res["sum_of_values"] = total; res["sum_of_values_closed_form"] = expect
    res["parity_full_size"] = bool(sample_ok and total == expect and prods == total_products)
    res["parity_what"] = (f"sum of all {nout} values of C == its closed form (exact), products == sum of row flops, and pattern + values of {len(S)} sampled rows against scipy")
    return res


def bench_spgemm_panels(ctx, *_):
    """SURVEY.md section 8(e), third form: C row panel g = L_g . L with L replicated, mask row-split with L; no collective on
    the data path, the per-panel nnz counts are all-gathered to form the global row pointer."""
    torch, dist, gb, args, stream, world, rank = ctx["torch"], ctx["dist"], ctx["gb"], ctx["args"], ctx["stream"], ctx["world"], ctx["rank"]
    from pygraphblas_b200 import Matrix, INT64, descriptor
    lib = gb.lib
    scale = args.spgemm_scale
    n, lp, lj = lower_triangle(scale)
    nnzL = len(lj)
    # panels balanced by products: flops(i) = sum over k in L(i,:) of nnz(L(k,:))
    rowlen = np.diff(lp)
    fl = np.add.reduceat(rowlen[lj].astype(np.int64), np.minimum(lp[:-1], nnzL - 1)) * (rowlen > 0)
    cum = np.concatenate(([0], np.cumsum(fl)))
    cuts = [int(np.searchsorted(cum, cum[-1] * g // world)) for g in range(world + 1)]
    cuts[0], cuts[-1] = 0, n
    r0, r1 = cuts[rank], cuts[rank + 1]
    k0, k1 = int(lp[r0]), int(lp[r1])
    Lg = Matrix.from_csr((lp[r0:r1 + 1] - k0).astype(np.int64), lj[k0:k1], np.ones(k1 - k0, np.int64), r1 - r0, n, INT64)
    Lfull = Matrix.from_csr(lp, lj, np.ones(nnzL, np.int64), n, n, INT64)
    C = None
    for _ in range(2):
        C = Lg.mxm(Lfull, mask=Lg, semiring=INT64.PLUS_PAIR, desc=descriptor.S)
    lib.B200_device_synchronize(); dist.barrier()
    reps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        C = Lg.mxm(Lfull, mask=Lg, semiring=INT64.PLUS_PAIR, desc=descriptor.S)
    e1.record(stream)
    lib.B200_device_synchronize(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    Cx = C.to_arrays()[2]
    stats = torch.tensor([int(C.nvals), int(Cx.sum())], device="cuda", dtype=torch.int64)
    per_panel = [torch.zeros_like(stats) for _ in range(world)]
    dist.all_gather(per_panel, stats)                     # "row-panel boundaries": the panels' nnz form the global row pointer
    nout = int(sum(int(p[0]) for p in per_panel)); tri = int(sum(int(p[1]) for p in per_panel))
    res = {"workload": f"R-MAT scale-{scale}: C<L> = L (+.pair) L split into {world} row panels by products, L replicated (SURVEY.md 8e)",
           "value": nout / (ms * 1e-3) / 1e6, "unit": "Mnnz-out/s", "ms": ms, "nnz_out": nout, "triangles": tri,
           "panel_nnz_out": [int(p[0]) for p in per_panel]}
    if rank == 0:
        import scipy.sparse as sp
        Ls = sp.csr_matrix((np.ones(nnzL, np.int64), lj, lp), shape=(n, n))
        ref = int((Ls @ Ls).multiply(Ls).sum()) if scale <= 18 else None
        cval = np.zeros(nnzL, np.int64); chas = np.zeros(nnzL, np.uint8)
        Lc = oracle_lib(); Lc.fast_set_threads(ctypes.c_int(host_cpu_budget()[0]))
        Lc.fast_masked_saxpy_plus_pair_i64(ctypes.c_int64(n), ctypes.c_int64(n), P(lp), P(lj), P(lp), P(lj), P(lp), P(lj), P(cval), P(chas))
        res["parity_full_size"] = bool(int(chas.sum()) == nout and int(cval.sum()) == tri and (ref is None or ref == tri))
        res["parity_what"] = "sum of the panels' nnz and of their values against the CPU port's full product"
    return res


# ------------------------------------------------------------------ configs[2]: BFS
def bench_bfs(ctx, n, indptr, indices):
    """BASELINE.json configs[2] shape on the bench graph: full BFS from the max-out-degree vertex,
    q<!visited, replace> = q' lor.land A per level (the hot path) + visited |= q; device time per level."""
    torch, gb, args, stream = ctx["torch"], ctx["gb"], ctx["args"], ctx["stream"]
    from pygraphblas_b200 import Matrix, Vector, BOOL, descriptor
    lib = gb.lib
    nnz = len(indices)
    A = Matrix.from_csr(indptr, indices, None, n, n, BOOL)
    I = Matrix.from_csr(np.arange(n + 1, dtype=np.int64), np.arange(n, dtype=np.uint32), None, n, n, BOOL)
    src = int(np.argmax(np.diff(indptr)))

    def bfs():
        q = Vector.sparse(BOOL, n); q[src] = True
        visited = Vector.sparse(BOOL, n); visited[src] = True
        level = np.full(n, -1, np.int32); level[src] = 0
        times, sizes, d = [], [], 0
        while True:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            q = q.vxm(A, mask=visited, desc=descriptor.RC, semiring=BOOL.LOR_LAND)
            e1.record(stream)
            nq = q.nvals
            lib.B200_device_synchronize(); torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1)); sizes.append(int(nq))
            if nq == 0:
                return level, times, sizes
            d += 1
            qi = q.to_arrays()[0]
            level[qi] = d
            I.mxv(q, out=visited, accum=BOOL.LOR, semiring=BOOL.LOR_LAND)

    bfs()                                       # builds the cached transpose
    level, times, sizes = bfs()
    # CPU port: same traversal with byte maps (oracle/grb_fast.c fast_bfs_step on the transposed graph)
    import scipy.sparse as sp
    Lc = oracle_lib()
    budget, info = host_cpu_budget()
    Lc.fast_set_threads(ctypes.c_int(budget))
    At = sp.csr_matrix((np.ones(nnz, np.int8), indices, indptr), shape=(n, n)).T.tocsr()
    tp, tc = At.indptr.astype(np.int64), At.indices.astype(np.uint32)
    front = np.zeros(n, np.uint8); front[src] = 1
    seen = front.copy()
    lev_cpu = np.full(n, -1, np.int32); lev_cpu[src] = 0
    d = 0
    t0 = time.perf_counter()
    while True:
        nxt = np.zeros(n, np.uint8)
        cnt = Lc.fast_bfs_step(ctypes.c_int64(n), P(tp), P(tc), P(front), P(seen), P(nxt))
        if cnt == 0:
            break
        d += 1
        lev_cpu[nxt != 0] = d
        seen |= nxt; front = nxt
    cpu_s = time.perf_counter() - t0
    return {"workload": f"R-MAT scale-{args.scale} BOOL pattern, full BFS from the max-out-degree vertex, LOR_LAND vxm with complemented mask + replace (BASELINE.json configs[2])",
            "ms_total": float(sum(times)), "ms_heaviest_step": float(max(times)), "levels": len(sizes) - 1, "reached": int((level >= 0).sum()),
            "step_ms": [round(t, 3) for t in times], "frontier_sizes": sizes,
            "value": nnz / (sum(times) * 1e-3) / 1e9, "unit": "GEdge/s (graph edges / whole-BFS device time)",
            "cpu_baseline": {"value": nnz / cpu_s / 1e9, "unit": "GEdge/s", "kind": "port", "cores": budget, "host": info,
                             "sample": "the same full BFS, oracle/grb_fast.c fast_bfs_step (OpenMP, byte maps, early exit)"},
            "parity_full_size": bool(np.array_equal(level, lev_cpu)), "parity_what": "the BFS level of every vertex against the CPU port"}


def bench_bfs_dist(ctx, n, indptr, indices):
    """configs[2] on N GPUs: the frontier step q<!visited, replace> = A' lor.land q as a row-split pull (rank r owns the rows of
    A' = the in-edges of its vertex block), ONE all-gather of the new frontier slices per level (values + presence bytes)."""
    torch, dist, gb, args, stream, world, rank, comm_f = ctx["torch"], ctx["dist"], ctx["gb"], ctx["args"], ctx["stream"], ctx["world"], ctx["rank"], None
    from pygraphblas_b200 import Matrix, Vector, BOOL, descriptor
    from pygraphblas_b200.distributed import Comm
    import scipy.sparse as sp
    lib = gb.lib
    nnz = len(indices)
    At = sp.csr_matrix((np.ones(nnz, np.int8), indices, indptr), shape=(n, n)).T.tocsr()
    At.sort_indices()
    gen = _generators()
    b = gen.row_block_bounds(At.indptr.astype(np.int64), world)
    b = [int(x) // 16 * 16 for x in b[:-1]] + [n]
    r0, r1 = b[rank], b[rank + 1]
    Al = At[r0:r1]
    A = Matrix.from_csr(Al.indptr.astype(np.int64), Al.indices.astype(np.uint32), None, r1 - r0, n, BOOL)
    src = int(np.argmax(np.diff(indptr)))
    comm = Comm(n, BOOL, rank, world)

    def bfs():
        qfull = Vector.sparse(BOOL, n); qfull[src] = True
        vis = np.zeros(r1 - r0, np.uint8)
        if r0 <= src < r1:
            vis[src - r0] = 1
        visited = Vector.from_numpy(vis.astype(np.bool_), present=vis)
        level = np.full(n, -1, np.int32); level[src] = 0
        times, d = [], 0
        while True:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ql = A.mxv(qfull, mask=visited, desc=descriptor.RC, semiring=BOOL.LOR_LAND)          # new frontier among my vertices
            qfull = comm.allgather(ql, r0)
            e1.record(stream)
            nq = qfull.nvals
            lib.B200_device_synchronize(); torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
            if nq == 0:
                return level, times
            d += 1
            level[qfull.to_arrays()[0]] = d
            visited = visited.eadd(ql, BOOL.LOR)
            qfull = qfull.dup()                              # the view is only valid until the next collective

    bfs()
    level, times = bfs()
    t = torch.tensor([float(sum(times))], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    res = {"workload": f"R-MAT scale-{args.scale} BOOL, full BFS, row-split pull over {world} GPUs, one library all-gather of the frontier per level (BASELINE.json configs[2])",
           "ms_total": ms_total, "levels": len(times) - 1, "reached": int((level >= 0).sum()), "value": nnz / (ms_total * 1e-3) / 1e9,
           "unit": "GEdge/s (graph edges / whole-BFS device time)"}
    if rank == 0:
        from scipy.sparse.csgraph import breadth_first_order
        S = sp.csr_matrix((np.ones(nnz, np.int8), indices, indptr), shape=(n, n))
        order, pred = breadth_first_order(S, src, directed=True, return_predecessors=True)
        lev = np.full(n, -1, np.int32); lev[src] = 0
        for v in order[1:]:
            lev[v] = lev[pred[v]] + 1
        res["parity_full_size"] = bool(np.array_equal(level, lev)); res["parity_what"] = "the BFS level of every vertex against scipy.sparse.csgraph"
    comm.close()
    return res


# ------------------------------------------------------------------ configs[4]: SSSP sweeps
def sssp_inputs(n, indptr, indices):
    rng = np.random.default_rng(3)
    wts = (np.float32(1.0) - rng.random(len(indices), dtype=np.float32)).astype(np.float32)
    return wts, int(np.argmax(np.diff(indptr)))


def cpu_sssp(n, indptr, indices, wts, src, sweeps):
    import scipy.sparse as sp
    Lc = oracle_lib()
    budget, info = host_cpu_budget()
    Lc.fast_set_threads(ctypes.c_int(budget))
    At = sp.csr_matrix((wts, indices, indptr), shape=(n, n)).T.tocsr(); At.sort_indices()
    tp, tc, tv = At.indptr.astype(np.int64), At.indices.astype(np.uint32), At.data.astype(np.float32)
    d = np.full(n, np.inf, np.float32); d[src] = 0
    t0 = time.perf_counter()
    for _ in range(sweeps):
        uu = d.copy()
        Lc.fast_spmv_min_plus_f32_accum(ctypes.c_int64(n), P(tp), P(tc), P(tv), P(uu), P(d))
    return d, (time.perf_counter() - t0) / sweeps, budget, info


def bench_sssp(ctx, n, indptr, indices):
    """BASELINE.json configs[4] shape on the bench graph (scale 22 here; tools/sssp_bench.py runs scale 24):
    16 sweeps of v = min(v, A' min.+ v), FP32 weights U(0,1], dense v, T0."""
    torch, gb, args, stream = ctx["torch"], ctx["gb"], ctx["args"], ctx["stream"]
    from pygraphblas_b200 import Matrix, Vector, FP32, descriptor
    lib = gb.lib
    nnz = len(indices)
    wts, src = sssp_inputs(n, indptr, indices)
    A = Matrix.from_csr(indptr, indices, wts, n, n, FP32)

    def fresh():
        d0 = np.full(n, np.inf, np.float32); d0[src] = 0
        return Vector.from_numpy(d0)

    def sweep(v):
        A.mxv(v, out=v, accum=FP32.MIN, semiring=FP32.MIN_PLUS, desc=descriptor.T0)

    v = fresh(); sweep(v); sweep(v); lib.B200_device_synchronize()
    v = fresh()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(16):
        sweep(v)
    e1.record(stream)
    lib.B200_device_synchronize(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 16
    d16 = v.to_numpy()[0]
    d, cpu_s, budget, info = cpu_sssp(n, indptr, indices, wts, src, 16)
    alg = nnz * 8 + (n + 1) * 4 + n * 4 * 3
    peak, _ = measured_peaks()
    return {"workload": f"R-MAT scale-{args.scale} FP32 weights, 16 Bellman-Ford sweeps v = min(v, A' min.+ v), dense v, T0 (BASELINE.json configs[4] shape)",
            "ms_per_sweep": ms, "value": nnz / (ms * 1e-3) / 1e9, "unit": "GEdge/s",
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes": int(alg)},
            "cpu_baseline": {"value": nnz / cpu_s / 1e9, "unit": "GEdge/s", "kind": "port", "cores": budget, "host": info,
                             "sample": "the same 16 sweeps, oracle/grb_fast.c OpenMP port"},
            "parity_full_size": bool(np.array_equal(d, d16)), "parity_what": "every distance after 16 sweeps, bit-exact against the CPU port"}


def bench_sssp_dist(ctx, n, indptr, indices):
    """configs[4] on N GPUs, the all-reduce form of SURVEY.md 8(e): A row-split, the sweep uses A' (INP0 = TRAN), so every rank
    folds its rows' contributions into a full-length partial and the library all-reduces the partials with MIN over peer
    memory (rank order); then v = min(v, result) on every rank."""
    torch, dist, gb, args, stream, world, rank = ctx["torch"], ctx["dist"], ctx["gb"], ctx["args"], ctx["stream"], ctx["world"], ctx["rank"]
    from pygraphblas_b200 import Matrix, Vector, FP32, descriptor
    from pygraphblas_b200.distributed import Comm
    lib = gb.lib
    nnz = len(indices)
    wts, src = sssp_inputs(n, indptr, indices)
    gen = _generators()
    b = gen.row_block_bounds(indptr, world)
    b = [int(x) // 16 * 16 for x in b[:-1]] + [n]
    r0, r1 = b[rank], b[rank + 1]
    k0, k1 = int(indptr[r0]), int(indptr[r1])
    A = Matrix.from_csr((indptr[r0:r1 + 1] - k0).astype(np.int64), indices[k0:k1], wts[k0:k1], r1 - r0, n, FP32)
    comm = Comm(n, FP32, rank, world)
    d0 = np.full(n, np.inf, np.float32); d0[src] = 0

    def run(sweeps):
        v = Vector.from_numpy(d0)
        for _ in range(sweeps):
            mine = v[r0:r1 - 1]                                 # my block of the replicated vector (device-side extract, inclusive stop)
            part = A.mxv(mine, semiring=FP32.MIN_PLUS, desc=descriptor.T0)      # full-length partial from my rows
            red = comm.allreduce(part, FP32.MIN_MONOID)
            v = v.eadd(red, FP32.MIN)
        return v

    run(2); lib.B200_device_synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    v = run(16)
    e1.record(stream)
    lib.B200_device_synchronize(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 16], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    res = {"workload": f"R-MAT scale-{args.scale} FP32, 16 sweeps v = min(v, A' min.+ v) on {world} GPUs: row-split A, T0, library all-reduce (MIN, rank order) of the partials (configs[4] shape)",
           "ms_per_sweep": ms, "value": nnz / (ms * 1e-3) / 1e9, "unit": "GEdge/s"}
    if rank == 0:
        d, _, _, _ = cpu_sssp(n, indptr, indices, wts, src, 16)
        res["parity_full_size"] = bool(np.array_equal(d, v.to_numpy()[0])); res["parity_what"] = "every distance after 16 sweeps, bit-exact against the CPU port"
    comm.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=int, default=22)
    ap.add_argument("--spgemm-scale", type=int, default=20)
    ap.add_argument("--spgemm-unmasked-scale", type=int, default=17)
    ap.add_argument("--spgemm-streamed-scale", type=int, default=20)
    ap.add_argument("--spgemm-streamed-cap", type=float, default=1.5e9, help="products per row panel of the streamed unmasked SpGEMM")
    ap.add_argument("--no-extras", "--no-spgemm", dest="no_extras", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--quick", action="store_true", help="timed SpMV loop only (for ncu): no e2e / CPU baseline / extras")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of the last timed step to DIR/*.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
