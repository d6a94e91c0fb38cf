#!/usr/bin/env python
"""Per-kernel times of bench.py's SpMV step (one in-place FP32 PLUS_TIMES GrB_mxv of the R-MAT graph) under torch.profiler.
    python tools/prof_spmv_step.py OUT_DIR [scale] [steps]
Writes OUT_DIR/launches_spmv_step.csv (step, kernel, grid, block, start relative to the step's first kernel, duration; ns, in launch
order) and prints, per kernel, the median duration, the median time by which it extends the step past the end of the kernel before
it, and the median share of the step's span (first start to last end) it is running.  The kernels of a step are launched with
programmatic dependent launch, so a kernel can start (and wait) before the one ahead of it ends: its duration then includes that
wait, and the time it adds to the step is what its end adds.  Run it on its own: tracing slows the host, not the kernels."""
import csv, json, os, sys, tempfile
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from torch.profiler import profile, ProfilerActivity
import pygraphblas_b200 as gb
from pygraphblas_b200 import Matrix, Vector, FP32
from bench import cached_graph, spmv_inputs

out_dir = sys.argv[1]
scale = int(sys.argv[2]) if len(sys.argv) > 2 else 22
steps = int(sys.argv[3]) if len(sys.argv) > 3 else 20
os.makedirs(out_dir, exist_ok=True)
n, indptr, indices = cached_graph(scale)
vals, u_host = spmv_inputs(len(indices), n)
A = Matrix.from_csr(indptr, indices, vals, n, n, FP32)
u, w = Vector.from_numpy(u_host), Vector.sparse(FP32, n)
for _ in range(10):
    A.mxv(u, semiring=FP32.PLUS_TIMES, out=w)
gb.lib.B200_device_synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(steps):
        A.mxv(u, semiring=FP32.PLUS_TIMES, out=w)
    gb.lib.B200_device_synchronize()
with tempfile.TemporaryDirectory() as tmp:
    trace = os.path.join(tmp, "t.pt.trace.json")
    prof.export_chrome_trace(trace)
    events = json.load(open(trace))["traceEvents"]
kernels = sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])
per_step = len(kernels) // steps
assert per_step * steps == len(kernels), (len(kernels), steps)
rows = []
for i, e in enumerate(kernels):
    a = e.get("args", {})
    t0 = kernels[i - i % per_step]["ts"]
    rows.append([i // per_step, e["name"], str(a.get("grid", "")), str(a.get("block", "")), int(round((e["ts"] - t0) * 1e3)),
                 int(round(e["dur"] * 1e3))])
with open(os.path.join(out_dir, "launches_spmv_step.csv"), "w", newline="") as f:
    wr = csv.writer(f)
    wr.writerow(["step", "kernel", "grid", "block", "start_ns", "duration_ns"])
    wr.writerows(rows)
span = [max(r[4] + r[5] for r in rows if r[0] == s) for s in range(steps)]
summary = {"scale": scale, "steps": steps, "kernels_per_step": per_step, "step_span_ns_median": float(np.median(span)), "kernels": []}
for k in range(per_step):
    mine = [rows[s * per_step + k] for s in range(steps)]
    adds = [r[4] + r[5] - (rows[r[0] * per_step + k - 1][4] + rows[r[0] * per_step + k - 1][5] if k else 0) for r in mine]
    summary["kernels"].append({"kernel": mine[0][1], "median_duration_ns": float(np.median([r[5] for r in mine])),
                               "median_adds_to_step_ns": float(np.median(adds)),
                               "median_share_of_step": float(np.median([r[5] / span[r[0]] for r in mine]))})
print(json.dumps(summary, indent=1))
json.dump(summary, open(os.path.join(out_dir, "launches_spmv_step_summary.json"), "w"), indent=1)
