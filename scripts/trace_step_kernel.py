"""Where the time of a k_step_tma launch goes: block 0's time stamps (bl_step_trace_*) over one forward + adjoint
of a lockstep batch of TRACE_PROBES runs (default 4) of the headline workload (n = 1M, depth 100, fp32), summarised
per phase."""
import ctypes as C
import json
import sys

import numpy as np

sys.path.insert(0, ".")
import experiments_lanczos_adjoints_b200 as bl
from experiments_lanczos_adjoints_b200 import _lib, plan as bl_plan, synthetic
import bench

row, col, data, dalpha, dbeta = bench.build_workload()
n, K, dtype = bench.N_ROWS, bench.DEPTH, np.float32
import os

P = int(os.environ.get("TRACE_PROBES", 4))  # runs of the lockstep batch (BatchedTridiagAdjointPlan)
if P < 2:
    sys.exit(f"TRACE_PROBES={P}: k_step_tma runs for lockstep batches of two or more runs only")
op = bl.operators.SparseOperator(row, col, (n, n))
pl = bl_plan.BatchedTridiagAdjointPlan(op, K, dtype, P)
pl.set_vectors(np.random.default_rng(0).standard_normal((P, n)).astype(dtype))
pl.set_params(data.astype(dtype))
pl.set_cotangents(np.stack([synthetic.slq_cotangent_dH(dalpha, dbeta, dtype)] * P))
for _ in range(3):
    pl.run()
bl.synchronize()
_lib.call("bl_step_trace_begin")
pl.run()
stamps = np.zeros((2048, 8), dtype=np.uint64)
count, pdl = C.c_int64(0), C.c_int(0)
_lib.call("bl_step_trace_end", stamps.ctypes.data, 2048, C.byref(count), C.byref(pdl))
st = stamps[: count.value].astype(np.float64)
sm_count = C.c_int(0)
clk_ghz = float(sys.argv[1]) if len(sys.argv) > 1 else 1.9  # SM clock under load (GHz), see bench clocks
d = np.diff(st[:, 1:], axis=1) / clk_ghz / 1e3  # us
names = ["phase0 loads", "phase0 reduce+epilogue", "phase1 stream", "phase1 reduce+epilogue", "phase2 stream", "exit sum"]
gap = np.diff(st[:, 0]) / 1e3  # us between consecutive kernel entries
total = (st[:, 7] - st[:, 1]) / clk_ghz / 1e3
out = {"probes": P, "launches": int(count.value), "pdl_accepted": int(pdl.value), "sm_clock_ghz_assumed": clk_ghz,
       "phases_us_mean": {nm: float(d[:, i].mean()) for i, nm in enumerate(names)},
       "phases_us_first_step": {nm: float(d[0, i]) for i, nm in enumerate(names)},
       "phases_us_step_50": {nm: float(d[50, i]) for i, nm in enumerate(names)},
       "phases_us_step_99": {nm: float(d[99, i]) for i, nm in enumerate(names)},
       "kernel_body_us_mean": float(total.mean()), "entry_to_entry_us_mean": float(gap.mean()),
       "entry_to_entry_us_fwd": [float(x) for x in gap[:99:10]], "body_us_fwd": [float(x) for x in total[:100:10]]}
print(json.dumps(out, indent=1))
