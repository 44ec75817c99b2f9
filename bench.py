#!/usr/bin/env python
"""Benchmark of the hot path: Lanczos (full re-orthogonalisation) forward + adjoint.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): sparse SPD operator, n = 1M rows, 11 entries per row
(COO layout of `suite_sparse_load`), Krylov depth 100, fp32, cotangents on the tridiagonal
coefficients (the SLQ case).  One forward + one adjoint sweep of one probe = 100 Krylov steps; the
metric is Krylov steps per second, `depth / (t_fwd + t_adj)`.

One bench "step" = the forward + adjoint of `lanes x probes` independent probe vectors per GPU (default
2 x 4): the probes of a lane advance in lockstep (`plan.BatchedTridiagAdjointPlan`: ONE launch per Krylov step
for the whole batch -- the multi-vector operator call and the Gram-Schmidt step, `k_step_tma`), the lanes run on
separate streams so that one batch's kernels fill the other's grid-wide reductions.  This is the product path of the SLQ /
Hutchinson estimator (`lanczos.probe_lockstep_sum`).  `config.single_probe` is ONE run alone.

N > 1 (launched by torchrun, one rank per GPU; the ranks meet over the library's own socket rendezvous and
NCCL, no torch): every rank runs its own probes on a replicated operator (probe sharding, SURVEY 8e); the
parameter cotangent accumulates on the device over the steps, as it does over the probes of an estimate, and
the timed region ends with ONE `ncclAllReduce` of it (hutchinson.py:54 over GPUs); weak scaling.

`--impl reference`: the reference's algorithm on the host CPUs (the NumPy/SciPy oracle port --
JAX is not installed in this image, so the reference itself cannot run), bounded sample.

`--dump-outputs DIR`: after the timed steps, rank 0 writes what they computed as `DIR/<name>.npy` in the run's
dtype (`dump_outputs`): `H` (lanes, probes, K, K) of the last forward, `dv` (lanes, probes, n) of the last adjoint
and `dparams` (nnz), the parameter cotangent summed over the probes, the lanes and the timed steps.  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ROWS = int(os.environ.get("BL_BENCH_N", 1_000_000))
DEPTH = int(os.environ.get("BL_BENCH_DEPTH", 100))
BANDS = 5
METRIC = "Lanczos fwd+adjoint steps/sec at n=1M, K=100; achieved HBM GB/s vs peak"
UNIT = "krylov_steps/s"


# DRAM traffic of the dominant kernel from `ncu --set full` captures: dram__bytes_read.sum + dram__bytes_write.sum
# of ONE launch, next to that launch's algorithmic bytes; each entry names the launch and the summary it comes from.
NCU_TRAFFIC = {"k_step_tma": {"traffic": 3103.660e6 + 26.833e6, "algorithmic": 4 * (3 + 100 + 98) * 4.0e6 + 82.6e6 + 48.0e6,
                              "launch": "forward step i=95 of a lockstep batch of 4 runs, operator call inside the launch (phase S: "
                                        "SELL operand 82.6 MB once + x, y, q per run; per run: phase 0 three vectors, phase 1 "
                                        "96 rows + 3 terms + out, phase 2 96 rows + v' + out), fp32, n=1M; 608.3 us = 5.50 TB/s",
                              "source": "profiles/r2d_lockstep_prof_step.md"},
               "k_xdots_tma": {"traffic": 396.5e6 + 11.7e6, "algorithmic": 100 * 4.0e6,
                               "launch": "forward pass B, i=95 (96 streamed rows + 3 terms + out), fp32, n=1M",
                               "source": "profiles/r1c_prof_xdots.md"},
               "k_fused_tma": {"traffic": 395.3e6 + 6.8e6, "algorithmic": 98 * 4.0e6,
                               "launch": "forward pass B, i=95 (96 resident rows), fp32, n=1M (before k_xdots_tma)",
                               "source": "profiles/r1b_prof_sym_fused.md"}}


def algorithmic_bytes(n, nnz, K, w):
    """SURVEY 8(d): compulsory traffic with the best legal fusion, active columns only."""
    fwd = 3 * n * w * K * (K + 1) / 2 + K * (nnz * (w + 4) + 4 * (n + 1)) + 8 * K * n * w
    adj = 3 * n * w * K * (K + 1) + K * (nnz * (3 * w + 4) + 4 * (n + 1)) + 10 * K * n * w
    return fwd, adj


DUMP_SAMPLE = 1 << 21  # elements kept of a larger output: three outputs stay under 64 MB even in fp64


def dump_outputs(directory, arrays, seed=0):
    """Write each array as `directory/<name>.npy`.  An array of more than DUMP_SAMPLE elements is written as its
    elements at DUMP_SAMPLE flat indices drawn from `seed` (ascending), the same indices on every run."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(seed).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a))


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (NVML; nvidia-smi fallback)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self._nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None

    def _sample(self):
        nv = self._nvml
        if nv is None:
            return
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
            names = {
                "hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap,
            }
            for name, bit in names.items():
                if mask & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while not self._stop_evt.is_set():
            self._sample()
            self._stop_evt.wait(0.05)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "source": "unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples), "source": "nvml"}  # fmt: skip


def build_workload(seed=0):
    from experiments_lanczos_adjoints_b200 import synthetic

    row, col, data = synthetic.banded_spd_coo(N_ROWS, bands=BANDS, seed=seed)
    rng = np.random.default_rng(seed + 1)
    dalpha, dbeta = rng.standard_normal(DEPTH), rng.standard_normal(DEPTH - 1)
    return row, col, data, dalpha, dbeta


# ---------------------------------------------------------------------------------------------
def cpu_reference_run(row, col, data, dalpha, dbeta, depth, dtype, seed=0):
    """One forward + adjoint of the reference's algorithm (oracle port) on the host CPUs: `lanczos.tridiag(reortho=
    "full")` and its VJP for cotangents on (alpha, beta), restricted to the columns that are non-zero at each step
    (`oracle.krylov.tridiag_full_active`: the reference's arithmetic without the identically-zero terms XLA would
    also stream -- optimistic for the CPU)."""
    from oracle import krylov, operators

    n = N_ROWS
    op = operators.CsrFastOperator(row, col, (n, n))
    v = np.random.default_rng(seed + 7).standard_normal(n).astype(dtype)
    t0 = time.perf_counter()
    _out, pull = krylov.tridiag_full_active(op, depth, v, data.astype(dtype))
    pull(((None, (dalpha[:depth].astype(dtype), dbeta[: depth - 1].astype(dtype))), (None, None)))
    return time.perf_counter() - t0


def cpu_baseline(row, col, data, dalpha, dbeta, sample_depth=40):
    cores = os.cpu_count() or 1
    t = cpu_reference_run(row, col, data, dalpha, dbeta, sample_depth, np.float32)
    return {
        "value": sample_depth / t, "unit": UNIT, "cores": cores, "kind": "port",
        "sample": f"n={N_ROWS}, nnz={len(data)}, fp32, one forward+adjoint at Krylov depth {sample_depth} "
                  f"({t:.1f} s; cost per Krylov step grows with depth, so depth {DEPTH} is slower per step -- "
                  "`bench.py --impl reference` times the full depth); NumPy/SciPy oracle port over the active "
                  "columns, BLAS threads = all cores (JAX not installed: the reference itself cannot run)",
    }  # fmt: skip


def run_reference(args):
    """The reference arm: the same workload at the SAME depth on the host cores.  One step (forward + adjoint at
    depth 100) takes the better part of a minute, so the arm times as many of the requested steps as fit a budget
    (BL_REF_BUDGET_S, default 150 s; at least one) and says how many it timed."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    row, col, data, dalpha, dbeta = build_workload()
    depth = int(os.environ.get("BL_REF_DEPTH", DEPTH))
    budget = float(os.environ.get("BL_REF_BUDGET_S", 150))
    t_start = time.perf_counter()
    times = []
    while len(times) < max(1, args.steps) and (not times or time.perf_counter() - t_start + times[-1] < budget):
        times.append(cpu_reference_run(row, col, data, dalpha, dbeta, depth, np.float32))
    t = float(np.mean(times))
    value = depth / t
    cores = os.cpu_count() or 1
    sampled = "" if depth == DEPTH else f" -- a depth-{depth} SAMPLE of the depth-{DEPTH} workload"
    sample = (f"{len(times)} timed step(s) of {args.steps} requested (budget {budget:.0f} s, no warm-up: a step takes "
              f"{t:.0f} s); each step = one forward+adjoint at Krylov depth {depth}{sampled} on n={N_ROWS}, "
              f"nnz={len(data)}, fp32; NumPy/SciPy oracle port of the reference algorithm over the active columns "
              "(JAX is not installed, the reference itself cannot be imported)")  # fmt: skip
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "steps_timed": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * t,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"sparse SPD COO operator n={N_ROWS} nnz={len(data)} ({2 * BANDS + 1}/row), Lanczos full "
                               f"reortho depth {depth}{sampled}, forward + adjoint (cotangents on alpha/beta)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))  # fmt: skip


# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--probes", type=int, default=int(os.environ.get("BL_BENCH_PROBES", 4)),
                    help="probe vectors per lockstep batch (mode lockstep) / per GPU on separate streams (mode streams)")
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("BL_BENCH_LANES", 2)),
                    help="lockstep batches in flight per GPU, each on its own stream")
    ap.add_argument("--mode", default=os.environ.get("BL_BENCH_MODE", "lockstep"), choices=["lockstep", "streams"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the other BASELINE configurations (`extra`)")
    ap.add_argument("--quick", action="store_true", help="device-timed steps only (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference keeps none")
        return run_reference(args)

    # stdout carries exactly ONE line, the JSON: whatever libraries print on file descriptor 1 while the
    # benchmark runs (NCCL's version banner, for one) goes to stderr; the descriptor is restored for the result
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

    import experiments_lanczos_adjoints_b200 as bl
    from experiments_lanczos_adjoints_b200 import comm as bl_comm
    from experiments_lanczos_adjoints_b200 import device as bl_dev
    from experiments_lanczos_adjoints_b200 import plan as bl_plan
    from experiments_lanczos_adjoints_b200 import synthetic

    group = bl_comm.init_from_env()  # socket rendezvous from RANK / WORLD_SIZE / MASTER_*; binds the GPU of LOCAL_RANK
    rank, world, local_rank = group.rank, group.world, group.local_rank
    dtype = np.float32 if args.dtype == "f32" else np.float64
    w = np.dtype(dtype).itemsize
    code = bl_dev.dtype_code(dtype)
    row, col, data, dalpha, dbeta = build_workload()
    nnz = len(data)
    lockstep = args.mode == "lockstep"
    P = max(1, args.probes)
    L = max(1, args.lanes) if lockstep else P
    per_lane = P if lockstep else 1
    probes_per_gpu = L * per_lane
    # several runs / batches in flight: one block per SM and kernel, so that kernels of different lanes share an SM
    # and fill each other's ramps and grid-wide reductions; a lane alone wants two
    blocks_in_flight = 0
    if "BL_BLOCKS_PER_SM" not in os.environ and ((lockstep and L >= 2) or (not lockstep and L >= 3)):
        blocks_in_flight = 1
    bl.set_blocks_per_sm(blocks_in_flight)
    plans = []
    for _lane in range(L):
        op = bl.operators.SparseOperator(row, col, (N_ROWS, N_ROWS))
        if lockstep:
            plans.append(bl_plan.BatchedTridiagAdjointPlan(op, DEPTH, dtype, P, stream=bl_dev.Stream()))
        else:
            plans.append(bl_plan.TridiagAdjointPlan(op, DEPTH, dtype, stream=bl_dev.Stream()))

    # pinned host buffers for the end-to-end path
    p_host = bl_plan.pinned_empty((nnz,), dtype)
    p_host[:] = data
    dH1 = synthetic.slq_cotangent_dH(dalpha, dbeta, dtype)
    dH_host = bl_plan.pinned_empty((per_lane, DEPTH, DEPTH) if lockstep else (DEPTH, DEPTH), dtype)
    dH_host[...] = dH1
    v_hosts, outs = [], []
    for li, pl in enumerate(plans):
        v_host = bl_plan.pinned_empty((per_lane, N_ROWS) if lockstep else (N_ROWS,), dtype)
        for b in range(per_lane):
            vec = np.random.default_rng(100 + (rank * L + li) * per_lane + b).standard_normal(N_ROWS)
            if lockstep:
                v_host[b] = vec
            else:
                v_host[:] = vec
        v_hosts.append(v_host)
        outs.append((bl_plan.pinned_empty(dH_host.shape, dtype), bl_plan.pinned_empty(v_host.shape, dtype),
                     [bl_plan.pinned_empty((nnz,), dtype)]))  # fmt: skip
        (pl.set_vectors if lockstep else pl.set_vector)(v_host)
        pl.set_params(p_host)
        (pl.set_cotangents if lockstep else pl.set_cotangent)(dH_host)
    main_stream = bl_dev.default_stream()
    grad_total = bl_dev.DeviceArray((nnz,), dtype)

    # Lanes half a cycle apart: every second lane runs [adjoint of its previous forward, next forward] while its
    # neighbour runs [forward, adjoint] -- one sweep with many active rows (bandwidth-bound) is then always in flight
    # beside one with few (bound by its grid-wide reductions), instead of both lanes being short of rows together.
    # Every step still is one forward + one adjoint of every probe batch.  BL_BENCH_STAGGER=1 switches it on; off by default:
    # measured +1.1 % on one box and -0.3 % on another, and a step whose lanes all run [forward, adjoint] is simpler to read.
    stagger = lockstep and L >= 2 and os.environ.get("BL_BENCH_STAGGER", "0") == "1"
    behind = [stagger and li % 2 == 1 for li in range(L)]
    for pl, late in zip(plans, behind):
        if late:
            pl.forward()  # primes the pipeline: the lane's first step starts with this forward's adjoint

    def step_device(active=None, first=False):
        """Forward + adjoint of every probe.  The parameter cotangent ACCUMULATES inside each lane's operator
        (zeroed on the first step only), as it does over the probes of an estimate (`lanczos.probe_lockstep_sum`)."""
        for pl in active or plans:
            if behind[plans.index(pl)]:
                pl.adjoint(zero=first, export=False)
                pl.forward()
            else:
                pl.forward()
                pl.adjoint(zero=first, export=False)

    def finish_estimate(active=None):
        """Close the estimate: export each lane's accumulated cotangent, add the lanes up, and -- probe sharding --
        ONE ncclAllReduce over the ranks (hutchinson.py:54 over GPUs)."""
        active = active or plans
        for pl in active:
            pl.export_grads()
        for pl in active:
            pl.stream.synchronize()
        s = main_stream.ptr
        bl_lib.call("bl_vec_axpby", code, nnz, 1.0, active[0].grads[0].ptr, 0.0, None, grad_total.ptr, s)
        for pl in active[1:]:
            bl_lib.call("bl_vec_axpby", code, nnz, 1.0, grad_total.ptr, 1.0, pl.grads[0].ptr, grad_total.ptr, s)
        group.allreduce_device(grad_total.ptr, nnz, dtype, main_stream)
        main_stream.synchronize()

    from experiments_lanczos_adjoints_b200 import _lib as bl_lib

    def barrier():
        bl.synchronize()
        group.barrier()
        bl.synchronize()

    def timed(step, steps, active=None, close=True):
        """`steps` steps + the closing reduction, device-timed (events on the launching streams), max over ranks."""
        active = active or plans
        barrier()
        e0, e1 = bl.Event(), bl.Event()
        launches0 = bl.launch_count()
        e0.record(main_stream)
        for pl in active:  # the lanes start after e0
            pl.stream.wait_event(e0)
        for k in range(steps):
            step(k == 0)
        if close:
            finish_estimate(active)
        else:
            for pl in active:
                pl.stream.synchronize()
        e1.record(main_stream)
        e1.synchronize()
        ms = e0.elapsed_ms(e1)
        launches = bl.launch_count() - launches0
        barrier()
        ms = float(group.allreduce_host(np.array(ms), op="max"))
        return ms, launches

    for k in range(args.warmup):
        step_device(first=(k == 0))
    finish_estimate()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_total, launches = timed(lambda first: step_device(first=first), args.steps)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:  # read before the end-to-end steps below reuse the plans and grad_total
        dump_outputs(args.dump_outputs, {
            "H": np.stack([pl.H.numpy(pl.stream) for pl in plans]).reshape(L, per_lane, DEPTH, DEPTH),
            "dv": np.stack([pl.dv.numpy(pl.stream) for pl in plans]).reshape(L, per_lane, N_ROWS),
            "dparams": grad_total.numpy(main_stream),
        })  # fmt: skip
    ms_per_step = ms_total / args.steps
    value = world * probes_per_gpu * DEPTH / (ms_per_step * 1e-3)

    def emit(obj):
        if rank == 0:
            sys.stdout.flush()
            os.dup2(stdout_fd, 1)
            print(json.dumps(obj), flush=True)

    if args.quick:
        emit({"value": value, "ms_per_step": ms_per_step, "gpu_launches": launches, "probes_per_gpu": probes_per_gpu,
              "mode": args.mode, "lanes": L, "stagger": bool(stagger), "quick": True})  # fmt: skip
        bl_comm.shutdown()
        return

    # end-to-end through the host-buffer entry point: per step H2D (v, params, dH) + fwd + adjoint + D2H (H, dv, dparams)
    io = {}

    def step_host(_first):
        h2d = d2h = 0
        for pl, late, v_host, (out_H, out_dv, out_g) in zip(plans, behind, v_hosts, outs):
            if late:
                a, b = pl.run_host(v_host, [p_host], dH_host, out_H, out_dv, out_g, sync=False, adjoint_first=True)
            else:
                a, b = pl.run_host(v_host, [p_host], dH_host, out_H, out_dv, out_g, sync=False)
            h2d, d2h = h2d + a, d2h + b
        for pl in plans:
            pl.stream.synchronize()  # the step's results (H, dv, dparams of every probe) are on the host
        io["h2d"], io["d2h"] = h2d, d2h

    for _ in range(2):
        step_host(False)
    e2e_steps = max(2, args.steps // 2)
    ms_e2e, _ = timed(step_host, e2e_steps)
    e2e_value = world * probes_per_gpu * DEPTH / (ms_e2e / e2e_steps * 1e-3)

    # ONE run alone (the latency of a single forward + adjoint; BASELINE configs[1] as literally stated)
    bl.set_blocks_per_sm(0)  # a run alone: the default two blocks per SM
    single = bl_plan.TridiagAdjointPlan(bl.operators.SparseOperator(row, col, (N_ROWS, N_ROWS)), DEPTH, dtype,
                                        stream=bl_dev.Stream())  # fmt: skip
    single.set_vector(v_hosts[0][0] if lockstep else v_hosts[0])
    single.set_params(p_host)
    single.set_cotangent(dH1)
    single.run()
    single.stream.synchronize()
    e0, e1 = bl.Event(), bl.Event()
    l0 = bl.launch_count()
    e0.record(single.stream)
    for _ in range(3):
        single.run()
    e1.record(single.stream)
    e1.synchronize()
    ms_single = e0.elapsed_ms(e1) / 3
    launches_single = (bl.launch_count() - l0) // 3

    # per-kernel-class timing of one more step of ONE lane (events around every launch, nothing else in flight)
    prof = bl_plan.profile(lambda: (plans[0].forward(), plans[0].adjoint(zero=True, export=True)))
    prof_single = bl_plan.profile(single.run)
    bl.set_blocks_per_sm(blocks_in_flight)
    peak, peak_src = measured_peaks()
    fwd_b, adj_b = (probes_per_gpu * b for b in algorithmic_bytes(N_ROWS, nnz, DEPTH, w))
    step_gbs = (fwd_b + adj_b) / (ms_per_step * 1e-3) / 1e9
    dom = max(prof, key=lambda k: prof[k]["ms"])
    d = prof[dom]
    dom_gbs = d["algorithmic_bytes"] / max(d["ms"], 1e-9) / 1e6
    prof_total = sum(c["ms"] for c in prof.values())
    streamed_b = L * sum(c["algorithmic_bytes"] for c in prof.values())  # per step = L lanes
    symmetric = all(os.environ.get(k, "1")[:1] != "0" for k in ("BL_SYMMETRIC_FORWARD", "BL_SYMMETRIC_ADJOINT", "BL_XDOTS"))
    stepk = lockstep and per_lane >= 2 and os.environ.get("BL_STEP", "1") != "0"
    KERNEL_OF = {"dots": "k_dots_few" if symmetric else "k_dots_tma", "combine": "k_combine_tma",
                 "matvec": "k_sell_spmv_multi" if lockstep and per_lane >= 2 else "k_sell_spmv_normalised",
                 "vjp": "k_sell_spmv_multi (A^T) + k_sell_grad_batch" if lockstep and per_lane >= 2 else "k_sell_spmv (A^T) + k_sell_grad_batch",
                 "other": "k_scale_copy",
                 "fused": "k_step_tma" if stepk else ("k_xdots_tma" if symmetric else "k_fused_tma")}  # fmt: skip

    def classes(pr):
        return {k: {"launches": c["launches"], "ms": round(c["ms"], 4),
                    "gbs": c["algorithmic_bytes"] / max(c["ms"], 1e-9) / 1e6} for k, c in pr.items()}  # fmt: skip

    single_streamed = sum(c["algorithmic_bytes"] for c in prof_single.values())
    roofline = {
        "bound": "hbm", "kernel": KERNEL_OF[dom],
        "achieved": dom_gbs, "peak": peak, "unit": "GB/s", "frac": dom_gbs / peak, "peak_source": peak_src,
        "traffic": NCU_TRAFFIC.get(KERNEL_OF[dom], {}).get("traffic"),
        "traffic_capture": NCU_TRAFFIC.get(KERNEL_OF[dom]), "launches_per_step": L * d["launches"],
        "avg_launch_ms": d["ms"] / max(1, d["launches"]), "share_of_step": d["ms"] / max(prof_total, 1e-9),
        "timing": "CUDA events around every launch of one lane's forward + adjoint, no other lane in flight",
        # streamed = the bytes this build's kernels account for; contract = SURVEY 8(d)'s figure for the general
        # (non-symmetric) loops, one operator read per probe.  The symmetric loops of tridiag(reortho="full") skip part of
        # the contract's traffic (local first Gram-Schmidt pass, one Lambda row, banded Gamma) and a lockstep batch reads
        # the operator once for all its probes, so contract_frac may exceed 1: the saving is reported as such, the
        # bandwidth claim is `frac` (streamed bytes / time / peak).
        "whole_step": {"streamed_gb": streamed_b / 1e9, "achieved": streamed_b / (ms_per_step * 1e-3) / 1e9,
                       "frac": streamed_b / (ms_per_step * 1e-3) / 1e9 / peak,
                       "contract_gb": (fwd_b + adj_b) / 1e9, "contract_equivalent_gbs": step_gbs,
                       "contract_frac": step_gbs / peak},
        "classes": classes(prof),
        "single_probe": {"streamed_gb": single_streamed / 1e9, "achieved": single_streamed / (ms_single * 1e-3) / 1e9,
                         "frac": single_streamed / (ms_single * 1e-3) / 1e9 / peak, "classes": classes(prof_single)},
    }  # fmt: skip

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {
            "workload": f"sparse SPD COO operator n={N_ROWS} nnz={nnz} ({2 * BANDS + 1}/row), Lanczos full "
                        f"reortho depth {DEPTH}, forward + adjoint (cotangents on alpha/beta)",
            "per_gpu": (f"{probes_per_gpu} independent probe vectors per GPU per step: {L} lockstep batch(es) of {per_lane} "
                        "(ONE k_step_tma launch per Krylov step and batch: operator call + Gram-Schmidt step), one stream per batch"
                        if lockstep else
                        f"{probes_per_gpu} independent probe vectors per GPU per step, each on its own stream") +
                       ("; every second batch runs half a cycle behind (its adjoint beside its neighbour's forward)" if stagger else "") +
                       "; the parameter cotangent accumulates on the device over the steps and the timed region ends with "
                       "one export + sum" + (" + ONE ncclAllReduce over the ranks" if world > 1 else ""),
            "mode": args.mode, "lanes": L, "probes_per_lane": per_lane, "probes_per_gpu": probes_per_gpu, "stagger": bool(stagger),
            "blocks_per_sm": {"timed_region": blocks_in_flight or 2, "single_probe_and_kernel_profile": 2},
            "single_probe": {"ms_per_forward_adjoint": ms_single, "krylov_steps_per_s": DEPTH / (ms_single * 1e-3),
                             "launches_per_run": int(launches_single)},
            "launches_per_probe_run": launches / args.steps / probes_per_gpu,
            "loops": ("symmetric loops of tridiag(reortho=full): BL_FWD_SYMMETRIC, BL_ADJ_SYMMETRIC, "
                      "BL_ADJ_TRIDIAG_COTANGENT (include/b200_lanczos.h); switched off by BL_SYMMETRIC_FORWARD=0 / "
                      "BL_SYMMETRIC_ADJOINT=0: " + ",".join(
                          f"{k}={os.environ[k]}" for k in ("BL_SYMMETRIC_FORWARD", "BL_SYMMETRIC_ADJOINT") if k in os.environ)),
            "l2": f"inputs larger than L2 (basis Q {DEPTH * N_ROWS * w / 1e6:.0f} MB per probe + adjoint basis, 126 MB L2)",
            "collectives": "libb200lanczos bl_dist_nccl_* (dlopen libnccl.so.2), socket rendezvous; no torch" if world > 1 else "none (1 GPU)",
        },
        "clocks": clocks, "gpu_launches": launches,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": io["h2d"], "d2h_bytes_per_step": io["d2h"],
                "ms_per_step": ms_e2e / e2e_steps},
        "roofline": roofline,
    }  # fmt: skip
    if world == 1 and not args.no_cpu_baseline and rank == 0:
        out["cpu_baseline"] = cpu_baseline(row, col, data, dalpha, dbeta)
    if not args.no_extra:
        del plans[:], single
        bl.empty_cache()
        bl.set_blocks_per_sm(0)  # the extras are single runs (or manage the setting themselves)
        import bench_extra

        extra = bench_extra.run_all(bl, group, row, col, data, N_ROWS, DEPTH, quick=bool(os.environ.get("BL_BENCH_EXTRA_QUICK")))
        out["extra"] = extra
    emit(out)
    bl_comm.shutdown()


if __name__ == "__main__":
    main()
