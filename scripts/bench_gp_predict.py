"""GP prediction at the UCI-protein shape of scripts/bench_gp_logml.py: n = 36 560 training points, d = 9,
Matérn-3/2, rank-100 pivoted-Cholesky preconditioner, fp32 (tensor-core sweeps), pcg_adaptive(atol 1e-2,
maxiter 1000, miniter 10), and M = 9 140 test points (a 80/20 split of the 45 730 protein rows).

Prints one JSON line: the device and its power limit, the time of the posterior mean (the solve for alpha and
one cross-covariance sweep), the time of the exact variances (cross-covariance columns and the lockstep
solves), the iterations of each variance batch and the cross sweep's kernel pairs per second.  Each time is a
host clock around work that ends in a device synchronise, after one warm-up call of the same shapes."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import experiments_lanczos_adjoints_b200 as bl
from experiments_lanczos_adjoints_b200 import cg, gp, low_rank

n, m, d = int(os.environ.get("GP_N", 36560)), int(os.environ.get("GP_M", 9140)), 9
block = int(os.environ.get("BLOCK", 1024))
rng = np.random.default_rng(0)
X = rng.standard_normal((n, d))
y = (np.sin(X[:, 0]) + 0.1 * rng.standard_normal(n)).astype(np.float32)
X_test = rng.standard_normal((m, d))

solve_p = cg.pcg_adaptive(rtol=0.0, atol=1e-2, maxiter=1000, miniter=10)
precondition = low_rank.preconditioner(low_rank.cholesky_partial_pivot(rank=100))
likelihood, _ = gp.likelihood_pdf_p(gp.gram_matvec(), gp.logpdf_krylov_p(solve_p=solve_p, logdet=None),
                                    precondition=precondition, constrain=gp.constraint_greater_than(1e-4))  # fmt: skip
mean_fun, _ = gp.mean_constant(shape_out=())
k, _ = gp.kernel_scaled_matern_32(shape_in=(d,), shape_out=())
model = gp.model_gp(mean_fun, k)
predict = gp.posterior(model, likelihood, block=block)
params = dict(params_mean={"constant_value": np.float32(0.0)},
              params_kernel={"raw_lengthscale": np.full(d, 1.0, np.float32), "raw_outputscale": np.float32(0.5)},
              params_likelihood={"raw_noise": np.float32(-1.0)})  # fmt: skip


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    bl.synchronize()
    return time.perf_counter() - t0, out


def device():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.splitlines()[0]  # fmt: skip
        name, power = (s.strip() for s in q.split(","))
        return name, power
    except Exception as exc:  # the JSON line says what could not be read
        return f"unknown ({exc})", "not read"


bl.set_device(0)
predict(X, y, X_test[:block], **params)  # warm-up of every kernel and shape: one variance block
t_mean, (mean, _, info_mean) = timed(lambda: predict(X, y, X_test, variance=False, **params))
t_all, (_, var, info) = timed(lambda: predict(X, y, X_test, **params))

# the cross sweep alone: K(X*, X) v, timed with device events over repeated launches
target = gp._TargetLogML(model, likelihood)
_, _, _, A, _, _, resid = target._setup(X, y, **params)
A.bind(np.float32)
cross = A.op.cross(X_test)
v = bl.device.asarray(resid)
cross.matvec(v)
reps = 20
e0, e1 = bl.device.Event(), bl.device.Event()
e0.record()
for _ in range(reps):
    cross.matvec(v)
e1.record()
e1.synchronize()
t_sweep = e0.elapsed_ms(e1) / 1e3 / reps

name, power = device()
print(json.dumps({
    "config": "GP posterior mean + exact variances", "device": name, "power_limit": power, "n": n, "d": d, "m": m,
    "dtype": "float32", "kernel": "matern32", "precond_rank": 100, "block": block,
    "mean_s": round(t_mean, 4), "mean_solve_steps": int(info_mean["solve"]["num_steps"]),
    "variance_s": round(t_all - t_mean, 3), "posterior_s": round(t_all, 3),
    "variance_batches": info["variance"]["batches"], "iterations_per_batch": info["variance"]["batch_num_steps"],
    "variance_reached_maxiter": info["variance"]["reached_maxiter"],
    "cross_sweep_ms": round(t_sweep * 1e3, 4), "cross_sweep_pairs_per_s": float(f"{n * m / t_sweep:.4g}"),
    "var_min": float(var.min()), "var_max": float(var.max()),
}))
