"""Gaussian-process log-marginal likelihood on the device: the model plumbing of
`/root/reference/src/matfree_extensions/util/gp_util.py` behind the same factory names, so that the wiring
of the reference's training script reads the same
(`experiments/applications/gaussian_process/train/optim_logml_adjoints_adaptive.py:110-140`):

    solve_p = cg.pcg_adaptive(rtol=0.0, atol=1e-2, maxiter=1000, miniter=10)
    sample = hutchinson.sampler_rademacher(np.ones(n), num=1)
    logdet = gp.krylov_logdet_slq(10, sample=sample, num_batches=10, checkpoint=True)
    precondition = low_rank.preconditioner(low_rank.cholesky_partial_pivot(rank=100))
    logpdf_p = gp.logpdf_krylov_p(solve_p=solve_p, logdet=logdet)
    likelihood, p_likelihood = gp.likelihood_pdf_p(gp.gram_matvec(), logpdf_p, precondition=precondition,
                                                   constrain=gp.constraint_greater_than(1e-4))
    m, p_mean = gp.mean_constant(shape_out=())
    k, p_kernel = gp.kernel_scaled_matern_32(shape_in=(d,), shape_out=())
    loss = gp.target_logml(gp.model_gp(m, k), likelihood)
    (value, info), grads = loss.value_and_grad(X, y, key, params_mean=..., params_kernel=..., params_likelihood=...)

What differs from the reference: kernels and means are descriptions (the matrix-free Gram operator of
`operators.GramOperator` evaluates them), and derivatives come from `value_and_grad` (hand-derived:
Lanczos adjoint for the log-determinant, `custom_linear_solve`'s implicit rule for the solve) instead of
`jax.grad`.
"""

from __future__ import annotations

import numpy as np

from experiments_lanczos_adjoints_b200 import _lib, cg, hutchinson, lanczos
from experiments_lanczos_adjoints_b200 import device as dev
from experiments_lanczos_adjoints_b200.operators import BoundOperator, GramOperator, check_test_inputs


# ---- parameter constraints (gp_util.py:187-201) ------------------------------------------------
class constraint_greater_than:
    """`minval + softplus(x)` (soft-plus with beta = 1, threshold 20); `.grad(x)` is its derivative."""

    def __init__(self, minval, /):
        self.minval = minval

    def __call__(self, x):
        x = np.asarray(x, dtype=np.float64)
        safe = np.where(x < 20.0, x, 1.0)
        return self.minval + np.where(x < 20.0, np.log(1.0 + np.exp(safe)), x)  # log(1 + exp), as gp_util.py:196

    def grad(self, x):
        x = np.asarray(x, dtype=np.float64)
        safe = np.where(x < 20.0, x, 1.0)
        return np.where(x < 20.0, 1.0 / (1.0 + np.exp(-safe)), 1.0)


# ---- model pieces --------------------------------------------------------------------------------
class _Kernel:
    def __init__(self, kind, raw_lengthscale, raw_outputscale):
        self.kind, self.raw_lengthscale, self.raw_outputscale = kind, raw_lengthscale, raw_outputscale


def _kernel_factory(kind):
    def make(*, shape_in, shape_out=()):
        """`gp_util.kernel_scaled_*` (`gp_util.py:69-184`): `(parametrize, params_like)`."""

        def parametrize(*, raw_lengthscale, raw_outputscale):
            return _Kernel(kind, raw_lengthscale, raw_outputscale)

        return parametrize, {"raw_lengthscale": np.empty(shape_in), "raw_outputscale": np.empty(shape_out)}

    return make


kernel_scaled_matern_32 = _kernel_factory("matern32")
kernel_scaled_matern_12 = _kernel_factory("matern12")
kernel_scaled_rbf = _kernel_factory("rbf")


class _ConstantMean:
    def __init__(self, constant_value):
        self.constant_value = constant_value


def mean_constant(*, shape_out):
    """`gp_util.mean_constant` (`gp_util.py:60-67`)."""

    def parametrize(*, constant_value):
        return _ConstantMean(constant_value)

    return parametrize, {"constant_value": np.empty(shape_out)}


def model_gp(mean_fun, kernel_fun):
    """`gp_util.model_gp` (`gp_util.py:49-57`)."""

    def prior(params_mean: dict, params_kernel: dict):
        return mean_fun(**params_mean), kernel_fun(**params_kernel)

    return prior


def gram_matvec():
    """`gp_util.gram_matvec` (`gp_util.py:525-543`): here a marker — the Gram matrix-vector product is
    the matrix-free device sweep of `operators.GramOperator` (no partitions needed: nothing is stored)."""
    return "device-sweep"


def gram_matvec_partitioned(num, *, checkpoint=True):  # noqa: ARG001
    """`gp_util.gram_matvec_partitioned`: partitioning bounds XLA's memory; the device sweep needs none."""
    return "device-sweep"


# ---- log-determinant (gp_util.py:550-575) --------------------------------------------------------
class _LogdetSLQ:
    def __init__(self, krylov_depth, sample, num_batches, vjp_reuse=False):
        self.K, self.sample, self.num_batches, self.vjp_reuse = krylov_depth, sample, num_batches, vjp_reuse

    def _estimator(self, A: BoundOperator):
        make = lanczos.integrand_spd_custom_vjp_reuse if self.vjp_reuse else lanczos.integrand_spd
        dtype = np.asarray(A.params[0]).dtype if len(A.params) else np.float64

        def sample(key):  # probes in the operator's dtype
            s = self.sample(key)
            return s if isinstance(s, dev.DeviceArray) else np.asarray(s, dtype=dtype)

        return hutchinson.hutchinson(make(np.log, self.K, A.op), sample)

    def _keys(self, key):
        return [key] if self.num_batches == 1 else list(hutchinson.split(key, num=self.num_batches))

    def __call__(self, A, /, key):
        est = self._estimator(A)
        values = np.asarray([est(k, *A.params) for k in self._keys(key)], dtype=np.float64)
        if self.num_batches == 1:
            return values[0], {"std": 0.0, "std_rel": 0.0}
        mean, std = values.mean(), values.std()
        return mean, {"std_abs": std, "std_rel": std / abs(mean)}

    def value_and_grad(self, A, /, key):
        """Value and the gradient w.r.t. the operator's parameters (Lanczos adjoint per probe)."""
        est = self._estimator(A)
        values, grads = [], None
        for k in self._keys(key):
            v, g = est.value_and_grad(k, *A.params)
            values.append(float(v))
            g = [np.asarray(x.numpy() if isinstance(x, dev.DeviceArray) else x, dtype=np.float64) for x in g]
            grads = g if grads is None else [a + b for a, b in zip(grads, g)]
        values = np.asarray(values)
        grads = [g / len(values) for g in grads]
        info = {"std": 0.0, "std_rel": 0.0} if self.num_batches == 1 else {
            "std_abs": values.std(), "std_rel": values.std() / abs(values.mean())}  # fmt: skip
        return values.mean(), info, grads


def krylov_logdet_slq(krylov_depth, /, *, sample, num_batches: int, checkpoint: bool = True):  # noqa: ARG001
    """`gp_util.krylov_logdet_slq` (`gp_util.py:550-575`): `logdet(A, key) -> (value, info)`.
    `checkpoint` is accepted for signature compatibility (the adjoint sweep stores what it needs)."""
    return _LogdetSLQ(krylov_depth, sample, num_batches)


def krylov_logdet_slq_vjp_reuse(krylov_depth, /, *, sample, num_batches: int, checkpoint: bool = True):  # noqa: ARG001
    """`gp_util.krylov_logdet_slq_vjp_reuse` (`gp_util.py:578-621`): cheap inexact gradients."""
    return _LogdetSLQ(krylov_depth, sample, num_batches, vjp_reuse=True)


# ---- log-pdf and likelihood (gp_util.py:243-276, 414-431) ----------------------------------------
class _LogpdfKrylovP:
    def __init__(self, solve_p, logdet):
        self.solve_p, self.logdet = solve_p, logdet


def logpdf_krylov_p(solve_p, logdet):
    """`gp_util.logpdf_krylov_p` (`gp_util.py:414-431`)."""
    return _LogpdfKrylovP(solve_p, logdet)


class _Likelihood:
    def __init__(self, logpdf_p, precondition, constrain):
        self.logpdf_p, self.precondition, self.constrain = logpdf_p, precondition, constrain
        self._ops = {}

    def operator(self, inputs, kind):
        key = (id(inputs), kind)
        if key not in self._ops:
            self._ops.clear()  # one data set at a time: the operator keeps X on the device
            self._ops[key] = (GramOperator(np.asarray(inputs), kind=kind), inputs)
        return self._ops[key][0]


def likelihood_pdf_p(matvec, logpdf_p, precondition, *, constrain):  # noqa: ARG001
    """`gp_util.likelihood_pdf_p` (`gp_util.py:243-276`): `(likelihood, {"raw_noise": ...})`."""
    return _Likelihood(logpdf_p, precondition, constrain), {"raw_noise": np.empty(())}


class _TargetLogML:
    def __init__(self, model, likelihood: _Likelihood):
        self.model, self.likelihood = model, likelihood

    def _setup(self, inputs, targets, params_mean, params_kernel, params_likelihood):
        mean, kernel = self.model(params_mean=params_mean, params_kernel=params_kernel)
        lk = self.likelihood
        targets = np.asarray(targets)
        dtype = targets.dtype if targets.dtype in (np.float32, np.float64) else np.dtype(np.float64)
        raw_noise = np.asarray(params_likelihood["raw_noise"], dtype=np.float64)
        noise = lk.constrain(raw_noise)  # gp_util.py:252-253
        op = lk.operator(inputs, kernel.kind)
        params = (np.asarray(kernel.raw_lengthscale, dtype), np.asarray(kernel.raw_outputscale, dtype).reshape(1),
                  np.asarray(noise, dtype).reshape(1))  # fmt: skip
        A = BoundOperator(op, *params)  # cov_matvec(v) + noise * v      (gp_util.py:270)
        pre, info_pre = lk.precondition(A, len(targets))  # lazy_kernel has no noise term (:257-258)
        resid = (targets - np.asarray(mean.constant_value, dtype)).astype(dtype)  # y - mean
        return dtype, raw_noise, noise, A, pre.bind(float(noise)), info_pre, resid

    def __call__(self, inputs, targets, *p_logpdf, params_mean, params_kernel, params_likelihood):
        dtype, _, _, A, P, info_pre, resid = self._setup(inputs, targets, params_mean, params_kernel, params_likelihood)
        lp = self.likelihood.logpdf_p
        logdet, info_logdet = lp.logdet(A, *p_logpdf)
        alpha, info_solve = lp.solve_p(A, resid, P)
        maha = float(np.dot(resid.astype(np.float64), alpha.numpy().astype(np.float64)))
        n = len(resid)
        value = -0.5 * logdet - 0.5 * maha - n / 2 * np.log(2 * np.pi)  # gp_util.py:417-428
        return dtype.type(value), {"precondition": info_pre, "logpdf": {"logdet": info_logdet, "solve": info_solve}}

    def value_and_grad(self, inputs, targets, *p_logpdf, params_mean, params_kernel, params_likelihood):
        """`jax.value_and_grad(mll, has_aux=True)` w.r.t. the three parameter dictionaries: returns
        `((value, info), (d params_mean, d params_kernel, d params_likelihood))`."""
        dtype, raw_noise, noise, A, P, info_pre, resid = self._setup(inputs, targets, params_mean, params_kernel,
                                                                     params_likelihood)  # fmt: skip
        lp = self.likelihood.logpdf_p
        logdet, info_logdet, (g_ls, g_os, g_noise) = lp.logdet.value_and_grad(A, *p_logpdf)
        alpha, info_solve = lp.solve_p(A, resid, P)
        alpha_h = alpha.numpy().astype(np.float64)
        maha = float(np.dot(resid.astype(np.float64), alpha_h))
        # d/dtheta [r^T A^{-1} r] = -alpha^T (dA/dtheta) alpha  (custom_linear_solve, symmetric A)
        op = A.op
        A.bind(dtype)
        op.grad_zero(dtype)
        op.vjp(alpha, alpha, want_z=False)
        m_ls, m_os, m_noise = (np.asarray(g.numpy(), dtype=np.float64) for g in op.grad_export(dtype))
        n = len(resid)
        value = -0.5 * logdet - 0.5 * maha - n / 2 * np.log(2 * np.pi)
        d_ls = -0.5 * np.asarray(g_ls).reshape(-1) + 0.5 * m_ls.reshape(-1)
        d_os = -0.5 * np.asarray(g_os).reshape(()) + 0.5 * m_os.reshape(())
        d_noise = (-0.5 * np.asarray(g_noise).reshape(()) + 0.5 * m_noise.reshape(())) * self.likelihood.constrain.grad(raw_noise)
        d_const = alpha_h.sum()  # d/dc [-(y - c)^T A^{-1} (y - c) / 2]
        info = {"precondition": info_pre, "logpdf": {"logdet": info_logdet, "solve": info_solve}}
        grads = ({"constant_value": dtype.type(d_const)},
                 {"raw_lengthscale": d_ls.astype(dtype), "raw_outputscale": dtype.type(d_os)},
                 {"raw_noise": dtype.type(d_noise)})  # fmt: skip
        return (dtype.type(value), info), grads


def target_logml(model, likelihood, /):
    """`gp_util.target_logml` (`gp_util.py:15-33`): `mll(inputs, targets, *p_logpdf, params_mean=,
    params_kernel=, params_likelihood=) -> (value, info)`, plus `.value_and_grad`."""
    return _TargetLogML(model, likelihood)


# ---- prediction ----------------------------------------------------------------------------------
class _Posterior:
    def __init__(self, model, likelihood: _Likelihood, block: int):
        self._target = _TargetLogML(model, likelihood)  # shares its operator / preconditioner / residual set-up
        self.block = int(block)

    def __call__(self, inputs, targets, test_inputs, *, params_mean, params_kernel, params_likelihood, variance=True):
        X_test = check_test_inputs(test_inputs, np.shape(inputs)[1])  # before any device work
        dtype, _, _, A, P, info_pre, resid = self._target._setup(inputs, targets, params_mean, params_kernel,
                                                                 params_likelihood)  # fmt: skip
        solve = self._target.likelihood.logpdf_p.solve_p
        alpha, info_solve = solve(A, resid, P)  # (K + s I)^{-1} (y - c); binds A
        cross = A.op.cross(X_test)
        c = float(np.asarray(params_mean["constant_value"], dtype=np.float64))
        mean = cross.matvec(alpha).numpy().astype(np.float64) + c
        info = {"precondition": info_pre, "solve": info_solve}
        if not variance:
            return mean.astype(dtype), None, info
        M, n = len(X_test), A.n
        prior = cross.prior_diag().numpy().astype(np.float64)
        quad = np.empty(M, np.float64)
        vsolve = cg.vmap_solver(solve)
        steps = []
        for t0 in range(0, M, self.block):
            count = min(self.block, M - t0)
            Kc = cross.columns(t0, count)  # rows k(x*_t, X)
            Xc, info_c = vsolve(A, Kc, P)
            q = dev.empty((count,), np.float64)
            _lib.call("bl_rows_dot_pairs", dev.dtype_code(dtype), n, count, Kc.ptr, Xc.ptr, Kc.ld, q.ptr,
                      dev.default_stream().ptr)  # fmt: skip
            quad[t0 : t0 + count] = q.numpy()
            if "num_steps" in info_c:
                steps.append(info_c["num_steps"])
        maxiter = vsolve._solver.max_steps
        batch_steps = [int(s.max()) for s in steps] if steps else [maxiter] * ((M + self.block - 1) // self.block)
        info["variance"] = {
            "batches": len(batch_steps),
            "batch_num_steps": batch_steps,  # the largest num_steps of each block
            "num_steps_max": max(batch_steps),
            "reached_maxiter": max(batch_steps) >= maxiter,
        }
        return mean.astype(dtype), (prior - quad).astype(dtype), info


def posterior(model, likelihood, /, *, block: int = 1024):
    """Posterior of the GP at test inputs: `(inputs, targets, test_inputs, *, params_mean=, params_kernel=,
    params_likelihood=, variance=True) -> (mean, var, info)`, for the model and likelihood of `target_logml`.

        mean_t = c + K(x*_t, X) alpha,                  alpha = (K + s I)^{-1} (y - c)
        var_t  = k(x*_t, x*_t) - k_t^T (K + s I)^{-1} k_t,  k_t = K(X, x*_t)

    This is the prediction half of the reference's GP utilities (its `likelihood_condition` /
    `target_posterior` build the same two quantities); the calling convention here follows `target_logml`.
    Every solve uses the likelihood's `solve_p` and preconditioner.  The variances are latent (no noise term)
    and exact up to the solver tolerance: one solve per test point, `block` test points in lockstep
    (`cg.vmap_solver`) sharing every Gram sweep; `k(x, x)` is the kernel formula at zero distance.  `info`
    has the mean solve's info and, for the variances, the number of blocks, the largest `num_steps` of each
    block and of all columns, and whether any column reached `maxiter` (a fixed-step solver reports its step
    count and True).

    fp32 on the tensor-core path: the squared distance of a test point that coincides with a training point
    is O(eps |x|^2), not 0, and the Matérn square root magnifies that; predict at training points in fp64."""
    return _Posterior(model, likelihood, block)
