"""GP prediction on the device: the cross-covariance sweep, the lockstep PCG and the posterior, against the
float64 oracle and against single-right-hand-side solves.

fp32 on the tensor-core path evaluates s2 = |x|^2 + |y|^2 - 2 x.y, which is exact only where the square sweep
forces it (its diagonal); the fp32 parity tests therefore keep test points at least 0.1 lengthscales from every
training point, and the coincident-point known answer runs in fp64."""

import numpy as np
import pytest
from conftest import rel_err
from gp_posterior_oracle import kernel_matrix, posterior, prior_diag

import experiments_lanczos_adjoints_b200 as bl
from experiments_lanczos_adjoints_b200 import cg, gp, low_rank, operators

pytestmark = pytest.mark.gpu

KINDS = ("matern32", "matern12", "rbf")
PATHS = [(np.float64, "alu"), (np.float32, "alu"), (np.float32, "tensor")]


def inv_softplus(x):
    return np.log(np.expm1(x))


def far_points(rng, X, m, ls, lo=-1.5, hi=1.5):
    """m points in [lo, hi]^d at least 0.1 lengthscales from every row of X (scaled distance)."""
    out = []
    while len(out) < m:
        cand = rng.uniform(lo, hi, (4 * m, X.shape[1]))
        d2 = ((cand / ls)[:, None, :] - (X / ls)[None, :, :]) ** 2
        keep = cand[np.sqrt(d2.sum(-1)).min(1) >= 0.1]
        out.extend(keep[: m - len(out)])
    return np.asarray(out)


def bound_gram(X, kind, path, dtype, raw_ls, raw_os, noise):
    op = operators.GramOperator(X, kind=kind, path=path)
    params = (np.asarray(raw_ls, dtype), np.asarray([raw_os], dtype), np.asarray([noise], dtype))
    op.bind(params, dtype)
    return op, params


# ---- 1. cross-covariance sweep, columns and prior diagonal ------------------------------------------
SHAPES = [(1000, 77, 9), (700, 1300, 1), (513, 300, 20), (600, 200, 21)]  # (n, M, d): M < 128, M > n, ...


@pytest.mark.parametrize("n,m,d", SHAPES)
@pytest.mark.parametrize("dtype,path", PATHS)
@pytest.mark.parametrize("kind", KINDS)
def test_cross_matvec_columns_and_prior_match_the_oracle(kind, dtype, path, n, m, d):
    if path == "tensor" and d > 20:
        pytest.skip("the tensor-core path takes d <= 20")
    rng = np.random.default_rng(n + m + d)
    ls = np.full(d, 0.4 * np.sqrt(d))
    X = rng.uniform(-1, 1, (n, d))
    Xt = far_points(rng, X, m, ls, lo=-1.0 if d > 1 else 1.05, hi=1.0 if d > 1 else 2.5)
    if d == 1:
        Xt[::2] *= -1  # both sides of the training interval
    raw_ls, raw_os = inv_softplus(ls), 0.3
    op, _ = bound_gram(X, kind, path, dtype, raw_ls, raw_os, 0.5)
    cross = op.cross(Xt)
    v = rng.standard_normal(n)
    eps = float(np.finfo(dtype).eps)  # the reference's eps is that of the working dtype
    Kx = kernel_matrix(kind, raw_ls, raw_os, Xt, X, eps)
    tol = 1e-10 if dtype == np.float64 else 1e-5
    assert rel_err(cross.matvec(v.astype(dtype)).numpy(), Kx @ v) < tol
    first, count = m // 3, min(37, m - m // 3)
    assert rel_err(cross.columns(first, count).numpy(), Kx[first : first + count]) < tol
    assert rel_err(cross.prior_diag().numpy(), prior_diag(kind, raw_os, m, eps)) < tol
    # a re-bind with other parameters re-prepares the test points (the noise plays no part)
    raw_ls2 = raw_ls + 0.2
    op.bind((np.asarray(raw_ls2, dtype), np.asarray([raw_os], dtype), np.asarray([2.0], dtype)), dtype)
    assert rel_err(cross.matvec(v.astype(dtype)).numpy(), kernel_matrix(kind, raw_ls2, raw_os, Xt, X, eps) @ v) < tol


# ---- 2. lockstep PCG against single solves -----------------------------------------------------------
def _operand(which, n, rng):
    if which == "dense64":
        M = rng.standard_normal((n, n)) / np.sqrt(n)
        op = operators.DenseOperator(n, sym=True)
        return operators.bound(op, (M @ M.T + np.eye(n)) / 2), np.float64, None
    dtype, path = (np.float64, "alu") if which == "gram64" else (np.float32, "tensor")
    X = rng.uniform(-1, 1, (n, 3))
    A = operators.bound(operators.GramOperator(X, "matern32", path=path), np.full(3, inv_softplus(0.3), dtype),
                        np.asarray([0.0], dtype), np.asarray([0.5], dtype))  # fmt: skip
    P = None
    if which == "gram32":
        pre, _ = low_rank.preconditioner(low_rank.cholesky_partial_pivot(rank=20))(A, n)
        P = pre.bind(0.5)
    return A, dtype, P


@pytest.mark.parametrize("count", [1, 5, 16, 17, 37])
@pytest.mark.parametrize("which", ["dense64", "gram64", "gram32"])
def test_lockstep_pcg_matches_single_solves_column_by_column(which, count):
    rng = np.random.default_rng(count)
    n = 700
    A, dtype, P = _operand(which, n, rng)
    # fp32: the sweep of one vector and the shared sweep of 16 sum k_ij v_j in different orders, and CG carries
    # such rounding into the recursive residual at about cond * 1e-7 |b|.  At a tolerance near that level (1e-4 |b|
    # here) the residuals of the two runs differ by ~10% and a column can stop one step apart, so the fp32
    # tolerances stay at 3e-3 |b| and above.
    atol = 1e-9 if dtype == np.float64 else 0.3
    solve = cg.pcg_adaptive(atol=atol, rtol=0.0, maxiter=400, miniter=1, check_every=5)
    scales = np.logspace(0, 2, count) if dtype == np.float64 else np.logspace(1, 2, count)
    B = rng.standard_normal((count, n)) * scales[:, None]  # columns freeze at different steps
    if count > 1:
        B[1] = 0.0  # frozen from the start
    if count > 2:
        B[2] = 0.01 * atol * rng.standard_normal(n)  # converges in the first step (miniter = 1)
    B = B.astype(dtype)
    X, info = cg.vmap_solver(solve)(A, B, P)
    Xh = X.numpy()
    tol = 1e-12 if dtype == np.float64 else 1e-5
    for c in range(count):
        x1, info1 = solve(A, B[c], P)
        assert info["num_steps"][c] == info1["num_steps"], (c, info["num_steps"], info1["num_steps"])
        ref = x1.numpy()
        assert np.linalg.norm(Xh[c] - ref) <= tol * max(np.linalg.norm(ref), 1e-30), c
    if count > 2:
        assert info["num_steps"][2] == 1 and len(set(info["num_steps"].tolist())) > 1


# ---- 3. - 6. the posterior ---------------------------------------------------------------------------------
def _predictor(kind, dtype, path, rank, atol, maxiter=2000):
    solve_p = cg.pcg_adaptive(atol=atol, rtol=0.0, maxiter=maxiter, miniter=1)
    precondition = low_rank.preconditioner(low_rank.cholesky_partial_pivot(rank=rank))
    likelihood, _ = gp.likelihood_pdf_p(gp.gram_matvec(), gp.logpdf_krylov_p(solve_p=solve_p, logdet=None),
                                        precondition=precondition, constrain=gp.constraint_greater_than(1e-4))  # fmt: skip
    m, _ = gp.mean_constant(shape_out=())
    k, _ = {"matern32": gp.kernel_scaled_matern_32, "matern12": gp.kernel_scaled_matern_12,
            "rbf": gp.kernel_scaled_rbf}[kind](shape_in=(3,), shape_out=())  # fmt: skip
    likelihood.operator = _with_path(likelihood.operator, path)
    return gp.posterior(gp.model_gp(m, k), likelihood), likelihood


def _with_path(make, path):
    def operator(inputs, kind):
        op = make(inputs, kind)
        bl._lib.call("bl_op_gram_set_path", op._handle, operators.GramOperator.PATHS[path])
        return op

    return operator


def _params(dtype, raw_ls, raw_os, raw_noise, const):
    return dict(params_mean={"constant_value": dtype(const)},
                params_kernel={"raw_lengthscale": np.asarray(raw_ls, dtype), "raw_outputscale": dtype(raw_os)},
                params_likelihood={"raw_noise": dtype(raw_noise)})  # fmt: skip


@pytest.mark.parametrize("m", [1, 300, 1000])
@pytest.mark.parametrize("n", [1000, 4097])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("dtype,path", [(np.float64, "alu"), (np.float32, "tensor")])
def test_posterior_matches_the_oracle(dtype, path, kind, n, m):
    rng = np.random.default_rng(n + m)
    ls = np.full(3, 0.3)
    X = rng.uniform(-1, 1, (n, 3))
    y = np.sin(3 * X).sum(1) + 0.1 * rng.standard_normal(n)
    Xt = far_points(rng, X, m, ls, lo=-1.0, hi=1.0)
    raw_ls, raw_os, const = inv_softplus(ls), 0.3, 0.2
    noise = 0.3
    raw_noise = inv_softplus(noise - 1e-4)
    fp64 = dtype == np.float64
    predict, _ = _predictor(kind, dtype, path, rank=50, atol=1e-12 if fp64 else 1e-6)
    mean, var, info = predict(X, y.astype(dtype), Xt, **_params(dtype, raw_ls, raw_os, raw_noise, const))
    eps = float(np.finfo(dtype).eps)
    mean_r, var_r, _ = posterior(kind, X, y.astype(dtype).astype(np.float64), Xt, raw_ls=raw_ls, raw_os=raw_os,
                                 noise=float(gp.constraint_greater_than(1e-4)(raw_noise)), const=const, eps=eps)  # fmt: skip
    assert not info["variance"]["reached_maxiter"]
    prior = prior_diag(kind, raw_os, m, eps)
    if fp64:
        assert rel_err(mean, mean_r) < 1e-8
        np.testing.assert_allclose(var, var_r, rtol=1e-8, atol=1e-8 * prior.max())
    else:
        assert rel_err(mean, mean_r) < 1e-4
        assert np.max(np.abs(var - var_r) / prior) < 1e-4


def test_known_answer_at_training_inputs_fp64():
    rng = np.random.default_rng(7)
    n = 500
    X = rng.uniform(0, 1, (n, 3))
    y = np.cos(4 * X.sum(1))
    raw_ls, raw_os, const = inv_softplus(np.full(3, 0.05)), 0.5, 0.1
    predict, _ = _predictor("matern32", np.float64, "alu", rank=20, atol=1e-13)
    mean, var, _ = predict(X, y, X, **_params(np.float64, raw_ls, raw_os, -40.0, const))  # noise at its floor
    noise = float(gp.constraint_greater_than(1e-4)(-40.0))
    np.testing.assert_allclose(mean, y, atol=2e-3 * np.abs(y).max())
    assert np.all(var < 10 * noise), var.max()


def test_posterior_is_deterministic():
    rng = np.random.default_rng(11)
    X = rng.uniform(-1, 1, (1000, 3))
    y = np.sin(X.sum(1))
    Xt = far_points(rng, X, 300, np.full(3, 0.3), lo=-1.0, hi=1.0)
    predict, _ = _predictor("matern32", np.float32, "tensor", rank=50, atol=1e-4)
    kw = _params(np.float32, inv_softplus(np.full(3, 0.3)), 0.3, inv_softplus(0.3), 0.2)
    m1, v1, _ = predict(X, y.astype(np.float32), Xt, **kw)
    m2, v2, _ = predict(X, y.astype(np.float32), Xt, **kw)
    assert np.array_equal(m1, m2) and np.array_equal(v1, v2)


def test_posterior_at_protein_scale():
    """n = 36 560, d = 9, fp32 tensor cores, M = 9 140 (the shape of scripts/bench_gp_predict.py)."""
    rng = np.random.default_rng(0)
    n, m, d = 36_560, 9_140, 9
    X = rng.standard_normal((n, d))
    y = np.sin(X[:, 0]) + 0.1 * rng.standard_normal(n)
    Xt = rng.standard_normal((m, d))
    raw_ls, raw_os, raw_noise, const = np.full(d, inv_softplus(1.5)), 0.5, inv_softplus(0.1), 0.05
    # a tight tolerance: the batched and the single solves are compared at well below it
    solve_p = cg.pcg_adaptive(atol=1e-5, rtol=0.0, maxiter=1000, miniter=10)
    precondition = low_rank.preconditioner(low_rank.cholesky_partial_pivot(rank=100))
    likelihood, _ = gp.likelihood_pdf_p(gp.gram_matvec(), gp.logpdf_krylov_p(solve_p=solve_p, logdet=None),
                                        precondition=precondition, constrain=gp.constraint_greater_than(1e-4))  # fmt: skip
    mean_fun, _ = gp.mean_constant(shape_out=())
    k, _ = gp.kernel_scaled_matern_32(shape_in=(d,), shape_out=())
    predict = gp.posterior(gp.model_gp(mean_fun, k), likelihood)
    kw = _params(np.float32, raw_ls, raw_os, raw_noise, const)
    mean, var, info = predict(X, y.astype(np.float32), Xt, **kw)
    assert mean.shape == var.shape == (m,) and not info["variance"]["reached_maxiter"]
    # the device's alpha (the same deterministic solve the posterior ran), then a float64 host evaluation
    target = gp._TargetLogML(gp.model_gp(mean_fun, k), likelihood)
    _, _, _, A, P, _, resid = target._setup(X, y.astype(np.float32), kw["params_mean"], kw["params_kernel"],
                                            kw["params_likelihood"])  # fmt: skip
    alpha, _ = solve_p(A, resid, P)
    alpha = alpha.numpy().astype(np.float64)
    rows = rng.choice(m, 64, replace=False)
    ref = const + kernel_matrix("matern32", raw_ls, raw_os, Xt[rows], X, float(np.finfo(np.float32).eps)) @ alpha
    assert rel_err(mean[rows], ref) < 1e-4
    # variances of 16 test points through single solves
    cross = A.op.cross(Xt)
    prior = cross.prior_diag().numpy().astype(np.float64)
    picks = rng.choice(m, 16, replace=False)
    single = []
    for t in picks:
        kt = cross.columns(int(t), 1).row(0)
        xt, info_t = solve_p(A, kt, P)
        q = float(np.dot(kt.numpy().astype(np.float64), xt.numpy().astype(np.float64)))
        single.append((prior[t] - q, info_t["num_steps"]))
    err = np.abs(var[picks] - [v for v, _ in single]) / prior[picks]
    assert err.max() < 1e-4, (err, [s for _, s in single], info["variance"])
