"""GPU parity tests: the CUDA path (through the host layer -> C ABI) against
 (1) the golden vectors produced by the reference's own sources (tests/golden),
 (2) the NumPy oracle on seeded inputs at sizes the oracle finishes in seconds,
 (3) size-independent properties at BASELINE.json's full size (n = 1M, K = 100).
Tolerances (BASELINE.json north_star): fp32 1e-5 on tridiagonal coefficients / log-dets and
1e-4 on gradients; fp64 1e-10 on all three; integer index work bit-exact."""

import os

import numpy as np
import pytest
from conftest import golden, golden_names, rel_err

import experiments_lanczos_adjoints_b200 as bl
from oracle import krylov, operators

pytestmark = pytest.mark.gpu

F32_VAL, F32_GRAD, F64 = 1e-5, 1e-4, 1e-10


def dt(g):
    return np.float64 if bool(g["x64"]) else np.float32


def tol(g, grad=False):
    return F64 if bool(g["x64"]) else (F32_GRAD if grad else F32_VAL)


def dense_op(g):
    return bl.operators.DenseOperator(len(g["v"]), sym=str(g["matvec"]) == "sym")


@pytest.mark.parametrize("name", golden_names("arnoldi_"))
def test_arnoldi_matches_reference_golden(name):
    g = golden(name)
    d, K, n = dt(g), int(g["K"]), len(g["v"])
    alg = bl.arnoldi.hessenberg(dense_op(g), K, reortho=str(g["reortho"]), reortho_vjp=str(g["reortho_vjp"]))
    (Q, H, r, c), pull = bl.vjp(alg, g["v"].astype(d), g["A"].astype(d))
    assert Q.shape == (n, K) and H.shape == (K, K) and r.shape == (n,) and c.shape == ()
    Qh, Hh, rh = Q.numpy(), H.numpy(), r.numpy()
    if "hilbert" in name:
        # cond ~ 1e13: only the reference's own identities hold (test_hessenberg_forward.py:58-66)
        A = g["A"] + g["A"].T if str(g["matvec"]) == "sym" else g["A"]
        small = np.sqrt(np.finfo(d).eps)
        assert np.allclose(A @ Qh - Qh @ Hh - np.outer(rh, np.eye(K)[-1]), 0.0, atol=small)
        assert np.allclose(Qh.T @ Qh, np.eye(K), atol=small)
        assert np.allclose(Qh[:, 0], float(c) * g["v"], atol=small)
        return
    for mine, ref in ((Qh, "Q"), (Hh, "H"), (float(c), "c")):
        assert rel_err(mine, g[ref]) < 2 * tol(g), ref
    if K < n:
        assert rel_err(rh, g["r"]) < 2 * tol(g)
    dv, dp = pull(tuple(g[k].astype(d) for k in ("dQ", "dH", "dr", "dc")))
    assert rel_err(dv.numpy(), g["dv_adjoint"]) < 2 * tol(g, True)
    assert rel_err(dp.numpy(), g["dp_adjoint"]) < 2 * tol(g, True)


@pytest.mark.parametrize("name", golden_names("tridiag_"))
def test_tridiag_matches_reference_golden(name):
    g = golden(name)
    d, K, n = dt(g), int(g["K"]), len(g["v"])
    alg = bl.lanczos.tridiag(dense_op(g), K, reortho=str(g["reortho"]))
    ((Qt, (alpha, beta)), (q_rem, b_rem)), pull = bl.vjp(alg, g["v"].astype(d), g["A"].astype(d))
    assert Qt.shape == (K, n) and alpha.shape == (K,) and beta.shape == (K - 1,)
    # 3-term Lanczos without re-orthogonalisation loses orthogonality: rounding-order
    # differences grow with K (the reference tests it at 1e-1, test_tridiag_forward.py:29-30)
    loose = 1e3 if (str(g["reortho"]) == "none" and K > 5) else 1.0
    assert rel_err(alpha, g["alpha"]) < loose * tol(g)
    assert rel_err(beta, g["beta"]) < loose * tol(g)
    assert rel_err(Qt.numpy(), g["Qt"]) < loose * 10 * tol(g)
    if K == n:
        return
    assert rel_err(q_rem.numpy(), g["q_rem"]) < loose * 10 * tol(g)
    assert rel_err(b_rem, g["b_rem"]) < loose * 10 * tol(g)
    cot = ((g["dQt"], (g["dalpha"], g["dbeta"])), (g["dq_rem"], g["db_rem"]))
    dv, dp = pull(cot)
    assert rel_err(dv.numpy(), g["dv_adjoint"]) < loose * 5 * tol(g, True)
    assert rel_err(dp.numpy(), g["dp_adjoint"]) < loose * 5 * tol(g, True)


@pytest.mark.parametrize("name", golden_names("sparse_coo_"))
def test_sparse_operand_matches_reference_golden(name):
    g = golden(name)
    d, K, n = dt(g), int(g["K"]), int(g["n"])
    op = bl.operators.SparseOperator(g["row"], g["col"], (n, n))
    # the matvec itself (BCOO @ x sums duplicates)
    x = g["v"].astype(d)
    y = op(x, g["data"].astype(d)).numpy()
    y_ref = operators.CooOperator(g["row"], g["col"], (n, n)).matvec(g["v"], g["data"])
    assert rel_err(y, y_ref) < tol(g)
    alg = bl.lanczos.tridiag(op, K, reortho=str(g["reortho"]))
    ((Qt, (alpha, beta)), _), pull = bl.vjp(alg, x, g["data"].astype(d))
    assert rel_err(alpha, g["alpha"]) < tol(g) and rel_err(beta, g["beta"]) < tol(g)
    cot = ((g["dQt"], (g["dalpha"], g["dbeta"])), (g["dq_rem"], g["db_rem"]))
    dv, dp = pull(cot)
    assert rel_err(dv.numpy(), g["dv"]) < 5 * tol(g, True)
    assert rel_err(dp.numpy(), g["dp"]) < 5 * tol(g, True)  # parameter gradient in COO order
    dv0, dp0 = pull(((None, (g["dalpha"], g["dbeta"])), (None, None)))  # SLQ-style cotangent
    assert rel_err(dv0.numpy(), g["dv_slqcot"]) < 5 * tol(g, True)
    assert rel_err(dp0.numpy(), g["dp_slqcot"]) < 5 * tol(g, True)


@pytest.mark.parametrize("name", golden_names("slq_"))
def test_slq_value_and_grad_match_reference_golden(name):
    g = golden(name)
    d, K = dt(g), int(g["K"])
    n = g["probes"].shape[1]
    op = bl.operators.DenseOperator(n, sym=str(g["matvec"]) == "sym")
    integrand = bl.lanczos.integrand_spd(np.log, K, op)
    probes = g["probes"].astype(d)
    A = g["A"].astype(d)
    vals = np.array([integrand(p, A) for p in probes])
    assert rel_err(vals, g["probe_values_adjoint"]) < tol(g)
    estimate = bl.hutchinson.hutchinson(integrand, lambda key: probes)
    assert rel_err(estimate(None, A), g["value_adjoint"]) < tol(g)
    value, grad = bl.value_and_grad(estimate, argnums=1)(None, A)
    assert rel_err(value, g["value_adjoint"]) < tol(g)
    assert rel_err(grad.numpy(), g["grad_adjoint"]) < tol(g, True)
    _, (dv0, _dA) = integrand.value_and_grad(probes[0], A)
    assert rel_err(dv0.numpy(), g["probe_dv0_adjoint"][0]) < 5 * tol(g, True)
    reuse = bl.lanczos.integrand_spd_custom_vjp_reuse(np.log, K, op)
    est_r = bl.hutchinson.hutchinson_nograd(reuse, lambda key: probes)
    with pytest.warns(UserWarning):
        value_r, (grad_r,) = est_r.value_and_grad(None, A)
    assert rel_err(value_r, g["value_reuse"]) < tol(g)
    assert rel_err(grad_r.numpy(), g["grad_reuse"]) < tol(g, True)


@pytest.mark.parametrize("name", golden_names("gp_kernels_"))
@pytest.mark.parametrize("kind", ["matern32", "matern12", "rbf"])
def test_gram_operator_matches_reference_golden(name, kind):
    g = golden(name)
    d = dt(g)
    amp = 1000.0 if kind == "matern12" else 5.0  # see tests/test_oracle_golden.py
    op = bl.operators.GramOperator(g["X"], kind=kind)
    params = (g["raw_lengthscale"].astype(d), g["raw_outputscale"].astype(d), np.zeros((), d))
    y = op(g["v"].astype(d), *params).numpy()
    assert rel_err(y, g[f"{kind}_y"]) < amp * tol(g)
    op.grad_zero(d)
    z = op.vjp(bl.asarray(g["v"].astype(d)), bl.asarray(g["lam"].astype(d))).numpy()
    dls, dos, dnoise = (a.numpy() for a in op.grad_export(d))
    assert rel_err(z, g[f"{kind}_dv"]) < amp * tol(g)
    if kind != "matern12":
        assert rel_err(dls, g[f"{kind}_dls"]) < amp * tol(g, True)
    assert rel_err(dos, g[f"{kind}_dos"]) < amp * tol(g, True)
    assert rel_err(dnoise, g["lam"] @ g["v"]) < tol(g, True)


def test_wave_operator_and_arnoldi_match_reference_golden():
    g = golden("pde_wave_g8_k6_f64")
    grid, K = int(g["g"]), int(g["K"])
    op = bl.operators.WaveStencilOperator(grid, g["stencil"])
    y0, lam, scale = g["y0"].ravel(), g["lam"].ravel(), g["scale"]
    assert rel_err(op(y0, scale).numpy(), g["rhs"].ravel()) < 1e-12
    op.grad_zero(np.float64)
    z = op.vjp(bl.asarray(y0), bl.asarray(lam)).numpy()
    (dscale,) = op.grad_export(np.float64)
    assert rel_err(z, g["rhs_dx"].ravel()) < 1e-12
    assert rel_err(dscale.numpy(), g["rhs_dscale"]) < 1e-12
    # expm action (1/c) Q expm(dt H) e1 and its gradient through the Arnoldi adjoint (pde_util.py:260-266)
    import scipy.linalg

    alg = bl.arnoldi.hessenberg(op, K, reortho="full")
    (Q, H, r, c), pull = bl.vjp(alg, y0, scale)
    Hh, ch, t1, u = H.numpy(), float(c), float(g["t1"]), g["u"].ravel()
    E = scipy.linalg.expm(t1 * Hh)
    out = (Q.numpy() @ E[:, 0]) / ch
    assert rel_err(out, g["expm_out"].ravel()) < 1e-10
    yv = E[:, 0]
    dQ = np.outer(u, yv) / ch
    dy = (Q.numpy().T @ u) / ch
    dc = -np.dot(u, Q.numpy() @ yv) / ch**2
    e1 = np.zeros(K)
    e1[0] = 1.0
    dH = t1 * scipy.linalg.expm_frechet(t1 * Hh.T, np.outer(dy, e1), compute_expm=False)
    dy0, dsc = pull((dQ, dH, None, dc))
    assert rel_err(dy0.numpy(), g["loss_dy0"].ravel()) < 1e-9
    assert rel_err(dsc.numpy(), g["loss_dscale"]) < 1e-9
    # the same through the drop-in factories (pde_util.py:240-268): solver_expm(expm_arnoldi)
    field, like = bl.pde.pde_wave_anisotropic(scale, g["stencil"], constrain="square", boundary="neumann")
    assert like["scale"].shape == scale.shape
    solve = bl.pde.solver_expm(0.0, t1, field, expm=bl.pde.expm_arnoldi(K))
    y1, info = solve(g["y0"], scale)
    assert info == {"num_matvecs": K} and rel_err(y1.numpy(), g["expm_out"].ravel()) < 1e-10
    (y1, _), pullback = bl.vjp(solve, g["y0"], scale)
    dy0_f, dsc_f = pullback(g["u"])
    assert rel_err(y1.numpy(), g["expm_out"].ravel()) < 1e-10
    assert rel_err(dy0_f.numpy(), g["loss_dy0"].ravel()) < 1e-9
    assert rel_err(dsc_f.numpy(), g["loss_dscale"]) < 1e-9


# ---- seeded random problems against the oracle ---------------------------------------------
def banded_spd(n, per_row, seed, max_off=2000):
    """Synthetic SPD operand in `suite_sparse_load` layout: diagonal, strict lower, mirrored."""
    rng = np.random.default_rng(seed)
    offs = np.sort(rng.choice(np.arange(1, min(max_off, n - 1) + 1), size=per_row, replace=False))
    lo_r = np.concatenate([np.arange(o, n) for o in offs])
    lo_c = np.concatenate([np.arange(0, n - o) for o in offs])
    vals = -rng.uniform(0.0, 1.0, lo_r.size)
    row = np.concatenate([np.arange(n), lo_r, lo_c]).astype(np.int32)
    col = np.concatenate([np.arange(n), lo_c, lo_r]).astype(np.int32)
    data = np.concatenate([np.full(n, 2.0 * per_row + 2.0), vals, vals])
    return row, col, data


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n,K", [(20000, 30), (4099, 17), (1, 1), (5, 5)])
def test_sparse_tridiag_and_adjoint_match_oracle(dtype, n, K):
    """Ragged sizes (n not a multiple of the vector width / slice height), n = 1, K = n."""
    rng = np.random.default_rng(n + K)
    if n >= 100:
        row, col, data = banded_spd(n, 4, seed=n)
    else:
        row = np.arange(n, dtype=np.int32)
        col = row.copy()
        data = 1.0 + np.arange(n, dtype=np.float64)
    v = rng.standard_normal(n) + 2.0
    op = bl.operators.SparseOperator(row, col, (n, n))
    alg = bl.lanczos.tridiag(op, K, reortho="full")
    ((Qt, (alpha, beta)), (q_rem, b_rem)), pull = bl.vjp(alg, v.astype(dtype), data.astype(dtype))
    ref = krylov.tridiag(operators.CsrFastOperator(row, col, (n, n)), K, reortho="full")
    ((Qt_r, (alpha_r, beta_r)), (q_r, b_r)), pull_r = ref.vjp(v, data)
    t_val, t_grad = (F64, F64) if dtype == np.float64 else (F32_VAL, F32_GRAD)
    assert rel_err(alpha, alpha_r) < t_val
    if K > 1:
        assert rel_err(beta, beta_r) < t_val
    if K == n:
        return
    dalpha, dbeta = rng.standard_normal(K), rng.standard_normal(K - 1)
    dv, dp = pull(((None, (dalpha, dbeta)), (None, None)))
    z = np.zeros_like
    dv_r, dp_r = pull_r(((z(Qt_r), (dalpha, dbeta)), (z(q_r), z(b_r))))
    assert rel_err(dv.numpy(), dv_r) < 10 * t_grad
    assert rel_err(dp.numpy(), dp_r) < 10 * t_grad
    # dense cotangent on every output (the published benchmark recipe, benchmark.py:95-96)
    cot = ((rng.standard_normal((K, n)), (dalpha, dbeta)), (rng.standard_normal(n), rng.standard_normal()))
    dv, dp = pull(cot)
    dv_r, dp_r = pull_r(cot)
    assert rel_err(dv.numpy(), dv_r) < 10 * t_grad
    assert rel_err(dp.numpy(), dp_r) < 10 * t_grad


def test_dense_basis_cotangent_beyond_depth_128():
    """The published benchmark sweeps the Krylov depth to 250 with a dense cotangent on Q
    (results/.../times_custom.npy[24], benchmark.py:95-96): `dQ^T Q` (arnoldi.py:127) is assembled in 128 x 128
    blocks, any depth."""
    n, K = 1500, 150
    row, col, data = banded_spd(n, 3, seed=5, max_off=40)
    rng = np.random.default_rng(6)
    v = rng.standard_normal(n)
    op = bl.operators.SparseOperator(row, col, (n, n))
    alg = bl.arnoldi.hessenberg(op, K, reortho="full")
    (Q, H, r, c), pull = bl.vjp(alg, v, data)
    ref = krylov.Hessenberg(operators.CsrFastOperator(row, col, (n, n)), K, reortho="full")
    (Q_r, H_r, r_r, c_r), pull_r = ref.vjp(v, data)
    cot = (rng.standard_normal((n, K)), rng.standard_normal((K, K)), rng.standard_normal(n), rng.standard_normal())
    dv, dp = pull(cot)
    dv_r, dp_r = pull_r(cot)
    assert rel_err(H.numpy(), H_r) < 1e-9
    assert rel_err(dv.numpy(), dv_r) < 1e-8 and rel_err(dp.numpy(), dp_r) < 1e-8


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_symmetric_adjoint_shortcuts_match_general_adjoint(dtype):
    """What `tridiag(reortho="full")` passes to the adjoint -- `BL_ADJ_SYMMETRIC` (`Lambda beta_plus`, arnoldi.py:218,
    keeps only its super-diagonal term) and `BL_ADJ_TRIDIAG_COTANGENT` (banded `Gamma`, arnoldi.py:213-217) --
    against the general adjoint, which carries the O(eps) entries of `H` and `Gamma` outside the bands like the
    reference (SURVEY Appendix B7).  Same operand, same cotangents."""
    n, K = 30011, 64
    row, col, data = banded_spd(n, 4, seed=11)
    rng = np.random.default_rng(12)
    v = rng.standard_normal(n)
    op = bl.operators.SparseOperator(row, col, (n, n))
    alg = bl.arnoldi.hessenberg(op, K, reortho="full")
    dalpha, dbeta = rng.standard_normal(K), rng.standard_normal(K - 1)
    dH = np.diag(dalpha) + 0.5 * (np.diag(dbeta, 1) + np.diag(dbeta, -1))
    cots = [(None, dH, None, None),
            (None, dH, rng.standard_normal(n), rng.standard_normal()),
            (rng.standard_normal((n, K)), dH, rng.standard_normal(n), rng.standard_normal())]  # fmt: skip
    results, Hs, Qs = {}, {}, {}
    for flags, (symmetric, tridiagonal) in {1: (False, False), 3: (True, False), 7: (True, True)}.items():
        alg.symmetric, alg.tridiagonal_cotangent = symmetric, tridiagonal
        assert alg._adjoint_flags == flags and alg._forward_flags == (3 if symmetric else 1)
        (Q, H, _, _), pull = bl.vjp(alg, v.astype(dtype), data.astype(dtype))
        Hs[flags], Qs[flags] = H.numpy(), Q.numpy()
        results[flags] = [tuple(x.numpy() for x in pull(c)) for c in cots]
    eps = np.finfo(dtype).eps
    # why the shortcuts are legal: the general forward's H is tridiagonal up to rounding
    assert np.abs(np.triu(Hs[1], 2)).max() < 100 * eps * np.abs(Hs[1]).max()
    # the symmetric forward (first Gram-Schmidt pass on rows i-1, i; BL_FWD_SYMMETRIC) against the general one
    t_val = F64 if dtype == np.float64 else F32_VAL
    # the local first pass skips rows j < i-1; the second pass's coefficients complete those entries of H (EPI_FWD_B)
    assert np.abs(np.triu(Hs[7], 2)).max() < 100 * eps * np.abs(Hs[7]).max()
    assert rel_err(np.diag(Hs[7]), np.diag(Hs[1])) < t_val and rel_err(np.diag(Hs[7], 1), np.diag(Hs[1], 1)) < t_val
    assert rel_err(Qs[7], Qs[1]) < 10 * t_val
    gram = Qs[7].astype(np.float64).T @ Qs[7].astype(np.float64)
    assert np.abs(gram - np.eye(K)).max() < 50 * eps
    t = F64 if dtype == np.float64 else F32_GRAD
    for flags in (3, 7):
        for general, short in zip(results[1], results[flags]):
            for a, b in zip(general, short):
                assert rel_err(b, a) < t, flags


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_lanczos3_matches_oracle(dtype):
    n, K = 3001, 12
    row, col, data = banded_spd(n, 3, seed=5)
    rng = np.random.default_rng(3)
    v = rng.standard_normal(n)
    op = bl.operators.SparseOperator(row, col, (n, n))
    alg = bl.lanczos.tridiag(op, K, reortho="none")
    ((xs, (a, b)), (x_last, b_last)), pull = bl.vjp(alg, v.astype(dtype), data.astype(dtype))
    ref = krylov.tridiag(operators.CsrFastOperator(row, col, (n, n)), K, reortho="none")
    ((xs_r, (a_r, b_r)), (xl_r, bl_r)), pull_r = ref.vjp(v, data)
    t_val, t_grad = (1e-9, 1e-8) if dtype == np.float64 else (5e-5, 5e-4)
    assert rel_err(a, a_r) < t_val and rel_err(b, b_r) < t_val and rel_err(b_last, bl_r) < t_val
    assert rel_err(xs.numpy(), xs_r) < 10 * t_val
    cot = ((rng.standard_normal((K, n)), (rng.standard_normal(K), rng.standard_normal(K - 1))),
           (rng.standard_normal(n), rng.standard_normal()))  # fmt: skip
    dv, dp = pull(cot)
    dv_r, dp_r = pull_r(cot)
    assert rel_err(dv.numpy(), dv_r) < t_grad and rel_err(dp.numpy(), dp_r) < t_grad


def test_callback_operator_runs_user_matvec():
    """An arbitrary user matvec written against DeviceArrays (the reference's `matvec` callable)."""
    n, K = 500, 6
    row, col, data = banded_spd(n, 2, seed=9, max_off=50)
    inner = bl.operators.SparseOperator(row, col, (n, n))
    inner.bind((data,), np.float64)

    def matvec(x):
        return inner.matvec(x)

    op = bl.operators.CallbackOperator(n, matvec)
    v = np.random.default_rng(0).standard_normal(n)
    Q, H, r, c = bl.arnoldi.hessenberg(op, K, reortho="full")(v)
    Q2, H2, r2, c2 = bl.arnoldi.hessenberg(inner, K, reortho="full")(v, data)
    assert rel_err(H.numpy(), H2.numpy()) < 1e-14 and rel_err(r.numpy(), r2.numpy()) < 1e-14

    def bad(x):
        raise KeyError("boom")

    with pytest.raises(KeyError, match="boom"):
        bl.arnoldi.hessenberg(bl.operators.CallbackOperator(n, bad), K, reortho="full")(v)


def test_row_sharded_path_with_one_rank_matches_plain_path():
    """The row-sharded code path (local reduction -> all-reduce hook -> separate epilogue kernel,
    operand = all-gather + rectangular local rows of A and A^T) on a single rank must reproduce the
    plain path; the 2-GPU run is `scripts/run_row_sharded.py` (profiles/r1_row_sharded.json)."""
    from experiments_lanczos_adjoints_b200 import parallel

    n, K = 20000, 12
    row, col, data = banded_spd(n, 4, seed=3)
    rng = np.random.default_rng(4)
    v = rng.standard_normal(n)
    dalpha, dbeta = rng.standard_normal(K), rng.standard_normal(K - 1)
    plain = bl.lanczos.tridiag(bl.operators.SparseOperator(row, col, (n, n)), K, reortho="full")
    ((_, (a0, b0)), _), pull0 = bl.vjp(plain, v, data)
    dv0, dp0 = pull0(((None, (dalpha, dbeta)), (None, None)))
    op = parallel.RowShardedSparseOperator(row, col, n)
    sharded = bl.lanczos.tridiag(op.callback, K, reortho="full")
    with parallel.row_sharded():
        ((_, (a1, b1)), _), pull1 = bl.vjp(sharded, op.local_slice(v), data)
        dv1, dp1 = pull1(((None, (dalpha, dbeta)), (None, None)))
    assert rel_err(a1, a0) < 1e-13 and rel_err(b1, b0) < 1e-13
    assert rel_err(dv1.numpy(), dv0.numpy()) < 1e-12
    assert rel_err(dp1, dp0.numpy()) < 1e-12


def test_wave_slab_operator_with_one_rank_matches_square_operator():
    """Row-sharded wave operand on a single rank (no neighbours) == the plain operand; the halo path
    itself needs two GPUs (`scripts/run_row_sharded_wave.py`, profiles/)."""
    from experiments_lanczos_adjoints_b200 import parallel

    g, K = 96, 5
    rng = np.random.default_rng(0)
    stencil = bl.operators.WaveStencilOperator.stencil_laplacian(1.0)
    y0 = rng.standard_normal((2, g, g))
    scale = 0.3 + 0.05 * rng.standard_normal((g, g))
    dH = rng.standard_normal((K, K))
    plain = bl.arnoldi.hessenberg(bl.operators.WaveStencilOperator(g, stencil), K, reortho="full")
    (Q0, H0, r0, c0), pull0 = bl.vjp(plain, y0.ravel(), scale)
    dv0, ds0 = pull0((None, dH, None, None))
    op = parallel.RowShardedWaveOperator(g, stencil)
    sharded = bl.arnoldi.hessenberg(op.callback, K, reortho="full")
    with parallel.row_sharded():
        (Q1, H1, r1, c1), pull1 = bl.vjp(sharded, op.local_slice(y0), scale)
        dv1, ds1 = pull1((None, dH, None, None))
    assert rel_err(H1.numpy(), H0.numpy()) < 1e-13 and rel_err(r1.numpy(), r0.numpy()) < 1e-12
    assert rel_err(dv1.numpy(), dv0.numpy()) < 1e-12 and rel_err(ds1, ds0.numpy()) < 1e-12


def test_depth_errors_match_reference():
    # /root/reference/tests/test_arnoldi/test_hessenberg_forward.py:69-78
    op = bl.operators.DenseOperator(2)
    for depth in (0, 3):
        with pytest.raises(ValueError, match="depth"):
            bl.arnoldi.hessenberg(op, depth, reortho="none")(np.ones(2), np.eye(2))


# ---- BASELINE.json full size: properties that need no oracle run ----------------------------
@pytest.mark.parametrize("dtype", [np.float32])
def test_full_size_properties(dtype):
    """n = 1M, ~10 nnz/row, K = 100 (BASELINE config 2): Arnoldi identities, orthogonality and
    linearity of the adjoint in its cotangent, checked with device reductions."""
    n, K = 1_000_000, 100
    row, col, data = banded_spd(n, 5, seed=0)  # 1 + 2*5 = 11 entries per row
    rng = np.random.default_rng(0)
    v = rng.standard_normal(n).astype(dtype)
    op = bl.operators.SparseOperator(row, col, (n, n))
    alg = bl.lanczos.tridiag(op, K, reortho="full")
    ((Qt, (alpha, beta)), (q_rem, b_rem)), pull = bl.vjp(alg, v, data.astype(dtype))
    Qh = Qt.numpy()  # (K, n) host copy, 400 MB
    gram = Qh[:, ::7].astype(np.float64) @ Qh[:, ::7].T.astype(np.float64)  # sampled rows only for speed
    full = Qh.astype(np.float64) @ Qh.T.astype(np.float64)
    assert np.abs(full - np.eye(K)).max() < 5e-5, np.abs(full - np.eye(K)).max()
    del gram
    # A Q^T = Q^T T + e_K (q b)^T on a few columns (test_tridiag_forward.py:56-58)
    A = operators.CsrFastOperator(row, col, (n, n))
    T = np.diag(alpha) + np.diag(beta, 1) + np.diag(beta, -1)
    for j in (0, K // 2, K - 1):
        lhs = A.matvec(Qh[j].astype(np.float64), data)
        rhs = T[j] @ Qh
        if j == K - 1:
            rhs = rhs + q_rem.numpy() * b_rem
        assert rel_err(lhs, rhs) < 5e-5
    assert np.all(beta > 0.1)  # no breakdown on this operand
    # linearity of the adjoint in the cotangent
    c1 = (rng.standard_normal(K), rng.standard_normal(K - 1))
    c2 = (rng.standard_normal(K), rng.standard_normal(K - 1))
    dv1, dp1 = pull(((None, c1), (None, None)))
    dv2, dp2 = pull(((None, c2), (None, None)))
    dv3, dp3 = pull(((None, (c1[0] + 2 * c2[0], c1[1] + 2 * c2[1])), (None, None)))
    assert rel_err(dv3.numpy(), dv1.numpy() + 2 * dv2.numpy()) < 1e-4
    assert rel_err(dp3.numpy(), dp1.numpy() + 2 * dp2.numpy()) < 1e-4
    # the symmetric / banded shortcuts of the adjoint (BL_ADJ_SYMMETRIC | BL_ADJ_TRIDIAG_COTANGENT, what `tridiag`
    # passes) against the general adjoint that carries every entry of H and Gamma, at the headline size
    alg.alg.symmetric = alg.alg.tridiagonal_cotangent = False
    dv1_general, dp1_general = pull(((None, c1), (None, None)))
    assert rel_err(dv1.numpy(), dv1_general.numpy()) < 1e-4
    assert rel_err(dp1.numpy(), dp1_general.numpy()) < 1e-4


@pytest.fixture(scope="module")
def headline_oracle():
    """ONE float64 oracle run at BASELINE config 2's full size (n = 1M, 11 entries per row, depth 100): forward,
    the adjoint for the SLQ cotangent (on alpha / beta only) and the adjoint for a dense cotangent on every output
    (the published benchmark recipe, benchmark.py:95-96).  About two minutes of host time; both dtypes of the test
    below compare with it (the float32 inputs are exactly representable in float64)."""
    n, K = 1_000_000, 100
    row, col, data = banded_spd(n, 5, seed=0)
    data = data.astype(np.float32).astype(np.float64)
    rng = np.random.default_rng(5)
    v = rng.standard_normal(n).astype(np.float32).astype(np.float64)
    dalpha = rng.standard_normal(K).astype(np.float32).astype(np.float64)
    dbeta = rng.standard_normal(K - 1).astype(np.float32).astype(np.float64)
    dQt = rng.standard_normal((K, n)).astype(np.float32)
    dq_rem = rng.standard_normal(n).astype(np.float32).astype(np.float64)
    dnorm = float(np.float32(rng.standard_normal()))
    op = operators.CsrFastOperator(row, col, (n, n))
    ((Qt, (alpha, beta)), (q_rem, b_rem)), pull = krylov.tridiag_full_active(op, K, v, data)
    ref = {"alpha": alpha, "beta": beta, "q_rem": q_rem, "b_rem": b_rem, "Q_last": Qt[K - 1].copy()}
    ref["slq"] = pull(((None, (dalpha, dbeta)), (None, None)))
    ref["dense"] = pull(((dQt.astype(np.float64), (dalpha, dbeta)), (dq_rem, dnorm)))
    # SLQ log-determinant integrand of this probe (lanczos.py:48-59)
    w, U = np.linalg.eigh(krylov.dense_tridiag(alpha, beta))
    ref["logdet"] = float(np.dot(v, v) * np.dot(U[0], np.log(w) * U[0]))
    return {"n": n, "K": K, "coo": (row, col, data), "v": v, "cot": (dalpha, dbeta, dQt, dq_rem, dnorm), "ref": ref}


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_headline_size_matches_oracle(headline_oracle, dtype):
    """The tolerance contract of BASELINE.json at the size it is quoted on (n = 1M, depth 100), CUDA path against
    the oracle: alpha, beta, SLQ log-det 1e-5 / 1e-10; gradients (dv, dtheta) 1e-4 / 1e-10 -- for the SLQ cotangent
    and for the dense cotangent.  lanczos.py:152-169, arnoldi.py:201-219."""
    h = headline_oracle
    n, K, ref = h["n"], h["K"], h["ref"]
    row, col, data = h["coo"]
    dalpha, dbeta, dQt, dq_rem, dnorm = h["cot"]
    t_val, t_grad = (F64, F64) if dtype == np.float64 else (F32_VAL, F32_GRAD)
    op = bl.operators.SparseOperator(row, col, (n, n))
    alg = bl.lanczos.tridiag(op, K, reortho="full")
    ((Qt, (alpha, beta)), (q_rem, b_rem)), pull = bl.vjp(alg, h["v"].astype(dtype), data.astype(dtype))
    assert rel_err(alpha, ref["alpha"]) < t_val
    assert rel_err(beta, ref["beta"]) < t_val
    assert np.max(np.abs(alpha - ref["alpha"]) / np.abs(ref["alpha"])) < 10 * t_val  # entry-wise too
    assert np.max(np.abs(beta - ref["beta"]) / np.abs(ref["beta"])) < 10 * t_val
    assert abs(float(b_rem) - ref["b_rem"]) < 10 * t_val * ref["b_rem"]
    assert rel_err(q_rem.numpy(), ref["q_rem"]) < 10 * t_grad
    assert rel_err(Qt.row(K - 1).numpy(), ref["Q_last"]) < 10 * t_grad  # last basis vector: 100 steps of rounding
    integrand = bl.lanczos.integrand_spd(np.log, K, op)
    value = integrand(h["v"].astype(dtype), data.astype(dtype))
    assert abs(float(value) - ref["logdet"]) < t_val * abs(ref["logdet"])
    dv, dp = pull(((None, (dalpha, dbeta)), (None, None)))
    assert rel_err(dv.numpy(), ref["slq"][0]) < t_grad
    assert rel_err(dp.numpy(), ref["slq"][1]) < t_grad
    del dv, dp
    dv, dp = pull(((dQt.astype(dtype), (dalpha, dbeta)), (dq_rem.astype(dtype), dnorm)))
    assert rel_err(dv.numpy(), ref["dense"][0]) < t_grad
    assert rel_err(dp.numpy(), ref["dense"][1]) < t_grad


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_tridiag_full_on_a_nonsymmetric_operand_matches_the_reference_loops(dtype):
    """`tridiag(reortho="full")` runs the symmetric loops by default (DESIGN 4b).  The reference runs general
    Arnoldi and symmetrises (lanczos.py:152-169), whatever the operand: for `lambda s, p: p @ s` with a
    non-symmetric `p` the library must notice (H is not tridiagonal) and return the gradient of the reference's
    output -- the oracle's general loops -- with a warning."""
    n, K = 257, 9
    rng = np.random.default_rng(41)
    A = np.diag(2.0 + np.arange(n) / n) + 0.3 * rng.standard_normal((n, n)) / np.sqrt(n)
    v = rng.standard_normal(n)
    op = bl.operators.DenseOperator(n, sym=False)
    alg = bl.lanczos.tridiag(op, K, reortho="full")
    ref = krylov.tridiag(operators.DenseOperator(), K, reortho="full")
    ((Qt_r, (alpha_r, beta_r)), (q_r, b_r)), pull_r = ref.vjp(v, A)
    t_val, t_grad = (F64, F64) if dtype == np.float64 else (F32_VAL, F32_GRAD)
    with pytest.warns(UserWarning, match="not symmetric"):
        ((Qt, (alpha, beta)), (q_rem, b_rem)), pull = bl.vjp(alg, v.astype(dtype), A.astype(dtype))
    assert rel_err(alpha, alpha_r) < t_val and rel_err(beta, beta_r) < t_val
    assert rel_err(Qt.numpy(), Qt_r) < 10 * t_val
    cot = ((rng.standard_normal((K, n)), (rng.standard_normal(K), rng.standard_normal(K - 1))),
           (rng.standard_normal(n), rng.standard_normal()))  # fmt: skip
    dv, dp = pull(cot)
    dv_r, dp_r = pull_r(cot)
    assert rel_err(dv.numpy(), dv_r) < 10 * t_grad
    assert rel_err(dp.numpy(), dp_r) < 10 * t_grad
    slq_cot = ((None, cot[0][1]), (None, None))
    dv, dp = pull(slq_cot)
    z = np.zeros_like
    dv_r, dp_r = pull_r(((z(Qt_r), cot[0][1]), (z(q_r), z(b_r))))
    assert rel_err(dv.numpy(), dv_r) < 10 * t_grad
    assert rel_err(dp.numpy(), dp_r) < 10 * t_grad
    # a symmetric operand through the same factory stays on the symmetric loops, silently
    import warnings as _w

    S = 0.5 * (A + A.T)
    with _w.catch_warnings():
        _w.simplefilter("error")
        (_, (alpha_s, _b)), _rem = alg(v.astype(dtype), S.astype(dtype))
    (_, (alpha_sr, _b)), _ = ref(v, S)
    assert rel_err(alpha_s, alpha_sr) < t_val


def test_concurrent_plans_on_separate_streams_match_their_solo_runs():
    """`bench.py` keeps several probes in flight per GPU: independent plans (own operator handle, workspace, stream)
    enqueued back to back, their kernels interleaving on the device.  Every plan must reproduce its solo result."""
    from experiments_lanczos_adjoints_b200 import device as dev
    from experiments_lanczos_adjoints_b200 import plan as bl_plan
    from experiments_lanczos_adjoints_b200 import synthetic

    n, K, P, dtype = 300_000, 24, 3, np.float32
    row, col, data = banded_spd(n, 4, seed=21)
    rng = np.random.default_rng(22)
    dH = synthetic.slq_cotangent_dH(rng.standard_normal(K), rng.standard_normal(K - 1), dtype)
    plans = []
    for p in range(P):
        pl = bl_plan.TridiagAdjointPlan(bl.operators.SparseOperator(row, col, (n, n)), K, dtype, stream=dev.Stream())
        pl.set_vector(np.random.default_rng(30 + p).standard_normal(n).astype(dtype))
        pl.set_params(data.astype(dtype))
        pl.set_cotangent(dH)
        plans.append(pl)
    solo = []
    for pl in plans:
        pl.run()
        pl.stream.synchronize()
        solo.append((*pl.coefficients(), pl.dv.numpy(pl.stream), pl.grads[0].numpy(pl.stream)))
    bl.synchronize()
    for _ in range(3):  # all plans in flight at once, several rounds
        for pl in plans:
            pl.run()
    bl.synchronize()
    for pl, (a0, b0, dv0, g0) in zip(plans, solo):
        a, b = pl.coefficients()
        assert rel_err(a, a0) < F32_VAL and rel_err(b, b0) < F32_VAL
        assert rel_err(pl.dv.numpy(pl.stream), dv0) < F32_GRAD and rel_err(pl.grads[0].numpy(pl.stream), g0) < F32_GRAD
    assert rel_err(solo[0][0], solo[1][0]) > 1e-3  # different probes: the comparison above is not vacuous


def _run_check_script(name):
    """A/B checks whose two sides are selected by an environment variable the library reads once per process."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "scripts", name)], cwd=root, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return res.stdout


def test_staged_cotangent_pass_is_bit_identical_to_the_gather_pass():
    """`k_sell_grad_tma` (pairs staged by TMA; banded operands) against `k_sell_grad_batch` (BL_GRAD_TMA=0): the same
    summation order, so the exported parameter cotangent must agree bit for bit -- banded (all blocks staged), random
    sparse (none) and banded with a few far entries (mixed), fp32 and fp64."""
    out = _run_check_script("check_grad_tma.py")
    assert out.count("bit-identical True") == 4, out


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_two_lockstep_lanes_in_flight_reproduce_their_solo_runs_bit_for_bit(dtype):
    """The bench configuration: two lockstep batches of four runs on two streams, one block per SM and kernel, so a
    block of each lane's step kernel shares every SM -- at the headline size (the failure this test pins needs both
    lanes' blocks resident together: phase S's mbarriers once lived in the x-tile buffer, and with another kernel's
    block on the SM the tile came back with barrier words in it; NaN rows in Q / Lambda a few steps later)."""
    from experiments_lanczos_adjoints_b200 import device as dev
    from experiments_lanczos_adjoints_b200 import plan as bl_plan
    from experiments_lanczos_adjoints_b200 import synthetic

    n, K, P, lanes = 1_000_000, 16 if dtype == np.float32 else 10, 4, 2
    row, col, data = synthetic.banded_spd_coo(n, 5, seed=0)
    rng = np.random.default_rng(1)
    ops = [bl.operators.SparseOperator(row, col, (n, n))]
    ops += [ops[0].clone() for _ in range(lanes - 1)]
    plans = [bl_plan.BatchedTridiagAdjointPlan(o, K, dtype, P, stream=dev.Stream()) for o in ops]
    dH = np.stack([synthetic.slq_cotangent_dH(rng.standard_normal(K), rng.standard_normal(K - 1), dtype) for _ in range(P)])
    vs = [(rng.integers(0, 2, size=(P, n)) * 2 - 1).astype(dtype) / np.sqrt(n) for _ in range(lanes)]

    def load():
        for pl, v in zip(plans, vs):
            pl.set_vectors(v)
            pl.set_params(data.astype(dtype))
            pl.set_cotangents(dH)
        bl.synchronize()

    def results(pl):
        return [a.numpy(pl.stream).copy() for a in (pl.H, pl.dv, pl.grads[0])]

    with dev.blocks_per_sm(1):
        load()
        solo = []
        for pl in plans:  # one lane at a time
            pl.run()
            bl.synchronize()
            solo.append(results(pl))
        assert all(np.isfinite(a).all() for res in solo for a in res)
        for rep in range(4):  # both lanes in flight
            load()
            for pl in plans:
                pl.forward()
            for pl in plans:
                pl.adjoint()
            bl.synchronize()
            for li, pl in enumerate(plans):
                for name, got, want in zip(("H", "dv", "dparams"), results(pl), solo[li]):
                    assert np.array_equal(got, want), f"rep {rep} lane {li}: {name} differs from the solo run"


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_slq_estimator_with_probes_in_flight_matches_the_sequential_loop(dtype):
    """`hutchinson(integrand_spd(log, K, sparse_op), sampler)`: with >= 8 probes the estimator runs the probes in
    lockstep batches of four (`lanczos.probe_lockstep_sum`: multi-vector SpMV + one Gram-Schmidt step kernel per
    batch, two batches in flight); value and gradient must equal the one-probe-at-a-time loop
    (`hutchinson.probe_loop_sum`, `jax.vmap(integrand)` + mean, hutchinson.py:14,54)."""
    from experiments_lanczos_adjoints_b200 import lanczos

    n, K, num = 20_003, 12, 9  # 9 = 4 + 4 + 1: the last group is ragged; n odd: rows 1..3 of a batch's (4, n) arrays are not 16-byte aligned
    row, col, data = banded_spd(n, 4, seed=31)
    probes = (np.random.default_rng(32).integers(0, 2, size=(num, n)) * 2 - 1).astype(dtype)
    integrand = bl.lanczos.integrand_spd(np.log, K, bl.operators.SparseOperator(row, col, (n, n)))
    estimate = bl.hutchinson.hutchinson(integrand, lambda key: probes)
    assert lanczos._lockstep_eligible(integrand, probes)
    value, (grad,) = estimate.value_and_grad(None, data.astype(dtype))
    lockstep = (float(value), grad.numpy(), float(estimate(None, data.astype(dtype))))
    loop_integrand = bl.lanczos.integrand_spd(np.log, K, bl.operators.SparseOperator(row, col, (n, n)))
    total, (grad,), count = bl.hutchinson.probe_loop_sum(loop_integrand, probes, (data.astype(dtype),), with_grad=True)
    value_nograd = bl.hutchinson.probe_loop_sum(loop_integrand, probes, (data.astype(dtype),), with_grad=False)[0]
    loop = (float(total) / count, grad.numpy() / count, float(value_nograd) / count)
    t_val, t_grad = (F64, F64) if dtype == np.float64 else (F32_VAL, F32_GRAD)
    assert abs(lockstep[0] - loop[0]) < t_val * abs(loop[0])
    assert abs(lockstep[2] - loop[2]) < t_val * abs(loop[2])
    assert rel_err(lockstep[1], loop[1]) < t_grad
    # and against the float64 oracle on the same probes
    ref = krylov.IntegrandSPD(np.log, lambda x: 1.0 / x, K, operators.CsrFastOperator(row, col, (n, n)))
    val_ref, (grad_ref,) = krylov.hutchinson_value_and_grad(ref, probes.astype(np.float64), data)
    assert abs(lockstep[0] - val_ref) < 10 * t_val * abs(val_ref)
    assert rel_err(lockstep[1], grad_ref) < 10 * t_grad


def test_peer_memory_route_two_ranks_on_one_gpu_matches_single_operator():
    """The native row-sharded route (peer-memory reductions fused with the epilogue + halo pushes,
    `bl_dist_comm_*`) with TWO ranks driven by two host threads on one GPU: each rank owns half of the
    grid rows; results must equal the single-operator run.  (The cross-process form of the same
    kernels runs under torchrun: `scripts/run_row_sharded_wave.py`, profiles/.)"""
    import threading

    from experiments_lanczos_adjoints_b200 import _lib, parallel

    g, K, world = 64, 6, 2
    rng = np.random.default_rng(0)
    stencil = bl.operators.WaveStencilOperator.stencil_laplacian(1.0)
    y0 = rng.standard_normal((2, g, g))
    scale = 0.3 + 0.05 * rng.standard_normal((g, g))
    dH = rng.standard_normal((K, K))
    dr = rng.standard_normal((2, g, g))
    plain = bl.arnoldi.hessenberg(bl.operators.WaveStencilOperator(g, stencil), K, reortho="full")
    (Q0, H0, r0, c0), pull0 = bl.vjp(plain, y0.ravel(), scale)
    dv0, ds0 = pull0((None, dH, dr.ravel(), None))
    H0, r0, dv0, ds0 = H0.numpy(), r0.numpy().reshape(2, g, g), dv0.numpy().reshape(2, g, g), ds0.numpy()
    bl.synchronize()

    # CUDA loads kernels lazily and a load may synchronise the context: with both ranks in ONE process a
    # rank spinning on its peer would block the peer's first launch of a kernel.  Load every kernel of
    # the sharded route first (same local shape, a one-rank communicator).  Separate processes (the
    # production set-up) have separate contexts and need none of this.
    local_n = g // world

    def one_rank_pass():
        solo = parallel.PeerComm(rank=0, world=1)
        slab = bl.operators.WaveStencilOperator(g, stencil, rows=local_n)
        _lib.call("bl_op_wave_set_comm", slab._handle, solo.handle)
        with parallel.row_sharded(comm=solo):
            warm = bl.arnoldi.hessenberg(slab, K, reortho="full")
            res, pull_w = bl.vjp(warm, y0[:, :local_n].ravel(), scale[:local_n])
            grads = pull_w((None, dH, dr[:, :local_n].ravel(), None))
        bl.synchronize()
        return solo, slab, res, grads

    # two passes whose buffers are alive at the same time: afterwards the allocation pool holds what BOTH
    # ranks need, so no rank calls cudaMalloc (which may wait for the peer's spinning kernel) while it runs
    keep = [one_rank_pass(), one_rank_pass()]
    del keep

    def attempt():
        comms = [parallel.PeerComm(rank=r, world=world) for r in range(world)]
        for c in comms:
            c.connect_local(comms)
        out, errors = {}, []
        ready = threading.Barrier(world)

        def rank_main(r):
            try:
                bl.default_stream()  # per-thread stream, operator and halo buffers exist before anyone spins
                op = parallel.RowShardedWaveOperator(g, stencil, comm=comms[r])
                alg = bl.arnoldi.hessenberg(op.callback, K, reortho="full")
                v_loc, s_loc, dr_loc = op.local_slice(y0), op.local_scale(scale), op.local_slice(dr)
                ready.wait(30)
                with parallel.row_sharded(comm=comms[r]):
                    (Q, H, rr, c), pull = bl.vjp(alg, v_loc, s_loc)
                    dv, ds = pull((None, dH, dr_loc, None))
                bl.default_stream().synchronize()
                out[r] = (H.numpy(), rr.numpy(), dv.numpy(), ds.numpy(), op)
            except Exception as exc:  # pragma: no cover
                errors.append(exc)

        threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(90)
        return out, errors, any(c.timed_out() for c in comms)

    out, errors, timed_out = attempt()
    if timed_out and not errors:  # a stalled host thread (not a protocol error): everything is resident now
        out, errors, timed_out = attempt()
    assert not errors, errors
    assert not timed_out
    assert np.array_equal(out[0][0], out[1][0])  # the same H, bit for bit, on both ranks
    for r in range(world):
        H, rr, dv, ds, op = out[r]
        assert rel_err(H, H0) < 1e-12
        assert rel_err(rr, op.local_slice(r0)) < 1e-11
        assert rel_err(dv, op.local_slice(dv0)) < 1e-9
        assert rel_err(ds, op.local_scale(ds0)) < 1e-9


def test_peer_memory_sharded_sparse_two_ranks_on_one_gpu_matches_single_operator():
    """Row-sharded SPARSE operand on the native route (`bl_op_sharded_sparse_create`: all-gather of the
    Lanczos vector through the communicator's peer-memory window, reductions fused with their epilogue),
    two ranks as two host threads on one GPU, against the unsharded operand: tridiagonal coefficients,
    dv and the parameter cotangent in COO order.  n is not a multiple of the chunk alignment."""
    import threading

    from experiments_lanczos_adjoints_b200 import parallel

    n, K, world = 20_011, 12, 2
    row, col, data = banded_spd(n, 4, seed=5, max_off=300)
    rng = np.random.default_rng(6)
    v = rng.standard_normal(n)
    dalpha, dbeta = rng.standard_normal(K), rng.standard_normal(K - 1)
    full = bl.lanczos.tridiag(bl.operators.SparseOperator(row, col, (n, n)), K, reortho="full")
    ((_, (a0, b0)), _), pull0 = bl.vjp(full, v, data)
    dv0, dp0 = pull0(((None, (dalpha, dbeta)), (None, None)))
    dv0, dp0 = dv0.numpy(), dp0.numpy()
    bl.synchronize()

    def attempt():
        comms = [parallel.PeerComm(rank=r, world=world) for r in range(world)]
        for c in comms:
            c.connect_local(comms)
        ops = [parallel.RowShardedSparseOperator(row, col, n, comm=comms[r]) for r in range(world)]
        for c in comms:
            c.connect_windows(comms)
        out, errors = {}, []
        ready = threading.Barrier(world)

        def rank_main(r):
            try:
                bl.default_stream()
                op = ops[r]
                alg = bl.lanczos.tridiag(op.callback, K, reortho="full")
                v_loc, params = op.local_slice(v), op.local_params(data)
                ready.wait(30)
                with parallel.row_sharded(comm=comms[r]):
                    ((_, (alpha, beta)), _), pull = bl.vjp(alg, v_loc, *params)
                    dv, dpa, _dpb = pull(((None, (dalpha, dbeta)), (None, None)))
                bl.default_stream().synchronize()
                out[r] = (np.asarray(alpha), np.asarray(beta), dv.numpy(), dpa.numpy())
            except Exception as exc:  # pragma: no cover
                errors.append(exc)

        threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(90)
        return ops, out, errors, any(c.timed_out() for c in comms)

    ops, out, errors, timed_out = attempt()
    if timed_out and not errors:
        ops, out, errors, timed_out = attempt()
    assert not errors, errors
    assert not timed_out
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    grad = np.zeros(len(data))
    for r in range(world):
        alpha, beta, dv, dpa = out[r]
        assert rel_err(alpha, a0) < 1e-12 and rel_err(beta, b0) < 1e-12
        lo = r * ops[r].chunk
        hi = min(n, lo + ops[r].chunk)
        assert rel_err(dv[: hi - lo], dv0[lo:hi]) < 1e-10
        grad[ops[r].idx_a] = dpa
    assert rel_err(grad, dp0) < 1e-10
