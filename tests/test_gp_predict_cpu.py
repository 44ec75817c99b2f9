"""GP prediction, host side: the float64 posterior oracle and the argument checks that run before any
device call."""

import types

import numpy as np
import pytest
from gp_posterior_oracle import kernel_matrix, posterior, prior_diag

import experiments_lanczos_adjoints_b200 as bl
from experiments_lanczos_adjoints_b200 import _lib, operators
from experiments_lanczos_adjoints_b200 import gp

KINDS = ("matern32", "matern12", "rbf")


def _problem(seed, n=60, m=25, d=3):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-1, 1, (n, d))
    y = np.sin(X.sum(1)) + 0.1 * rng.standard_normal(n)
    return X, y, rng.uniform(-1.2, 1.2, (m, d)), rng.standard_normal(d) * 0.3, 0.4


@pytest.mark.parametrize("kind", KINDS)
def test_oracle_posterior_matches_a_direct_solve(kind):
    X, y, Xt, raw_ls, raw_os = _problem(1)
    noise, const = 0.05, 0.3
    mean, var, _ = posterior(kind, X, y, Xt, raw_ls=raw_ls, raw_os=raw_os, noise=noise, const=const)
    K = kernel_matrix(kind, raw_ls, raw_os, X, X)
    np.fill_diagonal(K, prior_diag(kind, raw_os, len(X)))
    K += noise * np.eye(len(X))
    Kx = kernel_matrix(kind, raw_ls, raw_os, Xt, X)
    mean_d = const + Kx @ np.linalg.solve(K, y - const)
    var_d = np.array([prior_diag(kind, raw_os, 1)[0] - k @ np.linalg.solve(K, k) for k in Kx])
    np.testing.assert_allclose(mean, mean_d, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(var, var_d, rtol=1e-9, atol=1e-12)
    prior = prior_diag(kind, raw_os, len(Xt))
    assert np.all(var >= -1e-12) and np.all(var <= prior + 1e-12)
    # k(x, x) is the kernel formula at zero distance, which for the Matérn kinds is not the outputscale (the
    # expanded distance of a point to itself is O(eps |x|^2) in float64 here; sqrt turns that into ~1e-8)
    np.testing.assert_allclose(prior, np.diag(kernel_matrix(kind, raw_ls, raw_os, Xt, Xt)), rtol=1e-7)
    assert kind == "rbf" or np.all(prior < float(bl.gp.constraint_greater_than(0.0)(raw_os)))


@pytest.mark.parametrize("kind", KINDS)
def test_oracle_mean_reproduces_targets_with_noise_at_its_floor(kind):
    X, y, _, raw_ls, raw_os = _problem(2, n=30)
    noise = 1e-8
    mean, var, _ = posterior(kind, X, y, X, raw_ls=raw_ls, raw_os=raw_os, noise=noise, const=0.1)
    np.testing.assert_allclose(mean, y, atol=1e-5)
    assert np.all(var < 10 * noise)


@pytest.mark.parametrize("bad", [np.zeros((4, 2)), np.zeros((0, 3)), np.zeros(3), np.array([[0.0, np.nan, 1.0]]),
                                 np.array([[np.inf, 0.0, 0.0]])])  # fmt: skip
def test_bad_test_inputs_are_rejected_before_any_device_call(bad, monkeypatch):
    def no_device(*args, **kwargs):
        raise AssertionError("device call")

    monkeypatch.setattr(_lib, "call", no_device)
    parent = types.SimpleNamespace(d=3, n=10)
    with pytest.raises(ValueError):
        operators.GramCross(parent, bad)
    X, y, _, raw_ls, raw_os = _problem(3)
    likelihood, _ = gp.likelihood_pdf_p(gp.gram_matvec(), None, None, constrain=gp.constraint_greater_than(1e-4))
    m, _ = gp.mean_constant(shape_out=())
    k, _ = gp.kernel_scaled_matern_32(shape_in=(3,), shape_out=())
    predict = gp.posterior(gp.model_gp(m, k), likelihood)
    with pytest.raises(ValueError):
        predict(X, y, bad, params_mean={"constant_value": 0.0},
                params_kernel={"raw_lengthscale": raw_ls, "raw_outputscale": raw_os},
                params_likelihood={"raw_noise": 0.0})  # fmt: skip


def test_batched_pcg_workspace_query_is_a_pure_host_function():
    lib = _lib.load()
    one = lib.bl_pcg_batch_workspace_bytes(1000, 1, _lib.BL_F32)
    many = lib.bl_pcg_batch_workspace_bytes(1000, 37, _lib.BL_F32)
    wide = lib.bl_pcg_batch_workspace_bytes(36_576, 1024, _lib.BL_F64)
    assert 0 < one < many < wide
    assert wide >= 3 * 36_576 * 1024 * 8


def test_vmap_solver_takes_only_solvers_of_the_cg_module():
    with pytest.raises(TypeError):
        bl.cg.vmap_solver(lambda A, b: b)
    assert isinstance(bl.cg.vmap_solver(bl.cg.cg_adaptive(atol=1e-3, rtol=0.0, maxiter=5, miniter=0)),
                      bl.cg._VmapSolver)  # fmt: skip
