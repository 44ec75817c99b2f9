"""Lanczos tridiagonalisation and the SLQ integrands built on it.

Host-side mirror of `/root/reference/src/matfree_extensions/lanczos.py`:
`tridiag`, `integrand_spd`, `integrand_spd_custom_vjp_reuse` with the reference's signatures
and return structure.  `reortho="full"` runs Arnoldi and symmetrises (`lanczos.py:152-169`);
`reortho="none"` runs the three-term recurrence and its adjoint (`lanczos.py:172-335`).  The
O(n K) work is on the device; the K x K post-processing (`eigh`, `lanczos.py:48-59`) is host
NumPy, as the survey marks it ("stays in JAX/NumPy, not a kernel target").
"""

from __future__ import annotations

import ctypes as C
import warnings

import numpy as np

from experiments_lanczos_adjoints_b200 import _lib
from experiments_lanczos_adjoints_b200 import arnoldi
from experiments_lanczos_adjoints_b200 import device as dev
from experiments_lanczos_adjoints_b200 import synthetic
from experiments_lanczos_adjoints_b200.arnoldi import _cotangent_basis, _cotangent_vec, _ptr, _run, _Workspace


def _vec_ws():
    nbytes = _lib.load().bl_vec_workspace_bytes()
    return dev.DeviceArray(((nbytes + 3) // 4,), np.float32), nbytes


def device_dot(x: dev.DeviceArray, y: dev.DeviceArray, stream=None) -> float:
    stream = stream or dev.default_stream()
    out = dev.DeviceArray((), x.dtype)
    ws, nbytes = _vec_ws()
    _lib.call("bl_vec_dot", dev.dtype_code(x.dtype), x.size, x.ptr, y.ptr, out.ptr, ws.ptr, nbytes, stream.ptr)
    return float(out.numpy(stream))


def device_axpby(a, x, b, y, stream=None) -> dev.DeviceArray:
    stream = stream or dev.default_stream()
    out = dev.DeviceArray(x.shape, x.dtype)
    _lib.call("bl_vec_axpby", dev.dtype_code(x.dtype), x.size, float(a), x.ptr, float(b), _ptr(y), out.ptr, stream.ptr)
    return out


def hessenberg_is_tridiagonal(H: np.ndarray) -> bool:
    """Whether the Arnoldi matrix of a run is tridiagonal and symmetric up to rounding -- i.e. whether the operand
    behaved like a symmetric one on this Krylov space.  The symmetric loops (DESIGN 4b) complete `H` with the
    second pass's coefficients above the band (`EPI_FWD_B`), so every entry the adjoint shortcuts would drop is
    visible here: `|H[j, i]|, j < i-1` and `|H[i, i+1] - H[i+1, i]|` are `O(eps |H|)` for a symmetric operand and
    `O(|H|)` otherwise."""
    H = np.asarray(H)
    K = H.shape[0]
    if K < 2:
        return True
    scale = float(np.abs(H).max())
    bound = 1e3 * np.finfo(H.dtype).eps * scale
    asym = float(np.abs(np.diag(H, 1) - np.diag(H, -1)).max())
    above = float(np.abs(np.triu(H, 2)).max()) if K > 2 else 0.0
    return bool(np.isfinite(scale) and asym <= bound and above <= bound)


class _TridiagFull:
    """`_tridiag_reortho_full` (`lanczos.py:152-169`).

    The reference runs general Arnoldi and symmetrises `H`.  `assume_symmetric=None` (default) runs the symmetric
    loops and CHECKS the assumption on the `H` of every run (`hessenberg_is_tridiagonal`): an operand that is not
    symmetric gets the general adjoint loops (what the reference computes) and a warning.  `True` skips the check,
    `False` always runs the general loops."""

    def __init__(self, op, krylov_depth, custom_vjp, assume_symmetric=None):
        self.alg = arnoldi.hessenberg(op, krylov_depth, custom_vjp=custom_vjp, reortho="full")
        self.assume_symmetric = assume_symmetric
        # tridiagonalisation is defined for symmetric operands (lanczos.py:152-169)
        self.alg.symmetric = assume_symmetric is not False
        self.alg.tridiagonal_cotangent = self.alg.symmetric  # `pullback` below builds dH from (dalpha, dbeta)

    def _general_adjoint_needed(self, Hh) -> bool:
        if self.assume_symmetric is not None or hessenberg_is_tridiagonal(Hh):
            return False
        warnings.warn(
            "tridiag(reortho='full'): the operand is not symmetric on this Krylov space (H is not tridiagonal "
            "up to rounding); the adjoint runs the general Arnoldi loops, as the reference does.",
            stacklevel=3,
        )
        return True

    @staticmethod
    def _wrap(Qn, Hh, r, stream):
        T = 0.5 * (Hh + Hh.T)  # lanczos.py:162
        diags, offdiags = np.diag(T, 0).copy(), np.diag(T, 1).copy()
        norm = np.sqrt(device_dot(r, r, stream)).astype(Hh.dtype)
        remainder = (device_axpby(1.0 / norm, r, 0.0, None, stream), norm)
        return (Qn.T, (diags, offdiags)), remainder

    def __call__(self, vec, *params, stream=None):
        stream = stream or dev.default_stream()
        Qn, H, r, _c = self.alg(vec, *params, stream=stream)
        return self._wrap(Qn, H.numpy(stream), r, stream)

    def vjp(self, vec, *params, stream=None):
        stream = stream or dev.default_stream()
        (Qn, H, r, _c), pull = self.alg.vjp(vec, *params, stream=stream)
        Hh = H.numpy(stream)
        out = self._wrap(Qn, Hh, r, stream)
        K, dtype = H.shape[0], H.dtype
        norm = float(out[1][1])
        general = self._general_adjoint_needed(Hh)

        def pullback(cot):
            (dQt, (dalpha, dbeta)), (dq_rem, dnorm) = cot
            dH = synthetic.slq_cotangent_dH(dalpha, dbeta, dtype)
            # cotangent of (r/||r||, ||r||) (lanczos.py:166)
            dr = None
            dq = _cotangent_vec(dq_rem, r.size, dtype)
            dn = 0.0 if dnorm is None else float(np.asarray(dnorm))
            if dq is not None or dn != 0.0:
                coef_r = dn / norm
                if dq is not None:
                    coef_r -= device_dot(r, dq, stream) / norm**3
                    dr = device_axpby(1.0 / norm, dq, coef_r, r, stream)
                else:
                    dr = device_axpby(coef_r, r, 0.0, None, stream)
            dQ = None if dQt is None else _as_kn(dQt, K, r.size, dtype)
            if not general:
                return pull((dQ, dH, dr, None))
            saved = self.alg.symmetric, self.alg.tridiagonal_cotangent
            self.alg.symmetric = self.alg.tridiagonal_cotangent = False  # H is complete: general loops on it
            try:
                return pull((dQ, dH, dr, None))
            finally:
                self.alg.symmetric, self.alg.tridiagonal_cotangent = saved

        return out, pullback


def _as_kn(x, K, n, dtype):
    """A `(K, n)` cotangent handed to the Arnoldi pullback, which expects `(n, K)`."""
    if isinstance(x, dev.DeviceArray):
        return x.T
    return np.asarray(x, dtype=dtype).T


class _TridiagNone:
    """`_tridiag_reortho_none` (`lanczos.py:172-212`): three-term recurrence and its adjoint."""

    def __init__(self, op, krylov_depth, custom_vjp):
        arnoldi._require_operator(op)
        self.op, self.K, self.custom_vjp = op, krylov_depth, custom_vjp
        self._ws = _Workspace()

    def _forward(self, vec, params, stream):
        op, K = self.op, self.K
        v = dev.asarray(vec)
        n, dtype = v.shape[0], v.dtype
        if not isinstance(K, (int, np.integer)) or K < 1 or K > n:
            raise ValueError(f"Parameter depth {K} is outside the expected range")
        bound = op.bind(params, dtype, stream)
        ld = dev.basis_ld(n, dtype)
        xs = dev.DeviceArray((K + 1, n), dtype, ld=ld)
        alphas, betas = dev.DeviceArray((K,), dtype), dev.DeviceArray((K,), dtype)
        nbytes = _lib.load().bl_lanczos3_workspace_bytes(n, K, dev.dtype_code(dtype))
        ws = self._ws.get(("l3", n, K, dtype.str), nbytes)
        _run(op, "bl_lanczos3_forward", op._handle, dev.dtype_code(dtype), n, K, v.ptr, xs.ptr, ld,
             alphas.ptr, betas.ptr, ws.ptr, nbytes, stream.ptr)  # fmt: skip
        return (xs, alphas, betas), (v, n, dtype, ld, nbytes, ws, bound)

    @staticmethod
    def _wrap(xs, alphas, betas, K, n, stream):
        a, b = alphas.numpy(stream), betas.numpy(stream)
        basis = dev.DeviceArray((K, n), xs.dtype, ld=xs.ld, owner=xs._owner, ptr=xs.ptr)
        return (basis, (a, b[:-1].copy())), (xs.row(K), b[-1])  # lanczos.py:242-244

    def __call__(self, vec, *params, stream=None):
        stream = stream or dev.default_stream()
        (xs, alphas, betas), (_, n, *_rest) = self._forward(vec, params, stream)
        return self._wrap(xs, alphas, betas, self.K, n, stream)

    def vjp(self, vec, *params, stream=None):
        if not self.custom_vjp:
            raise NotImplementedError("autodiff through the loop is not available; use custom_vjp=True")
        if len(params) != 1:
            raise TypeError("the three-term adjoint supports exactly one parameter array (lanczos.py:329)")
        stream = stream or dev.default_stream()
        (xs, alphas, betas), (v, n, dtype, ld, nbytes, ws, bound) = self._forward(vec, params, stream)
        op, K = self.op, self.K
        out = self._wrap(xs, alphas, betas, K, n, stream)
        vnorm = dev.asarray(np.asarray([np.sqrt(device_dot(v, v, stream))], dtype=dtype))

        def pullback(cot):
            (dxs, (da, db)), (dx_last, db_last) = cot
            dxs_b = None
            dxs_h = None if dxs is None else np.asarray(dxs, dtype=dtype)
            dxl_h = None if dx_last is None else np.asarray(dx_last, dtype=dtype)
            if (dxs_h is not None and dxs_h.any()) or (dxl_h is not None and dxl_h.any()):
                full = np.zeros((K + 1, n), dtype)
                if dxs_h is not None:
                    full[:K] = dxs_h
                if dxl_h is not None:
                    full[K] = dxl_h
                dxs_b = dev.basis_from_host(full, dtype)
            dal = dev.asarray(np.asarray(da, dtype=dtype).reshape(K))
            dbe_h = np.zeros(K, dtype)
            if K > 1 and db is not None:
                dbe_h[: K - 1] = np.asarray(db, dtype=dtype)
            if db_last is not None:
                dbe_h[K - 1] = np.asarray(db_last, dtype=dtype)
            dbe = dev.asarray(dbe_h)
            op.bind(bound, dtype, stream)
            op.grad_zero(dtype, stream)
            dv = dev.DeviceArray((n,), dtype)
            _run(op, "bl_lanczos3_adjoint", op._handle, dev.dtype_code(dtype), n, K, xs.ptr, ld,
                 alphas.ptr, betas.ptr, _ptr(dxs_b), dal.ptr, dbe.ptr, vnorm.ptr, dv.ptr, ws.ptr,
                 nbytes, stream.ptr)  # fmt: skip
            (grad,) = op.grad_export(dtype, stream=stream)
            return dv, grad

        return out, pullback


def tridiag(matvec, krylov_depth, /, *, reortho: str, custom_vjp: bool = True, assume_symmetric=None):
    """Drop-in for `lanczos.tridiag` (`/root/reference/src/matfree_extensions/lanczos.py:142-149`):
    returns `estimate(vec, *params) -> ((Q.T (K,n), (diags, offdiags)), (r/||r||, ||r||))`.
    `assume_symmetric` (not in the reference) controls the symmetric loops of `reortho="full"`, see `_TridiagFull`."""
    if reortho == "full":
        return _TridiagFull(matvec, krylov_depth, custom_vjp, assume_symmetric)
    if reortho == "none":
        return _TridiagNone(matvec, krylov_depth, custom_vjp)
    msg = f"reortho={reortho} unsupported. Choose eiter {'full', 'none'}."
    raise ValueError(msg)  # lanczos.py:148-149 (ValueError here, TypeError in arnoldi: quirk B9)


# --------------------------------------------------------------------------------------------
# SLQ integrands
# --------------------------------------------------------------------------------------------


def _matfun_derivative(matfun, x):
    """f'(x) by the complex-step rule (exact to rounding for analytic NumPy functions such as
    log / sqrt / exp); JAX derives f' by autodiff in the reference (`lanczos.py:56`)."""
    h = 1e-30
    return np.imag(matfun(np.asarray(x, dtype=np.float64) + 1j * h)) / h


def _quadform_and_cotangents(matfun, matfun_grad, alpha, beta, want_grad):
    """`e1^T f(T) e1` through `eigh` (`lanczos.py:48-59`) and, for the gradient, the closed-form
    cotangents of `(diag, off_diag)` (Daleckii-Krein; the reference uses JAX autodiff of eigh)."""
    a64, b64 = np.asarray(alpha, np.float64), np.asarray(beta, np.float64)
    dense = np.diag(a64) + np.diag(b64, 1) + np.diag(b64, -1)
    w, U = np.linalg.eigh(dense)
    fw = np.asarray(matfun(w), dtype=np.float64)
    value = float(np.dot(U[0], fw * U[0]))
    if not want_grad:
        return value, None, None, (w, U)
    dfw = np.asarray((matfun_grad or (lambda x: _matfun_derivative(matfun, x)))(w), dtype=np.float64)
    dw = w[:, None] - w[None, :]
    with np.errstate(divide="ignore", invalid="ignore"):
        F = (fw[:, None] - fw[None, :]) / dw
    same = np.abs(dw) <= 1e-14 * max(1.0, float(np.abs(w).max()))
    F[same] = (0.5 * (dfw[:, None] + dfw[None, :]))[same]
    G = U @ (np.outer(U[0], U[0]) * F) @ U.T
    return value, np.diag(G).copy(), np.diag(G, 1) + np.diag(G, -1), (w, U)


class _IntegrandSPD:
    def __init__(self, matfun, krylov_depth, matvec, reortho, use_adjoints, matfun_grad):
        self.matfun, self.matfun_grad = matfun, matfun_grad
        self.alg = tridiag(matvec, krylov_depth, custom_vjp=use_adjoints, reortho=reortho)

    def __call__(self, v0, *parameters, stream=None):
        stream = stream or dev.default_stream()
        v0 = _flat(v0)
        scale = np.sqrt(device_dot(v0, v0, stream))  # lanczos.py:25
        u = device_axpby(1.0 / scale, v0, 0.0, None, stream)
        (_basis, (diag, off)), _ = self.alg(u, *parameters, stream=stream)
        value, *_ = _quadform_and_cotangents(self.matfun, self.matfun_grad, diag, off, False)
        return diag.dtype.type(scale**2 * value)  # lanczos.py:59

    def value_and_grad(self, v0, *parameters, stream=None, want_dv0=True):
        """`jax.value_and_grad(quadform, argnums=(0, 1, ...))`: `(value, (dv0, *dparams))`."""
        stream = stream or dev.default_stream()
        v0 = _flat(v0)
        scale = np.sqrt(device_dot(v0, v0, stream))
        u = device_axpby(1.0 / scale, v0, 0.0, None, stream)
        ((_basis, (diag, off)), _rem), pull = self.alg.vjp(u, *parameters, stream=stream)
        g, dalpha, dbeta, _ = _quadform_and_cotangents(self.matfun, self.matfun_grad, diag, off, True)
        s2 = scale**2
        du, *dparams = pull(((None, (s2 * dalpha, s2 * dbeta)), (None, None)))
        dv0 = None
        if want_dv0:  # chain rule through u = v0/||v0|| and the scale**2 factor (lanczos.py:24-26,59)
            udu = device_dot(u, du, stream)
            tmp = device_axpby(1.0 / scale, du, -udu / scale, u, stream)
            dv0 = device_axpby(2.0 * g, v0, 1.0, tmp, stream)
        return diag.dtype.type(s2 * g), (dv0, *dparams)


def _batch_eligible(integrand, dtype) -> bool:
    """Lockstep batching applies to the full-reorthogonalisation adjoint path on operators that defer
    their parameter cotangent (the Gram operator on the tensor-core path)."""
    import ctypes as C

    alg = getattr(integrand, "alg", None)
    if not isinstance(alg, _TridiagFull) or not alg.alg.custom_vjp:
        return False
    op = alg.alg.op
    if not hasattr(op, "_handle") or type(op).__name__ in ("CallbackOperator", "SparseOperator"):
        return False  # (the sparse operand defers its cotangent too, but shares no work between probes)
    yes = C.c_int(0)
    try:
        _lib.call("bl_op_deferred_grad", op._handle, dev.dtype_code(dtype), C.byref(yes))
    except Exception:
        return False
    return bool(yes.value)


LOCKSTEP_BATCH = 4  # runs per lockstep batch (one k_step_tma launch serves up to four runs)
LOCKSTEP_LANES = 2  # batches in flight: the host's K x K eigh of one batch runs under the other batch's kernels
LOCKSTEP_MIN_PROBES = 8  # two full batches, so that two are in flight; fewer probes run one at a time


def _lockstep_eligible(integrand, probes) -> bool:
    """Lockstep batches (`probe_lockstep_sum`) apply to the full-reorthogonalisation adjoint path on a square sparse
    operand (an operator that can be cloned: every lane needs its own values and cotangent accumulator), for at
    least `LOCKSTEP_MIN_PROBES` float32 or float64 probes."""
    alg = getattr(integrand, "alg", None)
    if not isinstance(alg, _TridiagFull) or not alg.alg.custom_vjp:
        return False
    op = alg.alg.op
    return (type(op).__name__ == "SparseOperator" and op.shape[0] == op.shape[1]
            and len(probes) >= LOCKSTEP_MIN_PROBES and probes.dtype in (np.float32, np.float64))  # fmt: skip


def _slq_batch(integrand, coefs, scales, with_grad, total, dH):
    """Adds `||v0||^2 e1^T f(T) e1` (`lanczos.py:25,59`) of each run of a batch to `total`, in run order, and returns
    the sum; with `with_grad`, `dH[b]` receives run b's cotangent of `H`.  `coefs[b]` is run b's `(diag, off_diag)`,
    `scales[b]` its `||v0||`."""
    for b, ((diag, off), scale) in enumerate(zip(coefs, scales)):
        g, dalpha, dbeta, _ = _quadform_and_cotangents(integrand.matfun, integrand.matfun_grad, diag, off, with_grad)
        s2 = scale**2
        total += s2 * g
        if with_grad:
            dH[b] = synthetic.slq_cotangent_dH(s2 * dalpha, s2 * dbeta, dH.dtype)
    return total


def probe_lockstep_sum(integrand, probes, parameters, *, with_grad, batch=None, lanes=None):
    """Sum over the rows of `probes (P, n)` of the SLQ integrand (and of its parameter gradient) on a sparse
    operand, the runs advancing in LOCKSTEP batches of `batch` probes (`plan.BatchedTridiagAdjointPlan`): per Krylov
    step one multi-vector SpMV -- the operand's values and indices are read once for the whole batch -- and one
    Gram-Schmidt step kernel whose grid-wide reductions serve all runs of the batch.  `lanes` batches are in flight
    on separate streams, so the host's `eigh` of one batch (`lanczos.py:48-59`) overlaps the other's kernels.  Same
    numbers as a loop of `integrand.value_and_grad` (`jax.vmap(integrand)`, hutchinson.py:14) up to summation
    order."""
    from experiments_lanczos_adjoints_b200 import plan as _plan

    if type(probes).__name__ != "LazyProbes":  # lazily drawn probes are materialised one batch at a time
        probes = np.asarray(probes)
    P, n = probes.shape
    dtype = np.dtype(probes.dtype)
    hess = integrand.alg.alg
    K = hess.K
    if not isinstance(K, (int, np.integer)) or K < 1 or K > n:
        raise ValueError(f"Parameter depth {K} is outside the expected range")
    B = max(1, min(batch or LOCKSTEP_BATCH, P))
    starts = list(range(0, P, B))
    L = max(1, min(lanes or LOCKSTEP_LANES, len(starts)))
    cache = integrand.__dict__.setdefault("_lockstep_plans", {})
    key = (L, B, dtype.str, n, K)
    if key not in cache:
        ops = [hess.op] + [hess.op.clone() for _ in range(L - 1)]
        cache[key] = ([_plan.BatchedTridiagAdjointPlan(o, K, dtype, B, stream=dev.Stream()) for o in ops],
                      _plan.PinnedBuffers([(B, n)] * len(ops), dtype))  # fmt: skip
    plans, staging = cache[key]  # per lane: the plan and a pinned buffer its normalised probes are copied from
    host_params = [p.numpy() if isinstance(p, dev.DeviceArray) else np.asarray(p) for p in parameters]
    dev.synchronize()  # the lanes' streams start after whatever the caller enqueued
    for pl in plans:
        pl.set_params(*host_params)
    total = 0.0
    used = [False] * L
    pending = [None] * L  # per lane: (scales, number of real probes) of the batch whose forward is enqueued

    def complete(li):
        nonlocal total
        scales, real = pending[li]
        pending[li] = None
        pl = plans[li]
        coefs, symmetric = pl.coefficients()  # synchronises this lane only
        if not symmetric and integrand.alg.assume_symmetric is None:
            warnings.warn("tridiag(reortho='full'): the operand is not symmetric on this Krylov space; the adjoint "
                          "runs the general Arnoldi loops, as the reference does.", stacklevel=3)  # fmt: skip
        dH = np.zeros((B, K, K), dtype)
        total = _slq_batch(integrand, coefs[:real], scales, with_grad, total, dH)
        if with_grad:
            pl.set_cotangents(dH)  # padding runs of a short last batch carry a zero cotangent: no contribution
            pl.adjoint(zero=not used[li], export=False,
                       general=not symmetric and integrand.alg.assume_symmetric is None)
            used[li] = True

    # two batches in flight: one block per SM and kernel, so that a block of each lane is resident on every SM and one
    # lane streams while the other sits in a grid-wide reduction (measured 4983 -> 5411 Krylov steps/s at n = 1M)
    bps = dev.blocks_per_sm(1 if L >= 2 else dev.get_blocks_per_sm())
    bps.__enter__()
    try:
        for gi, start in enumerate(starts):
            li = gi % L
            group = np.asarray(probes[start : start + B])  # (drawn now, while the other lane's kernels run)
            if pending[li] is not None:
                complete(li)
            real = len(group)
            if real < B:  # short last batch: repeat its last probe (zero cotangent, value ignored)
                group = np.concatenate([group, np.repeat(group[-1:], B - real, axis=0)])
            # lanczos.py:25: the norm accumulated in float64, the division in the working precision (as the reference's);
            # the lane's previous copy out of `staging[li]` finished before its coefficients were read (complete)
            scales = np.sqrt(np.einsum("ij,ij->i", group, group, dtype=np.float64))
            np.divide(group, scales.astype(dtype)[:, None], out=staging[li])
            plans[li].set_vectors(staging[li])
            plans[li].forward()
            pending[li] = (scales, real)
        for li in range(L):
            if pending[li] is not None:
                complete(li)
    finally:
        for pl in plans:
            pl.stream.synchronize()
        bps.__exit__(None, None, None)
    return total, (_lane_grad_sum(plans, used, dtype) if with_grad else None), P


def _lane_grad_sum(plans, used, dtype):
    """Exports the parameter cotangent each used lane accumulated in its operator and returns the sum over lanes."""
    active = [pl for pl, u in zip(plans, used) if u]
    for pl in active:
        pl.export_grads()
        pl.stream.synchronize()
    stream = dev.default_stream()
    grads = []
    for gi in range(len(active[0].grads)):
        acc = dev.DeviceArray(active[0].grads[gi].shape, dtype)
        _lib.call("bl_vec_axpby", dev.dtype_code(dtype), acc.size, 1.0, active[0].grads[gi].ptr, 0.0, None, acc.ptr, stream.ptr)
        for pl in active[1:]:
            _lib.call("bl_vec_axpby", dev.dtype_code(dtype), acc.size, 1.0, acc.ptr, 1.0, pl.grads[gi].ptr, acc.ptr, stream.ptr)
        grads.append(acc)
    stream.synchronize()
    return grads


def probe_batch_sum(integrand, probes, parameters, *, with_grad, stream=None, chunk=16):
    """Sum over the rows of `probes (P, n)` of the SLQ integrand (and of its parameter gradient), with the P
    Lanczos runs advancing in lockstep (`bl_arnoldi_{forward,adjoint}_batch`): one batched matvec per step
    for all probes and one batched parameter-cotangent pass per chunk.  Same numbers as P calls of
    `integrand.value_and_grad` (`jax.vmap(integrand)`, hutchinson.py:14)."""
    stream = stream or dev.default_stream()
    probes = np.asarray(probes)
    P, n = probes.shape
    dtype = probes.dtype
    hess = integrand.alg.alg  # HessenbergEstimate
    op, K = hess.op, hess.K
    if not isinstance(K, (int, np.integer)) or K < 1 or K > n:
        raise ValueError(f"Parameter depth {K} is outside the expected range")
    bound = op.bind(parameters, dtype, stream)
    ld = dev.basis_ld(n, dtype)
    code = dev.dtype_code(dtype)
    per = _lib.load().bl_arnoldi_workspace_bytes(n, K, code)
    total, grads = 0.0, None
    if with_grad:
        op.grad_zero(dtype, stream)
    for p0 in range(0, P, chunk):
        vs = probes[p0 : p0 + chunk]
        B = len(vs)
        scale = np.linalg.norm(vs.astype(np.float64), axis=1)  # lanczos.py:25
        U = dev.asarray(np.ascontiguousarray((vs / scale[:, None]).astype(dtype)))
        Q = dev.DeviceArray((B * K, n), dtype, ld=ld)
        H = dev.DeviceArray((B, K * K), dtype)
        r = dev.DeviceArray((B, n), dtype, ld=ld)
        c = dev.DeviceArray((B,), dtype)
        ws = dev.DeviceArray(((per * B + 7) // 8,), np.float64)
        _lib.call("bl_arnoldi_forward_batch", op._handle, code, n, K, arnoldi.forward_flags(True, True), B, U.ptr, n, Q.ptr, ld, H.ptr, r.ptr, c.ptr,
                  ws.ptr, per * B, stream.ptr)  # fmt: skip
        Hh = H.numpy(stream).reshape(B, K, K)
        coefs = [(np.diag(T, 0), np.diag(T, 1)) for T in 0.5 * (Hh + Hh.transpose(0, 2, 1))]  # lanczos.py:162
        dH = np.zeros((B, K, K), dtype=dtype)
        total = _slq_batch(integrand, coefs, scale, with_grad, total, dH)
        if with_grad:
            dHd = dev.asarray(dH.reshape(B, K * K))
            dv = dev.DeviceArray((B, n), dtype, ld=ld)
            Lam = dev.DeviceArray((B * K, n), dtype, ld=ld)
            _lib.call("bl_arnoldi_adjoint_batch", op._handle, code, n, K, arnoldi.adjoint_flags(True, True, True), B, Q.ptr, ld, H.ptr, r.ptr, c.ptr, None, dHd.ptr,
                      None, None, dv.ptr, ld, Lam.ptr, ws.ptr, per * B, stream.ptr)  # fmt: skip
            stream.synchronize()  # the buffers of this chunk go back to the pool
    if with_grad:
        grads = op.grad_export(dtype, stream=stream)
    del bound
    return total, grads, P


def _flat(v0):
    v0 = dev.asarray(v0)
    if v0.ndim != 1:  # ravel_pytree of a single array (lanczos.py:24)
        v0 = dev.DeviceArray((v0.size,), v0.dtype, owner=v0._owner, ptr=v0.ptr)
    return v0


def integrand_spd(matfun, krylov_depth, matvec, /, *, reortho: str = "full", use_adjoints_for_tridiag: bool = True,
                  matfun_grad=None):
    """Drop-in for `lanczos.integrand_spd` (`/root/reference/src/matfree_extensions/lanczos.py:14-61`):
    `quadform(v0, *parameters) -> ||v0||^2 e1^T f(T) e1`.  `matfun` acts on NumPy arrays
    (`np.log`, ...); its derivative defaults to the complex-step rule (`matfun_grad` overrides)."""
    return _IntegrandSPD(matfun, krylov_depth, matvec, reortho, use_adjoints_for_tridiag, matfun_grad)


class _IntegrandSPDReuse:
    def __init__(self, matfun, order, op, reortho, matfun_grad):
        self.matfun, self.matfun_grad, self.op = matfun, matfun_grad, op
        self.alg = tridiag(op, order, custom_vjp=False, reortho=reortho)  # lanczos.py:97

    def value_and_grad(self, v0, *parameters, stream=None, want_dv0=True):
        stream = stream or dev.default_stream()
        v0 = _flat(v0)
        scale = np.sqrt(device_dot(v0, v0, stream))
        u = device_axpby(1.0 / scale, v0, 0.0, None, stream)
        (basis, (diag, off)), _ = self.alg(u, *parameters, stream=stream)
        value, _, _, (w, U) = _quadform_and_cotangents(self.matfun, self.matfun_grad, diag, off, False)
        dfw = np.asarray((self.matfun_grad or (lambda x: _matfun_derivative(self.matfun, x)))(w))
        sol = U @ (dfw * U[0])  # lanczos.py:112-113
        # w1 = scale^2 * basis.T @ sol  (lanczos.py:114): a combination of basis rows
        K, n, dtype = basis.shape[0], basis.shape[1], basis.dtype
        w1 = dev.DeviceArray((n,), dtype)
        coef = np.ascontiguousarray(scale**2 * sol, dtype=np.float64)
        ws, nbytes = _vec_ws()
        _lib.call("bl_rows_combine", dev.dtype_code(dtype), n, K, basis.ptr, basis.ld, coef.ctypes.data, 0,
                  w1.ptr, ws.ptr, nbytes, stream.ptr)  # fmt: skip
        stream.synchronize()
        # gradient of  theta -> <w1, A(w2; theta)>  (lanczos.py:121), dv0 := 0 (lanczos.py:130-134)
        op = self.op
        op.grad_zero(dtype, stream)
        op.vjp(u, w1, want_z=False, stream=stream)
        grads = op.grad_export(dtype, stream=stream)
        warnings.warn("Todo: implement gradient wrt v correctly", stacklevel=1)  # lanczos.py:127-128
        dv0 = dev.zeros((n,), dtype) if want_dv0 else None
        return diag.dtype.type(scale**2 * value), (dv0, *grads)

    def __call__(self, v0, *parameters, stream=None):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return self.value_and_grad(v0, *parameters, stream=stream, want_dv0=False)[0]


def integrand_spd_custom_vjp_reuse(matfun, order, matvec, /, *, reortho: str = "full", matfun_grad=None):
    """Drop-in for `lanczos.integrand_spd_custom_vjp_reuse` (`lanczos.py:64-139`)."""
    arnoldi._require_operator(matvec)
    return _IntegrandSPDReuse(matfun, order, matvec, reortho, matfun_grad)
