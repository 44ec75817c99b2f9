"""Conjugate-gradient solvers: drop-ins for `/root/reference/src/matfree_extensions/cg.py`.

    solve = cg.pcg_adaptive(atol=1e-4, rtol=0.0, maxiter=1000, miniter=10)
    x, info = solve(A, b, P)           # A = operators.bound(op, *params), P = pre.bind(noise) or None

`A` is an operator with bound parameters (the reference passes a closure), `b` a host or device vector.
The whole iteration runs on the device (`bl_pcg_solve`, `csrc/solve.cu`): step lengths, the convergence
test of `pcg_adaptive` and `_safe_divide` never touch the host; the fixed-step solver does not
synchronise at all.  `solve.vjp(A, b, P)` is the `jax.lax.custom_linear_solve` rule of `cg.py:25-27`
(symmetric A): `db = A^{-1} xbar`, `dtheta = -d<db, A(x; theta)>/dtheta`.

`vmap_solver(solve)(A, B, P)` solves for every row of `B` in lockstep (`bl_pcg_solve_batch`): what
`jax.vmap(solve, in_axes=(None, 0, None))` gives in the reference.
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from experiments_lanczos_adjoints_b200 import _lib
from experiments_lanczos_adjoints_b200 import device as dev
from experiments_lanczos_adjoints_b200.operators import BoundOperator, Operator


class _Info(dict):
    """The reference's info dict; `residual_rel = r / |x|` (`cg.py:38`) is formed on first access."""

    def __init__(self, x, **items):
        super().__init__(**items)
        self._x = x

    def __missing__(self, key):
        if key != "residual_rel":
            raise KeyError(key)
        with np.errstate(divide="ignore", invalid="ignore"):
            value = self["residual_abs"].numpy() / np.abs(self._x.numpy())
        self[key] = value
        return value


def _as_bound(A) -> BoundOperator:
    if isinstance(A, BoundOperator):
        return A
    if isinstance(A, Operator):
        return BoundOperator(A)
    raise TypeError("A must be an operator object with bound parameters (operators.bound(op, *params)); "
                    "arbitrary Python closures cannot run on the device")  # fmt: skip


class _Solver:
    def __init__(self, *, max_steps, min_steps=0, atol=-1.0, rtol=0.0, check_every=8):
        self.max_steps, self.min_steps = int(max_steps), int(min_steps)
        self.atol, self.rtol, self.check_every = float(atol), float(rtol), int(check_every)
        self._ws = None

    def _solve(self, A: BoundOperator, b: dev.DeviceArray, P, stream):
        n, dtype = b.shape[0], b.dtype
        if P is not None and not hasattr(P, "_precond_handle"):
            raise TypeError("P must be a bound low-rank preconditioner (`pre.bind(noise)`) or None")
        A.bind(dtype, stream)
        nbytes = _lib.load().bl_pcg_workspace_bytes(n, dev.dtype_code(dtype))
        if self._ws is None or self._ws.size * self._ws.dtype.itemsize < nbytes:
            self._ws = dev.DeviceArray(((nbytes + 7) // 8,), np.float64)
        x, r = dev.DeviceArray((n,), dtype), dev.DeviceArray((n,), dtype)
        steps = C.c_int64(0)
        _lib.call("bl_pcg_solve", A.op._handle, dev.dtype_code(dtype), n, b.ptr,
                  P._precond_handle() if P is not None else None, self.max_steps, self.min_steps, self.atol, self.rtol,
                  self.check_every, x.ptr, r.ptr, C.byref(steps), self._ws.ptr, nbytes, stream.ptr)  # fmt: skip
        return x, r, steps.value

    def __call__(self, A, b, P=None, *, stream=None):
        A = _as_bound(A)  # argument errors first, before any device work
        stream = stream or dev.default_stream()
        b = dev.asarray(b)
        x, r, steps = self._solve(A, b, P, stream)
        info = _Info(x, residual_abs=r)
        if self.atol >= 0.0:
            info["num_steps"] = steps
        return x, info

    def vjp(self, A, b, P=None, *, stream=None):
        A = _as_bound(A)
        stream = stream or dev.default_stream()
        b = dev.asarray(b)
        x, info = self(A, b, P, stream=stream)

        def pullback(cotangent):
            xbar = cotangent[0] if isinstance(cotangent, tuple) else cotangent
            xbar = dev.asarray(xbar, dtype=b.dtype)
            db, _, _ = self._solve(A, xbar, P, stream)  # A^{-1} xbar (A symmetric)
            A.bind(b.dtype, stream)
            A.op.grad_zero(b.dtype, stream)
            A.op.vjp(x, db, want_z=False, stream=stream)
            grads = A.op.grad_export(b.dtype, stream=stream)
            for g in grads:  # dtheta = -<db, dA x>
                _lib.call("bl_vec_axpby", dev.dtype_code(g.dtype), g.size, -1.0, g.ptr, 0.0, None, g.ptr, stream.ptr)
            return tuple(grads), db

        return (x, info), pullback


class _NoPrecond:
    """`cg_*`: the solver with `P = identity` (`cg.py:9-17, 65-72`)."""

    def __init__(self, solver):
        self._solver = solver

    def __call__(self, A, b, *, stream=None):
        return self._solver(A, b, None, stream=stream)

    def vjp(self, A, b, *, stream=None):
        return self._solver.vjp(A, b, None, stream=stream)


def pcg_fixed_step(num_matvecs: int, /):
    """`cg.pcg_fixed_step` (`cg.py:20-62`): exactly `num_matvecs` iterations."""
    return _Solver(max_steps=num_matvecs)


def cg_fixed_step(num_matvecs: int, /):
    return _NoPrecond(pcg_fixed_step(num_matvecs))


def pcg_adaptive(*, atol: float, rtol, maxiter: int, miniter: int, check_every: int = 8):
    """`cg.pcg_adaptive` (`cg.py:75-131`).  `check_every`: how often the host polls the device's
    convergence flag (the device itself tests every iteration and freezes the state when it fails)."""
    return _Solver(max_steps=maxiter, min_steps=miniter, atol=atol, rtol=rtol, check_every=check_every)


def cg_adaptive(**kwargs):
    return _NoPrecond(pcg_adaptive(**kwargs))


class _VmapSolver:
    def __init__(self, solve):
        if isinstance(solve, _NoPrecond):
            self._solver, self._takes_p = solve._solver, False
        elif isinstance(solve, _Solver):
            self._solver, self._takes_p = solve, True
        else:
            raise TypeError("vmap_solver takes a solver of this module (pcg_* / cg_*)")
        self._ws = None

    def __call__(self, A, B, P=None, *, stream=None):
        A = _as_bound(A)
        if P is not None and not self._takes_p:
            raise TypeError("a cg_* solver takes no preconditioner")
        if P is not None and not hasattr(P, "_precond_handle"):
            raise TypeError("P must be a bound low-rank preconditioner (`pre.bind(noise)`) or None")
        stream = stream or dev.default_stream()
        if not isinstance(B, dev.DeviceArray):
            B = np.asarray(B)
            if B.ndim != 2 or B.shape[1] != A.n:
                raise ValueError(f"B must be (count, {A.n}), got shape {B.shape}")
            B = dev.basis_from_host(B, B.dtype if B.dtype in (np.float32, np.float64) else np.float64)
        if B.ndim != 2 or B.shape[1] != A.n:
            raise ValueError(f"B must be (count, {A.n}), got shape {B.shape}")
        count, n = B.shape
        if B.is_transposed or (B.ld * B.dtype.itemsize) % 16:
            B = dev.basis_from_host(B.numpy(), B.dtype)
        s, dtype, ld = self._solver, B.dtype, B.ld
        A.bind(dtype, stream)
        nbytes = _lib.load().bl_pcg_batch_workspace_bytes(ld, count, dev.dtype_code(dtype))
        if self._ws is None or self._ws.size * self._ws.dtype.itemsize < nbytes:
            self._ws = dev.DeviceArray(((nbytes + 7) // 8,), np.float64)
        X, R = dev.empty((count, n), dtype, ld=ld), dev.empty((count, n), dtype, ld=ld)
        steps = np.zeros(count, np.int64)
        _lib.call("bl_pcg_solve_batch", A.op._handle, dev.dtype_code(dtype), n, count, B.ptr, ld,
                  P._precond_handle() if P is not None else None, s.max_steps, s.min_steps, s.atol, s.rtol,
                  s.check_every, X.ptr, R.ptr, steps.ctypes.data_as(C.POINTER(C.c_int64)), self._ws.ptr, nbytes,
                  stream.ptr)  # fmt: skip
        info = _Info(X, residual_abs=R)
        if s.atol >= 0.0:
            info["num_steps"] = steps
        return X, info


def vmap_solver(solve, /):
    """`jax.vmap(solve, in_axes=(None, 0, None))` for a `pcg_*` / `cg_*` solver: `vmap_solver(solve)(A, B, P=None)`
    solves `A x = b` for every row `b` of `B` (count, n) and returns `(X (count, n), info)`; the info carries the
    residuals row by row and, for the adaptive solvers, `num_steps` per row.  Each row follows exactly the rules
    of `solve`; the rows share each operator sweep (the Gram operator evaluates a kernel tile once for up to 16
    rows)."""
    return _VmapSolver(solve)
