"""Matvec back-ends: device-resident operators that stand in for the reference's
user-supplied `matvec(v, *params)` callable.

The reference accepts any JAX-traceable callable and differentiates it with `jax.vjp`
(`/root/reference/src/matfree_extensions/arnoldi.py:207-209`).  Without a tracing compiler the
host layer recognises operator objects instead; each one is also a plain callable
`op(v, *params) -> A(v; params)` so code written against the reference reads the same.
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from experiments_lanczos_adjoints_b200 import _lib
from experiments_lanczos_adjoints_b200 import device as dev


class Operator:
    """Base class: owns a `bl_operator_t*`."""

    def __init__(self, handle: int, n: int):
        self._handle = handle
        self.n = int(n)
        self._bound = None  # (dtype code, [DeviceArray params]) kept alive while bound

    def __del__(self):
        h, self._handle = getattr(self, "_handle", None), None
        if h:
            try:
                _lib.load().bl_op_destroy(h)
            except Exception:
                pass

    # -- parameters ------------------------------------------------------------------
    @property
    def num_params(self) -> int:
        n = C.c_int(0)
        _lib.call("bl_op_num_params", self._handle, C.byref(n))
        return n.value

    def param_shapes(self):
        out = []
        for i in range(self.num_params):
            numel = C.c_int64(0)
            _lib.call("bl_op_param_size", self._handle, i, C.byref(numel))
            out.append((numel.value,))
        return out

    def bind(self, params, dtype, stream=None):
        """`set_params`: upload (if needed) and bind parameter values, reference order."""
        stream = stream or dev.default_stream()
        shapes = self.param_shapes()
        if len(params) != len(shapes):
            raise TypeError(f"operator takes {len(shapes)} parameter array(s), got {len(params)}")
        arrays = []
        for p, shape in zip(params, shapes):
            numel = int(np.prod(shape, dtype=np.int64))
            a = dev.asarray(p, dtype=dtype)
            if a.size != numel:
                raise ValueError(f"parameter has {a.size} elements, expected {numel}")
            arrays.append(a)
        ptrs = (C.c_void_p * max(1, len(arrays)))(*[a.ptr for a in arrays])
        _lib.call("bl_op_set_params", self._handle, dev.dtype_code(dtype), ptrs, len(arrays), stream.ptr)
        self._bound = (np.dtype(dtype), arrays)
        return arrays

    # -- the two maps ----------------------------------------------------------------
    def matvec(self, x: dev.DeviceArray, out: dev.DeviceArray | None = None, stream=None):
        stream = stream or dev.default_stream()
        out = out if out is not None else dev.empty(x.shape, x.dtype)
        _lib.call("bl_op_matvec", self._handle, dev.dtype_code(x.dtype), x.ptr, out.ptr, stream.ptr)
        return out

    def vjp(self, q: dev.DeviceArray, lam: dev.DeviceArray, want_z=True, stream=None):
        """`z = A^T lam`; the parameter cotangent accumulates inside the operator."""
        stream = stream or dev.default_stream()
        z = dev.empty(q.shape, q.dtype) if want_z else None
        _lib.call("bl_op_vjp", self._handle, dev.dtype_code(q.dtype), q.ptr, lam.ptr,
                  z.ptr if z is not None else None, stream.ptr)  # fmt: skip
        return z

    def grad_zero(self, dtype, stream=None):
        _lib.call("bl_op_grad_zero", self._handle, dev.dtype_code(dtype), (stream or dev.default_stream()).ptr)

    def grad_export(self, dtype, like=None, stream=None):
        stream = stream or dev.default_stream()
        shapes = like if like is not None else self.param_shapes()
        outs = [dev.empty(tuple(s), dtype) for s in shapes]
        ptrs = (C.c_void_p * max(1, len(outs)))(*[o.ptr for o in outs])
        _lib.call("bl_op_grad_export", self._handle, dev.dtype_code(dtype), ptrs, len(outs), stream.ptr)
        return outs

    # -- the reference's calling convention ----------------------------------------------
    def __call__(self, v, *params):
        x = dev.asarray(v)
        self.bind(params, x.dtype)
        return self.matvec(x)


class BoundOperator:
    """`lambda v: matvec(v, *params)` — an operator with its parameters bound: what the reference hands
    to CG, to the partial Cholesky (`lazy_kernel`) and to the SLQ log-determinant as `A`."""

    def __init__(self, op: Operator, *params):
        self.op, self.params = op, tuple(params)
        self.n = op.n

    def bind(self, dtype, stream=None):
        return self.op.bind(self.params, dtype, stream)

    def __call__(self, v):
        return self.op(v, *self.params)


def bound(op, *params) -> BoundOperator:
    return BoundOperator(op, *params)


class SparseOperator(Operator):
    """`BCOO((params, indices), shape) @ x` with `params` = COO data in COO order
    (`/root/reference/experiments/benchmarks/wall_times_vjp_through_lanczos_arnoldi/suite_sparse/benchmark.py:61-68`).
    Duplicate entries are summed by the matvec and stay independent parameters."""

    def __init__(self, row, col, shape):
        row = np.ascontiguousarray(np.asarray(row, dtype=np.int32))
        col = np.ascontiguousarray(np.asarray(col, dtype=np.int32))
        if row.shape != col.shape or row.ndim != 1:
            raise ValueError("row and col must be 1-D arrays of equal length")
        self.shape = (int(shape[0]), int(shape[1]))
        self.nnz = int(row.size)
        self._coo = (row, col)  # kept for `clone()`
        h = C.c_void_p()
        _lib.call("bl_op_sparse_create", self.shape[0], self.shape[1], self.nnz, row.ctypes.data,
                  col.ctypes.data, C.byref(h))  # fmt: skip
        super().__init__(h.value, self.shape[0])

    def clone(self):
        """A second handle on the same sparsity pattern with its own values and cotangent accumulator: independent
        Krylov runs (probes) on different streams need one operator each."""
        twin = object.__new__(SparseOperator)
        twin.shape, twin.nnz, twin._coo = self.shape, self.nnz, self._coo
        h = C.c_void_p()
        _lib.call("bl_op_sparse_clone", self._handle, C.byref(h))  # the finished index work is shared, not redone
        Operator.__init__(twin, h.value, self.shape[0])
        return twin

    @classmethod
    def from_matrix_market(cls, path):
        """`exp_util.suite_sparse_load` (`/root/reference/src/matfree_extensions/util/exp_util.py:35-42`):
        returns `(operator, data)` with `data` in the order `scipy.io.mmread` produces."""
        import scipy.io

        m = scipy.io.mmread(path)
        return cls(m.row, m.col, m.shape), np.asarray(m.data)

    def export_csr(self):
        row_ptr = np.empty(self.shape[0] + 1, np.int32)
        col_idx = np.empty(self.nnz, np.int32)
        perm = np.empty(self.nnz, np.int32)
        _lib.call("bl_op_sparse_export_csr", self._handle, row_ptr.ctypes.data, col_idx.ctypes.data, perm.ctypes.data)
        return row_ptr, col_idx, perm

    def export_sell(self, transpose=False):
        rows = self.shape[1] if transpose else self.shape[0]
        slice_ptr = np.empty((rows + 31) // 32 + 1, np.int64)
        slot = np.empty(self.nnz, np.int64)
        _lib.call("bl_op_sparse_export_sell", self._handle, int(transpose), slice_ptr.ctypes.data, slot.ctypes.data)
        return slice_ptr, slot


class DenseOperator(Operator):
    """`lambda s, p: p @ s` (`sym=False`) or `lambda s, p: (p + p.T) @ s` (`sym=True`): the operands
    of the reference's unit tests (`/root/reference/tests/test_lanczos/test_tridiag_adjoint.py:20-21`)."""

    def __init__(self, n, sym=False):
        h = C.c_void_p()
        _lib.call("bl_op_dense_create", int(n), int(bool(sym)), C.byref(h))
        super().__init__(h.value, n)
        self.sym = bool(sym)

    def param_shapes(self):
        return [(self.n, self.n)]

    def bind(self, params, dtype, stream=None):
        params = [np.asarray(p).reshape(-1) if not isinstance(p, dev.DeviceArray) else p for p in params]
        return super().bind(params, dtype, stream)

    def grad_export(self, dtype, like=None, stream=None):
        (g,) = super().grad_export(dtype, like=[(self.n * self.n,)], stream=stream)
        return [dev.DeviceArray((self.n, self.n), dtype, owner=g._owner, ptr=g.ptr)]


class GramOperator(Operator):
    """Matrix-free `(K(X, X) + noise I) v` for the scaled Matérn-3/2 / Matérn-1/2 / RBF kernels of
    `/root/reference/src/matfree_extensions/util/gp_util.py:69-184` (Gram matvec `:525-543`).
    Parameters, in order: `raw_lengthscale (d,)`, `raw_outputscale ()`, `noise ()`."""

    KINDS = {"matern32": 0, "matern12": 1, "rbf": 2}
    PATHS = {"auto": 0, "alu": 1, "tensor": 2}

    def __init__(self, X, kind="matern32", path="auto"):
        """`path`: which kernel evaluates the pairwise distances in fp32 -- "tensor" (tcgen05, TF32
        hi/lo split operands), "alu" (FP32 pipes) or "auto" (tensor cores when d <= 20)."""
        X = np.ascontiguousarray(np.asarray(X, dtype=np.float64))
        if X.ndim != 2:
            raise ValueError("X must be (n, d)")
        self.d = int(X.shape[1])
        h = C.c_void_p()
        _lib.call("bl_op_gram_create", X.shape[0], X.shape[1], self.KINDS[kind], X.ctypes.data, C.byref(h))
        super().__init__(h.value, X.shape[0])
        if path != "auto":
            _lib.call("bl_op_gram_set_path", self._handle, self.PATHS[path])

    def tile_distances(self, row_tile=0, col_tile=0, stream=None):
        """Diagnostic: the tensor-core accumulator `x_i.x_j - |x_j|^2 / 2` (scaled inputs) of one
        128 x 256 tile (after `bind`); `s2_ij = |x_i|^2 - 2 acc_ij`."""
        out = np.empty((128, 256), dtype=np.float32)
        s = stream or dev.default_stream()
        _lib.call("bl_op_gram_tile_distances", self._handle, int(row_tile), int(col_tile), out.ctypes.data, s.ptr)
        return out

    def param_shapes(self):
        return [(self.d,), (), ()]

    def bind(self, params, dtype, stream=None):
        params = [np.atleast_1d(np.asarray(p)) if not isinstance(p, dev.DeviceArray) else p for p in params]
        return super().bind(params, dtype, stream)

    def grad_export(self, dtype, like=None, stream=None):
        return super().grad_export(dtype, like=[(self.d,), (1,), (1,)], stream=stream)

    def cross(self, X_test):
        """The cross-covariance `K(X_test, X)` with this operator's kernel (see `GramCross`)."""
        return GramCross(self, X_test)


def check_test_inputs(X_test, d: int) -> np.ndarray:
    """`X_test` as a C-contiguous (M, d) float64 array; `ValueError` for another shape, no points or a
    non-finite entry."""
    X_test = np.ascontiguousarray(np.asarray(X_test, dtype=np.float64))
    if X_test.ndim != 2 or X_test.shape[1] != d:
        raise ValueError(f"X_test must be (M, {d}), got shape {X_test.shape}")
    if X_test.shape[0] == 0:
        raise ValueError("X_test has no points")
    if not np.all(np.isfinite(X_test)):
        raise ValueError("X_test has non-finite entries")
    return X_test


class GramCross:
    """Cross-covariance of a `GramOperator` with `M` test points: `matvec(v) = K(X*, X) v` (M values),
    `columns(first, count)` the rows `k(x*_t, X)` of `count` test points as a `(count, n)` device array (row
    stride 16-byte aligned), `prior_diag()` = `k(x*_t, x*_t)` (the kernel formula at zero distance, so
    `sigma (1 + sqrt(eps)) e^-sqrt(eps)` for Matérn-3/2).  Every call uses the kernel parameters the parent
    operator was last bound with, in that dtype (bind it first); the noise is never read.

    fp32 on the tensor-core path: `s2 = |x|^2 + |y|^2 - 2 x.y` is exact only on the square operator's diagonal,
    where it is forced to zero.  A test point that coincides with a training point gets `s2 = O(eps |x|^2)`
    instead of 0, which the Matérn square root magnifies; such points need fp64."""

    def __init__(self, gram: GramOperator, X_test):
        X_test = check_test_inputs(X_test, gram.d)
        self.parent, self.m, self.n = gram, int(X_test.shape[0]), gram.n
        h = C.c_void_p()
        _lib.call("bl_gram_cross_create", gram._handle, self.m, X_test.ctypes.data, C.byref(h))
        self._handle = h.value

    def __del__(self):
        h, self._handle = getattr(self, "_handle", None), None
        if h:
            try:
                _lib.load().bl_gram_cross_destroy(h)
            except Exception:
                pass

    def _dtype(self):
        if self.parent._bound is None:
            raise RuntimeError("bind the parent GramOperator first")
        return self.parent._bound[0]

    def matvec(self, v, stream=None):
        stream = stream or dev.default_stream()
        v = dev.asarray(v, dtype=self._dtype())
        if v.shape != (self.n,):
            raise ValueError(f"v must have {self.n} entries, got shape {v.shape}")
        out = dev.empty((self.m,), v.dtype)
        _lib.call("bl_gram_cross_matvec", self._handle, dev.dtype_code(v.dtype), v.ptr, out.ptr, stream.ptr)
        return out

    def columns(self, first, count, stream=None):
        first, count = int(first), int(count)
        if first < 0 or count < 1 or first + count > self.m:
            raise ValueError(f"columns [{first}, {first + count}) out of range for {self.m} test points")
        dtype = self._dtype()
        out = dev.empty((count, self.n), dtype, ld=dev.basis_ld(self.n, dtype))
        _lib.call("bl_gram_cross_columns", self._handle, dev.dtype_code(dtype), first, count, out.ptr, out.ld,
                  (stream or dev.default_stream()).ptr)  # fmt: skip
        return out

    def prior_diag(self, stream=None):
        dtype = self._dtype()
        out = dev.empty((self.m,), dtype)
        _lib.call("bl_gram_cross_prior_diag", self._handle, dev.dtype_code(dtype), out.ptr,
                  (stream or dev.default_stream()).ptr)  # fmt: skip
        return out


class WaveStencilOperator(Operator):
    """`(u, du) -> (du, scale^2 * conv3x3(stencil, edge_pad(u)))` on a `g x g` grid
    (`/root/reference/src/matfree_extensions/util/pde_util.py:126-157`).  Parameter: `scale (g, g)`."""

    def __init__(self, grid, stencil, *, rows=None, has_top=False, has_bottom=False):
        """`rows` (with `has_top` / `has_bottom`) builds the row-sharded form: a slab of `rows` grid
        rows x `grid` columns whose neighbours' boundary rows arrive through halo buffers
        (`parallel.RowShardedWaveOperator`)."""
        st = np.ascontiguousarray(np.asarray(stencil, dtype=np.float64))
        if st.shape != (3, 3):
            raise ValueError("stencil must be 3 x 3")
        self.g = int(grid)
        self.rows = self.g if rows is None else int(rows)
        h = C.c_void_p()
        _lib.call("bl_op_wave_slab_create", self.rows, self.g, int(bool(has_top)), int(bool(has_bottom)),
                  st.ctypes.data, C.byref(h))  # fmt: skip
        super().__init__(h.value, 2 * self.rows * self.g)

    def halo_ptr(self, which: int) -> int:
        p = C.c_void_p()
        _lib.call("bl_op_wave_halo", self._handle, int(which), C.byref(p))
        return p.value

    @staticmethod
    def stencil_laplacian(dx):
        """`pde_util.stencil_laplacian` (`pde_util.py:18-20`), centre weight -2 as in the reference."""
        return np.asarray([[0.0, 1.0, 0.0], [1.0, -2.0, 1.0], [0.0, 1.0, 0.0]]) / dx**2

    def param_shapes(self):
        return [(self.rows, self.g)]

    def bind(self, params, dtype, stream=None):
        params = [np.asarray(p).reshape(-1) if not isinstance(p, dev.DeviceArray) else p for p in params]
        return super().bind(params, dtype, stream)

    def grad_export(self, dtype, like=None, stream=None):
        (g,) = super().grad_export(dtype, like=[(self.rows * self.g,)], stream=stream)
        return [dev.DeviceArray((self.rows, self.g), dtype, owner=g._owner, ptr=g.ptr)]


class CallbackOperator(Operator):
    """An arbitrary user matvec written against `DeviceArray`s.

    `matvec_fn(x, *params) -> y` and `vjp_fn(q, lam, *params) -> (z, (dparam, ...))` receive and
    return `DeviceArray`s and must enqueue their work on `device.default_stream()`; parameter
    cotangents returned by `vjp_fn` are accumulated here on the host side."""

    def __init__(self, n, matvec_fn, vjp_fn=None, num_params=0):
        self._mv, self._vj = matvec_fn, vjp_fn
        self._nparams = int(num_params)
        self._params = []
        self._grads = None
        self._error = None

        def mv_cb(_user, dtype, x, y, stream):
            try:
                dt = np.float32 if dtype == _lib.BL_F32 else np.float64
                xin = dev.DeviceArray((n,), dt, ptr=x, owner=self)
                out = self._mv(xin, *self._params)
                _lib.call("bl_memcpy_d2d", y, out.ptr, n * np.dtype(dt).itemsize, stream)
                return 0
            except Exception as exc:  # surfaced by the caller
                self._error = exc
                return 1

        def vj_cb(_user, dtype, q, lam, z, stream):
            try:
                dt = np.float32 if dtype == _lib.BL_F32 else np.float64
                qin = dev.DeviceArray((n,), dt, ptr=q, owner=self)
                lin = dev.DeviceArray((n,), dt, ptr=lam, owner=self)
                zz, dps = self._vj(qin, lin, *self._params)
                if z:
                    _lib.call("bl_memcpy_d2d", z, zz.ptr, n * np.dtype(dt).itemsize, stream)
                dps = [np.asarray(d) for d in dps]
                self._grads = dps if self._grads is None else [g + d for g, d in zip(self._grads, dps)]
                return 0
            except Exception as exc:
                self._error = exc
                return 1

        self._mv_c = _lib.MATVEC_CB(mv_cb)
        self._vj_c = _lib.VJP_CB(vj_cb) if vjp_fn is not None else C.cast(None, _lib.VJP_CB)
        h = C.c_void_p()
        _lib.call("bl_op_callback_create", int(n), self._mv_c, self._vj_c, None, C.byref(h))
        super().__init__(h.value, n)

    @property
    def num_params(self):
        return self._nparams

    def param_shapes(self):
        return [np.shape(p) for p in self._params]

    def bind(self, params, dtype, stream=None):
        if len(params) != self._nparams:
            raise TypeError(f"operator takes {self._nparams} parameter array(s), got {len(params)}")
        self._params = list(params)
        return self._params

    def grad_zero(self, dtype, stream=None):
        self._grads = None

    def grad_export(self, dtype, like=None, stream=None):
        return list(self._grads or [])
