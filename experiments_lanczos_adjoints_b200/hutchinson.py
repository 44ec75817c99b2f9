"""Hutchinson / stochastic-Lanczos-quadrature estimators.

Host-side mirror of `/root/reference/src/matfree_extensions/hutchinson.py` plus the
`matfree.hutchinson.hutchinson` / `sampler_rademacher` pair the reference imports
(`/root/reference/src/matfree_extensions/util/gp_util.py:8,557`).  An estimator is
`sample(key, *parameters)`; `sample_fun(key)` returns the `(num, n)` probe matrix.  Probe
vectors are independent Lanczos runs, which `probe_sum` sums in one of three ways: lockstep
batches on a sparse operand (`lanczos.probe_lockstep_sum`, at least `lanczos.LOCKSTEP_MIN_PROBES`
probes), lockstep runs on the Gram operator, which shares work between vectors
(`lanczos.probe_batch_sum`), and one probe after the other otherwise (`probe_loop_sum`).
`parallel.hutchinson_sharded` shards the probes over GPUs.

PRNG note: JAX's threefry stream cannot be reproduced without JAX.  `sampler_rademacher` /
`sampler_normal` / `split` here are NumPy-based; parity tests always pass probes explicitly.
"""

from __future__ import annotations

import numpy as np

from experiments_lanczos_adjoints_b200 import device as dev


# ---- keys and samplers (NumPy stand-ins for jax.random) -----------------------------------
def prng_key(seed: int):
    return np.random.SeedSequence(int(seed))


def split(key, num: int = 2):
    """`jax.random.split` stand-in: `num` independent child keys."""
    if not isinstance(key, np.random.SeedSequence):
        key = np.random.SeedSequence(int(np.asarray(key).sum()))
    # a pure function of the key (SeedSequence.spawn is stateful): same key -> same children
    return [np.random.SeedSequence(entropy=key.entropy, spawn_key=tuple(key.spawn_key) + (i,)) for i in range(num)]


def _generator(key):
    if isinstance(key, np.random.Generator):
        return key
    if not isinstance(key, np.random.SeedSequence):
        key = np.random.SeedSequence(int(np.asarray(key).sum()))
    return np.random.default_rng(key)


def sampler_rademacher(x_like, /, *, num: int):
    """`matfree.hutchinson.sampler_rademacher(x_like, num=)`: `(num, n)` entries +-1."""
    n, dtype = int(np.size(x_like)), np.asarray(x_like).dtype

    def sample(key):
        return (_generator(key).integers(0, 2, size=(num, n)) * 2 - 1).astype(dtype)

    return sample


def sampler_normal(x_like, /, *, num: int):
    n, dtype = int(np.size(x_like)), np.asarray(x_like).dtype

    def sample(key):
        return _generator(key).standard_normal((num, n)).astype(dtype)

    return sample


# ---- estimators ------------------------------------------------------------------------------
def _probe_rows(samples):
    if isinstance(samples, dev.DeviceArray):
        if samples.ndim == 1:
            return [samples]
        return [samples.row(i) for i in range(samples._shape[0])]
    samples = np.asarray(samples)
    return list(samples.reshape(1, -1) if samples.ndim == 1 else samples)


def _mean(values):
    return np.mean(np.stack([np.asarray(v) for v in values]), axis=0)


def _resident(parameters, like):
    """Upload host parameter arrays once per estimate (not once per probe)."""
    dtype = like.dtype if hasattr(like, "dtype") else np.asarray(like).dtype
    if np.dtype(dtype) not in (np.dtype(np.float32), np.dtype(np.float64)):
        return parameters
    out = []
    for p in parameters:
        if isinstance(p, np.ndarray) and p.dtype.kind == "f" and p.ndim >= 1 and p.size >= 4096:
            p = dev.asarray(p.reshape(-1) if p.ndim > 1 else p, dtype=dtype) if p.ndim == 1 else p
        out.append(p)
    return tuple(out)


def probe_sum(integrand_fun, samples, parameters, *, with_grad=False):
    """Sum (not mean) of the integrand over probes, `(total, grads, count)`; gradients stay on the device."""
    from experiments_lanczos_adjoints_b200 import lanczos

    lazy = type(samples).__name__ == "LazyProbes"  # rows drawn on demand (parallel.sharded_sampler)
    matrix = (isinstance(samples, np.ndarray) or lazy) and samples.ndim == 2 and len(samples) > 1
    if matrix and lanczos._lockstep_eligible(integrand_fun, samples):  # lazy probes are drawn one batch at a time
        return lanczos.probe_lockstep_sum(integrand_fun, samples, parameters, with_grad=with_grad)
    if lazy:
        samples = np.asarray(samples)
    if matrix and samples.dtype in (np.float32, np.float64) and lanczos._batch_eligible(integrand_fun, samples.dtype):
        return lanczos.probe_batch_sum(integrand_fun, samples, parameters, with_grad=with_grad)
    return probe_loop_sum(integrand_fun, samples, parameters, with_grad=with_grad)


def probe_loop_sum(integrand_fun, samples, parameters, *, with_grad):
    """`probe_sum` one probe at a time (`jax.vmap(integrand)`, hutchinson.py:14): the path of every integrand the
    batched sums do not take, and their reference in tests."""
    total, grads, count = 0.0, None, 0
    rows = _probe_rows(samples)
    if len(rows):
        parameters = _resident(parameters, rows[0])
    for vec in rows:
        if with_grad:
            val, (_dv0, *dp) = integrand_fun.value_and_grad(vec, *parameters, want_dv0=False)
            if grads is None:
                grads = [_Accum(d) for d in dp]
            else:
                for g, d in zip(grads, dp):
                    g.add(d)
        else:
            val = integrand_fun(vec, *parameters)
        total = total + np.asarray(val, dtype=np.float64)
        count += 1
    return total, ([g.value for g in grads] if grads else None), count


class _Accum:
    """Running sum of per-probe gradients (device axpby when the gradient is a DeviceArray)."""

    def __init__(self, first):
        self.value = first

    def add(self, other):
        if isinstance(self.value, dev.DeviceArray):
            from experiments_lanczos_adjoints_b200 import _lib

            _lib.call("bl_vec_axpby", dev.dtype_code(self.value.dtype), self.value.size, 1.0, self.value.ptr,
                      1.0, other.ptr, self.value.ptr, dev.default_stream().ptr)  # fmt: skip
        else:
            self.value = self.value + other


def _scale(g, factor):
    if isinstance(g, dev.DeviceArray):
        from experiments_lanczos_adjoints_b200 import _lib

        _lib.call("bl_vec_axpby", dev.dtype_code(g.dtype), g.size, float(factor), g.ptr, 0.0, None, g.ptr,
                  dev.default_stream().ptr)  # fmt: skip
        return g
    return g * factor


class _Estimator:
    def __init__(self, integrand_fun, sample_fun):
        self.integrand_fun, self.sample_fun = integrand_fun, sample_fun

    def __call__(self, key, *parameters):
        total, _, count = probe_sum(self.integrand_fun, self.sample_fun(key), parameters)
        return total / count  # mean over probes (hutchinson.py:54)

    def value_and_grad(self, key, *parameters):
        """`jax.value_and_grad(estimate, argnums=(1, ...))`: probes are constants."""
        total, grads, count = probe_sum(self.integrand_fun, self.sample_fun(key), parameters, with_grad=True)
        return total / count, tuple(_scale(g, 1.0 / count) for g in grads)


def hutchinson(integrand_fun, /, sample_fun):
    """`matfree.hutchinson.hutchinson` == the reference's `_sample` (`hutchinson.py:51-54`)."""
    return _Estimator(integrand_fun, sample_fun)


def hutchinson_nograd(integrand_fun, /, sample_fun):
    """`hutchinson.hutchinson_nograd` (`hutchinson.py:8-17`): gradients never flow into the probes
    — true of every estimator here, the probes are host constants."""
    return _Estimator(integrand_fun, sample_fun)


class _CustomVJPEstimator:
    """`hutchinson.hutchinson_custom_vjp` (`hutchinson.py:20-48`): the forward pass samples with
    `key`, the backward pass with `split(key)[1]`; calling the primal outside a VJP raises."""

    def __init__(self, integrand_fun, sample_fun):
        self.integrand_fun, self.sample_fun = integrand_fun, sample_fun

    def __call__(self, _key, *_parameters):
        raise RuntimeError("oops")  # hutchinson.py:24-30

    def vjp(self, key, *parameters):
        _key_fwd, key_bwd = split(key, num=2)  # hutchinson.py:33
        total, _, count = probe_sum(self.integrand_fun, self.sample_fun(key), parameters)

        def pullback(cot):
            _, grads, cnt = probe_sum(self.integrand_fun, self.sample_fun(key_bwd), parameters, with_grad=True)
            return (None, *[_scale(g, float(cot) / cnt) for g in grads])

        return total / count, pullback


def hutchinson_custom_vjp(integrand_fun, /, sample_fun):
    return _CustomVJPEstimator(integrand_fun, sample_fun)


def hutchinson_batch(estimate_fun, /, num):
    """`hutchinson.hutchinson_batch` (`hutchinson.py:57-65`): mean of `num` estimates on split keys."""

    def estimate_b(key, *parameters):
        keys = split(key, num=num)
        return _mean([estimate_fun(k, *parameters) for k in keys])

    return estimate_b
