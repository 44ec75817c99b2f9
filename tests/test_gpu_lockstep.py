"""Lockstep Arnoldi batches (`bl_arnoldi_forward_batch` / `bl_arnoldi_adjoint_batch`) run by run against the float64
oracle, through every launch grouping of the step kernel `k_step_tma`.

`launch_step` (csrc/krylov.cu) hands the Gram-Schmidt step of up to `kStepBatch` runs to one cooperative launch.  How
many runs share a launch depends on the number of active basis rows m: the per-run shared-memory blocks grow with m,
so a batch of four is split 4 -> 3 + 1 -> 2 + 2 and finally runs on the separate kernels, in the middle of a sweep.
`step_groups` below restates that rule; a CPU test pins it to the source and checks that the depths of the GPU cases
pass through every grouping.  Each GPU case counts the `k_step_tma` launches of its forward and of its adjoint
(`bl_step_trace_*`) and compares them with the rule, so a case that quietly fell back to the separate kernels fails.

For every run p of a batch the GPU cases check H, Q, r, c and dv against `oracle.krylov.arnoldi_*_active` in float64,
and the parameter cotangent of run p alone: the adjoint is repeated with run p's cotangent and `dH = 0` for the others,
whose dv must then be exactly zero.  A kernel that mixed runs would leave sums over the batch unchanged; these checks
do not.  Rows of Q and Lambda must be zero in [n, ld) (the TMA kernels rely on it), and two identical calls must
return bit-identical results (the reductions run in a fixed order).
"""

import ctypes as C
import functools
import os

import numpy as np
import pytest
from conftest import rel_err

from oracle import krylov, operators

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "experiments_lanczos_adjoints_b200", "csrc")

# ---- launch_step's grouping rule, restated from the source --------------------------------------------------------
K_STEP_BATCH = 4  # kStepBatch, csrc/step_kernel.cuh:42
K_FEW_SLOTS = 40  # kFewSlots = kFewMax * kConsumerWarps + 8 = 4 * 8 + 8, csrc/step_kernel.cuh:43
K_GROUP = 8  # kGroup, csrc/stream_kernels.cuh:24
RING_BYTES = 26 * 4096  # (kStages * kGroup + 2) 4 KB tiles: the ring and the two x tiles, csrc/krylov.cu:565
BARRIER_BYTES = 256  # (2 * kStages + 2 + 2 * step::kOpStages) * 8 with kOpStages = 12, csrc/krylov.cu:565
SMEM_LIMIT = 112 * 1024  # the opt-in of k_step_tma, csrc/krylov.cu:617
TMA_MIN_N = 8192  # use_tma, csrc/krylov.cu:101
TILE_BYTES = 4096  # one block per 4 KB row segment (tma_grid), csrc/krylov.cu:119
TRACE_LAUNCHES = 2048  # kTraceLaunches, csrc/step_kernel.cuh:106

# the source text each constant above restates (a change there must change the restatement too)
SOURCE_QUOTES = [
    ("step_kernel.cuh", "constexpr int kFewMax = 4;"),
    ("step_kernel.cuh", "constexpr int kStepBatch = 4;"),
    ("step_kernel.cuh", "constexpr int kFewSlots = kFewMax * kConsumerWarps + 8;"),
    ("step_kernel.cuh", "constexpr int kTraceLaunches = 2048;"),
    ("step_kernel.cuh", "constexpr int kOpStageBytes = 8192;"),
    ("step_kernel.cuh", "constexpr int kOpStages = kStages * kGroup * kConsumerThreads * 16 / kOpStageBytes;"),
    ("stream_kernels.cuh", "constexpr int kGroup = 8;"),
    ("stream_kernels.cuh", "constexpr int kConsumerWarps = 8;"),
    ("stream_kernels.cuh", "constexpr int kStages = 3;"),
    ("krylov.cu", "return (size_t)(kStages * kGroup + 2) * TILE * sizeof(T) + (2 * kStages + 2 + 2 * step::kOpStages) * 8 +"),
    ("krylov.cu", "(size_t)count * acc_stride * 8 + (size_t)count * coef_stride * sizeof(T) + 16;"),
    ("krylov.cu", "int acc_stride = kFewSlots, coef_stride = kGroup;"),
    ("krylov.cu", "acc_stride = std::max(acc_stride, a.nrows1);"),
    ("krylov.cu", "coef_stride = std::max(coef_stride, (a.nrows2 + kGroup - 1) / kGroup * kGroup);"),
    ("krylov.cu", "int per_launch = std::min(total, kStepBatch);"),
    ("krylov.cu", "while (per_launch > 1 && step_smem_bytes<T>(per_launch, acc_stride, coef_stride) > 112 * 1024) --per_launch;"),
    ("krylov.cu", "if (per_launch < 2) return BL_OK;"),
    ("krylov.cu", "B.count = std::min(per_launch, total - first);"),
    ("krylov.cu", "bool use_tma(int64_t n) { return n >= 8192; }"),
]


def step_smem_bytes(count, acc_stride, coef_stride, itemsize):
    return RING_BYTES + BARRIER_BYTES + count * acc_stride * 8 + count * coef_stride * itemsize + 16


def step_groups(P, m, itemsize):
    """Runs per `k_step_tma` launch for one step of P lockstep runs with m active basis rows (n >= TMA_MIN_N): the
    forward's step i has m = i + 1 (nrows1 = nrows2 = m), the adjoint's step idx > 0 has m = idx + 1.  `()`: the step
    runs as separate kernels."""
    acc_stride = max(K_FEW_SLOTS, m)
    coef_stride = max(K_GROUP, -(-m // K_GROUP) * K_GROUP)
    per = min(P, K_STEP_BATCH)
    while per > 1 and step_smem_bytes(per, acc_stride, coef_stride, itemsize) > SMEM_LIMIT:
        per -= 1
    if P < 2 or per < 2:
        return ()
    return tuple(min(per, P - first) for first in range(0, P, per))


def sweep_groups(P, K, itemsize):
    """`(forward, adjoint)`: the grouping of every step of the two sweeps (forward m = 1..K, adjoint m = 2..K: step
    idx = 0 of the adjoint has no step-kernel form, `banded_step` in arnoldi_adjoint_t)."""
    return [step_groups(P, m, itemsize) for m in range(1, K + 1)], [step_groups(P, m, itemsize) for m in range(2, K + 1)]


def predicted_launches(n, P, K, itemsize):
    if n < TMA_MIN_N:
        return 0, 0
    fwd, adj = sweep_groups(P, K, itemsize)
    return sum(map(len, fwd)), sum(map(len, adj))


# ---- the cases (each GPU case below names the groupings its depth must pass through) -------------------------------
F64, F32 = np.float64, np.float32
CASES = {
    # n odd, just above the TMA threshold: 17 tiles of 4 KB, the last one partial; the depth reaches all four
    # groupings, and phase 1's reduction both with every block reducing every value and with block j reducing value j
    "A": dict(n=8221, dtype=F64, P=4, K=250),
    "B5": dict(n=8221, dtype=F64, P=5, K=250),  # 4 + 1, 3 + 2, 2 + 2 + 1
    "B7": dict(n=8221, dtype=F64, P=7, K=250),  # 4 + 3, 3 + 3 + 1, 2 + 2 + 2 + 1
    "C": dict(n=8221, dtype=F32, P=4, K=340, single_run_baseline=True),  # the fp32 crossovers (9 tiles)
    # the bench's launch shape (one block per SM): a large grid, block-per-value reductions, acc_stride > 40
    "D64": dict(n=150_001, dtype=F64, P=4, K=64, blocks_per_sm=1),
    "D32": dict(n=150_001, dtype=F32, P=4, K=64, blocks_per_sm=1),
    "E8191": dict(n=8191, dtype=F64, P=3, K=40),  # below use_tma: no step-kernel launch
    "E8192": dict(n=8192, dtype=F64, P=3, K=40),
}
ALL_GROUPINGS = {
    (8, 4): {(4,), (3, 1), (2, 2), ()},
    (8, 5): {(4, 1), (3, 2), (2, 2, 1), ()},
    (8, 7): {(4, 3), (3, 3, 1), (2, 2, 2, 1), ()},
    (4, 4): {(4,), (3, 1), (2, 2), ()},
}


def test_quoted_constants_match_the_source():
    for name, text in SOURCE_QUOTES:
        with open(os.path.join(CSRC, name)) as f:
            assert text in f.read(), f"{name} no longer contains {text!r}: update step_groups"
    # kOpStages = 3 * 8 * 256 * 16 / 8192 = 12 barriers of phase S, next to 2 * 3 + 2 of the ring
    assert BARRIER_BYTES == (2 * 3 + 2 + 2 * (3 * 8 * 256 * 16 // 8192)) * 8
    assert RING_BYTES == (3 * K_GROUP + 2) * TILE_BYTES


@pytest.mark.parametrize(
    "itemsize,P,spans",
    [
        (8, 4, [(1, 120, (4,)), (121, 162, (3, 1)), (163, 247, (2, 2)), (248, 400, ())]),
        (8, 5, [(1, 120, (4, 1)), (121, 162, (3, 2)), (163, 247, (2, 2, 1)), (248, 400, ())]),
        (4, 4, [(1, 163, (4,)), (164, 218, (3, 1)), (219, 328, (2, 2)), (329, 400, ())]),
        (8, 1, [(1, 400, ())]),
    ],
)
def test_step_groups_reproduce_the_crossover_table(itemsize, P, spans):
    for lo, hi, groups in spans:
        for m in range(lo, hi + 1):
            assert step_groups(P, m, itemsize) == groups, (itemsize, P, m)


def test_gpu_cases_pass_through_every_grouping():
    for (itemsize, P), want in ALL_GROUPINGS.items():
        fwd, adj = set(), set()
        for c in CASES.values():
            if np.dtype(c["dtype"]).itemsize == itemsize and c["P"] == P and c["n"] >= TMA_MIN_N:
                f, a = sweep_groups(P, c["K"], itemsize)
                fwd |= set(f)
                adj |= set(a)
        assert fwd == want and adj == want, (itemsize, P, fwd, adj)
    # case A: phase 1 of a launch reduces count * m values on G = 17 blocks; every block reduces all of them while
    # that is at most 2560 (grid_reduce), block j reduces value j above
    c = CASES["A"]
    G = -(-c["n"] * 8 // TILE_BYTES)
    regimes = {count * m * G <= 2560 for m in range(1, c["K"] + 1) for count in step_groups(c["P"], m, 8)}
    assert G == 17 and regimes == {True, False}
    for c in CASES.values():  # every traced sweep fits the trace
        assert max(predicted_launches(c["n"], c["P"], c["K"], np.dtype(c["dtype"]).itemsize)) < TRACE_LAUNCHES


# ---- GPU: inputs, oracle, runners ------------------------------------------------------------------------------------
# Contract bounds of tests/test_gpu_parity.py: fp64 1e-10 on the coefficients and 1e-9 on dv and the gradient (the bound
# of test_dense_basis_cotangent_beyond_depth_128), fp32 1e-5 / 1e-4 with x10 on dv.
BOUNDS = {
    F64: dict(alpha=1e-10, beta=1e-10, c=1e-10, Q=1e-8, orth=1e-12, r=1e-8, dv=1e-9, grad=1e-9),
    F32: dict(alpha=1e-5, beta=1e-5, c=1e-5, Q=1e-3, orth=1e-4, r=1e-3, dv=1e-3, grad=1e-4),
}
SENTINEL = {F64: np.uint64(0x7FF80000DEADBEEF), F32: np.uint32(0x7FC0BEEF)}  # quiet NaNs with a payload


def bits(a):
    a = np.asarray(a)
    return a.view(np.uint64 if a.dtype.itemsize == 8 else np.uint32)


@functools.lru_cache(maxsize=None)
def sparse_operand(n):
    from experiments_lanczos_adjoints_b200 import synthetic

    return synthetic.banded_spd_coo(n, 5, seed=n)


def probe(n, i):
    """Rademacher probe i of size n (exact in float32)."""
    return (np.random.default_rng([n, i]).integers(0, 2, n) * 2 - 1).astype(F64)


def cotangent(K, i, dtype=F64):
    """SLQ-type cotangent of run i: dH tridiagonal from seeded (dalpha, dbeta)."""
    from experiments_lanczos_adjoints_b200 import synthetic

    rng = np.random.default_rng([K, i, 7])
    return synthetic.slq_cotangent_dH(rng.standard_normal(K), rng.standard_normal(K - 1), dtype)


def oracle_run(op, params, v, dH, K):
    Qt, H, r, c = krylov.arnoldi_forward_active(op, K, v, *params)
    dv, dp = krylov.arnoldi_adjoint_active(op, params, Qt=Qt, H=H, r=r, c=c, dQt=None, dH=dH, dr=None, dc=0.0, reortho="full")
    return dict(Q=Qt, H=H, r=r, c=c, dv=dv, grad=dp[0])


@functools.lru_cache(maxsize=None)
def sparse_oracle(n, K, i):
    row, col, data = sparse_operand(n)
    return oracle_run(operators.CsrFastOperator(row, col, (n, n)), (data,), probe(n, i), cotangent(K, i), K)


def traced(fn):
    """Number of k_step_tma launches `fn()` enqueues."""
    from experiments_lanczos_adjoints_b200 import _lib

    stamps = (C.c_uint64 * (8 * TRACE_LAUNCHES))()
    count, pdl = C.c_int64(0), C.c_int(0)
    _lib.call("bl_step_trace_begin")
    try:
        fn()
    finally:
        _lib.call("bl_step_trace_end", stamps, TRACE_LAUNCHES, C.byref(count), C.byref(pdl))
    return count.value


def raw(a):
    """Every element of a device array's storage, the padding of its rows included: `(rows, ld)` for a 2-D array."""
    from experiments_lanczos_adjoints_b200 import _lib
    from experiments_lanczos_adjoints_b200 import device as dev

    host = np.empty(a.storage_elems, a.dtype)
    _lib.call("bl_memcpy_d2h", host.ctypes.data, a.ptr, host.nbytes, dev.default_stream().ptr)
    dev.default_stream().synchronize()
    return host.reshape(-1, a.ld) if a.ndim == 2 else host


def upload(a, host):
    from experiments_lanczos_adjoints_b200 import _lib
    from experiments_lanczos_adjoints_b200 import device as dev

    host = np.ascontiguousarray(host)
    assert host.nbytes == a.storage_elems * a.dtype.itemsize
    _lib.call("bl_memcpy_h2d", a.ptr, host.ctypes.data, host.nbytes, dev.default_stream().ptr)
    dev.default_stream().synchronize()


def fill_sentinel(a):
    upload(a, np.full(a.storage_elems, SENTINEL[a.dtype.type]).view(a.dtype))


def run_errors(H, Q, r, c, dv, ref):
    """Relative errors of one run against the oracle (`Q` is `(K, n)`); `orth` is `||Q Q^T - I||_F`."""
    T, Tr = 0.5 * (H + H.T), 0.5 * (ref["H"] + ref["H"].T)
    Q64 = np.asarray(Q, F64)
    return dict(
        alpha=rel_err(np.diag(T), np.diag(Tr)),
        beta=rel_err(np.diag(T, 1), np.diag(Tr, 1)),
        c=rel_err(c, ref["c"]),
        Q=rel_err(Q, ref["Q"]),
        orth=float(np.linalg.norm(Q64 @ Q64.T - np.eye(len(Q64)))),
        r=rel_err(r, ref["r"]),
        dv=rel_err(dv, ref["dv"]),
    )


def read(pl, K):
    P = pl.P
    return dict(H=pl.H.numpy().reshape(P, K, K), Q=raw(pl.Q), Lam=raw(pl.Lam), r=pl.r.numpy(), c=pl.c.numpy(),
                dv=pl.dv.numpy(), grad=pl.grads[0].numpy().ravel())  # fmt: skip


def run_plan(op, params, V, dHs, K, dtype):
    """The batch through `BatchedTridiagAdjointPlan`, with Q and Lambda filled with a NaN sentinel first.  Returns the
    results of forward + adjoint (with their traced launch counts), `(dv, gradient)` of the adjoint repeated with the
    cotangent of one run alone (`dH = 0` for the others), and the results of the whole call repeated."""
    from experiments_lanczos_adjoints_b200 import plan as bl_plan

    P = len(V)
    pl = bl_plan.BatchedTridiagAdjointPlan(op, K, dtype, P)
    fill_sentinel(pl.Q)
    fill_sentinel(pl.Lam)
    pl.set_vectors(V.astype(dtype))
    pl.set_params(*[p.astype(dtype) for p in params])
    pl.set_cotangents(dHs.astype(dtype))
    launches = (traced(pl.forward), traced(pl.adjoint))
    res = dict(read(pl, K), launches=launches)
    alone = []
    for p in range(P):
        dH = np.zeros_like(dHs)
        dH[p] = dHs[p]
        pl.set_cotangents(dH.astype(dtype))
        pl.adjoint()
        alone.append((pl.dv.numpy(), pl.grads[0].numpy().ravel()))
    pl.set_cotangents(dHs.astype(dtype))
    pl.run()
    return res, alone, read(pl, K)


def single_run_baseline(op, params, V, dHs, K, dtype, refs):
    """The same probes one at a time through `TridiagAdjointPlan` (the single-run path, which never launches
    k_step_tma): per-run errors against the oracle, and the error of the gradient summed over the runs."""
    from experiments_lanczos_adjoints_b200 import plan as bl_plan

    runs, summed = [], 0.0
    for v, dH, ref in zip(V, dHs, refs):
        pl = bl_plan.TridiagAdjointPlan(op, K, dtype)
        pl.set_vector(v.astype(dtype))
        pl.set_params(*[p.astype(dtype) for p in params])
        pl.set_cotangent(dH.astype(dtype))
        assert traced(pl.run) == 0
        grad = pl.grads[0].numpy().ravel()
        runs.append(dict(run_errors(pl.H.numpy(), pl.Q.numpy(), pl.r.numpy(), pl.c.numpy(), pl.dv.numpy(), ref),
                         grad=rel_err(grad, ref["grad"])))  # fmt: skip
        summed = summed + grad.astype(F64)
    return dict(runs=runs, grad_sum=rel_err(summed, sum(ref["grad"] for ref in refs)))


def limit(bound, base_err):
    """The contract bound; where the single-run path itself misses it (`base_err`), twice the single run's error."""
    return bound if base_err is None or base_err < bound else 2.0 * base_err


def check_runs(res, refs, dtype, n, K, expect_launches, base=None):
    """Per-run comparison with the oracle, the zero padding of Q and Lambda, and the traced launch counts."""
    P, bound = len(refs), BOUNDS[dtype]
    assert res["launches"] == expect_launches, f"k_step_tma launches (forward, adjoint) {res['launches']} != {expect_launches}"
    Q, Lam = res["Q"].reshape(P, K, -1), res["Lam"].reshape(P, K, -1)
    for name, B in (("Q", Q), ("Lambda", Lam)):
        assert not bits(B[:, :, n:]).any(), f"{name}: rows not zero in [n, ld)"
        assert np.isfinite(B[:, :, :n]).all(), name
    for p, ref in enumerate(refs):
        errs = run_errors(res["H"][p], Q[p, :, :n], res["r"][p], res["c"][p], res["dv"][p], ref)
        bad = {k: e for k, e in errs.items() if not e < limit(bound[k], base and base["runs"][p][k])}
        assert not bad, f"run {p}: {bad} (all: {errs})"
    err = rel_err(res["grad"], sum(ref["grad"] for ref in refs))
    assert err < limit(bound["grad"], base and base["grad_sum"]), f"summed gradient: {err}"


def check_attribution(res, alone, again, refs, dtype, base=None):
    """Run p's cotangent alone: run p's gradient and dv, exact zeros in every other run's dv.  And two identical
    calls: bit-identical H, dv and gradient."""
    for p, (dv, grad) in enumerate(alone):
        err = rel_err(grad, refs[p]["grad"])
        assert err < limit(BOUNDS[dtype]["grad"], base and base["runs"][p]["grad"]), f"run {p} alone: gradient error {err}"
        assert np.array_equal(bits(dv[p]), bits(res["dv"][p])), f"run {p} alone: dv differs from the batch's"
        for q in range(len(alone)):
            if q != p:
                assert not np.count_nonzero(dv[q]), f"run {p} alone: dv of run {q} is not zero"
    for name in ("H", "dv", "grad"):
        assert np.array_equal(bits(again[name]), bits(res[name])), f"{name} differs between two identical calls"


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_lockstep_batch_matches_the_oracle_run_by_run(case):
    """Case C (fp32, depth 340) is gated on the single-run path: at that depth the fp32 single run itself misses the
    contract bounds on dv and the gradient.  Measured on a B200 (1000 W), relative errors against the float64 oracle
    for probes 0..3, single run / batch: dv 2.1e-5 / 3.5e-5, 1.0e-3 / 1.1e-3, 6.2e-4 / 3.6e-4, 7.1e-5 / 2.2e-5;
    gradient 1.9e-5 / 4.8e-5, 8.6e-4 / 9.1e-4, 6.0e-4 / 3.5e-4, 7.9e-5 / 2.3e-5; gradient summed over the four runs,
    batch 4.4e-4.  Every other quantity, and every fp64 case up to depth 250, meets the contract bounds by orders of
    magnitude (fp64: dv and gradient <= 3.2e-12 in the batch and 4.7e-12 in the single run)."""
    import experiments_lanczos_adjoints_b200 as bl
    from experiments_lanczos_adjoints_b200 import device as dev

    c = CASES[case]
    n, dtype, P, K = c["n"], c["dtype"], c["P"], c["K"]
    row, col, data = sparse_operand(n)
    op = bl.operators.SparseOperator(row, col, (n, n))
    V = np.stack([probe(n, i) for i in range(P)])
    dHs = np.stack([cotangent(K, i) for i in range(P)])
    with dev.blocks_per_sm(c.get("blocks_per_sm", 0)):
        res, alone, again = run_plan(op, (data,), V, dHs, K, dtype)
    refs = [sparse_oracle(n, K, i) for i in range(P)]
    base = single_run_baseline(op, (data,), V, dHs, K, dtype, refs) if c.get("single_run_baseline") else None
    expect = predicted_launches(n, P, K, np.dtype(dtype).itemsize)
    assert (n < TMA_MIN_N) == (expect == (0, 0))
    check_runs(res, refs, dtype, n, K, expect, base)
    check_attribution(res, alone, again, refs, dtype, base)


class RecordingSymDense:
    """`operators.SymDenseOperator` (`(p + p^T) x`) with `p + p^T` formed once and the parameter cotangent
    `sum_k lam_k x_k^T + x_k lam_k^T` formed once from the recorded pairs (an n x n update per step is slow)."""

    def __init__(self, p):
        self.S = p + p.T
        self.pairs = []

    def matvec(self, x, _):
        return self.S @ x

    def vjp(self, x, lam, _):
        self.pairs.append((x, lam))
        return self.S @ lam, (np.zeros(1),)

    def grad(self):
        X, L = (np.array(a) for a in zip(*self.pairs))
        return (L.T @ X + X.T @ L).ravel()


@pytest.mark.gpu
def test_lockstep_batch_with_a_dense_operand_matches_the_oracle_run_by_run():
    """A dense operand has no SELL-32 form, so the step kernel runs without the operator call (no phase S): the
    forward's batched matvec is followed by k_step_tma, and the adjoint takes one vjp per run and then the step
    kernel."""
    import experiments_lanczos_adjoints_b200 as bl

    n, K, P, dtype = 8300, 40, 3, F64
    rng = np.random.default_rng(8300)
    G = rng.standard_normal((n, n))
    p = 0.25 * (G + G.T) / np.sqrt(n) + 2.0 * np.eye(n)  # p + p^T: spectrum within about 4 -+ 1.5
    del G
    V = rng.standard_normal((P, n))
    dHs = np.stack([cotangent(K, i) for i in range(P)])
    op = bl.operators.DenseOperator(n, sym=True)
    res, alone, again = run_plan(op, (p,), V, dHs, K, dtype)
    refs = []
    for i in range(P):
        rec = RecordingSymDense(p)
        refs.append(oracle_run(rec, (None,), V[i], dHs[i], K))
        refs[-1]["grad"] = rec.grad()
    expect = predicted_launches(n, P, K, 8)
    assert expect == (K, K - 1)
    check_runs(res, refs, dtype, n, K, expect)
    check_attribution(res, alone, again, refs, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("n,gap", [(8192, "n+1"), (8192, "ld+32"), (8221, "n+1")])
def test_batch_entries_leave_the_gaps_between_rows_untouched(n, gap):
    """`ldv`, `lddv` > n: the batch entries read v and write dv row by row and leave what lies between the rows alone.
    n = 8192 with a stride of n + 1 puts odd rows of dv off 16-byte alignment; n = 8221 with n + 1 leaves one element
    after a row whose last vector straddles n; ld + 32 is aligned with a wide gap."""
    import experiments_lanczos_adjoints_b200 as bl
    from experiments_lanczos_adjoints_b200 import _lib
    from experiments_lanczos_adjoints_b200 import device as dev
    from experiments_lanczos_adjoints_b200.arnoldi import adjoint_flags, forward_flags

    dtype, P, K = F64, 3, 40
    code, ld = dev.dtype_code(dtype), dev.basis_ld(n, dtype)
    ldv = n + 1 if gap == "n+1" else ld + 32
    row, col, data = sparse_operand(n)
    op = bl.operators.SparseOperator(row, col, (n, n))
    op.bind((data.astype(dtype),), dtype)
    V = np.stack([probe(n, i) for i in range(P)])
    dHs = np.stack([cotangent(K, i) for i in range(P)])
    v_host = np.full((P, ldv), SENTINEL[dtype]).view(dtype)
    v_host[:, :n] = V
    v, dv = dev.DeviceArray((P, ldv), dtype), dev.DeviceArray((P, ldv), dtype)
    upload(v, v_host)
    fill_sentinel(dv)
    Q, Lam = dev.DeviceArray((P * K, n), dtype, ld=ld), dev.DeviceArray((P * K, n), dtype, ld=ld)
    fill_sentinel(Q)
    fill_sentinel(Lam)
    H, r, c = dev.DeviceArray((P, K * K), dtype), dev.DeviceArray((P, n), dtype, ld=ld), dev.DeviceArray((P,), dtype)
    dH = dev.asarray(dHs.astype(dtype).reshape(P, K * K))
    ws_bytes = P * _lib.load().bl_arnoldi_workspace_bytes(n, K, code)
    ws = dev.DeviceArray(((ws_bytes + 3) // 4,), np.float32)
    s = dev.default_stream().ptr

    def forward():
        _lib.call("bl_arnoldi_forward_batch", op._handle, code, n, K, forward_flags(True, True), P, v.ptr, ldv, Q.ptr, ld,
                  H.ptr, r.ptr, c.ptr, ws.ptr, ws_bytes, s)  # fmt: skip

    def adjoint():
        op.grad_zero(dtype)
        _lib.call("bl_arnoldi_adjoint_batch", op._handle, code, n, K, adjoint_flags(True, True, True), P, Q.ptr, ld, H.ptr,
                  r.ptr, c.ptr, None, dH.ptr, None, None, dv.ptr, ldv, Lam.ptr, ws.ptr, ws_bytes, s)  # fmt: skip

    launches = (traced(forward), traced(adjoint))
    dv_raw = raw(dv)
    assert np.array_equal(bits(raw(v)), bits(v_host)), "v changed"
    assert (bits(dv_raw[:, n:]) == SENTINEL[dtype]).all(), "the gap between the rows of dv was written"
    res = dict(H=H.numpy().reshape(P, K, K), Q=raw(Q), Lam=raw(Lam), r=r.numpy(), c=c.numpy(), dv=dv_raw[:, :n],
               grad=op.grad_export(dtype)[0].numpy(), launches=launches)  # fmt: skip
    refs = [sparse_oracle(n, K, i) for i in range(P)]
    check_runs(res, refs, dtype, n, K, predicted_launches(n, P, K, 8))
