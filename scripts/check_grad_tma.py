"""k_sell_grad_tma (staged pairs) against k_sell_grad_batch (BL_GRAD_TMA=0): bit-identical parameter cotangents on a banded
operand (every block staged), a random sparse operand (no block staged) and a banded operand with a few far entries."""
import os
import subprocess
import sys
import tempfile

import numpy as np

sys.path.insert(0, ".")

if len(sys.argv) > 1 and sys.argv[1] == "child":
    import experiments_lanczos_adjoints_b200 as bl
    from experiments_lanczos_adjoints_b200 import plan as bl_plan, synthetic

    out = {}
    rng = np.random.default_rng(0)
    for name, n, K, dtype in [("banded_f32", 200_003, 20, np.float32), ("banded_f64", 100_001, 12, np.float64),
                              ("random_f32", 20_000, 10, np.float32), ("mixed_f32", 150_000, 10, np.float32)]:
        if name.startswith("random"):
            r = rng.integers(0, n, size=8 * n)
            c = rng.integers(0, n, size=8 * n)
            row = np.concatenate([r, c, np.arange(n)]).astype(np.int32)
            col = np.concatenate([c, r, np.arange(n)]).astype(np.int32)
            data = np.concatenate([0.01 * rng.standard_normal(8 * n)] * 2 + [20.0 + rng.random(n)])
        else:
            row, col, data = synthetic.banded_spd_coo(n, 5, seed=3, max_offset=100, long_range=0)
            if name.startswith("mixed"):  # a few symmetric far-away entries: their blocks fall back to gathers
                i = rng.integers(0, n // 2, size=40)
                j = i + n // 3
                row = np.concatenate([row, i, j]).astype(np.int32)
                col = np.concatenate([col, j, i]).astype(np.int32)
                data = np.concatenate([data, np.full(80, 0.01)])
        op = bl.operators.SparseOperator(row, col, (n, n))
        pl = bl_plan.TridiagAdjointPlan(op, K, dtype)
        pl.set_vector(rng.standard_normal(n).astype(dtype))
        pl.set_params(data.astype(dtype))
        pl.set_cotangent(synthetic.slq_cotangent_dH(rng.standard_normal(K), rng.standard_normal(K - 1), dtype))
        pl.run()
        pl.stream.synchronize()
        out[name] = pl.grads[0].numpy(pl.stream)
    np.savez(sys.argv[2], **out)
    sys.exit(0)

res = {}
tmp = tempfile.TemporaryDirectory()
for flag in ("0", "1"):
    path = os.path.join(tmp.name, f"grad_tma_{flag}.npz")
    subprocess.run([sys.executable, __file__, "child", path], check=True, env=dict(os.environ, BL_GRAD_TMA=flag))
    res[flag] = dict(np.load(path))
ok = True
for k in res["0"]:
    a, b = res["0"][k], res["1"][k]
    same = np.array_equal(a, b)
    ok = ok and same and np.isfinite(a).all() and np.abs(a).max() > 0
    print(f"{k}: bit-identical {same}; |grad| max {np.abs(a).max():.3e}; max |diff| {np.abs(a.astype(np.float64) - b).max():.3e}")
sys.exit(0 if ok else 1)
