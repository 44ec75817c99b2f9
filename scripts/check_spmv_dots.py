"""k_sell_spmv_dots (operator call + neighbouring-row dots of one run in one launch) against the separate k_dots_few launches
(BL_SPMV_DOTS=0): the dots are added up in another order, so H / dv / dparams agree to rounding, not bit for bit."""
import os
import subprocess
import sys
import tempfile

import numpy as np

sys.path.insert(0, ".")

CASES = [("f32", 200_003, 24, np.float32), ("f64", 100_001, 16, np.float64), ("f32_ragged", 33_333, 9, np.float32)]

if len(sys.argv) > 1 and sys.argv[1] == "child":
    import experiments_lanczos_adjoints_b200 as bl
    from experiments_lanczos_adjoints_b200 import plan as bl_plan, synthetic

    out = {}
    rng = np.random.default_rng(0)
    for name, n, K, dtype in CASES:
        row, col, data = synthetic.banded_spd_coo(n, 5, seed=3)
        op = bl.operators.SparseOperator(row, col, (n, n))
        pl = bl_plan.TridiagAdjointPlan(op, K, dtype)
        pl.set_vector(rng.standard_normal(n).astype(dtype))
        pl.set_params(data.astype(dtype))
        pl.set_cotangent(synthetic.slq_cotangent_dH(rng.standard_normal(K), rng.standard_normal(K - 1), dtype))
        l0 = bl.launch_count()
        pl.run()
        pl.stream.synchronize()
        out[name + "_launches"] = np.array(bl.launch_count() - l0)
        out[name + "_H"] = pl.H.numpy(pl.stream)
        out[name + "_dv"] = pl.dv.numpy(pl.stream)
        out[name + "_g"] = pl.grads[0].numpy(pl.stream)
    np.savez(sys.argv[2], **out)
    sys.exit(0)

res = {}
tmp = tempfile.TemporaryDirectory()
for flag in ("0", "1"):
    path = os.path.join(tmp.name, f"spmv_dots_{flag}.npz")
    subprocess.run([sys.executable, __file__, "child", path], check=True, env=dict(os.environ, BL_SPMV_DOTS=flag))
    res[flag] = dict(np.load(path))
ok = True
for name, n, K, dtype in CASES:
    tol = 2e-5 if dtype == np.float32 else 1e-11
    line = [f"{name}: launches {int(res['0'][name + '_launches'])} -> {int(res['1'][name + '_launches'])}"]
    ok = ok and int(res["1"][name + "_launches"]) < int(res["0"][name + "_launches"])
    for k in ("H", "dv", "g"):
        a, b = res["0"][f"{name}_{k}"].astype(np.float64), res["1"][f"{name}_{k}"].astype(np.float64)
        err = np.linalg.norm(a - b) / np.linalg.norm(a)
        ok = ok and np.isfinite(b).all() and err < tol
        line.append(f"{k} rel diff {err:.2e}")
    print("; ".join(line))
sys.exit(0 if ok else 1)
