"""CPU-side checks: the C-ABI library loads, exports every symbol `include/b200_lanczos.h`
declares, host logic (errors, index work) behaves like the reference — no compute calls."""

import ctypes
import os
import re

import numpy as np
import pytest
from conftest import ROOT

import experiments_lanczos_adjoints_b200 as bl
from experiments_lanczos_adjoints_b200 import _lib
from oracle import operators as oracle_ops


def header_symbols():
    text = open(os.path.join(ROOT, "include", "b200_lanczos.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(bl_[a-z0-9_]+)\s*\(", text)) - {"bl_matvec_cb", "bl_vjp_cb"})


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(_lib.library_path())
    names = header_symbols()
    assert len(names) >= 50
    for name in names:
        assert hasattr(lib, name), name
    assert set(names) == set(_lib.SIGNATURES), set(names) ^ set(_lib.SIGNATURES)
    assert b"sm_100a" in _lib.load().bl_version()


def test_up_to_date_library_is_reused_without_writing_to_the_tree(tmp_path, monkeypatch):
    """A built tree may be read-only: loading the library then creates no object directory or lock file."""
    from experiments_lanczos_adjoints_b200 import build

    build.build()
    stamp = os.stat(build.STAMP).st_mtime_ns
    monkeypatch.setattr(build, "OBJ", str(tmp_path / "objects"))
    assert build.build() == build.LIB
    assert not os.path.exists(tmp_path / "objects") and os.stat(build.STAMP).st_mtime_ns == stamp


def test_header_is_valid_c_and_library_links_from_c(tmp_path):
    """Compile tests/c_abi_smoke.c with gcc against include/b200_lanczos.h and run it."""
    import shutil
    import subprocess

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    lib = _lib.library_path()
    exe = str(tmp_path / "c_abi_smoke")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "c_abi_smoke.c"), "-o", exe, lib,
                    "-Wl,-rpath," + os.path.dirname(lib)], check=True)  # fmt: skip
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, (out.returncode, out.stdout, out.stderr)
    assert "c abi ok" in out.stdout


def test_workspace_queries_are_pure_host_functions():
    lib = _lib.load()
    small = lib.bl_arnoldi_workspace_bytes(1000, 10, _lib.BL_F32)
    big = lib.bl_arnoldi_workspace_bytes(1_000_000, 100, _lib.BL_F64)
    assert 0 < small < big < (1 << 31)
    assert lib.bl_lanczos3_workspace_bytes(1000, 10, _lib.BL_F32) > 0
    assert lib.bl_vec_workspace_bytes() > 0


@pytest.mark.parametrize("reortho_wrong", [True, "full_with_sparsity", "None"])
def test_hessenberg_raises_type_error_for_wrong_reortho(reortho_wrong):
    # /root/reference/tests/test_arnoldi/test_hessenberg_forward.py:81-84
    op = bl.operators.SparseOperator([0], [0], (2, 2))
    with pytest.raises(TypeError, match="Unexpected input"):
        bl.arnoldi.hessenberg(op, 1, reortho=reortho_wrong)


def test_tridiag_raises_value_error_for_wrong_reortho():
    # lanczos.py:148-149 raises ValueError for the same mistake (SURVEY quirk B9)
    op = bl.operators.SparseOperator([0], [0], (2, 2))
    with pytest.raises(ValueError, match="unsupported"):
        bl.lanczos.tridiag(op, 1, reortho="partial")


def test_plain_callable_is_rejected_loudly():
    with pytest.raises(TypeError, match="operator object"):
        bl.arnoldi.hessenberg(lambda s: s, 1, reortho="none")


def test_custom_vjp_estimator_raises_outside_vjp():
    est = bl.hutchinson.hutchinson_custom_vjp(lambda v, p: 0.0, lambda key: np.ones((1, 2)))
    with pytest.raises(RuntimeError, match="oops"):  # hutchinson.py:24-30
        est(0, 1.0)


@pytest.mark.parametrize("seed,n,nnz", [(0, 1, 1), (1, 33, 200), (2, 1000, 7000), (3, 64, 0), (4, 257, 5000)])
def test_sparse_index_work_is_bit_exact(seed, n, nnz):
    """COO -> CSR -> SELL-32 (A and A^T) against oracle/operators.py, including duplicates,
    empty rows, ragged last slice, nnz = 0."""
    rng = np.random.default_rng(seed)
    row = rng.integers(0, n, nnz).astype(np.int32)
    col = rng.integers(0, n, nnz).astype(np.int32)
    if nnz > 10:
        row[5], col[5] = row[2], col[2]  # a duplicate entry
    op = bl.operators.SparseOperator(row, col, (n, n))
    row_ptr, col_idx, perm = op.export_csr()
    r_ptr, c_idx, pm = oracle_ops.coo_to_csr(row, col, n)
    assert np.array_equal(row_ptr, r_ptr) and np.array_equal(col_idx, c_idx) and np.array_equal(perm, pm)
    slice_ptr, slot = op.export_sell()
    s_ptr, s_slot = oracle_ops.csr_to_sell(r_ptr, n)
    assert np.array_equal(slice_ptr, s_ptr) and np.array_equal(slot, s_slot)
    slice_ptr_t, slot_t = op.export_sell(transpose=True)
    rt_ptr, _, _ = oracle_ops.coo_to_csr(col, row, n)
    st_ptr, st_slot = oracle_ops.csr_to_sell(rt_ptr, n)
    assert np.array_equal(slice_ptr_t, st_ptr) and np.array_equal(slot_t, st_slot)


def test_sparse_create_rejects_out_of_range_indices():
    with pytest.raises(ValueError, match="out of range"):
        bl.operators.SparseOperator([0, 5], [0, 1], (3, 3))


def test_matrix_market_parameter_order_matches_mmread():
    """`suite_sparse_load` order: stored lower triangle, then mirrored strict part
    (/root/reference/src/matfree_extensions/util/exp_util.py:35-42)."""
    import io

    import scipy.io

    text = "%%MatrixMarket matrix coordinate real symmetric\n3 3 4\n1 1 2.0\n2 1 -1.0\n3 2 -0.5\n3 3 4.0\n"
    m = scipy.io.mmread(io.StringIO(text))
    r, c, d = oracle_ops.mm_expand_symmetric([0, 1, 2, 2], [0, 0, 1, 2], [2.0, -1.0, -0.5, 4.0])
    assert np.array_equal(m.row, r) and np.array_equal(m.col, c) and np.array_equal(m.data, d)


def test_quadform_cotangents_match_finite_differences():
    from experiments_lanczos_adjoints_b200.lanczos import _quadform_and_cotangents

    rng = np.random.default_rng(0)
    a, b = 2.0 + rng.uniform(size=6), 0.3 * rng.uniform(size=5)
    val, da, db, _ = _quadform_and_cotangents(np.log, None, a, b, True)
    eps = 1e-6
    for i in range(6):
        e = np.zeros(6)
        e[i] = eps
        fd = (_quadform_and_cotangents(np.log, None, a + e, b, False)[0]
              - _quadform_and_cotangents(np.log, None, a - e, b, False)[0]) / (2 * eps)  # fmt: skip
        assert abs(fd - da[i]) < 1e-8
    for i in range(5):
        e = np.zeros(5)
        e[i] = eps
        fd = (_quadform_and_cotangents(np.log, None, a, b + e, False)[0]
              - _quadform_and_cotangents(np.log, None, a, b - e, False)[0]) / (2 * eps)  # fmt: skip
        assert abs(fd - db[i]) < 1e-8


def test_loop_flags_match_the_header_and_only_tridiag_sets_the_symmetric_bits():
    """`second_pass` / `reortho_full` of the Krylov entry points are bit masks (include/b200_lanczos.h):
    the general loops of `arnoldi.hessenberg` pass 0/1, `lanczos.tridiag(reortho="full")` -- symmetric operand,
    tridiagonal cotangent (lanczos.py:152-169) -- adds the symmetric bits (SURVEY Appendix B7)."""
    import re

    from experiments_lanczos_adjoints_b200 import arnoldi

    header = open(os.path.join(ROOT, "include", "b200_lanczos.h")).read()
    consts = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (BL_(?:FWD|ADJ)_\w+) (\d+)", header)}
    assert consts == {"BL_FWD_SECOND_PASS": 1, "BL_FWD_SYMMETRIC": 2, "BL_ADJ_REORTHO_FULL": 1,
                      "BL_ADJ_SYMMETRIC": 2, "BL_ADJ_TRIDIAG_COTANGENT": 4}  # fmt: skip
    assert (arnoldi.BL_ADJ_REORTHO_FULL, arnoldi.BL_ADJ_SYMMETRIC, arnoldi.BL_ADJ_TRIDIAG_COTANGENT) == (1, 2, 4)
    assert [arnoldi.forward_flags(*a) for a in ((False, False), (True, False), (True, True), (False, True))] == [0, 1, 3, 0]
    assert arnoldi.adjoint_flags(False, True, True) == 0  # the shortcuts need the re-projection
    assert arnoldi.adjoint_flags(True, False, True) == 1
    assert arnoldi.adjoint_flags(True, True) == 3 and arnoldi.adjoint_flags(True, True, True) == 7

    op = bl.operators.DenseOperator(4)
    general = bl.arnoldi.hessenberg(op, 2, reortho="full")
    assert (general._forward_flags, general._adjoint_flags) == (1, 1)
    assert bl.arnoldi.hessenberg(op, 2, reortho="none")._adjoint_flags == 0
    assert bl.arnoldi.hessenberg(op, 2, reortho="full", reortho_vjp="none")._forward_flags == 0
    tri = bl.lanczos.tridiag(op, 2, reortho="full")
    assert (tri.alg._forward_flags, tri.alg._adjoint_flags) == (3, 7)


def test_sparse_operator_clone_shares_the_pattern_not_the_handle():
    """Probes in flight need one operator handle per lane (`SparseOperator.clone`): same index work, own handle."""
    rng = np.random.default_rng(5)
    n, nnz = 97, 400
    row, col = rng.integers(0, n, nnz).astype(np.int32), rng.integers(0, n, nnz).astype(np.int32)
    op = bl.operators.SparseOperator(row, col, (n, n))
    twin = op.clone()
    assert twin._handle != op._handle and twin.shape == op.shape and twin.nnz == op.nnz
    for a, b in zip(op.export_csr(), twin.export_csr()):
        assert np.array_equal(a, b)
    for t in (False, True):
        for a, b in zip(op.export_sell(t), twin.export_sell(t)):
            assert np.array_equal(a, b)


def test_probe_lockstep_eligibility_is_host_logic():
    """Which estimator calls run their probes in lockstep batches (`lanczos._lockstep_eligible`): full-
    reorthogonalisation SLQ on a square sparse operand with at least 8 probes; everything else takes the Gram batch
    or the one-probe-at-a-time route."""
    from experiments_lanczos_adjoints_b200 import lanczos

    n = 64
    idx = np.arange(n, dtype=np.int32)
    sparse = bl.operators.SparseOperator(idx, idx, (n, n))
    probes = np.ones((8, n), np.float32)
    full = bl.lanczos.integrand_spd(np.log, 4, sparse)
    assert lanczos._lockstep_eligible(full, probes)
    assert not lanczos._lockstep_eligible(full, probes[:-1])  # fewer than two batches of four
    assert not lanczos._lockstep_eligible(full, probes.astype(np.int32))
    assert not lanczos._lockstep_eligible(bl.lanczos.integrand_spd(np.log, 4, sparse, reortho="none"), probes)
    assert not lanczos._lockstep_eligible(bl.lanczos.integrand_spd(np.log, 4, bl.operators.DenseOperator(n)), probes)
    assert not lanczos._batch_eligible(full, np.float32)  # the sparse operand shares no work between probes


def test_ffi_shim_handlers_match_their_bindings(tmp_path):
    """`csrc/ffi_shim.cc` (the XLA-FFI layer north_star names) cannot be built here -- jaxlib's headers are absent --
    but it is type-checked: `tests/stubs/xla/ffi/api/ffi.h` declares the part of the FFI API the shim uses and its
    `Binding::To` static_asserts that every handler is invocable with exactly what its `.Ctx/.Arg/.Ret/.Attr` chain
    describes; the C ABI calls inside are checked against include/b200_lanczos.h."""
    import shutil
    import subprocess

    gxx = shutil.which("g++")
    cuda_inc = next((d for d in ("/usr/local/cuda/include", "/usr/include") if os.path.exists(os.path.join(d, "cuda_runtime_api.h"))), None)
    if gxx is None or cuda_inc is None:
        pytest.skip("g++ or cuda_runtime_api.h not available")
    shim = os.path.join(ROOT, "experiments_lanczos_adjoints_b200", "csrc", "ffi_shim.cc")
    base = [gxx, "-std=c++17", "-fsyntax-only", "-Wall", "-Werror", "-I", os.path.join(ROOT, "tests", "stubs"),
            "-I", os.path.join(ROOT, "include"), "-I", cuda_inc]  # fmt: skip
    res = subprocess.run(base + [shim], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    text = open(shim).read()
    handlers = re.findall(r"XLA_FFI_DEFINE_HANDLER_SYMBOL\((bl_ffi_[a-z0-9_]+)", text)
    assert {"bl_ffi_matvec", "bl_ffi_matvec_vjp", "bl_ffi_arnoldi_forward", "bl_ffi_arnoldi_adjoint",
            "bl_ffi_lanczos3_forward", "bl_ffi_lanczos3_adjoint", "bl_ffi_pcg_solve", "bl_ffi_precond_apply",
            "bl_ffi_cholesky_partial"} <= set(handlers)  # fmt: skip
    for entry in ("bl_arnoldi_forward_batch", "bl_arnoldi_adjoint_batch"):  # the batched handlers behind jax.vmap
        assert entry in text
    # the check has teeth: a handler whose parameters are out of order with its binding must not compile
    bad = tmp_path / "bad_shim.cc"
    good_sig = "ffi::Error PrecondApply(cudaStream_t stream, ffi::AnyBuffer v, ffi::Result<ffi::AnyBuffer> out, int64_t precond_handle)"
    assert good_sig in text
    bad.write_text(text.replace(good_sig, "ffi::Error PrecondApply(cudaStream_t stream, ffi::AnyBuffer v, int64_t precond_handle, ffi::Result<ffi::AnyBuffer> out)"))
    res = subprocess.run(base + [str(bad)], capture_output=True, text=True)
    assert res.returncode != 0 and "does not match" in res.stderr
