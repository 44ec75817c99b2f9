// XLA FFI shim: exposes the C ABI of libb200lanczos.so (include/b200_lanczos.h) as `jax.ffi` custom-call targets,
// one handler per entry point the reference's `custom_vjp` pairs need (INTEGRATION.md shows the Python side).
//
// NOT built in this image (JAX / jaxlib and their headers are not installed, see DESIGN.md): compile where
// `python -c "import jax.ffi; print(jax.ffi.include_dir())"` works,
//   g++ -O2 -fPIC -shared -std=c++17 -I$(python -c "import jax.ffi;print(jax.ffi.include_dir())") ...
//       -I$CUDA_HOME/include -I../../include ffi_shim.cc -L.. -lb200lanczos -o libb200lanczos_ffi.so
// Here it is type-checked against a stand-in for `xla/ffi/api/ffi.h` (tests/stubs/, `g++ -fsyntax-only`,
// tests/test_abi_cpu.py): every handler's signature must match its binding.
//
// The shim holds no logic.  Conventions:
//   * operator handles (bl_operator_t*, bl_precond_t*) are created once on the Python side through ctypes and
//     travel as int64 attributes;
//   * the operator's parameter arrays (`*params` of the reference's `matvec(v, *params)`; one for the sparse /
//     dense / stencil operands, three for the Gram operand) are the REMAINING arguments, their cotangents the
//     REMAINING results, in the same order -- any parameter count binds;
//   * scratch is an extra result buffer, so XLA owns it (`*_workspace_bytes` gives its size at trace time);
//   * every Krylov handler accepts a leading batch dimension (`vmap_method="expand_dims"`): `jax.vmap(integrand)`
//     over probes (hutchinson.py:14,53) and `jax.vmap(solve)` over initial conditions (train.py:109) become ONE
//     call of the lockstep drivers bl_arnoldi_{forward,adjoint}_batch, not a sequential loop.  Unbatched operands
//     arrive with a leading 1 under `expand_dims`; parameters are never batched.
#include <cuda_runtime_api.h>

#include <cstdint>
#include <string>
#include <vector>

#include "b200_lanczos.h"
#include "xla/ffi/api/ffi.h"

namespace ffi = xla::ffi;

namespace {

constexpr int kMaxParams = 8;

int dtype_of(ffi::DataType t) { return t == ffi::DataType::F32 ? BL_F32 : BL_F64; }

ffi::Error to_error(int rc) {
  if (rc == BL_OK) return ffi::Error::Success();
  return ffi::Error(rc == BL_EDEPTH || rc == BL_EINVAL ? ffi::ErrorCode::kInvalidArgument : ffi::ErrorCode::kInternal,
                    bl_last_error());
}

bl_operator_t* as_op(int64_t handle) { return reinterpret_cast<bl_operator_t*>(handle); }

// rank of `b` beyond its `core_rank` trailing dimensions = batch dimensions; returns the batch count
int64_t batch_of(const ffi::AnyBuffer& b, size_t core_rank) {
  const auto dims = b.dimensions();
  int64_t count = 1;
  for (size_t i = 0; i + core_rank < dims.size(); ++i) count *= dims[i];
  return count;
}
bool is_batched(const ffi::AnyBuffer& b, size_t core_rank) { return b.dimensions().size() > core_rank; }

// `*params` -> bl_op_set_params
ffi::Error bind_params(bl_operator_t* op, int dtype, const ffi::RemainingArgs& params, cudaStream_t stream) {
  if (params.size() > (size_t)kMaxParams) return ffi::Error::InvalidArgument("too many operator parameters");
  const void* p[kMaxParams] = {};
  for (size_t i = 0; i < params.size(); ++i) {
    auto buf = params.get<ffi::AnyBuffer>(i);
    if (!buf.has_value()) return ffi::Error::InvalidArgument("operator parameter is not a buffer");
    p[i] = buf.value().untyped_data();
  }
  return to_error(bl_op_set_params(op, dtype, p, (int)params.size(), stream));
}

// accumulated parameter cotangents -> the remaining results
ffi::Error export_grads(bl_operator_t* op, int dtype, ffi::RemainingRets& grads, cudaStream_t stream) {
  if (grads.size() > (size_t)kMaxParams) return ffi::Error::InvalidArgument("too many parameter cotangents");
  void* g[kMaxParams] = {};
  for (size_t i = 0; i < grads.size(); ++i) {
    auto buf = grads.get<ffi::AnyBuffer>(i);
    if (!buf.has_value()) return ffi::Error::InvalidArgument("parameter cotangent is not a buffer");
    g[i] = buf.value()->untyped_data();
  }
  return to_error(bl_op_grad_export(op, dtype, g, (int)grads.size(), stream));
}

#define BL_FFI_TRY(expr)               \
  do {                                 \
    ffi::Error _e = (expr);            \
    if (_e.failure()) return _e;       \
  } while (0)

// ---- the user matvec and its pullback (`matvec(v, *params)`, `jax.vjp(matvec)`: arnoldi.py:207-209) ----------
ffi::Error Matvec(cudaStream_t stream, ffi::AnyBuffer x, ffi::RemainingArgs params, ffi::Result<ffi::AnyBuffer> y,
                  int64_t op_handle) {
  bl_operator_t* op = as_op(op_handle);
  const int dtype = dtype_of(x.element_type());
  BL_FFI_TRY(bind_params(op, dtype, params, stream));
  return to_error(bl_op_matvec(op, dtype, x.untyped_data(), y->untyped_data(), stream));
}

ffi::Error MatvecVjp(cudaStream_t stream, ffi::AnyBuffer q, ffi::AnyBuffer lam, ffi::RemainingArgs params,
                     ffi::Result<ffi::AnyBuffer> z, ffi::RemainingRets dparams, int64_t op_handle) {
  bl_operator_t* op = as_op(op_handle);
  const int dtype = dtype_of(q.element_type());
  BL_FFI_TRY(bind_params(op, dtype, params, stream));
  BL_FFI_TRY(to_error(bl_op_grad_zero(op, dtype, stream)));
  BL_FFI_TRY(to_error(bl_op_vjp(op, dtype, q.untyped_data(), lam.untyped_data(), z->untyped_data(), stream)));
  return export_grads(op, dtype, dparams, stream);
}

// ---- arnoldi._forward (arnoldi.py:57-101) ---------------------------------------------------------------------
// v ([P,] n), *params -> Qt ([P,] K, ld), H ([P,] K, K), r ([P,] ld), c ([P]), workspace
// flags: BL_FWD_SECOND_PASS | BL_FWD_SYMMETRIC (b200_lanczos.h)
ffi::Error ArnoldiForward(cudaStream_t stream, ffi::AnyBuffer v, ffi::RemainingArgs params,
                          ffi::Result<ffi::AnyBuffer> Qt, ffi::Result<ffi::AnyBuffer> H, ffi::Result<ffi::AnyBuffer> r,
                          ffi::Result<ffi::AnyBuffer> c, ffi::Result<ffi::AnyBuffer> workspace, int64_t op_handle,
                          int64_t krylov_depth, int64_t flags) {
  bl_operator_t* op = as_op(op_handle);
  const int dtype = dtype_of(v.element_type());
  const int64_t n = v.dimensions().back();
  const int64_t ld = Qt->dimensions().back();
  BL_FFI_TRY(bind_params(op, dtype, params, stream));
  if (is_batched(v, 1))
    return to_error(bl_arnoldi_forward_batch(op, dtype, n, krylov_depth, (int)flags, batch_of(v, 1), v.untyped_data(), n,
                                             Qt->untyped_data(), ld, H->untyped_data(), r->untyped_data(),
                                             c->untyped_data(), workspace->untyped_data(), workspace->size_bytes(),
                                             stream));
  return to_error(bl_arnoldi_forward(op, dtype, n, krylov_depth, (int)flags, v.untyped_data(), Qt->untyped_data(), ld,
                                     H->untyped_data(), r->untyped_data(), c->untyped_data(),
                                     workspace->untyped_data(), workspace->size_bytes(), stream));
}

// ---- arnoldi._adjoint (arnoldi.py:104-220) --------------------------------------------------------------------
// residuals (Qt, H, r, c) + cotangents (dQt, dH, dr, dc), *params -> dv ([P,] n), Lambda scratch, workspace, *dparams.
// JAX materialises zero cotangents for a custom_vjp; `dense_cotangents` says which of them carry data
// (bit 0: dQt, bit 1: dr, bit 2: dc) -- the SLQ integrand's are all zero (SURVEY 3.3) and skip a basis-sized read.
// flags: BL_ADJ_REORTHO_FULL | BL_ADJ_SYMMETRIC | BL_ADJ_TRIDIAG_COTANGENT.  Batched: the parameter cotangent is
// the sum over the batch (what `jax.vmap` + a scalar loss gives).
ffi::Error ArnoldiAdjoint(cudaStream_t stream, ffi::AnyBuffer Qt, ffi::AnyBuffer H, ffi::AnyBuffer r, ffi::AnyBuffer c,
                          ffi::AnyBuffer dQt, ffi::AnyBuffer dH, ffi::AnyBuffer dr, ffi::AnyBuffer dc,
                          ffi::RemainingArgs params, ffi::Result<ffi::AnyBuffer> dv, ffi::Result<ffi::AnyBuffer> Lambda,
                          ffi::Result<ffi::AnyBuffer> workspace, ffi::RemainingRets dparams, int64_t op_handle,
                          int64_t flags, int64_t dense_cotangents) {
  bl_operator_t* op = as_op(op_handle);
  const int dtype = dtype_of(H.element_type());
  const int64_t K = H.dimensions().back(), ld = Qt.dimensions().back(), n = dv->dimensions().back();
  BL_FFI_TRY(bind_params(op, dtype, params, stream));
  BL_FFI_TRY(to_error(bl_op_grad_zero(op, dtype, stream)));
  const void* dQp = (dense_cotangents & 1) ? dQt.untyped_data() : nullptr;
  const void* drp = (dense_cotangents & 2) ? dr.untyped_data() : nullptr;
  const void* dcp = (dense_cotangents & 4) ? dc.untyped_data() : nullptr;
  int rc;
  if (is_batched(H, 2))
    rc = bl_arnoldi_adjoint_batch(op, dtype, n, K, (int)flags, batch_of(H, 2), Qt.untyped_data(), ld, H.untyped_data(),
                                  r.untyped_data(), c.untyped_data(), dQp, dH.untyped_data(), drp, dcp,
                                  dv->untyped_data(), n, Lambda->untyped_data(), workspace->untyped_data(),
                                  workspace->size_bytes(), stream);
  else
    rc = bl_arnoldi_adjoint(op, dtype, n, K, (int)flags, Qt.untyped_data(), ld, H.untyped_data(), r.untyped_data(),
                            c.untyped_data(), dQp, dH.untyped_data(), drp, dcp, dv->untyped_data(),
                            Lambda->untyped_data(), workspace->untyped_data(), workspace->size_bytes(), stream);
  BL_FFI_TRY(to_error(rc));
  return export_grads(op, dtype, dparams, stream);
}

// ---- three-term Lanczos (lanczos.py:215-285) and its adjoint (lanczos.py:288-335) -----------------------------
ffi::Error Lanczos3Forward(cudaStream_t stream, ffi::AnyBuffer v, ffi::RemainingArgs params,
                           ffi::Result<ffi::AnyBuffer> xs, ffi::Result<ffi::AnyBuffer> alphas,
                           ffi::Result<ffi::AnyBuffer> betas, ffi::Result<ffi::AnyBuffer> workspace, int64_t op_handle,
                           int64_t krylov_depth) {
  bl_operator_t* op = as_op(op_handle);
  const int dtype = dtype_of(v.element_type());
  BL_FFI_TRY(bind_params(op, dtype, params, stream));
  return to_error(bl_lanczos3_forward(op, dtype, v.dimensions().back(), krylov_depth, v.untyped_data(),
                                      xs->untyped_data(), xs->dimensions().back(), alphas->untyped_data(),
                                      betas->untyped_data(), workspace->untyped_data(), workspace->size_bytes(), stream));
}

// exactly one parameter array (lanczos.py:329); `dense_dxs` = 0 for a zero cotangent of the basis
ffi::Error Lanczos3Adjoint(cudaStream_t stream, ffi::AnyBuffer xs, ffi::AnyBuffer alphas, ffi::AnyBuffer betas,
                           ffi::AnyBuffer dxs, ffi::AnyBuffer dalphas, ffi::AnyBuffer dbetas, ffi::AnyBuffer vnorm,
                           ffi::RemainingArgs params, ffi::Result<ffi::AnyBuffer> dv,
                           ffi::Result<ffi::AnyBuffer> workspace, ffi::RemainingRets dparams, int64_t op_handle,
                           int64_t dense_dxs) {
  bl_operator_t* op = as_op(op_handle);
  const int dtype = dtype_of(alphas.element_type());
  if (params.size() != 1 || dparams.size() != 1)
    return ffi::Error::InvalidArgument("the three-term adjoint supports exactly one parameter array (lanczos.py:329)");
  const int64_t K = alphas.dimensions().back(), n = dv->dimensions().back();
  BL_FFI_TRY(bind_params(op, dtype, params, stream));
  BL_FFI_TRY(to_error(bl_op_grad_zero(op, dtype, stream)));
  BL_FFI_TRY(to_error(bl_lanczos3_adjoint(op, dtype, n, K, xs.untyped_data(), xs.dimensions().back(),
                                          alphas.untyped_data(), betas.untyped_data(),
                                          dense_dxs ? dxs.untyped_data() : nullptr, dalphas.untyped_data(),
                                          dbetas.untyped_data(), vnorm.untyped_data(), dv->untyped_data(),
                                          workspace->untyped_data(), workspace->size_bytes(), stream)));
  return export_grads(op, dtype, dparams, stream);
}

// ---- the solver half of the GP path (cg.py:20-131, low_rank.py:10-225) ----------------------------------------
// atol < 0: pcg_fixed_step(max_steps); atol >= 0: pcg_adaptive (the C entry point synchronises to read its flag).
ffi::Error PcgSolve(cudaStream_t stream, ffi::AnyBuffer b, ffi::RemainingArgs params, ffi::Result<ffi::AnyBuffer> x,
                    ffi::Result<ffi::AnyBuffer> r, ffi::Result<ffi::AnyBuffer> num_steps,
                    ffi::Result<ffi::AnyBuffer> workspace, int64_t op_handle, int64_t precond_handle, int64_t max_steps,
                    int64_t min_steps, double atol, double rtol, int64_t check_every) {
  bl_operator_t* op = as_op(op_handle);
  const int dtype = dtype_of(b.element_type());
  BL_FFI_TRY(bind_params(op, dtype, params, stream));
  int64_t steps = 0;
  BL_FFI_TRY(to_error(bl_pcg_solve(op, dtype, b.dimensions().back(), b.untyped_data(),
                                   reinterpret_cast<bl_precond_t*>(precond_handle), max_steps, min_steps, atol, rtol,
                                   (int)check_every, x->untyped_data(), r->untyped_data(), &steps,
                                   workspace->untyped_data(), workspace->size_bytes(), stream)));
  // `steps` is a stack variable: the copy must have completed before this frame returns
  if (cudaMemcpyAsync(num_steps->untyped_data(), &steps, sizeof(steps), cudaMemcpyHostToDevice, stream) != cudaSuccess ||
      cudaStreamSynchronize(stream) != cudaSuccess)
    return ffi::Error::Internal("copy of num_steps failed");
  return ffi::Error::Success();
}

// B, X, R (count, ld): the rows of B solved in lockstep (jax.vmap of the solve); num_steps (s64, count)
ffi::Error PcgSolveBatch(cudaStream_t stream, ffi::AnyBuffer B, ffi::RemainingArgs params, ffi::Result<ffi::AnyBuffer> X,
                         ffi::Result<ffi::AnyBuffer> R, ffi::Result<ffi::AnyBuffer> num_steps,
                         ffi::Result<ffi::AnyBuffer> workspace, int64_t op_handle, int64_t precond_handle,
                         int64_t max_steps, int64_t min_steps, double atol, double rtol, int64_t check_every) {
  bl_operator_t* op = as_op(op_handle);
  const int dtype = dtype_of(B.element_type());
  const int64_t count = B.dimensions()[0], ld = B.dimensions()[1];
  int64_t n = 0;
  BL_FFI_TRY(to_error(bl_op_size(op, &n)));
  BL_FFI_TRY(bind_params(op, dtype, params, stream));
  std::vector<int64_t> steps((size_t)count);
  BL_FFI_TRY(to_error(bl_pcg_solve_batch(op, dtype, n, count, B.untyped_data(), ld,
                                         reinterpret_cast<bl_precond_t*>(precond_handle), max_steps, min_steps, atol,
                                         rtol, (int)check_every, X->untyped_data(), R->untyped_data(), steps.data(),
                                         workspace->untyped_data(), workspace->size_bytes(), stream)));
  // `steps` lives in this frame: the copy must have completed before it returns
  if (cudaMemcpyAsync(num_steps->untyped_data(), steps.data(), sizeof(int64_t) * steps.size(), cudaMemcpyHostToDevice,
                      stream) != cudaSuccess ||
      cudaStreamSynchronize(stream) != cudaSuccess)
    return ffi::Error::Internal("copy of num_steps failed");
  return ffi::Error::Success();
}

// y = K(X*, X) v of a bl_gram_cross_t whose parent Gram operator is bound with `params` first
ffi::Error GramCrossMatvec(cudaStream_t stream, ffi::AnyBuffer v, ffi::RemainingArgs params,
                           ffi::Result<ffi::AnyBuffer> y, int64_t op_handle, int64_t cross_handle) {
  bl_operator_t* op = as_op(op_handle);
  const int dtype = dtype_of(v.element_type());
  BL_FFI_TRY(bind_params(op, dtype, params, stream));
  return to_error(bl_gram_cross_matvec(reinterpret_cast<bl_gram_cross_t*>(cross_handle), dtype, v.untyped_data(),
                                       y->untyped_data(), stream));
}

ffi::Error PrecondApply(cudaStream_t stream, ffi::AnyBuffer v, ffi::Result<ffi::AnyBuffer> out, int64_t precond_handle) {
  return to_error(bl_precond_apply(reinterpret_cast<bl_precond_t*>(precond_handle), dtype_of(v.element_type()),
                                   v.untyped_data(), out->untyped_data(), stream));
}

// L_rows (rank, ld), success (s32 scalar), pivots (s64, rank) -- low_rank.py:63-225
ffi::Error CholeskyPartial(cudaStream_t stream, ffi::RemainingArgs params, ffi::Result<ffi::AnyBuffer> L_rows,
                           ffi::Result<ffi::AnyBuffer> success, ffi::Result<ffi::AnyBuffer> pivots,
                           ffi::Result<ffi::AnyBuffer> workspace, int64_t op_handle, int64_t n, int64_t pivot) {
  bl_operator_t* op = as_op(op_handle);
  const int dtype = dtype_of(L_rows->element_type());
  const int64_t rank = L_rows->dimensions()[0], ld = L_rows->dimensions()[1];
  if (rank > 4096) return ffi::Error::InvalidArgument("rank too large for the shim's pivot buffer");
  BL_FFI_TRY(bind_params(op, dtype, params, stream));
  int ok = 0;
  int64_t piv[4096];
  BL_FFI_TRY(to_error(bl_cholesky_partial(op, dtype, n, rank, (int)pivot, L_rows->untyped_data(), ld, &ok, piv,
                                          workspace->untyped_data(), workspace->size_bytes(), stream)));
  if (cudaMemcpyAsync(success->untyped_data(), &ok, sizeof(ok), cudaMemcpyHostToDevice, stream) != cudaSuccess ||
      cudaMemcpyAsync(pivots->untyped_data(), piv, sizeof(int64_t) * (size_t)rank, cudaMemcpyHostToDevice, stream) !=
          cudaSuccess ||
      cudaStreamSynchronize(stream) != cudaSuccess)
    return ffi::Error::Internal("copy of the Cholesky flags failed");
  return ffi::Error::Success();
}

}  // namespace

#define BL_STREAM ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>()
using Buf = ffi::AnyBuffer;

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_matvec, Matvec,
                              BL_STREAM.Arg<Buf>().RemainingArgs().Ret<Buf>().Attr<int64_t>("op_handle"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_matvec_vjp, MatvecVjp,
                              BL_STREAM.Arg<Buf>().Arg<Buf>().RemainingArgs().Ret<Buf>().RemainingRets().Attr<int64_t>(
                                  "op_handle"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_arnoldi_forward, ArnoldiForward,
                              BL_STREAM.Arg<Buf>()  // v
                                  .RemainingArgs()  // *params
                                  .Ret<Buf>()       // Qt
                                  .Ret<Buf>()       // H
                                  .Ret<Buf>()       // r
                                  .Ret<Buf>()       // c
                                  .Ret<Buf>()       // workspace
                                  .Attr<int64_t>("op_handle")
                                  .Attr<int64_t>("krylov_depth")
                                  .Attr<int64_t>("flags"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_arnoldi_adjoint, ArnoldiAdjoint,
                              BL_STREAM.Arg<Buf>()  // Qt
                                  .Arg<Buf>()       // H
                                  .Arg<Buf>()       // r
                                  .Arg<Buf>()       // c
                                  .Arg<Buf>()       // dQt
                                  .Arg<Buf>()       // dH
                                  .Arg<Buf>()       // dr
                                  .Arg<Buf>()       // dc
                                  .RemainingArgs()  // *params
                                  .Ret<Buf>()       // dv
                                  .Ret<Buf>()       // Lambda
                                  .Ret<Buf>()       // workspace
                                  .RemainingRets()  // *dparams
                                  .Attr<int64_t>("op_handle")
                                  .Attr<int64_t>("flags")
                                  .Attr<int64_t>("dense_cotangents"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_lanczos3_forward, Lanczos3Forward,
                              BL_STREAM.Arg<Buf>()
                                  .RemainingArgs()
                                  .Ret<Buf>()  // xs (K+1, ld)
                                  .Ret<Buf>()  // alphas
                                  .Ret<Buf>()  // betas
                                  .Ret<Buf>()  // workspace
                                  .Attr<int64_t>("op_handle")
                                  .Attr<int64_t>("krylov_depth"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_lanczos3_adjoint, Lanczos3Adjoint,
                              BL_STREAM.Arg<Buf>()  // xs
                                  .Arg<Buf>()       // alphas
                                  .Arg<Buf>()       // betas
                                  .Arg<Buf>()       // dxs
                                  .Arg<Buf>()       // dalphas
                                  .Arg<Buf>()       // dbetas
                                  .Arg<Buf>()       // vnorm
                                  .RemainingArgs()
                                  .Ret<Buf>()  // dv
                                  .Ret<Buf>()  // workspace
                                  .RemainingRets()
                                  .Attr<int64_t>("op_handle")
                                  .Attr<int64_t>("dense_dxs"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_pcg_solve, PcgSolve,
                              BL_STREAM.Arg<Buf>()
                                  .RemainingArgs()
                                  .Ret<Buf>()  // x
                                  .Ret<Buf>()  // r
                                  .Ret<Buf>()  // num_steps (s64)
                                  .Ret<Buf>()  // workspace
                                  .Attr<int64_t>("op_handle")
                                  .Attr<int64_t>("precond_handle")
                                  .Attr<int64_t>("max_steps")
                                  .Attr<int64_t>("min_steps")
                                  .Attr<double>("atol")
                                  .Attr<double>("rtol")
                                  .Attr<int64_t>("check_every"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_pcg_solve_batch, PcgSolveBatch,
                              BL_STREAM.Arg<Buf>()  // B (count, ld)
                                  .RemainingArgs()
                                  .Ret<Buf>()  // X
                                  .Ret<Buf>()  // R
                                  .Ret<Buf>()  // num_steps (s64, count)
                                  .Ret<Buf>()  // workspace
                                  .Attr<int64_t>("op_handle")
                                  .Attr<int64_t>("precond_handle")
                                  .Attr<int64_t>("max_steps")
                                  .Attr<int64_t>("min_steps")
                                  .Attr<double>("atol")
                                  .Attr<double>("rtol")
                                  .Attr<int64_t>("check_every"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_gram_cross_matvec, GramCrossMatvec,
                              BL_STREAM.Arg<Buf>()  // v (n)
                                  .RemainingArgs()  // the parent's params
                                  .Ret<Buf>()       // y (M)
                                  .Attr<int64_t>("op_handle")
                                  .Attr<int64_t>("cross_handle"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_precond_apply, PrecondApply,
                              BL_STREAM.Arg<Buf>().Ret<Buf>().Attr<int64_t>("precond_handle"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(bl_ffi_cholesky_partial, CholeskyPartial,
                              BL_STREAM.RemainingArgs()
                                  .Ret<Buf>()  // L_rows
                                  .Ret<Buf>()  // success
                                  .Ret<Buf>()  // pivots
                                  .Ret<Buf>()  // workspace
                                  .Attr<int64_t>("op_handle")
                                  .Attr<int64_t>("n")
                                  .Attr<int64_t>("pivot"));
