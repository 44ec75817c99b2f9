// Linear solves of the GP path: preconditioned conjugate gradients, (pivoted) partial Cholesky of a
// lazily evaluated matrix, and the low-rank preconditioner built from it.
//
// Reference behaviour replaced (all under /root/reference/src/matfree_extensions/):
//   cg.py:20-62    pcg_fixed_step        cg.py:75-131   pcg_adaptive      cg.py:196-213  _safe_divide
//   low_rank.py:63-118  cholesky_partial      low_rank.py:120-225  cholesky_partial_pivot
//   low_rank.py:10-60   preconditioner: (s I + L L^T)^{-1} v by the Woodbury identity
//
// Everything stays on the stream: step lengths, residual norms, the convergence flag, the pivot
// permutation and the pivot index live in device memory; every kernel that reduces ends with the
// deterministic "partials + last block" scheme and lets that last block update the scalars.  The
// fixed-step solver never synchronises; the adaptive one reads the flags back every `check_every`
// iterations (iterations after convergence are frozen on the device, so the result is the state at
// exactly the iteration where the reference's while_loop stops).  Several right-hand sides run in
// lockstep as columns of one grid (blockIdx.y = column, each with its own scalars): every column follows
// exactly the rules of a single solve.
#include <climits>
#include <cmath>
#include <vector>

#include "operators.cuh"

namespace bl {
namespace {

constexpr int kThreads = 256;
constexpr int kMaxGrid = 296;  // 2 blocks per SM on 148 SMs

enum Scal { S_RZ = 0, S_PAP, S_ALPHA, S_BETA, S_ERR2, S_ACTIVE, S_NSTEPS, S_LII, S_SUCCESS, S_PIVOT, S_N };

template <typename T>
struct EpsSq;
template <>
struct EpsSq<float> {
  static __device__ float v() { return 1.1920928955078125e-07f * 1.1920928955078125e-07f; }
};
template <>
struct EpsSq<double> {
  static __device__ double v() { return 2.220446049250313e-16 * 2.220446049250313e-16; }
};
// cg.py:196-213: a / b where |b| > eps^2, else a (so a converged iteration divides 0 by 1)
template <typename T>
__device__ __forceinline__ T safe_divide(T a, T b) {
  return fabs(b) > EpsSq<T>::v() ? a / b : a;
}

int grid_for(int64_t n) { return (int)std::max<int64_t>(1, std::min<int64_t>(kMaxGrid, (n + kThreads - 1) / kThreads)); }

// block partial -> partials[blockIdx.x]; returns true in the last block (of this column's gridDim.x blocks)
// with the total in *total
__device__ __forceinline__ bool reduce_to_last(double v, double* partials, unsigned int* counter, double* total) {
  __shared__ double red[32];
  __shared__ double tot;
  double s = block_sum(v, red);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
  if (!last_block_done(counter, gridDim.x)) return false;
  double acc = 0.0;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) acc += partials[b];
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) tot = acc;
  __syncthreads();
  *total = tot;
  return true;
}

enum DotMode { DOT_INIT = 0, DOT_PAP = 1, DOT_RZ = 2 };

// Column c = blockIdx.y of a lockstep solve: its vectors start at row c (stride ld), its scalars, block
// partials and counter are its own.
struct Column {
  int64_t off;
  double* scal;
  double* partials;
  unsigned int* counter;
};
__device__ __forceinline__ Column column_of(int64_t ld, double* scal, double* partials, unsigned int* counter) {
  const int c = blockIdx.y;
  return Column{(int64_t)c * ld, scal + (size_t)c * S_N, partials + (size_t)c * kMaxGrid, counter + c};
}

// d = <x, y>, then (last block):
//   DOT_INIT : rz = d                                          cg.py:31-33 (the first dot(r, z))
//   DOT_PAP  : alpha = safe_divide(rz, d)                      cg.py:46
//   DOT_RZ   : beta = safe_divide(d, rz); rz = d               cg.py:55
// DOT_PAP / DOT_RZ of a frozen column are skipped: nothing reads their results any more.
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cg_dot(int64_t n, int64_t ld, const T* __restrict__ x,
                                                       const T* __restrict__ y, double* partials, unsigned int* counter,
                                                       double* scal_all, int mode) {
  const Column col = column_of(ld, scal_all, partials, counter);
  double* scal = col.scal;
  if (mode != DOT_INIT && scal[S_ACTIVE] == 0.0) return;  // uniform over the column's blocks
  x += col.off, y += col.off;
  double acc = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    acc += static_cast<double>(x[i]) * static_cast<double>(y[i]);
  double d;
  if (!reduce_to_last(acc, col.partials, col.counter, &d)) return;
  if (threadIdx.x != 0) return;
  const T dt = static_cast<T>(d);
  if (mode == DOT_INIT) {
    scal[S_RZ] = dt;
  } else if (mode == DOT_PAP) {
    scal[S_PAP] = dt;
    scal[S_ALPHA] = safe_divide<T>(static_cast<T>(scal[S_RZ]), dt);
  } else {
    scal[S_BETA] = safe_divide<T>(dt, static_cast<T>(scal[S_RZ]));
    scal[S_RZ] = dt;
  }
}

// x += alpha p ; r -= alpha Ap ; err2 = sum (r / (atol + |x| rtol))^2       cg.py:47-50, 104-111
// frozen (no update) once the convergence flag of the previous iteration is down.
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_cg_update_xr(int64_t n, int64_t ld, const T* __restrict__ p, const T* __restrict__ Ap, T* __restrict__ x,
               T* __restrict__ r, double atol, double rtol, long long miniter, long long maxiter, double* partials,
               unsigned int* counter, double* scal_all) {
  const Column col = column_of(ld, scal_all, partials, counter);
  double* scal = col.scal;
  p += col.off, Ap += col.off, x += col.off, r += col.off;
  const bool active = scal[S_ACTIVE] != 0.0;
  const bool adaptive = atol >= 0.0;
  if (!active) return;  // every block takes the same branch: the flag only changes in the last block below
  const T a = static_cast<T>(scal[S_ALPHA]);
  double acc = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const T xn = x[i] + a * p[i];
    const T rn = r[i] - a * Ap[i];
    x[i] = xn;
    r[i] = rn;
    if (adaptive) {
      const T e = rn / (static_cast<T>(atol) + fabs(xn) * static_cast<T>(rtol));
      acc += static_cast<double>(e) * static_cast<double>(e);
    }
  }
  double tot;
  if (!reduce_to_last(acc, col.partials, col.counter, &tot)) return;
  if (threadIdx.x != 0) return;
  const double steps = scal[S_NSTEPS] + 1.0;
  scal[S_NSTEPS] = steps;
  scal[S_ERR2] = tot;
  if (adaptive) {
    const bool large = sqrt(tot / (double)n) > 1.0;
    scal[S_ACTIVE] = ((large || steps < (double)miniter) && steps < (double)maxiter) ? 1.0 : 0.0;
  }
}

// the cond of the adaptive loop on the initial state x = 0, r = b            cg.py:104-113
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_cg_init(int64_t n, int64_t ld, const T* __restrict__ b, T* __restrict__ x, T* __restrict__ r, double atol,
          long long miniter, long long maxiter, double* partials, unsigned int* counter, double* scal_all) {
  const Column col = column_of(ld, scal_all, partials, counter);
  double* scal = col.scal;
  b += col.off, x += col.off, r += col.off;
  double acc = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    x[i] = T(0);
    r[i] = b[i];  // b - A(0)
    if (atol >= 0.0) {
      const T e = b[i] / static_cast<T>(atol);
      acc += static_cast<double>(e) * static_cast<double>(e);
    }
  }
  double tot;
  if (!reduce_to_last(acc, col.partials, col.counter, &tot)) return;
  if (threadIdx.x != 0) return;
  scal[S_NSTEPS] = 0.0;
  scal[S_ERR2] = tot;
  if (atol >= 0.0)
    scal[S_ACTIVE] = ((sqrt(tot / (double)n) > 1.0 || 0 < miniter) && 0 < maxiter) ? 1.0 : 0.0;
  else
    scal[S_ACTIVE] = 1.0;
}

// p = z + beta p   (beta == nullptr: p = z)                                  cg.py:56, 34
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cg_update_p(int64_t n, int64_t ld, const T* __restrict__ z,
                                                            T* __restrict__ p, const double* scal_all, bool first) {
  const int64_t off = (int64_t)blockIdx.y * ld;
  const double* scal = scal_all + (size_t)blockIdx.y * S_N;
  z += off, p += off;
  if (!first && scal[S_ACTIVE] == 0.0) return;
  const T b = first ? T(0) : static_cast<T>(scal[S_BETA]);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = first ? z[i] : z[i] + b * p[i];
}

// ---- low-rank preconditioner ------------------------------------------------------------------
// t[k] = <L_k, v_k>  (one block per row k; L_k = k-th column of the factor, stored as a row of length n;
// ldv = 0: one vector v for every row)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_rows_dot(int64_t n, const T* __restrict__ L, int64_t ld,
                                                         const T* __restrict__ v, int64_t ldv, double* __restrict__ t) {
  __shared__ double red[32];
  const T* row = L + (int64_t)blockIdx.x * ld;
  v += (int64_t)blockIdx.x * ldv;
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += static_cast<double>(row[i]) * static_cast<double>(v[i]);
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) t[blockIdx.x] = acc;
}
// G[a][b] = <L_a, L_b>
template <typename T>
__global__ void __launch_bounds__(kThreads) k_rows_gram(int64_t n, int rank, const T* __restrict__ L, int64_t ld,
                                                          double* __restrict__ G) {
  __shared__ double red[32];
  const int a = blockIdx.x, b = blockIdx.y;
  if (b > a) return;
  const T* ra = L + (int64_t)a * ld;
  const T* rb = L + (int64_t)b * ld;
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += static_cast<double>(ra[i]) * static_cast<double>(rb[i]);
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) G[(size_t)a * rank + b] = G[(size_t)b * rank + a] = acc;
}
// w = M t   (rank x rank doubles, one block)
__global__ void __launch_bounds__(kThreads) k_small_matvec(int rank, const double* __restrict__ M,
                                                             const double* __restrict__ t, double* __restrict__ w) {
  for (int a = threadIdx.x; a < rank; a += blockDim.x) {
    double acc = 0.0;
    for (int b = 0; b < rank; ++b) acc += M[(size_t)a * rank + b] * t[b];
    w[a] = acc;
  }
}
// out = (v - sum_k w_k L_k) / s
template <typename T>
__global__ void __launch_bounds__(kThreads) k_precond_combine(int64_t n, int rank, const T* __restrict__ L, int64_t ld,
                                                                const double* __restrict__ w, const T* __restrict__ v,
                                                                double s, T* __restrict__ out) {
  extern __shared__ double wsm[];
  for (int k = threadIdx.x; k < rank; k += blockDim.x) wsm[k] = w[k];
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double acc = static_cast<double>(v[i]);
    for (int k = 0; k < rank; ++k) acc -= wsm[k] * static_cast<double>(L[(int64_t)k * ld + i]);
    out[i] = static_cast<T>(acc / s);
  }
}

// ---- partial Cholesky -------------------------------------------------------------------------
// Step i, pivoted (low_rank.py:171-203): res[pos] = |diag[perm[pos]] - sum_k L_k[perm[pos]]^2|, first
// arg-max over positions, swap perm[i] <-> perm[kpos]; the last block then stores the pivot (original
// index), l_ii = sqrt(diag[piv] - |L[piv]|^2), the success flag and the coefficients c_k = L_k[piv].
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_chol_pivot(int64_t n, int i, bool pivot, const T* __restrict__ diag, const T* __restrict__ L, int64_t ld,
             long long* __restrict__ perm, double* pval, long long* ppos, unsigned int* counter, double* scal,
             long long* piv_out, double* coef) {
  __shared__ double sval[kThreads];
  __shared__ long long spos[kThreads];
  double best = -1.0;
  long long bpos = 0x7fffffffffffffffll;
  if (pivot) {
    for (int64_t pos = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pos < n; pos += (int64_t)gridDim.x * blockDim.x) {
      const long long j = perm[pos];
      T acc = T(0);
      for (int k = 0; k < i; ++k) {
        const T l = L[(int64_t)k * ld + j];
        acc = fma(l, l, acc);  // jax.vmap(jnp.dot)(L, L)
      }
      const double res = fabs(static_cast<double>(diag[j] - acc));
      if (res > best || (res == best && pos < bpos)) best = res, bpos = pos;
    }
  }
  sval[threadIdx.x] = best;
  spos[threadIdx.x] = bpos;
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      const double v2 = sval[threadIdx.x + o];
      const long long p2 = spos[threadIdx.x + o];
      if (v2 > sval[threadIdx.x] || (v2 == sval[threadIdx.x] && p2 < spos[threadIdx.x]))
        sval[threadIdx.x] = v2, spos[threadIdx.x] = p2;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) pval[blockIdx.x] = sval[0], ppos[blockIdx.x] = spos[0];
  if (!last_block_done(counter)) return;
  __shared__ long long piv_s;
  if (threadIdx.x == 0) {
    long long piv = i;
    if (pivot) {
      double bv = -1.0;
      long long bp = 0x7fffffffffffffffll;
      for (int b = 0; b < (int)gridDim.x; ++b)
        if (pval[b] > bv || (pval[b] == bv && ppos[b] < bp)) bv = pval[b], bp = ppos[b];
      const long long a = perm[i], c = perm[bp];
      perm[i] = c;
      perm[bp] = a;
      piv = c;
    }
    piv_s = piv;
    piv_out[0] = piv;
  }
  __syncthreads();
  const long long piv = piv_s;
  for (int k = threadIdx.x; k < i; k += blockDim.x) coef[k] = static_cast<double>(L[(int64_t)k * ld + piv]);
  __syncthreads();
  if (threadIdx.x == 0) {
    T acc = T(0);
    for (int k = 0; k < i; ++k) {
      const T l = static_cast<T>(coef[k]);
      acc = fma(l, l, acc);
    }
    const T lsq = diag[piv] - acc;  // low_rank.py:194
    scal[S_LII] = static_cast<double>(sqrt(lsq));
    if (!(lsq > T(0))) scal[S_SUCCESS] = 0.0;  // :198
    scal[S_PIVOT] = (double)piv;
  }
}

// L_i[j] = (col[j] - sum_k c_k L_k[j]) / l_ii                               low_rank.py:196-197
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_chol_update(int64_t n, int i, const T* __restrict__ col, T* __restrict__ L, int64_t ld, const double* __restrict__ coef,
              const double* __restrict__ scal) {
  extern __shared__ double csm[];
  for (int k = threadIdx.x; k < i; k += blockDim.x) csm[k] = coef[k];
  __syncthreads();
  const T lii = static_cast<T>(scal[S_LII]);
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
    T acc = T(0);
    for (int k = 0; k < i; ++k) acc = fma(L[(int64_t)k * ld + j], static_cast<T>(csm[k]), acc);  // L @ L[i, :]
    L[(int64_t)i * ld + j] = (col[j] - acc) / lii;
  }
}

__global__ void k_iota(int64_t n, long long* perm) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) perm[i] = i;
}

struct Carve {
  char* p;
  size_t left;
  void* take(size_t bytes) {
    bytes = align_up(bytes, 256);
    if (bytes > left) return nullptr;
    void* r = p;
    p += bytes;
    left -= bytes;
    return r;
  }
};

}  // namespace
}  // namespace bl

using namespace bl;

// (s I + L L^T)^{-1}: L as `rank` rows of length n; M = (s I + L^T L)^{-1} (rank x rank) is formed on the
// host from the device-computed Gram matrix whenever the shift changes.
struct bl_precond {
  int dtype = BL_F32;
  int64_t n = 0, rank = 0, ld = 0;
  const void* L = nullptr;
  std::vector<double> G;  // rank x rank, L^T L
  double shift = -1.0;
  DevBuf M, t, w;
};

namespace {

// in-place inverse of a symmetric positive definite matrix (Cholesky), row-major r x r
int spd_inverse(std::vector<double>& a, int r) {
  std::vector<double> c(a);
  for (int j = 0; j < r; ++j) {
    double d = c[(size_t)j * r + j];
    for (int k = 0; k < j; ++k) d -= c[(size_t)j * r + k] * c[(size_t)j * r + k];
    if (!(d > 0.0)) return BL_EINVAL;
    d = std::sqrt(d);
    c[(size_t)j * r + j] = d;
    for (int i = j + 1; i < r; ++i) {
      double v = c[(size_t)i * r + j];
      for (int k = 0; k < j; ++k) v -= c[(size_t)i * r + k] * c[(size_t)j * r + k];
      c[(size_t)i * r + j] = v / d;
    }
  }
  // solve C C^T X = I column by column
  std::vector<double> y(r);
  for (int col = 0; col < r; ++col) {
    for (int i = 0; i < r; ++i) {
      double v = i == col ? 1.0 : 0.0;
      for (int k = 0; k < i; ++k) v -= c[(size_t)i * r + k] * y[k];
      y[i] = v / c[(size_t)i * r + i];
    }
    for (int i = r - 1; i >= 0; --i) {
      double v = y[i];
      for (int k = i + 1; k < r; ++k) v -= c[(size_t)k * r + i] * a[(size_t)k * r + col];
      a[(size_t)i * r + col] = v / c[(size_t)i * r + i];
    }
  }
  return BL_OK;
}

template <typename T>
int precond_apply_t(bl_precond* p, const T* v, T* out, cudaStream_t s) {
  const int r = (int)p->rank;
  k_rows_dot<T><<<r, kThreads, 0, s>>>(p->n, static_cast<const T*>(p->L), p->ld, v, 0, p->t.as<double>());
  BL_LAUNCHED();
  k_small_matvec<<<1, kThreads, 0, s>>>(r, p->M.as<double>(), p->t.as<double>(), p->w.as<double>());
  BL_LAUNCHED();
  k_precond_combine<T><<<grid_for(p->n), kThreads, (size_t)r * 8, s>>>(p->n, r, static_cast<const T*>(p->L), p->ld,
                                                                        p->w.as<double>(), v, p->shift, out);
  BL_LAUNCHED();
  return BL_OK;
}

// `count` columns of n values, row stride ld, in lockstep (count == 1: bl_pcg_solve)
template <typename T>
int pcg_t(bl_operator* op, int dtype, int64_t n, int64_t count, int64_t ld, const T* b, bl_precond* pre,
          int64_t max_steps, int64_t min_steps, double atol, double rtol, int check_every, T* x, T* r,
          int64_t* num_steps_host, void* workspace, size_t workspace_bytes, cudaStream_t s) {
  Carve w{static_cast<char*>(workspace), workspace_bytes};
  double* scal = static_cast<double*>(w.take((size_t)count * S_N * 8));
  double* partials = static_cast<double*>(w.take((size_t)count * kMaxGrid * 8));
  unsigned int* counter = static_cast<unsigned int*>(w.take((size_t)count * 4));
  T* p = static_cast<T*>(w.take((size_t)count * ld * sizeof(T)));
  T* Ap = static_cast<T*>(w.take((size_t)count * ld * sizeof(T)));
  T* z = pre ? static_cast<T*>(w.take((size_t)count * ld * sizeof(T))) : nullptr;
  BL_REQUIRE(scal && partials && counter && p && Ap && (!pre || z), "pcg workspace too small");
  BL_CUDA(cudaMemsetAsync(workspace, 0, reinterpret_cast<char*>(p) - static_cast<char*>(workspace), s));
  const dim3 g(grid_for(n), (unsigned)count);
  const bool adaptive = atol >= 0.0;
  std::vector<int64_t> live((size_t)count);  // columns not yet seen frozen by the host
  for (int64_t c = 0; c < count; ++c) live[c] = c;
  std::vector<const void*> in;
  std::vector<void*> out;
  k_cg_init<T><<<g, kThreads, 0, s>>>(n, ld, b, x, r, atol, (long long)min_steps, (long long)max_steps, partials,
                                      counter, scal);
  BL_LAUNCHED();
  auto precond = [&]() -> int {  // z = P(r) for the live columns
    for (int64_t c : live) BL_CHECK(precond_apply_t<T>(pre, r + c * ld, z + c * ld, s));
    return BL_OK;
  };
  const T* zz = pre ? z : r;
  if (pre) BL_CHECK(precond());
  k_cg_update_p<T><<<g, kThreads, 0, s>>>(n, ld, zz, p, scal, true);
  BL_LAUNCHED();
  k_cg_dot<T><<<g, kThreads, 0, s>>>(n, ld, r, zz, partials, counter, scal, DOT_INIT);
  BL_LAUNCHED();
  std::vector<double> host((size_t)count * S_N);
  bool polled = false;
  for (int64_t it = 0; it < max_steps; ++it) {
    if (live.size() == 1) {
      BL_CHECK(op->matvec(dtype, p + live[0] * ld, Ap + live[0] * ld, s));
    } else {
      in.clear(), out.clear();
      for (int64_t c : live) in.push_back(p + c * ld), out.push_back(Ap + c * ld);
      BL_CHECK(op->matvec_batch(dtype, (int)live.size(), in.data(), out.data(), s));
    }
    k_cg_dot<T><<<g, kThreads, 0, s>>>(n, ld, p, Ap, partials, counter, scal, DOT_PAP);
    BL_LAUNCHED();
    k_cg_update_xr<T><<<g, kThreads, 0, s>>>(n, ld, p, Ap, x, r, atol, rtol, (long long)min_steps,
                                             (long long)max_steps, partials, counter, scal);
    BL_LAUNCHED();
    if (pre) BL_CHECK(precond());
    k_cg_dot<T><<<g, kThreads, 0, s>>>(n, ld, r, zz, partials, counter, scal, DOT_RZ);
    BL_LAUNCHED();
    k_cg_update_p<T><<<g, kThreads, 0, s>>>(n, ld, zz, p, scal, false);
    BL_LAUNCHED();
    if (adaptive && ((it + 1) % check_every == 0 || it + 1 == max_steps)) {
      BL_CUDA(cudaMemcpyAsync(host.data(), scal, host.size() * 8, cudaMemcpyDeviceToHost, s));
      BL_CUDA(cudaStreamSynchronize(s));
      polled = true;
      std::vector<int64_t> still;
      for (int64_t c : live)
        if (host[(size_t)c * S_N + S_ACTIVE] != 0.0) still.push_back(c);
      live.swap(still);
      if (live.empty()) break;
    }
  }
  if (num_steps_host)
    for (int64_t c = 0; c < count; ++c)  // fixed steps: every column runs max_steps iterations
      num_steps_host[c] = !adaptive ? max_steps : polled ? (int64_t)host[(size_t)c * S_N + S_NSTEPS] : 0;
  return BL_OK;
}

template <typename T>
int cholesky_t(bl_operator* op, int dtype, int64_t n, int64_t rank, bool pivot, T* L, int64_t ld, int* success_host,
               int64_t* pivots_host, void* workspace, size_t workspace_bytes, cudaStream_t s) {
  Carve w{static_cast<char*>(workspace), workspace_bytes};
  double* scal = static_cast<double*>(w.take(S_N * 8));
  double* pval = static_cast<double*>(w.take(kMaxGrid * 8));
  long long* ppos = static_cast<long long*>(w.take(kMaxGrid * 8));
  unsigned int* counter = static_cast<unsigned int*>(w.take(256));
  long long* piv = static_cast<long long*>(w.take((size_t)rank * 8));
  double* coef = static_cast<double*>(w.take((size_t)rank * 8));
  long long* perm = static_cast<long long*>(w.take((size_t)n * 8));
  T* diag = static_cast<T*>(w.take((size_t)n * sizeof(T)));
  T* col = static_cast<T*>(w.take((size_t)n * sizeof(T)));
  BL_REQUIRE(scal && pval && ppos && counter && piv && coef && perm && diag && col, "cholesky workspace too small");
  BL_CUDA(cudaMemsetAsync(workspace, 0, 256 * 4 + 2 * align_up(kMaxGrid * 8, 256), s));
  const double one = 1.0;
  BL_CUDA(cudaMemcpyAsync(scal + S_SUCCESS, &one, 8, cudaMemcpyHostToDevice, s));
  const int g = grid_for(n);
  k_iota<<<g, kThreads, 0, s>>>(n, perm);
  BL_LAUNCHED();
  BL_CHECK(op->element_diagonal(dtype, diag, s));
  for (int i = 0; i < (int)rank; ++i) {
    k_chol_pivot<T><<<pivot ? g : 1, kThreads, 0, s>>>(n, i, pivot, diag, L, ld, perm, pval, ppos, counter, scal, piv + i, coef);
    BL_LAUNCHED();
    BL_CHECK(op->element_column(dtype, reinterpret_cast<const int64_t*>(piv + i), col, s));
    k_chol_update<T><<<g, kThreads, (size_t)std::max(i, 1) * 8, s>>>(n, i, col, L, ld, coef, scal);
    BL_LAUNCHED();
  }
  if (success_host || pivots_host) {
    double ok = 1.0;
    BL_CUDA(cudaMemcpyAsync(&ok, scal + S_SUCCESS, 8, cudaMemcpyDeviceToHost, s));
    if (pivots_host) BL_CUDA(cudaMemcpyAsync(pivots_host, piv, (size_t)rank * 8, cudaMemcpyDeviceToHost, s));
    BL_CUDA(cudaStreamSynchronize(s));
    if (success_host) *success_host = ok != 0.0;
  }
  return BL_OK;
}

}  // namespace

extern "C" {

size_t bl_pcg_workspace_bytes(int64_t n, int dtype) {
  return 256 * 3 + align_up(kMaxGrid * 8, 256) + 3 * align_up((size_t)n * dtype_size(dtype), 256) + 1024;
}

size_t bl_pcg_batch_workspace_bytes(int64_t n, int64_t count, int dtype) {
  return align_up((size_t)count * S_N * 8, 256) + align_up((size_t)count * kMaxGrid * 8, 256) +
         align_up((size_t)count * 4, 256) + 3 * align_up((size_t)count * n * dtype_size(dtype), 256) + 1024;
}

int bl_pcg_solve(bl_operator_t* op, int dtype, int64_t n, const void* b, bl_precond_t* precond, int64_t max_steps,
                 int64_t min_steps, double atol, double rtol, int check_every, void* x, void* r,
                 int64_t* num_steps_host, void* workspace, size_t workspace_bytes, void* stream) {
  BL_REQUIRE(op && b && x && r && workspace && n >= 1 && op->n == n && max_steps >= 0, "bad pcg arguments");
  BL_REQUIRE(dtype == BL_F32 || dtype == BL_F64, "bad dtype");
  BL_REQUIRE(!precond || (precond->n == n && precond->dtype == dtype && precond->shift > 0.0),
             "preconditioner does not match (or has no shift: bl_precond_set_shift)");
  if (check_every < 1) check_every = 8;
  cudaStream_t s = as_stream(stream);
  if (dtype == BL_F32)
    return pcg_t<float>(op, dtype, n, 1, n, (const float*)b, precond, max_steps, min_steps, atol, rtol, check_every,
                        (float*)x, (float*)r, num_steps_host, workspace, workspace_bytes, s);
  return pcg_t<double>(op, dtype, n, 1, n, (const double*)b, precond, max_steps, min_steps, atol, rtol, check_every,
                       (double*)x, (double*)r, num_steps_host, workspace, workspace_bytes, s);
}

int bl_pcg_solve_batch(bl_operator_t* op, int dtype, int64_t n, int64_t count, const void* B, int64_t ld,
                       bl_precond_t* precond, int64_t max_steps, int64_t min_steps, double atol, double rtol,
                       int check_every, void* X, void* R, int64_t* num_steps_host, void* workspace,
                       size_t workspace_bytes, void* stream) {
  BL_REQUIRE(op && B && X && R && workspace && n >= 1 && op->n == n && max_steps >= 0 && count >= 1 && count <= 65535,
             "bad batched pcg arguments (1 <= count <= 65535)");
  BL_REQUIRE(dtype == BL_F32 || dtype == BL_F64, "bad dtype");
  BL_REQUIRE(ld >= n && (ld * (int64_t)dtype_size(dtype)) % 16 == 0, "row stride must be >= n and a multiple of 16 bytes");
  BL_REQUIRE(!precond || (precond->n == n && precond->dtype == dtype && precond->shift > 0.0),
             "preconditioner does not match (or has no shift: bl_precond_set_shift)");
  if (check_every < 1) check_every = 8;
  cudaStream_t s = as_stream(stream);
  if (dtype == BL_F32)
    return pcg_t<float>(op, dtype, n, count, ld, (const float*)B, precond, max_steps, min_steps, atol, rtol, check_every,
                        (float*)X, (float*)R, num_steps_host, workspace, workspace_bytes, s);
  return pcg_t<double>(op, dtype, n, count, ld, (const double*)B, precond, max_steps, min_steps, atol, rtol,
                       check_every, (double*)X, (double*)R, num_steps_host, workspace, workspace_bytes, s);
}

int bl_rows_dot_pairs(int dtype, int64_t n, int64_t count, const void* X, const void* Y, int64_t ld, double* out,
                      void* stream) {
  BL_REQUIRE(X && Y && out && n >= 1 && count >= 1 && count <= INT32_MAX && ld >= n, "bad rows_dot_pairs arguments");
  BL_REQUIRE(dtype == BL_F32 || dtype == BL_F64, "bad dtype");
  cudaStream_t s = as_stream(stream);
  if (dtype == BL_F32)
    k_rows_dot<float><<<(unsigned)count, kThreads, 0, s>>>(n, (const float*)X, ld, (const float*)Y, ld, out);
  else
    k_rows_dot<double><<<(unsigned)count, kThreads, 0, s>>>(n, (const double*)X, ld, (const double*)Y, ld, out);
  BL_LAUNCHED();
  return BL_OK;
}

size_t bl_cholesky_workspace_bytes(int64_t n, int64_t rank, int dtype) {
  return 256 * 2 + 2 * align_up(kMaxGrid * 8, 256) + 2 * align_up((size_t)rank * 8, 256) + align_up((size_t)n * 8, 256) +
         2 * align_up((size_t)n * dtype_size(dtype), 256) + 1024;
}

int bl_cholesky_partial(bl_operator_t* op, int dtype, int64_t n, int64_t rank, int pivot, void* L_rows, int64_t ld,
                        int* success_host, int64_t* pivots_host, void* workspace, size_t workspace_bytes,
                        void* stream) {
  BL_REQUIRE(op && L_rows && workspace && op->n == n && ld >= n, "bad cholesky arguments");
  BL_REQUIRE(dtype == BL_F32 || dtype == BL_F64, "bad dtype");
  if (rank > n) {  // low_rank.py:67-69 / 124-126
    set_error("Rank exceeds n: " + std::to_string(rank) + " >= " + std::to_string(n) + ".");
    return BL_EINVAL;
  }
  if (rank < 1) {
    set_error("Rank must be positive, but " + std::to_string(rank) + " < 1.");
    return BL_EINVAL;
  }
  BL_REQUIRE(rank <= 4096, "rank above 4096 is not supported");
  cudaStream_t s = as_stream(stream);
  if (dtype == BL_F32)
    return cholesky_t<float>(op, dtype, n, rank, pivot != 0, (float*)L_rows, ld, success_host, pivots_host, workspace,
                             workspace_bytes, s);
  return cholesky_t<double>(op, dtype, n, rank, pivot != 0, (double*)L_rows, ld, success_host, pivots_host, workspace,
                            workspace_bytes, s);
}

int bl_precond_create(int dtype, int64_t n, int64_t rank, const void* L_rows, int64_t ld, void* stream,
                      bl_precond_t** out) {
  BL_REQUIRE(out && L_rows && n >= 1 && rank >= 1 && rank <= n && rank <= 4096 && ld >= n, "bad preconditioner arguments");
  BL_REQUIRE(dtype == BL_F32 || dtype == BL_F64, "bad dtype");
  auto* p = new bl_precond();
  p->dtype = dtype, p->n = n, p->rank = rank, p->ld = ld, p->L = L_rows;
  cudaStream_t s = as_stream(stream);
  DevBuf G;
  int rc = G.ensure((size_t)rank * rank * 8);
  if (rc == BL_OK) rc = p->M.ensure((size_t)rank * rank * 8);
  if (rc == BL_OK) rc = p->t.ensure((size_t)rank * 8);
  if (rc == BL_OK) rc = p->w.ensure((size_t)rank * 8);
  if (rc != BL_OK) {
    delete p;
    return rc;
  }
  dim3 grid((unsigned)rank, (unsigned)rank);
  if (dtype == BL_F32)
    k_rows_gram<float><<<grid, kThreads, 0, s>>>(n, (int)rank, (const float*)L_rows, ld, G.as<double>());
  else
    k_rows_gram<double><<<grid, kThreads, 0, s>>>(n, (int)rank, (const double*)L_rows, ld, G.as<double>());
  g_launches.fetch_add(1, std::memory_order_relaxed);
  p->G.resize((size_t)rank * rank);
  if (cudaMemcpyAsync(p->G.data(), G.p, (size_t)rank * rank * 8, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess) {
    set_error("preconditioner: Gram matrix of the factor failed");
    delete p;
    return BL_ECUDA;
  }
  *out = p;
  return BL_OK;
}

int bl_precond_set_shift(bl_precond_t* p, double shift, void* stream) {
  BL_REQUIRE(p && shift > 0.0, "the shift (noise) must be positive");
  const int r = (int)p->rank;
  std::vector<double> m(p->G);
  for (int k = 0; k < r; ++k) m[(size_t)k * r + k] += shift;
  BL_REQUIRE(spd_inverse(m, r) == BL_OK, "capacitance matrix is not positive definite");
  cudaStream_t s = as_stream(stream);
  BL_CUDA(cudaMemcpyAsync(p->M.p, m.data(), (size_t)r * r * 8, cudaMemcpyHostToDevice, s));
  BL_CUDA(cudaStreamSynchronize(s));  // `m` is a host temporary
  p->shift = shift;
  return BL_OK;
}

int bl_precond_apply(bl_precond_t* p, int dtype, const void* v, void* out, void* stream) {
  BL_REQUIRE(p && v && out && dtype == p->dtype && p->shift > 0.0, "bad preconditioner call (set the shift first)");
  cudaStream_t s = as_stream(stream);
  return dtype == BL_F32 ? precond_apply_t<float>(p, (const float*)v, (float*)out, s)
                         : precond_apply_t<double>(p, (const double*)v, (double*)out, s);
}

int bl_precond_destroy(bl_precond_t* p) {
  delete p;
  return BL_OK;
}

}  // extern "C"
