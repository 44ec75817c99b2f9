// Matrix-free Gram operator (K(X,X) + noise I) v for scaled Matern-3/2 / Matern-1/2 / RBF kernels.
//
// Reference behaviour replaced: `gram_matvec()(k)(X, X, v)` and its `jax.vjp`
// (/root/reference/src/matfree_extensions/util/gp_util.py:525-543; kernels :69-184; soft-plus
// constraint :187-201).  The kernel matrix is never formed: each block owns a tile of rows
// and sweeps column tiles staged in shared memory, recomputing
//   s2_ij = max(0, |x_i|^2 + |x_j|^2 - 2 x_i.x_j)   (the reference's expanded form, :87-92)
// on the fly.  One sweep gives y = K v; the adjoint sweep gives K lam and the cotangents of
// (raw_lengthscale, raw_outputscale, noise) in the same pass.
//
// Bound: FP32/FP64 ALU + MUFU (sqrt, ex2) per pair, not HBM (n*(d+2) values are read per
// column tile and reused by every row of the block).
#include <vector>

#include <cstdlib>
#include <map>
#include <mutex>

#include "gram_tc.cuh"
#include "operators.cuh"
#include "tma_pipeline.cuh"

namespace bl {
namespace {

constexpr int kMaxDim = 32;
constexpr int kTileI = 128;  // threads per block; a block owns kTileI * RI rows
constexpr int kTileJ = 64;   // points per staged column tile

template <typename T>
__device__ __forceinline__ T softplus_t(T x) {  // gp_util.py:188-199 (beta = 1, threshold = 20)
  return x < T(20) ? log(T(1) + exp(x)) : x;
}
template <typename T>
__device__ __forceinline__ T softplus_grad_t(T x) {
  return x < T(20) ? T(1) / (T(1) + exp(-x)) : T(1);
}

template <typename T>
struct Eps;
template <>
struct Eps<float> {
  static __device__ __forceinline__ float v() { return 1.1920928955078125e-07f; }
};
template <>
struct Eps<double> {
  static __device__ __forceinline__ double v() { return 2.220446049250313e-16; }
};

// scaled inputs xs = fac * x / softplus(raw_ls) in a zero-padded [n][DP] layout (16-byte rows, so
// a column tile is one contiguous TMA bulk copy), squared norms, constrained scales
template <typename T>
__global__ void k_gram_prepare(int64_t n, int d, int dp, int kind, const double* __restrict__ X,
                               const T* __restrict__ raw_ls, const T* __restrict__ raw_os,
                               T* __restrict__ xs, T* __restrict__ xx, T* __restrict__ consts) {
  const T fac = kind == 0 ? sqrt(T(3)) : T(1);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    T s = T(0);
    for (int k = 0; k < dp; ++k) {
      T v = T(0);
      if (k < d) {
        const T ls = softplus_t(raw_ls[k]);
        v = fac * static_cast<T>(X[i * d + k]) / ls;
        s = fma(v, v, s);  // jnp.dot(x, x)
      }
      xs[i * dp + k] = v;
    }
    xx[i] = s;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) consts[0] = softplus_t(raw_os[0]);
}

// ---- two rows at a time -----------------------------------------------------------------------
// Blackwell issues packed FP32 pairs (`fma.rn.f32x2`, SASS FFMA2): one FMA-pipe slot does two
// multiply-adds.  Every thread owns RI rows; rows (2p, 2p+1) travel as one pair through the
// distance contraction and the kernel epilogue, which halves the FMA-pipe work per kernel entry.
// fp64 uses the same code with a plain two-element struct.
template <typename T>
struct P2 {
  T a, b;
};
template <>
struct P2<float> {
  float2 v;
};

__device__ __forceinline__ P2<float> p2_set(float x, float y) { return {make_float2(x, y)}; }
__device__ __forceinline__ P2<double> p2_set(double x, double y) { return {x, y}; }
template <typename T>
__device__ __forceinline__ P2<T> p2_splat(T x) { return p2_set(x, x); }
__device__ __forceinline__ float p2_lo(const P2<float>& p) { return p.v.x; }
__device__ __forceinline__ float p2_hi(const P2<float>& p) { return p.v.y; }
__device__ __forceinline__ double p2_lo(const P2<double>& p) { return p.a; }
__device__ __forceinline__ double p2_hi(const P2<double>& p) { return p.b; }
__device__ __forceinline__ P2<float> p2_fma(const P2<float>& x, const P2<float>& y, const P2<float>& z) {
  return {__ffma2_rn(x.v, y.v, z.v)};
}
__device__ __forceinline__ P2<double> p2_fma(const P2<double>& x, const P2<double>& y, const P2<double>& z) {
  return {fma(x.a, y.a, z.a), fma(x.b, y.b, z.b)};
}
__device__ __forceinline__ P2<float> p2_mul(const P2<float>& x, const P2<float>& y) { return {__fmul2_rn(x.v, y.v)}; }
__device__ __forceinline__ P2<double> p2_mul(const P2<double>& x, const P2<double>& y) { return {x.a * y.a, x.b * y.b}; }
__device__ __forceinline__ P2<float> p2_add(const P2<float>& x, const P2<float>& y) { return {__fadd2_rn(x.v, y.v)}; }
__device__ __forceinline__ P2<double> p2_add(const P2<double>& x, const P2<double>& y) { return {x.a + y.a, x.b + y.b}; }

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// exp(-s) for a pair: fp32 = ex2.approx(-s * log2(e)) per component (MUFU), fp64 = library exp
__device__ __forceinline__ P2<float> p2_exp_neg(const P2<float>& s) {
  const P2<float> t = p2_mul(s, p2_splat(-1.4426950408889634f));
  return p2_set(ex2_approx(p2_lo(t)), ex2_approx(p2_hi(t)));
}
__device__ __forceinline__ P2<double> p2_exp_neg(const P2<double>& s) { return {exp(-s.a), exp(-s.b)}; }
// sqrt of strictly positive numbers: fp32 = x * rsqrt.approx(x), fp64 = IEEE sqrt
__device__ __forceinline__ P2<float> p2_sqrt_pos(const P2<float>& x) {
  return p2_mul(x, p2_set(rsqrtf(p2_lo(x)), rsqrtf(p2_hi(x))));
}
__device__ __forceinline__ P2<double> p2_sqrt_pos(const P2<double>& x) { return {sqrt(x.a), sqrt(x.b)}; }
template <typename T>
__device__ __forceinline__ P2<T> p2_recip(const P2<T>& x) { return p2_set(T(1) / p2_lo(x), T(1) / p2_hi(x)); }

// value and derivative (w.r.t. the clamped squared distance) of two kernel entries
template <typename T, int KIND, bool ADJ>
__device__ __forceinline__ void kernel_eval2(const P2<T>& sigma, const P2<T>& s2, P2<T>& k, P2<T>& dk_ds2) {
  if (KIND == 2) {  // RBF: sigma exp(-s2/2)
    k = p2_mul(sigma, p2_exp_neg(p2_mul(s2, p2_splat(T(0.5)))));
    if (ADJ) dk_ds2 = p2_mul(k, p2_splat(T(-0.5)));
  } else {
    const P2<T> s = p2_sqrt_pos(p2_add(s2, p2_splat(Eps<T>::v())));
    const P2<T> e = p2_mul(sigma, p2_exp_neg(s));  // sigma e^{-s}
    if (KIND == 0) {  // Matern-3/2: sigma (1+s) e^{-s};  dk/ds2 = -sigma e^{-s} / 2
      k = p2_fma(s, e, e);
      if (ADJ) dk_ds2 = p2_mul(e, p2_splat(T(-0.5)));
    } else {  // Matern-1/2: sigma e^{-s};  dk/ds2 = -k / (2 s)
      k = e;
      if (ADJ) dk_ds2 = p2_mul(p2_mul(e, p2_splat(T(-0.5))), p2_recip(s));
    }
  }
}

// Register-tiled sweep: a block owns kTileI * RI rows (thread t: rows i0 + t + 128 r), column
// tiles of kTileJ points arrive by TMA bulk copies (double-buffered: scaled inputs, squared
// norms, v / lam, q); every staged point is reused for RI kernel evaluations from registers.
// grid = (row tiles, column splits).
//   ADJ == false: part[split][i] = sum_{j in split} k_ij v_j
//   ADJ == true : part[split][i] = sum_j k_ij lam_j ; block partial sums of
//                 d_sigma = sum lam_i q_j k_ij / sigma and  d_ls[k] = sum lam_i q_j dk_ij (x_ik - x_jk)^2
// CROSS == true: the rows are the m points (xsa, xxa) of another set (a cross-covariance K(X*, X) v,
// part[split][m]); the columns stay the n points (xs, xx).
template <typename T, int DP, int RI, bool ADJ, int KIND, bool CROSS = false>
__global__ void __launch_bounds__(kTileI)
k_gram_sweep(int64_t n, int d, const T* __restrict__ xs, const T* __restrict__ xx,
             const T* __restrict__ consts, const T* __restrict__ v, const T* __restrict__ q,
             T* __restrict__ part, double* __restrict__ gpart /* [blocks][d+1] */, int64_t m,
             const T* __restrict__ xsa, const T* __restrict__ xxa) {
  static_assert(!(CROSS && ADJ), "the cross-covariance sweep has no adjoint");
  using V = typename Vec<T>::type;
  constexpr int VN = Vec<T>::N;
  constexpr int NV = DP / VN;
  __shared__ __align__(128) T sx[2][kTileJ * DP];
  __shared__ __align__(16) T sxx[2][kTileJ];
  __shared__ __align__(16) T sv[2][kTileJ];
  __shared__ __align__(16) T sq[2][kTileJ];
  __shared__ uint64_t full[2];
  __shared__ double red_smem[32];

  const int tid = threadIdx.x;
  const int64_t i0 = (int64_t)blockIdx.x * (kTileI * RI);
  const int64_t rows = CROSS ? m : n;
  const T* xsr = CROSS ? xsa : xs;
  const T* xxr = CROSS ? xxa : xx;
  static_assert(RI % 2 == 0, "rows are processed in pairs");
  constexpr int RP = RI / 2;
  const P2<T> sigma2 = p2_splat(consts[0]);
  P2<T> xi[RP][DP], xxi[RP], lam_i[RP];  // rows (2p, 2p+1) of this thread as packed pairs
  bool live[RI];
#pragma unroll
  for (int p = 0; p < RP; ++p) {
    const int64_t ia = i0 + tid + (int64_t)kTileI * (2 * p), ib = ia + kTileI;
    live[2 * p] = ia < rows;
    live[2 * p + 1] = ib < rows;
#pragma unroll
    for (int k = 0; k < DP; ++k)
      xi[p][k] = p2_set(live[2 * p] ? xsr[ia * DP + k] : T(0), live[2 * p + 1] ? xsr[ib * DP + k] : T(0));
    xxi[p] = p2_set(live[2 * p] ? xxr[ia] : T(0), live[2 * p + 1] ? xxr[ib] : T(0));
    lam_i[p] = p2_set((ADJ && live[2 * p]) ? v[ia] : T(0), (ADJ && live[2 * p + 1]) ? v[ib] : T(0));
  }

  const int64_t per = ((n + gridDim.y - 1) / gridDim.y + kTileJ - 1) / kTileJ * kTileJ;
  const int64_t j0 = per * blockIdx.y;
  const int64_t j1 = j0 + per < n ? j0 + per : n;
  const int ntiles = j0 < j1 ? (int)((j1 - j0 + kTileJ - 1) / kTileJ) : 0;

  if (tid == 0) {
    tma::mbar_init(full + 0, 1);
    tma::mbar_init(full + 1, 1);
    tma::fence_barrier_init();
  }
  __syncthreads();
  auto issue = [&](int t) {
    const int b = t & 1;
    const int64_t jt = j0 + (int64_t)t * kTileJ;
    const int w = (int)((j1 - jt) < kTileJ ? (j1 - jt) : kTileJ);
    const uint32_t wv = (uint32_t)((w + VN - 1) / VN * VN) * sizeof(T);  // 16-byte granules
    const uint32_t bx = (uint32_t)w * DP * sizeof(T);
    tma::mbar_arrive_expect_tx(full + b, bx + wv * (ADJ ? 3u : 2u));
    tma::bulk_g2s(sx[b], xs + jt * DP, bx, full + b);
    tma::bulk_g2s(sxx[b], xx + jt, wv, full + b);
    tma::bulk_g2s(sv[b], v + jt, wv, full + b);
    if (ADJ) tma::bulk_g2s(sq[b], q + jt, wv, full + b);
  };
  if (tid == 0 && ntiles > 0) issue(0);

  double y_acc[RI], dsig_acc = 0.0, dls_acc[DP];
#pragma unroll
  for (int r = 0; r < RI; ++r) y_acc[r] = 0.0;
#pragma unroll
  for (int k = 0; k < DP; ++k) dls_acc[k] = 0.0;

  for (int t = 0; t < ntiles; ++t) {
    const int b = t & 1;
    if (tid == 0 && t + 1 < ntiles) issue(t + 1);  // stage (t+1)&1 was released by the barrier below
    tma::mbar_wait(full + b, (t >> 1) & 1);
    const int64_t jt = j0 + (int64_t)t * kTileJ;
    const int w = (int)((j1 - jt) < kTileJ ? (j1 - jt) : kTileJ);
    P2<T> y_t[RP], dsig_t = p2_splat(T(0)), dls_t[DP];
#pragma unroll
    for (int p = 0; p < RP; ++p) y_t[p] = p2_splat(T(0));
#pragma unroll
    for (int k = 0; k < DP; ++k) dls_t[k] = p2_splat(T(0));
    for (int jj = 0; jj < w; ++jj) {
      T xj[DP];
#pragma unroll
      for (int u = 0; u < NV; ++u) {
        T tmp[VN];
        vec_unpack(reinterpret_cast<const V*>(sx[b] + (size_t)jj * DP)[u], tmp);  // broadcast load
#pragma unroll
        for (int k = 0; k < VN; ++k) xj[u * VN + k] = tmp[k];
      }
      const P2<T> xxj = p2_splat(sxx[b][jj]), vj = p2_splat(sv[b][jj]);
      const P2<T> qj = p2_splat(ADJ ? sq[b][jj] : T(0));
#pragma unroll
      for (int p = 0; p < RP; ++p) {
        P2<T> dot = p2_splat(T(0));
#pragma unroll
        for (int k = 0; k < DP; ++k) dot = p2_fma(xi[p][k], p2_splat(xj[k]), dot);
        // s2 = |x|^2 + |y|^2 - 2 x.y, clamped at zero                          gp_util.py:92-95
        const P2<T> raw = p2_fma(dot, p2_splat(T(-2)), p2_add(xxi[p], xxj));
        const bool pos_a = p2_lo(raw) > T(0), pos_b = p2_hi(raw) > T(0);
        const P2<T> s2 = p2_set(pos_a ? p2_lo(raw) : T(0), pos_b ? p2_hi(raw) : T(0));
        P2<T> kij, dk;
        kernel_eval2<T, KIND, ADJ>(sigma2, s2, kij, dk);
        y_t[p] = p2_fma(kij, vj, y_t[p]);
        if (ADJ) {
          const P2<T> wgt = p2_mul(lam_i[p], qj);
          dsig_t = p2_fma(wgt, kij, dsig_t);
          // derivative of max(0, .) is zero where it clamps
          const P2<T> g = p2_mul(p2_mul(wgt, dk), p2_set(pos_a ? T(1) : T(0), pos_b ? T(1) : T(0)));
#pragma unroll
          for (int k = 0; k < DP; ++k) {
            const P2<T> diff = p2_add(xi[p][k], p2_splat(-xj[k]));
            dls_t[k] = p2_fma(g, p2_mul(diff, diff), dls_t[k]);
          }
        }
      }
    }
#pragma unroll
    for (int p = 0; p < RP; ++p) {
      y_acc[2 * p] += static_cast<double>(p2_lo(y_t[p]));
      y_acc[2 * p + 1] += static_cast<double>(p2_hi(y_t[p]));
    }
    if (ADJ) {
      dsig_acc += static_cast<double>(p2_lo(dsig_t)) + static_cast<double>(p2_hi(dsig_t));
#pragma unroll
      for (int k = 0; k < DP; ++k)
        dls_acc[k] += static_cast<double>(p2_lo(dls_t[k])) + static_cast<double>(p2_hi(dls_t[k]));
    }
    __syncthreads();  // everyone is done with stage b
  }
#pragma unroll
  for (int r = 0; r < RI; ++r) {
    const int64_t i = i0 + tid + (int64_t)kTileI * r;
    if (live[r]) part[(int64_t)blockIdx.y * rows + i] = static_cast<T>(y_acc[r]);
  }
  if (ADJ) {
    // rows that are not live carry lam_i = 0, so their sums are already zero
    const int blk = blockIdx.y * gridDim.x + blockIdx.x;
    double rsum = block_sum(dsig_acc, red_smem);
    if (tid == 0) gpart[(size_t)blk * (d + 1) + d] = rsum;
#pragma unroll
    for (int k = 0; k < DP; ++k)
      if (k < d) {
        rsum = block_sum(dls_acc[k], red_smem);
        if (tid == 0) gpart[(size_t)blk * (d + 1) + k] = rsum;
      }
  }
}

// out[b * ldo + j] = k(x_j, z_c), c = (index ? *index : 0) + b + zstep * j, b = blockIdx.y: the lazy kernel
// of gp_util.py:257-258, same expanded squared distance as the sweeps.  z = x with zstep 0 gives the column
// of point *index, with zstep 1 the diagonal; z = other points with zstep 0 gives cross-covariance columns.
template <typename T>
__global__ void k_gram_elements(int64_t n, int dp, int kind, const T* __restrict__ xs, const T* __restrict__ xx,
                                const T* __restrict__ zs, const T* __restrict__ zz, int64_t zstep,
                                const T* __restrict__ consts, const int64_t* __restrict__ index, int64_t ldo,
                                T* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int64_t c = (index ? index[0] : 0) + blockIdx.y + zstep * j;
  T dot = T(0);
  for (int k = 0; k < dp; ++k) dot = fma(xs[j * dp + k], zs[c * dp + k], dot);
  T s2 = xx[j] + zz[c] - T(2) * dot;
  s2 = s2 > T(0) ? s2 : T(0);
  const T sigma = consts[0];
  T val;
  if (kind == 2) {
    val = sigma * exp(-s2 / T(2));
  } else {
    const T s = sqrt(s2 + Eps<T>::v());
    val = kind == 0 ? sigma * (T(1) + s) * exp(-s) : sigma * exp(-s);
  }
  out[(int64_t)blockIdx.y * ldo + j] = val;
}

// y[i] = sum_s part[s][i] + noise * v[i]   (noise == nullptr: no noise term -- a cross-covariance, whose
// v is not indexed by the rows)
template <typename T>
__global__ void k_gram_finish(int64_t n, int jsplit, const T* __restrict__ part, const T* __restrict__ noise,
                              const T* __restrict__ v, T* __restrict__ y) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    T s = T(0);
    for (int sp = 0; sp < jsplit; ++sp) s += part[(int64_t)sp * n + i];
    y[i] = noise ? fma(noise[0], v[i], s) : s;
  }
}

// grad[0..d) += -2/ls_k * S_k * softplus'(raw_ls_k); grad[d] += S_sigma/sigma * softplus'(raw_os);
// grad[d+1] += lam . q
template <typename T>
__global__ void k_gram_grad_finish(int d, int nblocks, const double* __restrict__ gpart, const T* __restrict__ raw_ls,
                                   const T* __restrict__ raw_os, const T* __restrict__ consts, int64_t n,
                                   const T* __restrict__ lam, const T* __restrict__ q, T* __restrict__ grad) {
  __shared__ double red_smem[32];
  const int k = blockIdx.x;  // 0..d+1
  double s = 0.0;
  if (k <= d) {
    for (int b = threadIdx.x; b < nblocks; b += blockDim.x) s += gpart[(size_t)b * (d + 1) + k];
  } else {
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += static_cast<double>(lam[i]) * static_cast<double>(q[i]);
  }
  s = block_sum(s, red_smem);
  if (threadIdx.x != 0) return;
  if (k < d) {
    const double ls = static_cast<double>(softplus_t(raw_ls[k]));
    grad[k] += static_cast<T>(-2.0 / ls * s * static_cast<double>(softplus_grad_t(raw_ls[k])));
  } else if (k == d) {
    grad[d] += static_cast<T>(s / static_cast<double>(consts[0]) * static_cast<double>(softplus_grad_t(raw_os[0])));
  } else {
    grad[d + 1] += static_cast<T>(s);
  }
}

// y_p[i] = sum_s part[s][p][i] + noise * v_p[i]   (P vectors of one k_gram_tc_multi pass)
struct OutPtrs {
  float* p[gramtc::kBatchMax];
};
__global__ void k_gram_finish_multi(int64_t n, int jsplit, int P, const float* __restrict__ part,
                                    const float* __restrict__ noise, gramtc::VecPtrs v, OutPtrs y) {
  const int p = blockIdx.y;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int sp = 0; sp < jsplit; ++sp) s += part[((int64_t)sp * P + p) * n + i];
    y.p[p][i] = fmaf(noise[0], v.p[p][i], s);
  }
}

// sum_m <lam_m, q_m> (the noise parameter's cotangent), block shares in npart[gridDim.x]: the pairs are count * n elements
// -- one block walking them alone (as the finish kernel did) took 0.77 ms per pass of 16 pairs at n = 36 560
constexpr int kNoiseParts = 128;
template <typename T>
__global__ void k_gram_noise_partial(int64_t n, const T* __restrict__ Lam, int64_t ldl, const T* __restrict__ Q, int64_t ldq,
                                     int count, double* __restrict__ npart) {
  __shared__ double red_smem[32];
  double s = 0.0;
  const int64_t total = (int64_t)count * n;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = e / n, i = e - m * n;
    s += static_cast<double>(Lam[m * ldl + i]) * static_cast<double>(Q[m * ldq + i]);
  }
  s = block_sum(s, red_smem);
  if (threadIdx.x == 0) npart[blockIdx.x] = s;
}

// batched form: the partial sums come from one k_gram_tc_gradbatch pass over `count` (lam_m, q_m) pairs
template <typename T>
__global__ void k_gram_grad_finish_batch(int d, int nblocks, const double* __restrict__ gpart,
                                         const T* __restrict__ raw_ls, const T* __restrict__ raw_os,
                                         const T* __restrict__ consts, const double* __restrict__ npart, int nparts,
                                         T* __restrict__ grad) {
  __shared__ double red_smem[32];
  const int k = blockIdx.x;  // 0..d+1
  double s = 0.0;
  if (k <= d) {
    for (int b = threadIdx.x; b < nblocks; b += blockDim.x) s += gpart[(size_t)b * (d + 1) + k];
  } else {
    for (int b = threadIdx.x; b < nparts; b += blockDim.x) s += npart[b];
  }
  s = block_sum(s, red_smem);
  if (threadIdx.x != 0) return;
  if (k < d) {
    const double ls = static_cast<double>(softplus_t(raw_ls[k]));
    grad[k] += static_cast<T>(-2.0 / ls * s * static_cast<double>(softplus_grad_t(raw_ls[k])));
  } else if (k == d) {
    grad[d] += static_cast<T>(s / static_cast<double>(consts[0]) * static_cast<double>(softplus_grad_t(raw_os[0])));
  } else {
    grad[d + 1] += static_cast<T>(s);
  }
}

}  // namespace

// Test points of a cross-covariance K(X*, X) (bl_gram_cross_t): scaled and, on the tensor-core path, packed
// as the row operand with the kernel parameters bound to the parent operator (never its noise).  `binds`
// records which bind of the parent they were prepared for.
struct GramOperator;
struct GramCross {
  GramOperator* parent = nullptr;
  int64_t m = 0, mpad = 0;
  DevBuf X;  // m x d doubles
  DevBuf xs, xx, consts, opA, part;
  uint64_t binds = 0;
  int split = 1;  // column splits of the sweep
};

struct GramOperator : bl_operator {
  int64_t d = 0;
  int kind = 0;
  DevBuf X;  // n x d doubles
  DevBuf xs, xx, consts, part, gpart, npart, grad;
  const void* raw_ls = nullptr;
  const void* raw_os = nullptr;
  const void* noise = nullptr;
  int bound_dtype = -1;
  uint64_t binds = 0;  // set_params calls so far (cross objects re-prepare when it moves)
  int jsplit = 1;
  // tensor-core path (fp32, d <= 20): packed TF32 operands, see gram_tc.cuh
  int path = 0;  // 0 = automatic, 1 = FP32 ALU kernel, 2 = tcgen05 kernel
  DevBuf opA, opB, xt, dbg;
  int64_t npad = 0;
  int tc_split = 1;

  bool tc_eligible(int dtype) const { return dtype == BL_F32 && d <= 20; }
  bool use_tc(int dtype) const { return tc_eligible(dtype) && path != 1; }
  int tc_rowtiles() const { return (int)((n + gramtc::kM - 1) / gramtc::kM); }
  int tc_gparts() const { return tc_rowtiles() * tc_split; }

  int num_params() const override { return 3; }
  int64_t param_size(int i) const override { return i == 0 ? d : 1; }

  // padded point dimension (multiple of 4) and rows per thread
  int dp() const { return d <= 4 ? 4 : d <= 8 ? 8 : d <= 12 ? 12 : d <= 16 ? 16 : 32; }
  int ri() const { return dp() <= 16 ? 4 : 2; }
  int nblocks_for(int64_t rows) const { return (int)((rows + (int64_t)kTileI * ri() - 1) / ((int64_t)kTileI * ri())); }
  int nblocks_i() const { return nblocks_for(n); }
  // column splits of the ALU sweep: about four row blocks per SM
  int jsplit_for(int64_t rows) const {
    const int nb = nblocks_for(rows);
    return std::max(1, std::min<int>(64, (4 * sm_count() + nb - 1) / nb));
  }

  template <typename T>
  int set_params_t(cudaStream_t s) {
    BL_CHECK(xs.ensure(((size_t)n + kTileJ) * dp() * sizeof(T)));
    BL_CHECK(xx.ensure(((size_t)n + kTileJ) * sizeof(T)));
    BL_CHECK(consts.ensure(4 * sizeof(T)));
    jsplit = jsplit_for(n);
    const bool tc = use_tc(sizeof(T) == 4 ? BL_F32 : BL_F64);
    if (tc) plan_tc();
    BL_CHECK(part.ensure((size_t)std::max(jsplit, tc_split) * n * sizeof(T)));
    BL_CHECK(gpart.ensure((size_t)std::max(jsplit * nblocks_i(), tc_gparts()) * (d + 1) * sizeof(double)));
    BL_CHECK(grad.ensure((size_t)(d + 2) * sizeof(T)));
    k_gram_prepare<T><<<std::min<int>(1024, (int)((n + 255) / 256)), 256, 0, s>>>(
        n, (int)d, dp(), kind, X.as<double>(), static_cast<const T*>(raw_ls), static_cast<const T*>(raw_os),
        xs.as<T>(), xx.as<T>(), consts.as<T>());
    BL_LAUNCHED();
    if (tc) BL_CHECK(pack_tc(s));
    return BL_OK;
  }

  // ---- tensor-core path ------------------------------------------------------------------
  // column splits of a sweep over `rowtiles` row tiles: balance waves of one-CTA-per-SM blocks against the
  // per-CTA prologue (~1 tile)
  int tc_split_for(int rowtiles) const {
    const int tiles = (int)(npad / gramtc::kN), sms = sm_count();
    double best = 1e300;
    int split = 1;
    for (int sp = 1; sp <= std::min(tiles, 64); ++sp) {
      const int per = (tiles + sp - 1) / sp;
      const int waves = (rowtiles * sp + sms - 1) / sms;
      const double cost = (double)waves * (per + 1.0);
      if (cost < best - 1e-9) best = cost, split = sp;
    }
    return split;
  }
  void plan_tc() {
    npad = (n + gramtc::kN - 1) / gramtc::kN * gramtc::kN;
    tc_split = tc_split_for(tc_rowtiles());
  }
  int pack_tc(cudaStream_t s) {
    const int slots = gramtc::slots_for((int)d);
    BL_CHECK(opA.ensure((size_t)npad * slots * sizeof(float)));
    BL_CHECK(opB.ensure((size_t)npad * slots * sizeof(float)));
    BL_CHECK(xt.ensure((size_t)npad * gramtc::kXtRows * sizeof(float)));
    gramtc::k_gram_tc_pack<<<std::min<int>(1024, (int)((npad + 127) / 128)), 128, 0, s>>>(
        n, npad, (int)d, dp(), slots, xs.as<float>(), xx.as<float>(), opA.as<float>(), opB.as<float>(), xt.as<float>());
    BL_LAUNCHED();
    return BL_OK;
  }
  // CROSS: rows are the test points of `c`
  template <int KIND, bool ADJ, int D, bool CROSS = false>
  int launch_tc(const float* v, const float* q, float* dbg_out, int dbg_bx, int dbg_by, cudaStream_t s,
                const GramCross* c = nullptr) {
    const int slots = gramtc::slots_for((int)d);
    const gramtc::Plan pl = gramtc::make_plan(slots, ADJ);
    auto kernel = gramtc::k_gram_tc_sweep<KIND, ADJ, D, CROSS>;
    {
      static std::mutex mu;
      static std::map<int, bool> done;
      int dev = 0;
      BL_CUDA(cudaGetDevice(&dev));
      std::lock_guard<std::mutex> lk(mu);
      if (!done[dev]) {  // the request depends on d: opt in to the architectural maximum once
        cudaFuncAttributes fa;
        BL_CUDA(cudaFuncGetAttributes(&fa, kernel));
        BL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     227 * 1024 - (int)fa.sharedSizeBytes));
        done[dev] = true;
      }
    }
    if (CROSS)
      kernel<<<dim3((unsigned)(c->mpad / gramtc::kM), c->split), gramtc::kThreads, pl.total, s>>>(
          n, npad, (int)d, slots, c->opA.as<float>(), opB.as<float>(), nullptr, c->xx.as<float>(), consts.as<float>(), v,
          nullptr, c->part.as<float>(), nullptr, nullptr, 0, 0, c->m, c->mpad);
    else
      kernel<<<dim3(tc_rowtiles(), tc_split), gramtc::kThreads, pl.total, s>>>(
          n, npad, (int)d, slots, opA.as<float>(), opB.as<float>(), xt.as<float>(), xx.as<float>(), consts.as<float>(), v,
          q, part.as<float>(), gpart.as<double>(), dbg_out, dbg_bx, dbg_by, n, npad);
    BL_LAUNCHED();
    return BL_OK;
  }
  template <int KIND, bool ADJ>
  int launch_tc_d(const float* v, const float* q, float* dbg_out, int bx, int by, cudaStream_t s) {
    if (!ADJ) return launch_tc<KIND, false, 1>(v, q, dbg_out, bx, by, s);
    if (d <= 3) return launch_tc<KIND, ADJ, ADJ ? 3 : 1>(v, q, dbg_out, bx, by, s);
    if (d <= 4) return launch_tc<KIND, ADJ, ADJ ? 4 : 1>(v, q, dbg_out, bx, by, s);
    if (d <= 6) return launch_tc<KIND, ADJ, ADJ ? 6 : 1>(v, q, dbg_out, bx, by, s);
    if (d <= 8) return launch_tc<KIND, ADJ, ADJ ? 8 : 1>(v, q, dbg_out, bx, by, s);
    if (d <= 9) return launch_tc<KIND, ADJ, ADJ ? 9 : 1>(v, q, dbg_out, bx, by, s);
    if (d <= 12) return launch_tc<KIND, ADJ, ADJ ? 12 : 1>(v, q, dbg_out, bx, by, s);
    if (d <= 16) return launch_tc<KIND, ADJ, ADJ ? 16 : 1>(v, q, dbg_out, bx, by, s);
    return launch_tc<KIND, ADJ, ADJ ? 20 : 1>(v, q, dbg_out, bx, by, s);
  }
  template <bool ADJ>
  int sweep_tc(const float* v, const float* q, float* y, float* dbg_out, int bx, int by, cudaStream_t s) {
    if (kind == 0)
      BL_CHECK((launch_tc_d<0, ADJ>(v, q, dbg_out, bx, by, s)));
    else if (kind == 1)
      BL_CHECK((launch_tc_d<1, ADJ>(v, q, dbg_out, bx, by, s)));
    else
      BL_CHECK((launch_tc_d<2, ADJ>(v, q, dbg_out, bx, by, s)));
    if (y) BL_CHECK(finish<float>(n, tc_split, part.as<float>(), static_cast<const float*>(noise), v, y, s));
    return BL_OK;
  }
  // ---- deferred parameter cotangent (operators.cuh) ------------------------------------------
  bool deferred_grad(int dtype) const override {
    const char* env = std::getenv("BL_GRAM_DEFER");  // "0": per-step cotangent sweeps (A/B comparisons)
    return use_tc(dtype) && !(env && env[0] == '0');
  }
  int apply_transpose(int dtype, const void* lam, void* z, cudaStream_t s) override {
    return matvec(dtype, lam, z, s);  // the Gram matrix is symmetric
  }
  template <int KIND>
  int launch_multi(const gramtc::VecPtrs& vp, int P, cudaStream_t s) {
    const int slots = gramtc::slots_for((int)d);
    const gramtc::Plan pl = gramtc::make_plan_multi(slots);
    auto kernel = gramtc::k_gram_tc_multi<KIND>;
    {
      static std::mutex mu;
      static std::map<int, bool> done;
      int dev = 0;
      BL_CUDA(cudaGetDevice(&dev));
      std::lock_guard<std::mutex> lk(mu);
      if (!done[dev]) {
        cudaFuncAttributes fa;
        BL_CUDA(cudaFuncGetAttributes(&fa, kernel));
        BL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     227 * 1024 - (int)fa.sharedSizeBytes));
        done[dev] = true;
      }
    }
    kernel<<<dim3(tc_rowtiles(), tc_split), gramtc::kThreads, pl.total, s>>>(
        n, npad, slots, opA.as<float>(), opB.as<float>(), xx.as<float>(), consts.as<float>(), vp, P, part.as<float>());
    BL_LAUNCHED();
    return BL_OK;
  }
  int matvec_batch(int dtype, int count, const void* const* in, void* const* out, cudaStream_t s) override {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    if (!use_tc(dtype) || count == 1) return bl_operator::matvec_batch(dtype, count, in, out, s);
    BL_CHECK(part.ensure((size_t)tc_split * gramtc::kBatchMax * n * sizeof(float)));
    for (int p0 = 0; p0 < count; p0 += gramtc::kBatchMax) {
      const int P = std::min(gramtc::kBatchMax, count - p0);
      gramtc::VecPtrs vp{};
      OutPtrs op_{};
      for (int p = 0; p < P; ++p) vp.p[p] = static_cast<const float*>(in[p0 + p]), op_.p[p] = static_cast<float*>(out[p0 + p]);
      if (kind == 0)
        BL_CHECK(launch_multi<0>(vp, P, s));
      else if (kind == 1)
        BL_CHECK(launch_multi<1>(vp, P, s));
      else
        BL_CHECK(launch_multi<2>(vp, P, s));
      k_gram_finish_multi<<<dim3(std::min<int>(256, (int)((n + 255) / 256)), P), 256, 0, s>>>(
          n, tc_split, P, part.as<float>(), static_cast<const float*>(noise), vp, op_);
      BL_LAUNCHED();
    }
    return BL_OK;
  }
  int apply_transpose_batch(int dtype, int count, const void* const* in, void* const* out, cudaStream_t s) override {
    return matvec_batch(dtype, count, in, out, s);  // symmetric
  }

  template <int KIND, int D>
  int launch_batch(const float* Q, int64_t ldq, const float* Lam, int64_t ldl, int M, cudaStream_t s) {
    const int slots = gramtc::slots_for((int)d);
    const gramtc::Plan pl = gramtc::make_plan_batch(slots);
    auto kernel = gramtc::k_gram_tc_gradbatch<KIND, D>;
    {
      static std::mutex mu;
      static std::map<int, bool> done;
      int dev = 0;
      BL_CUDA(cudaGetDevice(&dev));
      std::lock_guard<std::mutex> lk(mu);
      if (!done[dev]) {
        cudaFuncAttributes fa;
        BL_CUDA(cudaFuncGetAttributes(&fa, kernel));
        BL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     227 * 1024 - (int)fa.sharedSizeBytes));
        done[dev] = true;
      }
    }
    kernel<<<dim3(tc_rowtiles(), tc_split), gramtc::kThreads, pl.total, s>>>(
        n, npad, (int)d, slots, opA.as<float>(), opB.as<float>(), xt.as<float>(), xx.as<float>(), consts.as<float>(), Q,
        ldq, Lam, ldl, M, gpart.as<double>());
    BL_LAUNCHED();
    return BL_OK;
  }
  template <int KIND>
  int launch_batch_d(const float* Q, int64_t ldq, const float* Lam, int64_t ldl, int M, cudaStream_t s) {
    if (d <= 3) return launch_batch<KIND, 3>(Q, ldq, Lam, ldl, M, s);
    if (d <= 4) return launch_batch<KIND, 4>(Q, ldq, Lam, ldl, M, s);
    if (d <= 6) return launch_batch<KIND, 6>(Q, ldq, Lam, ldl, M, s);
    if (d <= 8) return launch_batch<KIND, 8>(Q, ldq, Lam, ldl, M, s);
    if (d <= 9) return launch_batch<KIND, 9>(Q, ldq, Lam, ldl, M, s);
    if (d <= 12) return launch_batch<KIND, 12>(Q, ldq, Lam, ldl, M, s);
    if (d <= 16) return launch_batch<KIND, 16>(Q, ldq, Lam, ldl, M, s);
    return launch_batch<KIND, 20>(Q, ldq, Lam, ldl, M, s);
  }
  int vjp_batch(int dtype, const void* Q, int64_t ldq, const void* Lam, int64_t ldl, int count,
                cudaStream_t s) override {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    if (!use_tc(dtype)) return bl_operator::vjp_batch(dtype, Q, ldq, Lam, ldl, count, s);
    BL_REQUIRE((ldq * 4) % 16 == 0 && (ldl * 4) % 16 == 0 && ldq >= n && ldl >= n, "row strides must be 16-byte multiples");
    for (int m0 = 0; m0 < count; m0 += gramtc::kBatchMax) {
      const int M = std::min(gramtc::kBatchMax, count - m0);
      const float* q = static_cast<const float*>(Q) + (int64_t)m0 * ldq;
      const float* l = static_cast<const float*>(Lam) + (int64_t)m0 * ldl;
      if (kind == 0)
        BL_CHECK((launch_batch_d<0>(q, ldq, l, ldl, M, s)));
      else if (kind == 1)
        BL_CHECK((launch_batch_d<1>(q, ldq, l, ldl, M, s)));
      else
        BL_CHECK((launch_batch_d<2>(q, ldq, l, ldl, M, s)));
      BL_CHECK(npart.ensure(kNoiseParts * sizeof(double)));
      k_gram_noise_partial<float><<<kNoiseParts, 256, 0, s>>>(n, l, ldl, q, ldq, M, npart.as<double>());
      BL_LAUNCHED();
      k_gram_grad_finish_batch<float><<<(int)d + 2, 256, 0, s>>>(
          (int)d, tc_gparts(), gpart.as<double>(), static_cast<const float*>(raw_ls), static_cast<const float*>(raw_os),
          consts.as<float>(), npart.as<double>(), kNoiseParts, grad.as<float>());
      BL_LAUNCHED();
    }
    return BL_OK;
  }

  // diagnostic: the tensor-core accumulator (x_i.x_j - |x_j|^2/2) of the tile (rows 128 bi .., columns 256 bj ..)
  int tile_distances(int64_t bi, int64_t bj, float* out_host, cudaStream_t s) {
    BL_REQUIRE(bound_dtype == BL_F32 && use_tc(BL_F32), "tile distances need the fp32 tensor-core path (bind first)");
    const int64_t per = (npad / gramtc::kN + tc_split - 1) / tc_split;
    BL_REQUIRE(bi >= 0 && bi < tc_rowtiles() && bj >= 0 && bj < npad / gramtc::kN && bj % per == 0,
               "tile index out of range (column tile must be the first tile of a split)");
    BL_CHECK(dbg.ensure((size_t)gramtc::kM * gramtc::kN * sizeof(float)));
    BL_CUDA(cudaMemsetAsync(dbg.p, 0, dbg.bytes, s));
    // any vector works as v: only the accumulator is reported
    BL_CHECK((sweep_tc<false>(xx.as<float>(), nullptr, nullptr, dbg.as<float>(), (int)bi, (int)(bj / per), s)));
    BL_CUDA(cudaMemcpyAsync(out_host, dbg.p, dbg.bytes, cudaMemcpyDeviceToHost, s));
    BL_CUDA(cudaStreamSynchronize(s));
    return BL_OK;
  }

  int set_params(int dtype, const void* const* params, int num, cudaStream_t s) override {
    BL_REQUIRE(num == 3 && params && params[0] && params[1] && params[2],
               "gram operator takes (raw_lengthscale, raw_outputscale, noise)");
    raw_ls = params[0];
    raw_os = params[1];
    noise = params[2];
    bound_dtype = dtype;
    ++binds;
    return dtype == BL_F32 ? set_params_t<float>(s) : set_params_t<double>(s);
  }

  // CROSS: rows are the test points of `c`
  template <typename T, int DP, int RI, bool ADJ, bool CROSS = false>
  void launch_sweep(const T* v, const T* q, cudaStream_t s, const GramCross* c = nullptr) {
    dim3 grid(CROSS ? nblocks_for(c->m) : nblocks_i(), CROSS ? c->split : jsplit);
#define BL_GRAM_LAUNCH(KIND)                                                                                        \
  k_gram_sweep<T, DP, RI, ADJ, KIND, CROSS><<<grid, kTileI, 0, s>>>(                                                \
      n, (int)d, xs.as<T>(), xx.as<T>(), consts.as<T>(), v, q, (CROSS ? c->part : part).template as<T>(),            \
      gpart.as<double>(), CROSS ? c->m : n, (CROSS ? c->xs : xs).template as<T>(), (CROSS ? c->xx : xx).template as<T>())
    if (kind == 0)
      BL_GRAM_LAUNCH(0);
    else if (kind == 1)
      BL_GRAM_LAUNCH(1);
    else
      BL_GRAM_LAUNCH(2);
#undef BL_GRAM_LAUNCH
  }

  template <typename T, bool ADJ, bool CROSS = false>
  int sweep(const T* v, const T* q, T* y, cudaStream_t s, const GramCross* c = nullptr) {
    switch (dp()) {
      case 4: launch_sweep<T, 4, 4, ADJ, CROSS>(v, q, s, c); break;
      case 8: launch_sweep<T, 8, 4, ADJ, CROSS>(v, q, s, c); break;
      case 12: launch_sweep<T, 12, 4, ADJ, CROSS>(v, q, s, c); break;
      case 16: launch_sweep<T, 16, 4, ADJ, CROSS>(v, q, s, c); break;
      default: launch_sweep<T, 32, 2, ADJ, CROSS>(v, q, s, c); break;
    }
    BL_LAUNCHED();
    if (y) BL_CHECK(finish<T>(CROSS ? c->m : n, CROSS ? c->split : jsplit, (CROSS ? c->part : part).template as<T>(),
                              CROSS ? nullptr : static_cast<const T*>(noise), v, y, s));
    return BL_OK;
  }
  // y = sum of the column splits' partial products (+ noise v for the square operator: noise != nullptr)
  template <typename T>
  int finish(int64_t rows, int split, const T* partp, const T* noisep, const T* v, T* y, cudaStream_t s) {
    k_gram_finish<T><<<std::min<int>(1024, (int)((rows + 255) / 256)), 256, 0, s>>>(rows, split, partp, noisep, v, y);
    BL_LAUNCHED();
    return BL_OK;
  }

  int matvec(int dtype, const void* x, void* y, cudaStream_t s) override {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    if (use_tc(dtype)) return sweep_tc<false>((const float*)x, nullptr, (float*)y, nullptr, 0, 0, s);
    return dtype == BL_F32 ? sweep<float, false>((const float*)x, nullptr, (float*)y, s)
                           : sweep<double, false>((const double*)x, nullptr, (double*)y, s);
  }

  template <typename T>
  int vjp_t(const T* q, const T* lam, T* z, cudaStream_t s) {
    const bool tc = use_tc(sizeof(T) == 4 ? BL_F32 : BL_F64);
    if (tc)
      BL_CHECK((sweep_tc<true>((const float*)lam, (const float*)q, (float*)z, nullptr, 0, 0, s)));
    else
      BL_CHECK((sweep<T, true>(lam, q, z, s)));
    k_gram_grad_finish<T><<<(int)d + 2, 256, 0, s>>>((int)d, tc ? tc_gparts() : jsplit * nblocks_i(), gpart.as<double>(),
                                                      static_cast<const T*>(raw_ls), static_cast<const T*>(raw_os),
                                                      consts.as<T>(), n, lam, q, grad.as<T>());
    BL_LAUNCHED();
    return BL_OK;
  }

  int vjp(int dtype, const void* q, const void* lam, void* z, cudaStream_t s) override {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    return dtype == BL_F32 ? vjp_t<float>((const float*)q, (const float*)lam, (float*)z, s)
                           : vjp_t<double>((const double*)q, (const double*)lam, (double*)z, s);
  }

  // out[b][j] = k(x_j, z_c) for the `rows` points x, b < count (k_gram_elements)
  template <typename T>
  int elements_t(int64_t rows, const DevBuf& xsb, const DevBuf& xxb, const T* zs, const T* zz, int64_t zstep,
                 const int64_t* index, int64_t count, int64_t ldo, T* out, cudaStream_t s) {
    k_gram_elements<T><<<dim3((unsigned)((rows + 255) / 256), (unsigned)count), 256, 0, s>>>(
        rows, dp(), kind, xsb.as<T>(), xxb.as<T>(), zs, zz, zstep, consts.as<T>(), index, ldo, out);
    BL_LAUNCHED();
    return BL_OK;
  }
  int elements(int dtype, const int64_t* index, void* out, cudaStream_t s) {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    const int64_t zstep = index ? 0 : 1;
    if (dtype == BL_F32)
      return elements_t<float>(n, xs, xx, xs.as<float>(), xx.as<float>(), zstep, index, 1, n, static_cast<float*>(out), s);
    return elements_t<double>(n, xs, xx, xs.as<double>(), xx.as<double>(), zstep, index, 1, n, static_cast<double*>(out), s);
  }
  int element_diagonal(int dtype, void* out, cudaStream_t s) override { return elements(dtype, nullptr, out, s); }
  int element_column(int dtype, const int64_t* index, void* out, cudaStream_t s) override {
    return elements(dtype, index, out, s);
  }

  // ---- cross-covariance with the test points of a GramCross ------------------------------------
  template <typename T>
  int cross_prepare_t(GramCross& c, cudaStream_t s) {
    const int64_t m = c.m;
    BL_CHECK(c.xs.ensure((size_t)m * dp() * sizeof(T)));
    BL_CHECK(c.xx.ensure((size_t)m * sizeof(T)));
    BL_CHECK(c.consts.ensure(4 * sizeof(T)));  // k_gram_prepare's copy of the outputscale (the sweeps read the parent's)
    k_gram_prepare<T><<<std::min<int>(1024, (int)((m + 255) / 256)), 256, 0, s>>>(
        m, (int)d, dp(), kind, c.X.as<double>(), static_cast<const T*>(raw_ls), static_cast<const T*>(raw_os),
        c.xs.as<T>(), c.xx.as<T>(), c.consts.as<T>());
    BL_LAUNCHED();
    if (use_tc(sizeof(T) == 4 ? BL_F32 : BL_F64)) {
      const int slots = gramtc::slots_for((int)d);
      c.mpad = (m + gramtc::kM - 1) / gramtc::kM * gramtc::kM;
      c.split = tc_split_for((int)(c.mpad / gramtc::kM));
      BL_CHECK(c.opA.ensure((size_t)c.mpad * slots * sizeof(float)));
      gramtc::k_gram_tc_pack<<<std::min<int>(1024, (int)((c.mpad + 127) / 128)), 128, 0, s>>>(
          m, c.mpad, (int)d, dp(), slots, c.xs.as<float>(), c.xx.as<float>(), c.opA.as<float>(), nullptr, nullptr);
      BL_LAUNCHED();
    } else {
      c.split = jsplit_for(m);
    }
    BL_CHECK(c.part.ensure((size_t)c.split * m * sizeof(T)));
    c.binds = binds;
    return BL_OK;
  }
  int cross_prepare(GramCross& c, int dtype, cudaStream_t s) {
    BL_REQUIRE(dtype == bound_dtype, "bind the parent gram operator with the same dtype first");
    if (c.binds == binds) return BL_OK;
    return dtype == BL_F32 ? cross_prepare_t<float>(c, s) : cross_prepare_t<double>(c, s);
  }
  // y (m) = K(X*, X) v (n): no noise term
  int cross_matvec(GramCross& c, int dtype, const void* v, void* y, cudaStream_t s) {
    BL_CHECK(cross_prepare(c, dtype, s));
    if (use_tc(dtype)) {
      const float* vf = static_cast<const float*>(v);
      if (kind == 0)
        BL_CHECK((launch_tc<0, false, 1, true>(vf, nullptr, nullptr, 0, 0, s, &c)));
      else if (kind == 1)
        BL_CHECK((launch_tc<1, false, 1, true>(vf, nullptr, nullptr, 0, 0, s, &c)));
      else
        BL_CHECK((launch_tc<2, false, 1, true>(vf, nullptr, nullptr, 0, 0, s, &c)));
      return finish<float>(c.m, c.split, c.part.as<float>(), nullptr, vf, static_cast<float*>(y), s);
    }
    return dtype == BL_F32 ? sweep<float, false, true>((const float*)v, nullptr, (float*)y, s, &c)
                           : sweep<double, false, true>((const double*)v, nullptr, (double*)y, s, &c);
  }
  // out[b][j] = k(x*_{first+b}, x_j), b < count, row stride ldo
  int cross_columns(GramCross& c, int dtype, int64_t first, int64_t count, void* out, int64_t ldo, cudaStream_t s) {
    BL_CHECK(cross_prepare(c, dtype, s));
    if (dtype == BL_F32)
      return elements_t<float>(n, xs, xx, c.xs.as<float>() + first * dp(), c.xx.as<float>() + first, 0, nullptr, count,
                               ldo, static_cast<float*>(out), s);
    return elements_t<double>(n, xs, xx, c.xs.as<double>() + first * dp(), c.xx.as<double>() + first, 0, nullptr, count,
                              ldo, static_cast<double*>(out), s);
  }
  // out[t] = k(x*_t, x*_t): the kernel formula at s2 = 0
  int cross_prior_diag(GramCross& c, int dtype, void* out, cudaStream_t s) {
    BL_CHECK(cross_prepare(c, dtype, s));
    if (dtype == BL_F32)
      return elements_t<float>(c.m, c.xs, c.xx, c.xs.as<float>(), c.xx.as<float>(), 1, nullptr, 1, c.m,
                               static_cast<float*>(out), s);
    return elements_t<double>(c.m, c.xs, c.xx, c.xs.as<double>(), c.xx.as<double>(), 1, nullptr, 1, c.m,
                              static_cast<double*>(out), s);
  }

  int grad_zero(int dtype, cudaStream_t s) override {
    BL_CHECK(grad.ensure((size_t)(d + 2) * dtype_size(dtype)));
    BL_CUDA(cudaMemsetAsync(grad.p, 0, (size_t)(d + 2) * dtype_size(dtype), s));
    return BL_OK;
  }

  int grad_export(int dtype, void* const* grads, int num, cudaStream_t s) override {
    BL_REQUIRE(num == 3 && grads && grads[0] && grads[1] && grads[2], "gram operator has three gradient buffers");
    const size_t w = dtype_size(dtype);
    const char* g = static_cast<const char*>(grad.p);
    BL_CUDA(cudaMemcpyAsync(grads[0], g, d * w, cudaMemcpyDeviceToDevice, s));
    BL_CUDA(cudaMemcpyAsync(grads[1], g + d * w, w, cudaMemcpyDeviceToDevice, s));
    BL_CUDA(cudaMemcpyAsync(grads[2], g + (d + 1) * w, w, cudaMemcpyDeviceToDevice, s));
    return BL_OK;
  }
};

}  // namespace bl

struct bl_gram_cross {
  bl::GramCross cross;
};

extern "C" int bl_op_gram_set_path(bl_operator_t* op, int path) {
  auto* o = dynamic_cast<bl::GramOperator*>(op);
  BL_REQUIRE(o != nullptr && path >= 0 && path <= 2, "bad gram path (0 automatic, 1 ALU, 2 tensor cores)");
  BL_REQUIRE(path != 2 || o->d <= 20, "the tensor-core path supports d <= 20");
  o->path = path;
  o->bound_dtype = -1;  // operands are packed at bind time
  return BL_OK;
}

extern "C" int bl_op_gram_tile_distances(bl_operator_t* op, int64_t row_tile, int64_t col_tile, float* out_host,
                                         void* stream) {
  auto* o = dynamic_cast<bl::GramOperator*>(op);
  BL_REQUIRE(o != nullptr && out_host != nullptr, "bad arguments");
  return o->tile_distances(row_tile, col_tile, out_host, bl::as_stream(stream));
}

extern "C" int bl_op_gram_create(int64_t n, int64_t d, int kind, const double* X_host, bl_operator_t** op) {
  BL_REQUIRE(op && X_host && n > 0 && d > 0 && d <= bl::kMaxDim && kind >= 0 && kind <= 2,
             "bad gram operator arguments (d <= 32, kind in {0,1,2})");
  auto* o = new bl::GramOperator();
  o->n = n;
  o->d = d;
  o->kind = kind;
  int rc = o->X.ensure((size_t)n * d * sizeof(double));
  if (rc == BL_OK && cudaMemcpy(o->X.p, X_host, (size_t)n * d * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) {
    bl::set_error("cudaMemcpy of X failed");
    rc = BL_ECUDA;
  }
  if (rc != BL_OK) {
    delete o;
    return rc;
  }
  *op = o;
  return BL_OK;
}

extern "C" int bl_gram_cross_create(bl_operator_t* gram, int64_t m, const double* Xtest_host, bl_gram_cross_t** out) {
  auto* g = dynamic_cast<bl::GramOperator*>(gram);
  BL_REQUIRE(g != nullptr && out && Xtest_host && m > 0, "bad gram cross arguments (a gram operator and m >= 1 test points)");
  auto* c = new bl_gram_cross();
  c->cross.parent = g;
  c->cross.m = m;
  int rc = c->cross.X.ensure((size_t)m * g->d * sizeof(double));
  if (rc == BL_OK &&
      cudaMemcpy(c->cross.X.p, Xtest_host, (size_t)m * g->d * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) {
    bl::set_error("cudaMemcpy of the test points failed");
    rc = BL_ECUDA;
  }
  if (rc != BL_OK) {
    delete c;
    return rc;
  }
  *out = c;
  return BL_OK;
}

extern "C" int bl_gram_cross_destroy(bl_gram_cross_t* c) {
  delete c;
  return BL_OK;
}

extern "C" int bl_gram_cross_matvec(bl_gram_cross_t* c, int dtype, const void* v, void* y, void* stream) {
  BL_REQUIRE(c && v && y, "bad gram cross matvec arguments");
  return c->cross.parent->cross_matvec(c->cross, dtype, v, y, bl::as_stream(stream));
}

extern "C" int bl_gram_cross_columns(bl_gram_cross_t* c, int dtype, int64_t first, int64_t count, void* out, int64_t ld,
                                     void* stream) {
  BL_REQUIRE(c && out && first >= 0 && count >= 1 && first + count <= c->cross.m && count <= 65535 &&
                 ld >= c->cross.parent->n,
             "bad gram cross columns arguments (0 <= first, first + count <= m, count <= 65535, ld >= n)");
  return c->cross.parent->cross_columns(c->cross, dtype, first, count, out, ld, bl::as_stream(stream));
}

extern "C" int bl_gram_cross_prior_diag(bl_gram_cross_t* c, int dtype, void* out, void* stream) {
  BL_REQUIRE(c && out, "bad gram cross prior diagonal arguments");
  return c->cross.parent->cross_prior_diag(c->cross, dtype, out, bl::as_stream(stream));
}
