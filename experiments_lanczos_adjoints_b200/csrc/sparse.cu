// Sparse COO/BCOO operand -> SELL-32 SpMV, transposed SpMV and parameter cotangent.
//
// Reference behaviour replaced: `BCOO((params, M.indices), shape) @ x` and its `jax.vjp`
// (/root/reference/experiments/benchmarks/wall_times_vjp_through_lanczos_arnoldi/suite_sparse/benchmark.py:61-68,
//  /root/reference/src/matfree_extensions/util/exp_util.py:35-42).
//
// Layout in HBM (per operator, built once on the host):
//   SELL-32 ("sliced ELLPACK", slice height 32 = one warp, no row sorting) of A and of A^T:
//     slice_ptr[s]            int64   first slot of slice s
//     col[slot]               int32   column (A) / row (A^T) index; padding repeats a valid index
//     src[slot]               int32   COO position whose parameter lives in this slot, -1 = padding
//     val[slot]               T       gathered from the parameter vector by set_params
//   slot(row r, k-th entry) = slice_ptr[r/32] + k*32 + r%32  -> a warp reads 128 contiguous
//   bytes of `val` and of `col` per k: fully coalesced.
//   grad[slot] (T) accumulates lam[r]*q[col] in the same layout; grad_export scatters to COO order.
#include <algorithm>
#include <cstdlib>
#include <memory>
#include <mutex>
#include <numeric>
#include <set>
#include <vector>

#include "operators.cuh"
#include "tma_pipeline.cuh"

namespace bl {

namespace {

constexpr int kSlice = 32;

struct SellHost {
  std::vector<int64_t> slice_ptr;    // nslices + 1
  std::vector<int32_t> col;          // nslots
  std::vector<int32_t> src;          // nslots
  std::vector<int64_t> slot_of_csr;  // nnz
  int64_t nslots = 0;
};

struct CsrHost {
  std::vector<int32_t> row_ptr, col_idx, perm;
};

// Stable sort of COO entries by (row, col): counting sort on the row, stable sort on the
// column inside each row.  Same result as np.lexsort((col, row)) (oracle/operators.py).
CsrHost coo_to_csr(int64_t nrows, int64_t nnz, const int32_t* row, const int32_t* col) {
  CsrHost c;
  c.row_ptr.assign(nrows + 1, 0);
  for (int64_t e = 0; e < nnz; ++e) c.row_ptr[row[e] + 1]++;
  for (int64_t r = 0; r < nrows; ++r) c.row_ptr[r + 1] += c.row_ptr[r];
  c.perm.resize(nnz);
  std::vector<int32_t> fill(c.row_ptr.begin(), c.row_ptr.end() - 1);
  for (int64_t e = 0; e < nnz; ++e) c.perm[fill[row[e]]++] = (int32_t)e;
  for (int64_t r = 0; r < nrows; ++r)
    std::stable_sort(c.perm.begin() + c.row_ptr[r], c.perm.begin() + c.row_ptr[r + 1],
                     [&](int32_t a, int32_t b) { return col[a] < col[b]; });
  c.col_idx.resize(nnz);
  for (int64_t k = 0; k < nnz; ++k) c.col_idx[k] = col[c.perm[k]];
  return c;
}

SellHost csr_to_sell(int64_t nrows, const CsrHost& c) {
  SellHost s;
  const int64_t nslices = (nrows + kSlice - 1) / kSlice;
  s.slice_ptr.assign(nslices + 1, 0);
  for (int64_t sl = 0; sl < nslices; ++sl) {
    int64_t w = 0;
    for (int64_t r = sl * kSlice; r < std::min<int64_t>(nrows, (sl + 1) * kSlice); ++r)
      w = std::max<int64_t>(w, c.row_ptr[r + 1] - c.row_ptr[r]);
    s.slice_ptr[sl + 1] = s.slice_ptr[sl] + w * kSlice;
  }
  s.nslots = s.slice_ptr[nslices];
  s.col.assign(s.nslots, 0);
  s.src.assign(s.nslots, -1);
  s.slot_of_csr.resize(c.col_idx.size());
  for (int64_t r = 0; r < nrows; ++r) {
    const int64_t sl = r / kSlice, lane = r % kSlice;
    const int64_t w = (s.slice_ptr[sl + 1] - s.slice_ptr[sl]) / kSlice;
    const int64_t len = c.row_ptr[r + 1] - c.row_ptr[r];
    int32_t padcol = len > 0 ? c.col_idx[c.row_ptr[r]] : 0;
    for (int64_t k = 0; k < w; ++k) {
      const int64_t slot = s.slice_ptr[sl] + k * kSlice + lane;
      if (k < len) {
        s.col[slot] = c.col_idx[c.row_ptr[r] + k];
        s.src[slot] = c.perm[c.row_ptr[r] + k];
        s.slot_of_csr[c.row_ptr[r] + k] = slot;
      } else {
        s.col[slot] = padcol;
      }
    }
  }
  return s;
}

// ---- kernels ----
template <typename T>
__global__ void k_gather_values(int64_t nslots, const int32_t* __restrict__ src,
                                const T* __restrict__ params, T* __restrict__ val) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nslots;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t s = src[i];
    val[i] = s >= 0 ? params[s] : T(0);
  }
}

template <typename T>
__global__ void k_scatter_grad(int64_t nslots, const int32_t* __restrict__ src,
                               const T* __restrict__ grad, T* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nslots;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t s = src[i];
    if (s >= 0) out[s] = grad[i];
  }
}

__device__ __forceinline__ int ld_stream_i32(const int32_t* p) {
  int v;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream_t(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ double ld_stream_t(const double* p) {
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}

// Up to kSpmvBatch vectors per launch (lockstep Krylov runs over probes / initial conditions): the slice's values
// and column indices -- 8 of the ~9 bytes per non-zero a single-vector SpMV moves -- are read ONCE for all of them;
// the gathers of the P vectors are independent loads in flight together.  A single vector is a batch of one.
// NORM: the forward Krylov step's normalisation fused into the matvec, one length per run: q = v / len (true division
// as in arnoldi.py:80, written once per row, zero padded up to n_pad) and y = A q, one pass over the vector less.  The
// gathered entries are scaled with the reciprocal (a division per non-zero makes the kernel ALU-bound): they can
// differ from the stored q by one ulp, the size of the matvec's own rounding.
constexpr int kSpmvBatch = 4;
struct MultiVec {
  const void* x[kSpmvBatch];
  void* y[kSpmvBatch];
  const double* len[kSpmvBatch];
  void* q[kSpmvBatch];
};

// W slots of the row are in flight per lane: their column indices and values are loaded first, then all W x P
// gathers are issued before the first FMA.  (A loop over two slots per iteration leaves a lane with two
// dependent memory round trips per pair of entries: ~6 round trips for an 11-entry row, and the kernel runs at half
// of the HBM rate for want of loads in flight.)
template <typename T, int P, bool NORM, int W>
__global__ void __launch_bounds__(256)
k_sell_spmv_multi(int64_t nrows, const int64_t* __restrict__ slice_ptr, const int32_t* __restrict__ col,
                  const T* __restrict__ val, const MultiVec mv, int64_t n_pad) {
  const int lane = threadIdx.x & 31;
  const int64_t slice = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t r = slice * kSlice + lane;
  if (slice * kSlice >= nrows) return;
  const T* x[P];
  T inv[P], acc0[P], acc1[P];
#pragma unroll
  for (int pp = 0; pp < P; ++pp) {
    x[pp] = static_cast<const T*>(mv.x[pp]);
    inv[pp] = T(1);
    acc0[pp] = acc1[pp] = T(0);
    if (NORM) {
      const T d = static_cast<T>(*mv.len[pp]);
      inv[pp] = T(1) / d;
      if (r < n_pad) static_cast<T*>(mv.q[pp])[r] = r < nrows ? x[pp][r] * T(1) / d : T(0);
    }
  }
  const int64_t s0 = slice_ptr[slice], s1 = slice_ptr[slice + 1];
  const int width = (int)((s1 - s0) / kSlice);
  const int32_t* colp = col + s0 + lane;
  const T* valp = val + s0 + lane;
  int c[W], cn[W];
  T v[W], vn[W];
  auto load_chunk = [&](int k0, int (&cc)[W], T (&vv)[W]) {  // indices and values of slots k0 .. k0+W-1 of this row
#pragma unroll
    for (int j = 0; j < W; ++j) {
      const bool ok = k0 + j < width;
      const int off = (ok ? k0 + j : width - 1) * kSlice;  // clamped: a valid column, value 0
      cc[j] = ld_stream_i32(colp + off);
      vv[j] = ok ? ld_stream_t(valp + off) : T(0);
    }
  };
  if (width > 0) load_chunk(0, cn, vn);
  for (int k0 = 0; k0 < width; k0 += W) {
#pragma unroll
    for (int j = 0; j < W; ++j) {
      c[j] = cn[j];
      v[j] = vn[j];
    }
    T g[W][P];
#pragma unroll
    for (int j = 0; j < W; ++j)
#pragma unroll
      for (int pp = 0; pp < P; ++pp) g[j][pp] = __ldg(x[pp] + c[j]);
    // the next chunk's indices and values travel with this chunk's gathers: one dependent round trip per chunk
    if (k0 + W < width) load_chunk(k0 + W, cn, vn);
#pragma unroll
    for (int j = 0; j < W; ++j)
#pragma unroll
      for (int pp = 0; pp < P; ++pp) {
        const T gv = NORM ? g[j][pp] * inv[pp] : g[j][pp];
        if (j & 1)
          acc1[pp] = fma(v[j], gv, acc1[pp]);
        else
          acc0[pp] = fma(v[j], gv, acc0[pp]);
      }
  }
  if (r < nrows) {
#pragma unroll
    for (int pp = 0; pp < P; ++pp) static_cast<T*>(mv.y[pp])[r] = acc0[pp] + acc1[pp];
  }
}

// Adjoint of the sparse matvec in one launch:
//   z[r]       = sum_k valT[slot] * lam[colT[slot]]      (A^T lam, via SELL of A^T; optional)
//   grad[slot] += lam[r] * q[col[slot]]                   (d<lam, A q>/dparams, SELL of A)
template <typename T>
__global__ void __launch_bounds__(256)
k_sell_vjp(int64_t nrows, const int64_t* __restrict__ slice_ptr, const int32_t* __restrict__ col,
           T* __restrict__ grad, const int64_t* __restrict__ slice_ptr_t,
           const int32_t* __restrict__ col_t, const T* __restrict__ val_t, const T* __restrict__ q,
           const T* __restrict__ lam, T* __restrict__ z) {
  const int lane = threadIdx.x & 31;
  const int64_t slice = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t r = slice * kSlice + lane;
  if (slice * kSlice >= nrows) return;
  if (z != nullptr) {
    const int64_t s0 = slice_ptr_t[slice], s1 = slice_ptr_t[slice + 1];
    T acc0 = T(0), acc1 = T(0);
    int64_t p = s0 + lane;
    for (; p + kSlice < s1; p += 2 * kSlice) {
      const int c0 = ld_stream_i32(col_t + p), c1 = ld_stream_i32(col_t + p + kSlice);
      const T v0 = ld_stream_t(val_t + p), v1 = ld_stream_t(val_t + p + kSlice);
      acc0 = fma(v0, __ldg(lam + c0), acc0);
      acc1 = fma(v1, __ldg(lam + c1), acc1);
    }
    if (p < s1) acc0 = fma(ld_stream_t(val_t + p), __ldg(lam + ld_stream_i32(col_t + p)), acc0);
    if (r < nrows) z[r] = acc0 + acc1;
  }
  {
    const int64_t s0 = slice_ptr[slice], s1 = slice_ptr[slice + 1];
    const T lr = r < nrows ? __ldg(lam + r) : T(0);
    for (int64_t p = s0 + lane; p < s1; p += kSlice) {
      const int c = ld_stream_i32(col + p);
      grad[p] = fma(lr, __ldg(q + c), grad[p]);
    }
  }
}

// Deferred parameter cotangent of a whole adjoint sweep in ONE pass:
//   grad[slot] += sum_m Lam[m][r] * Q[m][col[slot]]       (d sum_m <Lam_m, A Q_m> / dparams)
// instead of a read-modify-write of `grad` (and a read of `col`) in every step.  One warp per slice, lane = row;
// W entries of the row are accumulated in registers while m runs over the K (lambda, q) pairs: `Lam[m][r]` is one
// coalesced load per m, `Q[m][col]` a gather that is coalesced for banded rows and mostly served by L2 (neighbouring
// slices read the same lines).  Same summation order as the per-step kernel (m = count-1 .. 0).
// acc[j] += sum_m Lam[m][rr] * Q[m][c[j]], m = count-1 .. 0.  U pairs per round: their U lambdas and U x W gathers are
// ISSUED before the first FMA.  (Left to the compiler, the loop kept two or three loads in flight per warp -- ncu: 24
// warps per issue on the long scoreboard, DRAM 17 %, L2 -> L1 4.7 TB/s -- and the pass was bound by the round trip of
// its gathers: 3.95 ms for the 400 pairs of a lockstep batch at C2, 1.80 ms with the loads batched.)
template <typename T, int W, int U>
__device__ __forceinline__ void grad_accumulate(T (&acc)[W], const int (&c)[W], const T* __restrict__ Lam, int64_t ldl,
                                                int64_t rr, bool live, const T* __restrict__ Q, int64_t ldq, int count) {
  int m = count - 1;
  for (; m >= U - 1; m -= U) {
    T lr[U], g[U][W];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      lr[u] = __ldg(Lam + (int64_t)(m - u) * ldl + rr);
      const T* qm = Q + (int64_t)(m - u) * ldq;
#pragma unroll
      for (int j = 0; j < W; ++j) g[u][j] = __ldg(qm + c[j]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const T l = live ? lr[u] : T(0);
#pragma unroll
      for (int j = 0; j < W; ++j) acc[j] = fma(l, g[u][j], acc[j]);
    }
  }
  for (; m >= 0; --m) {
    const T l = live ? __ldg(Lam + (int64_t)m * ldl + rr) : T(0);
    const T* qm = Q + (int64_t)m * ldq;
#pragma unroll
    for (int j = 0; j < W; ++j) acc[j] = fma(l, __ldg(qm + c[j]), acc[j]);
  }
}

template <typename T, int W, int U>
__global__ void __launch_bounds__(256, U >= 4 ? 2 : 3)
k_sell_grad_batch(int64_t nrows, const int64_t* __restrict__ slice_ptr, const int32_t* __restrict__ col,
                  T* __restrict__ grad, const T* __restrict__ Q, int64_t ldq, const T* __restrict__ Lam, int64_t ldl,
                  int count) {
  const int lane = threadIdx.x & 31;
  const int64_t slice = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (slice * kSlice >= nrows) return;
  const int64_t r = slice * kSlice + lane;
  const int64_t rr = r < nrows ? r : nrows - 1;  // padded lanes read a valid row, their lambda counts as zero
  const int64_t s0 = slice_ptr[slice], s1 = slice_ptr[slice + 1];
  const int width = (int)((s1 - s0) / kSlice);
  const bool live = r < nrows;
  for (int k0 = 0; k0 < width; k0 += W) {
    int c[W];
    T acc[W];
#pragma unroll
    for (int j = 0; j < W; ++j) {
      const int k = k0 + j < width ? k0 + j : width - 1;
      c[j] = ld_stream_i32(col + s0 + (int64_t)k * kSlice + lane);
      acc[j] = T(0);
    }
    grad_accumulate<T, W, U>(acc, c, Lam, ldl, rr, live, Q, ldq, count);
#pragma unroll
    for (int j = 0; j < W; ++j)
      if (k0 + j < width) grad[s0 + (int64_t)(k0 + j) * kSlice + lane] += acc[j];
  }
}

// The same pass with the (lambda, q) pairs STAGED by the TMA engine.  k_sell_grad_batch keeps two pairs in flight per
// warp and is bound by the round trip of its loads (3.96 ms for the 400 pairs of a lockstep batch at n = 1M, where the
// bytes take 0.5 ms).  Here a block owns kGradRows consecutive rows (8 slices); its rows of Lam[m] are one contiguous
// segment, and so is the WINDOW of columns its entries touch when the operand is banded or locally clustered: a
// producer thread streams both segments of pair m = count-1 .. 0 through a ring of shared-memory stages (bulk copies,
// mbarrier completion), the consumer warps read lambda and gather q from the stage -- no registers and no warp slots
// are spent on loads in flight, and a block keeps the whole ring outstanding.  Same summation order, same arithmetic:
// bit-identical to k_sell_grad_batch.  A block whose window does not fit (kGradWinMax columns) gathers from global
// memory as before.
constexpr int kGradRows = 256;    // rows of a block: 8 slices, one consumer warp each
constexpr int kGradWarps = kGradRows / kSlice;
constexpr int kGradWinMax = 512;  // columns of the q window a stage can hold
constexpr int kGradStageBytes = 48 * 1024;

template <typename T>
constexpr int grad_stages() {
  return kGradStageBytes / ((kGradRows + kGradWinMax) * (int)sizeof(T));
}

template <typename T, int W>
__global__ void __launch_bounds__((kGradWarps + 1) * 32)
k_sell_grad_tma(int64_t nrows, int64_t nslices, const int64_t* __restrict__ slice_ptr, const int32_t* __restrict__ col,
                T* __restrict__ grad, const T* __restrict__ Q, int64_t ldq, const T* __restrict__ Lam, int64_t ldl,
                int count) {
  constexpr int STAGES = grad_stages<T>();
  constexpr int STAGE_ELEMS = kGradRows + kGradWinMax;
  constexpr int ALIGN = 16 / (int)sizeof(T);  // elements per 16 bytes (bulk copies)
  extern __shared__ __align__(128) unsigned char grad_smem[];
  T* stages = reinterpret_cast<T*>(grad_smem);
  uint64_t* full = reinterpret_cast<uint64_t*>(stages + (size_t)STAGES * STAGE_ELEMS);
  uint64_t* empty = full + STAGES;
  __shared__ int win_s[3];  // min column, max column, max width over the block's slices
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row0 = (int64_t)blockIdx.x * kGradRows;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      tma::mbar_init(full + s, 1);
      tma::mbar_init(empty + s, kGradWarps);
    }
    tma::fence_barrier_init();
    win_s[0] = 0x7fffffff;
    win_s[1] = -1;
    win_s[2] = 0;
  }
  __syncthreads();
  const int64_t slice = (int64_t)blockIdx.x * kGradWarps + warp;
  const bool consumer = warp < kGradWarps;
  const bool active = consumer && slice < nslices;
  const int64_t r = slice * kSlice + lane;
  int64_t s0 = 0;
  int width = 0;
  if (active) {
    s0 = slice_ptr[slice];
    width = (int)((slice_ptr[slice + 1] - s0) / kSlice);
    int cmin = 0x7fffffff, cmax = -1;
    if (r < nrows)
      for (int k = 0; k < width; ++k) {
        const int c = ld_stream_i32(col + s0 + (int64_t)k * kSlice + lane);
        cmin = c < cmin ? c : cmin;
        cmax = c > cmax ? c : cmax;
      }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const int a = __shfl_xor_sync(0xffffffffu, cmin, o), b = __shfl_xor_sync(0xffffffffu, cmax, o);
      cmin = a < cmin ? a : cmin;
      cmax = b > cmax ? b : cmax;
    }
    if (lane == 0) {
      atomicMin(&win_s[0], cmin);
      atomicMax(&win_s[1], cmax);
      atomicMax(&win_s[2], width);
    }
  }
  __syncthreads();
  const int cmin = win_s[0], cmax = win_s[1], wmax = win_s[2];
  if (cmax < cmin || wmax == 0) return;  // nothing stored in these rows
  const int w0 = cmin / ALIGN * ALIGN;
  const int wlen = (cmax + 1 - w0 + ALIGN - 1) / ALIGN * ALIGN;
  const bool staged = wlen <= kGradWinMax;
  const int npass = (wmax + W - 1) / W;
  if (!consumer) {
    if (lane == 0 && staged) {  // ---- producer ----
      const int64_t lrows = ldl - row0 < kGradRows ? ldl - row0 : kGradRows;  // ld is a multiple of 16 bytes
      const uint32_t bytes_l = (uint32_t)(lrows * (int64_t)sizeof(T)), bytes_q = (uint32_t)wlen * (uint32_t)sizeof(T);
      int it = 0;
      for (int pass = 0; pass < npass; ++pass)
        for (int m = count - 1; m >= 0; --m, ++it) {
          const int s = it % STAGES;
          tma::mbar_wait(empty + s, ((it / STAGES) & 1) ^ 1);
          tma::mbar_arrive_expect_tx(full + s, bytes_l + bytes_q);
          T* dst = stages + (size_t)s * STAGE_ELEMS;
          tma::bulk_g2s(dst, Lam + (int64_t)m * ldl + row0, bytes_l, full + s);
          tma::bulk_g2s(dst + kGradRows, Q + (int64_t)m * ldq + w0, bytes_q, full + s);
        }
    }
    return;
  }
  const bool live = active && r < nrows;
  int it = 0;
  for (int pass = 0; pass < npass; ++pass) {
    const int k0 = pass * W;
    int c[W];
    T acc[W];
#pragma unroll
    for (int j = 0; j < W; ++j) {
      const int k = k0 + j < width ? k0 + j : width - 1;
      c[j] = active && width > 0 ? ld_stream_i32(col + s0 + (int64_t)k * kSlice + lane) : w0;
      if (staged) c[j] = live ? c[j] - w0 : 0;  // padded lanes hold a lambda of zero: any column of the window does
      acc[j] = T(0);
    }
    if (staged) {
      for (int m = count - 1; m >= 0; --m, ++it) {
        const int s = it % STAGES;
        tma::mbar_wait(full + s, (it / STAGES) & 1);
        const T* st = stages + (size_t)s * STAGE_ELEMS;
        const T lr = live ? st[warp * kSlice + lane] : T(0);
        const T* qs = st + kGradRows;
        if (k0 < width) {
#pragma unroll
          for (int j = 0; j < W; ++j) acc[j] = fma(lr, qs[c[j]], acc[j]);
        }
        __syncwarp();
        if (lane == 0) tma::mbar_arrive(empty + s);
      }
    } else if (active && k0 < width) {
      grad_accumulate<T, W, 2>(acc, c, Lam, ldl, r < nrows ? r : nrows - 1, r < nrows, Q, ldq, count);
    }
    if (active)
#pragma unroll
      for (int j = 0; j < W; ++j)
        if (k0 + j < width) grad[s0 + (int64_t)(k0 + j) * kSlice + lane] += acc[j];
  }
}

struct SellDev {
  DevBuf slice_ptr, col, src, val;
  int64_t nslots = 0, nslices = 0;
  int upload(const SellHost& h) {
    nslots = h.nslots;
    nslices = (int64_t)h.slice_ptr.size() - 1;
    BL_CHECK(slice_ptr.ensure(h.slice_ptr.size() * sizeof(int64_t)));
    BL_CHECK(col.ensure(std::max<size_t>(1, h.col.size()) * sizeof(int32_t)));
    BL_CHECK(src.ensure(std::max<size_t>(1, h.src.size()) * sizeof(int32_t)));
    BL_CUDA(cudaMemcpy(slice_ptr.p, h.slice_ptr.data(), h.slice_ptr.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
    if (!h.col.empty()) {
      BL_CUDA(cudaMemcpy(col.p, h.col.data(), h.col.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
      BL_CUDA(cudaMemcpy(src.p, h.src.data(), h.src.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    }
    return BL_OK;
  }
};

}  // namespace

struct SparseOperator : bl_operator {
  int64_t n_rows = 0, n_cols = 0, nnz = 0;
  struct HostIndex {  // the finished index work, shared by the clones of an operator
    CsrHost csr;                 // kept for the bit-exact export
    SellHost sell_h, sell_t_h;   // idem
  };
  std::shared_ptr<HostIndex> host = std::make_shared<HostIndex>();
  SellDev sell, sell_t;
  DevBuf grad;
  int bound_dtype = -1;

  int num_params() const override { return 1; }
  int64_t param_size(int) const override { return nnz; }
  // SURVEY 8(d): operator nnz(w+4)+4(n+1) (+ x, y); with cotangent nnz(3w+4)+4(n+1) (+ q, lam, z)
  double matvec_bytes(int dtype) const override {
    const double w = dtype == BL_F32 ? 4 : 8;
    return nnz * (w + 4) + 4.0 * (n_rows + 1) + 2.0 * n_rows * w;
  }
  double matvec_batch_bytes(int dtype, int count) const override {  // values + indices once per kSpmvBatch vectors
    const double w = dtype == BL_F32 ? 4 : 8;
    const int chunks = (count + kSpmvBatch - 1) / kSpmvBatch;
    return chunks * (nnz * (w + 4) + 4.0 * (n_rows + 1)) + 2.0 * count * n_rows * w;
  }
  double vjp_bytes(int dtype) const override {
    const double w = dtype == BL_F32 ? 4 : 8;
    return nnz * (3 * w + 4) + 4.0 * (n_rows + 1) + 3.0 * n_rows * w;
  }

  int build(const int32_t* row, const int32_t* col) {
    CsrHost& csr = host->csr;
    csr = coo_to_csr(n_rows, nnz, row, col);
    host->sell_h = csr_to_sell(n_rows, csr);
    CsrHost csr_t = coo_to_csr(n_cols, nnz, col, row);
    host->sell_t_h = csr_to_sell(n_cols, csr_t);
    // how many blocks of kGradRows rows keep their columns inside one window k_sell_grad_tma can stage
    int64_t blocks = 0, fit = 0;
    for (int64_t r0 = 0; r0 < n_rows; r0 += kGradRows, ++blocks) {
      const int64_t r1 = std::min<int64_t>(n_rows, r0 + kGradRows);
      int32_t lo = INT32_MAX, hi = -1;
      for (int64_t k = csr.row_ptr[r0]; k < csr.row_ptr[r1]; ++k) {
        lo = std::min(lo, csr.col_idx[k]);
        hi = std::max(hi, csr.col_idx[k]);
      }
      if (hi < lo || hi - lo + 8 <= kGradWinMax) ++fit;
    }
    grad_windows_fit = blocks > 0 && 4 * fit >= 3 * blocks;
    return BL_OK;  // pure host index work: testable without a GPU; upload happens on first bind
  }
  bool grad_windows_fit = false;  // banded / locally clustered rows: the deferred cotangent pass stages its pairs (TMA)

  bool uploaded = false;
  int ensure_uploaded() {
    if (uploaded) return BL_OK;
    BL_CHECK(sell.upload(host->sell_h));
    BL_CHECK(sell_t.upload(host->sell_t_h));
    uploaded = true;
    return BL_OK;
  }

  template <typename T>
  int set_params_t(const T* params, cudaStream_t s) {
    BL_CHECK(sell.val.ensure(std::max<int64_t>(1, sell.nslots) * sizeof(T)));
    BL_CHECK(sell_t.val.ensure(std::max<int64_t>(1, sell_t.nslots) * sizeof(T)));
    BL_CHECK(grad.ensure(std::max<int64_t>(1, sell.nslots) * sizeof(T)));
    const int blocks = 148 * 8;
    if (sell.nslots > 0) {
      k_gather_values<T><<<blocks, 256, 0, s>>>(sell.nslots, sell.src.as<int32_t>(), params, sell.val.as<T>());
      BL_LAUNCHED();
    }
    if (sell_t.nslots > 0) {
      k_gather_values<T><<<blocks, 256, 0, s>>>(sell_t.nslots, sell_t.src.as<int32_t>(), params, sell_t.val.as<T>());
      BL_LAUNCHED();
    }
    return BL_OK;
  }

  int set_params(int dtype, const void* const* params, int num, cudaStream_t s) override {
    BL_REQUIRE(num == 1 && params && params[0], "sparse operator takes one parameter (COO data)");
    BL_CHECK(ensure_uploaded());
    bound_dtype = dtype;
    return dtype == BL_F32 ? set_params_t<float>(static_cast<const float*>(params[0]), s)
                           : set_params_t<double>(static_cast<const double*>(params[0]), s);
  }

  template <typename T>
  int matvec_t(const T* x, T* y, cudaStream_t s) {
    const void* in[1] = {x};
    void* out[1] = {y};
    return spmv_multi_t<T, false>(sell, n_rows, 1, in, nullptr, nullptr, 0, out, s);
  }

  int matvec(int dtype, const void* x, void* y, cudaStream_t s) override {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    return dtype == BL_F32 ? matvec_t<float>(static_cast<const float*>(x), static_cast<float*>(y), s)
                           : matvec_t<double>(static_cast<const double*>(x), static_cast<double*>(y), s);
  }

  template <typename T>
  int matvec_normalised_t(const T* v, const double* len, T* q_out, int64_t n_pad, T* y, cudaStream_t s) {
    const void* in[1] = {v};
    const double* lens[1] = {len};
    void* q[1] = {q_out};
    void* out[1] = {y};
    return spmv_multi_t<T, true>(sell, n_rows, 1, in, lens, q, n_pad, out, s);
  }
  int matvec_normalised(int dtype, const void* v, const double* len, void* q_out, int64_t n_pad, void* y,
                        cudaStream_t s) override {
    // the fused kernel writes the padded row from its own threads: it needs a square operand whose slices
    // cover the padding, and in-place use (y aliasing v) is not possible
    if (dtype != bound_dtype || n_rows != n_cols || n_pad > sell.nslices * kSlice || v == y || n_rows == 0) return -1;
    return dtype == BL_F32
               ? matvec_normalised_t<float>(static_cast<const float*>(v), len, static_cast<float*>(q_out), n_pad,
                                            static_cast<float*>(y), s)
               : matvec_normalised_t<double>(static_cast<const double*>(v), len, static_cast<double*>(q_out), n_pad,
                                             static_cast<double*>(y), s);
  }

  // ---- several vectors per launch (lockstep runs): the operand's values and indices are read once per chunk ----
  template <typename T, bool NORM>
  int spmv_multi_t(const SellDev& m, int64_t rows, int count, const void* const* in, const double* const* len,
                   void* const* q_out, int64_t n_pad, void* const* out, cudaStream_t s) {
    const int64_t threads = m.nslices * kSlice;
    const int blocks = (int)((threads + 255) / 256);
    if (blocks <= 0) return BL_OK;
    for (int first = 0; first < count; first += kSpmvBatch) {
      const int P = std::min(kSpmvBatch, count - first);
      MultiVec mv = {};
      for (int pp = 0; pp < P; ++pp) {
        mv.x[pp] = in[first + pp];
        mv.y[pp] = out[first + pp];
        mv.len[pp] = NORM ? len[first + pp] : nullptr;
        mv.q[pp] = NORM ? q_out[first + pp] : nullptr;
      }
      const int64_t* sp = m.slice_ptr.as<int64_t>();
      const int32_t* cl = m.col.as<int32_t>();
      const T* vl = m.val.as<T>();
      switch (P) {
        case 1: k_sell_spmv_multi<T, 1, NORM, 6><<<blocks, 256, 0, s>>>(rows, sp, cl, vl, mv, n_pad); break;
        case 2: k_sell_spmv_multi<T, 2, NORM, 6><<<blocks, 256, 0, s>>>(rows, sp, cl, vl, mv, n_pad); break;
        case 3: k_sell_spmv_multi<T, 3, NORM, 4><<<blocks, 256, 0, s>>>(rows, sp, cl, vl, mv, n_pad); break;
        default: k_sell_spmv_multi<T, 4, NORM, 4><<<blocks, 256, 0, s>>>(rows, sp, cl, vl, mv, n_pad); break;
      }
      BL_LAUNCHED();
    }
    return BL_OK;
  }
  int matvec_batch(int dtype, int count, const void* const* in, void* const* out, cudaStream_t s) override {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    return dtype == BL_F32 ? spmv_multi_t<float, false>(sell, n_rows, count, in, nullptr, nullptr, 0, out, s)
                           : spmv_multi_t<double, false>(sell, n_rows, count, in, nullptr, nullptr, 0, out, s);
  }
  int apply_transpose_batch(int dtype, int count, const void* const* in, void* const* out, cudaStream_t s) override {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    BL_REQUIRE(n_rows == n_cols, "A^T lam needs a square operator");
    return dtype == BL_F32 ? spmv_multi_t<float, false>(sell_t, n_cols, count, in, nullptr, nullptr, 0, out, s)
                           : spmv_multi_t<double, false>(sell_t, n_cols, count, in, nullptr, nullptr, 0, out, s);
  }
  int matvec_normalised_batch(int dtype, int count, const void* const* v, const double* const* len, void* const* q_out,
                              int64_t n_pad, void* const* y, cudaStream_t s) override {
    if (dtype != bound_dtype || n_rows != n_cols || n_pad > sell.nslices * kSlice || n_rows == 0) return -1;
    for (int p = 0; p < count; ++p)
      if (v[p] == y[p]) return -1;
    return dtype == BL_F32 ? spmv_multi_t<float, true>(sell, n_rows, count, v, len, q_out, n_pad, y, s)
                           : spmv_multi_t<double, true>(sell, n_rows, count, v, len, q_out, n_pad, y, s);
  }

  template <typename T>
  int vjp_t(const T* q, const T* lam, T* z, cudaStream_t s) {
    const int64_t rows = z ? std::max(n_rows, n_cols) : n_rows;
    const int64_t threads = ((rows + kSlice - 1) / kSlice) * kSlice;
    const int blocks = (int)((threads + 255) / 256);
    if (blocks > 0) {
      k_sell_vjp<T><<<blocks, 256, 0, s>>>(rows, sell.slice_ptr.as<int64_t>(), sell.col.as<int32_t>(),
                                           grad.as<T>(), sell_t.slice_ptr.as<int64_t>(),
                                           sell_t.col.as<int32_t>(), sell_t.val.as<T>(), q, lam, z);
      BL_LAUNCHED();
    }
    return BL_OK;
  }

  int vjp(int dtype, const void* q, const void* lam, void* z, cudaStream_t s) override {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    BL_REQUIRE(n_rows == n_cols || z == nullptr, "A^T lam needs a square operator (pass z = NULL for the gradient only)");
    return dtype == BL_F32
               ? vjp_t<float>(static_cast<const float*>(q), static_cast<const float*>(lam), static_cast<float*>(z), s)
               : vjp_t<double>(static_cast<const double*>(q), static_cast<const double*>(lam), static_cast<double*>(z), s);
  }

  // Deferred cotangent (square operands): inside the adjoint loop only z = A^T lam (an SpMV with the SELL of
  // A^T: 92 MB per step instead of the 175 MB of the matvec-VJP at C2), then one batched pass over the K
  // (lambda, q) pairs.
  bool deferred_grad(int dtype) const override { return dtype == bound_dtype && n_rows == n_cols && n_rows > 0; }
  double apply_transpose_bytes(int dtype) const override { return matvec_bytes(dtype); }
  double vjp_batch_bytes(int dtype, int count) const override {  // Q and Lambda once, col, grad read + write
    const double w = dtype == BL_F32 ? 4 : 8;
    return 2.0 * count * n_rows * w + nnz * (4 + 2 * w) + 4.0 * (n_rows + 1);
  }
  template <typename T>
  int apply_transpose_t(const T* lam, T* z, cudaStream_t s) {
    const void* in[1] = {lam};
    void* out[1] = {z};
    return spmv_multi_t<T, false>(sell_t, n_cols, 1, in, nullptr, nullptr, 0, out, s);
  }
  int apply_transpose(int dtype, const void* lam, void* z, cudaStream_t s) override {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    BL_REQUIRE(n_rows == n_cols, "A^T lam needs a square operator");
    return dtype == BL_F32 ? apply_transpose_t<float>(static_cast<const float*>(lam), static_cast<float*>(z), s)
                           : apply_transpose_t<double>(static_cast<const double*>(lam), static_cast<double*>(z), s);
  }
  template <typename T>
  int vjp_batch_t(const T* Q, int64_t ldq, const T* Lam, int64_t ldl, int count, cudaStream_t s) {
    static const bool staged = [] {  // BL_GRAD_TMA=0: the register-staged pass everywhere (A/B measurements)
      const char* e = std::getenv("BL_GRAD_TMA");
      return !(e && e[0] == '0');
    }();
    // bulk copies: 16-byte aligned rows of Q and Lam (basis buffers of the drivers are)
    const bool aligned = (reinterpret_cast<uintptr_t>(Q) | reinterpret_cast<uintptr_t>(Lam)) % 16 == 0 &&
                         (ldq * sizeof(T)) % 16 == 0 && (ldl * sizeof(T)) % 16 == 0 && ldl >= n_rows && ldq >= n_cols;
    if (staged && grad_windows_fit && aligned && sell.nslices > 0 && count > 0) {
      constexpr size_t smem = (size_t)grad_stages<T>() * (kGradRows + kGradWinMax) * sizeof(T) + 2 * grad_stages<T>() * 8;
      {  // the opt-in is per device: one process may drive several GPUs from different host threads
        static std::mutex mu;
        static std::set<int> done;  // per instantiation (T)
        int dev = 0;
        BL_CUDA(cudaGetDevice(&dev));
        std::lock_guard<std::mutex> lk(mu);
        if (!done.count(dev)) {
          BL_CUDA(cudaFuncSetAttribute(k_sell_grad_tma<T, 12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
          done.insert(dev);
        }
      }
      const int blocks = (int)((sell.nslices + kGradWarps - 1) / kGradWarps);
      k_sell_grad_tma<T, 12><<<blocks, (kGradWarps + 1) * 32, smem, s>>>(n_rows, sell.nslices, sell.slice_ptr.as<int64_t>(),
                                                                       sell.col.as<int32_t>(), grad.as<T>(), Q, ldq, Lam,
                                                                       ldl, count);
      BL_LAUNCHED();
      return BL_OK;
    }
    const int64_t threads = sell.nslices * kSlice;
    const int blocks = (int)((threads + 255) / 256);
    if (blocks > 0 && count > 0) {
      // pairs per round: fp64 6.57 (1) -> 4.0 (2) -> 2.63 ms (4) for 400 pairs at C2
      constexpr int U = sizeof(T) == 8 ? 4 : 2;
      k_sell_grad_batch<T, 12, U><<<blocks, 256, 0, s>>>(n_rows, sell.slice_ptr.as<int64_t>(), sell.col.as<int32_t>(),
                                                         grad.as<T>(), Q, ldq, Lam, ldl, count);
      BL_LAUNCHED();
    }
    return BL_OK;
  }
  int vjp_batch(int dtype, const void* Q, int64_t ldq, const void* Lam, int64_t ldl, int count,
                cudaStream_t s) override {
    BL_REQUIRE(dtype == bound_dtype, "set_params must be called with the same dtype first");
    return dtype == BL_F32 ? vjp_batch_t<float>(static_cast<const float*>(Q), ldq, static_cast<const float*>(Lam), ldl, count, s)
                           : vjp_batch_t<double>(static_cast<const double*>(Q), ldq, static_cast<const double*>(Lam), ldl, count, s);
  }

  bool sell_view(int dtype, bool transpose, SellView* out) const override {
    if (dtype != bound_dtype || n_rows != n_cols || n_rows == 0 || !uploaded) return false;
    const SellDev& m = transpose ? sell_t : sell;
    if (m.nslots == 0 || m.val.p == nullptr) return false;
    out->slice_ptr = m.slice_ptr.as<int64_t>();
    out->col = m.col.as<int32_t>();
    out->val = m.val.p;
    out->nslices = m.nslices;
    out->nrows = n_rows;
    return true;
  }

  int grad_zero(int dtype, cudaStream_t s) override {
    BL_CHECK(grad.ensure(std::max<int64_t>(1, sell.nslots) * dtype_size(dtype)));
    BL_CUDA(cudaMemsetAsync(grad.p, 0, std::max<int64_t>(1, sell.nslots) * dtype_size(dtype), s));
    return BL_OK;
  }

  int grad_export(int dtype, void* const* grads, int num, cudaStream_t s) override {
    BL_REQUIRE(num == 1 && grads && grads[0], "sparse operator has one gradient buffer");
    if (sell.nslots == 0) return BL_OK;
    const int blocks = 148 * 8;
    if (dtype == BL_F32)
      k_scatter_grad<float><<<blocks, 256, 0, s>>>(sell.nslots, sell.src.as<int32_t>(), grad.as<float>(), static_cast<float*>(grads[0]));
    else
      k_scatter_grad<double><<<blocks, 256, 0, s>>>(sell.nslots, sell.src.as<int32_t>(), grad.as<double>(), static_cast<double*>(grads[0]));
    BL_LAUNCHED();
    return BL_OK;
  }
};

}  // namespace bl

extern "C" {

int bl_op_sparse_create(int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* coo_row_host,
                        const int32_t* coo_col_host, bl_operator_t** op) {
  BL_REQUIRE(op != nullptr, "op is NULL");
  BL_REQUIRE(n_rows > 0 && n_cols > 0 && nnz >= 0, "bad shape");
  BL_REQUIRE(nnz == 0 || (coo_row_host && coo_col_host), "index arrays are NULL");
  BL_REQUIRE(nnz < (int64_t)1 << 31, "nnz must fit int32");
  for (int64_t e = 0; e < nnz; ++e) {
    BL_REQUIRE(coo_row_host[e] >= 0 && coo_row_host[e] < n_rows, "row index out of range");
    BL_REQUIRE(coo_col_host[e] >= 0 && coo_col_host[e] < n_cols, "column index out of range");
  }
  auto* o = new bl::SparseOperator();
  o->n = n_rows;
  o->n_rows = n_rows;
  o->n_cols = n_cols;
  o->nnz = nnz;
  int rc = o->build(coo_row_host, coo_col_host);
  if (rc != BL_OK) {
    delete o;
    return rc;
  }
  *op = o;
  return BL_OK;
}

int bl_op_sparse_clone(const bl_operator_t* op, bl_operator_t** clone) {
  auto* src = dynamic_cast<const bl::SparseOperator*>(op);
  BL_REQUIRE(src != nullptr && clone != nullptr, "not a sparse operator");
  auto* o = new bl::SparseOperator();
  o->n = src->n;
  o->n_rows = src->n_rows;
  o->n_cols = src->n_cols;
  o->nnz = src->nnz;
  o->host = src->host;  // shared, read-only after build()
  o->grad_windows_fit = src->grad_windows_fit;
  *clone = o;  // device buffers are uploaded on the clone's first bind
  return BL_OK;
}

int bl_op_sparse_export_csr(const bl_operator_t* op, int32_t* row_ptr_host, int32_t* col_idx_host,
                            int32_t* perm_host) {
  auto* o = dynamic_cast<const bl::SparseOperator*>(op);
  BL_REQUIRE(o != nullptr, "not a sparse operator");
  if (row_ptr_host) std::copy(o->host->csr.row_ptr.begin(), o->host->csr.row_ptr.end(), row_ptr_host);
  if (col_idx_host) std::copy(o->host->csr.col_idx.begin(), o->host->csr.col_idx.end(), col_idx_host);
  if (perm_host) std::copy(o->host->csr.perm.begin(), o->host->csr.perm.end(), perm_host);
  return BL_OK;
}

int bl_op_sparse_export_sell(const bl_operator_t* op, int transpose, int64_t* slice_ptr_host,
                             int64_t* slot_of_csr_host) {
  auto* o = dynamic_cast<const bl::SparseOperator*>(op);
  BL_REQUIRE(o != nullptr, "not a sparse operator");
  const auto& h = transpose ? o->host->sell_t_h : o->host->sell_h;
  if (slice_ptr_host) std::copy(h.slice_ptr.begin(), h.slice_ptr.end(), slice_ptr_host);
  if (slot_of_csr_host) std::copy(h.slot_of_csr.begin(), h.slot_of_csr.end(), slot_of_csr_host);
  return BL_OK;
}

}  // extern "C"
