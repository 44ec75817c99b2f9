// TMA-staged versions of the basis-streaming kernels (sm_100a).
//
//   k_dots_tma    : red[j] = <row_j, x>                      pass A of CGS2, adjoint re-projection
//   k_combine_tma : out = s * (sum_k a_k vec_k + sum_j c_j row_j) (+ ||out||^2)   pass C, adjoint back-substitution
//   k_fused_tma   : out = combine(...)  AND  red[j] = <row_j, out> from ONE read of the rows  (pass B; adjoint)
//
// Persistent blocks (2 per SM): block b owns a contiguous, balanced range of columns and walks it
// in tiles.  Warp 8 lane 0 is the producer: for every tile and every group of 8 basis rows it
// issues one bulk copy per row segment into a shared-memory stage; warps 0-7 consume.  In
// k_fused_tma the rows that are needed twice stay resident for the tile, so the second use
// reads shared memory instead of HBM.
//
// Contract: row buffers are zero-padded up to `ld` (ld*sizeof(T) % 16 == 0), so the 16-byte
// vector that straddles `n` can be copied and multiplied without masking.
#pragma once

#include <cuda.h>

#include "krylov_kernels.cuh"
#include "tma_pipeline.cuh"

namespace bl {

constexpr int kGroup = 8;            // basis rows per pipeline stage (= consumer warps)
constexpr int kConsumerWarps = 8;
constexpr int kConsumerThreads = 32 * kConsumerWarps;
constexpr int kStreamThreads = kConsumerThreads + 32;  // + producer warp
constexpr int kStages = 3;
constexpr int kBoxesPerBarrier = 4;  // fused kernel: resident boxes ([8 x TILE]) that share one mbarrier

// Rows [0, n0) from block 0, [n0, n0 + n1) from block 1.  The kernels copy them with the L2 evict_first policy: a
// stream that is larger than L2 does not push the vectors (and the operand) out, which every step reads again
// (measured +4 % for one run alone).
struct RowSource {
  const char* base0 = nullptr;
  long long ldb0 = 0;  // bytes
  int n0 = 0;
  const char* base1 = nullptr;
  long long ldb1 = 0;
  int n1 = 0;
  __device__ __forceinline__ const char* row(int j) const {
    return j < n0 ? base0 + (long long)j * ldb0 : base1 + (long long)(j - n0) * ldb1;
  }
};

struct ColumnRange {
  long long c0, c1;  // [c0, c1) columns of this block, in elements; c1 - c0 multiple of the vector width
  int ntiles;
};

template <typename T>
__device__ __forceinline__ ColumnRange block_columns(long long n, int tile) {
  constexpr int VN = Vec<T>::N;
  const long long n_v = (n + VN - 1) / VN * VN;
  long long per = (n_v + gridDim.x - 1) / gridDim.x;
  per = (per + 31) / 32 * 32;
  ColumnRange r;
  r.c0 = per * blockIdx.x;
  r.c1 = r.c0 + per < n_v ? r.c0 + per : n_v;
  r.ntiles = r.c0 < r.c1 ? (int)((r.c1 - r.c0 + tile - 1) / tile) : 0;
  return r;
}

// This thread's column vector of p at column c, when `live`; zero otherwise.  Vectors of length n are not zero-padded:
// the one that straddles n is read element by element, its elements past n as zero.
template <typename T>
__device__ __forceinline__ typename Vec<T>::type load_colvec(const T* p, long long c, long long n, bool live) {
  constexpr int VN = Vec<T>::N;
  if (live && c + VN <= n) return *reinterpret_cast<const typename Vec<T>::type*>(p + c);
  T z[VN];
#pragma unroll
  for (int k = 0; k < VN; ++k) z[k] = T(0);
  if (live)
#pragma unroll
    for (int k = 0; k < VN; ++k)
      if (c + k < n) z[k] = p[c + k];
  return vec_pack(z);
}

// Stores this thread's column vector at column c of p; of the vector that straddles n, only the elements before n.
template <typename T>
__device__ __forceinline__ void store_colvec(T* p, long long c, long long n, const T (&v)[Vec<T>::N]) {
  constexpr int VN = Vec<T>::N;
  if (c + VN <= n) {
    *reinterpret_cast<typename Vec<T>::type*>(p + c) = vec_pack(v);
  } else {
#pragma unroll
    for (int k = 0; k < VN; ++k)
      if (c + k < n) p[c + k] = v[k];
  }
}

// Producer: group g of the rows [0, nrows) of src, columns [tc0, tc0 + len), into ring stage it % kStages once the
// consumers have released it.
template <typename T, int TILE>
__device__ __forceinline__ void stage_rows(T* stages, uint64_t* full, uint64_t* empty, int it, const RowSource& src,
                                           int g, int nrows, long long tc0, int len) {
  const uint32_t bytes = (uint32_t)len * sizeof(T);
  const int rows_here = nrows - g * kGroup < kGroup ? nrows - g * kGroup : kGroup;
  const int s = it % kStages;
  tma::mbar_wait(empty + s, ((it / kStages) & 1) ^ 1);
  tma::mbar_arrive_expect_tx(full + s, bytes * rows_here);
  T* dst = stages + (size_t)s * kGroup * TILE;
  const uint64_t pol = tma::policy_evict_first();
  for (int r = 0; r < rows_here; ++r)
    tma::bulk_g2s_hint(dst + (size_t)r * TILE, src.row(g * kGroup + r) + tc0 * (long long)sizeof(T), bytes, full + s,
                       pol);
}

// acc += sum_r cf[r] * (row r of a staged group) for this thread's column vector (st: its vector of row 0): a full
// group with all loads first.
template <typename T, int TILE>
__device__ __forceinline__ void fma_group(const typename Vec<T>::type* st, const T* cf, int rows, T (&acc)[Vec<T>::N]) {
  using V = typename Vec<T>::type;
  constexpr int VN = Vec<T>::N;
  if (rows == kGroup) {
    V q[kGroup];
#pragma unroll
    for (int r = 0; r < kGroup; ++r) q[r] = st[(size_t)r * (TILE / VN)];
#pragma unroll
    for (int r = 0; r < kGroup; ++r) {
      T e[VN];
      vec_unpack(q[r], e);
#pragma unroll
      for (int k = 0; k < VN; ++k) acc[k] = fma(cf[r], e[k], acc[k]);
    }
  } else {
    for (int r = 0; r < rows; ++r) {
      T e[VN];
      vec_unpack(st[(size_t)r * (TILE / VN)], e);
#pragma unroll
      for (int k = 0; k < VN; ++k) acc[k] = fma(cf[r], e[k], acc[k]);
    }
  }
}

// Fixed-order cross-block reduction + epilogue, run by the last block (all threads call it).
// Latency-bound (one block reads gridDim.x * nrows doubles from L2), so every lane issues all of
// its loads for two rows before the first add: <= 10 independent 16-byte loads in flight.
template <typename T>
__device__ __forceinline__ void reduce_partials_and_epilogue(int nrows, const double* __restrict__ partials,
                                                             const Epi& epi) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int G = gridDim.x;
  if ((G & 1) == 0 && G <= 320) {
    const int nv = G >> 1;  // 16-byte vectors per row
    for (int j = warp; j < nrows; j += 2 * nwarps) {
      const int j2 = j + nwarps < nrows ? j + nwarps : j;  // second row (or the same one again)
      const double2* p0 = reinterpret_cast<const double2*>(partials + (size_t)j * G);
      const double2* p1 = reinterpret_cast<const double2*>(partials + (size_t)j2 * G);
      double2 v0[5], v1[5];
#pragma unroll
      for (int k = 0; k < 5; ++k) {
        const int i = lane + 32 * k;
        const int ic = i < nv ? i : 0;
        v0[k] = __ldcg(p0 + ic);
        v1[k] = __ldcg(p1 + ic);
        if (i >= nv) v0[k] = v1[k] = make_double2(0.0, 0.0);
      }
      double s0 = 0.0, s1 = 0.0;
#pragma unroll
      for (int k = 0; k < 5; ++k) {
        s0 += v0[k].x + v0[k].y;
        s1 += v1[k].x + v1[k].y;
      }
      s0 = warp_sum(s0);
      s1 = warp_sum(s1);
      if (lane == 0) {
        epi.red[j] = s0;
        if (j2 != j) epi.red[j2] = s1;
      }
    }
  } else {
    for (int j = warp; j < nrows; j += nwarps) {
      const double* p = partials + (size_t)j * G;
      double s = 0.0;
      for (int b = lane; b < G; b += 32) s += __ldcg(p + b);
      s = warp_sum(s);
      if (lane == 0) epi.red[j] = s;
    }
  }
  __syncthreads();
  run_epilogue<T>(epi);
}

// ---------------------------------------------------------------------------------------------
// red[j] = <row_j, x>.  The x tile travels through its own double-buffered TMA slot so the
// consumers never wait on a global load; basis rows are prefetched before griddepcontrol.wait
// (they are older than the predecessor kernel), x — usually the predecessor's output — after it.
template <typename T, int TILE>
__global__ void __launch_bounds__(kStreamThreads, 2)
k_dots_tma(RowSource src, int nrows, const T* __restrict__ x, long long n, double* __restrict__ partials,
           unsigned int* counter, Epi epi, int reverse) {
  using V = typename Vec<T>::type;
  constexpr int VN = Vec<T>::N;
  constexpr int XV = TILE / (32 * VN);  // x vectors per lane
  extern __shared__ __align__(128) unsigned char smem_raw[];
  T* stages = reinterpret_cast<T*>(smem_raw);                       // [kStages][kGroup][TILE]
  T* xs = stages + (size_t)kStages * kGroup * TILE;                 // [2][TILE]
  uint64_t* full = reinterpret_cast<uint64_t*>(xs + 2 * TILE);
  uint64_t* empty = full + kStages;
  uint64_t* xfull = empty + kStages;   // [2]
  uint64_t* xempty = xfull + 2;        // [2]
  double* acc_s = reinterpret_cast<double*>(xempty + 2);            // [nrows]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      tma::mbar_init(full + s, 1);
      tma::mbar_init(empty + s, kConsumerWarps);
    }
    for (int s = 0; s < 2; ++s) {
      tma::mbar_init(xfull + s, 1);
      tma::mbar_init(xempty + s, kConsumerWarps);
    }
    tma::fence_barrier_init();
  }
  for (int j = threadIdx.x; j < nrows; j += blockDim.x) acc_s[j] = 0.0;
  __syncthreads();
  tma::griddep_launch_dependents();

  const ColumnRange cr = block_columns<T>(n, TILE);
  const int ngroups = (nrows + kGroup - 1) / kGroup;

  if (warp == kConsumerWarps) {
    if (lane == 0) {  // ---- producer ----
      const int total = cr.ntiles * ngroups;
      bool waited = false;
      auto issue_x = [&](int tt) {
        const int t = reverse ? cr.ntiles - 1 - tt : tt;
        const long long tc0 = cr.c0 + (long long)t * TILE;
        const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
        const int b = tt & 1;
        tma::mbar_wait(xempty + b, ((tt >> 1) & 1) ^ 1);
        tma::mbar_arrive_expect_tx(xfull + b, (uint32_t)len * sizeof(T));
        tma::bulk_g2s(xs + (size_t)b * TILE, x + tc0, (uint32_t)len * sizeof(T), xfull + b);
      };
      for (int it = 0; it < total; ++it) {
        const int tt = it / ngroups, gg = it - tt * ngroups;
        // x runs one tile ahead of the rows: x(0), x(1) right after the wait, x(tt+1) when tile tt starts
        if (!waited && (it == kStages || (gg == 0 && tt > 0))) {
          tma::griddep_wait();
          waited = true;
          issue_x(0);
          if (cr.ntiles > 1) issue_x(1);
        }
        if (gg == 0 && tt > 0 && tt + 1 < cr.ntiles) issue_x(tt + 1);
        const int t = reverse ? cr.ntiles - 1 - tt : tt;
        const int g = reverse ? ngroups - 1 - gg : gg;
        const long long tc0 = cr.c0 + (long long)t * TILE;
        const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
        stage_rows<T, TILE>(stages, full, empty, it, src, g, nrows, tc0, len);
      }
      if (!waited && total > 0) {
        tma::griddep_wait();
        issue_x(0);
        if (cr.ntiles > 1) issue_x(1);
      }
    }
  } else {  // ---- consumers: warp w takes row g*8 + w of every stage ----
    int it = 0;
    for (int tt = 0; tt < cr.ntiles; ++tt) {
      const int t = reverse ? cr.ntiles - 1 - tt : tt;
      const long long tc0 = cr.c0 + (long long)t * TILE;
      const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
      const int b = tt & 1;
      tma::mbar_wait(xfull + b, (tt >> 1) & 1);
      V xr[XV];
#pragma unroll
      for (int u = 0; u < XV; ++u) {
        const int e = (lane + 32 * u) * VN;
        T tmp[VN];
#pragma unroll
        for (int k = 0; k < VN; ++k) tmp[k] = T(0);
        if (e < len) {
          vec_unpack(reinterpret_cast<const V*>(xs + (size_t)b * TILE)[lane + 32 * u], tmp);
          if (tc0 + e + VN > n) {  // the vector that straddles n: x is not zero-padded
#pragma unroll
            for (int k = 0; k < VN; ++k)
              if (tc0 + e + k >= n) tmp[k] = T(0);
          }
        }
        xr[u] = vec_pack(tmp);
      }
      __syncwarp();
      if (lane == 0) tma::mbar_arrive(xempty + b);
      for (int gg = 0; gg < ngroups; ++gg, ++it) {
        const int g = reverse ? ngroups - 1 - gg : gg;
        const int s = it % kStages;
        tma::mbar_wait(full + s, (it / kStages) & 1);
        const int j = g * kGroup + warp;
        if (j < nrows) {
          const V* row = reinterpret_cast<const V*>(stages + ((size_t)s * kGroup + warp) * TILE);
          T a0 = T(0), a1 = T(0);
#pragma unroll
          for (int u = 0; u < XV; ++u) {
            if ((lane + 32 * u) * VN < len) {
              T q[VN], xx[VN];
              vec_unpack(row[lane + 32 * u], q);
              vec_unpack(xr[u], xx);
#pragma unroll
              for (int k = 0; k < VN; ++k) {
                if (u & 1)
                  a1 = fma(q[k], xx[k], a1);
                else
                  a0 = fma(q[k], xx[k], a0);
              }
            }
          }
          // release the stage before the (latency-bound) warp reduction: with three stages in
          // the ring every cycle a stage is held costs bytes in flight
          __syncwarp();
          if (lane == 0) tma::mbar_arrive(empty + s);
          double sacc = warp_sum(static_cast<double>(a0) + static_cast<double>(a1));
          if (lane == 0) acc_s[j] += sacc;  // row j is always handled by this warp: no race
        } else {
          __syncwarp();
          if (lane == 0) tma::mbar_arrive(empty + s);
        }
      }
    }
    tma::griddep_wait();  // blocks with no tile must still order their partial writes after the predecessor
  }
  __syncthreads();
  for (int j = threadIdx.x; j < nrows; j += blockDim.x) partials[(size_t)j * gridDim.x + blockIdx.x] = acc_s[j];
  if (!last_block_done(counter)) return;
  reduce_partials_and_epilogue<T>(nrows, partials, epi);
}

namespace step {
// fixed-order sum of one row of per-block partials by one warp; all loads of a lane are issued before the adds
__device__ __forceinline__ double row_sum(const double* __restrict__ p, int G, int lane) {
  double s = 0.0;
  if ((G & 1) == 0 && G <= 320) {
    const double2* p2 = reinterpret_cast<const double2*>(p);
    const int nv = G >> 1;
    double2 v[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const int i = lane + 32 * k;
      v[k] = __ldcg(p2 + (i < nv ? i : 0));
      if (i >= nv) v[k] = make_double2(0.0, 0.0);
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) s += v[k].x + v[k].y;
  } else {
    for (int k = lane; k < G; k += 32) s += __ldcg(p + k);
  }
  return warp_sum(s);
}

}  // namespace step

// ---------------------------------------------------------------------------------------------
// out = s * sum_j c_j row_j (+ ||out||^2): dense vector terms are rows too (src.nv leading
// single-row sources), so everything the consumers read arrives through the TMA pipeline.
// Row order inside a tile: basis groups first (prefetched before griddepcontrol.wait), the
// group(s) holding vector terms last (they may be the predecessor's output).
struct CombineTmaArgs {
  long long n = 0;
  void* out = nullptr;
  void* out2 = nullptr;
  int nvec = 0;
  VecTerm vec[kMaxVecTerms];
  RowSource src;                  // basis blocks only
  const double* coef0 = nullptr;  // coefficients of block 0 rows (already offset)
  double sign0 = 1.0;
  const double* coef1 = nullptr;
  double sign1 = 1.0;
  const double* out_div_ptr = nullptr;
  const double* out_mul_ptr = nullptr;
  double* partials = nullptr;
  unsigned int* counter = nullptr;
  int reverse = 0;  // walk tiles and row groups backwards (L2 "snake" order, see krylov.cu)
  Epi epi;
};

template <typename T, bool NORM>
__global__ void __launch_bounds__(kStreamThreads, 2)
k_combine_tma(CombineTmaArgs a) {
  using V = typename Vec<T>::type;
  constexpr int VN = Vec<T>::N;
  constexpr int TILE = kConsumerThreads * VN;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  T* stages = reinterpret_cast<T*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kStages * kGroup * TILE * sizeof(T));
  uint64_t* empty = full + kStages;
  T* coef = reinterpret_cast<T*>(empty + kStages);  // [ngb*8 + 8]: basis rows, then the vector group
  __shared__ double red_smem[32];
  __shared__ T oscale[2];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nbasis = a.src.n0 + a.src.n1;
  const int ngb = (nbasis + kGroup - 1) / kGroup;   // basis groups
  const int ngroups = ngb + (a.nvec > 0 ? 1 : 0);   // + one group of vector terms (nvec <= 8)
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      tma::mbar_init(full + s, 1);
      tma::mbar_init(empty + s, kConsumerWarps);
    }
    tma::fence_barrier_init();
  }
  __syncthreads();
  tma::griddep_launch_dependents();

  const ColumnRange cr = block_columns<T>(a.n, TILE);
  const int reverse = a.reverse;
  double ss = 0.0;

  if (warp == kConsumerWarps) {
    if (lane == 0) {
      int it = 0;
      bool waited = false;
      for (int tt = 0; tt < cr.ntiles; ++tt) {
        const int t = reverse ? cr.ntiles - 1 - tt : tt;
        const long long tc0 = cr.c0 + (long long)t * TILE;
        const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
        for (int gg = 0; gg < ngroups; ++gg, ++it) {
          if (gg < ngb) {
            stage_rows<T, TILE>(stages, full, empty, it, a.src, reverse ? ngb - 1 - gg : gg, nbasis, tc0, len);
            continue;
          }
          if (!waited) {
            tma::griddep_wait();
            waited = true;
          }
          const uint32_t bytes = (uint32_t)len * sizeof(T);
          const int s = it % kStages;
          tma::mbar_wait(empty + s, ((it / kStages) & 1) ^ 1);
          tma::mbar_arrive_expect_tx(full + s, bytes * a.nvec);
          T* dst = stages + (size_t)s * kGroup * TILE;
          for (int r = 0; r < a.nvec; ++r)
            tma::bulk_g2s(dst + (size_t)r * TILE, static_cast<const T*>(a.vec[r].ptr) + tc0, bytes, full + s);
        }
      }
    }
  } else {
    const int tid = threadIdx.x;  // 0..255: one 16-byte vector of every staged row
    // coefficients and scalars come from the predecessor's epilogue: wait for it first
    tma::griddep_wait();
    if (tid == 0) {
      oscale[0] = a.out_mul_ptr ? static_cast<T>(*a.out_mul_ptr) : T(1);
      oscale[1] = a.out_div_ptr ? static_cast<T>(*a.out_div_ptr) : T(1);
    }
    for (int j = tid; j < ngb * kGroup; j += kConsumerThreads)
      coef[j] = j >= nbasis ? T(0)
                            : (j < a.src.n0 ? static_cast<T>(a.sign0 * a.coef0[j])
                                            : static_cast<T>(a.sign1 * a.coef1[j - a.src.n0]));
    if (tid < kGroup) {
      T c = T(0);
      if (tid < a.nvec) {
        const VecTerm& v = a.vec[tid];
        c = static_cast<T>(v.coef_imm * (v.coef_ptr ? *v.coef_ptr : 1.0));
      }
      coef[ngb * kGroup + tid] = c;
    }
    tma::named_bar_sync(2, kConsumerThreads);
    int it = 0;
    for (int tt = 0; tt < cr.ntiles; ++tt) {
      const int t = reverse ? cr.ntiles - 1 - tt : tt;
      const long long tc0 = cr.c0 + (long long)t * TILE;
      const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
      const long long col = tc0 + (long long)tid * VN;
      const bool live = tid * VN < len;
      T acc[VN];
#pragma unroll
      for (int k = 0; k < VN; ++k) acc[k] = T(0);
      for (int gg = 0; gg < ngroups; ++gg, ++it) {
        const bool vec_group = gg >= ngb;
        const int g = vec_group ? gg : (reverse ? ngb - 1 - gg : gg);
        const int s = it % kStages;
        tma::mbar_wait(full + s, (it / kStages) & 1);
        const int rows_here = vec_group ? a.nvec : (nbasis - g * kGroup < kGroup ? nbasis - g * kGroup : kGroup);
        if (live)
          fma_group<T, TILE>(reinterpret_cast<const V*>(stages + (size_t)s * kGroup * TILE) + tid, coef + g * kGroup,
                             rows_here, acc);
        __syncwarp();
        if (lane == 0) tma::mbar_arrive(empty + s);
      }
      if (live) {
#pragma unroll
        for (int k = 0; k < VN; ++k) {
          acc[k] = acc[k] * oscale[0] / oscale[1];
          if (NORM && col + k < a.n) ss += static_cast<double>(acc[k] * acc[k]);
        }
        store_colvec(static_cast<T*>(a.out), col, a.n, acc);
        if (a.out2) store_colvec(static_cast<T*>(a.out2), col, a.n, acc);
      }
    }
  }
  if (!NORM) return;
  double bs = block_sum(ss, red_smem);
  if (threadIdx.x == 0) a.partials[blockIdx.x] = bs;
  if (!last_block_done(a.counter)) return;
  double s = 0.0;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) s += __ldcg(a.partials + b);
  s = block_sum(s, red_smem);
  if (threadIdx.x == 0) a.epi.red[0] = s;
  __syncthreads();
  run_epilogue<T>(a.epi);
}

// EPT consecutive elements of T as one 4/8/16-byte shared-memory load (conflict-free).
template <typename T, int EPT>
__device__ __forceinline__ void load_ept(const T* p, T (&e)[EPT]) {
  constexpr int BYTES = EPT * (int)sizeof(T);
  static_assert(BYTES == 4 || BYTES == 8 || BYTES == 16, "EPT * sizeof(T) must be 4, 8 or 16");
  if constexpr (BYTES == 4) {
    e[0] = p[0];
  } else if constexpr (BYTES == 8) {
    const uint2 v = *reinterpret_cast<const uint2*>(p);
    memcpy(e, &v, 8);
  } else {
    const uint4 v = *reinterpret_cast<const uint4*>(p);
    memcpy(e, &v, 16);
  }
}

// ---------------------------------------------------------------------------------------------
// Fused "combine, then dots against part of the rows" from ONE read of the basis:
//   out   = ( sum_v a_v vec_v + sum_{j < nres} c_j res_j + sum_k d_k str_k ) / div
//   red_j = < res_j , out >        for the resident rows j < nres
// Used for (i) the second Gram-Schmidt pass of the forward step (v' = v - Q h, h2 = Q^T v';
// arnoldi.py:88-92) and (ii) the adjoint's back-substitution fused with the next step's
// re-projection dots (lambda' = (...)/beta_minus, t = P lambda'; arnoldi.py:217-219 + 202-204).
//
// Data movement: 2-D tiled TMA through tensor maps — one instruction per [8 rows x TILE] box.
// The resident rows of a tile live in one of TWO shared-memory buffers, so the producer loads
// tile t+1 while the consumers run both sweeps over tile t (loads never drain); streamed-only
// rows go through a 3-slot ring; dense vector terms through a double-buffered slot.
// Sweep 1: thread <-> (column, row-split) accumulates the combination as boxes land.
// Sweep 2: warp w <-> row 8g+w takes the dots from shared memory and releases each box.
struct alignas(64) FusedArgs {
  CUtensorMap map_res;   // resident block: rows [0, nres) of one basis buffer (row extent = nres)
  CUtensorMap map_str0;  // streamed block 0 (rows [row_str0, row_str0 + nstr0))
  CUtensorMap map_str1;  // streamed block 1
  long long n = 0;
  void* out = nullptr;
  int nvec = 0;
  VecTerm vec[kMaxVecTerms];
  int nres = 0;
  const double* coef_res = nullptr;
  double sign_res = 1.0;
  int nstr0 = 0, row_str0 = 0;
  const double* coef_str0 = nullptr;
  double sign_str0 = 1.0;
  int nstr1 = 0, row_str1 = 0;
  const double* coef_str1 = nullptr;
  double sign_str1 = 1.0;
  const double* out_div_ptr = nullptr;
  double* partials = nullptr;
  unsigned int* counter = nullptr;
  int reverse = 0;
  int sr = kGroup;  // rows per streamed group (box rows of map_str0/1): 8, 16 or 32
  Epi epi;
};

struct FusedLayout {
  size_t res, ring, vec, part, xs, coef, elems;  // element offsets
  size_t bar_bytes, acc_bytes, total_bytes;
  int GR, GS0, GS1, GS;
};

template <typename T, int TILE>
__host__ __device__ inline FusedLayout fused_layout(int nres, int nstr0, int nstr1, int nvec, int sr) {
  constexpr int RS = kConsumerThreads * Vec<T>::N / TILE;  // row split of sweep 1
  FusedLayout L;
  L.GR = (nres + kGroup - 1) / kGroup;
  L.GS0 = (nstr0 + sr - 1) / sr;
  L.GS1 = (nstr1 + sr - 1) / sr;
  L.GS = L.GS0 + L.GS1;
  size_t o = 0;
  L.res = o;  o += (size_t)2 * L.GR * kGroup * TILE;
  L.ring = o; o += L.GS > 0 ? (size_t)kStages * sr * TILE : 0;
  L.vec = o;  o += (size_t)2 * (nvec > 0 ? nvec : 1) * TILE;
  L.part = o; o += (size_t)RS * TILE;
  L.xs = o;   o += (size_t)2 * TILE;
  L.coef = o; o += (size_t)L.GR * kGroup + (size_t)L.GS * sr + kGroup;
  L.elems = o;
  L.bar_bytes = (size_t)(4 * ((L.GR + 3) / 4) + 2 * kStages + 4) * 8;
  L.acc_bytes = (size_t)nres * 8;
  L.total_bytes = (L.elems * sizeof(T) + 127) / 128 * 128 + L.bar_bytes + L.acc_bytes + 64;
  return L;
}

// ---------------------------------------------------------------------------------------------
// red[j] = <row_j, x> for R <= 4 rows (the neighbouring-row dots of the symmetric loops, norms, single dots):
// two to five streams saturate nothing and need no staging -- every thread reads 16-byte vectors of x and of the
// rows straight into registers, one block-wide sum per row, last block reduces and runs the epilogue.  A launch
// is a few microseconds where the TMA pipeline's ramp costs more than the data.
struct FewRows {
  const void* row[4] = {nullptr, nullptr, nullptr, nullptr};
};

template <typename T, int R>
__global__ void __launch_bounds__(256)
k_dots_few(FewRows rows, const T* __restrict__ x, long long n, double* __restrict__ partials, unsigned int* counter,
           Epi epi) {
  using V = typename Vec<T>::type;
  constexpr int VN = Vec<T>::N;
  __shared__ double red_smem[32];
  tma::griddep_launch_dependents();
  tma::griddep_wait();  // x (and possibly the newest row) are the predecessor's output
  const long long ngroups = n / VN;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const V* xv = reinterpret_cast<const V*>(x);
  T acc[R];
#pragma unroll
  for (int r = 0; r < R; ++r) acc[r] = T(0);
  // U grid strides at a time: all (R + 1) * U loads are issued before the first FMA (the kernel is latency-bound)
  constexpr int U = R <= 2 ? 4 : 3;
  for (long long g0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; g0 < ngroups; g0 += U * stride) {
    V q[U][R], xx[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long g = g0 + u * stride;
      const long long gc = g < ngroups ? g : g0;  // clamped: a valid address, the product is masked below
#pragma unroll
      for (int r = 0; r < R; ++r) q[u][r] = ld_stream(static_cast<const V*>(rows.row[r]) + gc);
      xx[u] = ld_stream(xv + gc);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (g0 + u * stride < ngroups) {
        T b[VN];
        vec_unpack(xx[u], b);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          T a[VN];
          vec_unpack(q[u][r], a);
#pragma unroll
          for (int k = 0; k < VN; ++k) acc[r] = fma(a[k], b[k], acc[r]);
        }
      }
    }
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {  // scalar tail (n not a multiple of the vector width)
    for (long long c = ngroups * VN; c < n; ++c)
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r] = fma(static_cast<const T*>(rows.row[r])[c], x[c], acc[r]);
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const double bs = block_sum(static_cast<double>(acc[r]), red_smem);
    if (threadIdx.x == 0) partials[(size_t)r * gridDim.x + blockIdx.x] = bs;
  }
  if (!last_block_done(counter)) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp < R) {  // fixed-order reduction over blocks: warp r owns row r
    double s = 0.0;
    for (int b = lane; b < (int)gridDim.x; b += 32) s += __ldcg(partials + (size_t)warp * gridDim.x + b);
    s = warp_sum(s);
    if (lane == 0) epi.red[warp] = s;
  }
  __syncthreads();
  run_epilogue<T>(epi);
}

template <typename T, int TILE>
__global__ void __launch_bounds__(kStreamThreads, 2)
k_fused_tma(const __grid_constant__ FusedArgs a) {
  using V = typename Vec<T>::type;
  constexpr int VN = Vec<T>::N;
  constexpr int EPT = VN;                                // sweep 1: one 16-byte vector per thread and row
  constexpr int RS = kConsumerThreads * VN / TILE;       // ... rows r == h (mod RS) of every group
  constexpr int LV = TILE / (32 * VN);                   // vectors per lane (sweep 2)
  constexpr int GRMAX = 16;                              // sweep-2 lane accumulators (nres <= 128)
  static_assert(RS >= 1 && RS <= kGroup && TILE * RS == kConsumerThreads * VN, "bad tile");
  constexpr int BOXC = TILE > 256 ? 256 : TILE;                                // box columns (<= 256)
  constexpr int NBOX = TILE / BOXC;
  static_assert(LV >= 1, "tile too small");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int nres = a.nres, nvec = a.nvec;
  const int SR = a.sr;
  const FusedLayout L = fused_layout<T, TILE>(nres, a.nstr0, a.nstr1, nvec, SR);
  const int GR = L.GR, GS = L.GS, GS0 = L.GS0;
  T* base = reinterpret_cast<T*>(smem_raw);
  T* res_s = base + L.res;    // [2][GR*8][TILE]
  T* ring_s = base + L.ring;  // [3][SR][TILE]
  T* vec_s = base + L.vec;    // [2][nvec][TILE]
  T* part_s = base + L.part;  // [RS][TILE]
  T* xs = base + L.xs;        // [2][TILE]
  T* coef = base + L.coef;    // [GR*8][GS*SR][8]
  const int GQ = (GR + kBoxesPerBarrier - 1) / kBoxesPerBarrier;  // barrier groups of resident boxes
  uint64_t* res_full = reinterpret_cast<uint64_t*>(smem_raw + (L.elems * sizeof(T) + 127) / 128 * 128);  // [2][GQ]
  uint64_t* res_empty = res_full + 2 * GQ;      // [2][GQ]
  uint64_t* ring_full = res_empty + 2 * GQ;     // [3]
  uint64_t* ring_empty = ring_full + kStages;   // [3]
  uint64_t* x_full = ring_empty + kStages;      // [2]
  uint64_t* x_empty = x_full + 2;               // [2]
  double* acc_s = reinterpret_cast<double*>(x_empty + 2);  // [nres]
  __shared__ T oscale;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int g = 0; g < 2 * GQ; ++g) {
      tma::mbar_init(res_full + g, 1);
      tma::mbar_init(res_empty + g, kConsumerWarps);
    }
    for (int s = 0; s < kStages; ++s) {
      tma::mbar_init(ring_full + s, 1);
      tma::mbar_init(ring_empty + s, kConsumerWarps);
    }
    for (int s = 0; s < 2; ++s) {
      tma::mbar_init(x_full + s, 1);
      tma::mbar_init(x_empty + s, kConsumerWarps);
    }
    tma::fence_barrier_init();
  }
  for (int j = threadIdx.x; j < nres; j += blockDim.x) acc_s[j] = 0.0;
  __syncthreads();
  tma::griddep_launch_dependents();

  const ColumnRange cr = block_columns<T>(a.n, TILE);
  const int reverse = a.reverse;
  constexpr uint32_t kBoxBytes = (uint32_t)kGroup * TILE * sizeof(T);

  if (warp == kConsumerWarps) {
    if (lane == 0) {  // ---- producer ----
      tma::prefetch_tensormap(&a.map_res);
      if (GS > 0) {
        tma::prefetch_tensormap(&a.map_str0);
        tma::prefetch_tensormap(&a.map_str1);
      }
      bool waited = false;
      int its = 0;      // running index of streamed groups (ring position)
      int vec_next = 0; // next tile whose vector terms have to be issued
      auto issue_vec = [&](int tt) {
        if (nvec == 0) return;
        const int t = reverse ? cr.ntiles - 1 - tt : tt;
        const long long tc0 = cr.c0 + (long long)t * TILE;
        const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
        const uint32_t bytes = (uint32_t)len * sizeof(T);
        const int b = tt & 1;
        tma::mbar_wait(x_empty + b, ((tt >> 1) & 1) ^ 1);
        tma::mbar_arrive_expect_tx(x_full + b, bytes * nvec);
        for (int v = 0; v < nvec; ++v)
          tma::bulk_g2s(vec_s + ((size_t)b * nvec + v) * TILE, static_cast<const T*>(a.vec[v].ptr) + tc0, bytes,
                        x_full + b);
      };
      for (int tt = 0; tt < cr.ntiles; ++tt) {
        const int t = reverse ? cr.ntiles - 1 - tt : tt;
        const int tc0 = (int)(cr.c0 + (long long)t * TILE);
        const int b = tt & 1;
        const uint32_t ph = (tt >> 1) & 1;
        if (waited && vec_next <= tt) issue_vec(vec_next++);
        for (int qq = 0; qq < GQ; ++qq) {  // kBoxesPerBarrier boxes per mbarrier
          const int q = reverse ? GQ - 1 - qq : qq;
          const int g_lo = q * kBoxesPerBarrier;
          const int nb = GR - g_lo < kBoxesPerBarrier ? GR - g_lo : kBoxesPerBarrier;
          tma::mbar_wait(res_empty + b * GQ + q, ph ^ 1);  // sweep 2 of tile tt-2 released these boxes
          tma::mbar_arrive_expect_tx(res_full + b * GQ + q, kBoxBytes * nb);
          for (int gi = 0; gi < nb; ++gi) {
            const int g = g_lo + gi;
            T* dst = res_s + ((size_t)b * GR + g) * kGroup * TILE;
#pragma unroll
            for (int bx = 0; bx < NBOX; ++bx)
              tma::tensor_g2s_2d(dst + (size_t)bx * kGroup * BOXC, &a.map_res, tc0 + bx * BOXC, g * kGroup,
                                 res_full + b * GQ + q);
          }
        }
        if (!waited && (tt == 1 || cr.ntiles == 1 || GS > 0)) {
          // the resident rows of the first two tiles were prefetched; everything else may be the
          // predecessor's output and has to wait for it
          tma::griddep_wait();
          waited = true;
          issue_vec(vec_next++);
          if (tt == 1) issue_vec(vec_next++);
        }
        for (int gs = 0; gs < GS; ++gs, ++its) {
          const int s = its % kStages;
          tma::mbar_wait(ring_empty + s, ((its / kStages) & 1) ^ 1);
          tma::mbar_arrive_expect_tx(ring_full + s, (uint32_t)SR * TILE * sizeof(T));
          T* dst = ring_s + (size_t)s * SR * TILE;
          const bool first = gs < GS0;
          const void* map = first ? &a.map_str0 : &a.map_str1;
          const int row = first ? a.row_str0 + gs * SR : a.row_str1 + (gs - GS0) * SR;
#pragma unroll
          for (int bx = 0; bx < NBOX; ++bx)
            tma::tensor_g2s_2d(dst + (size_t)bx * SR * BOXC, map, tc0 + bx * BOXC, row, ring_full + s);
        }
      }
    }
  } else {
    const int tid = threadIdx.x;
    const int c = (tid % (TILE / VN)) * VN;  // first column of this thread inside the tile
    const int h = tid / (TILE / VN);         // row-split index: this thread takes rows r == h (mod RS)
    tma::griddep_wait();  // coefficients / scalars come from the predecessor's epilogue
    if (tid == 0) oscale = a.out_div_ptr ? static_cast<T>(*a.out_div_ptr) : T(1);
    for (int j = tid; j < GR * kGroup; j += kConsumerThreads)
      coef[j] = j < nres ? static_cast<T>(a.sign_res * a.coef_res[j]) : T(0);
    for (int j = tid; j < GS * SR; j += kConsumerThreads) {
      T cv = T(0);
      if (j < GS0 * SR) {
        if (j < a.nstr0) cv = static_cast<T>(a.sign_str0 * a.coef_str0[j]);
      } else if (j - GS0 * SR < a.nstr1) {
        cv = static_cast<T>(a.sign_str1 * a.coef_str1[j - GS0 * SR]);
      }
      coef[GR * kGroup + j] = cv;
    }
    if (tid < kGroup) {
      T cv = T(0);
      if (tid < nvec) {
        const VecTerm& v = a.vec[tid];
        cv = static_cast<T>(v.coef_imm * (v.coef_ptr ? *v.coef_ptr : 1.0));
      }
      coef[GR * kGroup + GS * SR + tid] = cv;
    }
    tma::named_bar_sync(2, kConsumerThreads);
    const T* cvec = coef + GR * kGroup + GS * SR;
    int its = 0;
    // sweep-2 partial dots stay in registers across tiles (one per group: row 8g + warp) and are
    // reduced across lanes once, after the last tile
    T lane_acc[GRMAX];
#pragma unroll
    for (int g = 0; g < GRMAX; ++g) lane_acc[g] = T(0);
    for (int tt = 0; tt < cr.ntiles; ++tt) {
      const int t = reverse ? cr.ntiles - 1 - tt : tt;
      const long long tc0 = cr.c0 + (long long)t * TILE;
      const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
      const int b = tt & 1;
      const uint32_t ph = (tt >> 1) & 1;
      // ---- sweep 1: thread <-> (one 16-byte vector of columns, rows r == h mod RS of every group) ----
      T acc[EPT];
#pragma unroll
      for (int k = 0; k < EPT; ++k) acc[k] = T(0);
      if (nvec > 0) {
        tma::mbar_wait(x_full + b, ph);
        if (h == 0 && c < len) {
          for (int v = 0; v < nvec; ++v) {
            T e[EPT];
            load_ept<T, EPT>(vec_s + ((size_t)b * nvec + v) * TILE + c, e);
#pragma unroll
            for (int k = 0; k < EPT; ++k) acc[k] = fma(cvec[v], e[k], acc[k]);
          }
        }
        __syncwarp();
        if (lane == 0) tma::mbar_arrive(x_empty + b);
      }
      // element (row r, column cc) of a [8][TILE] slot built from NBOX boxes of [8][BOXC]
      const int boff = (c / BOXC) * kGroup * BOXC + (c % BOXC);
      for (int qq = 0; qq < GQ; ++qq) {
        const int q = reverse ? GQ - 1 - qq : qq;
        const int g_lo = q * kBoxesPerBarrier;
        const int nb = GR - g_lo < kBoxesPerBarrier ? GR - g_lo : kBoxesPerBarrier;
        tma::mbar_wait(res_full + b * GQ + q, ph);
        for (int gi = 0; gi < nb; ++gi) {
          const int g = g_lo + gi;
          const T* st = res_s + ((size_t)b * GR + g) * kGroup * TILE + boff;
          const T* cf = coef + g * kGroup;
#pragma unroll
          for (int r = 0; r < kGroup / RS; ++r) {
            const int rr = r * RS + h;
            T e[EPT];
            load_ept<T, EPT>(st + (size_t)rr * BOXC, e);
#pragma unroll
            for (int k = 0; k < EPT; ++k) acc[k] = fma(cf[rr], e[k], acc[k]);
          }
        }
      }
      for (int gs = 0; gs < GS; ++gs, ++its) {
        const int s = its % kStages;
        tma::mbar_wait(ring_full + s, (its / kStages) & 1);
        const T* st = ring_s + (size_t)s * SR * TILE + (c / BOXC) * SR * BOXC + (c % BOXC);
        const T* cf = coef + GR * kGroup + gs * SR;
#pragma unroll 4
        for (int r = 0; r < SR / RS; ++r) {
          const int rr = r * RS + h;
          T e[EPT];
          load_ept<T, EPT>(st + (size_t)rr * BOXC, e);
#pragma unroll
          for (int k = 0; k < EPT; ++k) acc[k] = fma(cf[rr], e[k], acc[k]);
        }
        __syncwarp();
        if (lane == 0) tma::mbar_arrive(ring_empty + s);
      }
      if (RS > 1) {  // combine the row-split partial sums
#pragma unroll
        for (int k = 0; k < EPT; ++k) part_s[(size_t)h * TILE + c + k] = acc[k];
        tma::named_bar_sync(1, kConsumerThreads);
        if (h == 0) {
#pragma unroll
          for (int k = 0; k < EPT; ++k) {
            T sacc = T(0);
#pragma unroll
            for (int hh = 0; hh < RS; ++hh) sacc += part_s[(size_t)hh * TILE + c + k];
            acc[k] = sacc;
          }
        }
      }
      T* xcur = xs + (size_t)b * TILE;
      if (h == 0) {
        T val[EPT];
        bool all_ok = true;
#pragma unroll
        for (int k = 0; k < EPT; ++k) {
          const bool ok = c + k < len && tc0 + c + k < a.n;
          val[k] = ok ? acc[k] / oscale : T(0);
          all_ok = all_ok && ok;
        }
        *reinterpret_cast<V*>(xcur + c) = vec_pack(val);
        if (all_ok) {
          *reinterpret_cast<V*>(static_cast<T*>(a.out) + tc0 + c) = vec_pack(val);
        } else {
#pragma unroll
          for (int k = 0; k < EPT; ++k)
            if (c + k < len && tc0 + c + k < a.n) static_cast<T*>(a.out)[tc0 + c + k] = val[k];
        }
      }
      tma::named_bar_sync(1, kConsumerThreads);
      // ---- sweep 2: red[8g + w] += <row, out tile>; boxes released in the order they get refilled ----
      V xv[LV];
#pragma unroll
      for (int u = 0; u < LV; ++u) xv[u] = reinterpret_cast<const V*>(xcur)[lane + 32 * u];
#pragma unroll
      for (int qq = 0; qq < GRMAX / kBoxesPerBarrier; ++qq) {
        if (qq >= GQ) break;  // (unrolled for static register indexing; skip the unused copies)
        const int q = reverse ? GQ - 1 - qq : qq;
        const int g_lo = q * kBoxesPerBarrier;
        // all shared-memory loads of the (up to four) boxes first, then the FMAs
        V qv[kBoxesPerBarrier][LV];
#pragma unroll
        for (int gi = 0; gi < kBoxesPerBarrier; ++gi) {
          const int g = g_lo + gi;
          const bool on = g < GR && g * kGroup + warp < nres;
          const T* slot = res_s + ((size_t)b * GR + (on ? g : g_lo)) * kGroup * TILE;
#pragma unroll
          for (int u = 0; u < LV; ++u) {
            const int cc = (lane + 32 * u) * VN;  // column inside the tile
            qv[gi][u] = *reinterpret_cast<const V*>(slot + (cc / BOXC) * kGroup * BOXC + warp * BOXC + (cc % BOXC));
          }
        }
#pragma unroll
        for (int gi = 0; gi < kBoxesPerBarrier; ++gi) {
          const int g = g_lo + gi;
          if (g < GR && g * kGroup + warp < nres) {
            T p = T(0);
#pragma unroll
            for (int u = 0; u < LV; ++u) {
              T qq4[VN], xx[VN];
              vec_unpack(qv[gi][u], qq4);
              vec_unpack(xv[u], xx);
#pragma unroll
              for (int k = 0; k < VN; ++k) p = fma(qq4[k], xx[k], p);
            }
            lane_acc[qq * kBoxesPerBarrier + gi] += p;
          }
        }
        __syncwarp();
        if (lane == 0) tma::mbar_arrive(res_empty + b * GQ + q);
      }
    }
    // one cross-lane reduction per row for the whole block
#pragma unroll
    for (int qq = 0; qq < GRMAX / kBoxesPerBarrier; ++qq) {
      if (qq >= GQ) break;
      const int q = reverse ? GQ - 1 - qq : qq;
      double d[kBoxesPerBarrier];
#pragma unroll
      for (int gi = 0; gi < kBoxesPerBarrier; ++gi) d[gi] = static_cast<double>(lane_acc[qq * kBoxesPerBarrier + gi]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int gi = 0; gi < kBoxesPerBarrier; ++gi) d[gi] += __shfl_xor_sync(0xffffffffu, d[gi], o);
      }
      if (lane == 0) {
#pragma unroll
        for (int gi = 0; gi < kBoxesPerBarrier; ++gi) {
          const int j = (q * kBoxesPerBarrier + gi) * kGroup + warp;
          if (j < nres) acc_s[j] = d[gi];
        }
      }
    }
  }
  __syncthreads();
  for (int j = threadIdx.x; j < nres; j += blockDim.x) a.partials[(size_t)j * gridDim.x + blockIdx.x] = acc_s[j];
  if (!last_block_done(a.counter)) return;
  reduce_partials_and_epilogue<T>(nres, a.partials, a.epi);
}

}  // namespace bl
