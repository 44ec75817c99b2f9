// One Krylov step's worth of basis streaming in ONE launch, for up to kStepBatch independent runs (sm_100a).
//
// Per step and after the operator call, the symmetric loops of the forward (arnoldi.py:87-98) and of the adjoint
// (arnoldi.py:201-219) are
//
//   phase 0   red0[j] = <few_j, x0>                     two or three neighbouring basis rows      (k_dots_few)
//   phase 1   out1 = (sum_k a_k vec_k) / div ; red1[j] = <row_j, out1>  over the active rows      (k_xdots_tma)
//   phase 2   out2 = out1 + sum_j c_j row_j  (+ ||out2||^2)             over the active rows      (k_combine_tma)
//
// with a grid-wide reduction between the phases whose result (Gram-Schmidt coefficients) the next phase needs.
// Phases 1 and 2 run the same device code as k_xdots_tma and k_combine_tma: phase 1 of a run is step::xdots_run,
// the body of k_xdots_tma (defined below), and phase 2 folds the staged groups in with fma_group and writes out2
// with store_colvec, as k_combine_tma does.  As separate launches every reduction costs a kernel boundary (ramp,
// last-block pass, drain, launch: 8 us against 2-60 us of streaming), and a run is a chain of 800 of them.  Here
// the phases run in one cooperative grid: blocks meet at a counter in L2, every block (few values) or block j
// (value j, many values) reduces the per-block partials in a fixed order, and EVERY block runs the epilogue on
// identical numbers (its global writes are redundant and identical).  The TMA producer thread takes no part in the
// barriers: while the consumers wait it fills the 96 KB ring with the next phase's rows.
//
// Measured (block 0's time stamps, bl_step_trace_*), an in-kernel reduction costs ~6 us -- no less than a kernel
// boundary with programmatic dependent launch.  What pays is the BATCH: the lockstep drivers
// (bl_arnoldi_{forward,adjoint}_batch: Hutchinson probes, initial conditions) hand the step of up to kStepBatch runs
// to one launch; each phase loops over the runs, and ONE barrier per phase serves all of them, so a run's share
// of every fixed cost is divided by the batch size.
//
// Each block owns the same contiguous column range in all phases; thread t of the 256 consumers owns column
// vector t of every tile, so phase 2 reads back what the same thread wrote in phase 1 (program order, no
// fence), and phase 2 walks the tiles in the opposite direction (it starts on the rows phase 1 read last).
//
// Phase S (optional, StepOp): the OPERATOR CALL of the step rides in the same launch when the operand is stored as
// SELL-32 (sparse.cu) -- x0 = A x (forward: q = x / len is written on the way, x0 = A q) for every run.  A block
// computes the rows of its own column range: its slices' column indices are one contiguous range of `col`, which
// the producer streams through the ring (bulk copies of 8 KB); the consumer warps read them from shared memory, gather
// x from L2 and load the values alongside -- no dependent HBM round trip per slice, and the operand is read once for
// all runs of the batch.  A step is then ONE launch with three grid-wide reductions instead of two launches
// with four kernel boundaries.
#pragma once

#include "stream_kernels.cuh"

namespace bl {

constexpr int kFewMax = 4;
constexpr int kXTerms = 10;
constexpr int kStepBatch = 4;
constexpr int kFewSlots = kFewMax * kConsumerWarps + 8;  // per-run scratch of phase 0: warp partials, then block values

struct StepOp {  // the step's operator call, shared by the runs of a launch (phase S)
  const int64_t* slice_ptr = nullptr;  // nullptr: the operator ran as its own launch
  const int32_t* col = nullptr;
  const void* val = nullptr;
  long long nslices = 0, nrows = 0;
  long long n_pad = 0;  // norm: op_q is written up to n_pad entries (zero padding beyond nrows)
  int norm = 0;         // forward step: q = op_x / *op_len (true division, arnoldi.py:80-81), few_x = A q
  int wait_first = 0;   // the operand's values may be the predecessor's output: dependency wait before the first copy
};

struct StepArgs {
  long long n = 0;
  // ---- phase S (StepOp): few_x = A op_x ----
  const void* op_x = nullptr;
  void* op_q = nullptr;
  const double* op_len = nullptr;
  // ---- phase 0 ----
  int few_n = 0;
  const void* few_row[kFewMax] = {nullptr, nullptr, nullptr, nullptr};
  const void* few_x = nullptr;
  Epi epi0;
  // ---- phase 1 ----
  RowSource src1;
  int nrows1 = 0;
  void* out1 = nullptr;
  int nvec = 0;
  VecTerm vec[kXTerms];
  const double* out_div_ptr = nullptr;
  Epi epi1;
  // ---- phase 2 ----
  RowSource src2;
  int nrows2 = 0;
  const double* coef2 = nullptr;  // coefficient of row j: sign2 * coef2[j]
  double sign2 = 1.0;
  void* out2 = nullptr;
  int norm = 0;  // ||out2||^2 -> epi2 (run by the last block to leave)
  Epi epi2;
  // ---- reductions (per run) ----
  double* partials = nullptr;       // [rows][gridDim.x]: phase 1
  double* partials0 = nullptr;      // [kFewMax][gridDim.x]: phase 0 -- an area of its own: a block that is fast through a
                                    // short phase 1 must not overwrite shares a slow block is still adding up
  double* red_g = nullptr;          // [rows] reduced values of the distributed path
  double* partials_norm = nullptr;  // [gridDim.x]
  int wait_row = 1 << 30;  // rows >= wait_row of src1 are the predecessor kernel's output: the producer
                           // executes griddepcontrol.wait before it copies them
};

struct StepBatch {
  int count = 1;
  int reverse = 0;                      // direction of phase 1; phase 2 walks the other way
  int trace_slot = -1;                  // >= 0: block 0 writes its time stamps to g_step_trace[trace_slot]
  int acc_stride = 0, coef_stride = 0;  // per-run shared-memory strides (doubles / elements)
  unsigned int* bar = nullptr;          // arrival counter of the in-kernel barriers (0 between launches)
  unsigned int* exit_counter = nullptr;
  StepOp op;
  StepArgs a[kStepBatch];
};

// Optional time stamps of block 0 (bl_step_trace_*): 8 stamps per launch -- globaltimer at entry, then SM clocks
// after the dependency wait, phase 0's loads, phase 0's reduction, phase 1's stream, phase 1's reduction, phase 2, exit.
constexpr int kTraceStamps = 8;
constexpr int kTraceLaunches = 2048;
__device__ unsigned long long g_step_trace[kTraceStamps * kTraceLaunches];

#if defined(BL_STEP_DEBUG) || defined(BL_STEP_CYCLES)
// Debugging (-DBL_STEP_DEBUG): the FIRST non-finite value a k_step_tma launch meets, where it met it.
__device__ unsigned long long g_step_dbg[16];
__device__ __forceinline__ void dbg_record(int code, int p, int step_i, long long a, double v0, double v1) {
  if (atomicCAS(&g_step_dbg[0], 0ull, (unsigned long long)code) == 0ull) {
    g_step_dbg[1] = blockIdx.x;
    g_step_dbg[2] = threadIdx.x;
    g_step_dbg[3] = (unsigned long long)p;
    g_step_dbg[4] = (unsigned long long)step_i;
    g_step_dbg[5] = (unsigned long long)a;
    g_step_dbg[6] = (unsigned long long)__double_as_longlong(v0);
    g_step_dbg[7] = (unsigned long long)__double_as_longlong(v1);
    unsigned int smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    g_step_dbg[8] = smid;
    __threadfence();
  }
}
#ifdef BL_STEP_DEBUG
#define BL_DBG(cond, code, p, i, a, v0, v1) \
  do {                                      \
    if (cond) dbg_record(code, p, i, a, v0, v1); \
  } while (0)
#else
#define BL_DBG(cond, code, p, i, a, v0, v1) \
  do {                                      \
  } while (0)
#endif
template <typename X>
__device__ __forceinline__ bool dbg_bad(X v) { return !(fabs((double)v) < 1e30); }
// cycle counters of block 0 / warp 0 / lane 0 inside phase S: g_step_dbg[9 + k] accumulates section k
#define BL_CYC_DECL long long cyc_t0 = clock64(), cyc_acc[6] = {0, 0, 0, 0, 0, 0};
#define BL_CYC(k)                          \
  do {                                     \
    const long long cyc_t1 = clock64();    \
    cyc_acc[k] += cyc_t1 - cyc_t0;         \
    cyc_t0 = cyc_t1;                       \
  } while (0)
#define BL_CYC_FLUSH                                                                    \
  do {                                                                                  \
    if (blockIdx.x == 0 && warp == 0 && lane == 0)                                      \
      for (int k = 0; k < 6; ++k) atomicAdd(&g_step_dbg[9 + k], (unsigned long long)cyc_acc[k]); \
  } while (0)
#else
#define BL_CYC_DECL
#define BL_CYC(k) \
  do {            \
  } while (0)
#define BL_CYC_FLUSH \
  do {               \
  } while (0)
#define BL_DBG(cond, code, p, i, a, v0, v1) \
  do {                                      \
  } while (0)
#endif

namespace step {

__device__ __forceinline__ void stamp(int slot, int k, int tid) {
  if (slot >= 0 && blockIdx.x == 0 && tid == 0) {
    unsigned long long t;
    if (k == 0)
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    else
      t = (unsigned long long)clock64();
    g_step_trace[(size_t)slot * kTraceStamps + k] = t;
  }
}

__device__ __forceinline__ unsigned int ld_acquire(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

struct ConsumerSync {
  __device__ __forceinline__ void operator()() const { tma::named_bar_sync(1, kConsumerThreads); }
};

// Barrier among the consumer threads of all blocks (the producer warp is not involved).  The counter only
// grows inside a launch: block tickets of barrier k lie in [k G, (k+1) G), so the release value is the next
// multiple of G above the own ticket -- no generation flag, no reset, no host-side epoch.
__device__ __forceinline__ void grid_barrier(unsigned int* bar, int tid) {
  __threadfence();
  tma::named_bar_sync(1, kConsumerThreads);
  if (tid == 0) {
    const unsigned int G = gridDim.x;
    const unsigned int ticket = atomicAdd(bar, 1u);
    const unsigned int target = (ticket / G + 1u) * G;
    while ((int)(ld_acquire(bar) - target) < 0) {
    }
    __threadfence();
  }
  tma::named_bar_sync(1, kConsumerThreads);
}

// Sum over blocks of the per-block values of every run: run p has nvals(p) values at vals(p)[0..), reduced in
// place -- bit-identical in every block (fixed order).  Few values in total: one barrier, every block reduces all of
// them.  Many: block j reduces value j (j, j+G, ... over the runs' values laid end to end), a second barrier,
// everybody reads the results.  PHASE selects which count of StepArgs is meant (0: few_n, 1: nrows1).
template <int PHASE>
__device__ __forceinline__ int nvals_of(const StepArgs& a) {
  return PHASE == 0 ? a.few_n : a.nrows1;
}

template <int PHASE>
__device__ __forceinline__ void grid_reduce(const StepBatch& B, double* acc_base, int val_off, int tid) {
  const int G = gridDim.x, b = blockIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  int total = 0;
  for (int p = 0; p < B.count; ++p) {
    const int nv = nvals_of<PHASE>(B.a[p]);
    const double* src = acc_base + (size_t)p * B.acc_stride + val_off;
    double* part = PHASE == 0 ? B.a[p].partials0 : B.a[p].partials;
    for (int j = tid; j < nv; j += kConsumerThreads) __stcg(part + (size_t)j * G + b, src[j]);
    total += nv;
  }
  grid_barrier(B.bar, tid);
  const bool everyone = total * G <= 2560;
  for (int v = everyone ? warp : b + warp * G; v < total; v += everyone ? kConsumerWarps : kConsumerWarps * G) {
    int p = 0, j = v;
    while (j >= nvals_of<PHASE>(B.a[p])) j -= nvals_of<PHASE>(B.a[p++]);
    const double s = row_sum((PHASE == 0 ? B.a[p].partials0 : B.a[p].partials) + (size_t)j * G, G, lane);
    if (lane == 0) {
      if (everyone)
        acc_base[(size_t)p * B.acc_stride + val_off + j] = s;
      else
        __stcg(B.a[p].red_g + j, s);
    }
  }
  if (!everyone) {
    grid_barrier(B.bar, tid);
    for (int p = 0; p < B.count; ++p) {
      double* dst = acc_base + (size_t)p * B.acc_stride + val_off;
      for (int j = tid; j < nvals_of<PHASE>(B.a[p]); j += kConsumerThreads) dst[j] = __ldcg(B.a[p].red_g + j);
    }
  }
  tma::named_bar_sync(1, kConsumerThreads);
}

// ---- phase S: the operator call (SELL-32) ----
// Phase S uses the ring's memory as kOpStages FINE stages with barriers of their own: a stage is held by a consumer warp for a gather round trip (~2 us), so what stays
// in flight is (ring - held stages) -- with the three 32 KB stages of the basis stream that is one stage per block
// and the operand arrives at a fraction of the HBM rate.  Only the COLUMN INDICES go through the ring (the gathers
// depend on them); the values are plain coalesced loads issued together with the gathers, so they cost no round trip
// of their own and the ring holds twice as many slices.
constexpr int kOpStageBytes = 8192;
constexpr int kOpStages = kStages * kGroup * kConsumerThreads * 16 / kOpStageBytes;  // the ring: 96 KB = 12 fine stages
constexpr int kOpDepth = 8;                  // fine stages in use: what the producer keeps in flight
constexpr int kOpHold = kOpDepth / 2 - 1;    // stages a warp may span with the slices it has in flight
constexpr int kOpRing = kOpStages * kOpStageBytes / 4;  // slots in the ring
// The head of the stage in ring slot 0 is copied a second time behind the ring's end (into the x-tile buffer), so a
// chunk of up to kOpOverflow slots that starts in the last ring slot reads on linearly instead of wrapping.
constexpr int kOpOverflow = 16 * 32;
template <typename T>
__host__ __device__ constexpr int op_stage_slots() {
  return kOpStageBytes / 4;
}

template <typename T>
__device__ __forceinline__ T ld_stream(const T* p);
template <>
__device__ __forceinline__ float ld_stream<float>(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
template <>
__device__ __forceinline__ double ld_stream<double>(const double* p) {
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}

struct OpRange {
  long long s_lo = 0, s_hi = 0;  // slices of this block (rows of its column range)
  long long a0 = 0, a1 = 0;      // their slots in col / val
  int nstages = 0;
};

template <typename T>
__device__ __forceinline__ OpRange op_range(const StepOp& op, const ColumnRange& cr, long long n) {
  constexpr int VN = Vec<T>::N;
  OpRange o;
  if (op.slice_ptr == nullptr || cr.c0 >= cr.c1) return o;
  const long long n_v = (n + VN - 1) / VN * VN;
  o.s_lo = cr.c0 / 32;  // block ranges start on multiples of 32 columns
  o.s_hi = cr.c1 >= n_v ? op.nslices : cr.c1 / 32;  // the last block also owns the padding rows
  if (o.s_hi <= o.s_lo) return o;
  o.a0 = __ldg(op.slice_ptr + o.s_lo);
  o.a1 = __ldg(op.slice_ptr + o.s_hi);
  o.nstages = (int)((o.a1 - o.a0 + op_stage_slots<T>() - 1) / op_stage_slots<T>());
  return o;
}

// Loads of what a PREDECESSOR kernel wrote (x here, the vectors of phase 0) go through L2 (`ld.global.cg`): in a chain of
// programmatic dependent launches this kernel's lifetime overlaps the predecessor's, which is outside what `ld.global.nc`
// promises, and L1 buys nothing measurable here (gathers through `ld.global.nc` measured 5558 vs 5532 Krylov steps/s,
// within the noise).
// Consumer side: warp w takes the block's slices w, w + 8, ...; lane = row within the slice.  Summation order as in
// k_sell_spmv_multi (entries k of even / odd position in two accumulators, added at the end): bit-identical results.
// U slices of the warp are in flight together (their W x P gathers each are issued before the first FMA): with 16
// consumer warps per SM the gathers' round trip, not the operand stream, bounds the phase.  A warp holds at most
// kOpHold + 1 fine stages (lo .. hi): the slices of a group lie 8 slices apart; groups that span more fall back to one
// slice at a time (whose chunks release the stages behind them as they go).
template <typename T, int P, bool NORM, int W, int U>
__device__ __forceinline__ void op_phase(const StepBatch& B, const OpRange& o, const unsigned char* stages_raw,
                                         uint64_t* full, uint64_t* empty, int warp, int lane) {
  constexpr int SLOTS = op_stage_slots<T>();
  static_assert(W * 32 <= kOpOverflow && W * 32 <= SLOTS, "a chunk crosses at most one stage boundary");
  const StepOp& op = B.op;
  const T* x[P];
  T inv[P], dlen[P];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    x[p] = static_cast<const T*>(B.a[p].op_x);
    dlen[p] = NORM ? static_cast<T>(__ldcg(B.a[p].op_len)) : T(1);
    inv[p] = T(1) / dlen[p];
  }
  const T* valp = static_cast<const T*>(op.val) + o.a0 + lane;  // this lane's values of the block's slots
  const int* colp = reinterpret_cast<const int*>(stages_raw) + lane;
  constexpr int ring_slots = kOpDepth * SLOTS;
  int lo = 0, hi = -1;  // stages [lo, hi] of the operand stream are held by this warp
  int hi_ring = -1, lo_ring = 0, hi_par = 0;
  auto need = [&](int st) {
    while (hi < st) {
      ++hi;
      if (++hi_ring == kOpDepth) {
        hi_ring = 0;
        hi_par ^= hi > 0;
      }
      tma::mbar_wait(full + hi_ring, hi_par);
    }
  };
  auto done_below = [&](int st) {
    while (lo < st) {
      if (hi < lo) need(lo);  // every warp passes every stage
      __syncwarp();
      if (lane == 0) tma::mbar_arrive(empty + lo_ring);
      ++lo;
      lo_ring = lo_ring + 1 == kOpDepth ? 0 : lo_ring + 1;
    }
  };
  const long long first = o.s_lo + warp;
  const int nmine = o.s_hi > first ? (int)((o.s_hi - first + kConsumerWarps - 1) / kConsumerWarps) : 0;
  BL_CYC_DECL
  for (int base = 0; base < nmine; base += 32) {
    // lane l fetches the slot range of the warp's (base + l)-th slice (relative to the block's first slot: 32 bits)
    int sp0 = 0, sp1 = 0;
    if (base + lane < nmine) {
      const long long sl = first + (long long)(base + lane) * kConsumerWarps;
      sp0 = (int)(__ldg(op.slice_ptr + sl) - o.a0);
      sp1 = (int)(__ldg(op.slice_ptr + sl + 1) - o.a0);
    }
    const int cnt = nmine - base < 32 ? nmine - base : 32;
    int i = 0;
    while (i < cnt) {
      // ---- a group of up to U slices whose slots span at most kOpHold + 1 stages ----
      int rel[U], width[U];  // first slot of slice u (relative to the block's), entries per row
      long long r[U];
      int nu = 0, wmax = 0, head_st = 0;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        rel[u] = width[u] = 0;
        r[u] = 0;
        if (i + u < cnt) {
          const int a = __shfl_sync(0xffffffffu, sp0, (i + u) & 31), b = __shfl_sync(0xffffffffu, sp1, (i + u) & 31);
          const int last = b - 32 > a ? b - 32 : a;  // last slot row of the slice
          if (u == 0) head_st = a / SLOTS;
          if (u == 0 || (nu == u && last / SLOTS - head_st <= kOpHold)) {
            rel[u] = a;
            width[u] = (b - a) / 32;
            r[u] = (first + (long long)(base + i + u) * kConsumerWarps) * 32 + lane;
            wmax = width[u] > wmax ? width[u] : wmax;
            nu = u + 1;
          }
        }
      }
      T xr[U][P], acc0[U][P], acc1[U][P];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int p = 0; p < P; ++p) {
          xr[u][p] = NORM && u < nu && r[u] < op.nrows ? __ldcg(x[p] + r[u]) : T(0);
          acc0[u][p] = acc1[u][p] = T(0);
        }
      BL_CYC(0);  // group set-up (shuffles, row loads issued)
      for (int k0 = 0; k0 < wmax; k0 += W) {
        int rows[U];
        {  // stages below the first slot row that is still needed are finished with; wait for the last one of the round
          int low = -1, last = -1;
#pragma unroll
          for (int u = U - 1; u >= 0; --u) {
            rows[u] = width[u] - k0 < W ? width[u] - k0 : W;
            if (rows[u] > 0) {
              low = (rel[u] + k0 * 32) / SLOTS;
              const int e = (rel[u] + (k0 + rows[u] - 1) * 32) / SLOTS;
              last = e > last ? e : last;
            }
          }
          if (low >= 0) done_below(low);
          need(last);
        }
        BL_CYC(1);  // ring: release + wait
        int c[U][W];
        T v[U][W];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int s = rel[u] + k0 * 32;          // first slot of the chunk
          const int* cs = colp + s % ring_slots;   // linear in the ring (+ overflow copy behind its end)
          const T* vs = valp + s;
#pragma unroll
          for (int j = 0; j < W; ++j) {
            c[u][j] = 0;  // padding gathers x[0] with value 0
            v[u][j] = T(0);
            if (j < rows[u]) {
              c[u][j] = cs[j * 32];
              v[u][j] = ld_stream(vs + j * 32);
            }
          }
        }
        T g[U][W][P];
#ifdef BL_STEP_DEBUG
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int j = 0; j < W; ++j) {
            BL_DBG(c[u][j] < 0 || c[u][j] >= op.nrows, 1, u, B.a[0].epi0.i, c[u][j], (double)(rel[u] + k0 * 32), (double)j);
            if (c[u][j] < 0 || c[u][j] >= op.nrows) c[u][j] = 0;
            BL_DBG(dbg_bad(v[u][j]), 3, u, B.a[0].epi0.i, rel[u] + k0 * 32 + j * 32, (double)v[u][j], 0.0);
          }
#endif
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int j = 0; j < W; ++j)
#pragma unroll
            for (int p = 0; p < P; ++p) {  // through L2 (see the note above)
              g[u][j][p] = __ldcg(x[p] + c[u][j]);
              BL_DBG(dbg_bad(g[u][j][p]), 2, p, B.a[p].epi0.i, c[u][j], (double)g[u][j][p], (double)inv[p]);
            }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int j = 0; j < W; ++j)
#pragma unroll
            for (int p = 0; p < P; ++p) {
              const T gv = NORM ? g[u][j][p] * inv[p] : g[u][j][p];
              if (j & 1)
                acc1[u][p] = fma(v[u][j], gv, acc1[u][p]);
              else
                acc0[u][p] = fma(v[u][j], gv, acc0[u][p]);
            }
        BL_CYC(2);  // loads + FMAs of the round
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int p = 0; p < P; ++p) {
          BL_DBG(u < nu && r[u] < op.nrows && dbg_bad(acc0[u][p] + acc1[u][p]), 4, p, B.a[p].epi0.i, r[u], (double)acc0[u][p], (double)inv[p]);
          if (u < nu && r[u] < op.nrows) static_cast<T*>(const_cast<void*>(B.a[p].few_x))[r[u]] = acc0[u][p] + acc1[u][p];
          if (NORM && u < nu && r[u] < op.n_pad)
            static_cast<T*>(B.a[p].op_q)[r[u]] = r[u] < op.nrows ? xr[u][p] * T(1) / dlen[p] : T(0);
        }
      i += nu;
      BL_CYC(3);  // stores of the group
    }
  }
  done_below(o.nstages);  // every warp passes every stage of the operand stream
  BL_CYC(4);
  BL_CYC_FLUSH;
}

template <typename T, bool NORM>
__device__ __forceinline__ void op_phase_dispatch(const StepBatch& B, const OpRange& o, const unsigned char* stages_raw,
                                                  uint64_t* full, uint64_t* empty, int warp, int lane) {
  // slots per chunk (W, even) and slices in flight (U) by run count: what the register budget of the kernel carries
  constexpr bool F = sizeof(T) == 4;
  switch (B.count) {
    case 1: op_phase<T, 1, NORM, F ? 12 : 6, 2>(B, o, stages_raw, full, empty, warp, lane); break;
    case 2: op_phase<T, 2, NORM, 6, F ? 2 : 1>(B, o, stages_raw, full, empty, warp, lane); break;
    case 3: op_phase<T, 3, NORM, 4, F ? 2 : 1>(B, o, stages_raw, full, empty, warp, lane); break;
    default: op_phase<T, 4, NORM, 4, F ? 2 : 1>(B, o, stages_raw, full, empty, warp, lane); break;
  }
}

// One run's lane sums of <few_j, x0> over the block's tiles, TU tiles per round: the TU x (FN + 1) vector loads of a round
// are issued before the first FMA.  (One tile per round left a block with 4 runs x 13 tiles = 52 dependent L2 round trips
// in phase 0: 20-29 us of a launch whose phase 0 moves 64 MB.)
template <typename T, int TILE, int FN, int TU>
__device__ __forceinline__ void few_dots_run(const StepArgs& a, const ColumnRange& cr, long long n, int tid, T (&facc)[kFewMax]) {
  using V = typename Vec<T>::type;
  constexpr int VN = Vec<T>::N;
  const T* x0 = static_cast<const T*>(a.few_x);
  for (int t0 = 0; t0 < cr.ntiles; t0 += TU) {
    V xv[TU], qv[TU][FN];
    bool ok[TU];
#pragma unroll
    for (int u = 0; u < TU; ++u) {
      const long long c = cr.c0 + (long long)(t0 + u) * TILE + (long long)tid * VN;
      // whole vectors only (basis rows are zero-padded up to ld, x0 is not: the vector that straddles n goes below)
      ok[u] = t0 + u < cr.ntiles && c < cr.c1 && c + VN <= n;
      const long long cc = ok[u] ? c : cr.c0;
      xv[u] = __ldcg(reinterpret_cast<const V*>(x0 + cc));  // through L2 (op_phase's note)
#pragma unroll
      for (int r = 0; r < FN; ++r) qv[u][r] = __ldcg(reinterpret_cast<const V*>(static_cast<const T*>(a.few_row[r]) + cc));
    }
#pragma unroll
    for (int u = 0; u < TU; ++u) {
      if (ok[u]) {
        T xx[VN];
        vec_unpack(xv[u], xx);
#pragma unroll
        for (int r = 0; r < FN; ++r) {
          T q[VN];
          vec_unpack(qv[u][r], q);
#pragma unroll
          for (int k = 0; k < VN; ++k) facc[r] = fma(q[k], xx[k], facc[r]);
        }
      }
    }
  }
  // the vector that straddles n (at most one thread of one block)
  for (int tt = 0; tt < cr.ntiles; ++tt) {
    const long long c = cr.c0 + (long long)tt * TILE + (long long)tid * VN;
    if (c < cr.c1 && c < n && c + VN > n) {
#pragma unroll
      for (int r = 0; r < FN; ++r)
        for (int k = 0; c + k < n; ++k) facc[r] = fma(static_cast<const T*>(a.few_row[r])[c + k], __ldcg(x0 + c + k), facc[r]);
    }
  }
}

// Phase 0, block-local part: this block's share of <few_j, x0> for every run, left in the run's scratch area
// (acc_s + p * acc_stride + kFewMax * kConsumerWarps + j).
template <typename T, int TILE, typename Sync>
__device__ __forceinline__ void few_dots_local(const StepBatch& B, const ColumnRange& cr, long long n, double* acc_s,
                                         int tid, int warp, int lane, Sync csync) {
  const int P = B.count;
  for (int p = 0; p < P; ++p) {
    const StepArgs& a = B.a[p];
    if (a.few_n <= 0) continue;
    T facc[kFewMax];
#pragma unroll
    for (int r = 0; r < kFewMax; ++r) facc[r] = T(0);
    switch (a.few_n) {
      case 1: few_dots_run<T, TILE, 1, 4>(a, cr, n, tid, facc); break;
      case 2: few_dots_run<T, TILE, 2, 4>(a, cr, n, tid, facc); break;
      case 3: few_dots_run<T, TILE, 3, 3>(a, cr, n, tid, facc); break;
      default: few_dots_run<T, TILE, 4, 2>(a, cr, n, tid, facc); break;
    }
    double* scratch = acc_s + (size_t)p * B.acc_stride;
#pragma unroll
    for (int r = 0; r < kFewMax; ++r) {
      if (r < a.few_n) {
        const double w = warp_sum(static_cast<double>(facc[r]));
        if (lane == 0) scratch[r * kConsumerWarps + warp] = w;
      }
    }
  }
  csync();
  for (int p = 0; p < P; ++p) {
    double* scratch = acc_s + (size_t)p * B.acc_stride;
    if (tid < B.a[p].few_n) {
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < kConsumerWarps; ++w) s += scratch[tid * kConsumerWarps + w];
      BL_DBG(dbg_bad(s), 5, p, B.a[p].epi0.i, tid, s, 0.0);
      scratch[kFewMax * kConsumerWarps + tid] = s;  // this block's value of row tid
    }
  }
  csync();
}

// Phase 1 of one run, consumer side: out1 = (sum of the terms) / div, written to out1 and to the x tile, and
// acc[j] += <row j of src1, out1> over the block's tiles.  Thread t holds column vector t of every term, loaded a
// tile ahead; the rows come through the ring from the producer.  `it` (ring position) and `xt` (x-tile buffer) run
// on across runs.  IN_STEP: inside k_step_tma, where blocks of the same launch wrote the coefficients, so they are
// read through L2, and where the debug hooks record; p is the run's index there.
template <typename T, int TILE, bool IN_STEP>
__device__ __forceinline__ void xdots_run(const StepArgs& a, const ColumnRange& cr, int reverse, const T* stages,
                                          T* xs, uint64_t* full, uint64_t* empty, int& it, int& xt, double* acc_p,
                                          int p) {
  using V = typename Vec<T>::type;
  constexpr int VN = Vec<T>::N;
  constexpr int XV = TILE / (32 * VN);  // x vectors per lane
  static_assert(TILE == kConsumerThreads * VN, "one 16-byte column vector per consumer thread");
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long n = a.n;
  const int nrows1 = a.nrows1;
  const int ngroups1 = (nrows1 + kGroup - 1) / kGroup;
  T cv[kXTerms];
#pragma unroll
  for (int v = 0; v < kXTerms; ++v) {
    const double* cp = a.vec[v].coef_ptr;
    cv[v] = v < a.nvec ? static_cast<T>(a.vec[v].coef_imm * (cp ? (IN_STEP ? __ldcg(cp) : *cp) : 1.0)) : T(0);
  }
  const T oscale = a.out_div_ptr ? static_cast<T>(IN_STEP ? __ldcg(a.out_div_ptr) : *a.out_div_ptr) : T(1);
#ifdef BL_STEP_DEBUG
#pragma unroll
  for (int v = 0; v < kXTerms; ++v) BL_DBG(IN_STEP && tid == 0 && dbg_bad(cv[v]), 7, p, a.epi0.i, v, (double)cv[v], (double)oscale);
  BL_DBG(IN_STEP && tid == 0 && (dbg_bad(oscale) || oscale == T(0)), 7, p, a.epi0.i, 99, (double)oscale, 0.0);
#endif
  V term[kXTerms];
  auto load_terms = [&](int tt) {
    const int t = reverse ? cr.ntiles - 1 - tt : tt;
    const long long c = cr.c0 + (long long)t * TILE + (long long)tid * VN;
    const bool live = tt < cr.ntiles && c < cr.c1;
#pragma unroll
    for (int v = 0; v < kXTerms; ++v)
      term[v] = load_colvec(static_cast<const T*>(a.vec[v].ptr), c, n, live && v < a.nvec);
  };
  load_terms(0);
  for (int tt = 0; tt < cr.ntiles; ++tt, ++xt) {
    const int t = reverse ? cr.ntiles - 1 - tt : tt;
    const long long tc0 = cr.c0 + (long long)t * TILE;
    const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
    const bool live = tid * VN < len;
    T* x = xs + (size_t)(xt & 1) * TILE;
    {  // ---- build this thread's vector of the x tile ----
      T acc[VN];
#pragma unroll
      for (int k = 0; k < VN; ++k) acc[k] = T(0);
#pragma unroll
      for (int v = 0; v < kXTerms; ++v) {
        if (v < a.nvec) {
          T e[VN];
          vec_unpack(term[v], e);
#pragma unroll
          for (int k = 0; k < VN; ++k) {
            BL_DBG(IN_STEP && dbg_bad(e[k]), 8, p, a.epi0.i, v * 100000000ll + tc0 + tid * VN + k, (double)e[k], (double)cv[v]);
            acc[k] = fma(cv[v], e[k], acc[k]);
          }
        }
      }
      const long long c = tc0 + (long long)tid * VN;
#pragma unroll
      for (int k = 0; k < VN; ++k) acc[k] = live && c + k < n ? acc[k] / oscale : T(0);
      reinterpret_cast<V*>(x)[tid] = vec_pack(acc);
      if (live) store_colvec(static_cast<T*>(a.out1), c, n, acc);
    }
    load_terms(tt + 1);  // in flight while this tile's rows are consumed (in place: own columns only)
    tma::named_bar_sync(1, kConsumerThreads);
    V xr[XV];
#pragma unroll
    for (int u = 0; u < XV; ++u) xr[u] = reinterpret_cast<const V*>(x)[lane + 32 * u];
    for (int gg = 0; gg < ngroups1; ++gg, ++it) {
      const int g = reverse ? ngroups1 - 1 - gg : gg;
      const int s = it % kStages;
      tma::mbar_wait(full + s, (it / kStages) & 1);
      const int j = g * kGroup + warp;
      if (j < nrows1) {
        const V* row = reinterpret_cast<const V*>(stages + ((size_t)s * kGroup + warp) * TILE);
        T a0 = T(0), a1 = T(0);
#pragma unroll
        for (int u = 0; u < XV; ++u) {
          if ((lane + 32 * u) * VN < len) {
            T q[VN], xx[VN];
            vec_unpack(row[lane + 32 * u], q);
            vec_unpack(xr[u], xx);
#ifdef BL_STEP_DEBUG
#pragma unroll
            for (int k = 0; k < VN; ++k) {
              BL_DBG(IN_STEP && dbg_bad(q[k]), 9, p, a.epi0.i, j * 100000000ll + tc0 + (lane + 32 * u) * VN + k, (double)q[k], (double)s);
              BL_DBG(IN_STEP && dbg_bad(xx[k]), 10, p, a.epi0.i, j * 100000000ll + tc0 + (lane + 32 * u) * VN + k, (double)xx[k], 0.0);
            }
#endif
#pragma unroll
            for (int k = 0; k < VN; ++k) {
              if (u & 1)
                a1 = fma(q[k], xx[k], a1);
              else
                a0 = fma(q[k], xx[k], a0);
            }
          }
        }
        __syncwarp();
        if (lane == 0) tma::mbar_arrive(empty + s);
        double sacc = warp_sum(static_cast<double>(a0) + static_cast<double>(a1));
        if (lane == 0) acc_p[j] += sacc;  // row j is always handled by this warp: no race
      } else {
        __syncwarp();
        if (lane == 0) tma::mbar_arrive(empty + s);
      }
    }
  }
}

}  // namespace step

// ---------------------------------------------------------------------------------------------
// Phase 1 of a step as a launch of its own: out1 = (sum_k a_k vec_k) / div  AND  red[j] = <row_j, out1>.  k_dots_tma
// whose x tile is BUILT by the consumers instead of loaded.  The symmetric Krylov loops combine a handful of vectors
// (<= kXTerms: the iterate, two to five neighbouring basis rows, r, z, two rows of Lambda) and then need the dots of
// the result with every active basis row -- no row is used twice, so nothing has to stay resident (k_fused_tma's
// double-buffered [rows x 128] tiles and its two-sweep hand-over per tile go away) and the rows stream through the
// same 4 KB x 8 x 3 ring as in k_dots_tma.  Only the phase-1 fields of `a` are read; a.partials is the [nrows1][grid]
// area of the block shares.
template <typename T, int TILE>
__global__ void __launch_bounds__(kStreamThreads, 2)
k_xdots_tma(const __grid_constant__ StepArgs a, unsigned int* counter, int reverse) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  T* stages = reinterpret_cast<T*>(smem_raw);                       // [kStages][kGroup][TILE]
  T* xs = stages + (size_t)kStages * kGroup * TILE;                 // [2][TILE]
  uint64_t* full = reinterpret_cast<uint64_t*>(xs + 2 * TILE);
  uint64_t* empty = full + kStages;
  double* acc_s = reinterpret_cast<double*>(empty + kStages + 2);   // [nrows1]

  const int nrows = a.nrows1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      tma::mbar_init(full + s, 1);
      tma::mbar_init(empty + s, kConsumerWarps);
    }
    tma::fence_barrier_init();
  }
  for (int j = threadIdx.x; j < nrows; j += blockDim.x) acc_s[j] = 0.0;
  __syncthreads();
  tma::griddep_launch_dependents();

  const ColumnRange cr = block_columns<T>(a.n, TILE);
  const int ngroups = (nrows + kGroup - 1) / kGroup;

  if (warp == kConsumerWarps) {
    if (lane == 0) {  // ---- producer: basis rows only (older than the predecessor: no griddepcontrol.wait) ----
      const int total = cr.ntiles * ngroups;
      for (int it = 0; it < total; ++it) {
        const int tt = it / ngroups, gg = it - tt * ngroups;
        const int t = reverse ? cr.ntiles - 1 - tt : tt;
        const long long tc0 = cr.c0 + (long long)t * TILE;
        const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
        stage_rows<T, TILE>(stages, full, empty, it, a.src1, reverse ? ngroups - 1 - gg : gg, nrows, tc0, len);
      }
    }
  } else {
    tma::griddep_wait();  // the terms and their coefficients are the predecessor's output
    int it = 0, xt = 0;
    step::xdots_run<T, TILE, false>(a, cr, reverse, stages, xs, full, empty, it, xt, acc_s, 0);
  }
  __syncthreads();
  for (int j = threadIdx.x; j < nrows; j += blockDim.x) a.partials[(size_t)j * gridDim.x + blockIdx.x] = acc_s[j];
  if (!last_block_done(counter)) return;
  reduce_partials_and_epilogue<T>(nrows, a.partials, a.epi1);
}

template <typename T, int TILE>
__global__ void __launch_bounds__(kStreamThreads, 2)
k_step_tma(const __grid_constant__ StepBatch B) {
  using V = typename Vec<T>::type;
  constexpr int VN = Vec<T>::N;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  T* stages = reinterpret_cast<T*>(smem_raw);                       // [kStages][kGroup][TILE]
  T* xs = stages + (size_t)kStages * kGroup * TILE;                 // [2][TILE]
  uint64_t* full = reinterpret_cast<uint64_t*>(xs + 2 * TILE);
  uint64_t* empty = full + kStages;
  uint64_t* gate = empty + kStages;  // phase S done in this block: the ring is free, its rows of the newest basis vector are written
  // Phase S's barriers have memory of their OWN.  (They used to live in the x-tile buffer, which phase 1 overwrites
  // long after the last arrival -- with a block of another lane's kernel on the same SM the x tile then came back with
  // barrier words in it: 12 vectors of NaN exactly where the 24 barriers had been.  PTX wants mbarrier.inval before
  // an mbarrier's memory is put to another use; here the memory simply is not reused.)
  uint64_t* op_full = empty + kStages + 2;
  uint64_t* op_empty = op_full + step::kOpStages;
  double* acc_s = reinterpret_cast<double*>(op_empty + step::kOpStages);   // [count][acc_stride]: dots of phase 1, in place reduced
  T* coef_s = reinterpret_cast<T*>(acc_s + (size_t)B.count * B.acc_stride);  // [count][coef_stride]
  __shared__ double red_smem[32];

  const int P = B.count;
  const bool with_op = B.op.slice_ptr != nullptr;
  const int dir1 = B.reverse, dir2 = B.reverse ^ 1;
  const long long n = B.a[0].n;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      tma::mbar_init(full + s, 1);
      tma::mbar_init(empty + s, kConsumerWarps);
    }
    tma::mbar_init(gate, 1);
    if (B.op.slice_ptr != nullptr)
      for (int s = 0; s < step::kOpStages; ++s) {
        tma::mbar_init(op_full + s, 1);
        tma::mbar_init(op_empty + s, kConsumerWarps);
      }
    tma::fence_barrier_init();
  }
  for (int j = threadIdx.x; j < P * B.acc_stride; j += blockDim.x) acc_s[j] = 0.0;
  __syncthreads();
  // With the operator in the launch the successor may only start once every block has finished phase S: its
  // producer copies the basis rows written here before its own dependency wait (trigger after phase 0's barrier).
  if (!with_op) tma::griddep_launch_dependents();

  const ColumnRange cr = block_columns<T>(n, TILE);
  const step::OpRange orng = step::op_range<T>(B.op, cr, n);

  if (warp == kConsumerWarps) {
    if (lane == 0) {  // ---- producer: the rows of phase 1 of every run, then the rows of phase 2, one ring ----
      bool waited = false;
      bool gated = !with_op;  // with the operator in the launch the ring belongs to phase S first
      int it = 0;
      if (orng.nstages > 0) {  // ---- phase S: this block's slots of the operand, indices and values side by side ----
        constexpr int SLOTS = step::op_stage_slots<T>();
        if (B.op.wait_first) {
          tma::griddep_wait();
          waited = true;
        }
        for (int k = 0, s = 0, par = 1; k < orng.nstages; ++k) {
          const long long pos = orng.a0 + (long long)k * SLOTS;
          const uint32_t cnt = (uint32_t)((orng.a1 - pos) < SLOTS ? (orng.a1 - pos) : SLOTS);
          tma::mbar_wait(op_empty + s, par);
          const uint32_t over = s == 0 && k > 0 ? (cnt < (uint32_t)step::kOpOverflow ? cnt : (uint32_t)step::kOpOverflow) : 0u;
          tma::mbar_arrive_expect_tx(op_full + s, (cnt + over) * 4u);
          unsigned char* dst = smem_raw + (size_t)s * step::kOpStageBytes;
          tma::bulk_g2s(dst, B.op.col + pos, cnt * 4u, op_full + s);
          if (over)  // the ring's end reads on linearly
            tma::bulk_g2s(smem_raw + (size_t)step::kOpDepth * step::kOpStageBytes, B.op.col + pos, over * 4u, op_full + s);
          if (++s == step::kOpDepth) {
            s = 0;
            par ^= 1;
          }
        }
      }
      for (int phase = 1; phase <= 2; ++phase) {
        const int dir = phase == 1 ? dir1 : dir2;
        for (int pp = 0; pp < P; ++pp) {
          const int p = phase == 1 ? pp : P - 1 - pp;  // phase 2 starts with the run whose rows were read last (L2)
          const StepArgs& a = B.a[p];
          const RowSource& src = phase == 1 ? a.src1 : a.src2;
          const int nrows = phase == 1 ? a.nrows1 : a.nrows2;
          const int ngroups = (nrows + kGroup - 1) / kGroup;
          for (int tt = 0; tt < cr.ntiles; ++tt) {
            const int t = dir ? cr.ntiles - 1 - tt : tt;
            const long long tc0 = cr.c0 + (long long)t * TILE;
            const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
            for (int gg = 0; gg < ngroups; ++gg, ++it) {
              const int g = dir ? ngroups - 1 - gg : gg;
              const int rows_here = nrows - g * kGroup < kGroup ? nrows - g * kGroup : kGroup;
              if (!gated) {  // phase S is over in this block: the ring is free (and the newest row written)
                tma::mbar_wait(gate, 0);
                gated = true;
              }
              if (!waited && (phase == 2 || g * kGroup + rows_here > a.wait_row)) {
                tma::griddep_wait();
                waited = true;
              }
              stage_rows<T, TILE>(stages, full, empty, it, src, g, nrows, tc0, len);
            }
          }
        }
      }
    }
  } else {
    const int tid = threadIdx.x;  // 0..255: column vector tid of every tile
    step::stamp(B.trace_slot, 0, tid);
    tma::griddep_wait();          // everything below reads the predecessor's output
    step::ConsumerSync csync;
    step::stamp(B.trace_slot, 1, tid);

    // ================= phase S: x0 = A x, every run (the operator call of the step) =================
    if (with_op) {
      if (B.op.norm)
        step::op_phase_dispatch<T, true>(B, orng, smem_raw, op_full, op_empty, warp, lane);
      else
        step::op_phase_dispatch<T, false>(B, orng, smem_raw, op_full, op_empty, warp, lane);
      // the producer copies this block's columns of the rows written above (generic -> async proxy), the dots
      // below read them back
      asm volatile("fence.proxy.async;" ::: "memory");
      csync();
      if (tid == 0) tma::mbar_arrive(gate);
    }

    // ================= phase 0: dots of a few rows with x0, every run =================
    bool any_few = false;
    for (int p = 0; p < P; ++p) any_few = any_few || B.a[p].few_n > 0;
    if (any_few) {
      step::few_dots_local<T, TILE>(B, cr, n, acc_s, tid, warp, lane, csync);
      step::stamp(B.trace_slot, 2, tid);
      step::grid_reduce<0>(B, acc_s, kFewMax * kConsumerWarps, tid);
      for (int p = 0; p < P; ++p) {
        if (B.a[p].few_n <= 0) continue;
        BL_DBG(tid < B.a[p].few_n && dbg_bad(acc_s[(size_t)p * B.acc_stride + kFewMax * kConsumerWarps + tid]), 6, p,
               B.a[p].epi0.i, tid, acc_s[(size_t)p * B.acc_stride + kFewMax * kConsumerWarps + tid], 0.0);
        run_epilogue_impl<T>(B.a[p].epi0, acc_s + (size_t)p * B.acc_stride + kFewMax * kConsumerWarps, tid,
                             kConsumerThreads, csync);
      }
      __threadfence();  // the coefficients go through global memory (every block writes the same values)
      csync();
      for (int p = 0; p < P; ++p)
        if (tid < kFewSlots) acc_s[(size_t)p * B.acc_stride + tid] = 0.0;  // phase 1 accumulates into acc_s
      csync();
      step::stamp(B.trace_slot, 3, tid);
    }
    // every block is past phase S (phase 0's barrier)
    if (with_op) tma::griddep_launch_dependents();

    // ================= phase 1: out1 = (sum of terms) / div, red1[j] = <row_j, out1>, every run =================
    int it = 0, xt = 0;
    for (int p = 0; p < P; ++p)
      step::xdots_run<T, TILE, true>(B.a[p], cr, dir1, stages, xs, full, empty, it, xt, acc_s + (size_t)p * B.acc_stride, p);
    csync();
    step::stamp(B.trace_slot, 4, tid);
    step::grid_reduce<1>(B, acc_s, 0, tid);
    for (int p = 0; p < P; ++p) {
      BL_DBG(tid < B.a[p].nrows1 && dbg_bad(acc_s[(size_t)p * B.acc_stride + tid]), 11, p, B.a[p].epi0.i, tid,
             acc_s[(size_t)p * B.acc_stride + tid], 0.0);
      run_epilogue_impl<T>(B.a[p].epi1, acc_s + (size_t)p * B.acc_stride, tid, kConsumerThreads, csync);
    }
    __threadfence();
    csync();

    // ================= phase 2: out2 = out1 + sum_j c_j row_j (+ ||out2||^2), every run =================
    for (int p = 0; p < P; ++p) {
      const StepArgs& a = B.a[p];
      const int padded = (a.nrows2 + kGroup - 1) / kGroup * kGroup;
      T* cf = coef_s + (size_t)p * B.coef_stride;
      for (int j = tid; j < padded; j += kConsumerThreads)
        cf[j] = j < a.nrows2 ? static_cast<T>(a.sign2 * __ldcg(a.coef2 + j)) : T(0);
    }
    csync();
    step::stamp(B.trace_slot, 5, tid);
    for (int pp = 0; pp < P; ++pp) {
      const int p = P - 1 - pp;  // the producer's order
      const StepArgs& a = B.a[p];
      double ss = 0.0;
      const int nrows2 = a.nrows2;
      const int ngroups2 = (nrows2 + kGroup - 1) / kGroup;
      const T* coef_p = coef_s + (size_t)p * B.coef_stride;
      auto load_x = [&](int tt) {  // out1 as this very thread wrote it in phase 1
        const int t = dir2 ? cr.ntiles - 1 - tt : tt;
        const long long c = cr.c0 + (long long)t * TILE + (long long)tid * VN;
        return load_colvec(static_cast<const T*>(a.out1), c, n, tt < cr.ntiles && c < cr.c1);
      };
      V xnext = load_x(0);
      for (int tt = 0; tt < cr.ntiles; ++tt) {
        const int t = dir2 ? cr.ntiles - 1 - tt : tt;
        const long long tc0 = cr.c0 + (long long)t * TILE;
        const int len = (int)((cr.c1 - tc0) < TILE ? (cr.c1 - tc0) : TILE);
        const long long col = tc0 + (long long)tid * VN;
        const bool live = tid * VN < len;
        T acc[VN];
        vec_unpack(xnext, acc);
        xnext = load_x(tt + 1);
        for (int gg = 0; gg < ngroups2; ++gg, ++it) {
          const int g = dir2 ? ngroups2 - 1 - gg : gg;
          const int s = it % kStages;
          tma::mbar_wait(full + s, (it / kStages) & 1);
          const int rows_here = nrows2 - g * kGroup < kGroup ? nrows2 - g * kGroup : kGroup;
          if (live)
            fma_group<T, TILE>(reinterpret_cast<const V*>(stages + (size_t)s * kGroup * TILE) + tid, coef_p + g * kGroup,
                               rows_here, acc);
          __syncwarp();
          if (lane == 0) tma::mbar_arrive(empty + s);
        }
        if (live) {
          if (a.norm) {
#pragma unroll
            for (int k = 0; k < VN; ++k)
              if (col + k < n) ss += static_cast<double>(acc[k] * acc[k]);
          }
          store_colvec(static_cast<T*>(a.out2), col, n, acc);
        }
      }
      if (a.norm) {  // acc_s is free by now: warp sums of ||out2||^2, added up at the exit
        ss = warp_sum(ss);
        if (lane == 0) acc_s[(size_t)p * B.acc_stride + warp] = ss;
      }
    }
    step::stamp(B.trace_slot, 6, tid);
  }
  // ---- exit: the last block to leave re-arms the barrier counter and (norm) closes the reductions ----
  __syncthreads();
  if ((int)threadIdx.x < P && B.a[threadIdx.x].norm) {
    const double* w = acc_s + (size_t)threadIdx.x * B.acc_stride;
    double bs = 0.0;
#pragma unroll
    for (int k = 0; k < kConsumerWarps; ++k) bs += w[k];
    B.a[threadIdx.x].partials_norm[blockIdx.x] = bs;
  }
  step::stamp(B.trace_slot, 7, threadIdx.x);
  if (!last_block_done(B.exit_counter)) return;
  if (threadIdx.x == 0) *B.bar = 0u;
  for (int p = 0; p < P; ++p) {
    if (!B.a[p].norm) continue;
    double s = 0.0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) s += __ldcg(B.a[p].partials_norm + b);
    s = block_sum(s, red_smem);
    if (threadIdx.x == 0) B.a[p].epi2.red[0] = s;
    __syncthreads();
    run_epilogue<T>(B.a[p].epi2);
    __syncthreads();
  }
}

}  // namespace bl
