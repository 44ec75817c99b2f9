// Tensor-core (tcgen05 / TMEM) sweep of the matrix-free Gram operator, fp32 data.
//
// Reference behaviour replaced: the pairwise squared distance of
// /root/reference/src/matfree_extensions/util/gp_util.py:87-95 (Matern) and :168-176 (RBF),
//     s2_ij = max(0, |x_i|^2 + |x_j|^2 - 2 x_i.x_j),
// evaluated for a [128 x 256] tile of pairs by ONE group of `tcgen05.mma.kind::tf32` instructions.
//
// TF32 keeps 11 significand bits, the tolerance of this path is 1e-5, so every fp32 coordinate is
// split x = hi + lo (both exactly representable in TF32) and the contraction runs over the
// concatenated slots
//     A row i : [ hi(x) | lo(x) | hi(x) | 1     | 1      | 1      | 0.. ]
//     B row j : [ hi(y) | hi(y) | lo(y) | b_hi  | b_mid  | b_lo   | 0.. ]     b = -|y_j|^2 / 2 (exact 3-way split)
// so that the fp32 accumulator in TMEM holds  x.y - |y|^2/2  with an error of ~3 * 2^-24 |x||y| (the
// dropped lo*lo term and the last bit of lo) -- the level of an fp32 dot product.  The row term
// -|x_i|^2/2 is a per-thread constant of the epilogue (thread = row) and is folded into its first FMA,
// and the diagonal i == j is set to s2 = 0 exactly, as the fp32 evaluation of the reference's
// expression gives.  3d + 3 slots, padded to a multiple of 8 (one MMA consumes 8 TF32 slots):
// d = 9 -> 32 slots -> 4 MMAs of 128x256x8 per tile.
//
// Operands live in global memory in the canonical K-major no-swizzle core-matrix order
// ([16-byte slot chunk][point][4 floats]); a tile is a handful of contiguous 1-D TMA bulk copies and
// is consumed straight from shared memory by the tensor core.  Warp roles (one CTA per SM):
//   warp 0      TMA producer  (A tile once; B tile + v / q / x^T tile per stage)
//   warp 1      TMEM allocation + single-thread MMA issue, tcgen05.commit -> mbarriers
//   warps 2..9  epilogue: tcgen05.ld the accumulator (thread = row i, registers = columns j),
//               sqrt / exp on the MUFU, k_ij v_j accumulated per row.  Two accumulator buffers
//               (2 x 256 TMEM columns) let the MMA of tile t+1 run under the epilogue of tile t.
// The kernel is bound by the MUFU epilogue (rsqrt + ex2 per pair), not by the tensor pipe: the MMA
// group of a tile takes ~512 clocks, its epilogue ~4096.
#pragma once

#include "operators.cuh"
#include "tma_pipeline.cuh"

namespace bl {
namespace gramtc {

constexpr int kM = 128;          // rows per CTA  (UMMA M)
constexpr int kN = 256;          // columns per tile (UMMA N)
constexpr int kThreads = 320;    // 10 warps
constexpr int kEpiWarps = 8;
constexpr int kTmemCols = 512;   // two fp32 accumulators of kN columns
constexpr int kMaxSlots = 64;    // 3d + 3 <= 64  ->  d <= 20
constexpr int kXtRows = 20;      // rows of the transposed coordinate tile (adjoint sweep), >= d

__host__ __device__ inline int slots_for(int d) { return (3 * d + 3 + 7) / 8 * 8; }

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tma::smem_u32(slot_smem)),
               "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, no-swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, version 1):
// canonical layout ((8, m), 2) : ((16 B, SBO), LBO) -- LBO = distance between the two 16-byte slot
// chunks of one MMA, SBO = distance between groups of 8 rows.
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major
__host__ __device__ constexpr uint32_t instr_desc(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the mbarrier once every MMA issued so far by this thread has completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tma::smem_u32(bar))
               : "memory");
}
// 32 consecutive accumulator columns of this thread's TMEM lane (blocking)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      "tcgen05.wait::ld.sync.aligned;\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rsqf(float x) {
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---- operand packing ------------------------------------------------------------------------
// xs [n][dp] (scaled inputs), xx [n] (squared norms, same values as the ALU kernel uses)
//   -> opA / opB [slots/4][npad][4]   (points >= n are zero rows)
//   -> xt [kXtRows][npad]             (transposed fp32 coordinates for the adjoint epilogue)
// opB == nullptr: only the row operand and no xt (the test points of a cross-covariance sweep)
__global__ void k_gram_tc_pack(int64_t n, int64_t npad, int d, int dp, int slots, const float* __restrict__ xs,
                               const float* __restrict__ xx, float* __restrict__ opA, float* __restrict__ opB,
                               float* __restrict__ xt) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npad; i += (int64_t)gridDim.x * blockDim.x) {
    const bool live = i < n;
    float a[kMaxSlots], b[kMaxSlots];
#pragma unroll
    for (int s = 0; s < kMaxSlots; ++s) a[s] = b[s] = 0.f;
    if (live) {
      for (int k = 0; k < d; ++k) {
        const float x = xs[i * dp + k];
        const float hi = __uint_as_float(to_tf32(x));
        const float lo = __uint_as_float(to_tf32(x - hi));
        a[k] = hi, a[d + k] = lo, a[2 * d + k] = hi;
        b[k] = hi, b[d + k] = hi, b[2 * d + k] = lo;
      }
      const float h = -0.5f * xx[i];
      const float h0 = __uint_as_float(to_tf32(h));
      const float h1 = __uint_as_float(to_tf32(h - h0));
      const float h2 = __uint_as_float(to_tf32((h - h0) - h1));  // <= 2 bits left: exact
      a[3 * d] = 1.f, a[3 * d + 1] = 1.f, a[3 * d + 2] = 1.f;
      b[3 * d] = h0, b[3 * d + 1] = h1, b[3 * d + 2] = h2;
    }
    for (int c = 0; c < slots / 4; ++c) {
      float4 va, vb;
      va.x = a[4 * c], va.y = a[4 * c + 1], va.z = a[4 * c + 2], va.w = a[4 * c + 3];
      vb.x = b[4 * c], vb.y = b[4 * c + 1], vb.z = b[4 * c + 2], vb.w = b[4 * c + 3];
      reinterpret_cast<float4*>(opA)[(int64_t)c * npad + i] = va;
      if (opB) reinterpret_cast<float4*>(opB)[(int64_t)c * npad + i] = vb;
    }
    if (opB)
      for (int k = 0; k < kXtRows; ++k) xt[(int64_t)k * npad + i] = (live && k < d) ? xs[i * dp + k] : 0.f;
  }
}

// ---- shared-memory plan ---------------------------------------------------------------------
struct Plan {
  int ksteps;   // MMAs per tile (slots / 8)
  int stages;   // B-tile ring depth
  uint32_t a_bytes, b_bytes, aux_bytes, stage_bytes, bar_off, total;
};
// aux per stage: `aux_rows` rows of kN floats
__host__ __device__ inline Plan make_plan_rows(int slots, int aux_rows) {
  Plan p;
  p.ksteps = slots / 8;
  p.a_bytes = (uint32_t)slots * kM * 4;
  p.b_bytes = (uint32_t)slots * kN * 4;
  p.aux_bytes = (uint32_t)kN * 4 * aux_rows;
  p.stage_bytes = p.b_bytes + p.aux_bytes;
  const uint32_t budget = 220 * 1024;
  p.stages = 3;
  while (p.stages > 2 && p.a_bytes + p.stages * p.stage_bytes > budget) --p.stages;
  p.bar_off = p.a_bytes + p.stages * p.stage_bytes;
  p.total = p.bar_off + 256;
  if (p.total < 120 * 1024) p.total = 120 * 1024;  // one CTA per SM: each CTA owns all 512 TMEM columns
  return p;
}
// sweeps: v [kN] (+ q [kN] + x^T [kXtRows][kN] for the adjoint sweep)
__host__ __device__ inline Plan make_plan(int slots, bool adj) { return make_plan_rows(slots, adj ? 2 + kXtRows : 1); }
constexpr int kBatchMax = 16;  // vectors / (lambda, q) pairs per pass of the batched sweeps
__host__ __device__ inline Plan make_plan_batch(int slots) { return make_plan_rows(slots, kBatchMax + kXtRows); }
__host__ __device__ inline Plan make_plan_multi(int slots) { return make_plan_rows(slots, kBatchMax); }
struct VecPtrs {
  const float* p[kBatchMax];
};

// (unscaled) kernel values from the accumulator acc = x.y - |y|^2/2, two entries at a time.
//   KIND 0: Matern-3/2 (1+s) e^{-s}   KIND 1: Matern-1/2 e^{-s}   KIND 2: RBF e^{-s2/2}
// crow: per-row constant, (|x_i|^2 + eps) for the Matern kinds, (-|x_i|^2 / 2) for RBF.
struct Eval2 {
  float2 k;   // kernel value / sigma
  float2 e;   // e^{-s}  (Matern) or k (RBF)
  float2 ri;  // 1 / s   (Matern)
  bool pos0, pos1;  // s2 > 0 before the clamp (the clamp has zero derivative)   gp_util.py:92-95
};
template <int KIND>
__device__ __forceinline__ Eval2 kernel_from_acc(float2 acc, float2 crow) {
  Eval2 o;
  if (KIND == 2) {
    float2 a = __fadd2_rn(acc, crow);  // -s2/2
    o.pos0 = a.x < 0.f, o.pos1 = a.y < 0.f;
    a.x = fminf(a.x, 0.f), a.y = fminf(a.y, 0.f);  // clamp s2 at zero
    const float2 t = __fmul2_rn(a, make_float2(1.4426950408889634f, 1.4426950408889634f));
    o.k = make_float2(ex2f(t.x), ex2f(t.y));
    o.e = o.k;
    o.ri = make_float2(0.f, 0.f);
    return o;
  }
  const float eps = 1.1920928955078125e-07f;
  float2 t = __ffma2_rn(acc, make_float2(-2.f, -2.f), crow);  // s2 + eps
  o.pos0 = t.x > eps, o.pos1 = t.y > eps;
  t.x = fmaxf(t.x, eps), t.y = fmaxf(t.y, eps);  // max(s2, 0) + eps
  o.ri = make_float2(rsqf(t.x), rsqf(t.y));
  const float2 s = __fmul2_rn(t, o.ri);
  const float2 u = __fmul2_rn(s, make_float2(-1.4426950408889634f, -1.4426950408889634f));
  o.e = make_float2(ex2f(u.x), ex2f(u.y));
  o.k = KIND == 0 ? __ffma2_rn(s, o.e, o.e) : o.e;
  return o;
}
// d k / d s2 (divided by sigma), zero where the clamp is active
template <int KIND>
__device__ __forceinline__ float2 dkernel_from_eval(const Eval2& o) {
  float2 dk = __fmul2_rn(KIND == 2 ? o.k : o.e, make_float2(-0.5f, -0.5f));
  if (KIND == 1) dk = __fmul2_rn(dk, o.ri);
  dk.x = o.pos0 ? dk.x : 0.f;
  dk.y = o.pos1 ? dk.y : 0.f;
  return dk;
}

// ---- the pipeline shared by every sweep ---------------------------------------------------------
// One CTA per SM; grid = (row tiles of 128, column splits).  warp 0 = TMA producer, warp 1 = MMA issue,
// warps 2..9 = epilogue.  A stage of the ring holds the B operand tile (kN points) followed by the
// kernel-specific auxiliary rows (vectors, transposed coordinates); the accumulator is double-buffered in
// TMEM.  The kernels below differ in their auxiliary loader and in their epilogue only.
struct Pipe {
  Plan pl;
  uint8_t* smA;
  uint8_t* smS;
  uint64_t *full, *empty, *acc_full, *acc_empty, *a_full;  // see pipe_setup
  uint32_t tmem_base;
  int64_t i0, t0;  // first row of this CTA, first column tile of its split
  int ntiles;

  __device__ __forceinline__ uint8_t* stage(int s) const { return smS + (size_t)s * pl.stage_bytes; }
  __device__ __forceinline__ float* aux(int s) const { return reinterpret_cast<float*>(stage(s) + pl.b_bytes); }
};
struct Slot {  // ring stage / accumulator buffer and their mbarrier parities for tile `it`
  int s, b;
  uint32_t ph, bph;
};
__device__ __forceinline__ Slot slot_of(const Pipe& p, int it) {
  return Slot{it % p.pl.stages, it & 1, (uint32_t)(it / p.pl.stages) & 1u, (uint32_t)(it >> 1) & 1u};
}

// barriers, TMEM allocation, tile range; ends with a block-wide sync.  `full`: TMA -> MMA and epilogue;
// `empty`: MMA commit + 8 epilogue warps -> TMA; `acc_full`: MMA commit -> epilogue; `acc_empty`: 8 epilogue
// warps -> MMA; `a_full`: the A tile (loaded once).
__device__ __forceinline__ Pipe pipe_setup(uint8_t* smem, const Plan& pl, int64_t n) {
  Pipe p;
  p.pl = pl;
  p.smA = smem;
  p.smS = smem + pl.a_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + pl.bar_off);
  p.full = bars, p.empty = bars + 3, p.acc_full = bars + 6, p.acc_empty = bars + 8, p.a_full = bars + 10;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 11);
  p.i0 = (int64_t)blockIdx.x * kM;
  const int64_t tiles_total = (n + kN - 1) / kN;
  const int64_t per = (tiles_total + gridDim.y - 1) / gridDim.y;
  p.t0 = per * blockIdx.y;
  const int64_t t1 = p.t0 + per < tiles_total ? p.t0 + per : tiles_total;
  p.ntiles = p.t0 < t1 ? (int)(t1 - p.t0) : 0;
  if (threadIdx.x == 0) {
    for (int s = 0; s < pl.stages; ++s) {
      tma::mbar_init(p.full + s, 1);
      tma::mbar_init(p.empty + s, 1 + kEpiWarps);
    }
    for (int b = 0; b < 2; ++b) {
      tma::mbar_init(p.acc_full + b, 1);
      tma::mbar_init(p.acc_empty + b, kEpiWarps);
    }
    tma::mbar_init(p.a_full, 1);
    tma::fence_barrier_init();
  }
  if ((threadIdx.x >> 5) == 1) tmem_alloc(tmem_slot, kTmemCols);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  p.tmem_base = *tmem_slot;
  return p;
}
__device__ __forceinline__ void pipe_teardown(const Pipe& p) {
  fence_before_sync();
  __syncthreads();
  if ((threadIdx.x >> 5) == 1) {
    fence_after_sync();
    tmem_dealloc(p.tmem_base, kTmemCols);
  }
}

// A row of `kN` floats of a stage's auxiliary area filled from a global vector of `len` valid entries
// starting at column jt: whole 16-byte granules by TMA (`issue`), the ragged end and the zero padding by the
// producer warp (`fill`, generic stores that the arrive.expect_tx of lane 0 publishes).
struct RaggedRow {
  const float* src;  // element 0 of the vector
  int64_t len;       // entries that may be read (the rest of the tile is zero)
  __device__ __forceinline__ int granules(int64_t jt) const {
    const int64_t w = len - jt < kN ? len - jt : kN;
    return (int)(w > 0 ? w : 0) & ~3;
  }
  __device__ __forceinline__ void fill(float* dst, int64_t jt, int lane) const {
    for (int c = granules(jt) + lane; c < kN; c += 32) dst[c] = jt + c < len ? src[jt + c] : 0.f;
  }
  __device__ __forceinline__ uint32_t issue(float* dst, int64_t jt, uint64_t* bar) const {
    const uint32_t bytes = (uint32_t)granules(jt) * 4;
    if (bytes) tma::bulk_g2s(dst, src + jt, bytes, bar);
    return bytes;
  }
};

// warp 0.  Aux: `bool ragged(jt)`, `void fill(float* aux, jt, lane)`, `uint32_t bytes(jt)`,
// `void issue(float* aux, jt, bar)` for the auxiliary rows of one stage.  opA has `apad` points per slot
// chunk, opB `npad` (the same number unless the rows are another point set than the columns).
template <class Aux>
__device__ __forceinline__ void producer_warp(const Pipe& p, const float* __restrict__ opA, int64_t apad,
                                              const float* __restrict__ opB, int64_t npad, const Aux& aux) {
  const int lane = threadIdx.x & 31;
  if (lane == 0 && p.ntiles > 0) {
    tma::mbar_arrive_expect_tx(p.a_full, p.pl.a_bytes);
    for (int c = 0; c < 2 * p.pl.ksteps; ++c)
      tma::bulk_g2s(p.smA + (size_t)c * kM * 16, opA + ((int64_t)c * apad + p.i0) * 4, kM * 16, p.a_full);
  }
  for (int it = 0; it < p.ntiles; ++it) {
    const Slot sl = slot_of(p, it);
    tma::mbar_wait(p.empty + sl.s, sl.ph ^ 1u);
    const int64_t jt = (p.t0 + it) * kN;
    if (aux.ragged(jt)) {
      aux.fill(p.aux(sl.s), jt, lane);
      __syncwarp();
    }
    if (lane == 0) {
      tma::mbar_arrive_expect_tx(p.full + sl.s, p.pl.b_bytes + aux.bytes(jt));
      uint8_t* smB = p.stage(sl.s);
      for (int c = 0; c < 2 * p.pl.ksteps; ++c)
        tma::bulk_g2s(smB + (size_t)c * kN * 16, opB + ((int64_t)c * npad + jt) * 4, kN * 16, p.full + sl.s);
      aux.issue(p.aux(sl.s), jt, p.full + sl.s);
    }
  }
}

// warp 1: one group of `ksteps` TF32 MMAs (128 x 256 x 8 each) per tile, issued by lane 0
__device__ __forceinline__ void mma_warp(const Pipe& p) {
  const int lane = threadIdx.x & 31;
  const uint32_t idesc = instr_desc(kM, kN);
  if (p.ntiles > 0) tma::mbar_wait(p.a_full, 0);
  for (int it = 0; it < p.ntiles; ++it) {
    const Slot sl = slot_of(p, it);
    tma::mbar_wait(p.full + sl.s, sl.ph);
    tma::mbar_wait(p.acc_empty + sl.b, sl.bph ^ 1u);
    fence_after_sync();
    if (lane == 0) {
      const uint32_t sa = tma::smem_u32(p.smA), sb = tma::smem_u32(p.stage(sl.s));
      for (int k = 0; k < p.pl.ksteps; ++k) {
        const uint64_t da = smem_desc(sa + (uint32_t)k * 2 * kM * 16, kM * 16, 128);
        const uint64_t db = smem_desc(sb + (uint32_t)k * 2 * kN * 16, kN * 16, 128);
        mma_tf32(p.tmem_base + (uint32_t)sl.b * kN, da, db, idesc, k > 0 ? 1u : 0u);
      }
      mma_commit(p.empty + sl.s);
      mma_commit(p.acc_full + sl.b);
    }
    __syncwarp();
  }
}

// Epilogue warps 2..9: thread = row (TMEM lane `qd*32 + lane`), the two warpgroups split the kN columns.
struct EpiThread {
  int qd, half, row;
  bool live;
  float2 crow;        // per-row constant of kernel_from_acc
  uint32_t acc_diag;  // accumulator value that makes s2 exactly zero (the diagonal i == j)
};
template <int KIND>
__device__ __forceinline__ EpiThread epi_thread(const Pipe& p, int64_t n, const float* __restrict__ xx) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  EpiThread e;
  e.qd = warp & 3;            // TMEM lane quadrant this warp may access
  e.half = (warp - 2) >> 2;   // column half of the tile
  e.row = e.qd * 32 + lane;
  e.live = p.i0 + e.row < n;
  const float xxi = e.live ? xx[p.i0 + e.row] : 0.f;
  const float cr = KIND == 2 ? -0.5f * xxi : xxi + 1.1920928955078125e-07f;
  e.crow = make_float2(cr, cr);
  e.acc_diag = __float_as_uint(0.5f * xxi);
  return e;
}
__device__ __forceinline__ void epi_wait(const Pipe& p, const Slot& sl) {
  tma::mbar_wait(p.full + sl.s, sl.ph);
  tma::mbar_wait(p.acc_full + sl.b, sl.bph);
  fence_after_sync();
}
__device__ __forceinline__ void epi_release(const Pipe& p, const Slot& sl) {
  fence_before_sync();
  __syncwarp();
  if ((threadIdx.x & 31) == 0) {
    tma::mbar_arrive(p.acc_empty + sl.b);
    tma::mbar_arrive(p.empty + sl.s);
  }
}
// 32 accumulator columns (col0 ..) of this thread's row; on tiles that hold pairs with i == j the
// diagonal entry is replaced by the value that makes s2 exactly zero.  DIAG == false (rows and columns
// are different point sets): no replacement.
template <bool DIAG = true>
__device__ __forceinline__ void epi_load(const Pipe& p, const EpiThread& e, const Slot& sl, int it, int col0,
                                         uint32_t (&r)[32]) {
  tmem_ld32(p.tmem_base + ((uint32_t)(e.qd * 32) << 16) + (uint32_t)(sl.b * kN + col0), r);
  const int64_t jt = (p.t0 + it) * kN;
  if (DIAG && jt < p.i0 + kM && p.i0 < jt + kN) {
    const int jd = (int)(p.i0 + e.row - jt) - col0;  // column of this chunk with j == i (if any)
#pragma unroll
    for (int c = 0; c < 32; ++c) r[c] = c == jd ? e.acc_diag : r[c];
  }
}
// block-wide sums of the epilogue threads' `count` doubles -> gpart[cta][0..d) and gpart[cta][d] (slot `last`)
template <int D>
__device__ __forceinline__ void epi_reduce_grad(const double (&dacc)[D], double uacc, int d, double* __restrict__ gpart) {
  __shared__ double gred[kEpiWarps][kXtRows + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, ew = warp - 2;
  double t = warp_sum(uacc);
  if (lane == 0) gred[ew][D] = t;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    t = warp_sum(dacc[k]);
    if (lane == 0) gred[ew][k] = t;
  }
  tma::named_bar_sync(1, kEpiWarps * 32);
  if (warp == 2 && lane <= D) {
    double sacc = 0.0;
    for (int e = 0; e < kEpiWarps; ++e) sacc += gred[e][lane];
    const size_t blk = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
    if (lane == D)
      gpart[blk * (d + 1) + d] = sacc;
    else if (lane < d)
      gpart[blk * (d + 1) + lane] = sacc;
  }
}

// ---- auxiliary loaders --------------------------------------------------------------------------
// sweep: v [kN] (+ q [kN] + x^T [D][kN] for the adjoint sweep)
template <bool ADJ, int D>
struct SweepAux {
  RaggedRow v, q;
  const float* xt;
  int64_t npad;
  __device__ __forceinline__ bool ragged(int64_t jt) const { return v.granules(jt) < kN; }
  __device__ __forceinline__ void fill(float* aux, int64_t jt, int lane) const {
    v.fill(aux, jt, lane);
    if (ADJ) q.fill(aux + kN, jt, lane);
  }
  __device__ __forceinline__ uint32_t bytes(int64_t jt) const {
    return (uint32_t)v.granules(jt) * 4 * (ADJ ? 2 : 1) + (ADJ ? D * kN * 4 : 0);
  }
  __device__ __forceinline__ void issue(float* aux, int64_t jt, uint64_t* bar) const {
    v.issue(aux, jt, bar);
    if (ADJ) {
      q.issue(aux + kN, jt, bar);
      for (int k = 0; k < D; ++k) tma::bulk_g2s(aux + (size_t)(2 + k) * kN, xt + (int64_t)k * npad + jt, kN * 4, bar);
    }
  }
};
// batched sweeps: M rows (vectors, or the q rows of (lambda, q) pairs) [+ x^T [D][kN] after kBatchMax rows]
template <int D>
struct RowsAux {
  VecPtrs rows;
  int M;
  int64_t len;       // readable entries per row
  const float* xt;   // nullptr: no coordinate rows
  int64_t npad;
  __device__ __forceinline__ RaggedRow row(int m) const { return RaggedRow{rows.p[m], len}; }
  __device__ __forceinline__ bool ragged(int64_t jt) const { return row(0).granules(jt) < kN; }
  __device__ __forceinline__ void fill(float* aux, int64_t jt, int lane) const {
    for (int m = 0; m < M; ++m) row(m).fill(aux + (size_t)m * kN, jt, lane);
  }
  __device__ __forceinline__ uint32_t bytes(int64_t jt) const {
    return (uint32_t)row(0).granules(jt) * 4 * M + (xt ? D * kN * 4 : 0);
  }
  __device__ __forceinline__ void issue(float* aux, int64_t jt, uint64_t* bar) const {
    for (int m = 0; m < M; ++m) row(m).issue(aux + (size_t)m * kN, jt, bar);
    if (xt)
      for (int k = 0; k < D; ++k)
        tma::bulk_g2s(aux + (size_t)(kBatchMax + k) * kN, xt + (int64_t)k * npad + jt, kN * 4, bar);
  }
};

// ---- the sweeps -----------------------------------------------------------------------------------
//   ADJ == false: part[split][i] = sigma sum_{j in split} k_ij v_j
//   ADJ == true : the same with v = lam, plus per-CTA partial sums (layout of the ALU kernel)
//                 gpart[cta][d]  = sum lam_i q_j k_ij               (k includes sigma)
//                 gpart[cta][k]  = sum lam_i q_j dk_ij (x_ik - x_jk)^2,  k < d
// dbg != nullptr: CTA (dbg_bx, dbg_by) writes the raw accumulator (x.y - |y|^2/2) of its first tile to dbg[128][256].
// CROSS == true: the rows are another point set (a cross-covariance K(X*, X) v): m rows packed in opA with
// mpad points per slot chunk, xx = their squared norms, part[split][m]; the columns stay the n points of opB.
// Only the square sweep replaces the diagonal (it is exact only where the row and the column are one point).
template <int KIND, bool ADJ, int D, bool CROSS = false>
__global__ void __launch_bounds__(kThreads, 1)
k_gram_tc_sweep(int64_t n, int64_t npad, int d, int slots, const float* __restrict__ opA,
                const float* __restrict__ opB, const float* __restrict__ xt, const float* __restrict__ xx,
                const float* __restrict__ consts, const float* __restrict__ v, const float* __restrict__ q,
                float* __restrict__ part, double* __restrict__ gpart, float* __restrict__ dbg, int dbg_bx, int dbg_by,
                int64_t m, int64_t mpad) {
  static_assert(!(CROSS && ADJ), "the cross-covariance sweep has no adjoint");
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ double ycomb[kM];
  const int64_t rows = CROSS ? m : n;
  const Pipe p = pipe_setup(smem, make_plan(slots, ADJ), n);
  const int warp = threadIdx.x >> 5;
  if (warp == 0) {
    producer_warp(p, opA, CROSS ? mpad : npad, opB, npad, SweepAux<ADJ, D>{RaggedRow{v, n}, RaggedRow{q, n}, xt, npad});
  } else if (warp == 1) {
    mma_warp(p);
  } else {
    const EpiThread e = epi_thread<KIND>(p, rows, xx);
    double yacc = 0.0, uacc = 0.0, dacc[ADJ ? D : 1];
    float2 nxi[ADJ ? D : 1];  // (-x_ik, -x_ik)
#pragma unroll
    for (int k = 0; k < (ADJ ? D : 1); ++k) {
      const float x = ADJ ? xt[(int64_t)k * npad + p.i0 + e.row] : 0.f;
      nxi[k] = make_float2(-x, -x);
      dacc[k] = 0.0;
    }
    for (int it = 0; it < p.ntiles; ++it) {
      const Slot sl = slot_of(p, it);
      const float* smV = p.aux(sl.s);
      const float* smQ = smV + kN;
      const float* smX = smV + 2 * kN;
      epi_wait(p, sl);
      float2 y0 = make_float2(0.f, 0.f), y1 = y0, u0 = y0, u1 = y0, dl[ADJ ? D : 1];
#pragma unroll
      for (int k = 0; k < (ADJ ? D : 1); ++k) dl[k] = make_float2(0.f, 0.f);
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        const int col0 = e.half * 128 + cc * 32;
        uint32_t r[32];
        if (dbg != nullptr && it == 0 && (int)blockIdx.x == dbg_bx && (int)blockIdx.y == dbg_by) {
          tmem_ld32(p.tmem_base + ((uint32_t)(e.qd * 32) << 16) + (uint32_t)(sl.b * kN + col0), r);
#pragma unroll
          for (int c = 0; c < 32; ++c) dbg[(size_t)e.row * kN + col0 + c] = __uint_as_float(r[c]);
        }
        epi_load<!CROSS>(p, e, sl, it, col0, r);
#pragma unroll
        for (int pp = 0; pp < 8; ++pp) {
          const float4 v4 = *reinterpret_cast<const float4*>(smV + col0 + 4 * pp);
          const float2 a01 = make_float2(__uint_as_float(r[4 * pp]), __uint_as_float(r[4 * pp + 1]));
          const float2 a23 = make_float2(__uint_as_float(r[4 * pp + 2]), __uint_as_float(r[4 * pp + 3]));
          const Eval2 e01 = kernel_from_acc<KIND>(a01, e.crow), e23 = kernel_from_acc<KIND>(a23, e.crow);
          y0 = __ffma2_rn(e01.k, make_float2(v4.x, v4.y), y0);
          y1 = __ffma2_rn(e23.k, make_float2(v4.z, v4.w), y1);
          if (ADJ) {
            const float4 q4 = *reinterpret_cast<const float4*>(smQ + col0 + 4 * pp);
            const float2 q01 = make_float2(q4.x, q4.y), q23 = make_float2(q4.z, q4.w);
            u0 = __ffma2_rn(e01.k, q01, u0);
            u1 = __ffma2_rn(e23.k, q23, u1);
            const float2 g01 = __fmul2_rn(dkernel_from_eval<KIND>(e01), q01);
            const float2 g23 = __fmul2_rn(dkernel_from_eval<KIND>(e23), q23);
#pragma unroll
            for (int k = 0; k < D; ++k) {
              const float4 x4 = *reinterpret_cast<const float4*>(smX + (size_t)k * kN + col0 + 4 * pp);
              const float2 d01 = __fadd2_rn(make_float2(x4.x, x4.y), nxi[k]);
              const float2 d23 = __fadd2_rn(make_float2(x4.z, x4.w), nxi[k]);
              dl[k] = __ffma2_rn(g01, __fmul2_rn(d01, d01), dl[k]);
              dl[k] = __ffma2_rn(g23, __fmul2_rn(d23, d23), dl[k]);
            }
          }
        }
      }
      epi_release(p, sl);
      yacc += (double)(y0.x + y0.y) + (double)(y1.x + y1.y);
      if (ADJ) {
        uacc += (double)(u0.x + u0.y) + (double)(u1.x + u1.y);
#pragma unroll
        for (int k = 0; k < D; ++k) dacc[k] += (double)(dl[k].x + dl[k].y);
      }
    }
    // combine the two column halves, scale, store
    const double sigma = (double)consts[0];
    if (e.half == 1) ycomb[e.row] = yacc;
    tma::named_bar_sync(1, kEpiWarps * 32);
    if (e.half == 0 && e.live) part[(int64_t)blockIdx.y * rows + p.i0 + e.row] = (float)((yacc + ycomb[e.row]) * sigma);
    if (ADJ) {
      const double li = e.live ? (double)v[p.i0 + e.row] * sigma : 0.0;
#pragma unroll
      for (int k = 0; k < D; ++k) dacc[k] *= li;
      epi_reduce_grad<ADJ ? D : 1>(dacc, li * uacc, d, gpart);
    }
  }
  pipe_teardown(p);
}

// Deferred parameter cotangent of M <= kBatchMax matvec VJPs at once (the adjoint sweep of the Krylov
// loops defers them: arnoldi.py:207-209 only needs A^T lambda inside the loop):
//     sum_m d<lam_m, K(theta) q_m>/dtheta = sum_ij W_ij dk_ij/dtheta,   W_ij = sum_m lam_m[i] q_m[j],
// so the kernel tile (distances on the tensor pipe, sqrt / exp on the MUFU) and the per-dimension
// (x_ik - x_jk)^2 accumulation are paid ONCE for the M pairs; only the rank-M weight costs M FMAs per
// kernel entry.  Per-CTA partial sums in gpart (layout of the adjoint sweep).
template <int KIND, int D>
__global__ void __launch_bounds__(kThreads, 1)
k_gram_tc_gradbatch(int64_t n, int64_t npad, int d, int slots, const float* __restrict__ opA,
                    const float* __restrict__ opB, const float* __restrict__ xt, const float* __restrict__ xx,
                    const float* __restrict__ consts, const float* __restrict__ Qrows, int64_t ldq,
                    const float* __restrict__ Lrows, int64_t ldl, int M, double* __restrict__ gpart) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const Pipe p = pipe_setup(smem, make_plan_batch(slots), n);
  const int warp = threadIdx.x >> 5;
  if (warp == 0) {
    RowsAux<D> aux{{}, M, n, xt, npad};
    for (int m = 0; m < M; ++m) aux.rows.p[m] = Qrows + (int64_t)m * ldq;
    producer_warp(p, opA, npad, opB, npad, aux);
  } else if (warp == 1) {
    mma_warp(p);
  } else {
    const EpiThread e = epi_thread<KIND>(p, n, xx);
    double uacc = 0.0, dacc[D];
    float2 nxi[D], lam2[kBatchMax];
#pragma unroll
    for (int k = 0; k < D; ++k) {
      const float x = xt[(int64_t)k * npad + p.i0 + e.row];
      nxi[k] = make_float2(-x, -x);
      dacc[k] = 0.0;
    }
#pragma unroll
    for (int m = 0; m < kBatchMax; ++m) {
      const float l = (e.live && m < M) ? Lrows[(int64_t)m * ldl + p.i0 + e.row] : 0.f;
      lam2[m] = make_float2(l, l);
    }
    for (int it = 0; it < p.ntiles; ++it) {
      const Slot sl = slot_of(p, it);
      const float* smQ = p.aux(sl.s);
      const float* smX = smQ + kBatchMax * kN;
      epi_wait(p, sl);
      float2 u0 = make_float2(0.f, 0.f), u1 = u0, dl[D];
#pragma unroll
      for (int k = 0; k < D; ++k) dl[k] = make_float2(0.f, 0.f);
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        const int col0 = e.half * 128 + cc * 32;
        uint32_t r[32];
        epi_load(p, e, sl, it, col0, r);
#pragma unroll
        for (int pp = 0; pp < 8; ++pp) {
          const float2 a01 = make_float2(__uint_as_float(r[4 * pp]), __uint_as_float(r[4 * pp + 1]));
          const float2 a23 = make_float2(__uint_as_float(r[4 * pp + 2]), __uint_as_float(r[4 * pp + 3]));
          const Eval2 e01 = kernel_from_acc<KIND>(a01, e.crow), e23 = kernel_from_acc<KIND>(a23, e.crow);
          float2 w01 = make_float2(0.f, 0.f), w23 = w01;  // W_ij = sum_m lam_m[i] q_m[j]
#pragma unroll
          for (int m = 0; m < kBatchMax; ++m) {
            if (m < M) {
              const float4 q4 = *reinterpret_cast<const float4*>(smQ + (size_t)m * kN + col0 + 4 * pp);
              w01 = __ffma2_rn(lam2[m], make_float2(q4.x, q4.y), w01);
              w23 = __ffma2_rn(lam2[m], make_float2(q4.z, q4.w), w23);
            }
          }
          u0 = __ffma2_rn(e01.k, w01, u0);
          u1 = __ffma2_rn(e23.k, w23, u1);
          const float2 g01 = __fmul2_rn(dkernel_from_eval<KIND>(e01), w01);
          const float2 g23 = __fmul2_rn(dkernel_from_eval<KIND>(e23), w23);
#pragma unroll
          for (int k = 0; k < D; ++k) {
            const float4 x4 = *reinterpret_cast<const float4*>(smX + (size_t)k * kN + col0 + 4 * pp);
            const float2 d01 = __fadd2_rn(make_float2(x4.x, x4.y), nxi[k]);
            const float2 d23 = __fadd2_rn(make_float2(x4.z, x4.w), nxi[k]);
            dl[k] = __ffma2_rn(g01, __fmul2_rn(d01, d01), dl[k]);
            dl[k] = __ffma2_rn(g23, __fmul2_rn(d23, d23), dl[k]);
          }
        }
      }
      epi_release(p, sl);
      uacc += (double)(u0.x + u0.y) + (double)(u1.x + u1.y);
#pragma unroll
      for (int k = 0; k < D; ++k) dacc[k] += (double)(dl[k].x + dl[k].y);
    }
    const double sigma = (double)consts[0];
#pragma unroll
    for (int k = 0; k < D; ++k) dacc[k] *= sigma;
    epi_reduce_grad<D>(dacc, sigma * uacc, d, gpart);
  }
  pipe_teardown(p);
}

// Matvec of P <= kBatchMax vectors at once (lockstep Krylov runs over probes): every kernel tile --
// distances on the tensor pipe, sqrt / exp on the MUFU -- is evaluated ONCE and applied to the P
// vectors (P extra FMAs per entry), so P matvecs cost about as much as two.
//   part[split][p][i] = sigma sum_{j in split} k_ij v_p[j]
template <int KIND>
__global__ void __launch_bounds__(kThreads, 1)
k_gram_tc_multi(int64_t n, int64_t npad, int slots, const float* __restrict__ opA, const float* __restrict__ opB,
                const float* __restrict__ xx, const float* __restrict__ consts, VecPtrs vecs, int P,
                float* __restrict__ part) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ double ycomb[kBatchMax][kM];
  const Pipe p = pipe_setup(smem, make_plan_multi(slots), n);
  const int warp = threadIdx.x >> 5;
  if (warp == 0) {
    producer_warp(p, opA, npad, opB, npad, RowsAux<1>{vecs, P, n, nullptr, npad});
  } else if (warp == 1) {
    mma_warp(p);
  } else {
    const EpiThread e = epi_thread<KIND>(p, n, xx);
    double yacc[kBatchMax];
#pragma unroll
    for (int q = 0; q < kBatchMax; ++q) yacc[q] = 0.0;
    for (int it = 0; it < p.ntiles; ++it) {
      const Slot sl = slot_of(p, it);
      const float* smV = p.aux(sl.s);
      epi_wait(p, sl);
      float2 y[kBatchMax];
#pragma unroll
      for (int q = 0; q < kBatchMax; ++q) y[q] = make_float2(0.f, 0.f);
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        const int col0 = e.half * 128 + cc * 32;
        uint32_t r[32];
        epi_load(p, e, sl, it, col0, r);
#pragma unroll
        for (int pp = 0; pp < 8; ++pp) {
          const float2 a01 = make_float2(__uint_as_float(r[4 * pp]), __uint_as_float(r[4 * pp + 1]));
          const float2 a23 = make_float2(__uint_as_float(r[4 * pp + 2]), __uint_as_float(r[4 * pp + 3]));
          const Eval2 e01 = kernel_from_acc<KIND>(a01, e.crow), e23 = kernel_from_acc<KIND>(a23, e.crow);
#pragma unroll
          for (int q = 0; q < kBatchMax; ++q) {
            if (q < P) {
              const float4 v4 = *reinterpret_cast<const float4*>(smV + (size_t)q * kN + col0 + 4 * pp);
              y[q] = __ffma2_rn(e01.k, make_float2(v4.x, v4.y), y[q]);
              y[q] = __ffma2_rn(e23.k, make_float2(v4.z, v4.w), y[q]);
            }
          }
        }
      }
      epi_release(p, sl);
#pragma unroll
      for (int q = 0; q < kBatchMax; ++q) yacc[q] += (double)(y[q].x + y[q].y);
    }
    const double sigma = (double)consts[0];
    if (e.half == 1) {
#pragma unroll
      for (int q = 0; q < kBatchMax; ++q) ycomb[q][e.row] = yacc[q];
    }
    tma::named_bar_sync(1, kEpiWarps * 32);
    if (e.half == 0 && e.live) {
#pragma unroll
      for (int q = 0; q < kBatchMax; ++q)
        if (q < P) part[((int64_t)blockIdx.y * P + q) * n + p.i0 + e.row] = (float)((yacc[q] + ycomb[q][e.row]) * sigma);
    }
  }
  pipe_teardown(p);
}

}  // namespace gramtc
}  // namespace bl
