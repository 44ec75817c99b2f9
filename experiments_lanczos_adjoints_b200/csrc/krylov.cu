// Host-side drivers of the Krylov loops: they only enqueue kernels on the caller's stream.
//   bl_arnoldi_forward  <- arnoldi._forward / _forward_step   (arnoldi.py:57-101)
//   bl_arnoldi_adjoint  <- arnoldi._adjoint / _adjoint_step   (arnoldi.py:104-220)
//   bl_lanczos3_*       <- lanczos._forward / _adjoint        (lanczos.py:215-335)
#include <algorithm>
#include <mutex>
#include <set>
#include <utility>
#include <vector>
#include <type_traits>

#include <cstdlib>
#ifndef BL_DOTS_TILE_BYTES
#define BL_DOTS_TILE_BYTES 4096
#endif

#include "dist.cuh"
#include "krylov_kernels.cuh"
#include "stream_kernels.cuh"
#include "step_kernel.cuh"
#include "operators.cuh"

namespace bl {
namespace {

struct Grid {
  int dots = 1, combine = 1;
};

// Upper bounds the workspace is sized for (148 SMs on B200: 2 / 16 blocks per SM).
constexpr int kMaxDotsGrid = 296;
constexpr int kMaxCombineGrid = 2368;

int64_t gram_parts_for(int64_t n, int64_t K) {
  return std::max<int64_t>(1, std::min<int64_t>(kMaxDotsGrid, std::min<int64_t>((n + 1023) / 1024, (4 << 20) / (K * K) + 1)));
}

template <typename T>
Grid pick_grid(int64_t n) {
  constexpr int VN = Vec<T>::N;
  const int64_t groups = (n + VN - 1) / VN;
  Grid g;
  const int sms = sm_count();
  g.dots = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(2 * sms, kMaxDotsGrid), (groups + 255) / 256));
  g.combine = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(16 * sms, kMaxCombineGrid), (groups + kCombineThreads - 1) / kCombineThreads));
  return g;
}

// Carves the caller's workspace.
struct Workspace {
  unsigned char* base;
  size_t size, used = 0;
  Workspace(void* p, size_t bytes) : base(static_cast<unsigned char*>(p)), size(bytes) {}
  void* take(size_t bytes) {
    used = align_up(used, 256);
    void* p = base + used;
    used += bytes;
    return p;
  }
  bool ok() const { return used <= size; }
};

struct Common {
  unsigned int* counters;  // [0] dots, [1] combine
  double* scal;
  double* red;
  double* coefA;
  double* coefB;
  double* coefC;
  double* partials_dots;
  double* partials_comb;
  double* partials_few;  // [kFewMax][kMaxDotsGrid]: per-block shares of k_step_tma's phase 0
  long long partials_dots_count = 0;  // doubles behind partials_dots
};

size_t common_bytes(int64_t K) {
  size_t b = 0;
  b += 256;                                   // counters
  b += align_up(S_COUNT * 8, 256);            // scal
  b += 4 * align_up((K + 2) * 8, 256);        // red, coefA, coefB, coefC
  b += align_up((size_t)(K + 2) * kMaxDotsGrid * 8, 256);  // partials_dots
  b += align_up((size_t)kMaxCombineGrid * 8, 256);         // partials_comb
  b += align_up((size_t)kFewMax * kMaxDotsGrid * 8, 256);  // partials_few
  return b + 9 * 256;
}

void carve_common(Workspace& w, int64_t K, Common& c) {
  c.counters = static_cast<unsigned int*>(w.take(256));
  c.scal = static_cast<double*>(w.take(S_COUNT * 8));
  c.red = static_cast<double*>(w.take((K + 2) * 8));
  c.coefA = static_cast<double*>(w.take((K + 2) * 8));
  c.coefB = static_cast<double*>(w.take((K + 2) * 8));
  c.coefC = static_cast<double*>(w.take((K + 2) * 8));
  c.partials_dots = static_cast<double*>(w.take((size_t)(K + 2) * kMaxDotsGrid * 8));
  c.partials_dots_count = (long long)(K + 2) * kMaxDotsGrid;
  c.partials_comb = static_cast<double*>(w.take((size_t)kMaxCombineGrid * 8));
  c.partials_few = static_cast<double*>(w.take((size_t)kFewMax * kMaxDotsGrid * 8));
}

// TMA-staged kernels for n >= 8192; below that the register-staged (LDG) kernels.
bool use_tma(int64_t n) { return n >= 8192; }

template <typename T>
constexpr int dots_tile() { return BL_DOTS_TILE_BYTES / (int)sizeof(T); }  // row segment per copy

// Blocks per SM of the TMA-staged kernels (BL_BLOCKS_PER_SM = 1 or 2, default 2).  Two fill the shared memory
// of an SM; one leaves room for the successor's blocks to become resident and prefetch under the tail.
std::atomic<int> g_blocks_per_sm{0};  // bl_set_blocks_per_sm; 0 = environment / default
int blocks_per_sm() {
  static int v = [] {
    const char* e = std::getenv("BL_BLOCKS_PER_SM");
    return (e && e[0] == '1') ? 1 : 2;
  }();
  const int set = g_blocks_per_sm.load(std::memory_order_relaxed);
  return set ? set : v;
}
template <typename T>
int tma_grid(int64_t n, int tile) {
  return (int)std::max<int64_t>(1, std::min<int64_t>(std::min(blocks_per_sm() * sm_count(), kMaxDotsGrid), (n + tile - 1) / tile));
}

// Launch with the programmatic-dependent-launch attribute: the kernel's
// prologue and its first TMA loads overlap the tail (imbalance, last-block reduction) of the
// kernel in front of it; the kernel itself executes griddepcontrol.wait before reading anything
// its predecessor wrote.
// Row sharding: cross-rank SUM of the reduced values between a kernel's local reduction and the
// epilogue that consumes them (bl_dist_set_reduce_hook).
thread_local bl_allreduce_cb g_reduce_hook = nullptr;
thread_local void* g_reduce_user = nullptr;

// Runs `epi` after the hook: the kernel in front was launched with EPI_NONE and left the local
// sums in red[0..count).
bool is_sharded() { return g_reduce_hook != nullptr || dist::active(); }

// cross-rank sum over peer memory fused with the epilogue: one single-block kernel (dist.cuh)
template <typename T>
__global__ void __launch_bounds__(256) k_peer_reduce_epilogue(dist::PeerView pv, int count, Epi epi) {
  dist::peer_allreduce_block(pv, epi.red, count);
  run_epilogue<T>(epi);
}
__global__ void __launch_bounds__(256) k_peer_reduce(dist::PeerView pv, double* values, int count) {
  dist::peer_allreduce_block(pv, values, count);
}

// in-place cross-rank SUM of `count` device doubles on `s` (communicator first, then the hook)
int sharded_sum(double* values, int count, cudaStream_t s) {
  if (dist::active()) {
    BL_REQUIRE(count <= dist::kRedSlots, "reduction too large for the peer mailbox");
    dist::PeerView pv;
    BL_CHECK(dist::next_reduce(&pv));
    k_peer_reduce<<<1, 256, 0, s>>>(pv, values, count);
    BL_LAUNCHED();
    return BL_OK;
  }
  if (g_reduce_hook && g_reduce_hook(g_reduce_user, values, count, s) != 0) {
    set_error("all-reduce hook failed");
    return BL_ECALLBACK;
  }
  return BL_OK;
}

template <typename T>
int finish_sharded(const Common& c, Epi epi, int count, cudaStream_t s) {
  epi.red = c.red;
  epi.scal = c.scal;
  if (dist::active()) {
    BL_REQUIRE(count <= dist::kRedSlots, "reduction too large for the peer mailbox");
    dist::PeerView pv;
    BL_CHECK(dist::next_reduce(&pv));
    k_peer_reduce_epilogue<T><<<1, 256, 0, s>>>(pv, count, epi);
    BL_LAUNCHED();
    return BL_OK;
  }
  if (g_reduce_hook(g_reduce_user, c.red, count, s) != 0) {
    set_error("all-reduce hook failed");
    return BL_ECALLBACK;
  }
  k_epilogue_only<T><<<1, 256, 0, s>>>(epi);
  BL_LAUNCHED();
  return BL_OK;
}

// The epilogue of a streaming kernel's reduction, row sharding included: arm() before the launch, finish() after it.
// Peer-memory route: the cross-rank sum rides in the last block of the kernel itself (its epilogue carries the peer
// view), so a sharded reduction costs no extra launch.  All-reduce-hook route: the kernel runs with EPI_NONE and
// leaves its local sums in red[0..count); finish() runs the hook and then the epilogue as a launch of its own.
struct ShardedEpi {
  const Common* c = nullptr;
  Epi full;  // the epilogue as the caller built it
  int count = 0;
  bool split = false;  // hook route: finish() runs `full`

  // Points `epi` at the run's reduction buffers and, under row sharding, arms or splits it for `n` reduced values.
  int arm(const Common& common, Epi& epi, int n) {
    c = &common;
    epi.red = common.red;
    epi.scal = common.scal;
    full = epi;
    count = n;
    if (!dist::active()) {
      split = is_sharded();
      if (split) epi.mode = EPI_NONE;
      return BL_OK;
    }
    if (n > dist::kRedSlots) {
      set_error("reduction too large for the peer mailbox");
      return BL_EINVAL;
    }
    dist::PeerView pv;
    const int rc = dist::next_reduce(&pv);
    if (pv.world > 1) {  // one rank: the local sums are the global sums
      epi.peer_mail = pv.mail[pv.rank];
      epi.peer_seq = pv.seq;
      epi.peer_count = n;
    }
    return rc;
  }

  template <typename T>
  int finish(cudaStream_t s) const {
    return split ? finish_sharded<T>(*c, full, count, s) : BL_OK;
  }
};

// L2 "snake" order: consecutive streaming kernels walk the basis in
// opposite directions, so a kernel starts on the tiles its predecessor read last — the part of
// the basis that is still in the 126 MB L2.  Each block owns the same column range in every
// kernel (same grid, same partition), which makes the reuse exact.
thread_local int g_direction = 0;  // toggled per streaming launch; host-side launch order is the stream order
int next_direction() {
  g_direction ^= 1;
  return g_direction;
}

template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// The dynamic shared-memory opt-in is a per-device function attribute: cache it per (kernel,
// device) so that one process may drive several GPUs from different host threads.
template <typename F>
int set_smem(F* kernel, size_t bytes) {
  static std::mutex mu;
  static std::set<std::pair<const void*, int>> done;
  int dev = 0;
  BL_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  const auto key = std::make_pair(reinterpret_cast<const void*>(kernel), dev);
  if (done.count(key)) return BL_OK;
  BL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  done.insert(key);
  return BL_OK;
}

RowSource row_source(const RowBlock& b0, const RowBlock* b1, size_t w) {
  RowSource r;
  r.base0 = static_cast<const char*>(b0.base) + (long long)b0.row0 * b0.ld * (long long)w;
  r.ldb0 = b0.ld * (long long)w;
  r.n0 = b0.nrows;
  if (b1 && b1->nrows > 0) {
    r.base1 = static_cast<const char*>(b1->base) + (long long)b1->row0 * b1->ld * (long long)w;
    r.ldb1 = b1->ld * (long long)w;
    r.n1 = b1->nrows;
  }
  return r;
}

template <typename T>
int launch_dots(const Grid& g, const Common& c, RowBlock blk, const T* x, int64_t n, Epi epi, cudaStream_t s) {
  ShardedEpi se;
  BL_CHECK(se.arm(c, epi, blk.nrows));
  {
  ProfScope prof(BL_PROF_DOTS, (double)(blk.nrows + 1) * n * sizeof(T), s);
  if (use_tma(n) && blk.nrows <= 4) {
    FewRows fr;
    for (int j = 0; j < blk.nrows; ++j)
      fr.row[j] = static_cast<const char*>(blk.base) + (long long)(blk.row0 + j) * blk.ld * (long long)sizeof(T);
    // about two 16-byte vectors per thread and stream; the partials buffer holds (K+2) x kMaxDotsGrid doubles
    const long long vecs = n / Vec<T>::N;
    const int grid = (int)std::max<long long>(1, std::min<long long>({4LL * sm_count(), (vecs + 511) / 512,
                                                                      c.partials_dots_count / blk.nrows}));
    switch (blk.nrows) {
      case 1: BL_CUDA(launch_pdl(k_dots_few<T, 1>, grid, 256, 0, s, fr, x, (long long)n, c.partials_dots, c.counters + 0, epi)); break;
      case 2: BL_CUDA(launch_pdl(k_dots_few<T, 2>, grid, 256, 0, s, fr, x, (long long)n, c.partials_dots, c.counters + 0, epi)); break;
      case 3: BL_CUDA(launch_pdl(k_dots_few<T, 3>, grid, 256, 0, s, fr, x, (long long)n, c.partials_dots, c.counters + 0, epi)); break;
      default: BL_CUDA(launch_pdl(k_dots_few<T, 4>, grid, 256, 0, s, fr, x, (long long)n, c.partials_dots, c.counters + 0, epi)); break;
    }
  } else if (use_tma(n)) {
    constexpr int TILE = dots_tile<T>();
    const size_t smem = (size_t)(kStages * kGroup + 2) * TILE * sizeof(T) + (2 * kStages + 4) * 8 +
                        (size_t)blk.nrows * 8 + 16;
    BL_CHECK(set_smem(k_dots_tma<T, TILE>, 112 * 1024));
    BL_REQUIRE(smem <= 112 * 1024, "too many rows for k_dots_tma");
    BL_CUDA(launch_pdl(k_dots_tma<T, TILE>, tma_grid<T>(n, TILE), kStreamThreads, smem, s,
                       row_source(blk, nullptr, sizeof(T)), blk.nrows, x, (long long)n, c.partials_dots,
                       c.counters + 0, epi, next_direction()));
  } else {
    k_dots<T><<<g.dots, kDotsThreads, 0, s>>>(blk, x, n, c.partials_dots, c.counters + 0, epi);
  }
  BL_LAUNCHED();
  }
  return se.finish<T>(s);
}

template <typename T>
int launch_combine(const Grid& g, const Common& c, CombineArgs a, bool norm, cudaStream_t s) {
  a.partials = c.partials_comb;
  a.counter = c.counters + 1;
  a.epi.red = c.red;
  a.epi.scal = c.scal;
  ShardedEpi se;  // the reduction of ||out||^2 only
  if (norm) BL_CHECK(se.arm(c, a.epi, 1));
  const int nrows = a.blk[0].nrows + a.blk[1].nrows;
  {
  ProfScope prof(BL_PROF_COMBINE, (double)(nrows + a.nvec + 1 + (a.out2 ? 1 : 0)) * a.n * sizeof(T), s);
  if (use_tma(a.n) && nrows + a.nvec >= 4) {
    constexpr int TILE = kConsumerThreads * Vec<T>::N;
    CombineTmaArgs t;
    t.n = a.n;
    t.out = a.out;
    t.out2 = a.out2;
    t.nvec = a.nvec;
    for (int k = 0; k < a.nvec; ++k) t.vec[k] = a.vec[k];
    t.src = row_source(a.blk[0], &a.blk[1], sizeof(T));
    t.coef0 = a.blk[0].coef ? a.blk[0].coef + a.blk[0].coef0 : nullptr;
    t.sign0 = a.blk[0].sign;
    t.coef1 = a.blk[1].coef ? a.blk[1].coef + a.blk[1].coef0 : nullptr;
    t.sign1 = a.blk[1].sign;
    t.out_div_ptr = a.out_div_ptr;
    t.out_mul_ptr = a.out_mul_ptr;
    t.partials = a.partials;
    t.counter = a.counter;
    t.reverse = next_direction();
    t.epi = a.epi;
    const size_t smem = (size_t)kStages * kGroup * TILE * sizeof(T) + 2 * kStages * 8 +
                        (size_t)(nrows + 2 * kGroup) * sizeof(T) + 16;
    BL_CHECK(set_smem(k_combine_tma<T, true>, 100 * 1024));
    BL_CHECK(set_smem(k_combine_tma<T, false>, 100 * 1024));
    BL_REQUIRE(smem <= 100 * 1024, "too many rows for k_combine_tma");
    const int grid = tma_grid<T>(a.n, TILE);
    if (norm)
      BL_CUDA(launch_pdl(k_combine_tma<T, true>, grid, kStreamThreads, smem, s, t));
    else
      BL_CUDA(launch_pdl(k_combine_tma<T, false>, grid, kStreamThreads, smem, s, t));
  } else {
    const size_t smem = (size_t)(nrows + 1) * sizeof(T);
    if (norm)
      k_combine<T, true><<<g.combine, kCombineThreads, smem, s>>>(a);
    else
      k_combine<T, false><<<g.combine, kCombineThreads, smem, s>>>(a);
  }
  BL_LAUNCHED();
  }
  return se.finish<T>(s);
}

// ---- tensor maps (cuTensorMapEncodeTiled through the runtime's driver entry point) --------
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// Row-major [rows x ld] basis buffer, box = [8 rows x box_cols]; out-of-range elements read as 0.
int make_basis_map(CUtensorMap* map, int dtype, const void* base, int64_t ld, int64_t rows, int box_cols,
                   int box_rows = kGroup) {
  EncodeTiledFn fn = encode_tiled_fn();
  BL_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled is not available in this driver");
  const cuuint64_t gdim[2] = {(cuuint64_t)ld, (cuuint64_t)std::max<int64_t>(rows, 1)};
  const cuuint64_t gstride[1] = {(cuuint64_t)ld * dtype_size(dtype)};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  const cuuint32_t estride[2] = {1, 1};
  CUresult r = fn(map, dtype == BL_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2,
                  const_cast<void*>(base), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
    return BL_ECUDA;
  }
  return BL_OK;
}

// Host-side description of a fused combine + dots launch (k_fused_tma).
struct FusedSpec {
  int64_t n = 0;
  void* out = nullptr;
  int nvec = 0;
  VecTerm vec[kMaxVecTerms];
  RowBlock res;             // resident rows (dots wanted): coefficient of row j = sign * coef[coef0 + j]
  RowBlock str0, str1;      // streamed-only rows
  int64_t rows_total0 = 0;  // row extent of the buffers behind str0 / str1 (for the tensor maps)
  int64_t rows_total1 = 0;
  const double* out_div_ptr = nullptr;
  Epi epi;
};

template <typename T, int TILE>
int launch_fused_tile(const Common& c, const FusedSpec& f, int dtype, int sr, cudaStream_t s) {
  constexpr int BOXC = TILE > 256 ? 256 : TILE;
  const FusedLayout L = fused_layout<T, TILE>(f.res.nrows, f.str0.nrows, f.str1.nrows, f.nvec, sr);
  BL_CHECK(set_smem(k_fused_tma<T, TILE>, 225 * 1024));
  FusedArgs a;
  const char* res_base = static_cast<const char*>(f.res.base) + (int64_t)f.res.row0 * f.res.ld * (int64_t)sizeof(T);
  BL_CHECK(make_basis_map(&a.map_res, dtype, res_base, f.res.ld, f.res.nrows, BOXC));
  if (f.str0.nrows > 0)
    BL_CHECK(make_basis_map(&a.map_str0, dtype, f.str0.base, f.str0.ld, f.rows_total0, BOXC, sr));
  else
    a.map_str0 = a.map_res;
  if (f.str1.nrows > 0)
    BL_CHECK(make_basis_map(&a.map_str1, dtype, f.str1.base, f.str1.ld, f.rows_total1, BOXC, sr));
  else
    a.map_str1 = a.map_res;
  a.n = f.n;
  a.out = f.out;
  a.nvec = f.nvec;
  for (int k = 0; k < f.nvec; ++k) a.vec[k] = f.vec[k];
  a.nres = f.res.nrows;
  a.coef_res = f.res.coef + f.res.coef0;
  a.sign_res = f.res.sign;
  a.nstr0 = f.str0.nrows;
  a.row_str0 = f.str0.row0;
  a.coef_str0 = f.str0.coef ? f.str0.coef + f.str0.coef0 : nullptr;
  a.sign_str0 = f.str0.sign;
  a.nstr1 = f.str1.nrows;
  a.row_str1 = f.str1.row0;
  a.coef_str1 = f.str1.coef ? f.str1.coef + f.str1.coef0 : nullptr;
  a.sign_str1 = f.str1.sign;
  a.out_div_ptr = f.out_div_ptr;
  a.sr = sr;
  a.partials = c.partials_dots;
  a.counter = c.counters + 0;
  a.epi = f.epi;
  ShardedEpi se;
  BL_CHECK(se.arm(c, a.epi, f.res.nrows));
  a.reverse = next_direction();
  const int nrows = f.res.nrows + f.str0.nrows + f.str1.nrows;
  {
    ProfScope prof(BL_PROF_FUSED, (double)(nrows + f.nvec + 1) * f.n * sizeof(T), s);
    BL_CUDA(launch_pdl(k_fused_tma<T, TILE>, tma_grid<T>(f.n, TILE), kStreamThreads, L.total_bytes, s, a));
    BL_LAUNCHED();
  }
  return se.finish<T>(s);
}

// `*fused` is false on return when no tile shape fits shared memory or n is below the TMA threshold;
// the caller then runs combine and dots separately.
template <typename T>
int launch_fused(const Common& c, const FusedSpec& f, int dtype, cudaStream_t s, bool* fused) {
  *fused = false;
  // k_fused_tma keeps one register accumulator per resident box: at most 16 boxes = 128 rows
  if (!use_tma(f.n) || f.n >= ((int64_t)1 << 31) || f.res.nrows > 128) return BL_OK;
  // every tile pays a fixed chain (exchange, barriers, sweep hand-over) of about a microsecond: with
  // fewer than ~16 rows per tile that costs more than the second read of the rows it saves
  if (f.res.nrows + f.str0.nrows + f.str1.nrows < 16) return BL_OK;
  constexpr size_t two_per_sm = 113 * 1024;
  constexpr int TMAX = 4096 / (int)sizeof(T);  // 1024 floats / 512 doubles
  const int nr = f.res.nrows, n0 = f.str0.nrows, n1 = f.str1.nrows, nv = f.nvec;
  *fused = true;
  // widest tile that leaves room for two blocks per SM (the per-tile hand-over between the two
  // sweeps is a fixed cost); then the largest streamed-row group (32, 16 or 8 rows per ring stage)
  // that still fits
  auto pick_sr = [&](auto tile_tag) -> int {
    constexpr int TILE = decltype(tile_tag)::value;
    if (n0 + n1 == 0) return fused_layout<T, TILE>(nr, n0, n1, nv, kGroup).total_bytes <= two_per_sm ? kGroup : 0;
    for (int sr : {32, 16, 8})
      if (fused_layout<T, TILE>(nr, n0, n1, nv, sr).total_bytes <= two_per_sm) return sr;
    return 0;
  };
  if (int sr = pick_sr(std::integral_constant<int, TMAX>{})) return launch_fused_tile<T, TMAX>(c, f, dtype, sr, s);
  if (int sr = pick_sr(std::integral_constant<int, TMAX / 2>{})) return launch_fused_tile<T, TMAX / 2>(c, f, dtype, sr, s);
  if (int sr = pick_sr(std::integral_constant<int, TMAX / 4>{})) return launch_fused_tile<T, TMAX / 4>(c, f, dtype, sr, s);
  if (int sr = pick_sr(std::integral_constant<int, TMAX / 8>{})) return launch_fused_tile<T, TMAX / 8>(c, f, dtype, sr, s);
  *fused = false;
  return BL_OK;
}

// Phase 1 of a symmetric-loop step (StepArgs below) as a launch of its own: out1 = (sum of <= kXTerms vector
// terms) / div and red[j] = <row_j, out1> over the rows of src1 (k_xdots_tma, step_kernel.cuh).  `*done` stays
// false when n is below the TMA threshold or the shape does not fit; the caller then runs its general kernels.
template <typename T>
int launch_xdots(const Common& c, const StepArgs& f, cudaStream_t s, bool* done) {
  *done = false;
  constexpr int TILE = kConsumerThreads * Vec<T>::N;  // 4 KB row segments
  const size_t smem = (size_t)(kStages * kGroup + 2) * TILE * sizeof(T) + (2 * kStages + 4) * 8 +
                      (size_t)f.nrows1 * 8 + 16;
  if (!use_tma(f.n) || f.nvec > kXTerms || f.nrows1 < 1 || smem > 112 * 1024) return BL_OK;
  *done = true;
  StepArgs a = f;
  a.partials = c.partials_dots;
  ShardedEpi se;
  BL_CHECK(se.arm(c, a.epi1, f.nrows1));
  const int reverse = next_direction();
  BL_CHECK(set_smem(k_xdots_tma<T, TILE>, 112 * 1024));
  {
    ProfScope prof(BL_PROF_FUSED, (double)(f.nrows1 + f.nvec + 1) * f.n * sizeof(T), s);
    BL_CUDA(launch_pdl(k_xdots_tma<T, TILE>, tma_grid<T>(f.n, TILE), kStreamThreads, smem, s, a, c.counters + 0,
                       reverse));
    BL_LAUNCHED();
  }
  return se.finish<T>(s);
}

// One launch for the three basis-streaming phases of a symmetric-loop step (k_step_tma, step_kernel.cuh).  The kernel's
// blocks wait for one another, so the launch is cooperative (the driver starts the grid only when all of it is
// resident: kernels of other streams cannot wedge it) and the grid is capped at what fits the device.
std::atomic<int> g_step_pdl_ok{1};  // cleared when the driver refuses cooperative + programmatic launch together
std::atomic<int> g_step_trace_next{-1};  // bl_step_trace_begin arms it; every k_step_tma launch takes a slot

struct StepItem {  // one run's share of a k_step_tma launch
  const Common* c = nullptr;
  StepArgs a;
  double bytes = 0.0;  // algorithmic bytes of the three phases (profile classes)
  const StepOp* op = nullptr;  // the step's operator call rides in the launch (same for every run of a batch)
};

// The operator call of a Krylov step as phase S of k_step_tma: operands stored as SELL-32 only (SparseOperator).
// norm: the forward's q = v / len on the way, rows written up to n_pad.
bool make_step_op(bl_operator_t* op, int dtype, bool transpose, bool norm, int64_t n, int64_t n_pad, StepOp* so) {
  SellView v;
  if (!op->sell_view(dtype, transpose, &v)) return false;
  if (v.nrows != n || (norm && n_pad > v.nslices * 32)) return false;
  *so = StepOp();
  so->slice_ptr = v.slice_ptr;
  so->col = v.col;
  so->val = v.val;
  so->nslices = v.nslices;
  so->nrows = v.nrows;
  so->n_pad = n_pad;
  so->norm = norm ? 1 : 0;
  return true;
}

template <typename T>
size_t step_smem_bytes(int count, int acc_stride, int coef_stride) {
  constexpr int TILE = kConsumerThreads * Vec<T>::N;
  return (size_t)(kStages * kGroup + 2) * TILE * sizeof(T) + (2 * kStages + 2 + 2 * step::kOpStages) * 8 +
         (size_t)count * acc_stride * 8 + (size_t)count * coef_stride * sizeof(T) + 16;
}

// whether `blocks` blocks per SM of k_step_tma are co-resident on this device (cached per dtype and device)
template <typename T>
bool step_fits(int blocks) {
  constexpr int TILE = kConsumerThreads * Vec<T>::N;
  static std::mutex mu;
  static std::set<std::pair<int, int>> ok, bad;  // (device, blocks per SM), for the 112 KB opt-in size
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return false;
  std::lock_guard<std::mutex> lk(mu);
  const auto key = std::make_pair(dev, blocks);
  if (ok.count(key)) return true;
  if (bad.count(key)) return false;
  int coop = 0, per_sm = 0;
  cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
  if (coop && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_step_tma<T, TILE>, kStreamThreads, 112 * 1024) ==
                  cudaSuccess && per_sm >= blocks) {
    ok.insert(key);
    return true;
  }
  (void)cudaGetLastError();
  bad.insert(key);
  return false;
}

// The step of `count` runs (same n, same dtype) in ceil(count / kStepBatch) launches.  `*done` stays false -- nothing
// launched -- when the kernel does not apply (one run, row sharding, shape); the caller then runs the separate
// kernels for every run.  Batches of two or more runs only: for ONE run an in-kernel reduction costs what a kernel
// boundary with programmatic dependent launch costs (measured: 24.3 vs 23.6 ms per forward + adjoint at n = 1M,
// depth 100).
template <typename T>
int launch_step(std::vector<StepItem>& items, cudaStream_t s, bool* done) {
  *done = false;
  constexpr int TILE = kConsumerThreads * Vec<T>::N;
  const int total = (int)items.size();
  if (total < 2 || is_sharded()) return BL_OK;
  const StepOp* sop = items[0].op;
  const long long n = items[0].a.n;
  if (!use_tma(n)) return BL_OK;
  int acc_stride = kFewSlots, coef_stride = kGroup;
  for (const StepItem& it : items) {
    const StepArgs& a = it.a;
    if (a.n != n || a.nvec > kXTerms || a.few_n > kFewMax || a.nrows1 < 1 || a.nrows2 < 1) return BL_OK;
    if (it.op != sop || (sop && (a.few_n < 1 || a.op_x == nullptr || a.op_x == a.few_x))) return BL_OK;
    acc_stride = std::max(acc_stride, a.nrows1);
    coef_stride = std::max(coef_stride, (a.nrows2 + kGroup - 1) / kGroup * kGroup);
  }
  // largest batch per launch whose per-run coefficient blocks still fit beside the ring (two blocks per SM)
  int per_launch = std::min(total, kStepBatch);
  while (per_launch > 1 && step_smem_bytes<T>(per_launch, acc_stride, coef_stride) > 112 * 1024) --per_launch;
  if (per_launch < 2) return BL_OK;
  BL_CHECK(set_smem(k_step_tma<T, TILE>, 112 * 1024));
  if (!step_fits<T>(blocks_per_sm())) return BL_OK;
  *done = true;
  const int grid = tma_grid<T>(n, TILE);
  const bool pdl = g_step_pdl_ok.load(std::memory_order_relaxed) != 0;
  for (int first = 0; first < total; first += per_launch) {
    StepBatch B;
    B.count = std::min(per_launch, total - first);
    B.acc_stride = acc_stride;
    B.coef_stride = coef_stride;
    double bytes = 0.0;
    for (int p = 0; p < B.count; ++p) {
      StepItem& it = items[first + p];
      StepArgs& a = it.a;
      const Common& c = *it.c;
      a.partials = c.partials_dots;
      a.partials0 = c.partials_few;
      a.red_g = c.red;
      a.partials_norm = c.partials_comb;
      for (Epi* e : {&a.epi0, &a.epi1, &a.epi2}) {
        e->red = c.red;
        e->scal = c.scal;
      }
      B.a[p] = a;
      bytes += it.bytes;
    }
    B.bar = items[first].c->counters + 8;
    B.exit_counter = items[first].c->counters + 9;
    B.reverse = next_direction();
    (void)next_direction();  // phase 2 walks the other way: the next streaming kernel starts where it ended
    if (sop) {
      B.op = *sop;
      B.reverse = 0;  // old rows first: what the producer copies under phase S is older than the predecessor
    }
    if (g_step_trace_next.load(std::memory_order_relaxed) >= 0) {
      const int slot = g_step_trace_next.fetch_add(1, std::memory_order_relaxed);
      B.trace_slot = slot < kTraceLaunches ? slot : -1;
    }
    const size_t smem = step_smem_bytes<T>(B.count, acc_stride, coef_stride);
    ProfScope prof(BL_PROF_FUSED, bytes, s);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kStreamThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 2 : 1;
    cudaError_t err = cudaLaunchKernelEx(&cfg, k_step_tma<T, TILE>, B);
    if (err != cudaSuccess && pdl) {  // cooperative + programmatic refused together: cooperative alone
      (void)cudaGetLastError();
      g_step_pdl_ok.store(0, std::memory_order_relaxed);
      cfg.numAttrs = 1;
      err = cudaLaunchKernelEx(&cfg, k_step_tma<T, TILE>, B);
    }
    BL_CUDA(err);
    BL_LAUNCHED();
  }
  return BL_OK;
}

template <typename T>
int launch_scale_copy(int64_t n, const T* x, double mul, const double* div_ptr, T* out, int64_t n_pad, cudaStream_t s) {
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(16 * sm_count(), (n_pad + 255) / 256));
  ProfScope prof(BL_PROF_OTHER, 2.0 * n * sizeof(T), s);
  k_scale_copy<T><<<blocks, 256, 0, s>>>(n, x, mul, div_ptr, out, n_pad);
  BL_LAUNCHED();
  return BL_OK;
}

RowBlock rows(const void* base, int64_t ld, int row0, int nrows, const double* coef = nullptr,
              double sign = 1.0, int coef0 = 0) {
  RowBlock b;
  b.base = base;
  b.ld = ld;
  b.row0 = row0;
  b.nrows = nrows;
  b.coef = coef;
  b.sign = sign;
  b.coef0 = coef0;
  return b;
}

VecTerm term(const void* ptr, double imm = 1.0, const double* coef_ptr = nullptr) {
  VecTerm t;
  t.ptr = ptr;
  t.coef_imm = imm;
  t.coef_ptr = coef_ptr;
  return t;
}

int check_basis(int dtype, int64_t n, int64_t K, int64_t ld, const void* Q) {
  BL_REQUIRE(dtype == BL_F32 || dtype == BL_F64, "dtype must be BL_F32 or BL_F64");
  BL_REQUIRE(n >= 1, "n must be positive");
  if (K < 1 || K > n) {
    set_error("Parameter depth " + std::to_string(K) + " is outside the expected range");
    return BL_EDEPTH;
  }
  BL_REQUIRE(ld >= n && (ld * dtype_size(dtype)) % 16 == 0, "ld must be >= n and a multiple of 16 bytes");
  BL_REQUIRE(reinterpret_cast<uintptr_t>(Q) % 16 == 0, "basis pointer must be 16-byte aligned");
  return BL_OK;
}

// BL_FWD_SYMMETRIC of the caller's flags (needs the second pass)
bool symmetric_forward(int flags) {
  return (flags & BL_FWD_SYMMETRIC) != 0 && (flags & BL_FWD_SECOND_PASS) != 0;
}

// ---------------------------------------------------------------------------------------
// One Arnoldi forward run, split at the matvec so that several runs (probes) can advance in lockstep
// and share ONE batched matvec per step (arnoldi_forward_t): begin(), then per step
// [q_i = v / length, v = A q_i] -> post(i), or the whole step in one k_step_tma launch (step_item).
template <typename T>
struct FwdRun {
  bl_operator_t* op;
  int dtype;
  int64_t n;
  int K;
  bool second_pass;
  const T* v;
  T* Q;
  int64_t ld;
  T* H;
  T* r;
  T* c_out;
  void* workspace;
  size_t wbytes;
  cudaStream_t s;
  Common c;
  Grid g;
  T* alt = nullptr;    // spare vector: the fused normalise + matvec cannot run in place
  // BL_FWD_SYMMETRIC: the first Gram-Schmidt pass (arnoldi.py:87-88) takes rows i-1 and i only -- for a
  // symmetric operand the other entries of h = Q^H (A q_i) are O(eps |A|) while Q stays orthonormal, and the
  // second pass (arnoldi.py:91-92) removes what they would have removed: v'' = (I - Q Q^H) v' either way.
  bool local_first = false;
  int first_lo(int i) const { return local_first ? std::max(0, i - 1) : 0; }
  T* r_out = nullptr;  // the caller's remainder buffer (`r` is the CURRENT vector and may be `alt`)

  T* q_row(int i) const { return Q + (int64_t)i * ld; }

  int finish() {
    if (r != r_out) {
      BL_CUDA(cudaMemcpyAsync(r_out, r, (size_t)n * sizeof(T), cudaMemcpyDeviceToDevice, s));
      std::swap(r, alt);
    }
    return BL_OK;
  }

  int begin() {
  Workspace w(workspace, wbytes);
  carve_common(w, K, c);
  alt = static_cast<T*>(w.take((size_t)ld * sizeof(T)));
  r_out = r;
  BL_REQUIRE(w.ok(), "workspace too small (bl_arnoldi_workspace_bytes)");
  g = pick_grid<T>(n);

  BL_CUDA(cudaMemsetAsync(c.counters, 0, 256, s));
  BL_CUDA(cudaMemsetAsync(H, 0, (size_t)K * K * sizeof(T), s));
  BL_CUDA(cudaMemcpyAsync(r, v, (size_t)n * sizeof(T), cudaMemcpyDeviceToDevice, s));

  {  // initlength = sqrt(v . v); c = 1/initlength                              arnoldi.py:66,75
    Epi e;
    e.mode = EPI_INIT_NORM;
    e.m = 1;
    e.out_t = c_out;
    BL_CHECK(launch_dots<T>(g, c, rows(r, n, 0, 1), r, n, e, s));
  }
    return BL_OK;
  }
  // epilogue of the first pass's dots: h = Q^H v over the active rows        arnoldi.py:87
  Epi pass_a_epi(int i) const {
    Epi e;
    e.mode = EPI_FWD_A;
    e.i = i;
    e.K = K;
    e.j0 = first_lo(i);
    e.m = i + 1 - e.j0;
    e.H = H;
    e.coef = c.coefA;
    return e;
  }
  // epilogue of the second pass's dots: coefB = Q^H v'; with the local first pass also H[j < i-1, i]
  Epi pass_b_epi(int i) const {
    Epi e;
    e.mode = EPI_FWD_B;
    e.m = i + 1;
    e.coef = c.coefB;
    e.i = i;
    e.K = K;
    e.j0 = first_lo(i);
    e.H = local_first ? H : nullptr;
    return e;
  }
  // epilogue of the last combine: length = sqrt(v . v); h[i+1] = length       arnoldi.py:95-98
  Epi norm_epi(int i) const {
    Epi e;
    e.mode = EPI_FWD_NORM;
    e.i = i;
    e.K = K;
    e.H = H;
    return e;
  }
  int pre(int i) {
    T* qi = Q + (int64_t)i * ld;
    // v /= length; Q[:, i] = v                                                 arnoldi.py:80-81
    BL_CHECK(launch_scale_copy<T>(n, r, 1.0, c.scal + S_LEN, qi, ld, s));
    return BL_OK;
  }
  // symmetric loop (local_first), step i as ONE k_step_tma item on x = A q_i, updated in place:
  // h = (q_{i-1}, q_i)^H x | x' = x - h_{i-1} q_{i-1} - h_i q_i, h2 = Q^H x' | x'' = x' - Q h2, ||x''||   arnoldi.py:87-98
  StepItem step_item(int i, T* x) const {
    const int m = i + 1, j0 = first_lo(i);
    StepItem item{};
    item.c = &c;
    StepArgs& a = item.a;
    a.n = n;
    a.few_n = m - j0;
    for (int j = j0; j < m; ++j) a.few_row[j - j0] = q_row(j);
    a.few_x = x;
    a.epi0 = pass_a_epi(i);
    a.out1 = x;
    a.vec[a.nvec++] = term(x);
    for (int j = j0; j < m; ++j) a.vec[a.nvec++] = term(q_row(j), -1.0, c.coefA + j);
    a.src1 = row_source(rows(Q, ld, 0, m), nullptr, sizeof(T));
    a.nrows1 = m;
    a.epi1 = pass_b_epi(i);
    a.src2 = a.src1;
    a.nrows2 = m;
    a.coef2 = c.coefB;
    a.sign2 = -1.0;
    a.out2 = x;
    a.norm = 1;
    a.epi2 = norm_epi(i);
    a.wait_row = i;  // row i is the operator kernel's output (fused normalise + matvec)
    item.bytes = (double)((m - j0 + 1) + (m + a.nvec + 1) + (m + 2)) * n * sizeof(T);
    return item;
  }
  // The same with the operator call in the launch (phase S): q_i = v / length, x = A q_i, then the step.  x is the
  // spare buffer (the gathers of phase S read the whole input while other blocks write the output): after the
  // launch the caller swaps `r` and `alt`.                                                  arnoldi.py:80-98
  StepItem fused_item(int i, const StepOp* sop) const {
    StepItem item = step_item(i, alt);
    item.op = sop;
    item.a.op_x = r;
    item.a.op_q = q_row(i);
    item.a.op_len = c.scal + S_LEN;
    item.a.wait_row = std::max(0, i - 1);  // rows i-1 (the predecessor's phase S) and i (this launch's)
    item.bytes += op->matvec_bytes(dtype) + 1.0 * n * sizeof(T);
    return item;
  }
  // Step i as separate launches: the general loop, which for the symmetric loop is step_item(i) lowered -- phase 0
  // is the first dots launch, phase 1 k_xdots_tma (n below the TMA threshold: the general kernels), phase 2 the
  // second pass's combine.
  int post(int i) {
    const int m = i + 1, j0 = first_lo(i);
    BL_CHECK(launch_dots<T>(g, c, rows(Q, ld, j0, m - j0), r, n, pass_a_epi(i), s));
    bool fused = false;
    if (local_first) {
      // v = v - h_{i-1} q_{i-1} - h_i q_i is a three-vector combination, and h2 = Q^H v streams every active row
      // once (no row is needed twice: nothing stays resident)                 arnoldi.py:88,92
      BL_CHECK(launch_xdots<T>(c, step_item(i, r).a, s, &fused));
    }
    if (second_pass && !fused) {
      // v = v - Q h and, from the same read of Q, h2 = Q^H v (the second pass's coefficients;
      // h itself is not updated, arnoldi.py:92)
      FusedSpec f;
      f.n = n;
      f.out = r;
      f.nvec = 1;
      f.vec[0] = term(r);
      f.res = rows(Q, ld, 0, m, c.coefA, -1.0);
      f.epi = pass_b_epi(i);
      BL_CHECK(launch_fused<T>(c, f, dtype, s, &fused));
    }
    if (!fused) {  // v = v - Q h                                               arnoldi.py:88
      CombineArgs a;
      a.n = n;
      a.out = r;
      a.nvec = 1;
      a.vec[0] = term(r);
      a.blk[0] = rows(Q, ld, j0, m - j0, c.coefA, -1.0, j0);
      a.epi = norm_epi(i);
      BL_CHECK(launch_combine<T>(g, c, a, !second_pass, s));
      if (second_pass) {
        BL_CHECK(launch_dots<T>(g, c, rows(Q, ld, 0, m), r, n, pass_b_epi(i), s));
      }
    }
    if (second_pass) {  // v = v - Q (Q^H v)                                    arnoldi.py:91-92
      CombineArgs a;
      a.n = n;
      a.out = r;
      a.nvec = 1;
      a.vec[0] = term(r);
      a.blk[0] = rows(Q, ld, 0, m, c.coefB, -1.0);
      a.epi = norm_epi(i);
      BL_CHECK(launch_combine<T>(g, c, a, true, s));
    }
    return BL_OK;
  }
};

// P independent runs in lockstep (P = 1: bl_arnoldi_forward): per step one batched matvec for all of them, and
// for the symmetric loop the Gram-Schmidt step of all of them in one launch per kStepBatch runs.  Each run owns
// `per` bytes of the workspace.
template <typename T>
int arnoldi_forward_t(bl_operator_t* op, int dtype, int64_t n, int K, int flags, int P, const void* v_, int64_t ldv,
                      void* Q_, int64_t ld, void* H_, void* r_, void* c_, void* workspace, size_t per, cudaStream_t s) {
  const T* v = static_cast<const T*>(v_);
  T *Q = static_cast<T*>(Q_), *H = static_cast<T*>(H_), *r = static_cast<T*>(r_), *c_out = static_cast<T*>(c_);
  const bool symmetric = symmetric_forward(flags);
  std::vector<FwdRun<T>> runs;
  for (int p = 0; p < P; ++p) {
    runs.push_back(FwdRun<T>{op, dtype, n, K, (flags & BL_FWD_SECOND_PASS) != 0, v + (int64_t)p * ldv, Q + (int64_t)p * K * ld, ld,
                             H + (int64_t)p * K * K, r + (int64_t)p * ld, c_out + p,
                             static_cast<char*>(workspace) + per * p, per, s, {}, {}});
    runs.back().local_first = symmetric;
    BL_CHECK(runs.back().begin());
  }
  std::vector<const void*> in(P);
  std::vector<void*> out(P);
  std::vector<const double*> lens(P);
  std::vector<void*> qout(P);
  std::vector<StepItem> items(P);
  StepOp sop;
  const bool fuse = symmetric && make_step_op(op, dtype, false, true, n, ld, &sop);
  for (int i = 0; i < K; ++i) {
    bool stepped = false;
    if (fuse) {  // operator call + Gram-Schmidt step of all runs in one launch per kStepBatch runs
      sop.wait_first = i == 0;
      for (int p = 0; p < P; ++p) items[p] = runs[p].fused_item(i, &sop);
      for (StepItem& it : items) it.bytes += (op->matvec_batch_bytes(dtype, P) - P * op->matvec_bytes(dtype)) / P;
      BL_CHECK(launch_step<T>(items, s, &stepped));
      if (stepped) {
        for (FwdRun<T>& run : runs) std::swap(run.r, run.alt);
        continue;
      }
    }
    int rc = -1;
    {  // q_i = v / length and v = A q_i of every run in one batched operator call     arnoldi.py:80-84
      for (int p = 0; p < P; ++p) {
        in[p] = runs[p].r;
        lens[p] = runs[p].c.scal + S_LEN;
        qout[p] = runs[p].q_row(i);
        out[p] = runs[p].alt;
      }
      ProfScope prof(BL_PROF_MATVEC, op->matvec_batch_bytes(dtype, P) + 1.0 * P * n * sizeof(T), s);
      rc = op->matvec_normalised_batch(dtype, P, in.data(), lens.data(), qout.data(), ld, out.data(), s);
    }
    if (rc == BL_OK) {
      for (int p = 0; p < P; ++p) std::swap(runs[p].r, runs[p].alt);
    } else if (rc == -1) {
      for (int p = 0; p < P; ++p) {
        BL_CHECK(runs[p].pre(i));
        in[p] = runs[p].q_row(i);
        out[p] = runs[p].r;
      }
      ProfScope prof(BL_PROF_MATVEC, op->matvec_batch_bytes(dtype, P), s);
      BL_CHECK(op->matvec_batch(dtype, P, in.data(), out.data(), s));
    } else {
      return rc;
    }
    if (symmetric) {  // the Gram-Schmidt step of all runs in one launch per kStepBatch runs (k_step_tma)
      for (int p = 0; p < P; ++p) items[p] = runs[p].step_item(i, runs[p].r);
      BL_CHECK(launch_step<T>(items, s, &stepped));
      if (stepped) continue;
    }
    for (int p = 0; p < P; ++p) BL_CHECK(runs[p].post(i));
  }
  for (int p = 0; p < P; ++p) BL_CHECK(runs[p].finish());
  return BL_OK;
}

// BL_ADJ_SYMMETRIC of the caller's flags
bool symmetric_shortcut(int flags) { return (flags & BL_ADJ_SYMMETRIC) != 0; }

// ---------------------------------------------------------------------------------------
// One Arnoldi adjoint run, split at the operator call (see FwdRun): begin(), then for idx = K-1..0
// pre(idx) -> [z = A^T Lambda[idx] (+ parameter cotangent)] -> post(idx), then end().
template <typename T>
struct AdjRun {
  bl_operator_t* op;
  int dtype;
  int64_t n;
  int K;
  bool reortho_full;
  const T* Q;
  int64_t ld;
  const T* H;
  const T* r;
  const T* c_in;
  const T* dQ;
  const T* dH;
  const T* dr;
  const T* dc;
  T* dv;
  T* Lambda;
  void* workspace;
  size_t wbytes;
  cudaStream_t s;
  Common c;
  Grid g;
  double *eta = nullptr, *Gamma = nullptr, *PiGamma = nullptr, *Gmat = nullptr, *gram_partial = nullptr;
  int gram_parts = 0;
  T *z = nullptr, *lam = nullptr;
  bool defer_grad = false;
  // BL_ADJ_SYMMETRIC: the operand is symmetric, so H is tridiagonal up to rounding (full
  // re-orthogonalisation keeps |H[idx, j]| = O(eps |A|) for j > idx+1) and `Lambda beta_plus`
  // (arnoldi.py:218) reduces to its one O(1) term, -H[idx, idx+1] Lambda[idx+1]: K-idx-2 basis rows
  // per step are not read.  SURVEY Appendix B7; off unless the caller says the operand is symmetric.
  bool symmetric = false;
  // BL_ADJ_TRIDIAG_COTANGENT on top of it, no dQ: Gamma is banded.  After the re-projection
  // Q_{<=idx+1}^T lambda = dH[:idx+2, idx] exactly (arnoldi.py:201-204), and A q_j = Q H[:, j], so
  // Gamma[idx, j] = (H dH^T - dH^T H)[idx, j] up to rounding -- zero for j < idx-2 when H and dH are
  // tridiagonal.  The dots `Q^T (A^T lambda)` (arnoldi.py:213) then need rows idx-2..idx only and
  // `Q (Gamma + Gamma^T)[idx]` (arnoldi.py:217) rows idx-2..idx+2: the sweep reads the active basis
  // twice per step (the re-projection itself), like the forward's Gram-Schmidt passes.
  bool tridiag_cot = false, banded = false;
  int band_lo(int idx) const { return banded ? std::max(0, idx - 2) : 0; }
  int band_hi(int idx) const { return banded ? std::min(idx + 3, K) : K; }  // exclusive

  const T* q_row(int idx) const { return Q + (int64_t)idx * ld; }
  T* lam_row(int idx) const { return Lambda + (int64_t)idx * ld; }
  // terms of `- Lambda beta_plus`: every later row of Lambda, or (symmetric) row idx+1 as a vector term
  int lam_rows_streamed(int idx) const { return symmetric ? 0 : K - idx - 1; }
  // Vector terms of the back-substitution (its basis rows follow): dQ[idx] when given, eta[idx] r, -alpha Lambda[idx],
  // A^T lambda and, for a symmetric operand, -beta_plus Lambda[idx+1].  Returns their count.   arnoldi.py:212-218
  int back_terms(int idx, VecTerm* vec) const {
    int nv = 0;
    if (dQ) vec[nv++] = term(dQ + (int64_t)idx * ld);
    vec[nv++] = term(r, 1.0, c.scal + S_ETA_IDX);
    vec[nv++] = term(lam_row(idx), 1.0, c.scal + S_NEG_ALPHA);
    vec[nv++] = term(z);
    if (symmetric && idx + 1 < K) vec[nv++] = term(lam_row(idx + 1), 1.0, c.coefC + idx + 1);
    return nv;
  }
  // epilogue of the dots with A^T lambda: Gamma[idx, :] and the coefficients of the back-substitution   arnoldi.py:212-218
  Epi gamma_epi(int idx) const {
    Epi e;
    e.mode = EPI_ADJ_GAMMA;
    e.i = idx;
    e.K = K;
    e.j0 = band_lo(idx);
    e.m = idx + 1 - e.j0;
    e.Hc = H;
    e.Gamma = Gamma;
    e.PiGamma = PiGamma;
    e.eta = eta;
    e.coef = c.coefB;
    e.coef2 = c.coefC;
    return e;
  }
  // epilogue of the re-projection dots t = P lambda, rows <= idx+1 of P = Q^T: coefA = p - t   arnoldi.py:201-204
  Epi reproj_epi(int idx) const {
    Epi e;
    e.mode = EPI_ADJ_REPROJ;
    e.i = idx;
    e.K = K;
    e.m = std::min(idx + 2, K);
    e.dH = dH;
    e.coef = c.coefA;
    return e;
  }
  // What the step of idx+1 already did of pre(idx): k_step_tma wrote Lambda[idx] (its phase 2), or the separate
  // launches computed the re-projection coefficients (phase 1); otherwise pre(idx) runs both launches.
  enum Ahead { kNothing, kReproj, kLambdaRow };
  Ahead ahead = kNothing;

  int begin() {
  Workspace w(workspace, wbytes);
  carve_common(w, K, c);
  eta = static_cast<double*>(w.take((size_t)K * 8));
  Gamma = static_cast<double*>(w.take((size_t)K * K * 8));
  PiGamma = static_cast<double*>(w.take((size_t)K * K * 8));
  Gmat = static_cast<double*>(w.take((size_t)K * K * 8));
  gram_parts = (int)gram_parts_for(n, K);
  gram_partial = static_cast<double*>(w.take((size_t)gram_parts * K * K * 8));
  z = static_cast<T*>(w.take((size_t)ld * sizeof(T)));
  lam = static_cast<T*>(w.take((size_t)ld * sizeof(T)));
  BL_REQUIRE(w.ok(), "workspace too small (bl_arnoldi_workspace_bytes)");
  g = pick_grid<T>(n);
  defer_grad = op->deferred_grad(dtype);
  banded = symmetric && tridiag_cot && reortho_full && dQ == nullptr;

  BL_CUDA(cudaMemsetAsync(c.counters, 0, 256, s));
  BL_CUDA(cudaMemsetAsync(Gamma, 0, (size_t)K * K * 8, s));
  if (ld > n)  // row buffers are zero-padded up to ld (contract of the TMA-staged kernels)
    BL_CUDA(cudaMemset2DAsync(Lambda + n, (size_t)ld * sizeof(T), 0, (size_t)(ld - n) * sizeof(T), (size_t)K, s));

  // eta = dH e_K - Q^T dr ; lambda_K = dr + Q eta                             arnoldi.py:119-120
  {
    Epi e;
    e.mode = EPI_ADJ_ETA;
    e.K = K;
    e.dH = dH;
    e.eta = eta;
    e.coef = c.coefA;
    if (dr) {
      e.m = K;
      BL_CHECK(launch_dots<T>(g, c, rows(Q, ld, 0, K), dr, n, e, s));
    } else {
      e.m = 0;
      e.red = c.red;
      e.scal = c.scal;
      k_epilogue_only<T><<<1, 256, 0, s>>>(e);
      BL_LAUNCHED();
    }
    CombineArgs a;
    a.n = n;
    a.out = lam;
    if (dr) {
      a.nvec = 1;
      a.vec[0] = term(dr);
    }
    a.blk[0] = rows(Q, ld, 0, K, c.coefA, 1.0);
    BL_CHECK(launch_combine<T>(g, c, a, false, s));
  }
  // Pi_gamma = -dc c e1 e1^T + H dH^T - dQ^T Q                                arnoldi.py:127
  if (dQ) {
    constexpr int TK = 32, KB = 128;  // blocks of at most 128 x 128 entries of dQ^T Q per launch: any Krylov depth
    const size_t smem = 2 * (size_t)TK * kGramKP * sizeof(T);
    BL_CHECK(set_smem(k_gram_partial<T, TK>, smem));
    for (int a0 = 0; a0 < K; a0 += KB)
      for (int b0 = 0; b0 < K; b0 += KB) {
        k_gram_partial<T, TK><<<gram_parts, kGramThreads, smem, s>>>(std::min(KB, K - a0), std::min(KB, K - b0), K, n,
                                                            dQ + (int64_t)a0 * ld, Q + (int64_t)b0 * ld, ld,
                                                            gram_partial + (size_t)a0 * K + b0);
        BL_LAUNCHED();
      }
    k_gram_reduce<<<(K * K + 255) / 256, 256, 0, s>>>(K * K, gram_parts, gram_partial, Gmat);
    BL_LAUNCHED();
    BL_CHECK(sharded_sum(Gmat, (int)(K * K), s));
  }
  {
    dim3 grid(K, (K + 127) / 128);
    k_pi_gamma<T><<<grid, 128, 0, s>>>(K, H, dH, dc, c_in, dQ ? Gmat : nullptr, PiGamma);
    BL_LAUNCHED();
  }

    return BL_OK;
  }
  // Lambda[idx] = lambda + Q (p - P lambda): phase 2 of the step of idx+1        arnoldi.py:201-204, 216
  int pre(int idx) {
    T* Lrow = Lambda + (int64_t)idx * ld;
    if (ahead == kLambdaRow) return BL_OK;
    if (reortho_full) {
      // lambda -= P^T (P lambda) - P^T p, rows <= idx+1 of P = Q^T              arnoldi.py:201-204
      const int mact = std::min(idx + 2, K);
      if (ahead != kReproj) BL_CHECK(launch_dots<T>(g, c, rows(Q, ld, 0, mact), lam, n, reproj_epi(idx), s));
      CombineArgs a;
      a.n = n;
      a.out = Lrow;  // Lambda[:, idx] = lambda                                   arnoldi.py:216
      a.nvec = 1;
      a.vec[0] = term(lam);
      a.blk[0] = rows(Q, ld, 0, mact, c.coefA, 1.0);
      BL_CHECK(launch_combine<T>(g, c, a, false, s));
    } else {
      BL_CHECK(launch_scale_copy<T>(n, lam, 1.0, nullptr, Lrow, n, s));
    }
    return BL_OK;
  }
  // banded Gamma (idx > 0), step idx as ONE k_step_tma item: Gamma row from the dots of z with rows idx-2..idx |
  // back-substitution and the next step's re-projection dots | Lambda[idx-1] = lambda + Q (p - P lambda)
  //                                                                             arnoldi.py:212-219, 201-204, 216
  StepItem step_item(int idx) const {
    const int j0 = band_lo(idx);
    StepItem item{};
    item.c = &c;
    StepArgs& a = item.a;
    a.n = n;
    a.few_n = idx + 1 - j0;
    for (int j = j0; j <= idx; ++j) a.few_row[j - j0] = q_row(j);
    a.few_x = z;
    a.epi0 = gamma_epi(idx);
    a.out1 = lam;
    a.nvec = back_terms(idx, a.vec);
    for (int j = j0; j < band_hi(idx); ++j) a.vec[a.nvec++] = term(q_row(j), 1.0, c.coefB + j);
    a.out_div_ptr = c.scal + S_BETA_MINUS;
    a.src1 = row_source(rows(Q, ld, 0, idx + 1), nullptr, sizeof(T));
    a.nrows1 = idx + 1;
    a.epi1 = reproj_epi(idx - 1);
    a.src2 = a.src1;  // rows <= (idx-1)+1 of P = Q^T
    a.nrows2 = idx + 1;
    a.coef2 = c.coefA;
    a.sign2 = 1.0;
    a.out2 = lam_row(idx - 1);
    a.norm = 0;
    item.bytes = (double)((a.few_n + 1) + (idx + 1 + a.nvec + 1) + (idx + 1 + 2)) * n * sizeof(T);
    return item;
  }
  // The same with z = A^T Lambda[idx] in the launch (phase S; deferred parameter cotangent only).
  StepItem fused_item(int idx, const StepOp* sop) const {
    StepItem item = step_item(idx);
    item.op = sop;
    item.a.op_x = lam_row(idx);
    item.bytes += op->apply_transpose_bytes(dtype);
    return item;
  }
  // Step idx as separate launches: the general loop, which for banded Gamma is step_item(idx) lowered -- phase 0 is
  // the Gamma dots, phase 1 k_xdots_tma (n below the TMA threshold: the general kernels), phase 2 pre(idx - 1).
  int post(int idx) {
    // lambda = (Pi_xi[idx] + Q gamma_row - alpha lambda + A^T lambda - Lambda beta_plus) / beta_minus
    BL_CHECK(launch_dots<T>(g, c, rows(Q, ld, band_lo(idx), idx + 1 - band_lo(idx)), z, n, gamma_epi(idx), s));
    bool reproj = false;
    if (banded && idx > 0) {
      // banded Gamma: the back-substitution combines nine vectors at most, and the NEXT step's re-projection dots
      // t = P lambda stream rows 0..idx once                                    arnoldi.py:202,217-219
      BL_CHECK(launch_xdots<T>(c, step_item(idx).a, s, &reproj));
    }
    if (!reproj && reortho_full && idx > 0) {
      // ... fused with the NEXT step's re-projection dots t = P lambda (rows 0..idx of Q are the
      // active rows of P at idx-1): one read of those rows serves both          arnoldi.py:202,217-219
      FusedSpec f;
      f.n = n;
      f.out = lam;
      f.nvec = back_terms(idx, f.vec);
      // banded: rows idx+1, idx+2 ride as resident rows (their two extra dots are not read by the epilogue)
      const int nres = banded ? band_hi(idx) : idx + 1;
      f.res = rows(Q, ld, 0, nres, c.coefB, 1.0);
      f.str0 = rows(Q, ld, nres, K - nres, c.coefB, 1.0, nres);
      f.str1 = rows(Lambda, ld, idx + 1, lam_rows_streamed(idx), c.coefC, 1.0, idx + 1);
      f.rows_total0 = K;
      f.rows_total1 = K;
      f.out_div_ptr = c.scal + S_BETA_MINUS;
      f.epi = reproj_epi(idx - 1);
      BL_CHECK(launch_fused<T>(c, f, dtype, s, &reproj));
    }
    if (!reproj) {
      CombineArgs a;
      a.n = n;
      a.out = lam;
      a.nvec = back_terms(idx, a.vec);
      a.blk[0] = rows(Q, ld, band_lo(idx), band_hi(idx) - band_lo(idx), c.coefB, 1.0, band_lo(idx));
      a.blk[1] = rows(Lambda, ld, idx + 1, lam_rows_streamed(idx), c.coefC, 1.0, idx + 1);
      a.out_div_ptr = c.scal + S_BETA_MINUS;
      BL_CHECK(launch_combine<T>(g, c, a, false, s));
    }
    ahead = reproj ? kReproj : kNothing;
    return BL_OK;
  }
  int end() {
  // dv = lambda * c                                                              arnoldi.py:166
  k_load_scalar<T><<<1, 1, 0, s>>>(c_in, c.scal + S_C);
  BL_LAUNCHED();
  {
    CombineArgs a;
    a.n = n;
    a.out = dv;
    a.nvec = 1;
    a.vec[0] = term(lam, 1.0, c.scal + S_C);
    BL_CHECK(launch_combine<T>(g, c, a, false, s));
  }
    return BL_OK;
  }
};

// P independent adjoint runs in lockstep (P = 1: bl_arnoldi_adjoint; the bases of P forward runs are contiguous:
// Q[p][K][ld]): one batched A^T Lambda per step, and ONE batched parameter-cotangent pass over all P*K
// (lambda, q) pairs.  Each run owns `per` bytes of the workspace.
template <typename T>
int arnoldi_adjoint_t(bl_operator_t* op, int dtype, int64_t n, int K, int flags, int P, const void* Q_, int64_t ld,
                      const void* H_, const void* r_, const void* c_, const void* dQ_, const void* dH_, const void* dr_,
                      const void* dc_, void* dv_, int64_t lddv, void* Lambda_, void* workspace, size_t per,
                      cudaStream_t s) {
  const T *Q = static_cast<const T*>(Q_), *H = static_cast<const T*>(H_), *r = static_cast<const T*>(r_);
  const T *c_in = static_cast<const T*>(c_), *dQ = static_cast<const T*>(dQ_), *dH = static_cast<const T*>(dH_);
  const T *dr = static_cast<const T*>(dr_), *dc = static_cast<const T*>(dc_);
  T *dv = static_cast<T*>(dv_), *Lambda = static_cast<T*>(Lambda_);
  const bool deferred = op->deferred_grad(dtype);
  std::vector<AdjRun<T>> runs;
  std::vector<const void*> in(P);
  std::vector<void*> out(P);
  for (int p = 0; p < P; ++p) {
    runs.push_back(AdjRun<T>{op, dtype, n, K, (flags & BL_ADJ_REORTHO_FULL) != 0, Q + (int64_t)p * K * ld, ld, H + (int64_t)p * K * K,
                             r + (int64_t)p * ld, c_in + p, dQ ? dQ + (int64_t)p * K * ld : nullptr,
                             dH + (int64_t)p * K * K, dr ? dr + (int64_t)p * ld : nullptr, dc ? dc + p : nullptr,
                             dv + (int64_t)p * lddv, Lambda + (int64_t)p * K * ld,
                             static_cast<char*>(workspace) + per * p, per, s, {}, {}});
    runs.back().symmetric = symmetric_shortcut(flags);
    runs.back().tridiag_cot = (flags & BL_ADJ_TRIDIAG_COTANGENT) != 0;
    BL_CHECK(runs.back().begin());
    out[p] = runs[p].z;
  }
  std::vector<StepItem> items(P);
  StepOp sop;
  const bool fuse = deferred && runs[0].banded && make_step_op(op, dtype, true, false, n, ld, &sop);
  for (int idx = K - 1; idx >= 0; --idx) {
    for (int p = 0; p < P; ++p) {
      BL_CHECK(runs[p].pre(idx));
      in[p] = runs[p].lam_row(idx);
    }
    const bool banded_step = runs[0].banded && idx > 0;  // the step has a k_step_tma form (AdjRun::step_item)
    bool stepped = false;
    if (fuse && banded_step) {  // A^T lambda + back-substitution + the next re-projection of all runs in one launch
      sop.wait_first = idx == K - 1;
      for (int p = 0; p < P; ++p) items[p] = runs[p].fused_item(idx, &sop);
      for (StepItem& it : items) it.bytes += (op->matvec_batch_bytes(dtype, P) - P * op->matvec_bytes(dtype)) / P;
      BL_CHECK(launch_step<T>(items, s, &stepped));
    }
    if (!stepped) {
      {  // (A^T lambda, dparams += ...) = vjp of matvec at (q_idx, params)          arnoldi.py:207-209
        ProfScope prof(BL_PROF_VJP, deferred ? op->matvec_batch_bytes(dtype, P) : op->vjp_bytes(dtype) * P, s);
        if (deferred) {  // A^T lambda only; the parameter cotangent of all steps follows in one batched pass
          BL_CHECK(op->apply_transpose_batch(dtype, P, in.data(), out.data(), s));
        } else {  // the parameter cotangent accumulates in the operator over steps and runs (a sum over the batch)
          for (int p = 0; p < P; ++p) BL_CHECK(op->vjp(dtype, runs[p].q_row(idx), in[p], out[p], s));
        }
      }
      if (banded_step) {  // back-substitution, re-projection dots and the next Lambda row of all runs in one launch
        for (int p = 0; p < P; ++p) items[p] = runs[p].step_item(idx);
        BL_CHECK(launch_step<T>(items, s, &stepped));
      }
    }
    for (AdjRun<T>& run : runs) {
      if (stepped)
        run.ahead = AdjRun<T>::kLambdaRow;  // the launch also wrote Lambda[idx - 1] (its phase 2)
      else
        BL_CHECK(run.post(idx));
    }
  }
  if (deferred) {  // dparams = sum_idx d<Lambda[idx], A(Q[idx]; params)>/dparams   arnoldi.py:207-209, 168
    ProfScope prof(BL_PROF_VJP, op->vjp_batch_bytes(dtype, P * K), s);
    BL_CHECK(op->vjp_batch(dtype, Q, ld, Lambda, ld, P * K, s));
  }
  for (int p = 0; p < P; ++p) {
    // dv = lambda * c is written with 16-byte stores: a row of the caller's (count, lddv) array that is not aligned
    // (lddv = n, n odd) goes through the run's scratch vector
    T* dst = runs[p].dv;
    const bool misaligned = reinterpret_cast<uintptr_t>(dst) % 16 != 0;
    if (misaligned) runs[p].dv = runs[p].z;
    BL_CHECK(runs[p].end());
    if (misaligned) BL_CUDA(cudaMemcpyAsync(dst, runs[p].z, (size_t)n * sizeof(T), cudaMemcpyDeviceToDevice, s));
  }
  return BL_OK;
}

// ---------------------------------------------------------------------------------------
template <typename T>
int lanczos3_forward_t(bl_operator_t* op, int dtype, int64_t n, int K, const T* v, T* xs, int64_t ld,
                       T* alphas, T* betas, void* workspace, size_t wbytes, cudaStream_t s) {
  Workspace w(workspace, wbytes);
  Common c;
  carve_common(w, K, c);
  T* wv = static_cast<T*>(w.take((size_t)ld * sizeof(T)));
  BL_REQUIRE(w.ok(), "workspace too small (bl_lanczos3_workspace_bytes)");
  const Grid g = pick_grid<T>(n);
  BL_CUDA(cudaMemsetAsync(c.counters, 0, 256, s));
  {  // v0 = vec / ||vec||                                                        lanczos.py:222
    Epi e;
    e.mode = EPI_INIT_NORM;
    e.m = 1;
    BL_CHECK(launch_dots<T>(g, c, rows(v, n, 0, 1), v, n, e, s));
    BL_CHECK(launch_scale_copy<T>(n, v, 1.0, c.scal + S_LEN, xs, ld, s));
  }
  for (int i = 0; i < K; ++i) {
    const T* xi = xs + (int64_t)i * ld;
    BL_CHECK(op->matvec(dtype, xi, wv, s));
    {  // a = x . (A x)                                                           lanczos.py:256,280
      Epi e;
      e.mode = EPI_L3_ALPHA;
      e.i = i;
      e.m = 1;
      e.out_t = alphas;
      e.coef = c.coefA;
      BL_CHECK(launch_dots<T>(g, c, rows(xs, ld, i, 1), wv, n, e, s));
    }
    {  // r = A x - a x - b x_prev ; b = ||r||                                    lanczos.py:281-283
      CombineArgs a;
      a.n = n;
      a.out = wv;
      a.nvec = 1;
      a.vec[0] = term(wv);
      a.blk[0] = i == 0 ? rows(xs, ld, 0, 1, c.coefA, 1.0) : rows(xs, ld, i - 1, 2, c.coefA, 1.0);
      a.epi.mode = EPI_L3_BETA;
      a.epi.i = i;
      a.epi.out_t = betas;
      BL_CHECK(launch_combine<T>(g, c, a, true, s));
    }
    // x_next = r / b                                                              lanczos.py:284
    BL_CHECK(launch_scale_copy<T>(n, wv, 1.0, c.scal + S_LEN, xs + (int64_t)(i + 1) * ld, ld, s));
  }
  return BL_OK;
}

template <typename T>
int lanczos3_adjoint_t(bl_operator_t* op, int dtype, int64_t n, int K, const T* xs, int64_t ld,
                       const T* alphas, const T* betas, const T* dxs, const T* dalphas, const T* dbetas,
                       const T* vnorm, T* dv, void* workspace, size_t wbytes, cudaStream_t s) {
  Workspace w(workspace, wbytes);
  Common c;
  carve_common(w, K, c);
  T* xi = static_cast<T*>(w.take((size_t)ld * sizeof(T)));
  T* lamA = static_cast<T*>(w.take((size_t)ld * sizeof(T)));
  T* lamB = static_cast<T*>(w.take((size_t)ld * sizeof(T)));
  T* wv = static_cast<T*>(w.take((size_t)ld * sizeof(T)));
  BL_REQUIRE(w.ok(), "workspace too small (bl_lanczos3_workspace_bytes)");
  const Grid g = pick_grid<T>(n);
  BL_CUDA(cudaMemsetAsync(c.counters, 0, 256, s));
  // init: xi = -dxs[K], lambda_plus = 0                                          lanczos.py:303
  if (dxs)
    BL_CHECK(launch_scale_copy<T>(n, dxs + (int64_t)K * ld, -1.0, nullptr, xi, n, s));
  else
    BL_CUDA(cudaMemsetAsync(xi, 0, (size_t)n * sizeof(T), s));
  T* lam_plus = lamA;
  T* lam = lamB;
  BL_CUDA(cudaMemsetAsync(lam_plus, 0, (size_t)n * sizeof(T), s));
  for (int k = K - 1; k >= 0; --k) {
    {  // lambda_plus . x_k
      Epi e;
      e.mode = EPI_L3_ADJ_DOT;
      e.m = 1;
      e.slot = S_DOT0;
      BL_CHECK(launch_dots<T>(g, c, rows(xs, ld, k, 1), lam_plus, n, e, s));
    }
    {  // x_k . xi, x_{k+1} . xi -> mu, nu                                        lanczos.py:322-324
      Epi e;
      e.mode = EPI_L3_ADJ_MUNU;
      e.i = k;
      e.m = 2;
      e.in_t = dalphas;
      e.in_t2 = dbetas;
      e.in_t3 = alphas;
      e.in_t4 = betas;
      e.coef = c.coefA;
      e.coef2 = c.coefB;
      BL_CHECK(launch_dots<T>(g, c, rows(xs, ld, k, 2), xi, n, e, s));
    }
    {  // lambda = -xi/b + mu x_{k+1} + nu x_k                                    lanczos.py:325
      CombineArgs a;
      a.n = n;
      a.out = lam;
      a.nvec = 1;
      a.vec[0] = term(xi, 1.0, c.scal + S_INV_B);
      a.blk[0] = rows(xs, ld, k, 2, c.coefA, 1.0);
      BL_CHECK(launch_combine<T>(g, c, a, false, s));
    }
    // A lambda and dparams += d<x_k, A(lambda)>/dparams                          lanczos.py:328-329
    BL_CHECK(op->matvec(dtype, lam, wv, s));
    BL_CHECK(op->vjp(dtype, lam, xs + (int64_t)k * ld, nullptr, s));
    {  // xi = -dx_k - A lambda + a lambda + b lambda_plus - b nu x_{k+1}         lanczos.py:332
      CombineArgs a;
      a.n = n;
      a.out = xi;
      int nv = 0;
      if (dxs) a.vec[nv++] = term(dxs + (int64_t)k * ld, -1.0);
      a.vec[nv++] = term(wv, -1.0);
      a.vec[nv++] = term(lam, 1.0, c.scal + S_A);
      a.vec[nv++] = term(lam_plus, 1.0, c.scal + S_B);
      a.nvec = nv;
      a.blk[0] = rows(xs, ld, k, 2, c.coefB, 1.0);
      BL_CHECK(launch_combine<T>(g, c, a, false, s));
    }
    std::swap(lam, lam_plus);
  }
  {  // grad_initvec = ((xi . x0) x0 - xi) / ||v||   (xi is what the reference calls lambda_1)  :311
    Epi e;
    e.mode = EPI_L3_ADJ_FINAL;
    e.m = 1;
    e.in_t = vnorm;
    e.coef = c.coefA;
    BL_CHECK(launch_dots<T>(g, c, rows(xs, ld, 0, 1), xi, n, e, s));
    CombineArgs a;
    a.n = n;
    a.out = dv;
    a.nvec = 1;
    a.vec[0] = term(xi, 1.0, c.scal + S_TMP0);
    a.blk[0] = rows(xs, ld, 0, 1, c.coefA, 1.0);
    BL_CHECK(launch_combine<T>(g, c, a, false, s));
  }
  return BL_OK;
}

}  // namespace
}  // namespace bl

using namespace bl;

extern "C" {

int bl_dist_set_reduce_hook(bl_allreduce_cb hook, void* user) {
  g_reduce_hook = hook;
  g_reduce_user = user;
  return BL_OK;
}

size_t bl_arnoldi_workspace_bytes(int64_t n, int64_t K, int dtype) {
  const size_t ld = align_up((size_t)n, 64);
  size_t b = common_bytes(K);
  b += align_up((size_t)K * 8, 256);
  b += 3 * align_up((size_t)K * K * 8, 256);
  const int64_t gram_parts = gram_parts_for(n, K);
  b += align_up((size_t)gram_parts * K * K * 8, 256);
  b += 2 * align_up((ld + 64) * dtype_size(dtype), 256);
  return b + 16 * 256;
}

// One run is a lockstep batch of one whose slice is the caller's whole workspace (AdjRun / FwdRun::begin refuse a
// workspace that is too small before anything is launched).
int bl_arnoldi_forward(bl_operator_t* op, int dtype, int64_t n, int64_t K, int second_pass, const void* v,
                       void* Q, int64_t ld, void* H, void* r, void* c, void* workspace,
                       size_t workspace_bytes, void* stream) {
  BL_REQUIRE(op && v && Q && H && r && c && workspace, "NULL argument");
  BL_CHECK(check_basis(dtype, n, K, ld, Q));
  BL_REQUIRE(op->n == n, "operator size does not match n");
  const auto run = dtype == BL_F32 ? arnoldi_forward_t<float> : arnoldi_forward_t<double>;
  return run(op, dtype, n, (int)K, second_pass, 1, v, n, Q, ld, H, r, c, workspace, workspace_bytes, as_stream(stream));
}

int bl_arnoldi_adjoint(bl_operator_t* op, int dtype, int64_t n, int64_t K, int reortho_full, const void* Q,
                       int64_t ld, const void* H, const void* r, const void* c, const void* dQ,
                       const void* dH, const void* dr, const void* dc, void* dv, void* Lambda,
                       void* workspace, size_t workspace_bytes, void* stream) {
  BL_REQUIRE(op && Q && H && r && c && dH && dv && Lambda && workspace, "NULL argument");
  BL_CHECK(check_basis(dtype, n, K, ld, Q));
  BL_REQUIRE(reinterpret_cast<uintptr_t>(Lambda) % 16 == 0, "Lambda must be 16-byte aligned");
  BL_REQUIRE(dQ == nullptr || reinterpret_cast<uintptr_t>(dQ) % 16 == 0, "dQ must be 16-byte aligned");
  BL_REQUIRE(op->n == n, "operator size does not match n");
  BL_REQUIRE(ld <= (int64_t)align_up((size_t)n, 64), "ld must be at most n rounded up to 64");
  const auto run = dtype == BL_F32 ? arnoldi_adjoint_t<float> : arnoldi_adjoint_t<double>;
  return run(op, dtype, n, (int)K, reortho_full, 1, Q, ld, H, r, c, dQ, dH, dr, dc, dv, n, Lambda, workspace,
             workspace_bytes, as_stream(stream));
}

int bl_arnoldi_forward_batch(bl_operator_t* op, int dtype, int64_t n, int64_t K, int second_pass, int64_t count,
                             const void* v, int64_t ldv, void* Q, int64_t ld, void* H, void* r, void* c,
                             void* workspace, size_t workspace_bytes, void* stream) {
  BL_REQUIRE(op && v && Q && H && r && c && workspace && count >= 1 && count <= 4096 && ldv >= n, "bad batch arguments");
  BL_CHECK(check_basis(dtype, n, K, ld, Q));
  BL_REQUIRE(op->n == n, "operator size does not match n");
  const size_t per = bl_arnoldi_workspace_bytes(n, K, dtype);
  BL_REQUIRE(workspace_bytes >= per * (size_t)count, "workspace too small (P * bl_arnoldi_workspace_bytes)");
  const auto run = dtype == BL_F32 ? arnoldi_forward_t<float> : arnoldi_forward_t<double>;
  return run(op, dtype, n, (int)K, second_pass, (int)count, v, ldv, Q, ld, H, r, c, workspace, per, as_stream(stream));
}

int bl_arnoldi_adjoint_batch(bl_operator_t* op, int dtype, int64_t n, int64_t K, int reortho_full, int64_t count,
                             const void* Q, int64_t ld, const void* H, const void* r, const void* c, const void* dQ,
                             const void* dH, const void* dr, const void* dc, void* dv, int64_t lddv, void* Lambda,
                             void* workspace, size_t workspace_bytes, void* stream) {
  BL_REQUIRE(op && Q && H && r && c && dH && dv && Lambda && workspace && count >= 1 && count <= 4096 && lddv >= n,
             "bad batch arguments");
  BL_CHECK(check_basis(dtype, n, K, ld, Q));
  BL_REQUIRE(reinterpret_cast<uintptr_t>(Lambda) % 16 == 0, "Lambda must be 16-byte aligned");
  BL_REQUIRE(dQ == nullptr || reinterpret_cast<uintptr_t>(dQ) % 16 == 0, "dQ must be 16-byte aligned");
  BL_REQUIRE(op->n == n, "operator size does not match n");
  BL_REQUIRE(ld <= (int64_t)align_up((size_t)n, 64), "ld must be at most n rounded up to 64");
  const size_t per = bl_arnoldi_workspace_bytes(n, K, dtype);
  BL_REQUIRE(workspace_bytes >= per * (size_t)count, "workspace too small (P * bl_arnoldi_workspace_bytes)");
  const auto run = dtype == BL_F32 ? arnoldi_adjoint_t<float> : arnoldi_adjoint_t<double>;
  return run(op, dtype, n, (int)K, reortho_full, (int)count, Q, ld, H, r, c, dQ, dH, dr, dc, dv, lddv, Lambda,
             workspace, per, as_stream(stream));
}

#if defined(BL_STEP_DEBUG) || defined(BL_STEP_CYCLES)
extern "C" int bl_step_debug_read(unsigned long long* out16, int reset) {
  BL_CUDA(cudaDeviceSynchronize());
  BL_CUDA(cudaMemcpyFromSymbol(out16, bl::g_step_dbg, 16 * sizeof(unsigned long long)));
  if (reset) {
    unsigned long long z[16] = {0};
    BL_CUDA(cudaMemcpyToSymbol(bl::g_step_dbg, z, sizeof(z)));
  }
  return BL_OK;
}
#endif

int bl_step_trace_begin(void) {
  g_step_trace_next.store(0, std::memory_order_relaxed);
  return BL_OK;
}

int bl_step_trace_end(unsigned long long* stamps_host, int64_t max_launches, int64_t* launches, int* pdl_accepted) {
  BL_REQUIRE(stamps_host && launches, "NULL argument");
  const int taken = g_step_trace_next.exchange(-1, std::memory_order_relaxed);
  const int64_t count = std::max<int64_t>(0, std::min<int64_t>({(int64_t)taken, max_launches, (int64_t)kTraceLaunches}));
  BL_CUDA(cudaDeviceSynchronize());
  if (count > 0)
    BL_CUDA(cudaMemcpyFromSymbol(stamps_host, g_step_trace, (size_t)count * kTraceStamps * sizeof(unsigned long long)));
  *launches = count;
  if (pdl_accepted) *pdl_accepted = g_step_pdl_ok.load(std::memory_order_relaxed);
  return BL_OK;
}

int bl_set_blocks_per_sm(int blocks) {
  BL_REQUIRE(blocks >= 0 && blocks <= 2, "blocks per SM must be 0 (default), 1 or 2");
  g_blocks_per_sm.store(blocks, std::memory_order_relaxed);
  return BL_OK;
}

int bl_get_blocks_per_sm(int* blocks) {
  BL_REQUIRE(blocks != nullptr, "NULL argument");
  *blocks = g_blocks_per_sm.load(std::memory_order_relaxed);
  return BL_OK;
}

int bl_op_deferred_grad(bl_operator_t* op, int dtype, int* yes) {
  BL_REQUIRE(op && yes, "NULL argument");
  *yes = op->deferred_grad(dtype) ? 1 : 0;
  return BL_OK;
}

size_t bl_lanczos3_workspace_bytes(int64_t n, int64_t K, int dtype) {
  const size_t ld = align_up((size_t)n, 64);
  return common_bytes(K) + 4 * align_up((ld + 64) * dtype_size(dtype), 256) + 16 * 256;
}

int bl_lanczos3_forward(bl_operator_t* op, int dtype, int64_t n, int64_t K, const void* v, void* xs,
                        int64_t ld, void* alphas, void* betas, void* workspace, size_t workspace_bytes,
                        void* stream) {
  BL_REQUIRE(op && v && xs && alphas && betas && workspace, "NULL argument");
  BL_CHECK(check_basis(dtype, n, K, ld, xs));
  BL_REQUIRE(ld <= (int64_t)align_up((size_t)n, 64), "ld must be at most n rounded up to 64");
  BL_REQUIRE(op->n == n, "operator size does not match n");
  cudaStream_t s = as_stream(stream);
  if (dtype == BL_F32)
    return lanczos3_forward_t<float>(op, dtype, n, (int)K, (const float*)v, (float*)xs, ld, (float*)alphas,
                                     (float*)betas, workspace, workspace_bytes, s);
  return lanczos3_forward_t<double>(op, dtype, n, (int)K, (const double*)v, (double*)xs, ld, (double*)alphas,
                                    (double*)betas, workspace, workspace_bytes, s);
}

int bl_lanczos3_adjoint(bl_operator_t* op, int dtype, int64_t n, int64_t K, const void* xs, int64_t ld,
                        const void* alphas, const void* betas, const void* dxs, const void* dalphas,
                        const void* dbetas, const void* vnorm, void* dv, void* workspace,
                        size_t workspace_bytes, void* stream) {
  BL_REQUIRE(op && xs && alphas && betas && dalphas && dbetas && vnorm && dv && workspace, "NULL argument");
  BL_CHECK(check_basis(dtype, n, K, ld, xs));
  BL_REQUIRE(ld <= (int64_t)align_up((size_t)n, 64), "ld must be at most n rounded up to 64");
  BL_REQUIRE(op->n == n, "operator size does not match n");
  cudaStream_t s = as_stream(stream);
  if (dtype == BL_F32)
    return lanczos3_adjoint_t<float>(op, dtype, n, (int)K, (const float*)xs, ld, (const float*)alphas,
                                     (const float*)betas, (const float*)dxs, (const float*)dalphas,
                                     (const float*)dbetas, (const float*)vnorm, (float*)dv, workspace,
                                     workspace_bytes, s);
  return lanczos3_adjoint_t<double>(op, dtype, n, (int)K, (const double*)xs, ld, (const double*)alphas,
                                    (const double*)betas, (const double*)dxs, (const double*)dalphas,
                                    (const double*)dbetas, (const double*)vnorm, (double*)dv, workspace,
                                    workspace_bytes, s);
}

// ---- small vector helpers ---------------------------------------------------------------
size_t bl_vec_workspace_bytes(void) { return common_bytes(1024) + 16 * 256; }

}  // extern "C"

namespace bl {
namespace {
template <typename T>
int rows_dot_t(int64_t n, int nrows, const T* M, int64_t ld, const T* x, T* out, void* workspace, size_t wbytes,
               cudaStream_t s) {
  Workspace w(workspace, wbytes);
  Common c;
  carve_common(w, std::max(nrows, 1), c);
  BL_REQUIRE(w.ok(), "workspace too small (bl_vec_workspace_bytes)");
  BL_CUDA(cudaMemsetAsync(c.counters, 0, 256, s));
  Epi e;
  e.mode = EPI_STORE;
  e.m = nrows;
  e.out_t = out;
  return launch_dots<T>(pick_grid<T>(n), c, rows(M, ld, 0, nrows), x, n, e, s);
}

template <typename T>
int rows_combine_t(int64_t n, int nrows, const T* M, int64_t ld, const double* coef_host, bool accumulate, T* out,
                   void* workspace, size_t wbytes, cudaStream_t s) {
  Workspace w(workspace, wbytes);
  Common c;
  carve_common(w, std::max(nrows, 1), c);
  BL_REQUIRE(w.ok(), "workspace too small (bl_vec_workspace_bytes)");
  BL_CUDA(cudaMemcpyAsync(c.coefA, coef_host, (size_t)nrows * 8, cudaMemcpyHostToDevice, s));
  CombineArgs a;
  a.n = n;
  a.out = out;
  if (accumulate) {
    a.nvec = 1;
    a.vec[0] = term(out);
  }
  a.blk[0] = rows(M, ld, 0, nrows, c.coefA, 1.0);
  return launch_combine<T>(pick_grid<T>(n), c, a, false, s);
}

template <typename T>
__global__ void k_transpose(int64_t rows_, int64_t cols, const T* __restrict__ src, int64_t ld_src,
                            T* __restrict__ dst, int64_t ld_dst) {
  __shared__ T tile[32][33];
  const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
  for (int dy = threadIdx.y; dy < 32; dy += blockDim.y) {
    const int64_t r = r0 + dy, cidx = c0 + threadIdx.x;
    if (r < rows_ && cidx < cols) tile[dy][threadIdx.x] = src[r * ld_src + cidx];
  }
  __syncthreads();
  for (int dy = threadIdx.y; dy < 32; dy += blockDim.y) {
    const int64_t cidx = c0 + dy, r = r0 + threadIdx.x;
    if (r < rows_ && cidx < cols) dst[cidx * ld_dst + r] = tile[threadIdx.x][dy];
  }
}
}  // namespace
}  // namespace bl

extern "C" {

int bl_rows_dot(int dtype, int64_t n, int64_t nrows, const void* M, int64_t ld, const void* x, void* out,
                void* workspace, size_t workspace_bytes, void* stream) {
  BL_REQUIRE(M && x && out && workspace && n >= 1 && nrows >= 1 && nrows <= 1024, "bad rows_dot arguments");
  BL_REQUIRE((ld * dtype_size(dtype)) % 16 == 0 || nrows == 1, "ld must be a multiple of 16 bytes");
  cudaStream_t s = as_stream(stream);
  if (dtype == BL_F32)
    return rows_dot_t<float>(n, (int)nrows, (const float*)M, ld, (const float*)x, (float*)out, workspace, workspace_bytes, s);
  return rows_dot_t<double>(n, (int)nrows, (const double*)M, ld, (const double*)x, (double*)out, workspace, workspace_bytes, s);
}

int bl_vec_dot(int dtype, int64_t n, const void* x, const void* y, void* out, void* workspace,
               size_t workspace_bytes, void* stream) {
  return bl_rows_dot(dtype, n, 1, x, n, y, out, workspace, workspace_bytes, stream);
}

int bl_rows_combine(int dtype, int64_t n, int64_t nrows, const void* M, int64_t ld, const double* coef_host,
                    int accumulate, void* out, void* workspace, size_t workspace_bytes, void* stream) {
  BL_REQUIRE(M && coef_host && out && workspace && n >= 1 && nrows >= 1 && nrows <= 1024, "bad rows_combine arguments");
  BL_REQUIRE((ld * dtype_size(dtype)) % 16 == 0 || nrows == 1, "ld must be a multiple of 16 bytes");
  cudaStream_t s = as_stream(stream);
  if (dtype == BL_F32)
    return rows_combine_t<float>(n, (int)nrows, (const float*)M, ld, coef_host, accumulate != 0, (float*)out, workspace, workspace_bytes, s);
  return rows_combine_t<double>(n, (int)nrows, (const double*)M, ld, coef_host, accumulate != 0, (double*)out, workspace, workspace_bytes, s);
}

int bl_vec_axpby(int dtype, int64_t n, double a, const void* x, double b, const void* y, void* out, void* stream) {
  BL_REQUIRE(x && out && n >= 1, "bad axpby arguments");
  BL_REQUIRE(b == 0.0 || y != nullptr, "y is NULL with b != 0");
  cudaStream_t s = as_stream(stream);
  // reuse combine without coefficient rows; no workspace needed (no reduction)
  Common c{};
  CombineArgs args;
  args.n = n;
  args.out = out;
  args.nvec = 1;
  args.vec[0] = term(x, a);
  if (b != 0.0) {
    args.nvec = 2;
    args.vec[1] = term(y, b);
  }
  if (dtype == BL_F32) return launch_combine<float>(pick_grid<float>(n), c, args, false, s);
  return launch_combine<double>(pick_grid<double>(n), c, args, false, s);
}

int bl_transpose(int dtype, int64_t rows_, int64_t cols, const void* src, int64_t ld_src, void* dst,
                 int64_t ld_dst, void* stream) {
  BL_REQUIRE(src && dst && rows_ >= 1 && cols >= 1 && ld_src >= cols && ld_dst >= rows_, "bad transpose arguments");
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows_ + 31) / 32)), block(32, 8);
  cudaStream_t s = as_stream(stream);
  if (dtype == BL_F32)
    k_transpose<float><<<grid, block, 0, s>>>(rows_, cols, (const float*)src, ld_src, (float*)dst, ld_dst);
  else
    k_transpose<double><<<grid, block, 0, s>>>(rows_, cols, (const double*)src, ld_src, (double*)dst, ld_dst);
  BL_LAUNCHED();
  return BL_OK;
}

}  // extern "C"
