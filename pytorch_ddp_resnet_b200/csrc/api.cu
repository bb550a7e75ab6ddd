// libb200resnet.so — extern "C" entry points declared in include/b200resnet.h.
// Host-side planning (tile shapes, tap tables, TMA descriptors, split factors) + kernel launches.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>

#include "../../include/b200resnet.h"
#include "common.cuh"
#include "conv_direct.cuh"
#include "conv_tc.cuh"
#include "elementwise.cuh"
#include "head_sgd.cuh"
#include "input_pipeline.cuh"
#include "f32_path.cuh"

using namespace b200;

// -------------------------------------------------------------------------------------------------
// error handling
// -------------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define B200_REQUIRE(cond, ...) \
  do {                          \
    if (!(cond)) return fail(1, __VA_ARGS__); \
  } while (0)

#define B200_CUDA(...)                                                                   \
  do {                                                                                   \
    cudaError_t e__ = (__VA_ARGS__);                                                     \
    if (e__ != cudaSuccess) return fail(2, "%s failed: %s", #__VA_ARGS__, cudaGetErrorString(e__)); \
  } while (0)

static std::atomic<long long> g_launches{0};

#define B200_LAUNCH_CHECK(name)                                                          \
  do {                                                                                   \
    g_launches.fetch_add(1, std::memory_order_relaxed);                                  \
    cudaError_t e__ = cudaGetLastError();                                                \
    if (e__ != cudaSuccess) return fail(3, "launch of %s failed: %s", name, cudaGetErrorString(e__)); \
  } while (0)

static inline cudaStream_t as_stream(b200_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// Plain kernel launch through cudaLaunchKernelEx (one code path for ordinary and cluster launches).
// Programmatic dependent launch was tried here in round 1 (attribute on every launch, griddepcontrol
// wait at the top of every kernel): no gain on back-to-back kernels inside a CUDA graph and the full
// training graph hung, so it was removed.
template <typename... KArgs, typename... Args>
static cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                            cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// Experiment switches (DESIGN.md section 5) are environment variables read ONCE per process: every use below is
// a function-local `static const`, so no launch ever calls getenv.
static int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

// Deterministic mode (B200_ALGO_DETERMINISTIC or-ed into an entry point's `algo`): every cross-CTA / cross-warp fp32
// reduction runs in a fixed order - wgrad pixel-range splits and bias-gradient blocks store partials that
// wgrad_reduce_splits_kernel sums in order (instead of fp32 atomics into a zeroed gradient), the conv epilogues
// flush their statistics partials quadrant by quadrant (instead of shared-memory float atomics). The fp64
// accumulator atomics of the BN sums stay: their addends are fp32 values, whose fp64 sum is exact - hence
// independent of the order - unless the partials of one channel span more than ~2^21 in magnitude.
// The flag of the call being prepared by this thread (entry points set it, launch helpers read it):
static thread_local int g_det = 0;
static inline void take_det_flag(int& algo) {
  g_det = (algo & B200_ALGO_DETERMINISTIC) ? 1 : 0;
  algo &= ~B200_ALGO_DETERMINISTIC;
}

// partial-gradient workspace of a deterministic wgrad (dry: only report the split count the launch would use)
struct WgradDet {
  float* part;
  size_t bytes;
  bool dry;
  int splits;
};

// Per-device caches (one process may drive several GPUs): SM count, and "max dynamic shared memory
// already raised for this kernel on this device".
constexpr int MAX_DEVICES = 64;
static int cur_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEVICES) return 0;
  return dev;
}

static int num_sms() {
  static int n[MAX_DEVICES] = {0};
  const int dev = cur_device();
  if (n[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    n[dev] = v;
  }
  return n[dev];
}

template <auto Kernel>
static cudaError_t ensure_max_smem(int bytes) {
  static bool done[MAX_DEVICES] = {false};
  const int dev = cur_device();
  if (done[dev]) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done[dev] = true;
  return e;
}

static inline int ew_grid(size_t work_items, int per_block = EW_THREADS) {
  size_t b = (work_items + per_block - 1) / per_block;
  size_t cap = (size_t)num_sms() * 16;
  return (int)std::max<size_t>(1, std::min(b, cap));
}

extern "C" int b200_version(void) { return 100; }
extern "C" long long b200_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
extern "C" const char* b200_last_error(void) { return g_err; }

extern "C" int b200_device_check(void) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  int major = 0, minor = 0;
  B200_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  B200_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  B200_REQUIRE(major == 10, "device is sm_%d%d; this library only carries sm_100a code", major, minor);
  return 0;
}

// -------------------------------------------------------------------------------------------------
// TMA descriptors (driver entry point resolved at run time: no link-time libcuda dependency)
// -------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

static CUtensorMapSwizzle swizzle_for_bytes(int inner_bytes) {
  return inner_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                            : inner_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                : CU_TENSOR_MAP_SWIZZLE_32B;
}

// es = element size: 2 = bf16, 4 = fp32 (read by kind::tf32 MMAs). B200_TF32_TMA_ROUND=1 makes the TMA unit
// write TF32-rounded values (CU_TENSOR_MAP_DATA_TYPE_TFLOAT32) instead of raw fp32 bits, which the tensor core
// then truncates; which of the two matches cuDNN's TF32 convolutions is measured in tests/test_tf32_gpu.py.
static CUtensorMapDataType tmap_dtype(int es) {
  if (es == 2) return CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  static const int round = env_int("B200_TF32_TMA_ROUND", 1);
  return round ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
}

// bf16 tensor [N][H][W][C] with box (bc, bw, bh, bn)
// `pstride` > 1: the box takes every pstride-th pixel in w and h (TMA elementStrides): a stride-2 convolution
// reads its taps straight from the full-resolution tensor, bw x bh pixels land densely in shared memory.
static int make_tmap_nhwc(CUtensorMap* m, const void* ptr, int N, int H, int W, int C, int bc,
                          int bw, int bh, int bn, int pstride = 1, int es = 2) {
  EncodeTiledFn fn = encode_fn();
  B200_REQUIRE(fn, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * es, (cuuint64_t)W * C * es, (cuuint64_t)H * W * C * es};
  cuuint32_t box[4] = {(cuuint32_t)bc, (cuuint32_t)(bw * pstride), (cuuint32_t)(bh * pstride), (cuuint32_t)bn};
  cuuint32_t estr[4] = {1, (cuuint32_t)pstride, (cuuint32_t)pstride, 1};
  CUresult r = fn(m, tmap_dtype(es), 4, const_cast<void*>(ptr), dims, strides, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_bytes(bc * es),
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B200_REQUIRE(r == CUDA_SUCCESS,
               "cuTensorMapEncodeTiled(4d) failed: %d (N=%d H=%d W=%d C=%d box=%d,%d,%d,%d)", (int)r,
               N, H, W, C, bc, bw, bh, bn);
  return 0;
}

// bf16 matrix [rows][cols] (cols contiguous) with box (bc cols, br rows)
static int make_tmap_2d(CUtensorMap* m, const void* ptr, int rows, int cols, int bc, int br, int es = 2) {
  EncodeTiledFn fn = encode_fn();
  B200_REQUIRE(fn, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * es};
  cuuint32_t box[2] = {(cuuint32_t)bc, (cuuint32_t)br};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, tmap_dtype(es), 2, const_cast<void*>(ptr), dims, strides, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_bytes(bc * es),
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B200_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(2d) failed: %d (rows=%d cols=%d box=%d,%d)",
               (int)r, rows, cols, bc, br);
  return 0;
}

// -------------------------------------------------------------------------------------------------
// conv planning
// -------------------------------------------------------------------------------------------------
struct TilePlan {
  int bw, bh, bn, rows_valid, tiles_w, tiles_h, tiles_n;
};

static int largest_divisor_leq(int n, int cap) {
  for (int d = std::min(n, cap); d >= 1; --d)
    if (n % d == 0) return d;
  return 1;
}

// Box of output pixels (w, h, images) with at most 128 pixels.
static TilePlan plan_tiles(int Nimg, int P, int Q, int cap = 128) {
  TilePlan t;
  if (Q >= cap) {
    t.bw = cap; t.bh = 1; t.bn = 1;
  } else {
    t.bw = Q;
    const int mh = cap / Q;
    if (mh >= P) {
      t.bh = P;
      t.bn = largest_divisor_leq(Nimg, std::max(1, cap / (Q * P)));
    } else {
      int d = largest_divisor_leq(P, mh);
      t.bh = (2 * d > mh) ? d : mh;
      t.bn = 1;
    }
  }
  t.rows_valid = t.bw * t.bh * t.bn;
  t.tiles_w = (Q + t.bw - 1) / t.bw;
  t.tiles_h = (P + t.bh - 1) / t.bh;
  t.tiles_n = (Nimg + t.bn - 1) / t.bn;
  return t;
}

// wgrad reduces over the pixels of a tile in 16-pixel MMAs: its tiles must hold a multiple of 16 rows.
// Rows that fall outside the image are zero-filled by TMA in BOTH operands and add nothing, so tiles
// may overhang (e.g. 14x8 tiles on a 14x14 map). Picks the box with the best useful-row fraction.
static TilePlan plan_tiles_mult16(int Nimg, int P, int Q, int cap) {
  TilePlan best = plan_tiles(Nimg, P, Q, cap);
  if (best.rows_valid % 16 == 0) return best;
  double best_eff = -1.0;
  const int bw = std::min(Q, cap);
  for (int bh = 1; bh <= std::max(1, cap / bw) && bh <= P + 15; ++bh) {
    const int max_bn = (bh >= P) ? std::max(1, cap / (bw * bh)) : 1;
    for (int bn = 1; bn <= std::min(max_bn, Nimg); ++bn) {
      const int rows = bw * bh * bn;
      if (rows > cap || rows % 16 != 0) continue;
      const int th = (P + bh - 1) / bh, tn = (Nimg + bn - 1) / bn, tw = (Q + bw - 1) / bw;
      const double eff = (double)Nimg * P * Q / ((double)th * tn * tw * cap);
      if (eff > best_eff) {
        best_eff = eff;
        best.bw = bw; best.bh = bh; best.bn = bn; best.rows_valid = rows;
        best.tiles_w = tw; best.tiles_h = th; best.tiles_n = tn;
      }
    }
  }
  return best;
}

static int pick_kc(int C) { return (C % 64 == 0) ? 64 : (C % 32 == 0) ? 32 : 16; }

// largest divisor of K that is a multiple of `mult` and <= cap (0 if none)
static int pick_bn(int K, int mult, int cap) {
  for (int bn = std::min(K, cap) / mult * mult; bn >= mult; bn -= mult)
    if (K % bn == 0) return bn;
  return 0;
}

static inline int floordiv2(int e) { return (e >= 0) ? e / 2 : -((-e + 1) / 2); }
static inline int mod2(int e) { return ((e % 2) + 2) % 2; }

static bool same_geometry(int H, int W, int R, int S, int stride, int pad, int* P, int* Q) {
  *P = (H + 2 * pad - R) / stride + 1;
  *Q = (W + 2 * pad - S) / stride + 1;
  if (stride == 1) return *P == H && *Q == W;
  if (stride == 2) return (H % 2 == 0) && (W % 2 == 0) && *P == H / 2 && *Q == W / 2;
  return false;
}

extern "C" int b200_conv2d_tc_supported(int pass, int N, int H, int W, int C, int K, int R, int S,
                                        int stride, int pad) {
  int P, Q;
  if (N < 1 || R * S > TC_MAX_TAPS) return 0;
  if (!same_geometry(H, W, R, S, stride, pad, &P, &Q)) return 0;
  if (C % 16 != 0 || K % 16 != 0) return 0;
  if (pass == B200_PASS_WGRAD) {
    TilePlan t = plan_tiles_mult16(N, P, Q, 128);
    if (t.rows_valid % 16 != 0) return 0;
  }
  return 1;
}

// Few-input-channel convolutions (the 3-channel stems) run as im2col (K padded to a multiple of 32)
// followed by the tcgen05 GEMM path as a 1x1 convolution over Kpad channels.
static int im2col_kpad(int R, int S, int C) { return ((R * S * C + 31) / 32) * 32; }

static bool use_im2col(int algo, int pass, int N, int H, int W, int C, int K, int R, int S, int stride,
                       int pad) {
  if (algo == B200_ALGO_DIRECT || pass == B200_PASS_DGRAD) return false;
  if (b200_conv2d_tc_supported(pass, N, H, W, C, K, R, S, stride, pad)) return false;
  if (C >= 16 || K % 16 != 0 || R * S * C > 1024) return false;
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  if (P < 1 || Q < 1) return false;
  if (pass == B200_PASS_WGRAD && plan_tiles_mult16(N, P, Q, 128).rows_valid % 16 != 0) return false;
  return true;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static void wgrad_det_regions(int N, int H, int W, int C, int K, int R, int S, int stride, int pad, int algo,
                              size_t* dbias_bytes, size_t* part_bytes);

extern "C" size_t b200_conv2d_workspace_bytes(int pass, int N, int H, int W, int C, int K, int R,
                                              int S, int stride, int pad, int algo) {
  if (pass == B200_PASS_WGRAD && (algo & B200_ALGO_DETERMINISTIC)) {   // + the ordered-reduction partials
    algo &= ~B200_ALGO_DETERMINISTIC;
    size_t dbias_bytes = 0, part_bytes = 0;
    wgrad_det_regions(N, H, W, C, K, R, S, stride, pad, algo, &dbias_bytes, &part_bytes);
    return b200_conv2d_workspace_bytes(pass, N, H, W, C, K, R, S, stride, pad, algo) + dbias_bytes + part_bytes;
  }
  algo &= ~B200_ALGO_DETERMINISTIC;
  if (algo == B200_ALGO_DIRECT) return 0;
  if (use_im2col(algo, pass, N, H, W, C, K, R, S, stride, pad)) {
    const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
    const size_t kpad = im2col_kpad(R, S, C);
    return align_up((size_t)N * P * Q * kpad * 2, 1024) + align_up((size_t)K * kpad * 4, 1024);
  }
  if (stride != 2 || pass != B200_PASS_DGRAD) return 0;
  if (!b200_conv2d_tc_supported(pass, N, H, W, C, K, R, S, stride, pad)) return 0;
  return (size_t)N * H * W * C * 2;  // stride-2 dgrad: the four output phases before the merge
}

static bool use_tc(int algo, int pass, int N, int H, int W, int C, int K, int R, int S, int stride,
                   int pad) {
  if (algo == B200_ALGO_DIRECT) return false;
  return b200_conv2d_tc_supported(pass, N, H, W, C, K, R, S, stride, pad) != 0;
}

static int conv_cluster_size() {
  // B200_CONV_CLUSTER = 1 | 2 | 4 (default 2): CTAs per cluster sharing one multicast filter tile
  static const int v = env_int("B200_CONV_CLUSTER", 2);
  return (v == 1 || v == 2 || v == 4) ? v : 2;
}

template <int KC, int CS>
static int launch_conv_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, ConvTcArgs& a,
                          cudaStream_t st) {
  const int max_dyn = 228352;
  B200_CUDA(ensure_max_smem<conv_tc_kernel<KC, CS>>(max_dyn));
  a.a_bytes = 128u * KC * 2u;
  const uint32_t b_bytes = ((uint32_t)a.BN * KC * 2u + 1023u) & ~1023u;
  a.stage_bytes = a.a_bytes + b_bytes;
  a.stages = std::min<int>(TC_MAX_STAGES, (max_dyn - 1024) / (int)a.stage_bytes);
  B200_REQUIRE(a.stages >= 2, "conv_tc: tile does not fit in shared memory");
  a.tx_bytes = (uint32_t)a.rows_valid * KC * 2u + (uint32_t)a.BN * KC * 2u;
  size_t dyn = (size_t)a.stages * a.stage_bytes + 1024;
  dyn = std::max<size_t>(dyn, 120 * 1024);  // one CTA per SM: the CTA owns all 512 TMEM columns
  const int num_ctiles = a.num_tiles / CS;
  const int grid = std::min(num_ctiles, num_sms() / CS) * CS;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = dyn;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  B200_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<KC, CS>, tmA, tmB, a));
  B200_LAUNCH_CHECK("conv_tc_kernel");
  return 0;
}

// SM-pair (cta_group::2) launch: tmB's box holds BN/2 filter rows
template <int KC, int STATS, bool TF32 = false>
static int launch_conv_tc2(const CUtensorMap& tmA, const CUtensorMap& tmB, ConvTcArgs& a,
                           cudaStream_t st) {
  const int max_dyn = STATS ? 228352 - 6144 : 228352;   // STATS: 8 KB of static shared memory for the partial sums
  constexpr uint32_t ES = TF32 ? 4u : 2u;
  B200_CUDA(ensure_max_smem<conv_tc2_kernel<KC, STATS, TF32>>(max_dyn));
  a.a_bytes = 128u * KC * ES;
  const uint32_t b_bytes = ((uint32_t)(a.BN / 2) * KC * ES + 1023u) & ~1023u;
  a.block_bytes = a.a_bytes + b_bytes;
  a.tx_bytes = (uint32_t)a.rows_valid * KC * ES + (uint32_t)(a.BN / 2) * KC * ES;  // per CTA, per block
  // K-blocks per stage: at least 8 MMAs per barrier round trip (the issue loop costs ~500 cycles per
  // iteration), as long as three stages still fit
  const int budget = max_dyn - 1024;
  int gblk = std::max(1, 8 / (int)(KC * ES / 32));
  static const int gblk_env = env_int("B200_CONV_GBLK", 0);
  if (gblk_env > 0) gblk = gblk_env;
  gblk = std::min(gblk, a.taps.n * a.nkc);
  while (gblk > 1 && budget / (int)(gblk * a.block_bytes) < 3) --gblk;
  a.gblk = gblk;
  a.stage_bytes = (uint32_t)gblk * a.block_bytes;
  a.stages = std::min<int>(TC_MAX_STAGES, budget / (int)a.stage_bytes);
  B200_REQUIRE(a.stages >= 2, "conv_tc2: tile does not fit in shared memory");
  size_t dyn = (size_t)a.stages * a.stage_bytes + 1024;
  dyn = std::max<size_t>(dyn, 120 * 1024);
  const int num_ptiles = a.num_tiles / 2;
  const int grid = std::min(num_ptiles, num_sms() / 2) * 2;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(TC2_THREADS);
  cfg.dynamicSmemBytes = dyn;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  B200_CUDA(cudaLaunchKernelEx(&cfg, conv_tc2_kernel<KC, STATS, TF32>, tmA, tmB, a));
  B200_LAUNCH_CHECK("conv_tc2_kernel");
  return 0;
}

static bool conv_use_halo() {
  // B200_CONV_HALO=0 disables the halo-reuse kernel (3x3 / stride 1 / pad 1 layers fall back to conv_tc2)
  static const int v = env_int("B200_CONV_HALO", 1);
  return v != 0;
}

static thread_local int g_halo_relu = 0;   // epilogue ReLU flag of the halo launch being prepared by this thread
static thread_local EpiBnBwd g_halo_bb = {nullptr, 1.f, 0};   // STATS = 2 arguments of that launch

// Halo-reuse SM-pair launch (see conv_tc2h_kernel). MT pixel tiles per CTA share each filter stage.
template <int KC, int MT, int STATS, bool TAIL32 = false>
static int launch_conv_tc2h(const void* act, int Nact, int Ha, int Wa, int Cin, const void* wmat, int Cout,
                            int wcols, const TapTable& taps, void* out, const void* residual,
                            const float* bias, int Nimg, int P, int Q, int BN, int pw, double* stats,
                            const EpiStatsFinal& fin, cudaStream_t st) {
  const int max_dyn = STATS ? 228352 - 6144 : 228352;   // STATS: 8 KB of static shared memory for the partial sums
  B200_CUDA(ensure_max_smem<conv_tc2h_kernel<KC, MT, STATS, TAIL32>>(max_dyn));
  ConvHaloArgs a;
  memset(&a, 0, sizeof(a));
  a.tiles_w = Q / 8; a.tiles_h = P / 16;
  a.BN = BN; a.n_ntiles = Cout / BN; a.nkc = Cin / KC;
  a.P = P; a.Q = Q; a.Nimg = Nimg; a.ldo = Cout;
  a.num_tiles = a.tiles_w * a.tiles_h * Nimg * a.n_ntiles;
  a.ntaps = taps.n;
  a.pw = pw;
  a.patch_tx_bytes = (uint32_t)pw * HALO_PH * KC * 2u;
  a.patch_bytes = (a.patch_tx_bytes + 1023u) & ~1023u;
  a.btile_bytes = (((uint32_t)(BN / 2) * KC * 2u) + 1023u) & ~1023u;
  const int budget = max_dyn - 1024 - 2 * MT * (int)a.patch_bytes;
  // taps per filter stage: all 9 when three such stages fit (>= 18 MMAs per barrier round trip), else 3
  a.tpb = (budget / (int)(taps.n * a.btile_bytes) >= 3) ? taps.n : 3;
  static const int tpb_env = env_int("B200_HALO_TPB", 0);
  if (tpb_env > 0) a.tpb = std::min(tpb_env, taps.n);
  a.ntg = (taps.n + a.tpb - 1) / a.tpb;
  a.bstage_bytes = (uint32_t)a.tpb * a.btile_bytes;
  a.bstages = std::min(HALO_BSTAGES_MAX, budget / (int)a.bstage_bytes);
  B200_REQUIRE(a.bstages >= 2, "conv_tc2h: filter ring does not fit in shared memory");
  for (int t = 0; t < taps.n; ++t) {
    a.tap_rowoff[t] = (taps.dh[t] + 1) * pw + (taps.dw[t] + 1);
    a.tap_wcol[t] = taps.wcol[t];
  }
  a.out = reinterpret_cast<bf16*>(out);
  a.residual = reinterpret_cast<const bf16*>(residual);
  a.bias = bias;
  a.stats = stats;
  a.fin = fin;
  a.relu = g_halo_relu;
  a.bb = g_halo_bb;
  a.det = g_det;
  B200_REQUIRE(((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(residual)) & 31) == 0,
               "conv_tc2h: output and residual must be 32-byte aligned (256-bit epilogue accesses)");
  CUtensorMap tmA, tmB, tmA32, tmB32;
  if (int rc = make_tmap_nhwc(&tmA, act, Nact, Ha, Wa, Cin, KC, pw, HALO_PH, 1)) return rc;
  if (int rc = make_tmap_2d(&tmB, wmat, Cout, wcols, KC, BN / 2)) return rc;
  if (int rc = make_tmap_nhwc(&tmA32, act, Nact, Ha, Wa, Cin, 32, pw, HALO_PH, 1)) return rc;   // tail block maps
  if (int rc = make_tmap_2d(&tmB32, wmat, Cout, wcols, 32, BN / 2)) return rc;
  size_t dyn = 2 * MT * (size_t)a.patch_bytes + (size_t)a.bstages * a.bstage_bytes + 1024;
  dyn = std::max<size_t>(dyn, 120 * 1024);
  const int num_units = a.num_tiles / (2 * MT);
  const int grid = std::min(num_units, num_sms() / 2) * 2;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(TC2_THREADS);
  cfg.dynamicSmemBytes = dyn;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  B200_CUDA(cudaLaunchKernelEx(&cfg, conv_tc2h_kernel<KC, MT, STATS, TAIL32>, tmA, tmB, tmA32, tmB32, a));
  B200_LAUNCH_CHECK("conv_tc2h_kernel");
  return 0;
}

static bool conv_use_pair() {
  // B200_CONV_PAIR=0 disables the cta_group::2 kernel (falls back to the single-CTA kernel)
  static const int v = env_int("B200_CONV_PAIR", 1);
  return v != 0;
}

template <int KC>
static int launch_conv_tc_cs(int cs, const CUtensorMap& tmA, const CUtensorMap& tmB, ConvTcArgs& a,
                             cudaStream_t st) {
  switch (cs) {
    case 4: return launch_conv_tc<KC, 4>(tmA, tmB, a, st);
    case 2: return launch_conv_tc<KC, 2>(tmA, tmB, a, st);
    default: return launch_conv_tc<KC, 1>(tmA, tmB, a, st);
  }
}

// Output phases of a stride-2 dgrad run as ONE launch of the SM-pair kernel (see ConvTcArgs::nphase).
struct PhasePlan {
  int nphase;
  int tap0[5];
  int id[4];
};

// One shifted-window GEMM launch. act: [Nact][Ha][Wa][Cin] (bf16), wmat: [Cout][ntaps*Cin] (bf16),
// out: [Nimg][P][Q][Cout].
static int run_conv_tc(const void* act, int Nact, int Ha, int Wa, int Cin, const void* wmat, int Cout,
                       int wcols, const TapTable& taps, void* out, const void* residual,
                       const float* bias, int Nimg, int P, int Q, cudaStream_t st,
                       double* stats = nullptr, bool* stats_fused = nullptr,
                       const EpiStatsFinal* finp = nullptr, int cstride = 1,
                       const PhasePlan* phases = nullptr, int es = 2, int relu = 0,
                       const EpiBnBwd* bb = nullptr) {
  // bb != nullptr (with stats, finp): `residual` is the BN input x of the fused BN backward whose dy this launch
  // produces; the SM-pair kernels accumulate sum(g), sum(g * x) (STATS = 2) and *stats_fused says whether they did
  // es = 4: fp32 / TF32 precision mode (fp32 activations, filters, output; SM-pair kernel only)
  // phases != nullptr: (P, Q) is the FULL output extent, tiles are planned on the (P/2, Q/2) phase grid
  EpiStatsFinal fin;
  memset(&fin, 0, sizeof(fin));
  if (finp) fin = *finp;
  // stats != nullptr: the SM-pair kernels also accumulate the per-channel sum / sum of squares of the
  // output (fused BN statistics); *stats_fused says whether the kernel that ran did it
  if (stats_fused) *stats_fused = false;
  // a launch that cannot carry the fused BN backward runs as the plain conv (x is NOT a residual to add)
  auto plain_without_bb = [&]() {
    return run_conv_tc(act, Nact, Ha, Wa, Cin, wmat, Cout, wcols, taps, out, nullptr, bias, Nimg, P, Q, st, nullptr,
                       nullptr, nullptr, cstride, phases, es, relu, nullptr);
  };
  // The per-channel sums cost the epilogue ~200 instructions per 16-column chunk against ~30 for the plain one.
  // Behind a long main loop (3x3 filters: >= 1152 MACs per output) that hides under the next tile's MMAs; behind a
  // short one (1x1 filters of the bottleneck blocks, im2col'd stems) the epilogue IS the kernel. Measured at the
  // ImageNet shapes, batch 256 (tools/bench_conv.py): 128 -> 512 1x1 @56x56 fprop 244 us plain, 637 us with fused
  // sums, 165 us for the stand-alone statistics kernel on its output; its dgrad 244 / 1048 us; at a reduction
  // length of 512 the two ways tie, above it the fused sums cost 8 - 40 us. The fused sums cost ~0.5 us per MB of
  // output there, the stand-alone pass ~0.2 us per MB + ~8 us of launch and drain: on small tensors (ResNet-20,
  // ResNet-v2-164: launch-bound) fusing still wins. Hence: NOT fused below 512 MACs per output
  // (B200_FUSED_STATS_MIN_K) when the output is larger than 32 MB (B200_FUSED_STATS_MAX_MB).
  static const int fused_min_k = env_int("B200_FUSED_STATS_MIN_K", 512);
  static const int fused_max_mb = env_int("B200_FUSED_STATS_MAX_MB", 32);
  if ((stats || bb) && taps.n * Cin < fused_min_k &&
      (size_t)Nimg * P * Q * Cout * 2 > ((size_t)fused_max_mb << 20)) {
    if (bb) return plain_without_bb();
    stats = nullptr;
    finp = nullptr;
    memset(&fin, 0, sizeof(fin));
  }
  if (bb) {
    B200_REQUIRE(stats && stats_fused && finp && residual && es == 2 && !bias && !relu,
                 "conv_tc: the fused BN backward needs x, a statistics workspace and a plain bf16 dgrad");
    if (Cout % 16 != 0 || Cout > EPI_STATS_MAX_C) return plain_without_bb();
  }
  int KC = pick_kc(Cin);
  if (es == 4) KC = (Cin % 32 == 0) ? 32 : (Cin % 16 == 0) ? 16 : 8;   // 128 / 64 / 32-byte rows of fp32
  int BN = pick_bn(Cout, 16, 256);
  B200_REQUIRE(BN > 0, "conv_tc: no legal N tile for Cout=%d", Cout);
  // a fused residual is prefetched into registers: at most 80 columns per epilogue thread (N tile <= 160)
  if (residual && es == 2 && BN > 16 * EPI_RES_VECS) {
    const int bn2 = pick_bn(Cout, 32, 16 * EPI_RES_VECS);
    BN = bn2 > 0 ? bn2 : pick_bn(Cout, 16, 16 * EPI_RES_VECS);
    B200_REQUIRE(BN > 0, "conv_tc: no legal N tile for Cout=%d with a residual", Cout);
  }
  TilePlan t = phases ? plan_tiles(Nimg, P / 2, Q / 2) : plan_tiles(Nimg, P, Q);
  ConvTcArgs a;
  memset(&a, 0, sizeof(a));
  a.bw = t.bw; a.bh = t.bh; a.bn = t.bn; a.rows_valid = t.rows_valid;
  a.tiles_w = t.tiles_w; a.tiles_h = t.tiles_h; a.tiles_n = t.tiles_n;
  const int m_tiles_all = t.tiles_w * t.tiles_h * t.tiles_n;
  const bool pair = conv_use_pair() && m_tiles_all % 2 == 0 && BN % 32 == 0;
  B200_REQUIRE(!phases || pair, "conv_tc: the phased launch needs the SM-pair kernel");
  a.nphase = 1;
  a.phase_tap0[0] = 0;
  a.phase_tap0[1] = taps.n;
  if (phases) {
    a.nphase = phases->nphase;
    for (int i = 0; i < 5; ++i) a.phase_tap0[i] = phases->tap0[i];
    for (int i = 0; i < 4; ++i) a.phase_id[i] = phases->id[i];
  }
  // (tried: 64-channel blocks with a partial last block per tap for Cin = 160 - the extra predicate per
  //  MMA slowed the issue loop more than SWIZZLE_128B gained; KC stays a divisor of Cin)
  // halo-reuse kernel: 3x3 taps with unit displacements on an un-split input, maps that tile in 8x16
  {
    bool unit = taps.n == 9 && Ha == P && Wa == Q && Nact == Nimg && cstride == 1 && !phases && es == 2;
    for (int i = 0; unit && i < taps.n; ++i)
      unit = taps.dn[i] == 0 && taps.dh[i] >= -1 && taps.dh[i] <= 1 && taps.dw[i] >= -1 && taps.dw[i] <= 1;
    const int mt8x16 = (Q / 8) * (P / 16) * Nimg;
    if (unit && conv_use_halo() && conv_use_pair() && Q % 8 == 0 && P % 16 == 0 && mt8x16 % 2 == 0 &&
        BN % 32 == 0 && Cin % KC == 0 && KC >= 32) {
      // B200_HALO_MT = 1 | 2, B200_HALO_PW = 10 | 16. Measured (round 1, fprop TFLOP/s, 160@32x32 /
      // 320@16x16): MT=1 1183 / 1419, MT=2 983 / 1163 (halved filter traffic does not pay for the lost
      // accumulator double-buffering: the kernel is not L2->SM bound), PW=16 1168 / 1414.
      static const int mt_env = env_int("B200_HALO_MT", 1);
      static const int pw = std::max(10, std::min(16, env_int("B200_HALO_PW", 10)));
      const bool mt2 = mt_env == 2 && mt8x16 % 4 == 0 && 2 * BN <= 512 && (!residual || BN <= 8 * EPI_RES_VECS);
#define B200_HALO_ARGS act, Nact, Ha, Wa, Cin, wmat, Cout, wcols, taps, out, residual, bias, Nimg, P, Q, BN, pw
      // Cin = 64 n + 32 (the 160-channel layers): 64-channel blocks + one 32-channel tail block
      static const int mixed_env = env_int("B200_HALO_MIXED", 1);
      const bool mixed = mixed_env && !mt2 && Cin > 64 && Cin % 64 == 32;
      g_halo_relu = relu;
      if (bb) {
        if (mt2 || (BN / 2) % 16 != 0) return plain_without_bb();
        *stats_fused = true;
        g_halo_bb = *bb;
        if (mixed) return launch_conv_tc2h<64, 1, 2, true>(B200_HALO_ARGS, stats, fin, st);
        if (KC == 64) return launch_conv_tc2h<64, 1, 2>(B200_HALO_ARGS, stats, fin, st);
        return launch_conv_tc2h<32, 1, 2>(B200_HALO_ARGS, stats, fin, st);
      }
      if (stats && !mt2 && BN <= EPI_STATS_MAX_BN && Cout <= EPI_STATS_MAX_C) {
        *stats_fused = true;
        if (mixed) return launch_conv_tc2h<64, 1, true, true>(B200_HALO_ARGS, stats, fin, st);
        if (KC == 64) return launch_conv_tc2h<64, 1, true>(B200_HALO_ARGS, stats, fin, st);
        return launch_conv_tc2h<32, 1, true>(B200_HALO_ARGS, stats, fin, st);
      }
      if (mixed) return launch_conv_tc2h<64, 1, false, true>(B200_HALO_ARGS, nullptr, fin, st);
      if (KC == 64)
        return mt2 ? launch_conv_tc2h<64, 2, false>(B200_HALO_ARGS, nullptr, fin, st)
                   : launch_conv_tc2h<64, 1, false>(B200_HALO_ARGS, nullptr, fin, st);
      return mt2 ? launch_conv_tc2h<32, 2, false>(B200_HALO_ARGS, nullptr, fin, st)
                 : launch_conv_tc2h<32, 1, false>(B200_HALO_ARGS, nullptr, fin, st);
#undef B200_HALO_ARGS
    }
  }
  a.BN = BN; a.n_ntiles = Cout / BN; a.nkc = (Cin + KC - 1) / KC; a.cin = Cin;
  a.P = P; a.Q = Q; a.Nimg = Nimg; a.ldo = Cout;
  a.num_tiles = t.tiles_w * t.tiles_h * t.tiles_n * a.n_ntiles * a.nphase;
  a.taps = taps;
  a.cstride = cstride;
  a.relu = relu;
  a.det = g_det;
  B200_REQUIRE(cstride == 1 || (t.bw * cstride <= 256 && t.bh * cstride <= 256),
               "conv_tc: strided TMA box exceeds 256 elements");
  a.out = reinterpret_cast<bf16*>(out);
  a.residual = reinterpret_cast<const bf16*>(residual);
  a.bias = bias;
  B200_REQUIRE(((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(residual)) & 31) == 0,
               "conv_tc: output and residual must be 32-byte aligned (256-bit epilogue accesses)");
  if (es == 4) {
    B200_REQUIRE(pair, "conv_tc (tf32): shape needs the SM-pair kernel (even pixel-tile count, Cout %% 32 == 0)");
    CUtensorMap tmA, tmB;
    if (int rc = make_tmap_nhwc(&tmA, act, Nact, Ha, Wa, Cin, KC, t.bw, t.bh, t.bn, cstride, 4)) return rc;
    if (int rc = make_tmap_2d(&tmB, wmat, Cout, wcols, KC, BN / 2, 4)) return rc;
    switch (KC) {
      case 32: return launch_conv_tc2<32, false, true>(tmA, tmB, a, st);
      case 16: return launch_conv_tc2<16, false, true>(tmA, tmB, a, st);
      default: return launch_conv_tc2<8, false, true>(tmA, tmB, a, st);
    }
  }
  if (bb && (!pair || (BN / 2) % 16 != 0)) return plain_without_bb();
  if (pair) {
    // SM pair: every CTA stages BN/2 filter rows (whole 8-row swizzle atoms, UMMA N multiple of 16)
    CUtensorMap tmA, tmB;
    if (int rc = make_tmap_nhwc(&tmA, act, Nact, Ha, Wa, Cin, KC, t.bw, t.bh, t.bn, cstride)) return rc;
    if (int rc = make_tmap_2d(&tmB, wmat, Cout, wcols, KC, BN / 2)) return rc;
    if (bb) {
      *stats_fused = true;
      a.stats = stats;
      a.fin = fin;
      a.bb = *bb;
      switch (KC) {
        case 64: return launch_conv_tc2<64, 2>(tmA, tmB, a, st);
        case 32: return launch_conv_tc2<32, 2>(tmA, tmB, a, st);
        default: return launch_conv_tc2<16, 2>(tmA, tmB, a, st);
      }
    }
    if (stats && BN <= EPI_STATS_MAX_BN && Cout <= EPI_STATS_MAX_C) {
      *stats_fused = true;
      a.stats = stats;
      a.fin = fin;
      switch (KC) {
        case 64: return launch_conv_tc2<64, true>(tmA, tmB, a, st);
        case 32: return launch_conv_tc2<32, true>(tmA, tmB, a, st);
        default: return launch_conv_tc2<16, true>(tmA, tmB, a, st);
      }
    }
    switch (KC) {
      case 64: return launch_conv_tc2<64, false>(tmA, tmB, a, st);
      case 32: return launch_conv_tc2<32, false>(tmA, tmB, a, st);
      default: return launch_conv_tc2<16, false>(tmA, tmB, a, st);
    }
  }
  // cluster size: the pixel-tile count must split evenly and every filter slice must be whole 8-row
  // swizzle atoms
  int cs = conv_cluster_size();
  const int m_tiles = t.tiles_w * t.tiles_h * t.tiles_n;
  while (cs > 1 && (m_tiles % cs != 0 || (BN / cs) % 8 != 0 || BN % cs != 0)) cs /= 2;
  CUtensorMap tmA, tmB;
  if (int rc = make_tmap_nhwc(&tmA, act, Nact, Ha, Wa, Cin, KC, t.bw, t.bh, t.bn, cstride)) return rc;
  if (int rc = make_tmap_2d(&tmB, wmat, Cout, wcols, KC, BN / cs)) return rc;
  switch (KC) {
    case 64: return launch_conv_tc_cs<64>(cs, tmA, tmB, a, st);
    case 32: return launch_conv_tc_cs<32>(cs, tmA, tmB, a, st);
    default: return launch_conv_tc_cs<16>(cs, tmA, tmB, a, st);
  }
}

// taps of fprop / wgrad (window displacement on the input, column in the KRSC filter matrix)
// (for stride 2 the window origin is 2 * output pixel + displacement and the TMA map skips every other pixel)
static TapTable fprop_taps(int C, int R, int S, int pad) {
  TapTable tt;
  memset(&tt, 0, sizeof(tt));
  for (int r = 0; r < R; ++r)
    for (int s = 0; s < S; ++s) {
      const int i = tt.n++;
      tt.dh[i] = r - pad; tt.dw[i] = s - pad; tt.dn[i] = 0;
      tt.wcol[i] = (r * S + s) * C;
    }
  return tt;
}

static int conv2d_fprop_impl(const void* x, const void* w_krsc, const float* bias,
                             const void* residual, void* y, int N, int H, int W, int C, int K,
                             int R, int S, int stride, int pad, int algo, void* ws,
                             size_t ws_bytes, b200_stream_t stream, double* stats, bool* stats_fused,
                             const EpiStatsFinal* fin = nullptr, int relu = 0) {
  B200_REQUIRE(x && w_krsc && y, "conv2d_fprop: null pointer");
  B200_REQUIRE(stride == 1 || stride == 2, "conv2d_fprop: stride %d unsupported", stride);
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  B200_REQUIRE(P > 0 && Q > 0, "conv2d_fprop: empty output");
  cudaStream_t st = as_stream(stream);
  const bool tc = use_tc(algo, B200_PASS_FPROP, N, H, W, C, K, R, S, stride, pad);
  if (!tc && use_im2col(algo, B200_PASS_FPROP, N, H, W, C, K, R, S, stride, pad)) {
    const int kpad = im2col_kpad(R, S, C);
    const size_t col_bytes = align_up((size_t)N * P * Q * kpad * 2, 1024);
    B200_REQUIRE(ws && ws_bytes >= col_bytes + (size_t)K * kpad * 2, "conv2d_fprop: workspace too small");
    bf16* col = reinterpret_cast<bf16*>(ws);
    bf16* wpad = reinterpret_cast<bf16*>(reinterpret_cast<uint8_t*>(ws) + col_bytes);
    launch_k(im2col_kernel, ew_grid((size_t)N * P * Q * kpad), EW_THREADS, 0, st, (const bf16*)x, col, N, H, W, C, R, S, stride, pad, P, Q, kpad);
    B200_LAUNCH_CHECK("im2col_kernel");
    launch_k(repitch_rows_kernel<bf16>, ew_grid((size_t)K * kpad), EW_THREADS, 0, st, (const bf16*)w_krsc, wpad, K, R * S * C, kpad);
    B200_LAUNCH_CHECK("repitch_rows_kernel");
    TapTable tt;
    memset(&tt, 0, sizeof(tt));
    tt.n = 1;
    return run_conv_tc(col, N, P, Q, kpad, wpad, K, kpad, tt, y, residual, bias, N, P, Q, st, stats,
                       stats_fused, fin, 1, nullptr, 2, relu);
  }
  B200_REQUIRE(tc || algo != B200_ALGO_TC, "conv2d_fprop: shape not supported by the tcgen05 path");
  if (!tc) {
    ConvDims d{N, H, W, C, K, R, S, stride, pad, P, Q};
    const size_t total = (size_t)N * P * Q * K;
    launch_k(conv_fprop_direct_kernel, ew_grid(total), EW_THREADS, 0, st, (const bf16*)x, (const bf16*)w_krsc, bias, (const bf16*)residual, (bf16*)y, d, relu);
    B200_LAUNCH_CHECK("conv_fprop_direct_kernel");
    return 0;
  }
  // stride 2: ONE launch, the taps read every other pixel of x through the TMA map's elementStrides (round 1
  // made a parity-split copy of x first: 549 TFLOP/s against cuDNN's 724 on the 160->320 layer)
  TapTable tt = fprop_taps(C, R, S, pad);
  return run_conv_tc(x, N, H, W, C, w_krsc, K, R * S * C, tt, y, residual, bias, N, P, Q, st, stats,
                     stats_fused, fin, stride, nullptr, 2, relu);
}

extern "C" int b200_conv2d_fprop(const void* x, const void* w_krsc, const float* bias,
                                 const void* residual, void* y, int N, int H, int W, int C, int K,
                                 int R, int S, int stride, int pad, int relu, int algo, void* ws,
                                 size_t ws_bytes, b200_stream_t stream) {
  take_det_flag(algo);
  bool fused = false;
  return conv2d_fprop_impl(x, w_krsc, bias, residual, y, N, H, W, C, K, R, S, stride, pad, algo, ws,
                           ws_bytes, stream, nullptr, &fused, nullptr, relu);
}

static int bn_sums_launch(const void* x, int64_t rows, int C, void* ws, size_t ws_bytes, int finalize,
                          float eps, float momentum, float* mean, float* invstd, float* running_mean,
                          float* running_var, int64_t* num_batches_tracked, cudaStream_t st);

extern "C" int b200_conv2d_fprop_stats(const void* x, const void* w_krsc, const float* bias,
                                       const void* residual, void* y, int N, int H, int W, int C, int K,
                                       int R, int S, int stride, int pad, int algo, void* ws,
                                       size_t ws_bytes, void* stats_ws, size_t stats_ws_bytes, float eps,
                                       float* mean, float* invstd, b200_stream_t stream) {
  take_det_flag(algo);
  B200_REQUIRE(stats_ws && K % 8 == 0, "conv2d_fprop_stats: needs a statistics workspace and K %% 8 == 0");
  B200_REQUIRE(stats_ws_bytes >= b200_bn_workspace_bytes(0, K), "conv2d_fprop_stats: statistics workspace too small");
  B200_REQUIRE((reinterpret_cast<uintptr_t>(stats_ws) & 7) == 0, "conv2d_fprop_stats: statistics workspace must be 8-byte aligned");
  B200_REQUIRE((mean == nullptr) == (invstd == nullptr), "conv2d_fprop_stats: mean and invstd go together");
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  double* accum = reinterpret_cast<double*>(stats_ws);
  EpiStatsFinal fin;
  memset(&fin, 0, sizeof(fin));
  fin.ticket = reinterpret_cast<unsigned int*>(accum + BN_SLOTS * bn_slot_stride(K));
  fin.mean = mean; fin.invstd = invstd; fin.eps = eps; fin.rows = (long long)N * P * Q;
  bool fused = false;
  if (int rc = conv2d_fprop_impl(x, w_krsc, bias, residual, y, N, H, W, C, K, R, S, stride, pad, algo, ws,
                                 ws_bytes, stream, accum, &fused, &fin))
    return rc;
  if (fused) return 0;
  // kernels without the fused epilogue (direct, single-CTA): one reduction pass over y
  return bn_sums_launch(y, (int64_t)N * P * Q, K, stats_ws, stats_ws_bytes, mean ? 1 : 0, eps, 0.f, mean, invstd,
                        nullptr, nullptr, nullptr, as_stream(stream));
}

// merge of the parity-split dx with an optional addend
__global__ void parity_merge_add_kernel(const bf16* __restrict__ src, const bf16* __restrict__ addend,
                                        bf16* __restrict__ dst, int N, int H, int W, int C) {
  const int CG = C / 8;
  const size_t nvec = (size_t)N * H * W * CG;
  const int H2 = H / 2, W2 = W / 2;
  for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (size_t)gridDim.x * blockDim.x) {
    const int cg = (int)(v % CG);
    const size_t pix = v / CG;
    const int w = (int)(pix % W);
    const int h = (int)((pix / W) % H);
    const int n = (int)(pix / ((size_t)W * H));
    const int ph = (h & 1) * 2 + (w & 1);
    const size_t ppix = (((size_t)ph * N + n) * H2 + (h >> 1)) * W2 + (w >> 1);
    Vec8 a;
    a.raw = ldg_stream(src + ppix * C + (size_t)cg * 8);
    if (addend) {
      Vec8 b;
      b.raw = ldg_stream(addend + v * 8);
      float fa[8], fb[8];
      a.to_float(fa);
      b.to_float(fb);
#pragma unroll
      for (int j = 0; j < 8; ++j) fa[j] = round_bf16(fa[j] + fb[j]);
      a.from_float(fa);
    }
    stg_stream(dst + v * 8, a.raw);
  }
}

// Tap table of a stride-2 dgrad grouped by output parity phase, heaviest phase first (see ConvTcArgs::nphase).
// Returns false when some phase has no tap (such a phase is all zeros and cannot be a GEMM tile).
static bool build_dgrad_phases(int R, int S, int K, int pad, PhasePlan* pp, TapTable* all) {
  memset(pp, 0, sizeof(*pp));
  memset(all, 0, sizeof(*all));
  int cnt[4];
  for (int ph = 0; ph < 4; ++ph) {
    cnt[ph] = 0;
    for (int r = 0; r < R; ++r)
      for (int s = 0; s < S; ++s)
        if (mod2((ph >> 1) + pad - r) == 0 && mod2((ph & 1) + pad - s) == 0) ++cnt[ph];
  }
  if (R * S > TC_MAX_TAPS || !(cnt[0] > 0 && cnt[1] > 0 && cnt[2] > 0 && cnt[3] > 0)) return false;
  int order[4] = {0, 1, 2, 3};
  std::stable_sort(order, order + 4, [&](int x, int y) { return cnt[x] > cnt[y]; });   // heaviest first
  pp->nphase = 4;
  for (int i = 0; i < 4; ++i) {
    const int ph = order[i], pa = ph >> 1, pb = ph & 1;
    pp->id[i] = ph;
    pp->tap0[i] = all->n;
    for (int r = 0; r < R; ++r) {
      if (mod2(pa + pad - r) != 0) continue;
      for (int s = 0; s < S; ++s) {
        if (mod2(pb + pad - s) != 0) continue;
        const int t = all->n++;
        all->dh[t] = floordiv2(pa + pad - r); all->dw[t] = floordiv2(pb + pad - s); all->dn[t] = 0;
        all->wcol[t] = (r * S + s) * K;
      }
    }
  }
  pp->tap0[4] = all->n;
  return true;
}

// bb != nullptr: addend is the BN input x of the fused BN backward (see run_conv_tc); *fused reports whether the
// launch accumulated (and finalized) its sums
static int conv2d_dgrad_impl(const void* dy, const void* w_crsk, const void* addend, void* dx,
                             int N, int H, int W, int C, int K, int R, int S, int stride, int pad,
                             int algo, void* ws, size_t ws_bytes, b200_stream_t stream,
                             double* stats = nullptr, bool* fused = nullptr, const EpiStatsFinal* fin = nullptr,
                             const EpiBnBwd* bb = nullptr) {
  B200_REQUIRE(dy && w_crsk && dx, "conv2d_dgrad: null pointer");
  B200_REQUIRE(stride == 1 || stride == 2, "conv2d_dgrad: stride %d unsupported", stride);
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  cudaStream_t st = as_stream(stream);
  const bool tc = use_tc(algo, B200_PASS_DGRAD, N, H, W, C, K, R, S, stride, pad);
  B200_REQUIRE(tc || algo != B200_ALGO_TC, "conv2d_dgrad: shape not supported by the tcgen05 path");
  if (!tc) {
    ConvDims d{N, H, W, C, K, R, S, stride, pad, P, Q};
    const size_t total = (size_t)N * H * W * C;
    launch_k(conv_dgrad_direct_kernel, ew_grid(total), EW_THREADS, 0, st, (const bf16*)dy, (const bf16*)w_crsk, (const bf16*)(bb ? nullptr : addend), (bf16*)dx, d);
    B200_LAUNCH_CHECK("conv_dgrad_direct_kernel");
    return 0;
  }
  if (stride == 1) {
    // dx[h,w] = sum_{r,s} dy[h + pad - r, w + pad - s] . W[:, r, s, :]
    TapTable tt;
    memset(&tt, 0, sizeof(tt));
    for (int r = 0; r < R; ++r)
      for (int s = 0; s < S; ++s) {
        const int i = tt.n++;
        tt.dh[i] = pad - r; tt.dw[i] = pad - s; tt.dn[i] = 0;
        tt.wcol[i] = (r * S + s) * K;
      }
    return run_conv_tc(dy, N, P, Q, K, w_crsk, C, R * S * K, tt, dx, addend, nullptr, N, H, W, st, stats, fused, fin,
                       1, nullptr, 2, 0, bb);
  }
  // stride 2, ONE launch: the four output parity phases (a, b) are extra tiles of the SM-pair kernel, each
  // with its own subset of the taps; the epilogue writes dx (+ addend) in place at (2h' + a, 2w' + b).
  // (round 1: one launch per phase into a phase-split workspace + a merge kernel: 409 / 512 TFLOP/s)
  {
    PhasePlan pp;
    TapTable all;
    const bool all_phases = build_dgrad_phases(R, S, K, pad, &pp, &all);
    const int BNd = pick_bn(C, 16, 256);
    const TilePlan tp = plan_tiles(N, H / 2, W / 2);
    const bool pair_ok = conv_use_pair() && BNd > 0 && BNd % 32 == 0 &&
                         (tp.tiles_w * tp.tiles_h * tp.tiles_n) % 2 == 0 && R * S <= TC_MAX_TAPS;
    static const int single = env_int("B200_DGRAD_S2_SINGLE", 1);
    if (all_phases && pair_ok && single)
      return run_conv_tc(dy, N, P, Q, K, w_crsk, C, R * S * K, all, dx, addend, nullptr, N, H, W, st, stats,
                         fused, fin, 1, &pp, 2, 0, bb);
  }
  if (bb) addend = nullptr;   // the per-phase fallback below does not fuse: x must not be added
  // fallback: one launch per output parity phase (a, b), into the parity-split workspace
  const size_t need = (size_t)N * H * W * C * 2;
  B200_REQUIRE(ws && ws_bytes >= need, "conv2d_dgrad: workspace too small (%zu < %zu)", ws_bytes, need);
  const int H2 = H / 2, W2 = W / 2;
  const size_t phase_elems = (size_t)N * H2 * W2 * C;
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) {
      TapTable tt;
      memset(&tt, 0, sizeof(tt));
      for (int r = 0; r < R; ++r) {
        if (mod2(a + pad - r) != 0) continue;
        for (int s = 0; s < S; ++s) {
          if (mod2(b + pad - s) != 0) continue;
          const int i = tt.n++;
          tt.dh[i] = floordiv2(a + pad - r); tt.dw[i] = floordiv2(b + pad - s); tt.dn[i] = 0;
          tt.wcol[i] = (r * S + s) * K;
        }
      }
      bf16* dst = reinterpret_cast<bf16*>(ws) + (size_t)(a * 2 + b) * phase_elems;
      if (tt.n == 0) {
        B200_CUDA(cudaMemsetAsync(dst, 0, phase_elems * 2, st));
        continue;
      }
      if (int rc = run_conv_tc(dy, N, P, Q, K, w_crsk, C, R * S * K, tt, dst, nullptr, nullptr, N, H2,
                               W2, st))
        return rc;
    }
  launch_k(parity_merge_add_kernel, ew_grid((size_t)N * H * W * C / 8), EW_THREADS, 0, st, (const bf16*)ws, (const bf16*)addend, (bf16*)dx, N, H, W, C);
  B200_LAUNCH_CHECK("parity_merge_add_kernel");
  return 0;
}

extern "C" int b200_conv2d_dgrad(const void* dy, const void* w_crsk, const void* addend, void* dx,
                                 int N, int H, int W, int C, int K, int R, int S, int stride, int pad,
                                 int algo, void* ws, size_t ws_bytes, b200_stream_t stream) {
  take_det_flag(algo);
  return conv2d_dgrad_impl(dy, w_crsk, addend, dx, N, H, W, C, K, R, S, stride, pad, algo, ws, ws_bytes, stream);
}

// dgrad whose output dx is the dy of a BN + ReLU + dropout backward (b200_bn_act_bwd with a mask): the epilogue
// also accumulates sum(g) and sum(g * x_bn) per channel, g = dx masked (and scaled by 1/(1-p)), and the last CTA
// writes dbeta / dgamma - the whole reduce pass of that backward. *fused = 1 when this happened (then call
// b200_bn_act_bwd_apply), 0 when the shape ran on a kernel without the fused epilogue (then call b200_bn_act_bwd).
extern "C" int b200_conv2d_dgrad_bnbwd(const void* dy, const void* w_crsk, void* dx, int N, int H, int W, int C,
                                       int K, int R, int S, int stride, int pad, int algo, void* ws,
                                       size_t ws_bytes, const void* x_bn, const void* mask, const float* mean,
                                       const float* invstd, float dropout_p, float* dgamma, float* dbeta,
                                       void* stats_ws, size_t stats_ws_bytes, int* fused, b200_stream_t stream) {
  take_det_flag(algo);
  B200_REQUIRE(x_bn && mask && mean && invstd && dgamma && dbeta && stats_ws && fused,
               "conv2d_dgrad_bnbwd: null pointer");
  B200_REQUIRE(stats_ws_bytes >= b200_bn_workspace_bytes(0, C), "conv2d_dgrad_bnbwd: statistics workspace too small");
  B200_REQUIRE((reinterpret_cast<uintptr_t>(stats_ws) & 7) == 0 && (reinterpret_cast<uintptr_t>(mask) & 1) == 0,
               "conv2d_dgrad_bnbwd: statistics workspace must be 8-byte, the mask 2-byte aligned");
  B200_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "conv2d_dgrad_bnbwd: dropout_p out of range");
  double* accum = reinterpret_cast<double*>(stats_ws);
  EpiStatsFinal fin;
  memset(&fin, 0, sizeof(fin));
  fin.ticket = reinterpret_cast<unsigned int*>(accum + BN_SLOTS * bn_slot_stride(C));
  fin.mean = const_cast<float*>(mean); fin.invstd = const_cast<float*>(invstd);
  fin.rows = (long long)N * H * W;
  fin.dgamma = dgamma; fin.dbeta = dbeta;
  EpiBnBwd bb;
  bb.mask = reinterpret_cast<const uint8_t*>(mask);
  bb.inv_keep = 1.f / (1.f - dropout_p);
  bb.drop = dropout_p > 0.f ? 1 : 0;
  bool f = false;
  // stride 2 (four output phases per launch) is left to the separate reduction pass: measured at batch 128, the
  // fused epilogue costs 30.7 / 17.0 us on the 160<-320 @32x32 / 320<-640 @16x16 layers against 19.9 / 14.9 us
  // for b200_bn_act_bwd's own pass, while at stride 1 it costs 18.5 / 9.0 / 10.0 us against 19.9 / 14.9 / 14.0 us
  const bool fuse = stride == 1;
  const int rc = fuse ? conv2d_dgrad_impl(dy, w_crsk, x_bn, dx, N, H, W, C, K, R, S, stride, pad, algo, ws, ws_bytes,
                                          stream, accum, &f, &fin, &bb)
                      : conv2d_dgrad_impl(dy, w_crsk, nullptr, dx, N, H, W, C, K, R, S, stride, pad, algo, ws,
                                          ws_bytes, stream);
  *fused = f ? 1 : 0;
  return rc;
}

static int wgrad_cluster_size() {
  // B200_WGRAD_CLUSTER = 1 | 2 | 4 (default 2): CTAs per cluster sharing the multicast dY slabs
  static const int v = env_int("B200_WGRAD_CLUSTER", 1);  // measured: no gain from multicasting dY (round 1)
  return (v == 1 || v == 2 || v == 4) ? v : 1;
}

static int wgrad_mtiles_per_cta() {
  // B200_WGRAD_MT = 0 (auto) | 1 | 2: M tiles (TMEM accumulators) per CTA sharing each dY stage.
  // Measured in round 1 (after the producer's index math was hoisted): two tiles with 128-pixel stages
  // reach 928 / 902 TFLOP/s at C = 160 / 320 against 818 / 751 with one tile (28 % fewer bytes per MMA
  // through the TMA/L2 path), but 692 against 720 at C = 640, hence the auto rule in run_wgrad_tc.
  static const int v = env_int("B200_WGRAD_MT", 0);
  return (v < 0 || v > 2) ? 0 : v;
}

template <int SL, int CS, int MT, bool TF32 = false>
static int launch_wgrad_tc(const CUtensorMap& tmX, const CUtensorMap& tmDy, WgradTcArgs& a,
                           cudaStream_t st) {
  const int max_dyn = 228352;
  B200_CUDA(ensure_max_smem<wgrad_tc_kernel<SL, CS, MT, TF32>>(max_dyn));
  a.stage_bytes = (uint32_t)(MT * (128 / SL) + a.nb) * a.slab_bytes;
  a.stages = std::min<int>(8, (max_dyn - 1024) / (int)a.stage_bytes);
  static const int stages_env = env_int("B200_WGRAD_STAGES", 0);
  if (stages_env > 0) a.stages = std::max(2, std::min(a.stages, stages_env));
  B200_REQUIRE(a.stages >= 2, "wgrad_tc: tile does not fit in shared memory");
  a.tmem_cols = 32;
  while (a.tmem_cols < (MT - 1) * 256 + a.BN) a.tmem_cols *= 2;
  size_t dyn = (size_t)a.stages * a.stage_bytes + 1024;
  dyn = std::max<size_t>(dyn, 120 * 1024);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(a.n_mgroups * a.n_ntiles, a.splits);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = dyn;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  B200_CUDA(cudaLaunchKernelEx(&cfg, wgrad_tc_kernel<SL, CS, MT, TF32>, tmX, tmDy, a));
  B200_LAUNCH_CHECK("wgrad_tc_kernel");
  return 0;
}

template <int SL>
static int launch_wgrad_tc_cs(int cs, int mt, const CUtensorMap& tmX, const CUtensorMap& tmDy,
                              WgradTcArgs& a, cudaStream_t st) {
  if (mt == 2) {
    switch (cs) {
      case 4: return launch_wgrad_tc<SL, 4, 2>(tmX, tmDy, a, st);
      case 2: return launch_wgrad_tc<SL, 2, 2>(tmX, tmDy, a, st);
      default: return launch_wgrad_tc<SL, 1, 2>(tmX, tmDy, a, st);
    }
  }
  switch (cs) {
    case 4: return launch_wgrad_tc<SL, 4, 1>(tmX, tmDy, a, st);
    case 2: return launch_wgrad_tc<SL, 2, 1>(tmX, tmDy, a, st);
    default: return launch_wgrad_tc<SL, 1, 1>(tmX, tmDy, a, st);
  }
}

// Pixel-range splits of a wgrad launch. Cost model in units of one pipeline stage:
//   time(sp) = waves(cols * sp CTAs) * (stages per CTA + fixed), fixed = prologue + TMEM drain with
// atomics + launch tail expressed in stages. Minimising it fills whole waves of the SMs without paying
// the fixed part more often than needed (a 2-wave grid of half-length CTAs is slower than a 1-wave one).
static int pick_wgrad_splits(int cols, int num_ptiles, int fixed_units) {
  const int sms = num_sms();
  int best = 1;
  double best_cost = 1e30;
  const int max_splits = std::min(num_ptiles, 64);
  for (int sp = 1; sp <= max_splits; ++sp) {
    const int per = (num_ptiles + sp - 1) / sp;
    if ((num_ptiles + per - 1) / per != sp) continue;  // would leave empty splits
    const long total = (long)cols * sp;
    const long waves = (total + sms - 1) / sms;
    const double cost = (double)waves * (per + fixed_units) * (1.0 + 0.001 * sp);  // ties: fewer atomics
    if (cost < best_cost) { best_cost = cost; best = sp; }
  }
  static const int splits_env = env_int("B200_WGRAD_SPLITS", 0);
  if (splits_env > 0) best = std::min(splits_env, num_ptiles);
  const int per = (num_ptiles + best - 1) / best;
  return (num_ptiles + per - 1) / per;
}

// deterministic mode: sum `splits` partials of n floats (stride apart) in order into out
static int wgrad_reduce_splits(const float* part, float* out, size_t n, size_t stride, int splits, cudaStream_t st) {
  const size_t work = (n % 4 == 0) ? n / 4 : n;
  launch_k(wgrad_reduce_splits_kernel, ew_grid(work), EW_THREADS, 0, st, part, out, n, stride, splits);
  B200_LAUNCH_CHECK("wgrad_reduce_splits_kernel");
  return 0;
}

// Where the pixel-range splits of a wgrad launch put their results: into the partial buffer of a deterministic
// call (returns 1), else into dw, zeroed here when there is more than one split (returns 0); < 0: error.
static int wgrad_split_target(const WgradDet* det, int splits, size_t n, float* dw, cudaStream_t st, float** part,
                              size_t* part_stride) {
  *part = nullptr;
  *part_stride = 0;
  if (splits <= 1) return 0;
  if (det && det->part) {
    if (det->bytes < (size_t)splits * n * 4) {
      fail(1, "conv2d_wgrad: deterministic workspace too small (%zu < %zu bytes)", det->bytes, (size_t)splits * n * 4);
      return -2;
    }
    *part = det->part;
    *part_stride = n;
    return 1;
  }
  if (cudaMemsetAsync(dw, 0, n * 4, st) != cudaSuccess) {
    fail(2, "cudaMemsetAsync(dw) failed");
    return -2;
  }
  return 0;
}

static bool wgrad_use_halo() {
  // B200_WGRAD_HALO=0 falls back to the one-window-per-slab kernel
  static const int v = env_int("B200_WGRAD_HALO", 1);
  return v != 0;
}

// Halo-reuse SM-pair wgrad (3x3, stride 1, pad 1): see wgrad_tc2h_kernel. Returns -1 when the shape is
// not covered (the caller then uses the general kernel).
static int run_wgrad_tc2h(const void* act, const void* dy, int N, int P, int Q, int C, int K,
                          const TapTable& taps, float* dw, cudaStream_t st, WgradDet* det) {
  if (taps.n != 9 || C % 32 != 0 || K % 32 != 0 || Q % 8 != 0) return -1;
  for (int t = 0; t < 9; ++t)
    if (taps.dh[t] != t / 3 - 1 || taps.dw[t] != t % 3 - 1 || taps.dn[t] != 0) return -1;
  int bh, bn;
  if (P % 16 == 0) { bh = 16; bn = 1; }
  else if (P < 16 && 16 % P == 0 && N % (16 / P) == 0) { bh = P; bn = 16 / P; }
  else return -1;
  const int BN = pick_bn(K, 32, 160);
  if (BN <= 0) return -1;
  static const int pw_env = env_int("B200_WGRAD_PW", 10);
  const int pw = (pw_env == 16) ? 16 : 10;  // box bytes stay 1 KB multiples
  WgradHaloArgs a;
  memset(&a, 0, sizeof(a));
  a.bh = bh; a.bn = bn; a.pw = pw;
  a.tiles_w = Q / 8; a.tiles_h = P / bh;
  a.num_ptiles = a.tiles_w * a.tiles_h * (N / bn);
  a.ncombo = 3 * (C / 32);
  a.ncols = ((a.ncombo + 3) / 4 + 1) / 2 * 2;
  a.BN = BN; a.n_ntiles = K / BN;
  a.nbh = (BN / 2 + 31) / 32;
  a.ktot = 9 * C;
  a.box_bytes = (uint32_t)((16 * pw * 64 + 1023) / 1024 * 1024);
  a.slab_bytes = 128 * 64;
  a.stage_bytes = 4 * a.box_bytes + (uint32_t)a.nbh * a.slab_bytes;
  const int max_dyn = 228352;
  a.stages = std::min<int>(WGH_STAGES_MAX, (max_dyn - 1024) / (int)a.stage_bytes);
  static const int stages_env = env_int("B200_WGRAD_STAGES", 0);
  if (stages_env > 0) a.stages = std::max(2, std::min(a.stages, stages_env));
  if (a.stages < 2) return -1;
  a.splits = pick_wgrad_splits(a.ncols * a.n_ntiles, a.num_ptiles, 5);
  for (int t = 0; t < 9; ++t) a.wcol[t] = taps.wcol[t];
  a.dw = dw;
  if (det && det->dry) { det->splits = a.splits; return 0; }
  B200_CUDA(ensure_max_smem<wgrad_tc2h_kernel>(max_dyn));
  if (wgrad_split_target(det, a.splits, (size_t)K * a.ktot, dw, st, &a.part, &a.part_stride) < 0) return 1;
  CUtensorMap tmX, tmDy;
  if (int rc = make_tmap_nhwc(&tmX, act, N, P, Q, C, 32, pw, bh, bn)) return rc;
  if (int rc = make_tmap_nhwc(&tmDy, dy, N, P, Q, K, 32, 8, bh, bn)) return rc;
  size_t dyn = (size_t)a.stages * a.stage_bytes + 1024;
  dyn = std::max<size_t>(dyn, 120 * 1024);  // one CTA per SM (512 TMEM columns each)
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(a.ncols * a.n_ntiles, a.splits);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = dyn;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  B200_CUDA(cudaLaunchKernelEx(&cfg, wgrad_tc2h_kernel, tmX, tmDy, a));
  B200_LAUNCH_CHECK("wgrad_tc2h_kernel");
  if (a.part) return wgrad_reduce_splits(a.part, dw, (size_t)K * a.ktot, a.part_stride, a.splits, st);
  return 0;
}

// Shifted-window wgrad launch. act: [Nact][Ha][Wa][C] bf16, dy: [N][P][Q][K] bf16,
// dw: fp32 [K][ntaps*C] (row pitch = taps.n * C).
// fp32 / TF32 precision mode: fp32 x and dY, 16-channel slabs (64-byte rows, the byte geometry of the bf16
// kernel's 32-channel slabs), one M tile per CTA, N tile <= 80 so that two stages fit.
static int run_wgrad_tc_tf32(const void* act, int Nact, int Ha, int Wa, int C, const void* dy, int N, int P,
                             int Q, int K, const TapTable& taps, float* dw, cudaStream_t st, int cstride) {
  constexpr int SL = 16;
  B200_REQUIRE(C % SL == 0 && K % SL == 0, "wgrad_tc (tf32): C and K must be multiples of 16");
  const int BN = pick_bn(K, SL, 80);
  B200_REQUIRE(BN > 0, "wgrad_tc (tf32): no legal N tile for K=%d", K);
  TilePlan t = plan_tiles_mult16(N, P, Q, 128);
  B200_REQUIRE(t.rows_valid % 16 == 0, "wgrad_tc (tf32): pixel tile of %d rows is not a multiple of 16", t.rows_valid);
  WgradTcArgs a;
  memset(&a, 0, sizeof(a));
  a.bw = t.bw; a.bh = t.bh; a.bn = t.bn;
  a.tiles_w = t.tiles_w; a.tiles_h = t.tiles_h; a.tiles_n = t.tiles_n;
  a.num_ptiles = t.tiles_w * t.tiles_h * t.tiles_n;
  a.kmmas = t.rows_valid / 8;
  a.slab_bytes = (uint32_t)((t.rows_valid * SL * 4 + 1023) / 1024 * 1024);
  a.cin = C;
  a.slabs_per_tap = C / SL;
  a.nslabs_total = taps.n * a.slabs_per_tap;
  const int spm = 128 / SL;
  a.n_mtiles = (a.nslabs_total + spm - 1) / spm;
  a.n_mgroups = a.n_mtiles;
  a.BN = BN; a.n_ntiles = K / BN;
  a.nb = BN / SL;
  a.ktot = taps.n * C;
  a.splits = pick_wgrad_splits(a.n_mgroups * a.n_ntiles, a.num_ptiles, 8);
  a.taps = taps;
  a.dw = dw;
  a.cstride = cstride;
  if (a.splits > 1) B200_CUDA(cudaMemsetAsync(dw, 0, (size_t)K * a.ktot * 4, st));
  CUtensorMap tmX, tmDy;
  if (int rc = make_tmap_nhwc(&tmX, act, Nact, Ha, Wa, C, SL, t.bw, t.bh, t.bn, cstride, 4)) return rc;
  if (int rc = make_tmap_nhwc(&tmDy, dy, N, P, Q, K, SL, t.bw, t.bh, t.bn, 1, 4)) return rc;
  return launch_wgrad_tc<SL, 1, 1, true>(tmX, tmDy, a, st);
}

static int run_wgrad_tc(const void* act, int Nact, int Ha, int Wa, int C, const void* dy, int N, int P,
                        int Q, int K, const TapTable& taps, float* dw, cudaStream_t st, int cstride = 1,
                        WgradDet* det = nullptr) {
  if (wgrad_use_halo() && Nact == N && Ha == P && Wa == Q && cstride == 1) {
    const int rc = run_wgrad_tc2h(act, dy, N, P, Q, C, K, taps, dw, st, det);
    if (rc >= 0) return rc;
  }
  // slab width: 32 channels (64-byte TMA rows, SWIZZLE_64B) or 16; 64-channel slabs (SWIZZLE_128B, with
  // partial last slabs) are implemented and tested but were not faster (round 1), B200_WGRAD_SLAB=64
  int SL = (C % 32 == 0 && K % 32 == 0) ? 32 : 16;
  static const int slab_env = env_int("B200_WGRAD_SLAB", 0);
  if ((slab_env == 16 || slab_env == 32) && C % slab_env == 0 && K % slab_env == 0) SL = slab_env;
  if (slab_env == 64 && C >= 64 && K >= 64) SL = 64;
  int BN = pick_bn(K, 16, 160);
  if (SL < 64) BN = pick_bn(K, SL, 160);
  B200_REQUIRE(BN > 0, "wgrad_tc: no legal N tile for K=%d", K);
  const int cs = wgrad_cluster_size();
  int mt = wgrad_mtiles_per_cta();
  if (mt == 0) mt = (C <= 320) ? 2 : 1;
  static const int px_env = env_int("B200_WGRAD_PX", 128);
  const int px_cap = (px_env == 64) ? 64 : 128;
  TilePlan t = plan_tiles_mult16(N, P, Q, px_cap);
  if (t.rows_valid % 16 != 0 && mt == 2) { mt = 1; t = plan_tiles_mult16(N, P, Q, 128); }
  B200_REQUIRE(t.rows_valid % 16 == 0, "wgrad_tc: pixel tile of %d rows is not a multiple of 16",
               t.rows_valid);
  WgradTcArgs a;
  memset(&a, 0, sizeof(a));
  a.bw = t.bw; a.bh = t.bh; a.bn = t.bn;
  a.tiles_w = t.tiles_w; a.tiles_h = t.tiles_h; a.tiles_n = t.tiles_n;
  a.num_ptiles = t.tiles_w * t.tiles_h * t.tiles_n;
  a.kmmas = t.rows_valid / 16;
  a.slab_bytes = (uint32_t)((t.rows_valid * SL * 2 + 1023) / 1024 * 1024);
  a.cin = C;
  a.slabs_per_tap = (C + SL - 1) / SL;
  a.nslabs_total = taps.n * a.slabs_per_tap;
  const int spm = 128 / SL;
  a.n_mtiles = (a.nslabs_total + spm - 1) / spm;
  if (a.n_mtiles < 2) mt = 1;
  a.BN = BN;
  a.nb = (BN + SL - 1) / SL;
  if (mt == 2 && 2 * (size_t)(2 * spm + a.nb) * a.slab_bytes > 228352 - 1024) mt = 1;  // needs 2 stages
  a.n_mgroups = ((a.n_mtiles + mt - 1) / mt + cs - 1) / cs * cs;
  a.BN = BN; a.n_ntiles = K / BN;
  a.nb = (BN + SL - 1) / SL;
  a.ktot = taps.n * C;
  const int cols = a.n_mgroups * a.n_ntiles;
  a.splits = pick_wgrad_splits(cols, a.num_ptiles, 8);
  a.taps = taps;
  a.dw = dw;
  a.cstride = cstride;
  B200_REQUIRE(cstride == 1 || (t.bw * cstride <= 256 && t.bh * cstride <= 256),
               "wgrad_tc: strided TMA box exceeds 256 elements");
  if (det && det->dry) { det->splits = a.splits; return 0; }
  if (wgrad_split_target(det, a.splits, (size_t)K * a.ktot, dw, st, &a.part, &a.part_stride) < 0) return 1;
  CUtensorMap tmX, tmDy;
  if (int rc = make_tmap_nhwc(&tmX, act, Nact, Ha, Wa, C, SL, t.bw, t.bh, t.bn, cstride)) return rc;
  if (int rc = make_tmap_nhwc(&tmDy, dy, N, P, Q, K, SL, t.bw, t.bh, t.bn)) return rc;
  int rc;
  if (SL == 64) rc = launch_wgrad_tc_cs<64>(cs, mt, tmX, tmDy, a, st);
  else if (SL == 32) rc = launch_wgrad_tc_cs<32>(cs, mt, tmX, tmDy, a, st);
  else rc = launch_wgrad_tc_cs<16>(cs, mt, tmX, tmDy, a, st);
  if (rc) return rc;
  if (a.part) return wgrad_reduce_splits(a.part, dw, (size_t)K * a.ktot, a.part_stride, a.splits, st);
  return 0;
}

// geometry shared by b200_conv2d_wgrad and its workspace query
static int dbias_pix_per_block(size_t npix, int K) {
  // ONE block per SM: every block ends with K same-address atomics, which serialise (592 blocks took 46 us
  // for the 42 MB stem gradient in round 2's launch list, most of it in the atomics)
  // ... but a block streams only ~1.3 TB/s / 148 with its 256 x 8 16-byte loads in flight: tensors far beyond the
  // WRN stem's 42 MB (the 3.3 GB ImageNet-shape stem gradient took 2.5 ms per step, 5x its HBM time) get up to 8
  // blocks per SM, one more per 64 MB
  const size_t per_sm = std::min<size_t>(8, std::max<size_t>(1, (npix * (size_t)K * 2) >> 26));
  const size_t blocks = (size_t)num_sms() * per_sm;
  return (int)std::max<size_t>(64, (npix + blocks - 1) / blocks);
}
static int direct_wgrad_chunks(int total, size_t npix, int* pix_per_chunk) {
  const int bx = (total + 255) / 256;
  int chunks = (int)std::max<size_t>(1, std::min<size_t>((size_t)num_sms() * 8 / bx + 1, npix / 64 + 1));
  const int ppc = (int)((npix + chunks - 1) / chunks);
  *pix_per_chunk = ppc;
  return (int)((npix + ppc - 1) / ppc);
}

// Deterministic wgrad workspace = [im2col region][bias-gradient partials][filter-gradient partials]; sizes of the
// last two (0 when the launch would not split)
static void wgrad_det_regions(int N, int H, int W, int C, int K, int R, int S, int stride, int pad, int algo,
                              size_t* dbias_bytes, size_t* part_bytes) {
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  const size_t npix = (size_t)N * P * Q;
  const int ppc = dbias_pix_per_block(npix, K);
  *dbias_bytes = align_up((npix + ppc - 1) / ppc * (size_t)K * 4, 1024);
  *part_bytes = 0;
  WgradDet dry = {nullptr, 0, true, 1};
  const bool tc = use_tc(algo, B200_PASS_WGRAD, N, H, W, C, K, R, S, stride, pad);
  if (!tc && use_im2col(algo, B200_PASS_WGRAD, N, H, W, C, K, R, S, stride, pad)) {
    const int kpad = im2col_kpad(R, S, C);
    TapTable tt;
    memset(&tt, 0, sizeof(tt));
    tt.n = 1;
    if (run_wgrad_tc(nullptr, N, P, Q, kpad, nullptr, N, P, Q, K, tt, nullptr, nullptr, 1, &dry) == 0 && dry.splits > 1)
      *part_bytes = align_up((size_t)dry.splits * K * kpad * 4, 1024);
    return;
  }
  if (!tc) {
    int ppc_w;
    const int chunks = direct_wgrad_chunks(K * R * S * C, npix, &ppc_w);
    if (chunks > 1) *part_bytes = align_up((size_t)chunks * K * R * S * C * 4, 1024);
    return;
  }
  TapTable tt = fprop_taps(C, R, S, pad);
  if (run_wgrad_tc(nullptr, N, H, W, C, nullptr, N, P, Q, K, tt, nullptr, nullptr, stride, &dry) == 0 && dry.splits > 1)
    *part_bytes = align_up((size_t)dry.splits * K * R * S * C * 4, 1024);
}

extern "C" int b200_conv2d_wgrad(const void* dy, const void* x, float* dw_krsc, float* dbias, int N,
                                 int H, int W, int C, int K, int R, int S, int stride, int pad,
                                 int algo, void* ws, size_t ws_bytes, b200_stream_t stream) {
  take_det_flag(algo);
  const bool det = g_det != 0;
  B200_REQUIRE(dy && x && dw_krsc, "conv2d_wgrad: null pointer");
  B200_REQUIRE(stride == 1 || stride == 2, "conv2d_wgrad: stride %d unsupported", stride);
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  cudaStream_t st = as_stream(stream);
  const size_t npix = (size_t)N * P * Q;
  const bool tc = use_tc(algo, B200_PASS_WGRAD, N, H, W, C, K, R, S, stride, pad);
  const bool im2col = !tc && use_im2col(algo, B200_PASS_WGRAD, N, H, W, C, K, R, S, stride, pad);
  // workspace regions (see wgrad_det_regions)
  size_t base_bytes = 0, dbias_bytes = 0, part_bytes = 0;
  if (im2col) {
    const int kpad = im2col_kpad(R, S, C);
    base_bytes = align_up((size_t)N * P * Q * kpad * 2, 1024) + align_up((size_t)K * kpad * 4, 1024);
  }
  if (det) {
    wgrad_det_regions(N, H, W, C, K, R, S, stride, pad, algo, &dbias_bytes, &part_bytes);
    B200_REQUIRE(ws && ws_bytes >= base_bytes + dbias_bytes + part_bytes && (reinterpret_cast<uintptr_t>(ws) & 15) == 0,
                 "conv2d_wgrad: deterministic mode needs a 16-byte aligned workspace of %zu bytes (got %zu)",
                 base_bytes + dbias_bytes + part_bytes, ws_bytes);
  }
  float* dbias_part = det ? reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ws) + base_bytes) : nullptr;
  WgradDet wd = {det ? reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ws) + base_bytes + dbias_bytes) : nullptr,
                 part_bytes, false, 1};
  if (dbias) {
    B200_REQUIRE(K % 8 == 0, "conv2d_wgrad: dbias needs K %% 8 == 0 (K=%d)", K);
    const int ppc = dbias_pix_per_block(npix, K);
    const unsigned nblk = (unsigned)((npix + ppc - 1) / ppc);
    const bool part = det && nblk > 1;
    if (!part) B200_CUDA(cudaMemsetAsync(dbias, 0, (size_t)K * 4, st));
    launch_k(conv_dbias_kernel, dim3(nblk, 1), 256, 0, st, (const bf16*)dy, dbias, npix, K, ppc,
             part ? dbias_part : (float*)nullptr);
    B200_LAUNCH_CHECK("conv_dbias_kernel");
    if (part)
      if (int rc = wgrad_reduce_splits(dbias_part, dbias, (size_t)K, (size_t)K, (int)nblk, st)) return rc;
  }
  if (im2col) {
    const int kpad = im2col_kpad(R, S, C);
    const size_t col_bytes = align_up((size_t)N * P * Q * kpad * 2, 1024);
    B200_REQUIRE(ws && ws_bytes >= col_bytes + (size_t)K * kpad * 4, "conv2d_wgrad: workspace too small");
    bf16* col = reinterpret_cast<bf16*>(ws);
    float* dwpad = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ws) + col_bytes);
    launch_k(im2col_kernel, ew_grid((size_t)N * P * Q * kpad), EW_THREADS, 0, st, (const bf16*)x, col, N, H, W, C, R, S, stride, pad, P, Q, kpad);
    B200_LAUNCH_CHECK("im2col_kernel");
    TapTable tt;
    memset(&tt, 0, sizeof(tt));
    tt.n = 1;
    if (int rc = run_wgrad_tc(col, N, P, Q, kpad, dy, N, P, Q, K, tt, dwpad, st, 1, det ? &wd : nullptr)) return rc;
    launch_k(repitch_rows_kernel<float>, ew_grid((size_t)K * R * S * C), EW_THREADS, 0, st, dwpad, dw_krsc, K, kpad, R * S * C);
    B200_LAUNCH_CHECK("repitch_rows_kernel");
    return 0;
  }
  B200_REQUIRE(tc || algo != B200_ALGO_TC, "conv2d_wgrad: shape not supported by the tcgen05 path");
  if (!tc) {
    ConvDims d{N, H, W, C, K, R, S, stride, pad, P, Q};
    const int total = K * R * S * C;
    const int bx = (total + 255) / 256;
    int ppc;
    const int chunks = direct_wgrad_chunks(total, npix, &ppc);
    const bool part = det && chunks > 1;
    if (chunks > 1 && !part) B200_CUDA(cudaMemsetAsync(dw_krsc, 0, (size_t)total * 4, st));
    launch_k(conv_wgrad_direct_kernel, dim3(bx, chunks), 256, 0, st, (const bf16*)dy, (const bf16*)x,
                                                               dw_krsc, d, ppc, part ? wd.part : (float*)nullptr);
    B200_LAUNCH_CHECK("conv_wgrad_direct_kernel");
    if (part) return wgrad_reduce_splits(wd.part, dw_krsc, (size_t)total, (size_t)total, chunks, st);
    return 0;
  }
  TapTable tt = fprop_taps(C, R, S, pad);   // stride 2: strided TMA windows of x, no parity-split copy
  return run_wgrad_tc(x, N, H, W, C, dy, N, P, Q, K, tt, dw_krsc, st, stride, det ? &wd : nullptr);
}

// -------------------------------------------------------------------------------------------------
// fp32 / TF32 precision mode (the reference's evaluation path and its non-AMP training path)
// -------------------------------------------------------------------------------------------------
extern "C" int b200_conv2d_tf32_supported(int pass, int N, int H, int W, int C, int K, int R, int S, int stride,
                                          int pad) {
  int P, Q;
  if (N < 1 || R * S > TC_MAX_TAPS || (stride != 1 && stride != 2)) return 0;
  if (!same_geometry(H, W, R, S, stride, pad, &P, &Q)) return 0;
  if (pass == B200_PASS_WGRAD) {
    // The kind::tf32 wgrad (both operands MN-major fp32) is compiled in but returned all zeros on B200 in round 2
    // (gpurun_out/call10.out) and is switched off until that is understood: B200_TF32_WGRAD=1 enables it.
    static const int on = env_int("B200_TF32_WGRAD", 0);
    if (!on || C % 16 != 0 || K % 16 != 0) return 0;
    return plan_tiles_mult16(N, P, Q, 128).rows_valid % 16 == 0;
  }
  // fprop / dgrad run on the SM-pair kernel only: even pixel-tile count, N tile a multiple of 32
  const int Cin = pass == B200_PASS_DGRAD ? K : C, Cout = pass == B200_PASS_DGRAD ? C : K;
  if (Cin % 8 != 0) return 0;
  const int BN = pick_bn(Cout, 16, 256);
  if (BN <= 0 || BN % 32 != 0) return 0;
  const int Po = pass == B200_PASS_DGRAD ? H : P, Qo = pass == B200_PASS_DGRAD ? W : Q;
  TilePlan t = (pass == B200_PASS_DGRAD && stride == 2) ? plan_tiles(N, Po / 2, Qo / 2) : plan_tiles(N, Po, Qo);
  if ((t.tiles_w * t.tiles_h * t.tiles_n) % 2 != 0) return 0;
  if (pass == B200_PASS_DGRAD && stride == 2 && (R < 2 || S < 2)) return 0;
  return 1;
}

// im2col route of the few-input-channel stems in the fp32 mode: K = R*S*C padded to 32 fp32 columns
static bool tf32_use_im2col(int N, int H, int W, int C, int K, int R, int S, int stride, int pad) {
  if (C >= 8 || R * S * C > 1024) return false;
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  if (P < 1 || Q < 1) return false;
  return b200_conv2d_tf32_supported(B200_PASS_FPROP, N, P, Q, im2col_kpad(R, S, C), K, 1, 1, 1, 0) != 0;
}

extern "C" size_t b200_conv2d_tf32_workspace_bytes(int N, int H, int W, int C, int K, int R, int S, int stride,
                                                   int pad) {
  if (b200_conv2d_tf32_supported(B200_PASS_FPROP, N, H, W, C, K, R, S, stride, pad)) return 0;
  if (!tf32_use_im2col(N, H, W, C, K, R, S, stride, pad)) return 0;
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  const size_t kpad = im2col_kpad(R, S, C);
  return align_up((size_t)N * P * Q * kpad * 4, 1024) + align_up((size_t)K * kpad * 4, 1024);
}

extern "C" int b200_conv2d_fprop_tf32(const float* x, const float* w_krsc, const float* bias,
                                      const float* residual, float* y, int N, int H, int W, int C, int K,
                                      int R, int S, int stride, int pad, int relu, void* ws, size_t ws_bytes,
                                      b200_stream_t stream) {
  g_det = 0;
  B200_REQUIRE(x && w_krsc && y, "conv2d_fprop_tf32: null pointer");
  B200_REQUIRE(stride == 1 || stride == 2, "conv2d_fprop_tf32: stride %d unsupported", stride);
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  B200_REQUIRE(P > 0 && Q > 0, "conv2d_fprop_tf32: empty output");
  cudaStream_t st = as_stream(stream);
  if (b200_conv2d_tf32_supported(B200_PASS_FPROP, N, H, W, C, K, R, S, stride, pad)) {
    TapTable tt = fprop_taps(C, R, S, pad);
    return run_conv_tc(x, N, H, W, C, w_krsc, K, R * S * C, tt, y, residual, bias, N, P, Q, st, nullptr, nullptr,
                       nullptr, stride, nullptr, 4, relu);
  }
  if (tf32_use_im2col(N, H, W, C, K, R, S, stride, pad)) {
    const int kpad = im2col_kpad(R, S, C);
    const size_t col_bytes = align_up((size_t)N * P * Q * kpad * 4, 1024);
    B200_REQUIRE(ws && ws_bytes >= col_bytes + (size_t)K * kpad * 4, "conv2d_fprop_tf32: workspace too small");
    float* col = reinterpret_cast<float*>(ws);
    float* wpad = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ws) + col_bytes);
    launch_k(im2col_f32_kernel, ew_grid((size_t)N * P * Q * kpad), EW_THREADS, 0, st, x, col, N, H, W, C, R, S, stride, pad, P, Q, kpad);
    B200_LAUNCH_CHECK("im2col_f32_kernel");
    launch_k(repitch_rows_kernel<float>, ew_grid((size_t)K * kpad), EW_THREADS, 0, st, w_krsc, wpad, K, R * S * C, kpad);
    B200_LAUNCH_CHECK("repitch_rows_kernel");
    TapTable tt;
    memset(&tt, 0, sizeof(tt));
    tt.n = 1;
    return run_conv_tc(col, N, P, Q, kpad, wpad, K, kpad, tt, y, residual, bias, N, P, Q, st, nullptr, nullptr,
                       nullptr, 1, nullptr, 4, relu);
  }
  // shapes outside the TF32 tensor path (channel counts below 32, odd tile counts): exact fp32 on the CUDA cores
  ConvDims d{N, H, W, C, K, R, S, stride, pad, P, Q};
  launch_k(conv_fprop_direct_f32_kernel, ew_grid((size_t)N * P * Q * K), EW_THREADS, 0, st, x, w_krsc, bias, residual, y, d, relu);
  B200_LAUNCH_CHECK("conv_fprop_direct_f32_kernel");
  return 0;
}

extern "C" int b200_conv2d_dgrad_tf32(const float* dy, const float* w_crsk, const float* addend, float* dx,
                                      int N, int H, int W, int C, int K, int R, int S, int stride, int pad,
                                      b200_stream_t stream) {
  g_det = 0;
  B200_REQUIRE(dy && w_crsk && dx, "conv2d_dgrad_tf32: null pointer");
  B200_REQUIRE(b200_conv2d_tf32_supported(B200_PASS_DGRAD, N, H, W, C, K, R, S, stride, pad),
               "conv2d_dgrad_tf32: shape not supported in the fp32/TF32 mode");
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  cudaStream_t st = as_stream(stream);
  if (stride == 1) {
    TapTable tt;
    memset(&tt, 0, sizeof(tt));
    for (int r = 0; r < R; ++r)
      for (int s = 0; s < S; ++s) {
        const int i = tt.n++;
        tt.dh[i] = pad - r; tt.dw[i] = pad - s; tt.dn[i] = 0;
        tt.wcol[i] = (r * S + s) * K;
      }
    return run_conv_tc(dy, N, P, Q, K, w_crsk, C, R * S * K, tt, dx, addend, nullptr, N, H, W, st, nullptr,
                       nullptr, nullptr, 1, nullptr, 4);
  }
  PhasePlan pp;
  TapTable all;
  build_dgrad_phases(R, S, K, pad, &pp, &all);
  return run_conv_tc(dy, N, P, Q, K, w_crsk, C, R * S * K, all, dx, addend, nullptr, N, H, W, st, nullptr, nullptr,
                     nullptr, 1, &pp, 4);
}

extern "C" int b200_conv2d_wgrad_tf32(const float* dy, const float* x, float* dw_krsc, int N, int H, int W,
                                      int C, int K, int R, int S, int stride, int pad, b200_stream_t stream) {
  B200_REQUIRE(dy && x && dw_krsc, "conv2d_wgrad_tf32: null pointer");
  B200_REQUIRE(b200_conv2d_tf32_supported(B200_PASS_WGRAD, N, H, W, C, K, R, S, stride, pad),
               "conv2d_wgrad_tf32: shape not supported in the fp32/TF32 mode");
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  TapTable tt = fprop_taps(C, R, S, pad);
  return run_wgrad_tc_tf32(x, N, H, W, C, dy, N, P, Q, K, tt, dw_krsc, as_stream(stream), stride);
}

extern "C" int b200_nchw_to_nhwc_f32(const float* x, float* y, int N, int C, int H, int W, b200_stream_t stream) {
  B200_REQUIRE(x && y, "nchw_to_nhwc_f32: null pointer");
  launch_k(nchw_to_nhwc_f32_kernel, ew_grid((size_t)N * C * H * W), EW_THREADS, 0, as_stream(stream), x, y, N, C, H, W);
  B200_LAUNCH_CHECK("nchw_to_nhwc_f32_kernel");
  return 0;
}

extern "C" int b200_bn_act_fwd_f32(const float* x, float* y, int N, int H, int W, int C, const float* mean,
                                   const float* stat, int stat_is_var, float eps, const float* gamma,
                                   const float* beta, const float* skip, int skip_mode, int skip_C, int relu,
                                   b200_stream_t stream) {
  B200_REQUIRE(x && y && C % 4 == 0, "bn_act_fwd_f32: bad arguments");
  B200_REQUIRE(skip_mode == B200_SKIP_NONE || skip, "bn_act_fwd_f32: skip_mode set without skip tensor");
  B200_REQUIRE(skip_mode != B200_SKIP_SUBSAMPLE_PAD || (skip_C % 4 == 0 && skip_C <= C), "bn_act_fwd_f32: bad skip_C");
  BnActF32Args a;
  a.x = x; a.y = y; a.skip = skip; a.mean = mean; a.stat = stat; a.gamma = gamma; a.beta = beta;
  a.N = N; a.H = H; a.W = W; a.C = C; a.skip_mode = skip ? skip_mode : 0; a.skip_C = skip_C;
  a.stat_is_var = stat_is_var; a.relu = relu; a.affine = (gamma && beta && mean && stat) ? 1 : 0; a.eps = eps;
  launch_k(bn_act_fwd_f32_kernel, ew_grid((size_t)N * H * W * C / 4), EW_THREADS, 0, as_stream(stream), a);
  B200_LAUNCH_CHECK("bn_act_fwd_f32_kernel");
  return 0;
}

extern "C" int b200_subsample2_f32(const float* x, float* y, int N, int H, int W, int C, b200_stream_t stream) {
  B200_REQUIRE(x && y && C % 4 == 0, "subsample2_f32: bad arguments");
  launch_k(subsample2_f32_kernel, ew_grid((size_t)N * H * W * C / 4), EW_THREADS, 0, as_stream(stream), x, y, N, H, W, C);
  B200_LAUNCH_CHECK("subsample2_f32_kernel");
  return 0;
}

extern "C" int b200_pool_fwd_f32(const float* x, float* y, int N, int H, int W, int C, int k, int stride, int pad,
                                 int is_max, b200_stream_t stream) {
  B200_REQUIRE(x && y && C % 4 == 0 && stride >= 1, "pool_fwd_f32: bad arguments");
  const int P = (H + 2 * pad - k) / stride + 1, Q = (W + 2 * pad - k) / stride + 1;
  const int grid = ew_grid((size_t)N * P * Q * C / 4);
  if (is_max) launch_k(pool_fwd_f32_kernel<true>, grid, EW_THREADS, 0, as_stream(stream), x, y, N, H, W, C, k, stride, pad, P, Q);
  else launch_k(pool_fwd_f32_kernel<false>, grid, EW_THREADS, 0, as_stream(stream), x, y, N, H, W, C, k, stride, pad, P, Q);
  B200_LAUNCH_CHECK("pool_fwd_f32_kernel");
  return 0;
}

extern "C" int b200_linear_fwd_f32(const float* x, const float* w, const float* b, float* logits, int B, int I,
                                   int O, b200_stream_t stream) {
  B200_REQUIRE(x && w && logits, "linear_fwd_f32: null pointer");
  const size_t threads = (size_t)B * O * 32;
  launch_k(linear_fwd_f32_kernel, (unsigned)((threads + 255) / 256), 256, 0, as_stream(stream), x, w, b, logits, B, I, O);
  B200_LAUNCH_CHECK("linear_fwd_f32_kernel");
  return 0;
}

extern "C" int b200_ce_topk_f32(const float* logits, const int64_t* labels, float* out, int B, int O,
                                b200_stream_t stream) {
  B200_REQUIRE(logits && labels && out, "ce_topk_f32: null pointer");
  cudaStream_t st = as_stream(stream);
  B200_REQUIRE(B > 0 && O > 0, "ce_topk_f32: empty batch");
  launch_k(ce_topk_f32_kernel, 1, CE_WARPS * 32, 0, st, logits, labels, out, B, O);
  B200_LAUNCH_CHECK("ce_topk_f32_kernel");
  return 0;
}

// -------------------------------------------------------------------------------------------------
// layout / filters
// -------------------------------------------------------------------------------------------------
extern "C" int b200_weight_prep(const float* w_krsc, void* w_krsc_bf16, void* w_crsk_bf16, int K,
                                int RS, int C, b200_stream_t stream) {
  B200_REQUIRE(w_krsc, "weight_prep: null pointer");
  cudaStream_t st = as_stream(stream);
  const size_t n = (size_t)K * RS * C;
  if (w_krsc_bf16) {
    launch_k(weight_cast_kernel, ew_grid(n), EW_THREADS, 0, st, w_krsc, (bf16*)w_krsc_bf16, n);
    B200_LAUNCH_CHECK("weight_cast_kernel");
  }
  if (w_crsk_bf16) {
    dim3 grid((C + 31) / 32, (K + 31) / 32, RS);
    launch_k(weight_transpose_kernel, grid, dim3(32, 8), 0, st, w_krsc, (bf16*)w_crsk_bf16, K, RS, C);
    B200_LAUNCH_CHECK("weight_transpose_kernel");
  }
  return 0;
}

extern "C" int b200_weight_prep_multi(const void* table, int n, b200_stream_t stream) {
  B200_REQUIRE(table && n > 0, "weight_prep_multi: bad arguments");
  static_assert(sizeof(WeightPrepEntry) == 40, "table layout is part of the ABI: 3 pointers + 4 ints");
  dim3 grid(num_sms(), n);  // blocks beyond a small tensor's tile count exit at once
  launch_k(weight_prep_multi_kernel, grid, dim3(32, 8), 0, as_stream(stream), reinterpret_cast<const WeightPrepEntry*>(table));
  B200_LAUNCH_CHECK("weight_prep_multi_kernel");
  return 0;
}

extern "C" int b200_nchw_f32_to_nhwc_bf16(const float* x, void* y, int N, int C, int H, int W,
                                          b200_stream_t stream) {
  B200_REQUIRE(x && y, "nchw_f32_to_nhwc_bf16: null pointer");
  launch_k(nchw_f32_to_nhwc_bf16_kernel, ew_grid((size_t)N * H * W), EW_THREADS, 0, as_stream(stream), x, (bf16*)y, N, C, H, W);
  B200_LAUNCH_CHECK("nchw_f32_to_nhwc_bf16_kernel");
  return 0;
}

// -------------------------------------------------------------------------------------------------
// batch norm family
// -------------------------------------------------------------------------------------------------
// Grids of the HBM-bound BN kernels are ONE wave of resident blocks (measured: 1776 short blocks reach
// 4.0 TB/s on the 42 MB tensors, 592 long-lived ones with 4 loads in flight per thread 5.3 TB/s).
// One wave of at most num_sms * blocks_per_sm blocks in which every thread walks the same whole number
// of `unroll`-row batches (a ragged last batch is a full extra memory round trip for the whole grid).
static int bn_blocks(int64_t rows, int C, int blocks_per_sm, int unroll) {
  const int CG = C / 8;
  const int CGb = std::min(EW_THREADS, CG);
  const int RP = EW_THREADS / CGb;
  static const int balanced = env_int("B200_BN_BALANCED", 1);
  const int64_t cap = (int64_t)num_sms() * blocks_per_sm;
  if (balanced) {
    // a whole number of blocks per SM; the row passes are dealt out evenly (grid-stride loops / block_row_range)
    const int64_t passes = (rows + RP - 1) / RP;
    return (int)std::max<int64_t>(1, std::min(cap, passes));
  }
  const int64_t batches = (rows + (int64_t)RP * unroll - 1) / ((int64_t)RP * unroll);  // block-batches
  const int64_t per_block = (batches + cap - 1) / cap;
  return (int)std::max<int64_t>(1, (batches + per_block - 1) / per_block);
}

// BN_SLOTS copies of the fp64 accumulators [2][C] + the ticket counter of the last-block finalize
extern "C" size_t b200_bn_workspace_bytes(int64_t rows, int C) {
  (void)rows;
  return (size_t)BN_SLOTS * bn_slot_stride(C) * sizeof(double) + 16;
}

static int bn_sums_launch(const void* x, int64_t rows, int C, void* ws, size_t ws_bytes, int finalize,
                          float eps, float momentum, float* mean, float* invstd, float* running_mean,
                          float* running_var, int64_t* num_batches_tracked, cudaStream_t st) {
  B200_REQUIRE(C % 8 == 0, "bn_stats: C=%d must be a multiple of 8", C);
  B200_REQUIRE(ws && ws_bytes >= b200_bn_workspace_bytes(rows, C), "bn_stats: workspace too small");
  B200_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 7) == 0, "bn_stats: workspace must be 8-byte aligned");
  static const int bps = std::max(1, env_int("B200_BN_STATS_BPS", 4));
  BnStatsArgs a;
  a.x = (const bf16*)x; a.rows = rows; a.C = C; a.eps = eps; a.momentum = momentum;
  a.mean = mean; a.invstd = invstd; a.running_mean = running_mean; a.running_var = running_var;
  a.num_batches_tracked = num_batches_tracked;
  a.accum = reinterpret_cast<double*>(ws);
  a.ticket = reinterpret_cast<unsigned int*>(a.accum + BN_SLOTS * bn_slot_stride(C));
  a.finalize = finalize;
  const int CG = C / 8;
  dim3 grid(bn_blocks(rows, C, bps, 8), (CG + EW_THREADS - 1) / EW_THREADS);
  launch_k(bn_stats_kernel, grid, EW_THREADS, EW_THREADS * 16 * sizeof(float), st, a);
  B200_LAUNCH_CHECK("bn_stats_kernel");
  return 0;
}

extern "C" int b200_bn_stats(const void* x, int64_t rows, int C, float eps, float momentum,
                             float* mean, float* invstd, float* running_mean, float* running_var,
                             int64_t* num_batches_tracked, void* ws, size_t ws_bytes,
                             b200_stream_t stream) {
  B200_REQUIRE(x && mean && invstd && ws, "bn_stats: null pointer");
  return bn_sums_launch(x, rows, C, ws, ws_bytes, 1, eps, momentum, mean, invstd, running_mean,
                        running_var, num_batches_tracked, as_stream(stream));
}

extern "C" int b200_bn_stats_finalize(int64_t rows, int C, float eps, float momentum, float* mean,
                                      float* invstd, float* running_mean, float* running_var,
                                      int64_t* num_batches_tracked, void* ws, size_t ws_bytes,
                                      b200_stream_t stream) {
  B200_REQUIRE(mean && invstd && ws && rows > 0, "bn_stats_finalize: bad arguments");
  B200_REQUIRE(ws_bytes >= b200_bn_workspace_bytes(rows, C), "bn_stats_finalize: workspace too small");
  BnStatsArgs a;
  a.x = nullptr; a.rows = rows; a.C = C; a.eps = eps; a.momentum = momentum;
  a.mean = mean; a.invstd = invstd; a.running_mean = running_mean; a.running_var = running_var;
  a.num_batches_tracked = num_batches_tracked;
  a.accum = reinterpret_cast<double*>(ws);
  a.ticket = nullptr;
  a.finalize = 1;
  launch_k(bn_stats_finalize_kernel, (unsigned)((C + 255) / 256), 256, 0, as_stream(stream), a);
  B200_LAUNCH_CHECK("bn_stats_finalize_kernel");
  return 0;
}

extern "C" int b200_bn_running_update(const float* mean, const float* invstd, int64_t rows, int C, float eps,
                                      float momentum, float* running_mean, float* running_var,
                                      int64_t* num_batches_tracked, b200_stream_t stream) {
  B200_REQUIRE(mean && invstd && running_mean && running_var && rows > 0, "bn_running_update: bad arguments");
  launch_k(bn_running_update_kernel, (unsigned)((C + 255) / 256), 256, 0, as_stream(stream), mean, invstd, eps,
           momentum, rows, running_mean, running_var, num_batches_tracked, C);
  B200_LAUNCH_CHECK("bn_running_update_kernel");
  return 0;
}

static uint32_t drop_threshold(float p) {
  if (p <= 0.f) return 0;
  double t = (double)p * 65536.0 + 0.5;
  if (t > 65535.0) t = 65535.0;
  return (uint32_t)t;
}

extern "C" int b200_bn_act_fwd(const void* x, void* y, int N, int H, int W, int C, const float* mean,
                               const float* invstd, int stat_is_var, float eps, const float* gamma,
                               const float* beta, const void* skip, int skip_mode, int skip_C,
                               int relu, float dropout_p, uint64_t seed, const uint64_t* seed_offset,
                               float* running_mean, float* running_var, int64_t* num_batches_tracked,
                               float momentum, void* mask_out, b200_stream_t stream) {
  B200_REQUIRE(x && y, "bn_act_fwd: null pointer");
  B200_REQUIRE(!running_mean || (running_var && mean && invstd && !stat_is_var),
               "bn_act_fwd: the running-statistics update needs batch mean / invstd");
  B200_REQUIRE(C % 8 == 0, "bn_act_fwd: C=%d must be a multiple of 8", C);
  B200_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "bn_act_fwd: dropout_p out of range");
  B200_REQUIRE(skip_mode == B200_SKIP_NONE || skip, "bn_act_fwd: skip_mode set without skip tensor");
  B200_REQUIRE(skip_mode != B200_SKIP_SUBSAMPLE_PAD || (skip_C % 8 == 0 && skip_C <= C),
               "bn_act_fwd: bad skip_C=%d", skip_C);
  BnActFwdArgs a;
  a.x = (const bf16*)x; a.y = (bf16*)y; a.skip = (const bf16*)skip;
  a.mean = mean; a.invstd = invstd; a.gamma = gamma; a.beta = beta;
  a.N = N; a.H = H; a.W = W; a.C = C;
  a.skip_mode = skip ? skip_mode : 0; a.skip_C = skip_C;
  a.stat_is_var = stat_is_var; a.relu = relu;
  a.affine = (gamma && beta && mean && invstd) ? 1 : 0;
  a.eps = eps;
  a.inv_keep = 1.f / (1.f - dropout_p);
  a.drop_thr = drop_threshold(dropout_p);
  a.seed = seed;
  a.seed_offset = seed_offset;
  a.running_mean = running_mean; a.running_var = running_var; a.num_batches_tracked = num_batches_tracked;
  a.momentum = momentum;
  a.mask_out = reinterpret_cast<uint8_t*>(mask_out);
  {
    const int CG = C / 8;
    const int64_t rows = (int64_t)N * H * W;
    static const int bps = std::max(1, env_int("B200_BN_FWD_BPS", 4));
    cudaStream_t fst = as_stream(stream);
    const bool drop = a.drop_thr != 0;
    const bool keepbits = drop && !relu && a.mask_out;   // no fused ReLU to read the mask off the output
    if (a.skip_mode != 0) {
      dim3 grid(bn_blocks(rows, C, std::min(bps, 3), 2), (CG + EW_THREADS - 1) / EW_THREADS);
      if (drop) launch_k(bn_act_fwd_kernel<2, 3, true, 2>, grid, EW_THREADS, 0, fst, a);
      else launch_k(bn_act_fwd_kernel<2, 3, true, 0>, grid, EW_THREADS, 0, fst, a);
    } else if (!drop) {
      dim3 grid(bn_blocks(rows, C, bps, 4), (CG + EW_THREADS - 1) / EW_THREADS);
      launch_k(bn_act_fwd_kernel<4, 4, false, 0>, grid, EW_THREADS, 0, fst, a);
    } else if (keepbits) {
      dim3 grid(bn_blocks(rows, C, std::min(bps, 3), 4), (CG + EW_THREADS - 1) / EW_THREADS);
      launch_k(bn_act_fwd_kernel<4, 3, false, 2>, grid, EW_THREADS, 0, fst, a);
    } else {
      // two vectors in flight per thread: the four-vector variant spills at 64 registers once the RNG is in
      dim3 grid(bn_blocks(rows, C, bps, 2), (CG + EW_THREADS - 1) / EW_THREADS);
      launch_k(bn_act_fwd_kernel<2, 4, false, 1>, grid, EW_THREADS, 0, fst, a);
    }
  }
  B200_LAUNCH_CHECK("bn_act_fwd_kernel");
  return 0;
}

// reduce = false: dgamma / dbeta already hold the sums (b200_conv2d_dgrad_bnbwd produced them), apply pass only
static int bn_act_bwd_impl(const void* dy, const void* y, const void* mask, const void* x, void* dx,
                           void* dskip, const void* addend, int64_t rows, int C, const float* mean,
                           const float* invstd, const float* gamma, float* dgamma, float* dbeta,
                           int relu, float dropout_p, uint64_t seed, const uint64_t* seed_offset,
                           void* ws, size_t ws_bytes, b200_stream_t stream, bool reduce) {
  B200_REQUIRE(dy && dx, "bn_act_bwd: null pointer");
  B200_REQUIRE(C % 8 == 0, "bn_act_bwd: C=%d must be a multiple of 8", C);
  const bool gate_x = mask != nullptr;   // bit mask written by the forward: neither y nor the RNG is needed
  B200_REQUIRE(!relu || y || mask, "bn_act_bwd: relu needs the forward's mask bytes or its output y");
  cudaStream_t st = as_stream(stream);
  BnActBwdArgs a;
  a.dy = (const bf16*)dy; a.y = (const bf16*)y; a.x = (const bf16*)x;
  a.mask = reinterpret_cast<const uint8_t*>(mask);
  a.dx = (bf16*)dx; a.dskip = (bf16*)dskip; a.addend = (const bf16*)addend;
  a.mean = mean; a.invstd = invstd; a.gamma = gamma; a.dgamma = dgamma; a.dbeta = dbeta;
  a.rows = rows; a.C = C; a.relu = relu;
  a.affine = (gamma && mean && invstd) ? 1 : 0;
  a.inv_keep = 1.f / (1.f - dropout_p);
  a.drop_thr = drop_threshold(dropout_p);
  a.seed = seed;
  a.seed_offset = seed_offset;
  B200_REQUIRE(reduce || (a.affine && x && dgamma && dbeta), "bn_act_bwd_apply: needs the affine operands");
  if (a.affine && reduce) {
    B200_REQUIRE(x && dgamma && dbeta && ws, "bn_act_bwd: null pointer (affine path)");
    B200_REQUIRE(ws_bytes >= b200_bn_workspace_bytes(rows, C), "bn_act_bwd: workspace too small");
    B200_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 7) == 0, "bn_act_bwd: workspace must be 8-byte aligned");
    static const int rbps = std::max(1, env_int("B200_BN_REDUCE_BPS", 3));
    const int CG = C / 8;
    dim3 grid(bn_blocks(rows, C, rbps, gate_x ? 4 : 2), (CG + EW_THREADS - 1) / EW_THREADS);
    double* accum = reinterpret_cast<double*>(ws);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(accum + BN_SLOTS * bn_slot_stride(C));
    if (gate_x) launch_k(bn_act_bwd_reduce_kernel<true>, grid, EW_THREADS, EW_THREADS * 16 * sizeof(float), st, a, accum, ticket);
    else launch_k(bn_act_bwd_reduce_kernel<false>, grid, EW_THREADS, EW_THREADS * 16 * sizeof(float), st, a, accum, ticket);
    B200_LAUNCH_CHECK("bn_act_bwd_reduce_kernel");
  }
  {
    static const int abps = std::max(1, env_int("B200_BN_APPLY_BPS", 3));
    const int CG = C / 8;
    dim3 grid(bn_blocks(rows, C, abps, 2), (CG + EW_THREADS - 1) / EW_THREADS);
    if (!gate_x) launch_k(bn_act_bwd_apply_kernel<false, true, true>, grid, EW_THREADS, 0, st, a);
    else if (a.dskip) launch_k(bn_act_bwd_apply_kernel<true, true, true>, grid, EW_THREADS, 0, st, a);
    else if (a.addend) launch_k(bn_act_bwd_apply_kernel<true, true, false>, grid, EW_THREADS, 0, st, a);
    else launch_k(bn_act_bwd_apply_kernel<true, false, false>, grid, EW_THREADS, 0, st, a);
  }
  B200_LAUNCH_CHECK("bn_act_bwd_apply_kernel");
  return 0;
}

extern "C" int b200_bn_act_bwd(const void* dy, const void* y, const void* mask, const void* x, void* dx,
                               void* dskip, const void* addend, int64_t rows, int C, const float* mean,
                               const float* invstd, const float* gamma, float* dgamma, float* dbeta,
                               int relu, float dropout_p, uint64_t seed, const uint64_t* seed_offset,
                               void* ws, size_t ws_bytes, b200_stream_t stream) {
  return bn_act_bwd_impl(dy, y, mask, x, dx, dskip, addend, rows, C, mean, invstd, gamma, dgamma, dbeta, relu,
                         dropout_p, seed, seed_offset, ws, ws_bytes, stream, true);
}

// The apply pass alone: dgamma / dbeta are INPUTS (the per-channel sums b200_conv2d_dgrad_bnbwd finalized).
extern "C" int b200_bn_act_bwd_apply(const void* dy, const void* mask, const void* x, void* dx, void* dskip,
                                     const void* addend, int64_t rows, int C, const float* mean,
                                     const float* invstd, const float* gamma, const float* dgamma,
                                     const float* dbeta, int relu, float dropout_p, b200_stream_t stream) {
  B200_REQUIRE(mask, "bn_act_bwd_apply: needs the forward's mask bytes");
  return bn_act_bwd_impl(dy, nullptr, mask, x, dx, dskip, addend, rows, C, mean, invstd, gamma,
                         const_cast<float*>(dgamma), const_cast<float*>(dbeta), relu, dropout_p, 0, nullptr, nullptr, 0,
                         stream, false);
}

extern "C" int b200_subsample2(const void* x, void* y, int N, int H, int W, int C,
                               b200_stream_t stream) {
  B200_REQUIRE(x && y && C % 8 == 0, "subsample2: bad arguments");
  launch_k(subsample2_kernel, ew_grid((size_t)N * H * W * C / 8), EW_THREADS, 0, as_stream(stream), (const bf16*)x, (bf16*)y, N, H, W, C);
  B200_LAUNCH_CHECK("subsample2_kernel");
  return 0;
}

extern "C" int b200_upsample_add(void* dx, const void* g, int N, int H, int W, int C, int Cg, int ldg,
                                 b200_stream_t stream) {
  B200_REQUIRE(dx && g && C % 8 == 0 && Cg % 8 == 0 && Cg <= C && ldg >= Cg && ldg % 8 == 0,
               "upsample_add: bad arguments");
  launch_k(upsample_add_kernel, ew_grid((size_t)N * H * W * Cg / 8), EW_THREADS, 0, as_stream(stream), (bf16*)dx, (const bf16*)g, N, H, W, C, Cg, ldg);
  B200_LAUNCH_CHECK("upsample_add_kernel");
  return 0;
}

// -------------------------------------------------------------------------------------------------
// pooling
// -------------------------------------------------------------------------------------------------
static PoolDims pool_dims(int N, int H, int W, int C, int k, int stride, int pad) {
  PoolDims d{N, H, W, C, k, stride, pad, (H + 2 * pad - k) / stride + 1, (W + 2 * pad - k) / stride + 1};
  return d;
}

extern "C" int b200_avgpool_fwd(const void* x, void* y, int N, int H, int W, int C, int k, int stride,
                                int pad, b200_stream_t stream) {
  B200_REQUIRE(x && y && C % 8 == 0 && stride >= 1, "avgpool_fwd: bad arguments");
  PoolDims d = pool_dims(N, H, W, C, k, stride, pad);
  if (pad == 0 && k == H && k == W) {   // global pooling
    launch_k(avgpool_global_kernel, (unsigned)N, EW_THREADS, 0, as_stream(stream), (const bf16*)x, (bf16*)y, H * W, C);
    B200_LAUNCH_CHECK("avgpool_global_kernel");
    return 0;
  }
  launch_k(avgpool_fwd_kernel, ew_grid((size_t)N * d.P * d.Q * C / 8), EW_THREADS, 0, as_stream(stream), (const bf16*)x, (bf16*)y, d);
  B200_LAUNCH_CHECK("avgpool_fwd_kernel");
  return 0;
}

extern "C" int b200_avgpool_bwd(const void* dy, void* dx, int N, int H, int W, int C, int k,
                                int stride, int pad, b200_stream_t stream) {
  B200_REQUIRE(dy && dx && C % 8 == 0 && stride >= 1, "avgpool_bwd: bad arguments");
  PoolDims d = pool_dims(N, H, W, C, k, stride, pad);
  launch_k(avgpool_bwd_kernel, ew_grid((size_t)N * H * W * C / 8), EW_THREADS, 0, as_stream(stream), (const bf16*)dy, (bf16*)dx, d);
  B200_LAUNCH_CHECK("avgpool_bwd_kernel");
  return 0;
}

extern "C" int b200_maxpool_fwd(const void* x, void* y, void* argmax, int N, int H, int W, int C, int k,
                                int stride, int pad, b200_stream_t stream) {
  B200_REQUIRE(x && y && C % 8 == 0 && stride >= 1 && k * k <= 255, "maxpool_fwd: bad arguments");
  PoolDims d = pool_dims(N, H, W, C, k, stride, pad);
  // compile-time window / stride variants (k3 s2: the ImageNet-style stem pool; k2 s2; k3 s1): one block row per
  // output row, 256 threads over its (column, channel group) pairs
  const long long rows_f = (long long)N * d.P;
  const int per_row_f = d.Q * (C / 8);
  if (rows_f <= 0x7fffffffLL && per_row_f > 0 && ((k == 3 && (stride == 2 || stride == 1)) || (k == 2 && stride == 2))) {
    const dim3 grid((unsigned)rows_f, (unsigned)std::min(64, (per_row_f + 255) / 256));
#define B200_MP_FWD(K_, S_) launch_k(maxpool_fwd_ks_kernel<K_, S_>, grid, 256, 0, as_stream(stream), (const bf16*)x, (bf16*)y, reinterpret_cast<uint8_t*>(argmax), d)
    if (k == 3 && stride == 2) B200_MP_FWD(3, 2);
    else if (k == 3) B200_MP_FWD(3, 1);
    else B200_MP_FWD(2, 2);
#undef B200_MP_FWD
    B200_LAUNCH_CHECK("maxpool_fwd_ks_kernel");
    return 0;
  }
  launch_k(maxpool_fwd_kernel, ew_grid((size_t)N * d.P * d.Q * C / 8), EW_THREADS, 0, as_stream(stream), (const bf16*)x, (bf16*)y, reinterpret_cast<uint8_t*>(argmax), d);
  B200_LAUNCH_CHECK("maxpool_fwd_kernel");
  return 0;
}

extern "C" int b200_maxpool_bwd(const void* dy, const void* argmax, void* dx, int N, int H, int W, int C, int k,
                                int stride, int pad, b200_stream_t stream) {
  B200_REQUIRE(dy && argmax && dx && stride >= 1 && C % 8 == 0, "maxpool_bwd: bad arguments");
  PoolDims d = pool_dims(N, H, W, C, k, stride, pad);
  const long long rows_b = (long long)N * H;
  const int per_row_b = W * (C / 8);
  if (rows_b <= 0x7fffffffLL && per_row_b > 0 && ((k == 3 && (stride == 2 || stride == 1)) || (k == 2 && stride == 2))) {
    const dim3 grid((unsigned)rows_b, (unsigned)std::min(64, (per_row_b + 255) / 256));
#define B200_MP_BWD(K_, S_) launch_k(maxpool_bwd_ks_kernel<K_, S_>, grid, 256, 0, as_stream(stream), (const bf16*)dy, reinterpret_cast<const uint8_t*>(argmax), (bf16*)dx, d)
    if (k == 3 && stride == 2) B200_MP_BWD(3, 2);
    else if (k == 3) B200_MP_BWD(3, 1);
    else B200_MP_BWD(2, 2);
#undef B200_MP_BWD
    B200_LAUNCH_CHECK("maxpool_bwd_ks_kernel");
    return 0;
  }
  launch_k(maxpool_bwd_kernel, ew_grid((size_t)N * H * W * C / 8), EW_THREADS, 0, as_stream(stream), (const bf16*)dy, reinterpret_cast<const uint8_t*>(argmax), (bf16*)dx, d);
  B200_LAUNCH_CHECK("maxpool_bwd_kernel");
  return 0;
}

// -------------------------------------------------------------------------------------------------
// head
// -------------------------------------------------------------------------------------------------
extern "C" int b200_linear_fwd(const void* x, const float* w, const float* b, void* logits, int B,
                               int I, int O, b200_stream_t stream) {
  B200_REQUIRE(x && w && logits, "linear_fwd: null pointer");
  const size_t threads = (size_t)B * O * 32;
  launch_k(linear_fwd_kernel, (unsigned)((threads + 255) / 256), 256, 0, as_stream(stream), (const bf16*)x, w, b,
                                                                              (bf16*)logits, B, I, O);
  B200_LAUNCH_CHECK("linear_fwd_kernel");
  return 0;
}

extern "C" int b200_linear_bwd(const void* dlogits, const void* x, const float* w, void* dx,
                               float* dw, float* db, int B, int I, int O, b200_stream_t stream) {
  B200_REQUIRE(dlogits && x && w, "linear_bwd: null pointer");
  cudaStream_t st = as_stream(stream);
  if (dx) {
    launch_k(linear_bwd_dx_kernel, (unsigned)(((size_t)B * I + 255) / 256), 256, 0, st, (const bf16*)dlogits, w, (bf16*)dx, B, I, O);
    B200_LAUNCH_CHECK("linear_bwd_dx_kernel");
  }
  if (dw) {
    launch_k(linear_bwd_dw_kernel, (unsigned)(((size_t)O * I + 255) / 256), 256, 0, st, (const bf16*)dlogits, (const bf16*)x, dw, db, B, I, O);
    B200_LAUNCH_CHECK("linear_bwd_dw_kernel");
  }
  return 0;
}

extern "C" int b200_ce_topk(const void* logits, const int64_t* labels, float* out, void* dlogits,
                            const float* grad_scale, int B, int O, b200_stream_t stream) {
  B200_REQUIRE(logits && labels, "ce_topk: null pointer");
  cudaStream_t st = as_stream(stream);
  B200_REQUIRE(B > 0 && O > 0, "ce_topk: empty batch");
  launch_k(ce_topk_kernel, 1, CE_WARPS * 32, 0, st, (const bf16*)logits, labels, out, (bf16*)dlogits, grad_scale, B, O);
  B200_LAUNCH_CHECK("ce_topk_kernel");
  return 0;
}

// -------------------------------------------------------------------------------------------------
// input pipeline
// -------------------------------------------------------------------------------------------------
extern "C" int b200_augment_batch(const void* data, const int64_t* index, const void* flip, const int32_t* top,
                                  const int32_t* left, const float* mean, const float* stddev, int B, int H,
                                  int W, int C, int pad, int pad_mirror, int out_h, int out_w, int to_tensor,
                                  float* out_f32_nchw, void* out_bf16_nhwc, b200_stream_t stream) {
  B200_REQUIRE(data && index && (out_f32_nchw || out_bf16_nhwc), "augment_batch: null pointer");
  B200_REQUIRE(B > 0 && H > 0 && W > 0 && C > 0 && pad >= 0, "augment_batch: bad shape");
  B200_REQUIRE(!pad_mirror || (pad < H && pad < W), "augment_batch: mirror padding needs pad < H, W");
  B200_REQUIRE(out_h > 0 && out_w > 0 && out_h <= H + 2 * pad && out_w <= W + 2 * pad,
               "augment_batch: output %dx%d does not fit the padded %dx%d image", out_h, out_w, H + 2 * pad,
               W + 2 * pad);
  B200_REQUIRE(!stddev || mean, "augment_batch: stddev without mean");
  B200_REQUIRE((top == nullptr) == (left == nullptr), "augment_batch: top and left go together");
  B200_REQUIRE(top || (out_h == H + 2 * pad && out_w == W + 2 * pad),
               "augment_batch: a smaller output needs crop offsets");
  AugmentArgs a;
  a.data = reinterpret_cast<const uint8_t*>(data); a.index = index;
  a.flip = reinterpret_cast<const uint8_t*>(flip); a.top = top; a.left = left;
  a.mean = mean; a.stddev = stddev;
  a.B = B; a.H = H; a.W = W; a.C = C; a.pad = pad; a.mirror = pad_mirror; a.OH = out_h; a.OW = out_w;
  a.to_tensor = to_tensor;
  a.out_f32 = out_f32_nchw; a.out_bf16 = reinterpret_cast<bf16*>(out_bf16_nhwc);
  launch_k(augment_batch_kernel, ew_grid((size_t)B * out_h * out_w), EW_THREADS, 0, as_stream(stream), a);
  B200_LAUNCH_CHECK("augment_batch_kernel");
  return 0;
}

// -------------------------------------------------------------------------------------------------
// optimizer
// -------------------------------------------------------------------------------------------------
extern "C" int b200_sgd_step(float* const* params, const float* const* grads, float* const* bufs,
                             const int64_t* sizes, int n, int64_t max_size, float lr, float momentum,
                             float dampening, float weight_decay, int nesterov, int first_step,
                             const float* inv_scale, const float* found_inf, const float* lr_ptr,
                             b200_stream_t stream) {
  B200_REQUIRE(params && grads && bufs && sizes && n > 0, "sgd_step: bad arguments");
  SgdArgs a{params, grads, bufs, sizes, lr, momentum, dampening, weight_decay,
            nesterov, first_step, inv_scale, found_inf, lr_ptr};
  const int64_t chunk = (int64_t)SGD_THREADS * SGD_VEC_PER_THREAD * 4;
  dim3 grid((unsigned)((max_size + chunk - 1) / chunk), n);
  launch_k(sgd_step_kernel, grid, SGD_THREADS, 0, as_stream(stream), a);
  B200_LAUNCH_CHECK("sgd_step_kernel");
  return 0;
}

extern "C" int b200_adam_step(float* const* params, const float* const* grads, float* const* exp_avgs,
                              float* const* exp_avg_sqs, float* const* max_exp_avg_sqs, float* const* steps,
                              const int64_t* sizes, int n, int64_t max_size, double lr, double beta1,
                              double beta2, double eps, double weight_decay, int decoupled, int amsgrad,
                              const float* inv_scale, const float* found_inf, const float* lr_ptr,
                              unsigned* tickets, b200_stream_t stream) {
  B200_REQUIRE(params && grads && exp_avgs && exp_avg_sqs && steps && sizes && tickets && n > 0 && max_size >= 0,
               "adam_step: bad arguments");
  B200_REQUIRE(!amsgrad || max_exp_avg_sqs, "adam_step: amsgrad needs max_exp_avg_sqs");
  B200_REQUIRE(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0,
               "adam_step: betas must lie in [0, 1) and eps must be >= 0 (got %g, %g, %g)", beta1, beta2, eps);
  B200_REQUIRE(n <= 65535, "adam_step: %d tensors in one launch (at most 65535)", n);
  AdamArgs a{params, grads, exp_avgs, exp_avg_sqs, amsgrad ? max_exp_avg_sqs : nullptr, steps, sizes, tickets,
             lr, beta1, beta2, eps, weight_decay, decoupled, amsgrad, inv_scale, found_inf, lr_ptr};
  dim3 grid((unsigned)std::max<int64_t>(1, (max_size + ADAM_CHUNK - 1) / ADAM_CHUNK), n);
  launch_k(adam_step_kernel, grid, ADAM_THREADS, 0, as_stream(stream), a);
  B200_LAUNCH_CHECK("adam_step_kernel");
  return 0;
}

extern "C" int b200_tick(uint64_t* counter, b200_stream_t stream) {
  B200_REQUIRE(counter, "tick: null pointer");
  launch_k(tick_kernel, 1, 1, 0, as_stream(stream), counter);
  B200_LAUNCH_CHECK("tick_kernel");
  return 0;
}
