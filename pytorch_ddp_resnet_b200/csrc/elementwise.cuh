// HBM-bound kernels around the convolutions: batch-norm statistics, fused normalise + skip-add +
// ReLU + dropout (forward and backward), subsample / upsample, parity split, pooling, layout casts.
// All activations are NHWC bf16 handled as 16-byte vectors of 8 channels; per-channel quantities are
// fp32; reductions are warp-shuffle / shared-memory trees with deterministic per-block partials.
#pragma once
#include "common.cuh"

namespace b200 {

constexpr int EW_THREADS = 256;

// Inverted dropout on the 8 values of vector `v`: element j is dropped when its 16-bit uniform is
// below drop_thr, else scaled by 1/(1-p) and (ROUND) rounded to bf16 like the reference's bf16 multiply.
// Returns the keep mask (bit j set = element j kept).
template <bool ROUND>
__device__ __forceinline__ uint32_t dropout8(float* f, uint64_t seed, size_t v, uint32_t drop_thr,
                                             float inv_keep) {
  uint32_t keep = 0;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const uint2 d = rng_draw4(seed, (uint64_t)v * 2 + h);
    const uint32_t u[4] = {d.x & 0xffffu, d.x >> 16, d.y & 0xffffu, d.y >> 16};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float t = f[4 * h + j] * inv_keep;
      const bool k = u[j] >= drop_thr;
      keep |= (k ? 1u : 0u) << (4 * h + j);
      f[4 * h + j] = k ? (ROUND ? round_bf16(t) : t) : 0.f;
    }
  }
  return keep;
}

// -------------------------------------------------------------------------------------------------
// Block-level per-channel reduction helper. Each thread owns one 8-channel group `cg` (fixed for
// the whole kernel) and a row lane `rl`; acc[] holds NACC*8 per-channel partial sums of that thread.
// The block reduces over row lanes and writes partial[blockIdx.x][a][C] for a < NACC.
// -------------------------------------------------------------------------------------------------
template <int NACC>
__device__ __forceinline__ void block_channel_reduce(const float* acc, float* smem, int cgl, int rl,
                                                     int CGb, int RP, bool active, double* accum,
                                                     int C, int c_base) {
  // smem layout: [RP][CGb*8*NACC]; the block total of every channel goes to its slot with one fp64
  // atomic (fp32 inside a block: <= a few hundred terms; fp64 across blocks: E[x^2] - mean^2 cancels)
  const int width = CGb * 8 * NACC;
  if (active) {
#pragma unroll
    for (int a = 0; a < NACC; ++a)
#pragma unroll
      for (int j = 0; j < 8; ++j) smem[rl * width + (a * CGb + cgl) * 8 + j] = acc[a * 8 + j];
  }
  __syncthreads();
  double* slot = accum + (size_t)(blockIdx.x % BN_SLOTS) * bn_slot_stride(C);
  for (int i = threadIdx.x; i < width; i += blockDim.x) {
    float s = 0.f;
    for (int r = 0; r < RP; ++r) s += smem[r * width + i];
    const int a = i / (CGb * 8);
    const int c = c_base + (i % (CGb * 8));
    atomicAdd(slot + (size_t)a * C + c, (double)s);
  }
}

// Returns true in the block that finishes last; every other block's atomics are then visible to it
// (barrier, then one thread fences and takes a ticket: the pattern of a cooperative grid sync).
__device__ __forceinline__ bool last_block_done(unsigned int* ticket) {
  __shared__ int is_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int total = gridDim.x * gridDim.y;
    is_last = atomicAdd(ticket, 1u) == total - 1u;
    __threadfence();
  }
  __syncthreads();
  return is_last != 0;
}

// rows [r0, r1) of block blockIdx.x: the ceil(rows / RP) row passes are dealt out as evenly as integers allow
// (any grid size works). Round 1 rounded every block up to whole unrolled batches, which left 342 blocks for the
// 148 SMs at 128x8x8x640: SMs with three blocks against SMs with two, in kernels that are issue-bound.
__device__ __forceinline__ void block_row_range(int64_t rows, int RP, int64_t& r0, int64_t& r1) {
  const int64_t passes = (rows + RP - 1) / RP;
  r0 = passes * blockIdx.x / gridDim.x * RP;
  r1 = min(rows, passes * (blockIdx.x + 1) / gridDim.x * RP);
}

// geometry shared by the reduction kernels: blockIdx.y selects a chunk of <=256 channel groups
struct ReduceGeom {
  int CG;    // C / 8
  int CGb;   // channel groups handled by this block
  int cg0;   // first channel group of this block
  int RP;    // rows per pass
  int cgl, rl;
  bool active;
  __device__ __forceinline__ ReduceGeom(int C) {
    CG = C / 8;
    cg0 = blockIdx.y * EW_THREADS;
    CGb = min(EW_THREADS, CG - cg0);
    RP = EW_THREADS / CGb;
    cgl = threadIdx.x % CGb;
    rl = threadIdx.x / CGb;
    active = rl < RP;
  }
};

struct BnStatsArgs {
  const bf16* x;
  int64_t rows;
  int C;
  float eps, momentum;
  float* mean;
  float* invstd;
  float* running_mean;
  float* running_var;
  int64_t* num_batches_tracked;
  double* accum;          // BN_SLOTS x [2][C], zero on entry, zero again on exit
  unsigned int* ticket;   // zero on entry, zero again on exit
  int finalize;           // 0: accumulate only (the sums are finalized by bn_stats_finalize_kernel)
};

// running statistics of one channel from its batch mean / invstd (torch.nn.BatchNorm2d: momentum update with
// the UNBIASED batch variance). The biased variance is recovered as 1/invstd^2 - eps, in fp32: this runs at the head
// of ONE block of bn_act_fwd, eight channels per thread, and in fp64 (division) it made that block the last to
// finish; the fp32 result is within 3e-7 relative of the fp64 one for var >= eps.
__device__ __forceinline__ void bn_running_update_channel(float mean, float invstd, float eps, float momentum,
                                                          int64_t rows, float* running_mean, float* running_var,
                                                          int c) {
  float var = fmaxf(1.f / (invstd * invstd) - eps, 0.f);
  if (rows > 1) var *= (float)rows / (float)(rows - 1);
  running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
  running_var[c] = (1.f - momentum) * running_var[c] + momentum * var;
}

// one channel: mean / invstd from its drained sums, running-statistics update
__device__ __forceinline__ void bn_finalize_channel(const BnStatsArgs& a, int c, double s, double ss) {
  const double m = s / (double)a.rows;
  double var = ss / (double)a.rows - m * m;
  if (var < 0.0) var = 0.0;
  a.mean[c] = (float)m;
  a.invstd[c] = (float)(1.0 / sqrt(var + (double)a.eps));
  if (a.running_mean) {
    const double unbiased = a.rows > 1 ? var * (double)a.rows / (double)(a.rows - 1) : var;
    a.running_mean[c] = (1.f - a.momentum) * a.running_mean[c] + a.momentum * (float)m;
    a.running_var[c] = (1.f - a.momentum) * a.running_var[c] + a.momentum * (float)unbiased;
  }
}

// running statistics from mean / invstd that a conv kernel's tail produced (compatibility path: the
// training forward folds this update into bn_act_fwd)
__global__ void bn_running_update_kernel(const float* __restrict__ mean, const float* __restrict__ invstd,
                                         float eps, float momentum, int64_t rows, float* running_mean,
                                         float* running_var, int64_t* num_batches_tracked, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) bn_running_update_channel(mean[c], invstd[c], eps, momentum, rows, running_mean, running_var, c);
  if (c == 0 && num_batches_tracked) *num_batches_tracked += 1;
}

// Batch statistics in ONE launch: every block adds its per-channel sum / sum of squares to the fp64
// accumulators; the block that finishes last turns them into mean / invstd / running statistics and
// clears the accumulators for the next call (no partial buffer, no finalize kernel).
__global__ void __launch_bounds__(EW_THREADS, 4) bn_stats_kernel(const BnStatsArgs a) {
  extern __shared__ float red_smem[];
  const int C = a.C;
  ReduceGeom g(C);
  float acc[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) acc[j] = 0.f;
  if (g.active) {
    constexpr int U = 8;   // 8 independent 16-byte loads in flight per thread; rows past r1 are skipped
    int64_t r0, r1;
    block_row_range(a.rows, g.RP, r0, r1);
    const bf16* base = a.x + (size_t)(g.cg0 + g.cgl) * 8;
    for (int64_t r = r0 + g.rl; r < r1; r += U * (int64_t)g.RP) {
      Vec8 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t ru = r + u * (int64_t)g.RP;
        v[u].raw = make_uint4(0u, 0u, 0u, 0u);
        if (ru < r1) v[u].raw = ldg_stream(base + (size_t)ru * C);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float f[8];
        v[u].to_float(f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc[j] += f[j];
          acc[8 + j] = fmaf(f[j], f[j], acc[8 + j]);
        }
      }
    }
  }
  block_channel_reduce<2>(acc, red_smem, g.cgl, g.rl, g.CGb, g.RP, g.active, a.accum, C, g.cg0 * 8);
  if (!a.finalize || !last_block_done(a.ticket)) return;
  for (int c = threadIdx.x; c < C; c += blockDim.x)
    bn_finalize_channel(a, c, drain_slots(a.accum, C, 0, c), drain_slots(a.accum, C, 1, c));
  if (threadIdx.x == 0) {
    *a.ticket = 0u;
    if (a.num_batches_tracked) *a.num_batches_tracked += 1;
  }
}

// sums accumulated by a conv epilogue (or an accumulate-only pass) -> mean / invstd / running statistics
__global__ void bn_stats_finalize_kernel(const BnStatsArgs a) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < a.C) bn_finalize_channel(a, c, drain_slots(a.accum, a.C, 0, c), drain_slots(a.accum, a.C, 1, c));
  if (c == 0 && a.num_batches_tracked) *a.num_batches_tracked += 1;
}

// -------------------------------------------------------------------------------------------------
// forward: y = dropout(act(bn(x) [+ skip]))
// -------------------------------------------------------------------------------------------------
struct BnActFwdArgs {
  const bf16* x;
  bf16* y;
  const bf16* skip;
  const float* mean;
  const float* invstd;
  const float* gamma;
  const float* beta;
  int N, H, W, C;
  int skip_mode, skip_C;
  int stat_is_var, relu, affine;
  float eps;
  float inv_keep;
  uint32_t drop_thr;  // drop when u16 < drop_thr
  uint64_t seed;
  const uint64_t* seed_offset;  // device step counter folded into the seed (CUDA-graph replays)
  // optional: running-statistics update of the batch norm whose mean / invstd came out of a conv kernel's
  // tail (done by the blocks with blockIdx.x == 0, one thread per 8-channel group)
  float* running_mean;
  float* running_var;
  int64_t* num_batches_tracked;
  float momentum;
  // optional: one byte per (pixel, 8-channel group); bit j = unit j passed the ReLU gate AND was kept by the
  // dropout. The backward kernels read this instead of y (1/16 of the bytes) and regenerate nothing.
  uint8_t* mask_out;
};

// the running-statistics update of 8 channels, kept OUT of line: inlined, its fp64 arithmetic cost the hot
// loop of bn_act_fwd_kernel<4, 4, false> four spilled registers at its 64-register cap (16.3 -> 19.5 us at
// 128x32x32x160)
__device__ __noinline__ void bn_act_fwd_running_update(const float* mean, const float* invstd, float eps,
                                                       float momentum, int64_t rows, float* running_mean,
                                                       float* running_var, int64_t* num_batches_tracked,
                                                       int cgi) {
  for (int j = 0; j < 8; ++j) {
    const int c = cgi * 8 + j;
    bn_running_update_channel(mean[c], invstd[c], eps, momentum, rows, running_mean, running_var, c);
  }
  if (cgi == 0 && num_batches_tracked) *num_batches_tracked += 1;
}

// Thread mapping of the element-wise BN kernels: a thread owns ONE 8-channel group for the whole
// kernel (per-channel coefficients live in registers) and walks rows with stride RP * gridDim.x;
// the RP x CGb threads of a block touch RP consecutive rows = one contiguous 4 KB span per pass.
// bit j of the result = half-word j of the four packed bf16x2 words is non-zero (+0 / -0 count as zero).
// Per word: (w & 0x7fff7fff) + 0x7fff7fff carries into bit 15 / 31 exactly when the 15 magnitude bits of that
// half are non-zero, and never across the halves.
__device__ __forceinline__ uint32_t nonzero_bits8(const uint4& w) {
  const uint32_t k0 = ((w.x & 0x7fff7fffu) + 0x7fff7fffu) & 0x80008000u;
  const uint32_t k1 = ((w.y & 0x7fff7fffu) + 0x7fff7fffu) & 0x80008000u;
  const uint32_t k2 = ((w.z & 0x7fff7fffu) + 0x7fff7fffu) & 0x80008000u;
  const uint32_t k3 = ((w.w & 0x7fff7fffu) + 0x7fff7fffu) & 0x80008000u;
  const uint32_t b = (k0 >> 15) | (k1 >> 13) | (k2 >> 11) | (k3 >> 9);   // bits 0,2,4,6 and 16,18,20,22
  return (b | (b >> 15)) & 0xffu;
}

// DROP = false: no random numbers in the kernel at all, and the bf16 rounding of the affine result is the one
// the final pack does (ReLU commutes with rounding); DROP = true: round, gate, scale by 1/(1-p), round again,
// like the reference's bf16 dropout of a bf16 activation.
// The mask byte comes from the packed OUTPUT when a ReLU is fused (y != 0 exactly where the unit was active and
// kept): ~16 integer operations per 8 elements instead of a compare + select + merge per element and gate —
// ncu (round 2) had this kernel at 55 % issue-slot use cold, i.e. issue-bound once the data streams warm.
// DROP: 0 = no dropout, 1 = dropout, 2 = dropout that keeps its keep bits: they ARE the mask when no ReLU is fused.
template <int U, int MINB, bool SKIP, int DROP>
__global__ void __launch_bounds__(EW_THREADS, MINB) bn_act_fwd_kernel(const BnActFwdArgs a) {
  const int C = a.C;
  ReduceGeom g(C);
  if (!g.active) return;
  const int cgi = g.cg0 + g.cgl;
  const int64_t rows = (int64_t)a.N * a.H * a.W;
  if (a.running_mean && blockIdx.x == 0 && g.rl == 0)   // before anything is live in registers
    bn_act_fwd_running_update(a.mean, a.invstd, a.eps, a.momentum, rows, a.running_mean, a.running_var,
                              a.num_batches_tracked, cgi);
  float sc[8], sh[8];
  if (a.affine) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = cgi * 8 + j;
      const float is = a.stat_is_var ? rsqrtf(a.invstd[c] + a.eps) : a.invstd[c];
      sc[j] = a.gamma[c] * is;
      sh[j] = a.beta[c] - a.mean[c] * sc[j];
    }
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) { sc[j] = 1.f; sh[j] = 0.f; }
  }
  const uint64_t seed = DROP ? effective_seed(a.seed, a.seed_offset) : 0;
  const bool skip_here = SKIP && (a.skip_mode == 1 || (a.skip_mode == 2 && cgi * 8 < a.skip_C));
  const int64_t stride = (int64_t)g.RP * gridDim.x;
  for (int64_t r0 = (int64_t)blockIdx.x * g.RP + g.rl; r0 < rows; r0 += U * stride) {
    Vec8 xv[U], sv[SKIP ? U : 1];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t r = r0 + u * stride;
      if (r < rows) {
        xv[u].raw = ldg_stream(a.x + ((size_t)r * g.CG + cgi) * 8);
        if (SKIP && skip_here) {
          size_t so;
          if (a.skip_mode == 1) {
            so = ((size_t)r * g.CG + cgi) * 8;
          } else {
            const int w = (int)(r % a.W);
            const int h = (int)((r / a.W) % a.H);
            const int n = (int)(r / ((int64_t)a.W * a.H));
            so = (((size_t)n * (2 * a.H) + 2 * h) * (2 * a.W) + 2 * w) * a.skip_C + (size_t)cgi * 8;
          }
          sv[SKIP ? u : 0].raw = ldg_stream(a.skip + so);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t r = r0 + u * stride;
      if (r >= rows) break;
      const size_t v = (size_t)r * g.CG + cgi;
      float f[8];
      xv[u].to_float(f);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = fmaf(f[j], sc[j], sh[j]);   // sc = 1, sh = 0 without the affine part: exact
      if (SKIP && skip_here) {
        float sk[8];
        sv[SKIP ? u : 0].to_float(sk);
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = round_bf16(f[j]) + sk[j];
      }
      uint32_t bits = 0xffu;
      if (DROP) round_bf16_pairs8(f);
      if (a.relu) {
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], 0.f);
      }
      if (DROP) {   // the pack below rounds; the keep bits are dead code unless DROP == 2
        const uint32_t keep = dropout8<false>(f, seed, v, a.drop_thr, a.inv_keep);
        if (DROP == 2) bits = keep;
      }
      Vec8 o;
      o.from_float(f);
      if (a.mask_out) {
        // with a fused ReLU the packed output is non-zero exactly where the unit was active AND kept, for every
        // DROP (the skip route runs DROP == 2 with or without a ReLU); the keep bits alone are the mask without it
        if (a.relu) bits = nonzero_bits8(o.raw);
        a.mask_out[v] = (uint8_t)bits;
      }
      stg_stream(a.y + v * 8, o.raw);
    }
  }
}

// -------------------------------------------------------------------------------------------------
// backward
// -------------------------------------------------------------------------------------------------
struct BnActBwdArgs {
  const bf16* dy;
  const bf16* y;
  const uint8_t* mask;
  const bf16* x;
  bf16* dx;
  bf16* dskip;
  const bf16* addend;
  const float* mean;
  const float* invstd;
  const float* gamma;
  float* dgamma;
  float* dbeta;
  int64_t rows;
  int C;
  int relu, affine;
  float inv_keep;
  uint32_t drop_thr;
  uint64_t seed;
  const uint64_t* seed_offset;
};

// g = dy * mask / (1-p), mask = ReLU gate AND dropout keep.
//   BITS = true : the forward stored the combined mask as one byte per 8-channel group (bn_act_fwd mask_out):
//                 0.125 B/element instead of the 2 B/element of y, and no random numbers are regenerated
//                 (ncu, round 1: both backward kernels read 126 MB for a 42 MB tensor: dy, x and y);
//   BITS = false: with a fused ReLU the saved forward output y is non-zero exactly where the unit was both
//                 active and kept; without ReLU the dropout mask is regenerated from the counter RNG.
template <bool BITS>
__device__ __forceinline__ void masked_grad_from(const BnActBwdArgs& a, uint64_t seed, size_t v, const Vec8& dv,
                                                 const Vec8& yv, uint32_t bits, float* g) {
  dv.to_float(g);
  if (BITS) {
    if (a.drop_thr) {
#pragma unroll
      for (int j = 0; j < 8; ++j) g[j] *= a.inv_keep;
      round_bf16_pairs8(g);
#pragma unroll
      for (int j = 0; j < 8; ++j) g[j] = ((bits >> j) & 1u) ? g[j] : 0.f;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) g[j] = ((bits >> j) & 1u) ? g[j] : 0.f;
    }
  } else if (a.relu) {
    float yf[8];
    yv.to_float(yf);
    if (a.drop_thr) {
#pragma unroll
      for (int j = 0; j < 8; ++j) g[j] = (yf[j] != 0.f) ? round_bf16(g[j] * a.inv_keep) : 0.f;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) g[j] = (yf[j] != 0.f) ? g[j] : 0.f;
    }
  } else if (a.drop_thr) {
    dropout8<true>(g, seed, v, a.drop_thr, a.inv_keep);
  }
}

// accum[0][c] += sum g, accum[1][c] += sum g * x; the last block writes dbeta = sum g and
// dgamma = invstd * (sum g*x - mean * sum g) (= sum g * xhat, finished in fp64) and clears accum
template <bool BITS>
__global__ void __launch_bounds__(EW_THREADS, 3)
bn_act_bwd_reduce_kernel(const BnActBwdArgs a, double* __restrict__ accum, unsigned int* ticket) {
  extern __shared__ float red_smem[];
  ReduceGeom g(a.C);
  float acc[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) acc[j] = 0.f;
  const uint64_t seed = a.drop_thr ? effective_seed(a.seed, a.seed_offset) : 0;
  if (g.active) {
    const int cgi = g.cg0 + g.cgl;
    constexpr int U = BITS ? 4 : 2;
    int64_t r0, r1;
    block_row_range(a.rows, g.RP, r0, r1);
    for (int64_t rb = r0 + g.rl; rb < r1; rb += U * (int64_t)g.RP) {
      Vec8 dv[U], yv[BITS ? 1 : U], xv[U];
      uint32_t mb[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t r = rb + u * (int64_t)g.RP;
        if (r < r1) {
          const size_t v = (size_t)r * g.CG + cgi;
          dv[u].raw = ldg_stream(a.dy + v * 8);
          if (BITS) mb[u] = __ldg(a.mask + v);
          else if (a.relu) yv[BITS ? 0 : u].raw = ldg_stream(a.y + v * 8);
          xv[u].raw = ldg_stream(a.x + v * 8);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t r = rb + u * (int64_t)g.RP;
        if (r >= r1) break;
        const size_t v = (size_t)r * g.CG + cgi;
        float gr[8], xf[8];
        xv[u].to_float(xf);
        masked_grad_from<BITS>(a, seed, v, dv[u], yv[BITS ? 0 : u], BITS ? mb[u] : 0u, gr);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc[j] += gr[j];
          acc[8 + j] = fmaf(gr[j], xf[j], acc[8 + j]);
        }
      }
    }
  }
  block_channel_reduce<2>(acc, red_smem, g.cgl, g.rl, g.CGb, g.RP, g.active, accum, a.C, g.cg0 * 8);
  if (!last_block_done(ticket)) return;
  for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
    const double s0 = drain_slots(accum, a.C, 0, c), s1 = drain_slots(accum, a.C, 1, c);
    a.dbeta[c] = (float)s0;
    a.dgamma[c] = (float)((double)a.invstd[c] * (s1 - (double)a.mean[c] * s0));
  }
  if (threadIdx.x == 0) *ticket = 0u;
}

// dx = gamma * invstd * (g - (dbeta + xhat * dgamma) / rows) [+ addend]; dskip = g.
// Per channel this is dx = k1 * g + k2 * x + k3 with
//   k1 = gamma*invstd, k2 = -k1*invstd*dgamma/rows, k3 = -k1*dbeta/rows - k2*mean   (registers).
// ADD / DSKIP: the launch may carry an addend / a dskip output (false: the pointers are not even looked at, and
// the addend vectors cost no registers: with them the common no-addend launch spilled nine registers per vector
// at the 80-register cap).
template <bool BITS, bool ADD, bool DSKIP>
__global__ void __launch_bounds__(EW_THREADS, 3) bn_act_bwd_apply_kernel(const BnActBwdArgs a) {
  const int C = a.C;
  ReduceGeom g(C);
  if (!g.active) return;
  const int cgi = g.cg0 + g.cgl;
  float k1[8], k2[8], k3[8];
  if (a.affine) {
    const float inv_rows = 1.f / (float)a.rows;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = cgi * 8 + j;
      const float is = a.invstd[c];
      k1[j] = a.gamma[c] * is;
      k2[j] = -k1[j] * is * a.dgamma[c] * inv_rows;
      k3[j] = -k1[j] * a.dbeta[c] * inv_rows - k2[j] * a.mean[c];
    }
  }
  const uint64_t seed = (!BITS && a.drop_thr) ? effective_seed(a.seed, a.seed_offset) : 0;
  const bool add = ADD && a.addend != nullptr;
  const int64_t stride = (int64_t)g.RP * gridDim.x;
  constexpr int U = 2;
  for (int64_t r0 = (int64_t)blockIdx.x * g.RP + g.rl; r0 < a.rows; r0 += U * stride) {
    Vec8 dv[U], yv[BITS ? 1 : U], xv[U], av[ADD ? U : 1];
    uint32_t mb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t r = r0 + u * stride;
      if (r < a.rows) {
        const size_t v = (size_t)r * g.CG + cgi;
        dv[u].raw = ldg_stream(a.dy + v * 8);
        if (BITS) mb[u] = __ldg(a.mask + v);
        else if (a.relu) yv[BITS ? 0 : u].raw = ldg_stream(a.y + v * 8);
        if (a.affine) xv[u].raw = ldg_stream(a.x + v * 8);
        if (add) av[ADD ? u : 0].raw = ldg_stream(a.addend + v * 8);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t r = r0 + u * stride;
      if (r >= a.rows) break;
      const size_t v = (size_t)r * g.CG + cgi;
      float gr[8], d[8], xf[8];
      if (a.affine) xv[u].to_float(xf);
      masked_grad_from<BITS>(a, seed, v, dv[u], yv[BITS ? 0 : u], BITS ? mb[u] : 0u, gr);
      if (DSKIP && a.dskip) {
        Vec8 o;
        o.from_float(gr);
        stg_stream(a.dskip + v * 8, o.raw);
      }
      if (a.affine) {
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = fmaf(k1[j], gr[j], fmaf(k2[j], xf[j], k3[j]));
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = gr[j];
      }
      if (add) {   // bf16 dx, then the bf16 sum: two roundings (the second one is the pack below)
        float af[8];
        av[ADD ? u : 0].to_float(af);
        round_bf16_pairs8(d);
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] += af[j];
      }
      Vec8 o;
      o.from_float(d);
      stg_stream(a.dx + v * 8, o.raw);
    }
  }
}

__global__ void tick_kernel(uint64_t* counter) { *counter += 1; }

// -------------------------------------------------------------------------------------------------
// subsample / upsample-add / parity split and merge
// -------------------------------------------------------------------------------------------------
// y[n,h,w,:] = x[n,2h,2w,:]   (y is [N,H,W,C], x is [N,2H,2W,C])
__global__ void subsample2_kernel(const bf16* __restrict__ x, bf16* __restrict__ y, int N, int H,
                                  int W, int C) {
  const int CG = C / 8;
  const size_t nvec = (size_t)N * H * W * CG;
  for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (size_t)gridDim.x * blockDim.x) {
    const int cg = (int)(v % CG);
    const size_t pix = v / CG;
    const int w = (int)(pix % W);
    const int h = (int)((pix / W) % H);
    const int n = (int)(pix / ((size_t)W * H));
    const size_t spix = ((size_t)n * (2 * H) + 2 * h) * (2 * W) + 2 * w;
    const uint4 t = ldg_stream(x + spix * C + (size_t)cg * 8);
    stg_stream(y + v * 8, t);
  }
}

// dx[n,2h,2w,c] = bf16(dx + g[n,h,w,c]) for c < Cg; g has channel pitch ldg >= Cg
__global__ void upsample_add_kernel(bf16* __restrict__ dx, const bf16* __restrict__ g, int N, int H,
                                    int W, int C, int Cg, int ldg) {
  const int CGg = Cg / 8;
  const size_t nvec = (size_t)N * H * W * CGg;
  for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (size_t)gridDim.x * blockDim.x) {
    const int cg = (int)(v % CGg);
    const size_t pix = v / CGg;
    const int w = (int)(pix % W);
    const int h = (int)((pix / W) % H);
    const int n = (int)(pix / ((size_t)W * H));
    const size_t dpix = ((size_t)n * (2 * H) + 2 * h) * (2 * W) + 2 * w;
    bf16* dp = dx + dpix * C + (size_t)cg * 8;
    Vec8 a, b;
    a.raw = *reinterpret_cast<const uint4*>(dp);
    b.raw = ldg_stream(g + pix * ldg + (size_t)cg * 8);
    float fa[8], fb[8];
    a.to_float(fa);
    b.to_float(fb);
#pragma unroll
    for (int j = 0; j < 8; ++j) fa[j] = round_bf16(fa[j] + fb[j]);
    a.from_float(fa);
    *reinterpret_cast<uint4*>(dp) = a.raw;
  }
}

// parity split: xs[(h%2)*2 + (w%2)][n][h/2][w/2][:] = x[n][h][w][:]; merge is the inverse
template <bool MERGE>
__global__ void parity_kernel(const bf16* __restrict__ src, bf16* __restrict__ dst, int N, int H,
                              int W, int C) {
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
    const size_t po = ppix * C + (size_t)cg * 8;
    if (MERGE) stg_stream(dst + v * 8, ldg_stream(src + po));
    else stg_stream(dst + po, ldg_stream(src + v * 8));
  }
}

// -------------------------------------------------------------------------------------------------
// layout: fp32 NCHW images -> bf16 NHWC; fp32 KRSC filters -> bf16 KRSC + bf16 CRSK
// -------------------------------------------------------------------------------------------------
__global__ void nchw_f32_to_nhwc_bf16_kernel(const float* __restrict__ x, bf16* __restrict__ y,
                                             int N, int C, int H, int W) {
  const size_t npix = (size_t)N * H * W;
  const size_t hw = (size_t)H * W;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npix;
       p += (size_t)gridDim.x * blockDim.x) {
    const size_t n = p / hw, r = p % hw;
    for (int c = 0; c < C; ++c)
      y[p * C + c] = __float2bfloat16_rn(x[(n * C + c) * hw + r]);
  }
}

__global__ void weight_cast_kernel(const float* __restrict__ w, bf16* __restrict__ o, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    o[i] = __float2bfloat16_rn(w[i]);
}

// w[K][RS][C] -> wt[C][RS][K]; 32x32 tiles over (K, C) for each filter tap (blockIdx.z)
__global__ void weight_transpose_kernel(const float* __restrict__ w, bf16* __restrict__ wt, int K,
                                        int RS, int C) {
  __shared__ float tile[32][33];
  const int rs = blockIdx.z;
  const int k0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int k = k0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (k < K && c < C) ? w[((size_t)k * RS + rs) * C + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, k = k0 + threadIdx.x;
    if (k < K && c < C) wt[((size_t)c * RS + rs) * K + k] = __float2bfloat16_rn(tile[threadIdx.x][i]);
  }
}

// All filters of a model in ONE launch: blockIdx.y = tensor, blocks stride over its 32x32 (K x C) tiles
// per filter tap; every tile is read once (coalesced along C) and written twice: bf16 KRSC (same layout)
// and bf16 CRSK (transposed through shared memory).
struct WeightPrepEntry {
  const float* w;   // fp32 [K][RS][C]
  bf16* wk;         // bf16 [K][RS][C]
  bf16* wt;         // bf16 [C][RS][K]
  int K, RS, C;
  int pad_;
};

__global__ void weight_prep_multi_kernel(const WeightPrepEntry* __restrict__ table) {
  // 64 x 64 (K x C) tiles, two elements per thread: 256-byte reads, 128-byte writes in both layouts
  // (the 32 x 32 scalar version moved 64-byte rows and reached 2.2 TB/s); odd K or C: scalar 32 x 32.
  __shared__ float tile[64][65];
  const WeightPrepEntry e = table[blockIdx.y];
  if (((e.K | e.C) & 1) == 0) {
    const int tk = (e.K + 63) / 64, tc_ = (e.C + 63) / 64;
    const int ntiles = tk * tc_ * e.RS;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const int rs = t / (tk * tc_);
      const int k0 = ((t / tc_) % tk) * 64, c0 = (t % tc_) * 64;
      __syncthreads();
      for (int i = threadIdx.y; i < 64; i += blockDim.y) {
        const int k = k0 + i, c = c0 + 2 * threadIdx.x;
        float2 v = make_float2(0.f, 0.f);
        if (k < e.K && c < e.C) {
          const size_t o = ((size_t)k * e.RS + rs) * e.C + c;
          v = *reinterpret_cast<const float2*>(e.w + o);
          *reinterpret_cast<__nv_bfloat162*>(e.wk + o) = __floats2bfloat162_rn(v.x, v.y);
        }
        tile[i][2 * threadIdx.x] = v.x;
        tile[i][2 * threadIdx.x + 1] = v.y;
      }
      __syncthreads();
      for (int i = threadIdx.y; i < 64; i += blockDim.y) {
        const int c = c0 + i, k = k0 + 2 * threadIdx.x;
        if (k < e.K && c < e.C)
          *reinterpret_cast<__nv_bfloat162*>(e.wt + ((size_t)c * e.RS + rs) * e.K + k) =
              __floats2bfloat162_rn(tile[2 * threadIdx.x][i], tile[2 * threadIdx.x + 1][i]);
      }
    }
    return;
  }
  const int tk = (e.K + 31) / 32, tc_ = (e.C + 31) / 32;
  const int ntiles = tk * tc_ * e.RS;
  for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
    const int rs = t / (tk * tc_);
    const int k0 = ((t / tc_) % tk) * 32, c0 = (t % tc_) * 32;
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int k = k0 + i, c = c0 + threadIdx.x;
      float v = 0.f;
      if (k < e.K && c < e.C) {
        const size_t o = ((size_t)k * e.RS + rs) * e.C + c;
        v = e.w[o];
        e.wk[o] = __float2bfloat16_rn(v);
      }
      tile[i][threadIdx.x] = v;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int c = c0 + i, k = k0 + threadIdx.x;
      if (k < e.K && c < e.C)
        e.wt[((size_t)c * e.RS + rs) * e.K + k] = __float2bfloat16_rn(tile[threadIdx.x][i]);
    }
  }
}

// -------------------------------------------------------------------------------------------------
// im2col for convolutions with very few input channels (the 3-channel stems): col[pix][kk] with
// kk = (r*S + s)*C + c, zero padded to Kpad columns, so the conv becomes a 1x1 conv over Kpad channels
// that the tcgen05 GEMM path can run. Also the matching zero-padding of filter rows.
// -------------------------------------------------------------------------------------------------
__global__ void im2col_kernel(const bf16* __restrict__ x, bf16* __restrict__ col, int N, int H, int W,
                              int C, int R, int S, int stride, int pad, int P, int Q, int Kpad) {
  // one thread per (pixel, 8-column group): 16-byte stores, the (r, s, c) walk advances incrementally
  const int groups = Kpad / 8;
  const size_t total = (size_t)N * P * Q * groups;
  const int rsc = R * S * C;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int gi = (int)(idx % groups);
    const size_t pix = idx / groups;
    const int q = (int)(pix % Q);
    const int p = (int)((pix / Q) % P);
    const int n = (int)(pix / ((size_t)Q * P));
    int kk = gi * 8;
    int c = kk % C, s = (kk / C) % S, r = kk / (C * S);
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j, ++kk) {
      float v = 0.f;
      if (kk < rsc) {
        const int ih = p * stride + r - pad, iw = q * stride + s - pad;
        if (ih >= 0 && ih < H && iw >= 0 && iw < W)
          v = __bfloat162float(x[(((size_t)n * H + ih) * W + iw) * C + c]);
      }
      f[j] = v;
      if (++c == C) { c = 0; if (++s == S) { s = 0; ++r; } }
    }
    Vec8 o;
    o.from_float(f);
    *reinterpret_cast<uint4*>(col + pix * Kpad + (size_t)gi * 8) = o.raw;
  }
}

// dst[row][0..cols_dst) = src[row][0..cols_src) zero padded (cols_dst >= cols_src) or truncated
template <typename T>
__global__ void repitch_rows_kernel(const T* __restrict__ src, T* __restrict__ dst, int rows,
                                    int cols_src, int cols_dst) {
  const size_t total = (size_t)rows * cols_dst;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % cols_dst);
    const size_t r = idx / cols_dst;
    dst[idx] = (c < cols_src) ? src[r * cols_src + c] : T(0.f);
  }
}

// -------------------------------------------------------------------------------------------------
// pooling
// -------------------------------------------------------------------------------------------------
struct PoolDims {
  int N, H, W, C, k, stride, pad, P, Q;
};

// average pooling, count_include_pad = True (torch.nn.AvgPool2d default)
__global__ void avgpool_fwd_kernel(const bf16* __restrict__ x, bf16* __restrict__ y, PoolDims d) {
  const int CG = d.C / 8;
  const size_t nvec = (size_t)d.N * d.P * d.Q * CG;
  const float inv = 1.f / (float)(d.k * d.k);
  for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (size_t)gridDim.x * blockDim.x) {
    const int cg = (int)(v % CG);
    const size_t pix = v / CG;
    const int q = (int)(pix % d.Q);
    const int p = (int)((pix / d.Q) % d.P);
    const int n = (int)(pix / ((size_t)d.Q * d.P));
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int r = 0; r < d.k; ++r) {
      const int h = p * d.stride + r - d.pad;
      if (h < 0 || h >= d.H) continue;
      for (int s = 0; s < d.k; ++s) {
        const int w = q * d.stride + s - d.pad;
        if (w < 0 || w >= d.W) continue;
        Vec8 xv;
        xv.raw = ldg_stream(x + (((size_t)n * d.H + h) * d.W + w) * d.C + (size_t)cg * 8);
        float f[8];
        xv.to_float(f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += f[j];
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] *= inv;
    Vec8 o;
    o.from_float(acc);
    stg_stream(y + v * 8, o.raw);
  }
}

// Global average pooling (k == H == W, pad 0: the `ap8,1,0` head of the CIFAR nets): one block per image,
// thread = (8-channel group, pixel lane), 4 independent 16-byte loads in flight per thread, shared-memory
// reduction over the pixel lanes. (The generic kernel walks the 64 pixels serially in one thread: 39.6 us
// for the 10 MB WRN tensor in round 1.)
__global__ void __launch_bounds__(EW_THREADS) avgpool_global_kernel(const bf16* __restrict__ x,
                                                                    bf16* __restrict__ y, int HW, int C) {
  __shared__ float red[EW_THREADS * 8];
  const int CG = C / 8;
  const int CGb = min(EW_THREADS, CG);
  const int RP = EW_THREADS / CGb;
  const int cgl = threadIdx.x % CGb, part = threadIdx.x / CGb;
  const int n = blockIdx.x;
  const float inv = 1.f / (float)HW;
  for (int cg0 = 0; cg0 < CG; cg0 += CGb) {
    const int cg = cg0 + cgl;
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (part < RP && cg < CG) {
      const bf16* base = x + (size_t)n * HW * C + (size_t)cg * 8;
      for (int p = part; p < HW; p += 4 * RP) {
        Vec8 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          v[u].raw = make_uint4(0u, 0u, 0u, 0u);
          if (p + u * RP < HW) v[u].raw = ldg_stream(base + (size_t)(p + u * RP) * C);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          float f[8];
          v[u].to_float(f);
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] += f[j];
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) red[threadIdx.x * 8 + j] = acc[j];
    __syncthreads();
    if (part == 0 && cg < CG) {
      float s[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] = 0.f;
      for (int r = 0; r < RP; ++r)
#pragma unroll
        for (int j = 0; j < 8; ++j) s[j] += red[(r * CGb + cgl) * 8 + j];
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] *= inv;
      Vec8 o;
      o.from_float(s);
      *reinterpret_cast<uint4*>(y + (size_t)n * C + (size_t)cg * 8) = o.raw;
    }
    __syncthreads();
  }
}

__global__ void avgpool_bwd_kernel(const bf16* __restrict__ dy, bf16* __restrict__ dx, PoolDims d) {
  const int CG = d.C / 8;
  const size_t nvec = (size_t)d.N * d.H * d.W * CG;
  const float inv = 1.f / (float)(d.k * d.k);
  for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (size_t)gridDim.x * blockDim.x) {
    const int cg = (int)(v % CG);
    const size_t pix = v / CG;
    const int w = (int)(pix % d.W);
    const int h = (int)((pix / d.W) % d.H);
    const int n = (int)(pix / ((size_t)d.W * d.H));
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int r = 0; r < d.k; ++r) {
      const int hp = h + d.pad - r;
      if (hp < 0 || (hp % d.stride) != 0) continue;
      const int p = hp / d.stride;
      if (p >= d.P) continue;
      for (int s = 0; s < d.k; ++s) {
        const int wp = w + d.pad - s;
        if (wp < 0 || (wp % d.stride) != 0) continue;
        const int q = wp / d.stride;
        if (q >= d.Q) continue;
        Vec8 g;
        g.raw = ldg_stream(dy + (((size_t)n * d.P + p) * d.Q + q) * d.C + (size_t)cg * 8);
        float f[8];
        g.to_float(f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += round_bf16(f[j] * inv);
      }
    }
    Vec8 o;
    o.from_float(acc);
    stg_stream(dx + v * 8, o.raw);
  }
}

// max pooling (padding behaves as -inf). `idx` (optional, one byte per output element) records WHICH window
// position r*k + s held the first maximum in row-major scan order (torch's max_pool2d_with_indices rule), so
// that the backward pass needs neither x nor y.
__global__ void maxpool_fwd_kernel(const bf16* __restrict__ x, bf16* __restrict__ y, uint8_t* __restrict__ idx,
                                   PoolDims d) {
  const int CG = d.C / 8;
  const size_t nvec = (size_t)d.N * d.P * d.Q * CG;
  for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (size_t)gridDim.x * blockDim.x) {
    const int cg = (int)(v % CG);
    const size_t pix = v / CG;
    const int q = (int)(pix % d.Q);
    const int p = (int)((pix / d.Q) % d.P);
    const int n = (int)(pix / ((size_t)d.Q * d.P));
    float m[8];
    uint32_t arg[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      m[j] = -INFINITY;
      arg[j] = 0;
    }
    for (int r = 0; r < d.k; ++r) {
      const int h = p * d.stride + r - d.pad;
      if (h < 0 || h >= d.H) continue;
      for (int s = 0; s < d.k; ++s) {
        const int w = q * d.stride + s - d.pad;
        if (w < 0 || w >= d.W) continue;
        Vec8 xv;
        xv.raw = ldg_stream(x + (((size_t)n * d.H + h) * d.W + w) * d.C + (size_t)cg * 8);
        float f[8];
        xv.to_float(f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (f[j] > m[j]) {   // strict: the FIRST maximum in scan order wins
            m[j] = f[j];
            arg[j] = (uint32_t)(r * d.k + s);
          }
        }
      }
    }
    Vec8 o;
    o.from_float(m);
    stg_stream(y + v * 8, o.raw);
    if (idx) {
      uint2 packed;
      packed.x = arg[0] | (arg[1] << 8) | (arg[2] << 16) | (arg[3] << 24);
      packed.y = arg[4] | (arg[5] << 8) | (arg[6] << 16) | (arg[7] << 24);
      *reinterpret_cast<uint2*>(idx + v * 8) = packed;
    }
  }
}

// Backward of max pooling from the recorded argmax positions: an input element (h, w) gathers dy of every window
// (p, q) that contains it and whose recorded position is exactly (h, w). 8 channels per thread; per input element
// at most ceil(k/stride)^2 windows, each costing 8 index bytes + 16 dy bytes (round 1 re-read x and y and
// re-scanned each window for ties: 18 ms for the 3.3 GB ImageNet-shape stem output).
__global__ void maxpool_bwd_kernel(const bf16* __restrict__ dy, const uint8_t* __restrict__ idx,
                                   bf16* __restrict__ dx, PoolDims d) {
  const int CG = d.C / 8;
  const size_t nvec = (size_t)d.N * d.H * d.W * CG;
  for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (size_t)gridDim.x * blockDim.x) {
    const int cg = (int)(v % CG);
    const size_t pix = v / CG;
    const int w = (int)(pix % d.W);
    const int h = (int)((pix / d.W) % d.H);
    const int n = (int)(pix / ((size_t)d.W * d.H));
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int r = 0; r < d.k; ++r) {
      const int hp = h + d.pad - r;
      if (hp < 0 || (hp % d.stride) != 0) continue;
      const int p = hp / d.stride;
      if (p >= d.P) continue;
      for (int s = 0; s < d.k; ++s) {
        const int wp = w + d.pad - s;
        if (wp < 0 || (wp % d.stride) != 0) continue;
        const int q = wp / d.stride;
        if (q >= d.Q) continue;
        const size_t o = ((((size_t)n * d.P + p) * d.Q + q) * d.C) + (size_t)cg * 8;
        const uint2 ib = *reinterpret_cast<const uint2*>(idx + o);
        const uint32_t pos = (uint32_t)(r * d.k + s);
        // bytes of ib equal to pos?
        uint32_t hit = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          hit |= (((ib.x >> (8 * j)) & 0xffu) == pos ? 1u : 0u) << j;
          hit |= (((ib.y >> (8 * j)) & 0xffu) == pos ? 1u : 0u) << (4 + j);
        }
        if (!hit) continue;
        Vec8 gv;
        gv.raw = ldg_stream(dy + o);
        float gf[8];
        gv.to_float(gf);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += ((hit >> j) & 1u) ? gf[j] : 0.f;
      }
    }
    Vec8 ov;
    ov.from_float(acc);
    stg_stream(dx + v * 8, ov.raw);
  }
}

// Compile-time window / stride versions of the two kernels above (the ImageNet-shape stem pool is k = 3, stride 2,
// pad 1 over a 3.3 GB tensor). One block row per image row: blockIdx.x = n * rows + row, blockIdx.y tiles the
// (column, 8-channel group) pairs of that row, so the only runtime division left is one 32-bit divide by C / 8.
// The generic kernels did four 64-bit divisions per vector and `% stride` per tap, and ran issue-bound at ~1/3
// (forward) and ~1/8 (backward) of the HBM rate: 1.96 ms and 5.54 ms per step in round 2's launch list.
template <int K, int S>
__global__ void __launch_bounds__(256)
maxpool_fwd_ks_kernel(const bf16* __restrict__ x, bf16* __restrict__ y, uint8_t* __restrict__ idx, PoolDims d) {
  const int CG = d.C >> 3;
  const int n = blockIdx.x / d.P, p = blockIdx.x - n * d.P;
  const int qc = d.Q * CG;
  const bf16* xn = x + (size_t)n * d.H * d.W * d.C;
  const size_t orow = ((size_t)n * d.P + p) * d.Q * d.C;
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < qc; i += gridDim.y * blockDim.x) {
    const int q = i / CG, cg = i - q * CG;
    float m[8];
    uint32_t arg[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      m[j] = -INFINITY;
      arg[j] = 0;
    }
    Vec8 xv[K * K];
#pragma unroll
    for (int r = 0; r < K; ++r) {
      const int h = p * S + r - d.pad;
#pragma unroll
      for (int s2 = 0; s2 < K; ++s2) {
        const int w = q * S + s2 - d.pad;
        const bool in = h >= 0 && h < d.H && w >= 0 && w < d.W;
        // out-of-range taps load nothing and never win (bf16 -inf pattern 0xff80 in every half)
        xv[r * K + s2].raw = make_uint4(0xff80ff80u, 0xff80ff80u, 0xff80ff80u, 0xff80ff80u);
        if (in) xv[r * K + s2].raw = ldg_stream(xn + ((size_t)h * d.W + w) * d.C + (size_t)cg * 8);
      }
    }
#pragma unroll
    for (int t = 0; t < K * K; ++t) {
      float f[8];
      xv[t].to_float(f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (f[j] > m[j]) {   // strict: the FIRST maximum in scan order wins
          m[j] = f[j];
          arg[j] = (uint32_t)t;
        }
      }
    }
    Vec8 o;
    o.from_float(m);
    const size_t off = orow + (size_t)i * 8;
    stg_stream(y + off, o.raw);
    if (idx) {
      uint2 packed;
      packed.x = arg[0] | (arg[1] << 8) | (arg[2] << 16) | (arg[3] << 24);
      packed.y = arg[4] | (arg[5] << 8) | (arg[6] << 16) | (arg[7] << 24);
      *reinterpret_cast<uint2*>(idx + off) = packed;
    }
  }
}

template <int K, int S>
__global__ void __launch_bounds__(256)
maxpool_bwd_ks_kernel(const bf16* __restrict__ dy, const uint8_t* __restrict__ idx, bf16* __restrict__ dx,
                      PoolDims d) {
  const int CG = d.C >> 3;
  const int n = blockIdx.x / d.H, h = blockIdx.x - n * d.H;
  const int wc = d.W * CG;
  const size_t obase = (size_t)n * d.P * d.Q * d.C;
  const size_t irow = ((size_t)n * d.H + h) * d.W * d.C;
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < wc; i += gridDim.y * blockDim.x) {
    const int w = i / CG, cg = i - w * CG;
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int r = 0; r < K; ++r) {
      const int hp = h + d.pad - r;
      if (hp < 0 || (hp % S) != 0) continue;
      const int p = hp / S;
      if (p >= d.P) continue;
#pragma unroll
      for (int s2 = 0; s2 < K; ++s2) {
        const int wp = w + d.pad - s2;
        if (wp < 0 || (wp % S) != 0) continue;
        const int q = wp / S;
        if (q >= d.Q) continue;
        const size_t o = obase + ((size_t)p * d.Q + q) * d.C + (size_t)cg * 8;
        const uint2 ib = __ldg(reinterpret_cast<const uint2*>(idx + o));
        // bytes of ib equal to this tap's position r * K + s? (SIMD byte compare: 0xff per equal byte)
        const uint32_t pos4 = (uint32_t)(r * K + s2) * 0x01010101u;
        const uint32_t e0 = __vcmpeq4(ib.x, pos4), e1 = __vcmpeq4(ib.y, pos4);
        if ((e0 | e1) == 0u) continue;
        Vec8 gv;
        gv.raw = ldg_stream(dy + o);
        float gf[8];
        gv.to_float(gf);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc[j] += ((e0 >> (8 * j)) & 1u) ? gf[j] : 0.f;
          acc[4 + j] += ((e1 >> (8 * j)) & 1u) ? gf[4 + j] : 0.f;
        }
      }
    }
    Vec8 ov;
    ov.from_float(acc);
    stg_stream(dx + irow + (size_t)i * 8, ov.raw);
  }
}

}  // namespace b200
