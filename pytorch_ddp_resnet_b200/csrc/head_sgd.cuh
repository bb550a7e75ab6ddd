// Classifier head (Linear + cross-entropy + top-k) and the fused multi-tensor SGD and Adam updates.
// The head is tiny ([B,640] x [640,10] for WRN-28-10): latency matters, not throughput, so these
// are warp-per-output kernels with shuffle reductions. The SGD kernel is HBM-bound (20 B/param),
// so is the Adam kernel (28 B/param).
#pragma once
#include "common.cuh"

namespace b200 {

// logits[b][o] = bf16( sum_i x[b][i] * bf16(w[o][i]) + bf16(bias[o]) ); one warp per (b, o)
__global__ void linear_fwd_kernel(const bf16* __restrict__ x, const float* __restrict__ w,
                                  const float* __restrict__ bias, bf16* __restrict__ y, int B, int I,
                                  int O) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= B * O) return;
  const int b = warp / O, o = warp % O;
  float acc = 0.f;
  for (int i = lane; i < I; i += 32)
    acc = fmaf(__bfloat162float(x[(size_t)b * I + i]), round_bf16(w[(size_t)o * I + i]), acc);
  acc = warp_sum(acc);
  if (lane == 0) {
    if (bias) acc += round_bf16(bias[o]);
    y[(size_t)b * O + o] = __float2bfloat16_rn(acc);
  }
}

// dx[b][i] = bf16( sum_o dy[b][o] * bf16(w[o][i]) ); thread per (b, i)
__global__ void linear_bwd_dx_kernel(const bf16* __restrict__ dy, const float* __restrict__ w,
                                     bf16* __restrict__ dx, int B, int I, int O) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)B * I) return;
  const int b = (int)(idx / I), i = (int)(idx % I);
  float acc = 0.f;
  for (int o = 0; o < O; ++o)
    acc = fmaf(__bfloat162float(dy[(size_t)b * O + o]), round_bf16(w[(size_t)o * I + i]), acc);
  dx[idx] = __float2bfloat16_rn(acc);
}

// dw[o][i] = sum_b dy[b][o] * x[b][i]; thread per (o, i); db[o] = sum_b dy[b][o] (threads with i == 0)
__global__ void linear_bwd_dw_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ x,
                                     float* __restrict__ dw, float* __restrict__ db, int B, int I,
                                     int O) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)O * I) return;
  const int o = (int)(idx / I), i = (int)(idx % I);
  float acc = 0.f, accb = 0.f;
#pragma unroll 8
  for (int b = 0; b < B; ++b) {
    const float g = __bfloat162float(dy[(size_t)b * O + o]);
    acc = fmaf(g, __bfloat162float(x[(size_t)b * I + i]), acc);
    accb += g;
  }
  dw[idx] = acc;
  if (i == 0 && db) db[o] = accb;
}

// ONE block of CE_WARPS warps; warp w handles samples w, w + CE_WARPS, ... out[0] = mean loss, out[1] = fraction of
// labels that are not the top-1, out[2] = not in the top-5 (written, not accumulated: no zeroing needed).
// dlogits = (softmax - onehot) * scale / B. The sums run in a FIXED order (per warp over its samples, then over the
// warps): the reported loss is bit-reproducible (round 1 added one atomic per sample, in completion order).
constexpr int CE_WARPS = 32;

__device__ __forceinline__ void ce_block_sum3(float loss, float e1, float e5, float* __restrict__ out, int B) {
  __shared__ float s_acc[CE_WARPS][3];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { s_acc[warp][0] = loss; s_acc[warp][1] = e1; s_acc[warp][2] = e5; }
  __syncthreads();
  if (threadIdx.x < 3) {
    float t = 0.f;
    for (int w = 0; w < CE_WARPS; ++w) t += s_acc[w][threadIdx.x];
    out[threadIdx.x] = t / (float)B;
  }
}

__global__ void __launch_bounds__(CE_WARPS * 32)
ce_topk_kernel(const bf16* __restrict__ logits, const int64_t* __restrict__ labels,
               float* __restrict__ out, bf16* __restrict__ dlogits,
               const float* __restrict__ grad_scale, int B, int O) {
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  float loss = 0.f, e1 = 0.f, e5 = 0.f;
  for (int b = warp; b < B; b += CE_WARPS) {
    const bf16* row = logits + (size_t)b * O;
    const int label = (int)labels[b];
    float mx = -INFINITY;
    for (int o = lane; o < O; o += 32) mx = fmaxf(mx, __bfloat162float(row[o]));
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, s));
    float se = 0.f;
    for (int o = lane; o < O; o += 32) se += __expf(__bfloat162float(row[o]) - mx);
    se = warp_sum(se);
    const float lse = mx + __logf(se);
    const float zl = __bfloat162float(row[label]);
    if (out) {
      // rank of the label: logits strictly larger, ties broken towards the lower index
      float rank = 0.f;
      for (int o = lane; o < O; o += 32) {
        const float z = __bfloat162float(row[o]);
        rank += (z > zl || (z == zl && o < label)) ? 1.f : 0.f;
      }
      rank = warp_sum(rank);
      loss += lse - zl;
      e1 += rank >= 1.f ? 1.f : 0.f;
      e5 += rank >= 5.f ? 1.f : 0.f;
    }
    if (dlogits) {
      const float sc = (grad_scale ? *grad_scale : 1.f) / (float)B;
      for (int o = lane; o < O; o += 32) {
        const float p = __expf(__bfloat162float(row[o]) - lse);
        dlogits[(size_t)b * O + o] = __float2bfloat16_rn((p - (o == label ? 1.f : 0.f)) * sc);
      }
    }
  }
  if (out) ce_block_sum3(loss, e1, e5, out, B);
}

// -------------------------------------------------------------------------------------------------
// SGD with momentum / dampening / nesterov / weight decay over a list of tensors (torch.optim.SGD)
// grid = (chunks, n_tensors); each block handles 1024 float4 of one tensor
// -------------------------------------------------------------------------------------------------
struct SgdArgs {
  float* const* params;
  const float* const* grads;
  float* const* bufs;
  const int64_t* sizes;
  float lr, momentum, dampening, weight_decay;
  int nesterov, first_step;
  const float* inv_scale;
  const float* found_inf;
  const float* lr_ptr;  // device-resident learning rate (overrides lr when non-null)
};

constexpr int SGD_THREADS = 256;
constexpr int SGD_VEC_PER_THREAD = 4;

__device__ __forceinline__ float sgd_one(float& p, float g, float& buf, const SgdArgs& a, float is,
                                         float lr) {
  g *= is;
  g = fmaf(a.weight_decay, p, g);
  if (a.momentum != 0.f) {
    buf = a.first_step ? g : fmaf(a.momentum, buf, (1.f - a.dampening) * g);
    g = a.nesterov ? fmaf(a.momentum, buf, g) : buf;
  }
  p = fmaf(-lr, g, p);
  return p;
}

__global__ void __launch_bounds__(SGD_THREADS) sgd_step_kernel(const SgdArgs a) {
  if (a.found_inf && *a.found_inf != 0.f) return;
  const int t = blockIdx.y;
  const int64_t n = a.sizes[t];
  const int64_t chunk = (int64_t)SGD_THREADS * SGD_VEC_PER_THREAD * 4;
  const int64_t start = (int64_t)blockIdx.x * chunk;
  if (start >= n) return;
  float* p = a.params[t];
  const float* g = a.grads[t];
  float* m = a.bufs[t];
  const float is = a.inv_scale ? *a.inv_scale : 1.f;
  const float lr = a.lr_ptr ? *a.lr_ptr : a.lr;
  const bool aligned = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) |
                         reinterpret_cast<uintptr_t>(m)) & 15) == 0;
#pragma unroll
  for (int u = 0; u < SGD_VEC_PER_THREAD; ++u) {
    const int64_t i = start + ((int64_t)u * SGD_THREADS + threadIdx.x) * 4;
    if (i >= n) break;
    if (aligned && i + 4 <= n) {
      float4 pv = *reinterpret_cast<float4*>(p + i);
      const float4 gv = *reinterpret_cast<const float4*>(g + i);
      float4 mv = a.first_step ? make_float4(0, 0, 0, 0) : *reinterpret_cast<float4*>(m + i);
      sgd_one(pv.x, gv.x, mv.x, a, is, lr);
      sgd_one(pv.y, gv.y, mv.y, a, is, lr);
      sgd_one(pv.z, gv.z, mv.z, a, is, lr);
      sgd_one(pv.w, gv.w, mv.w, a, is, lr);
      *reinterpret_cast<float4*>(p + i) = pv;
      if (a.momentum != 0.f) *reinterpret_cast<float4*>(m + i) = mv;
    } else {
      for (int64_t j = i; j < min(n, i + 4); ++j) {
        float pv = p[j], mv = a.first_step ? 0.f : m[j];
        sgd_one(pv, g[j], mv, a, is, lr);
        p[j] = pv;
        if (a.momentum != 0.f) m[j] = mv;
      }
    }
  }
}

// -------------------------------------------------------------------------------------------------
// Adam / AdamW (torch.optim.Adam, torch.optim.AdamW) over a list of tensors, the grid shape of SGD:
// grid = (chunks, n_tensors); each block handles 2048 float4 of one tensor. 28 B / parameter
// (p, m, v read + written, g read), 36 B with amsgrad.
// The step counter lives on the device (one fp32 scalar per tensor, torch's fused / capturable format)
// and the launch advances it, so every CUDA-graph replay does. Every block computes with the value from
// before the launch; the block that finishes last for a tensor (ticket counter, zero on entry and on
// exit) writes step + 1.
// -------------------------------------------------------------------------------------------------
struct AdamArgs {
  float* const* params;
  const float* const* grads;
  float* const* exp_avgs;
  float* const* exp_avg_sqs;
  float* const* max_exp_avg_sqs;  // NULL unless amsgrad
  float* const* steps;
  const int64_t* sizes;
  unsigned* tickets;              // n zeroed counters
  double lr, beta1, beta2, eps, weight_decay;
  int decoupled, amsgrad;
  const float* inv_scale;
  const float* found_inf;
  const float* lr_ptr;  // device-resident learning rate (overrides lr when non-null)
};

constexpr int ADAM_THREADS = 256;
constexpr int ADAM_VEC_PER_THREAD = 8;  // 8192 elements per block: amortizes the fp64 bias-correction prologue
constexpr int64_t ADAM_CHUNK = (int64_t)ADAM_THREADS * ADAM_VEC_PER_THREAD * 4;

// Per-launch scalars, computed as torch computes them on the host (fp64, then rounded to fp32 where torch
// hands them to an fp32 kernel as a Python scalar).
struct AdamCoef {
  float is, wd, decay, b1c, b2, b2c, eps, bc2_sqrt, neg_step_size;
};

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, float& vmax, const AdamArgs& a,
                                         const AdamCoef& c) {
  g *= c.is;
  if (a.weight_decay != 0.0) {
    if (a.decoupled) p *= c.decay;            // param.mul_(1 - lr * wd)
    else g = fmaf(c.wd, p, g);                // grad = grad.add(param, alpha=wd)
  }
  m = fmaf(c.b1c, g - m, m);                  // exp_avg.lerp_(grad, 1 - beta1)
  v = fmaf(c.b2c * g, g, c.b2 * v);           // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
  float vv = v;
  if (a.amsgrad) {
    vmax = fmaxf(vmax, v);
    vv = vmax;
  }
  const float denom = sqrtf(vv) / c.bc2_sqrt + c.eps;
  p = fmaf(c.neg_step_size, m / denom, p);    // param.addcdiv_(exp_avg, denom, value=-step_size)
}

__global__ void __launch_bounds__(ADAM_THREADS) adam_step_kernel(const AdamArgs a) {
  if (a.found_inf && *a.found_inf != 0.f) return;
  const int t = blockIdx.y;
  const int64_t n = a.sizes[t];
  const int64_t start = (int64_t)blockIdx.x * ADAM_CHUNK;
  if (start >= n && blockIdx.x != 0) return;  // block 0 always takes part: an empty tensor still counts a step
  float* p = a.params[t];
  const float* g = a.grads[t];
  float* m = a.exp_avgs[t];
  float* v = a.exp_avg_sqs[t];
  float* vm = a.amsgrad ? a.max_exp_avg_sqs[t] : v;  // only touched with amsgrad
  const float step = *a.steps[t];
  // the pointers come from a table, so the compiler cannot tell their address space: say it (global
  // LDG / STG instead of generic LD / ST)
  __builtin_assume(__isGlobal(p) && __isGlobal(g) && __isGlobal(m) && __isGlobal(v) && __isGlobal(vm));

  AdamCoef c;
  {
    const double lr = a.lr_ptr ? (double)*a.lr_ptr : a.lr;
    const double s = (double)(step + 1.f);    // torch: step_t += 1 on the fp32 tensor, then its value
    const double bc1 = 1.0 - pow(a.beta1, s);
    const double bc2 = 1.0 - pow(a.beta2, s);
    c.is = a.inv_scale ? *a.inv_scale : 1.f;
    c.wd = (float)a.weight_decay;
    c.decay = (float)(1.0 - lr * a.weight_decay);
    c.b1c = (float)(1.0 - a.beta1);
    c.b2 = (float)a.beta2;
    c.b2c = (float)(1.0 - a.beta2);
    c.eps = (float)a.eps;
    c.bc2_sqrt = (float)sqrt(bc2);
    c.neg_step_size = (float)(-(lr / bc1));
  }

  const bool aligned = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) |
                         reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v) |
                         reinterpret_cast<uintptr_t>(vm)) & 15) == 0;
#pragma unroll
  for (int u = 0; u < ADAM_VEC_PER_THREAD; ++u) {
    const int64_t i = start + ((int64_t)u * ADAM_THREADS + threadIdx.x) * 4;
    if (i >= n) break;
    if (aligned && i + 4 <= n) {
      float4 pv = *reinterpret_cast<float4*>(p + i);
      const float4 gv = *reinterpret_cast<const float4*>(g + i);
      float4 mv = *reinterpret_cast<float4*>(m + i);
      float4 vv = *reinterpret_cast<float4*>(v + i);
      float4 xv = a.amsgrad ? *reinterpret_cast<float4*>(vm + i) : make_float4(0, 0, 0, 0);
      adam_one(pv.x, gv.x, mv.x, vv.x, xv.x, a, c);
      adam_one(pv.y, gv.y, mv.y, vv.y, xv.y, a, c);
      adam_one(pv.z, gv.z, mv.z, vv.z, xv.z, a, c);
      adam_one(pv.w, gv.w, mv.w, vv.w, xv.w, a, c);
      *reinterpret_cast<float4*>(p + i) = pv;
      *reinterpret_cast<float4*>(m + i) = mv;
      *reinterpret_cast<float4*>(v + i) = vv;
      if (a.amsgrad) *reinterpret_cast<float4*>(vm + i) = xv;
    } else {
      for (int64_t j = i; j < min(n, i + 4); ++j) {
        float pv = p[j], mv = m[j], vv = v[j], xv = a.amsgrad ? vm[j] : 0.f;
        adam_one(pv, g[j], mv, vv, xv, a, c);
        p[j] = pv;
        m[j] = mv;
        v[j] = vv;
        if (a.amsgrad) vm[j] = xv;
      }
    }
  }

  // last block of tensor t: every other block has read `step` (it took its ticket after its loads)
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned blocks = n > 0 ? (unsigned)((n + ADAM_CHUNK - 1) / ADAM_CHUNK) : 1u;
    __threadfence();
    if (atomicAdd(&a.tickets[t], 1u) == blocks - 1) {
      a.tickets[t] = 0u;
      *a.steps[t] = step + 1.f;
    }
  }
}

}  // namespace b200
