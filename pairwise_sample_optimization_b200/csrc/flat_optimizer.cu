// Optimizer boundary of the PSO training step over the FLAT LoRA buffers: global-norm clipping + AdamW + refresh of the
// 16-bit GEMM operand copies + zeroing of the gradient, in two launches for all 1120 adapter matrices.
//
// Replaces, at every accumulation boundary (train_online_pso_sdxl_turbo.py:858-861): accelerate's clip_grad_norm_ (one
// norm kernel per parameter + stack + norm + one scale per parameter), optimizer.step() (AdamW, :428-448) and
// optimizer.zero_grad(), plus this repo's own per-layer fp32 -> bf16 operand refresh.  Pure streaming work: 5 fp32 reads
// + 3 fp32 writes + one 16-bit write per parameter.
#include <atomic>
#include <cmath>

#include "common.cuh"

namespace psob200 {

constexpr int kOptThreads = 256;

// sum of squares of the gradient into ws[0] (double), block partials combined with one atomic per block
__global__ void __launch_bounds__(kOptThreads) flat_sumsq_kernel(const float* __restrict__ g, long long n, double* ws) {
  float acc = 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x * 4;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
    if (i + 4 <= n) {
      const float4 v = *reinterpret_cast<const float4*>(g + i);
      acc = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, acc))));
    } else {
      for (long long j = i; j < n; ++j) acc = fmaf(g[j], g[j], acc);
    }
  }
  acc = warp_sum(acc);
  __shared__ float s[kOptThreads / 32];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < kOptThreads / 32 ? s[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(ws, (double)v);
  }
}

// ---- data-parallel exchange fused into the optimizer boundary (NVLink SHARP through the multicast mapping) -------------
// The flat gradient buffer is symmetric memory, mapped at `mc` as a MULTICAST address: a load-reduce from it returns the
// sum of the N ranks' copies, computed inside the NVSwitch; a store to it lands in every rank's copy.  Rank r owns the
// slice [lo, hi): it pulls the reduced values (reduce-scatter), scales them to the mean, pushes them back to all ranks
// (all-gather) and, on the way, accumulates the sum of squares of its slice -- the global-norm pass of clip_grad_norm_
// costs no extra read.  Each rank's partial norm is added into slot `rank` of a small symmetric array on every rank.
// The caller brackets this launch with two cross-rank barriers (all backward passes done before; all slices written
// after); every rank ends up with bitwise-identical gradients and norm.
__device__ __forceinline__ float4 multimem_ld_reduce_add(const float* mc) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc) : "memory");
  return v;
}
__device__ __forceinline__ void multimem_st(float* mc, const float4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

__global__ void __launch_bounds__(kOptThreads)
flat_allreduce_sumsq_kernel(float* mc, double* mc_sumsq_slot, long long lo, long long hi, float scale) {
  float acc = 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x * 4;
  for (long long i = lo + ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < hi; i += stride) {
    float4 v = multimem_ld_reduce_add(mc + i);
    v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
    multimem_st(mc + i, v);
    acc = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, acc))));
  }
  acc = warp_sum(acc);
  __shared__ float s[kOptThreads / 32];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < kOptThreads / 32 ? s[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) {
      const double d = (double)v;
      asm volatile("multimem.red.relaxed.sys.global.add.f64 [%0], %1;" ::"l"(mc_sumsq_slot), "d"(d) : "memory");
    }
  }
}

struct AdamParams {
  float lr, beta1, beta2, eps, weight_decay, bc1, bc2_sqrt, max_norm, grad_scale;
  float* found_inf;
  long long* step_dev;
};

template <typename TO>
__global__ void __launch_bounds__(kOptThreads)
flat_adamw_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, TO* __restrict__ op,
                  long long n, AdamParams a, double* ws, float* norm_out, double* parts, int n_parts) {
  // global-norm clip coefficient (accelerate / torch clip_grad_norm_: coef = min(1, max_norm / (norm + 1e-6)))
  double sumsq = ws[0];
  for (int r = 0; r < n_parts; ++r) sumsq += parts[r];  // per-rank slices of the fused exchange (same order on every rank)
  const float norm = (float)sqrt(sumsq) * a.grad_scale;
  // a non-finite norm (overflowed fp16 gradients, or a NaN anywhere: fminf would silently drop it) skips the whole update,
  // as GradScaler.step does; torch's clip_grad_norm_ would instead smear the NaN over every parameter
  const bool skip = !(norm <= 3.4028234e38f);
  const float coef = a.max_norm > 0.f ? fminf(1.f, a.max_norm / (norm + 1e-6f)) * a.grad_scale : a.grad_scale;
  float bc1 = a.bc1, bc2_sqrt = a.bc2_sqrt;
  if (a.step_dev != nullptr) {  // device-side step count: read by every thread before the last block advances it
    const double t = (double)(*a.step_dev + 1);
    bc1 = (float)(1.0 - pow((double)a.beta1, t));
    bc2_sqrt = (float)sqrt(1.0 - pow((double)a.beta2, t));
  }
  const long long stride = (long long)gridDim.x * blockDim.x;
  if (skip) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) g[i] = 0.f;
  } else {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
      const float gi = g[i] * coef;
      float pi = p[i] * (1.f - a.lr * a.weight_decay);          // decoupled weight decay
      const float mi = fmaf(1.f - a.beta1, gi - m[i], m[i]);    // exp_avg.lerp_(g, 1 - beta1)
      const float vi = fmaf(a.beta2, v[i], (1.f - a.beta2) * gi * gi);
      const float denom = sqrtf(vi) / bc2_sqrt + a.eps;
      pi -= (a.lr / bc1) * (mi / denom);
      p[i] = pi;
      m[i] = mi;
      v[i] = vi;
      g[i] = 0.f;                                               // optimizer.zero_grad()
      if (op != nullptr) Vec8<TO>::store1(op + i, pi);          // the GEMM kernels' 16-bit operand copy
    }
  }
  // the last block to finish publishes the norm and leaves the workspace zeroed for the next boundary
  __shared__ unsigned ticket;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    ticket = atomicAdd(reinterpret_cast<unsigned*>(ws + 1), 1u);
  }
  __syncthreads();
  if (ticket == gridDim.x - 1 && threadIdx.x == 0) {
    if (norm_out != nullptr) *norm_out = norm;
    if (a.found_inf != nullptr) *a.found_inf = skip ? 1.f : 0.f;
    if (a.step_dev != nullptr && !skip) *a.step_dev += 1;  // every block has read it: this is the last one to finish
    ws[0] = 0.0;
    *reinterpret_cast<unsigned*>(ws + 1) = 0u;
    for (int r = 0; r < n_parts; ++r) parts[r] = 0.0;  // local copy only: peers zero theirs; next use is behind a barrier
  }
}

int launch_flat_sumsq(const float* g, long long n, double* ws, int n_sm, cudaStream_t st) {
  long long blocks = (n + kOptThreads * 4 - 1) / (kOptThreads * 4);
  if (blocks > n_sm * 8) blocks = n_sm * 8;
  flat_sumsq_kernel<<<(unsigned)blocks, kOptThreads, 0, st>>>(g, n, ws);
  return consume_launch_error("launch flat_sumsq_kernel", cudaSuccess);
}

}  // namespace psob200

using namespace psob200;

extern "C" int psob200_flat_adamw_step(const psob200_flat_adamw_args* args, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_flat_adamw_args& o = *args;
  if (!o.param || !o.grad || !o.exp_avg || !o.exp_avg_sq || !o.workspace || o.n <= 0 || (o.step <= 0 && !o.step_dev))
    return PSOB200_ERR_INVALID_ARG;
  if (o.operand && o.operand_dtype != PSOB200_BF16 && o.operand_dtype != PSOB200_F16) return PSOB200_ERR_DTYPE;
  if (!aligned16(o.grad) || !aligned16(o.workspace)) return PSOB200_ERR_ALIGNMENT;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  static PerDevice<int> sms_dev;
  std::atomic<int>& sms = sms_dev.here();
  int n_sm = sms.load(std::memory_order_relaxed);
  if (n_sm <= 0) {
    n_sm = psob200_device_sm_count();
    if (n_sm <= 0) n_sm = 148;
    sms.store(n_sm, std::memory_order_relaxed);
  }
  double* ws = reinterpret_cast<double*>(o.workspace);
  if (o.n_sumsq_parts < 0 || (o.n_sumsq_parts > 0 && !o.sumsq_parts)) return PSOB200_ERR_INVALID_ARG;
  if (o.n_sumsq_parts == 0 && (o.max_grad_norm > 0.f || o.norm_out != nullptr)) {
    const int rc = launch_flat_sumsq(o.grad, o.n, ws, n_sm, st);
    if (rc != PSOB200_OK) return rc;
  }
  AdamParams a;
  a.lr = o.lr; a.beta1 = o.beta1; a.beta2 = o.beta2; a.eps = o.eps; a.weight_decay = o.weight_decay;
  a.bc1 = (float)(1.0 - std::pow((double)o.beta1, (double)o.step));
  a.bc2_sqrt = (float)std::sqrt(1.0 - std::pow((double)o.beta2, (double)o.step));
  a.max_norm = o.max_grad_norm;
  a.grad_scale = o.grad_scale;
  a.found_inf = o.found_inf;
  a.step_dev = o.step_dev;
  long long blocks = (o.n + kOptThreads - 1) / kOptThreads;
  if (blocks > n_sm * 8) blocks = n_sm * 8;
  if (o.operand == nullptr || o.operand_dtype == PSOB200_BF16)
    flat_adamw_kernel<__nv_bfloat16><<<(unsigned)blocks, kOptThreads, 0, st>>>(
        o.param, o.grad, o.exp_avg, o.exp_avg_sq, reinterpret_cast<__nv_bfloat16*>(o.operand), o.n, a, ws, o.norm_out, o.sumsq_parts,
        o.n_sumsq_parts);
  else
    flat_adamw_kernel<__half><<<(unsigned)blocks, kOptThreads, 0, st>>>(
        o.param, o.grad, o.exp_avg, o.exp_avg_sq, reinterpret_cast<__half*>(o.operand), o.n, a, ws, o.norm_out, o.sumsq_parts, o.n_sumsq_parts);
  return consume_launch_error("launch flat_adamw_kernel", cudaSuccess);
}

extern "C" int psob200_flat_allreduce_sumsq(const psob200_flat_allreduce_args* args, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_flat_allreduce_args& o = *args;
  if (!o.grad_multicast || !o.sumsq_multicast || o.n <= 0 || o.world <= 0 || o.rank < 0 || o.rank >= o.world)
    return PSOB200_ERR_INVALID_ARG;
  if (!aligned16(o.grad_multicast) || (reinterpret_cast<uintptr_t>(o.sumsq_multicast) & 7u)) return PSOB200_ERR_ALIGNMENT;
  if (o.n % 4) return PSOB200_ERR_SHAPE;  // 128-bit multimem accesses
  // slices of whole 16-byte vectors; the last ranks may own less (or nothing)
  const long long vecs = o.n / 4, per = (vecs + o.world - 1) / o.world;
  long long lo = per * o.rank * 4, hi = per * (o.rank + 1) * 4;
  if (lo > o.n) lo = o.n;
  if (hi > o.n) hi = o.n;
  int n_sm = psob200_device_sm_count();
  if (n_sm <= 0) n_sm = 148;
  long long blocks = (hi - lo + kOptThreads * 4 - 1) / (kOptThreads * 4);
  if (blocks > n_sm * 4) blocks = n_sm * 4;
  if (blocks < 1) blocks = 1;  // an empty slice still launches: uniform launch sequence on every rank
  flat_allreduce_sumsq_kernel<<<(unsigned)blocks, kOptThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      o.grad_multicast, o.sumsq_multicast + o.rank, lo, hi, o.scale);
  return consume_launch_error("launch flat_allreduce_sumsq_kernel", cudaSuccess);
}
