// Optimizer boundary of the PSO training step over the FLAT LoRA buffers: global-norm clipping + AdamW + refresh of the
// 16-bit GEMM operand copies + zeroing of the gradient, in two launches for all 1120 adapter matrices.
//
// Replaces, at every accumulation boundary (train_online_pso_sdxl_turbo.py:858-861): accelerate's clip_grad_norm_ (one
// norm kernel per parameter + stack + norm + one scale per parameter), optimizer.step() (AdamW, :428-448) and
// optimizer.zero_grad(), plus this repo's own per-layer fp32 -> bf16 operand refresh.  Pure streaming work: 5 fp32 reads
// + 3 fp32 writes + one 16-bit write per parameter.
//
// Two update rules share the boundary (clip coefficient, overflow skip, bias corrections, device step counter, norm
// pieces, workspace reset; BoundaryParams, boundary_prologue / boundary_epilogue, begin_boundary on the host):
// flat_adamw_kernel (fp32 moments, torch.optim.AdamW) and flat_adamw8_kernel (bitsandbytes' blockwise 8-bit moments).
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

// ---- what both update rules share -------------------------------------------------------------------------------------
struct BoundaryParams {
  float lr, beta1, beta2, eps, weight_decay, max_norm, grad_scale, bc1, bc2_sqrt;  // bc*: host bias corrections of `step`
  float* found_inf;
  long long* step_dev;
  float* norm_out;
  double* ws;  // {sum of squares, ticket}
  double* parts;
  int n_parts;
  // device loss scaler (psob200_loss_scaler; amp_scale NULL = none): unscaled by in the prologue, updated in the epilogue
  float* amp_scale;
  int* amp_tracker;
  double amp_growth, amp_backoff;
  int amp_interval;
};

struct BoundaryScalars {
  float norm;
  bool skip;
  float coef, bc1, bc2_sqrt;
};

__device__ __forceinline__ BoundaryScalars boundary_prologue(const BoundaryParams& a) {
  // global-norm clip coefficient (accelerate / torch clip_grad_norm_: coef = min(1, max_norm / (norm + 1e-6)))
  double sumsq = a.ws[0];
  for (int r = 0; r < a.n_parts; ++r) sumsq += a.parts[r];  // per-rank slices of the fused exchange (same order on every rank)
  // unscale factor: with a device loss scaler torch's scale.double().reciprocal().float(), times grad_scale in fp32
  float grad_scale = a.grad_scale;
  if (a.amp_scale != nullptr) grad_scale = (float)(1.0 / (double)*a.amp_scale) * grad_scale;
  const float norm = (float)sqrt(sumsq) * grad_scale;
  // a non-finite norm (overflowed fp16 gradients, or a NaN anywhere: fminf would silently drop it) skips the whole update,
  // as GradScaler.step does; torch's clip_grad_norm_ would instead smear the NaN over every parameter
  const bool skip = !(norm <= 3.4028234e38f);
  const float coef = a.max_norm > 0.f ? fminf(1.f, a.max_norm / (norm + 1e-6f)) * grad_scale : grad_scale;
  float bc1 = a.bc1, bc2_sqrt = a.bc2_sqrt;
  if (a.step_dev != nullptr) {  // device-side step count: read by every thread before the last block advances it
    const double t = (double)(*a.step_dev + 1);
    bc1 = (float)(1.0 - pow((double)a.beta1, t));
    bc2_sqrt = (float)sqrt(1.0 - pow((double)a.beta2, t));
  }
  return {norm, skip, coef, bc1, bc2_sqrt};
}

// the last block to finish publishes the norm and leaves the workspace zeroed for the next boundary
__device__ __forceinline__ void boundary_epilogue(const BoundaryParams& a, float norm, bool skip) {
  __shared__ unsigned ticket;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    ticket = atomicAdd(reinterpret_cast<unsigned*>(a.ws + 1), 1u);
  }
  __syncthreads();
  if (ticket == gridDim.x - 1 && threadIdx.x == 0) {
    if (a.norm_out != nullptr) *a.norm_out = norm;
    if (a.found_inf != nullptr) *a.found_inf = skip ? 1.f : 0.f;
    if (a.step_dev != nullptr && !skip) *a.step_dev += 1;  // every block has read it: this is the last one to finish
    if (a.amp_scale != nullptr) {  // torch._amp_update_scale_ with found_inf = skip; read by every block, like step_dev
      const float s = *a.amp_scale;
      if (skip) {
        *a.amp_scale = (float)((double)s * a.amp_backoff);
        *a.amp_tracker = 0;
      } else if (*a.amp_tracker + 1 == a.amp_interval) {
        const float grown = (float)((double)s * a.amp_growth);
        if (isfinite(grown)) *a.amp_scale = grown;  // never grows past the fp32 range
        *a.amp_tracker = 0;
      } else {
        *a.amp_tracker += 1;
      }
    }
    a.ws[0] = 0.0;
    *reinterpret_cast<unsigned*>(a.ws + 1) = 0u;
    for (int r = 0; r < a.n_parts; ++r) a.parts[r] = 0.0;  // local copy only: peers zero theirs; next use is behind a barrier
  }
}

// ---- fp32 AdamW (torch.optim.AdamW) ------------------------------------------------------------------------------------
template <typename TO>
__global__ void __launch_bounds__(kOptThreads)
flat_adamw_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, TO* __restrict__ op,
                  long long n, BoundaryParams a) {
  const auto [norm, skip, coef, bc1, bc2_sqrt] = boundary_prologue(a);
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
  boundary_epilogue(a, norm, skip);
}

// ---- blockwise 8-bit AdamW (bitsandbytes, the Turbo recipe's `use_8bit_adam`, T:428-448) -------------------------------
// One update launch over every 8-bit block and every fp32-class range.  A group of block_size / 8 threads owns one block
// (256: one warp; 2048: one 256-thread CTA), 8 consecutive elements per thread: p and g as float4 pairs, 8 codes per moment
// as one 8-byte word.  The block's new absmax is a max over the bit patterns of |m| and |v| (non-negative floats order like
// unsigned integers).  The quantisation search runs over the 255 midpoints stored in breadth-first (Eytzinger) order: the
// 2^l candidates of probe l are adjacent words, so the lanes of a warp hit distinct banks where a sorted array would put
// every probe of one level in the same bank.
// Arithmetic is spelled with __f*_rn so that nvcc cannot contract it: the bitwise oracle (oracle/optim8bit.py) depends on it.
constexpr int kOpt8Threads = 256;

struct Adam8State {
  float* p;
  float* g;
  uint8_t* c1;
  uint8_t* c2;
  float* absmax1;
  float* absmax2;
  const float* map1;
  const float* map2;
  const long long* blocks8;  // {flat offset, length}
  long long n_blocks8;
  const long long* chunks32;  // {flat offset, length, compact offset}
  long long n_chunks32;
  float* m32;
  float* v32;
  long long n;
};

// in-order position k (0..254) of the perfect 255-node search tree -> its breadth-first slot (1..255)
__device__ __forceinline__ int eytzinger_slot(int k) {
  const int j = k + 1, tz = __ffs(j) - 1;
  return (1 << (7 - tz)) + (j >> (tz + 1));
}

// number of midpoints strictly below x (np.searchsorted(mid, x, "left"))
__device__ __forceinline__ int count_below(const float* tree, float x) {
  int i = 1;
#pragma unroll
  for (int l = 0; l < 8; ++l) i = 2 * i + (tree[i] < x ? 1 : 0);
  return i - 256;
}

// __grid_constant__: the fields are read from the parameter space where they are used; without it nvcc keeps every field of
// the two structs in registers for the whole kernel (5 more registers at GROUP 256, 16 more at GROUP 32)
template <int GROUP, typename TO>
__global__ void __launch_bounds__(kOpt8Threads)
flat_adamw8_kernel(const __grid_constant__ BoundaryParams h, const __grid_constant__ Adam8State a, TO* __restrict__ op) {
  constexpr int kUnits = kOpt8Threads / GROUP;  // blocks per CTA and iteration
  __shared__ float s_map1[256], s_map2[256], s_tree1[256], s_tree2[256];
  __shared__ unsigned s_red[2][kOpt8Threads / 32];
  if (a.n_blocks8 > 0) {
    for (int t = threadIdx.x; t < 256; t += kOpt8Threads) {
      s_map1[t] = a.map1[t];
      s_map2[t] = a.map2[t];
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 255; t += kOpt8Threads) {
      s_tree1[eytzinger_slot(t)] = __fmul_rn(__fadd_rn(s_map1[t], s_map1[t + 1]), 0.5f);
      s_tree2[eytzinger_slot(t)] = __fmul_rn(__fadd_rn(s_map2[t], s_map2[t + 1]), 0.5f);
    }
    __syncthreads();
  }
  const auto [norm, skip, coef, bc1, bc2] = boundary_prologue(h);
  const float step_size = __fdiv_rn(__fmul_rn(-h.lr, bc2), bc1);
  const float eps_bc2 = __fmul_rn(h.eps, bc2);
  const float omb1 = __fsub_rn(1.f, h.beta1), omb2 = __fsub_rn(1.f, h.beta2);
  const float decay = __fsub_rn(1.f, __fmul_rn(h.lr, h.weight_decay));

  const int grp = threadIdx.x / GROUP, lane = threadIdx.x % GROUP, i0 = lane * 8;
  const long long units = a.n_blocks8 + a.n_chunks32;
  for (long long base = (long long)blockIdx.x * kUnits; base < units; base += (long long)gridDim.x * kUnits) {
    const long long u = base + grp;
    const bool is8 = u < a.n_blocks8;
    long long off = 0, coff = 0;
    int len = 0;
    if (u < units) {
      if (is8) {
        off = a.blocks8[2 * u];
        len = (int)a.blocks8[2 * u + 1];
      } else {
        const long long* e = a.chunks32 + 3 * (u - a.n_blocks8);
        off = e[0];
        len = (int)e[1];
        coff = e[2];
      }
    }
    const int cnt = min(8, len - i0);  // elements of this thread (<= 0: none)
    const long long at = off + i0;
    const bool vec = cnt == 8 && (off & 7) == 0 && (coff & 7) == 0;
    if (skip) {  // gradient zeroed, everything else untouched
      for (int j = 0; j < 8; ++j)
        if (i0 < len && at + j < a.n) a.g[at + j] = 0.f;
      continue;
    }
    float pv[8], gv[8], mv[8], vv[8];
    unsigned char q1[8], q2[8];
    if (vec) {
      Vec8<float>::load(a.p + at, pv);
      Vec8<float>::load(a.g + at, gv);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        pv[j] = j < cnt ? a.p[at + j] : 0.f;
        gv[j] = j < cnt ? a.g[at + j] : 0.f;
      }
    }
    float am1 = 0.f, am2 = 0.f;
    if (is8) {
      if (u < units) {
        am1 = a.absmax1[u];
        am2 = a.absmax2[u];
      }
      if (vec) {
        const uint2 w1 = *reinterpret_cast<const uint2*>(a.c1 + at), w2 = *reinterpret_cast<const uint2*>(a.c2 + at);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          q1[j] = (unsigned char)(((j < 4 ? w1.x : w1.y) >> (8 * (j & 3))) & 0xffu);
          q2[j] = (unsigned char)(((j < 4 ? w2.x : w2.y) >> (8 * (j & 3))) & 0xffu);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          q1[j] = j < cnt ? a.c1[at + j] : (unsigned char)127;
          q2[j] = j < cnt ? a.c2[at + j] : (unsigned char)0;
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        mv[j] = j < cnt ? __fmul_rn(s_map1[q1[j]], am1) : 0.f;
        vv[j] = j < cnt ? __fmul_rn(s_map2[q2[j]], am2) : 0.f;
      }
    } else if (vec) {
      Vec8<float>::load(a.m32 + coff + i0, mv);
      Vec8<float>::load(a.v32 + coff + i0, vv);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        mv[j] = j < cnt ? a.m32[coff + i0 + j] : 0.f;
        vv[j] = j < cnt ? a.v32[coff + i0 + j] : 0.f;
      }
    }
    unsigned b1 = 0u, b2 = 0u;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float gj = __fmul_rn(gv[j], coef);
      mv[j] = __fadd_rn(__fmul_rn(mv[j], h.beta1), __fmul_rn(omb1, gj));
      vv[j] = __fadd_rn(__fmul_rn(vv[j], h.beta2), __fmul_rn(__fmul_rn(omb2, gj), gj));
      float pj = __fadd_rn(pv[j], __fmul_rn(step_size, __fdiv_rn(mv[j], __fadd_rn(__fsqrt_rn(vv[j]), eps_bc2))));
      if (h.weight_decay > 0.f) pj = __fmul_rn(pj, decay);  // bitsandbytes decays after the step (torch: before)
      pv[j] = pj;
      if (j < cnt) {
        b1 = max(b1, __float_as_uint(fabsf(mv[j])));
        b2 = max(b2, __float_as_uint(fabsf(vv[j])));
      }
    }
    if (is8) {
      b1 = __reduce_max_sync(0xffffffffu, b1);
      b2 = __reduce_max_sync(0xffffffffu, b2);
      if constexpr (GROUP > 32) {
        const int warp = threadIdx.x >> 5;
        if ((threadIdx.x & 31) == 0) {
          s_red[0][warp] = b1;
          s_red[1][warp] = b2;
        }
        __syncthreads();
#pragma unroll
        for (int w = 0; w < GROUP / 32; ++w) {
          b1 = max(b1, s_red[0][w]);
          b2 = max(b2, s_red[1][w]);
        }
        __syncthreads();  // s_red is reused by the next iteration
      }
      const float a1 = __uint_as_float(b1), a2 = __uint_as_float(b2);
      if (lane == 0 && u < units) {
        a.absmax1[u] = a1;
        a.absmax2[u] = a2;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        int c = count_below(s_tree1, a1 > 0.f ? __fdiv_rn(mv[j], a1) : 0.f);
        if (signbit(s_map1[c]) != signbit(mv[j])) c += mv[j] > 0.f ? 1 : -1;  // the momentum never flips sign
        q1[j] = (unsigned char)c;
        q2[j] = (unsigned char)count_below(s_tree2, a2 > 0.f ? __fdiv_rn(vv[j], a2) : 0.f);
      }
      if (vec) {
        uint2 w1 = make_uint2(0u, 0u), w2 = make_uint2(0u, 0u);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          (j < 4 ? w1.x : w1.y) |= (unsigned)q1[j] << (8 * (j & 3));
          (j < 4 ? w2.x : w2.y) |= (unsigned)q2[j] << (8 * (j & 3));
        }
        *reinterpret_cast<uint2*>(a.c1 + at) = w1;
        *reinterpret_cast<uint2*>(a.c2 + at) = w2;
      } else {
        for (int j = 0; j < cnt; ++j) {
          a.c1[at + j] = q1[j];
          a.c2[at + j] = q2[j];
        }
      }
    } else if (vec) {
      Vec8<float>::store(a.m32 + coff + i0, mv);
      Vec8<float>::store(a.v32 + coff + i0, vv);
    } else {
      for (int j = 0; j < cnt; ++j) {
        a.m32[coff + i0 + j] = mv[j];
        a.v32[coff + i0 + j] = vv[j];
      }
    }
    if (vec) {
      const float zero[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      Vec8<float>::store(a.p + at, pv);
      Vec8<float>::store(a.g + at, zero);  // optimizer.zero_grad()
      if (op != nullptr) Vec8<TO>::store(op + at, pv);
    } else if (i0 < len) {
      for (int j = 0; j < 8; ++j) {
        if (j < cnt) {
          a.p[at + j] = pv[j];
          if (op != nullptr) Vec8<TO>::store1(op + at + j, pv[j]);
        }
        if (at + j < a.n) a.g[at + j] = 0.f;  // also the flat layout's padding behind a short tail
      }
    }
  }
  boundary_epilogue(h, norm, skip);
}

// ---- host side shared by both entry points (their args structs name the shared fields alike) ---------------------------
// Validates the shared fields, in the order invalid argument, shape, dtype, alignment, after the entry's own checks
// `args_ok` (null pointers, tables), `shape_ok` and `aligned` (its 16-byte aligned pointers); launches flat_sumsq_kernel
// when the norm is needed and was not supplied (always with a loss scaler `sc`, already validated: the norm is its overflow
// check); fills `b`.  Returns the SM count for the grid clamp, or an error code (< 0).
template <typename Args>
int begin_boundary(const Args& o, const psob200_loss_scaler* sc, bool args_ok, bool shape_ok, bool aligned, cudaStream_t st,
                   BoundaryParams& b) {
  if (!args_ok || !o.param || !o.grad || !o.workspace || o.n <= 0 || (o.step <= 0 && !o.step_dev))
    return PSOB200_ERR_INVALID_ARG;
  if (o.n_sumsq_parts < 0 || (o.n_sumsq_parts > 0 && !o.sumsq_parts)) return PSOB200_ERR_INVALID_ARG;
  if (!shape_ok) return PSOB200_ERR_SHAPE;
  if (o.operand && o.operand_dtype != PSOB200_BF16 && o.operand_dtype != PSOB200_F16) return PSOB200_ERR_DTYPE;
  if (!aligned) return PSOB200_ERR_ALIGNMENT;
  const int n_sm = sm_count();
  double* ws = reinterpret_cast<double*>(o.workspace);
  if (o.n_sumsq_parts == 0 && (o.max_grad_norm > 0.f || o.norm_out != nullptr || sc != nullptr)) {
    long long blocks = (o.n + kOptThreads * 4 - 1) / (kOptThreads * 4);
    if (blocks > n_sm * 8) blocks = n_sm * 8;
    flat_sumsq_kernel<<<(unsigned)blocks, kOptThreads, 0, st>>>(o.grad, o.n, ws);
    const int rc = consume_launch_error("launch flat_sumsq_kernel", cudaSuccess);
    if (rc != PSOB200_OK) return rc;
  }
  b.lr = o.lr; b.beta1 = o.beta1; b.beta2 = o.beta2; b.eps = o.eps; b.weight_decay = o.weight_decay;
  b.max_norm = o.max_grad_norm; b.grad_scale = o.grad_scale;
  b.bc1 = (float)(1.0 - std::pow((double)o.beta1, (double)o.step));
  b.bc2_sqrt = (float)std::sqrt(1.0 - std::pow((double)o.beta2, (double)o.step));
  b.found_inf = o.found_inf; b.step_dev = o.step_dev; b.norm_out = o.norm_out;
  b.ws = ws; b.parts = o.sumsq_parts; b.n_parts = o.n_sumsq_parts;
  b.amp_scale = sc ? sc->scale : nullptr;
  b.amp_tracker = sc ? sc->growth_tracker : nullptr;
  b.amp_growth = sc ? sc->growth_factor : 1.0;
  b.amp_backoff = sc ? sc->backoff_factor : 1.0;
  b.amp_interval = sc ? sc->growth_interval : 0;
  return n_sm;
}

// the optimizer entry points' checks of a loss scaler: both state pointers, a growth that grows, a backoff that shrinks and
// stays positive, a reachable interval
inline bool scaler_ok(const psob200_loss_scaler* sc) {
  return sc != nullptr && sc->scale != nullptr && sc->growth_tracker != nullptr && sc->growth_interval > 0 &&
         sc->growth_factor > 1.0 && sc->backoff_factor > 0.0 && sc->backoff_factor < 1.0;
}

// calls f(TO{}) with the element type of the 16-bit operand copy (bf16 when there is none)
template <typename F>
void dispatch_operand(const void* operand, int32_t operand_dtype, F&& f) {
  if (operand == nullptr || operand_dtype == PSOB200_BF16)
    f(__nv_bfloat16{});
  else
    f(__half{});
}

}  // namespace psob200

using namespace psob200;

// sc: a validated loss scaler, or NULL (the unscaled entry points)
static int flat_adamw_step(const psob200_flat_adamw_args* args, const psob200_loss_scaler* sc, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_flat_adamw_args& o = *args;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  BoundaryParams b;
  const int n_sm = begin_boundary(o, sc, o.exp_avg && o.exp_avg_sq, true, aligned16(o.grad) && aligned16(o.workspace), st, b);
  if (n_sm < 0) return n_sm;
  long long blocks = (o.n + kOptThreads - 1) / kOptThreads;
  if (blocks > n_sm * 8) blocks = n_sm * 8;
  dispatch_operand(o.operand, o.operand_dtype, [&](auto t) {
    using TO = decltype(t);
    flat_adamw_kernel<TO><<<(unsigned)blocks, kOptThreads, 0, st>>>(o.param, o.grad, o.exp_avg, o.exp_avg_sq,
                                                                     reinterpret_cast<TO*>(o.operand), o.n, b);
  });
  return consume_launch_error("launch flat_adamw_kernel", cudaSuccess);
}

extern "C" int psob200_flat_adamw_step(const psob200_flat_adamw_args* args, void* stream) {
  return flat_adamw_step(args, nullptr, stream);
}

extern "C" int psob200_flat_adamw_step_scaled(const psob200_flat_adamw_args* args, const psob200_loss_scaler* scaler,
                                              void* stream) {
  if (!scaler_ok(scaler)) return PSOB200_ERR_INVALID_ARG;
  return flat_adamw_step(args, scaler, stream);
}

static int flat_adamw8_step(const psob200_flat_adamw8_args* args, const psob200_loss_scaler* sc, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_flat_adamw8_args& o = *args;
  const bool args_ok =
      o.n_blocks8 >= 0 && o.n_chunks32 >= 0 && o.n_blocks8 + o.n_chunks32 > 0 &&
      (o.n_blocks8 == 0 || (o.blocks8 && o.code1 && o.code2 && o.absmax1 && o.absmax2 && o.map1 && o.map2)) &&
      (o.n_chunks32 == 0 || (o.chunks32 && o.exp_avg32 && o.exp_avg_sq32));
  bool aligned = true;
  for (const void* p : {(const void*)o.param, (const void*)o.grad, (const void*)o.workspace, (const void*)o.operand,
                        (const void*)o.code1, (const void*)o.code2, (const void*)o.exp_avg32, (const void*)o.exp_avg_sq32})
    aligned = aligned && aligned16(p);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  BoundaryParams b;
  const int n_sm = begin_boundary(o, sc, args_ok, o.block_size == 256 || o.block_size == 2048, aligned, st, b);
  if (n_sm < 0) return n_sm;
  Adam8State a;
  a.p = o.param; a.g = o.grad; a.c1 = o.code1; a.c2 = o.code2; a.absmax1 = o.absmax1; a.absmax2 = o.absmax2;
  a.map1 = o.map1; a.map2 = o.map2;
  a.blocks8 = reinterpret_cast<const long long*>(o.blocks8); a.n_blocks8 = o.n_blocks8;
  a.chunks32 = reinterpret_cast<const long long*>(o.chunks32); a.n_chunks32 = o.n_chunks32;
  a.m32 = o.exp_avg32; a.v32 = o.exp_avg_sq32; a.n = o.n;
  const int group = o.block_size / 8, units_per_cta = kOpt8Threads / group;
  long long grid = (o.n_blocks8 + o.n_chunks32 + units_per_cta - 1) / units_per_cta;
  if (grid > n_sm * 8) grid = n_sm * 8;
  dispatch_operand(o.operand, o.operand_dtype, [&](auto t) {
    using TO = decltype(t);
    TO* op = reinterpret_cast<TO*>(o.operand);
    if (group == 32)
      flat_adamw8_kernel<32, TO><<<(unsigned)grid, kOpt8Threads, 0, st>>>(b, a, op);
    else
      flat_adamw8_kernel<256, TO><<<(unsigned)grid, kOpt8Threads, 0, st>>>(b, a, op);
  });
  return consume_launch_error("launch flat_adamw8_kernel", cudaSuccess);
}

extern "C" int psob200_flat_adamw8_step(const psob200_flat_adamw8_args* args, void* stream) {
  return flat_adamw8_step(args, nullptr, stream);
}

extern "C" int psob200_flat_adamw8_step_scaled(const psob200_flat_adamw8_args* args, const psob200_loss_scaler* scaler,
                                               void* stream) {
  if (!scaler_ok(scaler)) return PSOB200_ERR_INVALID_ARG;
  return flat_adamw8_step(args, scaler, stream);
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
  const int n_sm = sm_count();
  long long blocks = (hi - lo + kOptThreads * 4 - 1) / (kOptThreads * 4);
  if (blocks > n_sm * 4) blocks = n_sm * 4;
  if (blocks < 1) blocks = 1;  // an empty slice still launches: uniform launch sequence on every rank
  flat_allreduce_sumsq_kernel<<<(unsigned)blocks, kOptThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      o.grad_multicast, o.sumsq_multicast + o.rank, lo, hi, o.scale);
  return consume_launch_error("launch flat_allreduce_sumsq_kernel", cudaSuccess);
}
