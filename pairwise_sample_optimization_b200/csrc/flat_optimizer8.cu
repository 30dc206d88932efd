// Optimizer boundary with bitsandbytes' blockwise 8-bit AdamW state (the Turbo recipe's `use_8bit_adam`, T:428-448):
// clip + unscale + overflow skip + 8-bit AdamW + zero_grad + refresh of the 16-bit operand copies, in one update launch over
// every 8-bit block and every fp32-class range (plus flat_sumsq_kernel when the norm is not supplied).
//
// A group of block_size / 8 threads owns one block (256: one warp; 2048: one 256-thread CTA), 8 consecutive elements per
// thread: p and g as float4 pairs, 8 codes per moment as one 8-byte word.  The block's new absmax is a max over the bit
// patterns of |m| and |v| (non-negative floats order like unsigned integers).  The quantisation search runs over the 255
// midpoints stored in breadth-first (Eytzinger) order: the 2^l candidates of probe l are adjacent words, so the lanes of a
// warp hit distinct banks where a sorted array would put every probe of one level in the same bank.
// Arithmetic is spelled with __f*_rn so that nvcc cannot contract it: the bitwise oracle (oracle/optim8bit.py) depends on it.
#include <atomic>
#include <cmath>

#include "common.cuh"

namespace psob200 {

constexpr int kOpt8Threads = 256;

struct Adam8Params {
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
  float lr, beta1, beta2, eps, weight_decay, max_norm, grad_scale, bc1, bc2;
  float* found_inf;
  long long* step_dev;
  float* norm_out;
  double* ws;
  double* parts;
  int n_parts;
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

template <int GROUP, typename TO>
__global__ void __launch_bounds__(kOpt8Threads) flat_adamw8_kernel(Adam8Params a, TO* __restrict__ op) {
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
  // clip coefficient, overflow skip and bias corrections exactly as flat_adamw_kernel
  double sumsq = a.ws[0];
  for (int r = 0; r < a.n_parts; ++r) sumsq += a.parts[r];
  const float norm = (float)sqrt(sumsq) * a.grad_scale;
  const bool skip = !(norm <= 3.4028234e38f);
  const float coef = a.max_norm > 0.f ? fminf(1.f, a.max_norm / (norm + 1e-6f)) * a.grad_scale : a.grad_scale;
  float bc1 = a.bc1, bc2 = a.bc2;
  if (a.step_dev != nullptr) {
    const double t = (double)(*a.step_dev + 1);
    bc1 = (float)(1.0 - pow((double)a.beta1, t));
    bc2 = (float)sqrt(1.0 - pow((double)a.beta2, t));
  }
  const float step_size = __fdiv_rn(__fmul_rn(-a.lr, bc2), bc1);
  const float eps_bc2 = __fmul_rn(a.eps, bc2);
  const float omb1 = __fsub_rn(1.f, a.beta1), omb2 = __fsub_rn(1.f, a.beta2);
  const float decay = __fsub_rn(1.f, __fmul_rn(a.lr, a.weight_decay));

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
      mv[j] = __fadd_rn(__fmul_rn(mv[j], a.beta1), __fmul_rn(omb1, gj));
      vv[j] = __fadd_rn(__fmul_rn(vv[j], a.beta2), __fmul_rn(__fmul_rn(omb2, gj), gj));
      float pj = __fadd_rn(pv[j], __fmul_rn(step_size, __fdiv_rn(mv[j], __fadd_rn(__fsqrt_rn(vv[j]), eps_bc2))));
      if (a.weight_decay > 0.f) pj = __fmul_rn(pj, decay);  // bitsandbytes decays after the step (torch: before)
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
  // the last CTA to finish publishes the norm and leaves the workspace zeroed (as flat_adamw_kernel)
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
    if (a.step_dev != nullptr && !skip) *a.step_dev += 1;
    a.ws[0] = 0.0;
    *reinterpret_cast<unsigned*>(a.ws + 1) = 0u;
    for (int r = 0; r < a.n_parts; ++r) a.parts[r] = 0.0;
  }
}

template <int GROUP>
cudaError_t launch_adamw8(const Adam8Params& a, void* operand, int32_t operand_dtype, unsigned grid, cudaStream_t st) {
  if (operand == nullptr || operand_dtype == PSOB200_BF16)
    flat_adamw8_kernel<GROUP, __nv_bfloat16><<<grid, kOpt8Threads, 0, st>>>(a, reinterpret_cast<__nv_bfloat16*>(operand));
  else
    flat_adamw8_kernel<GROUP, __half><<<grid, kOpt8Threads, 0, st>>>(a, reinterpret_cast<__half*>(operand));
  return cudaSuccess;
}

}  // namespace psob200

using namespace psob200;

extern "C" int psob200_flat_adamw8_step(const psob200_flat_adamw8_args* args, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_flat_adamw8_args& o = *args;
  if (!o.param || !o.grad || !o.workspace || o.n <= 0 || (o.step <= 0 && !o.step_dev)) return PSOB200_ERR_INVALID_ARG;
  if (o.n_blocks8 < 0 || o.n_chunks32 < 0 || o.n_blocks8 + o.n_chunks32 == 0) return PSOB200_ERR_INVALID_ARG;
  if (o.n_blocks8 > 0 && (!o.blocks8 || !o.code1 || !o.code2 || !o.absmax1 || !o.absmax2 || !o.map1 || !o.map2))
    return PSOB200_ERR_INVALID_ARG;
  if (o.n_chunks32 > 0 && (!o.chunks32 || !o.exp_avg32 || !o.exp_avg_sq32)) return PSOB200_ERR_INVALID_ARG;
  if (o.n_sumsq_parts < 0 || (o.n_sumsq_parts > 0 && !o.sumsq_parts)) return PSOB200_ERR_INVALID_ARG;
  if (o.block_size != 256 && o.block_size != 2048) return PSOB200_ERR_SHAPE;
  if (o.operand && o.operand_dtype != PSOB200_BF16 && o.operand_dtype != PSOB200_F16) return PSOB200_ERR_DTYPE;
  for (const void* p : {(const void*)o.param, (const void*)o.grad, (const void*)o.workspace, (const void*)o.operand,
                        (const void*)o.code1, (const void*)o.code2, (const void*)o.exp_avg32, (const void*)o.exp_avg_sq32})
    if (!aligned16(p)) return PSOB200_ERR_ALIGNMENT;
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
  if (o.n_sumsq_parts == 0 && (o.max_grad_norm > 0.f || o.norm_out != nullptr)) {
    const int rc = launch_flat_sumsq(o.grad, o.n, ws, n_sm, st);
    if (rc != PSOB200_OK) return rc;
  }
  Adam8Params a;
  a.p = o.param; a.g = o.grad; a.c1 = o.code1; a.c2 = o.code2; a.absmax1 = o.absmax1; a.absmax2 = o.absmax2;
  a.map1 = o.map1; a.map2 = o.map2;
  a.blocks8 = reinterpret_cast<const long long*>(o.blocks8); a.n_blocks8 = o.n_blocks8;
  a.chunks32 = reinterpret_cast<const long long*>(o.chunks32); a.n_chunks32 = o.n_chunks32;
  a.m32 = o.exp_avg32; a.v32 = o.exp_avg_sq32; a.n = o.n;
  a.lr = o.lr; a.beta1 = o.beta1; a.beta2 = o.beta2; a.eps = o.eps; a.weight_decay = o.weight_decay;
  a.max_norm = o.max_grad_norm; a.grad_scale = o.grad_scale;
  a.bc1 = (float)(1.0 - std::pow((double)o.beta1, (double)o.step));
  a.bc2 = (float)std::sqrt(1.0 - std::pow((double)o.beta2, (double)o.step));
  a.found_inf = o.found_inf; a.step_dev = o.step_dev; a.norm_out = o.norm_out;
  a.ws = ws; a.parts = o.sumsq_parts; a.n_parts = o.n_sumsq_parts;
  const int group = o.block_size / 8, units_per_cta = kOpt8Threads / group;
  long long grid = (o.n_blocks8 + o.n_chunks32 + units_per_cta - 1) / units_per_cta;
  if (grid > n_sm * 8) grid = n_sm * 8;
  if (group == 32)
    launch_adamw8<32>(a, o.operand, o.operand_dtype, (unsigned)grid, st);
  else
    launch_adamw8<256>(a, o.operand, o.operand_dtype, (unsigned)grid, st);
  return consume_launch_error("launch flat_adamw8_kernel", cudaSuccess);
}
