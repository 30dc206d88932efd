// LayerNorm over the last dimension and GroupNorm over contiguous NCHW (optionally + SiLU and a per-(sample, channel) add
// before normalising), forward and backward.
//
// Replace torch.nn.LayerNorm / torch.nn.GroupNorm and the `F.silu(norm(x))` lines of diffusers==0.27.0
// `ResnetBlock2D.forward` (`h = nonlinearity(norm1(x))`; `h = nonlinearity(norm2(h + time_emb_proj(temb)[:, :, None, None]))`).
// Not rows of SURVEY.md section 8: the stock norm + SiLU kernels were 15 % of the measured dmd128 micro-step's kernel time
// (profiles/r02_bench_launches_dmd128.csv).  Pure streaming work: a few flops per element, one or two reductions per row
// or group.
//
// Arithmetic in fp32, one rounding per output element.  Variance without cancellation: LayerNorm is centred two-pass over
// the row held in registers; GroupNorm merges per-item (count, mean, M2) triples with Chan's parallel formula.  Every
// reduction has a fixed order (shuffle trees, fixed partitions, no floating-point atomics): results are bitwise
// reproducible, and the partition depends on the shape only, not on the device.
#include <algorithm>
#include <atomic>
#include <type_traits>

#include "common.cuh"

namespace psob200 {

constexpr int kNormThreads = 256;
constexpr int kNormWarps = kNormThreads / 32;
constexpr int kLnMaxC = 2048;           // 8 chunks of 8 per lane
constexpr long long kGnChunk = 8192;    // elements per CTA and group part: 256 threads x 4 items of 8

__device__ __forceinline__ float load_param(const void* p, int32_t dt, long long i) {
  if (dt == PSOB200_F32) return __ldg(reinterpret_cast<const float*>(p) + i);
  if (dt == PSOB200_BF16) return __bfloat162float(__ldg(reinterpret_cast<const __nv_bfloat16*>(p) + i));
  return __half2float(__ldg(reinterpret_cast<const __half*>(p) + i));
}

template <typename T>
__device__ __forceinline__ float round_to(float v) {
  if constexpr (std::is_same_v<T, __nv_bfloat16>) return __bfloat162float(__float2bfloat16_rn(v));
  else if constexpr (std::is_same_v<T, __half>) return __half2float(__float2half_rn(v));
  else return v;
}

// x / (1 + exp(-x)).  fp32 output: accurate exp and division (fp32 north star 1e-5); 16-bit output: the fast forms, whose
// error is far below a 16-bit ulp.
template <bool kPrecise>
__device__ __forceinline__ float sigmoidf(float z) {
  if constexpr (kPrecise) return 1.f / (1.f + expf(-z));
  else return __fdividef(1.f, 1.f + __expf(-z));
}

// kW = 8: one Vec8 item; kW = 1: one element (spans whose channel length H*W is not a multiple of 8)
template <typename T, int kW>
__device__ __forceinline__ void load_item(const T* p, float (&v)[kW]) {
  if constexpr (kW == 8) Vec8<T>::load(p, v);
  else v[0] = Vec8<T>::load1(p);
}

template <typename T, int kW>
__device__ __forceinline__ void store_item(T* p, const float (&v)[kW]) {
  if constexpr (kW == 8) Vec8<T>::store(p, v);
  else Vec8<T>::store1(p, v[0]);
}

// ---------------------------------------------------------------------------------------------------------------- LayerNorm
// One warp per row, the row in registers (lane l owns chunks l, l + 32, ... of 8 elements); weight and bias cached as fp32
// in shared memory once per CTA (the grid is one wave, so a CTA normalises many rows).
template <typename TI, typename TO, int kV>
__global__ void __launch_bounds__(kNormThreads)
layer_norm_fwd_kernel(const psob200_layer_norm_args a) {
  __shared__ __align__(16) float sw[kLnMaxC], sb[kLnMaxC];
  const int C = (int)a.C, nvec = C / 8, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < C; i += kNormThreads) {
    sw[i] = a.weight ? load_param(a.weight, a.param_dtype, i) : 1.f;
    sb[i] = a.bias ? load_param(a.bias, a.param_dtype, i) : 0.f;
  }
  __syncthreads();
  const float inv_c = 1.f / (float)C;
  for (long long row = (long long)blockIdx.x * kNormWarps + threadIdx.x / 32; row < a.rows;
       row += (long long)gridDim.x * kNormWarps) {
    const TI* x = reinterpret_cast<const TI*>(a.x) + row * a.ld_x;
    float v[kV][8];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kV; ++k) {
      const int j = lane + 32 * k;
      if (j < nvec) {
        Vec8<TI>::load(x + 8 * j, v[k]);
#pragma unroll
        for (int e = 0; e < 8; ++e) s += v[k][e];
      }
    }
    const float mean = warp_sum(s) * inv_c;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < kV; ++k) {
      if (lane + 32 * k < nvec) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float d = v[k][e] - mean;
          q = fmaf(d, d, q);
        }
      }
    }
    const float rstd = rsqrtf(warp_sum(q) * inv_c + a.eps);
    TO* y = reinterpret_cast<TO*>(a.y) + row * a.ld_y;
#pragma unroll
    for (int k = 0; k < kV; ++k) {
      const int j = lane + 32 * k;
      if (j < nvec) {
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = fmaf((v[k][e] - mean) * rstd, sw[8 * j + e], sb[8 * j + e]);
        Vec8<TO>::store(y + 8 * j, o);
      }
    }
    if (lane == 0) {
      a.mean[row] = mean;
      a.rstd[row] = rstd;
    }
  }
}

// dx = rstd (g - mean(g) - xhat mean(g xhat)),  g = dy w,  xhat = (x - mean) rstd.  x and dy stay in registers in their
// storage format and are decoded in both passes: half the registers of decoded fp32 rows, so twice the rows in flight
// (decoded, the 640-wide backward ran at 2 CTAs per SM and lost to the stock kernel).
template <typename TI, typename TO, int kV>
__global__ void __launch_bounds__(kNormThreads)
layer_norm_bwd_kernel(const psob200_layer_norm_args a) {
  __shared__ __align__(16) float sw[kLnMaxC];
  const int C = (int)a.C, nvec = C / 8, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < C; i += kNormThreads) sw[i] = a.weight ? load_param(a.weight, a.param_dtype, i) : 1.f;
  __syncthreads();
  const float inv_c = 1.f / (float)C;
  for (long long row = (long long)blockIdx.x * kNormWarps + threadIdx.x / 32; row < a.rows;
       row += (long long)gridDim.x * kNormWarps) {
    const TI* x = reinterpret_cast<const TI*>(a.x) + row * a.ld_x;
    const TO* dy = reinterpret_cast<const TO*>(a.dy) + row * a.ld_dy;
    const float mean = __ldg(a.mean + row), rstd = __ldg(a.rstd + row);
    typename Vec8<TI>::Raw rx[kV];
    typename Vec8<TO>::Raw rd[kV];
#pragma unroll
    for (int k = 0; k < kV; ++k) {
      const int j = lane + 32 * k;
      if (j < nvec) {
        rx[k] = Vec8<TI>::load_raw(x + 8 * j);
        rd[k] = Vec8<TO>::load_raw(dy + 8 * j);
      }
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < kV; ++k) {
      const int j = lane + 32 * k;
      if (j < nvec) {
        float xh[8], g[8];
        Vec8<TI>::decode(rx[k], xh);
        Vec8<TO>::decode(rd[k], g);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float gv = g[e] * sw[8 * j + e];
          s1 += gv;
          s2 = fmaf(gv, (xh[e] - mean) * rstd, s2);
        }
      }
    }
    const float c1 = warp_sum(s1) * inv_c, c2 = warp_sum(s2) * inv_c;
    TI* dx = reinterpret_cast<TI*>(a.dx) + row * a.ld_dx;
#pragma unroll
    for (int k = 0; k < kV; ++k) {
      const int j = lane + 32 * k;
      if (j < nvec) {
        float xh[8], g[8], o[8];
        Vec8<TI>::decode(rx[k], xh);
        Vec8<TO>::decode(rd[k], g);
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = rstd * (g[e] * sw[8 * j + e] - c1 - (xh[e] - mean) * rstd * c2);
        Vec8<TI>::store(dx + 8 * j, o);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------- GroupNorm
// Group gi = n G + g is the contiguous span [gi S, (gi + 1) S), S = (C / G) H W.  It is cut into P = ceil(S / kGnChunk)
// parts; CTA b handles part b % P of group b / P.  Two launches each way:
//   forward:  stats (per part: count, mean, M2 -> workspace)  |  apply (combine the P parts in order, normalise the part)
//   backward: sums  (per part: sum g, sum g xhat -> workspace) |  apply (combine in order, dx for the part)
// Every CTA of a group combines the same P partials in the same order, so all of them use bit-identical statistics.
struct Moments {
  float n, mean, m2;
};

// Chan et al.'s pairwise update: (n, mean, M2) of the union of two disjoint sets
__device__ __forceinline__ void merge(Moments& a, float nb, float mb, float m2b) {
  if (nb == 0.f) return;
  const float n = a.n + nb, d = mb - a.mean, f = nb / n;
  a.mean = fmaf(d, f, a.mean);
  a.m2 = a.m2 + m2b + d * d * a.n * f;
  a.n = n;
}

__device__ __forceinline__ void warp_merge(Moments& m) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float nb = __shfl_down_sync(0xffffffffu, m.n, o), mb = __shfl_down_sync(0xffffffffu, m.mean, o),
                m2b = __shfl_down_sync(0xffffffffu, m.m2, o);
    merge(m, nb, mb, m2b);
  }
}

__device__ __forceinline__ float warp_sum_down(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

struct GnShape {
  long long S, HW, Cg, P;
  int G;
};

__host__ __device__ inline long long gn_parts(long long S) { return (S + kGnChunk - 1) / kGnChunk; }

// x with the per-(sample, channel) term added and rounded to the input type, as the stock `h + temb` produces it
template <typename TI, int kW>
__device__ __forceinline__ void load_x(const psob200_group_norm_args& a, const GnShape& s, long long gi, long long e,
                                       int& c, float (&v)[kW]) {
  const TI* x = reinterpret_cast<const TI*>(a.x) + gi * s.S;
  load_item<TI, kW>(x + e, v);
  c = (int)((gi % s.G) * s.Cg + e / s.HW);
  if (a.channel_add) {
    const float t = Vec8<TI>::load1(reinterpret_cast<const TI*>(a.channel_add) + (gi / s.G) * a.C + c);
#pragma unroll
    for (int i = 0; i < kW; ++i) v[i] = round_to<TI>(v[i] + t);
  }
}

template <typename TI, int kW>
__global__ void __launch_bounds__(kNormThreads)
group_norm_stats_kernel(const psob200_group_norm_args a, const GnShape s) {
  const long long gi = blockIdx.x / s.P, part = blockIdx.x % s.P;
  const long long end = min(s.S, (part + 1) * kGnChunk);
  Moments m{0.f, 0.f, 0.f};
  for (long long e = part * kGnChunk + (long long)threadIdx.x * kW; e < end; e += kNormThreads * kW) {
    float v[kW];
    int c;
    load_x<TI, kW>(a, s, gi, e, c, v);
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < kW; ++i) sum += v[i];
    const float mb = sum * (1.f / kW);
    float m2b = 0.f;
#pragma unroll
    for (int i = 0; i < kW; ++i) m2b = fmaf(v[i] - mb, v[i] - mb, m2b);
    merge(m, (float)kW, mb, m2b);
  }
  __shared__ Moments sm[kNormWarps];
  warp_merge(m);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x / 32] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    Moments t = sm[0];
    for (int w = 1; w < kNormWarps; ++w) merge(t, sm[w].n, sm[w].mean, sm[w].m2);
    reinterpret_cast<float2*>(a.workspace)[blockIdx.x] = make_float2(t.mean, t.m2);
  }
}

// warp 0 combines the P parts of group gi in a fixed order; the result goes to shared memory
__device__ __forceinline__ void gn_group_moments(const psob200_group_norm_args& a, const GnShape& s, long long gi,
                                                 float& mean, float& rstd) {
  __shared__ float st[2];
  if (threadIdx.x < 32) {
    Moments m{0.f, 0.f, 0.f};
    const float2* ws = reinterpret_cast<const float2*>(a.workspace) + gi * s.P;
    for (long long p = threadIdx.x; p < s.P; p += 32) {
      const float2 q = ws[p];
      merge(m, (float)min(kGnChunk, s.S - p * kGnChunk), q.x, q.y);
    }
    warp_merge(m);
    if (threadIdx.x == 0) {
      st[0] = m.mean;
      st[1] = rsqrtf(m.m2 / (float)s.S + a.eps);
    }
  }
  __syncthreads();
  mean = st[0];
  rstd = st[1];
}

template <typename TI, typename TO, int kW>
__global__ void __launch_bounds__(kNormThreads)
group_norm_apply_kernel(const psob200_group_norm_args a, const GnShape s) {
  constexpr bool kPrecise = sizeof(TO) == 4;
  const long long gi = blockIdx.x / s.P, part = blockIdx.x % s.P;
  float mean, rstd;
  gn_group_moments(a, s, gi, mean, rstd);
  if (part == 0 && threadIdx.x == 0) {
    a.mean[gi] = mean;
    a.rstd[gi] = rstd;
  }
  const long long end = min(s.S, (part + 1) * kGnChunk);
  TO* y = reinterpret_cast<TO*>(a.y) + gi * s.S;
  for (long long e = part * kGnChunk + (long long)threadIdx.x * kW; e < end; e += kNormThreads * kW) {
    float v[kW];
    int c;
    load_x<TI, kW>(a, s, gi, e, c, v);
    const float w = a.weight ? load_param(a.weight, a.param_dtype, c) : 1.f;
    const float b = a.bias ? load_param(a.bias, a.param_dtype, c) : 0.f;
    const float sc = rstd * w;
#pragma unroll
    for (int i = 0; i < kW; ++i) {
      const float z = fmaf(v[i] - mean, sc, b);
      v[i] = a.silu ? z * sigmoidf<kPrecise>(z) : z;
    }
    store_item<TO, kW>(y + e, v);
  }
}

// g = dy w (dy times silu'(z) first when fused, z recomputed from x, mean, rstd and the affine);  xhat = (x - mean) rstd
template <typename TI, typename TO, int kW>
__device__ __forceinline__ void gn_grad_item(const psob200_group_norm_args& a, const GnShape& s, long long gi, long long e,
                                             float mean, float rstd, float (&xh)[kW], float (&g)[kW]) {
  constexpr bool kPrecise = sizeof(TO) == 4;
  int c;
  load_x<TI, kW>(a, s, gi, e, c, xh);
  load_item<TO, kW>(reinterpret_cast<const TO*>(a.dy) + gi * s.S + e, g);
  const float w = a.weight ? load_param(a.weight, a.param_dtype, c) : 1.f;
  const float b = a.bias ? load_param(a.bias, a.param_dtype, c) : 0.f;
#pragma unroll
  for (int i = 0; i < kW; ++i) {
    xh[i] = (xh[i] - mean) * rstd;
    if (a.silu) {
      const float z = fmaf(xh[i], w, b), sg = sigmoidf<kPrecise>(z);
      g[i] *= sg * fmaf(z, 1.f - sg, 1.f);  // silu'(z) = sigmoid(z) (1 + z (1 - sigmoid(z)))
    }
    g[i] *= w;
  }
}

template <typename TI, typename TO, int kW>
__global__ void __launch_bounds__(kNormThreads)
group_norm_bwd_sums_kernel(const psob200_group_norm_args a, const GnShape s) {
  const long long gi = blockIdx.x / s.P, part = blockIdx.x % s.P;
  const float mean = __ldg(a.mean + gi), rstd = __ldg(a.rstd + gi);
  const long long end = min(s.S, (part + 1) * kGnChunk);
  float s1 = 0.f, s2 = 0.f;
  for (long long e = part * kGnChunk + (long long)threadIdx.x * kW; e < end; e += kNormThreads * kW) {
    float xh[kW], g[kW];
    gn_grad_item<TI, TO, kW>(a, s, gi, e, mean, rstd, xh, g);
#pragma unroll
    for (int i = 0; i < kW; ++i) {
      s1 += g[i];
      s2 = fmaf(g[i], xh[i], s2);
    }
  }
  __shared__ float2 sm[kNormWarps];
  s1 = warp_sum_down(s1);
  s2 = warp_sum_down(s2);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x / 32] = make_float2(s1, s2);
  __syncthreads();
  if (threadIdx.x == 0) {
    float2 t = sm[0];
    for (int w = 1; w < kNormWarps; ++w) {
      t.x += sm[w].x;
      t.y += sm[w].y;
    }
    reinterpret_cast<float2*>(a.workspace)[blockIdx.x] = t;
  }
}

template <typename TI, typename TO, int kW>
__global__ void __launch_bounds__(kNormThreads)
group_norm_bwd_apply_kernel(const psob200_group_norm_args a, const GnShape s) {
  const long long gi = blockIdx.x / s.P, part = blockIdx.x % s.P;
  const float mean = __ldg(a.mean + gi), rstd = __ldg(a.rstd + gi);
  __shared__ float st[2];
  if (threadIdx.x < 32) {
    const float2* ws = reinterpret_cast<const float2*>(a.workspace) + gi * s.P;
    float s1 = 0.f, s2 = 0.f;
    for (long long p = threadIdx.x; p < s.P; p += 32) {
      const float2 q = ws[p];
      s1 += q.x;
      s2 += q.y;
    }
    s1 = warp_sum_down(s1);
    s2 = warp_sum_down(s2);
    if (threadIdx.x == 0) {
      st[0] = s1 / (float)s.S;
      st[1] = s2 / (float)s.S;
    }
  }
  __syncthreads();
  const float c1 = st[0], c2 = st[1];
  const long long end = min(s.S, (part + 1) * kGnChunk);
  TI* dx = reinterpret_cast<TI*>(a.dx) + gi * s.S;
  for (long long e = part * kGnChunk + (long long)threadIdx.x * kW; e < end; e += kNormThreads * kW) {
    float xh[kW], g[kW];
    gn_grad_item<TI, TO, kW>(a, s, gi, e, mean, rstd, xh, g);
#pragma unroll
    for (int i = 0; i < kW; ++i) g[i] = rstd * (g[i] - c1 - xh[i] * c2);
    store_item<TI, kW>(dx + e, g);
  }
}

// ---------------------------------------------------------------------------------------------------------------- host side
// Validation order of every entry point: invalid argument, dtype, shape, alignment (then workspace).
static int norm_dtypes_check(int32_t dt, int32_t out_dt, int32_t param_dt) {
  if (!valid_dtype(dt) || !valid_dtype(param_dt) || !(out_dt == dt || out_dt == PSOB200_F32)) return PSOB200_ERR_DTYPE;
  return PSOB200_OK;
}

static int layer_norm_check(const psob200_layer_norm_args& a, bool bwd) {
  if (!a.x || a.rows <= 0 || a.C <= 0 || !a.mean || !a.rstd) return PSOB200_ERR_INVALID_ARG;
  if (bwd ? (!a.dy || !a.dx) : !a.y) return PSOB200_ERR_INVALID_ARG;
  if (int rc = norm_dtypes_check(a.dtype, a.out_dtype, a.param_dtype)) return rc;
  // whole 8-element chunks per row, row starts on 16-byte boundaries
  if (a.C % 8 || a.C > kLnMaxC || a.ld_x < a.C || a.ld_x % 8) return PSOB200_ERR_SHAPE;
  if (bwd ? (a.ld_dy < a.C || a.ld_dy % 8 || a.ld_dx < a.C || a.ld_dx % 8) : (a.ld_y < a.C || a.ld_y % 8))
    return PSOB200_ERR_SHAPE;
  if (!aligned16(a.x) || (bwd ? (!aligned16(a.dy) || !aligned16(a.dx)) : !aligned16(a.y))) return PSOB200_ERR_ALIGNMENT;
  return PSOB200_OK;
}

static int group_norm_check(const psob200_group_norm_args& a, bool bwd) {
  if (!a.x || a.N <= 0 || a.C <= 0 || a.HW <= 0 || a.G <= 0 || !a.mean || !a.rstd || !a.workspace) return PSOB200_ERR_INVALID_ARG;
  if (bwd ? (!a.dy || !a.dx) : !a.y) return PSOB200_ERR_INVALID_ARG;
  if (int rc = norm_dtypes_check(a.dtype, a.out_dtype, a.param_dtype)) return rc;
  if (a.C % a.G) return PSOB200_ERR_SHAPE;
  if (!aligned16(a.x) || !aligned16(a.workspace) || (bwd ? (!aligned16(a.dy) || !aligned16(a.dx)) : !aligned16(a.y)))
    return PSOB200_ERR_ALIGNMENT;
  if (a.workspace_bytes < psob200_group_norm_workspace_bytes(a.N, a.C, a.HW, a.G)) return PSOB200_ERR_WORKSPACE;
  return PSOB200_OK;
}

// CTAs of `kernel` that fit on the device at once (queried once per kernel instantiation and device)
template <typename Kernel>
static long long one_wave(Kernel kernel) {
  static PerDevice<int> cached_dev;
  std::atomic<int>& cached = cached_dev.here();
  int per_sm = cached.load(std::memory_order_relaxed);
  if (per_sm <= 0) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kNormThreads, 0) != cudaSuccess || per_sm <= 0) {
      cudaGetLastError();
      per_sm = 4;
    }
    cached.store(per_sm, std::memory_order_relaxed);
  }
  return (long long)sm_count() * per_sm;
}

template <typename TI, typename TO, int kV>
static void launch_layer_norm(const psob200_layer_norm_args& a, bool bwd, cudaStream_t st) {
  const long long want = (a.rows + kNormWarps - 1) / kNormWarps;
  if (bwd) {
    const long long grid = std::min(want, one_wave(layer_norm_bwd_kernel<TI, TO, kV>));
    layer_norm_bwd_kernel<TI, TO, kV><<<(unsigned)grid, kNormThreads, 0, st>>>(a);
  } else {
    const long long grid = std::min(want, one_wave(layer_norm_fwd_kernel<TI, TO, kV>));
    layer_norm_fwd_kernel<TI, TO, kV><<<(unsigned)grid, kNormThreads, 0, st>>>(a);
  }
}

template <typename TI, typename TO>
static void dispatch_layer_norm(const psob200_layer_norm_args& a, bool bwd, cudaStream_t st) {
  const long long v = (a.C / 8 + 31) / 32;  // chunks of 8 per lane
  if (v <= 1) launch_layer_norm<TI, TO, 1>(a, bwd, st);
  else if (v == 2) launch_layer_norm<TI, TO, 2>(a, bwd, st);
  else if (v == 3) launch_layer_norm<TI, TO, 3>(a, bwd, st);
  else if (v == 4) launch_layer_norm<TI, TO, 4>(a, bwd, st);
  else if (v == 5) launch_layer_norm<TI, TO, 5>(a, bwd, st);
  else launch_layer_norm<TI, TO, 8>(a, bwd, st);
}

template <typename TI, typename TO, int kW>
static void launch_group_norm_w(const psob200_group_norm_args& a, const GnShape& s, bool bwd, cudaStream_t st) {
  const unsigned grid = (unsigned)(a.N * a.G * s.P);
  if (bwd) {
    group_norm_bwd_sums_kernel<TI, TO, kW><<<grid, kNormThreads, 0, st>>>(a, s);
    group_norm_bwd_apply_kernel<TI, TO, kW><<<grid, kNormThreads, 0, st>>>(a, s);
  } else {
    group_norm_stats_kernel<TI, kW><<<grid, kNormThreads, 0, st>>>(a, s);
    group_norm_apply_kernel<TI, TO, kW><<<grid, kNormThreads, 0, st>>>(a, s);
  }
}

template <typename TI, typename TO>
static void launch_group_norm(const psob200_group_norm_args& a, bool bwd, cudaStream_t st) {
  GnShape s;
  s.Cg = a.C / a.G;
  s.HW = a.HW;
  s.S = s.Cg * a.HW;
  s.P = gn_parts(s.S);
  s.G = a.G;
  // 8-element items never straddle a channel when H*W % 8 == 0 (then every group and part starts 16-byte aligned too)
  if (a.HW % 8 == 0) launch_group_norm_w<TI, TO, 8>(a, s, bwd, st);
  else launch_group_norm_w<TI, TO, 1>(a, s, bwd, st);
}

// (input, output) element types: 16-bit -> same or fp32 (autocast), fp32 -> fp32
template <template <typename, typename> class L, typename Args>
static void dispatch_io(const Args& a, bool bwd, cudaStream_t st) {
  const bool f32_out = a.out_dtype == PSOB200_F32;
  if (a.dtype == PSOB200_BF16) {
    if (f32_out) L<__nv_bfloat16, float>::run(a, bwd, st);
    else L<__nv_bfloat16, __nv_bfloat16>::run(a, bwd, st);
  } else if (a.dtype == PSOB200_F16) {
    if (f32_out) L<__half, float>::run(a, bwd, st);
    else L<__half, __half>::run(a, bwd, st);
  } else {
    L<float, float>::run(a, bwd, st);
  }
}

template <typename TI, typename TO>
struct LayerNormLauncher {
  static void run(const psob200_layer_norm_args& a, bool bwd, cudaStream_t st) { dispatch_layer_norm<TI, TO>(a, bwd, st); }
};
template <typename TI, typename TO>
struct GroupNormLauncher {
  static void run(const psob200_group_norm_args& a, bool bwd, cudaStream_t st) { launch_group_norm<TI, TO>(a, bwd, st); }
};

}  // namespace psob200

using namespace psob200;

extern "C" size_t psob200_group_norm_workspace_bytes(int64_t N, int64_t C, int64_t HW, int32_t G) {
  if (N <= 0 || C <= 0 || HW <= 0 || G <= 0 || C % G) return 0;
  return (size_t)(N * G * gn_parts((C / G) * HW)) * sizeof(float2);
}

static int layer_norm_entry(const psob200_layer_norm_args* args, bool bwd, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const int rc = layer_norm_check(*args, bwd);
  if (rc != PSOB200_OK) return rc;
  dispatch_io<LayerNormLauncher>(*args, bwd, reinterpret_cast<cudaStream_t>(stream));
  return consume_launch_error(bwd ? "launch layer_norm_bwd_kernel" : "launch layer_norm_fwd_kernel", cudaSuccess);
}

static int group_norm_entry(const psob200_group_norm_args* args, bool bwd, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const int rc = group_norm_check(*args, bwd);
  if (rc != PSOB200_OK) return rc;
  dispatch_io<GroupNormLauncher>(*args, bwd, reinterpret_cast<cudaStream_t>(stream));
  const int lrc = consume_launch_error(bwd ? "launch group_norm backward kernels" : "launch group_norm forward kernels",
                                       cudaSuccess);
  if (lrc == PSOB200_OK) count_launch();  // two kernels per call
  return lrc;
}

extern "C" int psob200_layer_norm_forward(const psob200_layer_norm_args* args, void* stream) {
  return layer_norm_entry(args, false, stream);
}
extern "C" int psob200_layer_norm_backward(const psob200_layer_norm_args* args, void* stream) {
  return layer_norm_entry(args, true, stream);
}
extern "C" int psob200_group_norm_forward(const psob200_group_norm_args* args, void* stream) {
  return group_norm_entry(args, false, stream);
}
extern "C" int psob200_group_norm_backward(const psob200_group_norm_args* args, void* stream) {
  return group_norm_entry(args, true, stream);
}
