// Gated GELU of the transformer feed-forward, forward and backward, one launch each.
//
// diffusers==0.27.0 `GEGLU.forward`: `hidden, gate = self.proj(x).chunk(2, dim=-1); return hidden * F.gelu(gate)`.
// The feed-forward is NOT one of the PSO hot-path rows of SURVEY.md section 8; it sits between two LoRA-wrapped attention
// blocks of every transformer layer, and the stock lowering of that one line (strided gelu + strided mul forward;
// gelu_backward + two strided muls + the concatenation of the two halves backward) was the largest single item of the
// measured training micro-step (22 % of the kernel time at 128x128 latents, profiles/r01_step_breakdown.md).  Pure
// streaming work: forward reads 2 I and writes I elements per row, backward reads 3 I and writes 2 I.
//
// Arithmetic in fp32 (exact erf GELU, torch's default `approximate="none"`), one rounding to the storage type.
#include <atomic>

#include "common.cuh"

namespace psob200 {

constexpr int kGegluThreads = 256;
constexpr int kGegluColThreads = 64;                             // threads along a row: 64 x 8 elements = 512 columns
constexpr int kGegluRows = kGegluThreads / kGegluColThreads;     // rows per CTA per iteration

// Standard normal CDF.  fp32 storage: erff (north_star tolerance 1e-5).  16-bit storage: the Chebyshev fit of erfc with
// fractional error < 1.2e-7 everywhere (W. H. Press et al., "erfcc") -- one rcp.approx, one ex2.approx and ten FMAs instead of
// erff's ~30 instructions: the kernel was issue-bound on erff (ncu: 36 instructions per element, issue slots 66 % busy at
// 44 % of the HBM roofline).  Accurate in the far negative tail too (it is a fit of erfc itself, not of 1 - erf).
template <bool kPrecise>
__device__ __forceinline__ float normal_cdf(float x) {
  if constexpr (kPrecise) {
    return 0.5f * (1.f + erff(x * 0.70710678118654752f));
  } else {
    // everything in base 2: coefficients pre-multiplied by log2(e), the factor 0.5 folded in as 2^-1, so the tail is
    // rcp.approx + 10 FMA + ex2.approx (the IEEE __frcp_rn / __expf variants cost more instructions than erff itself)
    const float ax = fabsf(x);
    const float w = ax * 0.8493218003f;  // |x| sqrt(log2(e) / 2): w^2 = z^2 log2(e), z = |x| / sqrt 2
    float t, e;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.35355339059327376f, ax, 1.f)));  // 1 / (1 + z / 2)
    float p = fmaf(t, 0.246517298f, -1.18611495f);
    p = fmaf(t, p, 2.14747446f);
    p = fmaf(t, p, -1.63775315f);
    p = fmaf(t, p, 0.402321582f);
    p = fmaf(t, p, -0.26875686f);
    p = fmaf(t, p, 0.139630057f);
    p = fmaf(t, p, 0.539700616f);
    p = fmaf(t, p, 1.4427292f);
    p = fmaf(t, p, -2.82574822f);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(fmaf(-w, w, p)));
    const float half_erfc = t * e;  // 0.5 erfc(|x| / sqrt 2) = Phi(-|x|)
    return x > 0.f ? 1.f - half_erfc : half_erfc;
  }
}

template <bool kPrecise>
__device__ __forceinline__ float gelu_erf(float x) { return x * normal_cdf<kPrecise>(x); }

// d/dx [x Phi(x)] = Phi(x) + x phi(x)
template <bool kPrecise>
__device__ __forceinline__ void gelu_erf_grad(float x, float& y, float& dy) {
  const float cdf = normal_cdf<kPrecise>(x);
  float pdf;  // phi(x) = 2^(-x^2 log2(e) / 2) / sqrt(2 pi)
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(pdf) : "f"(-0.7213475204444817f * x * x));
  pdf *= 0.3989422804014327f;
  y = x * cdf;
  dy = fmaf(x, pdf, cdf);
}

// Thread (tx, ty) of CTA (bx, by) owns columns [8 (64 bx + tx), +8) of rows 4 by + ty, + 4 gridDim.y, ...; two rows per
// iteration so that four (forward) / six (backward) 128-bit loads are in flight per thread.
template <typename T>
__global__ void __launch_bounds__(kGegluThreads)
geglu_fwd_kernel(const T* __restrict__ proj, T* __restrict__ out, long long M, long long I, long long ld_proj, long long ld_out) {
  constexpr bool kPrecise = sizeof(T) == 4;
  const int tx = threadIdx.x % kGegluColThreads, ty = threadIdx.x / kGegluColThreads;
  const long long col = ((long long)blockIdx.x * kGegluColThreads + tx) * 8;
  if (col >= I) return;
  const long long step = (long long)gridDim.y * kGegluRows;
  if (col + 8 <= I) {
    for (long long row = (long long)blockIdx.y * kGegluRows + ty; row < M; row += 2 * step) {
      const bool two = row + step < M;
      const long long row1 = two ? row + step : row;
      const T* p0 = proj + row * ld_proj + col;
      const T* p1 = proj + row1 * ld_proj + col;
      const typename Vec8<T>::Raw rh0 = Vec8<T>::load_raw(p0), rg0 = Vec8<T>::load_raw(p0 + I);
      const typename Vec8<T>::Raw rh1 = Vec8<T>::load_raw(p1), rg1 = Vec8<T>::load_raw(p1 + I);
      float h[8], g[8], o[8];
      Vec8<T>::decode(rh0, h);
      Vec8<T>::decode(rg0, g);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = h[j] * gelu_erf<kPrecise>(g[j]);
      Vec8<T>::store(out + row * ld_out + col, o);
      if (two) {
        Vec8<T>::decode(rh1, h);
        Vec8<T>::decode(rg1, g);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = h[j] * gelu_erf<kPrecise>(g[j]);
        Vec8<T>::store(out + row1 * ld_out + col, o);
      }
    }
  } else {  // ragged last columns (fp32 rows whose width is a multiple of 4 but not of 8)
    for (long long row = (long long)blockIdx.y * kGegluRows + ty; row < M; row += step)
      for (long long j = col; j < I; ++j)
        Vec8<T>::store1(out + row * ld_out + j, Vec8<T>::load1(proj + row * ld_proj + j) *
                                                    gelu_erf<kPrecise>(Vec8<T>::load1(proj + row * ld_proj + I + j)));
  }
}

template <typename T>
__global__ void __launch_bounds__(kGegluThreads)
geglu_bwd_kernel(const T* __restrict__ proj, const T* __restrict__ dout, T* __restrict__ dproj, long long M, long long I,
                 long long ld_proj, long long ld_dout, long long ld_dproj) {
  constexpr bool kPrecise = sizeof(T) == 4;
  const int tx = threadIdx.x % kGegluColThreads, ty = threadIdx.x / kGegluColThreads;
  const long long col = ((long long)blockIdx.x * kGegluColThreads + tx) * 8;
  if (col >= I) return;
  const long long step = (long long)gridDim.y * kGegluRows;
  if (col + 8 <= I) {
    for (long long row = (long long)blockIdx.y * kGegluRows + ty; row < M; row += 2 * step) {
      const bool two = row + step < M;
      const long long row1 = two ? row + step : row;
      const T* p0 = proj + row * ld_proj + col;
      const T* p1 = proj + row1 * ld_proj + col;
      const typename Vec8<T>::Raw rh0 = Vec8<T>::load_raw(p0), rg0 = Vec8<T>::load_raw(p0 + I),
                                  rd0 = Vec8<T>::load_raw(dout + row * ld_dout + col);
      const typename Vec8<T>::Raw rh1 = Vec8<T>::load_raw(p1), rg1 = Vec8<T>::load_raw(p1 + I),
                                  rd1 = Vec8<T>::load_raw(dout + row1 * ld_dout + col);
      float h[8], g[8], dy[8], dh[8], dg[8];
      Vec8<T>::decode(rh0, h);
      Vec8<T>::decode(rg0, g);
      Vec8<T>::decode(rd0, dy);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float y, yp;
        gelu_erf_grad<kPrecise>(g[j], y, yp);
        dh[j] = dy[j] * y;
        dg[j] = dy[j] * h[j] * yp;
      }
      Vec8<T>::store(dproj + row * ld_dproj + col, dh);
      Vec8<T>::store(dproj + row * ld_dproj + col + I, dg);
      if (two) {
        Vec8<T>::decode(rh1, h);
        Vec8<T>::decode(rg1, g);
        Vec8<T>::decode(rd1, dy);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float y, yp;
          gelu_erf_grad<kPrecise>(g[j], y, yp);
          dh[j] = dy[j] * y;
          dg[j] = dy[j] * h[j] * yp;
        }
        Vec8<T>::store(dproj + row1 * ld_dproj + col, dh);
        Vec8<T>::store(dproj + row1 * ld_dproj + col + I, dg);
      }
    }
  } else {
    for (long long row = (long long)blockIdx.y * kGegluRows + ty; row < M; row += step)
      for (long long j = col; j < I; ++j) {
        const float hv = Vec8<T>::load1(proj + row * ld_proj + j), gv = Vec8<T>::load1(proj + row * ld_proj + I + j);
        const float dv = Vec8<T>::load1(dout + row * ld_dout + j);
        float y, yp;
        gelu_erf_grad<kPrecise>(gv, y, yp);
        Vec8<T>::store1(dproj + row * ld_dproj + j, dv * y);
        Vec8<T>::store1(dproj + row * ld_dproj + I + j, dv * hv * yp);
      }
  }
}

static int geglu_check(const psob200_geglu_args& a, bool bwd) {
  if (a.M <= 0 || a.I <= 0 || !a.proj) return PSOB200_ERR_INVALID_ARG;
  if (bwd ? (!a.dout || !a.dproj) : !a.out) return PSOB200_ERR_INVALID_ARG;
  if (!valid_dtype(a.dtype)) return PSOB200_ERR_DTYPE;
  const long long vec = a.dtype == PSOB200_F32 ? 4 : 8;  // elements per 16 bytes
  // the vector path needs every row start and the column split on a 16-byte boundary
  if ((a.I % vec) || (a.ld_proj % vec) || a.ld_proj < 2 * a.I) return PSOB200_ERR_SHAPE;
  if (bwd ? ((a.ld_dout % vec) || (a.ld_dproj % vec) || a.ld_dout < a.I || a.ld_dproj < 2 * a.I) : ((a.ld_out % vec) || a.ld_out < a.I))
    return PSOB200_ERR_SHAPE;
  if (!aligned16(a.proj) || (bwd ? (!aligned16(a.dout) || !aligned16(a.dproj)) : !aligned16(a.out))) return PSOB200_ERR_ALIGNMENT;
  return PSOB200_OK;
}

// One wave exactly: never more CTAs than fit at once (first version: 8 per SM assumed and rounded UP -- 1190 CTAs on 1184 slots
// ran the forward as two waves, and the backward, limited to 5 CTAs per SM by registers, as 1.6).
template <typename Kernel>
static dim3 geglu_grid(const psob200_geglu_args& a, Kernel kernel) {
  const long long bx = (a.I + kGegluColThreads * 8 - 1) / (kGegluColThreads * 8);
  const int sms = sm_count();
  static PerDevice<int> cached_dev;  // per kernel instantiation (this function is a template) and device: queried once
  std::atomic<int>& cached = cached_dev.here();
  int per_sm = cached.load(std::memory_order_relaxed);
  if (per_sm <= 0) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kGegluThreads, 0) != cudaSuccess || per_sm <= 0) {
      cudaGetLastError();
      per_sm = 4;
    }
    cached.store(per_sm, std::memory_order_relaxed);
  }
  long long by = (long long)sms * per_sm / bx;  // rounded down
  const long long row_blocks = (a.M + 2 * kGegluRows - 1) / (2 * kGegluRows);  // two rows per thread per iteration
  if (by > row_blocks) by = row_blocks;
  if (by > 65535) by = 65535;
  if (by < 1) by = 1;
  return dim3((unsigned)bx, (unsigned)by);
}

template <typename T>
static void launch_geglu_fwd(const psob200_geglu_args& a, cudaStream_t st) {
  const dim3 grid = geglu_grid(a, geglu_fwd_kernel<T>);
  geglu_fwd_kernel<T><<<grid, kGegluThreads, 0, st>>>(reinterpret_cast<const T*>(a.proj), reinterpret_cast<T*>(a.out), a.M, a.I,
                                                       a.ld_proj, a.ld_out);
}

template <typename T>
static void launch_geglu_bwd(const psob200_geglu_args& a, cudaStream_t st) {
  const dim3 grid = geglu_grid(a, geglu_bwd_kernel<T>);
  geglu_bwd_kernel<T><<<grid, kGegluThreads, 0, st>>>(reinterpret_cast<const T*>(a.proj), reinterpret_cast<const T*>(a.dout),
                                                       reinterpret_cast<T*>(a.dproj), a.M, a.I, a.ld_proj, a.ld_dout, a.ld_dproj);
}

}  // namespace psob200

using namespace psob200;

extern "C" int psob200_geglu_forward(const psob200_geglu_args* args, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_geglu_args& a = *args;
  const int rc = geglu_check(a, false);
  if (rc != PSOB200_OK) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (a.dtype == PSOB200_BF16) launch_geglu_fwd<__nv_bfloat16>(a, st);
  else if (a.dtype == PSOB200_F16) launch_geglu_fwd<__half>(a, st);
  else launch_geglu_fwd<float>(a, st);
  return consume_launch_error("launch geglu_fwd_kernel", cudaSuccess);
}

extern "C" int psob200_geglu_backward(const psob200_geglu_args* args, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_geglu_args& a = *args;
  const int rc = geglu_check(a, true);
  if (rc != PSOB200_OK) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (a.dtype == PSOB200_BF16) launch_geglu_bwd<__nv_bfloat16>(a, st);
  else if (a.dtype == PSOB200_F16) launch_geglu_bwd<__half>(a, st);
  else launch_geglu_bwd<float>(a, st);
  return consume_launch_error("launch geglu_bwd_kernel", cudaSuccess);
}
