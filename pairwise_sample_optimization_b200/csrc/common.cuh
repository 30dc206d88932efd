// Shared device helpers for the PSO hot-path kernels (sm_100a).
#pragma once

#include <cooperative_groups.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/psob200.h"

#include <atomic>

namespace cg = cooperative_groups;

namespace psob200 {

// ---------------------------------------------------------------------------------------------
// Host-side caches of per-DEVICE facts (SM count, occupancy, "MaxDynamicSharedMemorySize already raised for this kernel"):
// keyed by the ordinal of the calling thread's current device -- the device the launch goes to -- so that a process which
// drives several GPUs configures every kernel on each of them (cudaFuncSetAttribute is per device).
// ---------------------------------------------------------------------------------------------
constexpr int kMaxDevices = 64;
inline int device_slot() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess) {
    cudaGetLastError();
    d = 0;
  }
  return (d >= 0 && d < kMaxDevices) ? d : kMaxDevices - 1;
}
template <typename T>
struct PerDevice {  // static storage: zero-initialised
  std::atomic<T> v[kMaxDevices];
  std::atomic<T>& here() { return v[device_slot()]; }
};

// SM count of the current device for grid sizing, queried once per device (148, a B200's, when the query fails).
inline int sm_count() {
  static PerDevice<int> per_device;
  std::atomic<int>& cached = per_device.here();
  int v = cached.load(std::memory_order_relaxed);
  if (v > 0) return v;
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    cudaGetLastError();
    return 148;
  }
  cached.store(n, std::memory_order_relaxed);
  return n;
}

// ---------------------------------------------------------------------------------------------
// 8-element (one "chunk") vector access.  bf16/fp16: one 128-bit transaction; fp32: two.
// Loads are streaming (read once): non-coherent path, no L1 allocation.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_stream_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ void stg_u4(void* p, const uint4& v) {
  asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

template <typename T>
struct Vec8;

template <>
struct Vec8<float> {
  static constexpr int kBytes = 32;
  struct Raw { uint4 a, b; };
  static __device__ __forceinline__ Raw load_raw(const float* p) { return Raw{ldg_stream_u4(p), ldg_stream_u4(p + 4)}; }
  static __device__ __forceinline__ void decode(const Raw& r, float (&v)[8]) {
    v[0] = __uint_as_float(r.a.x); v[1] = __uint_as_float(r.a.y); v[2] = __uint_as_float(r.a.z); v[3] = __uint_as_float(r.a.w);
    v[4] = __uint_as_float(r.b.x); v[5] = __uint_as_float(r.b.y); v[6] = __uint_as_float(r.b.z); v[7] = __uint_as_float(r.b.w);
  }
  static __device__ __forceinline__ void load(const float* p, float (&v)[8]) {
    uint4 a = ldg_stream_u4(p), b = ldg_stream_u4(p + 4);
    v[0] = __uint_as_float(a.x); v[1] = __uint_as_float(a.y); v[2] = __uint_as_float(a.z); v[3] = __uint_as_float(a.w);
    v[4] = __uint_as_float(b.x); v[5] = __uint_as_float(b.y); v[6] = __uint_as_float(b.z); v[7] = __uint_as_float(b.w);
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[8]) {
    uint4 a, b;
    a.x = __float_as_uint(v[0]); a.y = __float_as_uint(v[1]); a.z = __float_as_uint(v[2]); a.w = __float_as_uint(v[3]);
    b.x = __float_as_uint(v[4]); b.y = __float_as_uint(v[5]); b.z = __float_as_uint(v[6]); b.w = __float_as_uint(v[7]);
    stg_u4(p, a);
    stg_u4(p + 4, b);
  }
  static __device__ __forceinline__ float load1(const float* p) { return __ldg(p); }
  static __device__ __forceinline__ void store1(float* p, float v) { *p = v; }
};

template <>
struct Vec8<__nv_bfloat16> {
  static constexpr int kBytes = 16;
  struct Raw { uint4 a; };
  static __device__ __forceinline__ Raw load_raw(const __nv_bfloat16* p) { return Raw{ldg_stream_u4(p)}; }
  static __device__ __forceinline__ void decode(const Raw& r, float (&v)[8]) {
    const uint32_t w[4] = {r.a.x, r.a.y, r.a.z, r.a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[8]) {
    uint4 a = ldg_stream_u4(p);
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {  // bf16 -> fp32 is a 16-bit shift
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[8]) {
    uint4 a;
    uint32_t* w = &a.x;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    stg_u4(p, a);
  }
  static __device__ __forceinline__ float load1(const __nv_bfloat16* p) {
    return __bfloat162float(__ldg(p));
  }
  static __device__ __forceinline__ void store1(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

template <>
struct Vec8<__half> {
  static constexpr int kBytes = 16;
  struct Raw { uint4 a; };
  static __device__ __forceinline__ Raw load_raw(const __half* p) { return Raw{ldg_stream_u4(p)}; }
  static __device__ __forceinline__ void decode(const Raw& r, float (&v)[8]) {
    const uint32_t w[4] = {r.a.x, r.a.y, r.a.z, r.a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
      v[2 * i] = f.x;
      v[2 * i + 1] = f.y;
    }
  }
  static __device__ __forceinline__ void load(const __half* p, float (&v)[8]) {
    uint4 a = ldg_stream_u4(p);
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
      float2 f = __half22float2(h);
      v[2 * i] = f.x;
      v[2 * i + 1] = f.y;
    }
  }
  static __device__ __forceinline__ void store(__half* p, const float (&v)[8]) {
    uint4 a;
    uint32_t* w = &a.x;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    stg_u4(p, a);
  }
  static __device__ __forceinline__ float load1(const __half* p) { return __half2float(__ldg(p)); }
  static __device__ __forceinline__ void store1(__half* p, float v) { *p = __float2half_rn(v); }
};

// ---------------------------------------------------------------------------------------------
// Reductions
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------------
// Per-sample step coefficients (SURVEY.md App. A.2), resolved on the device so that the host
// never syncs (the reference does one .item() per sample, TS:63).
// ---------------------------------------------------------------------------------------------
struct StepCoef {
  float k;           // mean = k*x + a*eps
  float a;
  float s;           // std
  float inv_2s2n;    // 1 / (2 s^2 N)
  float log_s;       // log s
  float a_over_s2n;  // a / (s^2 N)   (d logp / d eps = a_over_s2n * (x' - mu))
  float next_input_scale;  // turbo only: 1/sqrt(sigma_to^2 + 1), the next UNet-input scaling (TP:121)
};

__device__ __forceinline__ double load_timestep(const void* ts, int32_t ts_dtype, int64_t i) {
  if (ts_dtype == PSOB200_TS_I64) return (double)reinterpret_cast<const long long*>(ts)[i];
  if (ts_dtype == PSOB200_TS_F32) return (double)reinterpret_cast<const float*>(ts)[i];
  return (double)reinterpret_cast<const int*>(ts)[i];
}

__device__ __forceinline__ StepCoef make_coef(double k, double a, double s, int64_t N, int32_t* status) {
  StepCoef c;
  c.k = (float)k;
  c.a = (float)a;
  c.s = (float)s;
  c.inv_2s2n = (float)(1.0 / (2.0 * s * s * (double)N));
  c.log_s = (float)log(s);
  c.a_over_s2n = (float)(a / (s * s * (double)N));
  c.next_input_scale = 1.f;
  // s == 0 (the deterministic last turbo step, TS:79 with sigma_to = 0) legitimately gives -inf/NaN
  // log-probs in the reference too, so only k and a are policed here.
  if (status != nullptr && !(isfinite(c.k) && isfinite(c.a))) atomicOr(status, PSOB200_STATUS_NONFINITE_COEFFICIENT);
  return c;
}

// Resolve (k,a,s) for sample `b`.  `row` indexes the timestep arrays (0 when one timestep is
// broadcast over the batch).  Scalars are evaluated in fp64: a handful of flops per CTA.
__device__ __forceinline__ StepCoef resolve_coef(const psob200_schedule& sc, const void* ts, const void* ts_prev,
                                                 const float* coef, int64_t row, int64_t b, int64_t B, int64_t N,
                                                 int32_t* status) {
  const double qnan = __longlong_as_double(0x7ff8000000000000ULL);
  if (sc.kind == PSOB200_SCHED_AFFINE) {
    return make_coef((double)coef[b], (double)coef[B + b], (double)coef[2 * B + b], N, status);
  }
  const double t = load_timestep(ts, sc.ts_dtype, row);
  if (sc.kind == PSOB200_SCHED_TURBO) {
    int idx = -1;
    for (int i = 0; i < sc.n_table; ++i) {  // first match, like (_t == timesteps).nonzero()[0]  (TS:63)
      if ((double)sc.sched_timesteps[i] == t) { idx = i; break; }
    }
    if (idx < 0) {
      if (status != nullptr) atomicOr(status, PSOB200_STATUS_TIMESTEP_NOT_IN_SCHEDULE);
      return make_coef(qnan, qnan, qnan, N, nullptr);
    }
    const double s_from = (double)sc.table[idx], s_to = (double)sc.table[idx + 1];     // TS:77-78
    const double s_up = sqrt(s_to * s_to * (s_from * s_from - s_to * s_to) / (s_from * s_from));  // TS:79
    const double s_down = sqrt(s_to * s_to - s_up * s_up);                             // TS:80
    StepCoef c = make_coef(1.0, s_down - s_from, s_up, N, status);                     // TS:88-92
    c.next_input_scale = (float)(1.0 / sqrt(s_to * s_to + 1.0));
    return c;
  }
  // DMD (DS:36-42, 102-112); negative indices wrap like torch indexing (t_prev = -1 at the last step)
  long long it = (long long)t, ip = (long long)load_timestep(ts_prev, sc.ts_dtype, row);
  if (it < 0) it += sc.n_table;
  if (ip < 0) ip += sc.n_table;
  if (it < 0 || it >= sc.n_table || ip < 0 || ip >= sc.n_table) {
    if (status != nullptr) atomicOr(status, PSOB200_STATUS_TIMESTEP_NOT_IN_SCHEDULE);
    return make_coef(qnan, qnan, qnan, N, nullptr);
  }
  const double a_t = (double)sc.table[it], a_p = (double)sc.table[ip];
  return make_coef(sqrt(a_p) / sqrt(a_t), -sqrt(a_p) * sqrt(1.0 - a_t) / sqrt(a_t), sqrt(1.0 - a_p), N, status);
}

// ---------------------------------------------------------------------------------------------
// Host-side helpers
// ---------------------------------------------------------------------------------------------
// Records what CUDA said about the last failed call of this thread (psob200_last_error_detail()).
void set_error_detail(const char* where, cudaError_t e);
// Bumps the library's launch counter (psob200_launch_count()).
void count_launch();
// Consumes the sticky-free last error; returns PSOB200_ERR_LAUNCH (and records the detail) if there was one.
inline int consume_launch_error(const char* where, cudaError_t e) {
  if (e == cudaSuccess) e = cudaPeekAtLastError();
  if (e == cudaSuccess) {
    count_launch();
    return PSOB200_OK;
  }
  set_error_detail(where, e);
  cudaGetLastError();
  return PSOB200_ERR_LAUNCH;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t dtype_size(int32_t dt) { return dt == PSOB200_F32 ? 4 : 2; }
inline bool valid_dtype(int32_t dt) { return dt == PSOB200_F32 || dt == PSOB200_BF16 || dt == PSOB200_F16; }

// Launch with an optional thread-block-cluster dimension (x only).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                  unsigned cluster, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// dtype dispatch: calls f(TP{}, TL{}) with the element types selected at run time.
template <typename F>
inline int dispatch2(int32_t dp, int32_t dl, F&& f) {
#define PSOB200_D2(DP, TPP)                                         \
  if (dp == DP) {                                                   \
    if (dl == PSOB200_F32) return f(TPP{}, float{});                \
    if (dl == PSOB200_BF16) return f(TPP{}, __nv_bfloat16{});       \
    if (dl == PSOB200_F16) return f(TPP{}, __half{});               \
  }
  PSOB200_D2(PSOB200_F32, float)
  PSOB200_D2(PSOB200_BF16, __nv_bfloat16)
  PSOB200_D2(PSOB200_F16, __half)
#undef PSOB200_D2
  return PSOB200_ERR_DTYPE;
}

}  // namespace psob200
