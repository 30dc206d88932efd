// Fused pairwise PSO loss + gradient (sm_100a).
//
// Per (win, lose) pair the eight tensors (policy / frozen-reference predictions, current and next latents, both
// branches) are processed in two passes with the residuals kept ON CHIP in between:
//
//   pass 1  stream the pair from HBM, form the policy residual r = x' - (k x + a eps) and, per branch, the sums needed
//           for  S_pol = sum r^2,  S_ref = sum r_ref^2,  D = S_ref - S_pol;
//   reduce  warp shuffles -> shared memory -> distributed shared memory over the cluster that shares the pair; the
//           pair's scalar loss function (clamp gate, log-sigmoid / hinge, prior) gives one multiplier per branch;
//           deterministic: fixed summation order, no atomics on the data path;
//   pass 2  write grad = g_k * r from the on-chip residuals.
//
// HBM traffic is the algorithmic 8N reads + 2N writes per pair (SURVEY.md section 8d).
//
// Two kernels share that structure (DESIGN.md section 3.1, profiles/r01_pair_loss.md; a third design -- a TMA ring with the
// residuals in registers, 44-57 % of HBM -- was measured in round 1 and is kept out of the product under tools/experiments/):
//   pair_loss_grad_tmem_kernel  (fast path, pair_loss_tmem.cuh) residuals parked in TENSOR MEMORY (tcgen05.st / ld),
//           1024 threads per SM, a per-thread cp.async ring of 192 KB, cluster of 1 (64^2 latents) or 2 (128^2);
//   pair_loss_grad_kernel       (general path, this file) vectorised or scalar LDG, residuals in shared memory;
//           any N, any alignment, up to 25600 elements per branch per CTA, one cluster per pair.
//
// Replaces: train_online_pso_sdxl_turbo.py:810-850,857 / train_online_pso_sdxl_dmd2.py:812-854,859
// (online) and train_pso_sdxl_turbo_dreambooth.py:1847-1865,1881-1935,1953 (DreamBooth).
#include <atomic>
#include <cmath>

#include "common.cuh"

namespace psob200 {

constexpr int kMaxCluster = 8;
constexpr int kMaxThreads = 512;
constexpr int kModeOnline = 0, kModeDbPso = 1, kModeDbPsoDb = 2;

struct PairKernelArgs {
  const void* pred[2];
  const void* ref[2];
  const void* x[2];
  const void* xn[2];
  void* grad[2];
  psob200_schedule sched;
  const void* ts[2];
  const void* ts_prev[2];
  const float* coef[2];
  const float* sigmas;  // dreambooth float[2B]
  const float* human_prefer;
  float* loss;
  float* stats;
  int32_t* status;
  unsigned int* counter;
  float* pair_loss;
  const float* amp_scale;  // device loss scale S (psob200_loss_scaler), NULL = none: multiplies the gradient multipliers
  long long B, N;
  long long stride[4][2];  // element stride between samples: pred, ref, x, xn
  double log_lo, log_hi;   // log(1-eps), log(1+eps): the clamp of T:844-845 expressed on delta
  int chunks_per_cta;
  int mode;
  float beta, eps, loss_scale, nu, lam;
};

__device__ __forceinline__ double softplus_neg(double z) {  // softplus(-z) = -log sigmoid(z)
  return log1p(exp(-fabs(z))) + fmax(-z, 0.0);
}
__device__ __forceinline__ double sigmoid_neg(double z) {  // sigmoid(-z)
  return 1.0 / (1.0 + exp(z));
}

__device__ __forceinline__ void resolve_pair_coefs(const PairKernelArgs& a, long long pair, int k, StepCoef* out) {
  if (a.mode == kModeOnline) {
    *out = resolve_coef(a.sched, a.ts[k], a.ts_prev[k], a.coef[k], pair, pair, a.B, a.N, a.status);
  } else {
    const double sg = (double)a.sigmas[(long long)k * a.B + pair];  // P:1855: x0_hat = -sigma*pred + noisy
    *out = make_coef(1.0, -sg, sg, a.N, a.status);
  }
}

// The pair's scalar function, evaluated by ONE thread of every CTA of the cluster on identical inputs
// (partials summed in rank order), so all CTAs obtain bit-identical gradient multipliers.
__device__ __forceinline__ void pair_scalar_function(const PairKernelArgs& a, long long pair, unsigned rank, unsigned C,
                                                     const float (*s_part)[8], const StepCoef* s_coef, float* s_g) {
  double S[2][3];
  for (int k = 0; k < 2; ++k)
    for (int j = 0; j < 3; ++j) {
      double v = 0.0;
      for (unsigned r = 0; r < C; ++r) v += (double)s_part[r][k * 3 + j];
      S[k][j] = v;
    }
  const StepCoef c0 = s_coef[0], c1 = s_coef[1];
  const double i0 = (double)c0.inv_2s2n, i1 = (double)c1.inv_2s2n;
  const double invB = 1.0 / (double)a.B;
  double g0, g1, per;
  float st[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (a.mode == kModeOnline) {
    const double kHalfLog2Pi = 0.91893853320467274178;
    const double d0 = S[0][2] * i0, d1 = S[1][2] * i1;  // delta_k = logp_pol,k - logp_ref,k
    const double beta = (double)a.beta, lo = a.log_lo, hi = a.log_hi;
    const bool open0 = (d0 >= lo) && (d0 <= hi), open1 = (d1 >= lo) && (d1 <= hi);
    // log(clamp(exp(d), 1-eps, 1+eps)): inside the clamp that is d itself (T:844-845); NaN propagates
    const double lr0 = open0 ? d0 : (d0 < lo ? lo : (d0 > hi ? hi : d0));
    const double lr1 = open1 ? d1 : (d1 < lo ? lo : (d1 > hi ? hi : d1));
    const double h0 = (double)a.human_prefer[pair * 2], h1 = (double)a.human_prefer[pair * 2 + 1];
    const double z = beta * (h0 * lr0 + h1 * lr1);  // T:847-850
    per = softplus_neg(z);
    const double common = -sigmoid_neg(z) * invB * beta * (double)a.loss_scale;
    g0 = open0 ? common * h0 * (double)c0.a_over_s2n : 0.0;  // torch.clamp passes grad on the closed interval
    g1 = open1 ? common * h1 * (double)c1.a_over_s2n : 0.0;
    st[0] = (float)(-S[0][0] * i0 - (double)c0.log_s - kHalfLog2Pi);  // TS:108-114 / DS:129-135
    st[1] = (float)(-S[0][1] * i0 - (double)c0.log_s - kHalfLog2Pi);
    st[2] = (float)(-S[1][0] * i1 - (double)c1.log_s - kHalfLog2Pi);
    st[3] = (float)(-S[1][1] * i1 - (double)c1.log_s - kHalfLog2Pi);
    st[4] = (float)d0;
    st[5] = (float)d1;
    st[6] = (float)z;
    st[7] = (float)per;
  } else {
    const double nu = (double)a.nu, beta = (double)a.beta;
    const double lam = a.lam > 0.f ? (double)a.lam : 0.0;           // P:1932
    const double Lw = 2.0 * S[0][0] * i0, Ll = 2.0 * S[1][0] * i1;  // P:1885-1891
    double logits, dl;
    if (a.mode == kModeDbPso) {
      logits = 2.0 * S[0][2] * i0 - nu * (2.0 * S[1][2] * i1);  // (Lref_w-L_w) - nu (Lref_l-L_l)  P:1919
      per = softplus_neg(beta * logits);                         // P:1925
      dl = -beta * sigmoid_neg(beta * logits) * invB;
      st[2] = (float)(2.0 * S[0][1] * i0);
      st[3] = (float)(2.0 * S[1][1] * i1);
    } else {
      logits = -(Lw - nu * Ll);  // P:1922
      const double m = 1.0 - beta * logits;
      per = m > 0.0 ? m : (m == m ? 0.0 : m);  // relu, NaN propagates   P:1927
      dl = m > 0.0 ? -beta * invB : 0.0;
    }
    per += lam * Ll;  // P:1932-1935
    const double Gw = -dl, Gl = nu * dl + lam * invB;
    g0 = (double)a.loss_scale * Gw * (-2.0 * (double)c0.a_over_s2n);
    g1 = (double)a.loss_scale * Gl * (-2.0 * (double)c1.a_over_s2n);
    st[0] = (float)Lw;
    st[1] = (float)Ll;
    st[4] = (float)logits;
    st[5] = (float)per;
  }
  float f0 = (float)g0, f1 = (float)g1;
  if (a.amp_scale != nullptr) {  // scaled in fp32 after the rounding: a power-of-two S gives exactly S x the unscaled grad
    const float S = *a.amp_scale;
    f0 *= S;
    f1 *= S;
  }
  s_g[0] = f0;
  s_g[1] = f1;
  if (rank == 0) {
    a.pair_loss[pair] = (float)per;
    if (a.stats != nullptr) {
      float4* dst = reinterpret_cast<float4*>(a.stats + pair * 8);
      dst[0] = make_float4(st[0], st[1], st[2], st[3]);
      dst[1] = make_float4(st[4], st[5], st[6], st[7]);
    }
  }
}

// CTA-level sum of the six accumulators and all-gather of the CTA partials over the cluster through
// distributed shared memory.  On return s_part[r][0..5] holds CTA r's partials in every CTA.
__device__ __forceinline__ void reduce_and_allgather(cg::cluster_group& cluster, const float (&acc)[2][3],
                                                     float (*s_warp)[kMaxThreads / 32], float (*s_part)[8]) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const unsigned C = cluster.num_blocks(), rank = cluster.block_rank();
#pragma unroll
  for (int k = 0; k < 2; ++k)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const float v = warp_sum(acc[k][j]);
      if (lane == 0) s_warp[k * 3 + j][warp] = v;
    }
  __syncthreads();
  float part = 0.f;
  if (tid < 6)
    for (int w = 0; w < nwarps; ++w) part += s_warp[tid][w];
  cluster.barrier_wait();  // pairs with barrier_arrive() at kernel entry: every CTA of the cluster is running
  if (tid < 6)
    for (unsigned r = 0; r < C; ++r) *cluster.map_shared_rank(&s_part[rank][tid], r) = part;
  cluster.sync();  // arrive.release / wait.acquire: the partials are visible in every CTA
}

// mean over pairs by the last cluster to finish (fixed summation order: deterministic); leaves the
// workspace counter zeroed for the next launch.
__device__ __forceinline__ void finalize_mean(const PairKernelArgs& a, int lane) {
  unsigned ticket = 0;
  if (lane == 0) {
    __threadfence();
    ticket = atomicAdd(a.counter, 1u);
  }
  ticket = __shfl_sync(0xffffffffu, ticket, 0);
  if (ticket == (unsigned)(a.B - 1)) {
    __threadfence();
    double s = 0.0;
    for (long long i = lane; i < a.B; i += 32) s += (double)__ldcg(a.pair_loss + i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      a.loss[0] = (float)((double)a.loss_scale * s / (double)a.B);
      *a.counter = 0u;
    }
  }
}

template <bool HAS_REF>
__device__ __forceinline__ void residual8(const float (&vx)[8], const float (&vn)[8], const float (&vp)[8],
                                          const float (&vr)[8], float kx, float ca, float (&r)[8], float& s_t,
                                          float& s_r, float& s_d) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float b0 = fmaf(-kx, vx[i], vn[i]);
    const float rt = fmaf(-ca, vp[i], b0);
    r[i] = rt;
    s_t = fmaf(rt, rt, s_t);
    if constexpr (HAS_REF) {
      const float rr = fmaf(-ca, vr[i], b0);
      s_r = fmaf(rr, rr, s_r);
      // sum(rr^2 - rt^2) = sum((rr-rt)(rr+rt)) with rr-rt = a*(eps_pol - eps_ref) formed from the
      // predictions themselves: no cancellation against the (much larger) latents
      s_d = fmaf(ca * (vp[i] - vr[i]), rr + rt, s_d);
    }
  }
}

}  // namespace psob200

#include "pair_loss_tmem.cuh"  // fast path: residuals in tensor memory, per-thread cp.async ring

namespace psob200 {

// =============================================================================================
// General path: LDG (vector or scalar), residuals in shared memory.
// =============================================================================================
template <typename TP, typename TL, bool HAS_REF, int W>
__global__ void __launch_bounds__(kMaxThreads) pair_loss_grad_kernel(const PairKernelArgs a) {
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned C = cluster.num_blocks();
  const unsigned rank = cluster.block_rank();
  const long long pair = blockIdx.x / C;
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* res = reinterpret_cast<float*>(smem_raw);  // [2 branches][chunks_per_cta * W] residuals
  __shared__ float s_warp[6][kMaxThreads / 32];
  __shared__ float s_part[kMaxCluster][8];
  __shared__ StepCoef s_coef[2];
  __shared__ float s_g[2];

  cluster.barrier_arrive();
  if (tid < 2) resolve_pair_coefs(a, pair, tid, &s_coef[tid]);
  __syncthreads();

  const int cpc = a.chunks_per_cta;
  const long long nchunk = (a.N + W - 1) / W;
  const long long cbeg = (long long)rank * cpc;
  const long long cend = (cbeg + cpc < nchunk) ? cbeg + cpc : nchunk;

  float acc[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const TP* pred = reinterpret_cast<const TP*>(a.pred[k]) + pair * a.stride[0][k];
    const TP* ref = HAS_REF ? reinterpret_cast<const TP*>(a.ref[k]) + pair * a.stride[1][k] : nullptr;
    const TL* x = reinterpret_cast<const TL*>(a.x[k]) + pair * a.stride[2][k];
    const TL* xn = reinterpret_cast<const TL*>(a.xn[k]) + pair * a.stride[3][k];
    const float kx = s_coef[k].k, ca = s_coef[k].a;
    float* resk = res + (size_t)k * cpc * W;
    float s_t = 0.f, s_r = 0.f, s_d = 0.f;
    if constexpr (W == 8) {
      float4* plane0 = reinterpret_cast<float4*>(resk);
      float4* plane1 = plane0 + cpc;
#pragma unroll 2
      for (long long c = cbeg + tid; c < cend; c += T) {
        float vx[8], vn[8], vp[8], vr[8], r[8];
        Vec8<TL>::load(x + c * 8, vx);
        Vec8<TL>::load(xn + c * 8, vn);
        Vec8<TP>::load(pred + c * 8, vp);
        if constexpr (HAS_REF) Vec8<TP>::load(ref + c * 8, vr);
        residual8<HAS_REF>(vx, vn, vp, vr, kx, ca, r, s_t, s_r, s_d);
        const int l = (int)(c - cbeg);
        plane0[l] = make_float4(r[0], r[1], r[2], r[3]);
        plane1[l] = make_float4(r[4], r[5], r[6], r[7]);
      }
    } else {
      for (long long c = cbeg + tid; c < cend; c += T) {
        const float b0 = fmaf(-kx, Vec8<TL>::load1(x + c), Vec8<TL>::load1(xn + c));
        const float ep = Vec8<TP>::load1(pred + c);
        const float rt = fmaf(-ca, ep, b0);
        s_t = fmaf(rt, rt, s_t);
        if constexpr (HAS_REF) {
          const float er = Vec8<TP>::load1(ref + c);
          const float rr = fmaf(-ca, er, b0);
          s_r = fmaf(rr, rr, s_r);
          s_d = fmaf(ca * (ep - er), rr + rt, s_d);
        }
        resk[c - cbeg] = rt;
      }
    }
    acc[k][0] = s_t;
    acc[k][1] = s_r;
    acc[k][2] = s_d;
  }

  reduce_and_allgather(cluster, acc, s_warp, s_part);
  if (tid == 0) pair_scalar_function(a, pair, rank, C, s_part, s_coef, s_g);
  __syncthreads();

#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const float g = s_g[k];
    TP* grad = reinterpret_cast<TP*>(a.grad[k]) + pair * a.N;
    const float* resk = res + (size_t)k * cpc * W;
    if constexpr (W == 8) {
      const float4* plane0 = reinterpret_cast<const float4*>(resk);
      const float4* plane1 = plane0 + cpc;
#pragma unroll 2
      for (long long c = cbeg + tid; c < cend; c += T) {
        const int l = (int)(c - cbeg);
        const float4 lo4 = plane0[l], hi4 = plane1[l];
        const float o[8] = {g * lo4.x, g * lo4.y, g * lo4.z, g * lo4.w, g * hi4.x, g * hi4.y, g * hi4.z, g * hi4.w};
        Vec8<TP>::store(grad + c * 8, o);
      }
    } else {
      for (long long c = cbeg + tid; c < cend; c += T) Vec8<TP>::store1(grad + c, g * resk[c - cbeg]);
    }
  }
  if (rank == 0 && warp == 0) finalize_mean(a, lane);
}

// ----------------------------------------------------------------------------------------------
template <typename K>
static int ensure_dynamic_smem(K kern, size_t smem, PerDevice<size_t>& per_device, const char* what) {
  std::atomic<size_t>& configured = per_device.here();  // 0 = untouched on this device: the 48 KB default applies
  if (smem <= 48 * 1024 || smem <= configured.load(std::memory_order_acquire)) return PSOB200_OK;
  cudaFuncAttributes fa;
  cudaError_t e = cudaFuncGetAttributes(&fa, kern);
  if (e != cudaSuccess) return consume_launch_error(what, e);
  const size_t limit = (size_t)227 * 1024 - fa.sharedSizeBytes;
  if (smem > limit) return PSOB200_ERR_SHAPE;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit);
  if (e != cudaSuccess) return consume_launch_error(what, e);
  configured.store(limit, std::memory_order_release);
  return PSOB200_OK;
}

template <typename TP, typename TL, bool HAS_REF, int W>
static int launch_pair_inst(const PairKernelArgs& ka, int threads, int cluster, size_t smem, cudaStream_t stream) {
  auto kern = pair_loss_grad_kernel<TP, TL, HAS_REF, W>;
  static PerDevice<size_t> configured;
  const int rc = ensure_dynamic_smem(kern, smem, configured, "configure pair_loss_grad_kernel");
  if (rc != PSOB200_OK) return rc;
  const cudaError_t e = launch_cluster(kern, dim3((unsigned)(ka.B * cluster)), dim3(threads), smem, stream,
                                       (unsigned)cluster, ka);
  return consume_launch_error("launch pair_loss_grad_kernel", e);
}

// Clusters of `cluster` CTAs that can be co-resident for this kernel (cached per instantiation and cluster size).
template <typename K>
static int max_active_clusters(K kern, int threads, size_t smem, int cluster, int sm_count, int ctas_per_sm,
                               PerDevice<int>* per_device) {
  int idx = cluster == 1 ? 0 : cluster == 2 ? 1 : cluster == 4 ? 2 : 3;
  std::atomic<int>& slot = per_device[idx].here();
  int v = slot.load(std::memory_order_relaxed);
  if (v > 0) return v;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(sm_count * ctas_per_sm / cluster * cluster));
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    n = sm_count * ctas_per_sm / cluster;  // optimistic fallback: the grid is still correct, only less balanced
  }
  slot.store(n, std::memory_order_relaxed);
  return n;
}

template <typename TP, typename TL, bool HAS_REF>
static int launch_pair_tmem_inst(const PairKernelArgs& ka, int cluster, int sm_count, cudaStream_t stream) {
  auto kern = pair_loss_grad_tmem_kernel<TP, TL, HAS_REF>;
  using Cfg = V3Cfg<TP, TL, HAS_REF>;
  constexpr size_t smem = Cfg::kSmemBytes;
  static PerDevice<size_t> configured;
  static PerDevice<int> active[4];
  const int rc = ensure_dynamic_smem(kern, smem, configured, "configure pair_loss_grad_tmem_kernel");
  if (rc != PSOB200_OK) return rc;
  long long clusters = max_active_clusters(kern, Cfg::kThreads, smem, cluster, sm_count, 1, active);
  if (clusters > ka.B) clusters = ka.B;  // persistent: every cluster loops over pairs cluster_id, +clusters, ...
  const cudaError_t e = launch_cluster(kern, dim3((unsigned)(clusters * cluster)), dim3(Cfg::kThreads), smem, stream,
                                       (unsigned)cluster, ka);
  return consume_launch_error("launch pair_loss_grad_tmem_kernel", e);
}

// Cluster size for the tensor-memory kernel: the smallest that fits a pair's residuals (at most kMaxIters/2 chunk
// iterations per branch per CTA), widened for small batches so that more SMs share a pair.  0 = does not fit.
template <typename TP, typename TL, bool HAS_REF>
static int tmem_cluster_for(long long nchunk, long long B, int sm_count, int tune_cluster) {
  using Cfg = V3Cfg<TP, TL, HAS_REF>;
  const long long cap = (long long)(Cfg::kMaxIters / 2) * Cfg::kThreads;  // chunks per branch per CTA
  if (tune_cluster != 0) return (nchunk + tune_cluster - 1) / tune_cluster <= cap ? tune_cluster : 0;
  int c = 1;
  while (c < kMaxCluster && (nchunk + c - 1) / c > cap) c <<= 1;
  if ((nchunk + c - 1) / c > cap) return 0;
  while (c < kMaxCluster && B * c * 2 <= sm_count && nchunk / (c * 2) >= Cfg::kThreads) c <<= 1;
  return c;
}

// tune_threads: 0 = heuristics (the tensor-memory kernel); >= 32 = the general (LDG) kernel with that many threads.
// tune_cluster: 0 = heuristics.
static int launch_pair(PairKernelArgs ka, bool has_ref, int32_t pred_dtype, int32_t latent_dtype, bool vec_ok,
                       int tune_threads, int tune_cluster, int sm_count, cudaStream_t stream) {
  if (tune_cluster != 0 && tune_cluster != 1 && tune_cluster != 2 && tune_cluster != 4 && tune_cluster != 8)
    return PSOB200_ERR_INVALID_ARG;
  if (tune_threads < 0 || (tune_threads > 0 && tune_threads < 32)) return PSOB200_ERR_INVALID_ARG;
  // ---- fast path: residuals in tensor memory
  if (vec_ok && tune_threads == 0) {
    const long long nchunk = ka.N / 8;
    const int rc = dispatch2(pred_dtype, latent_dtype, [&](auto tp, auto tl) -> int {
      using TP = decltype(tp);
      using TL = decltype(tl);
      const int cluster = has_ref ? tmem_cluster_for<TP, TL, true>(nchunk, ka.B, sm_count, tune_cluster)
                                  : tmem_cluster_for<TP, TL, false>(nchunk, ka.B, sm_count, tune_cluster);
      if (cluster == 0) return 1;  // does not fit: fall through to the general path
      PairKernelArgs k2 = ka;
      k2.chunks_per_cta = (int)((nchunk + cluster - 1) / cluster);
      return has_ref ? launch_pair_tmem_inst<TP, TL, true>(k2, cluster, sm_count, stream)
                     : launch_pair_tmem_inst<TP, TL, false>(k2, cluster, sm_count, stream);
    });
    if (rc != 1) return rc;
    if (tune_cluster != 0) return PSOB200_ERR_SHAPE;
  }
  // ---- general path
  const int W = vec_ok ? 8 : 1;
  const long long nchunk = (ka.N + W - 1) / W;
  const int threads = tune_threads >= 32 ? tune_threads : 256;
  if (threads > kMaxThreads || threads < 32 || (threads & 31)) return PSOB200_ERR_INVALID_ARG;
  // cluster size: keep the fp32 residual slab <= 64 KB per CTA (>= 3 CTAs per SM) when possible,
  // and spread small batches over more SMs for latency.
  const long long per_branch_cap = 8192, hard_cap = 25600;  // elements per branch per CTA
  int cluster = tune_cluster;
  if (cluster <= 0) {
    cluster = 1;
    while (cluster < kMaxCluster && (ka.N + cluster - 1) / cluster > per_branch_cap) cluster <<= 1;
    while (cluster < kMaxCluster && ka.B * cluster < 2LL * sm_count && nchunk / (cluster * 2) >= threads) cluster <<= 1;
  }
  const long long cpc = (nchunk + cluster - 1) / cluster;
  if (cpc * W > hard_cap) return PSOB200_ERR_SHAPE;
  ka.chunks_per_cta = (int)cpc;
  const size_t smem = (size_t)2 * cpc * W * sizeof(float);
  return dispatch2(pred_dtype, latent_dtype, [&](auto tp, auto tl) -> int {
    using TP = decltype(tp);
    using TL = decltype(tl);
    if (has_ref) {
      return W == 8 ? launch_pair_inst<TP, TL, true, 8>(ka, threads, cluster, smem, stream)
                    : launch_pair_inst<TP, TL, true, 1>(ka, threads, cluster, smem, stream);
    }
    return W == 8 ? launch_pair_inst<TP, TL, false, 8>(ka, threads, cluster, smem, stream)
                  : launch_pair_inst<TP, TL, false, 1>(ka, threads, cluster, smem, stream);
  });
}

}  // namespace psob200

using namespace psob200;

extern "C" size_t psob200_pair_loss_workspace_bytes(int64_t B) {
  if (B < 0) B = 0;
  return (size_t)16 + (((size_t)B * sizeof(float) + 15) & ~(size_t)15);
}

// amp_scale: the device loss scale of a psob200_loss_scaler, or NULL (the unscaled entry points)
static int online_pso_loss_grad(const psob200_schedule* sched, const psob200_online_pso_args* args, const float* amp_scale,
                                void* stream) {
  if (sched == nullptr || args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_online_pso_args& p = *args;
  if (p.B <= 0 || p.N <= 0 || p.loss == nullptr || p.human_prefer == nullptr || p.workspace == nullptr)
    return PSOB200_ERR_INVALID_ARG;
  if (!valid_dtype(p.pred_dtype) || !valid_dtype(p.latent_dtype)) return PSOB200_ERR_DTYPE;
  if (p.workspace_bytes < psob200_pair_loss_workspace_bytes(p.B)) return PSOB200_ERR_WORKSPACE;
  if (!aligned16(p.workspace) || (p.stats != nullptr && !aligned16(p.stats))) return PSOB200_ERR_ALIGNMENT;
  bool vec_ok = (p.N % 8) == 0;
  PairKernelArgs ka = {};
  for (int k = 0; k < 2; ++k) {
    if (!p.pred[k] || !p.ref[k] || !p.sample[k] || !p.next[k] || !p.grad[k]) return PSOB200_ERR_INVALID_ARG;
    if (sched->kind == PSOB200_SCHED_AFFINE) {
      if (!p.coef[k]) return PSOB200_ERR_INVALID_ARG;
    } else {
      if (!p.ts[k] || !sched->table || sched->n_table <= 0) return PSOB200_ERR_INVALID_ARG;
      if (sched->kind == PSOB200_SCHED_DMD && !p.ts_prev[k]) return PSOB200_ERR_INVALID_ARG;
      if (sched->kind == PSOB200_SCHED_TURBO && !sched->sched_timesteps) return PSOB200_ERR_INVALID_ARG;
    }
    vec_ok = vec_ok && aligned16(p.pred[k]) && aligned16(p.ref[k]) && aligned16(p.sample[k]) &&
             aligned16(p.next[k]) && aligned16(p.grad[k]);
    ka.pred[k] = p.pred[k]; ka.ref[k] = p.ref[k]; ka.x[k] = p.sample[k]; ka.xn[k] = p.next[k];
    ka.grad[k] = p.grad[k]; ka.ts[k] = p.ts[k]; ka.ts_prev[k] = p.ts_prev[k]; ka.coef[k] = p.coef[k];
    const int64_t st[4] = {p.stride_pred[k], p.stride_ref[k], p.stride_sample[k], p.stride_next[k]};
    for (int j = 0; j < 4; ++j) {
      if (st[j] < 0) return PSOB200_ERR_INVALID_ARG;
      ka.stride[j][k] = st[j] == 0 ? p.N : st[j];
      vec_ok = vec_ok && (ka.stride[j][k] % 8) == 0;
    }
  }
  if (sched->kind != PSOB200_SCHED_TURBO && sched->kind != PSOB200_SCHED_DMD && sched->kind != PSOB200_SCHED_AFFINE)
    return PSOB200_ERR_INVALID_ARG;
  ka.sched = *sched;
  ka.human_prefer = p.human_prefer;
  ka.loss = p.loss; ka.stats = p.stats; ka.status = p.status;
  ka.counter = reinterpret_cast<unsigned int*>(p.workspace);
  ka.pair_loss = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(p.workspace) + 16);
  ka.amp_scale = amp_scale;
  ka.B = p.B; ka.N = p.N; ka.mode = kModeOnline;
  ka.beta = p.beta; ka.eps = p.eps; ka.loss_scale = p.loss_scale;
  const double eps = (double)p.eps;
  ka.log_lo = (1.0 - eps > 0.0) ? std::log(1.0 - eps) : -HUGE_VAL;  // exp(d) > 0 >= 1-eps: never clamped from below
  ka.log_hi = std::log1p(eps);
  return launch_pair(ka, true, p.pred_dtype, p.latent_dtype, vec_ok, p.tune_threads, p.tune_cluster,
                     sm_count(), reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int psob200_online_pso_loss_grad(const psob200_schedule* sched, const psob200_online_pso_args* args,
                                            void* stream) {
  return online_pso_loss_grad(sched, args, nullptr, stream);
}

extern "C" int psob200_online_pso_loss_grad_scaled(const psob200_schedule* sched, const psob200_online_pso_args* args,
                                                   const psob200_loss_scaler* scaler, void* stream) {
  if (scaler == nullptr || scaler->scale == nullptr) return PSOB200_ERR_INVALID_ARG;
  return online_pso_loss_grad(sched, args, scaler->scale, stream);
}

static int dreambooth_pso_loss_grad(const psob200_dreambooth_args* args, const float* amp_scale, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_dreambooth_args& p = *args;
  if (p.b <= 0 || p.N <= 0 || !p.model_pred || !p.noisy || !p.target || !p.sigmas || !p.grad || !p.loss ||
      !p.workspace)
    return PSOB200_ERR_INVALID_ARG;
  if (p.loss_type != PSOB200_DB_PSO && p.loss_type != PSOB200_DB_PSO_DB) return PSOB200_ERR_INVALID_ARG;
  const bool has_ref = p.loss_type == PSOB200_DB_PSO;
  if (has_ref && !p.ref_pred) return PSOB200_ERR_INVALID_ARG;
  if (!valid_dtype(p.pred_dtype) || !valid_dtype(p.latent_dtype)) return PSOB200_ERR_DTYPE;
  if (p.workspace_bytes < psob200_pair_loss_workspace_bytes(p.b)) return PSOB200_ERR_WORKSPACE;
  if (!aligned16(p.workspace) || (p.stats != nullptr && !aligned16(p.stats))) return PSOB200_ERR_ALIGNMENT;
  const size_t ps = dtype_size(p.pred_dtype), ls = dtype_size(p.latent_dtype);
  const size_t half_p = (size_t)p.b * (size_t)p.N * ps, half_l = (size_t)p.b * (size_t)p.N * ls;
  bool vec_ok = (p.N % 8) == 0;
  PairKernelArgs ka = {};
  for (int k = 0; k < 2; ++k) {  // branch 0 = win rows [0,b), branch 1 = lose rows [b,2b)   (P:1891 chunk(2))
    ka.pred[k] = reinterpret_cast<const unsigned char*>(p.model_pred) + k * half_p;
    ka.ref[k] = has_ref ? reinterpret_cast<const unsigned char*>(p.ref_pred) + k * half_p : nullptr;
    ka.x[k] = reinterpret_cast<const unsigned char*>(p.noisy) + k * half_l;
    ka.xn[k] = reinterpret_cast<const unsigned char*>(p.target) + k * half_l;
    ka.grad[k] = reinterpret_cast<unsigned char*>(p.grad) + k * half_p;
    for (int j = 0; j < 4; ++j) ka.stride[j][k] = p.N;
    vec_ok = vec_ok && aligned16(ka.pred[k]) && (!has_ref || aligned16(ka.ref[k])) && aligned16(ka.x[k]) &&
             aligned16(ka.xn[k]) && aligned16(ka.grad[k]);
  }
  ka.sigmas = p.sigmas;
  ka.loss = p.loss; ka.stats = p.stats; ka.status = p.status;
  ka.counter = reinterpret_cast<unsigned int*>(p.workspace);
  ka.pair_loss = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(p.workspace) + 16);
  ka.amp_scale = amp_scale;
  ka.B = p.b; ka.N = p.N;
  ka.mode = has_ref ? kModeDbPso : kModeDbPsoDb;
  ka.beta = p.beta_pso; ka.nu = p.neg_defactor; ka.lam = p.prior_loss_weight; ka.loss_scale = p.loss_scale;
  return launch_pair(ka, has_ref, p.pred_dtype, p.latent_dtype, vec_ok, p.tune_threads, p.tune_cluster,
                     sm_count(), reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int psob200_dreambooth_pso_loss_grad(const psob200_dreambooth_args* args, void* stream) {
  return dreambooth_pso_loss_grad(args, nullptr, stream);
}

extern "C" int psob200_dreambooth_pso_loss_grad_scaled(const psob200_dreambooth_args* args,
                                                       const psob200_loss_scaler* scaler, void* stream) {
  if (scaler == nullptr || scaler->scale == nullptr) return PSOB200_ERR_INVALID_ARG;
  return dreambooth_pso_loss_grad(args, scaler->scale, stream);
}
