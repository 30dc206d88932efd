// Fast path of the fused pair-loss kernel, third design: residuals parked in TENSOR MEMORY.
//
// The two-pass structure (all 8N inputs of a pair must be reduced before any of its 2N gradient elements can be
// written) needs 2N fp32 residuals of on-chip storage per pair.  Registers force few warps per SM and shared memory
// competes with the load pipeline (profiles/r01_pair_loss.md: 16 warps/SM, SM-bound at 45-57 % of HBM).  Blackwell has
// a third on-chip memory that this kernel otherwise leaves idle: 256 KB of tensor memory per SM.  Every thread parks
// its residuals there with tcgen05.st (one instruction per 8-element chunk) and reads them back with tcgen05.ld for
// the gradient pass.  That frees
//   * the register file: 1024 threads per SM at <= 64 registers (32 warps hide the latencies), and
//   * all of shared memory for a deep cp.async ring (192 KB in flight per SM) in which every thread fetches and later
//     reads ONLY ITS OWN 16-byte pieces: no mbarrier, no producer role, no block barrier on the load path
//     (cp.async.wait_group is per thread),
// and shrinks the cluster: a pair of 4x128x128 latents fits two CTAs (148 SMs busy instead of 120), 4x64x64 fits one.
//
// Per pair: pass 1 (stream, residuals -> TMEM, 6 partial sums), block (+ cluster) reduction, the pair's scalar
// function on one thread, pass 2 (TMEM -> g*r -> global).  The ring runs ahead across pairs, so HBM stays busy while a
// pair is being finished.  Deterministic: fixed summation order, no atomics on the data path.
//
// Included by pair_loss.cu (needs PairKernelArgs and the shared helpers).
#pragma once

namespace psob200 {

constexpr int kTabPairs = 64;  // per-pair coefficients (fp64, dependent schedule-table loads) are resolved for 64 pairs at a time

struct PairEntry {
  StepCoef c[2];
  float h[2];
};

// fp32 evaluation of the pair's scalar function from values in registers / shared memory only.  Every lane of
// every warp of every CTA of the cluster runs it on identical inputs, so they all obtain the same multipliers.
// S = {S_pol0, S_ref0, D0, S_pol1, S_ref1, D1}.  Returns the per-pair loss term; stats (8 floats) when asked.
__device__ __forceinline__ float pair_scalar_function_fast(const PairKernelArgs& a, const float (&S)[6],
                                                           const PairEntry& e, float& g0, float& g1, float (&st)[8]) {
  const StepCoef c0 = e.c[0], c1 = e.c[1];
  const float i0 = c0.inv_2s2n, i1 = c1.inv_2s2n;
  const float invB = 1.0f / (float)a.B;
  float per;
#pragma unroll
  for (int i = 0; i < 8; ++i) st[i] = 0.f;
  if (a.mode == kModeOnline) {
    const float kHalfLog2Pi = 0.918938533204672742f;
    const float d0 = S[2] * i0, d1 = S[5] * i1;  // delta_k = logp_pol,k - logp_ref,k
    const float lo = (float)a.log_lo, hi = (float)a.log_hi;
    const bool open0 = (d0 >= lo) && (d0 <= hi), open1 = (d1 >= lo) && (d1 <= hi);
    const float lr0 = open0 ? d0 : (d0 < lo ? lo : (d0 > hi ? hi : d0));  // log clamp(exp d, 1-eps, 1+eps); NaN propagates
    const float lr1 = open1 ? d1 : (d1 < lo ? lo : (d1 > hi ? hi : d1));
    const float z = a.beta * (e.h[0] * lr0 + e.h[1] * lr1);  // T:847-850
    const float ez = expf(-fabsf(z));
    per = log1pf(ez) + fmaxf(-z, 0.f);                           // softplus(-z) = -log sigmoid(z)
    const float sig_neg = (z >= 0.f ? ez : 1.0f) / (1.0f + ez);  // sigmoid(-z), overflow-free
    const float common = -sig_neg * invB * a.beta * a.loss_scale;
    g0 = open0 ? common * e.h[0] * c0.a_over_s2n : 0.f;  // torch.clamp passes grad on the closed interval
    g1 = open1 ? common * e.h[1] * c1.a_over_s2n : 0.f;
    if (z != z) per = z;
    st[0] = -S[0] * i0 - c0.log_s - kHalfLog2Pi;  // TS:108-114 / DS:129-135
    st[1] = -S[1] * i0 - c0.log_s - kHalfLog2Pi;
    st[2] = -S[3] * i1 - c1.log_s - kHalfLog2Pi;
    st[3] = -S[4] * i1 - c1.log_s - kHalfLog2Pi;
    st[4] = d0; st[5] = d1; st[6] = z; st[7] = per;
  } else {
    const float nu = a.nu, beta = a.beta;
    const float lam = a.lam > 0.f ? a.lam : 0.f;              // P:1932
    const float Lw = 2.0f * S[0] * i0, Ll = 2.0f * S[3] * i1;  // P:1885-1891
    float logits, dl;
    if (a.mode == kModeDbPso) {
      logits = 2.0f * S[2] * i0 - nu * (2.0f * S[5] * i1);  // (Lref_w-L_w) - nu (Lref_l-L_l)   P:1919
      const float z = beta * logits;
      const float ez = expf(-fabsf(z));
      per = log1pf(ez) + fmaxf(-z, 0.f);  // P:1925
      const float sig_neg = (z >= 0.f ? ez : 1.0f) / (1.0f + ez);
      dl = -beta * sig_neg * invB;
      if (z != z) per = z;
      st[2] = 2.0f * S[1] * i0;
      st[3] = 2.0f * S[4] * i1;
    } else {
      logits = -(Lw - nu * Ll);  // P:1922
      const float m = 1.0f - beta * logits;
      per = m > 0.f ? m : (m == m ? 0.f : m);  // relu, NaN propagates   P:1927
      dl = m > 0.f ? -beta * invB : 0.f;
    }
    per += lam * Ll;  // P:1932-1935
    const float Gw = -dl, Gl = nu * dl + lam * invB;
    g0 = a.loss_scale * Gw * (-2.0f * c0.a_over_s2n);
    g1 = a.loss_scale * Gl * (-2.0f * c1.a_over_s2n);
    st[0] = Lw; st[1] = Ll; st[4] = logits; st[5] = per;
  }
  return per;
}


constexpr int kV3SmemRing = 192 * 1024;
constexpr int kV3TmemCols = 512;

__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
// 32 lanes x 8 consecutive 32-bit columns of tensor memory <-> 8 registers per thread.  SASS: STTM / LDTM
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
               "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
               "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Residual and partial sums in the "u form": with u = eps_pol - eps_ref the reference-branch residual is r + a*u, so
//   S_ref = S_pol + D,   D = a * (2 * sum(u r) + a * sum(u^2))
// needs only sum(r^2), sum(u r), sum(u^2): 6 instead of 9 flops per element, and D is still formed from the (small)
// prediction difference itself, never by cancelling the two large sums.
template <bool HAS_REF>
__device__ __forceinline__ void residual8_u(const float (&vx)[8], const float (&vn)[8], const float (&vp)[8],
                                            const float (&vr)[8], float kx, float ca, float (&r)[8], float& s_t,
                                            float& s_ur, float& s_uu) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float rt = fmaf(-ca, vp[i], fmaf(-kx, vx[i], vn[i]));
    r[i] = rt;
    s_t = fmaf(rt, rt, s_t);
    if constexpr (HAS_REF) {
      const float u = vp[i] - vr[i];
      s_ur = fmaf(u, rt, s_ur);
      s_uu = fmaf(u, u, s_uu);
    }
  }
}

// ---- packed fp32 pairs (sm_100 FFMA2 / FADD2 / FMUL2): two lanes per instruction, each lane rounds like the scalar op
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("sub.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// residual8_u on packed pairs: 24 instead of 48 floating-point instructions per 8-element chunk.  The three sums are
// kept as (even-element, odd-element) lane pairs and folded by the caller.
template <bool HAS_REF>
__device__ __forceinline__ void residual8_u2(const float (&vx)[8], const float (&vn)[8], const float (&vp)[8],
                                             const float (&vr)[8], f32x2 nkx, f32x2 nca, float (&r)[8], f32x2& s_t,
                                             f32x2& s_ur, f32x2& s_uu) {
#pragma unroll
  for (int i = 0; i < 8; i += 2) {
    const f32x2 p2 = pack2(vp[i], vp[i + 1]);
    const f32x2 rt = fma2(nca, p2, fma2(nkx, pack2(vx[i], vx[i + 1]), pack2(vn[i], vn[i + 1])));
    unpack2(rt, r[i], r[i + 1]);
    s_t = fma2(rt, rt, s_t);
    if constexpr (HAS_REF) {
      const f32x2 u = sub2(p2, pack2(vr[i], vr[i + 1]));
      s_ur = fma2(u, rt, s_ur);
      s_uu = fma2(u, u, s_uu);
    }
  }
}

template <typename TP, typename TL, bool HAS_REF>
struct V3Cfg {
  static constexpr int kNPred = HAS_REF ? 2 : 1;
  static constexpr int kBytesL = 8 * (int)sizeof(TL);  // one 8-element chunk of one latent tensor
  static constexpr int kBytesP = 8 * (int)sizeof(TP);
  static constexpr int kThreadBytes = 2 * kBytesL + kNPred * kBytesP;  // bf16/bf16: 64, fp32 preds + bf16 latents: 96
  static constexpr int kThreads = kThreadBytes <= 64 ? 1024 : 512;
  static constexpr int kSlotBytes = kThreads * kThreadBytes;
  static constexpr int kDepthRaw = kV3SmemRing / kSlotBytes;
  static constexpr int kDepth = kDepthRaw > 4 ? 4 : kDepthRaw;  // ring slots = chunk-iterations in flight
  static constexpr int kSmemBytes = kDepth * kSlotBytes;
  static constexpr int kWarpGroups = kThreads / 128;
  static constexpr int kMaxIters = kV3TmemCols / (8 * kWarpGroups);  // chunk-iterations per pair that fit in TMEM
  // tensor offsets inside a ring slot ([tensor][16-byte piece][thread])
  static constexpr int kOffX = 0;
  static constexpr int kOffXn = kThreads * kBytesL;
  static constexpr int kOffP = 2 * kThreads * kBytesL;
  static constexpr int kOffR = kOffP + kThreads * kBytesP;
};

// this thread's 8 elements of one tensor out of a ring slot (pieces of 16 bytes, thread-interleaved: conflict-free)
template <typename T, int kThreads>
__device__ __forceinline__ void lds_chunk(const unsigned char* sub, int tid, float (&v)[8]) {
  if constexpr (sizeof(T) == 4) {
    const float4 a = reinterpret_cast<const float4*>(sub)[tid], b = reinterpret_cast<const float4*>(sub)[kThreads + tid];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
    typename Vec8<T>::Raw raw{reinterpret_cast<const uint4*>(sub)[tid]};
    Vec8<T>::decode(raw, v);
  }
}

template <typename TP, typename TL, bool HAS_REF>
__global__ void __launch_bounds__(V3Cfg<TP, TL, HAS_REF>::kThreads, 1) pair_loss_grad_tmem_kernel(const PairKernelArgs a) {
  using Cfg = V3Cfg<TP, TL, HAS_REF>;
  constexpr int T = Cfg::kThreads;
  constexpr int D = Cfg::kDepth;
  constexpr int kWarps = T / 32;
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned C = cluster.num_blocks();
  const unsigned rank = cluster.block_rank();
  const long long cluster_id = blockIdx.x / C, n_clusters = gridDim.x / C;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  extern __shared__ __align__(128) unsigned char ring[];
  __shared__ float s_warp[kWarps][8];
  __shared__ __align__(16) float s_xch[2][kMaxCluster][8];  // CTA partial sums of the cluster, double-buffered by pair parity
  __shared__ float s_g[2];
  __shared__ PairEntry s_tab[2][kTabPairs];
  __shared__ uint32_t s_tmem_base;

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(&s_tmem_base)),
                 "n"(kV3TmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  // this thread's TMEM window: lanes 32*(warp%4).., columns of its warp group
  const uint32_t tmem_mine = s_tmem_base + ((uint32_t)((warp & 3) * 32) << 16);

  // ---- this CTA's slab of every sample: chunks [cbeg, cend) of each branch; Ib chunk-iterations per branch
  const int cpc = a.chunks_per_cta;
  const long long nchunk = a.N / 8;
  const long long cbeg = (long long)rank * cpc;
  const long long cend = (cbeg + cpc < nchunk) ? cbeg + cpc : nchunk;
  const int Ib = (cpc + T - 1) / T;  // host guarantees 2*Ib <= kMaxIters
  const int I = 2 * Ib;
  const uint32_t col0 = (uint32_t)((warp >> 2) * I * 8);
  const long long my_pairs = cluster_id < a.B ? (a.B - cluster_id + n_clusters - 1) / n_clusters : 0;
  const long long total = my_pairs * I;  // chunk-iterations of this CTA

  const int mine = cend > cbeg ? (int)(cend - cbeg) : 0;  // chunks per branch in this CTA's slab

  // ---- load cursor: the next chunk-iteration to fetch, kept incrementally (no divisions, no 64-bit per-thread
  // arithmetic on the hot path).  Addresses = CTA-uniform base of (pair, branch, tensor, slab) + 32-bit thread offset.
  long long c_it = 0;                  // pair ordinal of the cursor
  int c_j = 0, c_k = 0, c_slot = 0;    // chunk-iteration inside the branch, branch, ring slot
  int c_lc = tid;                      // this thread's chunk inside the slab for the cursor's iteration
  const unsigned char *ub_x = nullptr, *ub_n = nullptr, *ub_p = nullptr, *ub_r = nullptr;
  auto set_bases = [&]() {  // CTA-uniform
    const long long pair = cluster_id + c_it * n_clusters;
    const int k = c_k;
    ub_x = reinterpret_cast<const unsigned char*>(reinterpret_cast<const TL*>(a.x[k]) + pair * a.stride[2][k] + cbeg * 8);
    ub_n = reinterpret_cast<const unsigned char*>(reinterpret_cast<const TL*>(a.xn[k]) + pair * a.stride[3][k] + cbeg * 8);
    ub_p = reinterpret_cast<const unsigned char*>(reinterpret_cast<const TP*>(a.pred[k]) + pair * a.stride[0][k] + cbeg * 8);
    if constexpr (HAS_REF)
      ub_r = reinterpret_cast<const unsigned char*>(reinterpret_cast<const TP*>(a.ref[k]) + pair * a.stride[1][k] + cbeg * 8);
  };
  if (my_pairs > 0) set_bases();
  const uint32_t ring_base = (uint32_t)__cvta_generic_to_shared(ring) + (uint32_t)tid * 16u;
  auto issue = [&]() {  // start this thread's copies of the cursor's chunk-iteration (always commits a group)
    if (c_it < my_pairs) {
      const bool in = c_lc < mine;
      const uint32_t nb = in ? 16u : 0u;  // beyond the slab: zero-fill (src-size 0), address clamped to the slab start
      const uint32_t lc = in ? (uint32_t)c_lc : 0u;
      const uint32_t offL = lc * (uint32_t)Cfg::kBytesL, offP = lc * (uint32_t)Cfg::kBytesP;
      const uint32_t dst = ring_base + (uint32_t)c_slot * (uint32_t)Cfg::kSlotBytes;
      cp_async_16(dst + Cfg::kOffX, ub_x + offL, nb);
      if constexpr (sizeof(TL) == 4) cp_async_16(dst + Cfg::kOffX + T * 16u, ub_x + offL + 16, nb);
      cp_async_16(dst + Cfg::kOffXn, ub_n + offL, nb);
      if constexpr (sizeof(TL) == 4) cp_async_16(dst + Cfg::kOffXn + T * 16u, ub_n + offL + 16, nb);
      cp_async_16(dst + Cfg::kOffP, ub_p + offP, nb);
      if constexpr (sizeof(TP) == 4) cp_async_16(dst + Cfg::kOffP + T * 16u, ub_p + offP + 16, nb);
      if constexpr (HAS_REF) {
        cp_async_16(dst + Cfg::kOffR, ub_r + offP, nb);
        if constexpr (sizeof(TP) == 4) cp_async_16(dst + Cfg::kOffR + T * 16u, ub_r + offP + 16, nb);
      }
      c_lc += T;
      if (++c_j == Ib) {  // next branch / next pair (uniform branch, taken once per Ib iterations)
        c_j = 0;
        c_lc = tid;
        if (++c_k == 2) { c_k = 0; ++c_it; }
        if (c_it < my_pairs) set_bases();
      }
      if (++c_slot == D) c_slot = 0;
    }
    cp_async_commit();
  };

#pragma unroll
  for (int d = 0; d < D; ++d) issue();

  double loss_acc = 0.0;  // rank 0, thread 0
  int slot_i = 0;         // ring slot of the chunk-iteration being consumed
  for (long long it = 0; it < my_pairs; ++it) {
    const long long pair = cluster_id + it * n_clusters;
    const int tb = (int)((it / kTabPairs) & 1), slot_t = (int)(it % kTabPairs);
    if (slot_t == 0) {  // per-pair scalars of the next kTabPairs pairs, resolved in parallel (fp64, table look-ups)
      __syncthreads();
      if (tid < 2 * kTabPairs && it + (tid >> 1) < my_pairs) {
        const long long p = pair + (long long)(tid >> 1) * n_clusters;
        const int k = tid & 1;
        resolve_pair_coefs(a, p, k, &s_tab[tb][tid >> 1].c[k]);
        s_tab[tb][tid >> 1].h[k] = a.mode == kModeOnline ? a.human_prefer[p * 2 + k] : 0.f;
      }
      __syncthreads();
    }
    const PairEntry& ent = s_tab[tb][slot_t];

    // ------------------------------------------------------------------ pass 1
    float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    uint32_t tcol = tmem_mine + col0;
#pragma unroll 1
    for (int k = 0; k < 2; ++k) {
      const f32x2 nkx = pack2(-ent.c[k].k, -ent.c[k].k), nca = pack2(-ent.c[k].a, -ent.c[k].a);
      f32x2 s_t2 = 0ull, s_r2 = 0ull, s_d2 = 0ull;  // (+0.0f, +0.0f)
#pragma unroll 1
      for (int j = 0; j < Ib; ++j) {
        cp_async_wait<D - 1>();  // this thread's pieces of the oldest chunk-iteration in flight have landed
        const unsigned char* slot = ring + (size_t)slot_i * Cfg::kSlotBytes;
        float vx[8], vn[8], vp[8], vr[8], r[8];
        lds_chunk<TL, T>(slot + Cfg::kOffX, tid, vx);
        lds_chunk<TL, T>(slot + Cfg::kOffXn, tid, vn);
        lds_chunk<TP, T>(slot + Cfg::kOffP, tid, vp);
        if constexpr (HAS_REF) lds_chunk<TP, T>(slot + Cfg::kOffR, tid, vr);
        residual8_u2<HAS_REF>(vx, vn, vp, vr, nkx, nca, r, s_t2, s_r2, s_d2);  // (sum r^2, sum u r, sum u^2); zero-filled chunks add 0
        issue();  // refill the slot just drained (its values are in registers)
        tmem_st8(tcol, r);
        tcol += 8u;
        if (++slot_i == D) slot_i = 0;
      }
      float lo, hi, s_t, s_r, s_d;
      unpack2(s_t2, lo, hi); s_t = lo + hi;
      unpack2(s_r2, lo, hi); s_r = lo + hi;
      unpack2(s_d2, lo, hi); s_d = lo + hi;
      if (k == 0) { acc[0] = s_t; acc[1] = s_r; acc[2] = s_d; }  // (no runtime-indexed register array)
      else        { acc[3] = s_t; acc[4] = s_r; acc[5] = s_d; }
    }
    // ------------------------------------------------------------------ reduce: warp -> CTA -> cluster
#pragma unroll
    for (int j = 0; j < 6; ++j) acc[j] = warp_sum(acc[j]);
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < 6; ++j) s_warp[warp][j] = acc[j];
    }
    tmem_st_wait();
    __syncthreads();
    const int par = (int)(it & 1);
    if (warp == 0) {
      float part[6];
#pragma unroll
      for (int j = 0; j < 6; ++j) part[j] = warp_sum(lane < kWarps ? s_warp[lane][j] : 0.f);
      if (C == 1) {
        if (lane == 0) {
#pragma unroll
          for (int j = 0; j < 6; ++j) s_xch[par][0][j] = part[j];
        }
      } else if (lane < (int)C) {  // lane r pushes this CTA's partials into CTA r
        float* dst = cluster.map_shared_rank(&s_xch[par][rank][0], lane);
#pragma unroll
        for (int j = 0; j < 6; ++j) dst[j] = part[j];
      }
    }
    if (C > 1) cluster.sync();  // release/acquire: every CTA's partials are visible everywhere
    if (tid == 0) {
      float S[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (unsigned r = 0; r < C; ++r)  // rank order: identical in all CTAs
#pragma unroll
        for (int j = 0; j < 6; ++j) S[j] += s_xch[par][r][j];
#pragma unroll
      for (int k = 0; k < 2; ++k) {  // u form -> (S_pol, S_ref, D)
        const float ca = ent.c[k].a;
        const float d = ca * fmaf(ca, S[3 * k + 2], 2.f * S[3 * k + 1]);
        S[3 * k + 1] = S[3 * k] + d;
        S[3 * k + 2] = d;
      }
      float g0, g1, st[8];
      const float per = pair_scalar_function_fast(a, S, ent, g0, g1, st);
      if (a.amp_scale != nullptr) {  // device loss scale: the gradient is scaled before it is rounded to TP
        const float amp = *a.amp_scale;
        g0 *= amp;
        g1 *= amp;
      }
      s_g[0] = g0;
      s_g[1] = g1;
      if (rank == 0) {
        loss_acc += (double)per;
        if (a.stats != nullptr) {
          float4* dst = reinterpret_cast<float4*>(a.stats + pair * 8);
          dst[0] = make_float4(st[0], st[1], st[2], st[3]);
          dst[1] = make_float4(st[4], st[5], st[6], st[7]);
        }
      }
    }
    __syncthreads();
    // ------------------------------------------------------------------ pass 2: grad = g_k * r from tensor memory
    tcol = tmem_mine + col0;
#pragma unroll 1
    for (int k = 0; k < 2; ++k) {
      const float gk = s_g[k];
      const f32x2 gk2 = pack2(gk, gk);
      TP* gp = reinterpret_cast<TP*>(a.grad[k]) + pair * a.N + (cbeg + tid) * 8;
      int lc = tid;
#pragma unroll 1
      for (int j = 0; j < Ib; ++j, lc += T, gp += T * 8, tcol += 8u) {
        float r[8];
        tmem_ld8(tcol, r);
        if (lc < mine) {
          float o[8];
#pragma unroll
          for (int e = 0; e < 8; e += 2) unpack2(mul2(gk2, pack2(r[e], r[e + 1])), o[e], o[e + 1]);
          Vec8<TP>::store(gp, o);
        }
      }
    }
    // s_g / s_warp are rewritten only after the next pair's first __syncthreads: every thread has read them by then
  }
  cp_async_wait<0>();

  // ---- mean over pairs: one ticket per cluster; the last cluster sums the per-cluster sums in a fixed order
  if (rank == 0 && warp == 0 && my_pairs > 0) {
    unsigned ticket = 0;
    if (lane == 0) {
      reinterpret_cast<volatile float*>(a.pair_loss)[cluster_id] = (float)loss_acc;
      __threadfence();
      ticket = atomicAdd(a.counter, 1u);
    }
    ticket = __shfl_sync(0xffffffffu, ticket, 0);
    const long long active = a.B < n_clusters ? a.B : n_clusters;
    if (ticket == (unsigned)(active - 1)) {
      __threadfence();
      double s = 0.0;
      for (long long i = lane; i < active; i += 32) s += (double)__ldcg(a.pair_loss + i);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) {
        a.loss[0] = (float)((double)a.loss_scale * s / (double)a.B);
        *a.counter = 0u;
      }
    }
  }
  if (C > 1) cluster.sync();  // nobody leaves while a neighbour may still write its shared memory
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s_tmem_base), "n"(kV3TmemCols) : "memory");
  }
}

}  // namespace psob200
