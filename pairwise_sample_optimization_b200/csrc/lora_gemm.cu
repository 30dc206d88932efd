// LoRA projection GEMMs on the 5th-generation tensor cores (sm_100a): TMA-fed tcgen05.mma with the
// accumulators in tensor memory.
//
// One persistent, warp-specialised kernel runs a short LIST OF PROBLEMS per launch; each problem is
//
//     D[M,N] = alpha * sum_s  A_s[M,K_s] * B_s[N,K_s]^T  + bias[N]              (up to 4 reduction segments)
//
// * Two segments make the LoRA-wrapped projection ONE tensor-core pass over the frozen weight instead of the reference
//   stack's three GEMMs + scale + add (peft lora.Linear.forward, reached from train_online_pso_sdxl_turbo.py:338-345):
//   y = x W^T + b + (s x A^T) B^T  is  [x | T] [W | B]^T  with  T = s x A^T.
// * Several problems in one launch + a flag per row block make T a tile of the SAME launch: the tiles of the skinny
//   problem T = s x A^T come first in the tile list and release flags[m_blk] when their rows are stored; a tile of the
//   main problem waits for its flag only before the first TMA load of the adapter segment.  All CTAs of the persistent
//   grid are co-resident, so the wait cannot deadlock.  The backward uses the same scheme (U = s dY B, then
//   dX = dY W + U A); the weight gradients dA = U^T X and dB = dY^T T run as independent problems of one launch.
// * Projections that share their input (attention to_q / to_k / to_v, cross-attention to_k / to_v) are STACKED: one
//   problem over the concatenated weight [G N, K] whose adapter segment reads column group g of the stacked T, and in
//   the backward one dX problem whose segments walk the G gradients.
//
// Warp roles (256 threads, 1 CTA per SM, grid = min(tiles, SMs), static round-robin tile schedule):
//   warp 0      TMA producer: 128B-swizzled [128 x 64] A and [bn x 64] B boxes into a ring of stages
//   warp 1      MMA issuer: one thread, 4 x tcgen05.mma (128 x bn x 16) per stage, tcgen05.commit frees the stage
//   warp 2      tensor-memory allocator (512 columns = two accumulator buffers of <= 256 columns)
//   warps 4-7   epilogue: tcgen05.ld 32x32b -> alpha, bias, convert -> global (also a transposed copy, or
//               fp32 atomic accumulation for the split reductions); overlaps the next tile's MMAs.
#include <atomic>
#include <cstdlib>
#include <type_traits>
#include <mutex>

#include "common.cuh"
#include "ptx_sm100.cuh"

namespace psob200 {

constexpr int kBM = 128;            // UMMA M: rows of an output tile
constexpr int kBNMax = 256;         // widest UMMA N
constexpr int kBK = 64;             // reduction elements per stage = one 128-byte swizzle span of a 16-bit type
constexpr int kStages = 4;          // with the widest tile; narrower tiles get more (up to kMaxStages)
constexpr int kMaxStages = 8;
constexpr int kGemmThreads = 256;
constexpr int kStageABytes = kBM * kBK * 2;      // 16 KB
constexpr int kStageBBytes = kBNMax * kBK * 2;   // 32 KB
constexpr int kEpiStageDBytes = 32 * 128;         // output staging per epilogue warp: [32 rows][128 B] for the row-major output
constexpr int kEpiStageBytesPerWarp = kEpiStageDBytes + 32 * 64;  // + [32 columns][32 rows x 2 B] for the transposed copy
constexpr int kGemmSmemBytes = kStages * (kStageABytes + kStageBBytes) + 4 * kEpiStageBytesPerWarp + 1024;  // + 1024 B alignment slack
constexpr int kTmemCols = 512;

constexpr int kMaxSeg = 4;    // reduction segments per problem
constexpr int kMaxProb = 4;   // problems per launch
constexpr int kMaxMaps = 8;   // tensor maps per launch

struct GemmMaps {
  CUtensorMap m[kMaxMaps];
};

// One GEMM of the launch.  Tiles [tile0, tile0 + m_tiles * n_tiles * splits) of the launch's tile list belong to it,
// n fastest, then m, then the split of the reduction.
struct GemmProblem {
  long long M, N;           // output extent
  void* d;                  // row-major output [M, N] (may be null)
  void* dt;                 // transposed output [N, M] (may be null)
  const void* bias;
  long long ldd, lddt;
  long long group_n;        // stacked projections: output columns per group (>= N: one group); a tile never straddles groups
  int tile0, m_tiles, n_tiles, tiles_per_group, splits, kb_per_split;
  int bn;                   // tile width, multiple of 16, <= 256
  int n_seg, nk_total;
  int nk[kMaxSeg];          // 64-wide k-blocks per segment
  int map_a[kMaxSeg], map_b[kMaxSeg];
  int a_koff[kMaxSeg];      // A box: constant element offset along k (a column slice of a stacked buffer) ...
  int a_gkoff[kMaxSeg];     // ... plus this per column group of the tile (group g of the stacked T / U)
  int b_off[kMaxSeg];       // B box: constant offset along its row axis (the n coordinate; the k coordinate if B is reduction-major)
  float alpha;
  int bias_dtype;
  int m_fast;               // tile order: row blocks vary fastest (consecutive tiles share their B rows), else column tiles do
  int signal;               // != 0: every tile releases flags[m_blk] once its rows are stored
  int wait_seg, wait_count; // wait_seg >= 0: the first load of that segment waits until wait_count tiles released flags[m_blk]
};

struct GemmLaunch {
  GemmProblem prob[kMaxProb];
  int n_prob;
  int total_tiles;
  int ab_format, a_mn, b_mn, atomic, diag;
  int n_acc, acc_stride;    // CTA-pair kernel: tensor-memory accumulators and their column stride (2 x 256 or 3 x 160)
  int stages;               // even; stage = 16 KB of A + stage_b_bytes of B
  int stage_b_bytes;        // of the widest problem
  int pdl;                  // programmatic dependent launch role bits (psob200_gemm_args.pdl)
  int* flags;               // n_flags row-block counters + 1 exit ticket, zero on entry, zeroed again by the last CTA
  int n_flags;
};

struct TileInfo {
  int p, m_blk, group, kb0, kb1;
  long long n0, n_end;
};

__device__ __forceinline__ void decode_tile(const GemmLaunch& L, int t, TileInfo& ti) {
  int p = 0;
  while (p + 1 < L.n_prob && t >= L.prob[p + 1].tile0) ++p;
  const GemmProblem& P = L.prob[p];
  int loc = t - P.tile0;
  int n_blk, split;
  ti.p = p;
  if (P.m_fast) {
    ti.m_blk = loc % P.m_tiles;
    loc /= P.m_tiles;
    n_blk = loc % P.n_tiles;
    split = loc / P.n_tiles;
  } else {
    n_blk = loc % P.n_tiles;
    loc /= P.n_tiles;
    ti.m_blk = loc % P.m_tiles;
    split = loc / P.m_tiles;
  }
  ti.kb0 = split * P.kb_per_split;
  ti.kb1 = ti.kb0 + P.kb_per_split < P.nk_total ? ti.kb0 + P.kb_per_split : P.nk_total;
  ti.group = n_blk / P.tiles_per_group;
  ti.n0 = (long long)ti.group * P.group_n + (long long)(n_blk - ti.group * P.tiles_per_group) * P.bn;
  long long e = ti.n0 + P.bn;                         // a tile stops at the end of its column group and at N
  const long long ge = (long long)(ti.group + 1) * P.group_n;
  if (e > ge) e = ge;
  if (e > P.N) e = P.N;
  ti.n_end = e;
}

// Spin until `count` releases have reached *flag (acquire), then order the TMA (async proxy) reads behind it.
__device__ __forceinline__ void wait_flag(const int* flag, int count) {
  int v;
  do {
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
  } while (v < count);
  asm volatile("fence.proxy.async;" ::: "memory");
}

template <typename T>
__device__ __forceinline__ T cvt_out(float v);
template <> __device__ __forceinline__ float cvt_out<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 cvt_out<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half cvt_out<__half>(float v) { return __float2half_rn(v); }

// bias[n0 .. n0+32) as fp32, zero beyond N.  One uniform branch per chunk, 128-bit loads for whole chunks.
template <typename TB>
__device__ __forceinline__ void load_bias32(const void* bias, long long n0, long long N, float (&b)[32]) {
  const TB* src = reinterpret_cast<const TB*>(bias) + n0;
  if (n0 + 32 <= N && (reinterpret_cast<uintptr_t>(src) & 15u) == 0) {
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      float t[8];
      if constexpr (sizeof(TB) == 4) {
        const float4 lo = __ldg(reinterpret_cast<const float4*>(src + j)), hi = __ldg(reinterpret_cast<const float4*>(src + j + 4));
        t[0] = lo.x; t[1] = lo.y; t[2] = lo.z; t[3] = lo.w; t[4] = hi.x; t[5] = hi.y; t[6] = hi.z; t[7] = hi.w;
      } else {
        const uint4 w4 = __ldg(reinterpret_cast<const uint4*>(src + j));
        typename Vec8<TB>::Raw raw{w4};
        Vec8<TB>::decode(raw, t);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) b[j + i] = t[i];
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) b[j] = (n0 + j < N) ? Vec8<TB>::load1(src + j) : 0.f;
  }
}

// Epilogue mode (compile time): bits 0-1 = outputs (1: row-major d only, 2: transposed dt only, 3: whichever pointers are
// set, checked at run time), bit 2 = a bias may be present, bit 3 = it has the output's element type.  The hot launches of
// the training step get exact modes so that their instruction footprint stays small; mode 7 is the general case.
constexpr int kEpiD = 1, kEpiDt = 2, kEpiAnyOut = 3, kEpiBias = 4, kEpiGeneral = 7;
constexpr int kEpiBiasSameType = 8 | kEpiBias;  // the bias has the output's element type (nn.Linear in one dtype)
constexpr int kEpiFused = kEpiAnyOut | kEpiBiasSameType;  // problem lists: outputs and bias differ per problem

// One 32-column chunk of one accumulator row: v[j] belongs to (row, n0 + j).
template <typename TD, bool kAtomic, int kMode>
__device__ __forceinline__ void store_chunk(const GemmProblem& p, const float (&v)[32], long long row, long long n0,
                                            long long n_end, bool do_d = true, bool do_dt = true) {
  if (row >= p.M) return;
  const long long nleft = n_end - n0;  // columns of this chunk that belong to this tile and exist
  if ((kMode & kEpiD) && do_d && ((kMode & 3) != kEpiAnyOut || p.d != nullptr)) {
    TD* dst = reinterpret_cast<TD*>(p.d) + row * p.ldd + n0;
    if constexpr (kAtomic) {
      float* acc = reinterpret_cast<float*>(dst);
      if (nleft >= 32 && (reinterpret_cast<uintptr_t>(acc) & 15u) == 0) {
        // a thread owns 32 consecutive floats of its row: 8 vector reductions instead of 32 scalar ones (each lane
        // of a scalar atomic touches a different row = a different sector: a quarter of the L2 operations)
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(acc + j), "f"(v[j]), "f"(v[j + 1]), "f"(v[j + 2]),
                       "f"(v[j + 3])
                       : "memory");
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j < nleft) atomicAdd(acc + j, v[j]);
      }
    } else if (nleft >= 32 && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
      if constexpr (sizeof(TD) == 4) {
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(reinterpret_cast<float*>(dst) + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      } else {
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          const float o[8] = {v[j], v[j + 1], v[j + 2], v[j + 3], v[j + 4], v[j + 5], v[j + 6], v[j + 7]};
          Vec8<TD>::store(dst + j, o);
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < nleft) dst[j] = cvt_out<TD>(v[j]);
    }
  }
  if ((kMode & kEpiDt) && do_dt && ((kMode & 3) != kEpiAnyOut || p.dt != nullptr)) {  // lanes hold consecutive rows: coalesced columns
    TD* dst = reinterpret_cast<TD*>(p.dt) + n0 * p.lddt + row;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (j < nleft) {
        if constexpr (kAtomic) atomicAdd(reinterpret_cast<float*>(dst) + (long long)j * p.lddt, v[j]);
        else dst[(long long)j * p.lddt] = cvt_out<TD>(v[j]);
      }
    }
  }
}

// ---- row-major output through shared memory.  A lane of an epilogue warp owns one accumulator ROW: stored directly, one
// instruction writes 16 bytes to each of 32 different lines (32 L1 transactions, half-filled sectors) -- measured, draining a
// 256 x 224 tile took 2.3 us with the stores and 0.5 us without (tools/diag_timeline.py), and the drain of the last tile of a CTA
// is never hidden.  Staged: the lane writes its 16-byte pieces into the warp's [32 rows][128 B] buffer (piece index XOR row & 7:
// conflict-free both ways), then the warp writes whole 128-byte (64-byte) row segments, 4 (8) rows per instruction.
template <typename TD>
__device__ __forceinline__ void stage_chunk(unsigned char* stg, int lane, int piece0, const float (&v)[32]) {
  constexpr int kPer = 16 / (int)sizeof(TD);  // elements per 16-byte piece
#pragma unroll
  for (int q = 0; q < 32 / kPer; ++q) {
    uint4 w;
    if constexpr (sizeof(TD) == 4) {
      w = make_uint4(__float_as_uint(v[4 * q]), __float_as_uint(v[4 * q + 1]), __float_as_uint(v[4 * q + 2]), __float_as_uint(v[4 * q + 3]));
    } else {
      uint32_t* pw = &w.x;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if constexpr (std::is_same<TD, __nv_bfloat16>::value) {
          const __nv_bfloat162 h2 = __floats2bfloat162_rn(v[8 * q + 2 * i], v[8 * q + 2 * i + 1]);
          pw[i] = *reinterpret_cast<const uint32_t*>(&h2);
        } else {
          const __half2 h2 = __floats2half2_rn(v[8 * q + 2 * i], v[8 * q + 2 * i + 1]);
          pw[i] = *reinterpret_cast<const uint32_t*>(&h2);
        }
      }
    }
    *reinterpret_cast<uint4*>(stg + lane * 128 + (((piece0 + q) ^ (lane & 7)) << 4)) = w;
  }
}

// write the staged rows: `kPieces` (4 or 8) 16-byte pieces per row starting at column n0
template <typename TD, int kPieces>
__device__ __forceinline__ void flush_staged(const GemmProblem& p, const unsigned char* stg, int lane, long long row0, long long n0) {
  constexpr int kPer = 16 / (int)sizeof(TD);
  __syncwarp();
  const int q = lane % kPieces;
  TD* dst = reinterpret_cast<TD*>(p.d) + n0 + q * kPer;
#pragma unroll
  for (int r = lane / kPieces; r < 32; r += 32 / kPieces) {
    const uint4 w = *reinterpret_cast<const uint4*>(stg + r * 128 + ((q ^ (r & 7)) << 4));
    if (row0 + r < p.M) stg_u4(dst + (row0 + r) * p.ldd, w);
  }
  __syncwarp();
}

// The transposed copy (16-bit outputs) of a whole 32 x 32 chunk through the second part of the staging buffer: direct, a lane
// issues 32 two-byte stores per chunk (measured: + 1.5 us on the drain of a 256 x 64 t tile -- which every main tile of its row
// block waits for); staged as [column][row], the warp writes each column's 64 bytes as 16-byte pieces, 8 columns per instruction.
template <typename TD>
__device__ __forceinline__ void store_chunk_t_staged(const GemmProblem& p, unsigned char* stg_t, int lane, const float (&v)[32],
                                                     long long row0, long long n0) {
#pragma unroll
  for (int j = 0; j < 32; ++j) reinterpret_cast<TD*>(stg_t + j * 64)[lane] = cvt_out<TD>(v[j]);
  __syncwarp();
  TD* dst = reinterpret_cast<TD*>(p.dt) + row0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int idx = i * 32 + lane, col = idx >> 2, part = idx & 3;
    const uint4 w = *reinterpret_cast<const uint4*>(stg_t + idx * 16);
    stg_u4(dst + (n0 + col) * p.lddt + part * 8, w);
  }
  __syncwarp();
}

// Drain one accumulator tile: TMEM -> registers (the load of chunk c+1 is in flight while chunk c is converted and
// stored) -> alpha, bias -> global (row-major output through the warp's staging buffer `stg` when one is given).
template <typename TD, bool kAtomic, int kMode>
__device__ __forceinline__ void epilogue_tile(const GemmProblem& p, int diag, uint32_t taddr, long long row, long long n_tile0,
                                              long long n_end, bool add_bias, unsigned char* stg = nullptr) {
  const int chunks = (p.bn + 31) / 32;
  const int lane = threadIdx.x & 31;
  const long long row0 = row - lane;
  // uniform over the warp: this tile's row-major output can take the staged path (16-byte aligned row segments)
  const bool stage_ok = !kAtomic && (kMode & kEpiD) && stg != nullptr && p.d != nullptr && !(diag & 2) &&
                        ((reinterpret_cast<uintptr_t>(reinterpret_cast<TD*>(p.d) + n_tile0) & 15u) == 0) &&
                        (((unsigned long long)p.ldd * sizeof(TD)) & 15u) == 0;
  const bool stage_t_ok = !kAtomic && (kMode & kEpiDt) && sizeof(TD) == 2 && stg != nullptr && p.dt != nullptr && !(diag & 2) &&
                          row0 + 32 <= p.M && ((reinterpret_cast<uintptr_t>(reinterpret_cast<TD*>(p.dt) + row0) & 15u) == 0) &&
                          (((unsigned long long)p.lddt * sizeof(TD)) & 15u) == 0;
  uint32_t raw[2][32];
  ptx::tmem_ld_32x32(taddr, raw[0]);
#pragma unroll 1
  for (int c = 0; c < chunks; c += 2) {
    long long pending_n0 = -1;  // 16-bit outputs: the first chunk of a 64-column unit is staged and waits for the second
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int cc = c + h;
      const long long n0 = n_tile0 + (long long)cc * 32;
      if (cc < chunks && n0 < n_end) {  // uniform over the warp
        ptx::tmem_ld_wait();
        if (cc + 1 < chunks) ptx::tmem_ld_32x32(taddr + (uint32_t)(cc + 1) * 32, raw[h ^ 1]);
        float v[32];
        if ((kMode & kEpiBias) && add_bias) {
          float b[32];
          if constexpr ((kMode & 8) != 0) load_bias32<TD>(p.bias, n0, p.N, b);
          else if (p.bias_dtype == PSOB200_F32) load_bias32<float>(p.bias, n0, p.N, b);
          else if (p.bias_dtype == PSOB200_BF16) load_bias32<__nv_bfloat16>(p.bias, n0, p.N, b);
          else load_bias32<__half>(p.bias, n0, p.N, b);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaf(p.alpha, __uint_as_float(raw[h][j]), b[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = p.alpha * __uint_as_float(raw[h][j]);
        }
        if (stage_ok && n0 + 32 <= n_end) {
          if constexpr (sizeof(TD) == 4) {
            stage_chunk<TD>(stg, lane, 0, v);
            flush_staged<TD, 8>(p, stg, lane, row0, n0);
          } else if (h == 0) {
            stage_chunk<TD>(stg, lane, 0, v);
            if (cc + 1 < chunks && n0 + 64 <= n_end) pending_n0 = n0;  // flushed together with the next chunk
            else flush_staged<TD, 4>(p, stg, lane, row0, n0);
          } else {  // h == 1: chunk h == 0 of this unit was whole, staged and is pending
            stage_chunk<TD>(stg, lane, 4, v);
            flush_staged<TD, 8>(p, stg, lane, row0, pending_n0);
            pending_n0 = -1;
          }
          if constexpr ((kMode & kEpiDt) != 0) {
            if (stage_t_ok) {
              if constexpr (sizeof(TD) == 2) store_chunk_t_staged<TD>(p, stg + kEpiStageDBytes, lane, v, row0, n0);
            } else {
              store_chunk<TD, kAtomic, kMode>(p, v, row, n0, n_end, false);
            }
          }
        } else if (!(diag & 2)) {
          if constexpr ((kMode & kEpiDt) != 0 && sizeof(TD) == 2) {
            if (stage_t_ok && n0 + 32 <= n_end) {
              store_chunk_t_staged<TD>(p, stg + kEpiStageDBytes, lane, v, row0, n0);
              store_chunk<TD, kAtomic, kMode>(p, v, row, n0, n_end, true, false);
            } else {
              store_chunk<TD, kAtomic, kMode>(p, v, row, n0, n_end);
            }
          } else {
            store_chunk<TD, kAtomic, kMode>(p, v, row, n0, n_end);
          }
        }
      }
    }
  }
  ptx::tmem_ld_wait();
}

// One instantiation per output type / accumulation mode: the four epilogues together made this kernel 259 KB of SASS, and
// a launch that finds its code evicted from the instruction caches (any launch inside the training step: LayerNorm, SDPA,
// cuBLAS kernels run in between) paid ~10 us for it (tools/diag_cold.py: 15.7 us back to back, 26.6 us with three other
// kernels in between, only 18.4 us with the OPERANDS evicted instead).
template <typename TD, bool kAtomic, int kMode>
__global__ void __launch_bounds__(kGemmThreads, 1)
lora_gemm_kernel(const __grid_constant__ GemmMaps maps, const __grid_constant__ GemmLaunch L) {
  extern __shared__ unsigned char gemm_smem_raw[];
  // one "full" barrier per stage, one "empty" barrier per PAIR of stages: tcgen05.commit costs several hundred
  // cycles of tensor-pipe command time, so the MMA warp commits every second k-block only
  __shared__ __align__(8) uint64_t full_bar[kMaxStages], empty_bar[kMaxStages / 2], tmem_full_bar[2], tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;

  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(gemm_smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* smem_a = smem;
  const int n_stages = L.stages;
  const int stage_b_bytes = L.stage_b_bytes;
  unsigned char* smem_b = smem + n_stages * kStageABytes;
  unsigned char* smem_epi = smem + kStages * (kStageABytes + kStageBBytes);  // behind the operand ring at its largest

  // the warp index through a shuffle is PROVABLY warp-uniform: ptxas then keeps the role loops (barrier phases, stage counters,
  // UMMA / TMA descriptors) on the uniform datapath instead of moving ~20 per-thread registers to uniform ones (R2UR) per k-block
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int total_tiles = L.total_tiles;

  if (warp == 0 && lane == 0) {
    for (int p = 0; p < L.n_prob; ++p)
      for (int s = 0; s < L.prob[p].n_seg; ++s) {
        ptx::prefetch_tensormap(&maps.m[L.prob[p].map_a[s]]);
        ptx::prefetch_tensormap(&maps.m[L.prob[p].map_b[s]]);
      }
  }
  if (warp == 1 && lane == 0) {
#pragma unroll
    for (int s = 0; s < kMaxStages; ++s) ptx::mbar_init(&full_bar[s], 1);  // producer's arrive.expect_tx; TMA completes the bytes
#pragma unroll
    for (int s = 0; s < kMaxStages / 2; ++s) ptx::mbar_init(&empty_bar[s], 1);  // tcgen05.commit
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full_bar[a], 1);   // tcgen05.commit after the tile's last MMA
      ptx::mbar_init(&tmem_empty_bar[a], 4);  // one arrival per epilogue warp
    }
    ptx::fence_mbar_init();
  }
  // primary of a programmatic dependent launch: the dependent grid (the main GEMM that needs this launch's output only
  // for its last k-blocks) may start filling the SMs this small grid leaves idle
  if (L.pdl & 1) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (warp == 2) ptx::tmem_alloc<kTmemCols>(&tmem_base_slot);
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_slot;

  // The producer and MMA loops run WARP-UNIFORMLY (all 32 lanes keep the loop state) and only the issuing
  // instructions are predicated on elect.sync: UTMALDG / UTCHMMA take uniform-register operands, and a loop that
  // only lane 0 executes makes ptxas wrap every one of them in an ELECT / R2UR.BROADCAST waterfall (measured:
  // ~450 cycles per k-block, more than the MMAs themselves).
  if (warp == 0) {
    // ================================================================= TMA producer
    int stage = 0;
    uint32_t phase = 0;
    bool dep_pending = (L.pdl & 2) != 0;  // launched ahead of the grid that produces segment 1's A (or, bit 2, any operand)
    if (dep_pending && (L.pdl & 4)) {
      asm volatile("griddepcontrol.wait;" ::: "memory");
      asm volatile("fence.proxy.async;" ::: "memory");
      dep_pending = false;
    }
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      TileInfo ti;
      decode_tile(L, t, ti);
      const GemmProblem& P = L.prob[ti.p];
      const uint32_t tx = ((L.diag & 8) ? 0u : (uint32_t)kStageABytes) + ((L.diag & 4) ? 0u : (uint32_t)P.bn * kBK * 2u);
      const int m0 = ti.m_blk * kBM, n0 = (int)ti.n0;
      // segment of the tile's first k-block
      int seg = 0, kbs = ti.kb0;
      while (kbs >= P.nk[seg]) { kbs -= P.nk[seg]; ++seg; }
      bool need_wait = P.wait_seg >= 0;
      for (int kb = ti.kb0; kb < ti.kb1; ++kb) {
        if ((stage & 1) == 0) ptx::mbar_wait(&empty_bar[stage >> 1], phase ^ 1u);  // the pair (stage, stage+1) is free
        if (seg >= 1 && dep_pending) {  // first read of the previous launch's output: wait for that grid, then fence the
          asm volatile("griddepcontrol.wait;" ::: "memory");  // generic-proxy writes against the TMA (async proxy) reads
          asm volatile("fence.proxy.async;" ::: "memory");
          dep_pending = false;
        }
        if (need_wait && seg >= P.wait_seg) {  // the operand of this segment is produced by other tiles of THIS launch
          wait_flag(L.flags + ti.m_blk, P.wait_count * 4);
          need_wait = false;
        }
        const CUtensorMap* ma = &maps.m[P.map_a[seg]];
        const CUtensorMap* mb = &maps.m[P.map_b[seg]];
        const int ka = kbs * kBK + P.a_koff[seg] + ti.group * P.a_gkoff[seg];
        const int kk = kbs * kBK;
        const int boff = P.b_off[seg];
        unsigned char* sa = smem_a + stage * kStageABytes;
        unsigned char* sb = smem_b + stage * stage_b_bytes;
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(&full_bar[stage], tx);
          if (L.diag & 8) {
          } else if (L.a_mn) {  // A given reduction-major: two [64 k x 64 m] boxes, m contiguous
            ptx::tma_load_2d(sa, ma, m0, ka, &full_bar[stage]);
            ptx::tma_load_2d(sa + kStageABytes / 2, ma, m0 + 64, ka, &full_bar[stage]);
          } else {
            ptx::tma_load_2d(sa, ma, ka, m0, &full_bar[stage]);
          }
          if (L.diag & 4) {
          } else if (L.b_mn) {  // B given reduction-major: bn/64 boxes of [64 k x 64 n], n contiguous
            for (int j = 0; j < P.bn / 64; ++j)
              ptx::tma_load_2d(sb + j * (kBK * 128), mb, n0 + 64 * j, kk + boff, &full_bar[stage]);
          } else {
            ptx::tma_load_2d(sb, mb, kk, n0 + boff, &full_bar[stage]);
          }
        }
        __syncwarp();
        if (++stage == n_stages) { stage = 0; phase ^= 1u; }
        if (++kbs == P.nk[seg]) { kbs = 0; ++seg; }
      }
    }
  } else if (warp == 1) {
    // ================================================================= MMA issuer
    // per-k-step advance of the descriptor start address (>> 4) and the constant upper halves:
    //   K-major, 128B swizzle: 8-row atoms 1024 B apart (SBO); a 16-element k step is 32 B inside the swizzle span.
    //   reduction-major ("MN-major"): 64(mn) x 8(k) atoms, 1024 B between k atoms (SBO), 64 k-rows * 128 B between
    //   mn atoms (LBO); a 16-row k step is 2048 B.
    const uint64_t a_hi = ptx::smem_desc_sw128(0, L.a_mn ? kBK * 128 : 0, 1024);
    const uint64_t b_hi = ptx::smem_desc_sw128(0, L.b_mn ? kBK * 128 : 0, 1024);
    const uint32_t a_step = L.a_mn ? 2048u >> 4 : 32u >> 4, b_step = L.b_mn ? 2048u >> 4 : 32u >> 4;
    int stage = 0;
    uint32_t phase = 0;
    int iter = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++iter) {
      TileInfo ti;
      decode_tile(L, t, ti);
      const uint32_t idesc = ptx::umma_idesc_f16((uint32_t)L.ab_format, (uint32_t)L.a_mn, (uint32_t)L.b_mn, (uint32_t)L.prob[ti.p].bn);
      const int acc = iter & 1;
      const uint32_t acc_phase = (uint32_t)((iter >> 1) & 1);
      ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1u);  // epilogue has drained this accumulator
      ptx::tc_fence_after_sync();
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * kBNMax;
      for (int kb = ti.kb0; kb < ti.kb1; ++kb) {
        ptx::mbar_wait(&full_bar[stage], phase);
        ptx::tc_fence_after_sync();
        const uint64_t a_desc = a_hi | (uint64_t)((ptx::smem_addr(smem_a + stage * kStageABytes) >> 4) & 0x3FFFu);
        const uint64_t b_desc = b_hi | (uint64_t)((ptx::smem_addr(smem_b + stage * stage_b_bytes) >> 4) & 0x3FFFu);
        if (ptx::elect_one()) {
          if (!(L.diag & 1)) {
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k)
              ptx::umma_f16(d_tmem, a_desc + (uint64_t)(k * a_step), b_desc + (uint64_t)(k * b_step), idesc,
                            (kb > ti.kb0 || k > 0) ? 1u : 0u);
          }
          if (stage & 1) ptx::umma_commit(&empty_bar[stage >> 1]);      // the pair is reusable once these MMAs retire
          if (kb == ti.kb1 - 1) ptx::umma_commit(&tmem_full_bar[acc]);  // accumulator complete
        }
        __syncwarp();
        if (++stage == n_stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    // ================================================================= epilogue (TMEM lanes 32*(warp%4) ..)
    const int ew = warp - 4;
    int iter = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++iter) {
      TileInfo ti;
      decode_tile(L, t, ti);
      const GemmProblem& P = L.prob[ti.p];
      const int acc = iter & 1;
      const uint32_t acc_phase = (uint32_t)((iter >> 1) & 1);
      const long long row = (long long)ti.m_blk * kBM + ew * 32 + lane;
      const bool add_bias = P.bias != nullptr && ti.kb0 == 0;
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
      ptx::tc_fence_after_sync();
      const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)acc * kBNMax;
      epilogue_tile<TD, kAtomic, kMode>(P, L.diag, taddr, row, ti.n0, ti.n_end, add_bias, smem_epi + ew * kEpiStageBytesPerWarp);
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[acc]);
      if (P.signal) {  // these rows are an operand of other tiles of this launch: publish them (4 warps = one tile)
        __threadfence();
        __syncwarp();
        if (lane == 0) atomicAdd(L.flags + ti.m_blk, 1);
      }
    }
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc<kTmemCols>(tmem_base);
  }
  if (L.flags != nullptr && threadIdx.x == 0) {  // the last CTA to leave zeroes the flags for the next launch
    __threadfence();
    const int done = atomicAdd(L.flags + L.n_flags, 1);
    if (done == (int)gridDim.x - 1) {
      for (int i = 0; i <= L.n_flags; ++i) L.flags[i] = 0;
      __threadfence();
    }
  }
  // an independent dependent launch (bit 3): it never reads the previous grid's output, but it must not be seen as
  // complete before that grid is, so that later launches on the stream stay ordered after both
  if ((L.pdl & 8) && threadIdx.x == 0) asm volatile("griddepcontrol.wait;" ::: "memory");
}

}  // namespace psob200

#include "lora_gemm2.cuh"  // cta_group::2 variant (CTA pairs) for the large tensor-bound shapes

namespace psob200 {

// ---------------------------------------------------------------------------------------------- host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
  static std::once_flag once;
  static EncodeTiledFn fn = nullptr;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    else
      cudaGetLastError();
  });
  return fn;
}

// Tensor map of a row-major [rows, cols] 16-bit matrix with leading dimension ld (elements); box = 64 contiguous
// elements x box_rows rows, 128-byte swizzle, out-of-bounds elements read as zero.
static int make_map(CUtensorMap* map, const void* ptr, long long rows, long long cols, long long ld, int box_rows,
                    int ab_dtype) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (fn == nullptr) return PSOB200_ERR_DRIVER;
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 2u};
  const cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(map, ab_dtype == PSOB200_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                        const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? PSOB200_OK : PSOB200_ERR_DRIVER;
}

// Fewest pair tiles for which a launch goes to the CTA-pair kernel.  Tuning override: PSOB200_PAIR_MIN_TILES (read once).
static int pair_min_tiles(int sms) {
  static const int env = [] { const char* e = getenv("PSOB200_PAIR_MIN_TILES"); return e ? atoi(e) : 0; }();
  return env > 0 ? env : sms / 2;
}

// Diagnostics: bits OR-ed into every launch's `diag` (PSOB200_GEMM_DIAG, read once; e.g. 0x40000 = record the timeline).
static int env_diag() {
  static const int env = [] { const char* e = getenv("PSOB200_GEMM_DIAG"); return e ? (int)strtol(e, nullptr, 0) : 0; }();
  return env;
}

// Tuning experiment: tile width of the main problem of fused (in-launch dependency) CTA-pair launches (PSOB200_FUSED_BN).
static int env_fused_bn() {
  static const int env = [] { const char* e = getenv("PSOB200_FUSED_BN"); return e ? atoi(e) : 0; }();
  return env;
}

// per-tile fixed cost of the pair kernel in units of one accumulator column: measured per-wave times at K = 1344 are
// 6.7 us (bn 128) and 9.7 us (bn 256) = 3.7 us + 23.4 ns per column (tools/diag_lora_parts.py --bn ...)
constexpr int kTileFixedCols = 160;

static int choose_bn(long long N, bool b_mn) {
  if (b_mn && N < 256) return (int)(((N + 63) / 64) * 64);  // reduction-major B: whole 64-column boxes
  if (N >= 256) {
    // widest tile that wastes the fewest columns: 256, or 128-wide tiles when that divides N better
    const long long w256 = ((N + 255) / 256) * 256 - N, w128 = ((N + 127) / 128) * 128 - N;
    return w128 < w256 ? 128 : 256;
  }
  return (int)(((N + 15) / 16) * 16);
}

// Tile width of the CTA-pair kernel.  The kernel is persistent over `pairs` CTA pairs with a static tile order, so its time
// is (number of waves) x (time of one tile) and a tile costs ~ its width plus a fixed part (pipeline fill, drain of the last
// accumulator): pick the width that minimises waves x (bn + fixed) instead of always 256.  E.g. M = 8192, N = 1280 on 74
// pairs: 256 -> 160 tiles = 3 waves, 224 -> 192 tiles = 3 narrower waves (measured 29.0 -> 26.4 us).  Widths that are not
// multiples of 32 are excluded (bn = 144 measured 30 % slower than the model predicts).  `groups` column groups of `N` columns
// each are tiled separately (a tile never straddles two stacked projections); `other_tiles` = tiles of the launch's other problems.
static int choose_bn2(long long M, long long N, int groups, bool b_mn, int pairs, long long other_tiles) {
  const int unit = b_mn ? 128 : 32;
  if (N < 256) return (int)(((N + unit - 1) / unit) * unit);
  const long long m_tiles = (M + 255) / 256;
  int best = 256;
  long long best_cost = -1;
  for (int bn = 256; bn >= 128; bn -= unit) {
    const long long tiles = m_tiles * groups * ((N + bn - 1) / bn) + other_tiles;
    const long long waves = (tiles + pairs - 1) / pairs;
    const long long cost = waves * (bn + kTileFixedCols);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = bn; }
  }
  return best;
}

// ---- host description of a launch: what the C-ABI entry points assemble ---------------------------------------------
struct HostSeg {
  const void* a; long long lda, a_rows, a_cols;   // the matrix the A map describes ([M, cols] K-major, or [K, M] reduction-major)
  const void* b; long long ldb, b_rows, b_cols;   // the matrix the B map describes ([N.., K] K-major, or [K.., N] reduction-major)
  long long K;                                    // reduction length of the segment
  int a_koff, a_gkoff, b_off;
};
struct HostProblem {
  long long M, N;
  int n_seg;
  HostSeg seg[kMaxSeg];
  void* d; long long ldd; void* dt; long long lddt;
  const void* bias; int bias_dtype;
  float alpha;
  long long group_n;  // 0: one column group
  int signal, wait_seg, wait_count;
  int tune_bn;
};
struct HostLaunch {
  HostProblem prob[kMaxProb];
  int n_prob;
  int ab_dtype, d_dtype, a_mn, b_mn, accumulate, split_k, pdl, diag;
  int* flags; long long flags_len;
};

struct MapKey { const void* p; long long rows, cols, ld; int box; };

static int launch_problems(const HostLaunch& H, cudaStream_t stream) {
  if (H.n_prob < 1 || H.n_prob > kMaxProb) return PSOB200_ERR_INVALID_ARG;
  const int sms = sm_count();
  bool any_dep = false, any_dt = false, any_bias = false, bias_other = false, all_d = true;
  for (int i = 0; i < H.n_prob; ++i) {
    const HostProblem& hp = H.prob[i];
    if (hp.M <= 0 || hp.N <= 0 || hp.n_seg < 1 || hp.n_seg > kMaxSeg || (!hp.d && !hp.dt)) return PSOB200_ERR_INVALID_ARG;
    if ((hp.d && hp.ldd < hp.N) || (hp.dt && hp.lddt < hp.M)) return PSOB200_ERR_SHAPE;
    if (hp.M > 0x7fffffffLL - 256 || hp.N > 0x7fffffffLL - 256) return PSOB200_ERR_SHAPE;
    if (H.a_mn && hp.n_seg != 1) return PSOB200_ERR_INVALID_ARG;
    for (int s = 0; s < hp.n_seg; ++s) {
      const HostSeg& sg = hp.seg[s];
      if (!sg.a || !sg.b || sg.K <= 0 || sg.K > 0x7fffffffLL - 256) return PSOB200_ERR_INVALID_ARG;
      if (!aligned16(sg.a) || !aligned16(sg.b)) return PSOB200_ERR_ALIGNMENT;
      if (sg.lda <= 0 || (sg.lda % 8) != 0 || sg.ldb <= 0 || (sg.ldb % 8) != 0) return PSOB200_ERR_SHAPE;  // TMA: 16-byte row pitch
    }
    any_dep |= hp.signal != 0 || hp.wait_seg >= 0;
    any_dt |= hp.dt != nullptr;
    all_d &= hp.d != nullptr && hp.dt == nullptr;
    any_bias |= hp.bias != nullptr;
    bias_other |= hp.bias != nullptr && hp.bias_dtype != H.d_dtype;
    if (hp.bias && !valid_dtype(hp.bias_dtype)) return PSOB200_ERR_DTYPE;
  }
  if (H.ab_dtype != PSOB200_BF16 && H.ab_dtype != PSOB200_F16) return PSOB200_ERR_DTYPE;
  if (!valid_dtype(H.d_dtype)) return PSOB200_ERR_DTYPE;
  if (H.accumulate && H.d_dtype != PSOB200_F32) return PSOB200_ERR_DTYPE;
  if (H.split_k < 0 || (H.split_k > 1 && !H.accumulate)) return PSOB200_ERR_INVALID_ARG;
  if (any_dep && (H.accumulate || H.split_k > 1 || H.flags == nullptr)) return PSOB200_ERR_INVALID_ARG;

  // ---- kernel: CTA pairs (cta_group::2) when the launch has at least half a wave of 256-row pair tiles
  const HostProblem& big = H.prob[H.n_prob - 1];  // the main problem is listed last
  const int big_groups = big.group_n > 0 ? (int)((big.N + big.group_n - 1) / big.group_n) : 1;
  const long long big_gn = big.group_n > 0 ? big.group_n : big.N;
  bool pair = false;
  int big_bn2 = 0;
  {
    const int unit = H.b_mn ? 128 : 16;
    const bool eligible = !H.a_mn && !H.accumulate && H.split_k <= 1 &&
                          (big.tune_bn == 0 || (big.tune_bn % unit == 0 && big.tune_bn >= 32));
    long long other = 0;
    for (int i = 0; i + 1 < H.n_prob; ++i) other += (H.prob[i].M + 255) / 256;  // the skinny problems: one tile per row block
    big_bn2 = big.tune_bn > 0 ? big.tune_bn : choose_bn2(big.M, big_gn, big_groups, H.b_mn != 0, sms / 2, other);
    if (any_dep && big.tune_bn == 0 && env_fused_bn() > 0 && env_fused_bn() % unit == 0) big_bn2 = env_fused_bn();
    const long long pair_tiles = ((big.M + 255) / 256) * big_groups * ((big_gn + big_bn2 - 1) / big_bn2);
    const bool want = (H.diag & 0x10000) || (pair_tiles >= pair_min_tiles(sms) && big_gn >= 128 && !(H.diag & 0x20000));
    pair = eligible && want && big_bn2 <= kBNMax;
  }
  const int tile_m = pair ? 256 : kBM;

  GemmLaunch L = {};
  GemmMaps maps = {};
  MapKey keys[kMaxMaps];
  int n_maps = 0;
  auto get_map = [&](const void* p, long long rows, long long cols, long long ld, int box) -> int {
    for (int i = 0; i < n_maps; ++i)
      if (keys[i].p == p && keys[i].rows == rows && keys[i].cols == cols && keys[i].ld == ld && keys[i].box == box) return i;
    if (n_maps == kMaxMaps) return -1;
    if (make_map(&maps.m[n_maps], p, rows, cols, ld, box, H.ab_dtype) != PSOB200_OK) return -2;
    keys[n_maps] = {p, rows, cols, ld, box};
    return n_maps++;
  };

  L.n_prob = H.n_prob;
  int tile0 = 0, max_bn = 0, max_m_tiles = 0;
  long long base_tiles = 0;
  for (int i = 0; i < H.n_prob; ++i) {
    const HostProblem& hp = H.prob[i];
    const int groups = hp.group_n > 0 ? (int)((hp.N + hp.group_n - 1) / hp.group_n) : 1;
    const long long gn = hp.group_n > 0 ? hp.group_n : hp.N;
    int bn;
    if (pair) {
      bn = (i == H.n_prob - 1) ? big_bn2 : (hp.tune_bn > 0 ? hp.tune_bn : choose_bn2(hp.M, gn, groups, H.b_mn != 0, sms / 2, 0));
      if (bn < 32 || bn > kBNMax || (bn % (H.b_mn ? 128 : 16)) != 0) return PSOB200_ERR_INVALID_ARG;
    } else {
      bn = hp.tune_bn > 0 ? hp.tune_bn : choose_bn(gn, H.b_mn != 0);
      if (bn < 16 || bn > kBNMax || (bn % (H.b_mn ? 64 : 16)) != 0) return PSOB200_ERR_INVALID_ARG;
    }
    GemmProblem& P = L.prob[i];
    P.M = hp.M; P.N = hp.N;
    P.d = hp.d; P.ldd = hp.ldd; P.dt = hp.dt; P.lddt = hp.lddt;
    P.bias = hp.bias; P.bias_dtype = hp.bias_dtype; P.alpha = hp.alpha;
    P.group_n = gn;
    P.bn = bn;
    P.m_tiles = (int)((hp.M + tile_m - 1) / tile_m);
    P.tiles_per_group = (int)((gn + bn - 1) / bn);
    P.n_tiles = groups * P.tiles_per_group;
    P.n_seg = hp.n_seg;
    P.nk_total = 0;
    for (int s = 0; s < hp.n_seg; ++s) {
      const HostSeg& sg = hp.seg[s];
      P.nk[s] = pair ? (int)((sg.K + kBK2 - 1) / kBK2) : (int)((sg.K + kBK - 1) / kBK);  // stages: 128 deep (pairs) / 64 deep
      P.nk_total += P.nk[s];
      P.a_koff[s] = sg.a_koff; P.a_gkoff[s] = sg.a_gkoff; P.b_off[s] = sg.b_off;
      const int ma = H.a_mn ? get_map(sg.a, sg.a_rows, sg.a_cols, sg.lda, kBK) : get_map(sg.a, sg.a_rows, sg.a_cols, sg.lda, kBM);
      const int mb = H.b_mn ? get_map(sg.b, sg.b_rows, sg.b_cols, sg.ldb, kBK)
                            : get_map(sg.b, sg.b_rows, sg.b_cols, sg.ldb, pair ? bn / 2 : bn);
      if (ma == -2 || mb == -2) return PSOB200_ERR_DRIVER;
      if (ma < 0 || mb < 0) return PSOB200_ERR_INVALID_ARG;
      P.map_a[s] = ma; P.map_b[s] = mb;
    }
    P.signal = hp.signal; P.wait_seg = hp.wait_seg; P.wait_count = hp.wait_count;
    {  // A few row blocks against a weight matrix that L2 (126 MB) cannot hold -- the k / v of all cross-attention layers: 616 rows
       // x [153 600, 2048] -- : column tiles fastest streams the whole weight once PER ROW BLOCK (ncu: 1.99 GB of DRAM reads for 0.65 GB
       // of operands); row blocks fastest reads every weight tile once while the small x stays in L2
      const double esz = 2.0;
      const double b_bytes = (double)hp.N * (double)hp.seg[0].K * esz, a_bytes = (double)hp.M * (double)hp.seg[0].K * esz;
      P.m_fast = (!H.a_mn && b_bytes > 48e6 && a_bytes < 16e6 && P.m_tiles > 1) ? 1 : 0;
    }
    P.splits = 1; P.kb_per_split = P.nk_total;
    base_tiles += (long long)P.m_tiles * P.n_tiles;
    if (bn > max_bn) max_bn = bn;
    if (P.m_tiles > max_m_tiles) max_m_tiles = P.m_tiles;
  }
  // split the reduction only for accumulating launches that cannot fill the GPU: the largest split count whose tiles all fit
  // on the SMs at once (rounding UP gave e.g. 150 tiles on 148 SMs: two CTAs ran two tiles each and the launch took twice as
  // long; measured 12.2 -> 10.1 us for dA at M = 8192)
  int splits = H.split_k;
  if (splits == 0) {
    splits = 1;
    if (H.accumulate) {
      splits = (int)(sms / base_tiles);
      if (splits < 1) splits = 1;
    }
  }
  for (int i = 0; i < H.n_prob; ++i) {
    GemmProblem& P = L.prob[i];
    int sp = splits > P.nk_total ? P.nk_total : splits;
    P.kb_per_split = (P.nk_total + sp - 1) / sp;
    P.splits = (P.nk_total + P.kb_per_split - 1) / P.kb_per_split;
    P.tile0 = tile0;
    const long long nt = (long long)P.m_tiles * P.n_tiles * P.splits;
    if (nt + tile0 > 0x7fffffffLL) return PSOB200_ERR_SHAPE;
    tile0 += (int)nt;
  }
  L.total_tiles = tile0;
  {  // a waiting problem waits for EVERY tile of the signalling problems in its row block
    int released = 0;
    for (int i = 0; i < H.n_prob; ++i)
      if (L.prob[i].signal) released += L.prob[i].n_tiles;
    for (int i = 0; i < H.n_prob; ++i)
      if (L.prob[i].wait_seg >= 0) {
        if (released == 0 || L.prob[i].wait_seg >= L.prob[i].n_seg) return PSOB200_ERR_INVALID_ARG;
        L.prob[i].wait_count = released;
      }
  }
  L.ab_format = H.ab_dtype == PSOB200_BF16 ? 1 : 0;
  L.a_mn = H.a_mn ? 1 : 0;
  L.b_mn = H.b_mn ? 1 : 0;
  L.atomic = H.accumulate ? 1 : 0;
  L.diag = H.diag | env_diag();
  L.pdl = H.pdl;
  if (any_dep) {
    if (H.flags_len < max_m_tiles + 1) return PSOB200_ERR_WORKSPACE;
    L.flags = H.flags;
    L.n_flags = max_m_tiles;
  }

  typedef void (*KernelFn)(GemmMaps, GemmLaunch);
  const bool multi = H.n_prob > 1;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(kGemmThreads);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  if (H.pdl & (2 | 8)) {  // may begin while the previous kernel on the stream is still running (it waits on the device)
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  if (pair) {
    L.stages = kStages2;
    L.n_acc = max_bn <= 160 ? 3 : 2;
    L.acc_stride = max_bn <= 160 ? 160 : kBNMax;
    L.stage_b_bytes = 2 * (max_bn / 2) * kBK * 2;  // two 64-deep sub-tiles of this CTA's half of the widest B tile
    // 0-2: general per output type (any bias type); then per 16-bit type: bias of the same type, no bias, problem lists
    int variant;
    if (H.d_dtype == PSOB200_F32) variant = 0;
    else {
      const int t16 = H.d_dtype == PSOB200_BF16 ? 0 : 1;
      if (bias_other) variant = 1 + t16;
      else if (any_dt || (multi && any_bias)) variant = 7 + t16;
      else variant = 3 + 2 * t16 + (any_bias ? 0 : 1);
    }
    static const KernelFn kernels2[9] = {
        lora_gemm2_kernel<float, kEpiGeneral>, lora_gemm2_kernel<__nv_bfloat16, kEpiGeneral>, lora_gemm2_kernel<__half, kEpiGeneral>,
        lora_gemm2_kernel<__nv_bfloat16, kEpiD | kEpiBiasSameType>, lora_gemm2_kernel<__nv_bfloat16, kEpiD>,
        lora_gemm2_kernel<__half, kEpiD | kEpiBiasSameType>, lora_gemm2_kernel<__half, kEpiD>,
        lora_gemm2_kernel<__nv_bfloat16, kEpiFused>, lora_gemm2_kernel<__half, kEpiFused>};
    static PerDevice<int> max_clusters[9];  // 0: not configured on this device yet
    std::atomic<int>& cap = max_clusters[variant].here();
    int clusters = cap.load(std::memory_order_acquire);
    if (clusters == 0) {
      const cudaError_t e = cudaFuncSetAttribute(kernels2[variant], cudaFuncAttributeMaxDynamicSharedMemorySize, kGemm2SmemBytes);
      if (e != cudaSuccess) return consume_launch_error("configure lora_gemm2_kernel", e);
      // pairs that can be co-resident: a launch with in-kernel dependencies must never have more (its tiles spin-wait)
      cudaLaunchConfig_t oc = {};
      oc.gridDim = dim3((unsigned)(sms / 2 * 2));
      oc.blockDim = dim3(kGemmThreads);
      oc.dynamicSmemBytes = kGemm2SmemBytes;
      cudaLaunchAttribute oa[1];
      oa[0].id = cudaLaunchAttributeClusterDimension;
      oa[0].val.clusterDim.x = 2; oa[0].val.clusterDim.y = 1; oa[0].val.clusterDim.z = 1;
      oc.attrs = oa; oc.numAttrs = 1;
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, kernels2[variant], &oc) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        n = sms / 2;
      }
      if (n > sms / 2) n = sms / 2;
      clusters = n;
      cap.store(n, std::memory_order_release);
    }
    const long long want = L.total_tiles < clusters ? L.total_tiles : clusters;
    cfg.gridDim = dim3(2u * (unsigned)want);
    cfg.dynamicSmemBytes = kGemm2SmemBytes;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernels2[variant], maps, L);
    return consume_launch_error("launch lora_gemm2_kernel", e);
  }

  L.stages = (kStages * (kStageABytes + kStageBBytes)) / (kStageABytes + max_bn * kBK * 2);
  if (L.stages > kMaxStages) L.stages = kMaxStages;
  L.stages &= ~1;
  if ((H.diag >> 8) & 15) L.stages = (H.diag >> 8) & 14;
  L.stage_b_bytes = max_bn * kBK * 2;
  // exact epilogue modes for the single-problem launches of the training step, the fused mode for problem lists, the
  // general kernel for everything else
  int variant;
  if (L.atomic) {
    bool only_d = true, only_dt = true;
    for (int i = 0; i < H.n_prob; ++i) { only_d &= H.prob[i].d && !H.prob[i].dt; only_dt &= H.prob[i].dt && !H.prob[i].d; }
    variant = any_bias ? 0 : (only_d ? 1 : (only_dt ? 2 : 0));
  } else if (H.d_dtype == PSOB200_F32) variant = 3;
  else {
    const int base = H.d_dtype == PSOB200_BF16 ? 4 : 9;
    if (bias_other) variant = base;
    else if (multi) variant = (all_d && !any_bias) ? base + 2 : base + 4;
    else variant = base + (any_bias ? (all_d ? 1 : 0) : (all_d ? 2 : 3));
  }
  static const KernelFn kernels[14] = {
      lora_gemm_kernel<float, true, kEpiGeneral>, lora_gemm_kernel<float, true, kEpiD>, lora_gemm_kernel<float, true, kEpiDt>,
      lora_gemm_kernel<float, false, kEpiGeneral>,
      lora_gemm_kernel<__nv_bfloat16, false, kEpiGeneral>, lora_gemm_kernel<__nv_bfloat16, false, kEpiD | kEpiBiasSameType>,
      lora_gemm_kernel<__nv_bfloat16, false, kEpiD>, lora_gemm_kernel<__nv_bfloat16, false, kEpiAnyOut>,
      lora_gemm_kernel<__nv_bfloat16, false, kEpiFused>,
      lora_gemm_kernel<__half, false, kEpiGeneral>, lora_gemm_kernel<__half, false, kEpiD | kEpiBiasSameType>,
      lora_gemm_kernel<__half, false, kEpiD>, lora_gemm_kernel<__half, false, kEpiAnyOut>,
      lora_gemm_kernel<__half, false, kEpiFused>};
  static PerDevice<int> max_ctas[14];
  std::atomic<int>& cap = max_ctas[variant].here();
  int ctas = cap.load(std::memory_order_acquire);
  if (ctas == 0) {
    const cudaError_t e = cudaFuncSetAttribute(kernels[variant], cudaFuncAttributeMaxDynamicSharedMemorySize, kGemmSmemBytes);
    if (e != cudaSuccess) return consume_launch_error("configure lora_gemm_kernel", e);
    ctas = sms;  // one CTA per SM by design (~193 KB of shared memory each): every CTA of the grid is co-resident
    cap.store(ctas, std::memory_order_release);
  }
  cfg.gridDim = dim3((unsigned)(L.total_tiles < ctas ? L.total_tiles : ctas));
  cfg.dynamicSmemBytes = kGemmSmemBytes;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kernels[variant], maps, L);
  return consume_launch_error("launch lora_gemm_kernel", e);
}

}  // namespace psob200

using namespace psob200;

extern "C" int psob200_lora_gemm(const psob200_gemm_args* args, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_gemm_args& g = *args;
  if (g.M <= 0 || g.N <= 0 || g.K1 <= 0 || g.K2 < 0 || !g.a1 || !g.b1 || (!g.d && !g.dt)) return PSOB200_ERR_INVALID_ARG;
  if (g.K2 > 0 && (!g.a2 || !g.b2)) return PSOB200_ERR_INVALID_ARG;
  if (g.a_reduction_major && g.K2 > 0) return PSOB200_ERR_INVALID_ARG;
  if (g.bias && !valid_dtype(g.bias_dtype)) return PSOB200_ERR_DTYPE;
  HostLaunch H = {};
  H.n_prob = 1;
  H.ab_dtype = g.ab_dtype; H.d_dtype = g.d_dtype;
  H.a_mn = g.a_reduction_major; H.b_mn = g.b_reduction_major; H.accumulate = g.accumulate; H.split_k = g.split_k;
  H.pdl = g.pdl; H.diag = g.diag;
  HostProblem& P = H.prob[0];
  P.M = g.M; P.N = g.N;
  P.d = g.d; P.ldd = g.ldd; P.dt = g.dt; P.lddt = g.lddt;
  P.bias = g.bias; P.bias_dtype = g.bias_dtype; P.alpha = g.alpha;
  P.wait_seg = -1; P.tune_bn = g.tune_bn;
  P.n_seg = g.K2 > 0 ? 2 : 1;
  const void* as[2] = {g.a1, g.a2};
  const void* bs[2] = {g.b1, g.b2};
  const long long ldas[2] = {g.lda1, g.lda2}, ldbs[2] = {g.ldb1, g.ldb2}, ks[2] = {g.K1, g.K2};
  for (int s = 0; s < P.n_seg; ++s) {
    HostSeg& sg = P.seg[s];
    sg.a = as[s]; sg.lda = ldas[s]; sg.b = bs[s]; sg.ldb = ldbs[s]; sg.K = ks[s];
    if (g.a_reduction_major) { sg.a_rows = ks[s]; sg.a_cols = g.M; } else { sg.a_rows = g.M; sg.a_cols = ks[s]; }
    if (g.b_reduction_major) { sg.b_rows = ks[s]; sg.b_cols = g.N; } else { sg.b_rows = g.N; sg.b_cols = ks[s]; }
  }
  return launch_problems(H, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int psob200_lora_gemm_timeline(unsigned long long* host_out, long long capacity) {
  // diagnostics (diag bit 0x40000 of a CTA-pair launch): synchronous copy of the per-CTA time stamps of the last such launch
  const long long n = (long long)kTimelineCtas * kTimelineSlots * 2;
  if (host_out == nullptr || capacity < n) return PSOB200_ERR_INVALID_ARG;
  const cudaError_t e = cudaMemcpyFromSymbol(host_out, g_timeline, sizeof(unsigned long long) * n);
  return e == cudaSuccess ? (int)n : consume_launch_error("psob200_lora_gemm_timeline", e);
}

// ---------------------------------------------------------------------------------------------- stacked LoRA projections
namespace psob200 {

static HostSeg seg_kmajor(const void* a, long long lda, long long a_rows, long long a_cols, const void* b, long long ldb,
                          long long b_rows, long long b_cols, long long K) {
  HostSeg s = {};
  s.a = a; s.lda = lda; s.a_rows = a_rows; s.a_cols = a_cols;
  s.b = b; s.ldb = ldb; s.b_rows = b_rows; s.b_cols = b_cols;
  s.K = K;
  return s;
}

static HostLaunch launch_defaults(int32_t dtype) {
  HostLaunch H = {};
  H.ab_dtype = dtype;
  H.d_dtype = dtype;
  for (int i = 0; i < kMaxProb; ++i) { H.prob[i].alpha = 1.0f; H.prob[i].wait_seg = -1; }
  return H;
}

static int group_check(const psob200_lora_group_args& a, bool backward) {
  // the backward takes the G gradients as separate pointers (dy[PSOB200_MAX_GROUP]); the forward reads ONE input and writes one
  // stacked output, for any number of stacked projections (e.g. the k / v projections of every cross-attention layer at once)
  if (a.G < 1 || (backward && a.G > PSOB200_MAX_GROUP) || a.M <= 0 || a.K <= 0 || a.N <= 0 || !a.w) return PSOB200_ERR_INVALID_ARG;
  const bool lora = a.adapters_enabled != 0;
  if (lora && (!a.lora_a || !a.lora_b || a.r <= 0 || (backward && a.r * a.G > 4 * kBNMax))) return PSOB200_ERR_INVALID_ARG;
  if ((long long)a.G * a.N > 0x7fffffffLL - 256) return PSOB200_ERR_SHAPE;
  // column group g of the stacked t / u starts at g * r_stride: 16-byte aligned (ranks that are not multiples of 8 are
  // stacked with r_stride = r rounded up to 8: zero rows in lora_a, zero columns in t / u)
  const long long rs = a.r_stride > 0 ? a.r_stride : a.r;
  if (lora && (rs < a.r || (a.G > 1 && (rs % 8) != 0))) return PSOB200_ERR_SHAPE;
  if (a.G > 1 && a.bias) return PSOB200_ERR_INVALID_ARG;
  if (!backward && (!a.x || !a.y || (lora && !a.t))) return PSOB200_ERR_INVALID_ARG;
  if (backward) {
    for (int g = 0; g < a.G; ++g)
      if (!a.dy[g]) return PSOB200_ERR_INVALID_ARG;
    if (lora && !a.u) return PSOB200_ERR_INVALID_ARG;
    if (lora && a.d_lora_a && (!a.ut || !a.x)) return PSOB200_ERR_INVALID_ARG;
    if (lora && a.d_lora_b && !a.tt) return PSOB200_ERR_INVALID_ARG;
  }
  return PSOB200_OK;
}

}  // namespace psob200

extern "C" int psob200_lora_group_forward(const psob200_lora_group_args* args, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_lora_group_args& a = *args;
  int rc = group_check(a, false);
  if (rc != PSOB200_OK) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool lora = a.adapters_enabled != 0;
  const long long rs = a.r_stride > 0 ? a.r_stride : a.r;
  const long long GN = a.G * a.N, Gr = a.G * rs;  // width of the stacked t: G column groups of r_stride
  const int fph = a.forward_phases == 0 ? (PSOB200_FWD_DOWN | PSOB200_FWD_MAIN) : a.forward_phases;
  const bool fused = lora && fph == (PSOB200_FWD_DOWN | PSOB200_FWD_MAIN) && a.flags != nullptr;

  // t = scaling * x [A_1; ...; A_G]^T  (+ its transpose, the K-major operand of the dB reductions)
  HostProblem down = {};
  if (lora) {
    down.M = a.M; down.N = Gr; down.n_seg = 1;
    down.seg[0] = seg_kmajor(a.x, a.ldx, a.M, a.K, a.lora_a, a.lda, Gr, a.K, a.K);
    down.d = a.t; down.ldd = a.ldt; down.dt = a.tt; down.lddt = a.ldtt;
    down.alpha = a.scaling; down.wait_seg = -1;
  }
  // y = x [W_1; ...; W_G]^T + bias + t_g B_g^T for column group g  (ONE pass over the frozen weights)
  HostProblem main = {};
  main.M = a.M; main.N = GN; main.alpha = 1.0f; main.wait_seg = -1;
  main.group_n = a.G > 1 ? a.N : 0;
  main.n_seg = lora ? 2 : 1;
  main.seg[0] = seg_kmajor(a.x, a.ldx, a.M, a.K, a.w, a.ldw, GN, a.K, a.K);
  if (lora) {
    main.seg[1] = seg_kmajor(a.t, a.ldt, a.M, Gr, a.lora_b, a.ldb, GN, a.r, a.r);
    main.seg[1].a_gkoff = a.G > 1 ? (int)rs : 0;
  }
  main.bias = a.bias; main.bias_dtype = a.bias_dtype;
  main.d = a.y; main.ldd = a.ldy;

  if (fused) {  // one launch: the tiles of t come first and release a flag per row block; y's adapter segment waits for it
    HostLaunch H = launch_defaults(a.dtype);
    H.n_prob = 2;
    H.prob[0] = down; H.prob[0].signal = 1;
    H.prob[1] = main; H.prob[1].wait_seg = 1;
    H.flags = a.flags; H.flags_len = a.flags_len;
    if (a.launch_flags & 1) H.pdl = 2 | 4;
    return launch_problems(H, st);
  }
  if (lora && (fph & PSOB200_FWD_DOWN)) {
    HostLaunch H = launch_defaults(a.dtype);
    H.n_prob = 1; H.prob[0] = down;
    H.pdl = (fph & PSOB200_FWD_MAIN) ? 1 : 0;  // the main pass reads t only in its last k-blocks: let it start early
    if (a.launch_flags & 1) H.pdl |= 2 | 4;
    if ((rc = launch_problems(H, st)) != PSOB200_OK) return rc;
  }
  if (fph & PSOB200_FWD_MAIN) {
    HostLaunch H = launch_defaults(a.dtype);
    H.n_prob = 1; H.prob[0] = main;
    H.pdl = (lora && (fph & PSOB200_FWD_DOWN)) ? 2 : ((a.launch_flags & 1) ? (2 | 4) : 0);
    return launch_problems(H, st);
  }
  return PSOB200_OK;
}

extern "C" int psob200_lora_group_backward(const psob200_lora_group_args* args, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  const psob200_lora_group_args& a = *args;
  int rc = group_check(a, true);
  if (rc != PSOB200_OK) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool lora = a.adapters_enabled != 0;
  const int G = a.G;
  const long long rs = a.r_stride > 0 ? a.r_stride : a.r;
  const long long GN = G * a.N, Gr = G * rs;
  const int ph = a.backward_phases == 0 ? (PSOB200_BWD_INPUT_GRAD | PSOB200_BWD_WEIGHT_GRAD) : a.backward_phases;
  const bool need_u = lora && (ph & PSOB200_BWD_U) && (a.dx != nullptr || a.ut != nullptr || a.d_lora_a != nullptr);
  const bool need_dx = a.dx != nullptr && (ph & PSOB200_BWD_DX);

  // u_g = scaling * dy_g B_g   (B [N,r] consumed reduction-major out of the stacked [G N, r]: no transposed copy)
  HostProblem up[PSOB200_MAX_GROUP] = {};
  for (int g = 0; g < G && lora; ++g) {
    HostProblem& p = up[g];
    // N = r_stride: the columns beyond r are written as zeros (lora_b has only r columns: the TMA unit zero-fills), so that the
    // padding of the stacked u never holds stale bits when dx multiplies it with lora_a's zero rows
    p.M = a.M; p.N = rs; p.n_seg = 1; p.alpha = a.scaling; p.wait_seg = -1;
    p.seg[0] = seg_kmajor(a.dy[g], a.lddy[g], a.M, a.N, a.lora_b, a.ldb, GN, a.r, a.N);
    p.seg[0].b_off = (int)(g * a.N);
    p.d = reinterpret_cast<unsigned char*>(a.u) + (size_t)g * rs * 2; p.ldd = a.ldu;
    if (a.ut) { p.dt = reinterpret_cast<unsigned char*>(a.ut) + (size_t)g * rs * a.ldut * 2; p.lddt = a.ldut; }
  }
  // dx = sum_g dy_g W_g + [u_1 .. u_G] [A_1; ..; A_G]   (W [N,K], A [r,K] reduction-major)
  HostProblem dxp = {};
  if (need_dx) {
    dxp.M = a.M; dxp.N = a.K; dxp.alpha = 1.0f; dxp.wait_seg = -1;
    dxp.n_seg = G + (lora ? 1 : 0);
    for (int g = 0; g < G; ++g) {
      dxp.seg[g] = seg_kmajor(a.dy[g], a.lddy[g], a.M, a.N, a.w, a.ldw, GN, a.K, a.N);
      dxp.seg[g].b_off = (int)(g * a.N);
    }
    if (lora) dxp.seg[G] = seg_kmajor(a.u, a.ldu, a.M, Gr, a.lora_a, a.lda, Gr, a.K, Gr);
    dxp.d = a.dx; dxp.ldd = a.lddx;
  }
  const bool fuse_in = need_u && need_dx && a.flags != nullptr && G + 1 <= kMaxProb;
  if (fuse_in) {  // one launch: the u tiles release a flag per row block, dx's adapter segment waits for all G of them
    HostLaunch H = launch_defaults(a.dtype);
    H.b_mn = 1;
    H.n_prob = G + 1;
    for (int g = 0; g < G; ++g) { H.prob[g] = up[g]; H.prob[g].signal = 1; }
    H.prob[G] = dxp; H.prob[G].wait_seg = G;
    H.flags = a.flags; H.flags_len = a.flags_len;
    if (a.launch_flags & 1) H.pdl = 2 | 4;
    if ((rc = launch_problems(H, st)) != PSOB200_OK) return rc;
  } else {
    if (need_u) {
      HostLaunch H = launch_defaults(a.dtype);
      H.b_mn = 1; H.n_prob = G;
      for (int g = 0; g < G; ++g) H.prob[g] = up[g];
      H.pdl = (need_dx ? 1 : 0) | ((a.launch_flags & 1) ? (2 | 4) : 0);
      if ((rc = launch_problems(H, st)) != PSOB200_OK) return rc;
    }
    if (need_dx) {
      HostLaunch H = launch_defaults(a.dtype);
      H.b_mn = 1; H.n_prob = 1; H.prob[0] = dxp;
      H.pdl = (lora && need_u) ? 2 : ((a.launch_flags & 1) ? (2 | 4) : 0);
      if ((rc = launch_problems(H, st)) != PSOB200_OK) return rc;
    }
  }
  if (!lora) return PSOB200_OK;
  // dA[G r, K] += [u_1 .. u_G]^T x  (written transposed);  dB_g[N, r] += dy_g^T t_g : independent split reductions, one launch
  const bool want_da = (ph & PSOB200_BWD_DA) && a.d_lora_a != nullptr, want_db = (ph & PSOB200_BWD_DB) && a.d_lora_b != nullptr;
  if (!want_da && !want_db) return PSOB200_OK;
  // problems of the weight-gradient launches: dA as ONE problem over the stacked u when the gradient rows are packed like the
  // u columns (r_stride == r), else one per projection; then the G dB problems; at most kMaxProb per launch
  HostProblem wp[2 * PSOB200_MAX_GROUP] = {};
  int n = 0;
  if (want_da) {
    if (rs == a.r) {
      HostProblem& p = wp[n++];
      p.M = a.K; p.N = G * a.r; p.n_seg = 1; p.alpha = 1.0f; p.wait_seg = -1;
      p.seg[0] = seg_kmajor(a.x, a.ldx, a.M, a.K, a.ut, a.ldut, Gr, a.M, a.M);
      p.dt = a.d_lora_a; p.lddt = a.ld_da;
    } else {
      for (int g = 0; g < G; ++g) {
        HostProblem& p = wp[n++];
        p.M = a.K; p.N = a.r; p.n_seg = 1; p.alpha = 1.0f; p.wait_seg = -1;
        p.seg[0] = seg_kmajor(a.x, a.ldx, a.M, a.K, a.ut, a.ldut, Gr, a.M, a.M);
        p.seg[0].b_off = (int)(g * rs);
        p.dt = a.d_lora_a + (size_t)g * a.r * a.ld_da; p.lddt = a.ld_da;
      }
    }
  }
  if (want_db) {
    for (int g = 0; g < G; ++g) {
      HostProblem& p = wp[n++];
      p.M = a.N; p.N = a.r; p.n_seg = 1; p.alpha = 1.0f; p.wait_seg = -1;
      p.seg[0] = seg_kmajor(a.dy[g], a.lddy[g], a.M, a.N, a.tt, a.ldtt, Gr, a.M, a.M);
      p.seg[0].b_off = (int)(g * rs);
      p.d = a.d_lora_b + (size_t)g * a.N * a.ld_db; p.ldd = a.ld_db;
    }
  }
  for (int first = 0; first < n; first += kMaxProb) {
    const int cnt = n - first < kMaxProb ? n - first : kMaxProb;
    const bool more = first + cnt < n;
    HostLaunch H = launch_defaults(a.dtype);
    H.a_mn = 1; H.accumulate = 1; H.d_dtype = PSOB200_F32;
    H.n_prob = cnt;
    for (int i = 0; i < cnt; ++i) H.prob[i] = wp[first + i];
    // independent launches: the second may overlap the first entirely (it waits for it only before exiting)
    H.pdl = (more ? 1 : 0) | (first > 0 ? 8 : 0);
    if ((a.launch_flags & 1) && H.pdl == 0) H.pdl = 2 | 4;
    if (a.launch_flags & 2) H.split_k = 1;  // one accumulation per gradient element and launch: bit-reproducible
    if ((rc = launch_problems(H, st)) != PSOB200_OK) return rc;
  }
  return PSOB200_OK;
}

// ---------------------------------------------------------------------------------------------- LoRA-wrapped Linear (G = 1)
static psob200_lora_group_args group_of_linear(const psob200_lora_linear_args& a) {
  psob200_lora_group_args g = {};
  g.x = a.x; g.w = a.w; g.bias = a.bias; g.lora_a = a.lora_a; g.lora_b = a.lora_b;
  g.y = a.y; g.t = a.t; g.tt = a.tt; g.dy[0] = a.dy; g.dx = a.dx; g.u = a.u; g.ut = a.ut;
  g.d_lora_a = a.d_lora_a; g.d_lora_b = a.d_lora_b;
  g.flags = a.flags; g.flags_len = a.flags_len;
  g.ldx = a.ldx; g.ldw = a.ldw; g.lda = a.lda; g.ldb = a.ldb; g.ldy = a.ldy; g.ldt = a.ldt; g.ldtt = a.ldtt;
  g.lddy[0] = a.lddy; g.lddx = a.lddx; g.ldu = a.ldu; g.ldut = a.ldut; g.ld_da = a.ld_da; g.ld_db = a.ld_db;
  g.M = a.M; g.K = a.K; g.N = a.N; g.r = a.r; g.G = 1; g.r_stride = 0;
  g.scaling = a.scaling; g.dtype = a.dtype; g.bias_dtype = a.bias_dtype; g.adapters_enabled = a.adapters_enabled;
  g.forward_phases = a.forward_phases; g.backward_phases = a.backward_phases;
  return g;
}

extern "C" int psob200_lora_linear_forward(const psob200_lora_linear_args* args, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  if (args->adapters_enabled && args->r > kBNMax) return PSOB200_ERR_INVALID_ARG;
  const psob200_lora_group_args g = group_of_linear(*args);
  return psob200_lora_group_forward(&g, stream);
}

extern "C" int psob200_lora_linear_backward(const psob200_lora_linear_args* args, void* stream) {
  if (args == nullptr) return PSOB200_ERR_INVALID_ARG;
  if (!args->dy) return PSOB200_ERR_INVALID_ARG;
  if (args->adapters_enabled && args->r > kBNMax) return PSOB200_ERR_INVALID_ARG;
  const psob200_lora_group_args g = group_of_linear(*args);
  return psob200_lora_group_backward(&g, stream);
}
