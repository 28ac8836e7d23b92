// K3 — tcgen05 / TMEM / TMA GEMM family with fused epilogues (sm_100a).
//
// Replaces the cuBLASLt dispatches behind nn.Linear / nn.MultiheadAttention projections /
// einsum of the reference encoder (/root/reference/src/models/vit.py:197-206, 262-266, 289-292 and
// torch.nn.TransformerEncoderLayer), forward and backward:
//   fwd   : Y[M,N]  = X[M,K]  . W[N,K]^T      A K-major,  B K-major
//   dgrad : dX[M,K] = dY[M,N] . W[N,K]        A K-major,  B MN-major (W read in place, no transpose copy)
//   wgrad : dW[N,K] = dY[M,N]^T . X[M,K]      A MN-major, B MN-major (+ split-K over the token dimension)
//
// Structure: persistent CTAs (one per SM), 128 x BN output tile, BK = 64 (one 128-byte swizzle atom),
// kStages-deep TMA->smem ring, a single elected thread issues tcgen05.mma (M=128, N=BN, K=16) into a
// double-buffered TMEM accumulator (2 x BN columns) so that the epilogue warps (TMEM -> registers ->
// bias / activation / residual / mask -> global) of tile i overlap the main loop of tile i+1.
// Warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 4..11 = epilogue (coalesced through a per-warp
// smem transpose stage, see gemm_epilogue.cuh).
#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "sfcvit.h"
#include <string.h>

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kEpiWarps = 8;                 // two warps per TMEM lane quarter, each takes half of the tile's columns
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kNumThreads = 128 + kEpiThreads;

struct GemmParams {
  int M, N, K;
  int num_m_tiles, num_n_tiles, splits, kblocks_per_split, num_k_blocks;
  float* cs_ws;             // CS variant: fp32 [splits][M] partial row sums of A over K (wgrad: the bias gradient)
  EpiParams epi;
};

// CS ("column sums", wgrad only): db = dY^T . 1 is one more accumulator column of the GEMM that already streams dY —
// the units of n-tile 0 issue, per k-block, four extra M x 16 MMAs of their A tile against a constant all-ones B tile
// (1 KB of shared memory) into 16 TMEM columns behind the accumulator, and their epilogue writes that column per split.
// The accumulator is single-buffered in this variant (256 + 16 columns do not leave room for a second 256-column
// buffer); split-K weight gradients run one unit per CTA pair, so there is no next main loop to overlap with anyway.
template <int BN, int kStages, int CL, int EPI, bool CS = false>
struct SmemLayout {
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = (BN / CL) * BK * 2;                 // CL == 2: this CTA's half of the B tile
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kOnesOffset = kStages * kStageBytes;         // CS: 8 rows x 128 B of bf16 1.0 (1024-byte aligned)
  static constexpr int kEpiOffset = kOnesOffset + (CS ? 1024 : 0);  // per-epilogue-warp stage (transpose / TMA boxes)
  static constexpr int kEpiWarpBytes = EPI >= 3 ? 2 * kEpiStageBytes : kEpiStageBytes;   // + operand boxes
  static constexpr int kBarOffset = kEpiOffset + kEpiWarps * kEpiWarpBytes;
  static constexpr int kNumBars = 2 * kStages + 4 + 2 * kEpiWarps;  // full, empty, tmem_full[2], tmem_empty[2], operand[warp][2]
  static constexpr int kTotal = kBarOffset + kNumBars * 8 + 16 + 1024 /*alignment slack*/;
  static_assert(kTotal <= 232448, "exceeds the 227 KB dynamic shared memory of sm_100");
};

// EPI: 0 = general epilogue, 1 = lean transposed (coalesced st.global), 2 = lean + TMA store of bf16 boxes,
//      3 / 4 = 2 + residual / aux operand fetched by TMA into per-warp boxes.
// CL : 1 = one CTA per 128 x BN tile (tcgen05.mma.cta_group::1);
//      2 = CTA pairs (2-CTA clusters) on a 256 x BN tile with tcgen05.mma.cta_group::2: CTA r of the pair owns m-tile
//          2u + r (its A rows, its accumulator rows in its own TMEM) and loads only columns [r*BN/2, (r+1)*BN/2) of the
//          B tile — the tensor cores of the pair exchange the B halves, so shared-memory operand reads and L2 -> SM
//          traffic per FLOP drop by a third against CL = 1. The leader (rank 0) issues all MMAs; both CTAs' TMA loads
//          count their bytes on the leader's full barrier; tcgen05.commit multicasts to both CTAs' barriers.
template <int BN, int kStages, bool A_MN, bool B_MN, int EPI, int CL, bool CS = false>
__global__ void __launch_bounds__(kNumThreads, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_opnd, const GemmParams p) {
  using L = SmemLayout<BN, kStages, CL, EPI, CS>;
  constexpr int kAccBufs = CS ? 1 : 2;
  constexpr uint32_t kTmemCols = CS ? (BN == 256 ? 512u : 256u) : (uint32_t)(2 * BN);
  constexpr uint32_t kCsCol = BN;                                     // CS: 16 columns behind the (single) accumulator
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;        // [2]
  uint64_t* opnd_bar = tmem_empty + 2;         // [kEpiWarps][2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(opnd_bar + 2 * kEpiWarps);

  ptx::pdl_launch_dependents();
  const int warp = threadIdx.x >> 5;
  const int crank = CL > 1 ? (int)ptx::cluster_ctarank() : 0;
  const bool leader = crank == 0;
  const int num_m_units = (p.num_m_tiles + CL - 1) / CL;
  const int total_tiles = num_m_units * p.num_n_tiles * p.splits;      // units of CL m-tiles
  const int unit0 = (int)blockIdx.x / CL, unit_stride = (int)gridDim.x / CL;
  constexpr uint16_t kMask = (uint16_t)((1u << CL) - 1);
  constexpr int BNH = BN / CL;                                         // B columns held by this CTA

  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tmap(&tmap_a);
    ptx::prefetch_tmap(&tmap_b);
  }
  if (warp == 1 && ptx::elect_one()) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tmem_full[s], 1);
      ptx::mbar_init(&tmem_empty[s], CL * kEpiWarps);      // one arrival per epilogue warp (of both CTAs when CL == 2)
    }
    for (int s = 0; s < 2 * kEpiWarps; ++s) ptx::mbar_init(&opnd_bar[s], 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    if constexpr (CL == 2) ptx::tmem_alloc_2cta<kTmemCols>(tmem_ptr);
    else ptx::tmem_alloc<kTmemCols>(tmem_ptr);
  }
  if constexpr (CS) {
    if (warp == 3) {                                 // the all-ones B tile: every byte pattern of a swizzle is ones
      reinterpret_cast<uint4*>(smem + L::kOnesOffset)[threadIdx.x & 31] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
      reinterpret_cast<uint4*>(smem + L::kOnesOffset)[32 + (threadIdx.x & 31)] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
      ptx::fence_proxy_async_smem();
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (CL > 1) ptx::cluster_sync();       // peer barriers are initialised before any remote arrive / multicast commit
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  ptx::pdl_wait();                                 // set-up done; from here on global memory of the previous kernel is read

  if (warp == 0) {
    // ===================== TMA producer (every CTA: its A rows and its share of the B tile) =====================
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = unit0; t < total_tiles; t += unit_stride) {
        const int split = t % p.splits;
        const int tile = t / p.splits;
        const int n_tile = tile % p.num_n_tiles;
        const int m_tile = (tile / p.num_n_tiles) * CL + crank;      // may be one past the end for the odd CTA: TMA zero-fills
        const int kb0 = split * p.kblocks_per_split;
        const int kb1 = min(kb0 + p.kblocks_per_split, p.num_k_blocks);
        const int n0 = n_tile * BN + crank * BNH;
        for (int kb = kb0; kb < kb1; ++kb) {
          ptx::mbar_wait_sleep(&empty_bar[stage], phase ^ 1, 32);
          uint8_t* sa = smem + stage * L::kStageBytes;
          uint8_t* sb = sa + L::kABytes;
          if constexpr (CL == 1) {
            ptx::mbar_expect_tx(&full_bar[stage], L::kStageBytes);
            if constexpr (!A_MN) {
              ptx::tma_load_2d(&tmap_a, &full_bar[stage], sa, kb * BK, m_tile * BM);
            } else {
#pragma unroll
              for (int a = 0; a < BM / 64; ++a)
                ptx::tma_load_2d(&tmap_a, &full_bar[stage], sa + a * (BK * 128), m_tile * BM + a * 64, kb * BK);
            }
            if constexpr (!B_MN) {
              ptx::tma_load_2d(&tmap_b, &full_bar[stage], sb, kb * BK, n0);
            } else {
#pragma unroll
              for (int a = 0; a < BNH / 64; ++a)
                ptx::tma_load_2d(&tmap_b, &full_bar[stage], sb + a * (BK * 128), n0 + a * 64, kb * BK);
            }
          } else {
            // both CTAs of the pair count their bytes on the LEADER's full barrier (it issues the MMAs for both)
            if (leader) ptx::mbar_expect_tx(&full_bar[stage], 2 * L::kStageBytes);
            const uint32_t fb = ptx::mapa_u32(&full_bar[stage], 0);
            if constexpr (!A_MN) {
              ptx::tma_load_2d_2cta(&tmap_a, fb, sa, kb * BK, m_tile * BM);
            } else {
#pragma unroll
              for (int a = 0; a < BM / 64; ++a)
                ptx::tma_load_2d_2cta(&tmap_a, fb, sa + a * (BK * 128), m_tile * BM + a * 64, kb * BK);
            }
            if constexpr (!B_MN) {
              ptx::tma_load_2d_2cta(&tmap_b, fb, sb, kb * BK, n0);
            } else {
#pragma unroll
              for (int a = 0; a < BNH / 64; ++a)
                ptx::tma_load_2d_2cta(&tmap_b, fb, sb + a * (BK * 128), n0 + a * 64, kb * BK);
            }
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (CL == 2 && !leader) {
      // the peer CTA of a pair issues no MMAs (the leader's cta_group::2 instructions drive both tensor cores)
    } else if (ptx::elect_one()) {
      // ===================== MMA issuer =====================
      const uint32_t idesc = umma_idesc_bf16(BM * CL, BN, A_MN, B_MN);
      const uint32_t idesc_cs = umma_idesc_bf16(BM * CL, 16, A_MN, false);
      const uint64_t d_ones = umma_smem_desc_sw128(ptx::smem_u32(smem + L::kOnesOffset), 0, 1024);
      constexpr uint32_t kLboA = A_MN ? BK * 128 : 0, kLboB = B_MN ? BK * 128 : 0;
      constexpr uint32_t kAdvA = A_MN ? (16 * 128) >> 4 : (16 * 2) >> 4;   // per UMMA_K = 16, in 16-byte units
      constexpr uint32_t kAdvB = B_MN ? (16 * 128) >> 4 : (16 * 2) >> 4;
      int stage = 0;
      uint32_t phase = 0;
      int iter = 0;
      for (int t = unit0; t < total_tiles; t += unit_stride, ++iter) {
        const int split = t % p.splits;
        const int kb0 = split * p.kblocks_per_split;
        const int kb1 = min(kb0 + p.kblocks_per_split, p.num_k_blocks);
        const int acc = iter % kAccBufs;
        const uint32_t acc_phase = (iter / kAccBufs) & 1;
        const int cs_tile = CS ? (t / p.splits) % p.num_n_tiles : 0;   // CS: this unit takes the k-blocks kb % num_n_tiles == its n-tile
        bool cs_started = false;
        if constexpr (CL == 2) ptx::mbar_wait_cluster(&tmem_empty[acc], acc_phase ^ 1);
        else ptx::mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          if constexpr (CL == 2) ptx::mbar_wait_cluster(&full_bar[stage], phase);
          else ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(smem + stage * L::kStageBytes);
          const uint32_t sb = sa + L::kABytes;
          const uint64_t da = umma_smem_desc_sw128(sa, kLboA, 1024);
          const uint64_t db = umma_smem_desc_sw128(sb, kLboB, 1024);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint32_t accf = (kb > kb0 || k > 0) ? 1u : 0u;
            if constexpr (CL == 2) ptx::umma_f16_2cta(tmem_d, da + (uint64_t)(k * kAdvA), db + (uint64_t)(k * kAdvB), idesc, accf);
            else ptx::umma_f16(tmem_d, da + (uint64_t)(k * kAdvA), db + (uint64_t)(k * kAdvB), idesc, accf);
          }
          if constexpr (CS) {
            // the extra MMAs re-read the A tile from shared memory (+50 % operand traffic for the k-block), so the n-tiles
            // of an m-tile share them round-robin: every unit pays a third, none of them becomes the kernel's critical path
            if (kb % p.num_n_tiles == cs_tile) {
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) {
                const uint32_t accf = (cs_started || k > 0) ? 1u : 0u;
                if constexpr (CL == 2) ptx::umma_f16_2cta(tmem_base + kCsCol, da + (uint64_t)(k * kAdvA), d_ones, idesc_cs, accf);
                else ptx::umma_f16(tmem_base + kCsCol, da + (uint64_t)(k * kAdvA), d_ones, idesc_cs, accf);
              }
              cs_started = true;
            }
          }
          // frees the smem slot (in both CTAs of a pair) when these MMAs retire
          if constexpr (CL == 2) ptx::umma_commit_2cta(&empty_bar[stage], kMask);
          else ptx::umma_commit(&empty_bar[stage]);
          if (kb == kb1 - 1) {
            if constexpr (CL == 2) ptx::umma_commit_2cta(&tmem_full[acc], kMask);
            else ptx::umma_commit(&tmem_full[acc]);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================== epilogue (8 warps: lane quarter = warp % 4, column half = (warp - 4) / 4) =====================
    const int quarter = warp & 3;
    const int half = (warp - 4) >> 2;
    uint8_t* stage = smem + L::kEpiOffset + (warp - 4) * L::kEpiWarpBytes;
    uint32_t box_counter = 0;
    if (EPI >= 2 && (threadIdx.x & 31) == 0) {
      ptx::prefetch_tmap(&tmap_out);
      if (EPI >= 3) ptx::prefetch_tmap(&tmap_opnd);
    }
    int iter = 0;
    for (int t = unit0; t < total_tiles; t += unit_stride, ++iter) {
      const int split = t % p.splits;
      const int tile = t / p.splits;
      const int n_tile = tile % p.num_n_tiles;
      const int m_tile = (tile / p.num_n_tiles) * CL + crank;
      const int acc = iter % kAccBufs;
      const uint32_t acc_phase = (iter / kAccBufs) & 1;
      ptx::mbar_wait_sleep(&tmem_full[acc], acc_phase, 64);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + acc * BN + half * (BN / 2) + ((uint32_t)(quarter * 32) << 16);
      const int n0 = n_tile * BN + half * (BN / 2);
      const long long m0 = (long long)m_tile * BM + quarter * 32;
      if constexpr (EPI >= 2) epi_tile_tma<EPI - 2>(p.epi, &tmap_out, &tmap_opnd, taddr, n0, BN / 2, m0, stage, box_counter, opnd_bar + 2 * (warp - 4));
      else if constexpr (EPI == 1) epi_tile_fast(p.epi, taddr, n0, BN / 2, m0, (long long)p.M, EpiRowIdentity{}, split, stage);
      else epi_tile(p.epi, taddr, n0, BN / 2, m0, (long long)p.M, EpiRowIdentity{}, split, stage);
      if constexpr (CS) {
        if (half == 0) {                             // the row sums of this unit's A rows over ITS k-blocks (lane = row)
          uint32_t r16[16];
          ptx::tmem_ld_x16(tmem_base + kCsCol + ((uint32_t)(quarter * 32) << 16), r16);
          ptx::tmem_ld_wait();
          const int kb0 = split * p.kblocks_per_split, kb1 = min(kb0 + p.kblocks_per_split, p.num_k_blocks);
          const int first = kb0 + ((n_tile - kb0 % p.num_n_tiles) + p.num_n_tiles) % p.num_n_tiles;   // first k-block it owns
          const long long m = m0 + (threadIdx.x & 31);
          if (m < p.M) p.cs_ws[((long long)split * p.num_n_tiles + n_tile) * p.M + m] = first < kb1 ? __uint_as_float(r16[0]) : 0.f;
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if ((threadIdx.x & 31) == 0) {               // the accumulator buffer is drained: tell the (leader's) MMA issuer
        if constexpr (CL == 2) ptx::mbar_arrive_remote(&tmem_empty[acc], 0);
        else ptx::mbar_arrive(&tmem_empty[acc]);
      }
    }
    if constexpr (EPI >= 2) ptx::tma_store_wait_all<0>();     // staged boxes must be read out before the CTA retires
  }

  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (CL > 1) ptx::cluster_sync();       // no CTA exits (or frees TMEM) while its peer may still touch it
  if (warp == 2) {
    ptx::tc_fence_after();
    if constexpr (CL == 2) ptx::tmem_dealloc_2cta<kTmemCols>(tmem_base);
    else ptx::tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// out[m,n] (bf16 or fp32) = (accumulate ? out : 0) + act(alpha * sum_s ws[s,m,n] + bias[n])
// column-sum partials of the CS variant: cs_out[m] = sum_s cs_ws[s, m] (threads past the main range)
__device__ __forceinline__ void reduce_colsum(long long i, const float* __restrict__ cs_ws, int splits, int M, void* __restrict__ cs_out,
                                              int cs_fp32) {   // splits = number of partial rows (split count x n-tiles)
  if (cs_ws == nullptr || i >= M) return;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += cs_ws[(long long)k * M + i];            // `splits` here = split count x n-tiles
  if (cs_fp32) reinterpret_cast<float*>(cs_out)[i] = s;
  else reinterpret_cast<__nv_bfloat16*>(cs_out)[i] = __float2bfloat16(s);
}

__global__ void splitk_reduce_kernel(const float* __restrict__ ws, long long split_stride, int splits, void* __restrict__ out,
                                     long long ld_out, int M, int N, int out_fp32, int accumulate, float alpha,
                                     const __nv_bfloat16* __restrict__ bias, int act, const float* __restrict__ cs_ws,
                                     void* __restrict__ cs_out, int cs_fp32, int cs_parts) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)M * N;
  if (idx >= total) { reduce_colsum(idx - total, cs_ws, cs_parts, M, cs_out, cs_fp32); return; }
  const long long m = idx / N, n = idx % N;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += ws[k * split_stride + idx];
  s *= alpha;
  if (bias) s += __bfloat162float(bias[n]);
  if (act == SFC_ACT_RELU) s = fmaxf(s, 0.f);
  else if (act == SFC_ACT_GELU) s = gelu_erf(s);
  if (out_fp32) {
    float* o = reinterpret_cast<float*>(out) + m * ld_out + n;
    *o = accumulate ? (*o + s) : s;
  } else {
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out) + m * ld_out + n;
    *o = __float2bfloat16(accumulate ? (__bfloat162float(*o) + s) : s);
  }
}

// the common case (weight gradients: no bias / activation, N and ld_out multiples of 4): 4 columns per thread, 16-byte
// loads, four independent partial sums so that the loads of a thread are all in flight together
__global__ void __launch_bounds__(256) splitk_reduce_vec4_kernel(const float4* __restrict__ ws, long long split_stride4, int splits,
                                                                 void* __restrict__ out, long long ld_out, int M, int N4, int out_fp32,
                                                                 int accumulate, const float* __restrict__ cs_ws,
                                                                 void* __restrict__ cs_out, int cs_fp32, int cs_parts) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)M * N4) { reduce_colsum(idx - (long long)M * N4, cs_ws, cs_parts, M, cs_out, cs_fp32); return; }
  const long long m = idx / N4, n = (idx % N4) * 4;
  float4 a[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) a[u] = make_float4(0.f, 0.f, 0.f, 0.f);
  int k = 0;
  for (; k + 4 <= splits; k += 4) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float4 v = __ldg(ws + (long long)(k + u) * split_stride4 + idx);
      a[u].x += v.x; a[u].y += v.y; a[u].z += v.z; a[u].w += v.w;
    }
  }
  for (; k < splits; ++k) {
    const float4 v = __ldg(ws + (long long)k * split_stride4 + idx);
    a[0].x += v.x; a[0].y += v.y; a[0].z += v.z; a[0].w += v.w;
  }
  float4 t;
  t.x = (a[0].x + a[1].x) + (a[2].x + a[3].x); t.y = (a[0].y + a[1].y) + (a[2].y + a[3].y);
  t.z = (a[0].z + a[1].z) + (a[2].z + a[3].z); t.w = (a[0].w + a[1].w) + (a[2].w + a[3].w);
  if (out_fp32) {
    float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + m * ld_out + n);
    if (accumulate) { const float4 p = *o; t.x += p.x; t.y += p.y; t.z += p.z; t.w += p.w; }
    *o = t;
  } else {
    uint2* o = reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out) + m * ld_out + n);
    if (accumulate) {
      const uint2 p = *o;
      t.x += ptx::bf16_lo(p.x); t.y += ptx::bf16_hi(p.x); t.z += ptx::bf16_lo(p.y); t.w += ptx::bf16_hi(p.y);
    }
    *o = make_uint2(ptx::pack_bf16(t.x, t.y), ptx::pack_bf16(t.z, t.w));
  }
}

// smem ring depth: stage = 48 KB (CL 1) / 32 KB (CL 2) at BN 256, half of the B part at BN 128; EPI >= 3 needs 32 KB more
constexpr int gemm_stages(int bn, int cl, int epi) {
  const int stage_kb = 16 + (bn / cl) / 8;
  const int avail_kb = 224 - (epi >= 3 ? 64 : 32);
  const int s = avail_kb / stage_kb;
  return s > 8 ? 8 : s;
}

template <int BN, int kStages, bool A_MN, bool B_MN, int EPI, int CL, bool CS = false>
int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tout, const CUtensorMap& topnd, const GemmParams& p,
                cudaStream_t stream) {
  using L = SmemLayout<BN, kStages, CL, EPI, CS>;
  auto kern = gemm_bf16_kernel<BN, kStages, A_MN, B_MN, EPI, CL, CS>;
  static bool configured = false;
  if (!configured) {
    SFC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    configured = true;
  }
  const int units = ((p.num_m_tiles + CL - 1) / CL) * p.num_n_tiles * p.splits;
  const int max_clusters = sfc_num_sms() / CL;
  const int grid = (units < max_clusters ? units : max_clusters) * CL;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = L::kTotal;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = sfc_pdl_enabled() ? 2 : 1;
  SFC_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, ta, tb, tout, topnd, p));
  return 0;
}

}  // namespace

extern "C" int sfc_gemm_suggest_splits(int M, int N, int K);

extern "C" size_t sfc_gemm_workspace_bytes(int M, int N, int K, int splits) {
  if (splits <= 1) return 0;
  return (size_t)splits * (size_t)M * ((size_t)N + (size_t)sfc_ceil_div(N, 128)) * sizeof(float);   // partial tiles + partial column sums per n-tile
}

// Split-K factor for reductions over the token dimension (wgrad): the output has few tiles, so K is cut into `s`
// slices and the work units (tile pairs x slices, one per 2-CTA cluster) should fill whole waves of the 74 clusters.
// Cost model in units of one k-block of one wave: waves * (k-blocks per slice + fixed per-tile cost) + reduce traffic.
// Column-tile width: 256 (CTA pairs: 256 x 256 per pair) unless more than 15 % of a 256-wide tiling would be padding and a
// 128-wide one pads less (N = 384, ViT-S: 2 x 256 wastes a quarter of the MMAs and epilogue rows, 3 x 128 none). The
// ViT-B / ViT-L widths (768, 1024, 2304, 3072, 4096, 1000, 1536) keep 256.
static int gemm_pick_bn(int N, int K) {
  if (N <= 128) return 128;
  if (K < 256) return 256;     // very short K (ViT-Tiny, K = 192): per-tile fixed costs dominate, fewer larger tiles win (measured)
  const long long pad256 = (long long)sfc_ceil_div(N, 256) * 256, pad128 = (long long)sfc_ceil_div(N, 128) * 128;
  return (pad128 < pad256 && pad256 * 100 > (long long)N * 115) ? 128 : 256;
}

// Split count for a GEMM that also returns the row sums of A over K (ep->colsum_out; wgrad: the bias gradient) inside
// the same kernel, or 0 when no fused variant covers the shape (the caller then uses sfc_colsum). The fused variant is
// the split-K CTA-pair kernel with MN-major operands: M >= 2 row tiles, K >= 2 k-blocks, N % 32 == 0.
extern "C" int sfc_gemm_colsum_splits(int M, int N, int K, int a_mn_major, int b_mn_major) {
  if (!a_mn_major || !b_mn_major) return 0;
  if (sfc_ceil_div(M, BM) < 2 || sfc_ceil_div(K, BK) < 2 || N % 32 != 0 || N < 32) return 0;
  const int s = sfc_gemm_suggest_splits(M, N, K);
  return s < 2 ? 2 : s;
}

extern "C" int sfc_gemm_suggest_splits(int M, int N, int K) {
  const int bn = gemm_pick_bn(N, K);
  const int mt = sfc_ceil_div(M, BM), nt = sfc_ceil_div(N, bn);
  const int kblocks = sfc_ceil_div(K, BK);
  const int cl = mt >= 2 ? 2 : 1;
  const long long units = (long long)sfc_ceil_div(mt, cl) * nt;
  const int slots = sfc_num_sms() / cl;
  if (kblocks < 16) return 1;
  int max_s = kblocks / 8;
  if (max_s > 64) max_s = 64;
  double best = 1e30;
  int best_s = 1;
  for (int s = 1; s <= max_s; ++s) {
    const long long waves = (units * s + slots - 1) / slots;
    const double cost = (double)waves * (sfc_ceil_div(kblocks, s) + 16.0) + (s > 1 ? s * (0.06 * mt * nt) + 8.0 : 0.0);
    if (cost < best) { best = cost; best_s = s; }
  }
  return best_s;
}

extern "C" int sfc_gemm_bf16(const void* A, int a_mn_major, long long lda, const void* B, int b_mn_major, long long ldb,
                             int M, int N, int K, const SfcGemmEpilogue* ep, void* workspace, size_t workspace_bytes,
                             int splits, cudaStream_t stream) {
  SFC_REQUIRE(A && B && ep && ep->out, "sfc_gemm_bf16: null pointer argument");
  SFC_REQUIRE(M > 0 && N > 0 && K > 0, "sfc_gemm_bf16: bad shape M=%d N=%d K=%d", M, N, K);
  SFC_REQUIRE(lda % 8 == 0 && ldb % 8 == 0, "sfc_gemm_bf16: leading dimensions must be multiples of 8 elements (lda=%lld ldb=%lld)", lda, ldb);
  if (splits < 1) splits = 1;
  const int BN = gemm_pick_bn(N, K);
  GemmParams p;
  p.M = M; p.N = N; p.K = K;
  p.num_m_tiles = sfc_ceil_div(M, BM);
  p.num_n_tiles = sfc_ceil_div(N, BN);
  p.num_k_blocks = sfc_ceil_div(K, BK);
  if (splits > p.num_k_blocks) splits = p.num_k_blocks;
  p.kblocks_per_split = sfc_ceil_div(p.num_k_blocks, splits);
  splits = sfc_ceil_div(p.num_k_blocks, p.kblocks_per_split);   // no empty splits
  p.splits = splits;
  EpiParams& e = p.epi;
  e.N = N;
  e.bias = (const __nv_bfloat16*)ep->bias;
  e.residual = (const __nv_bfloat16*)ep->residual;
  e.aux = (const __nv_bfloat16*)ep->aux;
  e.out = ep->out;
  e.out_pre = (__nv_bfloat16*)ep->out_pre;
  e.ld_out = ep->ld_out; e.ld_res = ep->ld_res; e.ld_aux = ep->ld_aux;
  e.alpha = ep->alpha;
  e.act = ep->act; e.aux_mode = ep->aux_mode; e.out_fp32 = ep->out_fp32;
  e.drop_p = ep->drop_p; e.drop_seed = ep->drop_seed; e.drop_epoch = sfc_dropout_epoch_ptr();
  e.split_stride = 0;
  SFC_REQUIRE(e.aux_mode == SFC_AUX_NONE || e.aux != nullptr, "sfc_gemm_bf16: aux_mode set but aux is null");
  SFC_REQUIRE(e.drop_p >= 0.f && e.drop_p < 1.f, "sfc_gemm_bf16: dropout p out of range");

  p.cs_ws = nullptr;
  const bool want_cs = ep->colsum_out != nullptr;
  if (want_cs)
    SFC_REQUIRE(splits > 1 && a_mn_major && b_mn_major && p.num_m_tiles >= 2 && N % 32 == 0,
                "sfc_gemm_bf16: colsum_out needs the split-K MN-major (wgrad) path: ask sfc_gemm_colsum_splits first");
  GemmParams pk = p;
  if (splits > 1) {
    // bias and activation are applied by the reduce kernel (skinny weight-streaming GEMMs: the factorised head at small
    // batch); residual / aux / dropout / pre-activation copies stay single-pass only
    SFC_REQUIRE(!e.residual && e.aux_mode == SFC_AUX_NONE && !e.out_pre && e.drop_p == 0.f && !(ep->accumulate && (e.bias || e.act != SFC_ACT_NONE)),
                "sfc_gemm_bf16: split-K supports alpha, bias and an activation (or plain accumulation) only");
    pk.epi.bias = nullptr; pk.epi.act = SFC_ACT_NONE; pk.epi.alpha = 1.0f;
    const size_t need = (size_t)splits * (size_t)M * (size_t)N * sizeof(float);
    SFC_REQUIRE(workspace && workspace_bytes >= need, "sfc_gemm_bf16: split-K workspace too small (%zu < %zu)", workspace_bytes, need);
    pk.epi.out = workspace; pk.epi.out_fp32 = 1; pk.epi.ld_out = N; pk.epi.split_stride = (long long)M * N;
    if (want_cs) {
      SFC_REQUIRE(workspace_bytes >= need + (size_t)splits * (size_t)p.num_n_tiles * (size_t)M * sizeof(float), "sfc_gemm_bf16: workspace too small for the column sums");
      pk.cs_ws = reinterpret_cast<float*>(workspace) + (size_t)splits * (size_t)M * (size_t)N;
    }
  } else {
    SFC_REQUIRE(!ep->accumulate, "sfc_gemm_bf16: accumulate requires split-K (splits > 1)");
  }

  const bool fast = epi_fast_ok(pk.epi);
  const bool cl2 = fast && p.num_m_tiles >= 2;      // CTA pairs, tcgen05.mma.cta_group::2
  if (want_cs) SFC_REQUIRE(fast, "sfc_gemm_bf16: colsum_out: operands must be 16-byte aligned (fast epilogue)");
  // bf16 output: staged in swizzled smem boxes and stored by TMA (EPI 2); one [M, N] operand (residual or ReLU-mask
  // source) is fetched by TMA the same way (EPI 3 / 4). fp32 output (split-K partials) and residual + aux together keep
  // the transposed epilogue.
  const bool has_res = pk.epi.residual != nullptr, has_aux = pk.epi.aux_mode != SFC_AUX_NONE;
  int epi_mode = fast ? 1 : 0;
  if (fast && !pk.epi.out_fp32 && !(has_res && has_aux)) epi_mode = has_res ? 3 : (has_aux ? 4 : 2);
  CUtensorMap ta, tb, tout, topnd;
  memset(&tout, 0, sizeof(tout));
  memset(&topnd, 0, sizeof(topnd));
  if (epi_mode >= 2) {
    if (int e = sfc_make_tmap_2d_sw(&tout, pk.epi.out, 2, (uint64_t)N, (uint64_t)M, (uint64_t)pk.epi.ld_out * 2, 32, 32, 64)) return e;
  }
  if (epi_mode == 3) {
    if (int e = sfc_make_tmap_2d_sw(&topnd, pk.epi.residual, 2, (uint64_t)N, (uint64_t)M, (uint64_t)pk.epi.ld_res * 2, 32, 32, 64)) return e;
  } else if (epi_mode == 4) {
    if (int e = sfc_make_tmap_2d_sw(&topnd, pk.epi.aux, 2, (uint64_t)N, (uint64_t)M, (uint64_t)pk.epi.ld_aux * 2, 32, 32, 64)) return e;
  }
  if (!a_mn_major) { if (int e = sfc_make_tmap_2d(&ta, A, 2, (uint64_t)K, (uint64_t)M, (uint64_t)lda * 2, BK, BM, true)) return e; }
  else             { if (int e = sfc_make_tmap_2d(&ta, A, 2, (uint64_t)M, (uint64_t)K, (uint64_t)lda * 2, 64, BK, true)) return e; }
  if (!b_mn_major) { if (int e = sfc_make_tmap_2d(&tb, B, 2, (uint64_t)K, (uint64_t)N, (uint64_t)ldb * 2, BK, (uint32_t)(cl2 ? BN / 2 : BN), true)) return e; }
  else             { if (int e = sfc_make_tmap_2d(&tb, B, 2, (uint64_t)N, (uint64_t)K, (uint64_t)ldb * 2, 64, BK, true)) return e; }

  int rc = 0;
#define SFC_DISPATCH2(BN_, F_, CL_)                                                            \
  do {                                                                                          \
    if (!a_mn_major && !b_mn_major) rc = launch_gemm<BN_, gemm_stages(BN_, CL_, F_), false, false, F_, CL_>(ta, tb, tout, topnd, pk, stream); \
    else if (!a_mn_major && b_mn_major) rc = launch_gemm<BN_, gemm_stages(BN_, CL_, F_), false, true, F_, CL_>(ta, tb, tout, topnd, pk, stream); \
    else if (a_mn_major && b_mn_major) rc = launch_gemm<BN_, gemm_stages(BN_, CL_, F_), true, true, F_, CL_>(ta, tb, tout, topnd, pk, stream);  \
    else rc = launch_gemm<BN_, gemm_stages(BN_, CL_, F_), true, false, F_, CL_>(ta, tb, tout, topnd, pk, stream);                        \
  } while (0)
#define SFC_DISPATCH(BN_)                                                                   \
  do {                                                                                      \
    if (cl2 && epi_mode == 4) SFC_DISPATCH2(BN_, 4, 2);                                \
    else if (cl2 && epi_mode == 3) SFC_DISPATCH2(BN_, 3, 2);                           \
    else if (cl2 && epi_mode == 2) SFC_DISPATCH2(BN_, 2, 2);                           \
    else if (cl2) SFC_DISPATCH2(BN_, 1, 2);                                            \
    else if (epi_mode == 4) SFC_DISPATCH2(BN_, 4, 1);                                  \
    else if (epi_mode == 3) SFC_DISPATCH2(BN_, 3, 1);                                  \
    else if (epi_mode == 2) SFC_DISPATCH2(BN_, 2, 1);                                  \
    else if (fast) SFC_DISPATCH2(BN_, 1, 1);                                           \
    else SFC_DISPATCH2(BN_, 0, 1);                                                     \
  } while (0)
  if (want_cs) {
    if (BN == 256) rc = launch_gemm<256, gemm_stages(256, 2, 1), true, true, 1, 2, true>(ta, tb, tout, topnd, pk, stream);
    else rc = launch_gemm<128, gemm_stages(128, 2, 1), true, true, 1, 2, true>(ta, tb, tout, topnd, pk, stream);
  } else if (BN == 256) SFC_DISPATCH(256); else SFC_DISPATCH(128);
#undef SFC_DISPATCH2
#undef SFC_DISPATCH
  if (rc) return rc;

  if (splits > 1) {
    const long long total = (long long)M * N;
    const int threads = 256;
    const bool vec4 = N % 4 == 0 && ep->ld_out % 4 == 0 && !ep->bias && ep->act == SFC_ACT_NONE && ep->alpha == 1.0f &&
                      (reinterpret_cast<uintptr_t>(ep->out) & 15) == 0 && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0;
    const long long extra = want_cs ? M : 0;                  // threads past the main range reduce the column sums
    if (vec4)
      SFC_CUDA_OK(sfc_launch_pdl(splitk_reduce_vec4_kernel, dim3((unsigned)((total / 4 + extra + threads - 1) / threads)), dim3(threads), 0, stream,
          (const float4*)workspace, (long long)M * N / 4, splits, ep->out, ep->ld_out, M, N / 4, ep->out_fp32, ep->accumulate,
          (const float*)pk.cs_ws, ep->colsum_out, ep->colsum_fp32, splits * p.num_n_tiles));
    else
      SFC_CUDA_OK(sfc_launch_pdl(splitk_reduce_kernel, dim3((unsigned)((total + extra + threads - 1) / threads)), dim3(threads), 0, stream,
        (const float*)workspace, (long long)M * N, splits, ep->out, ep->ld_out, M, N, ep->out_fp32, ep->accumulate, ep->alpha,
        (const __nv_bfloat16*)ep->bias, ep->act, (const float*)pk.cs_ws, ep->colsum_out, ep->colsum_fp32, splits * p.num_n_tiles));
    SFC_LAUNCH_OK();
  }
  return 0;
}
