// K2 — fused curve-order patch gather + patch-embedding GEMM (sm_100a).
//
// Replaces, for every tokenizer of the reference,
//     rearrange 'b c (h p1)(w p2) -> b (h w)(p1 p2 c)'  ->  x[:, sfc_indices]  ->  'b (n g) d -> b n (g d)'  ->  Linear
// (/root/reference/src/tokenizers/multiscale/multi_hilbert.py:74-84, _1D/hilbert_embedding1D.py:30-43,
//  _2D/hilbert_embedding.py:80-91 Conv2d(k=s=p) + reorder) by ONE kernel: no permuted im2col tensor is written.
//
//   out[b, t, :] = W . concat_{q<g} patchvec(b, perm[t*g+q]) + bias (+ pos[t, :])
//
// K is ordered (q, c, p1, p2) — the image's own memory order, so every gathered run is a contiguous row segment of a
// patch — and the weight's K axis is permuted once on the host to match (never the data). Two kernels:
//  * patch_embed_tmem_kernel (K <= 768, p % 8 == 0, D % 128 == 0: every ViT-*/16 configuration): the gathered bf16 rows of
//    a 128-token tile are written ONCE into tensor memory (tcgen05.st) and are the A operand of all D / 64 column passes
//    (tcgen05.mma with A from TMEM); weights stream through a TMA ring, multicast inside a 4-CTA cluster.
//  * patch_embed_fwd_kernel (everything else: pixel-level p = 1 tokenizers, small pre-patches, long K): A tiles gathered
//    by 8 producer warps (two groups alternating pipeline stages) into the 128-byte-swizzled K-major shared-memory
//    layout, weights by TMA, double-buffered TMEM accumulators.
// Both convert fp32 -> bf16 in registers and fuse bias (+ position rows) in a row-per-lane epilogue.
#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "sfcvit.h"

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kThreads = 512;      // warps 0-3 control, 4-7 epilogue, 8-15 gather producers
constexpr int kEpiThreads = 128;
constexpr int kProdWarpsPerGroup = 4;
constexpr int kMaxTblKb = 64;      // k-blocks covered by the precomputed chunk-offset table (K <= 4096)

struct PatchParams {
  const void* img;
  const int* perm;       // [ntok * g] flat pre-patch index r*gw + c in curve order
  int B, C, H, W, p, g, gw;
  int in_fmt;            // SFC_IMG_F32_NCHW / SFC_IMG_BF16_NCHW / SFC_IMG_U8_NHWC
  int dual_epi;          // always 1: a runtime operand of the kernel's `dual` test (see patch_embed_fwd_kernel)
  int wide_ld, wide_st;  // 256-bit accesses: fp32 chunk = one 32-byte load (image 32-byte aligned), output rows 32-byte aligned
  int row_split;         // p == 4 (NCHW): an 8-element chunk is two 4-element patch rows, the second `row_split` (= W)
                         // elements after the first; 0 = the chunk is one contiguous run
  int ntok, K, Kpad;
  long long M;           // B * ntok
  int num_m_tiles, num_n_tiles, num_k_blocks;
  int rows_per_img, tok_off;
  EpiParams epi;         // epi.residual = position embedding rows (indexed by token), may be null
};

template <int BN, int kStages>
struct PeSmem {
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kEpiOffset = kStages * kStageBytes;          // 4 epilogue warps x transpose stage
  static constexpr int kBarOffset = kEpiOffset + 4 * kEpiStageBytes;
  static constexpr int kTblOffset = kBarOffset + (2 * kStages + 4) * 8 + 16;       // int32 [kMaxTblKb * 8 + kMaxTblKb]
  static constexpr int kTotal = kTblOffset + kMaxTblKb * 9 * 4 + 1024;
  static_assert(kTotal <= 232448, "exceeds the 227 KB dynamic shared memory of sm_100");
};

// accumulator row m = image * ntok + token  ->  output row (image-major, token offset) and position-embedding row
struct PeRowMap {
  int ntok, rows_per_img, tok_off;
  __device__ __forceinline__ void map(long long m, long long& m_out, long long& m_res) const {
    const long long bimg = m / ntok, tok = m % ntok;
    m_out = bimg * rows_per_img + tok_off + tok;
    m_res = tok;
  }
};

__device__ __forceinline__ uint4 pack8f(const float* f) {
  uint4 u;
  u.x = ptx::pack_bf16(f[0], f[1]); u.y = ptx::pack_bf16(f[2], f[3]);
  u.z = ptx::pack_bf16(f[4], f[5]); u.w = ptx::pack_bf16(f[6], f[7]);
  return u;
}

// Input formats (template parameter IN): 0 = fp32 NCHW, 1 = bf16 NCHW, 2 = uint8 NHWC (decoded image bytes; the
// (x / 255 - mean) / std normalisation is folded into the weight and bias on the host, the kernel converts exactly).
constexpr int IN_F32 = 0, IN_BF16 = 1, IN_U8 = 2;

struct ChunkRaw { uint4 a, b; };      // 8 consecutive K elements as loaded: fp32 a+b, bf16 a, uint8 a.x / a.y

template <int IN>
__device__ __forceinline__ void chunk_load(ChunkRaw& r, const void* img, long long off, int row_split = 0, bool wide = false) {
  if constexpr (IN == IN_BF16) {
    const __nv_bfloat16* src = reinterpret_cast<const __nv_bfloat16*>(img) + off;
    if (row_split == 0) {
      r.a = __ldg(reinterpret_cast<const uint4*>(src));
    } else {
      const uint2 lo = __ldg(reinterpret_cast<const uint2*>(src)), hi = __ldg(reinterpret_cast<const uint2*>(src + row_split));
      r.a = make_uint4(lo.x, lo.y, hi.x, hi.y);
    }
  } else if constexpr (IN == IN_F32) {
    const float* src = reinterpret_cast<const float*>(img) + off;
    if (wide) {                                  // warp-uniform: the 8 floats are one aligned 32-byte sector
      ptx::ldg256(src, r.a, r.b);
    } else {
      r.a = __ldg(reinterpret_cast<const uint4*>(src));
      r.b = __ldg(reinterpret_cast<const uint4*>(src + (row_split == 0 ? 4 : row_split)));
    }
  } else {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const uint8_t*>(img) + off));
    r.a.x = v.x; r.a.y = v.y;
  }
}

// byte k of w as an exact float: 0x4B000000 | byte is 2^23 + byte
__device__ __forceinline__ float u8_to_f32(uint32_t w, uint32_t sel) {
  return __uint_as_float(__byte_perm(w, 0x4B000000u, sel)) - 8388608.0f;
}

template <int IN>
__device__ __forceinline__ uint4 chunk_pack(const ChunkRaw& r) {
  uint4 o;
  if constexpr (IN == IN_BF16) {
    o = r.a;
  } else if constexpr (IN == IN_F32) {
    o.x = ptx::pack_bf16(__uint_as_float(r.a.x), __uint_as_float(r.a.y));
    o.y = ptx::pack_bf16(__uint_as_float(r.a.z), __uint_as_float(r.a.w));
    o.z = ptx::pack_bf16(__uint_as_float(r.b.x), __uint_as_float(r.b.y));
    o.w = ptx::pack_bf16(__uint_as_float(r.b.z), __uint_as_float(r.b.w));
  } else {
    o.x = ptx::pack_bf16(u8_to_f32(r.a.x, 0x7650u), u8_to_f32(r.a.x, 0x7651u));
    o.y = ptx::pack_bf16(u8_to_f32(r.a.x, 0x7652u), u8_to_f32(r.a.x, 0x7653u));
    o.z = ptx::pack_bf16(u8_to_f32(r.a.y, 0x7650u), u8_to_f32(r.a.y, 0x7651u));
    o.w = ptx::pack_bf16(u8_to_f32(r.a.y, 0x7652u), u8_to_f32(r.a.y, 0x7653u));
  }
  return o;
}

// Chunk-offset table (vectorised path, p % 8 == 0): K is ordered (q, c, p1, p2), so the image offset of the 8-element
// chunk j of k-block kb relative to the origin of pre-patch q is the same for EVERY token:
//   tbl[kb * 8 + j] = c * H * W + p1 * W + p2   (or -1 past K),   tblq[kb] = q   (p * p % 64 == 0: one (q, c) per k-block)
// It is built once per CTA, which leaves one add per 16-byte load in the gather loop (no per-chunk divisions).
__device__ __forceinline__ void build_chunk_table(const PatchParams& pp, int* tbl, int* tblq) {
  const int p = pp.p;
  for (int i = threadIdx.x; i < pp.num_k_blocks * 8; i += blockDim.x) {
    const int k0 = i * 8;
    int v = -1;
    if (k0 < pp.K) {
      if (pp.in_fmt == SFC_IMG_U8_NHWC) {            // K ordered (q, p1, p2, c): a patch row is p * C contiguous bytes
        const int rl = p * pp.C, e = k0 % rl, p1 = (k0 / rl) % p;
        v = p1 * pp.W * pp.C + e;
      } else {
        const int p2 = k0 % p, t1 = k0 / p, p1 = t1 % p, t2 = t1 / p, c = t2 % pp.C;
        v = c * pp.H * pp.W + p1 * pp.W + p2;
      }
    }
    tbl[i] = v;
  }
  for (int kb = threadIdx.x; kb < pp.num_k_blocks; kb += blockDim.x) tblq[kb] = (kb * 64) / (p * p * pp.C);
}

// element offset of the origin of pre-patch q of token row m (m < M)
__device__ __forceinline__ long long patch_origin(const PatchParams& pp, long long m, int q) {
  const int b = (int)(m / pp.ntok);
  const int t = (int)(m % pp.ntok);
  const int idx = __ldg(pp.perm + t * pp.g + q);
  const int r = idx / pp.gw, cc = idx % pp.gw;
  if (pp.in_fmt == SFC_IMG_U8_NHWC) return ((long long)b * pp.H * pp.W + (long long)(r * pp.p) * pp.W + cc * pp.p) * pp.C;
  return (long long)b * pp.C * pp.H * pp.W + (long long)(r * pp.p) * pp.W + cc * pp.p;
}

// Gathers the 64 K-elements [kb*64, kb*64+64) of one token row into its 128-byte swizzled smem row (vectorised path).
// `origin` = patch_origin of the k-block's q for this row (ignored when !row_ok).
template <int IN>
__device__ __forceinline__ void gather_row_vec(const PatchParams& pp, bool row_ok, long long origin, int row, int kb, const int* tbl,
                                               uint8_t* smem_a) {
  uint8_t* srow = smem_a + row * 128;
  const int sw = row & 7;
  ChunkRaw raw[8];
  int off[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    off[j] = tbl[kb * 8 + j];                     // broadcast shared-memory read
    if (row_ok && off[j] >= 0) chunk_load<IN>(raw[j], pp.img, origin + off[j], pp.row_split, pp.wide_ld != 0);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    uint4 o = make_uint4(0, 0, 0, 0);
    if (row_ok && off[j] >= 0) o = chunk_pack<IN>(raw[j]);
    *reinterpret_cast<uint4*>(srow + ((j ^ sw) << 4)) = o;
  }
}

// Generic element-wise gather (any p, g): pixel-level tokenizers (p = 1) and small pre-patches.
template <int IN>
__device__ __forceinline__ void gather_row(const PatchParams& pp, long long m, int row, int kb, uint8_t* smem_a) {
  static_assert(IN != IN_U8, "uint8 NHWC input is served by the vectorised paths only");
  constexpr bool BF16IN = IN == IN_BF16;
  uint8_t* srow = smem_a + row * 128;
  const int sw = row & 7;
  if (m >= pp.M) {
#pragma unroll
    for (int j = 0; j < 8; ++j) *reinterpret_cast<uint4*>(srow + ((j ^ sw) << 4)) = make_uint4(0, 0, 0, 0);
    return;
  }
  const int b = (int)(m / pp.ntok);
  const int t = (int)(m % pp.ntok);
  const int p = pp.p;
  const long long plane = (long long)pp.H * pp.W;
  {
    const int k_begin = kb * 64;
    int p2 = k_begin % p;
    int t1 = k_begin / p;
    int p1 = t1 % p;
    int t2 = t1 / p;
    int c = t2 % pp.C;
    int q = t2 / pp.C;
    int idx = (k_begin < pp.K) ? __ldg(pp.perm + t * pp.g + q) : 0;
    int r = idx / pp.gw, cc = idx % pp.gw;
#pragma unroll 1
    for (int j = 0; j < 8; ++j) {
      float f[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = k_begin + j * 8 + e;
        f[e] = 0.f;
        if (k < pp.K) {
          const long long off = ((long long)b * pp.C + c) * plane + (long long)(r * p + p1) * pp.W + cc * p + p2;
          if constexpr (BF16IN) f[e] = __bfloat162float(__ldg(reinterpret_cast<const __nv_bfloat16*>(pp.img) + off));
          else f[e] = __ldg(reinterpret_cast<const float*>(pp.img) + off);
          if (++p2 == p) {
            p2 = 0;
            if (++p1 == p) {
              p1 = 0;
              if (++c == pp.C) {
                c = 0;
                ++q;
                if (k + 1 < pp.K) {
                  idx = __ldg(pp.perm + t * pp.g + q);
                  r = idx / pp.gw; cc = idx % pp.gw;
                }
              }
            }
          }
        }
      }
      *reinterpret_cast<uint4*>(srow + ((j ^ sw) << 4)) = pack8f(f);
    }
  }
}

template <int BN, int kStages, bool VEC, int IN, bool FAST_EPI>
__global__ void __launch_bounds__(kThreads, 1)
patch_embed_fwd_kernel(const __grid_constant__ CUtensorMap tmap_w, const PatchParams pp) {
  static_assert(kStages % 2 == 0, "producer groups alternate stages by parity");
  using L = PeSmem<BN, kStages>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  int* tbl = reinterpret_cast<int*>(smem + L::kTblOffset);
  int* tblq = tbl + kMaxTblKb * 8;

  const int warp = threadIdx.x >> 5;
  const int total_tiles = pp.num_m_tiles * pp.num_n_tiles;
  // One k-block per tile (K <= 64: /4 pre-patches of small images): a tile costs one gather round but a full-width
  // epilogue, so the second producer group converts the upper half of the tile's columns instead of idling
  // (ViT-Tiny/4, B = 8192, same box: 0.198 -> 0.160 ms).
  // pp.dual_epi is always 1, but testing it keeps ptxas's register allocation of the row-per-lane epilogue: with `dual`
  // derived from num_k_blocks alone the FAST_EPI instantiations spill 48 / 60 bytes instead of 28 / 40, inside the
  // chunk loop, and bf16 ViT-Tiny/4 (B = 8192) slows from 0.110 to 0.127 ms (B200, 1000 W).
  const bool dual = FAST_EPI && pp.num_k_blocks == 1 && pp.dual_epi != 0;
  if constexpr (VEC) build_chunk_table(pp, tbl, tblq);

  if (warp == 0 && ptx::elect_one()) ptx::prefetch_tmap(&tmap_w);
  if (warp == 1 && ptx::elect_one()) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1 + kProdWarpsPerGroup);   // TMA expect_tx arrive + one arrive per producer warp
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tmem_full[s], 1);
      ptx::mbar_init(&tmem_empty[s], dual ? 2 * kEpiThreads : kEpiThreads);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc<2 * BN>(tmem_ptr);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer: weights =====================
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int n_tile = tile % pp.num_n_tiles;
        for (int kb = 0; kb < pp.num_k_blocks; ++kb) {
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sb = smem + stage * L::kStageBytes + L::kABytes;
          ptx::mbar_expect_tx(&full_bar[stage], L::kBBytes);
          ptx::tma_load_2d(&tmap_w, &full_bar[stage], sb, kb * BK, n_tile * BN);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (ptx::elect_one()) {
      const uint32_t idesc = umma_idesc_bf16(BM, BN, false, false);
      int stage = 0;
      uint32_t phase = 0;
      int iter = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++iter) {
        const int acc = iter & 1;
        const uint32_t acc_phase = (iter >> 1) & 1;
        ptx::mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int kb = 0; kb < pp.num_k_blocks; ++kb) {
          ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(smem + stage * L::kStageBytes);
          const uint32_t sb = sa + L::kABytes;
          const uint64_t da = umma_smem_desc_sw128(sa, 0, 1024);
          const uint64_t db = umma_smem_desc_sw128(sb, 0, 1024);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            ptx::umma_f16(tmem_d, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb > 0 || k > 0) ? 1u : 0u);
          ptx::umma_commit(&empty_bar[stage]);
          if (kb == pp.num_k_blocks - 1) ptx::umma_commit(&tmem_full[acc]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if ((warp >= 4 && warp < 8) || (dual && warp >= 12)) {
    // ===================== epilogue (dual: warps 12-15 take the upper column half of every tile) =====================
    const int ewarp = warp & 3;                  // TMEM lane quarter
    const int set = warp >= 12 ? 1 : 0;
    uint8_t* stage = smem + L::kEpiOffset + ewarp * kEpiStageBytes + set * (kEpiStageBytes / 2);
    PeRowMap rm{pp.ntok, pp.rows_per_img, pp.tok_off};
    int iter = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++iter) {
      const int n_tile = tile % pp.num_n_tiles;
      const int m_tile = tile / pp.num_n_tiles;
      const int acc = iter & 1;
      const uint32_t acc_phase = (iter >> 1) & 1;
      int col0 = 0, ncols = BN;
      if (dual) {
        const int valid = min(BN, pp.epi.N - n_tile * BN);
        const int lower = ((valid + 31) / 32 + 1) / 2 * 32;          // columns of set 0 (whole 32-column chunks)
        col0 = set ? lower : 0;
        ncols = set ? BN - lower : lower;
      }
      ptx::mbar_wait(&tmem_full[acc], acc_phase);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + acc * BN + col0 + ((uint32_t)(ewarp * 32) << 16);
      if constexpr (FAST_EPI) epi_tile_direct(pp.epi, taddr, n_tile * BN + col0, ncols, (long long)m_tile * BM + ewarp * 32, pp.M, rm, 0, reinterpret_cast<float*>(stage), pp.wide_st != 0);
      else epi_tile(pp.epi, taddr, n_tile * BN, BN, (long long)m_tile * BM + ewarp * 32, pp.M, rm, 0, stage);
      ptx::tc_fence_before();
      ptx::mbar_arrive(&tmem_empty[acc]);
    }
  } else if (warp >= 8) {
    // ===================== gather producers (2 groups x 4 warps, alternate stages) =====================
    const int pw = warp - 8;
    const int group = pw / kProdWarpsPerGroup;
    const int row = (pw % kProdWarpsPerGroup) * 32 + (threadIdx.x & 31);
    int it = 0;                                   // running k-block counter of this CTA
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int m_tile = tile / pp.num_n_tiles;
      const long long m = (long long)m_tile * BM + row;
      const bool row_ok = m < pp.M;
      int cur_q = -1;
      long long origin = 0;
      for (int kb = 0; kb < pp.num_k_blocks; ++kb, ++it) {
        if (!dual && (it & 1) != group) continue;           // dual: group 0 gathers every tile
        const int stage = it % kStages;
        const uint32_t phase = (it / kStages) & 1;
        if constexpr (VEC) {
          const int q = tblq[kb];
          if (row_ok && q != cur_q && q < pp.g) { origin = patch_origin(pp, m, q); cur_q = q; }
        }
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
        if constexpr (VEC) gather_row_vec<IN>(pp, row_ok, origin, row, kb, tbl, smem + stage * L::kStageBytes);
        else if constexpr (IN != IN_U8) gather_row<IN>(pp, m, row, kb, smem + stage * L::kStageBytes);
        ptx::fence_proxy_async_smem();            // generic-proxy smem writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (ptx::elect_one()) ptx::mbar_arrive(&full_bar[stage]);
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<2 * BN>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// TMEM-resident variant (K <= 768, vectorised gather): the gathered, converted patch rows of a 128-token tile are written
// ONCE into tensor memory (tcgen05.st: token = TMEM lane, two bf16 per column, K / 2 <= 384 columns) and serve as the A
// operand of every n-pass (tcgen05.mma with A from TMEM) — the image is gathered exactly once per token instead of once
// per 256-column n-tile, and no shared memory is spent on A. D = 2 x 64 columns (one accumulator per MMA issuer), the
// weights (B) stream through a 12-stage TMA ring of [64 features x 128 k] tiles (two 8 KB SWIZZLE_128B slabs).
//   warp 0 : TMA (weights)   warps 1, 3 : MMA issuers (even / odd passes)   warp 2 : TMEM allocator   warps 4-7 : epilogue
//   warps 8-15 : gather producers, warp w owns TMEM lane quarter w % 4; the two warps of a quarter alternate k-blocks
// A 128 x 64 x 16 MMA keeps the tensor pipe busy for 32 clocks, far less than one thread needs to wait for a stage and
// issue it, hence eight MMAs per barrier round trip and two issuers, each owning one accumulator and every other pass.
// The epilogue releases its accumulator as soon as tcgen05.ld has landed in registers, before converting and storing.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kTmBN = 64;            // output columns per pass
constexpr int kTmStages = 12;        // two passes of K = 768 in flight: one per MMA issuer
constexpr int kTmMaxKb = 12;         // K <= 768
constexpr int kTmDCol = 384;         // accumulators live in TMEM columns [384, 512)
constexpr int kTmMaxD = 2048;        // bias is staged once as fp32

struct PeTmSmem {
  static constexpr int kSlabBytes = kTmBN * BK * 2;                    // 8 KB: 64 features x 64 k
  static constexpr int kStageBytes = 2 * kSlabBytes;                   // two consecutive k-blocks
  static constexpr int kBiasOffset = kTmStages * kStageBytes;
  static constexpr int kBarOffset = kBiasOffset + kTmMaxD * 4;
  static constexpr int kNumBars = 2 * kTmStages + 2 * kTmMaxKb + 4;    // b_full/empty, a_full/empty per k-block, d_full/empty[2]
  static constexpr int kTblOffset = kBarOffset + kNumBars * 8 + 16;
  static constexpr int kTotal = kTblOffset + kMaxTblKb * 9 * 4 + 1024;
  static_assert(kTotal <= 232448, "exceeds the 227 KB dynamic shared memory of sm_100");
};

template <int IN, int CL>
__global__ void __launch_bounds__(kThreads, 1)
patch_embed_tmem_kernel(const __grid_constant__ CUtensorMap tmap_w, const PatchParams pp) {
  using L = PeTmSmem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* bias_s = reinterpret_cast<float*>(smem + L::kBiasOffset);
  uint64_t* b_full = reinterpret_cast<uint64_t*>(smem + L::kBarOffset);
  uint64_t* b_empty = b_full + kTmStages;
  uint64_t* a_full = b_empty + kTmStages;      // [kTmMaxKb]
  uint64_t* a_empty = a_full + kTmMaxKb;       // [kTmMaxKb]
  uint64_t* d_full = a_empty + kTmMaxKb;       // [2]
  uint64_t* d_empty = d_full + 2;              // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(d_empty + 2);
  int* tbl = reinterpret_cast<int*>(smem + L::kTblOffset);
  int* tblq = tbl + kMaxTblKb * 8;

  const int warp = threadIdx.x >> 5;
  const int nkb = pp.num_k_blocks;
  const int nst = (nkb + 1) >> 1;              // ring stages per pass (the last one holds a single k-block when nkb is odd)
  const int npass = pp.num_n_tiles;            // D / 64, even
  // every CTA of a cluster walks the same number of tiles: the weight stream is shared (multicast) and runs in lock step;
  // a CTA whose tile index is past the end gathers zeros and stores nothing
  const int rounds = (pp.num_m_tiles + (int)gridDim.x - 1) / (int)gridDim.x;
  const uint32_t crank = CL > 1 ? ptx::cluster_ctarank() : 0;
  constexpr uint16_t kMcMask = (uint16_t)((1u << CL) - 1);
  build_chunk_table(pp, tbl, tblq);
  for (int i = threadIdx.x; i < pp.epi.N; i += kThreads) bias_s[i] = pp.epi.bias ? __bfloat162float(pp.epi.bias[i]) : 0.0f;
  if (warp == 0 && ptx::elect_one()) ptx::prefetch_tmap(&tmap_w);
  if (warp == 1 && ptx::elect_one()) {
    for (int s = 0; s < kTmStages; ++s) { ptx::mbar_init(&b_full[s], 1); ptx::mbar_init(&b_empty[s], CL); }
    for (int k = 0; k < kTmMaxKb; ++k) { ptx::mbar_init(&a_full[k], 4); ptx::mbar_init(&a_empty[k], 2); }
    for (int s = 0; s < 2; ++s) { ptx::mbar_init(&d_full[s], 1); ptx::mbar_init(&d_empty[s], kEpiThreads); }
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc<512>(tmem_ptr);
  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (CL > 1) ptx::cluster_sync();   // peers' barriers are initialised before any multicast lands on them
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer: weight slabs [64 features x 64 k], each CTA multicasts its 64 / CL rows =====================
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int r = 0; r < rounds; ++r) {
        for (int n = 0; n < npass; ++n) {
          for (int st = 0; st < nst; ++st) {
            const int nslab = (2 * st + 1 < nkb) ? 2 : 1;
            ptx::mbar_wait_sleep(&b_empty[stage], phase ^ 1, 32);      // every CTA of the cluster has consumed this stage
            ptx::mbar_expect_tx(&b_full[stage], nslab * L::kSlabBytes);
            for (int h = 0; h < nslab; ++h) {
              uint8_t* dst = smem + stage * L::kStageBytes + h * L::kSlabBytes;
              if constexpr (CL > 1)
                ptx::tma_load_2d_mc(&tmap_w, &b_full[stage], dst + crank * (L::kSlabBytes / CL), (2 * st + h) * BK,
                                    n * kTmBN + (int)crank * (kTmBN / CL), kMcMask);
              else
                ptx::tma_load_2d(&tmap_w, &b_full[stage], dst, (2 * st + h) * BK, n * kTmBN);
            }
            if (++stage == kTmStages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1 || warp == 3) {
    // ===================== MMA issuers (A from TMEM): issuer i runs passes n = i, i + 2, ... into accumulator i =====================
    if (ptx::elect_one()) {
      const int iss = warp >> 1;
      const uint32_t idesc = umma_idesc_bf16(BM, kTmBN, false, false);
      const uint32_t tmem_d = tmem_base + kTmDCol + iss * kTmBN;
      int stage = iss * nst;                     // ring slots are handed out pass-major, so the issuers leapfrog by nst
      uint32_t phase = 0;
      if (stage >= kTmStages) { stage -= kTmStages; phase ^= 1; }
      int j = 0;                                 // passes issued by this thread
      for (int it = 0; it < rounds; ++it) {
        for (int n = iss; n < npass; n += 2, ++j) {
          ptx::mbar_wait(&d_empty[iss], (j & 1) ^ 1);
          ptx::tc_fence_after();
          for (int st = 0; st < nst; ++st) {
            const int nslab = (2 * st + 1 < nkb) ? 2 : 1;
            if (n == iss) {                                               // this tile's rows of the k-blocks are in TMEM
              ptx::mbar_wait(&a_full[2 * st], it & 1);
              if (nslab == 2) ptx::mbar_wait(&a_full[2 * st + 1], it & 1);
            }
            ptx::mbar_wait(&b_full[stage], phase);
            ptx::tc_fence_after();
            const uint64_t db = umma_smem_desc_sw128(ptx::smem_u32(smem + stage * L::kStageBytes), 0, 1024);
            const uint32_t ta = tmem_base + st * 64;
#pragma unroll
            for (int k = 0; k < 4; ++k) ptx::umma_f16_ts(tmem_d, ta + k * 8, db + (uint64_t)(k * 2), idesc, (st > 0 || k > 0) ? 1u : 0u);
            if (nslab == 2) {
#pragma unroll
              for (int k = 0; k < 4; ++k) ptx::umma_f16_ts(tmem_d, ta + 32 + k * 8, db + (uint64_t)(L::kSlabBytes / 16 + k * 2), idesc, 1u);
            }
            if constexpr (CL > 1) ptx::umma_commit_mc(&b_empty[stage], kMcMask);
            else ptx::umma_commit(&b_empty[stage]);
            if (n >= npass - 2) {                                         // this issuer's last read of the tile's k-blocks
              ptx::umma_commit(&a_empty[2 * st]);
              if (nslab == 2) ptx::umma_commit(&a_empty[2 * st + 1]);
            }
            if (++stage == kTmStages) { stage = 0; phase ^= 1; }
          }
          ptx::umma_commit(&d_full[iss]);
          stage += nst;                          // the other issuer's pass
          if (stage >= kTmStages) { stage -= kTmStages; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp >= 4 && warp < 8) {
    // ===================== epilogue: lane = token row, 64 columns per pass =====================
    const int ewarp = warp - 4;
    const int lane = threadIdx.x & 31;
    const EpiParams& e = pp.epi;
    const bool has_res = e.residual != nullptr, wide_st = pp.wide_st != 0;
    PeRowMap rm{pp.ntok, pp.rows_per_img, pp.tok_off};
    int pass = 0;
    for (int r = 0; r < rounds; ++r) {
      const long long m = ((long long)blockIdx.x + (long long)r * gridDim.x) * BM + ewarp * 32 + lane;
      const bool ok = m < pp.M;                                      // past-the-end tiles / rows store nothing
      long long m_out, m_res;
      rm.map(ok ? m : 0, m_out, m_res);
      const uint4* resp = reinterpret_cast<const uint4*>(e.residual + m_res * e.ld_res);
      uint4* outp = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(e.out) + m_out * e.ld_out);
      for (int n = 0; n < npass; ++n, ++pass) {
        const int acc = pass & 1;
        uint4 pos[8];
        if (has_res && ok) {
#pragma unroll
          for (int q = 0; q < 8; ++q) pos[q] = __ldg(resp + n * 8 + q);
        }
        ptx::mbar_wait_sleep(&d_full[acc], (pass >> 1) & 1, 32);
        ptx::tc_fence_after();
        const uint32_t taddr = tmem_base + kTmDCol + acc * kTmBN + ((uint32_t)(ewarp * 32) << 16);
        uint32_t raw[64];
        ptx::tmem_ld_x32(taddr, raw);
        ptx::tmem_ld_x32(taddr + 32, raw + 32);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        ptx::mbar_arrive(&d_empty[acc]);                             // the accumulator is in registers: release it now
        if (ok) {
          const float* bs = bias_s + n * kTmBN;
          uint4 prev = make_uint4(0, 0, 0, 0);
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float v[8];
            const float4 b0 = *reinterpret_cast<const float4*>(bs + q * 8);         // broadcast reads
            const float4 b1 = *reinterpret_cast<const float4*>(bs + q * 8 + 4);
            v[0] = __uint_as_float(raw[q * 8 + 0]) + b0.x; v[1] = __uint_as_float(raw[q * 8 + 1]) + b0.y;
            v[2] = __uint_as_float(raw[q * 8 + 2]) + b0.z; v[3] = __uint_as_float(raw[q * 8 + 3]) + b0.w;
            v[4] = __uint_as_float(raw[q * 8 + 4]) + b1.x; v[5] = __uint_as_float(raw[q * 8 + 5]) + b1.y;
            v[6] = __uint_as_float(raw[q * 8 + 6]) + b1.z; v[7] = __uint_as_float(raw[q * 8 + 7]) + b1.w;
            if (has_res) {
              float f[8];
              epi_unpack8(pos[q], f);
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] += f[i];
            }
            const uint4 o = epi_pack8(v);
            if (!wide_st) outp[n * 8 + q] = o;
            else if (q & 1) ptx::stg256(outp + n * 8 + q - 1, prev, o);       // one full 32-byte sector per lane
            else prev = o;
          }
        }
      }
    }
  } else if (warp >= 8) {
    // ===================== gather producers: image -> registers -> bf16 -> TMEM =====================
    const int pw = warp - 8;
    const int group = pw >> 2;                     // the two warps of a lane quarter alternate k-blocks
    const int quarter = pw & 3;                    // == warp % 4: the TMEM lanes this warp may write
    const int lane = threadIdx.x & 31;
    const int row = quarter * 32 + lane;
    const uint32_t t_a = tmem_base + ((uint32_t)(quarter * 32) << 16);
    for (int it = 0; it < rounds; ++it) {
      const long long m = ((long long)blockIdx.x + (long long)it * gridDim.x) * BM + row;
      const bool row_ok = m < pp.M;
      int cur_q = -1;
      long long origin = 0;
      for (int kb = group; kb < nkb; kb += 2) {
        const int q = tblq[kb];
        if (row_ok && q != cur_q && q < pp.g) { origin = patch_origin(pp, m, q); cur_q = q; }
        ChunkRaw raw[8];
        int off[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          off[j] = tbl[kb * 8 + j];
          if (row_ok && off[j] >= 0) chunk_load<IN>(raw[j], pp.img, origin + off[j], 0, pp.wide_ld != 0);
        }
        uint32_t packed[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          uint4 o = make_uint4(0, 0, 0, 0);
          if (row_ok && off[j] >= 0) o = chunk_pack<IN>(raw[j]);
          packed[j * 4 + 0] = o.x; packed[j * 4 + 1] = o.y; packed[j * 4 + 2] = o.z; packed[j * 4 + 3] = o.w;
        }
        ptx::mbar_wait_sleep(&a_empty[kb], (it & 1) ^ 1, 64);   // long wait (the previous tile's last passes)
        ptx::tc_fence_after();
        ptx::tmem_st_x32(t_a + kb * 32, packed);
        ptx::tmem_st_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&a_full[kb]);
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (CL > 1) ptx::cluster_sync();   // no CTA leaves while a peer may still multicast into it
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

template <int IN, int CL>
int launch_pe_tmem(const void* Wk, int D, const PatchParams& pp, cudaStream_t stream) {
  CUtensorMap tw;
  if (int err = sfc_make_tmap_2d(&tw, Wk, 2, (uint64_t)pp.Kpad, (uint64_t)D, (uint64_t)pp.Kpad * 2, BK, (uint32_t)(kTmBN / CL), true)) return err;
  auto kern = patch_embed_tmem_kernel<IN, CL>;
  static int max_clusters = 0;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = PeTmSmem::kTotal;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (max_clusters == 0) {
    SFC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, PeTmSmem::kTotal));
    cfg.gridDim = dim3(sfc_num_sms() / CL * CL);
    int n = 0;
    SFC_CUDA_OK(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));     // GPC boundaries can leave a few SMs out of 4-CTA clusters
    max_clusters = n > 0 ? n : 1;
  }
  const int want = sfc_ceil_div(pp.num_m_tiles, CL);
  cfg.gridDim = dim3((want < max_clusters ? want : max_clusters) * CL);
  SFC_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, tw, pp));
  return 0;
}

// A-only gather: writes the curve-ordered im2col matrix A[M, Kpad] (bf16). Used by the backward pass
// (weight gradient) only; the forward never materialises it.
template <int IN, bool VEC>
__global__ void __launch_bounds__(256) patch_gather_kernel(const PatchParams pp, __nv_bfloat16* __restrict__ A) {
  constexpr bool BF16IN = IN == IN_BF16;
  const int cpr = pp.Kpad / 8;                                   // 8-element chunks per row
  const long long total = pp.M * (long long)cpr;
  const int p = pp.p;
  const long long plane = (long long)pp.H * pp.W;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / cpr;
    const int k0 = (int)(i - m * cpr) * 8;
    const int b = (int)(m / pp.ntok), t = (int)(m - (long long)b * pp.ntok);
    uint4 o = make_uint4(0, 0, 0, 0);
    if constexpr (VEC) {
      // p % 8 == 0: the chunk is one contiguous run inside a patch row; p == 4: two consecutive patch rows (row_split)
      if (k0 < pp.K) {
        long long off;
        if constexpr (IN == IN_U8) {                  // K ordered (q, p1, p2, c), image NHWC
          const int rl = p * pp.C, e = k0 % rl, t1 = k0 / rl, p1 = t1 % p, q = t1 / p;
          const int idx = __ldg(pp.perm + t * pp.g + q);
          const int r = idx / pp.gw, cc = idx - r * pp.gw;
          off = (((long long)b * pp.H + (r * p + p1)) * pp.W + cc * p) * pp.C + e;
        } else {
          const int p2 = k0 % p, t1 = k0 / p, p1 = t1 % p, t2 = t1 / p, c = t2 % pp.C, q = t2 / pp.C;
          const int idx = __ldg(pp.perm + t * pp.g + q);
          const int r = idx / pp.gw, cc = idx - r * pp.gw;
          off = ((long long)b * pp.C + c) * plane + (long long)(r * p + p1) * pp.W + cc * p + p2;
        }
        ChunkRaw raw;
        chunk_load<IN>(raw, pp.img, off, pp.row_split, pp.wide_ld != 0);
        o = chunk_pack<IN>(raw);
      }
    } else if constexpr (IN != IN_U8) {
      float f[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = k0 + e;
        f[e] = 0.f;
        if (k < pp.K) {
          const int p2 = k % p, t1 = k / p, p1 = t1 % p, t2 = t1 / p, c = t2 % pp.C, q = t2 / pp.C;
          const int idx = __ldg(pp.perm + t * pp.g + q);
          const int r = idx / pp.gw, cc = idx % pp.gw;
          const long long off = ((long long)b * pp.C + c) * plane + (long long)(r * p + p1) * pp.W + cc * p + p2;
          if constexpr (BF16IN) f[e] = __bfloat162float(__ldg(reinterpret_cast<const __nv_bfloat16*>(pp.img) + off));
          else f[e] = __ldg(reinterpret_cast<const float*>(pp.img) + off);
        }
      }
      o = pack8f(f);
    }
    *reinterpret_cast<uint4*>(A + m * pp.Kpad + k0) = o;
  }
}

// vectorised gather: every 8-element K chunk is one contiguous, aligned run of the image (p % 8 == 0) or — p == 4, NCHW —
// two aligned 4-element patch rows one image row apart (a (q, c) plane is 16 elements, so a chunk never straddles two)
bool pe_vec_ok(const void* img, int fmt, int C, int H, int W, int p) {
  if (fmt == SFC_IMG_U8_NHWC)
    return ((p * C) % 8 == 0) && ((p * p * C) % 64 == 0) && ((W * C) % 8 == 0) && ((reinterpret_cast<uintptr_t>(img) & 7) == 0) &&
           ((long long)H * W * C < (1ll << 31));
  const int unit = (p == 4) ? 4 : 8;
  return (p % unit == 0) && (W % unit == 0) && ((reinterpret_cast<uintptr_t>(img) & 15) == 0) && (((long long)H * W) % unit == 0) &&
         ((long long)C * H * W < (1ll << 31));
}

int fill_params(PatchParams& pp, const void* img, int img_bf16, int B, int C, int H, int W, int p, int g, const int32_t* perm,
                int n_perm, int D) {
  SFC_REQUIRE(img && perm, "patch_embed: null pointer");
  SFC_REQUIRE(img_bf16 == SFC_IMG_F32_NCHW || img_bf16 == SFC_IMG_BF16_NCHW || img_bf16 == SFC_IMG_U8_NHWC,
              "patch_embed: unknown image format %d", img_bf16);
  pp.in_fmt = img_bf16;
  pp.row_split = (img_bf16 != SFC_IMG_U8_NHWC && p == 4) ? W : 0;
  // fp32 chunks as single 32-byte loads: every chunk offset is a multiple of 8 floats when the vectorised path applies
  pp.wide_ld = (img_bf16 == SFC_IMG_F32_NCHW && p % 8 == 0 && (reinterpret_cast<uintptr_t>(img) & 31) == 0) ? 1 : 0;
  pp.wide_st = 0;
  pp.dual_epi = 1;
  SFC_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && p > 0 && g > 0 && D > 0, "patch_embed: bad shape");
  SFC_REQUIRE(H % p == 0 && W % p == 0, "patch_embed: image %dx%d not divisible by pre-patch size %d", H, W, p);
  const int gh = H / p, gw = W / p;
  SFC_REQUIRE(n_perm > 0 && n_perm <= gh * gw && n_perm % g == 0, "patch_embed: permutation length %d must be in (0, %d] and divisible by group size %d", n_perm, gh * gw, g);
  pp.img = img; pp.perm = perm;
  pp.B = B; pp.C = C; pp.H = H; pp.W = W; pp.p = p; pp.g = g; pp.gw = gw;
  pp.ntok = n_perm / g;
  pp.K = g * C * p * p;
  pp.Kpad = sfc_ceil_div(pp.K, BK) * BK;
  pp.M = (long long)B * pp.ntok;
  pp.num_m_tiles = (int)sfc_ceil_div64(pp.M, BM);
  pp.num_k_blocks = pp.Kpad / BK;
  pp.rows_per_img = pp.ntok; pp.tok_off = 0;
  if (img_bf16 == SFC_IMG_U8_NHWC)
    SFC_REQUIRE(pe_vec_ok(img, img_bf16, C, H, W, p),
                "patch_embed: uint8 NHWC input needs (p * C) %% 8 == 0, (p * p * C) %% 64 == 0, (W * C) %% 8 == 0 and an 8-byte aligned buffer (p=%d C=%d W=%d)", p, C, W);
  return 0;
}

template <int BN, int kStages, bool VEC, int IN, bool FAST_EPI>
int launch_pe(const CUtensorMap& tw, const PatchParams& pp, cudaStream_t stream) {
  using L = PeSmem<BN, kStages>;
  auto kern = patch_embed_fwd_kernel<BN, kStages, VEC, IN, FAST_EPI>;
  static bool configured = false;
  if (!configured) {
    SFC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    configured = true;
  }
  const int total_tiles = pp.num_m_tiles * pp.num_n_tiles;
  const int grid = total_tiles < sfc_num_sms() ? total_tiles : sfc_num_sms();
  kern<<<grid, kThreads, L::kTotal, stream>>>(tw, pp);
  SFC_LAUNCH_OK();
  return 0;
}

}  // namespace

extern "C" int sfc_patch_embed_kpad(int C, int p, int g) { return sfc_ceil_div(g * C * p * p, BK) * BK; }

extern "C" int sfc_patch_embed_fwd(const void* img, int img_bf16, int B, int C, int H, int W, int p, int g, const int32_t* perm,
                                   int n_perm, const void* Wk, const void* bias, const void* pos, long long ld_pos, void* out,
                                   long long ld_out, int D, int rows_per_img, int tok_off, cudaStream_t stream) {
  PatchParams pp;
  if (int e = fill_params(pp, img, img_bf16, B, C, H, W, p, g, perm, n_perm, D)) return e;
  SFC_REQUIRE(Wk && out, "sfc_patch_embed_fwd: null pointer");
  SFC_REQUIRE(rows_per_img >= pp.ntok + tok_off && tok_off >= 0, "sfc_patch_embed_fwd: rows_per_img/tok_off inconsistent");
  pp.rows_per_img = rows_per_img; pp.tok_off = tok_off;
  const int BN = (D > 128) ? 256 : 128;
  pp.num_n_tiles = sfc_ceil_div(D, BN);
  pp.wide_st = ((reinterpret_cast<uintptr_t>(out) & 31) == 0 && (ld_out * 2) % 32 == 0 && D % 16 == 0) ? 1 : 0;
  EpiParams& e = pp.epi;
  e.N = D; e.bias = (const __nv_bfloat16*)bias; e.residual = (const __nv_bfloat16*)pos; e.aux = nullptr;
  e.out = out; e.out_pre = nullptr; e.ld_out = ld_out; e.ld_res = ld_pos; e.ld_aux = 0; e.split_stride = 0;
  e.alpha = 1.0f; e.act = SFC_ACT_NONE; e.aux_mode = SFC_AUX_NONE; e.out_fp32 = 0; e.drop_p = 0.f; e.drop_seed = 0; e.drop_epoch = nullptr;
  CUtensorMap tw;
  if (int err = sfc_make_tmap_2d(&tw, Wk, 2, (uint64_t)pp.Kpad, (uint64_t)D, (uint64_t)pp.Kpad * 2, BK, (uint32_t)BN, true)) return err;
  // the fused kernels take one pre-patch origin per 64-element k-block: p == 4 (48 elements per pre-patch at C = 3) only for g == 1
  const bool vec = pe_vec_ok(img, img_bf16, C, H, W, p) && pp.num_k_blocks <= kMaxTblKb && (pp.row_split == 0 || g == 1);
  const bool u8 = img_bf16 == SFC_IMG_U8_NHWC;
  SFC_REQUIRE(!u8 || vec, "sfc_patch_embed_fwd: uint8 NHWC input with K = %d exceeds the chunk table", pp.K);
  const bool fast = epi_fast_ok(pp.epi);
  if (vec && pp.row_split == 0 && fast && pp.num_k_blocks <= kTmMaxKb && D % (2 * kTmBN) == 0 && D <= kTmMaxD) {
    // TMEM-resident A: gather once per token, 64-column passes over the weights
    pp.num_n_tiles = D / kTmBN;
#define PE_TMEM(CL_)                                                                            \
  do {                                                                                          \
    if (u8) return launch_pe_tmem<IN_U8, CL_>(Wk, D, pp, stream);                               \
    return img_bf16 ? launch_pe_tmem<IN_BF16, CL_>(Wk, D, pp, stream) : launch_pe_tmem<IN_F32, CL_>(Wk, D, pp, stream); \
  } while (0)
    if (pp.num_m_tiles >= 4) PE_TMEM(4);
    if (pp.num_m_tiles >= 2) PE_TMEM(2);
    PE_TMEM(1);
#undef PE_TMEM
  }
#define PE_DISPATCH2(BN_, ST_, F_)                                                              \
  do {                                                                                          \
    if (u8) return launch_pe<BN_, ST_, true, IN_U8, F_>(tw, pp, stream);                        \
    if (vec && img_bf16) return launch_pe<BN_, ST_, true, IN_BF16, F_>(tw, pp, stream);         \
    if (vec && !img_bf16) return launch_pe<BN_, ST_, true, IN_F32, F_>(tw, pp, stream);         \
    if (!vec && img_bf16) return launch_pe<BN_, ST_, false, IN_BF16, F_>(tw, pp, stream);       \
    return launch_pe<BN_, ST_, false, IN_F32, F_>(tw, pp, stream);                              \
  } while (0)
#define PE_DISPATCH(BN_, ST_)                                                                   \
  do {                                                                                          \
    if (fast) PE_DISPATCH2(BN_, ST_, true); else PE_DISPATCH2(BN_, ST_, false);                 \
  } while (0)
  if (BN == 256) PE_DISPATCH(256, 4); else PE_DISPATCH(128, 6);
#undef PE_DISPATCH2
#undef PE_DISPATCH
}

// A[M, Kpad] = curve-ordered im2col (bf16), K order (q, c, p1, p2), zero padded to Kpad. Backward only.
extern "C" int sfc_patch_gather(const void* img, int img_bf16, int B, int C, int H, int W, int p, int g, const int32_t* perm,
                                int n_perm, void* A, cudaStream_t stream) {
  PatchParams pp;
  if (int e = fill_params(pp, img, img_bf16, B, C, H, W, p, g, perm, n_perm, 8)) return e;
  SFC_REQUIRE(A, "sfc_patch_gather: null output");
  const long long total = pp.M * (long long)(pp.Kpad / 8);
  long long blocks = sfc_ceil_div64(total, 256);
  const long long cap = 32ll * sfc_num_sms();
  if (blocks > cap) blocks = cap;
  const bool vec = pe_vec_ok(img, img_bf16, C, H, W, p);
  const unsigned nb = (unsigned)blocks;
  if (img_bf16 == SFC_IMG_U8_NHWC) patch_gather_kernel<IN_U8, true><<<nb, 256, 0, stream>>>(pp, (__nv_bfloat16*)A);
  else if (img_bf16 && vec) patch_gather_kernel<IN_BF16, true><<<nb, 256, 0, stream>>>(pp, (__nv_bfloat16*)A);
  else if (img_bf16) patch_gather_kernel<IN_BF16, false><<<nb, 256, 0, stream>>>(pp, (__nv_bfloat16*)A);
  else if (vec) patch_gather_kernel<IN_F32, true><<<nb, 256, 0, stream>>>(pp, (__nv_bfloat16*)A);
  else patch_gather_kernel<IN_F32, false><<<nb, 256, 0, stream>>>(pp, (__nv_bfloat16*)A);
  SFC_LAUNCH_OK();
  return 0;
}
