// Shared GEMM epilogue (used by gemm.cu and patch_embed.cu).
// order: *alpha -> +bias[n] -> (store out_pre) -> act -> dropout -> aux (relu mask / gelu') -> +residual -> store
//
// tcgen05.ld hands every lane one accumulator ROW (32 columns of it per chunk); writing global memory in that
// mapping touches 32 different 128-byte lines per instruction and made the epilogue, not the tensor pipe, the
// limiter of the K = 768 GEMMs. Each chunk is therefore transposed through a 4 KB per-warp shared-memory stage and
// finished in a mapping where 4 adjacent lanes cover 64 contiguous bytes of one output row, so residual / aux loads
// and all stores are sector-coalesced. The operands of chunk c+1 are fetched while chunk c is finished.
#pragma once
#include "common.cuh"
#include "sfcvit.h"

struct EpiParams {
  int N;                          // number of valid output columns
  const __nv_bfloat16* bias;      // [N] or null
  const __nv_bfloat16* residual;  // [*, ld_res] or null (added after activation)
  const __nv_bfloat16* aux;       // [*, ld_aux] or null
  void* out;                      // bf16 or fp32 [*, ld_out]
  __nv_bfloat16* out_pre;         // optional pre-activation copy (bf16, ld_out)
  long long ld_out, ld_res, ld_aux;
  long long split_stride;         // elements between split-K partial outputs (fp32)
  float alpha;
  int act;                        // SFC_ACT_*
  int aux_mode;                   // SFC_AUX_*
  int out_fp32;
  float drop_p;                   // dropout prob applied after activation (0 = off)
  unsigned long long drop_seed;
  const unsigned long long* drop_epoch;   // optional device counter mixed into the seed (null = none)
};

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_erf_grad(float x) {
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752f));
  const float pdf = 0.3989422804014327f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

// Counter-based dropout (same decisions in forward and backward, no mask tensor). The 64-bit seed is mixed once per
// thread (splitmix64) into two 32-bit keys; one 32-bit multiply-xorshift hash of (keys, index >> 1) then yields two
// 16-bit uniform lanes, and element `index` is kept iff its lane >= thr16 = floor(p * 65536). The keep probability is
// exactly 1 - thr16 / 65536, and that value (not the nominal p) is used for the rescale.
struct DropKey {
  uint32_t s0, s1, thr16;
  float inv_keep;
};
__host__ __device__ __forceinline__ uint32_t drop_thr16(float p) { return (uint32_t)(p * 65536.0f); }
__host__ __device__ __forceinline__ float drop_inv_keep(float p) {
  return p > 0.f ? 65536.0f / (65536.0f - (float)drop_thr16(p)) : 1.0f;
}
// The seed mixing of drop_key without the device-side epoch load (host-callable: tests/host/dropout_host.cu).
__host__ __device__ __forceinline__ DropKey drop_key_mixed(unsigned long long seed, float p) {
  unsigned long long z = seed + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  DropKey k;
  k.s0 = (uint32_t)z;
  k.s1 = (uint32_t)(z >> 32);
  k.thr16 = drop_thr16(p);
  k.inv_keep = drop_inv_keep(p);
  return k;
}
__host__ __device__ __forceinline__ unsigned long long drop_epoch_seed(unsigned long long seed, unsigned long long epoch) {
  return seed + epoch * 0xD1B54A32D192ED03ull;
}
__device__ __forceinline__ DropKey drop_key(unsigned long long seed, float p, const unsigned long long* epoch = nullptr) {
  if (epoch != nullptr) seed = drop_epoch_seed(seed, __ldg(epoch));   // CUDA-graph replays: fresh masks per replay
  return drop_key_mixed(seed, p);
}
__host__ __device__ __forceinline__ uint32_t drop_hash2(const DropKey& k, unsigned long long pair) {
  uint32_t x = ((uint32_t)pair ^ k.s0) * 0x9E3779B1u;
  x ^= x >> 15;
  x = (x + (uint32_t)(pair >> 32) * 0x632BE5ABu + k.s1) * 0x85EBCA77u;
  x ^= x >> 13;
  x *= 0xC2B2AE3Du;
  x ^= x >> 16;
  return x;
}
// Within an aligned group of G consecutive elements the lanes come from ONE hash (the group seed) expanded by G
// independent steps of a 32-bit LCG, x_i = seed * A^(i+1) + C_(i+1) (one multiply-add each, no dependency chain);
// element i of the group is kept iff x_i >= thr16 << 16, i.e. its top 16 bits are the uniform lane. Forward and
// backward of a dropout site must use the same G (8 for GEMM-output dropout, 16 for attention probabilities).
constexpr uint32_t kLcgA = 747796405u, kLcgC = 2891336453u;
__host__ __device__ constexpr uint32_t lcg_mul(int n) { uint32_t a = 1u; for (int i = 0; i < n; ++i) a *= kLcgA; return a; }
__host__ __device__ constexpr uint32_t lcg_add(int n) { uint32_t c = 0u; for (int i = 0; i < n; ++i) c = c * kLcgA + kLcgC; return c; }

template <int G>
__host__ __device__ __forceinline__ bool drop_keep(const DropKey& k, unsigned long long idx) {
  const uint32_t seed = drop_hash2(k, idx / G);
  uint32_t x = seed;
  const int pos = (int)(idx % G);
  for (int i = 0; i <= pos; ++i) x = x * kLcgA + kLcgC;
  return x >= (k.thr16 << 16);
}
// v[i] = keep(base + i) ? v[i] * inv_keep : 0 for NV consecutive elements
template <int NV, int G>
__device__ __forceinline__ void drop_apply(float* v, const DropKey& k, unsigned long long base) {
  static_assert(NV % G == 0, "NV must be a multiple of the group size");
  const uint32_t thr_hi = k.thr16 << 16;
  if (base % G == 0) {
#pragma unroll
    for (int g = 0; g < NV / G; ++g) {
      const uint32_t seed = drop_hash2(k, base / G + g);
#pragma unroll
      for (int i = 0; i < G; ++i) {
        const uint32_t x = seed * lcg_mul(i + 1) + lcg_add(i + 1);
        v[g * G + i] = (x >= thr_hi) ? v[g * G + i] * k.inv_keep : 0.f;
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = drop_keep<G>(k, base + i) ? v[i] * k.inv_keep : 0.f;
  }
}

// mask only: v[i] = keep(base + i) ? v[i] : 0 (the caller applies 1 / keep_prob once, downstream of a linear op)
template <int NV, int G>
__device__ __forceinline__ void drop_zero(float* v, const DropKey& k, unsigned long long base) {
  static_assert(NV % G == 0, "NV must be a multiple of the group size");
  const uint32_t thr_hi = k.thr16 << 16;
  if (base % G == 0) {
#pragma unroll
    for (int g = 0; g < NV / G; ++g) {
      const uint32_t seed = drop_hash2(k, base / G + g);
#pragma unroll
      for (int i = 0; i < G; ++i) {
        const uint32_t x = seed * lcg_mul(i + 1) + lcg_add(i + 1);
        v[g * G + i] = (x >= thr_hi) ? v[g * G + i] : 0.f;
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = drop_keep<G>(k, base + i) ? v[i] : 0.f;
  }
}

__device__ __forceinline__ void epi_unpack8(const uint4& b, float* f) {
  f[0] = ptx::bf16_lo(b.x); f[1] = ptx::bf16_hi(b.x); f[2] = ptx::bf16_lo(b.y); f[3] = ptx::bf16_hi(b.y);
  f[4] = ptx::bf16_lo(b.z); f[5] = ptx::bf16_hi(b.z); f[6] = ptx::bf16_lo(b.w); f[7] = ptx::bf16_hi(b.w);
}
__device__ __forceinline__ uint4 epi_pack8(const float* v) {
  uint4 o;
  o.x = ptx::pack_bf16(v[0], v[1]); o.y = ptx::pack_bf16(v[2], v[3]);
  o.z = ptx::pack_bf16(v[4], v[5]); o.w = ptx::pack_bf16(v[6], v[7]);
  return o;
}
__device__ __forceinline__ bool epi_al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Row mapping of a tile row (global accumulator row m) to the row of out / out_pre / aux (m_out) and of the
// residual (m_res). GEMM: identity. Patch embed: image-major output rows with a token offset, residual = pos[token].
struct EpiRowIdentity {
  __device__ __forceinline__ void map(long long m, long long& m_out, long long& m_res) const { m_out = m; m_res = m; }
};

// Per-tile, per-lane state of the transposed mapping: lane l owns, for it = 0..3, the 8 consecutive columns
// (l & 3) * 8 .. +7 of tile row it * 8 + (l >> 2) of every 32-column chunk.
struct EpiLane {
  long long m_out[4], m_res[4];
  bool ok[4];
  bool bias_vec, res_vec, aux_vec, out_vec, pre_vec;
  DropKey dkey;
};

struct EpiOps {                    // prefetched global operands of one 32-column chunk (vector path only)
  uint4 bias, res[4], aux[4];
};

__device__ __forceinline__ void epi_prefetch(const EpiParams& p, const EpiLane& L, EpiOps& o, int n, bool full) {
  if (!full) return;
  if (L.bias_vec) o.bias = __ldg(reinterpret_cast<const uint4*>(p.bias + n));
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    if (L.res_vec && L.ok[it]) o.res[it] = __ldg(reinterpret_cast<const uint4*>(p.residual + L.m_res[it] * p.ld_res + n));
    if (L.aux_vec && L.ok[it]) o.aux[it] = __ldg(reinterpret_cast<const uint4*>(p.aux + L.m_out[it] * p.ld_aux + n));
  }
}

// Finishes 8 consecutive columns n .. n+7 (nvalid of them inside N) of output row m_out and stores them.
__device__ __forceinline__ void epi_apply_store8(const EpiParams& p, const EpiLane& L, const EpiOps& o, int it, float (&v)[8], int n,
                                                 int nvalid, bool full, int split) {
  const long long m_out = L.m_out[it], m_res = L.m_res[it];
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] *= p.alpha;
  if (p.bias) {
    if (L.bias_vec && full) {
      float f[8];
      epi_unpack8(o.bias, f);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += f[j];
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < nvalid) v[j] += __bfloat162float(p.bias[n + j]);
    }
  }
  if (p.out_pre) {
    __nv_bfloat16* op = p.out_pre + m_out * p.ld_out + n;
    if (L.pre_vec && full) {
      *reinterpret_cast<uint4*>(op) = epi_pack8(v);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < nvalid) op[j] = __float2bfloat16(v[j]);
    }
  }
  if (p.act == SFC_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.0f);
  } else if (p.act == SFC_ACT_GELU) {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = gelu_erf(v[j]);
  }
  if (p.drop_p > 0.0f)
    drop_apply<8, 8>(v, L.dkey, (unsigned long long)m_out * (unsigned long long)p.N + (unsigned long long)n);
  if (p.aux_mode != SFC_AUX_NONE) {
    float a[8];
    if (L.aux_vec && full) {
      epi_unpack8(o.aux[it], a);
    } else {
      const __nv_bfloat16* ap = p.aux + m_out * p.ld_aux + n;
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] = (j < nvalid) ? __bfloat162float(ap[j]) : 0.0f;
    }
    if (p.aux_mode == SFC_AUX_RELU_MASK) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = a[j] > 0.0f ? v[j] : 0.0f;
    } else {  // SFC_AUX_GELU_GRAD: aux holds the pre-activation
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] *= gelu_erf_grad(a[j]);
    }
  }
  if (p.residual) {
    if (L.res_vec && full) {
      float f[8];
      epi_unpack8(o.res[it], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += f[j];
    } else {
      const __nv_bfloat16* rp = p.residual + m_res * p.ld_res + n;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < nvalid) v[j] += __bfloat162float(rp[j]);
    }
  }
  if (p.out_fp32) {
    float* op = reinterpret_cast<float*>(p.out) + (long long)split * p.split_stride + m_out * p.ld_out + n;
    if (L.out_vec && full) {
      reinterpret_cast<float4*>(op)[0] = make_float4(v[0], v[1], v[2], v[3]);
      reinterpret_cast<float4*>(op)[1] = make_float4(v[4], v[5], v[6], v[7]);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < nvalid) op[j] = v[j];
    }
  } else {
    __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + m_out * p.ld_out + n;
    if (L.out_vec && full) {
      *reinterpret_cast<uint4*>(op) = epi_pack8(v);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < nvalid) op[j] = __float2bfloat16(v[j]);
    }
  }
}

constexpr int kEpiStageBytes = 4096;   // per epilogue warp: 32 rows x 32 fp32, 16-byte chunks XOR-swizzled by (row & 7)

// Epilogue of one warp's share of an accumulator tile: TMEM lanes [quarter*32, +32) (the warp's lane quarter; `taddr`
// already carries the lane offset and the first column), columns [n_begin, n_begin + ncols) of the output, global
// accumulator rows m_base .. m_base+31. Each 32-column chunk is read from TMEM with one row per lane, transposed
// through the warp's private smem stage, and finished in a mapping where 4 adjacent lanes cover 64 contiguous bytes of
// one output row (8 rows per instruction): global loads of residual / aux and the stores are sector-coalesced.
// The global operands of chunk c+1 are in flight while chunk c is finished.
template <class RowMap>
__device__ __forceinline__ void epi_tile(const EpiParams& p, uint32_t taddr, int n_begin, int ncols, long long m_base, long long M,
                                         const RowMap& rm, int split, uint8_t* stage) {
  const int lane = (int)(threadIdx.x & 31);
  const int cg = lane & 3, rsub = lane >> 2;
  EpiLane L;
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const long long m = m_base + it * 8 + rsub;
    L.ok[it] = m < M;
    rm.map(L.ok[it] ? m : 0, L.m_out[it], L.m_res[it]);
  }
  L.bias_vec = p.bias && epi_al16(p.bias);
  L.res_vec = p.residual && (p.ld_res % 8 == 0) && epi_al16(p.residual);
  L.aux_vec = p.aux_mode != SFC_AUX_NONE && (p.ld_aux % 8 == 0) && epi_al16(p.aux);
  L.out_vec = p.out_fp32 ? ((p.ld_out % 4 == 0) && epi_al16(p.out) && (p.split_stride % 4 == 0))
                         : ((p.ld_out % 8 == 0) && epi_al16(p.out));
  L.pre_vec = p.out_pre && (p.ld_out % 8 == 0) && epi_al16(p.out_pre);
  L.dkey = drop_key(p.drop_seed, p.drop_p, p.drop_epoch);
  if (n_begin >= p.N) return;
  EpiOps cur, nxt;
  epi_prefetch(p, L, cur, n_begin + cg * 8, n_begin + 32 <= p.N);
  const int nchunks = ncols / 32;
#pragma unroll 1
  for (int c = 0; c < nchunks; ++c) {
    const int n0 = n_begin + c * 32;
    if (n0 >= p.N) break;                      // warp-uniform
    uint32_t raw[32];
    ptx::tmem_ld_x32(taddr + c * 32, raw);
    const bool more = (c + 1 < nchunks) && (n0 + 32 < p.N);
    if (more) epi_prefetch(p, L, nxt, n0 + 32 + cg * 8, n0 + 64 <= p.N);
    ptx::tmem_ld_wait();
    {
      uint8_t* srow = stage + lane * 128;
      const int sw = lane & 7;
#pragma unroll
      for (int q = 0; q < 8; ++q)
        *reinterpret_cast<uint4*>(srow + ((q ^ sw) << 4)) = make_uint4(raw[q * 4 + 0], raw[q * 4 + 1], raw[q * 4 + 2], raw[q * 4 + 3]);
    }
    __syncwarp();
    const bool full = n0 + 32 <= p.N;
    const int n = n0 + cg * 8;
    const int nvalid = p.N - n;                // may be <= 0 or > 8
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + rsub;
      const uint8_t* srow = stage + r * 128;
      const uint4 lo = *reinterpret_cast<const uint4*>(srow + (((2 * cg) ^ (r & 7)) << 4));
      const uint4 hi = *reinterpret_cast<const uint4*>(srow + (((2 * cg + 1) ^ (r & 7)) << 4));
      if (L.ok[it] && nvalid > 0) {
        float v[8] = {__uint_as_float(lo.x), __uint_as_float(lo.y), __uint_as_float(lo.z), __uint_as_float(lo.w),
                      __uint_as_float(hi.x), __uint_as_float(hi.y), __uint_as_float(hi.z), __uint_as_float(hi.w)};
        epi_apply_store8(p, L, cur, it, v, n, nvalid, full, split);
      }
    }
    __syncwarp();                              // stage is rewritten by the next chunk
    if (more) cur = nxt;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Lean variant for the encoder's hot GEMMs. Preconditions (checked on the host by epi_fast_ok): every 32-column chunk
// is full (N % 32 == 0), all operands 16-byte aligned with vectorisable leading dimensions, no pre-activation copy,
// activation in {none, ReLU}, aux in {none, ReLU mask}. Per-lane row pointers and all feature predicates are hoisted
// out of the chunk loop; bias is folded into one FFMA per element.
// ------------------------------------------------------------------------------------------------------------------
inline bool epi_fast_ok(const EpiParams& p) {
  auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  if (p.N % 32 != 0 || p.out_pre) return false;
  if (p.act != SFC_ACT_NONE && p.act != SFC_ACT_RELU) return false;
  if (p.aux_mode != SFC_AUX_NONE && p.aux_mode != SFC_AUX_RELU_MASK) return false;
  if (p.bias && !al(p.bias)) return false;
  if (p.residual && (!al(p.residual) || p.ld_res % 8 != 0)) return false;
  if (p.aux_mode != SFC_AUX_NONE && (!al(p.aux) || p.ld_aux % 8 != 0)) return false;
  if (!al(p.out)) return false;
  if (p.out_fp32) return p.ld_out % 4 == 0 && p.split_stride % 4 == 0;
  return p.ld_out % 8 == 0;
}

template <class RowMap>
__device__ __forceinline__ void epi_tile_fast(const EpiParams& p, uint32_t taddr, int n_begin, int ncols, long long m_base, long long M,
                                              const RowMap& rm, int split, uint8_t* stage) {
  const int lane = (int)(threadIdx.x & 31);
  const int cg = lane & 3, rsub = lane >> 2;
  const bool has_bias = p.bias != nullptr, has_res = p.residual != nullptr, has_aux = p.aux_mode != SFC_AUX_NONE;
  const bool has_drop = p.drop_p > 0.0f, f32 = p.out_fp32 != 0;
  // fp32 output (split-K partials): two 16-byte stores per lane would each half-fill 32 sectors per instruction
  const bool wide_f32 = f32 && (reinterpret_cast<uintptr_t>(p.out) & 31) == 0 && p.ld_out % 8 == 0 && p.split_stride % 8 == 0 &&
                        n_begin % 8 == 0;
  const float relu_lo = p.act == SFC_ACT_RELU ? 0.0f : -INFINITY;
  const float alpha = p.alpha;
  const DropKey dkey = drop_key(p.drop_seed, p.drop_p, p.drop_epoch);
  // per-lane row state: byte pointers at column n_begin + cg * 8 of rows it * 8 + rsub
  const char* resp[4];
  const char* auxp[4];
  char* outp[4];
  unsigned long long didx[4];
  bool ok[4];
  const int ncol0 = n_begin + cg * 8;
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const long long m = m_base + it * 8 + rsub;
    ok[it] = m < M;
    long long m_out, m_res;
    rm.map(ok[it] ? m : 0, m_out, m_res);
    resp[it] = reinterpret_cast<const char*>(p.residual) + (m_res * p.ld_res + ncol0) * 2;
    auxp[it] = reinterpret_cast<const char*>(p.aux) + (m_out * p.ld_aux + ncol0) * 2;
    outp[it] = reinterpret_cast<char*>(p.out) + (f32 ? ((long long)split * p.split_stride + m_out * p.ld_out + ncol0) * 4
                                                      : (m_out * p.ld_out + ncol0) * 2);
    didx[it] = (unsigned long long)m_out * (unsigned long long)p.N + (unsigned long long)ncol0;
  }
  const char* biasp = reinterpret_cast<const char*>(p.bias) + ncol0 * 2;
  uint4 cb = make_uint4(0, 0, 0, 0), cr[4], ca[4], nb = cb, nr[4], na[4];
  auto prefetch = [&](int coff, uint4& b, uint4 (&r)[4], uint4 (&a)[4]) {     // coff: column offset from n_begin
    if (has_bias) b = __ldg(reinterpret_cast<const uint4*>(biasp + coff * 2));
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      if (has_res && ok[it]) r[it] = __ldg(reinterpret_cast<const uint4*>(resp[it] + coff * 2));
      if (has_aux && ok[it]) a[it] = __ldg(reinterpret_cast<const uint4*>(auxp[it] + coff * 2));
    }
  };
  prefetch(0, cb, cr, ca);
  const int nchunks = ncols / 32;
  uint8_t* swrite = stage + lane * 128;
  const int sw = lane & 7;
#pragma unroll 1
  for (int c = 0; c < nchunks; ++c) {
    const int coff = c * 32;
    if (n_begin + coff >= p.N) break;          // warp-uniform
    uint32_t raw[32];
    ptx::tmem_ld_x32(taddr + coff, raw);
    const bool more = (c + 1 < nchunks) && (n_begin + coff + 32 < p.N);
    if (more) prefetch(coff + 32, nb, nr, na);
    ptx::tmem_ld_wait();
#pragma unroll
    for (int q = 0; q < 8; ++q)
      *reinterpret_cast<uint4*>(swrite + ((q ^ sw) << 4)) = make_uint4(raw[q * 4 + 0], raw[q * 4 + 1], raw[q * 4 + 2], raw[q * 4 + 3]);
    __syncwarp();
    float bf[8];
    epi_unpack8(cb, bf);
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + rsub;
      const uint8_t* srow = stage + r * 128;
      const uint4 lo = *reinterpret_cast<const uint4*>(srow + (((2 * cg) ^ (r & 7)) << 4));
      const uint4 hi = *reinterpret_cast<const uint4*>(srow + (((2 * cg + 1) ^ (r & 7)) << 4));
      if (ok[it]) {
        float v[8] = {__uint_as_float(lo.x), __uint_as_float(lo.y), __uint_as_float(lo.z), __uint_as_float(lo.w),
                      __uint_as_float(hi.x), __uint_as_float(hi.y), __uint_as_float(hi.z), __uint_as_float(hi.w)};
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaxf(fmaf(v[j], alpha, bf[j]), relu_lo);
        if (has_drop) drop_apply<8, 8>(v, dkey, didx[it] + (unsigned long long)coff);
        if (has_aux) {
          float a[8];
          epi_unpack8(ca[it], a);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = a[j] > 0.0f ? v[j] : 0.0f;
        }
        if (has_res) {
          float f[8];
          epi_unpack8(cr[it], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] += f[j];
        }
        if (f32) {
          float4* op = reinterpret_cast<float4*>(outp[it] + coff * 4);
          if (wide_f32) {                          // the lane's 8 fp32 = one 32-byte sector: a single 256-bit store
            ptx::stg256(op, make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3])),
                        make_uint4(__float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7])));
          } else {
            op[0] = make_float4(v[0], v[1], v[2], v[3]);
            op[1] = make_float4(v[4], v[5], v[6], v[7]);
          }
        } else {
          *reinterpret_cast<uint4*>(outp[it] + coff * 2) = epi_pack8(v);
        }
      }
    }
    __syncwarp();                              // stage is rewritten by the next chunk
    if (more) {
      cb = nb;
#pragma unroll
      for (int it = 0; it < 4; ++it) { cr[it] = nr[it]; ca[it] = na[it]; }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Direct variant (same preconditions as epi_tile_fast): no shared-memory transpose. Every lane finishes the 32 columns
// of ITS accumulator row and stores them with four 16-byte stores (64 contiguous bytes per row); residual / aux are
// read the same way. Needs ~50 fewer registers than the transposed variant (used where the CTA is register-tight:
// patch_embed.cu with 512 threads). `bias_s` = this warp's private fp32 copy of bias[n_begin .. n_begin + ncols) in
// shared memory (ncols floats; zeros when there is no bias).
// ------------------------------------------------------------------------------------------------------------------
template <class RowMap>
__device__ __forceinline__ void epi_tile_direct(const EpiParams& p, uint32_t taddr, int n_begin, int ncols, long long m_base, long long M,
                                                const RowMap& rm, int split, float* bias_s, bool wide_st = false) {
  const int lane = (int)(threadIdx.x & 31);
  const bool has_res = p.residual != nullptr, has_aux = p.aux_mode != SFC_AUX_NONE;
  const bool has_drop = p.drop_p > 0.0f, f32 = p.out_fp32 != 0;
  const float relu_lo = p.act == SFC_ACT_RELU ? 0.0f : -INFINITY;
  const float alpha = p.alpha;
  const DropKey dkey = drop_key(p.drop_seed, p.drop_p, p.drop_epoch);
  __syncwarp();
  for (int c0 = 0; c0 < ncols; c0 += 128) {       // lane l converts columns 4l .. 4l+3 of each 128-column group
    const int c = c0 + lane * 4;
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.bias && c < ncols && n_begin + c < p.N) {
      const uint2 u = __ldg(reinterpret_cast<const uint2*>(p.bias + n_begin + c));
      b4 = make_float4(ptx::bf16_lo(u.x), ptx::bf16_hi(u.x), ptx::bf16_lo(u.y), ptx::bf16_hi(u.y));
    }
    if (c < ncols) *reinterpret_cast<float4*>(bias_s + c) = b4;
  }
  __syncwarp();
  const long long m = m_base + lane;
  const bool ok = m < M;
  long long m_out, m_res;
  rm.map(ok ? m : 0, m_out, m_res);
  const char* resp = reinterpret_cast<const char*>(p.residual) + (m_res * p.ld_res + n_begin) * 2;
  const char* auxp = reinterpret_cast<const char*>(p.aux) + (m_out * p.ld_aux + n_begin) * 2;
  char* outp = reinterpret_cast<char*>(p.out) + (f32 ? ((long long)split * p.split_stride + m_out * p.ld_out + n_begin) * 4
                                                     : (m_out * p.ld_out + n_begin) * 2);
  const unsigned long long didx = (unsigned long long)m_out * (unsigned long long)p.N + (unsigned long long)n_begin;
  const int nchunks = ncols / 32;
#pragma unroll 1
  for (int c = 0; c < nchunks; ++c) {
    const int coff = c * 32;
    if (n_begin + coff >= p.N) break;          // warp-uniform
    uint32_t raw[32];
    ptx::tmem_ld_x32(taddr + coff, raw);
    uint4 cr[4], ca[4];
    if (ok) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (has_res) cr[q] = __ldg(reinterpret_cast<const uint4*>(resp + coff * 2) + q);
        if (has_aux) ca[q] = __ldg(reinterpret_cast<const uint4*>(auxp + coff * 2) + q);
      }
    }
    ptx::tmem_ld_wait();
    if (ok) {
      float v[32];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 b4 = *reinterpret_cast<const float4*>(bias_s + coff + q * 4);     // broadcast read
        v[q * 4 + 0] = fmaxf(fmaf(__uint_as_float(raw[q * 4 + 0]), alpha, b4.x), relu_lo);
        v[q * 4 + 1] = fmaxf(fmaf(__uint_as_float(raw[q * 4 + 1]), alpha, b4.y), relu_lo);
        v[q * 4 + 2] = fmaxf(fmaf(__uint_as_float(raw[q * 4 + 2]), alpha, b4.z), relu_lo);
        v[q * 4 + 3] = fmaxf(fmaf(__uint_as_float(raw[q * 4 + 3]), alpha, b4.w), relu_lo);
      }
      if (has_drop) drop_apply<32, 8>(v, dkey, didx + (unsigned long long)coff);
      if (has_aux) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float a[8];
          epi_unpack8(ca[q], a);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[q * 8 + j] = a[j] > 0.0f ? v[q * 8 + j] : 0.0f;
        }
      }
      if (has_res) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float f[8];
          epi_unpack8(cr[q], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[q * 8 + j] += f[j];
        }
      }
      if (f32) {
        float4* op = reinterpret_cast<float4*>(outp + coff * 4);
#pragma unroll
        for (int q = 0; q < 8; ++q) op[q] = make_float4(v[q * 4 + 0], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
      } else {
        uint4* op = reinterpret_cast<uint4*>(outp + coff * 2);
        if (wide_st) {                               // 256-bit stores: a full 32-byte sector per lane and instruction
          ptx::stg256(op, epi_pack8(&v[0]), epi_pack8(&v[8]));
          ptx::stg256(op + 2, epi_pack8(&v[16]), epi_pack8(&v[24]));
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q) op[q] = epi_pack8(&v[q * 8]);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// TMA-store variant (bf16 output, same preconditions as epi_tile_fast): each lane finishes the 32 columns of ITS
// accumulator row (bias by broadcast loads, residual / aux read 64 bytes per row), packs them to bf16 and writes them
// into a 32-row x 64-byte staging box (SWIZZLE_64B, conflict-free for row-per-lane 16-byte stores); one lane then
// issues a cp.async.bulk.tensor store of the box. Per 32 x 32 chunk this is 4 shared-memory stores per lane instead
// of 8 + 8 and no st.global at all: half the shared-memory traffic of the transposed variant (the single-CTA
// 128 x 256 MMA tile already takes ~75 % of the shared-memory bandwidth) and the store coalescing is done by the TMA
// unit. Two boxes per warp alternate, so a box is rewritten only after the store issued two chunks earlier has read it.
// Rows >= M and columns >= N are clipped by the tensor map.
// `stage` = this warp's 4 KB (two 2 KB boxes, 1024-byte aligned). The caller drains with tma_store_wait_all<0>().
// ------------------------------------------------------------------------------------------------------------------
// OPND: 0 = no [M, N] operand, 1 = residual, 2 = aux (ReLU mask source). The operand is fetched by TMA into per-warp
// 32 x 32 boxes (same SWIZZLE_64B layout, two boxes alternate, one mbarrier each) one chunk ahead, and every lane reads
// its own row from shared memory: no uncoalesced global loads, no transposed mapping.
template <int OPND>
__device__ __forceinline__ void epi_tile_tma(const EpiParams& p, const CUtensorMap* tmap_out, const CUtensorMap* tmap_opnd, uint32_t taddr,
                                             int n_begin, int ncols, long long m_base, uint8_t* stage, uint32_t& box_counter,
                                             uint64_t* obar) {
  const int lane = (int)(threadIdx.x & 31);
  const bool has_bias = p.bias != nullptr;
  const bool has_drop = p.drop_p > 0.0f;
  const float relu_lo = p.act == SFC_ACT_RELU ? 0.0f : -INFINITY;
  const float alpha = p.alpha;
  const DropKey dkey = drop_key(p.drop_seed, p.drop_p, p.drop_epoch);
  const long long m = m_base + lane;
  const char* biasp = reinterpret_cast<const char*>(p.bias) + (long long)n_begin * 2;
  const unsigned long long didx = (unsigned long long)m * (unsigned long long)p.N + (unsigned long long)n_begin;
  const int nchunks = ncols / 32;
  const int sw = (lane >> 1) & 3;                  // SWIZZLE_64B: 16-byte chunk index ^= (row >> 1) & 3
  uint8_t* obox = stage + 4096;                    // operand boxes follow the two output boxes
  if (n_begin >= p.N) return;
  if (OPND != 0 && lane == 0) {                    // operand box of chunk 0
    const uint32_t b = box_counter & 1u;
    ptx::mbar_expect_tx(&obar[b], 2048);
    ptx::tma_load_2d(tmap_opnd, &obar[b], obox + b * 2048, n_begin, (int)m_base);
  }
  uint4 cb[4] = {};
#pragma unroll 1
  for (int c = 0; c < nchunks; ++c) {
    const int coff = c * 32;
    if (n_begin + coff >= p.N) break;              // warp-uniform
    uint32_t raw[32];
    ptx::tmem_ld_x32(taddr + coff, raw);
    if (has_bias) {                                // same address in all lanes (broadcast, L1-resident): hidden by the TMEM load
#pragma unroll
      for (int q = 0; q < 4; ++q) cb[q] = __ldg(reinterpret_cast<const uint4*>(biasp + coff * 2) + q);
    }
    const bool more = (c + 1 < nchunks) && (n_begin + coff + 32 < p.N);
    const uint32_t cur = box_counter & 1u;
    if (OPND != 0 && more && lane == 0) {          // next chunk's operand box; its last readers passed the __syncwarp below
      const uint32_t nb = cur ^ 1u;
      ptx::mbar_expect_tx(&obar[nb], 2048);
      ptx::tma_load_2d(tmap_opnd, &obar[nb], obox + nb * 2048, n_begin + coff + 32, (int)m_base);
    }
    ptx::tmem_ld_wait();
    float v[32];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float bf[8];
      epi_unpack8(cb[q], bf);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[q * 8 + j] = fmaxf(fmaf(__uint_as_float(raw[q * 8 + j]), alpha, bf[j]), relu_lo);
    }
    if (has_drop) drop_apply<32, 8>(v, dkey, didx + (unsigned long long)coff);
    if constexpr (OPND != 0) {
      ptx::mbar_wait(&obar[cur], (box_counter >> 1) & 1u);
      const uint8_t* orow = obox + cur * 2048 + lane * 64;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float f[8];
        epi_unpack8(*reinterpret_cast<const uint4*>(orow + ((q ^ sw) << 4)), f);
        if constexpr (OPND == 1) {
#pragma unroll
          for (int j = 0; j < 8; ++j) v[q * 8 + j] += f[j];
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) v[q * 8 + j] = f[j] > 0.0f ? v[q * 8 + j] : 0.0f;
        }
      }
    }
    uint8_t* box = stage + cur * 2048;
    ptx::tma_store_wait_read<1>();                 // the store that read this box two chunks ago has finished reading
    __syncwarp();
#pragma unroll
    for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(box + lane * 64 + ((q ^ sw) << 4)) = epi_pack8(&v[q * 8]);
    ptx::fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
      ptx::tma_store_2d(tmap_out, box, n_begin + coff, (int)m_base);
      ptx::tma_store_commit();
    }
    ++box_counter;
  }
}
