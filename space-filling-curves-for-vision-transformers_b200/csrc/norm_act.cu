// K5 — memory-bound row/column kernels (sm_100a): LayerNorm forward/backward with warp-shuffle
// reductions, and column sums for bias gradients. These replace the ATen LayerNorm / reduction kernels
// behind nn.LayerNorm and the bias gradients of nn.Linear in the reference encoder
// (/root/reference/src/models/vit.py:197-206 -> torch TransformerEncoderLayer norm1/norm2; :253-254, :303).
// Residual adds, bias, ReLU/GELU and their derivatives are fused into the GEMM epilogues (gemm.cu).
//
// Layout: activations are bf16 [rows, D] row-major; one warp owns one row; each lane moves 16-byte
// vectors (8 bf16) so a warp reads/writes 512 contiguous bytes per instruction. Statistics are fp32.
#include "common.cuh"
#include "gemm_epilogue.cuh"   // drop_keep
#include "sfcvit.h"

namespace {

constexpr int kMaxVec = 8;        // per-lane 16-byte vectors: D <= 8 * 256 = 2048
constexpr int kLnWarps = 4;       // rows per CTA

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  f[0] = ptx::bf16_lo(u.x); f[1] = ptx::bf16_hi(u.x); f[2] = ptx::bf16_lo(u.y); f[3] = ptx::bf16_hi(u.y);
  f[4] = ptx::bf16_lo(u.z); f[5] = ptx::bf16_hi(u.z); f[6] = ptx::bf16_lo(u.w); f[7] = ptx::bf16_hi(u.w);
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  uint4 u;
  u.x = ptx::pack_bf16(f[0], f[1]); u.y = ptx::pack_bf16(f[2], f[3]);
  u.z = ptx::pack_bf16(f[4], f[5]); u.w = ptx::pack_bf16(f[6], f[7]);
  return u;
}

// y = (x - mean) * rstd * gamma + beta ; saves mean/rstd (fp32) for the backward pass
template <int NV>
__global__ void __launch_bounds__(kLnWarps * 32)
layernorm_fwd_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ gamma,
                     const __nv_bfloat16* __restrict__ beta, __nv_bfloat16* __restrict__ y, float* __restrict__ mean_out,
                     float* __restrict__ rstd_out, long long rows, int D, float eps) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * kLnWarps + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int nvec = D >> 3;                   // 16-byte vectors per row
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * D);
  float v[NV][8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vi = lane + i * 32;
    if (vi < nvec) {
      unpack8(__ldg(xr + vi), v[i]);
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[i][j];
    }
  }
  const float mean = warp_sum(s) / (float)D;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vi = lane + i * 32;
    if (vi < nvec) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { const float d = v[i][j] - mean; q += d * d; }
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)D + eps);
  uint4* yr = reinterpret_cast<uint4*>(y + row * D);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vi = lane + i * 32;
    if (vi < nvec) {
      float g[8], b[8], o[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(gamma) + vi), g);
      unpack8(__ldg(reinterpret_cast<const uint4*>(beta) + vi), b);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (v[i][j] - mean) * rstd * g[j] + b[j];
      yr[vi] = pack8(o);
    }
  }
  if (lane == 0) {
    if (mean_out) mean_out[row] = mean;
    if (rstd_out) rstd_out[row] = rstd;
  }
}

// dx = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma,  xhat = (x - mean) * rstd.
// Fused extras (all optional): dx_drop = dropout_mask(dx) / keep — the gradient that flows into the Linear whose
// output was dropped before the residual add (mask re-derived from (seed, row * D + col) exactly as the forward GEMM
// epilogue drew it) — and the column sums of that tensor (= bias gradient of that Linear).
// Per-CTA partial sums go to part[blockIdx.x][3][D] (fp32): dgamma = sum dy * xhat, dbeta = sum dy, colsum.
// Row data stay PACKED (bf16x8 uint4) in registers and are unpacked in each of the two passes, which keeps the
// kernel at 3 CTAs / SM for D = 768 (a memory-bound kernel needs the loads of many rows in flight).
template <int NV, bool DROP, bool CSUM>
__global__ void __launch_bounds__(kLnWarps * 32, 3)
layernorm_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x,
                     const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                     const __nv_bfloat16* __restrict__ gamma, __nv_bfloat16* __restrict__ dx,
                     __nv_bfloat16* __restrict__ dx_drop, float drop_p, unsigned long long drop_seed,
                     const unsigned long long* __restrict__ drop_epoch,
                     float* __restrict__ part, long long rows, int D) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  extern __shared__ float sred[];            // [kLnWarps][3][D]
  const DropKey dkey = drop_key(drop_seed, drop_p, drop_epoch);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nvec = D >> 3;
  float dg[NV][8], db[NV][8], cs[CSUM ? NV : 1][8];
  uint4 gmp[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vi = lane + i * 32;
#pragma unroll
    for (int j = 0; j < 8; ++j) { dg[i][j] = 0.f; db[i][j] = 0.f; if (CSUM) cs[i][j] = 0.f; }
    gmp[i] = (vi < nvec) ? __ldg(reinterpret_cast<const uint4*>(gamma) + vi) : make_uint4(0, 0, 0, 0);
  }
  for (long long row = (long long)blockIdx.x * kLnWarps + wid; row < rows; row += (long long)gridDim.x * kLnWarps) {
    const uint4* xr = reinterpret_cast<const uint4*>(x + row * D);
    const uint4* dyr = reinterpret_cast<const uint4*>(dy + row * D);
    uint4 xp[NV], dp[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int vi = lane + i * 32;
      if (vi < nvec) { xp[i] = __ldg(xr + vi); dp[i] = __ldg(dyr + vi); }
    }
    const float mean = mean_in[row], rstd = rstd_in[row];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int vi = lane + i * 32;
      if (vi < nvec) {
        float xv[8], dv[8], gm[8];
        unpack8(xp[i], xv); unpack8(dp[i], dv); unpack8(gmp[i], gm);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = (xv[j] - mean) * rstd;
          const float g = dv[j] * gm[j];
          s1 += g;
          s2 += g * xh;
          dg[i][j] += dv[j] * xh;
          db[i][j] += dv[j];
        }
      }
    }
    s1 = warp_sum(s1) / (float)D;
    s2 = warp_sum(s2) / (float)D;
    uint4* dxr = reinterpret_cast<uint4*>(dx + row * D);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int vi = lane + i * 32;
      if (vi < nvec) {
        float xv[8], dv[8], gm[8], o[8];
        unpack8(xp[i], xv); unpack8(dp[i], dv); unpack8(gmp[i], gm);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = (xv[j] - mean) * rstd;
          o[j] = rstd * (dv[j] * gm[j] - s1 - xh * s2);
        }
        dxr[vi] = pack8(o);
        if (DROP) {
          drop_apply<8, 8>(o, dkey, (unsigned long long)row * (unsigned long long)D + (unsigned long long)(vi * 8));
          reinterpret_cast<uint4*>(dx_drop + row * D)[vi] = pack8(o);
        }
        if (CSUM) {
#pragma unroll
          for (int j = 0; j < 8; ++j) cs[i][j] += o[j];
        }
      }
    }
  }
  // cross-warp reduction of the column partials
  constexpr int NP = CSUM ? 3 : 2;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vi = lane + i * 32;
    if (vi < nvec) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        sred[(wid * 3 + 0) * D + vi * 8 + j] = dg[i][j];
        sred[(wid * 3 + 1) * D + vi * 8 + j] = db[i][j];
        if (CSUM) sred[(wid * 3 + 2) * D + vi * 8 + j] = cs[i][j];
      }
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < NP * D; c += blockDim.x) {
    const int which = c / D, col = c % D;
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kLnWarps; ++w) s += sred[(w * 3 + which) * D + col];
    part[((long long)blockIdx.x * 3 + which) * D + col] = s;
  }
}

// column sums: x bf16 [rows, N] (ld) -> part[blockIdx.y][N] fp32. block (32 x 8): 32 lanes x 8 columns, 8 row lanes.
__global__ void __launch_bounds__(256)
colsum_partial_kernel(const __nv_bfloat16* __restrict__ x, long long ld, long long rows, int N, float* __restrict__ part,
                      long long rows_per_block) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  __shared__ float sred[8][256 + 8];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col0 = (blockIdx.x * 32 + tx) * 8;
  const long long r0 = (long long)blockIdx.y * rows_per_block;
  const long long r1 = min(r0 + rows_per_block, rows);
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (col0 < N) {
    const bool vec = (col0 + 8 <= N) && (ld % 8 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
    for (long long r = r0 + ty; r < r1; r += 8) {
      const __nv_bfloat16* p = x + r * ld + col0;
      if (vec) {
        float f[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(p)), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += f[j];
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (col0 + j < N) acc[j] += __bfloat162float(p[j]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) sred[ty][tx * 8 + j] = acc[j];
  __syncthreads();
  const int c = threadIdx.x;          // 256 columns per block
  const int col = blockIdx.x * 256 + c;
  if (col < N) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += sred[w][c];
    part[(long long)blockIdx.y * N + col] = s;
  }
}

// out_v[c] = (accumulate ? out_v[c] : 0) + sum_b part[b * stride + v * vstride + c]   for v < nvec output vectors.
// grid (ceil(N / 32), nvec), block (32 columns x kFinLanes part-lanes): the partials of a column are summed by kFinLanes
// threads with four independent loads in flight each instead of one long dependent loop (444 partials of a LayerNorm
// backward: 4 rounds of loads per thread).
struct FinalizeOut { void* ptr[3]; };
template <int kFinLanes>
__global__ void __launch_bounds__(32 * kFinLanes) partial_finalize_kernel(const float* __restrict__ part, int nparts, long long stride,
                                                                          long long vstride, int N, FinalizeOut outs, int out_fp32,
                                                                          int accumulate) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  __shared__ float sred[kFinLanes][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + tx;
  const int v = blockIdx.y;
  float s = 0.f;
  if (c < N) {
    const float* base = part + v * vstride + c;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int b = ty;
    for (; b + 3 * kFinLanes < nparts; b += 4 * kFinLanes) {
      s0 += base[(long long)b * stride];
      s1 += base[(long long)(b + kFinLanes) * stride];
      s2 += base[(long long)(b + 2 * kFinLanes) * stride];
      s3 += base[(long long)(b + 3 * kFinLanes) * stride];
    }
    for (; b < nparts; b += kFinLanes) s0 += base[(long long)b * stride];
    s = (s0 + s1) + (s2 + s3);
  }
  sred[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && c < N) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kFinLanes; ++w) t += sred[w][tx];
    void* out = outs.ptr[v];
    if (out_fp32) {
      float* o = reinterpret_cast<float*>(out) + c;
      *o = accumulate ? *o + t : t;
    } else {
      __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out) + c;
      *o = __float2bfloat16(accumulate ? __bfloat162float(*o) + t : t);
    }
  }
}

// out = alpha * dy * f'(aux) * dropout_mask: relu mask (aux > 0), exact-GELU derivative (aux = pre-activation) or
// identity; the dropout keep decision is re-derived from (seed, element index) exactly as in the GEMM epilogue.
__global__ void __launch_bounds__(256) act_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ aux,
                                                      __nv_bfloat16* __restrict__ out, long long nvec, int mode, float alpha,
                                                      float drop_p, unsigned long long seed,
                                                      const unsigned long long* __restrict__ drop_epoch) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const DropKey dkey = drop_key(seed, drop_p, drop_epoch);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    float d[8], a[8], o[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(dy) + i), d);
    if (mode != SFC_AUX_NONE) unpack8(__ldg(reinterpret_cast<const uint4*>(aux) + i), a);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = d[j] * alpha;
      if (mode == SFC_AUX_RELU_MASK) v = a[j] > 0.f ? v : 0.f;
      else if (mode == SFC_AUX_GELU_GRAD) {
        const float cdf = 0.5f * (1.0f + erff(a[j] * 0.70710678118654752f));
        const float pdf = 0.3989422804014327f * __expf(-0.5f * a[j] * a[j]);
        v *= (cdf + a[j] * pdf);
      }
      o[j] = v;
    }
    if (drop_p > 0.f) drop_apply<8, 8>(o, dkey, (unsigned long long)i * 8ull);
    reinterpret_cast<uint4*>(out)[i] = pack8(o);
  }
}

int ln_bwd_blocks(long long rows) {
  long long b = sfc_ceil_div64(rows, kLnWarps);
  const long long cap = 3ll * sfc_num_sms();
  return (int)(b < cap ? b : cap);
}

}  // namespace

extern "C" int sfc_layernorm_fwd(const void* x, const void* gamma, const void* beta, void* y, float* mean, float* rstd,
                                 long long rows, int D, float eps, cudaStream_t stream) {
  SFC_REQUIRE(x && gamma && beta && y, "sfc_layernorm_fwd: null pointer");
  SFC_REQUIRE(D % 8 == 0 && D >= 8 && D <= kMaxVec * 256, "sfc_layernorm_fwd: D=%d must be a multiple of 8 and <= %d", D, kMaxVec * 256);
  if (rows == 0) return 0;
  const unsigned grid = (unsigned)sfc_ceil_div64(rows, kLnWarps);
  const int nv = sfc_ceil_div(D / 8, 32);
#define LN_FWD(NV) SFC_CUDA_OK(sfc_launch_pdl(layernorm_fwd_kernel<NV>, dim3(grid), dim3(kLnWarps * 32), 0, stream, (const __nv_bfloat16*)x, \
      (const __nv_bfloat16*)gamma, (const __nv_bfloat16*)beta, (__nv_bfloat16*)y, mean, rstd, rows, D, eps))
  if (nv <= 1) LN_FWD(1); else if (nv <= 2) LN_FWD(2); else if (nv <= 3) LN_FWD(3); else if (nv <= 4) LN_FWD(4); else LN_FWD(8);
#undef LN_FWD
  SFC_LAUNCH_OK();
  return 0;
}

extern "C" size_t sfc_layernorm_bwd_scratch_bytes(long long rows, int D) {
  return (size_t)ln_bwd_blocks(rows) * 3 * (size_t)D * sizeof(float);
}

// dx_drop / dcolsum may be NULL. dcolsum = column sums of dx_drop (or of dx when dx_drop is NULL).
extern "C" int sfc_layernorm_bwd(const void* dy, const void* x, const float* mean, const float* rstd, const void* gamma,
                                 void* dx, void* dx_drop, float drop_p, unsigned long long drop_seed, void* dgamma,
                                 void* dbeta, void* dcolsum, int param_fp32, int accumulate, void* scratch,
                                 size_t scratch_bytes, long long rows, int D, cudaStream_t stream) {
  SFC_REQUIRE(dy && x && mean && rstd && gamma && dx && dgamma && dbeta, "sfc_layernorm_bwd: null pointer");
  SFC_REQUIRE(D % 8 == 0 && D >= 8 && D <= kMaxVec * 256, "sfc_layernorm_bwd: D=%d unsupported", D);
  SFC_REQUIRE(rows > 0, "sfc_layernorm_bwd: rows must be positive");
  SFC_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "sfc_layernorm_bwd: dropout p out of range");
  const bool drop = dx_drop != nullptr && drop_p > 0.f;
  SFC_REQUIRE(dx_drop == nullptr || drop, "sfc_layernorm_bwd: dx_drop given but drop_p == 0");
  const bool csum = dcolsum != nullptr;
  const int blocks = ln_bwd_blocks(rows);
  SFC_REQUIRE(scratch && scratch_bytes >= (size_t)blocks * 3 * D * sizeof(float), "sfc_layernorm_bwd: scratch too small");
  const size_t smem = (size_t)kLnWarps * 3 * D * sizeof(float);
  const int nv = sfc_ceil_div(D / 8, 32);
#define LN_BWD2(NV, DR, CS)                                                                                         \
  do {                                                                                                              \
    auto k = layernorm_bwd_kernel<NV, DR, CS>;                                                                      \
    if (smem > 48 * 1024) SFC_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    SFC_CUDA_OK(sfc_launch_pdl(k, dim3(blocks), dim3(kLnWarps * 32), smem, stream, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, mean, rstd, \
                               (const __nv_bfloat16*)gamma, (__nv_bfloat16*)dx, (__nv_bfloat16*)dx_drop,            \
                               drop_p, drop_seed, sfc_dropout_epoch_ptr(), (float*)scratch, rows, D));              \
  } while (0)
#define LN_BWD(NV)                                                                  \
  do {                                                                              \
    if (drop && csum) LN_BWD2(NV, true, true);                                      \
    else if (drop) LN_BWD2(NV, true, false);                                        \
    else if (csum) LN_BWD2(NV, false, true);                                        \
    else LN_BWD2(NV, false, false);                                                 \
  } while (0)
  if (nv <= 1) LN_BWD(1); else if (nv <= 2) LN_BWD(2); else if (nv <= 3) LN_BWD(3); else if (nv <= 4) LN_BWD(4); else LN_BWD(8);
#undef LN_BWD
#undef LN_BWD2
  SFC_LAUNCH_OK();
  FinalizeOut outs;
  outs.ptr[0] = dgamma; outs.ptr[1] = dbeta; outs.ptr[2] = dcolsum;
  dim3 grid(sfc_ceil_div(D, 32), csum ? 3 : 2);
  SFC_CUDA_OK(sfc_launch_pdl(partial_finalize_kernel<32>, grid, dim3(1024), 0, stream, (const float*)scratch, blocks, 3ll * D, (long long)D, D, outs, param_fp32, accumulate));
  SFC_LAUNCH_OK();
  return 0;
}

static int colsum_row_blocks(long long rows) {
  long long b = sfc_ceil_div64(rows, 256);
  if (b > 128) b = 128;
  return (int)(b < 1 ? 1 : b);
}

extern "C" size_t sfc_colsum_scratch_bytes(long long rows, int N) { return (size_t)colsum_row_blocks(rows) * (size_t)N * sizeof(float); }

// out[n] = sum_m x[m, n]   (bias gradients)
extern "C" int sfc_colsum(const void* x, long long ld, long long rows, int N, void* out, int out_fp32, int accumulate, void* scratch,
                          size_t scratch_bytes, cudaStream_t stream) {
  SFC_REQUIRE(x && out && rows > 0 && N > 0, "sfc_colsum: bad arguments");
  const int rb = colsum_row_blocks(rows);
  SFC_REQUIRE(scratch && scratch_bytes >= (size_t)rb * N * sizeof(float), "sfc_colsum: scratch too small");
  dim3 grid(sfc_ceil_div(N, 256), rb);
  colsum_partial_kernel<<<grid, 256, 0, stream>>>((const __nv_bfloat16*)x, ld, rows, N, (float*)scratch, sfc_ceil_div64(rows, rb));
  SFC_LAUNCH_OK();
  FinalizeOut outs;
  outs.ptr[0] = out; outs.ptr[1] = nullptr; outs.ptr[2] = nullptr;
  partial_finalize_kernel<8><<<dim3(sfc_ceil_div(N, 32), 1), 256, 0, stream>>>((const float*)scratch, rb, (long long)N, 0, N, outs, out_fp32, accumulate);
  SFC_LAUNCH_OK();
  return 0;
}

// out[i] = alpha * dy[i] * f'(aux[i]) * keep(seed, i) / (1 - drop_p)   (n % 8 == 0, contiguous bf16)
extern "C" int sfc_act_bwd(const void* dy, const void* aux, void* out, long long n, int aux_mode, float alpha, float drop_p,
                           unsigned long long drop_seed, cudaStream_t stream) {
  SFC_REQUIRE(dy && out && n >= 0 && n % 8 == 0, "sfc_act_bwd: bad arguments (n must be a multiple of 8)");
  SFC_REQUIRE(aux_mode == SFC_AUX_NONE || aux != nullptr, "sfc_act_bwd: aux is null");
  SFC_REQUIRE(aux_mode >= SFC_AUX_NONE && aux_mode <= SFC_AUX_GELU_GRAD, "sfc_act_bwd: bad mode");
  if (n == 0) return 0;
  long long blocks = sfc_ceil_div64(n / 8, 256);
  const long long cap = 16ll * sfc_num_sms();
  if (blocks > cap) blocks = cap;
  act_bwd_kernel<<<(unsigned)blocks, 256, 0, stream>>>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)aux, (__nv_bfloat16*)out, n / 8,
                                                       aux_mode, alpha, drop_p, drop_seed, sfc_dropout_epoch_ptr());
  SFC_LAUNCH_OK();
  return 0;
}
