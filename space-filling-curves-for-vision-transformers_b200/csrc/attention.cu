// K4 — tcgen05 flash attention, forward and backward, head_dim = 64, non-causal, no mask (sm_100a).
//
// Replaces F.scaled_dot_product_attention inside nn.MultiheadAttention of the reference encoder
// (/root/reference/src/models/vit.py:197-206 -> torch TransformerEncoderLayer._sa_block; enable_flash_sdp at
// main.py:158-159) and the explicit softmax(QK^T)V of altvit.py:129-141.
//
// Data layout: the packed in-projection output qkv[B*N, 3*D] (bf16) is read IN PLACE through one TMA tensor
// map: Q/K/V tile of head h = 64-column box at column h*64 / D+h*64 / 2D+h*64. Outputs: O[B*N, D] (heads
// concatenated, ready for out_proj) and LSE[B, H, N] (fp32, natural log) for the backward pass.
//
// Forward, one CTA per (128-query tile, head, image): S = Q K^T (tcgen05, fp32 in TMEM), each of the 128
// threads owns one query row (TMEM lane == row, so the row max / sum need no shuffles), exp2 online softmax,
// P (bf16) is written to shared memory in the swizzled K-major layout and O_j = P V_j runs on the tensor core
// with V read as an MN-major operand (no transpose); the running O is rescaled in registers.
// Backward, one CTA per (128-key tile, head, image), loop over query tiles: S and dP = dO V^T on the tensor
// core, P / dS in registers -> shared memory, dV += P^T dO, dK += dS^T Q (MN-major A operands, accumulators
// resident in TMEM across the loop) and dQ_i = dS K (red.global.add into an fp32 accumulator).
#include "common.cuh"
#include "gemm_epilogue.cuh"   // DropKey, drop_apply
#include "sfcvit.h"

namespace {

constexpr int DH = 64;
constexpr int BQ = 128;
constexpr int kTile = BQ * DH * 2;          // 16384 bytes: one 128 x 64 bf16 tile
constexpr float kLog2e = 1.4426950408889634f;

struct AttnParams {
  int B, H, N, D;
  float scale;
  float drop_p;
  unsigned long long drop_seed;
  const unsigned long long* drop_epoch;
  __nv_bfloat16* out;      // fwd: O [B*N, D]
  float* lse;              // [B, H, N]
  // backward
  const __nv_bfloat16* o;  // [B*N, D]
  const __nv_bfloat16* dout;  // [B*N, D]
  __nv_bfloat16* dqkv;     // [B*N, 3D]
  float* dq_acc;           // [B*N, D] fp32, zero-initialised (more than two key tiles: red.global.add)
  __nv_bfloat16* dq_part;  // one or two key tiles: bf16 [B*N, D] partial of key tile 0 when there are two (no atomics)
  int wide_st;             // backward read-out: 256-bit stores (dqkv and the partial buffer 32-byte aligned)
  int dq_mode;             // 0 = atomics into dq_acc, 1 = single key tile -> dqkv directly, 2 = tile 0 -> dq_part, tile 1 -> dqkv
  float* delta;            // [B, H, N] fp32 rowsum(dO * O)
  long long* dbg;          // optional timeline buffer (sfc_debug_set_timeline), CTA 0 only
};

// 16 consecutive values (columns c16*16 .. +15 of row r) as bf16 into the K-major SW128 operand buffer (buf = 32-bit
// shared-window address: st.shared, no generic-address arithmetic)
__device__ __forceinline__ void store_p_half(uint32_t buf, int r, int c16, const float* v) {
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int j8 = c16 * 2 + q;
    const uint32_t x = ptx::pack_bf16(v[q * 8 + 0], v[q * 8 + 1]), y = ptx::pack_bf16(v[q * 8 + 2], v[q * 8 + 3]);
    const uint32_t z = ptx::pack_bf16(v[q * 8 + 4], v[q * 8 + 5]), w = ptx::pack_bf16(v[q * 8 + 6], v[q * 8 + 7]);
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(buf + (uint32_t)((j8 >> 3) * kTile + r * 128 + (((j8 & 7) ^ (r & 7)) << 4))),
                 "r"(x), "r"(y), "r"(z), "r"(w)
                 : "memory");
  }
}

#ifdef SFC_ATTN_TIMELINE
#define SFC_TL(...) __VA_ARGS__
#else
#define SFC_TL(...)
#endif

// ================================================= forward =================================================
// Persistent, warp-specialised. Work item = (image b, head h, query pair qp): 256 query rows = two 128-row tiles A
// and B, each owned by one softmax warpgroup (thread <-> query row <-> TMEM lane), so the tensor core, the TMA engine
// and the other warpgroup always have independent work while one warpgroup is inside its exp loop.
//   warp 0 : TMA producer (Q tiles, K / V tiles of `bkv` keys; runs ahead across items)
//   warp 1 : MMA issuer   (S_w = Q_w K^T into TMEM region w; O_w = P_w V into the same region once P_w is in smem)
//   warp 2 : TMEM allocator;  warps 4-7 : softmax warpgroup A;  warps 8-11 : softmax warpgroup B
// The key tile size is a runtime value (any multiple of 16 up to 208): N <= 208 (the 14 x 14 grid: 196 -> 208) is a
// single pass without online-softmax rescaling; longer sequences use equal tiles of <= 192 keys, double buffered.
constexpr int kFwdThreads = 384;
constexpr int kFwdMaxSingleN = 208;   // longest sequence served in one key pass: the 14 x 14 grid's 196 keys padded to 208

struct FwdLayout {          // runtime shared-memory map (bytes), all tile bases 1024-byte aligned
  int bkv, nkv, stages, p_atoms;
  int off_k, off_v, off_p, off_bar, total;
};

inline FwdLayout fwd_layout(int N) {
  FwdLayout L;
  if (N <= kFwdMaxSingleN) { L.bkv = (N + 15) / 16 * 16; L.nkv = 1; L.stages = 1; }
  else {
    L.nkv = (N + 191) / 192;
    if (L.nkv < 2) L.nkv = 2;
    L.bkv = ((N + L.nkv - 1) / L.nkv + 15) / 16 * 16;
    L.stages = 2;
  }
  L.p_atoms = (L.bkv + 63) / 64;
  const int kv_bytes = (L.bkv * 128 + 1023) / 1024 * 1024;
  L.off_k = 2 * kTile;
  L.off_v = L.off_k + L.stages * kv_bytes;
  L.off_p = L.off_v + L.stages * kv_bytes;
  L.off_bar = L.off_p + 2 * L.p_atoms * kTile;
  L.total = L.off_bar + 32 * 8 + 16 + 1024;
  return L;
}

struct FwdBars {            // mbarrier indices
  static constexpr int q_full = 0, q_empty = 2, k_full = 4, k_empty = 6, v_full = 8, v_empty = 10, s_full = 12, p_full = 14,
                       o_full = 16, o_empty = 18, count = 20;
};

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---- the exp pass as an explicitly interleaved instruction stream -------------------------------------------------
// Measured (profiles/r2_attn_fwd_timeline.txt, tools/pipe_bench.cu): MUFU.EX2 occupies its pipe for 8 cycles per warp
// instruction but does NOT block the scheduler — other pipes keep issuing — provided the instruction stream offers them
// work BETWEEN the MUFUs. Left to ptxas, a 32-column chunk became 32 x (FFMA, MUFU, FADD) followed by ~140 integer / select
// / convert instructions of the dropout mask and the bf16 pack: two phases bound by different pipes that a warp executes
// one after the other (18 cycles per element instead of 8). Here the stream is written out by hand in units of 16 key
// columns (= one dropout group) as a software pipeline: while unit u's exponentials go down the MUFU pipe, the row sum,
// mask, pack and shared-memory store of unit u-1 are independent work for the issue slots in between (~6.5 instructions
// per MUFU); ptxas schedules the merged stream (measured: 7.8 SASS instructions per element, 0.169 -> 0.134 ms).
template <int I>
__device__ __forceinline__ void exp_post_elem(float& pv, float& psum, uint32_t seed, uint32_t thr_hi, bool drop) {
  asm("add.f32 %0, %0, %1;" : "+f"(psum) : "f"(pv));                 // the denominator sums the UNMASKED probabilities
  if (drop) {
    constexpr uint32_t A = lcg_mul(I + 1), C = lcg_add(I + 1);
    asm(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .u32 t;\n\t"
        "mad.lo.u32 t, %1, %2, %3;\n\t"
        "setp.ge.u32 p, t, %4;\n\t"
        "selp.f32 %0, %0, 0f00000000, p;\n\t"
        "}"
        : "+f"(pv)
        : "r"(seed), "n"(A), "n"(C), "r"(thr_hi));
  }
}
__device__ __forceinline__ uint32_t cvt_bf16x2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
// shared-memory address (32-bit window) of the 16-byte slot j8 (8 keys) of row r in the K-major SW128 P operand
__device__ __forceinline__ uint32_t p_slot_addr(uint32_t rowbase, int rx, int j8) {
  return rowbase + (uint32_t)((j8 >> 3) * kTile + (((j8 & 7) ^ rx) << 4));
}

// One pipeline step: exponentials of 16 raw scores s[0..15] into pn[] (stage A of the current unit) interleaved with the
// row sum / dropout mask / pack / store of the previous unit's probabilities pp[] (stage B). kDrop: pp's mask comes from
// `seed_prev` (one hash per aligned group of 16 keys, csrc/gemm_epilogue.cuh). st0 / st1: the previous unit's two slots.
template <bool kDrop, int I>
__device__ __forceinline__ void exp_step_elem(const uint32_t* s, float sl2, float nmb, float* pn, float* pp, float& psum,
                                              uint32_t seed_prev, uint32_t thr_hi, uint32_t* pk) {
  float x;
  asm("fma.rn.f32 %0, %1, %2, %3;" : "=f"(x) : "f"(__uint_as_float(s[I])), "f"(sl2), "f"(nmb));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(pn[I]) : "f"(x));
  exp_post_elem<I>(pp[I], psum, seed_prev, thr_hi, kDrop);
  if constexpr ((I & 1) == 1) pk[I >> 1] = cvt_bf16x2(pp[I - 1], pp[I]);
}
template <bool kDrop>
__device__ __forceinline__ void exp_step(const uint32_t* s, float sl2, float nmb, float (&pn)[16], float (&pp)[16], float& psum,
                                         uint32_t seed_prev, uint32_t thr_hi, uint32_t st0, uint32_t st1) {
  uint32_t pk[8];
  exp_step_elem<kDrop, 0>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 1>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 2>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 3>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 4>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 5>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 6>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 7>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  sts_v4(st0, pk[0], pk[1], pk[2], pk[3]);
  exp_step_elem<kDrop, 8>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 9>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 10>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 11>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 12>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 13>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 14>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  exp_step_elem<kDrop, 15>(s, sl2, nmb, pn, pp, psum, seed_prev, thr_hi, pk);
  sts_v4(st1, pk[4], pk[5], pk[6], pk[7]);
}
// drains the pipeline: stage B of the last unit
template <bool kDrop, int I>
__device__ __forceinline__ void exp_flush_elem(float* pp, float& psum, uint32_t seed_prev, uint32_t thr_hi, uint32_t* pk) {
  exp_post_elem<I>(pp[I], psum, seed_prev, thr_hi, kDrop);
  if constexpr ((I & 1) == 1) pk[I >> 1] = cvt_bf16x2(pp[I - 1], pp[I]);
}
template <bool kDrop>
__device__ __forceinline__ void exp_flush(float (&pp)[16], float& psum, uint32_t seed_prev, uint32_t thr_hi, uint32_t st0, uint32_t st1) {
  uint32_t pk[8];
  exp_flush_elem<kDrop, 0>(pp, psum, seed_prev, thr_hi, pk);   exp_flush_elem<kDrop, 1>(pp, psum, seed_prev, thr_hi, pk);
  exp_flush_elem<kDrop, 2>(pp, psum, seed_prev, thr_hi, pk);   exp_flush_elem<kDrop, 3>(pp, psum, seed_prev, thr_hi, pk);
  exp_flush_elem<kDrop, 4>(pp, psum, seed_prev, thr_hi, pk);   exp_flush_elem<kDrop, 5>(pp, psum, seed_prev, thr_hi, pk);
  exp_flush_elem<kDrop, 6>(pp, psum, seed_prev, thr_hi, pk);   exp_flush_elem<kDrop, 7>(pp, psum, seed_prev, thr_hi, pk);
  sts_v4(st0, pk[0], pk[1], pk[2], pk[3]);
  exp_flush_elem<kDrop, 8>(pp, psum, seed_prev, thr_hi, pk);   exp_flush_elem<kDrop, 9>(pp, psum, seed_prev, thr_hi, pk);
  exp_flush_elem<kDrop, 10>(pp, psum, seed_prev, thr_hi, pk);  exp_flush_elem<kDrop, 11>(pp, psum, seed_prev, thr_hi, pk);
  exp_flush_elem<kDrop, 12>(pp, psum, seed_prev, thr_hi, pk);  exp_flush_elem<kDrop, 13>(pp, psum, seed_prev, thr_hi, pk);
  exp_flush_elem<kDrop, 14>(pp, psum, seed_prev, thr_hi, pk);  exp_flush_elem<kDrop, 15>(pp, psum, seed_prev, thr_hi, pk);
  sts_v4(st1, pk[4], pk[5], pk[6], pk[7]);
}

template <bool kSingle, bool kDrop>
__global__ void __launch_bounds__(kFwdThreads, 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_kv,
                const __grid_constant__ CUtensorMap tmap_o, const AttnParams p, const FwdLayout L) {
  extern __shared__ __align__(1024) uint8_t smem_dyn[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.off_bar);
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + FwdBars::count);

  ptx::pdl_launch_dependents();
  const int tid = threadIdx.x, warp = tid >> 5;
  const int bkv = L.bkv, nkv = L.nkv, stages = L.stages;
  const int kv_bytes = (bkv * 128 + 1023) / 1024 * 1024;
  const int nqp = (p.N + 2 * BQ - 1) / (2 * BQ);
  const int n_items = p.B * p.H * nqp;

  if (tid == 0) {
    ptx::prefetch_tmap(&tmap_q);
    ptx::prefetch_tmap(&tmap_kv);
    ptx::prefetch_tmap(&tmap_o);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars[FwdBars::q_full + i], 1);
      ptx::mbar_init(&bars[FwdBars::q_empty + i], 1);
      ptx::mbar_init(&bars[FwdBars::k_full + i], 1);
      ptx::mbar_init(&bars[FwdBars::k_empty + i], 1);
      ptx::mbar_init(&bars[FwdBars::v_full + i], 1);
      ptx::mbar_init(&bars[FwdBars::v_empty + i], 1);
      ptx::mbar_init(&bars[FwdBars::s_full + i], 1);
      ptx::mbar_init(&bars[FwdBars::p_full + i], 128);
      ptx::mbar_init(&bars[FwdBars::o_full + i], 1);
      ptx::mbar_init(&bars[FwdBars::o_empty + i], 128);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc<512>(tmem_ptr);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  ptx::pdl_wait();                                 // set-up done; the previous kernel's qkv is read from here on
  // TMEM region w = columns [w * 256, w * 256 + 256). Single pass: S in [0, bkv <= 208), O overwrites [0, 64).
  // Multi-tile (bkv <= 192): S in [0, 192), O RESIDENT in [192, 256) across the key tiles of an item.
  constexpr uint32_t kOCol = kSingle ? 0u : 192u;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (ptx::elect_one()) {
      int ii = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++ii) {
        const int qp = item % nqp, h = (item / nqp) % p.H, b = item / (nqp * p.H);
        const int row0 = b * p.N;
        for (int w = 0; w < 2; ++w) {
          ptx::mbar_wait_relaxed(&bars[FwdBars::q_empty + w], (ii & 1) ^ 1);
          ptx::mbar_expect_tx(&bars[FwdBars::q_full + w], kTile);
          ptx::tma_load_2d(&tmap_q, &bars[FwdBars::q_full + w], smem + w * kTile, h * DH, row0 + qp * 2 * BQ + w * BQ);
        }
        for (int j = 0; j < nkv; ++j) {
          const int g = ii * nkv + j;
          const int st = g % stages;
          const uint32_t ph = (uint32_t)((g / stages) & 1);
          ptx::mbar_wait_relaxed(&bars[FwdBars::k_empty + st], ph ^ 1);
          ptx::mbar_expect_tx(&bars[FwdBars::k_full + st], (uint32_t)(bkv * 128));
          ptx::tma_load_2d(&tmap_kv, &bars[FwdBars::k_full + st], smem + L.off_k + st * kv_bytes, p.D + h * DH, row0 + j * bkv);
          ptx::mbar_wait_relaxed(&bars[FwdBars::v_empty + st], ph ^ 1);
          ptx::mbar_expect_tx(&bars[FwdBars::v_full + st], (uint32_t)(bkv * 128));
          ptx::tma_load_2d(&tmap_kv, &bars[FwdBars::v_full + st], smem + L.off_v + st * kv_bytes, 2 * p.D + h * DH, row0 + j * bkv);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (ptx::elect_one()) {
      const uint32_t idesc_s = umma_idesc_bf16(BQ, bkv, false, false);
      const uint32_t idesc_o = umma_idesc_bf16(BQ, DH, false, true);
      const int my_items = (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
      const int total = my_items * nkv;
      auto issue_s = [&](int w, int g) {
        const int j = g % nkv, ii = g / nkv, st = g % stages;
        if (j == 0) ptx::mbar_wait_relaxed(&bars[FwdBars::q_full + w], ii & 1);
        ptx::mbar_wait_relaxed(&bars[FwdBars::k_full + st], (g / stages) & 1);
        // single pass: S overwrites the columns O(g-1) was read from. Multi-tile: S has its own columns, which are free
        // once P(g-1) is complete — issue_pv(w, g-1) waited for that just before this call.
        if constexpr (kSingle) ptx::mbar_wait_relaxed(&bars[FwdBars::o_empty + w], (g & 1) ^ 1);
        ptx::tc_fence_after();
        const uint64_t dq = umma_smem_desc_sw128(ptx::smem_u32(smem + w * kTile), 0, 1024);
        const uint64_t dk = umma_smem_desc_sw128(ptx::smem_u32(smem + L.off_k + st * kv_bytes), 0, 1024);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          ptx::umma_f16(tmem_base + w * 256, dq + (uint64_t)(k * 2), dk + (uint64_t)(k * 2), idesc_s, k > 0 ? 1u : 0u);
        ptx::umma_commit(&bars[FwdBars::s_full + w]);
        if (w == 1) ptx::umma_commit(&bars[FwdBars::k_empty + st]);
        if (j == nkv - 1) ptx::umma_commit(&bars[FwdBars::q_empty + w]);
      };
      auto issue_pv = [&](int w, int g) {
        const int st = g % stages;
        const int j = g % nkv, ii = g / nkv;
        if constexpr (kSingle) ptx::mbar_wait_relaxed(&bars[FwdBars::p_full + w], g & 1);   // multi-tile: the caller waited (once)
        ptx::mbar_wait_relaxed(&bars[FwdBars::v_full + st], (g / stages) & 1);
        if constexpr (!kSingle) {
          if (j == 0) ptx::mbar_wait_relaxed(&bars[FwdBars::o_empty + w], (ii & 1) ^ 1);   // previous item's O has been read out
        }
        ptx::tc_fence_after();
        const uint32_t acc0 = (!kSingle && j > 0) ? 1u : 0u;          // multi-tile: O accumulates in TMEM across key tiles
        const uint32_t sp = ptx::smem_u32(smem + L.off_p + w * L.p_atoms * kTile);
        const uint32_t sv = ptx::smem_u32(smem + L.off_v + st * kv_bytes);
        const uint64_t da0 = umma_smem_desc_sw128(sp, 0, 1024);
        const uint64_t db0 = umma_smem_desc_sw128(sv, kTile, 1024);
        const uint32_t a_lo = (uint32_t)da0, a_hi = (uint32_t)(da0 >> 32), b_lo = (uint32_t)db0, b_hi = (uint32_t)(db0 >> 32);
        const int nk = bkv / 16;
#pragma unroll
        for (int k = 0; k < 13; ++k)                 // bkv <= 208; descriptor advances are compile-time constants
          if (k < nk)
            ptx::umma_f16_lohi(tmem_base + w * 256 + kOCol, a_lo + (uint32_t)((k >> 2) * (kTile >> 4) + (k & 3) * 2), a_hi,
                               b_lo + (uint32_t)(k * 128), b_hi, idesc_o, k > 0 ? 1u : acc0);
        ptx::umma_commit(&bars[FwdBars::o_full + w]);
        if (w == 1) ptx::umma_commit(&bars[FwdBars::v_empty + st]);
      };
      if (total > 0) {
        issue_s(0, 0);
        issue_s(1, 0);
        for (int g = 0; g < total; ++g) {
          if constexpr (kSingle) {
            SFC_TL(long long* dbg = (blockIdx.x == 0 && g < 32) ? p.dbg : nullptr;)
            issue_pv(0, g);
            SFC_TL(if (dbg) dbg[g * 32 + 16] = clock64();)
            if (g + 1 < total) issue_s(0, g + 1);
            SFC_TL(if (dbg) dbg[g * 32 + 17] = clock64();)
            issue_pv(1, g);
            SFC_TL(if (dbg) dbg[g * 32 + 18] = clock64();)
            if (g + 1 < total) issue_s(1, g + 1);
            SFC_TL(if (dbg) dbg[g * 32 + 19] = clock64();)
          } else {
            // P(g) complete = the S columns are free: the next S goes FIRST (the softmax warps wait for nothing else),
            // the PV product follows; O lives in its own columns
            for (int w = 0; w < 2; ++w) {
              ptx::mbar_wait_relaxed(&bars[FwdBars::p_full + w], g & 1);
              if (g + 1 < total) issue_s(w, g + 1);
              issue_pv(w, g);
            }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================== softmax warpgroups =====================
    const int w = (warp - 4) >> 2;                 // 0 = tile A, 1 = tile B
    const int quarter = warp & 3;
    const int lane = tid & 31;
    const int r = quarter * 32 + lane;             // row in tile == TMEM lane
    const uint32_t t_s = tmem_base + w * 256 + ((uint32_t)(quarter * 32) << 16);
    uint8_t* p_smem = smem + L.off_p + w * L.p_atoms * kTile;      // P operand; its first 16 KB double as the O staging tile
    const float sl2 = p.scale * kLog2e;
    const DropKey dkey = drop_key(p.drop_seed, p.drop_p, p.drop_epoch);
    const uint32_t thr_hi = dkey.thr16 << 16;
    const uint32_t p_s32 = ptx::smem_u32(p_smem);                  // 32-bit shared address: st.shared, no 64-bit address math
    const uint32_t p_row = p_s32 + (uint32_t)(r * 128);
    const int rx = r & 7;
    const bool store_owner = quarter == 0 && lane == 0;            // issues (and waits for) this tile's TMA stores
    int g = 0, ii = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++ii) {
      const int qp = item % nqp, h = (item / nqp) % p.H, b = item / (nqp * p.H);
      const int q_tile0 = qp * 2 * BQ + w * BQ;
      const int qi = q_tile0 + r;
      const bool warp_active = q_tile0 + quarter * 32 < p.N;     // warp-uniform: at least one valid query row
      // m_run = the row maximum the probabilities are scaled by. Multi-tile: it is raised (and O, l rescaled) only when
      // the true maximum exceeds it by more than 2^8 — P stays <= 256, the final O / l is unchanged.
      float m_run = -INFINITY, l_run = 0.f;
      for (int j = 0; j < nkv; ++j, ++g) {
        SFC_TL(long long* dbg = (blockIdx.x == 0 && g < 32 && (tid == 128 || tid == 256)) ? p.dbg + g * 32 + w * 8 : nullptr;)
        SFC_TL(if (dbg) dbg[0] = clock64();)
        ptx::mbar_wait_relaxed(&bars[FwdBars::s_full + w], g & 1);
        ptx::tc_fence_after();
        SFC_TL(if (dbg) dbg[1] = clock64();)
        uint32_t ra[32], rb[32];
        if (warp_active) {
          const int kv_valid = min(bkv, p.N - j * bkv);
          const int nch = (kv_valid + 31) / 32;
          // Both passes keep the TMEM load of the next 32-column chunk in flight while the current one is processed
          // (two register buffers, loop unrolled by two so that they stay in registers).
          float mx = -INFINITY, mx1 = -INFINITY;   // two chains of 3-input maxima: issue-bound, not latency-bound
          auto max_chunk = [&](const uint32_t (&rr)[32], int c) {
            if (c * 32 + 32 <= kv_valid) {
#pragma unroll
              for (int i = 0; i < 32; i += 8) {
                mx = fmaxf(mx, fmaxf(__uint_as_float(rr[i]), __uint_as_float(rr[i + 1])));
                mx1 = fmaxf(mx1, fmaxf(__uint_as_float(rr[i + 2]), __uint_as_float(rr[i + 3])));
                mx = fmaxf(mx, fmaxf(__uint_as_float(rr[i + 4]), __uint_as_float(rr[i + 5])));
                mx1 = fmaxf(mx1, fmaxf(__uint_as_float(rr[i + 6]), __uint_as_float(rr[i + 7])));
              }
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (c * 32 + i < kv_valid) mx = fmaxf(mx, __uint_as_float(rr[i]));
            }
          };
          ptx::tmem_ld_x32(t_s, ra);
#pragma unroll 1
          for (int c = 0; c < nch; c += 2) {
            ptx::tmem_ld_wait();
            if (c + 1 < nch) ptx::tmem_ld_x32(t_s + (c + 1) * 32, rb);
            max_chunk(ra, c);
            if (c + 1 < nch) {
              ptx::tmem_ld_wait();
              if (c + 2 < nch) ptx::tmem_ld_x32(t_s + (c + 2) * 32, ra);
              max_chunk(rb, c + 1);
            }
          }
          mx = fmaxf(mx, mx1);
          if constexpr (kSingle) {
            m_run = mx;
          } else {
            if (j == 0) {
              m_run = mx;
            } else {
              // PV(g-1) was issued right after S(g): every o_full phase is consumed exactly once, here or at the item's end
              ptx::mbar_wait_relaxed(&bars[FwdBars::o_full + w], (g - 1) & 1);
              ptx::tc_fence_after();
              const bool need = (mx - m_run) * sl2 > 8.0f;
              if (__any_sync(0xffffffffu, need)) {
                const float alpha = need ? ex2_approx((m_run - mx) * sl2) : 1.0f;
#pragma unroll
                for (int c = 0; c < DH / 32; ++c) {
                  ptx::tmem_ld_x32(t_s + kOCol + c * 32, ra);
                  ptx::tmem_ld_wait();
#pragma unroll
                  for (int i = 0; i < 32; ++i) ra[i] = __float_as_uint(__uint_as_float(ra[i]) * alpha);
                  ptx::tmem_st_x32(t_s + kOCol + c * 32, ra);
                  ptx::tmem_st_wait();
                }
                l_run *= alpha;
                if (need) m_run = mx;
              }
            }
          }
          ptx::tmem_ld_x32(t_s, ra);                    // first chunk of pass 2, in flight during the scalar work below
        }
        // The previous item's TMA store reads the staging tile that aliases this P operand: its owner waits for that read,
        // the tile-wide barrier hands the news to the other 127 threads before anybody writes P again.
        if (store_owner) ptx::tma_store_wait_read<0>();
        ptx::named_bar_sync(1 + w, 128);
        SFC_TL(if (dbg) dbg[2] = clock64();)
        if (warp_active) {
          const int kv_valid = min(bkv, p.N - j * bkv);
          const int nch = (kv_valid + 31) / 32;
          const float nmb = -m_run * sl2;
          float psum = 0.f;
          // dropout index space: (probability row) x (key index, row pitch padded to 16 so that 16-key groups are aligned)
          unsigned long long drop_grp = 0;
          if constexpr (kDrop)
            drop_grp = ((((unsigned long long)(b * p.H + h) * p.N + (unsigned long long)qi) * (unsigned long long)((p.N + 15) & ~15)) + (unsigned long long)(j * bkv)) >> 4;
          // software pipeline over 16-column units (see exp_step): pp = probabilities of the previous unit, still to be
          // summed / masked / packed / stored. It starts with an all-zero dummy unit aimed at unit 0's slots (which the
          // real unit 0 rewrites afterwards, same thread, program order).
          float pp[16], pq[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) pp[i] = 0.f;
          uint32_t seed_prev = 0, st0 = p_slot_addr(p_row, rx, 0), st1 = p_slot_addr(p_row, rx, 1);
          // one 32-column chunk = two units; the probability buffers swap roles (pp -> pq -> pp): no register copies
          auto chunk = [&](uint32_t* s32, int c) {
            const int nv = kv_valid - c * 32;
            if (nv < 32) {                              // keys past the sequence end: exp2(-inf) = 0
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (i >= nv) s32[i] = 0xff800000u;
            }
            exp_step<kDrop>(s32, sl2, nmb, pq, pp, psum, seed_prev, thr_hi, st0, st1);
            if constexpr (kDrop) seed_prev = drop_hash2(dkey, drop_grp + (unsigned long long)(2 * c));
            st0 = p_slot_addr(p_row, rx, 4 * c);
            st1 = p_slot_addr(p_row, rx, 4 * c + 1);
            exp_step<kDrop>(s32 + 16, sl2, nmb, pp, pq, psum, seed_prev, thr_hi, st0, st1);
            if constexpr (kDrop) seed_prev = drop_hash2(dkey, drop_grp + (unsigned long long)(2 * c + 1));
            st0 = p_slot_addr(p_row, rx, 4 * c + 2);
            st1 = p_slot_addr(p_row, rx, 4 * c + 3);
          };
#pragma unroll 1
          for (int c = 0; c < nch; c += 2) {
            ptx::tmem_ld_wait();
            if (c + 1 < nch) ptx::tmem_ld_x32(t_s + (c + 1) * 32, rb);
            chunk(ra, c);
            if (c + 1 < nch) {
              ptx::tmem_ld_wait();
              if (c + 2 < nch) ptx::tmem_ld_x32(t_s + (c + 2) * 32, ra);
              chunk(rb, c + 1);
            }
          }
          exp_flush<kDrop>(pp, psum, seed_prev, thr_hi, st0, st1);
          for (int u = 2 * nch; u < (bkv >> 4); ++u) {  // whole chunks past the sequence end inside [0, bkv): P = 0
            ptx::sts_zero16(p_slot_addr(p_row, rx, 2 * u));
            ptx::sts_zero16(p_slot_addr(p_row, rx, 2 * u + 1));
          }
          l_run += psum;
        }
        SFC_TL(if (dbg) dbg[3] = clock64();)
        ptx::tc_fence_before();
        ptx::fence_proxy_async_smem();
        ptx::mbar_arrive(&bars[FwdBars::p_full + w]);
        SFC_TL(if (dbg) dbg[4] = clock64();)
        // The softmax warps do not stall on a PV product between key tiles: S(g+1) goes to its own columns and O stays in
        // TMEM; the finished O is normalised and stored from TMEM after the item's last PV.
        if constexpr (!kSingle) {
          if (j < nkv - 1) continue;
        }
        ptx::mbar_wait_relaxed(&bars[FwdBars::o_full + w], g & 1);
        ptx::tc_fence_after();
        SFC_TL(if (dbg) dbg[5] = clock64();)
        if (warp_active) {
          ptx::tmem_ld_x32(t_s + kOCol, ra);
          ptx::tmem_ld_x32(t_s + kOCol + 32, rb);
          ptx::tmem_ld_wait();
        }
        // O sits in registers: the accumulator columns are released BEFORE the rows are normalised and stored, so the next
        // item's S product (single pass: it overwrites these columns) starts ~1.5 k cycles earlier
        ptx::tc_fence_before();
        ptx::mbar_arrive(&bars[FwdBars::o_empty + w]);
        if (warp_active) {
          const float inv_l = (kDrop ? dkey.inv_keep : 1.0f) / l_run;   // O = (keep . P / keep_prob) V / l: the mask zeroes, this scales
          // one 128-byte row per thread into the SW128 staging tile (16-byte slot ^= row & 7: conflict-free), then ONE TMA
          // store per tile — row-per-lane st.global touched 32 different lines per instruction (~1.7 k cycles per tile)
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const uint32_t* src = q < 4 ? ra + q * 8 : rb + (q - 4) * 8;
            sts_v4(p_row + (uint32_t)((q ^ rx) << 4),
                   ptx::pack_bf16(__uint_as_float(src[0]) * inv_l, __uint_as_float(src[1]) * inv_l),
                   ptx::pack_bf16(__uint_as_float(src[2]) * inv_l, __uint_as_float(src[3]) * inv_l),
                   ptx::pack_bf16(__uint_as_float(src[4]) * inv_l, __uint_as_float(src[5]) * inv_l),
                   ptx::pack_bf16(__uint_as_float(src[6]) * inv_l, __uint_as_float(src[7]) * inv_l));
          }
          if (qi < p.N && p.lse) p.lse[((long long)b * p.H + h) * p.N + qi] = m_run * p.scale + logf(l_run);
        }
        ptx::fence_proxy_async_smem();
        ptx::named_bar_sync(3 + w, 128);                            // the staging tile is complete
        if (store_owner && q_tile0 < p.N) {
          ptx::tma_store_3d(&tmap_o, p_smem, h * DH, q_tile0, b);   // rows past the image end are clipped by the tensor map
          ptx::tma_store_commit();
        }
        SFC_TL(if (dbg) dbg[6] = clock64();)
      }
    }
    if (store_owner) ptx::tma_store_wait_all<0>();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

// ================================================= backward =================================================
// Persistent, warp-specialised. Work item = (image b, head h, key tile jt of `bkv` <= 128 keys); inside an item the
// CTA walks the 128-row query tiles ("steps"). dV / dK of the item stay in TMEM across its steps, dQ of each step is
// reduced into an fp32 scratch with red.global.add (key tiles of one head run on different CTAs).
//   warp 0 : TMA producer (K, V per item, double buffered; Q, dO per step, 3 stages; runs ahead across items)
//   warp 1 : MMA issuer
//   warp 2 : TMEM allocator;  warps 4-19 : four element-wise warpgroups (thread <-> query row; warpgroup c owns the
//            32-column chunk c of the S / dP tile) — 4 warps per scheduler hide each other's TMEM / MUFU latencies
// TMEM (512 columns): S0 | S1 | dP | dV dK. Per step s the issuer runs
//   S(s+1) -> S[(s+1)&1]        early, so the exp pass of step s+1 overlaps the gradient MMAs of step s
//   dV += P^T dO, dK += dS^T Q, dQ(s) = dS K -> S[s&1] (dead by then)      after P / dS of step s are in smem
//   dP(s+1) = dO V^T -> dP
// and the warpgroups run  P = exp2(S - lse) (kept in registers)  ->  read dQ(s-1) out  ->  dS = P (dP - delta) scale.
// Per-step clock64 stamps of CTA 0 (tools/attn_timeline.py): compiled in only with -DSFC_ATTN_TIMELINE, they cost
// registers in a kernel that is 2 registers away from spilling.
constexpr int kBwdEwWarps = 16;                 // element-wise warps: 4 per TMEM lane quarter, one 32-column chunk each
constexpr int kBwdThreads = 64 + kBwdEwWarps * 32;   // warp 0: TMEM alloc + TMA, warp 1: MMA issuer; 18 warps leave 112 registers per thread
constexpr int kQdoStages = 3;

struct BwdSmem {
  static constexpr int kK = 0;                          // 2 stages x 16 KB
  static constexpr int kV = kK + 2 * kTile;             // 2 stages
  static constexpr int kQ = kV + 2 * kTile;             // 3 stages
  static constexpr int kDO = kQ + kQdoStages * kTile;   // 3 stages
  static constexpr int kP = kDO + kQdoStages * kTile;   // 128 x 128 bf16 (rows = query, cols = key)
  static constexpr int kDS = kP + 2 * kTile;
  static constexpr int kBar = kDS + 2 * kTile;
  static constexpr int kTotal = kBar + 24 * 8 + 16 + 1024;
  static_assert(kTotal <= 232448, "exceeds 227 KB");
};

struct BwdBars {
  static constexpr int kv_full = 0, kv_empty = 2, qdo_full = 4, qdo_empty = 7, s_full = 10, dp_full = 12, pds_full = 13,
                       dq_full = 14, dq_empty = 15, count = 16;
};

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// delta[b, h, n] = sum_d dO[b, n, h, d] * O[b, n, h, d]   (8 lanes per (row, head), fully coalesced)
__global__ void __launch_bounds__(256) attn_bwd_prep_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ dout,
                                                            float* __restrict__ delta, long long rows, int N, int H) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const long long total = rows * H * 8;
  const int lane = threadIdx.x & 31;
  // warp-uniform loop (the shuffles below need all 32 lanes)
  for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < total; base += (long long)gridDim.x * blockDim.x) {
    const long long t = base + lane;
    const bool ok = t < total;
    const long long rh = (ok ? t : total - 1) >> 3;
    const long long row = rh / H;
    const int h = (int)(rh % H);
    const long long off = (row * H + h) * DH + (t & 7) * 8;
    float s = 0.f;
    if (ok) {
      const uint4 a = __ldg(reinterpret_cast<const uint4*>(o + off)), d = __ldg(reinterpret_cast<const uint4*>(dout + off));
      s = ptx::bf16_lo(a.x) * ptx::bf16_lo(d.x) + ptx::bf16_hi(a.x) * ptx::bf16_hi(d.x) + ptx::bf16_lo(a.y) * ptx::bf16_lo(d.y) +
          ptx::bf16_hi(a.y) * ptx::bf16_hi(d.y) + ptx::bf16_lo(a.z) * ptx::bf16_lo(d.z) + ptx::bf16_hi(a.z) * ptx::bf16_hi(d.z) +
          ptx::bf16_lo(a.w) * ptx::bf16_lo(d.w) + ptx::bf16_hi(a.w) * ptx::bf16_hi(d.w);
    }
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    if (ok && (t & 7) == 0) {
      const long long b = row / N, n = row % N;
      delta[(b * H + h) * N + n] = s;
    }
  }
}

// Position in a CTA's step sequence, advanced without divisions: every warp role walks the same sequence, and with
// five warps per scheduler each scalar instruction of a role costs several cycles of wall time.
struct BwdCursor {
  int s, ii, qt, jt, h, b, st3, ph3;     // step, local item, query tile, (key tile, head, image), Q/dO stage and its phase
  int dh, db, n_kvt, H, nq;
  // head-major: the CTAs stride over heads, and the items of a CTA are (head, key tile 0), (head, key tile 1), ..., next
  // head — so that with two key tiles the second read-out can add the first one's dQ (see readout)
  __device__ __forceinline__ void init(int n_kvt_, int H_, int nq_) {
    n_kvt = n_kvt_; H = H_; nq = nq_;
    const int head = (int)blockIdx.x, g = (int)gridDim.x;
    jt = 0; h = head % H; b = head / H;
    dh = g % H; db = g / H;
    s = 0; ii = 0; qt = 0; st3 = 0; ph3 = 0;
  }
  __device__ __forceinline__ void advance() {
    ++s;
    if (++st3 == kQdoStages) { st3 = 0; ph3 ^= 1; }
    if (++qt == nq) {
      qt = 0; ++ii;
      if (++jt == n_kvt) {
        jt = 0;
        h += dh; if (h >= H) { h -= H; ++b; }
        b += db;
      }
    }
  }
};

// The element-wise warps' view of the same sequence: only what they use, so that the previous / current / next
// positions do not push the 16 warps (96 registers each) into local-memory spills inside the step loop.
struct EwPos {
  int s, qt, jt, h, b;
  __device__ __forceinline__ void advance(int dh, int db, int n_kvt, int H, int nq) {
    ++s;
    if (++qt == nq) {
      qt = 0;
      if (++jt == n_kvt) {
        jt = 0;
        h += dh; if (h >= H) { h -= H; ++b; }
        b += db;
      }
    }
  }
  // two registers for the previous position: qt, jt < 65536; heads < 256; images < 2^23 (checked on the host)
  __device__ __forceinline__ uint2 pack() const { return make_uint2((uint32_t)qt | ((uint32_t)jt << 16), (uint32_t)h | ((uint32_t)b << 8)); }
  __device__ __forceinline__ void unpack(uint2 v, int s_) { s = s_; qt = v.x & 0xffff; jt = v.x >> 16; h = v.y & 255; b = (int)(v.y >> 8); }
};

__global__ void __launch_bounds__(kBwdThreads, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_kv,
                const __grid_constant__ CUtensorMap tmap_do, const AttnParams p, const int bkv) {
  extern __shared__ __align__(1024) uint8_t smem_dyn[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BwdSmem::kBar);
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + BwdBars::count);

  ptx::pdl_launch_dependents();
  const int tid = threadIdx.x, warp = tid >> 5;
  const int nq = (p.N + BQ - 1) / BQ;                       // steps per item
  const int n_kvt = (p.N + bkv - 1) / bkv;
  const int n_heads = p.B * p.H;                              // the CTAs stride over heads
  const int my_heads = (int)blockIdx.x < n_heads ? (n_heads - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int my_items = my_heads * n_kvt;
  const int T = my_items * nq;                              // steps of this CTA

  if (tid == 0) {
    ptx::prefetch_tmap(&tmap_q);
    ptx::prefetch_tmap(&tmap_kv);
    ptx::prefetch_tmap(&tmap_do);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars[BwdBars::kv_full + i], 1);
      ptx::mbar_init(&bars[BwdBars::kv_empty + i], 1);
      ptx::mbar_init(&bars[BwdBars::s_full + i], 1);
    }
    for (int i = 0; i < kQdoStages; ++i) {
      ptx::mbar_init(&bars[BwdBars::qdo_full + i], 1);
      ptx::mbar_init(&bars[BwdBars::qdo_empty + i], 1);
    }
    ptx::mbar_init(&bars[BwdBars::dp_full], 1);
    ptx::mbar_init(&bars[BwdBars::pds_full], kBwdEwWarps * 32);
    ptx::mbar_init(&bars[BwdBars::dq_full], 1);
    ptx::mbar_init(&bars[BwdBars::dq_empty], kBwdEwWarps * 32);
    ptx::fence_barrier_init();
  }
  if (warp == 0) ptx::tmem_alloc<512>(tmem_ptr);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const uint32_t tmem_dp = tmem_base + 256, tmem_dv = tmem_base + 384, tmem_dk = tmem_base + 448;
  ptx::pdl_wait();                                 // set-up done; delta / qkv / dO of the previous kernels are read from here on

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (ptx::elect_one()) {
      BwdCursor c;
      c.init(n_kvt, p.H, nq);
      for (; c.s < T; c.advance()) {
        const int row0 = c.b * p.N;
        if (c.qt == 0) {
          const int kvst = c.ii & 1;
          ptx::mbar_wait_relaxed(&bars[BwdBars::kv_empty + kvst], ((c.ii >> 1) & 1) ^ 1);
          ptx::mbar_expect_tx(&bars[BwdBars::kv_full + kvst], (uint32_t)(2 * bkv * 128));
          ptx::tma_load_2d(&tmap_kv, &bars[BwdBars::kv_full + kvst], smem + BwdSmem::kK + kvst * kTile, p.D + c.h * DH, row0 + c.jt * bkv);
          ptx::tma_load_2d(&tmap_kv, &bars[BwdBars::kv_full + kvst], smem + BwdSmem::kV + kvst * kTile, 2 * p.D + c.h * DH, row0 + c.jt * bkv);
        }
        const int st = c.st3;
        ptx::mbar_wait_relaxed(&bars[BwdBars::qdo_empty + st], (uint32_t)(c.ph3 ^ 1));
        ptx::mbar_expect_tx(&bars[BwdBars::qdo_full + st], 2 * kTile);
        ptx::tma_load_2d(&tmap_q, &bars[BwdBars::qdo_full + st], smem + BwdSmem::kQ + st * kTile, c.h * DH, row0 + c.qt * BQ);
        ptx::tma_load_2d(&tmap_do, &bars[BwdBars::qdo_full + st], smem + BwdSmem::kDO + st * kTile, c.h * DH, row0 + c.qt * BQ);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (ptx::elect_one()) {
      const uint32_t idesc_s = umma_idesc_bf16(BQ, bkv, false, false);     // S, dP : K-major x K-major, N = bkv
      const uint32_t idesc_t = umma_idesc_bf16(128, DH, true, true);       // dV, dK: MN-major A (P^T / dS^T), MN-major B
      const uint32_t idesc_q = umma_idesc_bf16(BQ, DH, false, true);       // dQ    : K-major A (dS), MN-major B (K)
      auto s_issue = [&](const BwdCursor& c) {
        const int s = c.s, st = c.st3, kvst = c.ii & 1;
        ptx::mbar_wait_relaxed(&bars[BwdBars::qdo_full + st], (uint32_t)c.ph3);
        if (c.qt == 0) ptx::mbar_wait_relaxed(&bars[BwdBars::kv_full + kvst], (c.ii >> 1) & 1);
        if (s >= 2) ptx::mbar_wait_relaxed(&bars[BwdBars::dq_empty], s & 1);       // dQ(s-2) read out of S[s&1]
        ptx::tc_fence_after();
        const uint64_t dq = umma_smem_desc_sw128(ptx::smem_u32(smem + BwdSmem::kQ + st * kTile), 0, 1024);
        const uint64_t dk = umma_smem_desc_sw128(ptx::smem_u32(smem + BwdSmem::kK + kvst * kTile), 0, 1024);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          ptx::umma_f16(tmem_base + (s & 1) * 128, dq + (uint64_t)(k * 2), dk + (uint64_t)(k * 2), idesc_s, k > 0 ? 1u : 0u);
        ptx::umma_commit(&bars[BwdBars::s_full + (s & 1)]);
      };
      auto dp_issue = [&](const BwdCursor& c) {
        const int st = c.st3, kvst = c.ii & 1;
        const uint64_t ddo = umma_smem_desc_sw128(ptx::smem_u32(smem + BwdSmem::kDO + st * kTile), 0, 1024);
        const uint64_t dv = umma_smem_desc_sw128(ptx::smem_u32(smem + BwdSmem::kV + kvst * kTile), 0, 1024);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          ptx::umma_f16(tmem_dp, ddo + (uint64_t)(k * 2), dv + (uint64_t)(k * 2), idesc_s, k > 0 ? 1u : 0u);
        ptx::umma_commit(&bars[BwdBars::dp_full]);
      };
      auto grad_issue = [&](const BwdCursor& c) {
        const int s = c.s, qt = c.qt, st = c.st3, kvst = c.ii & 1;
        const int kv_valid = min(bkv, p.N - c.jt * bkv);
        const int q_valid = min(BQ, p.N - qt * BQ);
        const int nk_q = (q_valid + 15) / 16, nk_kv = (kv_valid + 15) / 16;
        const uint32_t sp = ptx::smem_u32(smem + BwdSmem::kP);
        const uint32_t sds = ptx::smem_u32(smem + BwdSmem::kDS);
        const uint32_t sq = ptx::smem_u32(smem + BwdSmem::kQ + st * kTile);
        const uint32_t sdo = ptx::smem_u32(smem + BwdSmem::kDO + st * kTile);
        const uint32_t sk = ptx::smem_u32(smem + BwdSmem::kK + kvst * kTile);
        // dV[kv, d] += sum_q P[q, kv] dO[q, d]   ;   dK[kv, d] += sum_q dS[q, kv] Q[q, d]     (reduction over q rows)
        // Descriptors as {lo, hi} words with compile-time advances: the single issuing thread shares its scheduler with
        // two element-wise warps, so every instruction it does not execute shortens the critical path of the step.
        auto lohi = [](uint64_t d, uint32_t& lo, uint32_t& hi) { lo = (uint32_t)d; hi = (uint32_t)(d >> 32); };
        uint32_t p_lo, p_hi, do_lo, do_hi, ds_lo, ds_hi, q_lo, q_hi, dsk_lo, dsk_hi, k_lo, k_hi;
        lohi(umma_smem_desc_sw128(sp, kTile, 1024), p_lo, p_hi);
        lohi(umma_smem_desc_sw128(sdo, kTile, 1024), do_lo, do_hi);
        lohi(umma_smem_desc_sw128(sds, kTile, 1024), ds_lo, ds_hi);
        lohi(umma_smem_desc_sw128(sq, kTile, 1024), q_lo, q_hi);
        lohi(umma_smem_desc_sw128(sds, 0, 1024), dsk_lo, dsk_hi);
        lohi(umma_smem_desc_sw128(sk, kTile, 1024), k_lo, k_hi);
        const uint32_t acc0 = qt > 0 ? 1u : 0u;
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k < nk_q) ptx::umma_f16_lohi(tmem_dv, p_lo + (uint32_t)(k * 128), p_hi, do_lo + (uint32_t)(k * 128), do_hi, idesc_t, k > 0 ? 1u : acc0);
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k < nk_q) ptx::umma_f16_lohi(tmem_dk, ds_lo + (uint32_t)(k * 128), ds_hi, q_lo + (uint32_t)(k * 128), q_hi, idesc_t, k > 0 ? 1u : acc0);
        // dQ[q, d] = sum_kv dS[q, kv] K[kv, d]  -> S[s & 1] columns 0..63
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k < nk_kv)
            ptx::umma_f16_lohi(tmem_base + (s & 1) * 128, dsk_lo + (uint32_t)((k >> 2) * (kTile >> 4) + (k & 3) * 2), dsk_hi,
                               k_lo + (uint32_t)(k * 128), k_hi, idesc_q, k > 0 ? 1u : 0u);
        ptx::umma_commit(&bars[BwdBars::dq_full]);
        ptx::umma_commit(&bars[BwdBars::qdo_empty + st]);
        if (qt == nq - 1) ptx::umma_commit(&bars[BwdBars::kv_empty + kvst]);
      };
      SFC_TL(long long* dbg = (blockIdx.x == 0) ? p.dbg : nullptr;)
      if (T > 0) {
        BwdCursor c0, c1;                                        // steps s and s + 1
        c0.init(n_kvt, p.H, nq);
        c1 = c0;
        s_issue(c0);
        dp_issue(c0);
        c1.advance();
        for (int s = 0; s < T; ++s) {
          SFC_TL(if (dbg && s < 64) dbg[s * 16 + 8] = clock64();)
          if (s + 1 < T) s_issue(c1);
          SFC_TL(if (dbg && s < 64) dbg[s * 16 + 9] = clock64();)
          ptx::mbar_wait_relaxed(&bars[BwdBars::pds_full], s & 1);       // P / dS of step s are in smem, dP(s) has been consumed
          SFC_TL(if (dbg && s < 64) dbg[s * 16 + 12] = clock64();)
          ptx::tc_fence_after();
          if (s + 1 < T) dp_issue(c1);                           // first: it is the input the warpgroups wait for next
          SFC_TL(if (dbg && s < 64) dbg[s * 16 + 11] = clock64();)
          grad_issue(c0);
          SFC_TL(if (dbg && s < 64) dbg[s * 16 + 10] = clock64();)
          c0 = c1;
          c1.advance();
        }
      }
    }
    __syncwarp();
  } else if (warp >= 2) {
    // ===================== element-wise warpgroups =====================
    const int ch = (warp - 2) >> 2;                // this warp's 32-column chunk of the S / dP tile (0..3)
    const int quarter = warp & 3;
    const int lane = tid & 31;
    const int r = quarter * 32 + lane;             // query row in tile == TMEM lane
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
    const float sl2 = p.scale * kLog2e;
    const float scale_ = p.scale;
    const DropKey dkey = drop_key(p.drop_seed, p.drop_p, p.drop_epoch);
    const bool has_drop = p.drop_p > 0.f;
    const uint32_t thr_hi = dkey.thr16 << 16;

    // readout of step sp (its dQ; and dV / dK when it was the last step of its item)
    auto readout = [&](const EwPos& cp) {
      const int sp = cp.s, qt = cp.qt, jt = cp.jt, h = cp.h;
      const int row0 = cp.b * p.N;
      const int qi = qt * BQ + r;
      ptx::mbar_wait_relaxed(&bars[BwdBars::dq_full], sp & 1);
      ptx::tc_fence_after();
      {
        uint32_t rr[16];
        ptx::tmem_ld_x16(tmem_base + (sp & 1) * 128 + lane_off + ch * 16, rr);
        ptx::tmem_ld_wait();
        if (qi < p.N) {
          if (p.dq_mode == 0) {
            float* dst = p.dq_acc + (long long)(row0 + qi) * p.D + h * DH + ch * 16;
#pragma unroll
            for (int e = 0; e < 16; e += 4)
              red_add_v4(dst + e, __uint_as_float(rr[e]), __uint_as_float(rr[e + 1]), __uint_as_float(rr[e + 2]), __uint_as_float(rr[e + 3]));
          } else {
            // one or two key tiles per head, no memset, no atomics: with two tiles the CTA walks them back to back
            // (head-major item order), the first tile's dQ goes to scratch as bf16 and the second tile's read-out — the
            // same thread, two steps later — adds it back and writes the final value
            const bool first_of_two = p.dq_mode == 2 && jt == 0;
            const bool second = p.dq_mode == 2 && jt != 0;
            __nv_bfloat16* part = p.dq_part + (long long)(row0 + qi) * p.D + h * DH + ch * 16;
            __nv_bfloat16* dst = first_of_two ? part : p.dqkv + (long long)(row0 + qi) * (3 * p.D) + h * DH + ch * 16;
            uint4 o2[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              float v[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(rr[q * 8 + e]);
              if (second) {
                const uint4 a = reinterpret_cast<const uint4*>(part)[q];
                v[0] += ptx::bf16_lo(a.x); v[1] += ptx::bf16_hi(a.x); v[2] += ptx::bf16_lo(a.y); v[3] += ptx::bf16_hi(a.y);
                v[4] += ptx::bf16_lo(a.z); v[5] += ptx::bf16_hi(a.z); v[6] += ptx::bf16_lo(a.w); v[7] += ptx::bf16_hi(a.w);
              }
              o2[q].x = ptx::pack_bf16(v[0], v[1]); o2[q].y = ptx::pack_bf16(v[2], v[3]);
              o2[q].z = ptx::pack_bf16(v[4], v[5]); o2[q].w = ptx::pack_bf16(v[6], v[7]);
            }
            // the lane's 16 columns are one 32-byte sector of its row: one 256-bit store (row-per-lane 16-byte stores
            // would touch 32 half-filled sectors per instruction, twice)
            if (p.wide_st) ptx::stg256(dst, o2[0], o2[1]);
            else { reinterpret_cast<uint4*>(dst)[0] = o2[0]; reinterpret_cast<uint4*>(dst)[1] = o2[1]; }
          }
        }
      }
      if (qt == nq - 1) {
        // dV (chunks 0, 1) / dK (chunks 2, 3), 32 columns per warp: TMEM lane == key row of this tile
        const int kvi = jt * bkv + r;
        const bool ok = r < bkv && kvi < p.N;
        const int half = ch & 1;
        const uint32_t t = (ch < 2 ? tmem_dv : tmem_dk) + lane_off + half * 32;
        __nv_bfloat16* dst = p.dqkv + (long long)(row0 + kvi) * (3 * p.D) + (ch < 2 ? 2 * p.D : p.D) + h * DH + half * 32;
        uint32_t rr[32];
        ptx::tmem_ld_x32(t, rr);
        ptx::tmem_ld_wait();
        if (ok) {
          uint4 o4[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            o4[q].x = ptx::pack_bf16(__uint_as_float(rr[q * 8 + 0]), __uint_as_float(rr[q * 8 + 1]));
            o4[q].y = ptx::pack_bf16(__uint_as_float(rr[q * 8 + 2]), __uint_as_float(rr[q * 8 + 3]));
            o4[q].z = ptx::pack_bf16(__uint_as_float(rr[q * 8 + 4]), __uint_as_float(rr[q * 8 + 5]));
            o4[q].w = ptx::pack_bf16(__uint_as_float(rr[q * 8 + 6]), __uint_as_float(rr[q * 8 + 7]));
          }
          if (p.wide_st) {
            ptx::stg256(dst, o4[0], o4[1]);
            ptx::stg256(dst + 16, o4[2], o4[3]);
          } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) reinterpret_cast<uint4*>(dst)[q] = o4[q];
          }
        }
      }
      ptx::tc_fence_before();
      ptx::mbar_arrive(&bars[BwdBars::dq_empty]);
    };

    // row statistics of a step: lse * log2e (+inf for rows past the sequence end, so that P = exp2(-inf) = 0 without a
    // branch) and delta. They are loaded one step ahead: the global-load latency hides behind the previous step.
    auto load_stats = [&](const EwPos& cn, float& l2, float& dl) {
      l2 = INFINITY; dl = 0.f;
      const int qi2 = cn.qt * BQ + r;
      if (cn.s < T && qi2 < p.N) {
        const long long si = ((long long)cn.b * p.H + cn.h) * p.N + qi2;
        // volatile asm: issued HERE (the compiler may not sink it to its use in the next step); the multiply by
        // log2e happens at use, so this step does not stall on the load
        asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(l2) : "l"(p.lse + si));
        asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(dl) : "l"(p.delta + si));
      }
    };
    EwPos cur;
    int dh, db;
    {
      const int head = (int)blockIdx.x, g = (int)gridDim.x;
      cur.s = 0; cur.qt = 0; cur.jt = 0;
      cur.h = head % p.H; cur.b = head / p.H;
      dh = g % p.H; db = g / p.H;
    }
    uint2 prev_packed = make_uint2(0, 0);
    float lse2_next, delta_next;
    load_stats(cur, lse2_next, delta_next);
    for (; cur.s < T; prev_packed = cur.pack(), cur.advance(dh, db, n_kvt, p.H, nq)) {
      {
        const int s = cur.s, qt = cur.qt, h = cur.h, b = cur.b;
        const int kv0 = cur.jt * bkv;
        const int kv_valid = min(bkv, p.N - kv0);
        const int qi = qt * BQ + r;
        const int q_valid = min(BQ, p.N - qt * BQ);
        const bool warp_active = quarter * 32 < ((q_valid + 15) / 16) * 16;   // rows read by the dV / dK MMAs
        const float lse2 = lse2_next * kLog2e, delta = delta_next;
        {
          EwPos nxt = cur;                                   // recomputed here instead of carried through the step
          nxt.advance(dh, db, n_kvt, p.H, nq);
          load_stats(nxt, lse2_next, delta_next);
        }
        // ---- phase A: P = exp2(S * scale * log2e - lse * log2e), kept in registers (+ dropout keep bits)
        float pr[32];
        SFC_TL(long long* dbg = (blockIdx.x == 0 && tid == 64 && s < 64) ? p.dbg : nullptr;)
        SFC_TL(if (dbg) dbg[s * 16 + 0] = clock64();)
        ptx::mbar_wait_relaxed(&bars[BwdBars::s_full + (s & 1)], (s >> 1) & 1);
        SFC_TL(if (dbg) dbg[s * 16 + 1] = clock64();)
        ptx::tc_fence_after();
        const int c = ch;
        const bool chunk_active = warp_active && c * 32 < bkv;   // against the kernel parameter: no live register
        if (chunk_active) {
          uint32_t rs[32];
          ptx::tmem_ld_x32(tmem_base + (s & 1) * 128 + lane_off + c * 32, rs);
          ptx::tmem_ld_wait();
          if (c * 32 + 32 <= kv_valid) {
#pragma unroll
            for (int e = 0; e < 32; ++e) pr[e] = ex2_approx(fmaf(__uint_as_float(rs[e]), sl2, -lse2));
          } else {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              pr[e] = (c * 32 + e < kv_valid) ? ex2_approx(fmaf(__uint_as_float(rs[e]), sl2, -lse2)) : 0.f;
          }
          if (has_drop) {
            // the keep decision travels to phase B in the sign of P (P >= 0): dropped elements are stored negated
            const unsigned long long base = (((unsigned long long)(b * p.H + h) * p.N + (unsigned long long)qi) * (unsigned long long)((p.N + 15) & ~15)) + (unsigned long long)(kv0 + c * 32);
            if ((base & 15ull) == 0) {
#pragma unroll
              for (int g2 = 0; g2 < 2; ++g2) {
                const uint32_t seed = drop_hash2(dkey, (base >> 4) + g2);
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                  const uint32_t x = seed * lcg_mul(e + 1) + lcg_add(e + 1);
                  pr[g2 * 16 + e] = (x >= thr_hi) ? pr[g2 * 16 + e] : -pr[g2 * 16 + e];
                }
              }
            } else {
#pragma unroll
              for (int e = 0; e < 32; ++e) pr[e] = drop_keep<16>(dkey, base + e) ? pr[e] : -pr[e];
            }
          }
        }
        // ---- dQ (and dV / dK) of the previous step leave TMEM; this also guarantees its MMAs no longer read P / dS smem
        SFC_TL(if (dbg) dbg[s * 16 + 2] = clock64();)
        if (s > 0) {
          EwPos prev;
          prev.unpack(prev_packed, s - 1);
          readout(prev);
        }
        SFC_TL(if (dbg) dbg[s * 16 + 3] = clock64();)
        // ---- phase B: dS = P * (dP - delta) * scale; P (dropped) and dS -> shared memory
        ptx::mbar_wait_relaxed(&bars[BwdBars::dp_full], s & 1);
        SFC_TL(if (dbg) dbg[s * 16 + 4] = clock64();)
        ptx::tc_fence_after();
        if (chunk_active) {
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            uint32_t rd[16];
            ptx::tmem_ld_x16(tmem_dp + lane_off + c * 32 + hf * 16, rd);
            ptx::tmem_ld_wait();
            float pv[16], dsv[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) {
              const float ps = pr[hf * 16 + e];
              const float pe = fabsf(ps);
              const float dp = __uint_as_float(rd[e]);
              if (has_drop) {
                const bool k = ps > 0.f;
                pv[e] = k ? pe * dkey.inv_keep : 0.f;
                dsv[e] = pe * scale_ * (k ? fmaf(dp, dkey.inv_keep, -delta) : -delta);
              } else {
                pv[e] = pe;
                dsv[e] = pe * scale_ * (dp - delta);       // pe == 0 outside the valid region
              }
            }
            store_p_half(ptx::smem_u32(smem) + BwdSmem::kP, r, c * 2 + hf, pv);
            store_p_half(ptx::smem_u32(smem) + BwdSmem::kDS, r, c * 2 + hf, dsv);
          }
        }
        SFC_TL(if (dbg) dbg[s * 16 + 5] = clock64();)
        ptx::tc_fence_before();
        ptx::fence_proxy_async_smem();
        SFC_TL(if (dbg) dbg[s * 16 + 6] = clock64();)
        ptx::mbar_arrive(&bars[BwdBars::pds_full]);
        SFC_TL(if (dbg) dbg[s * 16 + 7] = clock64();)
      }
    }
    if (T > 0) {
      EwPos prev;
      prev.unpack(prev_packed, T - 1);
      readout(prev);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

// dqkv[:, 0:D] = bf16(dq_acc)
__global__ void dq_finalize_kernel(const float* __restrict__ dq_acc, __nv_bfloat16* __restrict__ dqkv, long long rows, int D) {
  const long long total = rows * (D / 8);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / (D / 8);
    const int c = (int)(i % (D / 8)) * 8;
    const float4 a = *reinterpret_cast<const float4*>(dq_acc + m * D + c);
    const float4 bq = *reinterpret_cast<const float4*>(dq_acc + m * D + c + 4);
    uint4 o;
    o.x = ptx::pack_bf16(a.x, a.y); o.y = ptx::pack_bf16(a.z, a.w);
    o.z = ptx::pack_bf16(bq.x, bq.y); o.w = ptx::pack_bf16(bq.z, bq.w);
    *reinterpret_cast<uint4*>(dqkv + m * (3ll * D) + c) = o;
  }
}

long long* g_attn_dbg = nullptr;

int check_shape(int B, int H, int N, int D) {
  SFC_REQUIRE(B > 0 && H > 0 && N > 0 && D > 0 && D % H == 0, "attention: bad shape (D=%d, heads=%d)", D, H);
  SFC_REQUIRE((long long)B * N < (1ll << 31), "attention: too many rows");
  return 0;
}

}  // namespace

// attention_generic.cu: CUDA-core path for head dimensions other than 64 (small sequences)
int sfc_attn_generic_supported(int N, int dh, bool bwd);
int sfc_attn_generic_fwd(const void* qkv, void* out, float* lse, int B, int H, int N, int D, float scale, float drop_p,
                         unsigned long long drop_seed, cudaStream_t stream);
int sfc_attn_generic_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, int B, int H, int N,
                         int D, float scale, float drop_p, unsigned long long drop_seed, cudaStream_t stream);

extern "C" int sfc_attn_fwd(const void* qkv, void* out, float* lse, int B, int H, int N, int D, float scale, float drop_p,
                            unsigned long long drop_seed, cudaStream_t stream) {
  if (int e = check_shape(B, H, N, D)) return e;
  SFC_REQUIRE(qkv && out, "sfc_attn_fwd: null pointer");
  SFC_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "sfc_attn_fwd: dropout p out of range");
  if (D / H != DH) {
    SFC_REQUIRE(sfc_attn_generic_supported(N, D / H, false),
                "sfc_attn_fwd: head_dim %d is served by the generic path only for N <= 128 within shared memory (N=%d)", D / H, N);
    return sfc_attn_generic_fwd(qkv, out, lse, B, H, N, D, scale, drop_p, drop_seed, stream);
  }
  const FwdLayout L = fwd_layout(N);
  SFC_REQUIRE(L.total <= 232448, "sfc_attn_fwd: shared-memory plan of %d bytes exceeds 227 KB (N=%d)", L.total, N);
  CUtensorMap tq, tkv;
  if (int e = sfc_make_tmap_2d(&tq, qkv, 2, (uint64_t)3 * D, (uint64_t)B * N, (uint64_t)3 * D * 2, DH, BQ, true)) return e;
  if (int e = sfc_make_tmap_2d(&tkv, qkv, 2, (uint64_t)3 * D, (uint64_t)B * N, (uint64_t)3 * D * 2, DH, (uint32_t)L.bkv, true)) return e;
  CUtensorMap to;      // O [B][N][D]: a 128-row x 64-column box of one image; rows past N are clipped by the TMA unit
  if (int e = sfc_make_tmap_3d(&to, out, (uint64_t)D, (uint64_t)N, (uint64_t)B, (uint64_t)D * 2, (uint64_t)N * D * 2, DH, BQ)) return e;
  AttnParams p{};
  p.B = B; p.H = H; p.N = N; p.D = D; p.scale = scale; p.drop_p = drop_p; p.drop_seed = drop_seed; p.drop_epoch = sfc_dropout_epoch_ptr();
  p.out = (__nv_bfloat16*)out; p.lse = lse; p.dbg = g_attn_dbg;
  static bool configured = false;
  if (!configured) {
    SFC_CUDA_OK(cudaFuncSetAttribute(attn_fwd_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    SFC_CUDA_OK(cudaFuncSetAttribute(attn_fwd_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    SFC_CUDA_OK(cudaFuncSetAttribute(attn_fwd_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    SFC_CUDA_OK(cudaFuncSetAttribute(attn_fwd_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    configured = true;
  }
  const long long items = (long long)B * H * ((N + 2 * BQ - 1) / (2 * BQ));
  const int grid = (int)(items < sfc_num_sms() ? items : sfc_num_sms());
  const bool drop = drop_p > 0.f;
  if (L.nkv == 1 && drop) SFC_CUDA_OK(sfc_launch_pdl(attn_fwd_kernel<true, true>, dim3(grid), dim3(kFwdThreads), (size_t)L.total, stream, tq, tkv, to, p, L));
  else if (L.nkv == 1) SFC_CUDA_OK(sfc_launch_pdl(attn_fwd_kernel<true, false>, dim3(grid), dim3(kFwdThreads), (size_t)L.total, stream, tq, tkv, to, p, L));
  else if (drop) SFC_CUDA_OK(sfc_launch_pdl(attn_fwd_kernel<false, true>, dim3(grid), dim3(kFwdThreads), (size_t)L.total, stream, tq, tkv, to, p, L));
  else SFC_CUDA_OK(sfc_launch_pdl(attn_fwd_kernel<false, false>, dim3(grid), dim3(kFwdThreads), (size_t)L.total, stream, tq, tkv, to, p, L));
  SFC_LAUNCH_OK();
  return 0;
}

extern "C" size_t sfc_attn_bwd_scratch_bytes(int B, int N, int D) {
  return (size_t)B * N * D * sizeof(float) + (size_t)B * ((D + DH - 1) / DH) * N * sizeof(float);
}

// scratch = dQ workspace [B*N, D] (fp32 accumulator for > 2 key tiles, bf16 partial of tile 0 for 2, unused for 1) +
// delta [B, H, N].
extern "C" int sfc_attn_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, void* scratch,
                            size_t scratch_bytes, int B, int H, int N, int D, float scale, float drop_p,
                            unsigned long long drop_seed, cudaStream_t stream) {
  if (int e = check_shape(B, H, N, D)) return e;
  SFC_REQUIRE(qkv && out && dout && lse && dqkv, "sfc_attn_bwd: null pointer");
  SFC_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "sfc_attn_bwd: dropout p out of range");
  if (D / H != DH) {
    SFC_REQUIRE(sfc_attn_generic_supported(N, D / H, true),
                "sfc_attn_bwd: head_dim %d is served by the generic path only for N <= 128 within shared memory (N=%d)", D / H, N);
    return sfc_attn_generic_bwd(qkv, out, dout, lse, dqkv, B, H, N, D, scale, drop_p, drop_seed, stream);
  }
  SFC_REQUIRE(H < 256 && B < (1 << 23) && N <= 65536 * 16, "sfc_attn_bwd: heads < 256, images < 2^23 (H=%d, B=%d)", H, B);
  const size_t dq_bytes = (size_t)B * N * D * sizeof(float);
  const size_t need = sfc_attn_bwd_scratch_bytes(B, N, D);
  SFC_REQUIRE(scratch && scratch_bytes >= need, "sfc_attn_bwd: scratch too small (%zu < %zu)", scratch_bytes, need);
  // key tiles: equal sizes, multiple of 16, at most 128 (the M dimension of the dV / dK MMAs)
  const int n_kvt = (N + 127) / 128;
  const int bkv = ((N + n_kvt - 1) / n_kvt + 15) / 16 * 16;
  const int dq_mode = n_kvt == 1 ? 1 : (n_kvt == 2 ? 2 : 0);
  if (dq_mode == 0) SFC_CUDA_OK(cudaMemsetAsync(scratch, 0, dq_bytes, stream));
  const long long rows = (long long)B * N;
  float* delta = reinterpret_cast<float*>(reinterpret_cast<char*>(scratch) + dq_bytes);
  {
    long long blocks = sfc_ceil_div64(rows * H * 8, 256);
    const long long cap = 32ll * sfc_num_sms();
    if (blocks > cap) blocks = cap;
    SFC_CUDA_OK(sfc_launch_pdl(attn_bwd_prep_kernel, dim3((unsigned)blocks), dim3(256), 0, stream, (const __nv_bfloat16*)out, (const __nv_bfloat16*)dout,
                               delta, rows, N, H));
    SFC_LAUNCH_OK();
  }
  CUtensorMap tq, tkv, tdo;
  if (int e = sfc_make_tmap_2d(&tq, qkv, 2, (uint64_t)3 * D, (uint64_t)B * N, (uint64_t)3 * D * 2, DH, BQ, true)) return e;
  if (int e = sfc_make_tmap_2d(&tkv, qkv, 2, (uint64_t)3 * D, (uint64_t)B * N, (uint64_t)3 * D * 2, DH, (uint32_t)bkv, true)) return e;
  if (int e = sfc_make_tmap_2d(&tdo, dout, 2, (uint64_t)D, (uint64_t)B * N, (uint64_t)D * 2, DH, BQ, true)) return e;
  AttnParams p{};
  p.B = B; p.H = H; p.N = N; p.D = D; p.scale = scale; p.drop_p = drop_p; p.drop_seed = drop_seed; p.drop_epoch = sfc_dropout_epoch_ptr();
  p.lse = const_cast<float*>(lse); p.o = (const __nv_bfloat16*)out; p.dout = (const __nv_bfloat16*)dout;
  p.dqkv = (__nv_bfloat16*)dqkv; p.dq_acc = (float*)scratch; p.dq_part = (__nv_bfloat16*)scratch; p.dq_mode = dq_mode;
  p.wide_st = (((reinterpret_cast<uintptr_t>(dqkv) | reinterpret_cast<uintptr_t>(scratch)) & 31) == 0) ? 1 : 0;
  p.delta = delta; p.dbg = g_attn_dbg;
  static bool configured = false;
  if (!configured) {
    SFC_CUDA_OK(cudaFuncSetAttribute(attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BwdSmem::kTotal));
    configured = true;
  }
  const long long items = (long long)B * H;                  // the CTAs stride over heads (all key tiles of a head on one CTA)
  const int grid = (int)(items < sfc_num_sms() ? items : sfc_num_sms());
  SFC_CUDA_OK(sfc_launch_pdl(attn_bwd_kernel, dim3(grid), dim3(kBwdThreads), (size_t)BwdSmem::kTotal, stream, tq, tkv, tdo, p, bkv));
  SFC_LAUNCH_OK();
  if (dq_mode == 0) {
    long long blocks = sfc_ceil_div64(rows * (D / 8), 256);
    const long long cap = 16ll * sfc_num_sms();
    if (blocks > cap) blocks = cap;
    dq_finalize_kernel<<<(unsigned)blocks, 256, 0, stream>>>((const float*)scratch, (__nv_bfloat16*)dqkv, rows, D);
  }
  SFC_LAUNCH_OK();
  return 0;
}

// Debug: per-step clock64() timeline of CTA 0 of the next sfc_attn_bwd launches (>= 64 * 16 int64; NULL = off).
extern "C" void sfc_debug_set_timeline(void* dev_ptr) { g_attn_dbg = (long long*)dev_ptr; }
