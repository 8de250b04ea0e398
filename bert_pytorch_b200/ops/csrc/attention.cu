// Fused multi-head attention for BERT (non-causal, key-padding mask given as per-sequence valid length,
// head_dim 64, S <= 512 in blocks of 128) on tcgen05 tensor cores -- forward and backward.
// Replaces the reference's QK^T / scale / mask / softmax / dropout / PV chain that materialises three
// [B,h,S,S] tensors per layer (src/modeling.py:404-428; SURVEY.md K6-K12).
//
// Data layout: qkv is the QKV-GEMM output [B*S, 3H] (token-major, q|k|v, head-major inside), so Q/K/V
// tiles of one head are plain 2-D TMA boxes of that matrix -- no permute/contiguous copies (K6 is gone);
// the context is written as [B*S, H], ready for the output projection.
//
// In every kernel elected lanes of control warps issue the TMA loads and the tcgen05.mma, and the math warps work on
// rows of tensor memory (TMEM lane == query row).  Dropout draws Philox counter bits for the probabilities
// (element ((b * h + head) * S + q) * S + k); the backward regenerates the same bits instead of storing a mask.
//
// Forward: one thread per query row, P is written back into the S accumulator and feeds the P V MMA from TMEM
//   attn_fwd_row_kernel     S <= 128: persistent CTAs over (batch, head); S, P and the P V result share 128 TMEM
//                           columns, 48 KB -> four CTAs per SM
//   attn_fwd_stream_kernel  S > 128: persistent CTAs over (batch, head, 128-query block); K / V two-stage ring, the
//                           output accumulates in TMEM under a lazily raised running max; 256 columns -> two CTAs per SM
// Backward: S = Q K^T, dP = dO V^T -> threads form P~ (dropped probabilities / keep_prob) and dS -> dV = P~^T dO,
// dK = dS^T Q, dQ = dS K (the transposes are free: MN-major descriptors on the same tile)
//   attn_bwd_row2_kernel    S <= 128: persistent CTAs over (batch, head), two threads per query row, delta = <dO, O>
//                           in-kernel; dV / dK / dQ overwrite the consumed S / dP accumulators; 96 KB -> two CTAs per SM
//   attn_bwd_pipe_kernel    S > 128: one CTA per (batch, head, 128-key block) looping over the query blocks, software
//                           pipelined; dV, dK accumulate in TMEM, dQ goes out through fp32 atomics.  attn_delta_kernel
//                           (delta = <dO, O>) runs before it, attn_dq_convert_kernel (fp32 dQ -> bf16) after it
#include "common.cuh"
#include "gemm_sm100.h"
#include "kernels.h"

namespace b200 {

constexpr int ATT_BWD_THREADS = 288;   // 8 math warps (2 per TMEM lane quarter) + 1 control warp
constexpr int ATT_BWD16_THREADS = 544; // streaming backward: 16 math warps (4 per TMEM lane quarter) + 1 control warp
constexpr int TILE = 128;          // query rows / key rows per block
constexpr int HD = 64;             // head dim
constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct AttnArgs {
  int B, S, h, H;
  const int* seqlens;
  __nv_bfloat16* ctx;      // fwd out [B*S, H]
  float* lse;              // [B, h, S] natural-log LSE of the scaled scores
  float scale;
  Seed seed;
  unsigned int stream;
  unsigned int thresh16;
  float inv_keep;
  // backward
  const float* delta;      // [B, h, S]
  __nv_bfloat16* dqkv;     // [B*S, 3H]
  float* dq_acc;           // [B*S, H] fp32 (only when more than one key block)
  Fp8Out f8;               // optional fp8 copy of the output (ctx in the forward, dqkv in the backward)
};

// address of the 16-byte chunk holding columns [col8*8, col8*8+8) of row r inside a [128 x 128] bf16 tile
// stored as two [128 x 64] 128B-swizzled sub-tiles (the layout TMA/UMMA call SWIZZLE_128B)
__device__ __forceinline__ uint32_t p_chunk_offset(int r, int col8) {
  const int sub = col8 >> 3, ck = col8 & 7;
  return (uint32_t)(sub * 16384 + r * 128 + ((ck ^ (r & 7)) << 4));
}

// fp8 copy of NG*8 consecutive output elements held as raw fp32 bits in v[] (scaled by `mul`)
template <int NG>
__device__ __forceinline__ void emit_fp8_row(const Fp8Out& f8, size_t off, const uint32_t* v, float mul, float qscale,
                                             float& amax) {
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    float t8[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) t8[t] = __uint_as_float(v[g * 8 + t]) * mul;
    fp8_emit8(f8, off + g * 8, t8, qscale, amax);
  }
}

// ------------------------------------------------------------------------------------------------
// forward: one THREAD per query row, P stays in tensor memory, persistent CTAs.
//
// The softmax, not the MMA, is the cost of the forward: a two-threads-per-row layout measured 23-25 instructions per
// score element at ~55 % issue utilisation and 8-10 % tensor-pipe activity (profiles/ncu_hot_kernels_r1.md), half of
// it overhead of that mapping (two TMEM passes of 16-column loads, shared-memory exchanges and block barriers for the
// row statistics, swizzled shared-memory stores of P, Philox key schedule and 16-bit field extraction per element).
// Here
//   * thread r of the four softmax warps owns TMEM lane r = query row r: row max / row sum never leave the thread
//     (no exchange, no barrier), 3-input max, 32-column TMEM loads with the next chunk in flight;
//   * P (bf16) is written back into the first 64 columns of the S accumulator with tcgen05.st and feeds the PV MMA
//     as a TMEM A operand -- no shared-memory round trip, no proxy fence, and the Q / K tiles are free for the next
//     loads as soon as the S MMA has retired;
//   * the PV result lands in columns [64, 128) of the same accumulator: 128 TMEM columns and 48 KB per CTA ->
//     four (S <= 128) or three (streaming, 64 accumulator registers) co-resident CTAs per SM hide each other's
//     dependent MMA -> softmax -> MMA chains;
//   * CTAs are persistent over (batch, head, query block) items: TMEM allocation / barrier set-up once, the next
//     item's Q and K tiles stream in under the current softmax;
//   * dropout: 1 / keep_prob is folded into the exponent, the Philox round keys are precomputed, the 16-bit keep
//     fields are compared in place (one ISETP per element, same bits as dropout_keep8 so the backward kernels agree).
// ------------------------------------------------------------------------------------------------
constexpr int ATT_ROW_THREADS = 160;   // warps 0-3: softmax rows (TMEM lane quarter == warp), warp 4: control

__device__ __forceinline__ float max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// probabilities of one 32-key chunk of this thread's row: p' = 2^(s c - m + log2(1/keep)) (the dropout rescale rides
// in the exponent), rowsum over the valid keys BEFORE dropout, dropped entries zeroed, packed bf16 -> 16 words.
// NV: number of valid keys in the chunk (32 on the fast path; compile-time `FULL`)
template <bool FULL, bool DROP>
__device__ __forceinline__ void softmax_chunk(const uint32_t (&sv)[32], uint32_t (&pw)[16], float c_scale, float off,
                                              float& rowsum, int nvalid, const PhiloxKeys& keys, uint64_t e8,
                                              uint32_t stream, uint32_t T) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float pr[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      float e = ex2_approx(fmaf(__uint_as_float(sv[g * 8 + t]), c_scale, off));
      if (!FULL && g * 8 + t >= nvalid) e = 0.f;
      rowsum += e;
      pr[t] = e;
    }
    if (DROP) {
      const uint4 r = philox7(keys, e8 + (uint64_t)g, stream);
#pragma unroll
      for (int t = 0; t < 8; ++t) pr[t] = keep_bit(r, t, T) ? pr[t] : 0.f;
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) pw[g * 4 + t] = pack_bf16(pr[2 * t], pr[2 * t + 1]);
  }
}

// one 32-column chunk of the row maximum
__device__ __forceinline__ float chunk_max(const uint32_t (&v)[32], float mx, int nv) {
  if (nv >= 32) {
#pragma unroll
    for (int t = 0; t < 32; t += 2) mx = max3(mx, __uint_as_float(v[t]), __uint_as_float(v[t + 1]));
  } else if (nv > 0) {
#pragma unroll
    for (int t = 0; t < 32; ++t)
      if (t < nv) mx = fmaxf(mx, __uint_as_float(v[t]));
  }
  return mx;
}
// row maximum over the 128 score columns of this thread's TMEM lane (the next chunk is in flight while one is reduced)
__device__ __forceinline__ float row_max_128(uint32_t taddr, int kvalid) {
  float mx = -INFINITY;
  uint32_t a[32], b[32];
  tmem_ld_32x32(taddr, a);
  tmem_ld_wait();
  tmem_ld_32x32(taddr + 32, b);
  mx = chunk_max(a, mx, kvalid);
  tmem_ld_wait();
  tmem_ld_32x32(taddr + 64, a);
  mx = chunk_max(b, mx, kvalid - 32);
  tmem_ld_wait();
  tmem_ld_32x32(taddr + 96, b);
  mx = chunk_max(a, mx, kvalid - 64);
  tmem_ld_wait();
  mx = chunk_max(b, mx, kvalid - 96);
  return mx;
}
// probabilities of the 128 score columns -> dropout -> bf16 -> tcgen05.st into columns [0, 64) of the same lane.
// Words [16 c, 16 c + 16) of the P row overwrite S columns this thread has already consumed (chunk c + 1 starts at
// column 32 (c + 1) >= 16 (c + 1)).  Returns the row sum of the (1 / keep_prob scaled) probabilities before dropout.
__device__ __forceinline__ float row_softmax_128(uint32_t taddr, int kvalid, float c_scale, float off, bool drop,
                                                 const PhiloxKeys& keys, uint64_t e8, uint32_t stream, uint32_t T) {
  float rowsum = 0.f;
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    uint32_t v[32], pw[16];
    tmem_ld_32x32(taddr + c * 32, v);
    tmem_ld_wait();
    const int nv = kvalid - c * 32;
    if (nv >= 32) {
      if (drop) softmax_chunk<true, true>(v, pw, c_scale, off, rowsum, 32, keys, e8 + 4 * c, stream, T);
      else softmax_chunk<true, false>(v, pw, c_scale, off, rowsum, 32, keys, e8 + 4 * c, stream, T);
    } else if (nv > 0) {
      if (drop) softmax_chunk<false, true>(v, pw, c_scale, off, rowsum, nv, keys, e8 + 4 * c, stream, T);
      else softmax_chunk<false, false>(v, pw, c_scale, off, rowsum, nv, keys, e8 + 4 * c, stream, T);
    } else {
#pragma unroll
      for (int t = 0; t < 16; ++t) pw[t] = 0u;
    }
    tmem_st_32x16(taddr + c * 16, pw);
  }
  return rowsum;
}

// ---- S <= 128: one key block per item; S, P and the P V result share 128 TMEM columns -> four CTAs per SM
__global__ void __launch_bounds__(ATT_ROW_THREADS, 4)
attn_fwd_row_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const AttnArgs p, const int n_items) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                      // 16 KB each, 128B swizzle
  uint8_t* sK = smem + 16384;
  uint8_t* sV = smem + 32768;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 49152);
  uint64_t* qk_full = bars;                // Q and K tiles of an item landed
  uint64_t* v_full = bars + 1;             // V tile landed
  uint64_t* s_ready = bars + 2;            // S = Q K^T complete (Q and K are free)
  uint64_t* p_ready = bars + 3;            // 128 threads: P is in tensor memory
  uint64_t* o_ready = bars + 4;            // P V complete (V is free)
  uint64_t* o_read = bars + 5;             // 128 threads: the P V result has been read out -> S may be overwritten
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 128) {
    tma_prefetch_desc(&tmap_qkv);
    mbar_init(qk_full, 1);
    mbar_init(v_full, 1);
    mbar_init(s_ready, 1);
    mbar_init(p_ready, 128);
    mbar_init(o_ready, 1);
    mbar_init(o_read, 128);
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc(tmem_slot, 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tS = *tmem_slot, tO = tS + 64;
  pdl_trigger_small();
  pdl_wait();                              // PDL: the set-up above overlapped the previous kernel's tail

  if (warp == 4) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(128, 128, false, false);  // Q K^T : both K-major
      constexpr uint32_t idesc_o = umma_idesc_bf16(128, 64, false, true);    // P V   : P from TMEM, V MN-major
      const uint64_t dq = umma_smem_desc_sw128(smem_u32(sQ), 16, 1024);
      const uint64_t dk = umma_smem_desc_sw128(smem_u32(sK), 16, 1024);
      const uint32_t av = smem_u32(sV);
      auto load_qk = [&](int item) {
        const int b = item / p.h, head = item - b * p.h;
        mbar_arrive_expect_tx(qk_full, 32768);
        tma_load_2d(sQ, &tmap_qkv, qk_full, head * HD, b * p.S);
        tma_load_2d(sK, &tmap_qkv, qk_full, p.H + head * HD, b * p.S);
      };
      auto load_v = [&](int item) {
        const int b = item / p.h, head = item - b * p.h;
        mbar_arrive_expect_tx(v_full, 16384);
        tma_load_2d(sV, &tmap_qkv, v_full, 2 * p.H + head * HD, b * p.S);
      };
      int item = blockIdx.x;
      if (item < n_items) { load_qk(item); load_v(item); }
      for (uint32_t g = 0; item < n_items; item += gridDim.x, ++g) {
        const int nitem = item + gridDim.x;
        if (g > 0) mbar_wait(o_read, (g - 1) & 1);            // previous P V result drained out of [64, 128)
        mbar_wait(qk_full, g & 1);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < HD / 16; ++kk) umma_bf16_ss(tS, dq + 2 * kk, dk + 2 * kk, idesc_s, kk > 0);
        umma_commit(s_ready);
        mbar_wait(s_ready, g & 1);                            // Q and K may be refilled: next item streams in under the softmax
        if (nitem < n_items) load_qk(nitem);
        mbar_wait(p_ready, g & 1);
        mbar_wait(v_full, g & 1);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < TILE / 16; ++kk)
          umma_bf16_ts(tO, tS + kk * 8, umma_smem_desc_sw128(av + kk * 2048, 8192, 1024), idesc_o, kk > 0);
        umma_commit(o_ready);
        mbar_wait(o_ready, g & 1);                            // V may be refilled
        if (nitem < n_items) load_v(nitem);
      }
    }
  } else {
    const int r = warp * 32 + lane;                            // query row == TMEM lane
    const uint32_t lane_base = uint32_t(warp * 32) << 16;
    const float c_scale = p.scale * LOG2E;
    const bool drop = p.thresh16 != 0;
    const float lk = drop ? log2f(p.inv_keep) : 0.f;           // 1 / keep_prob rides in the exponent
    const uint32_t T = p.thresh16 << 16;
    const PhiloxKeys keys = philox_keys(drop ? p.seed.value() : 0ull);
    const bool q_ok = r < p.S;
    uint32_t g = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++g) {
      const int b = item / p.h, head = item - b * p.h;
      const int seqlen = min(__ldg(p.seqlens + b), p.S);
      const uint64_t e8row = (((uint64_t)item * p.S + (uint64_t)r) * (uint64_t)p.S) >> 3;   // dropout group base of the row
      mbar_wait(s_ready, g & 1);
      tc_fence_after();
      const float m = fmaxf(row_max_128(tS + lane_base, seqlen) * c_scale, -1e30f);   // an all-padding row stays finite
      const float l = row_softmax_128(tS + lane_base, seqlen, c_scale, lk - m, drop, keys, e8row, p.stream, T);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(p_ready);
      const float inv_l = (drop ? p.inv_keep : 1.f) / l;       // l and the P V result both carry 1 / keep_prob
      __nv_bfloat16* dst = p.ctx + (size_t)(b * p.S + r) * p.H + head * HD;
      float amax = 0.f;
      const float qscale = p.f8.q ? p.f8.meta[1] : 0.f;
      mbar_wait(o_ready, g & 1);
      tc_fence_after();
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        uint32_t o[32];
        tmem_ld_32x32(tO + lane_base + hh * 32, o);
        tmem_ld_wait();
        if (hh == 1) {                                         // accumulator drained: the next S MMA may go
          tc_fence_before();
          mbar_arrive(o_read);
        }
        if (q_ok) {
#pragma unroll
          for (int gq = 0; gq < 4; ++gq)
            *reinterpret_cast<uint4*>(dst + hh * 32 + gq * 8) = make_uint4(
                pack_bf16(__uint_as_float(o[gq * 8]) * inv_l, __uint_as_float(o[gq * 8 + 1]) * inv_l),
                pack_bf16(__uint_as_float(o[gq * 8 + 2]) * inv_l, __uint_as_float(o[gq * 8 + 3]) * inv_l),
                pack_bf16(__uint_as_float(o[gq * 8 + 4]) * inv_l, __uint_as_float(o[gq * 8 + 5]) * inv_l),
                pack_bf16(__uint_as_float(o[gq * 8 + 6]) * inv_l, __uint_as_float(o[gq * 8 + 7]) * inv_l));
          if (p.f8.q) emit_fp8_row<4>(p.f8, (size_t)(b * p.S + r) * p.H + head * HD + hh * 32, o, inv_l, qscale, amax);
        }
      }
      if (p.f8.q && amax > 0.f) atomicMax(reinterpret_cast<int*>(p.f8.meta), __float_as_int(isfinite(amax) ? amax : 3.0e38f));
      if (q_ok) p.lse[(size_t)item * p.S + r] = (m + log2f(l) - lk) * 0.6931471805599453f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tS, 128);
  }
}

// ---- S > 128: streaming kernel.  Per CTA: 4 softmax warps (thread == query row), one MMA warp, one TMA warp.
// TMEM: S | P in columns [0, 128), the output accumulator in [128, 192): the P V MMAs accumulate in tensor memory
// and S_{j+1} = Q K_{j+1}^T is issued right behind P_j V_j (tcgen05 executes in issue order), so the scores of the
// next key block are waiting when a softmax finishes -- the threads never wait for a P V.  The running maximum is
// only raised when a block exceeds it by more than 2^8 (probabilities stay below 256, exact in the fp32 row sum /
// accumulator); raising it rescales this thread's accumulator row in TMEM (tcgen05.ld -> mul -> tcgen05.st), which
// after the first key block is rare.  K / V ride a two-stage ring.  256 TMEM columns, 80 KB -> two CTAs per SM.
constexpr int ATT_STREAM_THREADS = 192;
__global__ void __launch_bounds__(ATT_STREAM_THREADS, 2)
attn_fwd_stream_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const AttnArgs p, const int n_items, const int nqb) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                      // 16 KB
  uint8_t* sK = smem + 16384;              // 2 x 16 KB
  uint8_t* sV = smem + 16384 * 3;          // 2 x 16 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 16384 * 5);
  uint64_t* q_full = bars;                 // once per item
  uint64_t* q_empty = bars + 1;            // last S MMA of an item retired
  uint64_t* k_full = bars + 2;             // [2]
  uint64_t* k_empty = bars + 4;            // [2]
  uint64_t* v_full = bars + 6;             // [2]
  uint64_t* v_empty = bars + 8;            // [2]
  uint64_t* s_ready = bars + 10;           // per key block
  uint64_t* p_ready = bars + 11;           // 128 threads, per key block
  uint64_t* o_ready = bars + 12;           // per item: last P V retired
  uint64_t* o_read = bars + 13;            // 128 threads, per item: accumulator read out
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 128) {
    tma_prefetch_desc(&tmap_qkv);
    mbar_init(q_full, 1);
    mbar_init(q_empty, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1); mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1); mbar_init(&v_empty[i], 1);
    }
    mbar_init(s_ready, 1);
    mbar_init(p_ready, 128);
    mbar_init(o_ready, 1);
    mbar_init(o_read, 128);
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc(tmem_slot, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tS = *tmem_slot, tO = tS + 128;

  auto coords = [&](int item, int& row0, int& qb, int& head, int& bh, int& seqlen, int& nkb) {
    bh = item / nqb;
    qb = item - bh * nqb;
    const int b = bh / p.h;
    head = bh - b * p.h;
    row0 = b * p.S;
    seqlen = min(__ldg(p.seqlens + b), p.S);
    nkb = max(1, (seqlen + TILE - 1) / TILE);
  };

  if (warp == 5) {
    if (lane == 0) {                       // ---------------- TMA producer
      uint32_t g = 0, n = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++n) {
        int row0, qb, head, bh, seqlen, nkb;
        coords(item, row0, qb, head, bh, seqlen, nkb);
        if (n > 0) mbar_wait(q_empty, (n - 1) & 1);
        mbar_arrive_expect_tx(q_full, 16384);
        tma_load_2d(sQ, &tmap_qkv, q_full, head * HD, row0 + qb * TILE);
        for (int j = 0; j < nkb; ++j, ++g) {
          const int st = g & 1;
          if (g >= 2) mbar_wait(&k_empty[st], ((g >> 1) - 1) & 1);
          mbar_arrive_expect_tx(&k_full[st], 16384);
          tma_load_2d(sK + st * 16384, &tmap_qkv, &k_full[st], p.H + head * HD, row0 + j * TILE);
          if (g >= 2) mbar_wait(&v_empty[st], ((g >> 1) - 1) & 1);
          mbar_arrive_expect_tx(&v_full[st], 16384);
          tma_load_2d(sV + st * 16384, &tmap_qkv, &v_full[st], 2 * p.H + head * HD, row0 + j * TILE);
        }
      }
    }
  } else if (warp == 4) {
    if (lane == 0) {                       // ---------------- MMA issuer
      constexpr uint32_t idesc_s = umma_idesc_bf16(128, 128, false, false);
      constexpr uint32_t idesc_o = umma_idesc_bf16(128, 64, false, true);
      const uint64_t dq = umma_smem_desc_sw128(smem_u32(sQ), 16, 1024);
      uint32_t g = 0, n = 0;
      auto issue_s = [&](uint32_t gg) {
        const int st = gg & 1;
        mbar_wait(&k_full[st], (gg >> 1) & 1);
        tc_fence_after();
        const uint64_t dk = umma_smem_desc_sw128(smem_u32(sK + st * 16384), 16, 1024);
#pragma unroll
        for (int kk = 0; kk < HD / 16; ++kk) umma_bf16_ss(tS, dq + 2 * kk, dk + 2 * kk, idesc_s, kk > 0);
        umma_commit(s_ready);
        umma_commit(&k_empty[st]);
      };
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++n) {
        int row0, qb, head, bh, seqlen, nkb;
        coords(item, row0, qb, head, bh, seqlen, nkb);
        mbar_wait(q_full, n & 1);
        issue_s(g);                                            // S_0 (the previous item's last P V is ahead of it in the pipe)
        for (int j = 0; j < nkb; ++j, ++g) {
          const int st = g & 1;
          if (j == 0 && n > 0) mbar_wait(o_read, (n - 1) & 1); // previous item's accumulator has been read out
          mbar_wait(p_ready, g & 1);
          mbar_wait(&v_full[st], (g >> 1) & 1);
          tc_fence_after();
          const uint32_t av = smem_u32(sV + st * 16384);
#pragma unroll
          for (int kk = 0; kk < TILE / 16; ++kk)
            umma_bf16_ts(tO, tS + kk * 8, umma_smem_desc_sw128(av + kk * 2048, 8192, 1024), idesc_o, (j > 0 || kk > 0));
          umma_commit(&v_empty[st]);
          if (j + 1 < nkb) {
            issue_s(g + 1);                                    // right behind the P V: overwrites S | P in issue order
          } else {
            umma_commit(o_ready);
            umma_commit(q_empty);
          }
        }
      }
    }
  } else {
    const int r = warp * 32 + lane;
    const uint32_t lane_base = uint32_t(warp * 32) << 16;
    const float c_scale = p.scale * LOG2E;
    const bool drop = p.thresh16 != 0;
    const float lk = drop ? log2f(p.inv_keep) : 0.f;
    const uint32_t T = p.thresh16 << 16;
    const PhiloxKeys keys = philox_keys(drop ? p.seed.value() : 0ull);
    uint32_t g = 0, n = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++n) {
      int row0, qb, head, bh, seqlen, nkb;
      coords(item, row0, qb, head, bh, seqlen, nkb);
      const int q = qb * TILE + r;
      const uint64_t e8row = (((uint64_t)bh * p.S + (uint64_t)q) * (uint64_t)p.S) >> 3;
      float m = -INFINITY, l = 0.f;
      for (int j = 0; j < nkb; ++j, ++g) {
        const int kvalid = seqlen - j * TILE;
        mbar_wait(s_ready, g & 1);
        tc_fence_after();
        const float mb = fmaxf(row_max_128(tS + lane_base, kvalid) * c_scale, -1e30f);
        // lazy running maximum: keep the old reference while this block stays within 2^8 of it
        const bool raise = mb > m + 8.f;
        if (j > 0 && __any_sync(0xffffffffu, raise)) {         // rescale this thread's accumulator row (warp-uniform branch)
          const float f = raise ? ex2_approx(m - mb) : 1.f;
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            uint32_t o[32];
            tmem_ld_32x32(tO + lane_base + hh * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int t = 0; t < 32; ++t) o[t] = __float_as_uint(__uint_as_float(o[t]) * f);
            tmem_st_32x32(tO + lane_base + hh * 32, o);
          }
          l *= f;
        }
        if (raise) m = mb;
        l += row_softmax_128(tS + lane_base, kvalid, c_scale, lk - m, drop, keys, e8row + (uint64_t)(j * (TILE / 8)),
                             p.stream, T);
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(p_ready);
      }
      // ---- epilogue: accumulator / row sum -> context
      mbar_wait(o_ready, n & 1);
      tc_fence_after();
      const float inv_l = (drop ? p.inv_keep : 1.f) / l;       // l and the accumulator both carry 1 / keep_prob
      const bool q_ok = q < p.S;
      __nv_bfloat16* dst = p.ctx + (size_t)(row0 + q) * p.H + head * HD;
      float amax = 0.f;
      const float qscale = p.f8.q ? p.f8.meta[1] : 0.f;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        uint32_t o[32];
        tmem_ld_32x32(tO + lane_base + hh * 32, o);
        tmem_ld_wait();
        if (hh == 1) {
          tc_fence_before();
          mbar_arrive(o_read);
        }
        if (q_ok) {
#pragma unroll
          for (int gq = 0; gq < 4; ++gq)
            *reinterpret_cast<uint4*>(dst + hh * 32 + gq * 8) = make_uint4(
                pack_bf16(__uint_as_float(o[gq * 8]) * inv_l, __uint_as_float(o[gq * 8 + 1]) * inv_l),
                pack_bf16(__uint_as_float(o[gq * 8 + 2]) * inv_l, __uint_as_float(o[gq * 8 + 3]) * inv_l),
                pack_bf16(__uint_as_float(o[gq * 8 + 4]) * inv_l, __uint_as_float(o[gq * 8 + 5]) * inv_l),
                pack_bf16(__uint_as_float(o[gq * 8 + 6]) * inv_l, __uint_as_float(o[gq * 8 + 7]) * inv_l));
          if (p.f8.q) emit_fp8_row<4>(p.f8, (size_t)(row0 + q) * p.H + head * HD + hh * 32, o, inv_l, qscale, amax);
        }
      }
      if (p.f8.q && amax > 0.f) atomicMax(reinterpret_cast<int*>(p.f8.meta), __float_as_int(isfinite(amax) ? amax : 3.0e38f));
      if (q_ok) p.lse[(size_t)bh * p.S + q] = (m + log2f(l) - lk) * 0.6931471805599453f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tS, 256);
  }
}

// ------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
attn_delta_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ dout, float* __restrict__ delta,
                  int B, int S, int h, int H) {
  // one 8-lane group per (token, head): 64 elements = 8 x 16 B
  const long long gid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const int sub = threadIdx.x & 7;
  const long long total = (long long)B * S * h;
  if (gid >= total) return;
  const int head = (int)(gid % h);
  const long long tok = gid / h;
  const size_t off = (size_t)tok * H + head * HD + sub * 8;
  const uint4 a = *reinterpret_cast<const uint4*>(o + off), d = *reinterpret_cast<const uint4*>(dout + off);
  const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, dw[4] = {d.x, d.y, d.z, d.w};
  float s = 0.f;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const float2 x = unpack_bf16(aw[t]), y = unpack_bf16(dw[t]);
    s += x.x * y.x + x.y * y.y;
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  if (sub == 0) {
    const int bb = (int)(tok / S), ss = (int)(tok % S);
    delta[((size_t)bb * h + head) * S + ss] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// backward, S > 128: one CTA per (batch, head, 128-key block), looping over the query blocks.  16 math warps: four
// threads per query row (TMEM lane quarter = warp & 3, 32-key column quarter = warp >> 2) -- at one CTA per SM the
// latency of the per-thread softmax-gradient chain bounds the kernel, and more threads per row shorten it; 16-column
// TMEM loads keep it under the 120 registers 544 threads allow.  TMEM (512 columns): S | dP | dV | dK | dQ.  Per query
// block the math warps write P~ and dS to shared memory (32 KB each, in the 128B-swizzled layout the MMAs read); dV +=
// P~^T dO and dK += dS^T Q accumulate in TMEM over all query blocks, dQ = dS K of the block is added to the fp32 dQ
// accumulator with vector atomics.  A key block that is all padding writes zero dK / dV and exits.  Pipelining:
//   * the math warps release S/dP as soon as they have pulled them out of TMEM (`sdp_free`), so the S/dP MMAs of
//     block i+1 run while block i's math is still in registers;
//   * block i's dQ is read back one iteration later (after block i+1's S/dP were loaded), so the dV/dK/dQ MMAs of
//     block i overlap the math of block i+1;
//   * Q/dO live in a 3-stage ring (blocks i, i+1 in use, i+2 landing); the reload of a stage is issued one iteration
//     after its last reader, when the wait is free.
// One P~ and one dS buffer serve every block: dq_ready(i-1) orders the stores of block i after the MMAs that read
// block i-1's, and ds_ready(i) orders the dQ MMA of block i after those stores.  192 KB shared memory, one CTA per SM.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(ATT_BWD16_THREADS, 1)
attn_bwd_pipe_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_do,
                     const AttnArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;                      // 16 KB
  uint8_t* sV = smem + 16384;              // 16 KB
  uint8_t* sQ = smem + 16384 * 2;          // 3 x 16 KB
  uint8_t* sDO = smem + 16384 * 5;         // 3 x 16 KB
  uint8_t* sPd = smem + 16384 * 8;         // 32 KB
  uint8_t* sDS = smem + 16384 * 10;        // 32 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 16384 * 12);
  uint64_t* kv_full = bars;
  uint64_t* qdo_full = bars + 1;           // 3
  uint64_t* qdo_empty = bars + 4;          // 3
  uint64_t* sdp_ready = bars + 7;
  uint64_t* sdp_free = bars + 8;
  uint64_t* ds_ready = bars + 9;
  uint64_t* dq_ready = bars + 10;
  uint64_t* fin = bars + 11;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kb = blockIdx.x, bh = blockIdx.y;
  const int b = bh / p.h, head = bh % p.h;
  const int seqlen = min(p.seqlens[b], p.S);
  const int nqb = (p.S + TILE - 1) / TILE;
  const int row0 = b * p.S;
  const bool dead = kb * TILE >= seqlen;     // every key of this block is padding: dK = dV = 0

  if (dead) {
    if (warp < 4) {
      const int key = kb * TILE + warp * 32 + lane;
      if (key < p.S) {
        __nv_bfloat16* dk = p.dqkv + (size_t)(row0 + key) * 3 * p.H + p.H + head * HD;
        __nv_bfloat16* dv = dk + p.H;
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          *reinterpret_cast<uint4*>(dk + g * 8) = make_uint4(0, 0, 0, 0);
          *reinterpret_cast<uint4*>(dv + g * 8) = make_uint4(0, 0, 0, 0);
        }
        if (p.f8.q) {
          unsigned char* qk = p.f8.q + (size_t)(row0 + key) * 3 * p.H + p.H + head * HD;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            *reinterpret_cast<uint4*>(qk + g * 16) = make_uint4(0, 0, 0, 0);
            *reinterpret_cast<uint4*>(qk + p.H + g * 16) = make_uint4(0, 0, 0, 0);
          }
        }
      }
    }
    return;
  }

  if (threadIdx.x == 512) {
    tma_prefetch_desc(&tmap_qkv);
    tma_prefetch_desc(&tmap_do);
    mbar_init(kv_full, 1);
    for (int i = 0; i < 3; ++i) { mbar_init(&qdo_full[i], 1); mbar_init(&qdo_empty[i], 1); }
    mbar_init(sdp_ready, 1);
    mbar_init(sdp_free, 512);
    mbar_init(ds_ready, 512);
    mbar_init(dq_ready, 1);
    mbar_init(fin, 1);
    fence_barrier_init();
  }
  if (warp == 16) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const unsigned long long seed = p.thresh16 != 0 ? p.seed.value() : 0ull;
  const uint32_t tS = tmem, tDP = tmem + 128, tDV = tmem + 256, tDK = tmem + 320, tDQ = tmem + 384;

  if (warp == 16) {
    if (lane == 0) {
      const int cq = head * HD, ck = p.H + head * HD, cv = 2 * p.H + head * HD;
      mbar_arrive_expect_tx(kv_full, 32768);
      tma_load_2d(sK, &tmap_qkv, kv_full, ck, row0 + kb * TILE);
      tma_load_2d(sV, &tmap_qkv, kv_full, cv, row0 + kb * TILE);
      for (int i = 0; i < min(3, nqb); ++i) {
        mbar_arrive_expect_tx(&qdo_full[i], 32768);
        tma_load_2d(sQ + i * 16384, &tmap_qkv, &qdo_full[i], cq, row0 + i * TILE);
        tma_load_2d(sDO + i * 16384, &tmap_do, &qdo_full[i], head * HD, row0 + i * TILE);
      }
      constexpr uint32_t id_kk = umma_idesc_bf16(128, 128, false, false);  // [q x keys], both K-major
      constexpr uint32_t id_tt = umma_idesc_bf16(128, 64, true, true);     // [keys x d] = X^T Y, both MN-major
      constexpr uint32_t id_kt = umma_idesc_bf16(128, 64, false, true);    // [q x d] = dS K, A K-major, B MN-major
      const uint32_t ak = smem_u32(sK), av = smem_u32(sV), apd = smem_u32(sPd), ads = smem_u32(sDS);
      // S = Q K^T and dPd = dO V^T of query block j (its Q / dO tiles sit in ring slot j % 3)
      auto issue_sdp = [&](int j) {
        const int sj = j % 3;
        mbar_wait(&qdo_full[sj], (j / 3) & 1);
        tc_fence_after();
        const uint32_t aq = smem_u32(sQ + sj * 16384), ado = smem_u32(sDO + sj * 16384);
#pragma unroll
        for (int kk = 0; kk < HD / 16; ++kk)
          umma_bf16_ss(tS, umma_smem_desc_sw128(aq + kk * 32, 16, 1024), umma_smem_desc_sw128(ak + kk * 32, 16, 1024),
                       id_kk, kk > 0);
#pragma unroll
        for (int kk = 0; kk < HD / 16; ++kk)
          umma_bf16_ss(tDP, umma_smem_desc_sw128(ado + kk * 32, 16, 1024), umma_smem_desc_sw128(av + kk * 32, 16, 1024),
                       id_kk, kk > 0);
        umma_commit(sdp_ready);
      };
      mbar_wait(kv_full, 0);
      issue_sdp(0);
      for (int i = 0; i < nqb; ++i) {
        const int st = i % 3;
        if (i + 1 < nqb) {                     // S/dP of the next block as soon as this block's left TMEM
          mbar_wait(sdp_free, i & 1);
          tc_fence_after();
          issue_sdp(i + 1);
        }
        mbar_wait(ds_ready, i & 1);
        tc_fence_after();
        const uint32_t aq = smem_u32(sQ + st * 16384), ado = smem_u32(sDO + st * 16384);
#pragma unroll
        for (int kk = 0; kk < TILE / 16; ++kk) {   // reduction over the 128 query rows of this block
          const uint64_t a_pd = umma_smem_desc_sw128(apd + kk * 2048, 16384, 1024);
          const uint64_t a_ds = umma_smem_desc_sw128(ads + kk * 2048, 16384, 1024);
          const uint64_t b_do = umma_smem_desc_sw128(ado + kk * 2048, 8192, 1024);
          const uint64_t b_q = umma_smem_desc_sw128(aq + kk * 2048, 8192, 1024);
          umma_bf16_ss(tDV, a_pd, b_do, id_tt, (i > 0 || kk > 0));   // dV += Pd^T dO
          umma_bf16_ss(tDK, a_ds, b_q, id_tt, (i > 0 || kk > 0));    // dK += dS^T Q
        }
#pragma unroll
        for (int kk = 0; kk < TILE / 16; ++kk) {   // dQ = dS K   (reduction over the 128 keys)
          const uint64_t a_ds = umma_smem_desc_sw128(ads + (kk >> 2) * 16384 + (kk & 3) * 32, 16, 1024);
          const uint64_t b_k = umma_smem_desc_sw128(ak + kk * 2048, 8192, 1024);
          umma_bf16_ss(tDQ, a_ds, b_k, id_kt, kk > 0);
        }
        umma_commit(dq_ready);
        umma_commit(&qdo_empty[st]);
        if (i >= 1 && i + 2 < nqb) {           // slot of block i-1 (its MMAs finished before ds_ready(i) could fire)
          const int sp = (i - 1) % 3;
          mbar_wait(&qdo_empty[sp], ((i - 1) / 3) & 1);
          mbar_arrive_expect_tx(&qdo_full[sp], 32768);
          tma_load_2d(sQ + sp * 16384, &tmap_qkv, &qdo_full[sp], cq, row0 + (i + 2) * TILE);
          tma_load_2d(sDO + sp * 16384, &tmap_do, &qdo_full[sp], head * HD, row0 + (i + 2) * TILE);
        }
      }
      umma_commit(fin);
    }
  } else {
    const int r = (warp & 3) * 32 + lane;        // query row inside the tile == TMEM lane
    const int ch = warp >> 2;                    // which 32-key column quarter this thread handles
    const uint32_t lane_base = uint32_t((warp & 3) * 32) << 16;
    const float c_scale = p.scale * LOG2E;
    const float qscale8 = p.f8.q ? p.f8.meta[1] : 0.f;
    float amax8 = 0.f;
    // dQ rows of query block j: read back from TMEM, reduce into the fp32 accumulator (several key blocks)
    auto drain_dq = [&](int j) {
      mbar_wait(dq_ready, j & 1);
      tc_fence_after();
      uint32_t v[16];                            // each thread owns 16 of the 64 dQ columns of its row
      tmem_ld_32x16(tDQ + lane_base + ch * 16, v);
      tmem_ld_wait();
      const int q = j * TILE + r;
      if (q < p.S) {
        float* dq = p.dq_acc + (size_t)(row0 + q) * p.H + head * HD + ch * 16;
#pragma unroll
        for (int g = 0; g < 4; ++g)
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dq + g * 4),
                       "f"(__uint_as_float(v[g * 4])), "f"(__uint_as_float(v[g * 4 + 1])),
                       "f"(__uint_as_float(v[g * 4 + 2])), "f"(__uint_as_float(v[g * 4 + 3]))
                       : "memory");
      }
      tc_fence_before();                         // dQ reads done before ds_ready lets the next dQ MMA overwrite it
    };
    // log-sum-exp and delta of the row one query block ahead (ncu round 2: 6 % of the stall samples sat on these two loads)
    float n_lse = r < p.S ? __ldg(p.lse + (size_t)bh * p.S + r) : 0.f;
    float n_dlt = r < p.S ? __ldg(p.delta + (size_t)bh * p.S + r) : 0.f;
    for (int i = 0; i < nqb; ++i) {
      const int q = i * TILE + r;
      const bool q_ok = q < p.S;
      const float lse2 = q_ok ? n_lse * LOG2E : 0.f;
      const float dlt = q_ok ? n_dlt : 0.f;
      if (q + TILE < p.S && i + 1 < nqb) {
        n_lse = __ldg(p.lse + (size_t)bh * p.S + q + TILE);
        n_dlt = __ldg(p.delta + (size_t)bh * p.S + q + TILE);
      }
      const uint64_t erow = ((uint64_t)bh * p.S + (uint64_t)q) * (uint64_t)p.S;
      uint4 ppd[4], pds[4];                      // this thread's 32 P~ / dS values, packed bf16
      mbar_wait(sdp_ready, i & 1);
      tc_fence_after();
#pragma unroll
      for (int sc = 0; sc < 2; ++sc) {           // two 16-column sub-chunks
        const int c16 = ch * 2 + sc;
        uint32_t sv[16], dv[16];
        tmem_ld_32x16(tS + lane_base + c16 * 16, sv);
        tmem_ld_32x16(tDP + lane_base + c16 * 16, dv);
        tmem_ld_wait();
        if (sc == 1) {                           // S / dP of this block are in registers: the next block's may land
          tc_fence_before();
          mbar_arrive(sdp_free);
        }
        const int k0 = kb * TILE + c16 * 16;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          Keep8 keep = Keep8::all();
          if (p.thresh16 != 0)
            keep = dropout_keep8(seed, p.stream, (erow + (uint64_t)(k0 + g * 8)) >> 3, p.thresh16);
          float pd[8], ds[8];
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            const int key = k0 + g * 8 + t;
            const bool ok = q_ok && key < seqlen;
            const float pr = ok ? ex2_approx(fmaf(__uint_as_float(sv[g * 8 + t]), c_scale, -lse2)) : 0.f;
            const bool kp = keep[t];
            const float dp = kp ? __uint_as_float(dv[g * 8 + t]) * p.inv_keep : 0.f;
            pd[t] = kp ? pr * p.inv_keep : 0.f;
            ds[t] = pr * (dp - dlt) * p.scale;
          }
          ppd[sc * 2 + g] = make_uint4(pack_bf16(pd[0], pd[1]), pack_bf16(pd[2], pd[3]), pack_bf16(pd[4], pd[5]),
                                       pack_bf16(pd[6], pd[7]));
          pds[sc * 2 + g] = make_uint4(pack_bf16(ds[0], ds[1]), pack_bf16(ds[2], ds[3]), pack_bf16(ds[4], ds[5]),
                                       pack_bf16(ds[6], ds[7]));
        }
      }
      // block i-1: its dV/dK/dQ MMAs ran while the values above were computed; once dq_ready(i-1) has fired they no
      // longer read the P~ / dS buffers either
      if (i > 0) drain_dq(i - 1);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint32_t off = p_chunk_offset(r, (ch * 2 + (c >> 1)) * 2 + (c & 1));
        *reinterpret_cast<uint4*>(sPd + off) = ppd[c];
        *reinterpret_cast<uint4*>(sDS + off) = pds[c];
      }
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(ds_ready);
    }
    drain_dq(nqb - 1);
    // dK / dV of this key block: column quarters 0,1 write the two halves of dK, quarters 2,3 those of dV
    mbar_wait(fin, 0);
    tc_fence_after();
    const int key = kb * TILE + r;
    {
      const int w = ch >> 1, c = ch & 1;
      const uint32_t src = w == 0 ? tDK : tDV;
      uint32_t v[32];
      tmem_ld_32x32(src + lane_base + c * 32, v);
      tmem_ld_wait();
      if (key < p.S) {
        __nv_bfloat16* dst = p.dqkv + (size_t)(row0 + key) * 3 * p.H + (w + 1) * p.H + head * HD + c * 32;
#pragma unroll
        for (int g = 0; g < 4; ++g)
          *reinterpret_cast<uint4*>(dst + g * 8) = make_uint4(
              pack_bf16(__uint_as_float(v[g * 8]), __uint_as_float(v[g * 8 + 1])),
              pack_bf16(__uint_as_float(v[g * 8 + 2]), __uint_as_float(v[g * 8 + 3])),
              pack_bf16(__uint_as_float(v[g * 8 + 4]), __uint_as_float(v[g * 8 + 5])),
              pack_bf16(__uint_as_float(v[g * 8 + 6]), __uint_as_float(v[g * 8 + 7])));
        if (p.f8.q)
          emit_fp8_row<4>(p.f8, (size_t)(row0 + key) * 3 * p.H + (w + 1) * p.H + head * HD + c * 32, v, 1.f, qscale8, amax8);
      }
    }
    if (p.f8.q) fp8_amax_commit(p.f8, amax8);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 16) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// backward, S <= 128: TWO threads per query row (64 key columns each, 8 math warps), persistent CTAs over
// (batch, head) items, dS PARKED IN TENSOR MEMORY.  The MMA chain: S = Q K^T, dP = dO V^T -> P~ -> dV = P~^T dO;
// dS -> dK = dS^T Q, dQ = dS K; dV / dK / dQ overwrite the consumed S / dP accumulators, one 32 KB buffer carries P~
// and then dS.  A one-thread-per-row layout of the same chain measured 19 % issue utilisation (NOTES.md): four math
// warps per CTA cannot hide the dependent MMA -> math -> MMA -> math -> MMA chain and the global loads of O / lse at
// the head of an item, and its 64 registers of packed dS forced full unrolling (instruction-cache misses).  Here
//   * ~12 instructions per score element (dsoftmax_chunk16): 1 / keep_prob in the exponent, dS = p' * select(keep,
//     dP * scale + c, c) with the row constants folded, hoisted Philox keys, in-place 16-bit keep compares;
//   * every 16-column chunk's dS (8 packed words) is written back with tcgen05.st into the upper half of the thread's
//     own, already consumed dP columns (chunks run right to left, so the target columns are always behind the read
//     pointer) and copied to shared memory once the dV MMA has released the P~ buffer: no register array survives the
//     chunk loop, which therefore stays rolled (small code, 16-byte shared-memory stores);
//   * the loop over items keeps TMEM / barriers alive, V of the next item streams in under the softmax-gradient math
//     and Q / K / dO under the epilogue stores; the O half-row and log-sum-exp of the NEXT item are fetched while this
//     item waits for its last MMAs;
//   * delta = <dO, O>: each thread of a row computes half, one shared-memory exchange + named barrier per item.
// 96 KB, 256 TMEM columns, 288 threads -> two CTAs per SM (16 math warps per SM).
// ------------------------------------------------------------------------------------------------
// P~ and dS of 16 score columns of one row, packed bf16: p' = 2^(s c + off) = P / keep_prob, u = dP a + bq
template <bool FULL, bool DROP>
__device__ __forceinline__ void dsoftmax_chunk16(const uint32_t (&sv)[16], const uint32_t (&dv)[16], uint32_t (&pw)[8],
                                                 uint32_t (&dw)[8], float c_scale, float off, float a, float bq, int nvalid,
                                                 const PhiloxKeys& keys, uint64_t e8, uint32_t stream, uint32_t T) {
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    float pd[8], ds[8];
    uint4 r = make_uint4(0, 0, 0, 0);
    if (DROP) r = philox7(keys, e8 + (uint64_t)g, stream);
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      float pr = ex2_approx(fmaf(__uint_as_float(sv[g * 8 + t]), c_scale, off));   // P / keep_prob
      if (!FULL && g * 8 + t >= nvalid) pr = 0.f;
      const float u = fmaf(__uint_as_float(dv[g * 8 + t]), a, bq);                   // (dP / keep - delta) scale keep
      const bool kp = DROP ? keep_bit(r, t, T) : true;
      pd[t] = kp ? pr : 0.f;
      ds[t] = pr * (kp ? u : bq);
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      pw[g * 4 + t] = pack_bf16(pd[2 * t], pd[2 * t + 1]);
      dw[g * 4 + t] = pack_bf16(ds[2 * t], ds[2 * t + 1]);
    }
  }
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}

__global__ void __launch_bounds__(ATT_BWD_THREADS, 2)
attn_bwd_row2_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_do,
                     const AttnArgs p, const int n_items) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;                      // 16 KB each
  uint8_t* sV = smem + 16384;
  uint8_t* sQ = smem + 16384 * 2;
  uint8_t* sDO = smem + 16384 * 3;
  uint8_t* sP = smem + 16384 * 4;          // 32 KB: P~, later dS
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 16384 * 6);
  uint64_t* qkd_full = bars;               // Q, K, dO of an item landed
  uint64_t* v_full = bars + 1;             // V landed
  uint64_t* sdp_ready = bars + 2;          // S and dP complete (V is free)
  uint64_t* pd_ready = bars + 3;           // 256 threads: P~ is in shared memory, S / dP consumed, dS parked
  uint64_t* dv_done = bars + 4;            // dV MMA retired: the buffer may be overwritten with dS
  uint64_t* ds_ready = bars + 5;           // 256 threads: dS is in shared memory
  uint64_t* fin = bars + 6;                // dK, dQ complete (Q, K, dO, the buffer are free)
  uint64_t* acc_read = bars + 7;           // 256 threads: dQ / dK / dV read out of tensor memory
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
  float* xch = reinterpret_cast<float*>(bars + 10);   // [2 halves][128 rows]: partial delta

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 256) {
    tma_prefetch_desc(&tmap_qkv);
    tma_prefetch_desc(&tmap_do);
    mbar_init(qkd_full, 1);
    mbar_init(v_full, 1);
    mbar_init(sdp_ready, 1);
    mbar_init(pd_ready, 256);
    mbar_init(dv_done, 1);
    mbar_init(ds_ready, 256);
    mbar_init(fin, 1);
    mbar_init(acc_read, 256);
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(tmem_slot, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tS = tmem, tDP = tmem + 128, tDV = tmem, tDK = tmem + 64, tDQ = tmem + 128;
  pdl_trigger_small();
  pdl_wait();                              // PDL: see attn_fwd_row_kernel

  if (warp == 8) {
    if (lane == 0) {
      constexpr uint32_t id_kk = umma_idesc_bf16(128, 128, false, false);  // [q x keys], both K-major
      constexpr uint32_t id_tt = umma_idesc_bf16(128, 64, true, true);     // [keys x d] = X^T Y, both MN-major
      constexpr uint32_t id_kt = umma_idesc_bf16(128, 64, false, true);    // [q x d] = dS K, A K-major, B MN-major
      const uint32_t aq = smem_u32(sQ), ado = smem_u32(sDO), ak = smem_u32(sK), av = smem_u32(sV), ap = smem_u32(sP);
      auto load_qkd = [&](int item) {
        const int b = item / p.h, head = item - b * p.h;
        mbar_arrive_expect_tx(qkd_full, 49152);
        tma_load_2d(sDO, &tmap_do, qkd_full, head * HD, b * p.S);
        tma_load_2d(sK, &tmap_qkv, qkd_full, p.H + head * HD, b * p.S);
        tma_load_2d(sQ, &tmap_qkv, qkd_full, head * HD, b * p.S);
      };
      auto load_v = [&](int item) {
        const int b = item / p.h, head = item - b * p.h;
        mbar_arrive_expect_tx(v_full, 16384);
        tma_load_2d(sV, &tmap_qkv, v_full, 2 * p.H + head * HD, b * p.S);
      };
      int item = blockIdx.x;
      if (item < n_items) { load_qkd(item); load_v(item); }
      for (uint32_t g = 0; item < n_items; item += gridDim.x, ++g) {
        const int nitem = item + gridDim.x;
        const uint32_t ph = g & 1;
        if (g > 0) mbar_wait(acc_read, (g - 1) & 1);           // previous dQ / dK / dV drained
        mbar_wait(qkd_full, ph);
        mbar_wait(v_full, ph);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < HD / 16; ++kk)   // S = Q K^T
          umma_bf16_ss(tS, umma_smem_desc_sw128(aq + kk * 32, 16, 1024), umma_smem_desc_sw128(ak + kk * 32, 16, 1024), id_kk, kk > 0);
#pragma unroll
        for (int kk = 0; kk < HD / 16; ++kk)   // dP = dO V^T
          umma_bf16_ss(tDP, umma_smem_desc_sw128(ado + kk * 32, 16, 1024), umma_smem_desc_sw128(av + kk * 32, 16, 1024), id_kk, kk > 0);
        umma_commit(sdp_ready);
        mbar_wait(sdp_ready, ph);                              // V is free: the next one streams in under the math
        if (nitem < n_items) load_v(nitem);
        mbar_wait(pd_ready, ph);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < TILE / 16; ++kk)   // dV = P~^T dO -> S[0,64)
          umma_bf16_ss(tDV, umma_smem_desc_sw128(ap + kk * 2048, 16384, 1024), umma_smem_desc_sw128(ado + kk * 2048, 8192, 1024), id_tt, kk > 0);
        umma_commit(dv_done);
        mbar_wait(ds_ready, ph);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < TILE / 16; ++kk)   // dK = dS^T Q -> S[64,128)
          umma_bf16_ss(tDK, umma_smem_desc_sw128(ap + kk * 2048, 16384, 1024), umma_smem_desc_sw128(aq + kk * 2048, 8192, 1024), id_tt, kk > 0);
#pragma unroll
        for (int kk = 0; kk < TILE / 16; ++kk)   // dQ = dS K -> dP[0,64)
          umma_bf16_ss(tDQ, umma_smem_desc_sw128(ap + (kk >> 2) * 16384 + (kk & 3) * 32, 16, 1024),
                       umma_smem_desc_sw128(ak + kk * 2048, 8192, 1024), id_kt, kk > 0);
        umma_commit(fin);
        mbar_wait(fin, ph);                                    // Q, K, dO free: next item streams in under the epilogue
        if (nitem < n_items) load_qkd(nitem);
      }
    }
  } else {
    const int r = (warp & 3) * 32 + lane;                      // query row == key row of the epilogue == TMEM lane
    const int hf = warp >> 2;                                  // key-column half [64 hf, 64 hf + 64)
    const uint32_t lane_base = uint32_t((warp & 3) * 32) << 16;
    const float c_scale = p.scale * LOG2E;
    const bool drop = p.thresh16 != 0;
    const float lk = drop ? log2f(p.inv_keep) : 0.f;
    const uint32_t T = p.thresh16 << 16;
    const PhiloxKeys keys = philox_keys(drop ? p.seed.value() : 0ull);
    const bool row_ok = r < p.S;
    const float qscale8 = p.f8.q ? p.f8.meta[1] : 0.f;
    const uint32_t tPark = tDP + lane_base + hf * 64 + 32;     // 32 words: this thread's 64 dS values, packed bf16
    float amax8 = 0.f;
    // O half-row (32 columns) and log-sum-exp of the first item
    uint4 ov[4];
    float lse_nat = 0.f;
    int seqlen_next = 0;                                         // sequence length of the item being fetched (ncu, round 2b:
    auto fetch = [&](int item) {                                 // 6.7 % of the stall samples sat on this load, issued per item
      const int b = item / p.h, head = item - b * p.h;           // right before its first use)
      const __nv_bfloat16* src = p.ctx + ((size_t)b * p.S + r) * p.H + head * HD + hf * 32;
#pragma unroll
      for (int c = 0; c < 4; ++c) ov[c] = row_ok ? __ldg(reinterpret_cast<const uint4*>(src + c * 8)) : make_uint4(0, 0, 0, 0);
      lse_nat = row_ok ? __ldg(p.lse + (size_t)item * p.S + r) : 0.f;
      seqlen_next = __ldg(p.seqlens + b);
    };
    if ((int)blockIdx.x < n_items) fetch(blockIdx.x);
    uint32_t g = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++g) {
      const uint32_t ph = g & 1;
      const int b = item / p.h, head = item - b * p.h;
      const int seqlen = min(seqlen_next, p.S);
      const size_t tok = (size_t)b * p.S + r;
      mbar_wait(qkd_full, ph);
      float part = 0.f;                                        // this thread's half of delta = <dO, O>
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint4 dv = *reinterpret_cast<const uint4*>(sDO + r * 128 + (((hf * 4 + c) ^ (r & 7)) << 4));
        const uint32_t aw[4] = {ov[c].x, ov[c].y, ov[c].z, ov[c].w}, dw[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float2 x = unpack_bf16(aw[t]), y = unpack_bf16(dw[t]);
          part = fmaf(x.x, y.x, fmaf(x.y, y.y, part));
        }
      }
      float* xb = xch + (g & 1) * 256;                         // double buffered by item parity
      xb[hf * 128 + r] = part;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      const float dlt = xb[r] + xb[128 + r];
      const float off = lk - lse_nat * LOG2E;                  // p' = 2^(s c + off) = P / keep_prob
      const float a = p.scale;                                 // dS = p' * (keep ? dP * scale + bq : bq)
      const float bq = -dlt * p.scale / p.inv_keep;
      const int kvalid = row_ok ? seqlen : 0;                  // rows beyond the sequence contribute nothing
      const uint64_t e8row = (((uint64_t)item * p.S + (uint64_t)r) * (uint64_t)p.S) >> 3;
      mbar_wait(sdp_ready, ph);
      tc_fence_after();
#pragma unroll 1
      for (int cl = 3; cl >= 0; --cl) {                        // right to left: parked dS lands in consumed columns only
        const int c = hf * 4 + cl;                             // 16-column chunk of the row
        uint32_t sv[16], dv[16], pw[8], dw[8];
        tmem_ld_32x16(tS + lane_base + c * 16, sv);
        tmem_ld_32x16(tDP + lane_base + c * 16, dv);
        tmem_ld_wait();
        const int nv = kvalid - c * 16;
        const uint64_t e8 = e8row + (uint64_t)(2 * c);
        if (nv >= 16) {
          if (drop) dsoftmax_chunk16<true, true>(sv, dv, pw, dw, c_scale, off, a, bq, 16, keys, e8, p.stream, T);
          else dsoftmax_chunk16<true, false>(sv, dv, pw, dw, c_scale, off, a, bq, 16, keys, e8, p.stream, T);
        } else if (nv > 0) {
          if (drop) dsoftmax_chunk16<false, true>(sv, dv, pw, dw, c_scale, off, a, bq, nv, keys, e8, p.stream, T);
          else dsoftmax_chunk16<false, false>(sv, dv, pw, dw, c_scale, off, a, bq, nv, keys, e8, p.stream, T);
        } else {
#pragma unroll
          for (int t = 0; t < 8; ++t) { pw[t] = 0u; dw[t] = 0u; }
        }
        *reinterpret_cast<uint4*>(sP + p_chunk_offset(r, c * 2)) = make_uint4(pw[0], pw[1], pw[2], pw[3]);
        *reinterpret_cast<uint4*>(sP + p_chunk_offset(r, c * 2 + 1)) = make_uint4(pw[4], pw[5], pw[6], pw[7]);
        tmem_st_32x8(tPark + cl * 8, dw);
      }
      tmem_st_wait();
      fence_proxy_async();
      tc_fence_before();                                       // S / dP reads retired before dV may overwrite S
      mbar_arrive(pd_ready);
      // the chunk registers are dead: the next item's O half-row, log-sum-exp and sequence length start their trip now
      if (item + (int)gridDim.x < n_items) fetch(item + gridDim.x);
      mbar_wait(dv_done, ph);                                  // the tensor core no longer reads P~
      tc_fence_after();
      {
        uint32_t w[32];
        tmem_ld_32x32(tPark, w);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 8; ++i)
          *reinterpret_cast<uint4*>(sP + p_chunk_offset(r, hf * 8 + i)) = make_uint4(w[i * 4], w[i * 4 + 1], w[i * 4 + 2], w[i * 4 + 3]);
      }
      fence_proxy_async();
      tc_fence_before();                                       // parked dS read out before dQ may overwrite dP[0,64)
      mbar_arrive(ds_ready);
      mbar_wait(fin, ph);
      tc_fence_after();
      // ---- epilogue: columns [32 hf, 32 hf + 32) of this row of dQ (query r), dK and dV (key r)
      __nv_bfloat16* drow = p.dqkv + tok * 3 * p.H + head * HD + hf * 32;
#pragma unroll
      for (int w = 0; w < 3; ++w) {
        const uint32_t src = w == 0 ? tDQ : (w == 1 ? tDK : tDV);
        uint32_t v[32];
        tmem_ld_32x32(src + lane_base + hf * 32, v);
        tmem_ld_wait();
        if (w == 2) {                                          // accumulators drained: the next item's MMAs may go
          tc_fence_before();
          mbar_arrive(acc_read);
        }
        if (row_ok) {
          __nv_bfloat16* dst = drow + w * p.H;
#pragma unroll
          for (int gq = 0; gq < 4; ++gq)
            *reinterpret_cast<uint4*>(dst + gq * 8) = make_uint4(
                pack_bf16(__uint_as_float(v[gq * 8]), __uint_as_float(v[gq * 8 + 1])),
                pack_bf16(__uint_as_float(v[gq * 8 + 2]), __uint_as_float(v[gq * 8 + 3])),
                pack_bf16(__uint_as_float(v[gq * 8 + 4]), __uint_as_float(v[gq * 8 + 5])),
                pack_bf16(__uint_as_float(v[gq * 8 + 6]), __uint_as_float(v[gq * 8 + 7])));
          if (p.f8.q) emit_fp8_row<4>(p.f8, tok * 3 * p.H + (size_t)(w * p.H + head * HD + hf * 32), v, 1.f, qscale8, amax8);
        }
      }
    }
    if (p.f8.q) fp8_amax_commit(p.f8, amax8);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem, 256);
  }
}

// dq_acc (fp32 [B*S, H]) -> q slots of dqkv (bf16 [B*S, 3H])
__global__ void __launch_bounds__(256)
attn_dq_convert_kernel(const float* __restrict__ acc, __nv_bfloat16* __restrict__ dqkv, long long rows, int H, const Fp8Out f8) {
  const int per_row = H / 8;
  const float qscale = f8.q ? f8.meta[1] : 0.f;
  float amax = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < rows * per_row;
       i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / per_row;
    const int col = (int)(i % per_row) * 8;
    const float4 a = *reinterpret_cast<const float4*>(acc + row * H + col);
    const float4 c = *reinterpret_cast<const float4*>(acc + row * H + col + 4);
    *reinterpret_cast<uint4*>(dqkv + row * 3 * H + col) =
        make_uint4(pack_bf16(a.x, a.y), pack_bf16(a.z, a.w), pack_bf16(c.x, c.y), pack_bf16(c.z, c.w));
    if (f8.q) {
      const float t8[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
      fp8_emit8(f8, (size_t)(row * 3 * H + col), t8, qscale, amax);
    }
  }
  if (f8.q) fp8_amax_commit(f8, amax);
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
static void fill_args(AttnArgs& a, int B, int S, int h, int d, const int* seqlens, float scale,
                      Seed seed, unsigned int stream, float p_drop) {
  if (d != HD) { fprintf(stderr, "[b200] attention kernels need head_dim 64 (got %d)\n", d); abort(); }
  if (S > 512 || S % 8 != 0) { fprintf(stderr, "[b200] attention kernels need S <= 512 and S %% 8 == 0 (got %d)\n", S); abort(); }
  a.B = B; a.S = S; a.h = h; a.H = h * d; a.seqlens = seqlens; a.scale = scale; a.seed = seed; a.stream = stream;
  a.thresh16 = p_drop > 0.f ? (unsigned)(p_drop * 65536.f + 0.5f) : 0u;
  a.inv_keep = p_drop > 0.f ? 65536.f / (65536.f - (float)a.thresh16) : 1.f;
  a.ctx = nullptr; a.lse = nullptr; a.delta = nullptr; a.dqkv = nullptr; a.dq_acc = nullptr;
}

// multiprocessor count of the current device: the persistent kernels launch a fixed number of CTAs per SM
static int sm_count() {
  static int sms = 0;
  if (sms == 0) {
    int dev;
    B200_CUDA_CHECK(cudaGetDevice(&dev));
    B200_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  return sms;
}

void attention_fwd(const void* qkv, const int* seqlens, void* ctx, float* lse, int B, int S, int h, int d,
                   float scale, Seed seed, unsigned int stream, float p_drop, Fp8Out f8, cudaStream_t st) {
  AttnArgs a;
  fill_args(a, B, S, h, d, seqlens, scale, seed, stream, p_drop);
  a.ctx = (__nv_bfloat16*)ctx; a.lse = lse; a.f8 = f8;
  const int H = h * d;
  CUtensorMap tm = make_tmap_2d_bf16(qkv, 3 * H, (uint64_t)B * S, 3 * H, 64, TILE);
  const int sms = sm_count();
  const int nqb = (S + TILE - 1) / TILE, n_items = nqb * B * h;
  if (S <= TILE) {
    constexpr int SMEMR = 16384 * 3 + 1024 + 128;
    static bool once = false;
    if (!once) { B200_CUDA_CHECK(cudaFuncSetAttribute(attn_fwd_row_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEMR)); once = true; }
    const int g = n_items < sms * 4 ? n_items : sms * 4;
    launch_pdl(attn_fwd_row_kernel, dim3(g), dim3(ATT_ROW_THREADS), SMEMR, st, tm, a, n_items);
  } else {
    constexpr int SMEMS = 16384 * 5 + 1024 + 256;
    static bool once = false;
    if (!once) { B200_CUDA_CHECK(cudaFuncSetAttribute(attn_fwd_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEMS)); once = true; }
    const int g = n_items < sms * 2 ? n_items : sms * 2;
    attn_fwd_stream_kernel<<<g, ATT_STREAM_THREADS, SMEMS, st>>>(tm, a, n_items, nqb);
  }
}

void attention_bwd(const void* qkv, const int* seqlens, const void* ctx, const void* dctx, const float* lse,
                   void* dqkv, float* delta_ws, float* dq_acc, int B, int S, int h, int d, float scale,
                   Seed seed, unsigned int stream, float p_drop, Fp8Out f8, cudaStream_t st) {
  AttnArgs a;
  fill_args(a, B, S, h, d, seqlens, scale, seed, stream, p_drop);
  a.f8 = f8;
  const int H = h * d;
  a.lse = const_cast<float*>(lse); a.delta = delta_ws; a.dqkv = (__nv_bfloat16*)dqkv; a.dq_acc = dq_acc;
  a.ctx = (__nv_bfloat16*)const_cast<void*>(ctx);
  CUtensorMap tq = make_tmap_2d_bf16(qkv, 3 * H, (uint64_t)B * S, 3 * H, 64, TILE);
  CUtensorMap td = make_tmap_2d_bf16(dctx, H, (uint64_t)B * S, H, 64, TILE);
  if (S <= TILE) {                               // one key block; the kernel computes delta itself
    constexpr int SMEM2 = 16384 * 6 + 1024 + 128 + 2048;
    static bool once = false;
    if (!once) { B200_CUDA_CHECK(cudaFuncSetAttribute(attn_bwd_row2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM2)); once = true; }
    const int n_items = B * h, sms = sm_count();
    const int g = n_items < sms * 2 ? n_items : sms * 2;
    launch_pdl(attn_bwd_row2_kernel, dim3(g), dim3(ATT_BWD_THREADS), SMEM2, st, tq, td, a, n_items);
    return;
  }
  if (dq_acc == nullptr) { fprintf(stderr, "[b200] attention_bwd needs a dq accumulation buffer when S > 128\n"); abort(); }
  const long long groups = (long long)B * S * h;
  attn_delta_kernel<<<(unsigned)((groups * 8 + 255) / 256), 256, 0, st>>>((const __nv_bfloat16*)ctx,
                                                                       (const __nv_bfloat16*)dctx, delta_ws, B, S, h, H);
  B200_CUDA_CHECK(cudaMemsetAsync(dq_acc, 0, sizeof(float) * (size_t)B * S * H, st));
  constexpr int SMEMP = 16384 * 12 + 1024 + 128;
  static bool once = false;
  if (!once) { B200_CUDA_CHECK(cudaFuncSetAttribute(attn_bwd_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEMP)); once = true; }
  attn_bwd_pipe_kernel<<<dim3((S + TILE - 1) / TILE, B * h), ATT_BWD16_THREADS, SMEMP, st>>>(tq, td, a);
  const long long work = (long long)B * S * (H / 8);
  int g = (int)((work + 255) / 256);
  if (g > 148 * 16) g = 148 * 16;
  attn_dq_convert_kernel<<<g, 256, 0, st>>>(dq_acc, (__nv_bfloat16*)dqkv, (long long)B * S, H, a.f8);
}

}  // namespace b200
