// Fused attention forward on tcgen05 for the GPS shapes (<= 384 keys, head dim 64):
//   O = dropout(softmax( Q K^T / sqrt(64) + spatial_log_bias + key_padding_mask )) V          per (scene, head)
// Replaces the attention core of
//   * MultiHeadAttentionSpatial, 'cond' fusion (modules/layers/transformers.py:188-237): the per-(head, query)
//     spatial gate  log(clamp(sigmoid(w . pairwise_loc + b), 1e-6))  is computed on the fly from the 5-dim pairwise
//     geometry and the 6 language-conditioned weights — the (H,B,L,T) attention / loc_attn / mask tensors of the
//     reference are never materialised;
//   * nn.MultiheadAttention's scaled-dot-product core incl. its attention-weight dropout (joint self-attention of
//     UnifiedSpatialCrossEncoderV2, self/cross attention of the V1 / Entity decoders; transformers.py:22-24,69-74,118-120).
// One CTA = one (scene, head), 8 warps: Q / K / V head slices arrive by TMA (128-byte swizzle, zero-filled past the
// sequence end), S = Q K^T is ONE tcgen05.mma chain into TMEM (N = keys rounded to 16), the softmax runs with one
// thread per (query row, half of the key columns) — two warpgroups share the 128 TMEM lanes and split the columns —,
// P goes back to shared memory as the K-major A operand of O = P V, whose B operand is the SAME staged V tile read
// MN-major (no transposed copy).  O reuses the TMEM columns of S.  All loops over keys are rolled 16-column units, so
// the kernel body stays inside the instruction cache.
// Keys past the last unmasked one of the scene (`kend`, from the key-padding mask) are skipped: the S MMA, the softmax
// units and the P V k-steps stop at round16(kend).  Their weights are exactly 0, so the output and lse are bit-identical
// to the same scene with those keys cut off.
#include "attn_common.cuh"
#include "svgps.h"

namespace {

using namespace attn;

struct FwdArgs {
  __nv_bfloat16 *out;              // (B,Lq,*) head h at columns [h*64, h*64+64)
  long long o_bs;
  int o_rs;
  const unsigned char *kpm;        // (B,Lk) 1 = masked key, or null
  const float *sw;                 // (B,Lq,SH*6) [bias, w1..w5] per spatial head (GATED)
  const float *locs;               // (B,Lq,Lk,5)
  int B, H, SH, Lq, Lk;
  float scale;
  float *lse;                      // (B,H,Lq) natural-log log-sum-exp of the logits per query, or null
  uint32_t tmem_cols;
  uint32_t t16;                    // dropout threshold (DROP)
  float inv_keep;
  unsigned long long seed;
  const unsigned long long *seed_offset;  // device counter added to the seed at run time (or null)
};

__device__ __forceinline__ float u2f(uint32_t x) { return __uint_as_float(x); }

template <bool GATED, bool DROP>
__global__ void __launch_bounds__(256, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap mq, const __grid_constant__ CUtensorMap mk,
                const __grid_constant__ CUtensorMap mv, const FwdArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int NK = (a.Lk + 15) & ~15;          // keys rounded to the MMA granularity
  const int nkbox = NK >> 4;                 // 16-row TMA boxes of K / V
  uint8_t *sQ = smem;                        // [128][64] sw128
  uint8_t *sK = sQ + 16384;                  // [NK][64]  sw128
  uint8_t *sV = sK + NK * 128;               // [NK][64]  sw128 (read MN-major)
  uint8_t *sP = sV + NK * 128;               // [NK/8][128][8] K-major, no swizzle
  float *kb = reinterpret_cast<float *>(sP + NK * 256);  // [384] additive key bias: 0 or -inf
  float *xmax = kb + 384;                    // [2][128] per-warpgroup row maxima
  float *xsum = xmax + 256;                  // [2][128] per-warpgroup row sums
  uint64_t *bars = reinterpret_cast<uint64_t *>(xsum + 256);  // 0: K/V landed, 1: Q tile landed, 2: MMA done
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 3);
  int *kend_s = reinterpret_cast<int *>(tmem_slot + 1);        // 1 + index of the last unmasked key

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, wg = warp >> 2, wq = warp & 3;
  const int row = wq * 32 + lane;            // tile row == TMEM lane of this thread
  const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    mbar_fence_init();
    *kend_s = 0;
    tma_prefetch_desc(&mq);
    tma_prefetch_desc(&mk);
    tma_prefetch_desc(&mv);
  }
  __syncthreads();
  if (tid == 0) {
    mbar_expect_tx(&bars[0], 2 * rows_bytes(0, nkbox, a.Lk));
    tma_rows(sK, &mk, h, 0, nkbox, a.Lk, b, &bars[0]);
    tma_rows(sV, &mv, h, 0, nkbox, a.Lk, b, &bars[0]);
    mbar_expect_tx(&bars[1], rows_bytes(0, 8, a.Lq));
    tma_rows(sQ, &mq, h, 0, 8, a.Lq, b, &bars[1]);
  }
  if (warp == 1) tmem_alloc_n(tmem_slot, a.tmem_cols);
  int last = 0;
  for (int j = tid; j < 384; j += 256) {
    const bool live = j < a.Lk && !(a.kpm != nullptr && a.kpm[(size_t)b * a.Lk + j]);
    kb[j] = live ? 0.f : -INFINITY;
    if (live) last = j + 1;
  }
  last = __reduce_max_sync(0xffffffffu, last);
  if (lane == 0 && last > 0) atomicMax(kend_s, last);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t trow = tmem + ((uint32_t)(wq * 32) << 16);
  const float c2 = a.scale * LOG2E;
  // keys swept: round16(kend), at least one unit so that a scene with every key masked still gets O = 0 from P V
  const int NKe = max(16, (*kend_s + 15) & ~15);
  const int nu = NKe >> 4;                   // 16-column units, split between the two warpgroups
  const int u_begin = wg == 0 ? 0 : (nu + 1) / 2, u_end = wg == 0 ? (nu + 1) / 2 : nu;
  const bool vec_loc = GATED && (a.Lk & 3) == 0;
  uint32_t ph_q = 0, ph_m = 0;

  for (int q0 = 0; q0 < a.Lq; q0 += 128) {
    const int qi = q0 + row;
    const bool qlive = qi < a.Lq;
    const bool wlive = q0 + wq * 32 < a.Lq;  // warp-uniform: this warp owns at least one query
    // ---- S = Q K^T ---------------------------------------------------------------------------------------------------
    if (tid < 32) {   // warp 0, converged: elect.sync picks the issuing lane (tc05.cuh: warp-converged issue)
      if (q0 == 0) mbar_wait(&bars[0], 0);
      mbar_wait(&bars[1], ph_q);
      fence_after_sync();
      const uint32_t aQ = smem_u32(sQ), aK = smem_u32(sK);
      for (int n0 = 0; n0 < NKe; n0 += 256) {  // one MMA covers at most 256 keys
        const uint32_t idesc = idesc_kk(min(256, NKe - n0));
#pragma unroll
        for (int ks = 0; ks < DH / 16; ++ks)
          mma_bf16_e(tmem + n0, make_desc_sw128(aQ + ks * 32), make_desc_sw128(aK + n0 * 128 + ks * 32), idesc, ks > 0);
      }
      mma_commit_e(&bars[2]);
    }
    ph_q ^= 1u;
    GateW gw;
    const float *loc = nullptr;
    uint32_t rk = 0;
    if (GATED && qlive) {
      gw.load(a.sw + ((size_t)b * a.Lq + qi) * (a.SH * 6) + (a.SH == 1 ? 0 : h) * 6);
      loc = a.locs + ((size_t)b * a.Lq + qi) * (size_t)a.Lk * 5;
    }
    if (DROP) rk = drop_row_key(attn::effective_seed(a.seed, a.seed_offset), ((unsigned long long)b * a.H + h) * a.Lq + qi);
    mbar_wait(&bars[2], ph_m);
    ph_m ^= 1u;
    fence_after_sync();
    if (tid == 0 && q0 + 128 < a.Lq) {  // sQ is free again: fetch the next query tile behind the softmax
      mbar_expect_tx(&bars[1], rows_bytes(q0 + 128, 8, a.Lq));
      tma_rows(sQ, &mq, h, q0 + 128, 8, a.Lq, b, &bars[1]);
    }

    // ---- pass 1: row maximum of the scaled, masked logits (the gate is <= 0, so this bounds the gated logits too) ----
    float m2 = -INFINITY;
    if (wlive) {
      // TMEM loads are software-pipelined: unit u + 1 is in flight while unit u is reduced (tcgen05.wait::ld retires every
      // load issued before it, so the next load is issued right after the wait)
      uint32_t ra[16], rb[16];
      if (u_begin < u_end) tmem_ld16_async(trow + u_begin * 16, ra);
#pragma unroll 1
      for (int u = u_begin; u < u_end; u += 2) {
        tmem_wait16(ra);
        if (u + 1 < u_end) tmem_ld16_async(trow + (u + 1) * 16, rb);
        {
          const float4 *kb4 = reinterpret_cast<const float4 *>(kb + u * 16);
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const float4 k4 = kb4[g];
            m2 = fmaxf(m2, fmaxf(fmaxf(fmaf(u2f(ra[4 * g]), c2, k4.x), fmaf(u2f(ra[4 * g + 1]), c2, k4.y)),
                                 fmaxf(fmaf(u2f(ra[4 * g + 2]), c2, k4.z), fmaf(u2f(ra[4 * g + 3]), c2, k4.w))));
          }
        }
        if (u + 1 < u_end) {
          tmem_wait16(rb);
          if (u + 2 < u_end) tmem_ld16_async(trow + (u + 2) * 16, ra);
          const float4 *kb4 = reinterpret_cast<const float4 *>(kb + (u + 1) * 16);
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const float4 k4 = kb4[g];
            m2 = fmaxf(m2, fmaxf(fmaxf(fmaf(u2f(rb[4 * g]), c2, k4.x), fmaf(u2f(rb[4 * g + 1]), c2, k4.y)),
                                 fmaxf(fmaf(u2f(rb[4 * g + 2]), c2, k4.z), fmaf(u2f(rb[4 * g + 3]), c2, k4.w))));
          }
        }
      }
    }
    xmax[wg * 128 + row] = m2;
    __syncthreads();
    m2 = fmaxf(xmax[row], xmax[128 + row]);
    if (m2 == -INFINITY) m2 = 0.f;  // every key masked: all weights 0, output row 0

    // ---- pass 2: p = 2^(x - max), row sum, dropout, bf16 P tile ------------------------------------------------------------
    float sum = 0.f;
    if (wlive) {
      uint32_t rn[16];                      // next unit's S columns (in flight behind the current unit's math)
      if (u_begin < u_end) tmem_ld16_async(trow + u_begin * 16, rn);
#pragma unroll 1
      for (int u = u_begin; u < u_end; ++u) {
        const int j0 = u * 16;
        uint32_t r[16];
        float g2[16];
        if (GATED) {
#pragma unroll
          for (int i = 0; i < 16; ++i) g2[i] = 0.f;
          if (loc != nullptr) {
            if (vec_loc) {
              const float4 *l4 = reinterpret_cast<const float4 *>(loc + (size_t)j0 * 5);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                if (j0 + q * 4 < a.Lk) {
                  const float4 A = __ldg(l4 + q * 5), B2 = __ldg(l4 + q * 5 + 1), C = __ldg(l4 + q * 5 + 2),
                               D = __ldg(l4 + q * 5 + 3), E = __ldg(l4 + q * 5 + 4);
                  g2[q * 4] = gw.log2gate(A.x, A.y, A.z, A.w, B2.x);
                  g2[q * 4 + 1] = gw.log2gate(B2.y, B2.z, B2.w, C.x, C.y);
                  g2[q * 4 + 2] = gw.log2gate(C.z, C.w, D.x, D.y, D.z);
                  g2[q * 4 + 3] = gw.log2gate(D.w, E.x, E.y, E.z, E.w);
                }
              }
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i)
                if (j0 + i < a.Lk) {
                  const float *l = loc + (size_t)(j0 + i) * 5;
                  g2[i] = gw.log2gate(l[0], l[1], l[2], l[3], l[4]);
                }
            }
          }
        }
        tmem_wait16(rn);
#pragma unroll
        for (int i = 0; i < 16; ++i) r[i] = rn[i];
        if (u + 1 < u_end) tmem_ld16_async(trow + j0 + 16, rn);
        const float4 *kb4 = reinterpret_cast<const float4 *>(kb + j0);
        float p[16];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float4 k4 = kb4[g];
          const float kk[4] = {k4.x, k4.y, k4.z, k4.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int i = g * 4 + e;
            float x = fmaf(u2f(r[i]), c2, kk[e]) - m2;
            if (GATED) x += g2[i];
            p[i] = ex2f(x);
            sum += p[i];
          }
        }
        if (DROP) {
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            const uint32_t hh = drop_pair_hash(rk, (uint32_t)(j0 + i) >> 1);
            p[i] = (hh & 0xFFFFu) >= a.t16 ? p[i] * a.inv_keep : 0.f;
            p[i + 1] = (hh >> 16) >= a.t16 ? p[i + 1] * a.inv_keep : 0.f;
          }
        }
        // unnormalised probabilities -> bf16 A operand; 1 / sum is applied to the fp32 output row
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          uint32_t w[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) w[e] = pack_bf16(p[hf * 8 + e * 2], p[hf * 8 + e * 2 + 1]);
          *reinterpret_cast<uint4 *>(sP + tile_off(128, row, j0 + hf * 8)) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
    }
    xsum[wg * 128 + row] = sum;
    fence_proxy_async_smem();
    fence_before_sync();
    __syncthreads();

    // ---- O = P V (V staged once, read MN-major); O overwrites the S columns ---------------------------------------------------
    if (tid < 32) {
      fence_after_sync();
      const uint32_t aP = smem_u32(sP), aV = smem_u32(sV);
      const uint32_t idesc = idesc_kmn(DH);
#pragma unroll 1
      for (int ks = 0; ks < nu; ++ks)
        mma_bf16_e(tmem, make_desc(aP + ks * 4096, 2048, 128), make_desc_sw128_mn(aV + ks * 2048), idesc, ks > 0);
      mma_commit_e(&bars[2]);
    }
    mbar_wait(&bars[2], ph_m);
    ph_m ^= 1u;
    fence_after_sync();
    if (wlive) {
      const float tot = xsum[row] + xsum[128 + row];
      const float inv = tot > 0.f ? 1.0f / tot : 0.f;
      uint32_t r0[16], r1[16];
      tmem_ld16_async(trow + wg * 32, r0);
      tmem_ld16_async(trow + wg * 32 + 16, r1);
      tmem_wait16(r0);
      tmem_wait16(r1);
      if (qlive) {
        if (wg == 0 && a.lse != nullptr)
          a.lse[((size_t)b * a.H + h) * a.Lq + qi] = tot > 0.f ? (m2 + lg2f(tot)) * LN2 : INFINITY;
        __nv_bfloat16 *o = a.out + (size_t)b * a.o_bs + (size_t)qi * a.o_rs + h * DH + wg * 32;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          uint32_t w[4], z[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            w[e] = pack_bf16(u2f(r0[hf * 8 + e * 2]) * inv, u2f(r0[hf * 8 + e * 2 + 1]) * inv);
            z[e] = pack_bf16(u2f(r1[hf * 8 + e * 2]) * inv, u2f(r1[hf * 8 + e * 2 + 1]) * inv);
          }
          *reinterpret_cast<uint4 *>(o + hf * 8) = make_uint4(w[0], w[1], w[2], w[3]);
          *reinterpret_cast<uint4 *>(o + 16 + hf * 8) = make_uint4(z[0], z[1], z[2], z[3]);
        }
      }
    }
    if (q0 + 128 < a.Lq) {  // the next tile's S overwrites O, xmax / xsum are reused
      fence_before_sync();
      __syncthreads();
      fence_after_sync();
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc_n(tmem, a.tmem_cols);
}

template <bool GATED, bool DROP>
int launch_fwd(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const FwdArgs &a, cudaStream_t st) {
  const int NK = (a.Lk + 15) & ~15;
  const size_t smem = 16384 + (size_t)NK * 128 * 2 + (size_t)NK * 256 + (384 + 512) * 4 + 64;
  constexpr size_t SMEM_MAX = 16384 + 384 * 128 * 2 + 384 * 256 + (384 + 512) * 4 + 64;
  auto kern = attn_fwd_kernel<GATED, DROP>;
  static bool configured[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return SV_ERR_INVALID_ARG;
  if (!configured[dev]) {
    int rc = sv::cuda_status(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX));
    if (rc) return rc;
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    configured[dev] = true;
  }
  kern<<<a.B * a.H, 256, smem, st>>>(mq, mk, mv, a);
  return sv::after_launch();
}

}  // namespace

extern "C" int sv_attention_fwd_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs, int k_rs,
                                     const void *v, long long v_bs, int v_rs, void *out, long long o_bs, int o_rs,
                                     const unsigned char *key_padding_mask, const float *spatial_w, int spatial_heads,
                                     const float *pairwise_locs, int B, int H, int Lq, int Lk, float scale,
                                     void *stream) {
  return sv_attention_fwd_dropout_bf16(q, q_bs, q_rs, k, k_bs, k_rs, v, v_bs, v_rs, out, o_bs, o_rs, key_padding_mask,
                                       spatial_w, spatial_heads, pairwise_locs, B, H, Lq, Lk, scale, nullptr, 0.f, 0ull,
                                       stream);
}

extern "C" int sv_attention_fwd_lse_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs, int k_rs,
                                         const void *v, long long v_bs, int v_rs, void *out, long long o_bs, int o_rs,
                                         const unsigned char *key_padding_mask, const float *spatial_w,
                                         int spatial_heads, const float *pairwise_locs, int B, int H, int Lq, int Lk,
                                         float scale, float *lse, void *stream) {
  return sv_attention_fwd_dropout_bf16(q, q_bs, q_rs, k, k_bs, k_rs, v, v_bs, v_rs, out, o_bs, o_rs, key_padding_mask,
                                       spatial_w, spatial_heads, pairwise_locs, B, H, Lq, Lk, scale, lse, 0.f, 0ull, stream);
}

extern "C" int sv_attention_fwd_dropout_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs,
                                             int k_rs, const void *v, long long v_bs, int v_rs, void *out, long long o_bs,
                                             int o_rs, const unsigned char *key_padding_mask, const float *spatial_w,
                                             int spatial_heads, const float *pairwise_locs, int B, int H, int Lq, int Lk,
                                             float scale, float *lse, float dropout_p, unsigned long long seed,
                                             void *stream) {
  if (!(dropout_p >= 0.f) || dropout_p >= 1.f) return SV_ERR_INVALID_ARG;
  if (B < 0 || H < 1 || Lq < 0 || Lk < 1 || Lk > 384) return SV_ERR_INVALID_ARG;
  if (B == 0 || Lq == 0) return SV_OK;
  if (!q || !k || !v || !out) return SV_ERR_INVALID_ARG;
  if ((q_rs % 8) || (k_rs % 8) || (v_rs % 8) || (o_rs % 8) || (q_bs % 8) || (k_bs % 8) || (v_bs % 8) || (o_bs % 8))
    return SV_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(q) & 15) || (reinterpret_cast<uintptr_t>(k) & 15) ||
      (reinterpret_cast<uintptr_t>(v) & 15) || (reinterpret_cast<uintptr_t>(out) & 15))
    return SV_ERR_INVALID_ARG;
  if (spatial_w && (!pairwise_locs || (spatial_heads != 1 && spatial_heads != H))) return SV_ERR_INVALID_ARG;
  if (spatial_w && dropout_p > 0.f) return SV_ERR_INVALID_ARG;  // the reference's spatial attention has no weight dropout
  FwdArgs a;
  a.out = (__nv_bfloat16 *)out; a.o_bs = o_bs; a.o_rs = o_rs;
  a.kpm = key_padding_mask; a.sw = spatial_w; a.locs = pairwise_locs;
  a.B = B; a.H = H; a.SH = spatial_heads; a.Lq = Lq; a.Lk = Lk; a.scale = scale;
  a.lse = lse;
  const int NK = (Lk + 15) & ~15;
  a.tmem_cols = pow2_cols(NK < 64 ? 64 : NK);
  a.t16 = drop_threshold(dropout_p);
  a.inv_keep = 1.0f / (1.0f - dropout_p);
  a.seed = seed; a.seed_offset = sv::g_seed_offset;
  CUtensorMap mq, mk, mv;
  int rc = make_map(&mq, q, B, Lq, H, q_rs, q_bs);
  if (rc) return rc;
  rc = make_map(&mk, k, B, Lk, H, k_rs, k_bs);
  if (rc) return rc;
  rc = make_map(&mv, v, B, Lk, H, v_rs, v_bs);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (spatial_w) return launch_fwd<true, false>(mq, mk, mv, a, st);
  if (a.t16) return launch_fwd<false, true>(mq, mk, mv, a, st);
  return launch_fwd<false, false>(mq, mk, mv, a, st);
}
