// Backward of the fused attention (csrc/attention.cu) on tcgen05.  P is recomputed from Q, K, the gate and the saved
// log-sum-exp; the dropout mask is regenerated from (seed, indices); no (B,H,L,T) tensor is ever stored.  Reference math:
// autograd of modules/layers/transformers.py:188-237 and of nn.MultiheadAttention's core
// (transformers.py:22-24,69-74,118-120).
// Plain and dropout attention: attn_bwd_fused_kernel, ONE launch per call (below).
// Spatially gated attention: attn_bwd_gated_kernel, launched twice per call — the gradient of the six gate weights is a
// per-query sum over keys, thread-local only when tile rows are queries:
//   SIDE 0 (tile rows = queries): S = Q K^T, dP = dO V^T -> dS = P o (dP - D) -> dQ = scale * dS K,
//                                 D = rowsum(dO o O), gradients of the 6 spatial-gate weights of each (query, head)
//   SIDE 1 (tile rows = keys):    S^T = K Q^T, dP^T = V dO^T -> P^T, dS^T -> dV = P^T dO, dK = scale * dS^T Q
// Structure (both sides): the "row" operand pair (Q,dO | K,V) is a 128-row TMA tile; the "column" operand pair
// (K,V | Q,dO) is streamed in blocks of 64 rows through a two-deep TMA ring (the next block lands behind the current
// element-wise stage).  Per block: two tcgen05.mma chains fill 2 x 64 TMEM columns, the element-wise stage (one thread
// per row, the two warpgroups split the block's 16-column units) writes the bf16 dS / P tiles, and the output MMAs
// accumulate over the blocks reading the SAME staged block MN-major.  TMEM: 4 x 64 columns, shared memory 80-110 KB
// independent of the sequence length -> two CTAs per SM for every shape up to 384 x 384.
#include "attn_common.cuh"
#include "svgps.h"

namespace {

using namespace attn;

struct BwdArgs {
  const __nv_bfloat16 *o, *d_o;      // (B,Lq,H*64) contiguous
  const unsigned char *kpm;          // (B,Lk) or null
  const float *sw, *locs, *lse;      // (B,Lq,H*6) | (B,Lq,Lk,5) | (B,H,Lq)
  int B, H, Lq, Lk;
  float scale;
  __nv_bfloat16 *dq, *dk, *dv;       // (B,L,H*64) with row stride d_rs (elements; rows of one tensor d_rs apart, scenes L * d_rs)
  int d_rs;
  float *dsw;                        // (B,Lq,H*6) or null
  float *dvec;                       // gated: (B,H,Lq) D, written by SIDE 0, read by SIDE 1
                                     // fused: (B,H,Lq,64) fp32 dQ partial sums (scenes with more than one live key tile)
  uint32_t t16;
  float inv_keep;
  unsigned long long seed;
  const unsigned long long *seed_offset;  // device counter added to the seed at run time (or null)
};

__device__ __forceinline__ float u2f(uint32_t x) { return __uint_as_float(x); }

constexpr uint32_t COL_S = 0, COL_DP = 64, COL_O1 = 128, COL_O2 = 192, TMEM_COLS = 256;

// 64 fp32 accumulator columns of this thread's row -> bf16 row of `dst` (64 contiguous elements)
__device__ __forceinline__ void store_row64(uint32_t taddr, __nv_bfloat16 *dst, bool live) {
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    uint32_t r0[16], r1[16];
    tmem_ld16_async(taddr + c * 32, r0);
    tmem_ld16_async(taddr + c * 32 + 16, r1);
    tmem_wait16(r0);
    tmem_wait16(r1);
    if (live) {
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        uint32_t w[4], z[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          w[e] = pack_bf16(u2f(r0[hf * 8 + e * 2]), u2f(r0[hf * 8 + e * 2 + 1]));
          z[e] = pack_bf16(u2f(r1[hf * 8 + e * 2]), u2f(r1[hf * 8 + e * 2 + 1]));
        }
        *reinterpret_cast<uint4 *>(dst + c * 32 + hf * 8) = make_uint4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<uint4 *>(dst + c * 32 + 16 + hf * 8) = make_uint4(z[0], z[1], z[2], z[3]);
      }
    }
  }
}

template <int SIDE>
__global__ void __launch_bounds__(256, 2)
attn_bwd_gated_kernel(const __grid_constant__ CUtensorMap mR1, const __grid_constant__ CUtensorMap mR2,
                const __grid_constant__ CUtensorMap mC1, const __grid_constant__ CUtensorMap mC2, const BwdArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int Lr = SIDE == 0 ? a.Lq : a.Lk;    // rows of the tiles
  const int Lc = SIDE == 0 ? a.Lk : a.Lq;    // columns swept in blocks of 64
  const int NC = (Lc + 15) & ~15;
  uint8_t *sR1 = smem;                       // [128][64] sw128   Q  | K
  uint8_t *sR2 = sR1 + 16384;                // [128][64] sw128   dO | V
  uint8_t *sC = sR2 + 16384;                 // 2 buffers x { [64][64] sw128 K | Q block, [64][64] sw128 V | dO block }
  uint8_t *sG1 = sC + 2 * 16384;             // [8][128][8] K-major   scale * dS (^T)
  uint8_t *sG2 = sG1 + 16384;                // [8][128][8] K-major   P^T (SIDE 1)
  float *vec = reinterpret_cast<float *>(sG2 + (SIDE == 1 ? 16384 : 0));
  // SIDE 0: vec = kb[NC] | red[128][6]      SIDE 1: vec = lse2[NC] | Dv[NC] | W[NC][6]
  float *kb = vec, *red = vec + NC;
  float *lse2s = vec, *Dv = vec + NC;
  float *Ws = vec + 2 * NC;
  // barriers 0,1: column block landed in buffer 0 / 1, 2: row tile landed, 3: MMA done
  uint64_t *bars = reinterpret_cast<uint64_t *>(vec + (SIDE == 0 ? NC + 768 : 8 * NC));
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 4);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, wg = warp >> 2, wq = warp & 3;
  const int row = wq * 32 + lane;
  const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
  const int E = a.H * DH;
  const int nblk = (NC + 63) >> 6;
  // column block `cb` of a tile (rows [64 cb, 64 cb + nb) of the column operands) -> staging buffer `buf`
  auto load_cblock = [&](int cb, int buf) {
    const int nb = min(64, NC - cb * 64);
    mbar_expect_tx(&bars[buf], 2 * rows_bytes(cb * 64, nb >> 4, Lc));
    tma_rows(sC + buf * 16384, &mC1, h, cb * 64, nb >> 4, Lc, b, &bars[buf]);
    tma_rows(sC + buf * 16384 + 8192, &mC2, h, cb * 64, nb >> 4, Lc, b, &bars[buf]);
  };

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    mbar_init(&bars[3], 1);
    mbar_fence_init();
    tma_prefetch_desc(&mR1);
    tma_prefetch_desc(&mR2);
    tma_prefetch_desc(&mC1);
    tma_prefetch_desc(&mC2);
  }
  __syncthreads();
  if (tid == 0) {
    load_cblock(0, 0);
    mbar_expect_tx(&bars[2], 2 * rows_bytes(0, 8, Lr));
    tma_rows(sR1, &mR1, h, 0, 8, Lr, b, &bars[2]);
    tma_rows(sR2, &mR2, h, 0, 8, Lr, b, &bars[2]);
  }
  if (warp == 1) tmem_alloc_n(tmem_slot, TMEM_COLS);
  // per-column vectors
  for (int c = tid; c < NC; c += 256) {
    if (SIDE == 0) {
      kb[c] = (c < a.Lk && !(a.kpm != nullptr && a.kpm[(size_t)b * a.Lk + c])) ? 0.f : -INFINITY;
    } else {
      const bool live = c < a.Lq;
      const size_t r = ((size_t)b * a.H + h) * a.Lq + c;
      lse2s[c] = live ? a.lse[r] * LOG2E : INFINITY;
      Dv[c] = live ? a.dvec[r] : 0.f;
      const float *w = a.sw + ((size_t)b * a.Lq + (live ? c : 0)) * (a.H * 6) + h * 6;
#pragma unroll
      for (int t = 0; t < 6; ++t) Ws[c * 6 + t] = live ? -LOG2E * w[t] : 0.f;
    }
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t trow = tmem + ((uint32_t)(wq * 32) << 16);
  const float c2 = a.scale * LOG2E;
  uint32_t ph_r = 0, ph_m = 0;
  int cbi = 0;  // running column-block counter: buffer = cbi & 1, phase of its barrier = (cbi >> 1) & 1

  for (int r0 = 0; r0 < Lr; r0 += 128) {
    const int ri = r0 + row;                     // query (SIDE 0) / key (SIDE 1) of this thread
    const bool rlive = ri < Lr;
    const bool wlive = r0 + wq * 32 < Lr;        // warp-uniform
    // ---- per-row state ------------------------------------------------------------------------------------------------
    float lse2 = INFINITY, D = 0.f;              // SIDE 0
    GateW gw;
    const float *loc = nullptr;
    bool klive = false;                          // SIDE 1: key takes part
    float gb = 0.f, g0 = 0.f, g1 = 0.f, g2a = 0.f, g3 = 0.f, g4 = 0.f;
    if (SIDE == 0) {
      if (rlive) {
        const size_t r = ((size_t)b * a.H + h) * a.Lq + ri;
        lse2 = a.lse[r] * LOG2E;
        const uint4 *po = reinterpret_cast<const uint4 *>(a.o + ((size_t)b * a.Lq + ri) * E + h * DH);
        const uint4 *pd = reinterpret_cast<const uint4 *>(a.d_o + ((size_t)b * a.Lq + ri) * E + h * DH);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint4 x = __ldg(po + c), y = __ldg(pd + c);
          const __nv_bfloat162 *xa = reinterpret_cast<const __nv_bfloat162 *>(&x);
          const __nv_bfloat162 *ya = reinterpret_cast<const __nv_bfloat162 *>(&y);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float2 u = __bfloat1622float2(xa[i]), w = __bfloat1622float2(ya[i]);
            D = fmaf(u.x, w.x, fmaf(u.y, w.y, D));
          }
        }
        if (wg == 0) a.dvec[r] = D;
        gw.load(a.sw + ((size_t)b * a.Lq + ri) * (a.H * 6) + h * 6);
        loc = a.locs + ((size_t)b * a.Lq + ri) * (size_t)a.Lk * 5;
      }
    } else {
      klive = rlive && !(a.kpm != nullptr && a.kpm[(size_t)b * a.Lk + ri]);
    }
    const bool vec_loc = SIDE == 0 && (a.Lk & 3) == 0;

    for (int blk = 0; blk < nblk; ++blk, ++cbi) {
      const int nb = min(64, NC - blk * 64);     // columns of this block (multiple of 16)
      const int buf = cbi & 1;
      // ---- S_blk, dP_blk ---------------------------------------------------------------------------------------------
      if (tid < 32) {   // warp 0, converged: elect.sync picks the issuing lane (tc05.cuh: warp-converged issue)
        if (blk == 0) mbar_wait(&bars[2], ph_r);
        mbar_wait(&bars[buf], (uint32_t)(cbi >> 1) & 1u);
        fence_after_sync();
        const uint32_t aR1 = smem_u32(sR1), aR2 = smem_u32(sR2);
        const uint32_t aC1 = smem_u32(sC) + buf * 16384, aC2 = aC1 + 8192;
        const uint32_t idesc = idesc_kk(nb);
#pragma unroll
        for (int ks = 0; ks < DH / 16; ++ks)
          mma_bf16_e(tmem + COL_S, make_desc_sw128(aR1 + ks * 32), make_desc_sw128(aC1 + ks * 32), idesc, ks > 0);
#pragma unroll
        for (int ks = 0; ks < DH / 16; ++ks)
          mma_bf16_e(tmem + COL_DP, make_desc_sw128(aR2 + ks * 32), make_desc_sw128(aC2 + ks * 32), idesc, ks > 0);
        mma_commit_e(&bars[3]);
      }
      mbar_wait(&bars[3], ph_m);
      ph_m ^= 1u;
      fence_after_sync();
      // every MMA issued before this commit has retired: the OTHER buffer (read last by the previous block's output MMAs) is
      // free -> stream the next column block (of this row tile or the first of the next) behind the element-wise stage
      if (tid == 0) {
        if (blk + 1 < nblk) load_cblock(blk + 1, buf ^ 1);
        else if (r0 + 128 < Lr) load_cblock(0, buf ^ 1);
      }
      if (tid == 0 && blk == nblk - 1 && r0 + 128 < Lr) {  // row operands are free: fetch the next tile
        mbar_expect_tx(&bars[2], 2 * rows_bytes(r0 + 128, 8, Lr));
        tma_rows(sR1, &mR1, h, r0 + 128, 8, Lr, b, &bars[2]);
        tma_rows(sR2, &mR2, h, r0 + 128, 8, Lr, b, &bars[2]);
      }

      // ---- element-wise stage: 16-column units, alternating between the warpgroups ----------------------------------------
      if (wlive) {
#pragma unroll 1
        for (int u = (wg + blk) & 1; u < (nb >> 4); u += 2) {
          const int cl = u * 16;                 // column inside the block
          const int c0 = blk * 64 + cl;          // global column (key for SIDE 0, query for SIDE 1)
          uint32_t rs[16], rd[16];
          tmem_ld16_async(trow + COL_S + cl, rs);
          tmem_ld16_async(trow + COL_DP + cl, rd);
          if constexpr (SIDE == 0) {
            // query-side unit: per group of 4 keys the 20 geometry floats are loaded ONCE and serve both the gate
            // and the six gate-weight gradients
            tmem_wait16(rs);
            tmem_wait16(rd);
            float ds[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int cq = c0 + q * 4;
              float l[4][5];
              bool have[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) have[e] = loc != nullptr && cq + e < a.Lk;
              if (vec_loc) {
                if (have[0]) {
                  const float4 *l4 = reinterpret_cast<const float4 *>(loc + (size_t)cq * 5);
                  const float4 A = __ldg(l4), B2 = __ldg(l4 + 1), C = __ldg(l4 + 2), Dd = __ldg(l4 + 3), Ee = __ldg(l4 + 4);
                  l[0][0] = A.x; l[0][1] = A.y; l[0][2] = A.z; l[0][3] = A.w; l[0][4] = B2.x;
                  l[1][0] = B2.y; l[1][1] = B2.z; l[1][2] = B2.w; l[1][3] = C.x; l[1][4] = C.y;
                  l[2][0] = C.z; l[2][1] = C.w; l[2][2] = Dd.x; l[2][3] = Dd.y; l[2][4] = Dd.z;
                  l[3][0] = Dd.w; l[3][1] = Ee.x; l[3][2] = Ee.y; l[3][3] = Ee.z; l[3][4] = Ee.w;
                }
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e)
                  if (have[e]) {
                    const float *lp = loc + (size_t)(cq + e) * 5;
#pragma unroll
                    for (int t = 0; t < 5; ++t) l[e][t] = __ldg(lp + t);
                  }
              }
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int i = q * 4 + e;
                const float gli = have[e] ? gw.log2gate(l[e][0], l[e][1], l[e][2], l[e][3], l[e][4]) : 0.f;
                const float p = ex2f(fmaf(u2f(rs[i]), c2, kb[c0 + i]) - lse2 + gli);
                const float dsi = p * (u2f(rd[i]) - D);
                if (have[e] && gli > LOG2_CLAMP) {                       // clamp(sigmoid, 1e-6) inactive
                  const float dz = dsi * (1.0f - ex2f(gli));            // d log(sigmoid(z)) / dz = 1 - sigmoid(z)
                  gb += dz;
                  g0 = fmaf(dz, l[e][0], g0);
                  g1 = fmaf(dz, l[e][1], g1);
                  g2a = fmaf(dz, l[e][2], g2a);
                  g3 = fmaf(dz, l[e][3], g3);
                  g4 = fmaf(dz, l[e][4], g4);
                }
                ds[i] = dsi * a.scale;
              }
            }
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              uint32_t w[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) w[e] = pack_bf16(ds[hf * 8 + e * 2], ds[hf * 8 + e * 2 + 1]);
              *reinterpret_cast<uint4 *>(sG1 + tile_off(128, row, cl + hf * 8)) = make_uint4(w[0], w[1], w[2], w[3]);
            }
          } else {  // key-side unit
            float gl[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) gl[i] = 0.f;
            if (klive) {
#pragma unroll
              for (int i = 0; i < 16; ++i)
                if (c0 + i < a.Lq) {
                  const float *w = Ws + (c0 + i) * 6;
                  const GateW g{w[0], w[1], w[2], w[3], w[4], w[5]};
                  const float *l = a.locs + (((size_t)b * a.Lq + c0 + i) * a.Lk + ri) * 5;
                  gl[i] = g.log2gate(__ldg(l), __ldg(l + 1), __ldg(l + 2), __ldg(l + 3), __ldg(l + 4));
                }
            }
            tmem_wait16(rs);
            tmem_wait16(rd);
            float ds[16], pd[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float p = klive ? ex2f(fmaf(u2f(rs[i]), c2, -lse2s[c0 + i]) + gl[i]) : 0.f;
              ds[i] = p * (u2f(rd[i]) - Dv[c0 + i]) * a.scale;
              pd[i] = p;
            }
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              uint32_t w[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) w[e] = pack_bf16(ds[hf * 8 + e * 2], ds[hf * 8 + e * 2 + 1]);
              *reinterpret_cast<uint4 *>(sG1 + tile_off(128, row, cl + hf * 8)) = make_uint4(w[0], w[1], w[2], w[3]);
#pragma unroll
              for (int e = 0; e < 4; ++e) w[e] = pack_bf16(pd[hf * 8 + e * 2], pd[hf * 8 + e * 2 + 1]);
              *reinterpret_cast<uint4 *>(sG2 + tile_off(128, row, cl + hf * 8)) = make_uint4(w[0], w[1], w[2], w[3]);
            }
          }
        }
      }
      if (SIDE == 0 && blk == nblk - 1 && wg == 1) {
        float *r = red + row * 6;
        r[0] = gb; r[1] = g0; r[2] = g1; r[3] = g2a; r[4] = g3; r[5] = g4;
      }
      fence_proxy_async_smem();
      fence_before_sync();
      __syncthreads();

      // ---- accumulate the outputs over this block's columns (column operand read MN-major) -------------------------------
      if (tid < 32) {
        fence_after_sync();
        const uint32_t aG1 = smem_u32(sG1), aG2 = smem_u32(sG2);
        const uint32_t aC1 = smem_u32(sC) + buf * 16384, aC2 = aC1 + 8192;
        const uint32_t idesc = idesc_kmn(DH);
#pragma unroll 1
        for (int ks = 0; ks < (nb >> 4); ++ks) {
          mma_bf16_e(tmem + COL_O1, make_desc(aG1 + ks * 4096, 2048, 128), make_desc_sw128_mn(aC1 + ks * 2048), idesc,
                   (blk | ks) != 0);
          if (SIDE == 1)
            mma_bf16_e(tmem + COL_O2, make_desc(aG2 + ks * 4096, 2048, 128), make_desc_sw128_mn(aC2 + ks * 2048), idesc,
                     (blk | ks) != 0);
        }
        if (blk == nblk - 1) mma_commit_e(&bars[3]);
      }
    }
    mbar_wait(&bars[3], ph_m);
    ph_m ^= 1u;
    fence_after_sync();
    ph_r ^= 1u;

    // ---- epilogue ----------------------------------------------------------------------------------------------------------
    if (wlive) {
      if (SIDE == 0) {
        // dQ: each warpgroup stores 32 of the 64 columns
        uint32_t q0[16], q1[16];
        tmem_ld16_async(trow + COL_O1 + wg * 32, q0);
        tmem_ld16_async(trow + COL_O1 + wg * 32 + 16, q1);
        tmem_wait16(q0);
        tmem_wait16(q1);
        if (rlive) {
          __nv_bfloat16 *o = a.dq + ((size_t)b * a.Lq + ri) * a.d_rs + h * DH + wg * 32;
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            uint32_t w[4], z[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              w[e] = pack_bf16(u2f(q0[hf * 8 + e * 2]), u2f(q0[hf * 8 + e * 2 + 1]));
              z[e] = pack_bf16(u2f(q1[hf * 8 + e * 2]), u2f(q1[hf * 8 + e * 2 + 1]));
            }
            *reinterpret_cast<uint4 *>(o + hf * 8) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4 *>(o + 16 + hf * 8) = make_uint4(z[0], z[1], z[2], z[3]);
          }
          if (wg == 0 && a.dsw != nullptr) {
            const float *r = red + row * 6;
            float *g = a.dsw + ((size_t)b * a.Lq + ri) * (a.H * 6) + h * 6;
            g[0] = gb + r[0]; g[1] = g0 + r[1]; g[2] = g1 + r[2]; g[3] = g2a + r[3]; g[4] = g3 + r[4]; g[5] = g4 + r[5];
          }
        }
      } else {
        // warpgroup 0 stores dV (from P^T), warpgroup 1 stores dK (from scale * dS^T)
        __nv_bfloat16 *o = (wg == 0 ? a.dv : a.dk) + ((size_t)b * a.Lk + ri) * a.d_rs + h * DH;
        store_row64(trow + (wg == 0 ? COL_O2 : COL_O1), o, rlive);
      }
    }
    if (r0 + 128 < Lr) {
      fence_before_sync();
      __syncthreads();
      fence_after_sync();
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc_n(tmem, TMEM_COLS);
}

// ---- one-pass backward of the plain / dropout attention ---------------------------------------------------------------
// Tile rows = keys: a 128-key tile of K, V is staged once, Q and dO stream through the two-deep ring in blocks of 64
// queries.  Per block S^T, dP^T, P^T and dS^T are computed ONCE (one exp2 and one dropout decision per (query, key) pair)
// and serve all three products:
//   dV += (P o mask)^T dO,  dK += scale dS^T Q     (A = the staged tiles K-major, accumulated over the blocks in TMEM)
//   dQ[block] = scale dS K                          (A = the SAME scale dS^T tile read MN-major, B = the staged K tile)
// dQ lands in the S^T columns (free once the element-wise stage has read them) and is drained right away: written as bf16
// when the scene has one live key tile, otherwise summed over the key tiles in the CTA-owned fp32 scratch (B,H,Lq,64) —
// no atomics, one CTA owns its (scene, head).  Key tiles past the last unmasked key (`kend`) do no MMA and no
// element-wise work; their dK / dV rows are written as zeros.  TMEM 4 x 64 columns, shared memory <= 102 KB: two CTAs per
// SM.
template <bool DROP>
__global__ void __launch_bounds__(256, 2)
attn_bwd_fused_kernel(const __grid_constant__ CUtensorMap mK, const __grid_constant__ CUtensorMap mV,
                      const __grid_constant__ CUtensorMap mQ, const __grid_constant__ CUtensorMap mO, const BwdArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int NC = (a.Lq + 15) & ~15;          // queries rounded to the MMA granularity
  uint8_t *sK = smem;                        // [128][64] sw128   K tile
  uint8_t *sV = sK + 16384;                  // [128][64] sw128   V tile
  uint8_t *sC = sV + 16384;                  // 2 buffers x { [64][64] sw128 Q block, [64][64] sw128 dO block }
  uint8_t *sG1 = sC + 2 * 16384;             // [8][128][8] K-major   scale * dS^T (read MN-major as scale * dS for dQ)
  uint8_t *sG2 = sG1 + 16384;                // [8][128][8] K-major   dropped P^T
  float *lse2s = reinterpret_cast<float *>(sG2 + 16384);  // [NC] lse * log2(e) of each query (+inf past Lq)
  float *Dv = lse2s + NC;                    // [NC] D = rowsum(dO o O)
  uint32_t *rks = reinterpret_cast<uint32_t *>(Dv + NC);  // [NC] dropout row keys
  // barriers 0,1: query block landed in buffer 0 / 1, 2: key tile landed, 3: MMA done
  uint64_t *bars = reinterpret_cast<uint64_t *>(rks + NC);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 4);
  int *kend_s = reinterpret_cast<int *>(tmem_slot + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, wg = warp >> 2, wq = warp & 3;
  const int row = wq * 32 + lane;
  const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
  const int E = a.H * DH;
  const int nblk = (NC + 63) >> 6;
  auto load_cblock = [&](int cb, int buf) {
    const int nb = min(64, NC - cb * 64);
    mbar_expect_tx(&bars[buf], 2 * rows_bytes(cb * 64, nb >> 4, a.Lq));
    tma_rows(sC + buf * 16384, &mQ, h, cb * 64, nb >> 4, a.Lq, b, &bars[buf]);
    tma_rows(sC + buf * 16384 + 8192, &mO, h, cb * 64, nb >> 4, a.Lq, b, &bars[buf]);
  };
  auto load_ktile = [&](int r0) {
    mbar_expect_tx(&bars[2], 2 * rows_bytes(r0, 8, a.Lk));
    tma_rows(sK, &mK, h, r0, 8, a.Lk, b, &bars[2]);
    tma_rows(sV, &mV, h, r0, 8, a.Lk, b, &bars[2]);
  };

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    mbar_init(&bars[3], 1);
    mbar_fence_init();
    *kend_s = 0;
    tma_prefetch_desc(&mK);
    tma_prefetch_desc(&mV);
    tma_prefetch_desc(&mQ);
    tma_prefetch_desc(&mO);
  }
  __syncthreads();
  if (tid == 0) {   // the first tile's operands fly while the prologue runs
    load_cblock(0, 0);
    load_ktile(0);
  }
  if (warp == 1) tmem_alloc_n(tmem_slot, TMEM_COLS);
  // ---- prologue: kend, and the per-query vectors of every query -------------------------------------------------------------
  int last = 0;
  for (int c = tid; c < a.Lk; c += 256)
    if (!(a.kpm != nullptr && a.kpm[(size_t)b * a.Lk + c])) last = c + 1;
  last = __reduce_max_sync(0xffffffffu, last);
  if (lane == 0 && last > 0) atomicMax(kend_s, last);
  const unsigned long long seed = DROP ? attn::effective_seed(a.seed, a.seed_offset) : 0ull;
  for (int c = tid; c < NC; c += 256) {
    const bool live = c < a.Lq;
    const size_t r = ((size_t)b * a.H + h) * a.Lq + c;
    float D = 0.f;
    if (live) {
      const uint4 *po = reinterpret_cast<const uint4 *>(a.o + ((size_t)b * a.Lq + c) * E + h * DH);
      const uint4 *pd = reinterpret_cast<const uint4 *>(a.d_o + ((size_t)b * a.Lq + c) * E + h * DH);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint4 x = __ldg(po + j), y = __ldg(pd + j);
        const __nv_bfloat162 *xa = reinterpret_cast<const __nv_bfloat162 *>(&x);
        const __nv_bfloat162 *ya = reinterpret_cast<const __nv_bfloat162 *>(&y);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 u = __bfloat1622float2(xa[i]), w = __bfloat1622float2(ya[i]);
          D = fmaf(u.x, w.x, fmaf(u.y, w.y, D));
        }
      }
    }
    lse2s[c] = live ? a.lse[r] * LOG2E : INFINITY;
    Dv[c] = D;
    rks[c] = DROP ? drop_row_key(seed, r) : 0u;
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t trow = tmem + ((uint32_t)(wq * 32) << 16);
  const float c2 = a.scale * LOG2E;
  const int kend = *kend_s;
  const int nkt = (kend + 127) >> 7;         // key tiles holding an unmasked key
  uint32_t ph_r = 0, ph_m = 0;
  int cbi = 0;  // running query-block counter: buffer = cbi & 1, phase of its barrier = (cbi >> 1) & 1

  for (int t = 0; t < nkt; ++t) {
    const int r0 = t * 128;
    const int ri = r0 + row;                     // key of this thread
    const bool klive = ri < kend && !(a.kpm != nullptr && a.kpm[(size_t)b * a.Lk + ri]);
    const bool wlive = r0 + wq * 32 < kend;      // warp-uniform: the warp holds a key at or before the last live one
    const int nks = min(8, (kend - r0 + 15) >> 4);  // 16-key steps of dS K holding a live key
    if (!wlive) {
      // rows past kend take no part, but dK / dV of every row and dQ's sum over the tile read them: zero once per tile
#pragma unroll
      for (int c = 0; c < 64; c += 8) {
        *reinterpret_cast<uint4 *>(sG1 + tile_off(128, row, c)) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4 *>(sG2 + tile_off(128, row, c)) = make_uint4(0, 0, 0, 0);
      }
    }

    for (int blk = 0; blk < nblk; ++blk, ++cbi) {
      const int nb = min(64, NC - blk * 64);     // queries of this block (multiple of 16)
      const int buf = cbi & 1;
      // ---- S^T, dP^T of the block -----------------------------------------------------------------------------------------
      if (tid < 32) {   // warp 0, converged: elect.sync picks the issuing lane (tc05.cuh: warp-converged issue)
        if (blk == 0) mbar_wait(&bars[2], ph_r);
        mbar_wait(&bars[buf], (uint32_t)(cbi >> 1) & 1u);
        fence_after_sync();
        const uint32_t aK = smem_u32(sK), aV = smem_u32(sV);
        const uint32_t aC1 = smem_u32(sC) + buf * 16384, aC2 = aC1 + 8192;
        const uint32_t idesc = idesc_kk(nb);
#pragma unroll
        for (int ks = 0; ks < DH / 16; ++ks)
          mma_bf16_e(tmem + COL_S, make_desc_sw128(aK + ks * 32), make_desc_sw128(aC1 + ks * 32), idesc, ks > 0);
#pragma unroll
        for (int ks = 0; ks < DH / 16; ++ks)
          mma_bf16_e(tmem + COL_DP, make_desc_sw128(aV + ks * 32), make_desc_sw128(aC2 + ks * 32), idesc, ks > 0);
        mma_commit_e(&bars[3]);
      }
      mbar_wait(&bars[3], ph_m);
      ph_m ^= 1u;
      fence_after_sync();
      // every earlier MMA has retired: the other buffer is free -> stream the next query block behind the element-wise stage
      if (tid == 0) {
        if (blk + 1 < nblk) load_cblock(blk + 1, buf ^ 1);
        else if (t + 1 < nkt) load_cblock(0, buf ^ 1);
      }

      // ---- element-wise stage: 16-query units, alternating between the warpgroups ---------------------------------------------
      if (wlive) {
#pragma unroll 1
        for (int u = (wg + blk) & 1; u < (nb >> 4); u += 2) {
          const int cl = u * 16;                 // query inside the block
          const int c0 = blk * 64 + cl;          // query
          uint32_t rs[16], rd[16];
          tmem_ld16_async(trow + COL_S + cl, rs);
          tmem_ld16_async(trow + COL_DP + cl, rd);
          uint32_t hh[16];
          if (DROP) {
            // keys 2k and 2k+1 (adjacent lanes) share every pair hash: each lane hashes half of the queries and swaps
#pragma unroll
            for (int i = 0; i < 16; i += 2) {
              const uint32_t mine = drop_pair_hash(rks[c0 + i + (ri & 1)], (uint32_t)ri >> 1);
              const uint32_t other = __shfl_xor_sync(0xffffffffu, mine, 1);
              hh[i] = (ri & 1) ? other : mine;
              hh[i + 1] = (ri & 1) ? mine : other;
            }
          }
          tmem_wait16(rs);
          tmem_wait16(rd);
          float ds[16], pd[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float dpi = u2f(rd[i]);
            const float p = klive ? ex2f(fmaf(u2f(rs[i]), c2, -lse2s[c0 + i])) : 0.f;
            float m = 1.f;
            if (DROP) {
              m = drop_keep(hh[i], (uint32_t)ri, a.t16) ? a.inv_keep : 0.f;
              dpi *= m;
            }
            ds[i] = klive ? p * (dpi - Dv[c0 + i]) * a.scale : 0.f;   // exact 0 for masked keys (dQ sums over them)
            pd[i] = p * m;
          }
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) w[e] = pack_bf16(ds[hf * 8 + e * 2], ds[hf * 8 + e * 2 + 1]);
            *reinterpret_cast<uint4 *>(sG1 + tile_off(128, row, cl + hf * 8)) = make_uint4(w[0], w[1], w[2], w[3]);
#pragma unroll
            for (int e = 0; e < 4; ++e) w[e] = pack_bf16(pd[hf * 8 + e * 2], pd[hf * 8 + e * 2 + 1]);
            *reinterpret_cast<uint4 *>(sG2 + tile_off(128, row, cl + hf * 8)) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
      }
      fence_proxy_async_smem();
      fence_before_sync();
      __syncthreads();

      // ---- dK, dV accumulate over the blocks (query operands read MN-major); dQ of the block into the S^T columns ------------
      if (tid < 32) {
        fence_after_sync();
        const uint32_t aG1 = smem_u32(sG1), aG2 = smem_u32(sG2);
        const uint32_t aC1 = smem_u32(sC) + buf * 16384, aC2 = aC1 + 8192;
        const uint32_t idesc = idesc_kmn(DH);
#pragma unroll 1
        for (int ks = 0; ks < (nb >> 4); ++ks) {
          mma_bf16_e(tmem + COL_O1, make_desc(aG1 + ks * 4096, 2048, 128), make_desc_sw128_mn(aC1 + ks * 2048), idesc,
                     (blk | ks) != 0);
          mma_bf16_e(tmem + COL_O2, make_desc(aG2 + ks * 4096, 2048, 128), make_desc_sw128_mn(aC2 + ks * 2048), idesc,
                     (blk | ks) != 0);
        }
        // A = scale dS (M = queries, K = keys) is the dS^T tile read MN-major: no-swizzle core matrices of 8 queries x 8 keys,
        // 8-key groups 128 B apart (leading byte offset), 8-query groups 2048 B apart (stride byte offset).  M = 128: rows
        // 64..127 read the P^T tile behind it and land in TMEM lanes that are never read.
        const uint32_t aK = smem_u32(sK);
#pragma unroll 1
        for (int ks = 0; ks < nks; ++ks)
          mma_bf16_e(tmem + COL_S, make_desc(aG1 + ks * 256, 128, 2048), make_desc_sw128_mn(aK + ks * 2048),
                     idesc_kmn(DH) | (1u << 15), ks > 0);
        mma_commit_e(&bars[3]);
      }
      mbar_wait(&bars[3], ph_m);
      ph_m ^= 1u;
      fence_after_sync();
      if (tid == 0 && blk == nblk - 1 && t + 1 < nkt) load_ktile(r0 + 128);  // K, V are free: fetch the next tile

      // ---- drain dQ of the block: TMEM lanes 0..63 = its queries, each warpgroup takes 32 of the 64 columns ------------------
      if (wq < 2) {
        const int q = blk * 64 + row;
        uint32_t v0[16], v1[16];
        tmem_ld16_async(trow + COL_S + wg * 32, v0);
        tmem_ld16_async(trow + COL_S + wg * 32 + 16, v1);
        tmem_wait16(v0);
        tmem_wait16(v1);
        if (q < a.Lq) {
          float f[32];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            f[i] = u2f(v0[i]);
            f[16 + i] = u2f(v1[i]);
          }
          float4 *sc = reinterpret_cast<float4 *>(a.dvec + ((((size_t)b * a.H + h) * a.Lq + q) * DH + wg * 32));
          if (t > 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 x = sc[i];
              f[4 * i] += x.x; f[4 * i + 1] += x.y; f[4 * i + 2] += x.z; f[4 * i + 3] += x.w;
            }
          }
          if (t + 1 < nkt) {
#pragma unroll
            for (int i = 0; i < 8; ++i) sc[i] = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
          } else {
            __nv_bfloat16 *o = a.dq + ((size_t)b * a.Lq + q) * a.d_rs + h * DH + wg * 32;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              uint32_t w[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) w[e] = pack_bf16(f[i * 8 + e * 2], f[i * 8 + e * 2 + 1]);
              *reinterpret_cast<uint4 *>(o + i * 8) = make_uint4(w[0], w[1], w[2], w[3]);
            }
          }
        }
      }
      fence_before_sync();
      __syncthreads();   // the S^T columns are read: the next block's S MMA may overwrite them
      fence_after_sync();
    }
    ph_r ^= 1u;

    // ---- epilogue: warpgroup 0 stores dV (from the dropped P^T), warpgroup 1 stores dK (from scale * dS^T) ---------------------
    if (r0 + wq * 32 < a.Lk) {
      __nv_bfloat16 *o = (wg == 0 ? a.dv : a.dk) + ((size_t)b * a.Lk + ri) * a.d_rs + h * DH;
      store_row64(trow + (wg == 0 ? COL_O2 : COL_O1), o, ri < a.Lk);
    }
    if (t + 1 < nkt) {   // the next tile's first output MMAs overwrite dK / dV
      fence_before_sync();
      __syncthreads();
      fence_after_sync();
    }
  }

  // ---- key tiles past the last unmasked key: zero dK / dV rows; every key masked: dQ = 0 --------------------------------------
  for (int r = nkt * 128 + (tid & 127); r < a.Lk; r += 128) {
    uint4 *o = reinterpret_cast<uint4 *>((wg == 0 ? a.dv : a.dk) + ((size_t)b * a.Lk + r) * a.d_rs + h * DH);
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = make_uint4(0, 0, 0, 0);
  }
  if (nkt == 0) {
    for (int q = tid; q < a.Lq; q += 256) {
      uint4 *o = reinterpret_cast<uint4 *>(a.dq + ((size_t)b * a.Lq + q) * a.d_rs + h * DH);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = make_uint4(0, 0, 0, 0);
    }
    if (tid < 32) {   // retire the prologue's operand loads before the CTA exits
      mbar_wait(&bars[0], 0);
      mbar_wait(&bars[2], 0);
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc_n(tmem, TMEM_COLS);
}

template <bool DROP>
int launch_fused(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const CUtensorMap &mo,
                 const BwdArgs &a, cudaStream_t st) {
  const int NC = (a.Lq + 15) & ~15;
  const size_t smem = 6 * 16384 + (size_t)3 * NC * 4 + 64;
  constexpr size_t SMEM_MAX = 6 * 16384 + 3 * 384 * 4 + 64;
  auto kern = attn_bwd_fused_kernel<DROP>;
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
  kern<<<a.B * a.H, 256, smem, st>>>(mk, mv, mq, mo, a);
  return sv::after_launch();
}

template <int SIDE>
int launch_side(const CUtensorMap &r1, const CUtensorMap &r2, const CUtensorMap &c1, const CUtensorMap &c2,
                const BwdArgs &a, cudaStream_t st) {
  const int Lc = SIDE == 0 ? a.Lk : a.Lq;
  const int NC = (Lc + 15) & ~15;
  const size_t smem = 32768 + 32768 + (SIDE == 1 ? 32768 : 16384) + (size_t)(SIDE == 0 ? NC + 768 : 8 * NC) * 4 + 64;
  constexpr size_t SMEM_MAX = 32768 + 32768 + 32768 + 8 * 384 * 4 + 64;
  auto kern = attn_bwd_gated_kernel<SIDE>;
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
  kern<<<a.B * a.H, 256, smem, st>>>(r1, r2, c1, c2, a);
  return sv::after_launch();
}

int launch_gated(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const CUtensorMap &mo,
                 const BwdArgs &a, cudaStream_t st) {
  int rc = launch_side<0>(mq, mo, mk, mv, a, st);
  if (rc) return rc;
  return launch_side<1>(mk, mv, mq, mo, a, st);
}

}  // namespace

extern "C" int sv_attention_bwd_scratch_floats(int B, int H, int Lq, int Lk) {
  if (B < 0 || H < 1 || Lq < 1 || Lk < 1) return 0;
  // D of the gated kernel (B,H,Lq); with more than one key tile also the fp32 dQ partial sums (B,H,Lq,64)
  const long long n = (long long)B * H * Lq * (Lk > 128 ? attn::DH : 1);
  return n > 0x7fffffffLL ? -1 : (int)n;
}

extern "C" int sv_attention_bwd_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs, int k_rs,
                                     const void *v, long long v_bs, int v_rs, const void *o, const void *d_o,
                                     const unsigned char *key_padding_mask, const float *spatial_w,
                                     const float *pairwise_locs, const float *lse, int B, int H, int Lq, int Lk,
                                     float scale, void *dq, void *dk, void *dv, float *d_spatial_w, float *dvec,
                                     void *stream) {
  return sv_attention_bwd_dropout_bf16(q, q_bs, q_rs, k, k_bs, k_rs, v, v_bs, v_rs, o, d_o, key_padding_mask, spatial_w,
                                       pairwise_locs, lse, B, H, Lq, Lk, scale, dq, dk, dv, d_spatial_w, dvec, 0.f, 0ull,
                                       stream);
}

extern "C" int sv_attention_bwd_dropout_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs,
                                             int k_rs, const void *v, long long v_bs, int v_rs, const void *o,
                                             const void *d_o, const unsigned char *key_padding_mask,
                                             const float *spatial_w, const float *pairwise_locs, const float *lse, int B,
                                             int H, int Lq, int Lk, float scale, void *dq, void *dk, void *dv,
                                             float *d_spatial_w, float *dvec, float dropout_p, unsigned long long seed,
                                             void *stream) {
  return sv_attention_bwd_strided_bf16(q, q_bs, q_rs, k, k_bs, k_rs, v, v_bs, v_rs, o, d_o, key_padding_mask, spatial_w,
                                       pairwise_locs, lse, B, H, Lq, Lk, scale, dq, dk, dv, H * attn::DH, d_spatial_w, dvec,
                                       dropout_p, seed, stream);
}

extern "C" int sv_attention_bwd_strided_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs,
                                             int k_rs, const void *v, long long v_bs, int v_rs, const void *o,
                                             const void *d_o, const unsigned char *key_padding_mask,
                                             const float *spatial_w, const float *pairwise_locs, const float *lse, int B,
                                             int H, int Lq, int Lk, float scale, void *dq, void *dk, void *dv, int d_rs,
                                             float *d_spatial_w, float *dvec, float dropout_p, unsigned long long seed,
                                             void *stream) {
  if (d_rs < H * attn::DH || (d_rs % 8)) return SV_ERR_INVALID_ARG;
  if (!(dropout_p >= 0.f) || dropout_p >= 1.f) return SV_ERR_INVALID_ARG;
  if (B < 0 || H < 1 || Lq < 1 || Lk < 1 || Lq > 384 || Lk > 384) return SV_ERR_INVALID_ARG;
  if (B == 0) return SV_OK;
  if (!q || !k || !v || !o || !d_o || !lse || !dq || !dk || !dv || !dvec) return SV_ERR_INVALID_ARG;
  if ((q_rs % 8) || (k_rs % 8) || (v_rs % 8) || (q_bs % 8) || (k_bs % 8) || (v_bs % 8)) return SV_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(q) & 15) || (reinterpret_cast<uintptr_t>(k) & 15) ||
      (reinterpret_cast<uintptr_t>(v) & 15) || (reinterpret_cast<uintptr_t>(o) & 15) ||
      (reinterpret_cast<uintptr_t>(d_o) & 15) || (reinterpret_cast<uintptr_t>(dq) & 15) ||
      (reinterpret_cast<uintptr_t>(dk) & 15) || (reinterpret_cast<uintptr_t>(dv) & 15))
    return SV_ERR_INVALID_ARG;
  if (spatial_w && (!pairwise_locs || !d_spatial_w)) return SV_ERR_INVALID_ARG;
  if (spatial_w && dropout_p > 0.f) return SV_ERR_INVALID_ARG;
  BwdArgs a;
  a.o = (const __nv_bfloat16 *)o; a.d_o = (const __nv_bfloat16 *)d_o;
  a.kpm = key_padding_mask; a.sw = spatial_w; a.locs = pairwise_locs; a.lse = lse;
  a.B = B; a.H = H; a.Lq = Lq; a.Lk = Lk; a.scale = scale;
  a.dq = (__nv_bfloat16 *)dq; a.dk = (__nv_bfloat16 *)dk; a.dv = (__nv_bfloat16 *)dv;
  a.d_rs = d_rs;
  a.dsw = d_spatial_w; a.dvec = dvec;
  a.t16 = drop_threshold(dropout_p);
  a.inv_keep = 1.0f / (1.0f - dropout_p);
  a.seed = seed; a.seed_offset = sv::g_seed_offset;
  CUtensorMap mq, mk, mv, mo;
  int rc = make_map(&mq, q, B, Lq, H, q_rs, q_bs);
  if (rc) return rc;
  rc = make_map(&mk, k, B, Lk, H, k_rs, k_bs);
  if (rc) return rc;
  rc = make_map(&mv, v, B, Lk, H, v_rs, v_bs);
  if (rc) return rc;
  rc = make_map(&mo, d_o, B, Lq, H, H * DH, (long long)Lq * H * DH);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (spatial_w) return launch_gated(mq, mk, mv, mo, a, st);
  if (a.t16) return launch_fused<true>(mq, mk, mv, mo, a, st);
  return launch_fused<false>(mq, mk, mv, mo, a, st);
}
