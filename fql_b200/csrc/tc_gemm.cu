// tc_gemm.cu -- generic tcgen05 GEMM for one Dense layer (forward, dgrad or wgrad) with fused epilogues.
//
//   D[M,N] = A[M,K] * B[K,N]   bf16 operands from HBM/L2 via TMA (4-D tensor maps: inner, rows, head, seed), fp32 accumulate
//   in TMEM, 128x64 output tile per CTA, 64-deep K blocks, 9-stage mbarrier pipeline (216 KB in flight per SM).
//
// Both operands may be K-major ([rows][K] row-major) or MN-major ([K][rows] row-major); with SWIZZLE_128B TMA boxes of
// 64 inner elements both land in smem as the canonical UMMA atoms, so every GEMM of the MLP reads the SAME row-major bf16
// tensors with no transposed copies:
//   forward  Y = X W        A = X  [batch][in]  K-major     B = W  [in][out]   MN-major   (utils/networks.py:54)
//   dgrad    dX = dY W^T    A = dY [batch][out] K-major     B = W  [in][out]   K-major    (n = in, k = out)
//   wgrad    dW = X^T dY    A = X  [batch][in]  MN-major    B = dY [batch][out] MN-major  (k = batch)
// A B=256 layer becomes 2 x 8 = 16 CTAs on 16 SMs: at small batch the step is latency-bound and spreading one layer over
// many SMs beats keeping it on the 2 SMs a row-tile-persistent kernel would use (see DESIGN.md).
#include "step.cuh"
#include "tc_prims.cuh"

#include <stdlib.h>

using namespace tc;

namespace {

// A/B switch (rebuild): 1 = one issuer warp and ONE accumulator (a quarter of the epilogue's TMEM reads).  Measured after the uniform-issue
// change: batch 256 step 0.2288 vs 0.2297 ms (noise), batch 8192 step 1.260 vs 1.208 ms (the K = batch loops of the weight gradients want
// four issuers) -- the default stays 4.
#ifndef FQL_TC_GEMM_NACC
#define FQL_TC_GEMM_NACC 4
#endif
constexpr int BM = 128, BN = 64, BK = 64;
constexpr int A_STAGE = BM * BK * 2;  // 16 KB
constexpr int B_STAGE = BN * BK * 2;  //  8 KB
constexpr int STAGE = A_STAGE + B_STAGE;
constexpr int NSTAGE = 9;
constexpr int NACC = FQL_TC_GEMM_NACC;                // MMA-issuer warps = independent TMEM accumulators (k-step ks of every block -> warp ks)
constexpr int NTHREADS = 32 * (1 + NACC + 4);  // TMA warp, NACC MMA warps, 4 epilogue warps
constexpr int SMEM_BYTES = NSTAGE * STAGE + 1024 + 256;

struct GPtrB {
  void* base;
  long long s0, s1;
  int ld;
  template <typename T>
  __device__ __forceinline__ T* at(int g0, int g1) const {
    return base ? reinterpret_cast<T*>(base) + g0 * s0 + g1 * s1 : nullptr;
  }
};

struct TcGemmArgs {
  int M, N, K;
  int G0, G1;
  int a_mn, b_mn, a_bcast0, b_bcast0;
  int mode;
  GPtrB bias;    // fp32 [N]
  GPtrB out_f;   // fp32 [M][ld]
  GPtrB out_h;   // bf16 [M][ld]
  GPtrB out_z;   // bf16 [M][ld]   pre-activation copy (forward) for the backward's gelu'
  GPtrB zin;     // bf16 [M][ld]   pre-activation of the layer below (dgrad)
  GPtrB act;     // fp32 [M][A]    Euler state (in/out)
  GPtrB xb;      // bf16 [M][ld]   first-layer operand whose action/time columns the Euler step rewrites
  GPtrB target;  // fp32 [M][A]
  int F, A, step, n_steps, clip;
  int ksplit;    // > 1: the K range is split over blockIdx.z, partial tiles are added into a zeroed fp32 output (red.global.add)
  GPtrB ln_s, ln_b, dbias, wmaster, dln_s, dln_b;   // TC_MODE_WGRAD_LN (see the epilogue)
  unsigned long long* dbg;  // optional [CTA][8] globaltimer stamps (diagnostics)
};

__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ float gelu_fast(float x) {
  const float u = FQL_GELU_C * (x + FQL_GELU_A * x * x * x);
  return 0.5f * x * (1.0f + tanh_approx(u));
}
__device__ __forceinline__ float gelu_grad_fast(float x) {
  const float x2 = x * x;
  const float u = FQL_GELU_C * (x + FQL_GELU_A * x2 * x);
  const float th = tanh_approx(u);
  const float du = FQL_GELU_C * (1.0f + 3.0f * FQL_GELU_A * x2);
  return 0.5f * (1.0f + th) + 0.5f * x * (1.0f - th * th) * du;
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// MODE (the fused epilogue) is a template parameter: one instantiation carries one epilogue, which keeps the code a short-lived
// launch has to fetch small (the 4-epilogue kernel was 58 KB)
template <int MODE>
__global__ void __launch_bounds__(NTHREADS, 1) tc_gemm_kernel(const __grid_constant__ CUtensorMap mapA,
                                                         const __grid_constant__ CUtensorMap mapB, const TcGemmArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NSTAGE * STAGE);
  uint64_t* full = bars;
  uint64_t* empty = bars + NSTAGE;
  uint64_t* acc_full = bars + 2 * NSTAGE;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NSTAGE + 1);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform to ptxas as well
  const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
  const int zg = blockIdx.z / a.ksplit, kz = blockIdx.z % a.ksplit;
  const int g0 = zg % a.G0, g1 = zg / a.G0;
  const int nkb_all = (a.K + BK - 1) / BK;
  const int kb0 = (int)((long long)nkb_all * kz / a.ksplit), kb1 = (int)((long long)nkb_all * (kz + 1) / a.ksplit);
  const int nkb = kb1 - kb0;   // this CTA's K blocks [kb0, kb1)
  unsigned long long* dbg = a.dbg ? a.dbg + ((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 8 : nullptr;
  if (dbg && threadIdx.x == 0) dbg[0] = gtime();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA);
    tma_prefetch_desc(&mapB);
    for (int i = 0; i < NSTAGE; i++) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], NACC);
    }
    mbar_init(acc_full, NACC);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 64 * NACC);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (dbg && threadIdx.x == 0) dbg[1] = gtime();
  // Programmatic dependent launch: everything above overlapped the previous kernel's tail; from here on we read what it
  // wrote.  Let the next kernel in the stream start its own prologue right away.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp == 0) {
    // TMA producer: one thread's role, all 32 lanes run the loop and the instructions are predicated on the elected lane (uniform-register
    // operands; under `if (lane == 0)` every TMA / tcgen05 instruction sits in an ELECT + R2UR.BROADCAST waterfall, tc_prims.cuh)
    const bool el = elect_one();
    {
      const int ga0 = a.a_bcast0 ? 0 : g0, gb0 = a.b_bcast0 ? 0 : g0;
      for (int kb = 0; kb < nkb; kb++) {
        const int st = kb % NSTAGE;
        if (kb >= NSTAGE) mbar_wait_u(&empty[st], ((kb / NSTAGE) - 1) & 1);
        uint8_t* sa = smem + st * STAGE;
        uint8_t* sb = sa + A_STAGE;
        const int kc = (kb0 + kb) * BK;
        if (el) {
          mbar_expect_tx(&full[st], STAGE);
          if (!a.a_mn) {
            tma_load_4d(sa, &mapA, &full[st], kc, m0, ga0, g1);
          } else {
            tma_load_4d(sa, &mapA, &full[st], m0, kc, ga0, g1);
            tma_load_4d(sa + A_STAGE / 2, &mapA, &full[st], m0 + 64, kc, ga0, g1);
          }
          if (!a.b_mn) tma_load_4d(sb, &mapB, &full[st], kc, n0, gb0, g1);
          else tma_load_4d(sb, &mapB, &full[st], n0, kc, gb0, g1);
        }
      }
    }
  } else if (warp <= NACC) {
    // ---------------- MMA issuers ----------------
    // Warp w owns k-step w of every 64-wide K block and accumulates into its own 64 TMEM columns; the epilogue adds the four partial
    // accumulators.  (Round 1 measured ~80 ns per tcgen05.mma per issuing warp and split the K steps over four warps for it; most of
    // that was the waterfall around every instruction of an `if (lane == 0)` loop -- profiles/micro/mma_dual_bench.cu.)
    const bool el = elect_one();
    {
      const int mw = warp - 1;
      const uint32_t idesc = make_idesc_bf16(BM, BN, a.a_mn != 0, a.b_mn != 0);
      const uint64_t a_t = (a.a_mn ? make_smem_desc(0, A_STAGE / 2, 1024) : make_smem_desc(0, 16, 1024)) + (uint64_t)(mw * (a.a_mn ? (2048 >> 4) : (32 >> 4)));
      const uint64_t b_t = (a.b_mn ? make_smem_desc(0, B_STAGE, 1024) : make_smem_desc(0, 16, 1024)) + (uint64_t)(mw * (a.b_mn ? (2048 >> 4) : (32 >> 4)));
      const uint32_t s0 = smem_u32(smem) >> 4;
      const uint32_t tacc = __shfl_sync(0xffffffffu, tmem_base, 0) + mw * 64;
      int st = 0;
      uint32_t ph = 0;
      for (int kb = 0; kb < nkb; kb++) {
        mbar_wait_u(&full[st], ph);
        tc_fence_after();
        if (dbg && el && mw == 0 && kb == 0) dbg[2] = gtime();
        if (dbg && el && mw == 0 && kb == nkb - 1) dbg[3] = gtime();
        if (el) {
          if constexpr (NACC == 1)   // one issuer: the four k-steps of the block into ONE accumulator (the epilogue reads a quarter of the TMEM data)
            umma_bf16_x4(tacc, a_t + (uint64_t)(s0 + st * (STAGE >> 4)), b_t + (uint64_t)(s0 + st * (STAGE >> 4) + (A_STAGE >> 4)),
                         a.a_mn ? (2048 >> 4) : (32 >> 4), a.b_mn ? (2048 >> 4) : (32 >> 4), idesc, kb != 0);
          else
            umma_bf16(tacc, a_t + (uint64_t)(s0 + st * (STAGE >> 4)), b_t + (uint64_t)(s0 + st * (STAGE >> 4) + (A_STAGE >> 4)), idesc, kb != 0);
          umma_commit(&empty[st]);
        }
        if (++st == NSTAGE) { st = 0; ph ^= 1; }
      }
      if (el) umma_commit(acc_full);
    }
  } else {
    // ---------------- epilogue: thread per row, 64 accumulator columns ----------------
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int m = m0 + row;
    const bool valid = m < a.M;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const float* bias = a.bias.at<const float>(g0, g1);
    mbar_wait(acc_full, 0);
    tc_fence_after();
    if (dbg && threadIdx.x == 32 * (1 + NACC)) dbg[4] = gtime();
#pragma unroll 1
    for (int j = 0; j < 2; j++) {
      // one 32-column half at a time keeps the live set at 64 registers: partial accumulators of the NACC MMA warps are added
      uint32_t r[32];
      tmem_ld32(t_lane + j * 32, r);
      tmem_wait_ld();
#pragma unroll
      for (int acc = 1; acc < NACC; acc++) {
        uint32_t t[32];
        tmem_ld32(t_lane + acc * 64 + j * 32, t);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; i++) r[i] = __float_as_uint(__uint_as_float(r[i]) + __uint_as_float(t[i]));
      }
      const int nb = n0 + j * 32;
      if (!valid || nb >= a.N) continue;
      float v[32];
#pragma unroll
      for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]) + ((bias && nb + i < a.N) ? bias[nb + i] : 0.f);
      if constexpr (MODE == TC_MODE_WGRAD_LN) {
        // Weight gradient of a Dense layer that follows a LayerNorm, from G = xhat^T dZ (this tile, this K split):
        //   h = gamma * xhat + beta   =>   dW[m][n] = gamma_m G[m][n] + beta_m db[n]        (db = column sums of dZ, already reduced)
        //   dgamma_m = sum_n W[m][n] G[m][n],   dbeta_m = sum_n W[m][n] db[n]              (the LayerNorm parameter gradients:
        //   sum_rows dH * xhat and sum_rows dH with dH = dZ W^T, re-associated so that no dH ever exists in HBM)
        const float gam = a.ln_s.at<const float>(g0, g1)[m], bet = a.ln_b.at<const float>(g0, g1)[m];
        const float* db = a.dbias.at<const float>(g0, g1);
        const float* wrow = a.wmaster.at<const float>(g0, g1) + (int64_t)m * a.out_f.ld + nb;
        float* o = a.out_f.at<float>(g0, g1) + (int64_t)m * a.out_f.ld + nb;
        float dg = 0.f, dbt = 0.f;
        const bool vec = (nb + 32 <= a.N) && ((a.out_f.ld & 3) == 0);
        if (vec) {
          // 16-byte accesses: a thread owns 32 consecutive floats of its row (one 128-byte line of W and of dW)
#pragma unroll
          for (int i4 = 0; i4 < 8; i4++) {
            const float4 w4 = __ldg(reinterpret_cast<const float4*>(wrow) + i4);
            const float4 d4 = __ldg(reinterpret_cast<const float4*>(db + nb) + i4);
            const float wv[4] = {w4.x, w4.y, w4.z, w4.w}, dv[4] = {d4.x, d4.y, d4.z, d4.w};
            float ov[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
              const float gacc = __uint_as_float(r[i4 * 4 + k]);
              dg = fmaf(wv[k], gacc, dg);
              if (kz == 0) dbt = fmaf(wv[k], dv[k], dbt);
              ov[k] = gam * gacc + (kz == 0 ? bet * dv[k] : 0.f);
            }
            if (a.ksplit > 1) atomicAdd(reinterpret_cast<float4*>(o) + i4, make_float4(ov[0], ov[1], ov[2], ov[3]));   // red.global.add.v4.f32
            else reinterpret_cast<float4*>(o)[i4] = make_float4(ov[0], ov[1], ov[2], ov[3]);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; i++) {
            if (nb + i < a.N) {
              const float gacc = __uint_as_float(r[i]);    // no bias in this mode: v[] == the accumulator
              const float w = wrow[i];
              const float dbn = db[nb + i];
              dg = fmaf(w, gacc, dg);
              if (kz == 0) dbt = fmaf(w, dbn, dbt);
              const float dw = gam * gacc + (kz == 0 ? bet * dbn : 0.f);
              if (a.ksplit > 1) atomicAdd(o + i, dw);      // K split over CTAs: partial tiles add into the zeroed leaf
              else o[i] = dw;
            }
          }
        }
        atomicAdd(a.dln_s.at<float>(g0, g1) + m, dg);
        if (kz == 0) atomicAdd(a.dln_b.at<float>(g0, g1) + m, dbt);
      } else if constexpr (MODE == TC_MODE_STORE_F32) {
        float* o = a.out_f.at<float>(g0, g1) + (int64_t)m * a.out_f.ld + nb;
        if (a.ksplit > 1 && nb + 32 <= a.N && (a.out_f.ld & 3) == 0) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) atomicAdd(reinterpret_cast<float4*>(o + i), make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
        } else if (a.ksplit > 1) {
#pragma unroll
          for (int i = 0; i < 32; i++)
            if (nb + i < a.N) atomicAdd(o + i, v[i]);
        } else if (nb + 32 <= a.N && (a.out_f.ld & 3) == 0) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            float4 w4 = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
            if (a.clip) {
              w4.x = fminf(fmaxf(w4.x, -1.0f), 1.0f); w4.y = fminf(fmaxf(w4.y, -1.0f), 1.0f);
              w4.z = fminf(fmaxf(w4.z, -1.0f), 1.0f); w4.w = fminf(fmaxf(w4.w, -1.0f), 1.0f);
            }
            *reinterpret_cast<float4*>(o + i) = w4;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; i++)
            if (nb + i < a.N) o[i] = a.clip ? fminf(fmaxf(v[i], -1.0f), 1.0f) : v[i];
        }
      } else if constexpr (MODE == TC_MODE_FWD_HIDDEN) {
        // utils/networks.py:54-56: z = xW + b ; h = gelu(z).  N is a multiple of 64 on this path.
        uint4* oz = a.out_z.base ? reinterpret_cast<uint4*>(a.out_z.at<__nv_bfloat16>(g0, g1) + (int64_t)m * a.out_z.ld + nb) : nullptr;
        uint4* oh = reinterpret_cast<uint4*>(a.out_h.at<__nv_bfloat16>(g0, g1) + (int64_t)m * a.out_h.ld + nb);
#pragma unroll
        for (int c = 0; c < 4; c++) {
          if (oz) oz[c] = make_uint4(pack2(v[c * 8], v[c * 8 + 1]), pack2(v[c * 8 + 2], v[c * 8 + 3]), pack2(v[c * 8 + 4], v[c * 8 + 5]),
                                     pack2(v[c * 8 + 6], v[c * 8 + 7]));
          float h[8];
#pragma unroll
          for (int i = 0; i < 8; i++) h[i] = gelu_fast(v[c * 8 + i]);
          oh[c] = make_uint4(pack2(h[0], h[1]), pack2(h[2], h[3]), pack2(h[4], h[5]), pack2(h[6], h[7]));
        }
      } else if constexpr (MODE == TC_MODE_DGRAD_GELU) {
        // dZ_{l-1} = (dZ_l W_l^T) * gelu'(Z_{l-1})
        const uint4* zi = reinterpret_cast<const uint4*>(a.zin.at<const __nv_bfloat16>(g0, g1) + (int64_t)m * a.zin.ld + nb);
        uint4* oh = reinterpret_cast<uint4*>(a.out_h.at<__nv_bfloat16>(g0, g1) + (int64_t)m * a.out_h.ld + nb);
        float* of = a.out_f.base ? a.out_f.at<float>(g0, g1) + (int64_t)m * a.out_f.ld + nb : nullptr;
#pragma unroll
        for (int c = 0; c < 4; c++) {
          const uint4 zz = zi[c];
          const uint32_t zw[4] = {zz.x, zz.y, zz.z, zz.w};
          float d[8];
#pragma unroll
          for (int i = 0; i < 4; i++) {
            const __nv_bfloat162 zb = *reinterpret_cast<const __nv_bfloat162*>(&zw[i]);
            d[2 * i] = v[c * 8 + 2 * i] * gelu_grad_fast(__low2float(zb));
            d[2 * i + 1] = v[c * 8 + 2 * i + 1] * gelu_grad_fast(__high2float(zb));
          }
          oh[c] = make_uint4(pack2(d[0], d[1]), pack2(d[2], d[3]), pack2(d[4], d[5]), pack2(d[6], d[7]));
          if (of) {
            *reinterpret_cast<float4*>(of + c * 8) = make_float4(d[0], d[1], d[2], d[3]);
            *reinterpret_cast<float4*>(of + c * 8 + 4) = make_float4(d[4], d[5], d[6], d[7]);
          }
        }
      } else if constexpr (MODE == TC_MODE_EULER) {
        // agents/fql.py:166-170: a += v / flow_steps; next t; after the last step target = clip(a)
        float* act = a.act.at<float>(g0, g1) + (int64_t)m * a.A;
        __nv_bfloat16* xb = a.xb.at<__nv_bfloat16>(g0, g1) + (int64_t)m * a.xb.ld;
        float* tg = a.target.at<float>(g0, g1) + (int64_t)m * a.A;
        const float inv = (float)a.n_steps;
#pragma unroll
        for (int i = 0; i < 32; i++) {
          const int n = nb + i;
          if (n < a.A) {
            const float an = act[n] + v[i] / inv;
            act[n] = an;
            xb[a.F + n] = __float2bfloat16(an);
            if (a.step == a.n_steps - 1) tg[n] = fminf(fmaxf(an, -1.0f), 1.0f);
          }
        }
        if (j == 0) xb[a.F + a.A] = __float2bfloat16((float)((double)(a.step + 1) / (double)a.n_steps));
      }
    }
  }
  if (dbg && threadIdx.x == 32 * (1 + NACC)) dbg[5] = gtime();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 64 * NACC);
  if (dbg && threadIdx.x == 32) dbg[6] = gtime();
}

int make_map_4d(CUtensorMap* m, const TcOperand& o, uint32_t box_rows) {
  auto enc = get_encode();
  FQL_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
  const int g0 = o.g0 > 0 ? o.g0 : 1, g1 = o.g1 > 0 ? o.g1 : 1;
  cuuint64_t dims[4] = {(cuuint64_t)o.inner, (cuuint64_t)o.rows, (cuuint64_t)g0, (cuuint64_t)g1};
  const long long s0 = (g0 > 1) ? o.s0 : (long long)o.ld * o.rows, s1 = (g1 > 1) ? o.s1 : s0 * g0;
  cuuint64_t strides[3] = {(cuuint64_t)o.ld * 2, (cuuint64_t)s0 * 2, (cuuint64_t)s1 * 2};
  cuuint32_t box[4] = {64, box_rows, 1, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  FQL_REQUIRE(((uintptr_t)o.ptr & 15) == 0 && (strides[0] & 15) == 0 && (strides[1] & 15) == 0 && (strides[2] & 15) == 0,
              "TMA operand not 16-byte aligned (ptr %p ld %lld s0 %lld s1 %lld)", o.ptr, (long long)o.ld, s0, s1);
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(o.ptr), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FQL_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(4d) failed (%d): inner %d rows %d ld %lld g0 %d s0 %lld g1 %d s1 %lld", (int)r,
              o.inner, o.rows, (long long)o.ld, g0, s0, g1, s1);
  return 0;
}

GPtrB gp(const TcPtr& p) { return GPtrB{p.base, p.s0, p.s1, p.ld}; }

const int g_tc_pdl = []() {
  const char* e = getenv("FQL_B200_PDL");
  return (e && e[0] == '0') ? 0 : 1;
}();

}  // namespace

int tc_gemm(const TcGemmSpec& s, cudaStream_t st) {
  if (s.M <= 0 || s.N <= 0 || s.K <= 0) return 0;
  TcGemmArgs a;
  memset(&a, 0, sizeof(a));
  a.M = s.M; a.N = s.N; a.K = s.K; a.G0 = s.G0 > 0 ? s.G0 : 1; a.G1 = s.G1 > 0 ? s.G1 : 1;
  a.a_mn = s.a_mn; a.b_mn = s.b_mn; a.a_bcast0 = (s.A.g0 <= 1); a.b_bcast0 = (s.B.g0 <= 1);
  a.mode = s.mode;
  a.bias = gp(s.bias); a.out_f = gp(s.out_f); a.out_h = gp(s.out_h); a.out_z = gp(s.out_z); a.zin = gp(s.zin);
  a.act = gp(s.act); a.xb = gp(s.xb); a.target = gp(s.target);
  a.F = s.F; a.A = s.Adim; a.step = s.step; a.n_steps = s.n_steps; a.clip = s.clip;
  a.ksplit = s.ksplit > 1 ? s.ksplit : 1;
  {
    const int nkb_all = (s.K + BK - 1) / BK;
    if (a.ksplit > nkb_all) a.ksplit = nkb_all;
  }
  FQL_REQUIRE(a.ksplit == 1 || s.mode == TC_MODE_STORE_F32 || s.mode == TC_MODE_WGRAD_LN, "tc_gemm: split-K needs an accumulating fp32 epilogue");
  FQL_REQUIRE(!(a.ksplit > 1 && s.bias.base), "tc_gemm: split-K with a bias");
  a.ln_s = gp(s.ln_s); a.ln_b = gp(s.ln_b); a.dbias = gp(s.dbias); a.wmaster = gp(s.wmaster); a.dln_s = gp(s.dln_s); a.dln_b = gp(s.dln_b);
  if (s.mode == TC_MODE_WGRAD_LN)
    FQL_REQUIRE(s.ln_s.base && s.ln_b.base && s.dbias.base && s.wmaster.base && s.dln_s.base && s.dln_b.base && s.out_f.base && !s.bias.base,
                "tc_gemm: TC_MODE_WGRAD_LN needs the LayerNorm parameters, db, the master weights and zeroed outputs");
  a.dbg = reinterpret_cast<unsigned long long*>(s.dbg);
  if (s.mode == TC_MODE_FWD_HIDDEN || s.mode == TC_MODE_DGRAD_GELU)
    FQL_REQUIRE(s.N % 64 == 0 && s.out_h.base, "tc_gemm: hidden/dgrad epilogues need N %% 64 == 0 and a bf16 output");
  CUtensorMap mapA, mapB;
  FQL_TRY(make_map_4d(&mapA, s.A, s.a_mn ? 64 : BM));
  FQL_TRY(make_map_4d(&mapB, s.B, 64));
  void (*kern)(const CUtensorMap, const CUtensorMap, const TcGemmArgs) = nullptr;
  switch (s.mode) {
    case TC_MODE_STORE_F32: kern = tc_gemm_kernel<TC_MODE_STORE_F32>; break;
    case TC_MODE_FWD_HIDDEN: kern = tc_gemm_kernel<TC_MODE_FWD_HIDDEN>; break;
    case TC_MODE_DGRAD_GELU: kern = tc_gemm_kernel<TC_MODE_DGRAD_GELU>; break;
    case TC_MODE_EULER: kern = tc_gemm_kernel<TC_MODE_EULER>; break;
    case TC_MODE_WGRAD_LN: kern = tc_gemm_kernel<TC_MODE_WGRAD_LN>; break;
    default: FQL_REQUIRE(false, "tc_gemm: unknown epilogue mode %d", s.mode);
  }
  static bool attr_set[FQL_MAX_DEVICES][8] = {};
  const int dev = fql_current_device();
  if (!attr_set[dev][s.mode & 7]) {
    FQL_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    attr_set[dev][s.mode & 7] = true;
  }
  dim3 grid((s.N + BN - 1) / BN, (s.M + BM - 1) / BM, a.G0 * a.G1 * a.ksplit);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = dim3(NTHREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_tc_pdl ? 1 : 0;
  FQL_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, mapA, mapB, a));
  FQL_CHECK_LAUNCH();
  return 0;
}
