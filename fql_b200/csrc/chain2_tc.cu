// chain2_tc.cu -- the throughput variant of the fused MLP chain (hidden = 512): one CTA runs a whole MLP forward -- for
// compute_flow_actions (agents/fql.py:155-171) the whole Euler loop -- or the whole input-gradient chain of its backward on a
// 128-row tile, with the epilogue of one layer overlapped with the tensor-core work of the same and the next layer.  Used
// where seeds x 128-row tiles fill the GPU (batch >= 1024-ish, vectorised seeds: BASELINE configs 3 and 4); euler_cluster.cu
// keeps the batch-256 latency path, and narrower widths run layer by layer through tc_gemm (tc_path.cu).
//
// The 128 x 512 fp32 accumulator of a layer is all of an SM's TMEM, so it cannot be double-buffered across layers.  Instead a
// layer is issued as two N-halves (TMEM columns [0,256) and [256,512)) and the K loop of the second half runs while the
// epilogue drains the first:
//
//   MMA   (l,h0) k=0..7 | (l,h1) k=0..7            | (l+1,h0) k=0..3 ... k=4..7   | (l+1,h1) ...
//   EPI                 | (l,h0): blocks 0..3 of   | (l,h1): blocks 4..7          | (l+1,h0) ...
//                       |  A_{l+1}, each written   |  (all reads of A_l are done) |
//                       |  once (l,h1) has passed  |
//                       |  that K block (a_free)   |
//
// Activations live in one K-major SWIZZLE_128B operand buffer sA (8 blocks of [128][64] bf16): block kb of the next layer's
// input overwrites block kb of this layer's input as soon as the second half's MMAs have consumed it (tcgen05.commit ->
// a_free[kb]); the next layer's MMAs start on block kb as soon as it is written (a_ready[kb]).
//   warp 0      TMA producer: one box per 16 KB weight stage, straight from the Flax [in,out] bf16 shadow --
//               forward: [32 k][256 n] MN-major (3-D box 64 n x 32 k x 4 chunks, SWIZZLE_128B);
//               backward (W^T): [256 n = in][32 k = out] K-major (2-D box, SWIZZLE_64B).  No transposed weight copy exists.
//   warp 1      MMA issuer: tcgen05.mma kind::f16 M=128 N=256 K=16, two per stage
//   warps 2-9   epilogue: warp (q, p) owns TMEM lanes [32q, 32q+32) (one row per thread) and the 32-column chunks of parity p
//     forward            + bias, GELU(tanh.approx) [, LayerNorm: two passes, gelu stashed in TMEM, row sums exchanged between
//                        the two warps of a row through smem], bf16 re-pack into sA; saves for the backward: H (or xhat), gelu'
//     backward           dZ_{l-1} = (dZ_l W_l^T) * gelu'(Z_{l-1})                          (utils/networks.py:54-56 reversed)
//     backward, LN       dZ_{l-1} = gelu' * rstd * (dx - mean(dx) - xhat * mean(dx * xhat)),  dx = gamma * (dZ_l W_l^T)
//                        from the forward's bf16 xhat / gelu' saves: no transcendental, no fp32 round trip through HBM
// Reference arithmetic: utils/networks.py:34-61 (MLP), :153-195 (Value), :198-235 (ActorVectorField); jax.grad of the same.
#include "step.cuh"
#include "tc_prims.cuh"

using namespace tc;

namespace {

constexpr int TILE_M = 128;
constexpr int KB_BYTES = TILE_M * 128;       // one K block of an A operand: [128 rows][64 bf16]
constexpr int KS = 32;                       // k rows of weights per pipeline stage
constexpr int NHALF = 256;                   // accumulator columns per N-half
constexpr int CHUNK_BYTES = KS * 128;        // one 64-column chunk of a forward stage
constexpr int STAGE_BYTES = 4 * CHUNK_BYTES; // 16 KB: [4 chunks][32 k][64 n] (forward) / [256 n][32 k] (backward)
constexpr int MAX_A = 32;
constexpr int EPI_WARPS = 8;
constexpr int C2_THREADS = 32 * (2 + EPI_WARPS);
constexpr int HID = 512;
constexpr int NKB = HID / 64;

enum { C2_FWD = 0, C2_EULER = 1, C2_FWD_LN = 2, C2_BWD = 3, C2_BWD_LN = 4 };

#ifdef FQL_C2_DBG   // diagnostics build only (make EXTRA=-DFQL_C2_DBG): per-stage %globaltimer stamps of CTA 0, iteration FQL_C2_DBG_N
__device__ unsigned long long g_c2_dbg[256];
__device__ __forceinline__ unsigned long long c2_gt() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#ifndef FQL_C2_DBG_N
#define FQL_C2_DBG_N 7
#endif
#define C2_STAMP(cond, idx) do { if ((cond) && el && blockIdx.x == 0) g_c2_dbg[idx] = c2_gt(); } while (0)
#else
#define C2_STAMP(cond, idx) do { } while (0)
#endif

struct Chain2Args {
  int NL, K0, K0pad, out_dim;
  int P, S, E, M, tiles;
  int x_row0[FQL_MAXP], x_rows_s, x_rows_e;
  int w_row[FQL_MAXP][FQL_MAXL], w_rows_s;   // rows of HID elements in the shadow
  int wl_row[FQL_MAXP], wl_rows_s;           // rows of 64 elements in the shadow (padded last layer)
  const float* params;
  long long arena;
  long long off_b[FQL_MAXP][FQL_MAXL], off_lns[FQL_MAXP][FQL_MAXL], off_lnb[FQL_MAXP][FQL_MAXL];
  float* out;            // forward: [G][Mcap][out_dim]; backward: dX0 [G][Mcap][K0] (optional)
  float* Zs[FQL_MAXL];   // forward: fp32 pre-activations (the per-layer LayerNorm backward of the small-batch schedule)
  float* mu[FQL_MAXL];
  float* rstd[FQL_MAXL]; // forward: out; backward (LN): in
  void* Hb[FQL_MAXL];    // forward: bf16 activations (wgrad operands); LN + XHb given: not written
  void* Zb[FQL_MAXL];    // forward: bf16 pre-activations (small-batch backward)
  void* DGb[FQL_MAXL];   // bf16 gelu'(z): forward out, backward in
  void* XHb[FQL_MAXL];   // bf16 xhat = (gelu(z) - mu) * rstd (LayerNorm): forward out, backward in (also the wgrad operand)
  void* dZb[FQL_MAXL];   // backward: bf16 dZ_l out (wgrad operands), optional
  int Mcap, r0;
  int Mcap_dz;           // backward: row capacity per group of the dZb buffers
  int save_mask;         // forward: bit p set = problem p writes its Hb / Zb / DGb / XHb / Zs / mu / rstd saves
  int n_steps, F, A;
  const float* a0;
  float* target;
  int clip_out;
  int nstage, w3d, has_dx0;
};

// gelu(x) and gelu'(x) with one MUFU tanh
__device__ __forceinline__ void gelu_and_grad(float x, float& g, float& dg) {
  const float x2 = x * x;
  const float th = tanh_approx(FQL_GELU_C * (x + FQL_GELU_A * x2 * x));
  g = 0.5f * x * (1.0f + th);
  dg = 0.5f * (1.0f + th) + 0.5f * x * (1.0f - th * th) * (FQL_GELU_C * (1.0f + 3.0f * FQL_GELU_A * x2));
}
__device__ __forceinline__ float gelu_fast(float x) {
  // 0.5 x (1 + tanh(c (x + a x^3))) as 3 FMUL + 2 FFMA + 1 MUFU
  const float p = fmaf(x * x, FQL_GELU_C * FQL_GELU_A, FQL_GELU_C);
  const float hx = 0.5f * x;
  return fmaf(hx, tanh_approx(x * p), hx);
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// 32 consecutive values of one row -> bf16, into block (j >> 1) of the K-major SWIZZLE_128B operand buffer (and optionally HBM)
__device__ __forceinline__ void store_chunk(uint8_t* sA, int row, int j, const float (&h)[32], __nv_bfloat16* gdst) {
  uint8_t* blk = sA + (j >> 1) * KB_BYTES;
  const int c0 = (j & 1) * 4;
#pragma unroll
  for (int c = 0; c < 4; c++) {
    const uint4 v = make_uint4(pack_bf16(h[c * 8 + 0], h[c * 8 + 1]), pack_bf16(h[c * 8 + 2], h[c * 8 + 3]),
                               pack_bf16(h[c * 8 + 4], h[c * 8 + 5]), pack_bf16(h[c * 8 + 6], h[c * 8 + 7]));
    *reinterpret_cast<uint4*>(blk + sw128_off(row, c0 + c)) = v;
    if (gdst) *reinterpret_cast<uint4*>(gdst + c * 8) = v;
  }
}
__device__ __forceinline__ void store_bf16x32(__nv_bfloat16* gdst, const float (&h)[32]) {
#pragma unroll
  for (int c = 0; c < 4; c++)
    *reinterpret_cast<uint4*>(gdst + c * 8) = make_uint4(pack_bf16(h[c * 8 + 0], h[c * 8 + 1]), pack_bf16(h[c * 8 + 2], h[c * 8 + 3]),
                                                         pack_bf16(h[c * 8 + 4], h[c * 8 + 5]), pack_bf16(h[c * 8 + 6], h[c * 8 + 7]));
}
// 32 consecutive bf16 of one row from HBM (zeros for rows outside the problem)
__device__ __forceinline__ void load_bf16x32(const __nv_bfloat16* src, bool valid, uint4 (&q)[4]) {
#pragma unroll
  for (int c = 0; c < 4; c++) q[c] = valid ? __ldg(reinterpret_cast<const uint4*>(src) + c) : make_uint4(0u, 0u, 0u, 0u);
}
__device__ __forceinline__ float bf16_at(const uint4 (&q)[4], int i) {
  const uint32_t w = (&q[i >> 3].x)[(i >> 1) & 3];
  return __uint_as_float((i & 1) ? (w & 0xffff0000u) : (w << 16));
}

template <int MODE>
__global__ void __launch_bounds__(C2_THREADS, 1) mlp_chain2_kernel(const __grid_constant__ CUtensorMap mapX,
                                                              const __grid_constant__ CUtensorMap mapW,
                                                              const __grid_constant__ CUtensorMap mapWL,
                                                              const __grid_constant__ CUtensorMap mapW0, const Chain2Args a) {
  constexpr bool LN = (MODE == C2_FWD_LN || MODE == C2_BWD_LN);
  constexpr bool BWD = (MODE == C2_BWD || MODE == C2_BWD_LN);
  constexpr bool EULER = (MODE == C2_EULER);
  constexpr int NPAR = BWD ? (LN ? 1 : 0) : (LN ? 3 : 1);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int nkb_x = BWD ? 1 : a.K0pad / 64;
  uint8_t* sA = smem;                                   // [8][16 KB]
  uint8_t* sX = sA + NKB * KB_BYTES;                    // [nkb_x][16 KB]
  uint8_t* sW = sX + nkb_x * KB_BYTES;                  // [nstage][16 KB]
  float* sPar = reinterpret_cast<float*>(sW + a.nstage * STAGE_BYTES);  // [2][NPAR][512]: bias (, LN scale, LN bias) / LN scale
  float* sStat = sPar + 2 * NPAR * HID;                 // [2][128][2] row sums of the two column parities (LayerNorm)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStat + (LN ? 2 * TILE_M * 2 : 0));
  uint64_t* full = bars;                 // [8]
  uint64_t* empty = bars + 8;            // [8]
  uint64_t* a_ready = bars + 16;         // [8]  block kb of the next layer's input is in sA            (8 epilogue warps)
  uint64_t* a_free = bars + 24;          // [4]  the second half's MMAs are done with block kb of sA    (tcgen05.commit)
  uint64_t* acc_full = bars + 28;        // [2]  half h of the accumulator is complete                  (tcgen05.commit)
  uint64_t* acc_free = bars + 30;        // [2]  half h of the accumulator has been read                (8 epilogue warps)
  uint64_t* x_full = bars + 32;
  uint64_t* x_ready = bars + 33;         //      the Euler update of the resident first-layer operand    (8 epilogue warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 34);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x % a.tiles, g = blockIdx.x / a.tiles;
  const int e = g % a.E, s = (g / a.E) % a.S, p = g / (a.E * a.S);
  // iterations of one pass: forward = NL layers (the last one narrow); backward = NL-1 hidden dZ's (+ the narrow dX0 GEMM)
  const int NIT = BWD ? (a.NL - 1 + (a.has_dx0 ? 1 : 0)) : a.NL;
  const int NWIDE = a.NL - 1;            // iterations with a 512-wide output
  const int total = a.n_steps * NIT;
  const int ntail = BWD ? a.K0pad : 64;  // output width of the narrow tail iteration

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapX);
    tma_prefetch_desc(&mapW);
    tma_prefetch_desc(&mapWL);
    if (BWD) tma_prefetch_desc(&mapW0);
    for (int i = 0; i < 8; i++) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
      mbar_init(&a_ready[i], EPI_WARPS);
    }
    for (int i = 0; i < 4; i++) mbar_init(&a_free[i], 1);
    for (int i = 0; i < 2; i++) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_free[i], EPI_WARPS);
    }
    mbar_init(x_full, 1);
    mbar_init(x_ready, EPI_WARPS);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // The TMA producer and the MMA issuer are ONE thread each, but all 32 lanes of their warps run the loops (waits, descriptor arithmetic):
  // warp-uniform control flow keeps the descriptors in uniform registers, and only the instruction itself is predicated on the elected
  // lane.  With the whole loop under `if (lane == 0)` ptxas wraps every tcgen05.mma / tcgen05.commit / TMA in an ELECT + 5 R2UR.BROADCAST
  // waterfall: 178 instead of 139 ns per two MMAs + commit in isolation (profiles/micro/mma_dual_bench.cu), 370 ns per stage in here.
  bool el = false;     // set at the top of the two roles' branches (straight from elect.sync: ptxas then knows the region is single-lane)
  // the producer and the issuer spin with the wait loop inside the asm block (see mbar_wait_u)
  auto wait_x = [&](uint64_t* bar, uint32_t parity) {
    if (warp <= 1) mbar_wait_u(bar, parity);
    else mbar_wait(bar, parity);
  };
  auto load2d = [&](void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    if (el) tma_load_2d(dst, m, bar, c0, c1);
  };

  if (warp == 0) {
    // ================= TMA producer =================
    el = elect_one();
    {
      if (el) mbar_expect_tx(x_full, nkb_x * KB_BYTES);
      const int xrow = a.x_row0[p] + s * a.x_rows_s + e * a.x_rows_e + tile * TILE_M;
      for (int kb = 0; kb < nkb_x; kb++) load2d(sX + kb * KB_BYTES, &mapX, x_full, kb * 64, xrow);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int n = 0; n < total; n++, it = (it + 1 == NIT) ? 0 : it + 1) {
        if (it < NWIDE) {
          // forward: layer it, K rows of W_it; backward: W^T of layer NL-1-it (it = 0: the padded last layer, K = 64 outputs)
          const int l = BWD ? a.NL - 1 - it : it;
          const int K = BWD ? (it == 0 ? 64 : HID) : (it == 0 ? a.K0 : HID);
          const int nst = (K + KS - 1) / KS;
          const int row0 = BWD ? (it == 0 ? a.wl_row[p] + s * a.wl_rows_s + e * HID : a.w_row[p][l] + s * a.w_rows_s + e * HID)
                               : a.w_row[p][l] + s * a.w_rows_s + e * K;
          for (int h = 0; h < 2; h++)
            for (int ks = 0; ks < nst; ks++) {
              wait_x(&empty[stage], phase ^ 1);
              C2_STAMP(n == FQL_C2_DBG_N && MODE == C2_EULER, 128 + h * 16 + ks);
              uint8_t* dst = sW + stage * STAGE_BYTES;
              if (el) mbar_expect_tx(&full[stage], STAGE_BYTES);
              if (BWD) {     // the 256 input rows of the half
                load2d(dst, it == 0 ? &mapWL : &mapW, &full[stage], ks * KS, row0 + h * NHALF);
              } else if (a.w3d) {
                if (el) tma_load_3d(dst, &mapW, &full[stage], 0, row0 + ks * KS, h * 4);
              } else {       // the 4 chunks of 64 output columns of the half
                for (int c = 0; c < 4; c++)
                  load2d(dst + c * CHUNK_BYTES, &mapW, &full[stage], (h * 4 + c) * 64, row0 + ks * KS);
              }
              if (++stage == a.nstage) { stage = 0; phase ^= 1; }
            }
        } else {
          // narrow tail: forward = the last Dense (padded to 64 outputs); backward = dX0 = dZ_0 W_0^T (K0pad inputs)
          const int row0 = BWD ? a.w_row[p][0] + s * a.w_rows_s + e * a.K0 : a.wl_row[p] + s * a.wl_rows_s + e * HID;
          for (int ks = 0; ks < HID / KS; ks++) {
            wait_x(&empty[stage], phase ^ 1);
            // backward: the K0pad input rows; forward: the padded 64 output columns
            if (el) mbar_expect_tx(&full[stage], BWD ? a.K0pad * 64 : KS * 128);
            if (BWD) load2d(sW + stage * STAGE_BYTES, &mapW0, &full[stage], ks * KS, row0);
            else load2d(sW + stage * STAGE_BYTES, &mapWL, &full[stage], 0, row0 + ks * KS);
            if (++stage == a.nstage) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    el = elect_one();
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);   // uniform copy (the shared-memory load is per-thread to ptxas)
    const uint32_t idesc_h = make_idesc_bf16(TILE_M, NHALF, false, !BWD);
    const uint32_t idesc_t = make_idesc_bf16(TILE_M, ntail, false, !BWD);
    auto mma = [&](uint32_t d, uint64_t ad, uint64_t bd, uint32_t id, uint32_t acc) {
      if (el) umma_bf16(d, ad, bd, id, acc);
    };
    auto mma_x2 = [&](uint32_t d, uint64_t ad, uint64_t bd, uint64_t as, uint64_t bs, uint32_t id, uint32_t acc) {
      if (el) umma_bf16_x2(d, ad, bd, as, bs, id, acc);
    };
    auto commit = [&](uint64_t* bar) {
      if (el) umma_commit(bar);
    };
    const uint64_t a_t = make_smem_desc(0, 16, 1024);
    // B: forward MN-major (64-column chunks CHUNK_BYTES apart, 8-k groups 1024 B apart); backward K-major rows of 64 B (SWIZZLE_64B)
    const uint64_t b_t = BWD ? make_smem_desc_sw64(0, 16, 512) : make_smem_desc(0, CHUNK_BYTES, 1024);
    const uint64_t b_k16 = BWD ? 2 : (2048 >> 4);      // second 16-k step inside a stage
    const uint32_t sa0 = smem_u32(sA) >> 4, sx0 = smem_u32(sX) >> 4, sw0 = smem_u32(sW) >> 4;
    int stage = 0;
    uint32_t phase = 0;
    int n_ar = 0, n_xr = 0;
    int uses[2] = {0, 0};
    int it = 0;
    for (int n = 0; n < total; n++, it = (it + 1 == NIT) ? 0 : it + 1) {
      if (it == 0) {
        if (n == 0) wait_x(x_full, 0);
        else wait_x(x_ready, (n_xr++) & 1);
        tc_fence_after();
      }
      if (it < NWIDE) {
        const int K = BWD ? (it == 0 ? 64 : HID) : (it == 0 ? a.K0 : HID);
        const int nst = (K + KS - 1) / KS;
        const uint32_t abase = (it == 0) ? sx0 : sa0;
        for (int h = 0; h < 2; h++) {
          if (uses[h] > 0) {
            wait_x(&acc_free[h], (uses[h] - 1) & 1);
            tc_fence_after();
          }
          const uint32_t tacc = tmem_u + h * NHALF;
          for (int ks = 0; ks < nst; ks++) {
            const int kb = ks >> 1;
            if (it > 0 && h == 0 && (ks & 1) == 0) {
              wait_x(&a_ready[kb], (n_ar - 1) & 1);
              tc_fence_after();
            }
            C2_STAMP(n == FQL_C2_DBG_N && MODE == C2_EULER, h * 48 + ks * 3 + 0);
            wait_x(&full[stage], phase);
            tc_fence_after();
            C2_STAMP(n == FQL_C2_DBG_N && MODE == C2_EULER, h * 48 + ks * 3 + 1);
            const uint64_t adesc = a_t + (uint64_t)(abase + kb * (KB_BYTES >> 4) + (ks & 1) * 4);
            const uint64_t bdesc = b_t + (uint64_t)(sw0 + stage * (STAGE_BYTES >> 4));
            // both K steps of a stage from ONE asm block (the second descriptor pair is a constant add inside PTX)
            if (K - ks * KS > 16) mma_x2(tacc, adesc, bdesc, 2, b_k16, idesc_h, ks > 0);
            else mma(tacc, adesc, bdesc, idesc_h, ks > 0);
            commit(&empty[stage]);
            C2_STAMP(n == FQL_C2_DBG_N && MODE == C2_EULER, h * 48 + ks * 3 + 2);
            if (++stage == a.nstage) { stage = 0; phase ^= 1; }
            if (it > 0 && h == 1 && (ks & 1) == 1 && kb < 4) commit(&a_free[kb]);
          }
          commit(&acc_full[h]);
          uses[h]++;
        }
        n_ar++;
      } else {
        if (uses[0] > 0) {
          wait_x(&acc_free[0], (uses[0] - 1) & 1);
          tc_fence_after();
        }
        for (int ks = 0; ks < HID / KS; ks++) {
          const int kb = ks >> 1;
          if ((ks & 1) == 0) wait_x(&a_ready[kb], (n_ar - 1) & 1);
          wait_x(&full[stage], phase);
          tc_fence_after();
          const uint64_t adesc = a_t + (uint64_t)(sa0 + kb * (KB_BYTES >> 4) + (ks & 1) * 4);
          const uint64_t bdesc = b_t + (uint64_t)(sw0 + stage * (STAGE_BYTES >> 4));
          mma_x2(tmem_u, adesc, bdesc, 2, b_k16, idesc_t, ks > 0);
          commit(&empty[stage]);
          if (++stage == a.nstage) { stage = 0; phase ^= 1; }
        }
        commit(&acc_full[0]);
        uses[0]++;
      }
    }
  } else {
    // ================= epilogue =================
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    const int pw = (warp - 2) >> 2;               // column-chunk parity of this warp
    const int row = q * 32 + lane;
    const int grow = tile * TILE_M + row;
    const bool valid = grow < a.M;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const int et = threadIdx.x - 64;              // 0..255
    const int64_t gidx = (int64_t)((p * a.S + s) * a.E + e) * a.Mcap + a.r0 + grow;
    const int64_t gidx_dz = (int64_t)(s * a.E + e) * a.Mcap_dz + grow;
    const bool vsave = valid && ((a.save_mask >> p) & 1);
    int nf[2] = {0, 0};
    int n_af = 0;
    float act[MAX_A];
    if (EULER) {
#pragma unroll
      for (int c = 0; c < MAX_A; c++) act[c] = (pw == 0 && valid && c < a.A) ? a.a0[((int64_t)s * a.M + grow) * a.A + c] : 0.f;
    }
    int it = 0, step = 0;
    for (int n = 0; n < total; n++, it = (it + 1 == NIT) ? 0 : it + 1, step += (it == 0)) {
      const bool wide = it < NWIDE;
      const int l = BWD ? a.NL - 2 - it : it;     // forward: the layer computed; backward: the hidden layer whose dZ is produced
      float* par = sPar + (n & 1) * NPAR * HID;
      if (NPAR > 0) {  // stage this iteration's per-column parameters while the MMAs run
        if (!BWD) {
          const int N = wide ? HID : a.out_dim;
          const float* b = a.params + (int64_t)s * a.arena + a.off_b[p][l] + (int64_t)e * N;
          for (int i = et; i < N; i += 32 * EPI_WARPS) par[i] = b[i];
          if (LN && wide) {
            const float* sc = a.params + (int64_t)s * a.arena + a.off_lns[p][l] + (int64_t)e * HID;
            const float* bi = a.params + (int64_t)s * a.arena + a.off_lnb[p][l] + (int64_t)e * HID;
            for (int i = et; i < HID; i += 32 * EPI_WARPS) {
              par[HID + i] = sc[i];
              par[2 * HID + i] = bi[i];
            }
          }
        } else if (wide) {
          const float* sc = a.params + (int64_t)s * a.arena + a.off_lns[p][l] + (int64_t)e * HID;
          for (int i = et; i < HID; i += 32 * EPI_WARPS) par[i] = sc[i];
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      uint32_t r[32];
      if (wide) {
        const int64_t rowoff = gidx * HID;
        if (MODE == C2_FWD || MODE == C2_EULER) {
          __nv_bfloat16* Hb = (vsave && a.Hb[l]) ? reinterpret_cast<__nv_bfloat16*>(a.Hb[l]) + rowoff : nullptr;
          __nv_bfloat16* Zb = (vsave && a.Zb[l]) ? reinterpret_cast<__nv_bfloat16*>(a.Zb[l]) + rowoff : nullptr;
          __nv_bfloat16* DGb = (vsave && a.DGb[l]) ? reinterpret_cast<__nv_bfloat16*>(a.DGb[l]) + rowoff : nullptr;
          for (int h = 0; h < 2; h++) {
            wait_x(&acc_full[h], (nf[h]++) & 1);
            tc_fence_after();
            // software-pipelined TMEM reads: chunk jj + 1 is in flight while chunk jj is evaluated (two register buffers)
            uint32_t rb[2][32];
            tmem_ld32(t_lane + (h * 8 + pw) * 32, rb[0]);
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
              const int j = h * 8 + jj * 2 + pw;
              tmem_wait_ld();
              if (jj < 3) tmem_ld32(t_lane + (j + 2) * 32, rb[(jj + 1) & 1]);
              const uint32_t (&rr)[32] = rb[jj & 1];
              float hv[32];
              if (DGb) {        // z -> gelu(z) for the next layer, gelu'(z) saved for the backward (the large-batch backward reads no z)
                float dv[32];
#pragma unroll
                for (int i = 0; i < 32; i++) gelu_and_grad(__uint_as_float(rr[i]) + par[j * 32 + i], hv[i], dv[i]);
                store_bf16x32(DGb + j * 32, dv);
              } else {
                float zv[32];
#pragma unroll
                for (int i = 0; i < 32; i++) {
                  zv[i] = __uint_as_float(rr[i]) + par[j * 32 + i];
                  hv[i] = gelu_fast(zv[i]);
                }
                if (Zb) store_bf16x32(Zb + j * 32, zv);
              }
              // block j >> 1 of sA still holds this layer's input until the second half's MMAs have consumed it
              if (it > 0 && h == 0) wait_x(&a_free[j >> 1], n_af & 1);
              store_chunk(sA, row, j, hv, Hb ? Hb + j * 32 : nullptr);
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) mbar_arrive(&a_ready[j >> 1]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_free[h]);
          }
          if (it > 0) n_af++;
        } else if (MODE == C2_BWD) {
          const __nv_bfloat16* DGb = reinterpret_cast<const __nv_bfloat16*>(a.DGb[l]) + rowoff;
          __nv_bfloat16* dZb = (valid && a.dZb[l]) ? reinterpret_cast<__nv_bfloat16*>(a.dZb[l]) + gidx_dz * HID : nullptr;
          for (int h = 0; h < 2; h++) {
            uint4 dq[4];
            load_bf16x32(DGb + (h * 8 + pw) * 32, valid, dq);   // the first chunk's gelu' is fetched while the MMAs run
            wait_x(&acc_full[h], (nf[h]++) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int jj = 0; jj < 4; jj++) {
              const int j = h * 8 + jj * 2 + pw;
              tmem_ld32(t_lane + j * 32, r);
              tmem_wait_ld();
              float hv[32];
#pragma unroll
              for (int i = 0; i < 32; i++) hv[i] = __uint_as_float(r[i]) * bf16_at(dq, i);
              if (jj < 3) load_bf16x32(DGb + (j + 2) * 32, valid, dq);
              if (it > 0 && h == 0) wait_x(&a_free[j >> 1], n_af & 1);
              store_chunk(sA, row, j, hv, dZb ? dZb + j * 32 : nullptr);
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) mbar_arrive(&a_ready[j >> 1]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_free[h]);
          }
          if (it > 0) n_af++;
        } else if (MODE == C2_FWD_LN) {
          // pass 1: g = gelu(z) stashed back into TMEM in place, row sums in registers
          float* Zs = (vsave && a.Zs[l]) ? a.Zs[l] + rowoff : nullptr;
          __nv_bfloat16* DGb = (vsave && a.DGb[l]) ? reinterpret_cast<__nv_bfloat16*>(a.DGb[l]) + rowoff : nullptr;
          float s1 = 0.f, s2 = 0.f;
          for (int h = 0; h < 2; h++) {
            wait_x(&acc_full[h], (nf[h]++) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int jj = 0; jj < 4; jj++) {
              const int j = h * 8 + jj * 2 + pw;
              tmem_ld32(t_lane + j * 32, r);
              tmem_wait_ld();
#pragma unroll
              for (int i = 0; i < 32; i++) r[i] = __float_as_uint(__uint_as_float(r[i]) + par[j * 32 + i]);   // z = xW + b
              if (Zs) {
#pragma unroll
                for (int i = 0; i < 32; i += 4)
                  *reinterpret_cast<float4*>(Zs + j * 32 + i) =
                      make_float4(__uint_as_float(r[i]), __uint_as_float(r[i + 1]), __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
              }
              if (DGb) {
                float dv[32];
#pragma unroll
                for (int i = 0; i < 32; i++) {
                  float gv;
                  gelu_and_grad(__uint_as_float(r[i]), gv, dv[i]);
                  s1 += gv;
                  s2 += gv * gv;
                  r[i] = __float_as_uint(gv);
                }
                store_bf16x32(DGb + j * 32, dv);
              } else {
#pragma unroll
                for (int i = 0; i < 32; i++) {
                  const float gv = gelu_fast(__uint_as_float(r[i]));
                  s1 += gv;
                  s2 += gv * gv;
                  r[i] = __float_as_uint(gv);
                }
              }
              tmem_st32(t_lane + j * 32, r);
            }
          }
          tmem_wait_st();
          sStat[(pw * TILE_M + row) * 2 + 0] = s1;
          sStat[(pw * TILE_M + row) * 2 + 1] = s2;
          asm volatile("bar.sync 1, 256;" ::: "memory");
          s1 += sStat[((pw ^ 1) * TILE_M + row) * 2 + 0];
          s2 += sStat[((pw ^ 1) * TILE_M + row) * 2 + 1];
          const float inv_n = 1.0f / (float)HID;
          const float mu = s1 * inv_n;
          const float var = fmaxf(0.f, s2 * inv_n - mu * mu);
          const float rstd = rsqrtf(var + FQL_LN_EPS);
          if (vsave && pw == 0) {
            if (a.mu[l]) a.mu[l][gidx] = mu;
            if (a.rstd[l]) a.rstd[l][gidx] = rstd;
          }
          // pass 2: normalise, re-pack.  Every MMA of this layer has completed (acc_full[1] was observed): sA is free.
          __nv_bfloat16* Hb = (vsave && a.Hb[l]) ? reinterpret_cast<__nv_bfloat16*>(a.Hb[l]) + rowoff : nullptr;
          __nv_bfloat16* XHb = (vsave && a.XHb[l]) ? reinterpret_cast<__nv_bfloat16*>(a.XHb[l]) + rowoff : nullptr;
          for (int h = 0; h < 2; h++) {
#pragma unroll 1
            for (int jj = 0; jj < 4; jj++) {
              const int j = h * 8 + jj * 2 + pw;
              tmem_ld32(t_lane + j * 32, r);
              tmem_wait_ld();
              float hv[32];
#pragma unroll
              for (int i = 0; i < 32; i++) hv[i] = (__uint_as_float(r[i]) - mu) * rstd;       // xhat
              if (XHb) store_bf16x32(XHb + j * 32, hv);
#pragma unroll
              for (int i = 0; i < 32; i++) hv[i] = hv[i] * par[HID + j * 32 + i] + par[2 * HID + j * 32 + i];
              store_chunk(sA, row, j, hv, Hb ? Hb + j * 32 : nullptr);
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) mbar_arrive(&a_ready[j >> 1]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_free[h]);
          }
        } else {  // C2_BWD_LN
          const __nv_bfloat16* XHb = reinterpret_cast<const __nv_bfloat16*>(a.XHb[l]) + rowoff;
          const __nv_bfloat16* DGb = reinterpret_cast<const __nv_bfloat16*>(a.DGb[l]) + rowoff;
          __nv_bfloat16* dZb = (valid && a.dZb[l]) ? reinterpret_cast<__nv_bfloat16*>(a.dZb[l]) + gidx_dz * HID : nullptr;
          const float rstd = valid ? a.rstd[l][gidx] : 0.f;
          // pass 1: dx = gamma * dH stashed in TMEM, row sums of dx and dx * xhat
          float m1 = 0.f, m2 = 0.f;
          for (int h = 0; h < 2; h++) {
            uint4 xq[4];
            load_bf16x32(XHb + (h * 8 + pw) * 32, valid, xq);
            wait_x(&acc_full[h], (nf[h]++) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int jj = 0; jj < 4; jj++) {
              const int j = h * 8 + jj * 2 + pw;
              tmem_ld32(t_lane + j * 32, r);
              tmem_wait_ld();
#pragma unroll
              for (int i = 0; i < 32; i++) {
                const float dx = __uint_as_float(r[i]) * par[j * 32 + i];
                m1 += dx;
                m2 = fmaf(dx, bf16_at(xq, i), m2);
                r[i] = __float_as_uint(dx);
              }
              if (jj < 3) load_bf16x32(XHb + (j + 2) * 32, valid, xq);
              tmem_st32(t_lane + j * 32, r);
            }
          }
          tmem_wait_st();
          sStat[(pw * TILE_M + row) * 2 + 0] = m1;
          sStat[(pw * TILE_M + row) * 2 + 1] = m2;
          asm volatile("bar.sync 1, 256;" ::: "memory");
          m1 = (m1 + sStat[((pw ^ 1) * TILE_M + row) * 2 + 0]) * (1.0f / (float)HID);
          m2 = (m2 + sStat[((pw ^ 1) * TILE_M + row) * 2 + 1]) * (1.0f / (float)HID);
          // pass 2: dz = gelu' * rstd * (dx - m1 - xhat * m2)       (flax LayerNorm backward, fast-variance form)
          for (int h = 0; h < 2; h++) {
#pragma unroll 1
            for (int jj = 0; jj < 4; jj++) {
              const int j = h * 8 + jj * 2 + pw;
              uint4 xq[4], dq[4];
              load_bf16x32(XHb + j * 32, valid, xq);
              load_bf16x32(DGb + j * 32, valid, dq);
              tmem_ld32(t_lane + j * 32, r);
              tmem_wait_ld();
              float hv[32];
#pragma unroll
              for (int i = 0; i < 32; i++) hv[i] = bf16_at(dq, i) * rstd * (__uint_as_float(r[i]) - m1 - bf16_at(xq, i) * m2);
              store_chunk(sA, row, j, hv, dZb ? dZb + j * 32 : nullptr);
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) mbar_arrive(&a_ready[j >> 1]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_free[h]);
          }
        }
      } else {
        // narrow tail
        wait_x(&acc_full[0], (nf[0]++) & 1);
        tc_fence_after();
        if (BWD) {
          // dX0 = dZ_0 W_0^T: columns [0, K0) in fp32 (the actor loss only reads the action columns)
          for (int j = pw; j * 32 < a.K0; j += 2) {
            tmem_ld32(t_lane + j * 32, r);
            tmem_wait_ld();
            if (valid && a.out) {
              float* o = a.out + gidx_dz * a.K0 + j * 32;
#pragma unroll
              for (int c = 0; c < 32; c++)
                if (j * 32 + c < a.K0) o[c] = __uint_as_float(r[c]);
            }
          }
        } else if (pw == 0) {
          // last Dense (linear): out_dim <= 32 columns of the padded N = 64 accumulator
          tmem_ld32(t_lane, r);
          tmem_wait_ld();
          if (!EULER) {
            if (valid && a.out) {
              float* o = a.out + gidx * a.out_dim;
#pragma unroll
              for (int c = 0; c < MAX_A; c++)
                if (c < a.out_dim) {
                  float v = __uint_as_float(r[c]) + par[c];
                  if (a.clip_out) v = fminf(fmaxf(v, -1.0f), 1.0f);
                  o[c] = v;
                }
            }
          } else {
            // Euler step (agents/fql.py:166-169): a += v / flow_steps, next t = (step+1)/flow_steps, written straight into the bf16
            // first-layer operand tile that stays resident in smem for the whole integration
            const float inv = (float)a.n_steps;
#pragma unroll
            for (int c = 0; c < MAX_A; c++)
              if (c < a.A) {
                act[c] += (__uint_as_float(r[c]) + par[c]) / inv;
                const int col = a.F + c;
                *reinterpret_cast<__nv_bfloat16*>(sX + (col >> 6) * KB_BYTES + sw128_off(row, (col & 63) >> 3) + (col & 7) * 2) = __float2bfloat16(act[c]);
              }
            {
              const int col = a.F + a.A;
              *reinterpret_cast<__nv_bfloat16*>(sX + (col >> 6) * KB_BYTES + sw128_off(row, (col & 63) >> 3) + (col & 7) * 2) =
                  __float2bfloat16((float)((double)(step + 1) / (double)a.n_steps));
            }
            if (step == a.n_steps - 1 && valid) {
#pragma unroll
              for (int c = 0; c < MAX_A; c++)
                if (c < a.A) a.target[((int64_t)s * a.M + grow) * a.A + c] = fminf(fmaxf(act[c], -1.0f), 1.0f);
            }
          }
        }
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&acc_free[0]);
          if (EULER) mbar_arrive(x_ready);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

#ifdef FQL_C2_DBG
}  // namespace
extern "C" int fql_debug_chain2_stamps(unsigned long long* host_out, int n) {
  FQL_CHECK_CUDA(cudaMemcpyFromSymbol(host_out, g_c2_dbg, (n < 256 ? n : 256) * sizeof(unsigned long long)));
  return 0;
}
namespace {
#endif

// The weight matrix [rows][512] as a 3-D tensor (64 n, row, chunk of 64 n): one box {64, KS, 4} lands a whole [4][KS][64] stage.
// The chunk dimension's stride (128 B) is smaller than the row dimension's (1024 B); returns false when the driver refuses that.
bool make_map_w3d(CUtensorMap* m, const void* base, uint64_t rows) {
  auto enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[3] = {64, rows, HID / 64};
  cuuint64_t strides[2] = {HID * 2, 128};
  cuuint32_t box[3] = {64, KS, 4};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

int fill_common(Chain2Args& a, const FqlDims* d, const Layout& L, int P, const int* net, int M, int Mcap0, int r0_in) {
  const NetView& n0 = L.net[net[0]];
  memset(&a, 0, sizeof(a));
  a.NL = n0.n_layers; a.K0 = n0.in_dim; a.K0pad = (int)round_up64(n0.in_dim, 64); a.out_dim = n0.out_dim;
  a.P = P; a.S = d->num_seeds; a.E = n0.ens; a.M = M; a.tiles = (M + TILE_M - 1) / TILE_M;
  FQL_REQUIRE(a.NL >= 3 && a.NL <= FQL_MAXL && a.out_dim <= MAX_A && a.K0pad <= 128, "tc_mlp_chain2: %d layers / output width %d / input width %d",
              a.NL, a.out_dim, a.K0);
  const int64_t seed_elems = tc_shadow_seed_elems(d, L);
  FQL_REQUIRE(seed_elems % HID == 0 && L.arena % 64 == 0, "shadow layout not row aligned");
  a.x_rows_s = Mcap0;
  a.w_rows_s = (int)(seed_elems / HID);
  a.wl_rows_s = (int)(seed_elems / 64);
  for (int p = 0; p < P; p++) {
    const NetView& nv = L.net[net[p]];
    a.x_row0[p] = p * a.S * Mcap0 + r0_in;
    for (int l = 0; l < nv.n_layers; l++) {
      a.w_row[p][l] = (int)(nv.off_w[l] / HID);
      a.off_b[p][l] = nv.off_b[l];
      a.off_lns[p][l] = nv.off_lns[l];
      a.off_lnb[p][l] = nv.off_lnb[l];
    }
    int64_t wl = L.arena;
    for (int t = 0; t < net[p]; t++) wl += (int64_t)L.net[t].ens * HID * 64;
    a.wl_row[p] = (int)(wl / 64);
  }
  a.arena = L.arena;
  a.n_steps = 1; a.F = d->obs_dim; a.A = d->action_dim;
  a.save_mask = 0xff;
  return 0;
}

template <int MODE>
int launch_chain2(const Chain2Args& a0, int nkb_x, int npar, bool ln, const CUtensorMap& mapX, const CUtensorMap& mapW, const CUtensorMap& mapWL,
                  const CUtensorMap& mapW0, cudaStream_t st) {
  Chain2Args a = a0;
  const int fixed = (NKB + nkb_x) * KB_BYTES + 2 * npar * HID * 4 + (ln ? 2 * TILE_M * 2 * 4 : 0) + 512 + 1024;
  int nstage = (232448 - fixed) / STAGE_BYTES;
  if (nstage > 8) nstage = 8;
  static const int cap = getenv("FQL_B200_CHAIN2_STAGES") ? atoi(getenv("FQL_B200_CHAIN2_STAGES")) : 0;   // diagnostics: shallower weight ring
  if (cap >= 2 && nstage > cap) nstage = cap;
  FQL_REQUIRE(nstage >= 2, "not enough shared memory for the weight pipeline");
  a.nstage = nstage;
  const int smem = fixed + nstage * STAGE_BYTES;
  auto kern = mlp_chain2_kernel<MODE>;
  static bool attr_set[FQL_MAX_DEVICES] = {};
  const int dev = fql_current_device();
  if (!attr_set[dev]) {
    FQL_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    attr_set[dev] = true;
  }
  const int grid = a.tiles * a.P * a.S * a.E;
  kern<<<grid, C2_THREADS, smem, st>>>(mapX, mapW, mapWL, mapW0, a);
  FQL_CHECK_LAUNCH();
  return 0;
}

}  // namespace

int tc_mlp_chain2(const TcChainSpec& f, cudaStream_t st) {
  const FqlDims* d = f.d;
  const Layout& L = *f.L;
  FQL_TRY(tc_supported(d));
  FQL_REQUIRE(d->hidden == HID, "tc_mlp_chain2 is built for hidden = 512");
  const NetView& n0 = L.net[f.net[0]];
  Chain2Args a;
  FQL_TRY(fill_common(a, d, L, f.P, f.net, f.M, f.Mcap0, f.r0_in));
  a.params = f.params;
  a.Mcap = f.buf ? f.buf->Mcap : f.M; a.r0 = f.r0;
  if (f.buf) {
    a.out = f.buf->out;
    for (int l = 0; l + 1 < n0.n_layers; l++) {
      a.Zs[l] = (f.save && n0.ln) ? f.buf->Z[l] : nullptr;
      a.mu[l] = (f.save && n0.ln) ? f.buf->mu[l] : nullptr;
      a.rstd[l] = (f.save && n0.ln) ? f.buf->rstd[l] : nullptr;
      a.Hb[l] = f.Hb ? f.Hb[l] : nullptr;
    }
    FQL_REQUIRE(!(f.save && !n0.ln), "tc_mlp_chain2: fp32 saves are for LayerNorm networks; actors save bf16 Z / H");
  } else {
    for (int l = 0; l + 1 < n0.n_layers; l++) {
      a.Hb[l] = f.Hb ? f.Hb[l] : nullptr;
      a.Zb[l] = f.Zb ? f.Zb[l] : nullptr;
    }
    if (f.Mcap_override > 0) a.Mcap = f.Mcap_override;
  }
  for (int l = 0; l + 1 < n0.n_layers; l++) {
    if (f.DGb) {            // large-batch backward: gelu' (and xhat for LayerNorm networks) instead of the pre-activations
      a.DGb[l] = f.DGb[l];
      a.Zb[l] = nullptr;
      a.Zs[l] = nullptr;
    }
    if (f.XHb) { a.XHb[l] = f.XHb[l]; a.Hb[l] = nullptr; }
  }
  if (f.save_mask) a.save_mask = f.save_mask;
  if (f.out_override) a.out = f.out_override;
  a.n_steps = f.n_steps > 0 ? f.n_steps : 1; a.a0 = f.a0; a.target = f.target;
  a.clip_out = f.clip_out;
  const bool euler = a.n_steps > 1;
  FQL_REQUIRE(!euler || (a.a0 && a.target && f.P == 1 && a.E == 1 && !n0.ln), "Euler chain needs a0/target and a single actor network");

  CUtensorMap mapX, mapW, mapWL;
  const int64_t x_rows = (int64_t)f.P * a.S * f.Mcap0;
  FQL_TRY(make_map_2d(&mapX, f.X0b, a.K0pad, x_rows, 64, TILE_M));
  static const bool no3d = getenv("FQL_B200_CHAIN2_W3D") && getenv("FQL_B200_CHAIN2_W3D")[0] == '0';
  a.w3d = (!no3d && make_map_w3d(&mapW, f.shadow, (uint64_t)a.S * a.w_rows_s)) ? 1 : 0;
  if (!a.w3d) FQL_TRY(make_map_2d(&mapW, f.shadow, HID, (uint64_t)a.S * a.w_rows_s, 64, KS));
  FQL_TRY(make_map_2d(&mapWL, f.shadow, 64, (uint64_t)a.S * a.wl_rows_s, 64, KS));
  const int nkb_x = a.K0pad / 64;
  if (n0.ln) return launch_chain2<C2_FWD_LN>(a, nkb_x, 3, true, mapX, mapW, mapWL, mapWL, st);
  if (euler) return launch_chain2<C2_EULER>(a, nkb_x, 1, false, mapX, mapW, mapWL, mapWL, st);
  return launch_chain2<C2_FWD>(a, nkb_x, 1, false, mapX, mapW, mapWL, mapWL, st);
}

// The input-gradient chain of one network's backward on M rows per group: dZ_{NL-2} ... dZ_0 as bf16 (operands of the weight
// gradients) and optionally dX0 = dZ_0 W_0^T in fp32 -- from the forward's bf16 gelu' (and xhat / rstd) saves.
int tc_mlp_chain2_backward(const TcChain2BwdSpec& f, cudaStream_t st) {
  const FqlDims* d = f.d;
  const Layout& L = *f.L;
  FQL_TRY(tc_supported(d));
  FQL_REQUIRE(d->hidden == HID, "tc_mlp_chain2_backward is built for hidden = 512");
  const NetView& nv = L.net[f.net];
  Chain2Args a;
  const int nets[1] = {f.net};
  FQL_TRY(fill_common(a, d, L, 1, nets, f.M, f.M * nv.ens, 0));
  a.params = f.params;
  a.Mcap = f.Mcap; a.r0 = f.r0; a.Mcap_dz = f.Mcap_dz > 0 ? f.Mcap_dz : f.M;
  // dOut: bf16 [S][E][M][64] zero padded; one 128-row tile of group (s, e) starts at row ((s * E + e) * M + tile * 128)
  a.x_row0[0] = 0; a.x_rows_s = f.M * nv.ens; a.x_rows_e = f.M;
  for (int l = 0; l + 1 < nv.n_layers; l++) {
    a.DGb[l] = f.DGb[l];
    a.XHb[l] = nv.ln ? f.XHb[l] : nullptr;
    a.rstd[l] = nv.ln ? f.rstd[l] : nullptr;
    a.dZb[l] = f.dZb ? f.dZb[l] : nullptr;
    FQL_REQUIRE(a.DGb[l] && (!nv.ln || (a.XHb[l] && a.rstd[l])), "tc_mlp_chain2_backward: missing forward saves of layer %d", l);
  }
  a.has_dx0 = f.dX0 ? 1 : 0;
  a.out = f.dX0;
  CUtensorMap mapX, mapW, mapWL, mapW0;
  FQL_TRY(make_map_2d(&mapX, f.dOutb, 64, (uint64_t)a.S * nv.ens * f.M, 64, TILE_M));
  FQL_TRY(make_map_2d(&mapW, f.shadow, HID, (uint64_t)a.S * a.w_rows_s, KS, NHALF, CU_TENSOR_MAP_SWIZZLE_64B));
  FQL_TRY(make_map_2d(&mapWL, f.shadow, 64, (uint64_t)a.S * a.wl_rows_s, KS, NHALF, CU_TENSOR_MAP_SWIZZLE_64B));
  FQL_TRY(make_map_2d(&mapW0, f.shadow, HID, (uint64_t)a.S * a.w_rows_s, KS, a.K0pad, CU_TENSOR_MAP_SWIZZLE_64B));
  if (nv.ln) return launch_chain2<C2_BWD_LN>(a, 1, 1, true, mapX, mapW, mapWL, mapW0, st);
  return launch_chain2<C2_BWD>(a, 1, 0, false, mapX, mapW, mapWL, mapW0, st);
}
