// euler_cluster.cu -- compute_flow_actions (agents/fql.py:155-171) as ONE persistent thread-block-cluster kernel.
//
// The Euler integration is the longest dependent chain of an update: flow_steps x 5 Dense layers on the same rows.  At
// batch 256 that is only two 128-row tiles, so the per-row-tile fused kernel (chain2_tc.cu) leaves 146 SMs idle and a
// kernel-per-layer schedule pays a launch + pipeline-fill per layer.  Here a cluster of NC (16, or 8 when the GPU cannot
// hold enough clusters of 16) CTAs owns one 128-row tile:
//
//   CTA j computes output columns [j*H/NC, (j+1)*H/NC) of every hidden layer with the FULL K: D_j = A[128 x K] * W_l[K x slice]
//     A: 16 sub-blocks ([128][32] bf16, SWIZZLE_64B) resident in smem; sub-block i holds input columns [32i, 32i+32), i.e. (part
//        of) the slice one CTA produced for the previous layer, all-gathered through L2 with TMA multicast: epilogue ->
//        st.global (bf16 row-major scratch) -> one cp.async.bulk.tensor ... .multicast::cluster per 32 columns that lands them
//        in all CTAs' smem and completes their per-sub-block mbarriers directly (MMAs start on the first sub-block that lands).
//        "smem may be overwritten" is a multicast tcgen05.commit from every CTA's MMA warps.  (Measured alternatives,
//        profiles/micro: DSMEM bulk copies 15 GB/s/SM, unicast gather + remote arrives 7.6 us/layer.)
//     B: the CTA's [K][H/NC] weight slice (MN-major, straight from the Flax [in,out] bf16 shadow), prefetched by TMA while the
//        previous layer's epilogue and exchange run (weights do not depend on activations)
//     D: fp32 in TMEM, one partial accumulator per issuing warp (NISS = 2 warps, each taking the sub-blocks of half the cluster as
//        they land), two sets so that layer l+1 can start while the epilogue still reads layer l.  TMEM reads run at 64 B/clk/SM, so
//        the epilogue's floor is (issuers x 128 x H/NC x 4 B) / 64 B/clk: 0.53 us at NC = 8, 0.27 us at NC = 16 -- with the
//        ~1.0 us issue-to-landed latency of the multicast this is what bounds a layer, hence the cluster of 16.
//        Epilogue: one thread per row: sum of the partials + bias, GELU(tanh), bf16.
//   the narrow last Dense (N = action_dim <= 32, zero-padded) is computed redundantly by every CTA, so each CTA applies
//   a += v / flow_steps to ITS copy of the first-layer operand tile (resident in smem for all steps) with no exchange.
//
// No kernel boundary, no global barrier: 4 L2 exchanges + 5 MMA chains per Euler step.
#include "step.cuh"
#include "tc_prims.cuh"

using namespace tc;

namespace {

constexpr int TILE_M = 128;
constexpr int KB = 64;                // K-block of the weight tiles (rows per TMA box)
constexpr int A_BLK = TILE_M * 128;   // 16 KB: [128][64] bf16 (first-layer operand tile, SWIZZLE_128B)
constexpr int SUB = 32;               // exchange granularity (columns)
constexpr int A_SUB = TILE_M * SUB * 2;  // 8 KB: [128][32] bf16, SWIZZLE_64B
constexpr int NSUB = 16;              // sub-blocks per hidden layer (H / SUB)
constexpr int MAX_A = 32;
constexpr int NMMA = 4;                // MMA warps in the launch (TMEM columns of an accumulator set = NMMA * NCOL)
#ifndef FQL_EULER_NISS
#define FQL_EULER_NISS 2
#endif
constexpr int NISS = FQL_EULER_NISS;   // warps that actually issue, each with its own partial accumulator (summed by the epilogue: its TMEM
                                       // reads, 64 B/clk, are the floor of a layer's epilogue).  4 when an `if (lane == 0)` issuer cost ~80 ns
                                       // per tcgen05.mma; with warp-uniform issue two warps keep up with the sub-blocks as they land.
static_assert(NISS == 1 || NISS == 2 || NISS == 4, "NISS");
constexpr int NEPI = 4;                // epilogue warps: one thread per row (TMEM-read bound: more warps were measured slower)
constexpr int NTHREADS = 32 * (1 + NMMA + NEPI);
constexpr int EPI0 = 32 * (1 + NMMA);  // first epilogue thread

struct EulerArgs {
  int H, K0, K0pad, A, F, n_steps, NL;
  int S, M, tiles;
  int x_rows_s;                 // rows of one seed in the X0b tensor
  int x_row0;                   // first row (inside a seed) of the Euler rows
  int w_row[FQL_MAXL];          // first shadow row (units of H elements) of layer l < NL-1
  int w_rows_s;
  int wl_row, wl_rows_s;        // padded last layer (units of 64 elements)
  const float* params;
  long long arena;
  long long off_b[FQL_MAXL];
  const float* c0;              // optional [S][M][H]: per-ROW additive term of layer 0 in place of its bias (pixel configs: the constant
                                // part obs_features @ W0[:F] + b0 of the first layer, hoisted out of the Euler loop; X0b then holds only
                                // the action / time columns and w_row[0] points at row F of W0)
  const float* a0;              // [S][M][A] initial actions (noise)
  float* target;                // [S][M][A] clip(final)
  __nv_bfloat16* hx;            // exchange scratch [2][S*tiles*128][H]
  long long hx_buf_elems;
  float* state;                 // fp32 Euler state between steps, per CTA: [CTA][MAX_A][128] (keeps 32 registers out of the epilogue)
  // MODE_FWD (one forward pass with the activations saved for the backward): bf16 [S][rows_cap][H] per hidden layer, element
  // (s, r0 + row, col); the H buffers double as the exchange buffers.  out: fp32 [S][rows_cap][A]
  __nv_bfloat16* Hsave[FQL_MAXL];
  __nv_bfloat16* Zsave[FQL_MAXL];
  float* out;
  int rows_cap, r0;
  float* Fsave[FQL_MAXL];       // MODE_DGRAD: fp32 copy of iteration it's output, same indexing as Hsave
  int z_rows_cap, z_r0;         // MODE_DGRAD: row geometry of Zsave (the forward pass's buffers)
  unsigned long long* dbg;  // optional [CTA][16] globaltimer stamps of iteration DBG_IT (diagnostics)
  unsigned long long* t_start;  // optional: kernel start / end time of CTA 0 (diagnostics)
  int dbg_it;                   // layer iteration the dbg stamps are taken at
};

struct HMaps {
  CUtensorMap m[4];  // MODE_EULER: m[0] = exchange scratch; MODE_FWD: m[l] = H buffer of layer l
};
// MODE_DGRAD: the input-gradient chain of a backward pass, dZ_{l-1} = (dZ_l W_l^T) * gelu'(Z_{l-1}): iteration `it` consumes
// W_{NL-it}^T (K-major slices straight from the [in,out] shadow: rows = this CTA's 32 inputs, k contiguous), multiplies by
// gelu' of the saved pre-activation and writes dZ as bf16 (exchange buffer = the wgrad operand) and fp32 (bias gradients).
constexpr int MODE_EULER = 0, MODE_FWD = 1, MODE_DGRAD = 2;

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

// AMAX: compile-time bound of action_dim (the Euler update is unrolled over it; the kernel's code must stay small -- the rarely
// executed last-layer path was measured at 3.5 us, mostly instruction fetch, when it was unrolled to 32 actions)
template <int NC, int AMAX, int MODE>
__global__ void __launch_bounds__(NTHREADS, 1) euler_cluster_kernel(const __grid_constant__ CUtensorMap mapX,
                                                               const __grid_constant__ CUtensorMap mapW,
                                                               const __grid_constant__ CUtensorMap mapWL,
                                                               const __grid_constant__ HMaps mapsH, const EulerArgs a) {
  constexpr int NCOL = 512 / NC;            // output columns per CTA (64 / 32)
  constexpr int HALVES = NCOL / SUB;        // 32-column exchange units per CTA (2 / 1)
  constexpr int B_ROWB = NCOL * 2;          // bytes per K row of the weight slice (128: SWIZZLE_128B, 64: SWIZZLE_64B)
  constexpr int B_BLK = KB * B_ROWB;        // one TMA box: [64 k][NCOL n] bf16
  constexpr int ACC_SET = NMMA * NCOL;      // TMEM columns of one accumulator set
  constexpr uint16_t MASK = (uint16_t)((1u << NC) - 1u);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int nkb = a.H / KB, nkb_x = a.K0pad / KB;
  uint8_t* sA = smem;                        // [NSUB][8 KB]: sub-block i = columns [32i, 32i+32) of the layer input
  uint8_t* sB = sA + NSUB * A_SUB;           // [nkb][B_BLK]  weight slice of the current layer
  uint8_t* sX = sB + nkb * B_BLK;            // [nkb_x][16 KB] first-layer operand tile, resident for all steps
  float* sBias = reinterpret_cast<float*>(sX + nkb_x * A_BLK);  // [NL][64]: this CTA's bias slice of every layer (constant over the steps)
  float* sT = sBias + a.NL * 64;  // [n_steps + 1]: the flow time i / n_steps as the reference rounds it (double quotient -> f32)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sT + 64);
  uint64_t* full_a = bars;          // [NSUB]
  uint64_t* full_b = bars + 16;
  uint64_t* acc_full = bars + 17;
  uint64_t* free_a = bars + 18;     // count NC*NMMA: every CTA's MMAs of the current layer are done -> sA may be overwritten
  uint64_t* a_ready = bars + 19;    // count NEPI: the Euler update of the resident X tile is done (local)
  uint64_t* x_full = bars + 20;
  uint64_t* half_ready = bars + 21; // [2] count NEPI: 32 columns of this CTA's layer output are in the exchange scratch
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 24);

  // warp index and cluster rank through a shuffle: warp-uniform to ptxas as well (operands of TMA / tcgen05 instructions derived from
  // them then live in uniform registers)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const uint32_t j = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);   // column slice
  const int cl = blockIdx.x / NC;                        // cluster id = (seed, tile)
  const int tile = cl % a.tiles, s = cl / a.tiles;
  const int NL = a.NL;
  const int total = a.n_steps * NL;
  const int hx_row = (s * a.tiles + tile) * TILE_M;      // this tile's rows in the exchange scratch
  unsigned long long* dbg = a.dbg ? a.dbg + blockIdx.x * 16 : nullptr;
  const int DBG_IT = a.dbg_it;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapX);
    tma_prefetch_desc(&mapW);
    tma_prefetch_desc(&mapWL);
    for (int i = 0; i < (MODE == MODE_EULER ? 1 : NL - 1); i++) tma_prefetch_desc(&mapsH.m[i]);
    for (int i = 0; i < NSUB; i++) mbar_init(&full_a[i], 1);
    mbar_init(&half_ready[0], NEPI);
    mbar_init(&half_ready[1], NEPI);
    mbar_init(full_b, 1);
    mbar_init(acc_full, NISS);
    mbar_init(free_a, NC * NISS);
    mbar_init(a_ready, NEPI);
    mbar_init(x_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 2 * ACC_SET);  // two accumulator sets
  for (int i = threadIdx.x; i < (MODE == MODE_DGRAD ? 0 : NL * 64); i += NTHREADS) {
    const int l = i >> 6, c = i & 63;
    const bool lastl = (l == NL - 1);
    const int N = lastl ? a.A : a.H;
    const int col = lastl ? c : (int)j * NCOL + c;
    sBias[i] = (c < NCOL && col < N && !(l == 0 && a.c0)) ? a.params[(int64_t)s * a.arena + a.off_b[l] + col] : 0.f;
  }
  if (threadIdx.x <= a.n_steps) sT[threadIdx.x] = (float)((double)threadIdx.x / (double)a.n_steps);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  cluster_sync_all();  // every CTA's barriers are initialised before any remote arrive
  const uint32_t tmem_base = *tmem_slot;
  if (a.t_start && blockIdx.x == 0 && threadIdx.x == 0) a.t_start[0] = gtime();

  if (warp == 0) {
    // ================= TMA producer / publisher =================
    // One thread's role, but all 32 lanes run the loop and only the instructions are predicated on the elected lane: with the loop
    // under `if (lane == 0)` ptxas wraps every TMA / tcgen05 instruction in an ELECT + R2UR.BROADCAST waterfall (tc_prims.cuh).
    const bool el = elect_one();
    {
      if (el) mbar_expect_tx(x_full, nkb_x * A_BLK);
      const int xrow = s * a.x_rows_s + a.x_row0 + tile * TILE_M;
      for (int kb = 0; kb < nkb_x; kb++)
        if (el) tma_load_2d(sX + kb * A_BLK, &mapX, x_full, kb * KB, xrow);
      int n_pub = 0;
      int l = 0;
      for (int it = 0; it < total; it++, l = (l + 1 == NL) ? 0 : l + 1) {
        const bool last = (l == NL - 1);
        const int K = (l == 0) ? a.K0 : a.H;
        const int kblocks = (K + KB - 1) / KB;
        // weights of this layer: sB is free once the previous layer's MMAs have completed
        if (it > 0) mbar_wait_u(acc_full, (it - 1) & 1);
        if (el) mbar_expect_tx(full_b, kblocks * B_BLK);
        for (int kb = 0; kb < kblocks; kb++) {
          if (!el) continue;
          if constexpr (MODE == MODE_DGRAD) {  // K-major: box = [NCOL input rows][64 k]
            if (l == 0) tma_load_2d(sB, &mapWL, full_b, 0, a.wl_row + s * a.wl_rows_s + (int)j * NCOL);
            else tma_load_2d(sB + kb * B_BLK, &mapW, full_b, kb * KB, a.w_row[l] + s * a.w_rows_s + (int)j * NCOL);
          } else {
            if (!last) tma_load_2d(sB + kb * B_BLK, &mapW, full_b, (int)j * NCOL, a.w_row[l] + s * a.w_rows_s + kb * KB);
            else tma_load_2d(sB + kb * B_BLK, &mapWL, full_b, 0, a.wl_row + s * a.wl_rows_s + kb * KB);
          }
        }
        if (l >= 1) {
          // arm the per-sub-block barriers, then publish this CTA's slice of the layer input (= the previous layer's output, which
          // its epilogue is producing right now) 32 columns at a time: one TMA multicast lands them in all CTAs' smem and
          // completes their barriers directly
          for (int sbk = 0; sbk < NSUB; sbk++)
            if (el) mbar_expect_tx(&full_a[sbk], A_SUB);
          const int buf = n_pub & 1;
          for (int h = 0; h < HALVES; h++) {
            mbar_wait_u(&half_ready[h], n_pub & 1);
            asm volatile("fence.proxy.async.global;" ::: "memory");  // the epilogue's st.global (acquired above) -> this thread's TMA read
            if (h == 0) mbar_wait_cluster_u(free_a, (it - 1) & 1);   // every CTA finished reading sA for the previous layer
            if (dbg && el && it == DBG_IT) dbg[3 + h] = gtime();
            const int sbk = (int)j * HALVES + h;
            if (el)
              asm volatile(
                  "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
                  ::"r"(smem_u32(sA + sbk * A_SUB)), "l"(reinterpret_cast<uint64_t>(MODE != MODE_EULER ? &mapsH.m[l - 1] : &mapsH.m[0])),
                  "r"(smem_u32(&full_a[sbk])), "r"(sbk * SUB),
                  "r"(MODE != MODE_EULER ? s * a.rows_cap + a.r0 + tile * TILE_M : buf * (a.S * a.tiles * TILE_M) + hx_row), "h"(MASK)
                  : "memory");
          }
          n_pub++;
        }
      }
    }
  } else if (warp <= NMMA) {
    // ================= MMA issuers =================
    // Four warps issue a quarter of the K range each into their own TMEM columns (summed by the epilogue): the sub-blocks of a layer's
    // input land one after the other, and a warp starts on its four as soon as they are there.  All 32 lanes of an issuer warp run
    // the loop; the tcgen05 instructions are predicated on the elected lane (uniform-register operands, no waterfall -- see above).
    const bool el = elect_one();
    if (warp <= NISS) {
      const int mw = warp - 1;
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc = make_idesc_bf16(TILE_M, NCOL, false, MODE != MODE_DGRAD);
      const uint64_t ax_t = make_smem_desc(0, 16, 1024);            // first-layer operand: [128][64] bf16 blocks, SWIZZLE_128B
      const uint64_t a64_t0 = make_smem_desc_sw64(0, 16, 512);      // [128][32] bf16 sub-blocks, SWIZZLE_64B: 8-row groups 512 B apart
      // B: MN-major [k][NCOL] tiles (forward) or K-major [NCOL][64 k] SWIZZLE_128B tiles (MODE_DGRAD: W^T)
      const uint64_t b_t0 = (MODE == MODE_DGRAD) ? make_smem_desc(0, 16, 1024)
                                                 : ((NC == 8) ? make_smem_desc(0, B_BLK, 1024) : make_smem_desc_sw64(0, B_BLK, 512));
      constexpr uint64_t B_KSTEP = (MODE == MODE_DGRAD) ? 2 : ((16 * B_ROWB) >> 4);   // 16 k: 32 B inside a row / 16 K rows
      constexpr uint64_t B_SUBH = (MODE == MODE_DGRAD) ? 4 : ((32 * B_ROWB) >> 4);    // second 32-k half of a 64-k block
      const uint32_t sa0 = smem_u32(sA) >> 4, sx0 = smem_u32(sX) >> 4, sb0 = smem_u32(sB) >> 4;
      int n_a = 0;  // uses of the full_a barriers
      int n_step = 0;
      int l = 0;
      for (int it = 0; it < total; it++, l = (l + 1 == NL) ? 0 : l + 1) {
        const int K = (l == 0) ? a.K0 : a.H;
        const int kblocks = (K + KB - 1) / KB;
        const uint32_t tacc = tmem_u + (it & 1) * ACC_SET + mw * NCOL;
        if (l == 0) {
          if (it == 0) mbar_wait_u(x_full, 0);
          else { mbar_wait_u(a_ready, (n_step - 1) & 1); }
          n_step++;
          if (dbg && el && mw == 0 && it == DBG_IT) dbg[8] = gtime();
        }
        mbar_wait_u(full_b, it & 1);
        tc_fence_after();
        if (dbg && el && mw == 0 && it == DBG_IT && l == 0) dbg[9] = gtime();
        if (l >= 1) {
          // hidden / last layers (K = H): warp w owns NSUB / NISS of the 16 sub-blocks, in the order they are published (clusters of 8:
          // every CTA publishes its first 32 columns, then its second)
          constexpr int PER = NSUB / NISS;
          for (int i = 0; i < PER; i++) {
            const int sbk = (NC == 8) ? (mw * (PER / 2) + (i % (PER / 2))) * 2 + (i / (PER / 2)) : mw * PER + i;
            mbar_wait_u(&full_a[sbk], n_a & 1);
            tc_fence_after();
            if (dbg && el && mw == 0 && it == DBG_IT && i == 0) dbg[5] = gtime();
            if (dbg && el && mw == NISS - 1 && it == DBG_IT && i == PER - 1) dbg[6] = gtime();
            if (el)
              umma_bf16_x2(tacc, a64_t0 + (uint64_t)(sa0 + sbk * (A_SUB >> 4)),
                           b_t0 + (uint64_t)(sb0 + (sbk >> 1) * (B_BLK >> 4) + (sbk & 1) * B_SUBH), 2, B_KSTEP, idesc, i != 0);
          }
        } else {
          // first layer (K0 <= 128): k-steps w, w + NISS, ... of every block -> warp w
          for (int kb = 0; kb < kblocks; kb++)
            for (int ks = mw; ks < 4; ks += NISS)
              if (el && ks < (a.K0 - kb * KB + 15) / 16)
                umma_bf16(tacc, ax_t + (uint64_t)(sx0 + kb * (A_BLK >> 4) + ks * 2), b_t0 + (uint64_t)(sb0 + kb * (B_BLK >> 4) + ks * B_KSTEP), idesc,
                          !(kb == 0 && ks == mw));
        }
        if (l >= 1) n_a++;
        if (dbg && el && mw == 0 && it == DBG_IT && l == 0) dbg[10] = gtime();
        if (el) {
          umma_commit(acc_full);
          asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(free_a)),
                       "h"(MASK)
                       : "memory");
        }
      }
    }
  } else {
    // ================= epilogue: one thread per row =================
    const int q = warp & 3;                          // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;
    const int grow = tile * TILE_M + row;
    const bool valid = grow < a.M;
    const uint32_t t_lane0 = tmem_base + ((uint32_t)(q * 32) << 16);
    const int et = threadIdx.x - EPI0;
    float* st_row = a.state + (int64_t)blockIdx.x * MAX_A * TILE_M + row;  // this row's Euler state, element c at st_row[c * 128]
    int n_exch = 0;
    int l = 0, step = 0;
    for (int it = 0; it < total; it++, l = (l + 1 == NL) ? 0 : l + 1, step += (l == 0)) {
      const bool last = (l == NL - 1);
      const float* sb = sBias + l * 64;
      uint4 zq[4];  // MODE_DGRAD: this row's 32 saved pre-activations, fetched while the MMAs run
      if constexpr (MODE == MODE_DGRAD) {
        static_assert(MODE != MODE_DGRAD || HALVES == 1, "the dgrad chain is built for clusters of 16");
        if (valid) {
          const uint4* zp = reinterpret_cast<const uint4*>(a.Zsave[l] + ((int64_t)s * a.z_rows_cap + a.z_r0 + grow) * a.H + j * NCOL);
#pragma unroll
          for (int c = 0; c < 4; c++) zq[c] = __ldg(zp + c);
        }
      }
      float ac[AMAX];  // Euler state of this row: fetched while the last layer's MMAs run (registers are free in this phase)
      if (MODE == MODE_EULER && last) {
#pragma unroll
        for (int c = 0; c < AMAX; c++)
          if (c < a.A) ac[c] = (step == 0) ? (valid ? __ldg(a.a0 + ((int64_t)s * a.M + grow) * a.A + c) : 0.f) : __ldcg(st_row + c * TILE_M);
      }
      mbar_wait(acc_full, it & 1);
      tc_fence_after();
      if (dbg && et == 0 && it == DBG_IT - 1) dbg[0] = gtime();
      if (dbg && et == 0 && it == DBG_IT) dbg[7] = gtime();
      // partial accumulators of the NISS issuer warps, loads issued in pairs (a first layer with K0 < 16 NISS has ceil(K0/16) of them)
      const int live = (l == 0 && (a.K0 + 15) / 16 < NISS) ? (a.K0 + 15) / 16 : NISS;
      const int buf = n_exch & 1;
      if (!last) n_exch++;
#pragma unroll 1
      for (int half = 0; half < HALVES; half++) {
        const uint32_t t_lane = t_lane0 + (it & 1) * ACC_SET + half * 32;
        uint32_t r0[32];
        if (!last || half == 0) {
          uint32_t t1[32];
          tmem_ld32(t_lane, r0);
          if (live > 1) tmem_ld32(t_lane + NCOL, t1);
          tmem_wait_ld();
          if (live > 1) {
#pragma unroll
            for (int i = 0; i < 32; i++) r0[i] = __float_as_uint(__uint_as_float(r0[i]) + __uint_as_float(t1[i]));
          }
          if (live > 2) {
            uint32_t t2[32];
            tmem_ld32(t_lane + 2 * NCOL, t1);
            if (live > 3) tmem_ld32(t_lane + 3 * NCOL, t2);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 32; i++) {
              float v = __uint_as_float(r0[i]) + __uint_as_float(t1[i]);
              if (live > 3) v += __uint_as_float(t2[i]);
              r0[i] = __float_as_uint(v);
            }
          }
        }
        if constexpr (MODE == MODE_DGRAD) {
          if (valid) {
            const int64_t e0 = ((int64_t)s * a.rows_cap + a.r0 + grow) * a.H + j * NCOL;
            uint4* dh = reinterpret_cast<uint4*>(a.Hsave[l] + e0);
            float4* df = reinterpret_cast<float4*>(a.Fsave[l] + e0);
#pragma unroll
            for (int c = 0; c < 4; c++) {
              const uint32_t zw[4] = {zq[c].x, zq[c].y, zq[c].z, zq[c].w};
              float dv[8];
#pragma unroll
              for (int i = 0; i < 4; i++) {
                const __nv_bfloat162 zb = *reinterpret_cast<const __nv_bfloat162*>(&zw[i]);
                dv[2 * i] = __uint_as_float(r0[c * 8 + 2 * i]) * gelu_grad_fast(__low2float(zb));
                dv[2 * i + 1] = __uint_as_float(r0[c * 8 + 2 * i + 1]) * gelu_grad_fast(__high2float(zb));
              }
              dh[c] = make_uint4(pack2(dv[0], dv[1]), pack2(dv[2], dv[3]), pack2(dv[4], dv[5]), pack2(dv[6], dv[7]));
              df[2 * c] = make_float4(dv[0], dv[1], dv[2], dv[3]);
              df[2 * c + 1] = make_float4(dv[4], dv[5], dv[6], dv[7]);
            }
          }
          if (!last) {  // the next layer's input: the producer thread multicasts it once all NEPI warps arrived
            __syncwarp();
            if (lane == 0) mbar_arrive(&half_ready[half]);
          }
        } else if (!last) {
          if constexpr (MODE == MODE_EULER) {
            uint4* dst = reinterpret_cast<uint4*>(a.hx + (int64_t)buf * a.hx_buf_elems + (int64_t)(hx_row + row) * a.H + j * NCOL + half * 32);
            if (l == 0 && a.c0) {   // hoisted first layer: + (features @ W0[:F] + b0) of this row (sBias of layer 0 is zero)
              const float4* cp = reinterpret_cast<const float4*>(a.c0 + ((int64_t)s * a.M + (valid ? grow : 0)) * a.H + j * NCOL + half * 32);
#pragma unroll
              for (int c = 0; c < 8; c++) {
                const float4 cv = __ldg(cp + c);
                r0[c * 4 + 0] = __float_as_uint(__uint_as_float(r0[c * 4 + 0]) + cv.x);
                r0[c * 4 + 1] = __float_as_uint(__uint_as_float(r0[c * 4 + 1]) + cv.y);
                r0[c * 4 + 2] = __float_as_uint(__uint_as_float(r0[c * 4 + 2]) + cv.z);
                r0[c * 4 + 3] = __float_as_uint(__uint_as_float(r0[c * 4 + 3]) + cv.w);
              }
            }
#pragma unroll
            for (int c = 0; c < 4; c++) {
              float h[8];
#pragma unroll
              for (int i = 0; i < 8; i++) h[i] = gelu_fast(__uint_as_float(r0[c * 8 + i]) + sb[half * 32 + c * 8 + i]);
              dst[c] = make_uint4(pack2(h[0], h[1]), pack2(h[2], h[3]), pack2(h[4], h[5]), pack2(h[6], h[7]));
            }
          } else if (valid) {
            // utils/networks.py:54-56: z = xW + b (saved for gelu' in the backward), h = gelu(z) (saved = the next layer's operand)
            const int64_t e0 = ((int64_t)s * a.rows_cap + a.r0 + grow) * a.H + j * NCOL + half * 32;
            uint4* dh = reinterpret_cast<uint4*>(a.Hsave[l] + e0);
            uint4* dz = reinterpret_cast<uint4*>(a.Zsave[l] + e0);
#pragma unroll
            for (int c = 0; c < 4; c++) {
              float z[8], h[8];
#pragma unroll
              for (int i = 0; i < 8; i++) {
                z[i] = __uint_as_float(r0[c * 8 + i]) + sb[half * 32 + c * 8 + i];
                h[i] = gelu_fast(z[i]);
              }
              dh[c] = make_uint4(pack2(h[0], h[1]), pack2(h[2], h[3]), pack2(h[4], h[5]), pack2(h[6], h[7]));
              dz[c] = make_uint4(pack2(z[0], z[1]), pack2(z[2], z[3]), pack2(z[4], z[5]), pack2(z[6], z[7]));
            }
          }
          // this warp's rows are in the scratch: the producer thread multicasts the 32 columns once all NEPI warps arrived
          __syncwarp();
          if (lane == 0) mbar_arrive(&half_ready[half]);
          if (dbg && et == 0 && it == DBG_IT - 1) dbg[1 + half] = gtime();
        } else if (MODE == MODE_FWD) {
          if (half == 0 && j == 0 && valid) {  // every CTA computes the narrow last layer; one writes it
            float* o = a.out + ((int64_t)s * a.rows_cap + a.r0 + grow) * a.A;
#pragma unroll
            for (int c = 0; c < AMAX; c++)
              if (c < a.A) o[c] = __uint_as_float(r0[c]) + sb[c];
          }
        } else if (half == 0) {
          // Euler step on this CTA's resident copy of the first-layer operand (every CTA computes the same last layer)
          if (dbg && et == 0 && it == DBG_IT - 1) dbg[13] = gtime();
          const float inv = (float)a.n_steps;
          const bool final_step = (step == a.n_steps - 1);
#pragma unroll
          for (int c = 0; c < AMAX; c++)
            if (c < a.A) {
              ac[c] += (__uint_as_float(r0[c]) + sb[c]) / inv;
              const int col = a.F + c;
              *reinterpret_cast<__nv_bfloat16*>(sX + (col >> 6) * A_BLK + sw128_off(row, (col & 63) >> 3) + (col & 7) * 2) = __float2bfloat16(ac[c]);
            }
          {
            const int col = a.F + a.A;
            *reinterpret_cast<__nv_bfloat16*>(sX + (col >> 6) * A_BLK + sw128_off(row, (col & 63) >> 3) + (col & 7) * 2) =
                __float2bfloat16(sT[step + 1]);
          }
          if (dbg && et == 0 && it == DBG_IT - 1) dbg[11] = gtime();
          // the MMA warps may start the next step's first layer as soon as the operand tile is updated; the state goes out after
          fence_proxy_async_smem();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(a_ready);
          if (dbg && et == 0 && it == DBG_IT - 1) dbg[12] = gtime();
#pragma unroll
          for (int c = 0; c < AMAX; c++)
            if (c < a.A) {
              if (!final_step) __stcg(st_row + c * TILE_M, ac[c]);
              else if (valid && j == 0) a.target[((int64_t)s * a.M + grow) * a.A + c] = fminf(fmaxf(ac[c], -1.0f), 1.0f);
            }
        }
      }  // halves
      if (!last) tc_fence_before();
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // no CTA may exit while a peer can still arrive on its barriers
  if (a.t_start && blockIdx.x == 0 && threadIdx.x == 0) a.t_start[1] = gtime();
  if (warp == 1) tmem_dealloc(tmem_base, 2 * ACC_SET);
}

}  // namespace

size_t tc_euler_scratch_elems(const FqlDims* d, int M) {
  const int tiles = (M + TILE_M - 1) / TILE_M;
  // two exchange buffers [S*tiles*128][H] bf16 + the per-CTA fp32 Euler state [S*tiles*16][MAX_A][128]
  return (size_t)2 * d->num_seeds * tiles * TILE_M * d->hidden + (size_t)2 * d->num_seeds * tiles * 16 * MAX_A * TILE_M;
}

namespace {
template <int NC, int AMAX, int MODE>
int launch_euler(const EulerArgs& a, const TcEulerSpec& f, cudaStream_t st, bool query_only, int* max_clusters) {
  constexpr int NCOL = 512 / NC;
  const FqlDims* d = f.d;
  const int smem = NSUB * A_SUB + (a.H / KB) * (KB * NCOL * 2) + (a.K0pad / KB) * A_BLK + a.NL * 64 * 4 + 64 * 4 + 256 + 1024;
  FQL_REQUIRE(smem <= 232448, "euler_cluster_kernel: shared memory %d > 227 KB", smem);
  auto kern = euler_cluster_kernel<NC, AMAX, MODE>;
  static bool attr_set[FQL_MAX_DEVICES] = {};
  const int dev = fql_current_device();
  if (!attr_set[dev]) {
    FQL_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    if (NC > 8) FQL_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    attr_set[dev] = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(NC * a.tiles * a.S);
  cfg.blockDim = dim3(NTHREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = NC;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (query_only) {
    cfg.stream = nullptr;
    if (cudaOccupancyMaxActiveClusters(max_clusters, kern, &cfg) != cudaSuccess) {
      cudaGetLastError();
      *max_clusters = 0;
    }
    return 0;
  }
  const CUtensorMapSwizzle wsw = (NC == 8 || MODE == MODE_DGRAD) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUtensorMap mapX, mapW, mapWL;
  HMaps mapsH;
  memset(&mapsH, 0, sizeof(mapsH));
  FQL_TRY(make_map_2d(&mapX, f.X0b, a.K0pad, (uint64_t)a.S * f.Mcap0, 64, TILE_M));
  if (MODE == MODE_DGRAD) {  // K-major W^T slices: [NCOL input rows][64 k]
    FQL_TRY(make_map_2d(&mapW, f.shadow, d->hidden, (uint64_t)a.S * a.w_rows_s, 64, NCOL, wsw));
    FQL_TRY(make_map_2d(&mapWL, f.shadow, 64, (uint64_t)a.S * a.wl_rows_s, 64, NCOL, wsw));
  } else {
    FQL_TRY(make_map_2d(&mapW, f.shadow, d->hidden, (uint64_t)a.S * a.w_rows_s, NCOL, KB, wsw));
    FQL_TRY(make_map_2d(&mapWL, f.shadow, 64, (uint64_t)a.S * a.wl_rows_s, NCOL, KB, wsw));  // NC = 16: the first 32 (>= action_dim) columns
  }
  if (MODE == MODE_EULER) {
    FQL_TRY(make_map_2d(&mapsH.m[0], f.scratch, d->hidden, (uint64_t)2 * a.S * a.tiles * TILE_M, SUB, TILE_M, CU_TENSOR_MAP_SWIZZLE_64B));
  } else {
    for (int l = 0; l + 1 < a.NL; l++)
      FQL_TRY(make_map_2d(&mapsH.m[l], a.Hsave[l], d->hidden, (uint64_t)a.S * a.rows_cap, SUB, TILE_M, CU_TENSOR_MAP_SWIZZLE_64B));
  }
  FQL_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, mapX, mapW, mapWL, mapsH, a));
  FQL_CHECK_LAUNCH();
  return 0;
}
}  // namespace

namespace {
int fill_args(EulerArgs& a, const FqlDims* d, const Layout& L, int net, const float* params, int M, int Mcap0, int r0_in, bool hoisted = false) {
  FQL_TRY(tc_supported(d, !hoisted));
  FQL_REQUIRE(d->hidden == 512, "euler_cluster_kernel is built for hidden = 512 (16 exchange units of 32 columns)");
  const NetView& nv = L.net[net];
  memset(&a, 0, sizeof(a));
  a.H = d->hidden; a.K0 = nv.in_dim; a.K0pad = (int)round_up64(nv.in_dim, 64); a.A = nv.out_dim; a.F = d->obs_dim;
  a.n_steps = 1; a.NL = nv.n_layers;
  a.S = d->num_seeds; a.M = M; a.tiles = (M + TILE_M - 1) / TILE_M;
  a.x_rows_s = Mcap0; a.x_row0 = r0_in;
  const int64_t seed_elems = tc_shadow_seed_elems(d, L);
  a.w_rows_s = (int)(seed_elems / d->hidden);
  a.wl_rows_s = (int)(seed_elems / 64);
  for (int l = 0; l < nv.n_layers; l++) {
    a.w_row[l] = (int)(nv.off_w[l] / d->hidden);
    a.off_b[l] = nv.off_b[l];
  }
  int64_t wl = L.arena;
  for (int t = 0; t < net; t++) wl += (int64_t)L.net[t].ens * d->hidden * 64;
  a.wl_row = (int)(wl / 64);
  a.params = params; a.arena = L.arena;
  FQL_REQUIRE(a.A <= MAX_A, "euler_cluster_kernel: output width %d > %d", a.A, MAX_A);
  a.dbg_it = 7;  // layer iteration the optional phase stamps (FQL_B200_STAMPS) are taken at
  return 0;
}
// clusters of 16 CTAs the GPU can hold at once (one per GPC); 0 when FQL_B200_EULER_NC=8 forces clusters of 8
int max_clusters16(const EulerArgs& a, const TcEulerSpec& f) {
  static int max16_dev[FQL_MAX_DEVICES];
  static bool known[FQL_MAX_DEVICES] = {};
  const int dev = fql_current_device();
  int& max16 = max16_dev[dev];
  if (!known[dev]) {
    const char* e = getenv("FQL_B200_EULER_NC");
    if (e && atoi(e) == 8) max16 = 0;
    else if (launch_euler<16, 8, MODE_EULER>(a, f, nullptr, true, &max16)) max16 = 0;
    if (getenv("FQL_B200_VERBOSE")) fprintf(stderr, "fql_b200: clusters of 16 CTAs resident at once (device %d): %d\n", dev, max16);
    known[dev] = true;
  }
  return max16;
}
}  // namespace

int tc_euler_cluster(const TcEulerSpec& f, cudaStream_t st) {
  const FqlDims* d = f.d;
  EulerArgs a;
  FQL_TRY(fill_args(a, d, *f.L, FQL_NET_ACTOR_BC_FLOW, f.params, f.M, f.Mcap0, f.r0_in, f.c0 != nullptr));
  a.A = d->action_dim; a.n_steps = d->flow_steps;
  if (f.c0) {
    // hoisted first layer (agents/fql.py:162-169: the observation features are constant over the flow steps): the kernel's first layer
    // is [action | t] @ W0[F:] + c0[row], X0b holds those A + 1 columns only
    a.c0 = f.c0;
    a.K0 = d->action_dim + 1; a.K0pad = 64; a.F = 0;
    a.w_row[0] += d->obs_dim;
  }
  a.a0 = f.a0; a.target = f.target;
  a.hx = reinterpret_cast<__nv_bfloat16*>(f.scratch);
  a.hx_buf_elems = (long long)a.S * a.tiles * TILE_M * a.H;
  a.state = reinterpret_cast<float*>(a.hx + 2 * a.hx_buf_elems);
  a.dbg = reinterpret_cast<unsigned long long*>(f.dbg);
  a.t_start = reinterpret_cast<unsigned long long*>(f.t_start);
  FQL_REQUIRE(f.scratch != nullptr && f.a0 && f.target, "tc_euler_cluster: NULL argument");
  FQL_REQUIRE(a.n_steps < 64, "euler_cluster_kernel: flow_steps %d >= 64", a.n_steps);
  // clusters of 16 (one per GPC) halve the per-layer epilogue; fall back to clusters of 8 when there are more row tiles than the
  // GPU can hold clusters of 16 at once
  const bool c16 = a.tiles * a.S <= max_clusters16(a, f);
  if (a.A <= 8) return c16 ? launch_euler<16, 8, MODE_EULER>(a, f, st, false, nullptr) : launch_euler<8, 8, MODE_EULER>(a, f, st, false, nullptr);
  if (a.A <= 16) return c16 ? launch_euler<16, 16, MODE_EULER>(a, f, st, false, nullptr) : launch_euler<8, 16, MODE_EULER>(a, f, st, false, nullptr);
  return c16 ? launch_euler<16, 32, MODE_EULER>(a, f, st, false, nullptr) : launch_euler<8, 32, MODE_EULER>(a, f, st, false, nullptr);
}

// One forward pass of an actor network (no LayerNorm) on M rows as a cluster-of-16 chain, activations saved for the backward.
// other_clusters: clusters of 16 that run at the same time (the Euler chain).  Returns 1 when the kernel cannot take the problem
// (the caller then uses the layer-by-layer path), 0 on success, -1 on error.
int tc_cluster_forward(const TcClusterFwdSpec& f, int other_clusters, cudaStream_t st) {
  const FqlDims* d = f.d;
  const NetView& nv = f.L->net[f.net];
  if (d->hidden != 512 || nv.ln || nv.n_layers > 5 || nv.n_layers < 2 || nv.out_dim > MAX_A || nv.in_dim > 128) return 1;
  EulerArgs a;
  if (fill_args(a, d, *f.L, f.net, f.params, f.M, f.rows_cap, f.r0)) return -1;
  TcEulerSpec e;
  memset(&e, 0, sizeof(e));
  e.d = d; e.L = f.L; e.params = f.params; e.shadow = f.shadow; e.X0b = f.X0b; e.Mcap0 = f.rows_cap; e.r0_in = f.r0; e.M = f.M;
  if (a.tiles * a.S + other_clusters > max_clusters16(a, e)) return 1;
  for (int l = 0; l + 1 < nv.n_layers; l++) {
    a.Hsave[l] = reinterpret_cast<__nv_bfloat16*>(f.Hb[l]);
    a.Zsave[l] = reinterpret_cast<__nv_bfloat16*>(f.Zb[l]);
    if (!a.Hsave[l] || !a.Zsave[l]) return 1;
  }
  a.out = f.out; a.rows_cap = f.rows_cap; a.r0 = f.r0;
  a.t_start = reinterpret_cast<unsigned long long*>(f.t_start);
  if (a.A <= 8) return launch_euler<16, 8, MODE_FWD>(a, e, st, false, nullptr) ? -1 : 0;
  if (a.A <= 16) return launch_euler<16, 16, MODE_FWD>(a, e, st, false, nullptr) ? -1 : 0;
  return launch_euler<16, 32, MODE_FWD>(a, e, st, false, nullptr) ? -1 : 0;
}

// The input-gradient chain of an actor network's backward (no LayerNorm) on M rows as one cluster-of-16 launch:
// dZ_{NL-2} = (dOut W_last^T) * gelu'(Z_{NL-2}), then dZ_{l-1} = (dZ_l W_l^T) * gelu'(Z_{l-1}) down to dZ_0 (bf16 + fp32 copies).
// Returns 1 when the kernel cannot take the problem (the caller then uses the layer-by-layer path), 0 on success, -1 on error.
int tc_cluster_dgrad(const TcClusterBwdSpec& f, int other_clusters, cudaStream_t st) {
  const FqlDims* d = f.d;
  const NetView& nv = f.L->net[f.net];
  if (d->hidden != 512 || nv.ln || nv.n_layers > 5 || nv.n_layers < 3 || nv.out_dim > 64) return 1;
  EulerArgs a;
  if (fill_args(a, d, *f.L, f.net, nullptr, f.M, f.M, 0)) return -1;
  const int NLn = nv.n_layers;
  a.NL = NLn - 1;          // chain GEMMs
  a.K0 = 64; a.K0pad = 64; // dOut zero-padded to 64 columns
  for (int it = 1; it < a.NL; it++) a.w_row[it] = (int)(nv.off_w[NLn - 1 - it] / d->hidden);  // iteration it multiplies by W_{NL-it}^T
  TcEulerSpec e;
  memset(&e, 0, sizeof(e));
  e.d = d; e.L = f.L; e.shadow = f.shadow; e.X0b = f.dOutb; e.Mcap0 = f.M; e.r0_in = 0; e.M = f.M;
  if (a.tiles * a.S + other_clusters > max_clusters16(a, e)) return 1;
  for (int it = 0; it < a.NL; it++) {
    const int lo = NLn - 2 - it;  // iteration it produces dZ_lo
    a.Hsave[it] = reinterpret_cast<__nv_bfloat16*>(f.dZb[lo]);
    a.Fsave[it] = f.dZf[lo];
    a.Zsave[it] = reinterpret_cast<__nv_bfloat16*>(f.Zb[lo]);
    if (!a.Hsave[it] || !a.Fsave[it] || !a.Zsave[it]) return 1;
  }
  a.rows_cap = f.M; a.r0 = 0; a.z_rows_cap = f.z_rows_cap; a.z_r0 = f.z_r0;
  a.t_start = reinterpret_cast<unsigned long long*>(f.t_start);
  return launch_euler<16, 8, MODE_DGRAD>(a, e, st, false, nullptr) ? -1 : 0;
}
