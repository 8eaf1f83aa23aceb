// encoder_tc.cu -- ImpalaEncoder('impala_small') forward / backward (utils/encoders.py:10-57, 60-100) on the 5th-generation
// tensor cores: every 3x3 SAME convolution is an implicit GEMM on tcgen05 (bf16 operands, fp32 accumulation in TMEM).
//   x = u8/255 -> 3 x [conv3x3 -> max_pool 3x3/2 SAME(-inf) -> (relu -> conv -> relu -> conv) + skip] -> relu -> flatten
//     -> Dense(2048 -> 512) -> gelu(tanh)                                   (encoders.py:83-100, networks.py:34-61 activate_final)
//
// conv_tc_kernel<CT_CONV>   D[128 pixels][64] = im2col(X)[128][9 Cin] * Wb[9 Cin][64]    forward AND input gradient (the same kernel
//                           on dY with the taps flipped and the channel roles swapped in the prepared weights)
// conv_tc_kernel<CT_WGRAD>  dW[9 Cin (+1)][Cout] += im2col(X)^T[9 Cin (+1)][128 pixels] * dY[128 pixels][Cout], accumulated in TMEM
//                           over all pixel tiles of a persistent CTA; row 9 Cin of the operand is a column of ones, so the same
//                           MMAs produce the bias gradient; per-CTA partials are reduced in CTA order (deterministic)
// Activations are NHWC bf16 with 16 or 32 channels (the uint8 frames become 16-channel bf16 INTEGERS 0..255, exact in bf16; the
// 1/255 of encoders.py:84 is applied in fp32 to the accumulator).  Nothing is ever materialised as an im2col matrix in HBM:
//   producers  NGRP groups of four warps.  A tile's zero-padded neighbourhood [R + 2][W + 2][Cin] arrives by ONE 4-D TMA per tile into a
//              small ring (out-of-bounds elements read as zero = SAME padding), prefetched a tile ahead, and the producers copy it
//              shared -> shared (odd image sizes: direct gather from L2, one round trip per tile): thread r owns pixel r of the tile; for each of the 9 taps it copies that
//              neighbour's channels (16-byte chunks, zeros outside the image = SAME padding) straight from L2/HBM into the K-major
//              SWIZZLE_128B operand blocks ([128 rows][64 k] bf16) the MMAs read -- the same blocks serve as the MN-major A operand
//              of the weight gradient;
//   2 issuers  (warp 0 and the last warp) one thread each issues tcgen05.mma (M=128, N=64, K=16) for every second tile of the CTA into its own accumulator set
//              (each issuing warp serialises its own barrier waits and instructions); the prepared weights [Kpad][64] arrive once per CTA by TMA and stay
//              resident; operand buffers and accumulators are double-buffered so tile i+1 is gathered while tile i multiplies;
//   4 warps    epilogue: thread per pixel reads its accumulator row from TMEM: x scale + bias, x relu-mask of a saved tensor,
//              + skip / upstream gradient, relu, bf16 NHWC stores (16-byte vectors).
// Pooling (3x3/2, first maximum wins, argmax routing in the backward) and the element-wise pieces are bf16 kernels below; the final
// Dense runs through tc_gemm.cu.
#include "step.cuh"
#include "tc_prims.cuh"

using namespace tc;
typedef __nv_bfloat16 bf16;

namespace {

constexpr int kStacks[3] = {16, 32, 32};
constexpr int TM = 128;
constexpr int BLK = TM * 128;            // one operand block: [128 rows][64 bf16]
#ifndef FQL_CONV_NBUF16
#define FQL_CONV_NBUF16 2   // a multiple of NGRP (see below); the halo ring prefetches the gathers, the operand buffers only cover the MMAs
#endif
// operand buffers = producer groups of a kernel instantiation: the 16-channel forward / input-gradient kernels (48 KB buffers) keep three
__host__ __device__ constexpr int conv_nbuf(int mode, int cin) { return (mode == 0 && cin == 16) ? FQL_CONV_NBUF16 : 2; }
// warps: NGRP MMA issuers | NGRP producer groups of 4 warps | 4 epilogue warps.  Tile i of a CTA uses operand buffer i % NBUF and
// belongs to lane i % NGRP (one producer group, one issuing warp, one accumulator set per lane).  NBUF is a multiple of NGRP, so a
// buffer is always filled and consumed by the same lane: every mbarrier has ONE waiter that sees every one of its phases (a waiter that
// skipped a phase would take the parity of an older phase for the one it waits for -- the failure an odd NBUF produced).
constexpr int NGRP = 2;
__host__ __device__ constexpr int conv_threads(int, int) { return 32 * (5 * NGRP + 4); }
constexpr int KPAD_MAX = 320;            // round_up(9 * 32, 64)
constexpr int WSLOT = KPAD_MAX * 64;     // elements of one prepared weight matrix [Kpad][64]
enum { CT_CONV = 0, CT_WGRAD = 1 };

struct ConvTcArgs {
  const bf16* x;        // input activations, NHWC [npix][CIN]
  int H, W;
  long long npix;
  int tiles;
  // CT_CONV epilogue: v = acc * scale + bias; v = mask > 0 ? v : 0; v += add; v = relu_out ? max(v, 0) : v
  float scale;
  const float* bias;
  const bf16* mask;
  const bf16* add;
  bf16* out;
  bf16* out_relu;       // optional second output max(v, 0)
  int relu_out;
  // CT_WGRAD
  const bf16* dy;       // [npix][COUT]
  float* partial;       // [gridDim.x][krows][COUT]
  int krows;            // 9 * CIN + 1
  // halo staging (halo != 0): a tile = NB images x R rows x W pixels; its zero-padded neighbourhood [NB][R + 2][W + 2][CIN] arrives by ONE
  // TMA (mapX: the NHWC tensor, box {CIN, W + 2, R + 2, NB}, out-of-bounds = zeros = SAME padding) into a ring slot
  int halo, R, NB, tiles_per_image, halo_bytes;
};

__device__ __forceinline__ uint4 ldg16(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// halo ring: slots per lane and bytes per slot (W <= 64 for 16 channels: 4 x 66 pixels; W <= 32 for 32 channels: 6 x 34 pixels)
__host__ __device__ constexpr int halo_nstg(int cin) { return cin == 16 ? 2 : 1; }
__host__ __device__ constexpr int halo_slot(int cin) { return cin == 16 ? 9216 : 13312; }

template <int MODE, int CIN, int COUT>
__global__ void __launch_bounds__(conv_threads(MODE, CIN), 1) conv_tc_kernel(const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapX, const ConvTcArgs a) {
  constexpr int CH = CIN / 8;                       // 16-byte chunks per (pixel, tap)
  constexpr int NCH = 9 * CH;                       // chunks of real K per pixel row
  constexpr int NK16 = (9 * CIN + 15) / 16;         // MMA K steps (CT_CONV)
  constexpr int NKB = (9 * CIN + 1 + 63) / 64;      // operand blocks per buffer that hold data
  constexpr int NMT = (9 * CIN + 1 + 127) / 128;    // M tiles of the weight gradient
  // blocks per buffer.  The weight gradient's last M tile reads a second 64-column chunk one block past the buffer: whatever lies there
  // (the next buffer / the dY tiles: finite bf16 data) only reaches accumulator rows >= 9 CIN + 1, which nobody reads
  constexpr int NBLK = NKB;
  constexpr int NSTG = halo_nstg(CIN), HSLOT = halo_slot(CIN);
  // operand buffers: a tile's gather (one L2 round trip) and its MMAs (~0.7 us) overlap with other tiles only across buffers, so the
  // 16-channel forward / input-gradient kernels, whose buffers are 48 KB, keep three of them
  constexpr int NBUF = conv_nbuf(MODE, CIN);
  constexpr int NTHR = conv_threads(MODE, CIN);
  constexpr int W_EPI = 5 * NGRP;              // first epilogue warp (warps [0, NGRP): MMA issuers, [NGRP, 5 NGRP): producers)
  static_assert(NBUF % NGRP == 0, "a buffer must always belong to the same producer group / MMA issuer");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;                                         // [NBUF][NBLK][BLK]
  uint8_t* sB = sA + NBUF * NBLK * BLK;                       // CT_CONV: weights [NKB * 64 k][64 n]; CT_WGRAD: dY tiles [NBUF][BLK]
  constexpr int NBOX = (NK16 + 1) / 2;                         // 32-row boxes of the prepared weights that hold real K rows
  constexpr int SB_BYTES = (MODE == CT_WGRAD) ? NBUF * BLK : NBOX * 4096;
  uint8_t* sH = sB + ((SB_BYTES + 1023) & ~1023);             // halo ring [NGRP][NSTG][HSLOT]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sH + NGRP * NSTG * HSLOT);
  uint64_t* a_full = bars;          // [4] operand buffer gathered                 (4 producer warps)
  uint64_t* a_empty = bars + 4;     // [4] the MMAs have consumed the buffer       (tcgen05.commit)
  uint64_t* acc_full = bars + 8;    // [4] accumulator complete                    (tcgen05.commit)
  uint64_t* acc_free = bars + 12;   // [4] accumulator read                        (4 epilogue warps)
  uint64_t* b_full = bars + 16;     //     weights landed                          (TMA)
  uint64_t* h_full = bars + 17;     // [NGRP][2] halo slot landed                  (TMA)
  uint64_t* h_empty = bars + 21;    // [NGRP][2] halo slot copied into the operand (4 producer warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 25);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform to ptxas as well
  const int ntl = (a.tiles > (int)blockIdx.x) ? (a.tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;   // tiles of this CTA

  if (warp == 0 && lane == 0) {
    if (MODE == CT_CONV) tma_prefetch_desc(&mapW);
    for (int i = 0; i < 4; i++) {
      mbar_init(&a_full[i], 4);
      mbar_init(&a_empty[i], 1);
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_free[i], 4);
    }
    mbar_init(b_full, 1);
    for (int i = 0; i < 4; i++) {
      mbar_init(&h_full[i], 1);
      mbar_init(&h_empty[i], 4);
    }
    if (a.halo) tma_prefetch_desc(&mapX);
    fence_barrier_init();
  }
  // accumulators: CT_CONV one 64-column set per slot, CT_WGRAD NMT x 64 columns per slot
  constexpr uint32_t TCOLS = (MODE == CT_WGRAD) ? 512u : 128u;
  static_assert(NGRP * NMT * 64 <= 512, "weight-gradient accumulators exceed TMEM");
  if (warp == NGRP) tmem_alloc(tmem_slot, TCOLS);
  // the padding columns of the operand blocks are written once: zeros (and never touched by the gather)
  {
    uint4* z = reinterpret_cast<uint4*>(sA);
    const int n16 = (NBUF * NBLK * BLK + ((MODE == CT_WGRAD) ? NBUF * BLK : 0)) / 16;
    for (int i = threadIdx.x; i < n16; i += NTHR) z[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // programmatic dependent launch: everything above (barriers, TMEM, zeroed operand padding) overlapped the previous kernel's tail; from
  // here on this kernel reads what its predecessors wrote, and its successor may start its own prologue
  FQL_PDL_SYNC();

  if (warp < NGRP) {
    // ================= MMA issuers (+ the one-time weight load) =================
    // Warp g issues the tiles of slot g into accumulator set g.  All 32 lanes run the loop (waits, descriptor arithmetic in uniform
    // registers); the tcgen05 / TMA instructions are predicated on the elected lane -- under `if (lane == 0)` each of them sat in an
    // ELECT + R2UR.BROADCAST waterfall (tc_prims.cuh, profiles/micro/mma_dual_bench.cu).
    const int g = warp;
    const bool el = elect_one();
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    if (ntl > 0) {
      if (MODE == CT_CONV) {
        if (g == 0 && el) {
          // rows [0, NK16 * 16) of the prepared matrix as boxes of 32 rows
          mbar_expect_tx(b_full, NBOX * 4096);
          for (int i = 0; i < NBOX; i++) tma_load_2d(sB + i * 4096, &mapW, b_full, 0, i * 32);
        }
        mbar_wait_u(b_full, 0);
      }
      const uint32_t sa0 = smem_u32(sA) >> 4, sb0 = smem_u32(sB) >> 4;
      if (MODE == CT_CONV) {
        const uint32_t idesc = make_idesc_bf16(128, 64, false, true);
        const uint64_t a_t = make_smem_desc(0, 16, 1024) + (uint64_t)sa0;
        const uint64_t bb = make_smem_desc(0, 4096, 1024) + (uint64_t)sb0;
        const uint32_t tacc = tmem_u + g * 64;
        for (int it = g; it < ntl; it += NGRP) {
          const int buf = it % NBUF, use = it / NGRP;
          mbar_wait_u(&a_full[buf], (it / NBUF) & 1);
          if (use >= 1) mbar_wait_u(&acc_free[g], (use - 1) & 1);
          tc_fence_after();
          const uint64_t ab = a_t + (uint64_t)(buf * NBLK * (BLK >> 4));
          if (el) {
#pragma unroll
            for (int kb = 0; kb < NK16 / 4; kb++)      // one 64-wide K block = four K steps (A: +32 B, B: +16 rows of 128 B)
              umma_bf16_x4(tacc, ab + (uint64_t)(kb * (BLK >> 4)), bb + (uint64_t)(kb * 4 * (2048 >> 4)), 2, 2048 >> 4, idesc, kb > 0);
            if (NK16 % 4 >= 2)
              umma_bf16_x2(tacc, ab + (uint64_t)((NK16 / 4) * (BLK >> 4)), bb + (uint64_t)((NK16 / 4) * 4 * (2048 >> 4)), 2, 2048 >> 4, idesc, 1);
            if (NK16 % 2 == 1)
              umma_bf16(tacc, ab + (uint64_t)((NK16 / 4) * (BLK >> 4) + ((NK16 % 4) - 1) * 2), bb + (uint64_t)((NK16 - 1) * (2048 >> 4)), idesc, 1);
            umma_commit(&a_empty[buf]);
            umma_commit(&acc_full[g]);
          }
        }
      } else {
        const uint32_t idesc = make_idesc_bf16(128, 64, true, true);
        const uint64_t a_t = make_smem_desc(0, BLK, 1024) + (uint64_t)(sa0 + g * NBLK * (BLK >> 4));
        const uint64_t bb = make_smem_desc(0, BLK, 1024) + (uint64_t)(sb0 + g * (BLK >> 4));
        const uint32_t tacc = tmem_u + g * NMT * 64;
        static_assert(MODE != 1 || NBUF == NGRP, "the weight-gradient kernel keeps one buffer per lane");
        for (int it = g; it < ntl; it += NGRP) {
          mbar_wait_u(&a_full[g], (it / NBUF) & 1);
          tc_fence_after();
          if (el) {
#pragma unroll
            for (int mt = 0; mt < NMT; mt++) {
              const uint64_t ab = a_t + (uint64_t)(2 * mt * (BLK >> 4));
              umma_bf16_x4(tacc + mt * 64, ab, bb, 2048 >> 4, 2048 >> 4, idesc, it >= NBUF);
              umma_bf16_x4(tacc + mt * 64, ab + (uint64_t)(4 * (2048 >> 4)), bb + (uint64_t)(4 * (2048 >> 4)), 2048 >> 4, 2048 >> 4, idesc, 1);
            }
            umma_commit(&a_empty[g]);
          }
        }
        if (ntl > g && el) umma_commit(&acc_full[g]);
      }
    }
  } else if (warp < W_EPI) {
    // ================= producers: implicit im2col into the swizzled operand blocks =================
    const int grp = (warp - NGRP) >> 2;        // group g gathers tiles g, g + NGRP, ...
    const int r = ((warp - NGRP) & 3) * 32 + lane;
    const int HW = a.H * a.W;
    const bool issuer = ((warp - NGRP) & 3) == 0 && lane == 0;   // the group's TMA thread (halo staging)
    // halo staging: this pixel's position inside the tile's zero-padded neighbourhood is the same for every tile
    const int PI = a.R * a.W;                  // pixels of one image inside a tile
    const int hb = a.halo ? r / PI : 0, hr = a.halo ? (r % PI) / a.W : 0, hw = a.halo ? r % a.W : 0;
    const int hrow = (a.W + 2) * CIN * 2;      // bytes of one halo row
    const uint32_t hoff = (uint32_t)((hb * (a.R + 2) + hr) * hrow + hw * CIN * 2);
    auto halo_fetch = [&](int it, int slot) {  // TMA of tile it's neighbourhood into ring slot `slot` of this group
      const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
      const int b0 = (a.NB > 1) ? (int)(tile * a.NB) : (int)(tile / a.tiles_per_image);
      const int h0 = (a.NB > 1) ? 0 : (int)(tile % a.tiles_per_image) * a.R;
      uint64_t* bar = &h_full[grp * 2 + slot];
      mbar_expect_tx(bar, a.halo_bytes);
      tma_load_4d(sH + (grp * NSTG + slot) * HSLOT, &mapX, bar, 0, -1, h0 - 1, b0);
    };
    if (a.halo && issuer)
      for (int k = 0; k < NSTG && grp + k * NGRP < ntl; k++) halo_fetch(grp + k * NGRP, k);
    int k = 0;                                 // this group's tile counter
    for (int it = grp; it < ntl; it += NGRP, k++) {
      const int buf = it % NBUF;
      const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
      const long long p = tile * TM + r;
      const bool valid = p < a.npix;
      uint4 dyv[COUT / 8];
      if (MODE == CT_WGRAD) {                  // the dY row of this pixel: in flight while the waits below pass
#pragma unroll
        for (int c = 0; c < COUT / 8; c++) dyv[c] = valid ? ldg16(a.dy + p * COUT + c * 8) : make_uint4(0u, 0u, 0u, 0u);
      }
      if (it >= NBUF) mbar_wait(&a_empty[buf], ((it / NBUF) - 1) & 1);
      uint8_t* A = sA + buf * NBLK * BLK;
      if (a.halo) {
        const int slot = k % NSTG;
        mbar_wait(&h_full[grp * 2 + slot], (k / NSTG) & 1);
        const uint8_t* hp = sH + (grp * NSTG + slot) * HSLOT + hoff;
#pragma unroll
        for (int tap = 0; tap < 9; tap++) {
          const uint8_t* src = hp + (tap / 3) * hrow + (tap % 3) * CIN * 2;
#pragma unroll
          for (int c = 0; c < CH; c++) {
            const int kc = tap * CH + c;
            *reinterpret_cast<uint4*>(A + (kc >> 3) * BLK + sw128_off(r, kc & 7)) = *reinterpret_cast<const uint4*>(src + c * 16);
          }
        }
      } else {
        const int pin = valid ? (int)(p % HW) : 0;
        const int h = pin / a.W, w = pin - h * a.W;
        const bf16* img = a.x + (valid ? (p - pin) : 0) * CIN;
#pragma unroll
        for (int tap = 0; tap < 9; tap++) {
          const int hh = h + tap / 3 - 1, ww = w + tap % 3 - 1;
          const bool inb = valid && hh >= 0 && hh < a.H && ww >= 0 && ww < a.W;
          const bf16* src = img + (long long)(hh * a.W + ww) * CIN;
#pragma unroll
          for (int c = 0; c < CH; c++) {
            const int kc = tap * CH + c;
            const uint4 v = inb ? ldg16(src + c * 8) : make_uint4(0u, 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(A + (kc >> 3) * BLK + sw128_off(r, kc & 7)) = v;
          }
        }
      }
      if (MODE == CT_WGRAD) {
        // column 9*CIN of the operand = 1 (bias gradient), then the dY tile [128 pixels][COUT]
        *reinterpret_cast<uint4*>(A + (NCH >> 3) * BLK + sw128_off(r, NCH & 7)) = make_uint4(valid ? 0x3F80u : 0u, 0u, 0u, 0u);
        uint8_t* Bt = sB + buf * BLK;
#pragma unroll
        for (int c = 0; c < COUT / 8; c++) *reinterpret_cast<uint4*>(Bt + sw128_off(r, c)) = dyv[c];
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&a_full[buf]);
      if (a.halo) {
        // the slot is free once all four warps have copied it out; the group's TMA thread then refills it NSTG tiles ahead
        const int slot = k % NSTG;
        if (lane == 0) mbar_arrive(&h_empty[grp * 2 + slot]);
        if (issuer && it + NSTG * NGRP < ntl) {
          mbar_wait(&h_empty[grp * 2 + slot], (k / NSTG) & 1);
          halo_fetch(it + NSTG * NGRP, slot);
        }
      }
    }
  } else {
    // ================= epilogue =================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t rg[32];
    if (MODE == CT_CONV) {
      float bias[COUT];
#pragma unroll
      for (int c = 0; c < COUT; c++) bias[c] = a.bias ? __ldg(a.bias + c) : 0.f;
      for (int it = 0; it < ntl; it++) {
        const int buf = it % NGRP;               // accumulator set of the tile's lane
        const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
        const long long p = tile * TM + row;
        const bool valid = p < a.npix;
        mbar_wait(&acc_full[buf], (it / NGRP) & 1);
        tc_fence_after();
        tmem_ld32(t_lane + buf * 64, rg);
        tmem_wait_ld();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_free[buf]);
        if (!valid) continue;
#pragma unroll
        for (int c8 = 0; c8 < COUT / 8; c8++) {
          float v[8];
#pragma unroll
          for (int i = 0; i < 8; i++) v[i] = fmaf(__uint_as_float(rg[c8 * 8 + i]), a.scale, bias[c8 * 8 + i]);
          if (a.mask) {
            const uint4 m = ldg16(a.mask + p * COUT + c8 * 8);
            const uint32_t mw[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
            for (int i = 0; i < 4; i++) {
              // bf16 > 0: sign bit clear and not zero
              const uint32_t lo = mw[i] & 0xffffu, hi = mw[i] >> 16;
              if (!(lo != 0u && lo < 0x8000u)) v[2 * i] = 0.f;
              if (!(hi != 0u && hi < 0x8000u)) v[2 * i + 1] = 0.f;
            }
          }
          if (a.add) {
            const uint4 s = ldg16(a.add + p * COUT + c8 * 8);
            const uint32_t sw[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
            for (int i = 0; i < 4; i++) {
              v[2 * i] += __uint_as_float(sw[i] << 16);
              v[2 * i + 1] += __uint_as_float(sw[i] & 0xffff0000u);
            }
          }
          if (a.relu_out) {
#pragma unroll
            for (int i = 0; i < 8; i++) v[i] = fmaxf(v[i], 0.f);
          }
          uint32_t o[4];
#pragma unroll
          for (int i = 0; i < 4; i++) {
            __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
            o[i] = *reinterpret_cast<uint32_t*>(&t);
          }
          *reinterpret_cast<uint4*>(a.out + p * COUT + c8 * 8) = make_uint4(o[0], o[1], o[2], o[3]);
          if (a.out_relu) {
#pragma unroll
            for (int i = 0; i < 4; i++) {
              __nv_bfloat162 t = __floats2bfloat162_rn(fmaxf(v[2 * i], 0.f), fmaxf(v[2 * i + 1], 0.f));
              o[i] = *reinterpret_cast<uint32_t*>(&t);
            }
            *reinterpret_cast<uint4*>(a.out_relu + p * COUT + c8 * 8) = make_uint4(o[0], o[1], o[2], o[3]);
          }
        }
      }
    } else if (ntl > 0) {
      for (int g = 0; g < NGRP && g < ntl; g++) mbar_wait(&acc_full[g], 0);
      tc_fence_after();
      float* part = a.partial + (long long)blockIdx.x * a.krows * COUT;
#pragma unroll 1
      for (int mt = 0; mt < NMT; mt++) {
        tmem_ld32(t_lane + mt * 64, rg);
        tmem_wait_ld();
        for (int g = 1; g < NGRP && g < ntl; g++) {      // the other lanes' tiles accumulated into their own sets
          uint32_t r2[32];
          tmem_ld32(t_lane + (g * NMT + mt) * 64, r2);
          tmem_wait_ld();
#pragma unroll
          for (int c = 0; c < 32; c++) rg[c] = __float_as_uint(__uint_as_float(rg[c]) + __uint_as_float(r2[c]));
        }
        const int kr = mt * 128 + row;
        if (kr < a.krows) {
#pragma unroll
          for (int c = 0; c < COUT; c += 4)
            *reinterpret_cast<float4*>(part + (long long)kr * COUT + c) =
                make_float4(__uint_as_float(rg[c]), __uint_as_float(rg[c + 1]), __uint_as_float(rg[c + 2]), __uint_as_float(rg[c + 3]));
        }
      }
    } else {
      // a CTA without tiles still owns a slot of the partial buffer
      float* part = a.partial + (long long)blockIdx.x * a.krows * COUT;
      for (int i = row; i < a.krows * COUT; i += 128) part[i] = 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == NGRP) tmem_dealloc(tmem_base, TCOLS);
}

// gw[tap][ci][co] = scale * sum_cta partial[cta][tap * CIN + ci][co] (ci < cin_real); gb[co] = sum_cta partial[cta][9 * CIN][co].
// 32 outputs per block; the CTA partials of an output are split over 32 threads (<= 5 independent loads each at 148 CTAs: the
// 8-way split of round 2 was a chain of 19 dependent L2 round trips = 22 us per launch, 27 launches per step) and combined in a
// fixed order (deterministic).
constexpr int WR_SPLIT = 32;
__global__ void __launch_bounds__(32 * WR_SPLIT) wgrad_reduce_kernel(const float* __restrict__ partial, int nctas, int krows, int CIN, int cin_real,
                                                                     int COUT, float scale, float* __restrict__ gw, float* __restrict__ gb) {
  __shared__ float red[WR_SPLIT][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + tx;
  const int n_w = 9 * cin_real * COUT;
  const bool live = i < n_w + COUT;
  int kr = 0, co = 0;
  if (live) {
    if (i < n_w) {
      co = i % COUT;
      const int t = i / COUT, ci = t % cin_real, tap = t / cin_real;
      kr = tap * CIN + ci;
    } else {
      co = i - n_w;
      kr = 9 * CIN;
    }
  }
  float s = 0.f;
  if (live) {
    const float* src = partial + (long long)kr * COUT + co;
    const long long stride = (long long)krows * COUT;
    int c = ty;
    for (; c + 3 * WR_SPLIT < nctas; c += 4 * WR_SPLIT) {
      const float v0 = src[c * stride], v1 = src[(c + WR_SPLIT) * stride], v2 = src[(c + 2 * WR_SPLIT) * stride], v3 = src[(c + 3 * WR_SPLIT) * stride];
      s += v0; s += v1; s += v2; s += v3;
    }
    for (; c < nctas; c += WR_SPLIT) s += src[c * stride];
  }
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && live) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < WR_SPLIT; k++) t += red[k][tx];
    if (i < n_w) gw[i] = t * scale;
    else gb[co] = t;
  }
}

// ---- prepared bf16 weights of one encoder -----------------------------------------------------------------------
struct PrepJob {
  long long off_w;       // fp32 HWIO kernel [3][3][cin][cout] in the arena
  int cin, cin_p, cout;  // cin_p: channels of the activation tensor the forward reads (16 for the 9-channel frames)
};
struct PrepArgs {
  PrepJob job[9];
  long long off_dense;
  int flat_dim, feat;
};
// grid (x, 19): y < 9 forward matrix of conv y, 9 <= y < 18 input-gradient matrix of conv y - 9, y == 18 the Dense kernel
//   forward   Wf[k = tap * cin_p + ci][n = co] = W[tap][ci][co]
//   dgrad     Wd[k = tap * cout + co][n = ci]  = W[8 - tap][ci][co]      (flipped taps: encoders.py conv is its own transpose up to that)
__global__ void enc_prep_weights_kernel(const float* __restrict__ params, PrepArgs pa, bf16* __restrict__ wf, bf16* __restrict__ wd,
                                        bf16* __restrict__ dense) {
  const int y = blockIdx.y;
  if (y == 18) {
    const long long n = (long long)pa.flat_dim * pa.feat;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
      dense[i] = __float2bfloat16(params[pa.off_dense + i]);
    return;
  }
  const PrepJob j = pa.job[y % 9];
  if (j.cout == 0) return;
  const float* W = params + j.off_w;
  const bool fwd = y < 9;
  bf16* dst = (fwd ? wf : wd) + (long long)(y % 9) * WSLOT;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < WSLOT; i += gridDim.x * blockDim.x) {
    const int k = i >> 6, n = i & 63;
    float v = 0.f;
    if (fwd) {
      const int tap = k / j.cin_p, ci = k - tap * j.cin_p;
      if (tap < 9 && ci < j.cin && n < j.cout) v = W[(tap * j.cin + ci) * j.cout + n];
    } else {
      const int tap = k / j.cout, co = k - tap * j.cout;
      if (tap < 9 && n < j.cin) v = W[((8 - tap) * j.cin + n) * j.cout + co];
    }
    dst[i] = __float2bfloat16(v);
  }
}

// uint8 frames [npix][C] -> bf16 [npix][16], the integer values themselves (exact), channels >= C zero
__global__ void enc_image_kernel(const uint8_t* __restrict__ img, bf16* __restrict__ out, long long npix, int C) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npix) return;
  uint32_t o[8];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const float v0 = (2 * i < C) ? (float)img[p * C + 2 * i] : 0.f, v1 = (2 * i + 1 < C) ? (float)img[p * C + 2 * i + 1] : 0.f;
    __nv_bfloat162 t = __floats2bfloat162_rn(v0, v1);
    o[i] = *reinterpret_cast<uint32_t*>(&t);
  }
  uint4* q = reinterpret_cast<uint4*>(out + p * 16);
  q[0] = make_uint4(o[0], o[1], o[2], o[3]);
  q[1] = make_uint4(o[4], o[5], o[6], o[7]);
}

__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

// max_pool 3x3 stride 2 'SAME' (-inf padding; first maximum in row-major order wins, as encoder.cu / the oracle), 8 channels per
// thread.  Writes p (skip connection), relu(p) (operand of the first residual convolution) and the argmax (backward routing).
__global__ void pool_fwd_bf16_kernel(const bf16* __restrict__ in, bf16* __restrict__ out, bf16* __restrict__ out_relu, uint8_t* __restrict__ arg,
                                     long long B, int H, int W, int C) {
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2, C8 = C / 8;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * Ho * Wo * C8) return;
  const int c8 = (int)(i % C8), xo = (int)((i / C8) % Wo), yo = (int)((i / ((long long)C8 * Wo)) % Ho);
  const long long b = i / ((long long)C8 * Wo * Ho);
  const int lo_h = ((Ho - 1) * 2 + 3 - H) / 2, lo_w = ((Wo - 1) * 2 + 3 - W) / 2;
  float best[8];
  int bk[8];
#pragma unroll
  for (int k = 0; k < 8; k++) { best[k] = -INFINITY; bk[k] = -1; }
  for (int ky = 0; ky < 3; ky++) {
    const int iy = 2 * yo + ky - lo_h;
    if (iy < 0 || iy >= H) continue;
    for (int kx = 0; kx < 3; kx++) {
      const int ix = 2 * xo + kx - lo_w;
      if (ix < 0 || ix >= W) continue;
      const uint4 q = ldg16(in + ((b * H + iy) * W + ix) * C + c8 * 8);
      const uint32_t qw[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const float v0 = bf_lo(qw[k]), v1 = bf_hi(qw[k]);
        if (v0 > best[2 * k] || bk[2 * k] < 0) { best[2 * k] = v0; bk[2 * k] = ky * 3 + kx; }
        if (v1 > best[2 * k + 1] || bk[2 * k + 1] < 0) { best[2 * k + 1] = v1; bk[2 * k + 1] = ky * 3 + kx; }
      }
    }
  }
  uint32_t o[4], orl[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    __nv_bfloat162 t = __floats2bfloat162_rn(best[2 * k], best[2 * k + 1]);
    o[k] = *reinterpret_cast<uint32_t*>(&t);
    __nv_bfloat162 u = __floats2bfloat162_rn(fmaxf(best[2 * k], 0.f), fmaxf(best[2 * k + 1], 0.f));
    orl[k] = *reinterpret_cast<uint32_t*>(&u);
  }
  const long long o8 = ((b * Ho + yo) * Wo + xo) * C + c8 * 8;
  *reinterpret_cast<uint4*>(out + o8) = make_uint4(o[0], o[1], o[2], o[3]);
  *reinterpret_cast<uint4*>(out_relu + o8) = make_uint4(orl[0], orl[1], orl[2], orl[3]);
  uint32_t a0 = 0, a1 = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) { a0 |= (uint32_t)bk[k] << (8 * k); a1 |= (uint32_t)bk[4 + k] << (8 * k); }
  *reinterpret_cast<uint2*>(arg + o8) = make_uint2(a0, a1);
}

// gather form of the pooling gradient: an input pixel sums the windows whose argmax points at it (fixed order: deterministic)
__global__ void pool_bwd_bf16_kernel(const bf16* __restrict__ dout, const uint8_t* __restrict__ arg, bf16* __restrict__ din, long long B, int H,
                                     int W, int C) {
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2, C8 = C / 8;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * H * W * C8) return;
  const int c8 = (int)(i % C8), x = (int)((i / C8) % W), y = (int)((i / ((long long)C8 * W)) % H);
  const long long b = i / ((long long)C8 * W * H);
  const int lo_h = ((Ho - 1) * 2 + 3 - H) / 2, lo_w = ((Wo - 1) * 2 + 3 - W) / 2;
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int yo = (y + lo_h) / 2 - 1; yo <= (y + lo_h) / 2; yo++) {
    const int ky = y + lo_h - 2 * yo;
    if (yo < 0 || yo >= Ho || ky < 0 || ky > 2) continue;
    for (int xo = (x + lo_w) / 2 - 1; xo <= (x + lo_w) / 2; xo++) {
      const int kx = x + lo_w - 2 * xo;
      if (xo < 0 || xo >= Wo || kx < 0 || kx > 2) continue;
      const long long o8 = ((b * Ho + yo) * Wo + xo) * C + c8 * 8;
      const uint2 ag = *reinterpret_cast<const uint2*>(arg + o8);
      const uint4 q = ldg16(dout + o8);
      const uint32_t qw[4] = {q.x, q.y, q.z, q.w};
      const uint32_t me = (uint32_t)(ky * 3 + kx);
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const uint32_t ak = ((k < 4 ? ag.x : ag.y) >> (8 * (k & 3))) & 0xffu;
        if (ak == me) s[k] += (k & 1) ? bf_hi(qw[k >> 1]) : bf_lo(qw[k >> 1]);
      }
    }
  }
  uint32_t o[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    __nv_bfloat162 t = __floats2bfloat162_rn(s[2 * k], s[2 * k + 1]);
    o[k] = *reinterpret_cast<uint32_t*>(&t);
  }
  *reinterpret_cast<uint4*>(din + i * 8) = make_uint4(o[0], o[1], o[2], o[3]);
}

// features = gelu(z)                                                        (networks.py:56, activate_final)
__global__ void enc_gelu_kernel(const float* __restrict__ z, float* __restrict__ feat, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) feat[i] = gelu_tanh_f(z[i]);
}
// dz = dfeat * gelu'(z), in fp32 (bias gradient) and bf16 (GEMM operand)
__global__ void enc_dz_kernel(const float* __restrict__ dfeat, const float* __restrict__ z, float* __restrict__ dz, bf16* __restrict__ dzb, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = dfeat[i] * gelu_tanh_grad_f(z[i]);
  dz[i] = v;
  dzb[i] = __float2bfloat16(v);
}
// dx = dflat * (relu(x_last) > 0) -> bf16
__global__ void enc_relu_mask_kernel(const float* __restrict__ d, const bf16* __restrict__ xr, bf16* __restrict__ out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float2bfloat16(__bfloat162float(xr[i]) > 0.f ? d[i] : 0.f);
}

// prepared weights [rows][64] bf16 as boxes of [32 k][64 n]
int make_map_w(CUtensorMap* m, const void* base, int rows) {
  auto enc = get_encode();
  FQL_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {64, (cuuint64_t)rows};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {64, 32};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FQL_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(conv weights) failed (%d)", (int)r);
  return 0;
}

// Halo staging applies when a 128-pixel tile is R full rows of one image (W divides 128, R = 128 / W divides H) or NB whole images
// (H W divides 128), and the neighbourhood fits the ring slot; other geometries (odd image sizes) use the direct gather.
// mapX: the NHWC activation tensor {C, W, H, B} with box {C, W + 2, R + 2, NB}, no swizzle, out-of-bounds elements read as zero.
int conv_halo_setup(ConvTcArgs& a, CUtensorMap* mapX, const void* x, int cin, long long B) {
  memset(mapX, 0, sizeof(*mapX));
  a.halo = 0; a.R = 1; a.NB = 1; a.tiles_per_image = 1; a.halo_bytes = 0;
  static const bool off = getenv("FQL_B200_CONV_HALO") && getenv("FQL_B200_CONV_HALO")[0] == '0';
  if (off) return 0;
  const int H = a.H, W = a.W;
  int R = 0, NB = 0;
  if (W <= TM && TM % W == 0 && H % (TM / W) == 0) { R = TM / W; NB = 1; }
  else if (H * W < TM && TM % (H * W) == 0) { R = H; NB = TM / (H * W); }
  else return 0;
  const long long bytes = (long long)NB * (R + 2) * (W + 2) * cin * 2;
  if (bytes > halo_slot(cin) || W + 2 > 256 || R + 2 > 256) return 0;
  auto enc = get_encode();
  FQL_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[4] = {(cuuint64_t)cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)cin * 2, (cuuint64_t)W * cin * 2, (cuuint64_t)H * W * cin * 2};
  cuuint32_t box[4] = {(cuuint32_t)cin, (cuuint32_t)(W + 2), (cuuint32_t)(R + 2), (cuuint32_t)NB};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(mapX, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FQL_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(conv halo) failed (%d): C %d W %d H %d B %lld box %d x %d x %d", (int)r, cin, W, H, B, W + 2, R + 2, NB);
  a.halo = 1; a.R = R; a.NB = NB; a.tiles_per_image = (NB == 1) ? H / R : 1; a.halo_bytes = (int)bytes;
  return 0;
}

template <int MODE, int CIN, int COUT>
int launch_conv_t(const CUtensorMap& mapW, const CUtensorMap& mapX, const ConvTcArgs& a, int grid, cudaStream_t st) {
  constexpr int NKB = (9 * CIN + 1 + 63) / 64, NK16 = (9 * CIN + 15) / 16, NBOX = (NK16 + 1) / 2;
  constexpr int NBUF = conv_nbuf(MODE, CIN);
  constexpr int SB = ((MODE == CT_WGRAD) ? NBUF * BLK : NBOX * 4096);
  constexpr int SMEM = NBUF * NKB * BLK + ((SB + 1023) & ~1023) + NGRP * halo_nstg(CIN) * halo_slot(CIN) + 256 + 1024;
  static_assert(SMEM <= 232448, "conv_tc_kernel: shared memory");
  auto kern = conv_tc_kernel<MODE, CIN, COUT>;
  static bool attr_set[FQL_MAX_DEVICES] = {};
  const int dev = fql_current_device();
  if (!attr_set[dev]) {
    FQL_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    attr_set[dev] = true;
  }
  FQL_CHECK_CUDA(fql_launch_pdl(kern, dim3(grid), dim3(conv_threads(MODE, CIN)), SMEM, st, mapW, mapX, a));
  FQL_CHECK_LAUNCH();
  return 0;
}

int num_sms() {
  static int n[FQL_MAX_DEVICES] = {};
  const int dev = fql_current_device();
  if (!n[dev]) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, dev) == cudaSuccess) n[dev] = p.multiProcessorCount;
    if (n[dev] <= 0) n[dev] = 148;
  }
  return n[dev];
}

// out[npix][cout] = epilogue(conv3x3(x[npix][cin]) with the prepared matrix wb [Kpad][64])
int conv_tc(const bf16* x, int cin, int cout, const bf16* wb, long long B, int H, int W, float scale, const float* bias, const bf16* mask,
            const bf16* add, int relu_out, bf16* out, bf16* out_relu, cudaStream_t st) {
  ConvTcArgs a;
  memset(&a, 0, sizeof(a));
  a.x = x; a.H = H; a.W = W; a.npix = B * H * W; a.tiles = (int)((a.npix + TM - 1) / TM);
  a.scale = scale; a.bias = bias; a.mask = mask; a.add = add; a.relu_out = relu_out; a.out = out; a.out_relu = out_relu;
  const int grid = a.tiles < num_sms() ? a.tiles : num_sms();
  if (grid <= 0) return 0;
  CUtensorMap mapW, mapX;
  FQL_TRY(make_map_w(&mapW, wb, KPAD_MAX));
  FQL_TRY(conv_halo_setup(a, &mapX, x, cin, B));
  if (cin == 16 && cout == 16) return launch_conv_t<CT_CONV, 16, 16>(mapW, mapX, a, grid, st);
  if (cin == 16 && cout == 32) return launch_conv_t<CT_CONV, 16, 32>(mapW, mapX, a, grid, st);
  if (cin == 32 && cout == 32) return launch_conv_t<CT_CONV, 32, 32>(mapW, mapX, a, grid, st);
  if (cin == 32 && cout == 16) return launch_conv_t<CT_CONV, 32, 16>(mapW, mapX, a, grid, st);
  FQL_REQUIRE(false, "conv_tc: unsupported channel counts %d -> %d", cin, cout);
  return 1;
}

// gw [3][3][cin_real][cout], gb [cout] from x [npix][cin] and dY [npix][cout]
int conv_wgrad_tc(const bf16* x, int cin, int cin_real, int cout, const bf16* dy, long long B, int H, int W, float scale, float* partial,
                  float* gw, float* gb, cudaStream_t st) {
  ConvTcArgs a;
  memset(&a, 0, sizeof(a));
  a.x = x; a.H = H; a.W = W; a.npix = B * H * W; a.tiles = (int)((a.npix + TM - 1) / TM);
  a.dy = dy; a.partial = partial; a.krows = 9 * cin + 1;
  const int grid = a.tiles < num_sms() ? a.tiles : num_sms();
  if (grid <= 0) return 0;
  CUtensorMap mapW, mapX;
  memset(&mapW, 0, sizeof(mapW));
  FQL_TRY(conv_halo_setup(a, &mapX, x, cin, B));
  if (cin == 16 && cout == 16) FQL_TRY((launch_conv_t<CT_WGRAD, 16, 16>(mapW, mapX, a, grid, st)));
  else if (cin == 16 && cout == 32) FQL_TRY((launch_conv_t<CT_WGRAD, 16, 32>(mapW, mapX, a, grid, st)));
  else if (cin == 32 && cout == 32) FQL_TRY((launch_conv_t<CT_WGRAD, 32, 32>(mapW, mapX, a, grid, st)));
  else FQL_REQUIRE(false, "conv_wgrad_tc: unsupported channel counts %d -> %d", cin, cout);
  const int n = 9 * cin_real * cout + cout;
  wgrad_reduce_kernel<<<(n + 31) / 32, 32 * WR_SPLIT, 0, st>>>(partial, grid, a.krows, cin, cin_real, cout, scale, gw, gb);
  FQL_CHECK_LAUNCH();
  return 0;
}

template <typename K, typename... Args>
int launch1d(K kern, long long n, cudaStream_t st, Args... args) {
  if (n <= 0) return 0;
  kern<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(args...);
  FQL_CHECK_LAUNCH();
  return 0;
}

TcOperand opnd(const void* p, int inner, int rows) {
  TcOperand o;
  memset(&o, 0, sizeof(o));
  o.ptr = p; o.inner = inner; o.rows = rows; o.ld = inner; o.g0 = 1; o.g1 = 1;
  return o;
}
TcPtr tptr(void* p, int ld) {
  TcPtr t;
  memset(&t, 0, sizeof(t));
  t.base = p; t.ld = ld;
  return t;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// buffers of one tensor-core encoder pass (bf16 activations)
// ---------------------------------------------------------------------------------------------------------------
size_t enc_tc_carve(const FqlDims* d, int64_t B, void* base, EncBuf* e, bool for_backward) {
  char* p = reinterpret_cast<char*>(base);
  size_t off = 0;
  auto take = [&](int64_t nbytes) {
    off = (off + 255) & ~(size_t)255;
    void* r = base ? reinterpret_cast<void*>(p + off) : nullptr;
    off += (size_t)nbytes;
    return r;
  };
  int H = d->reserved[0], W = d->reserved[1];
  EncTc& t = e->tc;
  t.img = take(B * H * W * 16 * 2);
  t.y0 = take(B * H * W * 32 * 2);      // pre-pool convolution output / its gradient (largest: 16 channels at full resolution)
  for (int i = 0; i < 3; i++) {
    const int f = kStacks[i];
    const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
    const int64_t n = B * Ho * Wo * f;
    t.p[i] = take(n * 2);
    t.r1[i] = take(n * 2);
    t.r2[i] = take(n * 2);
    t.xs[i] = take(n * 2);
    e->arg[i] = reinterpret_cast<uint8_t*>(take(n));
    H = Ho; W = Wo;
  }
  e->flat_dim = H * W * kStacks[2];
  t.flat = take(B * e->flat_dim * 2);
  e->z = reinterpret_cast<float*>(take(B * d->obs_dim * 4));
  t.wf = take((int64_t)9 * WSLOT * 2);
  t.wd = take((int64_t)9 * WSLOT * 2);
  t.wdense = take((int64_t)e->flat_dim * d->obs_dim * 2);
  if (for_backward) {
    e->dz = reinterpret_cast<float*>(take(B * d->obs_dim * 4));
    t.dzb = take(B * d->obs_dim * 2);
    e->dflat = reinterpret_cast<float*>(take(B * e->flat_dim * 4));
    const int64_t big2 = B * ((d->reserved[0] + 1) / 2) * ((d->reserved[1] + 1) / 2) * 32;
    t.da = take(big2 * 2);
    t.db = take(big2 * 2);
    t.dc = take(big2 * 2);
    e->partial = reinterpret_cast<float*>(take((int64_t)160 * (9 * 32 + 1) * 32 * 4));
  }
  return off + 256;
}

int enc_tc_forward(const FqlDims* d, const EncView& v, const float* params, const uint8_t* obs, int64_t B, const EncBuf& e, float* feat,
                   cudaStream_t st) {
  int H = d->reserved[0], W = d->reserved[1], C = d->reserved[2];
  FQL_REQUIRE(C <= 16 && d->obs_dim % 64 == 0, "tensor-core encoder: %d image channels (max 16), feature width %d", C, d->obs_dim);
  const EncTc& t = e.tc;
  bf16* wf = reinterpret_cast<bf16*>(t.wf);
  // prepared bf16 operands of this encoder's weights (forward + input-gradient matrices of the 9 convolutions, the Dense kernel)
  PrepArgs pa;
  memset(&pa, 0, sizeof(pa));
  {
    int cin = C;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) {
        PrepJob& jb = pa.job[i * 3 + j];
        jb.off_w = v.off_cw[i][j];
        jb.cin = (j == 0) ? cin : kStacks[i];
        jb.cin_p = (i == 0 && j == 0) ? 16 : jb.cin;
        jb.cout = kStacks[i];
        if (j == 2) cin = kStacks[i];
      }
    pa.off_dense = v.off_dw; pa.flat_dim = e.flat_dim; pa.feat = d->obs_dim;
  }
  enc_prep_weights_kernel<<<dim3(64, 19), 256, 0, st>>>(params, pa, wf, reinterpret_cast<bf16*>(t.wd), reinterpret_cast<bf16*>(t.wdense));
  FQL_CHECK_LAUNCH();
  FQL_TRY(launch1d(enc_image_kernel, B * H * W, st, obs, reinterpret_cast<bf16*>(t.img), (long long)B * H * W, C));
  const bf16* xin = reinterpret_cast<const bf16*>(t.img);
  int cin = 16;
  for (int i = 0; i < 3; i++) {
    const int f = kStacks[i];
    const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
    bf16 *y0 = reinterpret_cast<bf16*>(t.y0), *p = reinterpret_cast<bf16*>(t.p[i]), *r1 = reinterpret_cast<bf16*>(t.r1[i]),
         *r2 = reinterpret_cast<bf16*>(t.r2[i]), *xs = reinterpret_cast<bf16*>(t.xs[i]);
    FQL_TRY(conv_tc(xin, cin, f, wf + (i * 3 + 0) * WSLOT, B, H, W, i == 0 ? 1.0f / 255.0f : 1.0f, params + v.off_cb[i][0], nullptr, nullptr, 0,
                    y0, nullptr, st));
    FQL_TRY(launch1d(pool_fwd_bf16_kernel, B * Ho * Wo * (f / 8), st, (const bf16*)y0, p, r1, e.arg[i], (long long)B, H, W, f));
    FQL_TRY(conv_tc(r1, f, f, wf + (i * 3 + 1) * WSLOT, B, Ho, Wo, 1.0f, params + v.off_cb[i][1], nullptr, nullptr, 1, r2, nullptr, st));
    FQL_TRY(conv_tc(r2, f, f, wf + (i * 3 + 2) * WSLOT, B, Ho, Wo, 1.0f, params + v.off_cb[i][2], nullptr, p, 0, xs,
                    i == 2 ? reinterpret_cast<bf16*>(t.flat) : nullptr, st));
    xin = xs; cin = f; H = Ho; W = Wo;
  }
  // z = relu(x).flatten() @ Wd + bd ; features = gelu(z)
  TcGemmSpec g;
  memset(&g, 0, sizeof(g));
  g.M = (int)B; g.N = d->obs_dim; g.K = e.flat_dim; g.G0 = 1; g.G1 = 1; g.a_mn = 0; g.b_mn = 1;
  g.A = opnd(t.flat, e.flat_dim, (int)B);
  g.B = opnd(t.wdense, d->obs_dim, e.flat_dim);
  g.mode = TC_MODE_STORE_F32;
  g.bias = tptr(const_cast<float*>(params + v.off_db), 0);
  g.out_f = tptr(e.z, d->obs_dim);
  FQL_TRY(tc_gemm(g, st));
  FQL_TRY(launch1d(enc_gelu_kernel, B * d->obs_dim, st, (const float*)e.z, feat, (long long)B * d->obs_dim));
  return 0;
}

int enc_tc_backward(const FqlDims* d, const EncView& v, const float* params, float* grads, const uint8_t* obs, int64_t B, const EncBuf& e,
                    const float* dfeat, cudaStream_t st) {
  (void)obs; (void)params;
  const int F = d->obs_dim;
  const EncTc& t = e.tc;
  bf16* wdg = reinterpret_cast<bf16*>(t.wd);
  FQL_TRY(launch1d(enc_dz_kernel, B * F, st, dfeat, (const float*)e.z, e.dz, reinterpret_cast<bf16*>(t.dzb), (long long)B * F));
  TcGemmSpec g;
  memset(&g, 0, sizeof(g));   // dWd = flat^T dz
  g.M = e.flat_dim; g.N = F; g.K = (int)B; g.G0 = 1; g.G1 = 1; g.a_mn = 1; g.b_mn = 1;
  g.A = opnd(t.flat, e.flat_dim, (int)B);
  g.B = opnd(t.dzb, F, (int)B);
  g.mode = TC_MODE_STORE_F32;
  g.out_f = tptr(grads + v.off_dw, F);
  FQL_TRY(tc_gemm(g, st));
  ColSumArgs c;
  memset(&c, 0, sizeof(c));
  c.P = 1; c.S = 1; c.E = 1; c.M = (int)B; c.N = F; c.ld = F;
  c.X.base[0] = e.dz;
  c.out.base[0] = grads + v.off_db;
  FQL_TRY(launch_colsum(c, st));
  memset(&g, 0, sizeof(g));   // dflat = dz Wd^T  (the [flat, 512] kernel read as a K-major operand: n = flat, k = 512)
  g.M = (int)B; g.N = e.flat_dim; g.K = F; g.G0 = 1; g.G1 = 1; g.a_mn = 0; g.b_mn = 0;
  g.A = opnd(t.dzb, F, (int)B);
  g.B = opnd(t.wdense, F, e.flat_dim);
  g.mode = TC_MODE_STORE_F32;
  g.out_f = tptr(e.dflat, e.flat_dim);
  FQL_TRY(tc_gemm(g, st));
  int Hs[4], Ws[4], Cs[4];
  Hs[0] = d->reserved[0]; Ws[0] = d->reserved[1]; Cs[0] = 16;
  for (int i = 0; i < 3; i++) { Hs[i + 1] = (Hs[i] + 1) / 2; Ws[i + 1] = (Ws[i] + 1) / 2; Cs[i + 1] = kStacks[i]; }
  bf16 *dx = reinterpret_cast<bf16*>(t.da), *other = reinterpret_cast<bf16*>(t.dc), *dc1 = reinterpret_cast<bf16*>(t.db);
  bf16* dy0 = reinterpret_cast<bf16*>(t.y0);
  FQL_TRY(launch1d(enc_relu_mask_kernel, B * e.flat_dim, st, (const float*)e.dflat, reinterpret_cast<const bf16*>(t.flat), dx,
                   (long long)B * e.flat_dim));
  for (int i = 2; i >= 0; i--) {
    const int f = kStacks[i], Ho = Hs[i + 1], Wo = Ws[i + 1], H = Hs[i], W = Ws[i], C = Cs[i];
    const bf16 *p = reinterpret_cast<const bf16*>(t.p[i]), *r1 = reinterpret_cast<const bf16*>(t.r1[i]), *r2 = reinterpret_cast<const bf16*>(t.r2[i]);
    (void)p;
    // conv2: input relu(c1) = r2, output gradient dx
    FQL_TRY(conv_wgrad_tc(r2, f, f, f, dx, B, Ho, Wo, 1.0f, e.partial, grads + v.off_cw[i][2], grads + v.off_cb[i][2], st));
    // dc1 = dgrad(dx, W2) * (c1 > 0)
    FQL_TRY(conv_tc(dx, f, f, wdg + (i * 3 + 2) * WSLOT, B, Ho, Wo, 1.0f, nullptr, r2, nullptr, 0, dc1, nullptr, st));
    // conv1: input relu(pool) = r1, output gradient dc1
    FQL_TRY(conv_wgrad_tc(r1, f, f, f, dc1, B, Ho, Wo, 1.0f, e.partial, grads + v.off_cw[i][1], grads + v.off_cb[i][1], st));
    // dpool = dx (skip) + dgrad(dc1, W1) * (pool > 0)
    FQL_TRY(conv_tc(dc1, f, f, wdg + (i * 3 + 1) * WSLOT, B, Ho, Wo, 1.0f, nullptr, r1, dx, 0, other, nullptr, st));
    // dc0 = pool_bwd(dpool)
    FQL_TRY(launch1d(pool_bwd_bf16_kernel, B * H * W * (f / 8), st, (const bf16*)other, (const uint8_t*)e.arg[i], dy0, (long long)B, H, W, f));
    // conv0: input = previous stack's output (or the frames), output gradient dc0
    const bf16* xin = i ? reinterpret_cast<const bf16*>(t.xs[i - 1]) : reinterpret_cast<const bf16*>(t.img);
    FQL_TRY(conv_wgrad_tc(xin, C, i ? C : d->reserved[2], f, dy0, B, H, W, i ? 1.0f : 1.0f / 255.0f, e.partial, grads + v.off_cw[i][0],
                          grads + v.off_cb[i][0], st));
    if (i > 0)  // gradient w.r.t. the previous stack's output (no relu between stacks)
      FQL_TRY(conv_tc(dy0, f, C, wdg + (i * 3 + 0) * WSLOT, B, H, W, 1.0f, nullptr, nullptr, nullptr, 0, dx, nullptr, st));
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Stand-alone entry points of the convolution kernels (include/fql_b200.h): what the encoder passes above are made of, exposed so
// that the tensor-core arithmetic can be checked exactly (bf16-representable inputs, fp32 accumulation) -- tests/test_conv_tc_gpu.py
// ---------------------------------------------------------------------------------------------------------------
extern "C" size_t fql_conv3x3_workspace_bytes(void) { return (size_t)2 * 9 * WSLOT * 2 + (size_t)160 * (9 * 32 + 1) * 32 * 4 + 1024; }

extern "C" int fql_conv3x3_bf16(const void* x, const float* w_hwio, const float* bias, int32_t B, int32_t H, int32_t W, int32_t cin, int32_t cout,
                                int32_t input_gradient, const void* mask, const void* add, int32_t relu_out, void* out, void* workspace,
                                size_t ws_bytes, void* stream) {
  FQL_REQUIRE(x && w_hwio && out && workspace && ws_bytes >= fql_conv3x3_workspace_bytes(), "fql_conv3x3_bf16: NULL argument / workspace too small");
  FQL_REQUIRE((cin == 16 || cin == 32) && (cout == 16 || cout == 32) && B >= 1 && H >= 1 && W >= 1, "fql_conv3x3_bf16: %d -> %d channels", cin, cout);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  bf16* wf = reinterpret_cast<bf16*>(workspace);
  bf16* wd = wf + 9 * WSLOT;
  PrepArgs pa;
  memset(&pa, 0, sizeof(pa));
  pa.job[0].off_w = 0; pa.job[0].cin = cin; pa.job[0].cin_p = cin; pa.job[0].cout = cout;
  enc_prep_weights_kernel<<<dim3(16, 18), 256, 0, st>>>(w_hwio, pa, wf, wd, nullptr);
  FQL_CHECK_LAUNCH();
  // input gradient: x is dY [B,H,W,cout] and out is dX [B,H,W,cin] of the convolution whose kernel is w_hwio [3,3,cin,cout]
  if (input_gradient)
    return conv_tc(reinterpret_cast<const bf16*>(x), cout, cin, wd, B, H, W, 1.0f, bias, reinterpret_cast<const bf16*>(mask),
                   reinterpret_cast<const bf16*>(add), relu_out, reinterpret_cast<bf16*>(out), nullptr, st);
  return conv_tc(reinterpret_cast<const bf16*>(x), cin, cout, wf, B, H, W, 1.0f, bias, reinterpret_cast<const bf16*>(mask),
                 reinterpret_cast<const bf16*>(add), relu_out, reinterpret_cast<bf16*>(out), nullptr, st);
}

extern "C" int fql_conv3x3_wgrad_bf16(const void* x, const void* dy, int32_t B, int32_t H, int32_t W, int32_t cin, int32_t cout, float* gw, float* gb,
                                      void* workspace, size_t ws_bytes, void* stream) {
  FQL_REQUIRE(x && dy && gw && gb && workspace && ws_bytes >= fql_conv3x3_workspace_bytes(), "fql_conv3x3_wgrad_bf16: NULL argument / workspace too small");
  FQL_REQUIRE((cin == 16 || cin == 32) && (cout == 16 || cout == 32) && !(cin == 32 && cout == 16), "fql_conv3x3_wgrad_bf16: %d -> %d channels", cin, cout);
  float* partial = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + (size_t)2 * 9 * WSLOT * 2);
  return conv_wgrad_tc(reinterpret_cast<const bf16*>(x), cin, cin, cout, reinterpret_cast<const bf16*>(dy), B, H, W, 1.0f, partial, gw, gb,
                       reinterpret_cast<cudaStream_t>(stream));
}
