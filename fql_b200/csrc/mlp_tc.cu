// mlp_tc.cu -- the tensor-core (FQL_PRECISION_BF16_TC) forward path: ONE persistent kernel runs a whole MLP -- and, for
// compute_flow_actions (agents/fql.py:155-171), the whole flow_steps-long Euler loop -- for a 128-row tile:
//
//   warp 0   TMA producer : streams the bf16 shadow weights of every layer as MN-major SWIZZLE_128B B-tiles
//                           (kernel leaves are Flax [in,out] row-major, so a [16 k][64 n] box IS the canonical MN-major atom)
//   warps 1-2 MMA issuers : tcgen05.mma kind::f16, M=128, N<=256 per instruction, one 256-column half of the accumulator each
//                           ; fp32 accumulators in all 512 TMEM columns
//   warps 3-6 epilogue    : one thread per row (tcgen05.ld 32x32b): + bias, GELU(tanh), optional LayerNorm with per-thread row
//                           statistics (the 128x512 fp32 accumulator is exactly one SM's TMEM, so LN needs no cross-thread
//                           reduction), bf16 re-pack straight into the next layer's K-major SWIZZLE_128B A operand in smem.
//
// Activations never leave the SM between layers (or Euler steps); optional fp32 / bf16 copies of Z / H go to HBM for the backward.
// Used where there are enough 128-row tiles to fill the GPU (large batch, many seeds) and for sample_actions; at batch 256 the
// cluster kernels of euler_cluster.cu split one tile over 16 SMs instead.
// Reference arithmetic: utils/networks.py:34-61 (MLP), :153-195 (Value), :198-235 (ActorVectorField).
#include "step.cuh"
#include "tc_prims.cuh"

#include <map>
#include <vector>

using namespace tc;

namespace {

constexpr int TILE_M = 128;
constexpr int KB_BYTES = TILE_M * 128;  // one K-block of an A operand: [128 rows][64 bf16]
constexpr int STAGE_K = 16;             // k-rows of weights per pipeline stage (= one UMMA k-step)
constexpr int CHUNK_BYTES = STAGE_K * 128;
constexpr int MAX_A = 32;

struct ChainArgs {
  int n_layers, H, K0, K0pad, out_dim, ln;
  int P, S, E, M, tiles;
  int x_row0[FQL_MAXP], x_rows_s;
  int w_row[FQL_MAXP][FQL_MAXL], w_rows_s;   // rows of H elements in the shadow
  int wl_row[FQL_MAXP], wl_rows_s;           // rows of 64 elements in the shadow (padded last layer)
  const float* params;
  long long arena;
  long long off_b[FQL_MAXP][FQL_MAXL], off_lns[FQL_MAXP][FQL_MAXL], off_lnb[FQL_MAXP][FQL_MAXL];
  float* out;
  float* Zs[FQL_MAXL];
  float* Hs[FQL_MAXL];
  float* mu[FQL_MAXL];
  float* rstd[FQL_MAXL];
  void* Hb[FQL_MAXL];  // bf16 copies of H (operands of the tensor-core backward)
  void* Zb[FQL_MAXL];  // bf16 copies of Z (gelu' in the tensor-core backward; non-LayerNorm networks)
  int Mcap, r0;
  int n_steps, F, A;   // Euler: n_steps > 1
  const float* a0;     // [S][M][A] initial actions (noise) for the Euler chain
  float* target;       // [S][M][A] clip(final action)
  int clip_out;        // out = clip(out) (sample_actions)
  int nstage;
};

__device__ __forceinline__ float gelu_fast(float x) {
  const float u = FQL_GELU_C * (x + FQL_GELU_A * x * x * x);
  return 0.5f * x * (1.0f + tanh_approx(u));
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

constexpr int CH_NMMA = 2;   // MMA-issuer warps: one per 256-column half of the accumulator
constexpr int CH_THREADS = 32 * (1 + CH_NMMA + 4);
constexpr int CH_EPI0 = 32 * (1 + CH_NMMA);

__global__ void __launch_bounds__(CH_THREADS, 1) mlp_chain_tc_kernel(const __grid_constant__ CUtensorMap mapX,
                                                              const __grid_constant__ CUtensorMap mapW,
                                                              const __grid_constant__ CUtensorMap mapWL, const ChainArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int nkb_a = a.H / 64, nkb_x = a.K0pad / 64, nchunk = a.H / 64;
  uint8_t* sA = smem;                                   // [nkb_a][128][128 B]
  uint8_t* sX = sA + nkb_a * KB_BYTES;                  // [nkb_x][128][128 B]
  uint8_t* sB = sX + nkb_x * KB_BYTES;                  // [nstage][nchunk][16][128 B]
  const int stage_bytes = nchunk * CHUNK_BYTES;
  float* sPar = reinterpret_cast<float*>(sB + a.nstage * stage_bytes);  // [2][3][H]: bias, ln scale, ln bias (double buffered)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sPar + 2 * 3 * a.H);
  uint64_t* full = bars;                 // [nstage]
  uint64_t* empty = bars + 8;            // [nstage]
  uint64_t* x_full = bars + 16;
  uint64_t* acc_full = bars + 17;
  uint64_t* a_ready = bars + 18;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 20);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform to ptxas as well
  const int tile = blockIdx.x % a.tiles, g = blockIdx.x / a.tiles;
  const int e = g % a.E, s = (g / a.E) % a.S, p = g / (a.E * a.S);
  const int NL = a.n_layers;
  const int total_iters = a.n_steps * NL;
  const int n_issuers = (a.H > 256) ? CH_NMMA : 1;  // hidden layers: issuer h owns N-half h; the narrow last layer: issuer 0

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapX);
    tma_prefetch_desc(&mapW);
    tma_prefetch_desc(&mapWL);
    for (int i = 0; i < a.nstage; i++) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], n_issuers);
    }
    mbar_init(x_full, 1);
    mbar_init(acc_full, n_issuers);
    mbar_init(a_ready, 4);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer =================
    // (single-thread roles run warp-uniform, the instruction predicated on the elected lane: tc_prims.cuh)
    const bool el = elect_one();
    {
      if (el) mbar_expect_tx(x_full, nkb_x * KB_BYTES);
      const int xrow = a.x_row0[p] + s * a.x_rows_s + tile * TILE_M;
      for (int kb = 0; kb < nkb_x; kb++)
        if (el) tma_load_2d(sX + kb * KB_BYTES, &mapX, x_full, kb * 64, xrow);
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < total_iters; it++) {
        const int l = it % NL;
        const bool last = (l == NL - 1);
        const int K = (l == 0) ? a.K0 : a.H;
        const int ksteps = (K + STAGE_K - 1) / STAGE_K;
        for (int ks = 0; ks < ksteps; ks++) {
          mbar_wait_u(&empty[stage], phase ^ 1);
          uint8_t* dst = sB + stage * stage_bytes;
          if (el) {
            if (!last) {
              mbar_expect_tx(&full[stage], stage_bytes);
              const int row = a.w_row[p][l] + s * a.w_rows_s + e * K + ks * STAGE_K;
              for (int c = 0; c < nchunk; c++) tma_load_2d(dst + c * CHUNK_BYTES, &mapW, &full[stage], c * 64, row);
            } else {
              mbar_expect_tx(&full[stage], CHUNK_BYTES);
              const int row = a.wl_row[p] + s * a.wl_rows_s + e * a.H + ks * STAGE_K;
              tma_load_2d(dst, &mapWL, &full[stage], 0, row);
            }
          }
          if (++stage == a.nstage) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp <= CH_NMMA) {
    // ================= MMA issuers =================
    const int mw = warp - 1;
    const bool el = elect_one();
    if (mw < n_issuers) {
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      int stage = 0;
      uint32_t phase = 0;
      const int n_mma = (a.H > 256) ? 256 : a.H;          // N per instruction for hidden layers
      const uint32_t idesc_h = make_idesc_bf16(128, n_mma, false, true);
      const uint32_t idesc_l = make_idesc_bf16(128, 64, false, true);
      const uint64_t a_t = make_smem_desc(0, 16, 1024), b_t = make_smem_desc(0, CHUNK_BYTES, 1024);
      const uint32_t sa0 = smem_u32(sA) >> 4, sx0 = smem_u32(sX) >> 4, sb0 = smem_u32(sB) >> 4;
      for (int it = 0; it < total_iters; it++) {
        const int l = it % NL;
        const bool last = (l == NL - 1);
        if (it == 0) mbar_wait_u(x_full, 0);
        else mbar_wait_u(a_ready, (it - 1) & 1);
        tc_fence_after();
        const int K = (l == 0) ? a.K0 : a.H;
        const int ksteps = (K + STAGE_K - 1) / STAGE_K;
        const uint32_t a0 = (l == 0) ? sx0 : sa0;
        for (int ks = 0; ks < ksteps; ks++) {
          mbar_wait_u(&full[stage], phase);
          tc_fence_after();
          const uint64_t adesc = a_t + (uint64_t)(a0 + (ks >> 2) * (KB_BYTES >> 4) + (ks & 3) * 2);
          const uint32_t b0 = sb0 + stage * (stage_bytes >> 4);
          if (el) {
            if (!last) {
              umma_bf16(tmem_u + mw * n_mma, adesc, b_t + (uint64_t)(b0 + mw * (n_mma / 64) * (CHUNK_BYTES >> 4)), idesc_h, ks > 0);
            } else if (mw == 0) {
              umma_bf16(tmem_u, adesc, b_t + (uint64_t)b0, idesc_l, ks > 0);
            }
            umma_commit(&empty[stage]);
          }
          if (++stage == a.nstage) { stage = 0; phase ^= 1; }
        }
        if (el) umma_commit(acc_full);
      }
    }
  } else {
    // ================= epilogue: one thread per row =================
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;                // row inside the tile
    const int grow = tile * TILE_M + row;         // row inside the group
    const bool valid = grow < a.M;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const int et = threadIdx.x - CH_EPI0;         // 0..127
    const int64_t gidx = (int64_t)((p * a.S + s) * a.E + e) * a.Mcap + a.r0 + grow;  // row index into [G][Mcap][*] buffers
    const float* bias_g[FQL_MAXL];
    float act[MAX_A];
#pragma unroll
    for (int c = 0; c < MAX_A; c++) act[c] = 0.f;
    if (a.n_steps > 1 && valid) {
#pragma unroll
      for (int c = 0; c < MAX_A; c++)
        if (c < a.A) act[c] = a.a0[((int64_t)s * a.M + grow) * a.A + c];
    }
    (void)bias_g;
    for (int it = 0; it < total_iters; it++) {
      const int l = it % NL, step = it / NL;
      const bool last = (l == NL - 1);
      const int N = last ? a.out_dim : a.H;
      float* par = sPar + (it & 1) * 3 * a.H;
      {  // stage this layer's bias / LN parameters while the MMAs run
        const float* b = a.params + (int64_t)s * a.arena + a.off_b[p][l] + (int64_t)e * N;
        for (int i = et; i < N; i += 128) par[i] = b[i];
        if (a.ln && !last) {
          const float* sc = a.params + (int64_t)s * a.arena + a.off_lns[p][l] + (int64_t)e * N;
          const float* bi = a.params + (int64_t)s * a.arena + a.off_lnb[p][l] + (int64_t)e * N;
          for (int i = et; i < N; i += 128) {
            par[a.H + i] = sc[i];
            par[2 * a.H + i] = bi[i];
          }
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      mbar_wait(acc_full, it & 1);
      tc_fence_after();
      uint32_t r[32];
      if (!last) {
        float* Zs = a.Zs[l] ? a.Zs[l] + gidx * a.H : nullptr;
        float* Hs = a.Hs[l] ? a.Hs[l] + gidx * a.H : nullptr;
        if (!a.ln) {
          for (int j = 0; j < a.H / 32; j++) {
            tmem_ld32(t_lane + j * 32, r);
            tmem_wait_ld();
            float h[32];
#pragma unroll
            for (int i = 0; i < 32; i++) {
              const float z = __uint_as_float(r[i]) + par[j * 32 + i];
              r[i] = __float_as_uint(z);
              h[i] = gelu_fast(z);
            }
            if (valid && Zs) {
#pragma unroll
              for (int i = 0; i < 32; i += 4)
                *reinterpret_cast<float4*>(Zs + j * 32 + i) = make_float4(__uint_as_float(r[i]), __uint_as_float(r[i + 1]),
                                                                          __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
            }
            if (valid && Hs) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(Hs + j * 32 + i) = make_float4(h[i], h[i + 1], h[i + 2], h[i + 3]);
            }
            if (valid && a.Zb[l]) {
#pragma unroll
              for (int c = 0; c < 4; c++)
                *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(a.Zb[l]) + gidx * a.H + j * 32 + c * 8) =
                    make_uint4(pack_bf16(__uint_as_float(r[c * 8 + 0]), __uint_as_float(r[c * 8 + 1])),
                               pack_bf16(__uint_as_float(r[c * 8 + 2]), __uint_as_float(r[c * 8 + 3])),
                               pack_bf16(__uint_as_float(r[c * 8 + 4]), __uint_as_float(r[c * 8 + 5])),
                               pack_bf16(__uint_as_float(r[c * 8 + 6]), __uint_as_float(r[c * 8 + 7])));
            }
            uint8_t* blk = sA + ((j * 32) >> 6) * KB_BYTES;
            const int c0 = ((j * 32) & 63) >> 3;
#pragma unroll
            for (int c = 0; c < 4; c++) {
              uint4 v = make_uint4(pack_bf16(h[c * 8 + 0], h[c * 8 + 1]), pack_bf16(h[c * 8 + 2], h[c * 8 + 3]),
                                   pack_bf16(h[c * 8 + 4], h[c * 8 + 5]), pack_bf16(h[c * 8 + 6], h[c * 8 + 7]));
              *reinterpret_cast<uint4*>(blk + sw128_off(row, c0 + c)) = v;
              if (valid && a.Hb[l]) *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(a.Hb[l]) + gidx * a.H + j * 32 + c * 8) = v;
            }
          }
        } else {
          // pass 1: g = gelu(z) stashed back into TMEM in place, row statistics in registers
          float s1 = 0.f, s2 = 0.f;
          for (int j = 0; j < a.H / 32; j++) {
            tmem_ld32(t_lane + j * 32, r);
            tmem_wait_ld();
            float zz[32];
#pragma unroll
            for (int i = 0; i < 32; i++) {
              const float z = __uint_as_float(r[i]) + par[j * 32 + i];
              zz[i] = z;
              const float gv = gelu_fast(z);
              s1 += gv;
              s2 += gv * gv;
              r[i] = __float_as_uint(gv);
            }
            tmem_st32(t_lane + j * 32, r);
            if (valid && Zs) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(Zs + j * 32 + i) = make_float4(zz[i], zz[i + 1], zz[i + 2], zz[i + 3]);
            }
          }
          tmem_wait_st();
          const float inv_n = 1.0f / (float)a.H;
          const float mu = s1 * inv_n;
          const float var = fmaxf(0.f, s2 * inv_n - mu * mu);
          const float rstd = rsqrtf(var + FQL_LN_EPS);
          if (valid && a.mu[l]) {
            a.mu[l][gidx] = mu;
            a.rstd[l][gidx] = rstd;
          }
          for (int j = 0; j < a.H / 32; j++) {
            tmem_ld32(t_lane + j * 32, r);
            tmem_wait_ld();
            float h[32];
#pragma unroll
            for (int i = 0; i < 32; i++)
              h[i] = (__uint_as_float(r[i]) - mu) * rstd * par[a.H + j * 32 + i] + par[2 * a.H + j * 32 + i];
            if (valid && Hs) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(Hs + j * 32 + i) = make_float4(h[i], h[i + 1], h[i + 2], h[i + 3]);
            }
            uint8_t* blk = sA + ((j * 32) >> 6) * KB_BYTES;
            const int c0 = ((j * 32) & 63) >> 3;
#pragma unroll
            for (int c = 0; c < 4; c++) {
              uint4 v = make_uint4(pack_bf16(h[c * 8 + 0], h[c * 8 + 1]), pack_bf16(h[c * 8 + 2], h[c * 8 + 3]),
                                   pack_bf16(h[c * 8 + 4], h[c * 8 + 5]), pack_bf16(h[c * 8 + 6], h[c * 8 + 7]));
              *reinterpret_cast<uint4*>(blk + sw128_off(row, c0 + c)) = v;
              if (valid && a.Hb[l]) *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(a.Hb[l]) + gidx * a.H + j * 32 + c * 8) = v;
            }
          }
        }
      } else {
        // last Dense (linear): out_dim <= 32 columns of the padded N=64 accumulator
        tmem_ld32(t_lane, r);
        tmem_wait_ld();
        if (a.n_steps == 1) {
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
          // Euler step (agents/fql.py:166-169): a += v / flow_steps, next t = (step+1)/flow_steps, written straight into
          // the bf16 first-layer operand tile that stays resident in smem for the whole integration.
          const float inv = (float)a.n_steps;
#pragma unroll
          for (int c = 0; c < MAX_A; c++)
            if (c < a.A) {
              act[c] += (__uint_as_float(r[c]) + par[c]) / inv;
              const int col = a.F + c;
              *reinterpret_cast<__nv_bfloat16*>(sX + (col >> 6) * KB_BYTES + sw128_off(row, (col & 63) >> 3) + (col & 7) * 2) =
                  __float2bfloat16(act[c]);
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
      // publish: smem operand written (generic proxy) -> async proxy; TMEM reads done -> accumulator may be overwritten
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_ready);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------------------------
// bf16 shadow of the parameter arena (+ zero-padded [H][64] copies of the narrow last-layer kernels)
// ---------------------------------------------------------------------------------------------------------------
__global__ void shadow_convert_kernel(const float* __restrict__ params, __nv_bfloat16* __restrict__ shadow, int64_t arena,
                                      int64_t shadow_seed, int S) {
  const int64_t i4 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const int s = blockIdx.y;
  if (i4 >= arena) return;
  const float4 v = *reinterpret_cast<const float4*>(params + (int64_t)s * arena + i4);
  uint2 o = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
  *reinterpret_cast<uint2*>(shadow + (int64_t)s * shadow_seed + i4) = o;
}

__global__ void shadow_lastlayer_kernel(const float* __restrict__ params, __nv_bfloat16* __restrict__ shadow, Layout L,
                                        int64_t shadow_seed, int H) {
  const int net = blockIdx.y, s = blockIdx.z;
  const NetView& v = L.net[net];
  const int64_t n = (int64_t)v.ens * H * 64;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = (int)(i % 64);
  const int64_t ek = i / 64;  // e*H + k
  const float* W = params + (int64_t)s * L.arena + v.off_w[v.n_layers - 1];
  const float val = c < v.out_dim ? W[ek * v.out_dim + c] : 0.f;
  int64_t base = L.arena;
  for (int t = 0; t < net; t++) base += (int64_t)L.net[t].ens * H * 64;
  shadow[(int64_t)s * shadow_seed + base + i] = __float2bfloat16(val);
}

// bf16 first-layer operands [rows][K0pad] from fp32 [rows][K0] (zero padded): one thread per 8 output columns (one 16-byte store)
__global__ void pad_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int64_t rows, int K0, int K0pad) {
  FQL_PDL_SYNC();
  const int per_row = K0pad >> 3;             // K0pad is a multiple of 64
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * per_row) return;
  const int64_t r = i / per_row;
  const int c0 = (int)(i - r * per_row) * 8;
  const float* xr = x + r * K0;
  float v[8];
#pragma unroll
  for (int k = 0; k < 8; k++) v[k] = (c0 + k < K0) ? xr[c0 + k] : 0.f;
  *reinterpret_cast<uint4*>(y + r * K0pad + c0) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// host: tensor maps (shared by every tensor-core source)
// ---------------------------------------------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

int make_map_2d(CUtensorMap* m, const void* base, uint64_t inner, uint64_t rows, uint32_t box_inner, uint32_t box_rows,
                CUtensorMapSwizzle swz) {
  auto enc = get_encode();
  FQL_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {inner * 2};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FQL_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) inner=%llu rows=%llu", (int)r, (unsigned long long)inner,
              (unsigned long long)rows);
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// public (library-internal) API
// ---------------------------------------------------------------------------------------------------------------
int64_t tc_shadow_seed_elems(const FqlDims* d, const Layout& L) {
  int64_t n = L.arena;
  for (int t = 0; t < FQL_NUM_NETS; t++) n += (int64_t)L.net[t].ens * d->hidden * 64;
  return n;
}

int tc_supported(const FqlDims* d, bool fused_kernels) {
  FQL_REQUIRE(d->hidden % 64 == 0 && d->hidden >= 64 && d->hidden <= 512 && (d->hidden & (d->hidden - 1)) == 0,
              "FQL_PRECISION_BF16_TC needs hidden in {64,128,256,512} (got %d)", d->hidden);
  // the fused chain / cluster kernels keep the first-layer operand tile resident in shared memory (two 64-wide K blocks); wider
  // inputs (pixel configs: 512 encoder features + action + time) run layer by layer through tc_gemm
  FQL_REQUIRE(!fused_kernels || !tc_wide_input(d), "the fused tensor-core MLP kernels need obs_dim+action_dim+1 <= 128");
  FQL_REQUIRE(d->action_dim <= MAX_A, "FQL_PRECISION_BF16_TC needs action_dim <= %d", MAX_A);
  FQL_REQUIRE(!d->actor_layer_norm, "FQL_PRECISION_BF16_TC does not implement actor_layer_norm=True (non-default, agents/fql.py:260); "
                                    "use FQL_PRECISION_FP32");
  return 0;
}

int tc_refresh_shadow(const FqlDims* d, const Layout& L, const float* params, void* shadow, cudaStream_t st) {
  FQL_TRY(tc_supported(d, false));
  FQL_REQUIRE(shadow != nullptr, "shadow buffer is NULL (FQL_PRECISION_BF16_TC needs fql_shadow_bytes() bytes)");
  const int64_t seed = tc_shadow_seed_elems(d, L);
  dim3 g1((unsigned)((L.arena / 4 + 255) / 256), d->num_seeds);
  shadow_convert_kernel<<<g1, 256, 0, st>>>(params, reinterpret_cast<__nv_bfloat16*>(shadow), L.arena, seed, d->num_seeds);
  FQL_CHECK_LAUNCH();
  dim3 g2((unsigned)((2 * d->hidden * 64 + 255) / 256), FQL_NUM_NETS, d->num_seeds);
  shadow_lastlayer_kernel<<<g2, 256, 0, st>>>(params, reinterpret_cast<__nv_bfloat16*>(shadow), L, seed, d->hidden);
  FQL_CHECK_LAUNCH();
  return 0;
}

int tc_refresh_shadow_lastlayer(const FqlDims* d, const Layout& L, const float* params, void* shadow, cudaStream_t st) {
  const int64_t seed = tc_shadow_seed_elems(d, L);
  dim3 g2((unsigned)((2 * d->hidden * 64 + 255) / 256), FQL_NUM_NETS, d->num_seeds);
  shadow_lastlayer_kernel<<<g2, 256, 0, st>>>(params, reinterpret_cast<__nv_bfloat16*>(shadow), L, seed, d->hidden);
  FQL_CHECK_LAUNCH();
  return 0;
}

int tc_pad_bf16(const float* x, void* y, int64_t rows, int K0, int K0pad, cudaStream_t st) {
  const int64_t n = rows * (K0pad / 8);
  if (n == 0) return 0;
  FQL_REQUIRE(K0pad % 8 == 0, "tc_pad_bf16: K0pad=%d", K0pad);
  FQL_CHECK_CUDA(fql_launch_pdl(pad_bf16_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, x, reinterpret_cast<__nv_bfloat16*>(y), rows, K0,
                                K0pad));
  FQL_CHECK_LAUNCH();
  return 0;
}

int tc_mlp_chain(const TcChainSpec& f, cudaStream_t st) {
  const FqlDims* d = f.d;
  const Layout& L = *f.L;
  FQL_TRY(tc_supported(d));
  if (tc_mlp_chain2_supported(d)) return tc_mlp_chain2(f, st);   // hidden = 512: the epilogue-overlapped variant (chain2_tc.cu)
  const NetView& n0 = L.net[f.net[0]];
  ChainArgs a;
  memset(&a, 0, sizeof(a));
  a.n_layers = n0.n_layers; a.H = d->hidden; a.K0 = n0.in_dim; a.K0pad = (int)round_up64(n0.in_dim, 64);
  a.out_dim = n0.out_dim; a.ln = n0.ln;
  a.P = f.P; a.S = d->num_seeds; a.E = n0.ens; a.M = f.M; a.tiles = (f.M + TILE_M - 1) / TILE_M;
  const int64_t seed_elems = tc_shadow_seed_elems(d, L);
  FQL_REQUIRE(seed_elems % d->hidden == 0 && L.arena % 64 == 0, "shadow layout not row aligned");
  a.x_rows_s = f.Mcap0;
  a.w_rows_s = (int)(seed_elems / d->hidden);
  a.wl_rows_s = (int)(seed_elems / 64);
  for (int p = 0; p < f.P; p++) {
    const NetView& nv = L.net[f.net[p]];
    a.x_row0[p] = p * a.S * f.Mcap0 + f.r0_in;
    for (int l = 0; l < nv.n_layers; l++) {
      a.w_row[p][l] = (int)(nv.off_w[l] / d->hidden);
      a.off_b[p][l] = nv.off_b[l];
      a.off_lns[p][l] = nv.off_lns[l];
      a.off_lnb[p][l] = nv.off_lnb[l];
    }
    int64_t wl = L.arena;
    for (int t = 0; t < f.net[p]; t++) wl += (int64_t)L.net[t].ens * d->hidden * 64;
    a.wl_row[p] = (int)(wl / 64);
  }
  a.params = f.params; a.arena = L.arena;
  a.Mcap = f.buf ? f.buf->Mcap : f.M; a.r0 = f.r0;
  if (f.buf) {
    a.out = f.buf->out;
    for (int l = 0; l + 1 < n0.n_layers; l++) {
      a.Zs[l] = f.save ? f.buf->Z[l] : nullptr;
      a.Hs[l] = f.save ? f.buf->Hh[l] : nullptr;
      a.mu[l] = (f.save && n0.ln) ? f.buf->mu[l] : nullptr;
      a.rstd[l] = (f.save && n0.ln) ? f.buf->rstd[l] : nullptr;
      a.Hb[l] = f.Hb ? f.Hb[l] : nullptr;
    }
  }
  if (!f.buf) {
    for (int l = 0; l + 1 < n0.n_layers; l++) {
      a.Hb[l] = f.Hb ? f.Hb[l] : nullptr;
      a.Zb[l] = f.Zb ? f.Zb[l] : nullptr;
    }
    if (f.Mcap_override > 0) a.Mcap = f.Mcap_override;
  }
  if (f.out_override) a.out = f.out_override;
  a.n_steps = f.n_steps > 0 ? f.n_steps : 1; a.F = d->obs_dim; a.A = d->action_dim; a.a0 = f.a0; a.target = f.target;
  a.clip_out = f.clip_out;
  FQL_REQUIRE(a.n_steps == 1 || (a.a0 && a.target && f.P == 1 && a.E == 1), "Euler chain needs a0/target and a single actor network");
  const int fixed = (a.H / 64 + a.K0pad / 64) * KB_BYTES + 2 * 3 * a.H * 4 + 256 + 1024;
  const int stage_bytes = (a.H / 64) * CHUNK_BYTES;
  int nstage = (232448 - fixed) / stage_bytes;
  if (nstage > 8) nstage = 8;
  FQL_REQUIRE(nstage >= 2, "not enough shared memory for the weight pipeline");
  a.nstage = nstage;
  const int smem = fixed + nstage * stage_bytes;

  CUtensorMap mapX, mapW, mapWL;
  const int64_t x_rows = (int64_t)f.P * a.S * f.Mcap0;
  FQL_TRY(make_map_2d(&mapX, f.X0b, a.K0pad, x_rows, 64, TILE_M));
  FQL_TRY(make_map_2d(&mapW, f.shadow, d->hidden, (uint64_t)a.S * a.w_rows_s, 64, STAGE_K));
  FQL_TRY(make_map_2d(&mapWL, f.shadow, 64, (uint64_t)a.S * a.wl_rows_s, 64, STAGE_K));
  static bool attr_set[FQL_MAX_DEVICES] = {};
  const int dev = fql_current_device();
  if (!attr_set[dev]) {
    FQL_CHECK_CUDA(cudaFuncSetAttribute(mlp_chain_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    attr_set[dev] = true;
  }
  const int grid = a.tiles * a.P * a.S * a.E;
  mlp_chain_tc_kernel<<<grid, CH_THREADS, smem, st>>>(mapX, mapW, mapWL, a);
  FQL_CHECK_LAUNCH();
  return 0;
}
