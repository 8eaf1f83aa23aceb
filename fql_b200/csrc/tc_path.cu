// tc_path.cu -- layer-by-layer tensor-core schedules built from tc_gemm (+ the SIMT row/column kernels):
//   actor networks (no LayerNorm by default): forward incl. the Euler integration, backward (dgrad chain + wgrads); at small
//     batch the Euler integration, the one-step actor's forward and its dgrad chain are cluster launches instead (euler_cluster.cu)
//   critic (LayerNorm): forward (GEMM + GELU/LayerNorm row kernel per layer, one chain per problem) and backward
// Reference: utils/networks.py:34-61 (layer arithmetic), agents/fql.py:155-171 (Euler), utils/flax_utils.py:137 (jax.grad).
#include "step.cuh"

#include <cuda_bf16.h>

namespace {
typedef __nv_bfloat16 bf16;

// bf16 mode: MUFU tanh (2^-11 abs error) instead of the ~25-instruction tanhf; these kernels sit on the critic chain
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float gelu_fast(float x) {
  return 0.5f * x * (1.0f + tanh_fast(FQL_GELU_C * (x + FQL_GELU_A * x * x * x)));
}
__device__ __forceinline__ void gelu_and_grad_fast(float x, float* g, float* dg) {
  const float x2 = x * x;
  const float th = tanh_fast(FQL_GELU_C * (x + FQL_GELU_A * x2 * x));
  *g = 0.5f * x * (1.0f + th);
  *dg = 0.5f * (1.0f + th) + 0.5f * x * (1.0f - th * th) * (FQL_GELU_C * (1.0f + 3.0f * FQL_GELU_A * x2));
}

TcOperand op(const void* ptr, int inner, int rows, long long ld, int g0, long long s0, int g1, long long s1) {
  TcOperand o;
  o.ptr = ptr; o.inner = inner; o.rows = rows; o.ld = ld; o.g0 = g0; o.s0 = s0; o.g1 = g1; o.s1 = s1;
  return o;
}
TcPtr tp(const void* base, long long s0, long long s1, int ld) {
  TcPtr p;
  p.base = const_cast<void*>(base); p.s0 = s0; p.s1 = s1; p.ld = ld;
  return p;
}
int64_t wl_offset(const FqlDims* d, const Layout& L, int net) {
  int64_t o = L.arena;
  for (int t = 0; t < net; t++) o += (int64_t)L.net[t].ens * d->hidden * 64;
  return o;
}

// Row kernels of the critic chain: one warp per row, the whole row (N <= 512, N % 4 == 0) in registers as four float4 per lane
// (lane owns columns 128 i + 4 lane .. + 3): one trip to memory, 16-byte loads, 8/16-byte stores, gelu / gelu' evaluated once.
constexpr int ROW_V = 4;        // float4 per lane
constexpr int ROW_WARPS = 4;    // rows per CTA

__device__ __forceinline__ uint2 pack4_bf16(float a, float b, float c, float d) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  return make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
}

// H = [LayerNorm](gelu(Z)) -> bf16 (+ row statistics).  Z: fp32 [rows][N] contiguous; scale/bias per (s, e).
__global__ void __launch_bounds__(32 * ROW_WARPS) act_ln_bf16_kernel(const float* __restrict__ Z, const float* __restrict__ scale_base,
                                                                     const float* __restrict__ bias_base, int64_t par_s, int64_t par_e,
                                                                     bf16* __restrict__ Hb, float* __restrict__ mu_out,
                                                                     float* __restrict__ rstd_out, int M, int N, int S, int E, int ln) {
  FQL_PDL_SYNC();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * ROW_WARPS + warp;
  if (row >= (int64_t)S * E * M) return;
  const int g = (int)(row / M), e = g % E, s = g / E;
  const float* z = Z + row * N;
  bf16* h = Hb + row * N;
  float gv[ROW_V][4];
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < ROW_V; i++) {
    const int c = i * 128 + lane * 4;
    if (c < N) {
      const float4 zz = *reinterpret_cast<const float4*>(z + c);
      gv[i][0] = gelu_fast(zz.x); gv[i][1] = gelu_fast(zz.y); gv[i][2] = gelu_fast(zz.z); gv[i][3] = gelu_fast(zz.w);
#pragma unroll
      for (int k = 0; k < 4; k++) { s1 += gv[i][k]; s2 += gv[i][k] * gv[i][k]; }
    }
  }
  if (!ln) {
#pragma unroll
    for (int i = 0; i < ROW_V; i++) {
      const int c = i * 128 + lane * 4;
      if (c < N) *reinterpret_cast<uint2*>(h + c) = pack4_bf16(gv[i][0], gv[i][1], gv[i][2], gv[i][3]);
    }
    return;
  }
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  const float inv_n = 1.0f / (float)N;
  const float mu = s1 * inv_n;
  const float var = fmaxf(0.f, s2 * inv_n - mu * mu);
  const float rstd = rsqrtf(var + FQL_LN_EPS);
  const float* sc = scale_base + s * par_s + e * par_e;
  const float* bi = bias_base + s * par_s + e * par_e;
#pragma unroll
  for (int i = 0; i < ROW_V; i++) {
    const int c = i * 128 + lane * 4;
    if (c < N) {
      const float4 s4 = *reinterpret_cast<const float4*>(sc + c), b4 = *reinterpret_cast<const float4*>(bi + c);
      *reinterpret_cast<uint2*>(h + c) = pack4_bf16((gv[i][0] - mu) * rstd * s4.x + b4.x, (gv[i][1] - mu) * rstd * s4.y + b4.y,
                                                    (gv[i][2] - mu) * rstd * s4.z + b4.z, (gv[i][3] - mu) * rstd * s4.w + b4.w);
    }
  }
  if (lane == 0 && mu_out) {
    mu_out[row] = mu;
    rstd_out[row] = rstd;
  }
}

// dZ rows kernel for LayerNorm nets with an extra bf16 copy: dZ = LNbwd(dH; Z) * gelu'(Z)
__global__ void __launch_bounds__(32 * ROW_WARPS) ln_bwd_bf16_kernel(const float* __restrict__ dH, const float* __restrict__ Z,
                                                                     const float* __restrict__ scale_base, int64_t scale_s, int64_t scale_e,
                                                                     float* __restrict__ dZ, bf16* __restrict__ dZb, int M, int N, int S, int E,
                                                                     int64_t z_rows_e, int64_t z_rows_s) {
  FQL_PDL_SYNC();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * ROW_WARPS + warp;
  if (row >= (int64_t)S * E * M) return;
  const int r = (int)(row % M), g = (int)(row / M), e = g % E, s = g / E;
  const float* z = Z + ((int64_t)s * z_rows_s + (int64_t)e * z_rows_e + r) * N;
  const float* dh = dH + row * N;
  float* dz = dZ + row * N;
  bf16* dzb = dZb + row * N;
  const float* sc = scale_base + s * scale_s + e * scale_e;
  float gv[ROW_V][4], dg[ROW_V][4], dx[ROW_V][4];
  float s1 = 0.f, s2 = 0.f, m1 = 0.f;
#pragma unroll
  for (int i = 0; i < ROW_V; i++) {
    const int c = i * 128 + lane * 4;
#pragma unroll
    for (int k = 0; k < 4; k++) gv[i][k] = dg[i][k] = dx[i][k] = 0.f;
    if (c < N) {
      const float4 zz = *reinterpret_cast<const float4*>(z + c), dd = *reinterpret_cast<const float4*>(dh + c),
                   s4 = *reinterpret_cast<const float4*>(sc + c);
      const float zv[4] = {zz.x, zz.y, zz.z, zz.w}, dv[4] = {dd.x, dd.y, dd.z, dd.w}, sv[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
      for (int k = 0; k < 4; k++) {
        gelu_and_grad_fast(zv[k], &gv[i][k], &dg[i][k]);
        dx[i][k] = dv[k] * sv[k];
        s1 += gv[i][k];
        s2 += gv[i][k] * gv[i][k];
        m1 += dx[i][k];
      }
    }
  }
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  m1 = warp_sum(m1);
  const float inv_n = 1.0f / (float)N;
  const float mu = s1 * inv_n;
  const float var = fmaxf(0.f, s2 * inv_n - mu * mu);
  const float rstd = rsqrtf(var + FQL_LN_EPS);
  float m2 = 0.f;
#pragma unroll
  for (int i = 0; i < ROW_V; i++) {
    const int c = i * 128 + lane * 4;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      gv[i][k] = (gv[i][k] - mu) * rstd;  // xhat
      if (c < N) m2 += dx[i][k] * gv[i][k];
    }
  }
  m1 *= inv_n;
  m2 = warp_sum(m2) * inv_n;
#pragma unroll
  for (int i = 0; i < ROW_V; i++) {
    const int c = i * 128 + lane * 4;
    if (c < N) {
      float v[4];
#pragma unroll
      for (int k = 0; k < 4; k++) v[k] = rstd * (dx[i][k] - m1 - gv[i][k] * m2) * dg[i][k];
      *reinterpret_cast<float4*>(dz + c) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<uint2*>(dzb + c) = pack4_bf16(v[0], v[1], v[2], v[3]);
    }
  }
}

// dZ = dH * gelu'(Z) (no LayerNorm) with a bf16 copy
__global__ void gelu_bwd_bf16_kernel(const float* __restrict__ dH, const float* __restrict__ Z, float* __restrict__ dZ,
                                     bf16* __restrict__ dZb, int M, int N, int S, int E, int64_t z_rows_e, int64_t z_rows_s) {
  FQL_PDL_SYNC();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)S * E * M * N) return;
  const int c = (int)(i % N);
  const int64_t row = i / N;
  const int r = (int)(row % M), g = (int)(row / M), e = g % E, s = g / E;
  float gg, dgg;
  gelu_and_grad_fast(Z[((int64_t)s * z_rows_s + (int64_t)e * z_rows_e + r) * N + c], &gg, &dgg);
  const float v = dH[i] * dgg;
  dZ[i] = v;
  dZb[i] = __float2bfloat16(v);
}

// Column sums over rows of a bf16 tensor [G][M][N] (N % 64 == 0), ADDED into fp32 out (zeroed by the caller): bias gradients from
// the bf16 dZ saves of the large-batch backward.  grid (N / 64, row chunks, G); a warp reads 128 contiguous bytes of one row.
constexpr int CS_ROWS = 256;
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const bf16* __restrict__ X, int64_t M, int N, float* __restrict__ out, int64_t os0, int G0,
                                                          int64_t os1) {
  const int g = blockIdx.z, g0 = g % G0, g1 = g / G0;
  const int c = blockIdx.x * 64 + (threadIdx.x & 31) * 2;
  const int rl = threadIdx.x >> 5;
  const int64_t r0 = (int64_t)blockIdx.y * CS_ROWS, r1 = (r0 + CS_ROWS < M) ? r0 + CS_ROWS : M;
  const bf16* x = X + (int64_t)g * M * N + c;
  float a0 = 0.f, a1 = 0.f;
  int64_t r = r0 + rl;
  for (; r + 24 < r1; r += 32) {   // four independent loads in flight per thread
    __nv_bfloat162 v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) v[u] = *reinterpret_cast<const __nv_bfloat162*>(x + (r + 8 * u) * N);
#pragma unroll
    for (int u = 0; u < 4; u++) {
      a0 += __low2float(v[u]);
      a1 += __high2float(v[u]);
    }
  }
  for (; r < r1; r += 8) {
    const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(x + r * N);
    a0 += __low2float(v);
    a1 += __high2float(v);
  }
  __shared__ float sh[8][64];
  sh[rl][(threadIdx.x & 31) * 2] = a0;
  sh[rl][(threadIdx.x & 31) * 2 + 1] = a1;
  __syncthreads();
  if (threadIdx.x < 64) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) t += sh[i][threadIdx.x];
    atomicAdd(out + g0 * os0 + g1 * os1 + blockIdx.x * 64 + threadIdx.x, t);
  }
}

}  // namespace

int launch_colsum_bf16(const void* X, int64_t G, int64_t M, int N, float* out, int64_t out_stride_g0, int G0, int64_t out_stride_g1, cudaStream_t st) {
  FQL_REQUIRE(N % 64 == 0 && G >= 1 && M >= 1, "launch_colsum_bf16: N=%d", N);
  dim3 grid(N / 64, (unsigned)((M + CS_ROWS - 1) / CS_ROWS), (unsigned)G);
  colsum_bf16_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const bf16*>(X), M, N, out, out_stride_g0, G0, out_stride_g1);
  FQL_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// actor forward (optionally one Euler step: the last layer's epilogue applies a += v/n and rewrites the operand tile)
// ---------------------------------------------------------------------------------------------------------------
int tc_actor_forward(const TcActor& t, float* out, long long out_ss, int clip, const TcEuler* eu, cudaStream_t st) {
  const FqlDims* d = t.d;
  const Layout& L = *t.L;
  const NetView& nv = L.net[t.net];
  const int H = d->hidden, NL = nv.n_layers, S = d->num_seeds;
  const int64_t seed_elems = tc_shadow_seed_elems(d, L);
  const bf16* sh = reinterpret_cast<const bf16*>(t.shadow);
  FQL_REQUIRE(!nv.ln && nv.ens == 1, "tc_actor_forward: LayerNorm / ensemble networks go through tc_critic_forward");
  for (int l = 0; l < NL; l++) {
    const bool last = (l == NL - 1);
    TcGemmSpec g;
    memset(&g, 0, sizeof(g));
    g.M = t.M; g.K = nv.k_of(l); g.G0 = 1; g.G1 = S; g.a_mn = 0; g.b_mn = 1;
    if (l == 0) g.A = op(t.X0b, t.K0pad, t.M, t.K0pad, 1, 0, S, t.x_ss);
    else g.A = op(t.Hb[l - 1], H, t.M, H, 1, 0, S, t.h_ss);
    g.bias = tp(t.params + nv.off_b[l], 0, L.arena, 0);
    if (!last) {
      g.N = H;
      g.B = op(sh + nv.off_w[l], H, g.K, H, 1, 0, S, seed_elems);
      g.mode = TC_MODE_FWD_HIDDEN;
      g.out_h = tp(t.Hb[l], 0, t.h_ss, H);
      if (t.Zb[l]) g.out_z = tp(t.Zb[l], 0, t.h_ss, H);
    } else {
      g.N = nv.out_dim;
      g.B = op(sh + wl_offset(d, L, t.net), 64, H, 64, 1, 0, S, seed_elems);
      if (!eu) {
        g.mode = TC_MODE_STORE_F32;
        g.out_f = tp(out, 0, out_ss, nv.out_dim);
        g.clip = clip;
      } else {
        g.mode = TC_MODE_EULER;
        g.act = tp(eu->act, 0, (long long)t.M * nv.out_dim, nv.out_dim);
        g.xb = tp(t.X0b, 0, t.x_ss, t.K0pad);
        g.target = tp(eu->target, 0, (long long)t.M * nv.out_dim, nv.out_dim);
        g.F = d->obs_dim; g.Adim = d->action_dim; g.step = eu->step; g.n_steps = eu->n_steps;
      }
    }
    FQL_TRY(tc_gemm(g, st));
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// actor backward: dOut fp32 [S][M][A] -> parameter gradients (fp32, into the arena)
// ---------------------------------------------------------------------------------------------------------------
// dX0 [S][M][K0] = dZ_0 W_0^T in fp32: the gradient of an actor's loss with respect to its first-layer input (pixel configs: the first
// obs_dim columns are the encoder features, agents/fql.py:58, 65 -> utils/encoders.py backward)
int tc_actor_input_grad(const TcActor& t, const void* dZ0b, float* dX0, cudaStream_t st) {
  const FqlDims* d = t.d;
  const Layout& L = *t.L;
  const NetView& nv = L.net[t.net];
  const int H = d->hidden, S = d->num_seeds, K0 = nv.in_dim;
  const bf16* sh = reinterpret_cast<const bf16*>(t.shadow);
  TcGemmSpec g;
  memset(&g, 0, sizeof(g));
  g.M = t.M; g.N = K0; g.K = H; g.G0 = 1; g.G1 = S; g.a_mn = 0; g.b_mn = 0;
  g.A = op(dZ0b, H, t.M, H, 1, 0, S, (long long)t.M * H);
  g.B = op(sh + nv.off_w[0], H, K0, H, 1, 0, S, tc_shadow_seed_elems(d, L));
  g.mode = TC_MODE_STORE_F32;
  g.out_f = tp(dX0, 0, (long long)t.M * K0, K0);
  return tc_gemm(g, st);
}

int tc_actor_backward(const TcActor& t, const float* dOut, void* dOutb, void* const dZb[FQL_MAXL], float* const dZf[FQL_MAXL],
                      cudaStream_t st, cudaStream_t side, cudaStream_t side2, cudaEvent_t* ev, bool dOutb_ready) {
  // side: weight-gradient GEMMs, side2: bias-gradient column sums (one stream for both was measured to be the longest chain of
  // the backward: 8 us of side work per 5 us dgrad step)
  if (!side2) side2 = side;
  // st carries the dependent dgrad chain dZ_4 -> dZ_3 -> ... -> dZ_0; the weight/bias gradients of layer l only need dZ_l,
  // so they go to `side` behind an event (every layer has its own dZ buffer, nothing is overwritten).
  const FqlDims* d = t.d;
  const Layout& L = *t.L;
  const NetView& nv = L.net[t.net];
  const int H = d->hidden, NL = nv.n_layers, S = d->num_seeds, A = nv.out_dim;
  const int64_t seed_elems = tc_shadow_seed_elems(d, L);
  const bf16* sh = reinterpret_cast<const bf16*>(t.shadow);
  const long long dz_ss = (long long)t.M * H;
  auto colsum = [&](const float* X, int N, int ld, long long ss, int64_t goff) {
    ColSumArgs c;
    memset(&c, 0, sizeof(c));
    c.P = 1; c.S = S; c.E = 1; c.M = t.M; c.N = N; c.ld = ld;
    c.X.base[0] = X; c.X.stride_s = ss;
    c.out.base[0] = t.grads + goff; c.out.stride_s = L.arena;
    return launch_colsum(c, side2, t.cs_scratch, t.cs_scratch ? 65536 : 0);
  };
  if (!dOutb_ready) FQL_TRY(tc_pad_bf16(dOut, dOutb, (int64_t)S * t.M, A, 64, st));  // else: written by the loss kernel
  FQL_CHECK_CUDA(cudaEventRecord(ev[0], st));
  {  // dZ_{NL-2} = (dOut W^T) * gelu'(Z)
    TcGemmSpec g;
    memset(&g, 0, sizeof(g));
    g.M = t.M; g.N = H; g.K = 64; g.G0 = 1; g.G1 = S; g.a_mn = 0; g.b_mn = 0;
    g.A = op(dOutb, 64, t.M, 64, 1, 0, S, (long long)t.M * 64);
    g.B = op(sh + wl_offset(d, L, t.net), 64, H, 64, 1, 0, S, seed_elems);
    g.mode = TC_MODE_DGRAD_GELU;
    g.zin = tp(t.Zb[NL - 2], 0, t.h_ss, H);
    g.out_h = tp(dZb[NL - 2], 0, dz_ss, H);
    g.out_f = tp(dZf[NL - 2], 0, dz_ss, H);
    FQL_TRY(tc_gemm(g, st));
    FQL_CHECK_CUDA(cudaEventRecord(ev[1], st));
  }
  for (int l = NL - 2; l >= 1; l--) {  // dZ_{l-1} = (dZ_l W_l^T) * gelu'(Z_{l-1})
    TcGemmSpec g;
    memset(&g, 0, sizeof(g));
    g.M = t.M; g.N = H; g.K = H; g.G0 = 1; g.G1 = S; g.a_mn = 0; g.b_mn = 0;
    g.A = op(dZb[l], H, t.M, H, 1, 0, S, dz_ss);
    g.B = op(sh + nv.off_w[l], H, nv.k_of(l), H, 1, 0, S, seed_elems);
    g.mode = TC_MODE_DGRAD_GELU;
    g.zin = tp(t.Zb[l - 1], 0, t.h_ss, H);
    g.out_h = tp(dZb[l - 1], 0, dz_ss, H);
    g.out_f = tp(dZf[l - 1], 0, dz_ss, H);
    FQL_TRY(tc_gemm(g, st));
    FQL_CHECK_CUDA(cudaEventRecord(ev[2 + (NL - 2 - l)], st));
  }
  // ---- side streams: parameter gradients
  FQL_CHECK_CUDA(cudaStreamWaitEvent(side, ev[0], 0));
  if (side2 != side) FQL_CHECK_CUDA(cudaStreamWaitEvent(side2, ev[0], 0));
  FQL_TRY(colsum(dOut, A, A, (long long)t.M * A, nv.off_b[NL - 1]));
  {  // dW_last = H^T dOut
    TcGemmSpec g;
    memset(&g, 0, sizeof(g));
    g.M = H; g.N = A; g.K = t.M; g.G0 = 1; g.G1 = S; g.a_mn = 1; g.b_mn = 1;
    g.A = op(t.Hb[NL - 2], H, t.M, H, 1, 0, S, t.h_ss);
    g.B = op(dOutb, 64, t.M, 64, 1, 0, S, (long long)t.M * 64);
    g.mode = TC_MODE_STORE_F32;
    g.out_f = tp(t.grads + nv.off_w[NL - 1], 0, L.arena, A);
    FQL_TRY(tc_gemm(g, side));
  }
  for (int l = NL - 2; l >= 0; l--) {
    FQL_CHECK_CUDA(cudaStreamWaitEvent(side, ev[1 + (NL - 2 - l)], 0));
    if (side2 != side) FQL_CHECK_CUDA(cudaStreamWaitEvent(side2, ev[1 + (NL - 2 - l)], 0));
    FQL_TRY(colsum(dZf[l], H, H, dz_ss, nv.off_b[l]));
    TcGemmSpec g;  // dW_l = A_l^T dZ_l
    memset(&g, 0, sizeof(g));
    g.M = nv.k_of(l); g.N = H; g.K = t.M; g.G0 = 1; g.G1 = S; g.a_mn = 1; g.b_mn = 1;
    if (l == 0) g.A = op(t.X0b, t.K0pad, t.M, t.K0pad, 1, 0, S, t.x_ss);
    else g.A = op(t.Hb[l - 1], H, t.M, H, 1, 0, S, t.h_ss);
    g.B = op(dZb[l], H, t.M, H, 1, 0, S, dz_ss);
    g.mode = TC_MODE_STORE_F32;
    g.out_f = tp(t.grads + nv.off_w[l], 0, L.arena, H);
    FQL_TRY(tc_gemm(g, side));
  }
  return 0;
}

// Parameter gradients only (the dgrad chain already ran, e.g. as one cluster launch): the weight-gradient GEMMs and the bias column
// sums are independent of each other, so they are dealt round-robin onto the caller's streams (which the caller forked / joins).
int tc_actor_param_grads(const TcActor& t, const float* dOut, const void* dOutb, void* const dZb[FQL_MAXL], float* const dZf[FQL_MAXL],
                         cudaStream_t* streams, int n_streams) {
  const FqlDims* d = t.d;
  const Layout& L = *t.L;
  const NetView& nv = L.net[t.net];
  const int H = d->hidden, NL = nv.n_layers, S = d->num_seeds, A = nv.out_dim;
  const long long dz_ss = (long long)t.M * H;
  int k = 0;
  auto next = [&]() { return streams[(k++) % n_streams]; };
  auto colsum = [&](const float* X, int N, int ld, long long ss, int64_t goff) {
    ColSumArgs c;
    memset(&c, 0, sizeof(c));
    c.P = 1; c.S = S; c.E = 1; c.M = t.M; c.N = N; c.ld = ld;
    c.X.base[0] = X; c.X.stride_s = ss;
    c.out.base[0] = t.grads + goff; c.out.stride_s = L.arena;
    return launch_colsum(c, next(), nullptr, 0);
  };
  for (int l = 0; l <= NL - 1; l++) {  // weight gradients first (the longer launches), layer 0 .. last
    TcGemmSpec g;
    memset(&g, 0, sizeof(g));
    g.K = t.M; g.G0 = 1; g.G1 = S; g.a_mn = 1; g.b_mn = 1; g.mode = TC_MODE_STORE_F32;
    if (l == 0) g.A = op(t.X0b, t.K0pad, t.M, t.K0pad, 1, 0, S, t.x_ss);
    else g.A = op(t.Hb[l - 1], H, t.M, H, 1, 0, S, t.h_ss);
    if (l == NL - 1) {
      g.M = H; g.N = A;
      g.B = op(dOutb, 64, t.M, 64, 1, 0, S, (long long)t.M * 64);
      g.out_f = tp(t.grads + nv.off_w[l], 0, L.arena, A);
    } else {
      g.M = nv.k_of(l); g.N = H;
      g.B = op(dZb[l], H, t.M, H, 1, 0, S, dz_ss);
      g.out_f = tp(t.grads + nv.off_w[l], 0, L.arena, H);
    }
    FQL_TRY(tc_gemm(g, next()));
  }
  FQL_TRY(colsum(dOut, A, A, (long long)t.M * A, nv.off_b[NL - 1]));
  for (int l = NL - 2; l >= 0; l--) FQL_TRY(colsum(dZf[l], H, H, dz_ss, nv.off_b[l]));
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// critic backward (2 heads, optional LayerNorm) on saved fp32 Z / mu / rstd and bf16 H of one problem of the grouped pass
//   grads != NULL : full backward (critic loss, fql.py:36-37)
//   grads == NULL : input gradient only, stored params (actor Q loss, fql.py:70) -> dX0 [S][2][M][K0]
// ---------------------------------------------------------------------------------------------------------------
int tc_critic_backward(const TcCritic& t, cudaStream_t st, cudaStream_t side, cudaStream_t side2, cudaEvent_t* ev) {
  if (!side2) side2 = side;  // side: weight-gradient GEMMs, side2: bias / LayerNorm-parameter column sums
  // st: the dependent chain  dZ_4 -> dgrad -> [LN/GELU bwd] -> dZ_3 -> ...   side: everything that only CONSUMES dZ_l / dH_l
  // (weight, bias and LayerNorm-parameter gradients).  Every layer has its own dH / dZ buffers, nothing is overwritten.
  const FqlDims* d = t.d;
  const Layout& L = *t.L;
  const NetView& nv = L.net[FQL_NET_CRITIC];
  const int H = d->hidden, NL = nv.n_layers, S = d->num_seeds, E = 2, M = t.M, K0 = nv.in_dim;
  const int64_t seed_elems = tc_shadow_seed_elems(d, L);
  const bf16* sh = reinterpret_cast<const bf16*>(t.shadow);
  const long long dz_se = (long long)M * H, dz_ss = (long long)E * M * H;
  const int64_t Mcap = t.buf->Mcap;
  const int64_t prow = (int64_t)t.p * S * E * Mcap;  // first row of the problem inside the grouped pass buffers
  const long long z_se = Mcap * H, z_ss = (long long)E * Mcap * H;
  auto colsum = [&](const float* X, int N, int ld, long long se, long long ss, int64_t goff, const float* Z, const float* mu,
                    const float* rstd) {
    ColSumArgs c;
    memset(&c, 0, sizeof(c));
    c.P = 1; c.S = S; c.E = E; c.M = M; c.N = N; c.ld = ld;
    c.X.base[0] = X; c.X.stride_s = ss; c.X.stride_e = se;
    if (Z) {
      c.Z.base[0] = Z; c.Z.stride_s = z_ss; c.Z.stride_e = z_se;
      c.mu.base[0] = mu; c.mu.stride_s = (long long)E * Mcap; c.mu.stride_e = Mcap;
      c.rstd.base[0] = rstd; c.rstd.stride_s = c.mu.stride_s; c.rstd.stride_e = Mcap;
    }
    c.out.base[0] = t.grads + goff; c.out.stride_s = L.arena; c.out.stride_e = N;
    return launch_colsum(c, side2, t.cs_scratch, t.cs_scratch ? 65536 : 0);
  };
  // ---- chain
  FQL_TRY(tc_pad_bf16(t.dOut, t.dOutb, (int64_t)S * E * M, 1, 64, st));
  FQL_CHECK_CUDA(cudaEventRecord(ev[0], st));
  for (int l = NL - 1; l >= 0; l--) {
    const bool last = (l == NL - 1);
    if (l == 0 && !t.dX0) break;
    const void* dzb = last ? t.dOutb : t.dZb[l];
    const int dz_inner = last ? 64 : H;
    const long long dzb_se = (long long)M * dz_inner, dzb_ss = (long long)E * M * dz_inner;
    TcGemmSpec g;  // dH_{l-1} [M][K_l] = dZ_l W_l^T   (raw, fp32)
    memset(&g, 0, sizeof(g));
    g.M = M; g.N = nv.k_of(l); g.K = last ? 64 : H; g.G0 = E; g.G1 = S; g.a_mn = 0; g.b_mn = 0;
    g.A = op(dzb, dz_inner, M, dz_inner, E, dzb_se, S, dzb_ss);
    if (last) g.B = op(sh + wl_offset(d, L, FQL_NET_CRITIC), 64, H, 64, E, (long long)H * 64, S, seed_elems);
    else g.B = op(sh + nv.off_w[l], H, nv.k_of(l), H, E, (long long)nv.k_of(l) * H, S, seed_elems);
    g.mode = TC_MODE_STORE_F32;
    if (l == 0) {
      g.out_f = tp(t.dX0, (long long)M * K0, (long long)E * M * K0, K0);
      FQL_TRY(tc_gemm(g, st));
      break;
    }
    g.out_f = tp(t.dHf[l - 1], dz_se, dz_ss, H);
    FQL_TRY(tc_gemm(g, st));
    const float* Zp = t.buf->Z[l - 1] + prow * H;
    if (nv.ln) {
      const int64_t rows = (int64_t)S * E * M;
      FQL_CHECK_CUDA(fql_launch_pdl(ln_bwd_bf16_kernel, dim3((unsigned)((rows + ROW_WARPS - 1) / ROW_WARPS)), dim3(32 * ROW_WARPS), 0, st, t.dHf[l - 1], Zp,
                                    t.params + nv.off_lns[l - 1], L.arena, H, t.dZf[l - 1], reinterpret_cast<bf16*>(t.dZb[l - 1]), M, H, S, E, Mcap,
                                    (int64_t)E * Mcap));
      FQL_CHECK_LAUNCH();
    } else {
      const int64_t n = (int64_t)S * E * M * H;
      FQL_CHECK_CUDA(fql_launch_pdl(gelu_bwd_bf16_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, t.dHf[l - 1], Zp, t.dZf[l - 1],
                                    reinterpret_cast<bf16*>(t.dZb[l - 1]), M, H, S, E, Mcap, (int64_t)E * Mcap));
      FQL_CHECK_LAUNCH();
    }
    FQL_CHECK_CUDA(cudaEventRecord(ev[1 + (NL - 1 - l)], st));  // dZ_{l-1} (and dH_{l-1}) ready
  }
  if (!t.grads) return 0;
  // ---- side: parameter gradients
  FQL_CHECK_CUDA(cudaStreamWaitEvent(side, ev[0], 0));
  if (side2 != side) FQL_CHECK_CUDA(cudaStreamWaitEvent(side2, ev[0], 0));
  FQL_TRY(colsum(t.dOut, 1, 1, M, (long long)E * M, nv.off_b[NL - 1], nullptr, nullptr, nullptr));
  for (int l = NL - 1; l >= 0; l--) {
    const bool last = (l == NL - 1);
    if (!last) {
      FQL_CHECK_CUDA(cudaStreamWaitEvent(side, ev[1 + (NL - 2 - l)], 0));  // dZ_l
      if (side2 != side) FQL_CHECK_CUDA(cudaStreamWaitEvent(side2, ev[1 + (NL - 2 - l)], 0));
      FQL_TRY(colsum(t.dZf[l], H, H, dz_se, dz_ss, nv.off_b[l], nullptr, nullptr, nullptr));
      if (nv.ln) {
        const float* Zl = t.buf->Z[l] + prow * H;
        FQL_TRY(colsum(t.dHf[l], H, H, dz_se, dz_ss, nv.off_lnb[l], nullptr, nullptr, nullptr));
        FQL_TRY(colsum(t.dHf[l], H, H, dz_se, dz_ss, nv.off_lns[l], Zl, t.buf->mu[l] + prow, t.buf->rstd[l] + prow));
      }
    }
    const void* dzb = last ? t.dOutb : t.dZb[l];
    const int dz_inner = last ? 64 : H;
    const long long dzb_se = (long long)M * dz_inner, dzb_ss = (long long)E * M * dz_inner;
    TcGemmSpec g;  // dW_l [K_l][N_l] = A_l^T dZ_l
    memset(&g, 0, sizeof(g));
    g.M = nv.k_of(l); g.N = nv.n_of(l); g.K = M; g.G0 = E; g.G1 = S; g.a_mn = 1; g.b_mn = 1;
    if (l == 0) g.A = op(t.X0b, t.K0pad, M, t.K0pad, 1, 0, S, t.x_ss);  // input shared by both heads
    else g.A = op(reinterpret_cast<const bf16*>(t.Hb[l - 1]) + prow * H, H, M, H, E, z_se, S, z_ss);
    g.B = op(dzb, dz_inner, M, dz_inner, E, dzb_se, S, dzb_ss);
    g.mode = TC_MODE_STORE_F32;
    g.out_f = tp(t.grads + nv.off_w[l], (long long)nv.k_of(l) * nv.n_of(l), L.arena, nv.n_of(l));
    FQL_TRY(tc_gemm(g, side));
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// critic forward of ONE problem of the grouped pass (2 heads), layer by layer: tc_gemm (+bias, fp32 Z) -> fused GELU+LayerNorm
// row kernel (bf16 H, fp32 row statistics).  The three problems {target(s',a'), critic(s,a), critic(s,a_pi)} are independent
// chains and run on three streams.
// ---------------------------------------------------------------------------------------------------------------
int tc_critic_forward(const TcCritic& t, int net, float* out, cudaStream_t st) {
  const FqlDims* d = t.d;
  const Layout& L = *t.L;
  const NetView& nv = L.net[net];
  const int H = d->hidden, NL = nv.n_layers, S = d->num_seeds, E = 2, M = t.M;
  const int64_t seed_elems = tc_shadow_seed_elems(d, L);
  const bf16* sh = reinterpret_cast<const bf16*>(t.shadow);
  const int64_t Mcap = t.buf->Mcap;
  FQL_REQUIRE(Mcap == M, "tc_critic_forward: the grouped pass buffers must be dense (Mcap == M)");
  const int64_t prow = (int64_t)t.p * S * E * Mcap;
  const long long z_se = Mcap * H, z_ss = (long long)E * Mcap * H;
  for (int l = 0; l < NL; l++) {
    const bool last = (l == NL - 1);
    TcGemmSpec g;
    memset(&g, 0, sizeof(g));
    g.M = M; g.K = nv.k_of(l); g.G0 = E; g.G1 = S; g.a_mn = 0; g.b_mn = 1;
    if (l == 0) g.A = op(t.X0b, t.K0pad, M, t.K0pad, 1, 0, S, t.x_ss);
    else g.A = op(reinterpret_cast<const bf16*>(t.Hb[l - 1]) + prow * H, H, M, H, E, z_se, S, z_ss);
    g.mode = TC_MODE_STORE_F32;
    g.bias = tp(t.params + nv.off_b[l], nv.n_of(l), L.arena, 0);
    if (!last) {
      g.N = H;
      g.B = op(sh + nv.off_w[l], H, g.K, H, E, (long long)g.K * H, S, seed_elems);
      g.out_f = tp(t.buf->Z[l] + prow * H, z_se, z_ss, H);
      FQL_TRY(tc_gemm(g, st));
      const int64_t rows = (int64_t)S * E * M;
      FQL_CHECK_CUDA(fql_launch_pdl(act_ln_bf16_kernel, dim3((unsigned)((rows + ROW_WARPS - 1) / ROW_WARPS)), dim3(32 * ROW_WARPS), 0, st, t.buf->Z[l] + prow * H,
                                    nv.ln ? t.params + nv.off_lns[l] : nullptr, nv.ln ? t.params + nv.off_lnb[l] : nullptr, L.arena, (int64_t)H,
                                    reinterpret_cast<bf16*>(t.Hb[l]) + prow * H, nv.ln ? t.buf->mu[l] + prow : nullptr,
                                    nv.ln ? t.buf->rstd[l] + prow : nullptr, M, H, S, E, (int)nv.ln));
      FQL_CHECK_LAUNCH();
    } else {
      g.N = 1;
      g.B = op(sh + wl_offset(d, L, net), 64, H, 64, E, (long long)H * 64, S, seed_elems);
      g.out_f = tp(out + prow, Mcap, (long long)E * Mcap, 1);
      FQL_TRY(tc_gemm(g, st));
    }
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Large-batch backward (seeds x 128-row tiles fill the GPU): the whole input-gradient chain is ONE chain2 launch per network
// reading the forward's bf16 gelu' (/ xhat / rstd) saves; bias gradients are column sums of the bf16 dZ saves; weight gradients are
// split-K tc_gemm launches (LayerNorm networks: TC_MODE_WGRAD_LN on the xhat saves, which also yields the LayerNorm parameter
// gradients).  No fp32 dH / dZ tensor, no LayerNorm row kernel and no per-layer dgrad launch remains.
// ---------------------------------------------------------------------------------------------------------------
namespace {
// One launch zeroes a list of gradient leaves of every seed (the leaves that are accumulated with atomics: bias / LayerNorm
// gradients and split-K weight gradients).  Leaf lengths are multiples of 4 floats except the narrow last-layer ones.
struct ZeroList {
  int n;
  long long off[24];
  long long len[24];
};
__global__ void zero_list_kernel(float* __restrict__ base, ZeroList z, int64_t stride) {
  const int seg = blockIdx.y;
  float* p = base + (int64_t)blockIdx.z * stride + z.off[seg];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < z.len[seg]; i += (int64_t)gridDim.x * blockDim.x) p[i] = 0.f;
}
struct Zeroer {
  ZeroList z;
  int64_t longest = 0;
  Zeroer() { z.n = 0; }
  void add(int64_t off, int64_t len) {
    if (z.n < 24 && len > 0) {
      z.off[z.n] = off; z.len[z.n] = len; z.n++;
      if (len > longest) longest = len;
    }
  }
  int run(float* grads, int64_t stride, int S, cudaStream_t st) {
    if (z.n == 0) return 0;
    int bx = (int)((longest + 1023) / 1024);
    if (bx > 256) bx = 256;
    zero_list_kernel<<<dim3(bx, z.n, S), 256, 0, st>>>(grads, z, stride);
    FQL_CHECK_LAUNCH();
    return 0;
  }
};
// K splits that bring a weight-gradient GEMM to about two CTAs per SM
int wgrad_ksplit(int Mw, int N, int groups, int K) {
  const int base = ((Mw + 127) / 128) * ((N + 63) / 64) * groups;
  int ks = 296 / (base > 0 ? base : 1);
  const int nkb = (K + 63) / 64;
  if (ks > nkb / 4) ks = nkb / 4;     // at least four K blocks per CTA
  return ks < 1 ? 1 : ks;
}
}  // namespace

int tc_actor_backward_big(const TcActor& t, const float* dOut, void* dOutb, void* const dZb[FQL_MAXL], bool dOutb_ready, cudaStream_t st) {
  const FqlDims* d = t.d;
  const Layout& L = *t.L;
  const NetView& nv = L.net[t.net];
  const int H = d->hidden, NL = nv.n_layers, S = d->num_seeds, A = nv.out_dim;
  const long long dz_ss = (long long)t.M * H;
  FQL_REQUIRE(!nv.ln && nv.ens == 1, "tc_actor_backward_big: actor networks only");
  if (!dOutb_ready) FQL_TRY(tc_pad_bf16(dOut, dOutb, (int64_t)S * t.M, A, 64, st));
  TcChain2BwdSpec b;
  memset(&b, 0, sizeof(b));
  b.d = d; b.L = &L; b.net = t.net; b.params = t.params; b.shadow = t.shadow; b.dOutb = dOutb;
  b.M = t.M; b.Mcap = (int)(t.h_ss / H); b.r0 = 0; b.Mcap_dz = t.M;
  b.DGb = t.Zb;                 // the forward saved gelu'(z) in the pre-activation buffers
  b.dZb = dZb;
  FQL_TRY(tc_mlp_chain2_backward(b, st));
  // bias gradients
  {
    ColSumArgs c;
    memset(&c, 0, sizeof(c));
    c.P = 1; c.S = S; c.E = 1; c.M = t.M; c.N = A; c.ld = A;
    c.X.base[0] = dOut; c.X.stride_s = (long long)t.M * A;
    c.out.base[0] = t.grads + nv.off_b[NL - 1]; c.out.stride_s = L.arena;
    FQL_TRY(launch_colsum(c, st, t.cs_scratch, t.cs_scratch ? 65536 : 0));
  }
  Zeroer zr;
  int ksp[FQL_MAXL];
  for (int l = 0; l < NL; l++) {
    const int Mw = (l == NL - 1) ? H : nv.k_of(l), Nw = (l == NL - 1) ? A : H;
    ksp[l] = wgrad_ksplit(Mw, Nw, S, t.M);
    if (l + 1 < NL) zr.add(nv.off_b[l], H);
    if (ksp[l] > 1) zr.add(nv.off_w[l], (int64_t)Mw * Nw);
  }
  FQL_TRY(zr.run(t.grads, L.arena, S, st));
  for (int l = 0; l + 1 < NL; l++) FQL_TRY(launch_colsum_bf16(dZb[l], S, t.M, H, t.grads + nv.off_b[l], 0, 1, L.arena, st));
  // weight gradients dW_l = A_l^T dZ_l
  for (int l = 0; l < NL; l++) {
    TcGemmSpec g;
    memset(&g, 0, sizeof(g));
    g.K = t.M; g.G0 = 1; g.G1 = S; g.a_mn = 1; g.b_mn = 1; g.mode = TC_MODE_STORE_F32;
    if (l == 0) g.A = op(t.X0b, t.K0pad, t.M, t.K0pad, 1, 0, S, t.x_ss);
    else g.A = op(t.Hb[l - 1], H, t.M, H, 1, 0, S, t.h_ss);
    if (l == NL - 1) {
      g.M = H; g.N = A;
      g.B = op(dOutb, 64, t.M, 64, 1, 0, S, (long long)t.M * 64);
    } else {
      g.M = nv.k_of(l); g.N = H;
      g.B = op(dZb[l], H, t.M, H, 1, 0, S, dz_ss);
    }
    g.out_f = tp(t.grads + nv.off_w[l], 0, L.arena, g.N);
    g.ksplit = ksp[l];
    FQL_TRY(tc_gemm(g, st));
  }
  return 0;
}

// Critic (2 heads, LayerNorm) on the saves of problem t.p of the grouped forward.
//   grads != NULL: critic-loss backward (agents/fql.py:36-37): every parameter gradient of the critic
//   grads == NULL: input gradient only with the stored parameters (actor Q loss, agents/fql.py:70) -> dX0 [S][2][M][K0]
int tc_critic_backward_big(const TcCritic& t, void* const* XHb, void* const* DGb, cudaStream_t st) {
  const FqlDims* d = t.d;
  const Layout& L = *t.L;
  const NetView& nv = L.net[FQL_NET_CRITIC];
  const int H = d->hidden, NL = nv.n_layers, S = d->num_seeds, E = 2, M = t.M, K0 = nv.in_dim;
  FQL_REQUIRE(nv.ln, "tc_critic_backward_big: built for the LayerNorm critic (config['layer_norm'] = True)");
  const int64_t Mcap = t.buf->Mcap;
  const int64_t prow = (int64_t)t.p * S * E * Mcap;   // first row of the problem inside the grouped pass buffers
  const long long z_se = Mcap * H, z_ss = (long long)E * Mcap * H;
  const long long dz_se = (long long)M * H, dz_ss = (long long)E * M * H;
  FQL_TRY(tc_pad_bf16(t.dOut, t.dOutb, (int64_t)S * E * M, 1, 64, st));
  void* xh[FQL_MAXL] = {};
  void* dg[FQL_MAXL] = {};
  float* rs[FQL_MAXL] = {};
  for (int l = 0; l + 1 < NL; l++) {
    xh[l] = reinterpret_cast<bf16*>(XHb[l]) + prow * H;
    dg[l] = reinterpret_cast<bf16*>(DGb[l]) + prow * H;
    rs[l] = t.buf->rstd[l] + prow;
  }
  TcChain2BwdSpec b;
  memset(&b, 0, sizeof(b));
  b.d = d; b.L = &L; b.net = FQL_NET_CRITIC; b.params = t.params; b.shadow = t.shadow; b.dOutb = t.dOutb;
  b.M = M; b.Mcap = (int)Mcap; b.r0 = 0; b.Mcap_dz = M;
  b.DGb = dg; b.XHb = xh; b.rstd = rs;
  b.dZb = t.grads ? t.dZb : nullptr;
  b.dX0 = t.dX0;
  FQL_TRY(tc_mlp_chain2_backward(b, st));
  if (!t.grads) return 0;
  // bias gradients: last layer from the fp32 dQ, hidden layers from the bf16 dZ saves
  {
    ColSumArgs c;
    memset(&c, 0, sizeof(c));
    c.P = 1; c.S = S; c.E = E; c.M = M; c.N = 1; c.ld = 1;
    c.X.base[0] = t.dOut; c.X.stride_s = (long long)E * M; c.X.stride_e = M;
    c.out.base[0] = t.grads + nv.off_b[NL - 1]; c.out.stride_s = L.arena; c.out.stride_e = 1;
    FQL_TRY(launch_colsum(c, st, t.cs_scratch, t.cs_scratch ? 65536 : 0));
  }
  Zeroer zr;
  int ksp[FQL_MAXL];
  for (int l = 0; l < NL; l++) {
    ksp[l] = wgrad_ksplit(nv.k_of(l), nv.n_of(l), S * E, M);
    if (l + 1 < NL) {
      zr.add(nv.off_b[l], (int64_t)E * H);
      zr.add(nv.off_lns[l], (int64_t)E * H);
      zr.add(nv.off_lnb[l], (int64_t)E * H);
    }
    if (ksp[l] > 1) zr.add(nv.off_w[l], (int64_t)E * nv.k_of(l) * nv.n_of(l));
  }
  FQL_TRY(zr.run(t.grads, L.arena, S, st));
  for (int l = 0; l + 1 < NL; l++) FQL_TRY(launch_colsum_bf16(t.dZb[l], (int64_t)S * E, M, H, t.grads + nv.off_b[l], H, E, L.arena, st));
  for (int l = 0; l < NL; l++) {
    const bool last = (l == NL - 1);
    const void* dzb = last ? t.dOutb : t.dZb[l];
    const int dz_inner = last ? 64 : H;
    const long long dzb_se = (long long)M * dz_inner, dzb_ss = (long long)E * M * dz_inner;
    TcGemmSpec g;
    memset(&g, 0, sizeof(g));
    g.M = nv.k_of(l); g.N = nv.n_of(l); g.K = M; g.G0 = E; g.G1 = S; g.a_mn = 1; g.b_mn = 1;
    g.B = op(dzb, dz_inner, M, dz_inner, E, dzb_se, S, dzb_ss);
    g.out_f = tp(t.grads + nv.off_w[l], (long long)nv.k_of(l) * nv.n_of(l), L.arena, nv.n_of(l));
    g.ksplit = ksp[l];
    if (l == 0) {
      g.A = op(t.X0b, t.K0pad, M, t.K0pad, 1, 0, S, t.x_ss);  // input shared by both heads
      g.mode = TC_MODE_STORE_F32;
    } else {
      // h_{l-1} = gamma * xhat + beta feeds this layer: G = xhat^T dZ_l, transformed in the epilogue (tc_gemm.cu)
      g.A = op(xh[l - 1], H, M, H, E, z_se, S, z_ss);
      g.mode = TC_MODE_WGRAD_LN;
      g.ln_s = tp(t.params + nv.off_lns[l - 1], H, L.arena, 0);
      g.ln_b = tp(t.params + nv.off_lnb[l - 1], H, L.arena, 0);
      g.dbias = tp(t.grads + nv.off_b[l], nv.n_of(l), L.arena, 0);
      g.wmaster = tp(t.params + nv.off_w[l], (long long)H * nv.n_of(l), L.arena, 0);
      g.dln_s = tp(t.grads + nv.off_lns[l - 1], H, L.arena, 0);
      g.dln_b = tp(t.grads + nv.off_lnb[l - 1], H, L.arena, 0);
    }
    FQL_TRY(tc_gemm(g, st));
  }
  return 0;
}

// Diagnostics (not part of the product ABI surface used by the agent): one GEMM on caller buffers with chosen operand
// majorness (timing only: the buffers are interpreted as whatever layout the flags say).
extern "C" int fql_debug_tc_gemm(const void* X, const void* W, const float* bias, void* Hout, int M, int N, int K, void* dbg, void* stream,
                                 int a_mn, int b_mn) {
  TcGemmSpec g;
  memset(&g, 0, sizeof(g));
  g.M = M; g.N = N; g.K = K; g.G0 = 1; g.G1 = 1; g.a_mn = a_mn; g.b_mn = b_mn;
  g.A = a_mn ? op(X, M, K, M, 1, 0, 1, 0) : op(X, K, M, K, 1, 0, 1, 0);
  g.B = b_mn ? op(W, N, K, N, 1, 0, 1, 0) : op(W, K, N, K, 1, 0, 1, 0);
  g.mode = TC_MODE_FWD_HIDDEN;
  g.bias = tp(bias, 0, 0, 0);
  g.out_h = tp(Hout, 0, 0, N);
  g.dbg = dbg;
  return tc_gemm(g, reinterpret_cast<cudaStream_t>(stream));
}

// ---------------------------------------------------------------------------------------------------------------
// Test hooks (include/fql_b200.h): one tc_gemm or one row / column kernel on caller buffers, with the argument meaning the step
// uses, so that each kernel can be checked on its own against a reference.  tc_gemm's own FQL_REQUIRE checks are the validation.
// ---------------------------------------------------------------------------------------------------------------
namespace {
TcOperand test_op(const FqlTestOperand& o) { return op(o.ptr, o.inner, o.rows, o.ld, o.g0, o.s0, o.g1, o.s1); }
TcPtr test_ptr(const FqlTestPtr& p) { return tp(p.base, p.s0, p.s1, p.ld); }
}  // namespace

extern "C" int fql_test_tc_gemm(const FqlTestGemm* t, void* stream) {
  FQL_REQUIRE(t != nullptr, "fql_test_tc_gemm: spec is NULL");
  TcGemmSpec g;
  memset(&g, 0, sizeof(g));
  g.mode = t->mode; g.M = t->M; g.N = t->N; g.K = t->K; g.G0 = t->G0; g.G1 = t->G1; g.a_mn = t->a_mn; g.b_mn = t->b_mn;
  g.ksplit = t->ksplit;
  g.A = test_op(t->A); g.B = test_op(t->B);
  g.bias = test_ptr(t->bias); g.out_f = test_ptr(t->out_f); g.out_h = test_ptr(t->out_h); g.out_z = test_ptr(t->out_z);
  g.zin = test_ptr(t->zin); g.act = test_ptr(t->act); g.xb = test_ptr(t->xb); g.target = test_ptr(t->target);
  g.ln_s = test_ptr(t->ln_s); g.ln_b = test_ptr(t->ln_b); g.dbias = test_ptr(t->dbias); g.wmaster = test_ptr(t->wmaster);
  g.dln_s = test_ptr(t->dln_s); g.dln_b = test_ptr(t->dln_b);
  g.F = t->F; g.Adim = t->Adim; g.step = t->step; g.n_steps = t->n_steps; g.clip = t->clip;
  return tc_gemm(g, reinterpret_cast<cudaStream_t>(stream));
}

// rows = S * E * M, one warp per row (tc_critic_forward / tc_critic_backward launch them the same way)
extern "C" int fql_test_act_ln_bf16(const float* Z, const float* scale, const float* bias, int64_t par_s, int64_t par_e, void* Hb, float* mu,
                                    float* rstd, int32_t M, int32_t N, int32_t S, int32_t E, int32_t ln, void* stream) {
  FQL_REQUIRE(M >= 1 && S >= 1 && E >= 1 && N >= 4 && N <= 128 * ROW_V && N % 4 == 0, "fql_test_act_ln_bf16: M=%d N=%d S=%d E=%d", M, N, S, E);
  FQL_REQUIRE(!ln || (scale && bias), "fql_test_act_ln_bf16: LayerNorm needs scale and bias");
  const int64_t rows = (int64_t)S * E * M;
  FQL_CHECK_CUDA(fql_launch_pdl(act_ln_bf16_kernel, dim3((unsigned)((rows + ROW_WARPS - 1) / ROW_WARPS)), dim3(32 * ROW_WARPS), 0,
                                reinterpret_cast<cudaStream_t>(stream), Z, scale, bias, par_s, par_e, reinterpret_cast<bf16*>(Hb), mu, rstd, M,
                                N, S, E, ln));
  FQL_CHECK_LAUNCH();
  return 0;
}

extern "C" int fql_test_ln_bwd_bf16(const float* dH, const float* Z, const float* scale, int64_t scale_s, int64_t scale_e, float* dZ, void* dZb,
                                    int32_t M, int32_t N, int32_t S, int32_t E, int64_t z_rows_e, int64_t z_rows_s, void* stream) {
  FQL_REQUIRE(M >= 1 && S >= 1 && E >= 1 && N >= 4 && N <= 128 * ROW_V && N % 4 == 0, "fql_test_ln_bwd_bf16: M=%d N=%d S=%d E=%d", M, N, S, E);
  const int64_t rows = (int64_t)S * E * M;
  FQL_CHECK_CUDA(fql_launch_pdl(ln_bwd_bf16_kernel, dim3((unsigned)((rows + ROW_WARPS - 1) / ROW_WARPS)), dim3(32 * ROW_WARPS), 0,
                                reinterpret_cast<cudaStream_t>(stream), dH, Z, scale, scale_s, scale_e, dZ, reinterpret_cast<bf16*>(dZb), M, N, S,
                                E, z_rows_e, z_rows_s));
  FQL_CHECK_LAUNCH();
  return 0;
}

extern "C" int fql_test_gelu_bwd_bf16(const float* dH, const float* Z, float* dZ, void* dZb, int32_t M, int32_t N, int32_t S, int32_t E,
                                      int64_t z_rows_e, int64_t z_rows_s, void* stream) {
  FQL_REQUIRE(M >= 1 && S >= 1 && E >= 1 && N >= 1, "fql_test_gelu_bwd_bf16: M=%d N=%d S=%d E=%d", M, N, S, E);
  const int64_t n = (int64_t)S * E * M * N;
  FQL_CHECK_CUDA(fql_launch_pdl(gelu_bwd_bf16_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream), dH, Z,
                                dZ, reinterpret_cast<bf16*>(dZb), M, N, S, E, z_rows_e, z_rows_s));
  FQL_CHECK_LAUNCH();
  return 0;
}

extern "C" int fql_test_colsum_bf16(const void* X, int64_t G, int64_t M, int32_t N, float* out, int64_t out_stride_g0, int32_t G0,
                                    int64_t out_stride_g1, void* stream) {
  FQL_REQUIRE(G0 >= 1 && G % G0 == 0, "fql_test_colsum_bf16: G=%lld G0=%d", (long long)G, G0);
  return launch_colsum_bf16(X, G, M, N, out, out_stride_g0, G0, out_stride_g1, reinterpret_cast<cudaStream_t>(stream));
}
