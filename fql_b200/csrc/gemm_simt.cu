// gemm_simt.cu -- fp32 (FFMA) grouped GEMM family with fused epilogues + the row/column kernels around it.
// This is the FQL_PRECISION_FP32 ("parity") arithmetic of the MLP passes of FQLAgent.update:
//   forward  Dense            utils/networks.py:54      x @ kernel + bias          (launch_gemm, bias/act epilogue)
//   GELU(tanh) + LayerNorm    utils/networks.py:55-58                              (launch_act_ln_fwd)
//   backward (jax.grad)       utils/flax_utils.py:137   dgrad / wgrad / LN+GELU bwd (launch_gemm trans_*, launch_act_ln_bwd,
//                                                                                   launch_colsum)
// Groups (blockIdx.z) batch the 2-head ensemble (utils/networks.py:14-24), independent seeds and up to three
// problems that share shapes, so one launch covers e.g. {target critic, critic(s,a), critic(s,a_pi)} x 2 heads.
#include "common.cuh"

namespace {

template <int BM, int BN, int BK, int KS>
__global__ void __launch_bounds__(KS*(BM / 4) * (BN / 4)) gemm_kernel(GemmArgs a) {
  constexpr int NTK = (BM / 4) * (BN / 4);  // threads per k-group
  constexpr int NT = KS * NTK;
  constexpr int KPG = BK / KS;              // k per group per tile
  constexpr int LDA_S = BM + 4, LDB_S = BN + 4;
  constexpr int TILE_F = BK * LDA_S + BK * LDB_S;
  constexpr int RED_F = (KS > 1) ? (KS - 1) * BM * BN : 0;
  constexpr int SMEM_F = TILE_F > RED_F ? TILE_F : RED_F;
  __shared__ __align__(16) float smem[SMEM_F];
  float* As = smem;                  // [BK][LDA_S]
  float* Bs = smem + BK * LDA_S;     // [BK][LDB_S]

  const int g = blockIdx.z;
  const int e = g % a.E, s = (g / a.E) % a.S, p = g / (a.E * a.S);
  const float* __restrict__ A = a.A.at(p, s, e);
  const float* __restrict__ B = a.B.at(p, s, e);
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int t = threadIdx.x;
  const int kg = t / NTK, tin = t % NTK;
  const int tx = tin % (BN / 4), ty = tin / (BN / 4);

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < a.K; k0 += BK) {
    // ---- A tile -> As[k][m]
    if (!a.trans_a) {
#pragma unroll 4
      for (int idx = t; idx < BM * BK; idx += NT) {
        int k = idx % BK, m = idx / BK;
        int gm = m0 + m, gk = k0 + k;
        As[k * LDA_S + m] = (gm < a.M && gk < a.K) ? A[(int64_t)gm * a.lda + gk] : 0.f;
      }
    } else {
#pragma unroll 4
      for (int idx = t; idx < BM * BK; idx += NT) {
        int m = idx % BM, k = idx / BM;
        int gm = m0 + m, gk = k0 + k;
        As[k * LDA_S + m] = (gm < a.M && gk < a.K) ? A[(int64_t)gk * a.lda + gm] : 0.f;
      }
    }
    // ---- B tile -> Bs[k][n]
    if (!a.trans_b) {
#pragma unroll 4
      for (int idx = t; idx < BN * BK; idx += NT) {
        int n = idx % BN, k = idx / BN;
        int gn = n0 + n, gk = k0 + k;
        Bs[k * LDB_S + n] = (gn < a.N && gk < a.K) ? B[(int64_t)gk * a.ldb + gn] : 0.f;
      }
    } else {
#pragma unroll 4
      for (int idx = t; idx < BN * BK; idx += NT) {
        int k = idx % BK, n = idx / BK;
        int gn = n0 + n, gk = k0 + k;
        Bs[k * LDB_S + n] = (gn < a.N && gk < a.K) ? B[(int64_t)gn * a.ldb + gk] : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < KPG; kk++) {
      const int k = kg * KPG + kk;
      float4 av = *reinterpret_cast<const float4*>(&As[k * LDA_S + ty * 4]);
      float4 bv = *reinterpret_cast<const float4*>(&Bs[k * LDB_S + tx * 4]);
      float ar[4] = {av.x, av.y, av.z, av.w};
      float br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
    }
    __syncthreads();
  }

  if (KS > 1) {  // in-CTA split-K reduction (deterministic order kg = 1..KS-1 added onto kg 0)
    if (kg > 0) {
      float* r = smem + (kg - 1) * BM * BN + tin * 16;
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) r[i * 4 + j] = acc[i][j];
    }
    __syncthreads();
    if (kg > 0) return;
#pragma unroll
    for (int q = 0; q < KS - 1; q++) {
      const float* r = smem + q * BM * BN + tin * 16;
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] += r[i * 4 + j];
    }
  }

  // ---- epilogue
  const float* __restrict__ bias = a.bias.base[p] ? a.bias.at(p, s, e) : nullptr;
  const float* __restrict__ mulz = a.mulz.base[p] ? a.mulz.at(p, s, e) : nullptr;
  float* __restrict__ out_pre = a.out_pre.at(p, s, e);
  float* __restrict__ out = a.out.at(p, s, e);
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= a.M) continue;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int gn = n0 + tx * 4 + j;
      if (gn >= a.N) continue;
      float v = acc[i][j];
      if (bias) v += bias[gn];
      if (out_pre) out_pre[(int64_t)gm * a.ld_pre + gn] = v;
      if (mulz) v *= gelu_tanh_grad_f(mulz[(int64_t)gm * a.ld_mulz + gn]);
      if (a.act_gelu) v = gelu_tanh_f(v);
      if (out) out[(int64_t)gm * a.ldo + gn] = v;
    }
  }
}

// one warp per row: H = [LN](gelu(Z))
__global__ void __launch_bounds__(256) act_ln_fwd_kernel(ActLnArgs a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + warp;
  const int64_t total = (int64_t)a.P * a.S * a.E * a.M;
  if (row >= total) return;
  const int g = (int)(row / a.M), r = (int)(row % a.M);
  const int e = g % a.E, s = (g / a.E) % a.S, p = g / (a.E * a.S);
  const float* __restrict__ z = a.Z.at(p, s, e) + (int64_t)r * a.ld;
  float* __restrict__ h = a.H.at(p, s, e) + (int64_t)r * a.ld;
  if (!a.ln) {
    for (int c = lane; c < a.N; c += 32) h[c] = gelu_tanh_f(z[c]);
    return;
  }
  float s1 = 0.f, s2 = 0.f;
  for (int c = lane; c < a.N; c += 32) {
    float gv = gelu_tanh_f(z[c]);
    s1 += gv;
    s2 += gv * gv;
  }
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  const float inv_n = 1.0f / (float)a.N;
  const float mu = s1 * inv_n;
  const float var = fmaxf(0.f, s2 * inv_n - mu * mu);  // flax use_fast_variance
  const float rstd = rsqrtf(var + FQL_LN_EPS);
  const float* __restrict__ sc = a.scale.at(p, s, e);
  const float* __restrict__ bi = a.lnbias.at(p, s, e);
  for (int c = lane; c < a.N; c += 32) {
    float gv = gelu_tanh_f(z[c]);
    h[c] = (gv - mu) * rstd * sc[c] + bi[c];
  }
  if (lane == 0) {
    float* m = a.mu.at(p, s, e);
    float* rs = a.rstd.at(p, s, e);
    if (m) m[r] = mu;
    if (rs) rs[r] = rstd;
  }
}

// one warp per row: dZ = LNbwd(dH) * gelu'(Z)
__global__ void __launch_bounds__(256) act_ln_bwd_kernel(ActLnBwdArgs a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + warp;
  const int64_t total = (int64_t)a.P * a.S * a.E * a.M;
  if (row >= total) return;
  const int g = (int)(row / a.M), r = (int)(row % a.M);
  const int e = g % a.E, s = (g / a.E) % a.S, p = g / (a.E * a.S);
  const float* __restrict__ z = a.Z.at(p, s, e) + (int64_t)r * a.ld;
  const float* __restrict__ dh = a.dH.at(p, s, e) + (int64_t)r * a.ld;
  float* __restrict__ dz = a.dZ.at(p, s, e) + (int64_t)r * a.ld;
  const float* __restrict__ sc = a.scale.at(p, s, e);
  float s1 = 0.f, s2 = 0.f;
  for (int c = lane; c < a.N; c += 32) {
    float gv = gelu_tanh_f(z[c]);
    s1 += gv;
    s2 += gv * gv;
  }
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  const float inv_n = 1.0f / (float)a.N;
  const float mu = s1 * inv_n;
  const float var = fmaxf(0.f, s2 * inv_n - mu * mu);
  const float rstd = rsqrtf(var + FQL_LN_EPS);
  float m1 = 0.f, m2 = 0.f;
  for (int c = lane; c < a.N; c += 32) {
    float xh = (gelu_tanh_f(z[c]) - mu) * rstd;
    float dx = dh[c] * sc[c];
    m1 += dx;
    m2 += dx * xh;
  }
  m1 = warp_sum(m1) * inv_n;
  m2 = warp_sum(m2) * inv_n;
  for (int c = lane; c < a.N; c += 32) {
    float zc = z[c];
    float xh = (gelu_tanh_f(zc) - mu) * rstd;
    float dx = dh[c] * sc[c];
    dz[c] = rstd * (dx - m1 - xh * m2) * gelu_tanh_grad_f(zc);
  }
}

// out[c] = sum_r X[r,c] * (Z ? xhat(Z)[r,c] : 1); block = 32 columns x 32 row lanes, 4 independent accumulators per
// thread (the loop is latency-bound otherwise); deterministic tree
__global__ void __launch_bounds__(1024) colsum_kernel(ColSumArgs a, int rows_per_chunk, float* __restrict__ partial) {
  const int g = blockIdx.y;
  const int r_begin = blockIdx.z * rows_per_chunk, r_end = min(a.M, r_begin + rows_per_chunk);
  const int e = g % a.E, s = (g / a.E) % a.S, p = g / (a.E * a.S);
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cx;
  const float* __restrict__ X = a.X.at(p, s, e);
  const float* __restrict__ Z = a.Z.base[p] ? a.Z.at(p, s, e) : nullptr;
  const float* __restrict__ mu = Z ? a.mu.at(p, s, e) : nullptr;
  const float* __restrict__ rstd = Z ? a.rstd.at(p, s, e) : nullptr;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  if (c < a.N) {
    if (!Z) {
      for (int r0 = r_begin + ry; r0 < r_end; r0 += 128) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int r = r0 + u * 32;
          if (r < r_end) acc[u] += X[(int64_t)r * a.ld + c];
        }
      }
    } else {
      for (int r0 = r_begin + ry; r0 < r_end; r0 += 128) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int r = r0 + u * 32;
          if (r < r_end) acc[u] += X[(int64_t)r * a.ld + c] * ((gelu_tanh_f(Z[(int64_t)r * a.ld + c]) - mu[r]) * rstd[r]);
        }
      }
    }
  }
  __shared__ float red[32][33];
  red[ry][cx] = (acc[0] + acc[1]) + (acc[2] + acc[3]);
  __syncthreads();
  if (ry == 0 && c < a.N) {
    float v = 0.f;
#pragma unroll
    for (int q = 0; q < 32; q++) v += red[q][cx];
    if (partial) partial[((int64_t)blockIdx.z * gridDim.y + g) * a.N + c] = v;
    else a.out.at(p, s, e)[c] = v;
  }
}

// second stage: out[g][c] = sum over chunks (fixed order)
__global__ void colsum_final_kernel(ColSumArgs a, const float* __restrict__ partial, int chunks) {
  const int g = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= a.N) return;
  const int e = g % a.E, s = (g / a.E) % a.S, p = g / (a.E * a.S);
  float v = 0.f;
  for (int k = 0; k < chunks; k++) v += partial[((int64_t)k * gridDim.y + g) * a.N + c];
  a.out.at(p, s, e)[c] = v;
}

}  // namespace

int launch_gemm(const GemmArgs& a, cudaStream_t st) {
  if (a.tf32x3) return launch_gemm_tf32x3(a, st);
  if (a.M <= 0 || a.N <= 0) return 0;
  const int G = a.P * a.S * a.E;
  const int64_t big_tiles = (int64_t)((a.M + 63) / 64) * ((a.N + 63) / 64) * G;
  if (big_tiles >= 120 && a.N >= 48) {
    dim3 grid((a.N + 63) / 64, (a.M + 63) / 64, G);
    gemm_kernel<64, 64, 16, 1><<<grid, 256, 0, st>>>(a);
  } else {
    dim3 grid((a.N + 31) / 32, (a.M + 31) / 32, G);
    gemm_kernel<32, 32, 64, 4><<<grid, 256, 0, st>>>(a);
  }
  FQL_CHECK_LAUNCH();
  return 0;
}

int launch_act_ln_fwd(const ActLnArgs& a, cudaStream_t st) {
  const int64_t rows = (int64_t)a.P * a.S * a.E * a.M;
  if (rows == 0) return 0;
  act_ln_fwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(a);
  FQL_CHECK_LAUNCH();
  return 0;
}

int launch_act_ln_bwd(const ActLnBwdArgs& a, cudaStream_t st) {
  const int64_t rows = (int64_t)a.P * a.S * a.E * a.M;
  if (rows == 0) return 0;
  act_ln_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(a);
  FQL_CHECK_LAUNCH();
  return 0;
}

int launch_colsum(const ColSumArgs& a, cudaStream_t st, float* scratch, size_t scratch_floats) {
  const int G = a.P * a.S * a.E;
  const int col_blocks = (a.N + 31) / 32;
  // few rows: one pass.  Many rows: split the rows over enough CTAs to fill the GPU, then a deterministic second stage.
  int chunks = 1;
  if (scratch && a.M >= 1024) {
    chunks = (a.M + 511) / 512;
    while (chunks > 1 && (int64_t)chunks * G * col_blocks > 1184) chunks = (chunks + 1) / 2;
    if ((size_t)chunks * G * a.N > scratch_floats) chunks = 1;
  }
  if (chunks == 1) {
    colsum_kernel<<<dim3(col_blocks, G, 1), 1024, 0, st>>>(a, a.M, nullptr);
    FQL_CHECK_LAUNCH();
    return 0;
  }
  const int rows = (a.M + chunks - 1) / chunks;
  colsum_kernel<<<dim3(col_blocks, G, chunks), 1024, 0, st>>>(a, rows, scratch);
  FQL_CHECK_LAUNCH();
  colsum_final_kernel<<<dim3((a.N + 127) / 128, G), 128, 0, st>>>(a, scratch, chunks);
  FQL_CHECK_LAUNCH();
  return 0;
}
