// losses.cu -- the non-GEMM arithmetic of FQLAgent.total_loss (agents/fql.py:22-111): input assembly, TD target,
// loss reductions and the loss-side gradients.  One CTA per seed for the reductions (deterministic order).
#include "step.cuh"
#include "dp_comm.cuh"

#include <cuda_bf16.h>

namespace {

__device__ __forceinline__ float clip1(float x) { return fminf(fmaxf(x, -1.0f), 1.0f); }

template <int OP>  // 0 sum, 1 max
__device__ float block_reduce(float v, float* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = OP == 0 ? warp_sum(v) : warp_max(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  if (w == 0) {
    float x = lane < nw ? sh[lane] : (OP == 0 ? 0.f : -INFINITY);
    x = OP == 0 ? warp_sum(x) : warp_max(x);
    if (lane == 0) sh[0] = x;
  }
  __syncthreads();
  float r = sh[0];
  return r;
}

// Builds every first-layer input of the step (concats of networks.py:191,229-231) + vel (fql.py:55-56).
__global__ void prep_kernel(StepShape sh, FqlBatch b, WsPtrs w) {
  const int row = blockIdx.x;  // s*B + r
  const int s = row / sh.B, r = row % sh.B;
  const int F = sh.F, A = sh.A, B = sh.B;
  const int KO = F + A, KF = F + A + 1, KC = F + A;
  // what each call site sees as its observation: the batch itself, or (pixel configs) that network's encoder output
  const float* sOn = w.src[0] + (int64_t)row * F;   // onestep(next_obs)        fql.py:25
  const float* sO = w.src[1] + (int64_t)row * F;    // onestep(obs)             fql.py:65,82
  const float* sTn = w.src[2] + (int64_t)row * F;   // target critic(next_obs)  fql.py:28
  const float* sC = w.src[3] + (int64_t)row * F;    // critic(obs)              fql.py:36,70
  const float* sF = w.src[4] + (int64_t)row * F;    // bc flow(obs)             fql.py:58,64
  const float* act = b.actions + (int64_t)row * A;
  const float* zn = b.z_next + (int64_t)row * A;
  const float* x0 = b.x0 + (int64_t)row * A;
  const float* z = b.z + (int64_t)row * A;
  const float* zm = b.z_metric + (int64_t)row * A;
  const float t = b.t[row];
  float* xo0 = w.XO + ((int64_t)s * 3 * B + r) * KO;
  float* xo1 = xo0 + (int64_t)B * KO;
  float* xo2 = xo1 + (int64_t)B * KO;
  float* xf0 = w.XF + ((int64_t)s * 2 * B + r) * KF;
  float* xf1 = xf0 + (int64_t)B * KF;
  float* xc0 = w.XC + ((int64_t)(0 * sh.S + s) * B + r) * KC;
  float* xc1 = w.XC + ((int64_t)(1 * sh.S + s) * B + r) * KC;
  float* xc2 = w.XC + ((int64_t)(2 * sh.S + s) * B + r) * KC;
  for (int c = threadIdx.x; c < F; c += blockDim.x) {
    const float o = sO[c], f = sF[c], cc = sC[c];
    xo0[c] = sOn[c]; xo1[c] = o; xo2[c] = o;
    xf0[c] = f; xf1[c] = f;
    xc0[c] = sTn[c]; xc1[c] = cc; xc2[c] = cc;
  }
  for (int c = threadIdx.x; c < A; c += blockDim.x) {
    float a = act[c], x = x0[c];
    xo0[F + c] = zn[c]; xo1[F + c] = z[c]; xo2[F + c] = zm[c];
    xf0[F + c] = (1.0f - t) * x + t * a;
    xf1[F + c] = z[c];
    xc1[F + c] = a;
    w.vel[(int64_t)row * A + c] = a - x;
    if (w.euler_a) w.euler_a[(int64_t)row * A + c] = z[c];
  }
  if (threadIdx.x == 0) {
    xf0[F + A] = t;
    xf1[F + A] = 0.0f;  // Euler step 0: t = 0/flow_steps (fql.py:167)
  }
}

// After the one-step actor pass on rows {(s',z_next), (s,z), (s,z')}: clip and scatter the actions into the critic
// inputs (fql.py:25-26, 69-70) and reduce the logging mse (fql.py:82-83).
// parts: bit 0 = the critic inputs (row groups (s',z') and (s,z)), bit 1 = the mse metric (row group (s,z''))
__global__ void post_onestep_kernel(StepShape sh, FqlBatch b, WsPtrs w, float* raw, int parts) {
  __shared__ float red[32];
  const int s = blockIdx.x;
  const int F = sh.F, A = sh.A, B = sh.B, KC = F + A;
  const float* out = w.O_out + (int64_t)s * 3 * B * A;
  float mse = 0.f;
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < B * A; i += gridDim.y * blockDim.x) {
    const int r = i / A, c = i % A;
    if (parts & 1) {
      w.XC[((int64_t)(0 * sh.S + s) * B + r) * KC + F + c] = clip1(out[i]);
      w.XC[((int64_t)(2 * sh.S + s) * B + r) * KC + F + c] = clip1(out[(int64_t)B * A + i]);
    }
    if (parts & 2) {
      float d = clip1(out[(int64_t)2 * B * A + i]) - b.actions[(int64_t)s * B * A + i];
      mse += d * d;
    }
  }
  if (!(parts & 2)) return;
  mse = block_reduce<0>(mse, red);
  if (threadIdx.x == 0) atomicAdd(&raw[s * FQL_NUM_RAW + RAW_MSE], mse);  // raw is zeroed at the start of the step
}

// TD target + critic loss gradient (fql.py:28-44) and the actor's Q statistics / dQ seed (fql.py:70-76).
// qout: [3][S][2][B]  (0: target critic on (s',a'), 1: critic on (s,a), 2: critic on (s, clip a_pi))
// parts: bit 0 = TD / critic-loss half (problems 0, 1), bit 1 = actor-Q half (problem 2)
// Sum of one float per rank over the data-parallel ranks, identical bits on every rank (rank order): thread 0 of the CTA stores a
// {epoch, value} word into slot [rank][s] of every peer (one aligned 8-byte store: the flag travels with the datum, no fence)
// and collects the world words of its own pad.
__device__ float dp_sum_over_ranks(const DpLamArgs& l, int s, int S, float mine) {
  const uint32_t ep = l.epoch[s] + 1;
  const unsigned long long word = ((unsigned long long)ep << 32) | (unsigned long long)__float_as_uint(mine);
  for (int r = 0; r < l.world; r++)
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(l.slots[r] + (int64_t)l.rank * S + s), "l"(word) : "memory");
  float tot = 0.f;
  for (int r = 0; r < l.world; r++) {
    const unsigned long long* src = l.slots[l.rank] + (int64_t)r * S + s;
    unsigned long long v;
    unsigned long long t0 = 0;
    for (;;) {
      asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(src) : "memory");
      if ((uint32_t)(v >> 32) == ep) break;
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      if (t0 == 0) t0 = t;
      if (t - t0 > 60ull * 1000000000ull) {
        printf("fql_b200: data-parallel |q| exchange timed out waiting for rank %d (seed %d)\n", r, s);
        __trap();
      }
    }
    tot += __uint_as_float((uint32_t)v);
  }
  l.epoch[s] = ep;
  return tot;
}

__global__ void critic_post_kernel(StepShape sh, FqlHparams hp, FqlBatch b, WsPtrs w, float* raw, int parts, DpLamArgs dpl) {
  // grid (S, nc): CTA c of seed s reduces rows c, c + nc, ... ; the partial sums of the nc CTAs are combined in CTA order by the
  // last one to finish (ticket counter), so the result does not depend on scheduling
  __shared__ float red[32];
  __shared__ int s_last;
  const int s = blockIdx.x, cta = blockIdx.y, nc = gridDim.y;
  const int B = sh.B, S = sh.S;
  const float* q_t = w.C_out + ((int64_t)(0 * S + s) * 2) * B;
  const float* q_c = w.C_out + ((int64_t)(1 * S + s) * 2) * B;
  const float* q_p = w.C_out + ((int64_t)(2 * S + s) * 2) * B;
  const float inv_2gb = 1.0f / (2.0f * (float)sh.GB);
  float sq = 0.f, qs = 0.f, qmx = -INFINITY, qmn = INFINITY, ps = 0.f, pa = 0.f;
  for (int r = cta * blockDim.x + threadIdx.x; r < B; r += nc * blockDim.x) {
    if (parts & 1) {
      const float t0 = q_t[r], t1 = q_t[B + r];
      const float nq = sh.q_agg_min ? fminf(t0, t1) : (t0 + t1) * 0.5f;
      const float y = b.rewards[(int64_t)s * B + r] + hp.discount * b.masks[(int64_t)s * B + r] * nq;
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const float q = q_c[h * B + r];
        const float d = q - y;
        sq += d * d;
        qs += q;
        qmx = fmaxf(qmx, q);
        qmn = fminf(qmn, q);
        w.dq[((int64_t)s * 2 + h) * B + r] = 2.0f * d * inv_2gb;
      }
    }
    if (parts & 2) {
      const float qp = (q_p[r] + q_p[B + r]) * 0.5f;
      ps += qp;
      pa += fabsf(qp);
    }
  }
  // per-CTA partials: [half][S][64][4]
  float* part1 = w.cpost_part + ((int64_t)(0 * S + s) * 64 + cta) * 4;
  float* part2 = w.cpost_part + ((int64_t)(1 * S + s) * 64 + cta) * 4;
  if (parts & 1) {
    sq = block_reduce<0>(sq, red);
    qs = block_reduce<0>(qs, red);
    qmx = block_reduce<1>(qmx, red);
    qmn = -block_reduce<1>(-qmn, red);
    if (threadIdx.x == 0) { part1[0] = sq; part1[1] = qs; part1[2] = qmx; part1[3] = -qmn; }
  }
  if (parts & 2) {
    ps = block_reduce<0>(ps, red);
    pa = block_reduce<0>(pa, red);
    if (threadIdx.x == 0) { part2[0] = ps; part2[1] = pa; }
  }
  if (threadIdx.x == 0) {
    __threadfence();
    int* ticket = w.cpost_ticket + ((parts & 3) - 1) * S + s;      // one counter per (call variant, seed)
    const int t = atomicAdd(ticket, 1);
    s_last = (t == nc - 1);
    if (s_last) *ticket = 0;                                        // ready for the next step
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  float* rw = raw + s * FQL_NUM_RAW;
  if ((parts & 1) && threadIdx.x == 0) {
    float a0 = 0.f, a1 = 0.f, a2 = -INFINITY, a3 = -INFINITY;
    for (int c = 0; c < nc; c++) {
      const float* p = w.cpost_part + ((int64_t)(0 * S + s) * 64 + c) * 4;
      a0 += __ldcg(p); a1 += __ldcg(p + 1); a2 = fmaxf(a2, __ldcg(p + 2)); a3 = fmaxf(a3, __ldcg(p + 3));
    }
    rw[RAW_CRITIC_SQ] = a0; rw[RAW_Q_SUM] = a1; rw[RAW_Q_MAX] = a2; rw[RAW_Q_NEGMIN] = a3;
  }
  if (parts & 2) {
    __shared__ float s_pa;
    if (threadIdx.x == 0) {
      float a0 = 0.f, a1 = 0.f;
      for (int c = 0; c < nc; c++) {
        const float* p = w.cpost_part + ((int64_t)(1 * S + s) * 64 + c) * 4;
        a0 += __ldcg(p); a1 += __ldcg(p + 1);
      }
      rw[RAW_QPI_SUM] = a0; rw[RAW_QPI_ABS] = a1;
      // lam = 1/mean|q| over the GLOBAL batch, stop-gradient (fql.py:74-76): data-parallel ranks exchange their sums here
      if (sh.normalize_q_loss && dpl.world > 1) a1 = dp_sum_over_ranks(dpl, s, sh.S, a1);
      s_pa = a1;
    }
    __syncthreads();
    float lam = 1.0f;
    if (sh.normalize_q_loss) lam = 1.0f / (s_pa / (float)sh.GB);
    const float dqs = -lam * inv_2gb;
    for (int i = threadIdx.x; i < 2 * B; i += blockDim.x) w.dqs[(int64_t)s * 2 * B + i] = dqs;
  }
}

// BC flow-matching loss gradient (fql.py:58-59): pred rows are rows [0,B) of the bc-flow pass output.
__global__ void bc_post_kernel(StepShape sh, WsPtrs w, float* raw) {
  __shared__ float red[32];
  const int s = blockIdx.x;
  const int A = sh.A, B = sh.B;
  const float* pred = w.F_out + (int64_t)s * 2 * B * A;
  const float scale = 2.0f / ((float)sh.GB * (float)A);
  float sq = 0.f;
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < B * A; i += gridDim.y * blockDim.x) {
    float d = pred[i] - w.vel[(int64_t)s * B * A + i];
    sq += d * d;
    w.dpred[(int64_t)s * B * A + i] = scale * d;
  }
  sq = block_reduce<0>(sq, red);
  if (threadIdx.x == 0) atomicAdd(&raw[s * FQL_NUM_RAW + RAW_BC_SQ], sq);
}

// One Euler step (fql.py:166-169): a += v / flow_steps on the Euler rows of XF; t column <- (i+1)/flow_steps;
// after the last step: target = clip(a) (fql.py:170).
__global__ void euler_update_kernel(StepShape sh, WsPtrs w, int step) {
  const int A = sh.A, B = sh.B, KF = sh.F + sh.A + 1;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)sh.S * B * A) return;
  const int c = (int)(i % A);
  const int64_t row = i / A;
  const int s = (int)(row / B), r = (int)(row % B);
  float* xf = w.XF + ((int64_t)s * 2 * B + B + r) * KF;
  const float v = w.F_out[((int64_t)s * 2 * B + B + r) * A + c];
  const float a = xf[sh.F + c] + v / (float)sh.flow_steps;
  xf[sh.F + c] = a;
  if (c == 0) xf[sh.F + A] = (float)((double)(step + 1) / (double)sh.flow_steps);
  if (step == sh.flow_steps - 1) w.target[i] = clip1(a);
}

// Distillation loss + dL/da_pi (fql.py:65-79): da = alpha*2(a_pi-target)/(GB*A) + [dQ/da through clip].
// dX0: [S][2][B][KC] input-gradient of the critic(s, clip a_pi) pass; the two heads are summed (input broadcast).
__global__ void actor_grad_kernel(StepShape sh, FqlHparams hp, WsPtrs w, float* raw, __nv_bfloat16* dapib) {
  __shared__ float red[32];
  const int s = blockIdx.x;
  const int A = sh.A, B = sh.B, KC = sh.F + sh.A;
  const float* api = w.O_out + ((int64_t)s * 3 * B + B) * A;
  const float scale = hp.alpha * 2.0f / ((float)sh.GB * (float)A);
  float sq = 0.f;
  // dapib (tensor-core mode): the same gradient as the zero-padded bf16 [B][64] operand of the first dgrad GEMM
  if (dapib) {
    const int P = 64 - A;
    for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < B * P; i += gridDim.y * blockDim.x)
      dapib[((int64_t)s * B + i / P) * 64 + A + i % P] = __float2bfloat16(0.f);
  }
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < B * A; i += gridDim.y * blockDim.x) {
    const int r = i / A, c = i % A;
    const float a = api[i];
    const float d = a - w.target[(int64_t)s * B * A + i];
    sq += d * d;
    const float g0 = w.dX0[(((int64_t)s * 2 + 0) * B + r) * KC + sh.F + c];
    const float g1 = w.dX0[(((int64_t)s * 2 + 1) * B + r) * KC + sh.F + c];
    const float inside = (a >= -1.0f && a <= 1.0f) ? 1.0f : 0.0f;
    const float g = scale * d + (g0 + g1) * inside;
    w.dapi[(int64_t)s * B * A + i] = g;
    if (dapib) dapib[((int64_t)s * B + r) * 64 + c] = __float2bfloat16(g);
  }
  sq = block_reduce<0>(sq, red);
  if (threadIdx.x == 0) atomicAdd(&raw[s * FQL_NUM_RAW + RAW_DISTILL_SQ], sq);
}

// info[13] from the (all-reduced) raw accumulators + gradient statistics.
__global__ void finalize_info_kernel(StepShape sh, FqlHparams hp, const float* raw, int ranks, const float* gstats, float* info,
                                     int with_grad_stats) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= sh.S) return;
  fql_finalize_info_seed(sh, hp, raw, ranks, gstats, info, s, with_grad_stats);
}

// clip(x) elementwise (fql.py:152)
__global__ void clip_kernel(const float* in, float* out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = clip1(in[i]);
}

// generic concat of up to 3 row blocks into X [rows, k0+k1+k2]; x2 may be a scalar constant column
__global__ void concat_kernel(const float* x0, int k0, const float* x1, int k1, float c2, int k2, float* out, int64_t rows) {
  const int K = k0 + k1 + k2;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * K) return;
  const int64_t r = i / K;
  const int c = (int)(i % K);
  out[i] = c < k0 ? x0[r * k0 + c] : (c < k0 + k1 ? x1[r * k1 + (c - k0)] : c2);
}

// Euler step for the standalone compute_flow_actions entry: X [rows, F+A+1] in place
__global__ void euler_inplace_kernel(float* X, const float* v, int F, int A, int64_t rows, int step, int nsteps, float* out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * A) return;
  const int64_t r = i / A;
  const int c = (int)(i % A);
  float* x = X + r * (F + A + 1);
  const float a = x[F + c] + v[i] / (float)nsteps;
  x[F + c] = a;
  if (c == 0) x[F + A] = (float)((double)(step + 1) / (double)nsteps);
  if (step == nsteps - 1) out[i] = clip1(a);
}

}  // namespace

// CTAs per seed of the elementwise loss kernels: one per 8192 (row, action) elements; a single CTA (deterministic sum order)
// for small batches, several + one float atomicAdd each for large ones
static int loss_ctas(const StepShape& sh) {
  const int64_t n = (int64_t)sh.B * sh.A;
  int c = (int)((n + 8191) / 8192);
  return c < 1 ? 1 : (c > 64 ? 64 : c);
}

int launch_prep(const StepShape& sh, const FqlBatch& b, const WsPtrs& w, cudaStream_t st) {
  prep_kernel<<<sh.S * sh.B, 64, 0, st>>>(sh, b, w);
  FQL_CHECK_LAUNCH();
  return 0;
}
int launch_post_onestep(const StepShape& sh, const FqlBatch& b, const WsPtrs& w, float* raw, cudaStream_t st, int parts) {
  post_onestep_kernel<<<dim3(sh.S, loss_ctas(sh)), 1024, 0, st>>>(sh, b, w, raw, parts);
  FQL_CHECK_LAUNCH();
  return 0;
}
int launch_critic_post(const StepShape& sh, const FqlHparams& hp, const FqlBatch& b, const WsPtrs& w, float* raw, cudaStream_t st, int parts,
                       const DpLamArgs* dpl) {
  DpLamArgs l;
  memset(&l, 0, sizeof(l));
  if (dpl) l = *dpl;
  int nc = (sh.B + 2047) / 2048;
  nc = nc < 1 ? 1 : (nc > 64 ? 64 : nc);
  critic_post_kernel<<<dim3(sh.S, nc), 1024, 0, st>>>(sh, hp, b, w, raw, parts, l);
  FQL_CHECK_LAUNCH();
  return 0;
}
int launch_bc_post(const StepShape& sh, const WsPtrs& w, float* raw, cudaStream_t st) {
  bc_post_kernel<<<dim3(sh.S, loss_ctas(sh)), 1024, 0, st>>>(sh, w, raw);
  FQL_CHECK_LAUNCH();
  return 0;
}
int launch_euler_update(const StepShape& sh, const WsPtrs& w, int step, cudaStream_t st) {
  const int64_t n = (int64_t)sh.S * sh.B * sh.A;
  euler_update_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(sh, w, step);
  FQL_CHECK_LAUNCH();
  return 0;
}
int launch_actor_grad(const StepShape& sh, const FqlHparams& hp, const WsPtrs& w, float* raw, cudaStream_t st, void* dapib) {
  actor_grad_kernel<<<dim3(sh.S, loss_ctas(sh)), 1024, 0, st>>>(sh, hp, w, raw, reinterpret_cast<__nv_bfloat16*>(dapib));
  FQL_CHECK_LAUNCH();
  return 0;
}
int launch_finalize_info(const StepShape& sh, const FqlHparams& hp, const float* raw, int ranks, const float* gstats, float* info,
                         int with_grad_stats, cudaStream_t st) {
  finalize_info_kernel<<<(sh.S + 63) / 64, 64, 0, st>>>(sh, hp, raw, ranks, gstats, info, with_grad_stats);
  FQL_CHECK_LAUNCH();
  return 0;
}
int launch_clip(const float* in, float* out, int64_t n, cudaStream_t st) {
  if (n == 0) return 0;
  clip_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(in, out, n);
  FQL_CHECK_LAUNCH();
  return 0;
}
int launch_concat(const float* x0, int k0, const float* x1, int k1, float c2, int k2, float* out, int64_t rows, cudaStream_t st) {
  const int64_t n = rows * (k0 + k1 + k2);
  if (n == 0) return 0;
  concat_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x0, k0, x1, k1, c2, k2, out, rows);
  FQL_CHECK_LAUNCH();
  return 0;
}
int launch_euler_inplace(float* X, const float* v, int F, int A, int64_t rows, int step, int nsteps, float* out, cudaStream_t st) {
  const int64_t n = rows * A;
  if (n == 0) return 0;
  euler_inplace_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(X, v, F, A, rows, step, nsteps, out);
  FQL_CHECK_LAUNCH();
  return 0;
}
