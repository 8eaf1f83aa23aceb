// optim.cu -- fused multi-tensor optimizer pass over the flat arenas (north_star #5):
//   gradient statistics   utils/flax_utils.py:139-149  (per-leaf max / min / L2 -> max, min, L1-of-L2)
//   optax.adam apply      utils/flax_utils.py:120-130, agents/fql.py:237 (b1 .9, b2 .999, eps 1e-8, eps_root 0)
//   Polyak target update  agents/fql.py:113-120 -- from the PRE-step critic and PRE-step target (SURVEY F6)
// One pass: each CTA owns one FQL_LEAF_PAD-float block (never straddles a leaf), reads g,p,m,v once, writes p,m,v
// (+ target block for critic leaves).  Target-critic leaves have exactly-zero gradients (SURVEY F7) so Adam is the
// identity on them; they are only written by the Polyak half.  HBM-bound: 28 B/param (+8 B/critic param).
#include "step.cuh"

#include <cuda_bf16.h>

namespace {

// ADAM_U consecutive blocks per CTA, all loads issued before the first use.  Measured on B200 (110 MB pass, cold L2): U = 1
// 21.8 us, U = 4 27.3 us (registers halve the resident CTAs) -- more CTAs beat more loads per thread.
constexpr int ADAM_U = 1;
template <bool TABLE>
__global__ void __launch_bounds__(256) adam_polyak_stats_kernel(Layout L, FqlHparams hp, float* __restrict__ params,
                                                                float* __restrict__ mu, float* __restrict__ nu,
                                                                const float* __restrict__ grads,
                                                                const float* __restrict__ bc,
                                                                float* __restrict__ partials, __nv_bfloat16* __restrict__ shadow,
                                                                int64_t shadow_seed, int blk0, int blk1, int nblk) {
  const int s = blockIdx.y;
  const int b0 = blk0 + blockIdx.x * ADAM_U;
  const int64_t base = (int64_t)s * L.arena;
  const NetView& tgt = L.net[FQL_NET_TARGET_CRITIC];
  const NetView& cri = L.net[FQL_NET_CRITIC];
  float4 g[ADAM_U], p[ADAM_U], m[ADAM_U], v[ADAM_U], tp[ADAM_U];
  bool act[ADAM_U], pol[ADAM_U];
#pragma unroll
  for (int u = 0; u < ADAM_U; u++) {
    const int64_t off = (int64_t)(b0 + u) * FQL_LEAF_PAD + threadIdx.x * 4;
    act[u] = (b0 + u < blk1) && !(off >= tgt.begin && off < tgt.end);  // block-uniform
    pol[u] = act[u] && off >= cri.begin && off < cri.end;
    if (act[u]) {
      g[u] = *reinterpret_cast<const float4*>(grads + base + off);
      p[u] = *reinterpret_cast<const float4*>(params + base + off);
      m[u] = *reinterpret_cast<const float4*>(mu + base + off);
      v[u] = *reinterpret_cast<const float4*>(nu + base + off);
    }
    if (pol[u]) tp[u] = *reinterpret_cast<const float4*>(params + base + off - cri.begin + tgt.begin);
  }
  // optax bias_correction: 1 - decay**count in float32, correctly rounded -- computed once per step by zero_bc_kernel (a double
  // pow in every CTA of this pass cost ~3 us per CTA wave)
  const float bc1 = bc[0], bc2 = bc[1];
  const float lr = seed_hp<TABLE>(hp, s, &FqlHparams::lr), tau = seed_hp<TABLE>(hp, s, &FqlHparams::tau),
              omt = seed_hp<TABLE>(hp, s, &FqlHparams::one_minus_tau);
  __shared__ float smx[ADAM_U][8], smn[ADAM_U][8], ssq[ADAM_U][8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int u = 0; u < ADAM_U; u++) {
    if (!act[u]) continue;
    const int64_t off = (int64_t)(b0 + u) * FQL_LEAF_PAD + threadIdx.x * 4;
    float gr[4] = {g[u].x, g[u].y, g[u].z, g[u].w}, pr[4] = {p[u].x, p[u].y, p[u].z, p[u].w}, mr[4] = {m[u].x, m[u].y, m[u].z, m[u].w},
          vr[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
    float pn[4];
    float mx = -INFINITY, mn = INFINITY, sq = 0.f;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const float gi = gr[i];
      mx = fmaxf(mx, gi);
      mn = fminf(mn, gi);
      sq += gi * gi;
      mr[i] = hp.beta1 * mr[i] + hp.one_minus_beta1 * gi;
      vr[i] = hp.beta2 * vr[i] + hp.one_minus_beta2 * gi * gi;
      const float mhat = mr[i] / bc1;
      const float vhat = vr[i] / bc2;
      pn[i] = pr[i] + (-lr * (mhat / (sqrtf(vhat) + hp.eps)));
    }
    *reinterpret_cast<float4*>(params + base + off) = make_float4(pn[0], pn[1], pn[2], pn[3]);
    if (shadow) {  // bf16 tensor-core operand copy of the fresh parameters (same [in,out] layout)
      __nv_bfloat162 lo = __floats2bfloat162_rn(pn[0], pn[1]), hi = __floats2bfloat162_rn(pn[2], pn[3]);
      *reinterpret_cast<uint2*>(shadow + (int64_t)s * shadow_seed + off) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
    }
    *reinterpret_cast<float4*>(mu + base + off) = make_float4(mr[0], mr[1], mr[2], mr[3]);
    *reinterpret_cast<float4*>(nu + base + off) = make_float4(vr[0], vr[1], vr[2], vr[3]);
    if (pol[u]) {  // Polyak with the pre-step critic values still in registers
      const int64_t toff = base + off - cri.begin + tgt.begin;
      float4 t4 = tp[u];
      t4.x = pr[0] * tau + t4.x * omt;
      t4.y = pr[1] * tau + t4.y * omt;
      t4.z = pr[2] * tau + t4.z * omt;
      t4.w = pr[3] * tau + t4.w * omt;
      *reinterpret_cast<float4*>(params + toff) = t4;
      if (shadow) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(t4.x, t4.y), hi = __floats2bfloat162_rn(t4.z, t4.w);
        *reinterpret_cast<uint2*>(shadow + (int64_t)s * shadow_seed + (toff - base)) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
      }
    }
    mx = warp_max(mx);
    mn = warp_min(mn);
    sq = warp_sum(sq);
    if (lane == 0) { smx[u][w] = mx; smn[u][w] = mn; ssq[u][w] = sq; }
  }
  __syncthreads();
  if (threadIdx.x < ADAM_U && b0 + (int)threadIdx.x < blk1) {
    const int u = threadIdx.x;
    float* part = partials + ((int64_t)s * nblk + b0 + u) * 4;
    // act[] is indexed with a compile-time constant everywhere else; recompute the flag for the runtime index here
    const int64_t off = (int64_t)(b0 + u) * FQL_LEAF_PAD;
    const bool a_u = !(off >= tgt.begin && off < tgt.end);
    float a = 0.f, b = 0.f, c = 0.f;
    if (a_u) {
      a = smx[u][0]; b = smn[u][0]; c = ssq[u][0];
#pragma unroll
      for (int i = 1; i < 8; i++) { a = fmaxf(a, smx[u][i]); b = fminf(b, smn[u][i]); c += ssq[u][i]; }
    }
    part[0] = a; part[1] = b; part[2] = c;
  }
}

// one CTA per seed, one WARP per leaf (lanes stride over the leaf's block partials): per-leaf L2 norms, then the three
// scalars of flax_utils.py:147-149
template <bool TABLE>
__global__ void __launch_bounds__(1024) grad_stats_final_kernel(Layout L, const float* __restrict__ partials,
                                                                float* __restrict__ gstats, int32_t* count_inc, FinArgs fin) {
  const int s = blockIdx.x;
  const int nblk = L.leaf_blk[L.n_leaves];
  const float* part = partials + (int64_t)s * nblk * 4;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __shared__ float smx[32], smn[32], snorm[32];
  float wmx = 0.f, wmn = 0.f, wnorm = 0.f;  // the target critic's zero gradients are leaves too (SURVEY F7)
  for (int leaf = w; leaf < L.n_leaves; leaf += 32) {
    if (L.leaf_net[leaf] == FQL_NET_TARGET_CRITIC) continue;
    float mx = -INFINITY, mn = INFINITY, sq = 0.f;
    const int bend = L.leaf_blk[leaf + 1];
    const float4* p4 = reinterpret_cast<const float4*>(part);
    for (int b0 = L.leaf_blk[leaf] + lane; b0 < bend; b0 += 256) {  // eight independent 16-byte loads in flight per lane: a 512 x 512 leaf
      float4 v[8];                                                   // (256 blocks) is ONE round trip, the critic's [2,512,512] two
#pragma unroll
      for (int u = 0; u < 8; u++) v[u] = (b0 + 32 * u < bend) ? p4[b0 + 32 * u] : make_float4(-INFINITY, INFINITY, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < 8; u++) {
        mx = fmaxf(mx, v[u].x);
        mn = fminf(mn, v[u].y);
        sq += v[u].z;
      }
    }
    mx = warp_max(mx);
    mn = warp_min(mn);
    sq = warp_sum(sq);
    wmx = fmaxf(wmx, mx);
    wmn = fminf(wmn, mn);
    wnorm += sqrtf(sq);
  }
  if (lane == 0) { smx[w] = wmx; smn[w] = wmn; snorm[w] = wnorm; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = smx[0], b = smn[0], c = snorm[0];
    for (int i = 1; i < 32; i++) { a = fmaxf(a, smx[i]); b = fminf(b, smn[i]); c += snorm[i]; }
    gstats[s * 4 + 0] = a;
    gstats[s * 4 + 1] = b;
    gstats[s * 4 + 2] = c;
    if (s == 0 && count_inc) count_inc[0] += 1;  // optax count / TrainState.step advance (flax_utils.py:126)
    if (fin.info) fql_finalize_info_seed<TABLE>(fin.sh, fin.hp, fin.raw, fin.ranks, gstats, fin.info, s, 1);
  }
}

// A correctly rounded float pow (via double): one ulp of pow(0.999f, t) is 7.5e-6 of (1 - 0.999^8), so a sloppy powf would show
// up in the parameters at the fp32 mode's 1e-5 tolerance.
__global__ void zero_bc_kernel(float4* p, int64_t n4, const int32_t* __restrict__ count, float beta1, float beta2, float* bc, int* tickets,
                               int n_tickets) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n4) p[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (tickets && i < n_tickets) tickets[i] = 0;   // arrival counters of the multi-CTA loss kernel (the workspace is not zero-initialised)
  if (i == 0 && count) {
    const double t = (double)(count[0] + 1);
    bc[0] = 1.0f - (float)pow((double)beta1, t);
    bc[1] = 1.0f - (float)pow((double)beta2, t);
  }
}

// FQLAgent.target_update (agents/fql.py:113-120) on its own: target <- tau * critic + (1 - tau) * target, plus the bf16 shadow.
template <bool TABLE>
__global__ void target_update_kernel(float* __restrict__ params, __nv_bfloat16* __restrict__ shadow, int64_t arena, int64_t shadow_seed,
                                     int64_t cri0, int64_t tgt0, int64_t n, FqlHparams hp) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const int s = blockIdx.y;
  if (i >= n) return;
  const float tau = seed_hp<TABLE>(hp, s, &FqlHparams::tau), omt = seed_hp<TABLE>(hp, s, &FqlHparams::one_minus_tau);
  const float4 p = *reinterpret_cast<const float4*>(params + s * arena + cri0 + i);
  float4 t = *reinterpret_cast<const float4*>(params + s * arena + tgt0 + i);
  t.x = p.x * tau + t.x * omt;
  t.y = p.y * tau + t.y * omt;
  t.z = p.z * tau + t.z * omt;
  t.w = p.w * tau + t.w * omt;
  *reinterpret_cast<float4*>(params + s * arena + tgt0 + i) = t;
  if (shadow) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(t.x, t.y), hi = __floats2bfloat162_rn(t.z, t.w);
    *reinterpret_cast<uint2*>(shadow + s * shadow_seed + tgt0 + i) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
  }
}

__global__ void zero_kernel(float4* p, int64_t n4) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n4) p[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

}  // namespace

int launch_adam_polyak_stats(const Layout& L, const FqlHparams& hp, int S, float* params, float* mu, float* nu,
                             const float* grads, const float* bc, float* partials, void* shadow, int64_t shadow_seed, cudaStream_t st,
                             int blk0, int blk1) {
  const int nblk = L.leaf_blk[L.n_leaves];
  if (blk1 < 0) blk1 = nblk;
  if (blk1 <= blk0) return 0;
  dim3 grid((blk1 - blk0 + ADAM_U - 1) / ADAM_U, S);
  (hp.per_seed ? adam_polyak_stats_kernel<true> : adam_polyak_stats_kernel<false>)<<<grid, 256, 0, st>>>(L, hp, params, mu, nu, grads, bc, partials, reinterpret_cast<__nv_bfloat16*>(shadow), shadow_seed, blk0, blk1,
                                                 nblk);
  FQL_CHECK_LAUNCH();
  return 0;
}

int launch_grad_stats_final(const Layout& L, int S, const float* partials, float* gstats, int32_t* count_inc, cudaStream_t st,
                            const FinArgs* fin) {
  FinArgs f;
  memset(&f, 0, sizeof(f));
  if (fin) f = *fin;
  (f.hp.per_seed ? grad_stats_final_kernel<true> : grad_stats_final_kernel<false>)<<<S, 1024, 0, st>>>(L, partials, gstats, count_inc, f);
  FQL_CHECK_LAUNCH();
  return 0;
}

int launch_zero_bc(float* p, int64_t n, const int32_t* count, const FqlHparams& hp, float* bc, cudaStream_t st, int* tickets, int n_tickets) {
  const int64_t n4 = n / 4;
  const int64_t work = n4 > n_tickets ? n4 : n_tickets;
  const unsigned blocks = (unsigned)((work + 255) / 256);
  zero_bc_kernel<<<blocks ? blocks : 1, 256, 0, st>>>(reinterpret_cast<float4*>(p), n4, count, hp.beta1, hp.beta2, bc, tickets, n_tickets);
  FQL_CHECK_LAUNCH();
  return 0;
}

extern "C" int fql_target_update(const FqlDims* d, const FqlHparams* hp, float* params, void* shadow, void* stream) {
  Layout L;
  FQL_TRY(fql_build_layout(d, &L));
  FQL_REQUIRE(hp && params, "fql_target_update: NULL argument");
  FQL_TRY(check_seed_table(hp));
  const NetView& cri = L.net[FQL_NET_CRITIC];
  const NetView& tgt = L.net[FQL_NET_TARGET_CRITIC];
  const int64_t n = cri.end - cri.begin;
  FQL_REQUIRE(n == tgt.end - tgt.begin && n % 4 == 0, "critic / target critic ranges differ");
  const bool tcm = d->precision == FQL_PRECISION_BF16_TC;
  FQL_REQUIRE(!tcm || shadow, "FQL_PRECISION_BF16_TC needs the bf16 shadow");
  dim3 grid((unsigned)((n / 4 + 255) / 256), d->num_seeds);
  (hp->per_seed ? target_update_kernel<true> : target_update_kernel<false>)<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      params, tcm ? reinterpret_cast<__nv_bfloat16*>(shadow) : nullptr, L.arena, tcm ? tc_shadow_seed_elems(d, L) : 0, cri.begin, tgt.begin, n,
      *hp);
  FQL_CHECK_LAUNCH();
  if (tcm) FQL_TRY(tc_refresh_shadow_lastlayer(d, L, params, shadow, reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int launch_zero(float* p, int64_t n, cudaStream_t st) {
  if (n == 0) return 0;
  const int64_t n4 = n / 4;  // arenas and workspace slices are multiples of 4 floats
  zero_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(reinterpret_cast<float4*>(p), n4);
  FQL_CHECK_LAUNCH();
  return 0;
}
