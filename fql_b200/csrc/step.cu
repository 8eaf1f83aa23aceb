// step.cu -- arena layout, workspace map and the stream-level schedule of FQLAgent.update (agents/fql.py:122-133).
//
// Two schedules of one step, both forked/joined with events on the context's internal streams and capturable into a CUDA graph:
//   fp32 parity mode (enqueue_step): three streams
//     S0: prep -> onestep actor on {(s',z_next),(s,z),(s,z')} (fql.py:25,65,82) -> {target critic, critic(s,a),
//         critic(s,clip a_pi)} x 2 heads as ONE grouped pass (fql.py:28,36,70) -> TD/Q post -> critic input-gradient
//         -> [join Euler] distill + dL/da_pi -> onestep backward
//     S1: bc-flow on {(s,x_t,t), Euler step 0} -> Euler steps 1..n-1 (fql.py:155-171)      <- longest dependent chain
//     S2: BC loss + bc-flow backward (fql.py:58-59); critic backward (fql.py:36-37)
//     S0: join -> grad stats + Adam + Polyak (optim.cu) -> info
//   bf16 tensor-core mode (enqueue_grads_tc): the same dependency graph with the dependent chains on the high-priority streams
//     S0/S1 and everything that only consumes on low-priority side streams; timeline in DESIGN.md section 5.
#include "step.cuh"
#include "dp_comm.cuh"

#include <cuda_bf16.h>
#include <stdarg.h>

#include <vector>

// ---------------------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
thread_local long long g_fql_launches = 0;
void fql_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---------------------------------------------------------------------------------------------------------
// layout
// ---------------------------------------------------------------------------------------------------------
int fql_validate_dims(const FqlDims* d) {
  FQL_REQUIRE(d != nullptr, "dims is NULL");
  FQL_REQUIRE(d->batch >= 1 && d->global_batch >= d->batch, "batch=%d global_batch=%d", d->batch, d->global_batch);
  FQL_REQUIRE(d->obs_dim >= 1 && d->action_dim >= 1, "obs_dim=%d action_dim=%d", d->obs_dim, d->action_dim);
  FQL_REQUIRE(d->hidden >= 1 && d->num_hidden >= 1 && d->num_hidden + 1 <= FQL_MAXL, "hidden=%d num_hidden=%d", d->hidden, d->num_hidden);
  FQL_REQUIRE(d->num_seeds >= 1, "num_seeds=%d", d->num_seeds);
  FQL_REQUIRE(d->flow_steps >= 1, "flow_steps=%d", d->flow_steps);
  FQL_REQUIRE(d->precision == FQL_PRECISION_FP32 || d->precision == FQL_PRECISION_BF16_TC || d->precision == FQL_PRECISION_BF16_ENC,
              "precision=%d", d->precision);
  FQL_REQUIRE(d->precision != FQL_PRECISION_BF16_ENC || d->reserved[0] > 0, "FQL_PRECISION_BF16_ENC is a pixel-config mode (encoder='impala_small')");
  if (d->reserved[0] > 0) {  // pixel observations through ImpalaEncoder('impala_small')
    FQL_REQUIRE(d->reserved[1] > 0 && d->reserved[2] > 0 && d->reserved[2] <= 32, "image dims %dx%dx%d", d->reserved[0], d->reserved[1], d->reserved[2]);
    FQL_REQUIRE(d->obs_dim == 512, "pixel configs: obs_dim is the encoder output width and must be 512 (got %d)", d->obs_dim);
    FQL_REQUIRE(d->num_seeds == 1, "pixel configs are built for num_seeds == 1");
    // FQL_PRECISION_FP32: fp32 CUDA-core encoders and MLPs; FQL_PRECISION_BF16_ENC: tcgen05 encoders, fp32 MLPs;
    // FQL_PRECISION_BF16_TC: tcgen05 encoders and MLPs (the MLPs layer by layer: their first-layer input is 512 + A (+ 1) wide)
  }
  return 0;
}

int fql_build_layout(const FqlDims* d, Layout* L) {
  FQL_TRY(fql_validate_dims(d));
  memset(L, 0, sizeof(*L));
  const int F = d->obs_dim, A = d->action_dim, H = d->hidden, NL = d->num_hidden + 1;
  int64_t off = 0;
  int nl = 0;
  auto add_leaf = [&](int net, int64_t n) {
    int64_t o = off;
    L->leaf_blk[nl] = (int)(off / FQL_LEAF_PAD);
    L->leaf_net[nl] = net;
    nl++;
    off += round_up64(n, FQL_LEAF_PAD);
    return o;
  };
  // arena order: bc_flow | critic | onestep | target.  The first two networks' gradients are complete long before the one-step
  // actor's (which waits for the Euler target), so a data-parallel run all-reduces [0, onestep.begin) early; the target critic
  // (zero gradients) stays last.
  static const int kOrder[FQL_NUM_NETS] = {FQL_NET_ACTOR_BC_FLOW, FQL_NET_CRITIC, FQL_NET_ACTOR_ONESTEP_FLOW, FQL_NET_TARGET_CRITIC};
  for (int oi = 0; oi < FQL_NUM_NETS; oi++) {
    const int n = kOrder[oi];
    NetView& v = L->net[n];
    v.n_layers = NL;
    v.hidden = H;
    const bool critic = (n == FQL_NET_CRITIC || n == FQL_NET_TARGET_CRITIC);
    v.ens = critic ? 2 : 1;
    v.ln = critic ? d->critic_layer_norm : d->actor_layer_norm;
    v.in_dim = (n == FQL_NET_ACTOR_BC_FLOW) ? F + A + 1 : F + A;
    v.out_dim = critic ? 1 : A;
    v.begin = off;
    const int extra = v.ln ? 4 : 2;
    FQL_REQUIRE(nl + NL * extra + 20 <= FQL_MAX_LEAVES, "too many leaves");
    for (int l = 0; l < NL; l++) {
      const int64_t K = v.k_of(l), N = v.n_of(l);
      v.off_w[l] = add_leaf(n, v.ens * K * N);
      v.off_b[l] = add_leaf(n, v.ens * N);
      if (v.ln && l + 1 < NL) {
        v.off_lns[l] = add_leaf(n, v.ens * N);
        v.off_lnb[l] = add_leaf(n, v.ens * N);
      }
    }
    if (d->reserved[0] > 0) {  // encoder of this network (the bc-flow one is the separate `actor_bc_flow_encoder` module, fql.py:230-232)
      v.has_enc = 1;
      static const int stacks[3] = {16, 32, 32};
      int c = d->reserved[2], h = d->reserved[0], w = d->reserved[1];
      for (int i = 0; i < 3; i++) {
        const int f = stacks[i];
        const int cin[3] = {c, f, f};
        for (int j = 0; j < 3; j++) {
          v.enc.off_cw[i][j] = add_leaf(n, 9 * cin[j] * f);
          v.enc.off_cb[i][j] = add_leaf(n, f);
        }
        c = f; h = (h + 1) / 2; w = (w + 1) / 2;
      }
      v.enc.off_dw = add_leaf(n, (int64_t)h * w * c * d->obs_dim);  // MLP((512,)): the encoder output width is obs_dim
      v.enc.off_db = add_leaf(n, d->obs_dim);
    }
    v.end = off;
  }
  L->arena = off;
  L->n_leaves = nl;
  L->leaf_blk[nl] = (int)(off / FQL_LEAF_PAD);
  return 0;
}

StepShape make_shape(const FqlDims* d) {
  StepShape s;
  s.S = d->num_seeds; s.B = d->batch; s.GB = d->global_batch; s.F = d->obs_dim; s.A = d->action_dim;
  s.H = d->hidden; s.NH = d->num_hidden;
  s.q_agg_min = d->q_agg_min; s.normalize_q_loss = d->normalize_q_loss; s.flow_steps = d->flow_steps;
  return s;
}

// ---------------------------------------------------------------------------------------------------------
// workspace
// ---------------------------------------------------------------------------------------------------------
namespace {
struct Carver {
  char* base;
  size_t off = 0;
  float* take(int64_t nfloats) {
    off = (off + 255) & ~(size_t)255;
    float* p = base ? reinterpret_cast<float*>(base + off) : nullptr;
    off += (size_t)nfloats * sizeof(float);
    return p;
  }
};

void carve_pass(Carver& c, PassBuf* pb, int G, int Mcap, int H, int NH, int out_dim, bool ln, bool need_z, bool need_h = true) {
  pb->G = G;
  pb->Mcap = Mcap;
  for (int l = 0; l < NH; l++) {
    pb->Z[l] = (need_z || ln) ? c.take((int64_t)G * Mcap * H) : nullptr;
    pb->Hh[l] = need_h ? c.take((int64_t)G * Mcap * H) : nullptr;
    pb->mu[l] = ln ? c.take((int64_t)G * Mcap) : nullptr;
    pb->rstd[l] = ln ? c.take((int64_t)G * Mcap) : nullptr;
  }
  pb->out = c.take((int64_t)G * Mcap * out_dim);
}
}  // namespace

size_t carve_workspace(const FqlDims* d, const Layout& L, void* base, WsPtrs* w) {
  Carver c{reinterpret_cast<char*>(base)};
  const int64_t S = d->num_seeds, B = d->batch, F = d->obs_dim, A = d->action_dim, H = d->hidden;
  const int NH = d->num_hidden;
  memset(w, 0, sizeof(*w));
  w->XO = c.take(S * 3 * B * (F + A));
  w->XF = c.take(S * 2 * B * (F + A + 1));
  w->XC = c.take(3 * S * B * (F + A));
  w->vel = c.take(S * B * A);
  // fp32 post-activations: only the SIMT MLPs read them; the tensor-core step keeps bf16 copies (O_Hb, F_Hb, C_Hb below)
  const bool simt = d->precision != FQL_PRECISION_BF16_TC;
  carve_pass(c, &w->pO, (int)S, (int)(3 * B), (int)H, NH, (int)A, d->actor_layer_norm, true, simt);
  carve_pass(c, &w->pF, (int)S, (int)(2 * B), (int)H, NH, (int)A, d->actor_layer_norm, true, simt);
  carve_pass(c, &w->pC, (int)(3 * S * 2), (int)B, (int)H, NH, 1, d->critic_layer_norm, true, simt);
  w->O_out = w->pO.out;
  w->F_out = w->pF.out;
  w->C_out = w->pC.out;
  w->dq = c.take(S * 2 * B);
  w->dqs = c.take(S * 2 * B);
  w->dpred = c.take(S * B * A);
  w->dapi = c.take(S * B * A);
  w->target = c.take(S * B * A);
  w->dX0 = c.take(S * 2 * B * (F + A));
  w->raw_local = c.take(S * FQL_NUM_RAW);
  w->gstats = c.take(S * 4 + 4);  // + Adam bias corrections {1 - b1^t, 1 - b2^t} of the step in flight
  w->partials = c.take(S * (int64_t)L.leaf_blk[L.n_leaves] * 4);
  w->cpost_part = c.take(2 * S * 64 * 4);
  w->cpost_ticket = reinterpret_cast<int*>(c.take(3 * S + 4));
  if (d->reserved[0] > 0) {
    for (int i = 0; i < 5; i++) w->feat[i] = c.take(S * B * F);
    for (int i = 0; i < 3; i++) w->dfeat[i] = c.take(S * B * F);
    w->dX0F = c.take(S * B * (F + A + 1));
    w->dX0O = c.take(S * B * (F + A));
    w->dX0C = c.take(S * 2 * B * (F + A));
    const bool bwd[5] = {false, true, false, true, true};
    for (int i = 0; i < 5; i++) {
      c.off = (c.off + 255) & ~(size_t)255;
      c.off += enc_carve(d, B, base ? c.base + c.off : nullptr, &w->enc[i], bwd[i]);
    }
  }
  if (d->precision == FQL_PRECISION_BF16_TC) {
    const int64_t kO = round_up64(F + A, 64), kF = round_up64(F + A + 1, 64);
    w->XOb = c.take((S * 3 * B * kO + 1) / 2);
    w->XFb = c.take((S * 2 * B * kF + 1) / 2);
    w->XCb = c.take((3 * S * B * kO + 1) / 2);
    for (int l = 0; l < NH; l++) {
      w->O_Hb[l] = c.take(S * 3 * B * H / 2);
      w->O_Zb[l] = c.take(S * 3 * B * H / 2);
      w->F_Hb[l] = c.take(S * 2 * B * H / 2);
      w->F_Zb[l] = c.take(S * 2 * B * H / 2);
      w->C_Hb[l] = c.take(3 * S * 2 * B * H / 2);
      w->C_XHb[l] = c.take(3 * S * 2 * B * H / 2);
      w->C_DGb[l] = c.take(3 * S * 2 * B * H / 2);
    }
    for (int i = 0; i < NH; i++) {
      w->O_dZb[i] = c.take(S * B * H / 2);
      w->F_dZb[i] = c.take(S * B * H / 2);
      w->O_dZf[i] = c.take(S * B * H);
      w->F_dZf[i] = c.take(S * B * H);
    }
    w->O_dOutb = c.take(S * B * 64 / 2);
    w->F_dOutb = c.take(S * B * 64 / 2);
    for (int i = 0; i < NH; i++) {
      w->C1_dZb[i] = c.take(S * 2 * B * H / 2);
      w->C2_dZb[i] = c.take(S * 2 * B * H / 2);
      w->C1_dZf[i] = c.take(S * 2 * B * H);
      w->C1_dHf[i] = c.take(S * 2 * B * H);
      w->C2_dZf[i] = c.take(S * 2 * B * H);
      w->C2_dHf[i] = c.take(S * 2 * B * H);
    }
    w->C1_dOutb = c.take(S * 2 * B * 64 / 2);
    w->C2_dOutb = c.take(S * 2 * B * 64 / 2);
    w->euler_a = c.take(S * B * A);
    for (int i = 0; i < 3; i++) w->cs_scratch[i] = c.take(65536);
    w->euler_hx = c.take((int64_t)(tc_euler_scratch_elems(d, (int)B) / 2 + 4));
  }
  for (int i = 0; i < 2; i++) {
    w->dC[i] = c.take(S * 2 * B * H);
    w->dCp[i] = c.take(S * 2 * B * H);
    w->dF[i] = c.take(S * B * H);
    w->dO[i] = c.take(S * B * H);
  }
  return c.off + 256;
}

// ---------------------------------------------------------------------------------------------------------
// grouped MLP forward / backward in FQL_PRECISION_FP32
// ---------------------------------------------------------------------------------------------------------
namespace {

struct FwdSpec {
  int P;
  const NetView* nv[FQL_MAXP];
  const float* params;
  int64_t arena;
  int S, E, M, H;
  const float* X0;  // [P][S][Mcap0][K0]
  int Mcap0, r0_in;
  PassBuf* buf;
  int r0;
  int save_z;
};

int mlp_forward(const FwdSpec& f, cudaStream_t st) {
  const NetView& n0 = *f.nv[0];
  const int NL = n0.n_layers;
  const int64_t Mcap = f.buf->Mcap;
  for (int l = 0; l < NL; l++) {
    const int K = n0.k_of(l), N = n0.n_of(l);
    const bool last = (l == NL - 1);
    GemmArgs a;
    memset(&a, 0, sizeof(a));
    a.P = f.P; a.S = f.S; a.E = f.E; a.M = f.M; a.N = N; a.K = K;
    for (int p = 0; p < f.P; p++) {
      if (l == 0) a.A.base[p] = f.X0 + ((int64_t)p * f.S * f.Mcap0 + f.r0_in) * K;
      else a.A.base[p] = f.buf->Hh[l - 1] + ((int64_t)p * f.S * f.E * Mcap + f.r0) * f.H;
      a.B.base[p] = f.params + f.nv[p]->off_w[l];
      a.bias.base[p] = f.params + f.nv[p]->off_b[l];
    }
    if (l == 0) { a.A.stride_s = (int64_t)f.Mcap0 * K; a.A.stride_e = 0; a.lda = K; }
    else { a.A.stride_s = (int64_t)f.E * Mcap * f.H; a.A.stride_e = Mcap * f.H; a.lda = f.H; }
    a.B.stride_s = f.arena; a.B.stride_e = (int64_t)K * N; a.ldb = N;
    a.bias.stride_s = f.arena; a.bias.stride_e = N;
    a.out.stride_s = (int64_t)f.E * Mcap * N; a.out.stride_e = Mcap * N; a.ldo = N;
    a.out_pre.stride_s = a.out.stride_s; a.out_pre.stride_e = a.out.stride_e; a.ld_pre = N;
    for (int p = 0; p < f.P; p++) {
      const int64_t goff = ((int64_t)p * f.S * f.E * Mcap + f.r0) * N;
      if (last) a.out.base[p] = f.buf->out + goff;
      else if (n0.ln) a.out.base[p] = f.buf->Z[l] + goff;
      else {
        a.out.base[p] = f.buf->Hh[l] + goff;
        a.out_pre.base[p] = f.save_z ? f.buf->Z[l] + goff : nullptr;
      }
    }
    a.act_gelu = (!last && !n0.ln) ? 1 : 0;
    FQL_TRY(launch_gemm(a, st));
    if (!last && n0.ln) {
      ActLnArgs r;
      memset(&r, 0, sizeof(r));
      r.P = f.P; r.S = f.S; r.E = f.E; r.M = f.M; r.N = N; r.ld = N; r.ln = 1;
      for (int p = 0; p < f.P; p++) {
        const int64_t goff = ((int64_t)p * f.S * f.E * Mcap + f.r0);
        r.Z.base[p] = f.buf->Z[l] + goff * N;
        r.H.base[p] = f.buf->Hh[l] + goff * N;
        r.mu.base[p] = f.buf->mu[l] + goff;
        r.rstd.base[p] = f.buf->rstd[l] + goff;
        r.scale.base[p] = f.params + f.nv[p]->off_lns[l];
        r.lnbias.base[p] = f.params + f.nv[p]->off_lnb[l];
      }
      r.Z.stride_s = (int64_t)f.E * Mcap * N; r.Z.stride_e = Mcap * N;
      r.H.stride_s = r.Z.stride_s; r.H.stride_e = r.Z.stride_e;
      r.mu.stride_s = (int64_t)f.E * Mcap; r.mu.stride_e = Mcap;
      r.rstd.stride_s = r.mu.stride_s; r.rstd.stride_e = r.mu.stride_e;
      r.scale.stride_s = f.arena; r.scale.stride_e = N;
      r.lnbias.stride_s = f.arena; r.lnbias.stride_e = N;
      FQL_TRY(launch_act_ln_fwd(r, st));
    }
  }
  return 0;
}

struct BwdSpec {
  const NetView* nv;
  const float* params;
  float* grads;  // NULL: no parameter gradients (dgrad-only pass)
  int64_t arena;
  int S, E, M, H;
  const float* X0;  // already offset to (problem, first row); [S][Mcap0][K0]
  int Mcap0;
  const PassBuf* buf;
  int p, r0;        // problem index / first row inside buf
  const float* dOut;  // [S][E][M][out_dim]
  float* dpp[2];      // [S][E][M][H]
  float* dX0;         // optional [S][E][M][K0]
};

int mlp_backward(const BwdSpec& b, cudaStream_t st) {
  const NetView& n = *b.nv;
  const int NL = n.n_layers;
  const int64_t Mcap = b.buf->Mcap;
  const int64_t goff_rows = ((int64_t)b.p * b.S * b.E * Mcap + b.r0);  // row offset of this problem inside buf
  const float* dZ = b.dOut;
  int ldz = n.out_dim;
  int cur = 0;
  for (int l = NL - 1; l >= 0; l--) {
    const int K = n.k_of(l), N = n.n_of(l);
    const int64_t dz_ss = (int64_t)b.E * b.M * ldz, dz_se = (int64_t)b.M * ldz;
    if (b.grads) {
      GemmArgs a;  // dW[K,N] = A_l^T[K,M] * dZ[M,N]
      memset(&a, 0, sizeof(a));
      a.P = 1; a.S = b.S; a.E = b.E; a.M = K; a.N = N; a.K = b.M;
      a.trans_a = 1;
      if (l == 0) { a.A.base[0] = b.X0; a.A.stride_s = (int64_t)b.Mcap0 * K; a.A.stride_e = 0; a.lda = K; }
      else { a.A.base[0] = b.buf->Hh[l - 1] + goff_rows * b.H; a.A.stride_s = (int64_t)b.E * Mcap * b.H; a.A.stride_e = Mcap * b.H; a.lda = b.H; }
      a.B.base[0] = dZ; a.B.stride_s = dz_ss; a.B.stride_e = dz_se; a.ldb = ldz;
      a.out.base[0] = b.grads + n.off_w[l]; a.out.stride_s = b.arena; a.out.stride_e = (int64_t)K * N; a.ldo = N;
      FQL_TRY(launch_gemm(a, st));
      ColSumArgs c;  // db[N] = sum_rows dZ
      memset(&c, 0, sizeof(c));
      c.P = 1; c.S = b.S; c.E = b.E; c.M = b.M; c.N = N; c.ld = ldz;
      c.X.base[0] = dZ; c.X.stride_s = dz_ss; c.X.stride_e = dz_se;
      c.out.base[0] = b.grads + n.off_b[l]; c.out.stride_s = b.arena; c.out.stride_e = N;
      FQL_TRY(launch_colsum(c, st));
    }
    if (l == 0 && !b.dX0) break;
    GemmArgs a;  // dH_{l-1}[M,K] = dZ[M,N] * W_l^T
    memset(&a, 0, sizeof(a));
    a.P = 1; a.S = b.S; a.E = b.E; a.M = b.M; a.N = K; a.K = N;
    a.A.base[0] = dZ; a.A.stride_s = dz_ss; a.A.stride_e = dz_se; a.lda = ldz;
    a.trans_b = 1;
    a.B.base[0] = b.params + n.off_w[l]; a.B.stride_s = b.arena; a.B.stride_e = (int64_t)K * N; a.ldb = N;
    if (l == 0) {
      a.out.base[0] = b.dX0; a.out.stride_s = (int64_t)b.E * b.M * K; a.out.stride_e = (int64_t)b.M * K; a.ldo = K;
      FQL_TRY(launch_gemm(a, st));
      break;
    }
    float* dst = b.dpp[cur];
    a.out.base[0] = dst; a.out.stride_s = (int64_t)b.E * b.M * b.H; a.out.stride_e = (int64_t)b.M * b.H; a.ldo = b.H;
    const float* Zprev = b.buf->Z[l - 1] + goff_rows * b.H;
    const int64_t z_ss = (int64_t)b.E * Mcap * b.H, z_se = Mcap * b.H;
    if (!n.ln) {  // dZ_{l-1} = dH_{l-1} * gelu'(Z_{l-1}) fused into the dgrad epilogue
      a.mulz.base[0] = Zprev; a.mulz.stride_s = z_ss; a.mulz.stride_e = z_se; a.ld_mulz = b.H;
      FQL_TRY(launch_gemm(a, st));
    } else {
      FQL_TRY(launch_gemm(a, st));
      if (b.grads) {
        ColSumArgs c;
        memset(&c, 0, sizeof(c));
        c.P = 1; c.S = b.S; c.E = b.E; c.M = b.M; c.N = b.H; c.ld = b.H;
        c.X.base[0] = dst; c.X.stride_s = a.out.stride_s; c.X.stride_e = a.out.stride_e;
        c.out.base[0] = b.grads + n.off_lnb[l - 1]; c.out.stride_s = b.arena; c.out.stride_e = b.H;
        FQL_TRY(launch_colsum(c, st));
        // NB: colsum addresses Z/mu/rstd rows with X's row index, so they must share X's row pitch: Z rows of this
        // problem are contiguous per (s,e) with pitch H, same as dst.
        c.Z.base[0] = Zprev; c.Z.stride_s = z_ss; c.Z.stride_e = z_se;
        c.mu.base[0] = b.buf->mu[l - 1] + goff_rows; c.mu.stride_s = (int64_t)b.E * Mcap; c.mu.stride_e = Mcap;
        c.rstd.base[0] = b.buf->rstd[l - 1] + goff_rows; c.rstd.stride_s = c.mu.stride_s; c.rstd.stride_e = c.mu.stride_e;
        c.out.base[0] = b.grads + n.off_lns[l - 1];
        FQL_TRY(launch_colsum(c, st));
      }
      ActLnBwdArgs r;
      memset(&r, 0, sizeof(r));
      r.P = 1; r.S = b.S; r.E = b.E; r.M = b.M; r.N = b.H; r.ld = b.H;
      r.dH.base[0] = dst; r.dH.stride_s = a.out.stride_s; r.dH.stride_e = a.out.stride_e;
      r.dZ.base[0] = dst; r.dZ.stride_s = a.out.stride_s; r.dZ.stride_e = a.out.stride_e;
      r.Z.base[0] = Zprev; r.Z.stride_s = z_ss; r.Z.stride_e = z_se;
      r.scale.base[0] = b.params + n.off_lns[l - 1]; r.scale.stride_s = b.arena; r.scale.stride_e = b.H;
      FQL_TRY(launch_act_ln_bwd(r, st));
    }
    dZ = dst;
    ldz = b.H;
    cur ^= 1;
  }
  return 0;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// context: internal streams / events / cached graphs
// ---------------------------------------------------------------------------------------------------------
struct GraphEntry {
  std::vector<unsigned char> key;
  cudaGraphExec_t exec;
  long long kernels;  // kernel nodes in the captured graph
};
struct FqlContext {
  cudaStream_t sc = nullptr;  // data-parallel exchange (dp_comm.cu): bucket reductions overlap the rest of the backward
  DpState dp;                 // attached peer-memory communicator (fql_dp_attach)
  cudaStream_t s0 = nullptr, s1 = nullptr, s2 = nullptr, s3 = nullptr, s4 = nullptr, s5 = nullptr, s6 = nullptr, s7 = nullptr, s8 = nullptr, s9 = nullptr;  // s0 stands in for the caller's stream when that is the legacy default
  cudaEvent_t ev[64] = {};
  std::vector<GraphEntry> graphs;
  int use_graph = 1;
  int use_euler_cluster = 1;
  int use_cluster_fwd = 1;   // FQL_B200_CLUSTER_FWD=0: one-step actor forward layer by layer
  int use_cluster_bwd = 1;   // FQL_B200_CLUSTER_BWD=0: one-step actor dgrad chain layer by layer
  unsigned long long* stamps = nullptr;  // FQL_B200_STAMPS=1: %globaltimer at schedule points (diagnostics, profiles/dbg_timeline.py)
  int adam_done_blk = 0;     // blocks [0, adam_done_blk) were already applied by enqueue_grads_tc in this enqueue
  int euler_hoist = 1;       // FQL_B200_EULER_HOIST=0: pixel configs, Euler integration layer by layer instead of hoisted first layer + cluster kernel
  int enc_streams = 1;       // FQL_B200_ENC_STREAMS=0: pixel configs, the five tensor-core encoder forwards on one stream
  int dp_early_adam = 1;     // FQL_B200_DP_EARLY_ADAM=0: data parallel, one optimizer pass at the end.  Default: the bc-flow + critic part
                             // runs behind their bucket reductions, under the one-step actor's bucket exchange
  int dp_bc_late = 0;        // FQL_B200_DP_BC_LATE=1: bc-flow's bucket is exchanged together with the critic's (one launch) instead of
                             // under the Euler chain
  int use_big_bwd = 1;       // FQL_B200_BIG_BWD=0: per-layer backward (tc_gemm + row kernels) also at large batch
  int chain_min_tiles = 48;  // row tiles (x seeds) from which the fused per-tile chain kernels (hidden 512) replace the per-layer GEMMs
  cudaEvent_t early_event = nullptr;  // optional: recorded when the bc-flow and critic gradients of fql_step_grads are complete
  long long launches = 0;  // kernels enqueued through this context
};

extern "C" long long fql_launch_count(FqlContext* c) { return c ? c->launches : -1; }
extern "C" int fql_set_early_grads_event(FqlContext* c, void* event) {
  FQL_REQUIRE(c != nullptr, "context is NULL");
  c->early_event = reinterpret_cast<cudaEvent_t>(event);
  for (auto& g : c->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  c->graphs.clear();  // the event is baked into captured graphs
  return 0;
}
extern "C" int64_t fql_early_grads_floats(const FqlDims* d) {
  Layout L;
  if (fql_build_layout(d, &L)) return -1;
  return L.net[FQL_NET_ACTOR_ONESTEP_FLOW].begin;
}
extern "C" int fql_dp_allreduce(FqlContext* c, int32_t bucket, int64_t off, int64_t n, void* stream) {
  FQL_REQUIRE(c && c->dp.active, "fql_dp_allreduce: no communicator attached (fql_dp_attach)");
  const long long before = g_fql_launches;
  const int rc = dp_allreduce_range(c->dp, bucket, off, n, reinterpret_cast<cudaStream_t>(stream));
  c->launches += g_fql_launches - before;
  return rc;
}
extern "C" int fql_dp_attach(FqlContext* c, const FqlDims* d, const FqlDpComm* comm) {
  FQL_REQUIRE(c != nullptr, "context is NULL");
  for (auto& g : c->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  c->graphs.clear();  // the communicator's pointers are baked into captured graphs
  c->dp = DpState();
  if (!comm) return 0;
  Layout L;
  FQL_TRY(fql_build_layout(d, &L));
  FQL_REQUIRE(comm->world >= 2 && comm->world <= FQL_DP_MAX_RANKS && comm->rank >= 0 && comm->rank < comm->world, "fql_dp_attach: rank %d of %d",
              comm->rank, comm->world);
  for (int r = 0; r < comm->world; r++) FQL_REQUIRE(comm->base[r] != nullptr && ((uintptr_t)comm->base[r] & 15) == 0, "fql_dp_attach: base[%d] is NULL / unaligned", r);
  c->dp.comm = *comm;
  c->dp.S = d->num_seeds;
  c->dp.arena = L.arena;
  c->dp.lay = dp_layout(d->num_seeds, L.arena);
  c->dp.active = 1;
  return 0;
}

__global__ void stamp_kernel(unsigned long long* slot) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  *slot = t;
}
static int stamp(FqlContext* ctx, int idx, cudaStream_t st) {
  if (!ctx->stamps) return 0;
  stamp_kernel<<<1, 1, 0, st>>>(ctx->stamps + idx);
  FQL_CHECK_LAUNCH();
  return 0;
}
extern "C" int fql_debug_stamps(FqlContext* c, unsigned long long* host_out, int n) {
  FQL_REQUIRE(c && c->stamps && n <= 576, "stamps are off (FQL_B200_STAMPS=1)");
  FQL_CHECK_CUDA(cudaMemcpy(host_out, c->stamps, n * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return 0;
}
static int record_early(FqlContext* ctx, cudaStream_t st) {
  if (!ctx->early_event) return 0;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  FQL_CHECK_CUDA(cudaStreamIsCapturing(st, &cap));
  FQL_CHECK_CUDA(cudaEventRecordWithFlags(ctx->early_event, st, cap == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault));
  return 0;
}

extern "C" int fql_context_create(FqlContext** out) {
  FQL_REQUIRE(out != nullptr, "out is NULL");
  FqlContext* c = new FqlContext();
  // the dependent chains that bound a small-batch step (S0: one-step actor / critic / tail, s1: Euler) get the highest
  // priority so that their CTAs are placed before those of the bulk side work (weight gradients, early optimizer pass)
  int prio_lo = 0, prio_hi = 0;
  FQL_CHECK_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  const char* pr = getenv("FQL_B200_PRIO");
  if (pr && pr[0] == '0') prio_hi = prio_lo;
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->s0, cudaStreamNonBlocking, prio_hi));
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->s1, cudaStreamNonBlocking, prio_hi));
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->s2, cudaStreamNonBlocking, prio_lo));
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->s3, cudaStreamNonBlocking, prio_lo));
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->s4, cudaStreamNonBlocking, prio_lo));
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->s5, cudaStreamNonBlocking, prio_lo));
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->s6, cudaStreamNonBlocking, prio_lo));
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->s7, cudaStreamNonBlocking, prio_lo));
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->s8, cudaStreamNonBlocking, prio_lo));
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->s9, cudaStreamNonBlocking, prio_lo));
  FQL_CHECK_CUDA(cudaStreamCreateWithPriority(&c->sc, cudaStreamNonBlocking, prio_hi));
  for (auto& e : c->ev) FQL_CHECK_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  const char* g = getenv("FQL_B200_GRAPH");
  if (g && g[0] == '0') c->use_graph = 0;
  const char* ec = getenv("FQL_B200_EULER_CLUSTER");
  if (ec && ec[0] == '0') c->use_euler_cluster = 0;
  const char* cbw = getenv("FQL_B200_CLUSTER_BWD");
  if (cbw && cbw[0] == '0') c->use_cluster_bwd = 0;
  const char* cfw = getenv("FQL_B200_CLUSTER_FWD");
  if (cfw && cfw[0] == '0') c->use_cluster_fwd = 0;
  const char* stp = getenv("FQL_B200_STAMPS");
  if (stp && stp[0] == '1') {
    FQL_CHECK_CUDA(cudaMalloc(&c->stamps, 576 * sizeof(unsigned long long)));  // 64 schedule points + [32 CTAs][16] Euler phases
    FQL_CHECK_CUDA(cudaMemset(c->stamps, 0, 576 * sizeof(unsigned long long)));
  }
  const char* ehs = getenv("FQL_B200_EULER_HOIST");
  if (ehs) c->euler_hoist = atoi(ehs);
  const char* ens = getenv("FQL_B200_ENC_STREAMS");
  if (ens) c->enc_streams = atoi(ens);
  const char* dea = getenv("FQL_B200_DP_EARLY_ADAM");
  if (dea) c->dp_early_adam = atoi(dea);
  const char* dbl = getenv("FQL_B200_DP_BC_LATE");
  if (dbl) c->dp_bc_late = atoi(dbl);
  const char* cm = getenv("FQL_B200_CHAIN_MIN_TILES");
  if (cm) c->chain_min_tiles = atoi(cm);
  const char* bb = getenv("FQL_B200_BIG_BWD");
  if (bb && bb[0] == '0') c->use_big_bwd = 0;
  *out = c;
  return 0;
}

extern "C" int fql_context_destroy(FqlContext* c) {
  if (!c) return 0;
  for (auto& g : c->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  for (auto& e : c->ev) if (e) cudaEventDestroy(e);
  if (c->s0) cudaStreamDestroy(c->s0);
  if (c->s1) cudaStreamDestroy(c->s1);
  if (c->s2) cudaStreamDestroy(c->s2);
  if (c->s3) cudaStreamDestroy(c->s3);
  if (c->s4) cudaStreamDestroy(c->s4);
  if (c->s5) cudaStreamDestroy(c->s5);
  if (c->s6) cudaStreamDestroy(c->s6);
  if (c->s7) cudaStreamDestroy(c->s7);
  if (c->s8) cudaStreamDestroy(c->s8);
  if (c->s9) cudaStreamDestroy(c->s9);
  if (c->sc) cudaStreamDestroy(c->sc);
  if (c->stamps) cudaFree(c->stamps);
  delete c;
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// the step
// ---------------------------------------------------------------------------------------------------------
namespace {

struct StepCall {
  const FqlDims* d;
  const FqlHparams* hp;
  const FqlBatch* b;
  const FqlState* st;
  float* raw;
  float* info;
  void* ws;
  size_t ws_bytes;
  int do_grads, do_backward, do_apply;
  int raw_ranks;  // fql_step_apply: `raw` holds the all-gathered accumulators of this many ranks [ranks][S][FQL_NUM_RAW]
};

int check_common(const FqlDims* d, const void* ws, size_t ws_bytes, Layout* L, WsPtrs* w) {
  FQL_TRY(fql_build_layout(d, L));
  const size_t need = carve_workspace(d, *L, nullptr, w);
  FQL_REQUIRE(ws != nullptr && ws_bytes >= need, "workspace too small: have %zu need %zu", ws_bytes, need);
  FQL_REQUIRE(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  carve_workspace(d, *L, const_cast<void*>(ws), w);
  return 0;
}

// What every call site reads as "observations": the batch itself (state configs) or the output of that network's encoder.
// Five unique encoder forwards per step (SURVEY 8d): onestep(next_obs), onestep(obs), target critic(next_obs), critic(obs), bc flow(obs).
int encode_observations(const StepCall& c, const Layout& L, WsPtrs& w, cudaStream_t st, FqlContext* ctx = nullptr) {
  const FqlBatch& b = *c.b;
  if (c.d->reserved[0] == 0) {
    w.src[0] = w.src[2] = b.next_observations;
    w.src[1] = w.src[3] = w.src[4] = b.observations;
    return 0;
  }
  const uint8_t* obs = reinterpret_cast<const uint8_t*>(b.observations);
  const uint8_t* nobs = reinterpret_cast<const uint8_t*>(b.next_observations);
  const float* P = c.st->params;
  const int64_t B = c.d->batch;
  // tensor-core encoders: the five independent forwards on three streams (a pass is ~30 short launches, many of them smaller than
  // the GPU: the tails and the small layers of one pass fill the gaps of another)
  cudaStream_t sa = st, sb = st;
  const bool fork = ctx && c.d->precision != FQL_PRECISION_FP32 && ctx->enc_streams;
  if (fork) {
    sa = ctx->s5; sb = ctx->s6;
    FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[60], st));
    FQL_CHECK_CUDA(cudaStreamWaitEvent(sa, ctx->ev[60], 0));
    FQL_CHECK_CUDA(cudaStreamWaitEvent(sb, ctx->ev[60], 0));
  }
  FQL_TRY(enc_forward(c.d, L.net[FQL_NET_ACTOR_ONESTEP_FLOW].enc, P, nobs, B, w.enc[0], w.feat[0], st));
  FQL_TRY(enc_forward(c.d, L.net[FQL_NET_TARGET_CRITIC].enc, P, nobs, B, w.enc[2], w.feat[2], sa));
  FQL_TRY(enc_forward(c.d, L.net[FQL_NET_ACTOR_BC_FLOW].enc, P, obs, B, w.enc[4], w.feat[4], sb));
  FQL_TRY(enc_forward(c.d, L.net[FQL_NET_ACTOR_ONESTEP_FLOW].enc, P, obs, B, w.enc[1], w.feat[1], st));
  FQL_TRY(enc_forward(c.d, L.net[FQL_NET_CRITIC].enc, P, obs, B, w.enc[3], w.feat[3], sa));
  if (fork) {
    FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[61], sa));
    FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[62], sb));
    FQL_CHECK_CUDA(cudaStreamWaitEvent(st, ctx->ev[61], 0));
    FQL_CHECK_CUDA(cudaStreamWaitEvent(st, ctx->ev[62], 0));
  }
  for (int i = 0; i < 5; i++) w.src[i] = w.feat[i];
  return 0;
}

// Encoder backward of one trainable network from its MLP's first-layer input gradient dX0 [E][B][K0] (feature columns first).
int encoder_grads(const StepCall& c, const Layout& L, const WsPtrs& w, int net, const float* dX0, int E, int K0, float* dfeat, int enc_idx,
                  cudaStream_t st) {
  const int64_t B = c.d->batch;
  FQL_TRY(launch_extract_feat_grad(dX0, dfeat, E, B, K0, c.d->obs_dim, st));
  return enc_backward(c.d, L.net[net].enc, c.st->params, c.st->grads, reinterpret_cast<const uint8_t*>(c.b->observations), B, w.enc[enc_idx],
                      dfeat, st);
}

// ---------------------------------------------------------------------------------------------------------
// FQL_PRECISION_BF16_TC schedule of the loss/gradient half of the step: every contraction on tcgen05.
//   S1: Euler integration, layer by layer (each layer = 16 CTAs of tc_gemm at B=256)              <- longest chain
//   S2: bc-flow forward on the BC rows, BC loss, bc-flow backward; then the critic backward
//   S0: one-step actor forward, grouped critic forward (tc_gemm + LayerNorm row kernel per layer; at large batch one fused
//       chain launch, LayerNorm in the epilogue), TD/Q post, critic input gradient, [join Euler] distillation, one-step actor backward
// ---------------------------------------------------------------------------------------------------------
int enqueue_grads_tc(FqlContext* ctx, const StepCall& c, const Layout& L, WsPtrs& w, const StepShape& sh, const FqlHparams& hp,
                     float* raw, cudaStream_t S0) {
  const FqlBatch& b = *c.b;
  const FqlDims* d = c.d;
  const int S = sh.S, B = sh.B, H = sh.H, NH = sh.NH;
  const float* P = c.st->params;
  const void* shadow = c.st->shadow;
  typedef __nv_bfloat16 bf16;
  cudaStream_t S1 = ctx->s1, S2 = ctx->s2;
  cudaEvent_t ev_prep = ctx->ev[0], ev_f0 = ctx->ev[1], ev_cpost = ctx->ev[2], ev_euler = ctx->ev[3], ev_s2 = ctx->ev[4], ev_pad = ctx->ev[5];
  const int kO = (int)round_up64(sh.F + sh.A, 64), kF = (int)round_up64(sh.F + sh.A + 1, 64);
  const bool dp_grads = ctx->dp.active && c.do_backward;   // data parallel: per-network bucket reductions on ctx->sc
  // pixel configs (512 encoder features in front of the action columns): every MLP layer by layer through tc_gemm, and the
  // first-layer input gradients of the three trainable networks feed their encoders' backward
  const bool wide = tc_wide_input(d), pix = d->reserved[0] > 0;
  // data parallel: state configs exchange per-network buckets as soon as each is final; pixel configs (encoder gradients finish on other
  // streams) exchange the whole trainable prefix of the arena once, behind the complete backward
  const bool dp_bucketed = dp_grads && !pix;
  bool bc_enc_forked = false;
  FQL_TRY(stamp(ctx, 0, S0));   // step start
  FQL_TRY(launch_zero_bc(raw, (int64_t)S * FQL_NUM_RAW, c.do_apply ? c.st->count : nullptr, hp, w.gstats + S * 4, S0, w.cpost_ticket, 3 * S));
  FQL_TRY(encode_observations(c, L, w, S0, ctx));
  FQL_TRY(launch_prep(sh, b, w, S0));
  FQL_TRY(stamp(ctx, 1, S0));   // prep done
  FQL_CHECK_CUDA(cudaEventRecord(ev_prep, S0));
  FQL_CHECK_CUDA(cudaStreamWaitEvent(S1, ev_prep, 0));

  auto actor = [&](int net, const void* X0b, int K0pad, int rows_cap, int r0, int M, void* const* Hb, void* const* Zb, bool with_z) {
    TcActor t;
    memset(&t, 0, sizeof(t));
    t.d = d; t.L = &L; t.net = net; t.params = P; t.shadow = shadow; t.grads = c.st->grads; t.M = M;
    t.X0b = reinterpret_cast<const bf16*>(X0b) + (int64_t)r0 * K0pad; t.K0pad = K0pad; t.x_ss = (long long)rows_cap * K0pad;
    for (int l = 0; l < NH; l++) {
      t.Hb[l] = reinterpret_cast<bf16*>(Hb[l]) + (int64_t)r0 * H;
      t.Zb[l] = with_z ? reinterpret_cast<bf16*>(Zb[l]) + (int64_t)r0 * H : nullptr;
    }
    t.h_ss = (long long)rows_cap * H;
    t.cs_scratch = (net == FQL_NET_ACTOR_BC_FLOW) ? w.cs_scratch[0] : w.cs_scratch[1];
    return t;
  };

  // ---- S1: Euler (agents/fql.py:155-171) on rows [B, 2B) of the bc-flow buffers
  FQL_TRY(tc_pad_bf16(w.XF, w.XFb, (int64_t)S * 2 * B, sh.F + sh.A + 1, kF, S1));
  FQL_CHECK_CUDA(cudaEventRecord(ev_pad, S1));
  const int row_tiles = S * ((B + 127) / 128);
  // enough 128-row tiles to fill the GPU: fused per-tile chain kernels (chain2_tc.cu, hidden 512 only; narrower MLPs run layer by
  // layer at every batch size)
  const bool many_tiles = H == 512 && row_tiles >= ctx->chain_min_tiles && !wide;
  // ... and the whole backward as chain launches on bf16 gelu' / xhat saves (chain2_tc.cu, tc_path.cu "large-batch backward")
  const bool big_bwd = many_tiles && ctx->use_big_bwd && d->critic_layer_norm && d->reserved[0] == 0;
  auto chain = [&](int net, const void* X0b, int rows_cap, int r0_in, int M, void* const* Hb, void* const* Zb, float* out, int n_steps,
                   cudaStream_t st) {
    TcChainSpec t;
    memset(&t, 0, sizeof(t));
    t.d = d; t.L = &L; t.P = 1; t.net[0] = net; t.params = P; t.shadow = shadow; t.M = M; t.X0b = X0b; t.Mcap0 = rows_cap; t.r0_in = r0_in;
    t.r0 = r0_in; t.Hb = Hb; t.Zb = Zb; t.Mcap_override = rows_cap; t.out_override = out; t.n_steps = n_steps;
    if (big_bwd && Zb) { t.DGb = Zb; t.Zb = nullptr; }   // the pre-activation buffers hold gelu'(z) on this path
    if (n_steps > 1) { t.a0 = b.z; t.target = w.target; }
    return tc_mlp_chain2(t, st);
  };
  if (many_tiles) {
    FQL_TRY(chain(FQL_NET_ACTOR_BC_FLOW, w.XFb, 2 * B, B, B, nullptr, nullptr, nullptr, sh.flow_steps, S1));
  } else if (H == 512 && ctx->use_euler_cluster && wide && S == 1 && ctx->euler_hoist) {
    // pixel configs: the observation features are constant over the flow steps (agents/fql.py:162-169), so their part of the first
    // layer, c0 = features @ W0[:F] + b0, is one GEMM in front of the loop and the cluster kernel integrates with the first layer
    // reduced to [action | t] @ W0[F:] + c0[row]  (10 x 5 layer-by-layer GEMM launches -> one GEMM + one persistent launch)
    const NetView& nb = L.net[FQL_NET_ACTOR_BC_FLOW];
    const bf16* sh16 = reinterpret_cast<const bf16*>(shadow);
    float* c0 = w.dF[0];                                   // fp32 scratch of the SIMT schedule, free in this one
    TcGemmSpec g;
    memset(&g, 0, sizeof(g));
    g.M = B; g.N = H; g.K = sh.F; g.G0 = 1; g.G1 = 1; g.a_mn = 0; g.b_mn = 1;
    g.A.ptr = reinterpret_cast<const bf16*>(w.XFb) + (int64_t)B * kF; g.A.inner = sh.F; g.A.rows = B; g.A.ld = kF; g.A.g0 = 1; g.A.g1 = 1;
    g.B.ptr = sh16 + nb.off_w[0]; g.B.inner = H; g.B.rows = sh.F; g.B.ld = H; g.B.g0 = 1; g.B.g1 = 1;
    g.mode = TC_MODE_STORE_F32;
    g.bias.base = const_cast<float*>(P + nb.off_b[0]);
    g.out_f.base = c0; g.out_f.ld = H;
    FQL_TRY(tc_gemm(g, S1));
    float* xa = w.dF[1];                                   // [B][A + 1] = (noise | t = 0)
    void* xab = w.dO[0];                                   // bf16 [B][64]
    FQL_TRY(launch_concat(b.z, sh.A, b.z, 0, 0.f, 1, xa, B, S1));
    FQL_TRY(tc_pad_bf16(xa, xab, B, sh.A + 1, 64, S1));
    TcEulerSpec e;
    memset(&e, 0, sizeof(e));
    e.d = d; e.L = &L; e.params = P; e.shadow = shadow; e.X0b = xab; e.Mcap0 = B; e.r0_in = 0; e.M = B;
    e.a0 = b.z; e.c0 = c0; e.target = w.target; e.scratch = w.euler_hx;
    FQL_TRY(tc_euler_cluster(e, S1));
  } else if (H == 512 && ctx->use_euler_cluster && !wide) {
    TcEulerSpec e;
    memset(&e, 0, sizeof(e));
    e.d = d; e.L = &L; e.params = P; e.shadow = shadow; e.X0b = w.XFb; e.Mcap0 = 2 * B; e.r0_in = B; e.M = B;
    e.a0 = b.z; e.target = w.target; e.scratch = w.euler_hx;
    e.t_start = ctx->stamps ? ctx->stamps + 13 : nullptr;
    e.dbg = (ctx->stamps && S * ((B + 127) / 128) <= 2) ? ctx->stamps + 64 : nullptr;
    FQL_TRY(tc_euler_cluster(e, S1));
  } else {
    TcActor e = actor(FQL_NET_ACTOR_BC_FLOW, w.XFb, kF, 2 * B, B, B, w.F_Hb, w.F_Zb, false);
    for (int i = 0; i < sh.flow_steps; i++) {
      TcEuler eu{w.euler_a, w.target, i, sh.flow_steps};
      FQL_TRY(tc_actor_forward(e, nullptr, 0, 0, &eu, S1));
    }
  }
  FQL_TRY(stamp(ctx, 2, S1));   // Euler done
  FQL_CHECK_CUDA(cudaEventRecord(ev_euler, S1));
  if (getenv("FQL_B200_EULER_ALONE")) {  // diagnostics: serialise everything else behind the Euler chain
    const int m = atoi(getenv("FQL_B200_EULER_ALONE"));
    if (m & 1) FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ev_euler, 0));
    if (m & 2) FQL_CHECK_CUDA(cudaStreamWaitEvent(S2, ev_euler, 0));
  }

  // ---- S2: bc-flow on the BC rows [0, B), BC loss, backward
  FQL_CHECK_CUDA(cudaStreamWaitEvent(S2, ev_pad, 0));
  TcActor fbc = actor(FQL_NET_ACTOR_BC_FLOW, w.XFb, kF, 2 * B, 0, B, w.F_Hb, w.F_Zb, true);
  if (many_tiles) FQL_TRY(chain(FQL_NET_ACTOR_BC_FLOW, w.XFb, 2 * B, 0, B, w.F_Hb, w.F_Zb, w.F_out, 1, S2));
  else FQL_TRY(tc_actor_forward(fbc, w.F_out, (long long)2 * B * sh.A, 0, nullptr, S2));
  FQL_TRY(launch_bc_post(sh, w, raw, S2));
  if (c.do_backward && big_bwd) {
    FQL_TRY(tc_actor_backward_big(fbc, w.dpred, w.F_dOutb, w.F_dZb, false, S2));
    FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[16], S2));
    if (dp_bucketed && !ctx->dp_bc_late) {
      const NetView& nb = L.net[FQL_NET_ACTOR_BC_FLOW];
      FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->sc, ctx->ev[16], 0));
      FQL_TRY(dp_reduce_bucket(ctx->dp, 0, nb.begin, nb.end - nb.begin, nullptr, ctx->sc));
    }
    FQL_TRY(stamp(ctx, 4, S2));
  } else if (c.do_backward) {
    FQL_TRY(tc_actor_backward(fbc, w.dpred, w.F_dOutb, w.F_dZb, w.F_dZf, S2, ctx->s3, ctx->s7, &ctx->ev[8]));
    if (pix) {  // d(BC loss)/d(features) -> actor_bc_flow_encoder (agents/fql.py:58, 230-232), on its own stream: S2 goes on to the
                // critic's backward (the three encoder backwards are ~30 short launches each and overlap each other's gaps)
      FQL_TRY(tc_actor_input_grad(fbc, w.F_dZb[0], w.dX0F, S2));
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[63], S2));
      FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->sc, ctx->ev[63], 0));   // (the communication stream: idle in pixel configs)
      FQL_TRY(encoder_grads(c, L, w, FQL_NET_ACTOR_BC_FLOW, w.dX0F, 1, sh.F + sh.A + 1, w.dfeat[1], 4, ctx->sc));
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[37], ctx->sc));
      bc_enc_forked = true;
    }
    FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[53], ctx->s7));
    FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->s3, ctx->ev[53], 0));
    FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[16], ctx->s3));
    if (dp_bucketed && !ctx->dp_bc_late) {  // bc-flow's gradients are final long before the rest: its bucket crosses NVLink under the remaining backward
      const NetView& nb = L.net[FQL_NET_ACTOR_BC_FLOW];
      FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->sc, ctx->ev[16], 0));
      FQL_TRY(stamp(ctx, 20, ctx->sc));   // bc-flow bucket: gradients final
      FQL_TRY(dp_reduce_bucket(ctx->dp, 0, nb.begin, nb.end - nb.begin, nullptr, ctx->sc));
      FQL_TRY(stamp(ctx, 21, ctx->sc));   // bc-flow bucket reduced
    }
    FQL_TRY(stamp(ctx, 4, S2));   // bc-flow dgrad chain done (weight gradients on s3 may still run)
  }
  (void)ev_f0;

  // ---- S0: one-step actor on {(s',z_next), (s,z), (s,z')}, grouped critic pass
  FQL_TRY(tc_pad_bf16(w.XO, w.XOb, (int64_t)S * 3 * B, sh.F + sh.A, kO, S0));
  TcActor fo = actor(FQL_NET_ACTOR_ONESTEP_FLOW, w.XOb, kO, 3 * B, 0, 3 * B, w.O_Hb, w.O_Zb, true);
  bool split_metric = false;
  if (many_tiles) {
    FQL_TRY(chain(FQL_NET_ACTOR_ONESTEP_FLOW, w.XOb, 3 * B, 0, 3 * B, w.O_Hb, w.O_Zb, w.O_out, 1, S0));
  } else {
    // small batch: the same cluster-of-16 chain kernel as the Euler integration (2.7 us per layer instead of a GEMM launch each)
    int rc = 1;
    if (ctx->use_euler_cluster && ctx->use_cluster_fwd && !wide) {
      // rows (s',z') and (s,z) feed the critic passes that everything else waits for; the (s,z'') rows only feed the mse metric
      // and go layer by layer on a side stream (the GPU holds 7 clusters of 16: 2 Euler + 4 here)
      TcClusterFwdSpec cf;
      memset(&cf, 0, sizeof(cf));
      cf.d = d; cf.L = &L; cf.params = P; cf.shadow = shadow; cf.net = FQL_NET_ACTOR_ONESTEP_FLOW; cf.X0b = w.XOb; cf.rows_cap = 3 * B; cf.r0 = 0;
      cf.M = 2 * B; cf.Hb = w.O_Hb; cf.Zb = w.O_Zb; cf.out = w.O_out;
      cf.t_start = ctx->stamps ? ctx->stamps + 15 : nullptr;
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[56], S0));  // XOb padded
      rc = tc_cluster_forward(cf, row_tiles, S0);
      if (rc < 0) return -1;
      if (rc == 0) {
        FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->s9, ctx->ev[56], 0));
        TcActor fm = actor(FQL_NET_ACTOR_ONESTEP_FLOW, w.XOb, kO, 3 * B, 2 * B, B, w.O_Hb, w.O_Zb, true);
        FQL_TRY(tc_actor_forward(fm, w.O_out + (int64_t)2 * B * sh.A, (long long)3 * B * sh.A, 0, nullptr, ctx->s9));
        FQL_TRY(launch_post_onestep(sh, b, w, raw, ctx->s9, 2));
        FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[57], ctx->s9));
        split_metric = true;
      }
    }
    if (rc == 1) FQL_TRY(tc_actor_forward(fo, w.O_out, (long long)3 * B * sh.A, 0, nullptr, S0));
  }
  FQL_TRY(stamp(ctx, 3, S0));   // one-step actor forward done
  FQL_TRY(launch_post_onestep(sh, b, w, raw, S0, split_metric ? 1 : 3));
  FQL_TRY(tc_pad_bf16(w.XC, w.XCb, (int64_t)3 * S * B, sh.F + sh.A, kO, S0));
  TcCritic cr;
  memset(&cr, 0, sizeof(cr));
  cr.d = d; cr.L = &L; cr.params = P; cr.shadow = shadow; cr.M = B; cr.K0pad = kO; cr.x_ss = (long long)B * kO; cr.buf = &w.pC; cr.Hb = w.C_Hb;
  cr.cs_scratch = w.cs_scratch[2];
  bool split_cpost = false;
  if (many_tiles) {   // enough row tiles to fill the GPU: the three critic problems x 2 heads as ONE fused launch
    TcChainSpec t;
    memset(&t, 0, sizeof(t));
    t.d = d; t.L = &L; t.P = 3; t.net[0] = FQL_NET_TARGET_CRITIC; t.net[1] = FQL_NET_CRITIC; t.net[2] = FQL_NET_CRITIC;
    t.params = P; t.shadow = shadow; t.M = B; t.X0b = w.XCb; t.Mcap0 = B; t.buf = &w.pC; t.save = 1; t.n_steps = 1; t.Hb = w.C_Hb;
    if (big_bwd) { t.DGb = w.C_DGb; t.XHb = w.C_XHb; t.save_mask = 6; }   // problems 1 (critic loss) and 2 (actor Q loss) have a backward
    FQL_TRY(tc_mlp_chain2(t, S0));
  } else {
    // three independent chains {target critic(s',a'), critic(s,a), critic(s,clip a_pi)}: S0 + two forked streams
    FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[40], S0));
    // problem 2 = critic(s, a_pi) heads the longest chain of the step (-> dQ/da -> one-step actor backward): it stays on the
    // high-priority main stream, the two TD problems go to the side streams
    cudaStream_t cs[3] = {ctx->s6, ctx->s5, S0};
    const int nets[3] = {FQL_NET_TARGET_CRITIC, FQL_NET_CRITIC, FQL_NET_CRITIC};
    for (int p = 0; p < 3; p++) {
      if (cs[p] != S0) FQL_CHECK_CUDA(cudaStreamWaitEvent(cs[p], ctx->ev[40], 0));
      TcCritic f = cr;
      f.p = p; f.X0b = reinterpret_cast<const bf16*>(w.XCb) + (int64_t)p * S * B * kO;
      FQL_TRY(tc_critic_forward(f, nets[p], w.C_out, cs[p]));
      if (cs[p] != S0) FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[41 + p], cs[p]));
    }
    // the TD half of the loss kernel follows problems 0 and 1 on their side stream; the main stream only waits for problem 2
    FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->s5, ctx->ev[41], 0));
    FQL_TRY(launch_critic_post(sh, hp, b, w, raw, ctx->s5, 1));
    FQL_CHECK_CUDA(cudaEventRecord(ev_cpost, ctx->s5));
    split_cpost = true;
  }
  FQL_TRY(stamp(ctx, 5, S0));   // critic forward (problem 2) done
  const DpLamArgs dpl = dp_lam_args(ctx->dp);
  FQL_TRY(launch_critic_post(sh, hp, b, w, raw, S0, split_cpost ? 2 : 3, &dpl));
  if (!split_cpost) FQL_CHECK_CUDA(cudaEventRecord(ev_cpost, S0));

  if (c.do_backward) {
    // critic backward (fql.py:36-37) on S2, after the bc-flow backward
    FQL_CHECK_CUDA(cudaStreamWaitEvent(S2, ev_cpost, 0));
    TcCritic t = cr;
    t.grads = c.st->grads; t.p = 1; t.X0b = reinterpret_cast<const bf16*>(w.XCb) + (int64_t)1 * S * B * kO;
    t.dOut = w.dq; t.dOutb = w.C1_dOutb;
    for (int l = 0; l < NH; l++) { t.dZb[l] = w.C1_dZb[l]; t.dZf[l] = w.C1_dZf[l]; t.dHf[l] = w.C1_dHf[l]; }
    if (pix) t.dX0 = w.dX0C;   // d(critic loss)/d(features) of both heads -> the critic's encoder (agents/fql.py:36)
    if (big_bwd) {
      FQL_TRY(tc_critic_backward_big(t, w.C_XHb, w.C_DGb, S2));
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[36], S2));
    } else {
      FQL_TRY(tc_critic_backward(t, S2, ctx->s5, ctx->s8, &ctx->ev[28]));
      if (pix) FQL_TRY(encoder_grads(c, L, w, FQL_NET_CRITIC, w.dX0C, 2, sh.F + sh.A, w.dfeat[0], 3, S2));
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[54], ctx->s8));
      FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->s5, ctx->ev[54], 0));
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[36], ctx->s5));
    }
    if (dp_bucketed) {
      const NetView& nc = L.net[FQL_NET_CRITIC];
      FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->sc, ctx->ev[36], 0));
      int64_t b0 = nc.begin;
      if (ctx->dp_bc_late) {              // bc-flow | critic are adjacent in the arena: one exchange for both
        FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->sc, ctx->ev[16], 0));
        b0 = L.net[FQL_NET_ACTOR_BC_FLOW].begin;
        FQL_REQUIRE(L.net[FQL_NET_ACTOR_BC_FLOW].end == nc.begin, "arena order: bc-flow is not followed by the critic");
      }
      FQL_TRY(stamp(ctx, 22, ctx->sc));   // critic bucket: gradients final
      FQL_TRY(dp_reduce_bucket(ctx->dp, 1, b0, nc.end - b0, nullptr, ctx->sc));
      FQL_TRY(stamp(ctx, 23, ctx->sc));   // critic bucket reduced
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[59], ctx->sc));
    }
    FQL_CHECK_CUDA(cudaStreamWaitEvent(S2, ctx->ev[36], 0));
    FQL_CHECK_CUDA(cudaStreamWaitEvent(S2, ctx->ev[16], 0));  // bc-flow weight gradients (side stream s3)
    FQL_TRY(stamp(ctx, 8, S2));   // bc-flow + critic gradients complete
    FQL_TRY(record_early(ctx, S2));
    // critic input gradient with stored params (fql.py:70) on S0
    TcCritic q = cr;
    q.grads = nullptr; q.p = 2; q.X0b = reinterpret_cast<const bf16*>(w.XCb) + (int64_t)2 * S * B * kO;
    q.dOut = w.dqs; q.dOutb = w.C2_dOutb; q.dX0 = w.dX0;
    for (int l = 0; l < NH; l++) { q.dZb[l] = w.C2_dZb[l]; q.dZf[l] = w.C2_dZf[l]; q.dHf[l] = w.C2_dHf[l]; }
    if (big_bwd) FQL_TRY(tc_critic_backward_big(q, w.C_XHb, w.C_DGb, S0));
    else FQL_TRY(tc_critic_backward(q, S0, nullptr, nullptr, &ctx->ev[44]));
    FQL_TRY(stamp(ctx, 6, S0));   // critic input-gradient chain done
    if (dp_bucketed && c.do_apply && ctx->dp_early_adam) {
      // data parallel: bc-flow's and the critic's part of the optimizer pass (+ Polyak) right behind their bucket exchanges on the
      // communication stream, under the one-step actor's backward and bucket exchange.  Last readers of their weights: the Euler
      // chain (bc-flow) and the critic input-gradient chain that S0 has just enqueued; the critic's own backward precedes ev[36].
      const int blk1 = (int)(L.net[FQL_NET_ACTOR_ONESTEP_FLOW].begin / FQL_LEAF_PAD);
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[52], S0));
      FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->sc, ctx->ev[52], 0));
      FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->sc, ev_euler, 0));
      FQL_TRY(launch_adam_polyak_stats(L, hp, S, c.st->params, c.st->mu, c.st->nu, c.st->grads, w.gstats + S * 4, w.partials, c.st->shadow,
                                       tc_shadow_seed_elems(d, L), ctx->sc, 0, blk1));
      FQL_TRY(stamp(ctx, 9, ctx->sc));  // early optimizer pass done
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[59], ctx->sc));
      ctx->adam_done_blk = blk1;
    }
  }
  if (bc_enc_forked) FQL_CHECK_CUDA(cudaStreamWaitEvent(S2, ctx->ev[37], 0));
  FQL_CHECK_CUDA(cudaEventRecord(ev_s2, S2));
  FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ev_euler, 0));
  if (split_metric) FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ctx->ev[57], 0));
  if (split_cpost) FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ev_cpost, 0));
  FQL_TRY(launch_actor_grad(sh, hp, w, raw, S0, w.O_dOutb));
  FQL_TRY(stamp(ctx, 7, S0));   // joined Euler, dL/da done
  if (c.do_backward) {
    TcActor bo = actor(FQL_NET_ACTOR_ONESTEP_FLOW, w.XOb, kO, 3 * B, B, B, w.O_Hb, w.O_Zb, true);
    int rc = 1;
    if (!many_tiles && ctx->use_euler_cluster && ctx->use_cluster_bwd && !wide) {
      // small batch: the dgrad chain as ONE cluster-of-16 launch (the Euler chain has finished: its clusters are free), then the
      // ten independent parameter-gradient launches dealt onto five idle side streams
      TcClusterBwdSpec cb;
      memset(&cb, 0, sizeof(cb));
      cb.d = d; cb.L = &L; cb.shadow = shadow; cb.net = FQL_NET_ACTOR_ONESTEP_FLOW; cb.dOutb = w.O_dOutb; cb.M = B;
      cb.Zb = w.O_Zb; cb.z_rows_cap = 3 * B; cb.z_r0 = B; cb.dZb = w.O_dZb; cb.dZf = w.O_dZf;
      cb.t_start = ctx->stamps ? ctx->stamps + 17 : nullptr;
      rc = tc_cluster_dgrad(cb, 0, S0);
      if (rc < 0) return -1;
      if (rc == 0) {
        cudaStream_t ss[5] = {ctx->s4, ctx->s9, ctx->s3, ctx->s7, ctx->s1};  // one weight gradient + one column sum each
        FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[18], S0));
        for (int i = 0; i < 5; i++) FQL_CHECK_CUDA(cudaStreamWaitEvent(ss[i], ctx->ev[18], 0));
        FQL_TRY(tc_actor_param_grads(bo, w.dapi, w.O_dOutb, w.O_dZb, w.O_dZf, ss, 5));
        for (int i = 0; i < 5; i++) {
          FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[19 + i], ss[i]));
          FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ctx->ev[19 + i], 0));
        }
      }
    }
    if (rc == 1 && big_bwd) {
      FQL_TRY(tc_actor_backward_big(bo, w.dapi, w.O_dOutb, w.O_dZb, true, S0));
    } else if (rc == 1) {
      FQL_TRY(tc_actor_backward(bo, w.dapi, w.O_dOutb, w.O_dZb, w.O_dZf, S0, ctx->s4, ctx->s9, &ctx->ev[18], true));
      if (pix) {  // d(alpha distill + Q loss)/d(features) -> the one-step actor's encoder (agents/fql.py:65)
        FQL_TRY(tc_actor_input_grad(bo, w.O_dZb[0], w.dX0O, S0));
        FQL_TRY(encoder_grads(c, L, w, FQL_NET_ACTOR_ONESTEP_FLOW, w.dX0O, 1, sh.F + sh.A, w.dfeat[2], 1, S0));
      }
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[55], ctx->s9));
      FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->s4, ctx->ev[55], 0));
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[26], ctx->s4));
      FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ctx->ev[26], 0));
    }
    FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ctx->ev[16], 0));
    FQL_TRY(stamp(ctx, 10, S0));  // one-step actor gradients complete
  }
  FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ev_s2, 0));
  if (dp_grads && !dp_bucketed) {
    const int64_t t0 = L.net[FQL_NET_TARGET_CRITIC].begin;
    FQL_TRY(dp_reduce_bucket(ctx->dp, 3, 0, t0, raw, S0));
  }
  if (dp_bucketed) {  // the one-step actor's bucket + the metric accumulators close the exchange; the optimizer pass follows on S0
    const NetView& no = L.net[FQL_NET_ACTOR_ONESTEP_FLOW];
    FQL_TRY(stamp(ctx, 24, S0));          // one-step bucket: gradients final
    FQL_TRY(dp_reduce_bucket(ctx->dp, 2, no.begin, no.end - no.begin, raw, S0));
    FQL_TRY(stamp(ctx, 25, S0));          // one-step bucket reduced
    FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ctx->ev[59], 0));
  }
  return 0;
}

int enqueue_step(FqlContext* ctx, const StepCall& c, cudaStream_t S0) {
  Layout L;
  WsPtrs w;
  FQL_TRY(check_common(c.d, c.ws, c.ws_bytes, &L, &w));
  const bool tcm = c.d->precision == FQL_PRECISION_BF16_TC;
  if (tcm) {
    FQL_TRY(tc_supported(c.d, false));
    FQL_REQUIRE(c.st->shadow != nullptr, "FQL_PRECISION_BF16_TC needs FqlState.shadow (fql_shadow_bytes() bytes, kept by fql_refresh_shadow)");
  }
  const StepShape sh = make_shape(c.d);
  const FqlHparams hp = *c.hp;
  const int S = sh.S, B = sh.B, H = sh.H;
  FQL_REQUIRE(!(c.d->normalize_q_loss && c.d->global_batch != c.d->batch) || ctx->dp.active,
              "normalize_q_loss with a data-parallel split needs the global mean|q| inside the step (agents/fql.py:74-76): attach a peer-memory "
              "communicator (fql_dp_attach); the fql_step_grads / fql_step_apply split cannot provide it");
  if (ctx->dp.active && c.do_grads) {
    FQL_REQUIRE(c.st->grads == ctx->dp.comm.base[ctx->dp.comm.rank], "data parallel: FqlState.grads must be this rank's symmetric buffer (base[rank])");
    FQL_REQUIRE(c.d->global_batch == (int64_t)c.d->batch * ctx->dp.comm.world && ctx->dp.S == S && !c.raw,
                "data parallel: global_batch must be world x batch (%d x %d), seeds as attached, and the raw accumulators internal", ctx->dp.comm.world, c.d->batch);
  }
  float* raw = c.raw ? c.raw : w.raw_local;
  const float* P = c.st->params;

  if (c.do_grads && !tcm) {
    const FqlBatch& b = *c.b;
    cudaStream_t S1 = ctx->s1, S2 = ctx->s2;
    cudaEvent_t ev_prep = ctx->ev[0], ev_f0 = ctx->ev[1], ev_cpost = ctx->ev[2], ev_euler = ctx->ev[3], ev_s2 = ctx->ev[4];
    FQL_TRY(launch_zero_bc(raw, (int64_t)S * FQL_NUM_RAW, c.do_apply ? c.st->count : nullptr, hp, w.gstats + S * 4, S0, w.cpost_ticket, 3 * S));
    FQL_TRY(encode_observations(c, L, w, S0, ctx));
    FQL_TRY(launch_prep(sh, b, w, S0));
    const bool pix = c.d->reserved[0] > 0;
    FQL_CHECK_CUDA(cudaEventRecord(ev_prep, S0));
    FQL_CHECK_CUDA(cudaStreamWaitEvent(S1, ev_prep, 0));
    FQL_CHECK_CUDA(cudaStreamWaitEvent(S2, ev_prep, 0));

    // ---- S1: bc-flow network on {BC rows, Euler rows}, then the Euler chain
    FwdSpec fF;
    memset(&fF, 0, sizeof(fF));
    fF.P = 1; fF.nv[0] = &L.net[FQL_NET_ACTOR_BC_FLOW]; fF.params = P; fF.arena = L.arena;
    fF.S = S; fF.E = 1; fF.M = 2 * B; fF.H = H; fF.X0 = w.XF; fF.Mcap0 = 2 * B; fF.r0_in = 0;
    fF.buf = &w.pF; fF.r0 = 0; fF.save_z = 1;
    {
      FQL_TRY(mlp_forward(fF, S1));
      FQL_CHECK_CUDA(cudaEventRecord(ev_f0, S1));
      fF.M = B; fF.r0_in = B; fF.r0 = B; fF.save_z = 0;
      for (int i = 0; i < sh.flow_steps; i++) {
        FQL_TRY(launch_euler_update(sh, w, i, S1));
        if (i + 1 < sh.flow_steps) FQL_TRY(mlp_forward(fF, S1));
      }
    }
    FQL_CHECK_CUDA(cudaEventRecord(ev_euler, S1));

    // ---- S0: one-step actor, then the grouped critic pass
    FwdSpec fO;
    memset(&fO, 0, sizeof(fO));
    fO.P = 1; fO.nv[0] = &L.net[FQL_NET_ACTOR_ONESTEP_FLOW]; fO.params = P; fO.arena = L.arena;
    fO.S = S; fO.E = 1; fO.M = 3 * B; fO.H = H; fO.X0 = w.XO; fO.Mcap0 = 3 * B; fO.r0_in = 0;
    fO.buf = &w.pO; fO.r0 = 0; fO.save_z = 1;
    FQL_TRY(mlp_forward(fO, S0));
    FQL_TRY(launch_post_onestep(sh, b, w, raw, S0));
    FwdSpec fC;
    memset(&fC, 0, sizeof(fC));
    fC.P = 3; fC.nv[0] = &L.net[FQL_NET_TARGET_CRITIC]; fC.nv[1] = &L.net[FQL_NET_CRITIC]; fC.nv[2] = &L.net[FQL_NET_CRITIC];
    fC.params = P; fC.arena = L.arena; fC.S = S; fC.E = 2; fC.M = B; fC.H = H; fC.X0 = w.XC; fC.Mcap0 = B; fC.r0_in = 0;
    fC.buf = &w.pC; fC.r0 = 0; fC.save_z = 1;
    FQL_TRY(mlp_forward(fC, S0));
    {
      const DpLamArgs dpl = dp_lam_args(ctx->dp);
      FQL_TRY(launch_critic_post(sh, hp, b, w, raw, S0, 3, &dpl));
    }
    FQL_CHECK_CUDA(cudaEventRecord(ev_cpost, S0));

    // ---- S2: BC loss + bc-flow backward, critic backward
    FQL_CHECK_CUDA(cudaStreamWaitEvent(S2, ev_f0, 0));
    FQL_TRY(launch_bc_post(sh, w, raw, S2));
    if (c.do_backward) {
      BwdSpec bF;
      memset(&bF, 0, sizeof(bF));
      bF.nv = &L.net[FQL_NET_ACTOR_BC_FLOW]; bF.params = P; bF.grads = c.st->grads; bF.arena = L.arena;
      bF.S = S; bF.E = 1; bF.M = B; bF.H = H; bF.X0 = w.XF; bF.Mcap0 = 2 * B; bF.buf = &w.pF; bF.p = 0; bF.r0 = 0;
      bF.dOut = w.dpred; bF.dpp[0] = w.dF[0]; bF.dpp[1] = w.dF[1];
      if (pix) bF.dX0 = w.dX0F;
      FQL_TRY(mlp_backward(bF, S2));
      if (pix) FQL_TRY(encoder_grads(c, L, w, FQL_NET_ACTOR_BC_FLOW, w.dX0F, 1, sh.F + sh.A + 1, w.dfeat[1], 4, S2));
      FQL_CHECK_CUDA(cudaStreamWaitEvent(S2, ev_cpost, 0));
      BwdSpec bC;
      memset(&bC, 0, sizeof(bC));
      bC.nv = &L.net[FQL_NET_CRITIC]; bC.params = P; bC.grads = c.st->grads; bC.arena = L.arena;
      bC.S = S; bC.E = 2; bC.M = B; bC.H = H; bC.X0 = w.XC + (int64_t)1 * S * B * (sh.F + sh.A); bC.Mcap0 = B;
      bC.buf = &w.pC; bC.p = 1; bC.r0 = 0; bC.dOut = w.dq; bC.dpp[0] = w.dC[0]; bC.dpp[1] = w.dC[1];
      if (pix) bC.dX0 = w.dX0C;
      FQL_TRY(mlp_backward(bC, S2));
      if (pix) FQL_TRY(encoder_grads(c, L, w, FQL_NET_CRITIC, w.dX0C, 2, sh.F + sh.A, w.dfeat[0], 3, S2));
      FQL_TRY(record_early(ctx, S2));
    }
    FQL_CHECK_CUDA(cudaEventRecord(ev_s2, S2));

    // ---- S0: critic input gradient (stored params: no weight grads, fql.py:70), distill, onestep backward
    if (c.do_backward) {
      BwdSpec bQ;
      memset(&bQ, 0, sizeof(bQ));
      bQ.nv = &L.net[FQL_NET_CRITIC]; bQ.params = P; bQ.grads = nullptr; bQ.arena = L.arena;
      bQ.S = S; bQ.E = 2; bQ.M = B; bQ.H = H; bQ.X0 = w.XC + (int64_t)2 * S * B * (sh.F + sh.A); bQ.Mcap0 = B;
      bQ.buf = &w.pC; bQ.p = 2; bQ.r0 = 0; bQ.dOut = w.dqs; bQ.dpp[0] = w.dCp[0]; bQ.dpp[1] = w.dCp[1]; bQ.dX0 = w.dX0;
      FQL_TRY(mlp_backward(bQ, S0));
    }
    FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ev_euler, 0));
    FQL_TRY(launch_actor_grad(sh, hp, w, raw, S0));
    if (c.do_backward) {
      BwdSpec bO;
      memset(&bO, 0, sizeof(bO));
      bO.nv = &L.net[FQL_NET_ACTOR_ONESTEP_FLOW]; bO.params = P; bO.grads = c.st->grads; bO.arena = L.arena;
      bO.S = S; bO.E = 1; bO.M = B; bO.H = H; bO.X0 = w.XO + (int64_t)B * (sh.F + sh.A); bO.Mcap0 = 3 * B;
      bO.buf = &w.pO; bO.p = 0; bO.r0 = B; bO.dOut = w.dapi; bO.dpp[0] = w.dO[0]; bO.dpp[1] = w.dO[1];
      if (pix) bO.dX0 = w.dX0O;
      FQL_TRY(mlp_backward(bO, S0));
      if (pix) FQL_TRY(encoder_grads(c, L, w, FQL_NET_ACTOR_ONESTEP_FLOW, w.dX0O, 1, sh.F + sh.A, w.dfeat[2], 1, S0));
    }
    FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ev_s2, 0));
    if (ctx->dp.active && c.do_backward) {  // parity mode: one reduction over the trainable prefix of the arena (+ metric gather)
      const int64_t t0 = L.net[FQL_NET_TARGET_CRITIC].begin;
      FQL_TRY(dp_reduce_bucket(ctx->dp, 3, 0, t0, raw, S0));
    }
  }

  ctx->adam_done_blk = 0;
  if (c.do_grads && tcm) FQL_TRY(enqueue_grads_tc(ctx, c, L, w, sh, hp, raw, S0));
  int raw_ranks = c.raw_ranks > 1 ? c.raw_ranks : 1;
  const float* raw_fin = raw;
  if (ctx->dp.active && c.do_grads) {
    // forward-only calls (fql_total_loss) still gather the accumulators so that info describes the GLOBAL batch
    if (!c.do_backward) FQL_TRY(dp_reduce_bucket(ctx->dp, 2, 0, 0, raw, S0));
    raw_fin = dp_raw_all(ctx->dp);
    raw_ranks = ctx->dp.comm.world;
  }
  if (c.do_apply) {
    if (!c.do_grads) FQL_TRY(launch_zero_bc(nullptr, 0, c.st->count, hp, w.gstats + S * 4, S0));
    // Adam + Polyak + gradient statistics (+ the bf16 operand shadow of the new parameters) in one pass over the arenas
    // (the target critic's blocks carry no gradient and are written by the critic's CTAs: skipped when the pass is split)
    const int blk0 = ctx->adam_done_blk;
    const int blk1 = blk0 ? (int)(L.net[FQL_NET_TARGET_CRITIC].begin / FQL_LEAF_PAD) : -1;
    FQL_TRY(launch_adam_polyak_stats(L, hp, S, c.st->params, c.st->mu, c.st->nu, c.st->grads, w.gstats + S * 4, w.partials,
                                     tcm ? c.st->shadow : nullptr, tcm ? tc_shadow_seed_elems(c.d, L) : 0, S0, blk0, blk1));
    FQL_TRY(stamp(ctx, 11, S0));  // optimizer pass done
    if (tcm) {  // the zero-padded narrow last-layer copies, beside the statistics tail
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[50], S0));
      FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->s1, ctx->ev[50], 0));
      FQL_TRY(tc_refresh_shadow_lastlayer(c.d, L, c.st->params, c.st->shadow, ctx->s1));
      FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[51], ctx->s1));
    }
    FinArgs fin;
    memset(&fin, 0, sizeof(fin));
    fin.sh = sh; fin.hp = hp; fin.raw = raw_fin; fin.ranks = raw_ranks; fin.info = c.info;
    FQL_TRY(launch_grad_stats_final(L, S, w.partials, w.gstats, c.st->count, S0, c.info ? &fin : nullptr));
    if (tcm) FQL_CHECK_CUDA(cudaStreamWaitEvent(S0, ctx->ev[51], 0));
  }
  if (c.info && !c.do_apply) FQL_TRY(launch_finalize_info(sh, hp, raw_fin, raw_ranks, w.gstats, c.info, 0, S0));
  FQL_TRY(stamp(ctx, 12, S0));    // step end
  return 0;
}

// Run `c` through a cached CUDA graph when possible (the ~150 launches of a B=256 step are launch-bound otherwise).
int run_step_on(FqlContext* ctx, const StepCall& c, cudaStream_t S0) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  FQL_CHECK_CUDA(cudaStreamIsCapturing(S0, &cap));
  if (!ctx->use_graph || cap != cudaStreamCaptureStatusNone) {
    const long long before = g_fql_launches;
    const int rc0 = enqueue_step(ctx, c, S0);
    ctx->launches += g_fql_launches - before;
    return rc0;
  }

  std::vector<unsigned char> key;
  auto push = [&](const void* p, size_t n) { key.insert(key.end(), (const unsigned char*)p, (const unsigned char*)p + n); };
  push(c.d, sizeof(FqlDims));
  push(c.hp, sizeof(FqlHparams));
  if (c.b) push(c.b, sizeof(FqlBatch));
  push(c.st, sizeof(FqlState));
  push(&c.raw, sizeof(void*)); push(&c.info, sizeof(void*)); push(&c.ws, sizeof(void*)); push(&c.ws_bytes, sizeof(size_t));
  int flags[4] = {c.do_grads, c.do_backward, c.do_apply, c.raw_ranks};
  push(flags, sizeof(flags));
  push(&S0, sizeof(S0));
  GraphEntry* seen = nullptr;
  for (auto& g : ctx->graphs)
    if (g.key == key) {
      if (g.exec) {
        FQL_CHECK_CUDA(cudaGraphLaunch(g.exec, S0));
        ctx->launches += g.kernels;
        return 0;
      }
      seen = &g;
    }
  if (!seen) {
    // First sight of this argument set: run eagerly (this also lets the driver load every kernel outside a capture);
    // the second call captures, later calls replay.
    if (ctx->graphs.size() >= 16) {
      if (ctx->graphs.front().exec) cudaGraphExecDestroy(ctx->graphs.front().exec);
      ctx->graphs.erase(ctx->graphs.begin());
    }
    ctx->graphs.push_back({key, nullptr, 0});
    const long long before = g_fql_launches;
    const int rc0 = enqueue_step(ctx, c, S0);
    ctx->launches += g_fql_launches - before;
    return rc0;
  }
  // validate eagerly (errors must not surface in the middle of a capture)
  {
    Layout L;
    WsPtrs w;
    FQL_TRY(check_common(c.d, c.ws, c.ws_bytes, &L, &w));
    if (c.d->precision == FQL_PRECISION_BF16_TC) {
      FQL_TRY(tc_supported(c.d, false));
      FQL_REQUIRE(c.st->shadow != nullptr, "FQL_PRECISION_BF16_TC needs FqlState.shadow");
    }
  }
  FQL_CHECK_CUDA(cudaStreamBeginCapture(S0, cudaStreamCaptureModeThreadLocal));
  const long long before = g_fql_launches;
  int rc = enqueue_step(ctx, c, S0);
  const long long nk = g_fql_launches - before;
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaStreamEndCapture(S0, &graph);
  if (rc) {
    if (graph) cudaGraphDestroy(graph);
    return rc;
  }
  FQL_CHECK_CUDA(e);
  cudaGraphExec_t exec = nullptr;
  FQL_CHECK_CUDA(cudaGraphInstantiate(&exec, graph, 0));
  cudaGraphDestroy(graph);
  seen->exec = exec;
  seen->kernels = nk;
  FQL_CHECK_CUDA(cudaGraphLaunch(exec, S0));
  ctx->launches += nk;
  return 0;
}


// The legacy default stream (what torch hands out by default) can neither be captured nor forked from with non-blocking
// streams safely, so the step runs on the context's own stream, ordered after / before the caller's stream with events.
int run_step(FqlContext* ctx, const StepCall& c, void* stream) {
  FQL_REQUIRE(ctx != nullptr, "context is NULL");
  FQL_REQUIRE(c.d && c.hp && c.st, "NULL argument");
  cudaStream_t user = reinterpret_cast<cudaStream_t>(stream);
  if (user != nullptr && user != cudaStreamLegacy) return run_step_on(ctx, c, user);
  FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[6], user));
  FQL_CHECK_CUDA(cudaStreamWaitEvent(ctx->s0, ctx->ev[6], 0));
  const int rc = run_step_on(ctx, c, ctx->s0);
  FQL_CHECK_CUDA(cudaEventRecord(ctx->ev[7], ctx->s0));
  FQL_CHECK_CUDA(cudaStreamWaitEvent(user, ctx->ev[7], 0));
  return rc;
}

}  // namespace

extern "C" int fql_update_step(FqlContext* ctx, const FqlDims* d, const FqlHparams* hp, const FqlBatch* batch,
                               const FqlState* st, float* info, void* workspace, size_t ws_bytes, void* stream) {
  FQL_REQUIRE(batch != nullptr, "batch is NULL");
  StepCall c{d, hp, batch, st, nullptr, info, workspace, ws_bytes, 1, 1, 1, 1};
  return run_step(ctx, c, stream);
}

extern "C" int fql_step_grads(FqlContext* ctx, const FqlDims* d, const FqlHparams* hp, const FqlBatch* batch,
                              const FqlState* st, float* raw, void* workspace, size_t ws_bytes, void* stream) {
  FQL_REQUIRE(batch != nullptr && raw != nullptr, "batch/raw is NULL");
  StepCall c{d, hp, batch, st, raw, nullptr, workspace, ws_bytes, 1, 1, 0, 1};
  return run_step(ctx, c, stream);
}

extern "C" int fql_step_apply(FqlContext* ctx, const FqlDims* d, const FqlHparams* hp, const FqlState* st, const float* raw,
                              float* info, void* workspace, size_t ws_bytes, void* stream) {
  FQL_REQUIRE(raw != nullptr, "raw is NULL");
  StepCall c{d, hp, nullptr, st, const_cast<float*>(raw), info, workspace, ws_bytes, 0, 0, 1, 1};
  return run_step(ctx, c, stream);
}

extern "C" int fql_step_apply_gathered(FqlContext* ctx, const FqlDims* d, const FqlHparams* hp, const FqlState* st, const float* raw_all,
                                       int32_t ranks, float* info, void* workspace, size_t ws_bytes, void* stream) {
  FQL_REQUIRE(raw_all != nullptr && ranks >= 1, "raw_all is NULL / ranks < 1");
  StepCall c{d, hp, nullptr, st, const_cast<float*>(raw_all), info, workspace, ws_bytes, 0, 0, 1, ranks};
  return run_step(ctx, c, stream);
}

extern "C" int fql_total_loss(FqlContext* ctx, const FqlDims* d, const FqlHparams* hp, const FqlBatch* batch,
                              const FqlState* st, float* info, void* workspace, size_t ws_bytes, void* stream) {
  FQL_REQUIRE(batch != nullptr && info != nullptr, "batch/info is NULL");
  StepCall c{d, hp, batch, st, nullptr, info, workspace, ws_bytes, 1, 0, 0, 1};
  return run_step(ctx, c, stream);
}

// ---------------------------------------------------------------------------------------------------------
// standalone forward entry points
// ---------------------------------------------------------------------------------------------------------
namespace {
struct FwdWs {          // workspace of the stand-alone forward entry points
  float* X;             // fp32 first-layer input [S][rows][in_dim]
  void* Xb;             // bf16 copy, zero padded to K0pad <= 128 columns (tensor cores)
  void* Hx;             // exchange scratch of the cluster Euler kernel (tensor cores, hidden = 512)
  void* Hb[FQL_MAXL];   // bf16 hidden activations [S][rows][H] per hidden layer (tensor cores, hidden < 512: layer by layer)
  float* act;           // fp32 Euler state [S][rows][A] of the same
  float* feat;          // pixel observations: encoder output and pass buffers
  EncBuf eb;
  PassBuf pb;           // fp32 activations / output of the SIMT path
};

size_t carve_forward(const FqlDims* d, int rows, int ens, int in_dim, int out_dim, bool ln, void* base, FwdWs* f) {
  Carver c{reinterpret_cast<char*>(base)};
  memset(f, 0, sizeof(*f));
  f->X = c.take((int64_t)d->num_seeds * rows * in_dim);
  f->Xb = c.take((int64_t)d->num_seeds * rows * 128 / 2 + 4);
  const bool tc = d->precision == FQL_PRECISION_BF16_TC;
  if (tc && d->hidden == 512) f->Hx = c.take((int64_t)(tc_euler_scratch_elems(d, rows) / 2 + 4));
  if (tc && d->hidden < 512) {
    for (int l = 0; l < d->num_hidden; l++) f->Hb[l] = c.take((int64_t)d->num_seeds * rows * d->hidden / 2);
    f->act = c.take((int64_t)d->num_seeds * rows * d->action_dim);
  }
  if (d->reserved[0] > 0) {  // pixel observations: encoder pass buffers + its output
    f->feat = c.take((int64_t)rows * d->obs_dim);
    c.off = (c.off + 255) & ~(size_t)255;
    c.off += enc_carve(d, rows, base ? c.base + c.off : nullptr, &f->eb, false);
  }
  carve_pass(c, &f->pb, d->num_seeds * ens, rows, d->hidden, d->num_hidden, out_dim, ln, false);
  return c.off + 256;
}

// the one-step / bc-flow actor layer by layer on the tensor cores (hidden < 512), first-layer operand f.Xb
TcActor fwd_actor(const FqlDims* d, const Layout& L, int net, const float* params, const void* shadow, int rows, const FwdWs& f) {
  TcActor t;
  memset(&t, 0, sizeof(t));
  t.d = d; t.L = &L; t.net = net; t.params = params; t.shadow = shadow; t.M = rows;
  t.X0b = f.Xb; t.K0pad = (int)round_up64(L.net[net].in_dim, 64); t.x_ss = (long long)rows * t.K0pad;
  for (int l = 0; l < d->num_hidden; l++) t.Hb[l] = f.Hb[l];
  t.h_ss = (long long)rows * d->hidden;
  return t;
}
}  // namespace

extern "C" size_t fql_forward_workspace_bytes(const FqlDims* d, int32_t rows) {
  if (fql_validate_dims(d)) return 0;
  FwdWs f;
  return carve_forward(d, rows, 2, d->obs_dim + d->action_dim + 1, d->action_dim > 1 ? d->action_dim : 1, true, nullptr, &f);
}

static int forward_net(const FqlDims* d, const Layout& L, int net, const float* params, const float* X, PassBuf* pb, int rows,
                       cudaStream_t st) {
  FwdSpec f;
  memset(&f, 0, sizeof(f));
  f.P = 1; f.nv[0] = &L.net[net]; f.params = params; f.arena = L.arena;
  f.S = d->num_seeds; f.E = L.net[net].ens; f.M = rows; f.H = d->hidden; f.X0 = X; f.Mcap0 = rows; f.buf = pb;
  return mlp_forward(f, st);
}

extern "C" int fql_mlp_forward(FqlContext*, const FqlDims* d, int32_t net, const float* params, const float* x, float* y,
                               int32_t rows, void* workspace, size_t ws_bytes, void* stream) {
  Layout L;
  FQL_TRY(fql_build_layout(d, &L));
  FQL_REQUIRE(net >= 0 && net < FQL_NUM_NETS && rows >= 1, "bad net/rows");
  FQL_REQUIRE(d->precision == FQL_PRECISION_FP32, "fql_mlp_forward: FP32 only");
  const NetView& nv = L.net[net];
  FwdWs f;
  const size_t need = carve_forward(d, rows, nv.ens, nv.in_dim, nv.out_dim, nv.ln, nullptr, &f);
  FQL_REQUIRE(workspace && ws_bytes >= need, "workspace too small: have %zu need %zu", ws_bytes, need);
  carve_forward(d, rows, nv.ens, nv.in_dim, nv.out_dim, nv.ln, workspace, &f);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  FQL_TRY(forward_net(d, L, net, params, x, &f.pb, rows, st));
  FQL_CHECK_CUDA(cudaMemcpyAsync(y, f.pb.out, sizeof(float) * (size_t)d->num_seeds * nv.ens * rows * nv.out_dim,
                                 cudaMemcpyDeviceToDevice, st));
  return 0;
}

extern "C" int fql_sample_actions(FqlContext*, const FqlDims* d, const float* params, const void* shadow, const float* obs,
                                  const float* noise, float* actions_out, int32_t rows, void* workspace, size_t ws_bytes,
                                  void* stream) {
  Layout L;
  FQL_TRY(fql_build_layout(d, &L));
  FQL_REQUIRE(rows >= 1, "rows=%d", rows);
  const NetView& nv = L.net[FQL_NET_ACTOR_ONESTEP_FLOW];
  FwdWs f;
  const size_t need = carve_forward(d, rows, 1, nv.in_dim, nv.out_dim, nv.ln, nullptr, &f);
  FQL_REQUIRE(workspace && ws_bytes >= need, "workspace too small: have %zu need %zu", ws_bytes, need);
  carve_forward(d, rows, 1, nv.in_dim, nv.out_dim, nv.ln, workspace, &f);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t R = (int64_t)d->num_seeds * rows;
  if (d->reserved[0] > 0) {  // obs is uint8 [rows,H,W,C]: encode with the one-step actor's encoder (networks.py:226-227)
    FQL_TRY(enc_forward(d, nv.enc, params, reinterpret_cast<const uint8_t*>(obs), rows, f.eb, f.feat, st));
    obs = f.feat;
  }
  FQL_TRY(launch_concat(obs, d->obs_dim, noise, d->action_dim, 0.f, 0, f.X, R, st));
  if (d->precision == FQL_PRECISION_BF16_TC && !tc_wide_input(d)) {
    FQL_REQUIRE(shadow != nullptr, "FQL_PRECISION_BF16_TC needs the bf16 shadow");
    const int kp = (int)round_up64(nv.in_dim, 64);
    FQL_TRY(tc_pad_bf16(f.X, f.Xb, R, nv.in_dim, kp, st));
    if (d->hidden == 512) {
      TcChainSpec t;
      memset(&t, 0, sizeof(t));
      t.d = d; t.L = &L; t.P = 1; t.net[0] = FQL_NET_ACTOR_ONESTEP_FLOW; t.params = params; t.shadow = shadow;
      t.M = rows; t.X0b = f.Xb; t.Mcap0 = rows; t.n_steps = 1; t.out_override = actions_out; t.clip_out = 1;
      return tc_mlp_chain2(t, st);
    }
    const TcActor t = fwd_actor(d, L, FQL_NET_ACTOR_ONESTEP_FLOW, params, shadow, rows, f);
    return tc_actor_forward(t, actions_out, (long long)rows * d->action_dim, 1, nullptr, st);
  }
  FQL_TRY(forward_net(d, L, FQL_NET_ACTOR_ONESTEP_FLOW, params, f.X, &f.pb, rows, st));
  FQL_TRY(launch_clip(f.pb.out, actions_out, R * d->action_dim, st));
  return 0;
}

extern "C" int fql_compute_flow_actions(FqlContext*, const FqlDims* d, const float* params, const void* shadow, const float* obs,
                                        const float* noise, float* actions_out, int32_t rows, void* workspace, size_t ws_bytes,
                                        void* stream) {
  Layout L;
  FQL_TRY(fql_build_layout(d, &L));
  FQL_REQUIRE(rows >= 1, "rows=%d", rows);
  const NetView& nv = L.net[FQL_NET_ACTOR_BC_FLOW];
  FwdWs f;
  const size_t need = carve_forward(d, rows, 1, nv.in_dim, nv.out_dim, nv.ln, nullptr, &f);
  FQL_REQUIRE(workspace && ws_bytes >= need, "workspace too small: have %zu need %zu", ws_bytes, need);
  carve_forward(d, rows, 1, nv.in_dim, nv.out_dim, nv.ln, workspace, &f);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t R = (int64_t)d->num_seeds * rows;
  if (d->reserved[0] > 0) {  // fql.py:162-163: encode once with actor_bc_flow_encoder, then is_encoded=True
    FQL_TRY(enc_forward(d, nv.enc, params, reinterpret_cast<const uint8_t*>(obs), rows, f.eb, f.feat, st));
    obs = f.feat;
  }
  FQL_TRY(launch_concat(obs, d->obs_dim, noise, d->action_dim, 0.f, 1, f.X, R, st));
  if (d->precision == FQL_PRECISION_BF16_TC && !tc_wide_input(d)) {
    FQL_REQUIRE(shadow != nullptr, "FQL_PRECISION_BF16_TC needs the bf16 shadow");
    const int kp = (int)round_up64(nv.in_dim, 64);
    FQL_TRY(tc_pad_bf16(f.X, f.Xb, R, nv.in_dim, kp, st));
    if (d->hidden == 512) {
      TcEulerSpec e;
      memset(&e, 0, sizeof(e));
      e.d = d; e.L = &L; e.params = params; e.shadow = shadow; e.X0b = f.Xb; e.Mcap0 = rows; e.r0_in = 0; e.M = rows;
      e.a0 = noise; e.target = actions_out; e.scratch = f.Hx;
      return tc_euler_cluster(e, st);
    }
    // agents/fql.py:155-171: the fp32 Euler state starts as the noise; each step's last layer adds v / flow_steps to it and
    // rewrites the action and time columns of the bf16 first-layer operand
    FQL_CHECK_CUDA(cudaMemcpyAsync(f.act, noise, sizeof(float) * (size_t)R * d->action_dim, cudaMemcpyDeviceToDevice, st));
    const TcActor t = fwd_actor(d, L, FQL_NET_ACTOR_BC_FLOW, params, shadow, rows, f);
    for (int i = 0; i < d->flow_steps; i++) {
      TcEuler eu{f.act, actions_out, i, d->flow_steps};
      FQL_TRY(tc_actor_forward(t, nullptr, 0, 0, &eu, st));
    }
    return 0;
  }
  for (int i = 0; i < d->flow_steps; i++) {
    FQL_TRY(forward_net(d, L, FQL_NET_ACTOR_BC_FLOW, params, f.X, &f.pb, rows, st));
    FQL_TRY(launch_euler_inplace(f.X, f.pb.out, d->obs_dim, d->action_dim, R, i, d->flow_steps, actions_out, st));
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// misc API
// ---------------------------------------------------------------------------------------------------------
extern "C" int fql_version(void) { return FQL_ABI_VERSION; }
extern "C" const char* fql_last_error(void) { return g_err; }
extern "C" const char* fql_info_name(int i) {
  static const char* names[FQL_NUM_INFO] = {
      "critic/critic_loss", "critic/q_mean", "critic/q_max", "critic/q_min", "actor/actor_loss", "actor/bc_flow_loss",
      "actor/distill_loss", "actor/q_loss", "actor/q", "actor/mse", "grad/max", "grad/min", "grad/norm"};
  return (i >= 0 && i < FQL_NUM_INFO) ? names[i] : nullptr;
}
extern "C" int64_t fql_arena_floats(const FqlDims* d) {
  Layout L;
  if (fql_build_layout(d, &L)) return -1;
  return L.arena;
}
extern "C" size_t fql_workspace_bytes(const FqlDims* d) {
  Layout L;
  if (fql_build_layout(d, &L)) return 0;
  WsPtrs w;
  return carve_workspace(d, L, nullptr, &w);
}
extern "C" size_t fql_shadow_bytes(const FqlDims* d) {
  Layout L;
  if (fql_build_layout(d, &L)) return 0;
  if (d->precision != FQL_PRECISION_BF16_TC) return 0;
  return (size_t)d->num_seeds * (size_t)tc_shadow_seed_elems(d, L) * 2;
}
extern "C" int fql_refresh_shadow(const FqlDims* d, const float* params, void* shadow, void* stream) {
  Layout L;
  FQL_TRY(fql_build_layout(d, &L));
  if (d->precision != FQL_PRECISION_BF16_TC) return 0;
  return tc_refresh_shadow(d, L, params, shadow, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int fql_layout(const FqlDims* d, FqlLeaf* leaves, int32_t cap, int32_t* n_leaves) {
  Layout L;
  FQL_TRY(fql_build_layout(d, &L));
  int n = 0;
  auto put = [&](int net, int layer, int kind, int ens, int rows, int cols, int64_t off) {
    if (leaves && n < cap) leaves[n] = FqlLeaf{net, layer, kind, ens, rows, cols, off};
    n++;
  };
  static const int kOrder[FQL_NUM_NETS] = {FQL_NET_ACTOR_BC_FLOW, FQL_NET_CRITIC, FQL_NET_ACTOR_ONESTEP_FLOW, FQL_NET_TARGET_CRITIC};
  for (int oi = 0; oi < FQL_NUM_NETS; oi++) {  // arena order
    const int t = kOrder[oi];
    const NetView& v = L.net[t];
    for (int l = 0; l < v.n_layers; l++) {
      put(t, l, FQL_LEAF_KERNEL, v.ens, v.k_of(l), v.n_of(l), v.off_w[l]);
      put(t, l, FQL_LEAF_BIAS, v.ens, 1, v.n_of(l), v.off_b[l]);
      if (v.ln && l + 1 < v.n_layers) {
        put(t, l, FQL_LEAF_LN_SCALE, v.ens, 1, v.n_of(l), v.off_lns[l]);
        put(t, l, FQL_LEAF_LN_BIAS, v.ens, 1, v.n_of(l), v.off_lnb[l]);
      }
    }
    if (v.has_enc) {
      static const int stacks[3] = {16, 32, 32};
      int c = d->reserved[2], h = d->reserved[0], w = d->reserved[1];
      for (int i = 0; i < 3; i++) {
        const int f = stacks[i];
        const int cin[3] = {c, f, f};
        for (int j = 0; j < 3; j++) {
          put(t, 3 * i + j, FQL_LEAF_CONV_KERNEL, 1, 9 * cin[j], f, v.enc.off_cw[i][j]);
          put(t, 3 * i + j, FQL_LEAF_CONV_BIAS, 1, 1, f, v.enc.off_cb[i][j]);
        }
        c = f; h = (h + 1) / 2; w = (w + 1) / 2;
      }
      put(t, 0, FQL_LEAF_ENC_DENSE_KERNEL, 1, h * w * c, d->obs_dim, v.enc.off_dw);
      put(t, 0, FQL_LEAF_ENC_DENSE_BIAS, 1, 1, d->obs_dim, v.enc.off_db);
    }
  }
  if (n_leaves) *n_leaves = n;
  FQL_REQUIRE(!leaves || n <= cap, "leaf table too small: need %d", n);
  return 0;
}
