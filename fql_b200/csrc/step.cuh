// step.cuh -- shapes, workspace map and launcher prototypes of one FQLAgent.update (agents/fql.py:122-133).
#pragma once
#include "common.cuh"

#include <cudaTypedefs.h>

enum {  // raw accumulators per seed (all-reduced across data-parallel ranks: [0..8] SUM, [9..10] MAX)
  RAW_CRITIC_SQ = 0, RAW_Q_SUM = 1, RAW_BC_SQ = 2, RAW_DISTILL_SQ = 3, RAW_QPI_SUM = 4, RAW_QPI_ABS = 5, RAW_MSE = 6,
  RAW_Q_MAX = 9, RAW_Q_NEGMIN = 10,
};

struct StepShape {
  int S, B, GB, F, A, H, NH;  // seeds, local batch, global batch, obs, action, hidden width, hidden layers
  int q_agg_min, normalize_q_loss, flow_steps;
};

struct PassBuf {               // activations of one grouped MLP pass: [G][Mcap][H] per hidden layer
  float* Z[FQL_MAXL];          // pre-activation (kept for backward / LN)
  float* Hh[FQL_MAXL];         // post activation (+LN): next layer's input
  float* mu[FQL_MAXL];         // LN row statistics [G][Mcap]
  float* rstd[FQL_MAXL];
  float* out;                  // [G][Mcap][out_dim]
  int G, Mcap;
};

struct EncTc {                // bf16 NHWC activations / prepared weights of one tensor-core encoder pass (encoder_tc.cu)
  void *img, *y0, *p[3], *r1[3], *r2[3], *xs[3], *flat;
  void *wf, *wd, *wdense;     // [9][320][64] forward / input-gradient matrices of the convolutions, [flat][512] Dense kernel
  void *dzb, *da, *db, *dc;
};
struct EncBuf {               // activations of one encoder pass over B images (encoder.cu)
  EncTc tc;                   // FQL_PRECISION_BF16_ENC
  float *pl[3], *c1[3], *x[3];
  uint8_t* arg[3];
  float *flat, *z, *scratch;
  float *dz, *dflat, *da, *db, *dc, *partial;
  int flat_dim;
};

struct WsPtrs {
  float *XO, *XF, *XC, *vel;   // first-layer inputs [S][3B][F+A], [S][2B][F+A+1], [3][S][B][F+A]; vel [S][B][A]
  float *O_out, *F_out, *C_out;
  float *dq, *dqs, *dpred, *dapi, *target, *dX0;
  float *raw_local;            // [S][FQL_NUM_RAW] when the caller passes none
  float *gstats;               // [S][4]: grad max, min, L1-of-L2 norm
  float *partials;             // [S][blocks][4] per 1024-float arena block: max, min, sumsq
  float *cpost_part;           // [2][S][64][4] per-CTA partial sums of the TD / actor-Q loss kernel
  int *cpost_ticket;           // [3][S] arrival counters of the same (zero between steps)
  PassBuf pO, pF, pC;
  float *dC[2], *dCp[2], *dF[2], *dO[2];  // backward ping-pong [S][E][B][H]
  void *XOb, *XFb, *XCb;       // bf16 zero-padded copies of the first-layer inputs (FQL_PRECISION_BF16_TC)
  // per-layer tensor-core path (actor networks): bf16 activations / pre-activations, backward ping-pong, Euler state
  void *O_Hb[FQL_MAXL], *O_Zb[FQL_MAXL], *F_Hb[FQL_MAXL], *F_Zb[FQL_MAXL], *E_Hb[FQL_MAXL];
  void *C_Hb[FQL_MAXL];        // bf16 post-LN activations of the grouped critic pass [3][S][2][B][H]
  void *C_XHb[FQL_MAXL], *C_DGb[FQL_MAXL];  // large-batch backward: bf16 xhat and gelu' of the same pass
  void *O_dZb[FQL_MAXL], *F_dZb[FQL_MAXL], *O_dOutb, *F_dOutb;
  float *O_dZf[FQL_MAXL], *F_dZf[FQL_MAXL];
  void *C1_dZb[FQL_MAXL], *C1_dOutb, *C2_dZb[FQL_MAXL], *C2_dOutb;
  float *C1_dZf[FQL_MAXL], *C1_dHf[FQL_MAXL], *C2_dZf[FQL_MAXL], *C2_dHf[FQL_MAXL];
  float *euler_a;
  float *cs_scratch[3];        // column-sum scratch per backward side stream
  // pixel configs: encoder outputs that replace the observations per call site, encoder pass buffers, feature gradients
  float *feat[5];              // [S][B][512]: onestep(next_obs), onestep(obs), target critic(next_obs), critic(obs), bc_flow(obs)
  float *dfeat[3];             // gradients w.r.t. feat[3] (critic), feat[4] (bc flow), feat[1] (onestep)
  float *dX0F, *dX0O, *dX0C;   // first-layer input gradients of the three trainable MLPs
  EncBuf enc[5];
  const float *src[5];         // what prep reads as `observations` for the 5 call sites (features, or the batch itself)
  void *euler_hx;              // exchange scratch of the cluster Euler kernel
};

StepShape make_shape(const FqlDims* d);
size_t carve_workspace(const FqlDims* d, const Layout& L, void* base, WsPtrs* w);  // returns bytes needed

int launch_prep(const StepShape& sh, const FqlBatch& b, const WsPtrs& w, cudaStream_t st);
int launch_post_onestep(const StepShape& sh, const FqlBatch& b, const WsPtrs& w, float* raw, cudaStream_t st, int parts = 3);
struct DpLamArgs;
int launch_critic_post(const StepShape& sh, const FqlHparams& hp, const FqlBatch& b, const WsPtrs& w, float* raw, cudaStream_t st, int parts = 3,
                       const DpLamArgs* dpl = nullptr);
int launch_bc_post(const StepShape& sh, const WsPtrs& w, float* raw, cudaStream_t st);
int launch_euler_update(const StepShape& sh, const WsPtrs& w, int step, cudaStream_t st);
int launch_actor_grad(const StepShape& sh, const FqlHparams& hp, const WsPtrs& w, float* raw, cudaStream_t st, void* dapib = nullptr);
int launch_finalize_info(const StepShape& sh, const FqlHparams& hp, const float* raw, int ranks, const float* gstats, float* info,
                         int with_grad_stats, cudaStream_t st);
int launch_clip(const float* in, float* out, int64_t n, cudaStream_t st);
int launch_concat(const float* x0, int k0, const float* x1, int k1, float c2, int k2, float* out, int64_t rows, cudaStream_t st);
int launch_euler_inplace(float* X, const float* v, int F, int A, int64_t rows, int step, int nsteps, float* out, cudaStream_t st);

// optim.cu
int launch_adam_polyak_stats(const Layout& L, const FqlHparams& hp, int S, float* params, float* mu, float* nu,
                             const float* grads, const float* bc, float* partials, void* shadow, int64_t shadow_seed, cudaStream_t st,
                             int blk0 = 0, int blk1 = -1);  // CTA range in FQL_LEAF_PAD blocks (default: the whole arena)
// fin != NULL: the same launch also writes the info vector (finalize_info_kernel folded in: one launch less at the end of the step)
struct FinArgs {
  StepShape sh;
  FqlHparams hp;
  const float* raw;
  int ranks;
  float* info;
};
int launch_grad_stats_final(const Layout& L, int S, const float* partials, float* gstats, int32_t* count_inc, cudaStream_t st,
                            const FinArgs* fin = nullptr);

#ifdef __CUDACC__
// info[13] of one seed from the (all-gathered) raw accumulators + gradient statistics (agents/fql.py:38-44, 78-90, flax_utils.py:147-149).
// data parallel: `raw` is the all-gather of every rank's accumulators [ranks][S][FQL_NUM_RAW]: sums add, max / -min take the max
__device__ __forceinline__ void fql_finalize_info_seed(const StepShape& sh, const FqlHparams& hp, const float* raw, int ranks, const float* gstats,
                                                       float* info, int s, int with_grad_stats) {
  float rw[FQL_NUM_RAW];
  for (int i = 0; i < FQL_NUM_RAW; i++) rw[i] = raw[s * FQL_NUM_RAW + i];
  for (int r = 1; r < ranks; r++) {
    const float* o = raw + ((int64_t)r * sh.S + s) * FQL_NUM_RAW;
    for (int i = 0; i < 9; i++) rw[i] += o[i];
    rw[RAW_Q_MAX] = fmaxf(rw[RAW_Q_MAX], o[RAW_Q_MAX]);
    rw[RAW_Q_NEGMIN] = fmaxf(rw[RAW_Q_NEGMIN], o[RAW_Q_NEGMIN]);
  }
  float* o = info + s * FQL_NUM_INFO;
  const float gb = (float)sh.GB, A = (float)sh.A;
  const float critic_loss = rw[RAW_CRITIC_SQ] / (2.0f * gb);
  const float bc = rw[RAW_BC_SQ] / (gb * A);
  const float distill = rw[RAW_DISTILL_SQ] / (gb * A);
  const float q = rw[RAW_QPI_SUM] / gb;
  float q_loss = -q;
  if (sh.normalize_q_loss) q_loss = (1.0f / (rw[RAW_QPI_ABS] / gb)) * q_loss;
  o[0] = critic_loss;
  o[1] = rw[RAW_Q_SUM] / (2.0f * gb);
  o[2] = rw[RAW_Q_MAX];
  o[3] = -rw[RAW_Q_NEGMIN];
  o[4] = bc + hp.alpha * distill + q_loss;
  o[5] = bc;
  o[6] = distill;
  o[7] = q_loss;
  o[8] = q;
  o[9] = rw[RAW_MSE] / (gb * A);
  if (with_grad_stats) {
    o[10] = gstats[s * 4 + 0];
    o[11] = gstats[s * 4 + 1];
    o[12] = gstats[s * 4 + 2];
  } else {
    o[10] = o[11] = o[12] = 0.f;
  }
}
#endif
int launch_zero(float* p, int64_t n, cudaStream_t st);
// zero p[0..n) and (count != NULL) write optax's float32 bias corrections {1 - b1^(count+1), 1 - b2^(count+1)} to bc[0..1]
int launch_zero_bc(float* p, int64_t n, const int32_t* count, const FqlHparams& hp, float* bc, cudaStream_t st, int* tickets = nullptr,
                   int n_tickets = 0);

// chain2_tc.cu -- fused per-tile MLP chains (hidden = 512): one forward pass, or the whole Euler loop, per 128-row tile and launch
struct TcChainSpec {
  const FqlDims* d;
  const Layout* L;
  int P;
  int net[FQL_MAXP];
  const float* params;
  const void* shadow;
  int M;             // valid rows per group
  const void* X0b;   // bf16 [P][S][Mcap0][K0pad]
  int Mcap0, r0_in;
  PassBuf* buf;      // fp32 saves / output (optional)
  int r0, save;
  float* out_override;
  void* const* Hb;   // optional bf16 copies of the hidden activations [G][Mcap][H] per layer (tensor-core backward operands)
  void* const* Zb;   // optional bf16 copies of the pre-activations (buf == NULL only)
  int Mcap_override; // row capacity of the Hb/Zb/out buffers when buf == NULL
  int n_steps;       // > 1: Euler integration of compute_flow_actions
  const float* a0;
  float* target;
  int clip_out;
  void* const* DGb;  // optional: save bf16 gelu'(z) per hidden layer instead of the pre-activations (large-batch backward)
  void* const* XHb;  // LayerNorm only: save bf16 xhat per hidden layer instead of the normalised activations
  int save_mask;     // bit p set = problem p writes its saves (0 = all)
};
int tc_mlp_chain2(const TcChainSpec& f, cudaStream_t st);
// chain2_tc.cu: the whole input-gradient chain of one network's backward, one launch.  Every pointer is already offset to the
// first row of the problem; rows of group (s, e) start at ((s * ens + e) * Mcap + r0).
struct TcChain2BwdSpec {
  const FqlDims* d;
  const Layout* L;
  int net;
  const float* params;   // LayerNorm scales
  const void* shadow;
  const void* dOutb;     // bf16 [S][ens][M][64]: dL/d(output), zero padded
  int M, Mcap, r0;       // rows per group, row capacity per group and first row of the forward's saves
  int Mcap_dz;           // row capacity per group of dZb / dX0 (0: M)
  void* const* DGb;      // bf16 gelu'(z_l)           [S][ens][Mcap][H] per hidden layer
  void* const* XHb;      // bf16 xhat_l (LayerNorm)
  float* const* rstd;    // fp32 [S][ens][Mcap]   (LayerNorm)
  void* const* dZb;      // out (optional): bf16 dZ_l [S][ens][Mcap_dz][H] -- operands of the weight gradients
  float* dX0;            // out (optional): fp32 [S][ens][Mcap_dz][K0] input gradient
};
int tc_mlp_chain2_backward(const TcChain2BwdSpec& f, cudaStream_t st);
// mlp_tc.cu -- shared by every tensor-core MLP kernel: shape limits, bf16 shadow, padded first-layer operands, TMA tensor maps
int tc_supported(const FqlDims* d, bool fused_kernels = true);   // fused_kernels: also the limits of the chain / cluster kernels
inline bool tc_wide_input(const FqlDims* d) { return d->obs_dim + d->action_dim + 1 > 128; }   // pixel configs: 512 encoder features
int64_t tc_shadow_seed_elems(const FqlDims* d, const Layout& L);
int tc_refresh_shadow(const FqlDims* d, const Layout& L, const float* params, void* shadow, cudaStream_t st);
int tc_refresh_shadow_lastlayer(const FqlDims* d, const Layout& L, const float* params, void* shadow, cudaStream_t st);
int tc_pad_bf16(const float* x, void* y, int64_t rows, int K0, int K0pad, cudaStream_t st);
// TMA tensor maps: the driver's cuTensorMapEncodeTiled (NULL when the driver does not provide it), and a bf16 [rows][inner] row-major
// tensor read in boxes of [box_rows][box_inner]
PFN_cuTensorMapEncodeTiled_v12000 get_encode();
int make_map_2d(CUtensorMap* m, const void* base, uint64_t inner, uint64_t rows, uint32_t box_inner, uint32_t box_rows,
                CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B);

// tc_gemm.cu -- generic tcgen05 GEMM (one Dense layer: forward / dgrad / wgrad)
enum { TC_MODE_STORE_F32 = 0, TC_MODE_FWD_HIDDEN = 1, TC_MODE_DGRAD_GELU = 2, TC_MODE_EULER = 3, TC_MODE_WGRAD_LN = 4 };
struct TcOperand {   // bf16 tensor [g1][g0][rows][inner] with pitches ld / s0 / s1 (elements)
  const void* ptr;
  int inner, rows;
  long long ld;
  int g0;
  long long s0;
  int g1;
  long long s1;
};
struct TcPtr {       // epilogue operand addressed as base + g0*s0 + g1*s1 (elements of its own type), row pitch ld
  void* base;
  long long s0, s1;
  int ld;
};
struct TcGemmSpec {
  int M, N, K, G0, G1;
  int a_mn, b_mn;    // operand is MN-major ([K][rows] row-major) instead of K-major ([rows][K])
  TcOperand A, B;
  int mode;
  TcPtr bias, out_f, out_h, out_z, zin, act, xb, target;
  int F, Adim, step, n_steps, clip;
  int ksplit;        // > 1: split K over CTAs, partial tiles ADDED into a zeroed fp32 output (STORE_F32 / WGRAD_LN)
  TcPtr ln_s, ln_b, dbias, wmaster, dln_s, dln_b;   // TC_MODE_WGRAD_LN: LayerNorm scale / bias [M], db [N], fp32 weights [M][N], out dgamma / dbeta [M]
  void* dbg;  // optional device buffer for per-CTA timestamps
};
// column sums over rows of a bf16 tensor [G][M][N] ADDED into fp32 out[g * out_stride + n] (bias gradients from the bf16 dZ saves)
int launch_colsum_bf16(const void* X, int64_t G, int64_t M, int N, float* out, int64_t out_stride_g0, int G0, int64_t out_stride_g1, cudaStream_t st);
int tc_gemm(const TcGemmSpec& s, cudaStream_t st);
struct TcActor;
int tc_actor_input_grad(const TcActor& t, const void* dZ0b, float* dX0, cudaStream_t st);

// tc_path.cu -- layer-by-layer tensor-core schedules
struct TcActor {
  const FqlDims* d;
  const Layout* L;
  int net;
  const float* params;
  const void* shadow;
  float* grads;
  int M;                 // valid rows per seed
  const void* X0b;       // bf16 [S][..][K0pad], already offset to the first row
  int K0pad;
  long long x_ss;        // seed pitch (elements)
  void* Hb[FQL_MAXL];    // bf16 [S][..][H] per hidden layer, already offset to the first row
  void* Zb[FQL_MAXL];
  long long h_ss;
  float* cs_scratch;     // scratch of the two-stage column sums (65536 floats)
};
struct TcEuler {
  float* act;
  float* target;
  int step, n_steps;
};
struct TcCritic {
  const FqlDims* d;
  const Layout* L;
  const float* params;
  const void* shadow;
  float* grads;          // NULL: input gradient only
  int M, p;
  const void* X0b;       // bf16 [S][M][K0pad] of problem p
  int K0pad;
  long long x_ss;
  const PassBuf* buf;    // fp32 Z / mu / rstd of the grouped pass
  void* const* Hb;       // bf16 H per layer [P][S][E][Mcap][H]
  const float* dOut;     // [S][2][M]
  void* dOutb;
  void* dZb[FQL_MAXL];     // per hidden layer: bf16 dZ_l  [S][2][M][H]
  float* dZf[FQL_MAXL];    //                   fp32 dZ_l
  float* dHf[FQL_MAXL];    //                   fp32 dH_l (before the LayerNorm/GELU backward)
  float* dX0;
  float* cs_scratch;
};
int tc_actor_forward(const TcActor& t, float* out, long long out_ss, int clip, const TcEuler* eu, cudaStream_t st);
int tc_actor_backward(const TcActor& t, const float* dOut, void* dOutb, void* const dZb[FQL_MAXL], float* const dZf[FQL_MAXL],
                      cudaStream_t st, cudaStream_t side, cudaStream_t side2, cudaEvent_t* ev, bool dOutb_ready = false);
int tc_critic_backward(const TcCritic& t, cudaStream_t st, cudaStream_t side, cudaStream_t side2, cudaEvent_t* ev);
int tc_critic_forward(const TcCritic& t, int net, float* out, cudaStream_t st);
// large-batch backward: one chain2 launch per network + split-K weight gradients (tc_path.cu)
int tc_actor_backward_big(const TcActor& t, const float* dOut, void* dOutb, void* const dZb[FQL_MAXL], bool dOutb_ready, cudaStream_t st);
int tc_critic_backward_big(const TcCritic& t, void* const* XHb, void* const* DGb, cudaStream_t st);

// euler_cluster.cu -- compute_flow_actions as one persistent thread-block-cluster kernel (hidden = 512)
struct TcEulerSpec {
  const FqlDims* d;
  const Layout* L;
  const float* params;
  const void* shadow;
  const void* X0b;     // bf16 [S][Mcap0][K0pad] first-layer operand (obs | noise | t = 0)
  int Mcap0, r0_in, M;
  const float* a0;     // [S][M][A]
  const float* c0;     // optional fp32 [S][M][H]: features @ W0[:F] + b0 (pixel configs); X0b is then bf16 [S][Mcap0][64] = (noise | t = 0)
  float* target;       // [S][M][A]
  void* scratch;       // tc_euler_scratch_elems() bf16 elements
  void* dbg;           // optional timestamp buffer (diagnostics)
  void* t_start;       // optional: %globaltimer when CTA 0 starts / ends (2 x u64, diagnostics)
};
size_t tc_euler_scratch_elems(const FqlDims* d, int M);
struct TcClusterFwdSpec {
  const FqlDims* d;
  const Layout* L;
  const float* params;
  const void* shadow;
  int net;
  const void* X0b;          // bf16 [S][rows_cap][K0pad]
  int rows_cap, r0, M;      // rows [r0, r0 + M) of every seed
  void* const* Hb;          // bf16 [S][rows_cap][H] per hidden layer (saved activations)
  void* const* Zb;          // bf16 pre-activations
  float* out;               // fp32 [S][rows_cap][out_dim]
  void* t_start;            // optional: %globaltimer at start / end of CTA 0 (diagnostics)
};
int tc_cluster_forward(const TcClusterFwdSpec& f, int other_clusters, cudaStream_t st);
struct TcClusterBwdSpec {
  const FqlDims* d;
  const Layout* L;
  const void* shadow;
  int net;
  const void* dOutb;        // bf16 [S][M][64]: dL/d(output), zero padded
  int M;
  void* const* Zb;          // bf16 pre-activations saved by the forward: [S][z_rows_cap][H], rows [z_r0, z_r0 + M)
  int z_rows_cap, z_r0;
  void* const* dZb;         // out: bf16 [S][M][H] per hidden layer
  float* const* dZf;        // out: fp32 copies (bias gradients)
  void* t_start;            // optional diagnostics
};
int tc_cluster_dgrad(const TcClusterBwdSpec& f, int other_clusters, cudaStream_t st);
// parameter gradients of an actor network from finished dZ buffers: 2 * n_layers independent launches spread over `streams`
int tc_actor_param_grads(const TcActor& t, const float* dOut, const void* dOutb, void* const dZb[FQL_MAXL], float* const dZf[FQL_MAXL],
                         cudaStream_t* streams, int n_streams);
int tc_euler_cluster(const TcEulerSpec& f, cudaStream_t st);

// encoder.cu
size_t enc_carve(const FqlDims* d, int64_t B, void* base, EncBuf* e, bool for_backward);
int enc_forward(const FqlDims* d, const EncView& v, const float* params, const uint8_t* obs, int64_t B, const EncBuf& e, float* feat,
                cudaStream_t st);
int enc_backward(const FqlDims* d, const EncView& v, const float* params, float* grads, const uint8_t* obs, int64_t B, const EncBuf& e,
                 const float* dfeat, cudaStream_t st);
// encoder_tc.cu -- the same three entry points on tcgen05 (FQL_PRECISION_BF16_ENC); encoder.cu dispatches to them
size_t enc_tc_carve(const FqlDims* d, int64_t B, void* base, EncBuf* e, bool for_backward);
int enc_tc_forward(const FqlDims* d, const EncView& v, const float* params, const uint8_t* obs, int64_t B, const EncBuf& e, float* feat,
                   cudaStream_t st);
int enc_tc_backward(const FqlDims* d, const EncView& v, const float* params, float* grads, const uint8_t* obs, int64_t B, const EncBuf& e,
                    const float* dfeat, cudaStream_t st);
int launch_extract_feat_grad(const float* dX0, float* out, int E, int64_t M, int K0, int F, cudaStream_t st);
