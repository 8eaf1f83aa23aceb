/*
 * fql_b200.h -- C ABI of libfql_b200.so: the B200 (sm_100a) implementation of the FQL training hot path.
 *
 * The reference (zhouzypaul/fql) is pure Python/JAX and has NO FFI today; this boundary is what a
 * `jax.ffi` custom call (or the ctypes shim in fql_b200/_lib.py) binds.  Every entry point below names the
 * reference interface it replaces (paths relative to the reference repo root).
 *
 * Conventions
 *   - plain C: POD structs, raw device pointers, sizes, a cudaStream_t passed as void*.  No torch/jax types.
 *   - enqueue-only: no entry point synchronises the device or allocates on the hot path; scratch memory is a
 *     caller-owned workspace sized by fql_workspace_bytes().
 *   - returns 0 on success; non-zero => fql_last_error() holds a thread-local message.  Nothing throws.
 *   - all floating tensors are float32, row-major; Dense kernels are [in,out] exactly as Flax stores them;
 *     ensemble (critic) leaves keep the leading axis 2; a leading "seed" axis of length num_seeds vectorises
 *     independent agents (seed stride = fql_arena_floats()).
 *   - parameters / Adam moments / gradients live in flat float32 "arenas" with one common leaf layout, queried
 *     with fql_layout().  In-place updates (params, mu, nu, count) are aliased in/out buffers
 *     (jax.ffi input_output_aliases).
 */
#ifndef FQL_B200_H_
#define FQL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FQL_ABI_VERSION 1

/* Networks inside an arena, in arena order.  Names follow agents/fql.py:224-229 (`modules_<name>`). */
enum { FQL_NET_ACTOR_BC_FLOW = 0, FQL_NET_ACTOR_ONESTEP_FLOW = 1, FQL_NET_CRITIC = 2, FQL_NET_TARGET_CRITIC = 3, FQL_NUM_NETS = 4 };
/* Leaf kinds inside a network (utils/networks.py:54,58). */
enum { FQL_LEAF_KERNEL = 0, FQL_LEAF_BIAS = 1, FQL_LEAF_LN_SCALE = 2, FQL_LEAF_LN_BIAS = 3,
       /* encoder leaves (utils/encoders.py): layer = 3*stack + conv for the convolutions */
       FQL_LEAF_CONV_KERNEL = 4, FQL_LEAF_CONV_BIAS = 5, FQL_LEAF_ENC_DENSE_KERNEL = 6, FQL_LEAF_ENC_DENSE_BIAS = 7 };
/* Arithmetic mode of the contractions. */
enum { FQL_PRECISION_FP32 = 0,      /* fp32 FFMA everywhere: parity mode (1e-5 vs the fp32/fp64 oracle)          */
       FQL_PRECISION_BF16_TC = 1,   /* bf16 operands on tcgen05, fp32 accumulate/epilogue, fp32 master weights   */
       FQL_PRECISION_BF16_ENC = 2 };/* pixel configs: the ImpalaEncoders (89 % of the FLOPs) as bf16 implicit-GEMM
                                     * convolutions on tcgen05 (fp32 accumulate, bf16 activations), MLPs in fp32  */

/* Static problem description: agents/fql.py:249-270 (get_config) + shapes fixed at create() (:192-194). */
typedef struct FqlDims {
  int32_t batch;             /* rows per seed held by THIS rank                                             */
  int32_t global_batch;      /* rows per seed over all data-parallel ranks (loss denominators); >= batch     */
  int32_t obs_dim;           /* F: observation features fed to the MLPs                                      */
  int32_t action_dim;        /* A                                                                            */
  int32_t hidden;            /* width of the hidden layers (512)                                             */
  int32_t num_hidden;        /* number of hidden layers (4); MLP = num_hidden+1 Dense layers                 */
  int32_t critic_layer_norm; /* config['layer_norm']                                                         */
  int32_t actor_layer_norm;  /* config['actor_layer_norm']                                                   */
  int32_t q_agg_min;         /* config['q_agg']=='min'                                                       */
  int32_t normalize_q_loss;  /* config['normalize_q_loss']                                                   */
  int32_t flow_steps;        /* config['flow_steps']                                                         */
  int32_t num_seeds;         /* independent agents vectorised on the leading axis (1 = the reference)        */
  int32_t precision;         /* FQL_PRECISION_*                                                              */
  int32_t reserved[3];       /* pixel configs (config['encoder']=='impala_small'): {img_h, img_w, img_c}, observations are
                              * uint8 [S,B,img_h,img_w,img_c] (passed through the float* fields) and obs_dim must be 512;
                              * {0,0,0} = state-based */
} FqlDims;

/* Hyper-parameters that are runtime scalars. agents/fql.py:255-264, optax.adam defaults. */
typedef struct FqlHparams {
  float lr, beta1, beta2, eps;
  float discount, tau, alpha;
  /* (1-beta1), (1-beta2), (1-tau) evaluated in double on the host and then rounded, as the reference's Python-float
   * arithmetic does (optax `(1 - decay) * g`, fql.py:116 `tp * (1 - tau)`): 1.0f-0.999f differs from (float)0.001 by 1.3e-5. */
  float one_minus_beta1, one_minus_beta2, one_minus_tau;
  float reserved[2];
} FqlHparams;

typedef struct FqlLeaf {
  int32_t net;        /* FQL_NET_*                                  */
  int32_t layer;      /* Dense_<layer> / LayerNorm_<layer>          */
  int32_t kind;       /* FQL_LEAF_*                                 */
  int32_t ens;        /* leading ensemble axis (1 = none, 2 critic) */
  int32_t rows, cols; /* kernel: [in,out]; vectors: rows=1          */
  int64_t offset;     /* float offset inside one seed's arena       */
} FqlLeaf;

/* One training batch (utils/datasets.py:68-92 output) + the five noise draws of one update (SURVEY 8a "RNG
 * derivation"): device pointers, leading seed axis if num_seeds>1. */
typedef struct FqlBatch {
  const float* observations;      /* [S,B,F]  */
  const float* actions;           /* [S,B,A]  */
  const float* next_observations; /* [S,B,F]  */
  const float* rewards;           /* [S,B]    */
  const float* masks;             /* [S,B]    */
  const float* z_next;            /* [S,B,A] N(0,1): critic_loss sample_actions   (agents/fql.py:25)  */
  const float* x0;                /* [S,B,A] N(0,1): BC flow x_0                  (agents/fql.py:52)  */
  const float* t;                 /* [S,B,1] U[0,1): BC flow time                 (agents/fql.py:54)  */
  const float* z;                 /* [S,B,A] N(0,1): distillation noises          (agents/fql.py:63)  */
  const float* z_metric;          /* [S,B,A] N(0,1): logging sample_actions       (agents/fql.py:82)  */
} FqlBatch;

/* Train state (utils/flax_utils.py:53-70 TrainState + optax ScaleByAdamState): aliased in/out. */
typedef struct FqlState {
  float* params;   /* [S, arena]                                   */
  float* mu;       /* [S, arena]                                   */
  float* nu;       /* [S, arena]                                   */
  float* grads;    /* [S, arena] out: d(total_loss)/d(params)      */
  int32_t* count;  /* [1] optax count (pre-update value on entry)  */
  void* shadow;    /* bf16 operand copies for FQL_PRECISION_BF16_TC, fql_shadow_bytes() bytes; else NULL */
} FqlState;

#define FQL_NUM_INFO 13 /* order == fql_info_name(i); names of agents/fql.py:39-44,85-92 + flax_utils.py:151-157 */
#define FQL_NUM_RAW 16  /* raw per-rank accumulators, see fql_step_grads() */

typedef struct FqlContext FqlContext; /* owns internal streams/events/graphs; one per (thread, device) */

/* ---- library ------------------------------------------------------------------------------------------ */
int fql_version(void);
const char* fql_last_error(void);
const char* fql_info_name(int i);
int fql_context_create(FqlContext** out);
int fql_context_destroy(FqlContext* ctx);
long long fql_launch_count(FqlContext* ctx); /* kernels enqueued through ctx so far (graph replays included) */

/* ---- layout: replaces the pytree structure built by FQLAgent.create (agents/fql.py:205-242) ------------- */
int64_t fql_arena_floats(const FqlDims* d);                         /* floats per seed (leaves padded to 32) */
int fql_layout(const FqlDims* d, FqlLeaf* leaves, int32_t cap, int32_t* n_leaves);
size_t fql_workspace_bytes(const FqlDims* d);
size_t fql_shadow_bytes(const FqlDims* d);
size_t fql_forward_workspace_bytes(const FqlDims* d, int32_t rows); /* for the standalone forward entry points */

/* ---- the hot path: FQLAgent.update (agents/fql.py:122-133) ---------------------------------------------- */
/* Whole step on one rank: total_loss grads (fql.py:94-111 via flax_utils.py:137), grad stats (:139-157),
 * optax.adam apply (:120-130), Polyak from the pre-step critic (fql.py:113-120).  info: 13 floats (device). */
int fql_update_step(FqlContext* ctx, const FqlDims* d, const FqlHparams* hp, const FqlBatch* batch,
                    const FqlState* st, float* info, void* workspace, size_t ws_bytes, void* stream);
/* Data-parallel split of the same step.  fql_step_grads leaves d(loss)/d(params) for this rank's rows
 * (already divided by global_batch) in st->grads and FQL_NUM_RAW raw accumulators in `raw`
 * ([0..8] sums to all-reduce with SUM, [9] max, [10] -min to all-reduce with MAX); the caller all-reduces both,
 * then fql_step_apply does stats + Adam + Polyak and finalises info. */
int fql_step_grads(FqlContext* ctx, const FqlDims* d, const FqlHparams* hp, const FqlBatch* batch,
                   const FqlState* st, float* raw, void* workspace, size_t ws_bytes, void* stream);
int fql_step_apply(FqlContext* ctx, const FqlDims* d, const FqlHparams* hp, const FqlState* st, const float* raw,
                   float* info, void* workspace, size_t ws_bytes, void* stream);
/* Same as fql_step_apply on the ALL-GATHERED accumulators [ranks][S][FQL_NUM_RAW]: the SUM / MAX reduction over ranks happens in
 * the info kernel (no extra collectives or host-side reductions). */
int fql_step_apply_gathered(FqlContext* ctx, const FqlDims* d, const FqlHparams* hp, const FqlState* st, const float* raw_all,
                            int32_t ranks, float* info, void* workspace, size_t ws_bytes, void* stream);
/* Overlap hook for data parallelism: `event` (a cudaEvent_t, or NULL to disable) is recorded by fql_step_grads as soon as the
 * gradients of the first fql_early_grads_floats() floats of the arena (bc-flow actor + critic) are final, i.e. while the one-step
 * actor's backward is still running; the caller may start all-reducing that prefix on another stream behind the event. */
int fql_set_early_grads_event(FqlContext* ctx, void* event);
int64_t fql_early_grads_floats(const FqlDims* d);
/* ---- data parallel over NVLink peer memory (no NCCL on the step) --------------------------------------------
 * Every rank maps every rank's "symmetric" buffer (fql_dp_symmetric_bytes() bytes: [gradient arena S x arena floats | metric
 * gather | lam exchange | flags]) into its address space -- CUDA IPC / VMM peer mappings, plus the NVLS multicast mapping of the
 * same allocations when the fabric offers one (torch.distributed._symmetric_memory.rendezvous provides both; any allocator
 * that yields the pointers below works).  The caller zero-fills its buffer once, synchronises all ranks, and attaches.  From
 * then on fql_update_step / fql_total_loss on this context ARE the data-parallel step (FqlDims.global_batch = world x batch,
 * FqlState.grads must be base[rank]): as soon as a network's gradients are final, one kernel of this library reduces that
 * bucket across ranks -- rank r owns 1/world of it: multimem.ld_reduce through the switch (or loads from the world peer
 * mappings, summed in rank order) and multimem.st (or peer stores) of the sum back into every rank's arena -- overlapped with
 * the rest of the backward; the metric accumulators are gathered by the last bucket's kernel; config['normalize_q_loss'] gets its
 * global mean|q| (agents/fql.py:74-76) from a one-word-per-rank exchange inside the loss kernel.  Ranks synchronise through
 * release/acquire flags in the peer-mapped buffers; every rank applies the identical Adam / Polyak step (replicas stay
 * bit-identical, no parameter broadcast).  The whole step stays one CUDA graph. */
#define FQL_DP_MAX_RANKS 8
typedef struct FqlDpComm {
  int32_t rank, world;
  void* base[FQL_DP_MAX_RANKS]; /* this process's mapping of rank i's symmetric buffer; base[rank] is the local one */
  void* base_mc;                /* NVLS multicast mapping of the same buffers, or NULL (peer loads / stores are used instead) */
} FqlDpComm;
size_t fql_dp_symmetric_bytes(const FqlDims* d, int32_t world);
int fql_dp_attach(FqlContext* ctx, const FqlDims* d, const FqlDpComm* comm); /* comm == NULL detaches */
/* Stand-alone exchange: floats [off, off + n) of every seed's gradient arena are summed over the ranks, in place on every rank
 * (what an ncclAllReduce of that range would do; SURVEY 8e).  bucket in [0, 4) selects the flag set: launches that may be in
 * flight at the same time must use different buckets.  Enqueue-only; every rank calls it with the same arguments. */
int fql_dp_allreduce(FqlContext* ctx, int32_t bucket, int64_t off, int64_t n, void* stream);

/* Forward-only total_loss(grad_params=None) (agents/fql.py:94-111 as called from main.py:284): 10 info floats
 * [0..9] and the scalar loss in info[FQL_NUM_INFO-3] slot order documented in fql_info_name. */
int fql_total_loss(FqlContext* ctx, const FqlDims* d, const FqlHparams* hp, const FqlBatch* batch,
                   const FqlState* st, float* info, void* workspace, size_t ws_bytes, void* stream);

/* ---- pieces of the path, individually callable ---------------------------------------------------------- */
/* FQLAgent.sample_actions (agents/fql.py:135-153) with the noise draw explicit: out = clip(pi(obs, noise)). */
int fql_sample_actions(FqlContext* ctx, const FqlDims* d, const float* params, const void* shadow, const float* obs,
                       const float* noise, float* actions_out, int32_t rows, void* workspace, size_t ws_bytes, void* stream);
/* FQLAgent.compute_flow_actions (agents/fql.py:155-171): flow_steps Euler steps of actor_bc_flow, then clip. */
int fql_compute_flow_actions(FqlContext* ctx, const FqlDims* d, const float* params, const void* shadow, const float* obs,
                             const float* noise, float* actions_out, int32_t rows, void* workspace, size_t ws_bytes, void* stream);
/* One network forward (utils/networks.py MLP/Value/ActorVectorField __call__): x [S,rows,in] -> y [S,ens,rows,out]. */
int fql_mlp_forward(FqlContext* ctx, const FqlDims* d, int32_t net, const float* params, const float* x, float* y,
                    int32_t rows, void* workspace, size_t ws_bytes, void* stream);
/* FQLAgent.target_update(network, 'critic') (agents/fql.py:113-120) on its own: target_critic <- tau * critic + (1 - tau) * target_critic
 * in place in the parameter arena (fql_update_step already contains it, fused into the optimizer pass). */
int fql_target_update(const FqlDims* d, const FqlHparams* hp, float* params, void* shadow, void* stream);
/* Rebuild the bf16 operand shadow from fp32 params (after create()/restore; the step keeps it current itself). */
int fql_refresh_shadow(const FqlDims* d, const float* params, void* shadow, void* stream);

/* ---- either side of the path --------------------------------------------------------------------------- */
/* Dataset.sample gather + frame stack + random crop (utils/datasets.py:68-112, 17-33) on a device-resident
 * dataset.  idxs/init_idxs are int64 [B] drawn on the host (MT19937 order preserved); crop_from int64 [B,2] or
 * NULL.  elem_bytes: bytes of one scalar; row_elems: scalars per stored row (H*W*C for images); for images
 * (img_h>0) frames are concatenated on the channel axis and cropped with edge padding `pad`. */
int fql_gather_rows(const void* src, void* dst, const int64_t* idxs, int64_t n_idx, int64_t row_bytes, void* stream);
int fql_gather_frames(const uint8_t* obs_src, const uint8_t* next_src, uint8_t* obs_out, uint8_t* next_out,
                      const int64_t* idxs, const int64_t* init_idxs, const int64_t* crop_from, int64_t n_idx,
                      int32_t img_h, int32_t img_w, int32_t img_c, int32_t frame_stack, int32_t pad, void* stream);
/* Device noise for production runs (own Philox-4x32-10 generator; jax threefry streams are version-dependent,
 * SURVEY 8c): fills the five noise tensors of one update from (seed, step). */
int fql_fill_noise(const FqlDims* d, uint64_t seed, uint64_t step, float* z_next, float* x0, float* t, float* z,
                   float* z_metric, void* stream);
/* The same for a data-parallel rank holding rows [row_offset, row_offset + batch) of the global batch: the Philox counters are
 * indices into the GLOBAL [S][global_batch][A] tensors, so R ranks draw exactly the noise one device would draw for the global
 * batch (SURVEY 8e) and no two ranks share a row.  fql_fill_noise == row_offset 0 with global_batch == batch. */
int fql_fill_noise_rows(const FqlDims* d, uint64_t seed, uint64_t step, int64_t row_offset, float* z_next, float* x0, float* t,
                        float* z, float* z_metric, void* stream);


/* ---- diagnostics -------------------------------------------------------------------------------------- */
/* %globaltimer stamps taken at the schedule points of the last step when the context was created with FQL_B200_STAMPS=1
 * (profiles/dbg_timeline.py); fails otherwise.  Synchronises the device: not for the hot path. */
int fql_debug_stamps(FqlContext* ctx, unsigned long long* host_out, int n);

/* ---- 3x3 SAME convolutions of ImpalaEncoder (utils/encoders.py:17-57) on tcgen05, stand-alone -------------------------
 * x: bf16 NHWC [B,H,W,cin] (cin, cout in {16, 32}); w_hwio: fp32 [3,3,cin,cout] (nn.Conv kernel layout), rounded to bf16 for the
 * tensor cores; fp32 accumulation.  out = epilogue(conv(x) + bias): optional relu-mask of a saved bf16 tensor (mask > 0), optional
 * bf16 addend (skip connection / upstream gradient), optional relu; bf16 NHWC.  input_gradient != 0: x is dY [B,H,W,cout] and out
 * is dX [B,H,W,cin] (jax.grad of the same convolution with respect to its input).  The weight gradient returns fp32
 * gw [3,3,cin,cout] and gb [cout] (sums over all pixels, reduced in a fixed order).  These are the kernels FQL_PRECISION_BF16_ENC
 * runs inside fql_update_step; they are exported for exact arithmetic checks. */
size_t fql_conv3x3_workspace_bytes(void);
int fql_conv3x3_bf16(const void* x, const float* w_hwio, const float* bias, int32_t B, int32_t H, int32_t W, int32_t cin, int32_t cout,
                     int32_t input_gradient, const void* mask, const void* add, int32_t relu_out, void* out, void* workspace,
                     size_t ws_bytes, void* stream);
int fql_conv3x3_wgrad_bf16(const void* x, const void* dy, int32_t B, int32_t H, int32_t W, int32_t cin, int32_t cout, float* gw, float* gb,
                           void* workspace, size_t ws_bytes, void* stream);

/* ---- test hooks: the tensor-core MLP kernels of FQL_PRECISION_BF16_TC one at a time on caller buffers ---------------------------
 * Not used by the step; they exist so that each kernel can be compared with a reference on its own.  The arguments mean what they
 * mean inside the step (fql_b200/csrc/step.cuh: TcGemmSpec, and the row / column kernels of tc_path.cu); enqueue-only. */
typedef struct FqlTestOperand { /* bf16 TMA operand [g1][g0][rows][inner], pitches ld / s0 / s1 in elements */
  const void* ptr;
  int32_t inner, rows;
  int64_t ld;
  int32_t g0;
  int64_t s0;
  int32_t g1;
  int64_t s1;
} FqlTestOperand;
typedef struct FqlTestPtr {     /* epilogue tensor at base + g0 * s0 + g1 * s1 (elements of its own type), row pitch ld */
  void* base;
  int64_t s0, s1;
  int32_t ld;
} FqlTestPtr;
typedef struct FqlTestGemm {    /* D[M,N] = A[M,K] B[K,N] over G1 x G0 groups with the epilogue `mode` (TC_MODE_*) */
  int32_t mode, M, N, K, G0, G1, a_mn, b_mn, ksplit;
  FqlTestOperand A, B;
  FqlTestPtr bias, out_f, out_h, out_z, zin, act, xb, target, ln_s, ln_b, dbias, wmaster, dln_s, dln_b;
  int32_t F, Adim, step, n_steps, clip;
} FqlTestGemm;
int fql_test_tc_gemm(const FqlTestGemm* g, void* stream);
/* H = [LayerNorm](gelu(Z)) -> bf16 (+ mu / rstd when ln); Z fp32 [S][E][M][N] dense, scale / bias at s * par_s + e * par_e */
int fql_test_act_ln_bf16(const float* Z, const float* scale, const float* bias, int64_t par_s, int64_t par_e, void* Hb, float* mu,
                         float* rstd, int32_t M, int32_t N, int32_t S, int32_t E, int32_t ln, void* stream);
/* dZ = LayerNorm_bwd(dH; gelu(Z)) * gelu'(Z) (fp32 + bf16 copy); row r of group (s, e) of Z at (s * z_rows_s + e * z_rows_e + r) * N */
int fql_test_ln_bwd_bf16(const float* dH, const float* Z, const float* scale, int64_t scale_s, int64_t scale_e, float* dZ, void* dZb,
                         int32_t M, int32_t N, int32_t S, int32_t E, int64_t z_rows_e, int64_t z_rows_s, void* stream);
/* dZ = dH * gelu'(Z) (fp32 + bf16 copy), Z addressed as above */
int fql_test_gelu_bwd_bf16(const float* dH, const float* Z, float* dZ, void* dZb, int32_t M, int32_t N, int32_t S, int32_t E,
                           int64_t z_rows_e, int64_t z_rows_s, void* stream);
/* column sums of bf16 X [G][M][N] (N % 64 == 0) ADDED into out[g0 * out_stride_g0 + g1 * out_stride_g1 + n], g = g1 * G0 + g0 */
int fql_test_colsum_bf16(const void* X, int64_t G, int64_t M, int32_t N, float* out, int64_t out_stride_g0, int32_t G0,
                         int64_t out_stride_g1, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FQL_B200_H_ */
