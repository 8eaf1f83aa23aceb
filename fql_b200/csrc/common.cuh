// common.cuh -- shared declarations of libfql_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/fql_b200.h"

#define FQL_MAXL 8   // max Dense layers per MLP
#define FQL_MAXP 3   // max problems batched into one grouped pass

void fql_set_error(const char* fmt, ...);

#define FQL_CHECK_CUDA(x)                                                                          \
  do {                                                                                             \
    cudaError_t e__ = (x);                                                                         \
    if (e__ != cudaSuccess) {                                                                      \
      fql_set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #x, cudaGetErrorString(e__));   \
      return 1;                                                                                    \
    }                                                                                              \
  } while (0)
extern thread_local long long g_fql_launches;  // kernels enqueued by this thread (diagnostics: fql_launch_count)
#define FQL_CHECK_LAUNCH()                 \
  do {                                     \
    g_fql_launches++;                      \
    FQL_CHECK_CUDA(cudaGetLastError());    \
  } while (0)
// Programmatic dependent launch for the small kernels that sit between the tensor-core GEMMs of a dependent chain: the kernel may
// be scheduled while its predecessor in the stream is still running; FQL_PDL_SYNC() (first statement that matters in the kernel)
// blocks until the predecessor's writes are visible and lets the successor start its own prologue.  Without the launch
// attribute both instructions are no-ops.
#define FQL_PDL_SYNC()                                             \
  do {                                                             \
    asm volatile("griddepcontrol.wait;" ::: "memory");             \
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); \
  } while (0)
inline bool fql_pdl_enabled() {
  static const bool on = []() {
    const char* e = getenv("FQL_B200_PDL");
    return !(e && e[0] == '0');
  }();
  return on;
}
template <typename... KArgs, typename... Args>
inline cudaError_t fql_launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = fql_pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
// cudaFuncSetAttribute / occupancy results are per DEVICE: caches of them are indexed by the current device (FQLAgent.create(device=...)
// may put a second GPU under the same process)
#define FQL_MAX_DEVICES 64
inline int fql_current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev >= 0 && dev < FQL_MAX_DEVICES ? dev : 0;
}
#define FQL_REQUIRE(cond, ...)       \
  do {                               \
    if (!(cond)) {                   \
      fql_set_error(__VA_ARGS__);    \
      return 1;                      \
    }                                \
  } while (0)
#define FQL_TRY(x)          \
  do {                      \
    int r__ = (x);          \
    if (r__) return r__;    \
  } while (0)

// ---------------------------------------------------------------------------------------------------------
// arena layout
// ---------------------------------------------------------------------------------------------------------
struct EncView {            // ImpalaEncoder('impala_small') leaves of one network (utils/encoders.py)
  int64_t off_cw[3][3], off_cb[3][3];  // stack_blocks_i / Conv_j kernel [3,3,cin,cout] and bias
  int64_t off_dw, off_db;              // MLP_0 / Dense_0 kernel [flat,512] and bias
};
struct NetView {
  int n_layers;           // Dense layers
  int in_dim, out_dim;    // first-layer fan-in, last-layer fan-out
  int hidden;
  int ens;                // 1 or 2
  int ln;                 // LayerNorm after each hidden activation
  int64_t off_w[FQL_MAXL], off_b[FQL_MAXL], off_lns[FQL_MAXL], off_lnb[FQL_MAXL];
  int has_enc;
  EncView enc;
  int64_t begin, end;     // float range of this network inside one seed's arena
  __host__ __device__ int k_of(int l) const { return l == 0 ? in_dim : hidden; }
  __host__ __device__ int n_of(int l) const { return l == n_layers - 1 ? out_dim : hidden; }
};
#define FQL_LEAF_PAD 1024  // every leaf is padded to a multiple of this many floats: one optimizer CTA = one leaf
#define FQL_MAX_LEAVES 160
struct Layout {
  NetView net[FQL_NUM_NETS];
  int64_t arena;                       // floats per seed
  int n_leaves;
  int leaf_blk[FQL_MAX_LEAVES + 1];    // first FQL_LEAF_PAD-block of each leaf (arena order); [n_leaves] = total blocks
  int leaf_net[FQL_MAX_LEAVES];
};
int fql_build_layout(const FqlDims* d, Layout* L);
int fql_validate_dims(const FqlDims* d);

// ---------------------------------------------------------------------------------------------------------
// grouped operand addressing: group g = (problem p, seed s, head e), g = (p*S + s)*E + e
// ---------------------------------------------------------------------------------------------------------
struct GPtr {             // read-only operand selected per group
  const float* base[FQL_MAXP];
  int64_t stride_s, stride_e;
  __device__ __forceinline__ const float* at(int p, int s, int e) const {
    return base[p] + (int64_t)s * stride_s + (int64_t)e * stride_e;
  }
};
struct GPtrW {            // writable operand selected per group
  float* base[FQL_MAXP];
  int64_t stride_s, stride_e;
  __device__ __forceinline__ float* at(int p, int s, int e) const {
    return base[p] ? base[p] + (int64_t)s * stride_s + (int64_t)e * stride_e : nullptr;
  }
};

// C[M,N] = opA(A)[M,K] * opB(B)[K,N] (+ epilogue), one problem per blockIdx.z
struct GemmArgs {
  GPtr A, B, bias, mulz;  // bias: [N] added to acc (optional); mulz: [M,N] pre-activation, acc *= gelu'(mulz) (optional)
  GPtrW out_pre, out;     // out_pre: acc(+bias) before activation (optional); out: final
  int M, N, K;
  int lda, ldb, ldo, ld_mulz, ld_pre;
  int trans_a, trans_b;   // trans_a: A stored [K,M]; trans_b: B stored [N,K]
  int act_gelu;           // out = gelu(acc+bias)
  int S, E;               // seeds, heads (groups = P*S*E)
  int P;
  int tf32x3;             // FQL_PRECISION_FP32_TC: 3xTF32 on tcgen05 (gemm_tf32x3.cu) instead of FFMA
};
int launch_gemm(const GemmArgs& a, cudaStream_t st);
int launch_gemm_tf32x3(const GemmArgs& a, cudaStream_t st);

// rows kernel: H = LN(gelu(Z)) (or just gelu), per group scale/bias
struct ActLnArgs {
  GPtr Z, scale, lnbias;
  GPtrW H, mu, rstd;      // mu/rstd optional ([M] per group)
  int M, N, ld;
  int ln;
  int P, S, E;
};
int launch_act_ln_fwd(const ActLnArgs& a, cudaStream_t st);

// rows kernel: dZ = LNbwd(dH; Z) * gelu'(Z)
struct ActLnBwdArgs {
  GPtr dH, Z, scale;
  GPtrW dZ;
  int M, N, ld;
  int P, S, E;
};
int launch_act_ln_bwd(const ActLnBwdArgs& a, cudaStream_t st);

// column reductions over rows: out0[c] = sum_r X[r,c] (* xhat(Z)[r,c] if Z given -> LN scale grad)
struct ColSumArgs {
  GPtr X, Z;              // Z optional: multiply by xhat recomputed from Z rows (needs mu/rstd)
  GPtr mu, rstd;
  GPtrW out;              // [N]
  int M, N, ld;
  int P, S, E;
};
int launch_colsum(const ColSumArgs& a, cudaStream_t st, float* scratch = nullptr, size_t scratch_floats = 0);

// ---------------------------------------------------------------------------------------------------------
// device math shared by every kernel (must match oracle/fql_oracle.py gelu_tanh / gelu_tanh_grad)
// ---------------------------------------------------------------------------------------------------------
#define FQL_GELU_C 0.7978845608028654f
#define FQL_GELU_A 0.044715f
#define FQL_LN_EPS 1e-6f

__device__ __forceinline__ float gelu_tanh_f(float x) {
  float u = FQL_GELU_C * (x + FQL_GELU_A * x * x * x);
  return 0.5f * x * (1.0f + tanhf(u));
}
__device__ __forceinline__ float gelu_tanh_grad_f(float x) {
  float x2 = x * x;
  float u = FQL_GELU_C * (x + FQL_GELU_A * x2 * x);
  float th = tanhf(u);
  float du = FQL_GELU_C * (1.0f + 3.0f * FQL_GELU_A * x2);
  return 0.5f * (1.0f + th) + 0.5f * x * (1.0f - th * th) * du;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
static inline int64_t round_up64(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
