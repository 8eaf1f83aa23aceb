// mlp_tc.cu -- what every tensor-core (FQL_PRECISION_BF16_TC) MLP kernel shares:
//   the bf16 shadow of the fp32 parameter arena, plus zero-padded [H][64] copies of the narrow last-layer kernels (the B operands);
//   bf16 first-layer operands, zero padded to a multiple of 64 columns (the A operands);
//   the TMA tensor maps; and tc_supported(), the shapes the tensor-core path implements.
// The MLPs themselves run in chain2_tc.cu (fused per-tile chains: hidden = 512, enough 128-row tiles to fill the GPU), in
// euler_cluster.cu (cluster kernels: hidden = 512, small batch) and otherwise layer by layer through tc_gemm (tc_path.cu), which
// is the only tensor-core route at hidden 64, 128 and 256.
#include "step.cuh"

#include <cuda_bf16.h>

namespace {

constexpr int MAX_A = 32;

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
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
