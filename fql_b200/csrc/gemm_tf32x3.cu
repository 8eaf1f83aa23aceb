// gemm_tf32x3.cu -- the GemmArgs grouped GEMM (gemm_simt.cu) on tcgen05 tensor cores with 3xTF32 operand splitting: the
// FQL_PRECISION_FP32_TC arithmetic of every Dense contraction of the MLP passes.
//
//   x ~= hi + lo,  hi = cvt.rna.tf32(x) (11 significant bits),  lo = cvt.rna.tf32(x - hi)  (x - hi is exact in fp32, |.| <= 2^-11 |x|)
//   A B ~= A_lo B_hi + A_hi B_lo + A_hi B_hi          (A_lo B_lo, <= 2^-22 |A||B| per product, is dropped)
//
// lo is rounded to tf32 as well, so the tensor core reads both halves exactly: what x - hi loses is <= 2^-11 |x - hi| <= 2^-22 |x|
// and, rounded to nearest, has no sign bias (a tf32 view of an fp32 lo would truncate, with the same sign for every element).
//
// The tensor core's fp32 accumulation is the larger error: every MMA that adds into an accumulator costs up to ~2^-23 of the
// accumulator's magnitude, with a consistent sign (measured on a B200: one accumulator taking all three products of every k-step
// ended 4.6e-7 of sum |a b| off at K = 64 and 1.8e-6 at K = 16384, 3-17x the FFMA kernel, and a B = 4096 backward pass 1.2e-5 off on a
// bias gradient).  So the adds are spread: hi.hi of k-step j goes to main accumulator j (of NMAIN = 4), the two small products to a
// correction accumulator of their own (their rounding is relative to a sum 2^-11 smaller), and the epilogue adds the eight partial
// tiles in fp32 in a fixed order.  Each main accumulator takes one MMA per 32 of K instead of three per 8.
//
// One CTA computes a 128 x 64 output tile of one group (p, s, e):
//   warps 0-7   producers: fp32 from global memory (any pitch, either orientation, out-of-range elements zero) -> hi / lo ->
//               K-major SWIZZLE_128B tiles in shared memory (32 fp32 = one 128-byte row per output row).  Warps 0-3 fill the even
//               K blocks, warps 4-7 the odd ones, so two blocks' global loads are in flight at once.  Plain loads rather than TMA:
//               the operands have row pitches such as 38 floats that TMA cannot address, and the producer has to split them anyway.
//   warp 8      TMEM allocation and the MMA issuer (warp-uniform, the instruction predicated on elect.sync).
//   warps 0-7   epilogue: TMEM -> shared memory -> (split-K: fixed-order sum over the cluster through DSMEM) -> the epilogue of
//               gemm_kernel in the same order (+bias, out_pre, *gelu'(mulz), gelu, out) with coalesced global stores.
// Split-K (weight gradients: K = batch, few output tiles): the K blocks are spread over a cluster of R CTAs along blockIdx.z and
// rank r sums the partial tiles of ranks 0..R-1 in that order for 1/R of the tile: deterministic, no atomics, no workspace.
#include "common.cuh"
#include "tc_prims.cuh"

using namespace tc;

namespace {

constexpr int BM = 128, BN = 64, BK = 32;
constexpr int A_TILE = BM * BK * 4;                  // 16 KB (hi or lo)
constexpr int B_TILE = BN * BK * 4;                  //  8 KB
constexpr int STAGE = 2 * A_TILE + 2 * B_TILE;       // A_hi | A_lo | B_hi | B_lo = 48 KB
constexpr int NSTAGE = 4;
constexpr int NPROD = 256;                           // producer / epilogue threads (warps 0-7), two groups of 128
constexpr int NTHREADS = NPROD + 32;                 // + MMA warp
constexpr int RED_LD = BN + 1;                       // row pitch (floats) of the partial tile in shared memory
constexpr int SMEM_BYTES = NSTAGE * STAGE + 1024 + 256;
constexpr int MAX_SPLIT = 8;                         // portable cluster size
constexpr int NMAIN = BK / 8;                        // main (hi.hi) accumulators, one per k-step of a K block; as many correction ones
constexpr int TMEM_COLS = 2 * NMAIN * BN;            // 512: all of TMEM (one CTA per SM: the operand ring takes 193 KB of shared memory)
static_assert(BM * RED_LD * 4 <= NSTAGE * STAGE, "the partial tile reuses the operand ring");

// instruction descriptor, kind::tf32: A/B TF32, D F32, both K-major (PTX ISA, tcgen05 instruction descriptor)
constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

// One 32-deep K block = four k-steps of 8 from ONE asm block (the descriptors advance by 32 bytes per k-step inside the swizzle atom,
// so ptxas materialises the uniform-register operands once, see umma_bf16_x4).  k-step j puts hi.hi into main accumulator j and
// lo.hi + hi.lo into correction accumulator NMAIN + j (TMEM columns 64 x slot).
__device__ __forceinline__ void umma_tf32x3_k32(uint32_t d, uint64_t ahi, uint64_t alo, uint64_t bhi, uint64_t blo, uint32_t acc_first) {
#define FQL_X3_STEP(J)                                                                                                       \
  "add.u64 ah, %1, 2*" #J ";\n\tadd.u64 al, %2, 2*" #J ";\n\tadd.u64 bh, %3, 2*" #J ";\n\tadd.u64 bl, %4, 2*" #J ";\n\t" \
  "add.u32 dm, %0, 64*" #J ";\n\tadd.u32 dl, %0, 256+64*" #J ";\n\t"                                                      \
  "tcgen05.mma.cta_group::1.kind::tf32 [dm], ah, bh, %5, p;\n\t"                                                          \
  "tcgen05.mma.cta_group::1.kind::tf32 [dl], al, bh, %5, p;\n\t"                                                          \
  "tcgen05.mma.cta_group::1.kind::tf32 [dl], ah, bl, %5, q;\n\t"
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 ah, al, bh, bl;\n\t.reg .b32 dm, dl;\n\t"
      "setp.ne.b32 p, %6, 0;\n\tsetp.eq.b32 q, 0, 0;\n\t"
      FQL_X3_STEP(0) FQL_X3_STEP(1) FQL_X3_STEP(2) FQL_X3_STEP(3)
      "}\n"
      ::"r"(d), "l"(ahi), "l"(alo), "l"(bhi), "l"(blo), "r"(IDESC), "r"(acc_first)
      : "memory");
#undef FQL_X3_STEP
}

__device__ __forceinline__ float tf32_hi(float x) {
  uint32_t h;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(x));
  return __uint_as_float(h);
}

// Global loads of one operand tile: R rows (M or N) x BK k, element (r, k) at src[r * rs + k * ks].  Item i of thread t covers four
// consecutive k of one row (one 16-byte chunk of the swizzled row).  Items are ordered so that a warp's loads are coalesced: along k
// when k is contiguous in memory (rs = ld), along rows when rows are (ks = ld).
template <int R>
struct TileLoad {
  static constexpr int ITEMS = R * (BK / 4) / 128;
  float v[ITEMS][4];
  __device__ __forceinline__ static void item(int i, bool kmaj, int& r, int& c) {
    if (kmaj) { c = i & 7; r = i >> 3; }
    else { r = i % R; c = i / R; }
  }
  __device__ __forceinline__ void load(const float* __restrict__ src, int64_t rs, int64_t ks, bool kmaj, int rows_left, int k_left, int t) {
#pragma unroll
    for (int u = 0; u < ITEMS; u++) {
      int r, c;
      item(t + 128 * u, kmaj, r, c);
      const float* p = src + (int64_t)r * rs + (int64_t)(c * 4) * ks;
#pragma unroll
      for (int j = 0; j < 4; j++) v[u][j] = (r < rows_left && c * 4 + j < k_left) ? __ldg(p + (int64_t)j * ks) : 0.f;
    }
  }
  __device__ __forceinline__ void store(uint8_t* hi, uint8_t* lo, bool kmaj, int t) const {
#pragma unroll
    for (int u = 0; u < ITEMS; u++) {
      int r, c;
      item(t + 128 * u, kmaj, r, c);
      float h[4], l[4];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        h[j] = tf32_hi(v[u][j]);
        l[j] = tf32_hi(v[u][j] - h[j]);
      }
      const uint32_t o = sw128_off((uint32_t)r, (uint32_t)c);
      *reinterpret_cast<float4*>(hi + o) = make_float4(h[0], h[1], h[2], h[3]);
      *reinterpret_cast<float4*>(lo + o) = make_float4(l[0], l[1], l[2], l[3]);
    }
  }
};

__global__ void __launch_bounds__(NTHREADS, 1) gemm_tf32x3_kernel(const GemmArgs a, int split) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NSTAGE * STAGE);
  uint64_t* full = bars;
  uint64_t* empty = bars + NSTAGE;
  uint64_t* acc_full = bars + 2 * NSTAGE;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NSTAGE + 1);
  float* red = reinterpret_cast<float*>(smem);  // [BM][RED_LD] partial tile, after the last MMA has read the ring

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
  const int g = blockIdx.z / split, kz = blockIdx.z % split;   // cluster (1, 1, split): kz is the CTA's rank in it
  const int e = g % a.E, s = (g / a.E) % a.S, p = g / (a.E * a.S);
  const int nkb_all = (a.K + BK - 1) / BK;
  const int kb0 = (int)((int64_t)nkb_all * kz / split), kb1 = (int)((int64_t)nkb_all * (kz + 1) / split);
  const int nkb = kb1 - kb0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTAGE; i++) {
      mbar_init(&full[i], 128);
      mbar_init(&empty[i], 1);
    }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 8) {
    // ---------------- producers: group pg fills K blocks pg, pg + 2, ... ----------------
    const int pg = warp >> 2, t = threadIdx.x & 127;
    const float* __restrict__ A = a.A.at(p, s, e);
    const float* __restrict__ B = a.B.at(p, s, e);
    // A element (m, k): trans_a ? A[k * lda + m] : A[m * lda + k];  B element (n, k): trans_b ? B[n * ldb + k] : B[k * ldb + n]
    const bool a_km = !a.trans_a, b_km = a.trans_b;
    const int64_t a_rs = a_km ? a.lda : 1, a_ks = a_km ? 1 : a.lda;
    const int64_t b_rs = b_km ? a.ldb : 1, b_ks = b_km ? 1 : a.ldb;
    TileLoad<BM> la;
    TileLoad<BN> lb;
    for (int kb = pg; kb < nkb; kb += 2) {
      const int st = kb % NSTAGE;
      const int k0 = (kb0 + kb) * BK;
      la.load(A + (int64_t)m0 * a_rs + (int64_t)k0 * a_ks, a_rs, a_ks, a_km, a.M - m0, a.K - k0, t);
      lb.load(B + (int64_t)n0 * b_rs + (int64_t)k0 * b_ks, b_rs, b_ks, b_km, a.N - n0, a.K - k0, t);
      if (kb >= NSTAGE) mbar_wait(&empty[st], ((kb / NSTAGE) - 1) & 1);
      uint8_t* sa = smem + st * STAGE;
      la.store(sa, sa + A_TILE, a_km, t);
      lb.store(sa + 2 * A_TILE, sa + 2 * A_TILE + B_TILE, b_km, t);
      fence_proxy_async_smem();
      mbar_arrive(&full[st]);
    }
  } else {
    // ---------------- MMA issuer ----------------
    const bool el = elect_one();
    const uint64_t d0 = make_smem_desc(smem_u32(smem), 16, 1024);
    const uint32_t tacc = __shfl_sync(0xffffffffu, tmem_base, 0);
    int st = 0;
    uint32_t ph = 0;
    for (int kb = 0; kb < nkb; kb++) {
      mbar_wait_u(&full[st], ph);
      tc_fence_after();
      if (el) {
        const uint64_t ds = d0 + (uint64_t)(st * (STAGE >> 4));
        umma_tf32x3_k32(tacc, ds, ds + (A_TILE >> 4), ds + (2 * A_TILE >> 4), ds + ((2 * A_TILE + B_TILE) >> 4), kb != 0);
        umma_commit(&empty[st]);
      }
      if (++st == NSTAGE) { st = 0; ph ^= 1; }
    }
    if (el) umma_commit(acc_full);
  }

  // ---------------- accumulator -> shared memory ----------------
  if (warp < 8) {
    const int q = warp & 3, h = warp >> 2;
    const int row = q * 32 + lane;
    mbar_wait(acc_full, 0);
    tc_fence_after();
    // (m0 + m1) + (m2 + m3) + ((c0 + c1) + (c2 + c3)): main accumulators in slots 0-3, correction accumulators in slots 4-7
    const uint32_t t0 = tmem_base + ((uint32_t)(q * 32) << 16) + h * 32;
    float sum[2][32];
#pragma unroll
    for (int half = 0; half < 2; half++) {
      float pair[2][32];
#pragma unroll
      for (int pr = 0; pr < 2; pr++) {
        uint32_t x[32], y[32];
        tmem_ld32(t0 + (uint32_t)((half * NMAIN + 2 * pr) * BN), x);
        tmem_ld32(t0 + (uint32_t)((half * NMAIN + 2 * pr + 1) * BN), y);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; i++) pair[pr][i] = __uint_as_float(x[i]) + __uint_as_float(y[i]);
      }
#pragma unroll
      for (int i = 0; i < 32; i++) sum[half][i] = pair[0][i] + pair[1][i];
    }
    float* dst = red + row * RED_LD + h * 32;
#pragma unroll
    for (int i = 0; i < 32; i++) dst[i] = sum[0][i] + sum[1][i];
  }
  tc_fence_before();
  if (split > 1) cluster_sync_all();
  else __syncthreads();

  // ---------------- fixed-order reduction over the cluster + the epilogue of gemm_kernel ----------------
  if (warp < 8) {
    const uint32_t lbase = smem_u32(red);
    const float* __restrict__ bias = a.bias.base[p] ? a.bias.at(p, s, e) : nullptr;
    const float* __restrict__ mulz = a.mulz.base[p] ? a.mulz.at(p, s, e) : nullptr;
    float* __restrict__ out_pre = a.out_pre.at(p, s, e);
    float* __restrict__ out = a.out.at(p, s, e);
    const int part = BM * BN / split;
    for (int idx = kz * part + (int)threadIdx.x; idx < (kz + 1) * part; idx += NPROD) {
      const int row = idx / BN, col = idx % BN;
      const int gm = m0 + row, gn = n0 + col;
      if (gm >= a.M || gn >= a.N) continue;
      const uint32_t off = (uint32_t)(row * RED_LD + col) * 4u;
      float v;
      if (split == 1) {
        v = red[row * RED_LD + col];
      } else {
        v = 0.f;
#pragma unroll
        for (int i = 0; i < MAX_SPLIT; i++) {
          if (i < split) {
            uint32_t ra;
            float x;
            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(lbase + off), "r"(i));
            asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(x) : "r"(ra) : "memory");
            v += x;
          }
        }
      }
      if (bias) v += bias[gn];
      if (out_pre) out_pre[(int64_t)gm * a.ld_pre + gn] = v;
      if (mulz) v *= gelu_tanh_grad_f(mulz[(int64_t)gm * a.ld_mulz + gn]);
      if (a.act_gelu) v = gelu_tanh_f(v);
      if (out) out[(int64_t)gm * a.ldo + gn] = v;
    }
  }
  if (split > 1) cluster_sync_all();  // no CTA leaves while a peer may still read its partial tile
  else __syncthreads();
  tc_fence_after();
  if (warp == 8) tmem_dealloc(tmem_base, TMEM_COLS);
}

}  // namespace

int launch_gemm_tf32x3(const GemmArgs& a, cudaStream_t st) {
  if (a.M <= 0 || a.N <= 0) return 0;
  FQL_REQUIRE(a.K >= 1, "gemm_tf32x3: K=%d", a.K);
  const int G = a.P * a.S * a.E;
  static int sms[FQL_MAX_DEVICES] = {};
  static bool attr_set[FQL_MAX_DEVICES] = {};
  const int dev = fql_current_device();
  if (!attr_set[dev]) {
    FQL_CHECK_CUDA(cudaFuncSetAttribute(gemm_tf32x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    FQL_CHECK_CUDA(cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev));
    attr_set[dev] = true;
  }
  // Split K over a cluster while the output tiles leave SMs idle and every split keeps at least 4 K blocks (128 of K).
  const int64_t tiles = (int64_t)((a.M + BM - 1) / BM) * ((a.N + BN - 1) / BN) * G;
  const int nkb = (a.K + BK - 1) / BK;
  int split = 1;
  while (split < MAX_SPLIT && tiles * split < sms[dev] && nkb >= 8 * split) split *= 2;
  FQL_REQUIRE((a.M + BM - 1) / BM <= 65535 && (int64_t)G * split <= 65535, "gemm_tf32x3: grid too large (M=%d, %d groups)", a.M, G);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((a.N + BN - 1) / BN, (a.M + BM - 1) / BM, G * split);
  cfg.blockDim = dim3(NTHREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = split;
  cfg.attrs = attr;
  cfg.numAttrs = split > 1 ? 1 : 0;
  FQL_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_tf32x3_kernel, a, split));
  FQL_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// test hook: launch_gemm on caller buffers in the arithmetic of `precision`
// ---------------------------------------------------------------------------------------------------------
extern "C" int fql_test_gemm_f32(const FqlTestGemmF32* t, int32_t precision, void* stream) {
  FQL_REQUIRE(t != nullptr, "fql_test_gemm_f32: spec is NULL");
  FQL_REQUIRE(precision == FQL_PRECISION_FP32 || precision == FQL_PRECISION_FP32_TC, "fql_test_gemm_f32: precision %d (FP32 or FP32_TC)", precision);
  FQL_REQUIRE(t->P >= 1 && t->P <= FQL_MAXP && t->S >= 1 && t->E >= 1 && t->M >= 1 && t->N >= 1 && t->K >= 1,
              "fql_test_gemm_f32: P=%d S=%d E=%d M=%d N=%d K=%d", t->P, t->S, t->E, t->M, t->N, t->K);
  GemmArgs a;
  memset(&a, 0, sizeof(a));
  auto ro = [&](GPtr& d, const FqlTestGPtr& g) {
    for (int i = 0; i < FQL_MAXP; i++) d.base[i] = reinterpret_cast<const float*>(g.base[i]);
    d.stride_s = g.stride_s; d.stride_e = g.stride_e;
  };
  auto rw = [&](GPtrW& d, const FqlTestGPtr& g) {
    for (int i = 0; i < FQL_MAXP; i++) d.base[i] = reinterpret_cast<float*>(const_cast<void*>(g.base[i]));
    d.stride_s = g.stride_s; d.stride_e = g.stride_e;
  };
  ro(a.A, t->A); ro(a.B, t->B); ro(a.bias, t->bias); ro(a.mulz, t->mulz);
  rw(a.out_pre, t->out_pre); rw(a.out, t->out);
  for (int i = 0; i < t->P; i++) FQL_REQUIRE(a.A.base[i] && a.B.base[i], "fql_test_gemm_f32: A / B of problem %d is NULL", i);
  a.M = t->M; a.N = t->N; a.K = t->K;
  a.lda = t->lda; a.ldb = t->ldb; a.ldo = t->ldo; a.ld_mulz = t->ld_mulz; a.ld_pre = t->ld_pre;
  a.trans_a = t->trans_a; a.trans_b = t->trans_b; a.act_gelu = t->act_gelu;
  a.S = t->S; a.E = t->E; a.P = t->P;
  a.tf32x3 = precision == FQL_PRECISION_FP32_TC;
  return launch_gemm(a, reinterpret_cast<cudaStream_t>(stream));
}
