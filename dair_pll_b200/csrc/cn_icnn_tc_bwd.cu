// Weight gradients of the support-function network (backward of HomogeneousICNN.forward,
// dair_pll/deep_support_function.py:238-266) on the tensor cores, for the rows of a batch that carry a cotangent.
//
// With the slope masks m0 (layer 0) and m1 (layer 1) of the visited rows constant, every weight gradient of
// L = sum_r gp[r] . p[r] follows from three (W x W) matrices and two (3 x W) vectors (dair_pll_b200/deep_support_function.py):
//   C_k[j,i] = sum_r gp_k[r] m0[r,j] m1[r,i]            g1[k,i] = sum_r gp_k[r] m1[r,i]
//   G[j,i] = sum_k Wd0[k,j] C_k[j,i]     gWd0[k,j] = sum_i |wout|_i |Wh|[j,i] C_k[j,i]
// and with m = s + (1 - s) b (b the mask BIT, s the LeakyReLU slope)
//   C_k = s^2 S_k + s (1 - s) (R0_k[j] + R1_k[i]) + (1 - s)^2 N_k[j,i],        g1[k,i] = s S_k + (1 - s) R1_k[i]
//   N_k[j,i] = sum_r gp_k[r] b0[r,j] b1[r,i]    R0_k[j] = sum_r gp_k[r] b0[r,j]    R1_k[i] = sum_r gp_k[r] b1[r,i]    S_k = sum_r gp_k[r].
// N_k is the only contraction of size rows x W x W.  gp_k[r] splits exactly into TCB_NS balanced base-128 int8 digits of
// a power-of-two scale per coordinate (56-bit fixed point: 14 bits of headroom for outlier rows on top of the 42 bits the
// forward works with), so each digit plane of N_k is an int8 x int8 -> int32 product of
//   A[j][r] = digit[r] AND m0t[j][r]   (m0t = layer-0 bits as bytes 0x00 / 0xFF, transposed: K-major)   and   B[i][r] = m1t[i][r]  (0 / 1),
// two planes per accumulator through the -128 copy of B, exactly as in the forward kernel (cn_icnn_tc.cuh).  Integer
// accumulation is exact and order independent: the result does not depend on how the rows are chunked.
//
// No host read anywhere: the row count is a device scalar (the compaction is torch.nonzero_static), every grid is fixed.
//   dpll_icnn_tc_bwd_digits_f64    digit planes of gp (rows beyond the count: zero)
//   dpll_icnn_tc_bwd_sums_f64      R0, R1, S (CUDA cores, fixed summation order)
//   dpll_icnn_tc_bwd_gram_f64      N_k partial accumulators: CTA = (output block of 128 x 256, row chunk), tcgen05.mma M 128 N 256
//   dpll_icnn_tc_bwd_finish_f64    chunks and planes -> C_k (3, W, W) in fp64
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/dair_pll_b200.h"
#include "cn_icnn_tc.cuh"
#include "cn_launch.cuh"

namespace {

using namespace cn;

constexpr int TCB_NS = 8;                       // digit planes of the cotangent (56-bit fixed point per coordinate)
constexpr int TCB_NT = TCB_NS / 2;              // plane pairs = accumulators per (coordinate, output block)
constexpr int TCB_BLOCKS = 3 * TCB_NT * 2;      // (k, pair, half of the j range): 24 output blocks of 128 x 256
constexpr int TCB_CHUNKS = 6;                   // row chunks: 24 x 6 = 144 CTAs
constexpr int kStageRows = 128;                 // K bytes per pipeline stage
constexpr int kGramThreads = 256;
constexpr int kOffAhi = 0, kOffAlo = 16384, kOffBlo = 32768, kOffBhi = 65536, kStageBytes = 98304;
constexpr int kGramSmem = 2 * kStageBytes + 64;
// instruction descriptor, kind::i8, M 128, N 256
constexpr uint32_t kIdescGram = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  for (uint32_t spin = 0; spin < (1u << 22); ++spin) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) return;
  }
  __trap();
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 rx;\n"
      ".reg .pred px;\n"
      "elect.sync rx|px, %1;\n"
      "@px mov.s32 %0, 1;\n"
      "}\n"
      : "+r"(pred)
      : "r"(0xffffffffu));
  return pred != 0;
}
// K-major, no swizzle, 128 K-bytes per row: LBO 128 B, SBO 1024 B
__device__ __forceinline__ uint64_t umma_desc128(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(128u >> 4) << 16) | ((uint64_t)(1024u >> 4) << 32) |
         ((uint64_t)1 << 46);
}
__device__ __forceinline__ void umma_i8_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(kIdescGram), "r"(accumulate), "r"(0), "r"(0), "r"(0), "r"(0)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, int32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, "
      "%18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ int64_t round_up128(int64_t n) { return (n + 127) & ~(int64_t)127; }

// balanced base-128 digits of g / 2^e (|g| <= 2^e), most significant first, stored with the even planes negated
__device__ __forceinline__ void cotangent_digits(double g, int e, int8_t* dig) {
  long long I = llrint(ldexp(g, 7 * TCB_NS - 1 - e));
#pragma unroll
  for (int s = TCB_NS - 1; s >= 1; --s) {
    const int dd = (int)((I + 64) & 127) - 64;
    dig[s] = (int8_t)((s & 1) ? dd : -dd);
    I = (I - dd) >> 7;
  }
  dig[0] = (int8_t)(-I);
}

// digit planes dw[k][s][row] (row stride ldk) of the gathered cotangent gp (capacity, 3); amax (3) = max |gp_k|
__global__ void bwd_digits_kernel(const double* __restrict__ gp, const int64_t* __restrict__ n_ptr, const double* __restrict__ amax,
                                  int64_t ldk, int8_t* __restrict__ dw) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= ldk) return;
  const bool live = r < *n_ptr;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    int8_t dig[TCB_NS];
    int e = 0;
    const double m = amax[k];
    if (m > 0) (void)frexp(m, &e);                     // m = f 2^e, f in [0.5, 1): |g| < 2^e
    cotangent_digits(live ? gp[3 * r + k] : 0.0, e, dig);
#pragma unroll
    for (int s = 0; s < TCB_NS; ++s) dw[((int64_t)(k * TCB_NS + s)) * ldk + r] = dig[s];
  }
}

// sums[0..3W) = R0_k[j], [3W..6W) = R1_k[i], [6W..6W+3) = S_k.  Block x < 2W: one mask row; block 2W: S.
__global__ void __launch_bounds__(256)
bwd_sums_kernel(const double* __restrict__ gp, const int64_t* __restrict__ n_ptr, const uint8_t* __restrict__ m0t,
                const uint8_t* __restrict__ m1t, int64_t ldk, double* __restrict__ sums) {
  __shared__ double red[3][256];
  const int64_t n = *n_ptr;
  const int row = blockIdx.x;
  const uint8_t* mask = row < TC_W ? m0t + (int64_t)row * ldk : (row < 2 * TC_W ? m1t + (int64_t)(row - TC_W) * ldk : nullptr);
  double a0 = 0, a1 = 0, a2 = 0;
  for (int64_t r = threadIdx.x; r < n; r += blockDim.x) {
    if (!mask || mask[r]) { a0 += gp[3 * r]; a1 += gp[3 * r + 1]; a2 += gp[3 * r + 2]; }
  }
  red[0][threadIdx.x] = a0; red[1][threadIdx.x] = a1; red[2][threadIdx.x] = a2;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o)
      for (int k = 0; k < 3; ++k) red[k][threadIdx.x] += red[k][threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x < 3) {
    const int k = threadIdx.x;
    if (row < TC_W) sums[k * TC_W + row] = red[k][0];
    else if (row < 2 * TC_W) sums[3 * TC_W + k * TC_W + (row - TC_W)] = red[k][0];
    else sums[6 * TC_W + k] = red[k][0];
  }
}

// partial[chunk][block][j (128)][i (256)] int32
__global__ void __launch_bounds__(kGramThreads, 1)
bwd_gram_kernel(const int64_t* __restrict__ n_ptr, const uint8_t* __restrict__ m0t, const uint8_t* __restrict__ m1t,
                const int8_t* __restrict__ dw, int64_t ldk, int32_t* __restrict__ partial) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * kStageBytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 2 * kStageBytes + 32);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int ob = blockIdx.x % TCB_BLOCKS, rc = blockIdx.x / TCB_BLOCKS;
  const int half = ob & 1, t = (ob >> 1) % TCB_NT, k = ob / (2 * TCB_NT);
  if (tid == 0) {
    mbar_init(smem_u32(&bars[0]), 1);
    mbar_init(smem_u32(&bars[1]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(256u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int64_t n128 = round_up128(*n_ptr);
  const int64_t per = round_up128((n128 + TCB_CHUNKS - 1) / TCB_CHUNKS);
  const int64_t r_begin = rc * per < n128 ? rc * per : n128;
  const int64_t r_end = r_begin + per < n128 ? r_begin + per : n128;
  const int nstages = (int)((r_end - r_begin) / kStageRows);

  const int c16 = tid & 7;                                  // this thread's 16-byte K chunk of every operand row
  const int8_t* dhi = dw + (int64_t)(k * TCB_NS + 2 * t) * ldk;
  const int8_t* dlo = dw + (int64_t)(k * TCB_NS + 2 * t + 1) * ldk;
  const uint8_t* m0 = m0t + (int64_t)(half * 128) * ldk;
  for (int st = 0; st < nstages; ++st) {
    const int buf = st & 1;
    uint8_t* sb = smem + buf * kStageBytes;
    if (st >= 2) mbar_wait(smem_u32(&bars[buf]), (uint32_t)((st >> 1) - 1) & 1u);     // the MMAs that read this buffer are done
    const int64_t r0 = r_begin + (int64_t)st * kStageRows + 16 * c16;
    const uint4 ghi = *reinterpret_cast<const uint4*>(dhi + r0);
    const uint4 glo = *reinterpret_cast<const uint4*>(dlo + r0);
#pragma unroll 4
    for (int j = tid >> 3; j < 128; j += kGramThreads / 8) {
      const uint4 m = *reinterpret_cast<const uint4*>(m0 + (int64_t)j * ldk + r0);
      const int off = (j >> 3) * 1024 + c16 * 128 + (j & 7) * 16;
      *reinterpret_cast<uint4*>(sb + kOffAhi + off) = make_uint4(m.x & ghi.x, m.y & ghi.y, m.z & ghi.z, m.w & ghi.w);
      *reinterpret_cast<uint4*>(sb + kOffAlo + off) = make_uint4(m.x & glo.x, m.y & glo.y, m.z & glo.z, m.w & glo.w);
    }
#pragma unroll 4
    for (int i = tid >> 3; i < 256; i += kGramThreads / 8) {
      const uint4 m = *reinterpret_cast<const uint4*>(m1t + (int64_t)i * ldk + r0);
      const int off = (i >> 3) * 1024 + c16 * 128 + (i & 7) * 16;
      *reinterpret_cast<uint4*>(sb + kOffBlo + off) = m;
      *reinterpret_cast<uint4*>(sb + kOffBhi + off) = make_uint4(m.x << 7, m.y << 7, m.z << 7, m.w << 7);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        const uint32_t base = smem_u32(sb);
#pragma unroll
        for (int ks = 0; ks < kStageRows / 32; ++ks) {
          umma_i8_ss(tmem, umma_desc128(base + kOffAhi + ks * 256), umma_desc128(base + kOffBhi + ks * 256),
                     (st | ks) != 0 ? 1u : 0u);
          umma_i8_ss(tmem, umma_desc128(base + kOffAlo + ks * 256), umma_desc128(base + kOffBlo + ks * 256), 1u);
        }
        umma_commit(smem_u32(&bars[buf]));
      }
      __syncwarp();
    }
  }
  // all MMAs done -> accumulator to global (zeros for an empty chunk)
  if (nstages >= 1) {
    const int last = (nstages - 1) & 1;
    mbar_wait(smem_u32(&bars[last]), (uint32_t)((nstages - 1) >> 1) & 1u);
    if (nstages >= 2) mbar_wait(smem_u32(&bars[last ^ 1]), (uint32_t)((nstages - 2) >> 1) & 1u);
  }
  __syncwarp();
  tc_fence_after();
  {
    const int quad = warp & 3, ch = warp >> 2;                      // TMEM lane quadrant, column half
    const int j = quad * 32 + (tid & 31);
    int32_t* out = partial + (((int64_t)rc * TCB_BLOCKS + ob) * 128 + j) * 256 + ch * 128;
#pragma unroll 1
    for (int g = 0; g < 4; ++g) {
      int32_t a[32];
      if (nstages >= 1) {
        tmem_ld32(tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(ch * 128 + g * 32), a);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      } else {
#pragma unroll
        for (int q = 0; q < 32; ++q) a[q] = 0;
      }
#pragma unroll
      for (int q = 0; q < 32; q += 4)
        *reinterpret_cast<int4*>(out + g * 32 + q) = make_int4(a[q], a[q + 1], a[q + 2], a[q + 3]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(256u) : "memory");
}

// C[k][j][i] from the partial accumulators, the 1-D sums and the coordinate scales.  Block = (k, j), thread = i.
__global__ void __launch_bounds__(TC_W)
bwd_finish_kernel(const int32_t* __restrict__ partial, const double* __restrict__ sums, const double* __restrict__ amax,
                  double slope, double* __restrict__ C) {
  const int k = blockIdx.x / TC_W, j = blockIdx.x % TC_W, i = threadIdx.x;
  const int half = j >> 7, jj = j & 127;
  double v = 0;
#pragma unroll
  for (int t = 0; t < TCB_NT; ++t) {
    const int ob = (k * TCB_NT + t) * 2 + half;
    long long acc = 0;
#pragma unroll
    for (int rc = 0; rc < TCB_CHUNKS; ++rc) acc += partial[(((int64_t)rc * TCB_BLOCKS + ob) * 128 + jj) * 256 + i];
    v = v * 16384.0 + (double)acc;
  }
  int e = 0;
  const double m = amax[k];
  if (m > 0) (void)frexp(m, &e);
  const double N = ldexp(v, e - (7 * TCB_NS - 1));
  const double S = sums[6 * TC_W + k], R0 = sums[k * TC_W + j], R1 = sums[3 * TC_W + k * TC_W + i];
  C[((int64_t)k * TC_W + j) * TC_W + i] = slope * slope * S + slope * (1.0 - slope) * (R0 + R1) + (1.0 - slope) * (1.0 - slope) * N;
}

}  // namespace

extern "C" {

size_t dpll_icnn_tc_bwd_partial_bytes(void) { return (size_t)TCB_CHUNKS * TCB_BLOCKS * 128 * 256 * sizeof(int32_t); }
int32_t dpll_icnn_tc_bwd_planes(void) { return 3 * TCB_NS; }

int dpll_icnn_tc_bwd_f64(const double* gp, const int64_t* n_rows, const double* amax, const uint8_t* m0t, const uint8_t* m1t,
                         int64_t ldk, double slope, int8_t* planes, int32_t* partial, double* sums, double* C, void* stream) {
  if (!gp || !n_rows || !amax || !m0t || !m1t || !planes || !partial || !sums || !C || ldk <= 0 || (ldk & 127)) return DPLL_EINVAL;
  // int32 accumulators: a chunk of rows x (128 * 64 + 64) must stay below 2^31
  if (ldk > (int64_t)TCB_CHUNKS * 250000) return DPLL_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  bwd_digits_kernel<<<(unsigned)((ldk + 255) / 256), 256, 0, st>>>(gp, n_rows, amax, ldk, planes);
  bwd_sums_kernel<<<2 * TC_W + 1, 256, 0, st>>>(gp, n_rows, m0t, m1t, ldk, sums);
  cudaError_t e = cudaFuncSetAttribute(bwd_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kGramSmem);
  if (e != cudaSuccess) return (int)e;
  bwd_gram_kernel<<<TCB_BLOCKS * TCB_CHUNKS, kGramThreads, kGramSmem, st>>>(n_rows, m0t, m1t, planes, ldk, partial);
  bwd_finish_kernel<<<3 * TC_W, TC_W, 0, st>>>(partial, sums, amax, slope, C);
  return cn::launch_status();
}

}  // extern "C"
