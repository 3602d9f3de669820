// Support points of the depth-2 homogeneous ICNN (HomogeneousICNN.forward, dair_pll/deep_support_function.py:238-266;
// called per contact by DeepSupportConvex.get_vertices, geometry.py:309-325) for ALL direction rows of a batch in one
// kernel on the sm_100a tensor cores: tcgen05.mma kind::i8 with int32 accumulators in TMEM.  See cn_icnn_tc.cuh for
// the mathematics (layer Jacobian = binary mask x constant matrix, as exact int8 digit-plane products).
//
// One persistent CTA per SM, 128-row tiles, warp-specialised (320 threads):
//   warps 0-7   prologue + epilogue.  Thread = (TMEM lane = direction row, column half).  Prologue: slope-mask bits of
//               layer 0 as the two byte-valued A operands ({0, 1} and {0, -128}), written straight into TENSOR MEMORY
//               (tcgen05.st; the MMA then takes A from TMEM and reads only the 1 KB B tile from shared memory -- with A
//               in shared memory a 128 x 32 B re-read per MMA made the N = 32 products four times slower).  Epilogue:
//               accumulators -> fp64 Jacobian (exact integer Horner) -> z1, layer-1 mask, support point, in registers.
//   warp 8      producer: digit planes of one (chunk of 32 hidden units, input coordinate k) unit = 6 planes x (32 x 256)
//               int8 = 48 KB per cp.async.bulk from the prepared image (L2-resident, 1.18 MB) into a 3-slot ring.
//   warp 9      MMA issuer: 48 MMAs (M 128, N 32, K 32) per unit into that k's three accumulators; tcgen05.commit
//               releases the ring slot and publishes the accumulators.
// The three accumulator sets (one per k) are handed back by the epilogue as soon as they are in registers, so the
// tensor pipe works on (chunk c, k+1 ...) while the CUDA cores finish (chunk c, k).
// TMEM columns: [0, 64) A {0,1}; [64, 128) A {0,-128}; [128 + 96 k + 32 t, +32) accumulator t of coordinate k.
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/dair_pll_b200.h"
#include "cn_icnn_tc.cuh"
#include "cn_launch.cuh"

namespace {

using namespace cn;

#ifndef TC_SPLIT
#define TC_SPLIT 4
#endif
constexpr int kSplit = TC_SPLIT;                     // threads per direction row (column groups of a chunk)
constexpr int kCols = TC_NC / kSplit;              // hidden units per thread and unit
constexpr int kEpiWarps = 4 * kSplit, kEpiThreads = kEpiWarps * 32, kThreads = kEpiThreads + 64;
constexpr int kTileRows = 128;
constexpr int kSlots = 3;
constexpr int kOffB = 0, kOffC = kOffB + kSlots * TC_UNIT_BYTES, kOffP = kOffC + TC_NCONST_SMEM * 8,
              kOffBar = kOffP + 2 * (kSplit - 1) * kTileRows * 3 * 8, kSmemBytes = kOffBar + 128;
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColAlo = 0, kColAhi = 64, kColAcc = 128;
// instruction descriptor, kind::i8: D s32 (2 << 4), A s8 (1 << 7), B s8 (1 << 10), both K-major, N >> 3 at 17, M >> 4 at 24
constexpr uint32_t kIdesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TC_NC >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
// barrier indices
constexpr int kBarFull = 0, kBarEmpty = kSlots, kBarAccFull = 2 * kSlots, kBarAccEmpty = 2 * kSlots + 3,
              kBarAReady = 2 * kSlots + 6, kNumBars = 2 * kSlots + 7;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// bounded spin (a protocol error must not hang the device): traps after a few seconds
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
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
  // K-major, no swizzle: LBO (K-adjacent core matrices) 128 B, SBO (8-row groups) 2048 B, descriptor version 1
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(128u >> 4) << 16) | ((uint64_t)(2048u >> 4) << 32) |
         ((uint64_t)1 << 46);
}
// D[tmem] (+)= A[tmem] . B[smem]
__device__ __forceinline__ void umma_i8_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, {%5, %6, %7, %8}, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(kIdesc), "r"(accumulate), "r"(0), "r"(0), "r"(0), "r"(0)
      : "memory");
}
// one lane of a converged warp (the compiler then issues the uniform-datapath instruction once, without a lane loop)
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
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, int32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, int32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory"); }

// sum_t acc_t 128^(2 (NACC-1-t)) as a double: integer Horner on the integer pipe (|result| < 2^51), then the 2^52 + 2^51
// bias trick instead of the conversion unit (exact)
__device__ __forceinline__ double horner_i2d(const int32_t* a) {
  long long v = a[0];
#pragma unroll
  for (int t = 1; t < TC_NACC; ++t) v = v * 16384 + a[t];
  return __longlong_as_double(v + 0x4338000000000000LL) - 6755399441055744.0;
}

// Rare-path correction, run AFTER a tile's hot loop for the entries whose |z1| fell below the tolerance (a 42-bit Jacobian
// must not decide the mask there; about one entry in 4e9): bit (8 c + q) of `flagged` marks hidden unit
// i = 32 c + 8 ch + q of this thread, `positive` the sign the hot loop used.  z1_i and Y_k[i] are recomputed in plain fp64
// from the weights (one pass over the 256 units of layer 0); if the exact sign differs, p is corrected by the difference
// of the two slopes and the recorded mask bit is rewritten.
template <bool RECORD>
__device__ __noinline__ void redo_entries(const double* sW0, const double* __restrict__ consts, const double* __restrict__ Wh,
                                          double dx, double dy, double dz, double slope, int ch, unsigned long long flagged,
                                          unsigned long long positive, double& p0, double& p1, double& p2,
                                          uint8_t* __restrict__ m1t, int64_t ldk, int64_t row) {
  const double* Wd1 = consts + TC_C_WD1;
  while (flagged) {
    const int bit = __ffsll((long long)flagged) - 1;
    flagged &= flagged - 1;
    const int i = (bit / kCols) * TC_NC + ch * kCols + (bit % kCols);
    double y0 = Wd1[i], y1 = Wd1[TC_W + i], y2 = Wd1[2 * TC_W + i], z = 0;
    for (int j = 0; j < TC_W; ++j) {
      const double lin = dx * sW0[j] + dy * sW0[TC_W + j] + dz * sW0[2 * TC_W + j];
      const double m0 = lin > 0 ? 1.0 : slope, wh = fabs(Wh[j * TC_W + i]);
      y0 += m0 * sW0[j] * wh; y1 += m0 * sW0[TC_W + j] * wh; y2 += m0 * sW0[2 * TC_W + j] * wh;
      z += (lin > 0 ? lin : slope * lin) * wh;
    }
    z += dx * Wd1[i] + dy * Wd1[TC_W + i] + dz * Wd1[2 * TC_W + i];
    const bool was = (positive >> bit) & 1ull, is = z > 0;
    if (was == is) continue;
    const double dm = (is ? 1.0 - slope : slope - 1.0) * consts[TC_C_COL + 8 * i + 7];      // (m_exact - m_used) |w_out|_i
    p0 = fma(dm, y0, p0); p1 = fma(dm, y1, p1); p2 = fma(dm, y2, p2);
    if (RECORD) m1t[(int64_t)i * ldk + row] = is ? 1 : 0;
  }
}

// RECORD = false: support points p of all D rows.  RECORD = true (the backward's first pass over the compacted active
// rows): the row count comes from device memory (*n_ptr <= D, no host read), and instead of p the two layers' slope-mask
// bits are written as TRANSPOSED byte matrices -- m0t[j][row] in {0x00, 0xFF}, m1t[i][row] in {0, 1}, row stride ldk --
// the K-major operands of the weight-gradient kernel.
template <bool RECORD>
__global__ void __launch_bounds__(kThreads, 1)
icnn_tc_kernel(const double* __restrict__ d, int64_t D, const int64_t* __restrict__ n_ptr, const uint8_t* __restrict__ img,
               const double* __restrict__ consts, const double* __restrict__ Wh, double slope, double* __restrict__ p,
               uint8_t* __restrict__ m0t, uint8_t* __restrict__ m1t, int64_t ldk) {
  if (RECORD) { const int64_t n = *n_ptr; D = n < D ? n : D; }
  extern __shared__ __align__(1024) uint8_t smem[];
  double* sC = reinterpret_cast<double*>(smem + kOffC);
  double* sP = reinterpret_cast<double*>(smem + kOffP);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBar + 8 * kNumBars);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t bar0 = smem_u32(bars);
  auto bar = [bar0](int i) { return bar0 + 8u * (uint32_t)i; };

  if (tid == 0) {
    for (int s = 0; s < kSlots; ++s) { mbar_init(bar(kBarFull + s), 1); mbar_init(bar(kBarEmpty + s), 1); }
    for (int k = 0; k < 3; ++k) { mbar_init(bar(kBarAccFull + k), 1); mbar_init(bar(kBarAccEmpty + k), kEpiWarps); }
    mbar_init(bar(kBarAReady), kEpiWarps);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  for (int i = tid; i < TC_NCONST_SMEM; i += kThreads) sC[i] = consts[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int64_t ntiles = (D + kTileRows - 1) / kTileRows;
  const int64_t my_tiles = (int64_t)blockIdx.x < ntiles ? (ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;

  if (warp == kEpiWarps) {
    // ===== producer (whole warp runs the loop, one elected lane issues) =====
    const uint32_t sB = smem_u32(smem + kOffB);
    const int64_t total = my_tiles * TC_UNITS;
    int s = 0, unit = 0;
    uint32_t use = 0;
    for (int64_t g = 0; g < total; ++g) {
      if (use >= 1) mbar_wait(bar(kBarEmpty + s), (use - 1) & 1u);
      if (elect_one()) {
        mbar_expect_tx(bar(kBarFull + s), TC_UNIT_BYTES);
        bulk_g2s(sB + (uint32_t)s * TC_UNIT_BYTES, img + (size_t)unit * TC_UNIT_BYTES, TC_UNIT_BYTES, bar(kBarFull + s));
      }
      __syncwarp();
      if (++s == kSlots) { s = 0; ++use; }
      if (++unit == TC_UNITS) unit = 0;
    }
  } else if (warp == kEpiWarps + 1) {
    // ===== MMA issuer (whole warp runs the loop, one elected lane issues) =====
    const uint32_t sB = smem_u32(smem + kOffB);
    // descriptor of byte 0 of the ring: K-major, no swizzle, LBO 128 B, SBO 2048 B, version 1; +1 per 16 bytes
    const uint64_t desc0 = umma_desc(sB);
    int s = 0;
    uint32_t use = 0;
    for (int64_t it = 0; it < my_tiles; ++it) {
      mbar_wait(bar(kBarAReady), (uint32_t)it & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < TC_CHUNKS; ++c) {
        const uint32_t n = (uint32_t)(it * TC_CHUNKS + c);       // uses of each accumulator set so far
#pragma unroll 1
        for (int k = 0; k < 3; ++k) {
          if (n >= 1) mbar_wait(bar(kBarAccEmpty + k), (n - 1) & 1u);
          mbar_wait(bar(kBarFull + s), use & 1u);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t desc_u = desc0 + (uint64_t)((uint32_t)s * (TC_UNIT_BYTES >> 4));
#pragma unroll
            for (int t = 0; t < TC_NACC; ++t) {
              const uint32_t acc = tmem + kColAcc + (uint32_t)((k * TC_NACC + t) * TC_NC);
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const uint32_t a_base = tmem + (h == 0 ? kColAhi : kColAlo);
#pragma unroll
                for (int ks = 0; ks < TC_W / 32; ++ks)
                  umma_i8_ts(acc, a_base + ks * 8, desc_u + (uint64_t)(((2 * t + h) * TC_SLICE_BYTES + ks * 256) >> 4),
                             (h | ks) != 0 ? 1u : 0u);
              }
            }
            umma_commit(bar(kBarEmpty + s));
            umma_commit(bar(kBarAccFull + k));
          }
          __syncwarp();
          if (++s == kSlots) { s = 0; ++use; }
        }
      }
    }
  } else {
    // ===== prologue + epilogue warps =====
    const int quad = warp & 3, ch = warp >> 2;                 // TMEM lane quadrant, column group
    const int r_in = quad * 32 + lane;
    const uint32_t tmem_lane = tmem + ((uint32_t)(quad * 32) << 16);
    const double* sW0 = sC + TC_C_WD0;
    constexpr int kWords = 64 / kSplit;                        // words of each A copy written by this thread
    for (int64_t it = 0; it < my_tiles; ++it) {
      const int64_t tile = blockIdx.x + it * gridDim.x;
      const int64_t row = tile * kTileRows + r_in;
      const bool valid = row < D;
      double dx = 0, dy = 0, dz = 0;
      if (valid) { dx = d[3 * row]; dy = d[3 * row + 1]; dz = d[3 * row + 2]; }
      // ---- prologue: this thread's mask bits of layer 0 (hidden units ch * 4 kWords ..) -> kWords words of A in TMEM ----
      {
        uint32_t w[kWords];
#pragma unroll
        for (int wi = 0; wi < kWords; ++wi) {
          uint32_t v = 0;
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            const int j = (ch * kWords + wi) * 4 + b;
            const double lin = dx * sW0[j] + dy * sW0[TC_W + j] + dz * sW0[2 * TC_W + j];
            v |= (lin > 0 ? 1u : 0u) << (8 * b);
          }
          w[wi] = v;
          if (RECORD) {
#pragma unroll
            for (int b = 0; b < 4; ++b)
              m0t[(int64_t)((ch * kWords + wi) * 4 + b) * ldk + row] = ((v >> (8 * b)) & 1u) ? 0xFF : 0x00;
          }
        }
        // (the previous tile's MMAs have all completed: its last accumulator set was awaited below)
        if constexpr (kWords == 32) tmem_st32(tmem_lane + kColAlo + (uint32_t)(ch * kWords), w);
        else tmem_st16(tmem_lane + kColAlo + (uint32_t)(ch * kWords), w);
#pragma unroll
        for (int wi = 0; wi < kWords; ++wi) w[wi] <<= 7;
        if constexpr (kWords == 32) tmem_st32(tmem_lane + kColAhi + (uint32_t)(ch * kWords), w);
        else tmem_st16(tmem_lane + kColAhi + (uint32_t)(ch * kWords), w);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(kBarAReady));
      }
      double p0 = 0, p1 = 0, p2 = 0;
      unsigned long long flagged = 0, positive = 0;
      static_assert(TC_CHUNKS * kCols <= 64, "one flag bit per (chunk, column) of a thread");
#pragma unroll 1
      for (int c = 0; c < TC_CHUNKS; ++c) {
        const uint32_t n = (uint32_t)(it * TC_CHUNKS + c);
        double Y0[kCols], Y1[kCols];
        // reconstructed Jacobian entry |w_out|_i Y_k[i] of column q from its three accumulators
        auto entry = [&](const int32_t (&a)[TC_NACC][kCols], int k, int q) {
          const int i = c * TC_NC + ch * kCols + q;
          int32_t aq[TC_NACC];
#pragma unroll
          for (int t = 0; t < TC_NACC; ++t) aq[t] = a[t][q];
          const double v = horner_i2d(aq);
          const double2 cb = *reinterpret_cast<const double2*>(sC + TC_C_COL + 8 * i + 2 * k);
          return fma(cb.x, v, cb.y);
        };
        auto load_set = [&](int32_t (&a)[TC_NACC][kCols], int k) {
#pragma unroll
          for (int t = 0; t < TC_NACC; ++t) {
            const uint32_t ta = tmem_lane + kColAcc + (uint32_t)((k * TC_NACC + t) * TC_NC + ch * kCols);
            if constexpr (kCols == 16) tmem_ld16(ta, a[t]);
            else tmem_ld8(ta, a[t]);
          }
        };
        {
          // the accumulator sets of k = 0 and k = 1 are fetched TOGETHER (one exposed TMEM-load latency instead of two: the
          // tensor pipe runs ahead of this epilogue, so both are normally complete) and handed back at once
          int32_t a0[TC_NACC][kCols], a1[TC_NACC][kCols];
          mbar_wait(bar(kBarAccFull + 0), n & 1u);
          mbar_wait(bar(kBarAccFull + 1), n & 1u);
          __syncwarp();
          tc_fence_after();
          load_set(a0, 0);
          load_set(a1, 1);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { mbar_arrive(bar(kBarAccEmpty + 0)); mbar_arrive(bar(kBarAccEmpty + 1)); }
#pragma unroll
          for (int q = 0; q < kCols; ++q) { Y0[q] = entry(a0, 0, q); Y1[q] = entry(a1, 1, q); }
        }
        {
          int32_t a[TC_NACC][kCols];
          mbar_wait(bar(kBarAccFull + 2), n & 1u);
          __syncwarp();
          tc_fence_after();
          load_set(a, 2);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar(kBarAccEmpty + 2));     // the tensor pipe may overwrite this set
#pragma unroll
          for (int q = 0; q < kCols; ++q) {
            const int i = c * TC_NC + ch * kCols + q;
            const double y = entry(a, 2, q);
            const double z = dx * Y0[q] + dy * Y1[q] + dz * y;
            // |z1| below the tolerance: the entry is flagged and settled in plain fp64 AFTER the tile's hot loop
            // (redo_entries) -- a call inside this loop cost 160-260 bytes of spills around it
            if (fabs(z) < sC[TC_C_COL + 8 * i + 6]) {
              flagged |= 1ull << (c * kCols + q);
              if (z > 0) positive |= 1ull << (c * kCols + q);
            }
            const double m = z > 0 ? 1.0 : slope;
            if (RECORD) m1t[(int64_t)i * ldk + row] = z > 0 ? 1 : 0;
            p0 = fma(m, Y0[q], p0);
            p1 = fma(m, Y1[q], p1);
            p2 = fma(m, y, p2);
          }
        }
      }
      if (flagged && valid) redo_entries<RECORD>(sW0, consts, Wh, dx, dy, dz, slope, ch, flagged, positive, p0, p1, p2, m1t, ldk, row);
      if (RECORD) continue;
      // the column groups of a row meet in shared memory
      double* sPt = sP + (it & 1) * ((kSplit - 1) * kTileRows * 3);
      if (ch > 0) {
        double* dst = sPt + ((ch - 1) * kTileRows + r_in) * 3;
        dst[0] = p0; dst[1] = p1; dst[2] = p2;
      }
      epi_barrier();
      if (ch == 0 && valid) {
#pragma unroll
        for (int o = 0; o < kSplit - 1; ++o) {
          const double* src = sPt + (o * kTileRows + r_in) * 3;
          p0 += src[0]; p1 += src[1]; p2 += src[2];
        }
        p[3 * row] = p0; p[3 * row + 1] = p1; p[3 * row + 2] = p2;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
}

// one block per hidden unit i (column of the three Q_k): scales, digit planes, epilogue constants
__global__ void __launch_bounds__(TC_W)
icnn_tc_prepare_kernel(const double* __restrict__ Wd0, const double* __restrict__ Wd1, const double* __restrict__ Wh,
                       const double* __restrict__ wout, double slope, uint8_t* __restrict__ img, double* __restrict__ consts) {
  __shared__ double red_max[TC_W / 32], red_sum[TC_W / 32], red_abs[TC_W / 32];
  __shared__ double bc[3];
  const int i = blockIdx.x, j = threadIdx.x, lane = j & 31, w = j >> 5;
  const double wh = fabs(Wh[j * TC_W + i]);
  const double wo = fabs(wout[i]);
  double abs_total = 0;
  for (int k = 0; k < 3; ++k) {
    const double q = Wd0[k * TC_W + j] * wh;
    double mx = fabs(q), sm = q, ab = fabs(q);
    for (int o = 16; o > 0; o >>= 1) {
      mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      sm += __shfl_xor_sync(0xffffffffu, sm, o);
      ab += __shfl_xor_sync(0xffffffffu, ab, o);
    }
    if (lane == 0) { red_max[w] = mx; red_sum[w] = sm; red_abs[w] = ab; }
    __syncthreads();
    if (j == 0) {
      double m2 = 0, s2 = 0, a2 = 0;
      for (int x = 0; x < TC_W / 32; ++x) { m2 = fmax(m2, red_max[x]); s2 += red_sum[x]; a2 += red_abs[x]; }
      bc[0] = m2; bc[1] = s2; bc[2] = a2;
    }
    __syncthreads();
    int e;
    const double sigma = tc_column_scale(bc[0], &e);
    int8_t dig[TC_NS];
    tc_digits(q, e, dig);
    for (int s = 0; s < TC_NS; ++s) img[tc_image_offset(k, s, j, i)] = (uint8_t)dig[s];
    if (j == 0) {
      consts[TC_C_COL + 8 * i + 2 * k] = wo * ((1.0 - slope) * ldexp(sigma, -(7 * TC_NS - 1)));
      consts[TC_C_COL + 8 * i + 2 * k + 1] = wo * (Wd1[k * TC_W + i] + slope * bc[1]);
      consts[TC_C_WD0 + k * TC_W + i] = Wd0[k * TC_W + i];
      consts[TC_C_WD1 + k * TC_W + i] = Wd1[k * TC_W + i];
    }
    abs_total += bc[2] + fabs(Wd1[k * TC_W + i]);
    __syncthreads();
  }
  if (j == 0) {
    consts[TC_C_COL + 8 * i + 6] = wo * (TC_ZTOL_REL * abs_total);
    consts[TC_C_COL + 8 * i + 7] = wo;                      // read by redo_columns only
  }
}

}  // namespace

extern "C" {

size_t dpll_icnn_tc_image_bytes(void) { return (size_t)cn::TC_IMG_BYTES; }
size_t dpll_icnn_tc_const_bytes(void) { return (size_t)cn::TC_NCONST * sizeof(double); }

int dpll_icnn_tc_prepare_f64(const double* Wd0, const double* Wd1, const double* Wh, const double* wout, int32_t W,
                             double slope, void* image, double* consts, void* stream) {
  if (W != cn::TC_W || !Wd0 || !Wd1 || !Wh || !wout || !image || !consts) return DPLL_EINVAL;
  icnn_tc_prepare_kernel<<<cn::TC_W, cn::TC_W, 0, static_cast<cudaStream_t>(stream)>>>(
      Wd0, Wd1, Wh, wout, slope, static_cast<uint8_t*>(image), consts);
  return cn::launch_status();
}

int dpll_icnn_tc_support_f64(const double* d, int64_t D, const void* image, const double* consts, const double* Wh,
                             int32_t W, double slope, double* p, void* stream) {
  if (W != cn::TC_W || D < 0 || !image || !consts || !Wh) return DPLL_EINVAL;
  if (D == 0) return DPLL_OK;
  if (!d || !p) return DPLL_EINVAL;
  cudaError_t e = cudaFuncSetAttribute(icnn_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e != cudaSuccess) return (int)e;
  const int64_t ntiles = (D + kTileRows - 1) / kTileRows;
  int sms = 0;
  if (int rc = cn::sm_count(&sms)) return rc;
  const int grid = (int)(ntiles < sms ? ntiles : sms);
  icnn_tc_kernel<false><<<grid, kThreads, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(
      d, D, nullptr, static_cast<const uint8_t*>(image), consts, Wh, slope, p, nullptr, nullptr, 0);
  return cn::launch_status();
}

int dpll_icnn_tc_record_f64(const double* d, int64_t capacity, const int64_t* n_rows, const void* image, const double* consts,
                            const double* Wh, int32_t W, double slope, uint8_t* m0t, uint8_t* m1t, int64_t ldk, void* stream) {
  if (W != cn::TC_W || capacity < 0 || !n_rows || !image || !consts || !Wh || (ldk & 127) || ldk < capacity) return DPLL_EINVAL;
  if (capacity == 0) return DPLL_OK;
  if (!d || !m0t || !m1t) return DPLL_EINVAL;
  cudaError_t e = cudaFuncSetAttribute(icnn_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e != cudaSuccess) return (int)e;
  const int64_t ntiles = (capacity + kTileRows - 1) / kTileRows;
  int sms = 0;
  if (int rc = cn::sm_count(&sms)) return rc;
  const int grid = (int)(ntiles < sms ? ntiles : sms);
  icnn_tc_kernel<true><<<grid, kThreads, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(
      d, capacity, n_rows, static_cast<const uint8_t*>(image), consts, Wh, slope, nullptr, m0t, m1t, ldk);
  return cn::launch_status();
}

}  // extern "C"
