// Wavefront kernel for the two-body (elbow) ContactNets loss + envelope backward: the scheduling of
// cube_loss_wf_kernel (cn_kernels.cu) over the closed-form articulated terms of cn_elbow_wf.cuh.
//
// Each WARP owns a pool of kEwSlots sample slots in shared memory (96 doubles each, field-major: the 17 numbers of the
// mass matrix, lever arms, hinge columns, QP vector, the Newton state), two ring queues of slots (active / done) and
// a FIFO of sample indices, and runs warp-uniform phases:
//   T   triage of the next 32 input samples in registers (elbow_loss_free_flight): free flight -- 62% of a toss data
//       set -- is finalised on the spot, the others queue their index for a slot
//   N   one Newton visit (elbow_newton_visit: one gradient / packed-Hessian evaluation, 7x7 Cholesky in registers)
//       for the active slots
//   PE  for slots of the done queue: pass 0 finalises the finished samples (problem rebuilt from x, x+; loss +
//       envelope backward), pass 1 refills the emptied slots with triaged samples (problem built and parked)
// With 96-double records a warp gets 32 slots (8 warps per SM), so phases run at least half a warp wide (PE when
// >= 16 slots wait, N otherwise) instead of always 32 as for the cube.  No per-thread arrays outlive a phase: the
// dense 7x7 objects of the first elbow kernels (5 KB of local memory per thread, 1.2 GB of DRAM writes per launch)
// are gone -- the record is the only per-sample state.
#include <cuda_runtime.h>

#include "../../include/dair_pll_b200.h"
#include "cn_elbow_wf.cuh"
#include "cn_launch.cuh"
#include "cn_reduce.cuh"

namespace {

#ifndef CN_EW_SLOTS
#define CN_EW_SLOTS 32
#endif
#ifndef CN_EW_WARPS
#define CN_EW_WARPS 4
#endif
constexpr int kEwSlots = CN_EW_SLOTS;
#ifndef CN_EW_PE_MIN
#define CN_EW_PE_MIN (kEwSlots / 2)
#endif
constexpr int kEwPeMin = CN_EW_PE_MIN;     // a PE phase runs once this many slots wait in the done queue
constexpr int kEwWarps = CN_EW_WARPS;
constexpr int kEwQin = 64;
constexpr int kEwNAcc = 32;       // 28 parameter gradients + loss sum + pad
constexpr int kEwMaxBlocks = 148 * 16;
static_assert((size_t)kEwMaxBlocks * kEwNAcc * sizeof(double) <= cn::kWsPartialsBytes, "elbow partials exceed the workspace");

template <typename T> struct EwWarpPool {
  T field[cn::EW_FIELDS][kEwSlots];
  int32_t sample[kEwSlots];       // offset of the slot's sample in the warp's range; -1 = empty
  int32_t iters[kEwSlots];
  uint8_t q_act[kEwSlots], q_done[kEwSlots];
  int32_t q_in[kEwQin];
};

template <typename T> __device__ __forceinline__ T ew_warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Warp reduce-scatter of 32 per-lane values: on return lane l holds sum over lanes of v[bitrev5(l)]... precisely, the
// value index owned by a lane is built from its lane bits stage by stage (bit 4 first): after the stage with offset
// o the lane keeps the half of its remaining values selected by (lane & o).  31 shuffle-adds per lane instead of
// 32 x 5; all array indices are compile-time constants (registers).  Deterministic (fixed tree).
template <typename T> __device__ __forceinline__ T ew_reduce_scatter32(T* v, int lane) {
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const bool up = lane & 16;
    const T keep = up ? v[i + 16] : v[i], give = up ? v[i] : v[i + 16];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, give, 16);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const bool up = lane & 8;
    const T keep = up ? v[i + 8] : v[i], give = up ? v[i] : v[i + 8];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, give, 8);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool up = lane & 4;
    const T keep = up ? v[i + 4] : v[i], give = up ? v[i] : v[i + 4];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, give, 4);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const bool up = lane & 2;
    const T keep = up ? v[i + 2] : v[i], give = up ? v[i] : v[i + 2];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, give, 2);
  }
  {
    const bool up = lane & 1;
    const T keep = up ? v[1] : v[0], give = up ? v[0] : v[1];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, give, 1);
  }
  return v[0];      // lane l owns value index (l & 16) + (l & 8) + (l & 4) + (l & 2) + (l & 1) = l
}

template <typename T, typename IO>
__device__ __forceinline__ void ew_load_params(cn::ElbowParams<T>& P, const IO* inertia, const IO* mu, const IO* half,
                                               const IO* kin, T dt, T eps) {
  T in[20], m[2], h[6], kn[cn::EL_NKIN];
  for (int i = 0; i < 20; ++i) in[i] = T(inertia[i]);
  for (int i = 0; i < 2; ++i) m[i] = T(mu[i]);
  for (int i = 0; i < 6; ++i) h[i] = half ? T(half[i]) : T(0);
  for (int i = 0; i < cn::EL_NKIN; ++i) kn[i] = T(kin[i]);
  cn::elbow_params_init(P, in, m, h, kn, dt, eps);
}

template <typename T, typename IO>
__global__ void __launch_bounds__(kEwWarps * 32)
elbow_loss_wf_kernel(const IO* __restrict__ x, const IO* __restrict__ xp, const IO* __restrict__ weight,
                     const IO* __restrict__ inertia, const IO* __restrict__ mu, const IO* __restrict__ half,
                     const IO* __restrict__ kin, const IO* __restrict__ pts, T dt, T eps, int64_t B,
                     IO* __restrict__ loss, IO* __restrict__ force, IO* __restrict__ grad_pts,
                     int32_t* __restrict__ iters, T* __restrict__ partials, int want_grad,
                     const int32_t* __restrict__ skip_flag, unsigned long long* __restrict__ dyn_counter) {
  // dyn_counter != nullptr (DPLL_LOSS_DYNAMIC): warps draw their 32-sample chunks from a global counter, in batch
  // order (cost-ordered batches: uniform chunks, longest solves first), as cube_loss_wf_kernel does.
  if (skip_flag && *skip_flag) return;
  extern __shared__ __align__(16) unsigned char ew_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  EwWarpPool<T>* pool = reinterpret_cast<EwWarpPool<T>*>(ew_smem) + warp;
  const unsigned lt_mask = (1u << lane) - 1u;

  cn::ElbowParams<T> P;
  ew_load_params<T, IO>(P, inertia, mu, half, kin, dt, eps);
  const cn::SolverCfg<T> cfg = cn::default_cfg<T>();
  // Accumulators: lane l owns accumulator l ([0, 28) parameter gradients, 28 = loss sum); every finalising phase
  // reduce-scatters its 32 lanes' contributions (ew_reduce_scatter32), so one register replaces 29 per thread.
  T acc_lane = T(0);

  const int64_t gw = (int64_t)blockIdx.x * kEwWarps + warp, W = (int64_t)gridDim.x * kEwWarps;
  const int64_t base = B / W, rem = B % W;
  const int64_t lo = dyn_counter ? 0 : gw * base + (gw < rem ? gw : rem);
  const int64_t hi = dyn_counter ? B : lo + base + (gw < rem ? 1 : 0);
  int64_t next = lo;

  for (int s = lane; s < kEwSlots; s += 32) { pool->q_done[s] = (uint8_t)s; pool->sample[s] = -1; }
  int n_act = 0, n_done = kEwSlots, h_act = 0, h_done = 0, n_in = 0, h_in = 0;
  __syncwarp();

  while (true) {
    int phase;   // 0 = PE, 1 = N, 2 = T
    const bool drain = next >= hi && n_in == 0;
    if (next < hi && n_in < 32) phase = 2;
    else if (drain) {
      if (n_act > 0) phase = 1;
      else if (n_done > 0) phase = 0;
      else break;
    } else if (n_done >= kEwPeMin) phase = 0;
    else phase = 1;

    if (phase == 2) {
      int64_t first = next;
      if (dyn_counter) {
        unsigned long long t = 0;
        if (lane == 0) t = atomicAdd(dyn_counter, 32ull);
        first = (int64_t)__shfl_sync(0xffffffffu, t, 0);
        if (first >= B) first = B;
      }
      const int64_t left = hi - first;
      const int cnt = left < 32 ? (int)left : 32;
      bool queue = false;
      const int64_t b = first + lane;
      T gs[kEwNAcc];
#pragma unroll
      for (int i = 0; i < kEwNAcc; ++i) gs[i] = T(0);
      if (lane < cnt) {
        T xs[15], xps[15];
#pragma unroll
        for (int i = 0; i < 15; ++i) { xs[i] = T(x[b * 15 + i]); xps[i] = T(xp[b * 15 + i]); }
        T l = T(0);
        const T w = weight ? T(weight[b]) : T(1);
        if (cn::elbow_loss_free_flight<T, IO>(P, xs, xps, pts ? pts + b * 24 : (const IO*)nullptr,
                                              want_grad ? gs : (T*)nullptr, grad_pts ? grad_pts + b * 24 : (IO*)nullptr, w,
                                              &l)) {
          if (force) {
#pragma unroll 1
            for (int i = 0; i < 24; ++i) force[b * 24 + i] = IO(0);
          }
#pragma unroll
          for (int i = 0; i < DPLL_ELBOW_NPARAM; ++i) gs[i] *= w;
          if (loss) loss[b] = IO(l);
          gs[DPLL_ELBOW_NPARAM] = l;
          if (iters) iters[b] = 0;
        } else {
          queue = true;
        }
      }
      acc_lane += ew_reduce_scatter32(gs, lane);
      const unsigned m_q = __ballot_sync(0xffffffffu, queue);
      if (queue) pool->q_in[(h_in + n_in + __popc(m_q & lt_mask)) % kEwQin] = (int32_t)(b - lo);
      n_in += __popc(m_q);
      next = dyn_counter ? (first >= B ? B : lo) : next + cnt;
    } else if (phase == 1) {
      const int k = n_act < 32 ? n_act : 32;
      const bool on = lane < k;
      int st = -1;
      int slot = 0;
      if (on) {
        slot = pool->q_act[(h_act + lane) % kEwSlots];
        const cn::ElbowRec<T> S{&pool->field[0][slot], kEwSlots};
        T u[7], d[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) { u[i] = pool->field[77 + i][slot]; d[i] = pool->field[84 + i][slot]; }
        T best = pool->field[91][slot], d0 = pool->field[92][slot];
        cn::CubeTrial<T> tr{pool->field[93][slot], pool->field[94][slot], pool->field[95][slot]};
        int it = pool->iters[slot];
        st = cn::elbow_newton_visit<T>(P, S, cfg, u, d, d0, best, tr, it);
        pool->iters[slot] = it;
        pool->field[91][slot] = best;
#pragma unroll
        for (int i = 0; i < 7; ++i) { pool->field[77 + i][slot] = u[i]; pool->field[84 + i][slot] = d[i]; }
        pool->field[92][slot] = d0;
        pool->field[93][slot] = tr.alpha; pool->field[94][slot] = tr.lo; pool->field[95][slot] = tr.hi;
      }
      __syncwarp();
      const unsigned m_done = __ballot_sync(0xffffffffu, st == cn::NEWTON_DONE);
      const unsigned m_act = __ballot_sync(0xffffffffu, st == cn::NEWTON_CONTINUE);
      h_act = (h_act + k) % kEwSlots; n_act -= k;
      if (st == cn::NEWTON_DONE) pool->q_done[(h_done + n_done + __popc(m_done & lt_mask)) % kEwSlots] = (uint8_t)slot;
      else if (st == cn::NEWTON_CONTINUE) pool->q_act[(h_act + n_act + __popc(m_act & lt_mask)) % kEwSlots] = (uint8_t)slot;
      n_done += __popc(m_done); n_act += __popc(m_act);
    } else {
      const int k = n_done < 32 ? n_done : 32;
      const bool on = lane < k;
      int slot = 0, old = -1;
      if (on) { slot = pool->q_done[(h_done + lane) % kEwSlots]; old = pool->sample[slot]; }
      bool to_active = false;
      int n_new = 0;
#pragma unroll 1
      for (int pass = 0; pass < 2; ++pass) {
        if (pass == 0) {
          if (!__any_sync(0xffffffffu, on && old >= 0)) continue;
        } else {
          n_new = n_in < k ? n_in : k;
          if (n_new == 0) break;
        }
        const bool work = pass == 0 ? (on && old >= 0) : (lane < n_new);
        T gs[kEwNAcc];
#pragma unroll
        for (int i = 0; i < kEwNAcc; ++i) gs[i] = T(0);
        if (work) {
          const int64_t b = lo + (pass == 0 ? old : pool->q_in[(h_in + lane) % kEwQin]);
          T xs[15], xps[15];
#pragma unroll
          for (int i = 0; i < 15; ++i) { xs[i] = T(x[b * 15 + i]); xps[i] = T(xp[b * 15 + i]); }
          const cn::ElbowRec<T> S{&pool->field[0][slot], kEwSlots};
          cn::ElbowSetup<T> E;
          cn::ElbowLossCore<T> A;
          cn::elbow_loss_prologue_wf<T, IO>(P, xs, xps, pts ? pts + b * 24 : (const IO*)nullptr, S, E, A);
          if (pass == 0) {
            T u[7];
#pragma unroll
            for (int i = 0; i < 7; ++i) u[i] = pool->field[77 + i][slot];
            const T w = weight ? T(weight[b]) : T(1);
            const T l = cn::elbow_loss_epilogue_wf<T, IO>(P, S, E, A, u, want_grad ? gs : (T*)nullptr,
                                                          force ? force + b * 24 : (IO*)nullptr,
                                                          grad_pts ? grad_pts + b * 24 : (IO*)nullptr, w);
#pragma unroll
            for (int i = 0; i < DPLL_ELBOW_NPARAM; ++i) gs[i] *= w;
            if (loss) loss[b] = IO(l);
            gs[DPLL_ELBOW_NPARAM] = l;
            if (iters) iters[b] = pool->iters[slot] & 0xff;
            pool->sample[slot] = -1;
          } else {
#pragma unroll
            for (int i = 0; i < 7; ++i) pool->field[77 + i][slot] = (T(1) - A.a_start) * A.dv[i];
            pool->field[91][slot] = T(-1);
            pool->field[92][slot] = T(0);
            pool->sample[slot] = (int32_t)(b - lo);
            pool->iters[slot] = 0;
            to_active = true;
          }
        }
        if (pass == 0) acc_lane += ew_reduce_scatter32(gs, lane);
      }
      h_in = (h_in + n_new) % kEwQin; n_in -= n_new;
      const bool more = next < hi || n_in > 0;
      __syncwarp();
      const unsigned m_act = __ballot_sync(0xffffffffu, to_active);
      const unsigned m_keep = __ballot_sync(0xffffffffu, on && !to_active && more);
      h_done = (h_done + k) % kEwSlots; n_done -= k;
      if (to_active) pool->q_act[(h_act + n_act + __popc(m_act & lt_mask)) % kEwSlots] = (uint8_t)slot;
      else if (on && more) pool->q_done[(h_done + n_done + __popc(m_keep & lt_mask)) % kEwSlots] = (uint8_t)slot;
      n_act += __popc(m_act); n_done += __popc(m_keep);
    }
    __syncwarp();
  }

  if (!partials) return;
  __shared__ T red[kEwWarps][kEwNAcc];
  red[warp][lane] = acc_lane;
  __syncthreads();
  if (threadIdx.x < kEwNAcc) {
    T s = T(0);
#pragma unroll
    for (int w = 0; w < kEwWarps; ++w) s += red[w][threadIdx.x];
    partials[(int64_t)blockIdx.x * kEwNAcc + threadIdx.x] = s;
  }
}

template <typename T, typename IO>
int launch_elbow_loss(const IO* x, const IO* xp, const IO* weight, const IO* inertia, const IO* mu, const IO* half,
                      const IO* kin, const IO* pts, T dt, T eps, int64_t B, IO* loss, IO* force, IO* grad_pts,
                      int32_t* iters, IO* grad, IO* loss_sum,
                      const int32_t* skip_flag, void* workspace, size_t workspace_bytes, void* stream, int flags) {
  if (B < 0 || !inertia || !mu || (!half && !pts) || !kin || (grad_pts && (!pts || !grad))) return DPLL_EINVAL;
  if (B > 0 && (!x || !xp)) return DPLL_EINVAL;
  const bool want_red = grad || loss_sum;
  if (want_red && !cn::workspace_ok(workspace, workspace_bytes)) return DPLL_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  T* partials = want_red ? static_cast<T*>(workspace) : nullptr;
  unsigned long long* dyn = nullptr;
  if (flags & DPLL_LOSS_DYNAMIC) {
    if (!cn::workspace_ok(workspace, workspace_bytes)) return DPLL_EWORKSPACE;
    if (int rc = cn::dynamic_counter(workspace, st, &dyn)) return rc;
  }
  const size_t smem = sizeof(EwWarpPool<T>) * kEwWarps;
  cudaError_t ea = cudaFuncSetAttribute(elbow_loss_wf_kernel<T, IO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (ea != cudaSuccess) return (int)ea;
  // at most one resident set; a warp wants >= 128 samples to keep its pool busy
  int blocks;
  int64_t cap;
  if (int rc = cn::resident_blocks(elbow_loss_wf_kernel<T, IO>, kEwWarps * 32, smem, (B + kEwWarps * 128 - 1) / (kEwWarps * 128),
                                   kEwMaxBlocks, &blocks, &cap))
    return rc;
  elbow_loss_wf_kernel<T, IO><<<blocks, kEwWarps * 32, smem, st>>>(x, xp, weight, inertia, mu, half, kin, pts, dt, eps, B,
                                                                   loss, force, grad_pts, iters, partials, grad ? 1 : 0,
                                                                   skip_flag, dyn);
  if (int rc = cn::launch_status()) return rc;
  if (!want_red) return DPLL_OK;
  reduce_partials_kernel<T, IO, kEwNAcc, DPLL_ELBOW_NPARAM><<<1, 32 * kEwNAcc, 0, st>>>(partials, blocks, grad, loss_sum,
                                                                                       skip_flag);
  return cn::launch_status();
}

}  // namespace

extern "C" {

int dpll_elbow_loss_f64(const double* x, const double* x_plus, const double* weight, const double* inertia,
                        const double* mu_pair, const double* half, const double* kin, const double* pts, double dt,
                        double eps, int64_t B, int32_t flags, double* loss, double* force, double* grad_pts,
                        int32_t* iters, double* grad, double* loss_sum, const int32_t* skip_flag, void* workspace,
                        size_t workspace_bytes, void* stream) {
  return launch_elbow_loss<double, double>(x, x_plus, weight, inertia, mu_pair, half, kin, pts, dt, eps, B, loss, force,
                                           grad_pts, iters, grad, loss_sum, skip_flag, workspace, workspace_bytes, stream,
                                           flags);
}

int dpll_elbow_loss_f32(const float* x, const float* x_plus, const float* weight, const float* inertia,
                        const float* mu_pair, const float* half, const float* kin, const float* pts, float dt, float eps,
                        int64_t B, int32_t flags, float* loss, float* force, float* grad_pts, int32_t* iters, float* grad,
                        float* loss_sum, const int32_t* skip_flag, void* workspace, size_t workspace_bytes,
                        void* stream) {
  return launch_elbow_loss<double, float>(x, x_plus, weight, inertia, mu_pair, half, kin, pts, (double)dt, (double)eps, B,
                                          loss, force, grad_pts, iters, grad, loss_sum, skip_flag, workspace,
                                          workspace_bytes, stream, flags);
}

}  // extern "C"
