// CUDA kernels + C ABI (include/dair_pll_b200.h) for the ContactNets hot path, sm_100a.
//
// One sample per thread: the whole per-sample pipeline (terms -> QP build -> Newton solve
// -> loss -> envelope backward) lives in registers; no tensor cores (the per-sample
// systems are 6x6), no shared-memory tiles; HBM traffic is 2*13 loads + 1 store per
// sample.  Parameter gradients are accumulated per thread across a grid-stride loop and
// reduced warp -> block -> grid in a fixed order (deterministic).
#include <cuda_runtime.h>

#include "../../include/dair_pll_b200.h"
#include "../../include/dair_pll_b200_warm_body_tree.h"
#include "cn_cube.cuh"
#include "cn_params.cuh"
#include "cn_elbow.cuh"
#include "cn_elbow_wf.cuh"
#include "cn_comm.cuh"
#include "cn_launch.cuh"
#include "cn_reduce.cuh"

namespace {

constexpr int kLossThreads = 128;
constexpr int kNAcc = 16;            // 14 parameter gradients + loss sum + pad
constexpr int kMaxBlocks = 148 * 16; // most blocks of a loss launch (box and witness points)
static_assert((size_t)kMaxBlocks * kNAcc * sizeof(double) <= cn::kWsPartialsBytes, "box partials exceed the workspace");

// Tosses per warp of a rollout launch.  A toss is a chain of dependent steps, so a warp is issue-bound by its own
// instruction stream whatever its number of active lanes (ncu, 4,096 x 80 at four tosses per warp: 2.2 lanes per instruction
// with the FP64 pipe 64% busy), and two warps on one SM sub-partition slow each other down.  Small batches therefore get ONE
// block per SM -- one warp per sub-partition -- with as many tosses per warp as that takes (4,096 x 80: 7 per warp; measured
// 2.61 ms at 4 per warp, 2.04 at 8, 2.32 at 12, 2.45 at 16); only when that would put more than 12 tosses on a warp (the warp
// advances at the pace of its slowest toss) are all resident warps used.
inline int rollout_tosses_per_warp(int64_t B, int sms, int64_t resident_warps) {
  const int64_t warps1 = (int64_t)sms * (kLossThreads / 32);
  int64_t lpw = (B + warps1 - 1) / warps1;
  if (lpw > 12) lpw = (B + resident_warps - 1) / resident_warps;
  if (lpw < 1) lpw = 1;
  if (lpw > 32) lpw = 32;
  return (int)lpw;
}

// load the callable-level parameters (stored as IO) into the compute type
template <typename T, typename IO>
__device__ __forceinline__ void load_cube_params(cn::CubeParams<T>& P, const IO* inertia, const IO* mu, const IO* half,
                                                 T dt, T eps) {
  T in[10], m[1], h[3];
#pragma unroll
  for (int i = 0; i < 10; ++i) in[i] = T(inertia[i]);
  m[0] = T(mu[0]);
#pragma unroll
  for (int i = 0; i < 3; ++i) h[i] = T(half[i]);
  cn::cube_params_init(P, in, m, h, dt, eps);
}

// T = arithmetic type, IO = storage type of states / parameters / outputs.  The fp32 variant is
// IO = float with T = double: on this latency-bound path fp32 arithmetic buys no speed (measured:
// a pure-fp32 build is slower, its Newton needs more steps) and cannot hold 1e-4 on the gradients
// (cond(H) ~ 1e4-1e5), while fp32 storage halves the HBM traffic.
template <typename T, typename IO>
__global__ void __launch_bounds__(kLossThreads)
cube_loss_kernel(const IO* __restrict__ x, const IO* __restrict__ xp, const IO* __restrict__ weight,
                 const IO* __restrict__ inertia,
                 const IO* __restrict__ mu, const IO* __restrict__ half, T dt, T eps, int64_t B,
                 IO* __restrict__ loss, IO* __restrict__ force, int32_t* __restrict__ iters,
                 T* __restrict__ partials, int want_grad, const int32_t* __restrict__ skip_flag, int64_t ldx,
                 int64_t ldxp) {
  if (skip_flag && *skip_flag) return;
  cn::CubeParams<T> P;
  load_cube_params<T, IO>(P, inertia, mu, half, dt, eps);
  const cn::SolverCfg<T> cfg = cn::default_cfg<T>();
  T acc[kNAcc];
#pragma unroll
  for (int i = 0; i < kNAcc; ++i) acc[i] = T(0);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += stride) {
    T xs[13], xps[13];
#pragma unroll
    for (int i = 0; i < 13; ++i) { xs[i] = T(x[b * ldx + i]); xps[i] = T(xp[b * ldxp + i]); }
    int it;
    T gs[DPLL_CUBE_NPARAM], fo[12];
#pragma unroll
    for (int i = 0; i < DPLL_CUBE_NPARAM; ++i) gs[i] = T(0);
    const T l = cn::cube_loss_sample<T>(P, cfg, xs, xps, want_grad ? gs : nullptr, force ? fo : nullptr, &it);
    if (force) {
#pragma unroll
      for (int i = 0; i < 12; ++i) force[b * 12 + i] = IO(fo[i]);
    }
    const T w = weight ? T(weight[b]) : T(1);
#pragma unroll
    for (int i = 0; i < DPLL_CUBE_NPARAM; ++i) acc[i] += w * gs[i];
    if (loss) loss[b] = IO(l);
    acc[14] += l;
    if (iters) iters[b] = it;
  }
  if (!partials) return;
  __shared__ T red[kLossThreads / 32][kNAcc];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < kNAcc; ++i) {
    const T s = warp_sum(acc[i]);
    if (lane == 0) red[warp][i] = s;
  }
  __syncthreads();
  if (threadIdx.x < kNAcc) {
    T s = T(0);
#pragma unroll
    for (int w = 0; w < kLossThreads / 32; ++w) s += red[w][threadIdx.x];
    partials[(int64_t)blockIdx.x * kNAcc + threadIdx.x] = s;
  }
}

// ---------------------------------------------------------------------------
// Racing warps for the EXPENSIVE head of a cost-ordered batch (DPLL_LOSS_RACE); see cube_loss_wf_kernel.
//
// A launch lasts at least as long as its longest Newton chain (~45 dependent visits of ~2.5 us on the bench batch), which
// is all that is left of a small launch -- the strong-scaling shard of a data-parallel step.  How long a chain gets depends
// on where it starts: over eight different start points on the feasible segment (cube_loss_start) the SHORTEST chain of the
// worst sample is 26 visits instead of 47 (over the best four: 28), and only 92 of 39,016 solves still need 20 or more.
// The optimum is unique, so any of them gives the same answer.
// ---------------------------------------------------------------------------
constexpr int kRaceLanes = 4;                          // start points per sample: factors 7, 2, 60 of a_min and the fraction 0.3
constexpr int kRaceSamples = 32 / kRaceLanes;          // samples per racing warp

// ---------------------------------------------------------------------------
// Wavefront variant of the loss kernel.
//
// A solve needs 0 .. ~45 Newton visits depending on the sample (free-flight samples need none), so
// one-sample-per-thread leaves ~80% of the lanes idle (ncu: 5.8 active threads per instruction,
// profiles/).  Here each WARP owns a pool of kWfSlots sample slots in shared memory, two ring queues of
// slots (active / done) and a FIFO of sample indices, and runs warp-uniform phases over 32 samples:
//   T   triage of the next 32 input samples in registers: free flight (u = 0, f = 0 optimal) is finalised
//       on the spot by cube_loss_free_flight; the others queue their index for a slot
//   N   one Newton visit (one gradient/Hessian evaluation, cube_newton_visit) for 32 active slots
//   PE  for 32 slots of the done queue: pass 0 finalises the finished samples (problem rebuilt from
//       x, x+ -> loss + envelope backward -> outputs), pass 1 refills the emptied slots with triaged
//       samples (problem built and parked in the slot).  One code instance of the prologue serves both.
// Slots are conserved (active + done = kWfSlots until the input runs out), so one of the two queues
// always holds a full warp's worth: phases run 32 wide until the warp drains.  The phase choice depends
// only on warp-uniform counters; there is no divergence between phases and the per-sample arithmetic is
// the same code as the simple kernel.  Samples are assigned to warps statically (contiguous ranges),
// which keeps the gradient reduction deterministic.  The hot loops are kept small (rolled per-contact
// loops over the shared-memory slot) because warps of one SM sit in different phases and share the
// instruction cache.
// ---------------------------------------------------------------------------
#ifndef CN_WF_UNR
#define CN_WF_UNR 1
#endif
constexpr int kWfUnr = CN_WF_UNR;   // unroll factor of the per-contact loops inside the Newton step
#ifndef CN_WF_UNR_PE
#define CN_WF_UNR_PE 1
#endif
constexpr int kWfUnrPE = CN_WF_UNR_PE;   // ... and inside the prologue / epilogue
#ifndef CN_WF_MIN_PER_WARP
#define CN_WF_MIN_PER_WARP 128
#endif
constexpr int kWfMinPerWarp = CN_WF_MIN_PER_WARP;   // fewest samples a warp should get before more warps are used
#ifndef CN_WF_SLOTS
#define CN_WF_SLOTS 64
#endif
#ifndef CN_WF_PE_MIN
#define CN_WF_PE_MIN 32
#endif
#ifndef CN_WF_MIN_BLOCKS
#define CN_WF_MIN_BLOCKS 1
#endif
constexpr int kWfSlots = CN_WF_SLOTS;      // sample slots per warp
constexpr int kWfPeMin = CN_WF_PE_MIN;     // a PE phase runs once this many slots wait in the done queue
constexpr int kWfQin = 64;                 // FIFO of triaged samples waiting for a slot (< 32 + 32 entries)
constexpr int kWfWarps = 4;
constexpr int kWfFields = 50;   // IW 6 | mcW 3 | rho 12 | q 12 | u 6 | best_res2 1 | d 6 | d0 1 | alpha, lo, hi

template <typename T> struct WfWarpPool {
  T field[kWfFields][kWfSlots];
  int32_t sample[kWfSlots];     // offset of the slot's sample in the warp's range; -1 = empty
  int32_t iters[kWfSlots];
  uint8_t q_act[kWfSlots], q_done[kWfSlots];
  int32_t q_in[kWfQin];         // offsets of triaged samples that need the solver, waiting for a slot
};

template <typename T, typename IO, int UNR, bool RACE = false, bool PTS = false>
__global__ void __launch_bounds__(kWfWarps * 32, CN_WF_MIN_BLOCKS)
cube_loss_wf_kernel(const IO* __restrict__ x, const IO* __restrict__ xp, const IO* __restrict__ weight,
                    const IO* __restrict__ inertia, const IO* __restrict__ mu, const IO* __restrict__ half, T dt,
                    T eps, int64_t B, IO* __restrict__ loss, IO* __restrict__ force, int32_t* __restrict__ iters,
                    T* __restrict__ partials, int want_grad, const int32_t* __restrict__ skip_flag,
                    unsigned long long* __restrict__ dyn_counter, int64_t ldx, int64_t ldxp,
                    const IO* __restrict__ u_init, IO* __restrict__ u_out, int race_blocks, int64_t head) {
  // u_init / u_out (nullable, (B, 6)): start point of every sample's Newton solve and its optimum (world-frame
  // twist).  A training loop revisits the same pairs with slowly moving parameters: started from the previous
  // epoch's optimum the solve takes a few visits instead of ~11 (the optimum is unique, so only the visit count
  // depends on the start).
  // dyn_counter != nullptr (DPLL_LOSS_DYNAMIC / variant 2): warps take their triage chunks of 32 samples from a
  // global counter, in batch order, instead of a static range -- removes the load imbalance between warps and
  // lets a cost-ordered batch start its longest solves first, but the assignment of samples to warps (and with it
  // the rounding of the gradient sums) then depends on timing.  (Measured and dropped: a two-ended queue in which
  // the second block of every SM consumes the batch from its cheap end, so that no two warps of long chains share
  // an SM sub-partition -- 0.427 vs 0.398 ms at 1,048,576 pairs, 0.143 vs 0.129 ms at 131,072.)
  // PTS (the witness-point instance, T = IO): the lever arms come from per-sample body-frame points instead of selected box
  // corners (body_*_pts in cn_cube.cuh).  It takes its extra arguments through parameters the box instances have and it
  // does not use -- extra kernel parameters change ptxas's register allocation of the box instances -- so that their
  // code stays as it is:  half = the points (B, 4, 3), of which the first n_c are used;  u_out = grad_pts (B, 4, 3),
  // w_b d loss_b / d pts_b (nullable);  want_grad = bit 0 as for the box | n_c << 1.  u_init must be null and RACE false.
  // Accumulators: [d/d inertia 10 | d/d mu | loss sum].  Its code sits in `if constexpr` branches in front of the box
  // statements, which keep their text: even a dead statement's line information changes the box instances' allocation.
  static_assert(!(PTS && RACE), "no racing warps for witness points");
  if (skip_flag && *skip_flag) return;
  // DPLL_LOSS_RACE (the RACE instantiation): the warps of blocks [0, race_blocks) are RACING warps for the first `head`
  // samples (the expensive head of a cost-ordered batch); the other blocks run the wavefront scheduler over the rest.  A
  // racing warp takes eight samples and gives each four slots with different start points; it then runs through the very
  // same phases -- PE pass 1 builds and parks the problems, N visits all slots, after every visit the slots of one sample
  // vote: the first to converge wins, its siblings are dropped, PE pass 0 finalises the winner.  The same code instances as
  // the wavefront warps, so the two kinds of warps share the instruction cache (a first version with a per-thread racing
  // body in the same launch spent 21% of its stall samples waiting for instructions).
  const bool race_warp = RACE && (int)blockIdx.x < race_blocks;
  if (!race_warp) {
    x += head * ldx; xp += head * ldxp; B -= head;
    if (weight) weight += head;
    if (loss) loss += head;
    if (force) force += head * 12;
    if (iters) iters += head;
    if (u_init) u_init += head * 6;
    if (u_out) u_out += head * 6;
  }
  const int wf_block = (int)blockIdx.x - race_blocks, wf_blocks = (int)gridDim.x - race_blocks;
  extern __shared__ __align__(16) unsigned char wf_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WfWarpPool<T>* pool = reinterpret_cast<WfWarpPool<T>*>(wf_smem) + warp;
  const unsigned lt_mask = (1u << lane) - 1u;

  cn::CubeParams<T> P;
  if constexpr (PTS) {
    T in[10], m[1], h[3] = {T(0), T(0), T(0)};
#pragma unroll
    for (int i = 0; i < 10; ++i) in[i] = T(inertia[i]);
    m[0] = T(mu[0]);
    cn::cube_params_init(P, in, m, h, dt, eps);
  } else
  load_cube_params<T, IO>(P, inertia, mu, half, dt, eps);
  const cn::SolverCfg<T> cfg = cn::default_cfg<T>();
  T acc[kNAcc];
#pragma unroll
  for (int i = 0; i < kNAcc; ++i) acc[i] = T(0);

  // static contiguous sample range of this warp
  const int64_t gw = (int64_t)wf_block * kWfWarps + warp, W = (int64_t)wf_blocks * kWfWarps;
  const int64_t base = B / W, rem = B % W;
  const int64_t lo = (dyn_counter || race_warp) ? 0 : gw * base + (gw < rem ? gw : rem);
  const int64_t hi = race_warp ? 0 : (dyn_counter ? B : lo + base + (gw < rem ? 1 : 0));
  int64_t next = lo;               // static: next unread sample of the range; dynamic: B once the counter ran out

  for (int s = lane; s < kWfSlots; s += 32) { pool->q_done[s] = (uint8_t)s; pool->sample[s] = -1; }
  int n_act = 0, n_done = kWfSlots, h_act = 0, h_done = 0, n_in = 0, h_in = 0;
  if (race_warp) {
    // no triage: the warp's kRaceSamples samples x kRaceLanes start points wait in q_in (entry = sample | start << 28)
    const int64_t first = ((int64_t)blockIdx.x * kWfWarps + warp) * kRaceSamples;
    const int64_t left = head - first;
    const int cnt = left <= 0 ? 0 : (left < kRaceSamples ? (int)left : kRaceSamples);
    if (lane < cnt * kRaceLanes) pool->q_in[lane] = (int32_t)(first + lane / kRaceLanes) | ((lane % kRaceLanes) << 28);
    n_in = cnt * kRaceLanes;
  }
  __syncwarp();

  while (true) {
    int phase;   // 0 = PE, 1 = N, 2 = T (triage)
    // Slots are conserved while input remains (active + done = kWfSlots), so one of the two queues
    // always holds a full warp's worth.  Once the input is exhausted (drain) the remaining samples'
    // Newton chains are the critical path: N runs at whatever width is left and the finished samples
    // are finalised in full-width PE batches at the very end.
    const bool drain = next >= hi && n_in == 0;
    if (next < hi && n_in < 32) phase = 2;     // keep a warp's worth of solver samples queued
    else if (drain) {
      if (n_act > 0) phase = 1;
      else if (n_done > 0) phase = 0;
      else break;
    } else if (n_done >= kWfPeMin) phase = 0;
    else phase = 1;

    if (phase == 2) {
      // T: the next 32 input samples, in registers only.  Free flight (u = 0, f = 0 optimal) is finalised
      // here at a third of the generic cost; the others wait in q_in for a slot.
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
      if (lane < cnt) {
        T xs[13], xps[13];
#pragma unroll
        for (int i = 0; i < 13; ++i) { xs[i] = T(x[b * ldx + i]); xps[i] = T(xp[b * ldxp + i]); }
        T gs[DPLL_CUBE_NPARAM];
#pragma unroll
        for (int i = 0; i < DPLL_CUBE_NPARAM; ++i) gs[i] = T(0);
        T l = T(0);
        if constexpr (PTS) {
          const T w = weight ? T(weight[b]) : T(1);
          if (cn::body_loss_free_flight_pts<T>(P, xs, xps, half + b * 12, want_grad >> 1, w, (want_grad & 1) ? gs : (T*)nullptr,
                                               u_out ? u_out + b * 12 : (IO*)nullptr, &l)) {
            if (force) {
#pragma unroll
              for (int i = 0; i < 12; ++i) force[b * 12 + i] = IO(0);
            }
#pragma unroll
            for (int i = 0; i < 11; ++i) acc[i] += w * gs[i];
            if (loss) loss[b] = IO(l);
            acc[11] += l;
            if (iters) iters[b] = 0;
          } else {
            queue = true;
          }
        } else
        if (cn::cube_loss_free_flight<T>(P, xs, xps, want_grad ? gs : (T*)nullptr, &l)) {
          if (force) {
#pragma unroll
            for (int i = 0; i < 12; ++i) force[b * 12 + i] = IO(0);
          }
          const T w = weight ? T(weight[b]) : T(1);
#pragma unroll
          for (int i = 0; i < DPLL_CUBE_NPARAM; ++i) acc[i] += w * gs[i];
          if (loss) loss[b] = IO(l);
          acc[14] += l;
          if (iters) iters[b] = 0;
          if (u_out) {
#pragma unroll
            for (int i = 0; i < 6; ++i) u_out[b * 6 + i] = IO(0);
          }
        } else {
          queue = true;
        }
      }
      const unsigned m_q = __ballot_sync(0xffffffffu, queue);
      if (queue) pool->q_in[(h_in + n_in + __popc(m_q & lt_mask)) % kWfQin] = (int32_t)(b - lo);
      n_in += __popc(m_q);
      next = dyn_counter ? (first >= B ? B : lo) : next + cnt;
#ifndef CN_NO_PREFETCH
      if (!dyn_counter && next + lane < hi) {       // the rows of the next triage visit: pull them into L2
        const char* px = reinterpret_cast<const char*>(x + (next + lane) * ldx);
        const char* pp = reinterpret_cast<const char*>(xp + (next + lane) * ldxp);
        asm volatile("prefetch.global.L2 [%0];" ::"l"(px));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(px + 13 * sizeof(IO) - 1));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(pp));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(pp + 13 * sizeof(IO) - 1));
      }
#endif
    } else if (phase == 1) {
      const int k = n_act < 32 ? n_act : 32;
      const bool on = lane < k;
      int st = -1;
      int slot = 0;
      if (on) {
        slot = pool->q_act[(h_act + lane) % kWfSlots];
        const cn::CubeProb<T> S{&pool->field[0][slot], kWfSlots};
        T u[6], d[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) { u[i] = pool->field[33 + i][slot]; d[i] = pool->field[40 + i][slot]; }
        T best = pool->field[39][slot], d0 = pool->field[46][slot];
        cn::CubeTrial<T> tr{pool->field[47][slot], pool->field[48][slot], pool->field[49][slot]};
        int it = pool->iters[slot];
        st = cn::cube_newton_visit<T, UNR>(P, S, cfg, u, d, d0, best, tr, it);
        pool->iters[slot] = it;
        pool->field[39][slot] = best;
#pragma unroll
        for (int i = 0; i < 6; ++i) { pool->field[33 + i][slot] = u[i]; pool->field[40 + i][slot] = d[i]; }
        pool->field[46][slot] = d0;
        pool->field[47][slot] = tr.alpha; pool->field[48][slot] = tr.lo; pool->field[49][slot] = tr.hi;
      }
      if (race_warp) {
        // the slots of one sample vote: the first finisher wins, its siblings give their slots back unfinalised
        const int sid = on ? pool->sample[slot] : -2 - lane;
        const unsigned grp = __match_any_sync(0xffffffffu, sid);
        const unsigned fin = __ballot_sync(0xffffffffu, on && st == cn::NEWTON_DONE);
        if (on && (grp & fin) && lane != __ffs(grp & fin) - 1) { pool->sample[slot] = -1; st = cn::NEWTON_DONE; }
      }
      __syncwarp();          // ring entries read above may be overwritten below (queue full): order the accesses
      const unsigned m_done = __ballot_sync(0xffffffffu, st == cn::NEWTON_DONE);
      const unsigned m_act = __ballot_sync(0xffffffffu, st == cn::NEWTON_CONTINUE);
      h_act = (h_act + k) % kWfSlots; n_act -= k;
      if (st == cn::NEWTON_DONE) pool->q_done[(h_done + n_done + __popc(m_done & lt_mask)) % kWfSlots] = (uint8_t)slot;
      else if (st == cn::NEWTON_CONTINUE) pool->q_act[(h_act + n_act + __popc(m_act & lt_mask)) % kWfSlots] = (uint8_t)slot;
      n_done += __popc(m_done); n_act += __popc(m_act);
    } else {
      // PE: up to 32 slots of the done queue, two passes over ONE code instance of the prologue.  Pass 0
      // finalises the finished samples (problem rebuilt from x, x+; loss + envelope backward; outputs) and
      // their slots become empty; pass 1 gives the batch's empty slots the next triaged samples (problem
      // built and parked) and sends them to the active queue -- so in steady state both passes run 32 wide.
      const int k = n_done < 32 ? n_done : 32;
      const bool on = lane < k;
      int slot = 0, old = -1;
      if (on) { slot = pool->q_done[(h_done + lane) % kWfSlots]; old = pool->sample[slot]; }
      bool to_active = false;
      int n_new = 0;
#pragma unroll 1
      for (int pass = 0; pass < 2; ++pass) {
        if (pass == 0) {
          if (!__any_sync(0xffffffffu, on && old >= 0)) continue;
        } else {
          n_new = n_in < k ? n_in : k;                     // after pass 0 every slot of the batch is empty
          if (n_new == 0) break;
        }
        const bool work = pass == 0 ? (on && old >= 0) : (lane < n_new);
        if (work) {
          const int32_t ent = pass == 0 ? old : pool->q_in[(h_in + lane) % kWfQin];
          const int start = race_warp ? (ent >> 28) & 7 : 0;          // (pass 1 of a racing warp: which start point)
          const int64_t b = lo + (race_warp ? (ent & 0x0fffffff) : ent);
          T xs[13], xps[13];
#pragma unroll
          for (int i = 0; i < 13; ++i) { xs[i] = T(x[b * ldx + i]); xps[i] = T(xp[b * ldxp + i]); }
          const cn::CubeProb<T> S{&pool->field[0][slot], kWfSlots};
          cn::CubeLossAux<T> A;
          if constexpr (PTS) cn::body_loss_prologue_pts<T, kWfUnrPE>(P, xs, xps, half + b * 12, want_grad >> 1, S, A);
          else
          cn::cube_loss_prologue<T, kWfUnrPE>(P, xs, xps, S, A);      // (re)builds IW, mcW, rho, q in the slot
          if (pass == 0) {
            if constexpr (PTS) {
              T u[6], gs[11], fo[12];
#pragma unroll
              for (int i = 0; i < 6; ++i) u[i] = pool->field[33 + i][slot];
#pragma unroll
              for (int i = 0; i < 11; ++i) gs[i] = T(0);
              const T w = weight ? T(weight[b]) : T(1);
              const T l = cn::body_loss_epilogue_pts<T, kWfUnrPE, true>(P, S, A, u, want_grad >> 1, w,
                                                                        (want_grad & 1) ? gs : (T*)nullptr,
                                                                        u_out ? u_out + b * 12 : (IO*)nullptr,
                                                                        force ? fo : (T*)nullptr);
              if (force) {
#pragma unroll
                for (int i = 0; i < 12; ++i) force[b * 12 + i] = IO(fo[i]);
              }
#pragma unroll
              for (int i = 0; i < 11; ++i) acc[i] += w * gs[i];
              if (loss) loss[b] = IO(l);
              acc[11] += l;
              if (iters) iters[b] = pool->iters[slot] & 0xff;
            } else {
            T u[6];
#pragma unroll
            for (int i = 0; i < 6; ++i) u[i] = pool->field[33 + i][slot];
            T gs[DPLL_CUBE_NPARAM];
#pragma unroll
            for (int i = 0; i < DPLL_CUBE_NPARAM; ++i) gs[i] = T(0);
            T fo[12];
            const T l = cn::cube_loss_epilogue<T, kWfUnrPE, true>(P, S, A, u, want_grad ? gs : (T*)nullptr, force ? fo : (T*)nullptr);
            if (force) {
#pragma unroll
              for (int i = 0; i < 12; ++i) force[b * 12 + i] = IO(fo[i]);
            }
            const T w = weight ? T(weight[b]) : T(1);
#pragma unroll
            for (int i = 0; i < DPLL_CUBE_NPARAM; ++i) acc[i] += w * gs[i];
            if (loss) loss[b] = IO(l);
            acc[14] += l;
            if (iters) iters[b] = pool->iters[slot] & 0xff;
            if (u_out) {
#pragma unroll
              for (int i = 0; i < 6; ++i) u_out[b * 6 + i] = IO(u[i]);
            }
            }
            pool->sample[slot] = -1;
          } else {
            T us[6];
            if (start == 3) cn::cube_loss_start_fraction<T>(A, T(0.3), us);
            else cn::cube_loss_start<T>(A, start == 1 ? T(2) : start == 2 ? T(60) : T(CN_LOSS_START_FACTOR), us);
#pragma unroll
            for (int i = 0; i < 6; ++i) pool->field[33 + i][slot] = u_init ? T(u_init[b * 6 + i]) : us[i];
            pool->field[39][slot] = T(-1);
            pool->field[46][slot] = T(0);
            pool->sample[slot] = (int32_t)(b - lo);
            pool->iters[slot] = 0;
            to_active = true;
          }
        }
      }
      h_in = (h_in + n_new) % kWfQin; n_in -= n_new;
      const bool more = next < hi || n_in > 0;             // empty slots are only kept while input remains
      __syncwarp();
      const unsigned m_act = __ballot_sync(0xffffffffu, to_active);
      const unsigned m_keep = __ballot_sync(0xffffffffu, on && !to_active && more);
      h_done = (h_done + k) % kWfSlots; n_done -= k;
      if (to_active) pool->q_act[(h_act + n_act + __popc(m_act & lt_mask)) % kWfSlots] = (uint8_t)slot;
      else if (on && more) pool->q_done[(h_done + n_done + __popc(m_keep & lt_mask)) % kWfSlots] = (uint8_t)slot;
      n_act += __popc(m_act); n_done += __popc(m_keep);
    }
    __syncwarp();
  }

  if (!partials) return;
  __shared__ T red[kWfWarps][kNAcc];
#pragma unroll 1
  for (int i = 0; i < kNAcc; ++i) {
    T v = T(0);
#pragma unroll
    for (int j = 0; j < kNAcc; ++j) v = (j == i) ? acc[j] : v;
    const T s = warp_sum(v);
    if (lane == 0) red[warp][i] = s;
  }
  __syncthreads();
  if (threadIdx.x < kNAcc) {
    T s = T(0);
#pragma unroll
    for (int w = 0; w < kWfWarps; ++w) s += red[w][threadIdx.x];
    partials[(int64_t)blockIdx.x * kNAcc + threadIdx.x] = s;
  }
}

// Warm-started witness-point loss of the single body (dpll_body_loss_pts_warm_f64): the PTS instance of
// cube_loss_wf_kernel -- same triage, slots, Newton visits and PE passes, same accumulators -- with a start point and an
// optimum per sample.  u_init (nullable, (B, 6)): PE pass 1 seeds the slot's u from row b instead of the feasible-segment
// point; u_out (nullable, (B, 6)): PE pass 0 writes the slot's u, the triage writes zeros for free flight (its exact
// optimum).  Row b is read when its sample gets a slot and written when that sample is finalised, so u_init == u_out
// works.  A kernel of its own: statements added to cube_loss_wf_kernel, even in discarded `if constexpr` branches, changed
// ptxas's register allocation of its box instances.
template <int UNR>
__global__ void __launch_bounds__(kWfWarps * 32, CN_WF_MIN_BLOCKS)
body_loss_pts_warm_kernel(const double* __restrict__ x, const double* __restrict__ xp, const double* __restrict__ weight,
                          const double* __restrict__ inertia, const double* __restrict__ mu,
                          const double* __restrict__ pts, int n_c, double dt, double eps, int64_t B,
                          double* __restrict__ loss, double* __restrict__ force, double* __restrict__ grad_pts,
                          int32_t* __restrict__ iters, double* __restrict__ partials, int want_grad,
                          const int32_t* __restrict__ skip_flag, unsigned long long* __restrict__ dyn_counter,
                          const double* u_init, double* u_out) {
  using T = double;
  if (skip_flag && *skip_flag) return;
  extern __shared__ __align__(16) unsigned char wf_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WfWarpPool<T>* pool = reinterpret_cast<WfWarpPool<T>*>(wf_smem) + warp;
  const unsigned lt_mask = (1u << lane) - 1u;

  cn::CubeParams<T> P;
  {
    T in[10], m[1], h[3] = {T(0), T(0), T(0)};
#pragma unroll
    for (int i = 0; i < 10; ++i) in[i] = inertia[i];
    m[0] = mu[0];
    cn::cube_params_init(P, in, m, h, dt, eps);
  }
  const cn::SolverCfg<T> cfg = cn::default_cfg<T>();
  T acc[12];                       // [d/d inertia 10 | d/d mu | loss sum], as the PTS instance
#pragma unroll
  for (int i = 0; i < 12; ++i) acc[i] = T(0);

  const int64_t gw = (int64_t)blockIdx.x * kWfWarps + warp, W = (int64_t)gridDim.x * kWfWarps;
  const int64_t base = B / W, rem = B % W;
  const int64_t lo = dyn_counter ? 0 : gw * base + (gw < rem ? gw : rem);
  const int64_t hi = dyn_counter ? B : lo + base + (gw < rem ? 1 : 0);
  int64_t next = lo;

  for (int s = lane; s < kWfSlots; s += 32) { pool->q_done[s] = (uint8_t)s; pool->sample[s] = -1; }
  int n_act = 0, n_done = kWfSlots, h_act = 0, h_done = 0, n_in = 0, h_in = 0;
  __syncwarp();

  while (true) {
    int phase;   // 0 = PE, 1 = N, 2 = T (triage): the scheduling of cube_loss_wf_kernel
    const bool drain = next >= hi && n_in == 0;
    if (next < hi && n_in < 32) phase = 2;
    else if (drain) {
      if (n_act > 0) phase = 1;
      else if (n_done > 0) phase = 0;
      else break;
    } else if (n_done >= kWfPeMin) phase = 0;
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
      if (lane < cnt) {
        T xs[13], xps[13], gs[11];
#pragma unroll
        for (int i = 0; i < 13; ++i) { xs[i] = x[b * 13 + i]; xps[i] = xp[b * 13 + i]; }
#pragma unroll
        for (int i = 0; i < 11; ++i) gs[i] = T(0);
        T l = T(0);
        const T w = weight ? weight[b] : T(1);
        if (cn::body_loss_free_flight_pts<T>(P, xs, xps, pts + b * 12, n_c, w, want_grad ? gs : (T*)nullptr,
                                             grad_pts ? grad_pts + b * 12 : (T*)nullptr, &l)) {
          if (force) {
#pragma unroll
            for (int i = 0; i < 12; ++i) force[b * 12 + i] = T(0);
          }
#pragma unroll
          for (int i = 0; i < 11; ++i) acc[i] += w * gs[i];
          if (loss) loss[b] = l;
          acc[11] += l;
          if (iters) iters[b] = 0;
          if (u_out) {
#pragma unroll 1
            for (int i = 0; i < 6; ++i) u_out[b * 6 + i] = T(0);
          }
        } else {
          queue = true;
        }
      }
      const unsigned m_q = __ballot_sync(0xffffffffu, queue);
      if (queue) pool->q_in[(h_in + n_in + __popc(m_q & lt_mask)) % kWfQin] = (int32_t)(b - lo);
      n_in += __popc(m_q);
      next = dyn_counter ? (first >= B ? B : lo) : next + cnt;
    } else if (phase == 1) {
      const int k = n_act < 32 ? n_act : 32;
      const bool on = lane < k;
      int st = -1;
      int slot = 0;
      if (on) {
        slot = pool->q_act[(h_act + lane) % kWfSlots];
        const cn::CubeProb<T> S{&pool->field[0][slot], kWfSlots};
        T u[6], d[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) { u[i] = pool->field[33 + i][slot]; d[i] = pool->field[40 + i][slot]; }
        T best = pool->field[39][slot], d0 = pool->field[46][slot];
        cn::CubeTrial<T> tr{pool->field[47][slot], pool->field[48][slot], pool->field[49][slot]};
        int it = pool->iters[slot];
        st = cn::cube_newton_visit<T, UNR>(P, S, cfg, u, d, d0, best, tr, it);
        pool->iters[slot] = it;
        pool->field[39][slot] = best;
#pragma unroll
        for (int i = 0; i < 6; ++i) { pool->field[33 + i][slot] = u[i]; pool->field[40 + i][slot] = d[i]; }
        pool->field[46][slot] = d0;
        pool->field[47][slot] = tr.alpha; pool->field[48][slot] = tr.lo; pool->field[49][slot] = tr.hi;
      }
      __syncwarp();
      const unsigned m_done = __ballot_sync(0xffffffffu, st == cn::NEWTON_DONE);
      const unsigned m_act = __ballot_sync(0xffffffffu, st == cn::NEWTON_CONTINUE);
      h_act = (h_act + k) % kWfSlots; n_act -= k;
      if (st == cn::NEWTON_DONE) pool->q_done[(h_done + n_done + __popc(m_done & lt_mask)) % kWfSlots] = (uint8_t)slot;
      else if (st == cn::NEWTON_CONTINUE) pool->q_act[(h_act + n_act + __popc(m_act & lt_mask)) % kWfSlots] = (uint8_t)slot;
      n_done += __popc(m_done); n_act += __popc(m_act);
    } else {
      // PE: pass 0 finalises the finished samples (optimum to u_out), pass 1 parks the next triaged ones (start from
      // u_init)
      const int k = n_done < 32 ? n_done : 32;
      const bool on = lane < k;
      int slot = 0, old = -1;
      if (on) { slot = pool->q_done[(h_done + lane) % kWfSlots]; old = pool->sample[slot]; }
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
        if (work) {
          const int32_t ent = pass == 0 ? old : pool->q_in[(h_in + lane) % kWfQin];
          const int64_t b = lo + ent;
          T xs[13], xps[13];
#pragma unroll
          for (int i = 0; i < 13; ++i) { xs[i] = x[b * 13 + i]; xps[i] = xp[b * 13 + i]; }
          const cn::CubeProb<T> S{&pool->field[0][slot], kWfSlots};
          cn::CubeLossAux<T> A;
          cn::body_loss_prologue_pts<T, kWfUnrPE>(P, xs, xps, pts + b * 12, n_c, S, A);
          if (pass == 0) {
            T u[6], gs[11], fo[12];
#pragma unroll
            for (int i = 0; i < 6; ++i) u[i] = pool->field[33 + i][slot];
#pragma unroll
            for (int i = 0; i < 11; ++i) gs[i] = T(0);
            const T w = weight ? weight[b] : T(1);
            const T l = cn::body_loss_epilogue_pts<T, kWfUnrPE, true>(P, S, A, u, n_c, w, want_grad ? gs : (T*)nullptr,
                                                                      grad_pts ? grad_pts + b * 12 : (T*)nullptr,
                                                                      force ? fo : (T*)nullptr);
            if (force) {
#pragma unroll
              for (int i = 0; i < 12; ++i) force[b * 12 + i] = fo[i];
            }
#pragma unroll
            for (int i = 0; i < 11; ++i) acc[i] += w * gs[i];
            if (loss) loss[b] = l;
            acc[11] += l;
            if (iters) iters[b] = pool->iters[slot] & 0xff;
            if (u_out) {
#pragma unroll
              for (int i = 0; i < 6; ++i) u_out[b * 6 + i] = u[i];
            }
            pool->sample[slot] = -1;
          } else {
            T us[6];
            if (u_init) {
#pragma unroll
              for (int i = 0; i < 6; ++i) us[i] = u_init[b * 6 + i];
            } else {
              cn::cube_loss_start<T>(A, T(CN_LOSS_START_FACTOR), us);
            }
#pragma unroll
            for (int i = 0; i < 6; ++i) pool->field[33 + i][slot] = us[i];
            pool->field[39][slot] = T(-1);
            pool->field[46][slot] = T(0);
            pool->sample[slot] = (int32_t)(b - lo);
            pool->iters[slot] = 0;
            to_active = true;
          }
        }
      }
      h_in = (h_in + n_new) % kWfQin; n_in -= n_new;
      const bool more = next < hi || n_in > 0;
      __syncwarp();
      const unsigned m_act = __ballot_sync(0xffffffffu, to_active);
      const unsigned m_keep = __ballot_sync(0xffffffffu, on && !to_active && more);
      h_done = (h_done + k) % kWfSlots; n_done -= k;
      if (to_active) pool->q_act[(h_act + n_act + __popc(m_act & lt_mask)) % kWfSlots] = (uint8_t)slot;
      else if (on && more) pool->q_done[(h_done + n_done + __popc(m_keep & lt_mask)) % kWfSlots] = (uint8_t)slot;
      n_act += __popc(m_act); n_done += __popc(m_keep);
    }
    __syncwarp();
  }

  if (!partials) return;
  __shared__ T red[kWfWarps][kNAcc];
#pragma unroll 1
  for (int i = 0; i < 12; ++i) {
    T v = T(0);
#pragma unroll
    for (int j = 0; j < 12; ++j) v = (j == i) ? acc[j] : v;
    const T s = warp_sum(v);
    if (lane == 0) red[warp][i] = s;
  }
  __syncthreads();
  if (threadIdx.x < kNAcc) {
    T s = T(0);
    if (threadIdx.x < 12) {
#pragma unroll
      for (int w = 0; w < kWfWarps; ++w) s += red[w][threadIdx.x];
    }
    partials[(int64_t)blockIdx.x * kNAcc + threadIdx.x] = s;
  }
}

// ---- leaf-level parameter preparation / chain rule (cube: theta 10, friction 2 [box, ground], length 3) ----

template <typename T, typename IO>
__global__ void cube_prep_kernel(const IO* __restrict__ theta, const IO* __restrict__ friction,
                                 const IO* __restrict__ length, IO* __restrict__ params /* [inertia 10 | mu 1 | half 3] */,
                                 const int32_t* __restrict__ skip_flag) {
  if (skip_flag && *skip_flag) return;
  if (threadIdx.x == 0) {
    T th[10], out[10];
    for (int i = 0; i < 10; ++i) th[i] = T(theta[i]);
    cn::theta_to_inertia_vector<T>(th, out);
    for (int i = 0; i < 10; ++i) params[i] = IO(out[i]);
    const T a = cn::t_abs(T(friction[0])), b = cn::t_abs(T(friction[1]));
    params[10] = IO(T(2) * a * b / (a + b));
    for (int i = 0; i < 3; ++i) params[11 + i] = IO(cn::t_abs(T(length[i])));
  }
}

// Sums the per-block partials (fixed order) and pushes the callable-level gradient through the
// parameter preparation: grad_leaf = [d/d theta (10) | d/d friction (2) | d/d length (3)].
// Data-parallel step (comm != nullptr): the same block then performs the step's only exchange itself --
// [grad_leaf 15 | loss sum | sample count] is pushed into every peer's buffer over NVLink and the world's rows
// are summed in rank order (cn_comm.cuh), so no host-launched collective follows the kernel.  `sums` (17) /
// `means` (16) receive the (global) sums and the sums divided by the sample count; `local_out` (16, nullable)
// keeps this rank's own [grad_leaf | loss sum].
template <typename T, typename IO>
__global__ void reduce_partials_leaf_kernel(const T* __restrict__ partials, int nblocks, const IO* __restrict__ theta,
                                            const IO* __restrict__ friction, const IO* __restrict__ length,
                                            IO* __restrict__ grad_leaf, IO* __restrict__ loss_sum,
                                            const int32_t* __restrict__ skip_flag, cn::CommDev* comm, double count,
                                            IO* __restrict__ sums, IO* __restrict__ means, IO* __restrict__ local_out) {
  if (skip_flag && *skip_flag) return;
  __shared__ T g[kNAcc];
  __shared__ double o[cn::COMM_MAX_ELEMS];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (w < kNAcc) {
    T s = T(0);
    for (int b = lane; b < nblocks; b += 32) s += partials[(int64_t)b * kNAcc + w];
    s = warp_sum(s);
    if (lane == 0) g[w] = s;
  }
  __syncthreads();
  const int t = threadIdx.x;
  if (t < 10) {
    cn::Dual<T> th[10], out[10];
    for (int i = 0; i < 10; ++i) th[i] = cn::Dual<T>(T(theta[i]), i == t ? T(1) : T(0));
    cn::theta_to_inertia_vector<cn::Dual<T>>(th, out);
    T s = T(0);
    for (int i = 0; i < 10; ++i) s += g[i] * out[i].d;
    o[t] = (double)s;
  } else if (t == 10) {
    const T fa = T(friction[0]), fb = T(friction[1]);
    const T a = cn::t_abs(fa), b = cn::t_abs(fb), den = (a + b) * (a + b);
    const T sa = fa > T(0) ? T(1) : (fa < T(0) ? T(-1) : T(0)), sb = fb > T(0) ? T(1) : (fb < T(0) ? T(-1) : T(0));
    o[10] = (double)(g[10] * (T(2) * b * b / den) * sa);
    o[11] = (double)(g[10] * (T(2) * a * a / den) * sb);
  } else if (t >= 11 && t < 14) {
    const T l = T(length[t - 11]);
    o[12 + (t - 11)] = (double)(g[t] * (l > T(0) ? T(1) : (l < T(0) ? T(-1) : T(0))));
  } else if (t == 14) {
    o[15] = (double)g[14];
  } else if (t == 15) {
    o[16] = count;
  }
  __syncthreads();
  if (local_out && t < 16) local_out[t] = IO(o[t]);
  if (comm) cn::comm_allreduce_block(comm, o, 17);
  if (t < 15 && grad_leaf) grad_leaf[t] = IO(o[t]);
  else if (t == 15 && loss_sum) *loss_sum = IO(o[15]);
  if (sums && t < 17) sums[t] = IO(o[t]);                    // [grad_leaf 15 | loss sum | sample count]
  if (means && t < 16) means[t] = IO(o[t] / o[16]);          // the same per sample: loss.mean() and its gradient
}

template <typename T, typename IO>
__global__ void __launch_bounds__(kLossThreads)
cube_rollout_kernel(const IO* __restrict__ x0, const IO* __restrict__ inertia, const IO* __restrict__ mu,
                    const IO* __restrict__ half, T dt, T eps, int64_t B, int steps, IO* __restrict__ traj,
                    IO* __restrict__ force, int32_t* __restrict__ iters, int lanes_per_warp, IO* __restrict__ usol) {
  // A toss is a sequential chain of `steps` solves whose lengths differ per toss, and a warp advances
  // at the pace of its slowest lane: small batches are therefore spread thinly (lanes_per_warp < 32
  // tosses per warp) so that every SM sub-partition holds warps and each waits for few neighbours.
  const int lane = threadIdx.x & 31;
  if (lane >= lanes_per_warp) return;
  cn::CubeParams<T> P;
  load_cube_params<T, IO>(P, inertia, mu, half, dt, eps);
  const cn::SolverCfg<T> cfg = cn::default_cfg<T>();
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t stride = (((int64_t)gridDim.x * blockDim.x) >> 5) * lanes_per_warp;
  for (int64_t b = warp * lanes_per_warp + lane; b < B; b += stride) {
    T xc[13], xn[13], fo[12];
    IO* out = traj + b * (int64_t)(steps + 1) * 13;
#pragma unroll
    for (int i = 0; i < 13; ++i) { xc[i] = T(x0[b * 13 + i]); out[i] = IO(xc[i]); }
    int total = 0;
    T warm[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
    for (int s = 0; s < steps; ++s) {
      total += cn::cube_step_sample<T>(P, cfg, xc, xn, force ? fo : nullptr, warm);
      if (usol) {                      // the step's QP optimum, for the reverse-mode backward (cn_cube_adjoint.cuh)
#pragma unroll
        for (int i = 0; i < 6; ++i) usol[(b * steps + s) * 6 + i] = IO(warm[i]);
      }
      if (force) {
#pragma unroll
        for (int i = 0; i < 12; ++i) force[(b * steps + s) * 12 + i] = IO(fo[i]);
      }
#pragma unroll
      for (int i = 0; i < 13; ++i) { xc[i] = xn[i]; out[(int64_t)(s + 1) * 13 + i] = IO(xn[i]); }
    }
    if (iters) iters[b] = total;
  }
}

template <typename T, typename IO>
__global__ void __launch_bounds__(kLossThreads)
body_pts_step_kernel(const IO* __restrict__ x, const IO* __restrict__ inertia, const IO* __restrict__ mu,
                     const IO* __restrict__ pts, int n_c, T dt, T eps, int64_t B, IO* __restrict__ xn,
                     IO* __restrict__ force) {
  cn::CubeParams<T> P;
  {
    T in[10], m[1], h[3] = {T(0), T(0), T(0)};
#pragma unroll
    for (int i = 0; i < 10; ++i) in[i] = T(inertia[i]);
    m[0] = T(mu[0]);
    cn::cube_params_init(P, in, m, h, dt, eps);
  }
  const cn::SolverCfg<T> cfg = cn::default_cfg<T>();
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  T xs[13], pt[12], xo[13], fo[12];
#pragma unroll
  for (int i = 0; i < 13; ++i) xs[i] = T(x[b * 13 + i]);
#pragma unroll
  for (int i = 0; i < 12; ++i) pt[i] = T(pts[b * 12 + i]);
  cn::body_step_sample_pts<T>(P, cfg, xs, pt, n_c, xo, force ? fo : (T*)nullptr);
#pragma unroll
  for (int i = 0; i < 13; ++i) xn[b * 13 + i] = IO(xo[i]);
  if (force) {
#pragma unroll
    for (int i = 0; i < 12; ++i) force[b * 12 + i] = IO(fo[i]);
  }
}

// Dense terms export (MultibodyTerms.forward, multibody_terms.py:584-609): one sample per thread.
template <typename T, typename IO>
__global__ void __launch_bounds__(kLossThreads)
cube_terms_kernel(const IO* __restrict__ q, const IO* __restrict__ v, const IO* __restrict__ inertia,
                  const IO* __restrict__ mu, const IO* __restrict__ half, int64_t B, IO* __restrict__ M,
                  IO* __restrict__ J, IO* __restrict__ phi, IO* __restrict__ acc, IO* __restrict__ D) {
  cn::CubeParams<T> P;
  load_cube_params<T, IO>(P, inertia, mu, half, T(1), T(1));
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  T qs[7], vs[6], Mo[36], Jo[72], po[4], ao[6], Do[144];
  for (int i = 0; i < 7; ++i) qs[i] = T(q[b * 7 + i]);
  for (int i = 0; i < 6; ++i) vs[i] = T(v[b * 6 + i]);
  cn::cube_terms_sample<T>(P, qs, vs, Mo, Jo, po, ao, D ? Do : (T*)nullptr);
  for (int i = 0; i < 36; ++i) M[b * 36 + i] = IO(Mo[i]);
  for (int i = 0; i < 72; ++i) J[b * 72 + i] = IO(Jo[i]);
  for (int i = 0; i < 4; ++i) phi[b * 4 + i] = IO(po[i]);
  for (int i = 0; i < 6; ++i) acc[b * 6 + i] = IO(ao[i]);
  if (D) for (int i = 0; i < 144; ++i) D[b * 144 + i] = IO(Do[i]);
}

// ---------------------------------------------------------------------------
// Elbow (floating base + hinge, 8 contacts): the loss kernel is the wavefront kernel in cn_elbow_wf.cu; rollout
// and terms run one sample per thread, problem in thread-local arrays.
// ---------------------------------------------------------------------------
template <typename T, typename IO>
__device__ __forceinline__ void load_elbow_params(cn::ElbowParams<T>& P, const IO* inertia, const IO* mu, const IO* half,
                                                  const IO* kin, T dt, T eps) {
  T in[20], m[2], h[6], kn[cn::EL_NKIN];
  for (int i = 0; i < 20; ++i) in[i] = T(inertia[i]);
  for (int i = 0; i < 2; ++i) m[i] = T(mu[i]);
  for (int i = 0; i < 6; ++i) h[i] = half ? T(half[i]) : T(0);
  for (int i = 0; i < cn::EL_NKIN; ++i) kn[i] = T(kin[i]);
  cn::elbow_params_init(P, in, m, h, kn, dt, eps);
}

template <typename T, typename IO>
__global__ void __launch_bounds__(kLossThreads)
elbow_rollout_kernel(const IO* __restrict__ x0, const IO* __restrict__ inertia, const IO* __restrict__ mu,
                     const IO* __restrict__ half, const IO* __restrict__ kin, const IO* __restrict__ pts, T dt, T eps,
                     int64_t B, int steps, IO* __restrict__ traj, IO* __restrict__ force, int32_t* __restrict__ iters,
                     int lanes_per_warp, IO* __restrict__ usol) {
  const int lane = threadIdx.x & 31;              // small batches are spread thinly, as in cube_rollout_kernel
  if (lane >= lanes_per_warp) return;
  cn::ElbowParams<T> P;
  load_elbow_params<T, IO>(P, inertia, mu, half, kin, dt, eps);
  const cn::SolverCfg<T> cfg = cn::default_cfg<T>();
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t stride = (((int64_t)gridDim.x * blockDim.x) >> 5) * lanes_per_warp;
  for (int64_t b = warp * lanes_per_warp + lane; b < B; b += stride) {
    T xc[15], xn[15], fo[24], pt[24];
    IO* out = traj + b * (int64_t)(steps + 1) * 15;
    for (int i = 0; i < 15; ++i) { xc[i] = T(x0[b * 15 + i]); out[i] = IO(xc[i]); }
    if (pts) for (int i = 0; i < 24; ++i) pt[i] = T(pts[b * 24 + i]);
    int total = 0;
    for (int s = 0; s < steps; ++s) {
      T us[7];
      total += cn::elbow_step_sample_wf<T>(P, cfg, xc, pts ? pt : (const T*)nullptr, xn, force ? fo : (T*)nullptr,
                                           usol ? us : (T*)nullptr);
      if (usol) for (int i = 0; i < 7; ++i) usol[(b * steps + s) * 7 + i] = IO(us[i]);
      if (force) for (int i = 0; i < 24; ++i) force[(b * steps + s) * 24 + i] = IO(fo[i]);
      for (int i = 0; i < 15; ++i) { xc[i] = xn[i]; out[(int64_t)(s + 1) * 15 + i] = IO(xn[i]); }
    }
    if (iters) iters[b] = total;
  }
}

// Dense terms export for the two-body system (MultibodyTerms.forward, multibody_terms.py:584-609).  One sample per
// thread; the 24x24 Delassus block makes it 6.9 KB written per sample -- an HBM-bound export for callers that ask
// for the matrices (the loss / step kernels never form them).
template <typename T, typename IO>
__global__ void __launch_bounds__(64)
elbow_terms_kernel(const IO* __restrict__ q, const IO* __restrict__ v, const IO* __restrict__ inertia,
                   const IO* __restrict__ mu, const IO* __restrict__ half, const IO* __restrict__ kin, int64_t B,
                   IO* __restrict__ M, IO* __restrict__ J, IO* __restrict__ phi, IO* __restrict__ acc, IO* __restrict__ D) {
  cn::ElbowParams<T> P;
  load_elbow_params<T, IO>(P, inertia, mu, half, kin, T(1), T(1));
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  T qs[8], vs[7], Mo[49], Jo[168], po[8], ao[7];
  for (int i = 0; i < 8; ++i) qs[i] = T(q[b * 8 + i]);
  for (int i = 0; i < 7; ++i) vs[i] = T(v[b * 7 + i]);
  T* Do = D ? reinterpret_cast<T*>(D + b * 576) : (T*)nullptr;        // T == IO here: assembled in place
  cn::elbow_terms_sample<T>(P, qs, vs, Mo, Jo, po, ao, Do);
  for (int i = 0; i < 49; ++i) M[b * 49 + i] = IO(Mo[i]);
  for (int i = 0; i < 168; ++i) J[b * 168 + i] = IO(Jo[i]);
  for (int i = 0; i < 8; ++i) phi[b * 8 + i] = IO(po[i]);
  for (int i = 0; i < 7; ++i) acc[b * 7 + i] = IO(ao[i]);
}

template <typename T>
__global__ void __launch_bounds__(256) fma_peak_kernel(T* out, int64_t iters) {
  T a[16];
  const T m = T(1) + T(1e-9) * T(threadIdx.x), c = T(1e-12);
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = T(i) + T(blockIdx.x) * T(1e-6);
  for (int64_t k = 0; k < iters; ++k) {
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = a[i] * m + c;
  }
  T s = T(0);
#pragma unroll
  for (int i = 0; i < 16; ++i) s += a[i];
  out[(int64_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// Grid and tosses per warp of a rollout launch (rollout_tosses_per_warp): at most one resident set of blocks.
template <typename K>
int rollout_grid(K kernel, int64_t B, int* blocks, int* lpw) {
  int sms = 0;
  int64_t cap;
  if (int rc = cn::sm_count(&sms)) return rc;
  if (int rc = cn::resident_cap(kernel, kLossThreads, 0, INT64_MAX, &cap)) return rc;
  *lpw = rollout_tosses_per_warp(B, sms, cap * (kLossThreads / 32));
  const int64_t per_block = (int64_t)*lpw * (kLossThreads / 32);
  const int64_t need = (B + per_block - 1) / per_block;
  *blocks = (int)(need < cap ? need : cap);
  return DPLL_OK;
}

constexpr int64_t kRaceMaxBatch = 300000;     // larger launches are bound by throughput, not by their longest chain
constexpr int64_t kRaceMaxHead = 2048;

// Wavefront loss launch of the single body: box corners, or witness points (PTS; the arguments are packed as
// cube_loss_wf_kernel describes).  Sets the shared-memory size of every instance it may launch, picks the grid and the
// instance by batch size, resets the chunk counter of the dynamic schedule and launches.  *rows = the number of blocks
// that write partials.
template <typename T, typename IO, bool PTS>
int launch_cube_wf(bool dynamic, int flags, const IO* x, const IO* xp, const IO* weight, const IO* inertia, const IO* mu,
                   const IO* half, T dt, T eps, int64_t B, IO* loss, IO* force, int32_t* iters, T* partials,
                   int want_grad, const int32_t* skip_flag, void* workspace, size_t workspace_bytes, cudaStream_t st,
                   int64_t ldx, int64_t ldxp, const IO* u_init, IO* u_out, int* rows) {
  const size_t smem = sizeof(WfWarpPool<T>) * kWfWarps;
  cudaError_t ea = cudaFuncSetAttribute(cube_loss_wf_kernel<T, IO, kWfUnr, false, PTS>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (ea == cudaSuccess)
    ea = cudaFuncSetAttribute(cube_loss_wf_kernel<T, IO, 4, false, PTS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)smem);
  if constexpr (!PTS) {
    if (ea == cudaSuccess)
      ea = cudaFuncSetAttribute(cube_loss_wf_kernel<T, IO, 4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  if (ea != cudaSuccess) return (int)ea;
  // at most one resident set of blocks, fewer for small batches -- a warp needs a few hundred samples to keep its pool
  // full; with fewer, every SM would run many mostly-empty warps at the issue rate of full ones
  int blocks;
  int64_t cap;
  if (int rc = cn::resident_blocks(cube_loss_wf_kernel<T, IO, kWfUnr, false, PTS>, kWfWarps * 32, smem,
                                   (B + kWfWarps * kWfMinPerWarp - 1) / (kWfWarps * kWfMinPerWarp), kMaxBlocks,
                                   &blocks, &cap))
    return rc;
  unsigned long long* dyn = nullptr;
  if (dynamic) {
    if (!cn::workspace_ok(workspace, workspace_bytes)) return DPLL_EWORKSPACE;
    if (int rc = cn::dynamic_counter(workspace, st, &dyn)) return rc;
  }
  // Up to ~320 samples per warp (crossover measured around 400) the launch is a few long Newton chains per warp: the
  // instance with the per-contact loop of the Newton visit unrolled overlaps the four contacts (measured -8% at
  // 65,536 pairs, -5% at 262,144).  Larger batches keep every warp's pool full and run the rolled instance,
  // which is smaller in the instruction cache (the unrolled one is +5% at 1M pairs, +15% at 4M).
  const bool small = B <= cap * kWfWarps * 320;
  if constexpr (!PTS) {
    // DPLL_LOSS_RACE: the head of a cost-ordered batch goes to racing blocks at the front of the same grid, the
    // wavefront blocks take the rest.  Only for launches bounded by their longest chain (small shards), and only for
    // cold solves.
    if ((flags & DPLL_LOSS_RACE) && dynamic && small && !u_init && B >= 4096 && B <= kRaceMaxBatch) {
      int64_t head = B / 64;
      if (head > kRaceMaxHead) head = kRaceMaxHead;
      head -= head % (kWfWarps * kRaceSamples);
      const int race_blocks = (int)(head / (kWfWarps * kRaceSamples));
      // an SM holds two blocks: leave the racing blocks their share of the resident set
      if (blocks > cap - race_blocks) blocks = (int)(cap - race_blocks > 1 ? cap - race_blocks : 1);
      if (race_blocks > 0) {
        cube_loss_wf_kernel<T, IO, 4, true><<<race_blocks + blocks, kWfWarps * 32, smem, st>>>(
            x, xp, weight, inertia, mu, half, dt, eps, B, loss, force, iters, partials, want_grad, skip_flag, dyn, ldx,
            ldxp, u_init, u_out, race_blocks, head);
        *rows = race_blocks + blocks;
        return cn::launch_status();
      }
    }
  }
  auto kernel = small ? cube_loss_wf_kernel<T, IO, 4, false, PTS> : cube_loss_wf_kernel<T, IO, kWfUnr, false, PTS>;
  kernel<<<blocks, kWfWarps * 32, smem, st>>>(x, xp, weight, inertia, mu, half, dt, eps, B, loss, force, iters, partials,
                                              want_grad, skip_flag, dyn, ldx, ldxp, u_init, u_out, 0, 0);
  *rows = blocks;
  return cn::launch_status();
}

template <typename T, typename IO>
int launch_cube_loss(int variant, const IO* x, const IO* xp, const IO* weight, const IO* inertia, const IO* mu,
                     const IO* half, const IO* theta, const IO* friction, const IO* length, T dt, T eps, int64_t B,
                     IO* loss, IO* force, int32_t* iters, IO* grad, IO* loss_sum,
                     const int32_t* skip_flag, void* workspace, size_t workspace_bytes, void* stream, int flags = 0,
                     cn::CommDev* comm = nullptr, IO* sums = nullptr, IO* means = nullptr, IO* local_out = nullptr,
                     int64_t ldx = 13, int64_t ldxp = 13, const IO* u_init = nullptr, IO* u_out = nullptr) {
  const bool leaf = theta != nullptr;
  if (ldx < 13 || ldxp < 13) return DPLL_EINVAL;
  if ((u_init || u_out) && variant == 1) return DPLL_EINVAL;      // warm starts live in the wavefront kernel
  if (flags & DPLL_LOSS_DYNAMIC) variant = 2;
  if (comm && (!leaf || skip_flag)) return DPLL_EINVAL;   // the exchange lives in the leaf reduction and is unconditional
  if (B < 0 || (leaf ? (!friction || !length) : (!inertia || !mu || !half))) return DPLL_EINVAL;
  if (B > 0 && (!x || !xp)) return DPLL_EINVAL;
  const bool want_red = grad || loss_sum || comm || sums || means;
  if ((want_red || leaf) && !cn::workspace_ok(workspace, workspace_bytes)) return DPLL_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  T* partials = want_red ? static_cast<T*>(workspace) : nullptr;
  if (leaf) {
    // callable-level parameters are produced on the device, behind the partials in the workspace
    IO* params = reinterpret_cast<IO*>(static_cast<char*>(workspace) + cn::kWsParamsOffset);
    cube_prep_kernel<T, IO><<<1, 32, 0, st>>>(theta, friction, length, params, skip_flag);
    inertia = params; mu = params + 10; half = params + 11;
  }
  const int want_grad = (grad || sums || means) ? 1 : 0;
  int rows;
  if (variant == 0 || variant == 2) {
    if (int rc = launch_cube_wf<T, IO, false>(variant == 2, flags, x, xp, weight, inertia, mu, half, dt, eps, B, loss,
                                              force, iters, partials, want_grad, skip_flag, workspace, workspace_bytes,
                                              st, ldx, ldxp, u_init, u_out, &rows))
      return rc;
  } else {
    int64_t cap;
    if (int rc = cn::resident_blocks(cube_loss_kernel<T, IO>, kLossThreads, 0, (B + kLossThreads - 1) / kLossThreads,
                                     kMaxBlocks, &rows, &cap))
      return rc;
    cube_loss_kernel<T, IO><<<rows, kLossThreads, 0, st>>>(x, xp, weight, inertia, mu, half, dt, eps, B, loss, force,
                                                           iters, partials, want_grad, skip_flag, ldx, ldxp);
    if (int rc = cn::launch_status()) return rc;
  }
  if (!want_red) return DPLL_OK;
  if (leaf) reduce_partials_leaf_kernel<T, IO><<<1, 32 * kNAcc, 0, st>>>(partials, rows, theta, friction, length, grad,
                                                                        loss_sum, skip_flag, comm, (double)B, sums, means,
                                                                        local_out);
  else reduce_partials_kernel<T, IO, kNAcc, DPLL_CUBE_NPARAM><<<1, 32 * kNAcc, 0, st>>>(partials, rows, grad, loss_sum,
                                                                                       skip_flag);
  return cn::launch_status();
}

template <typename T, typename IO>
int launch_cube_rollout(const IO* x0, const IO* inertia, const IO* mu, const IO* half, T dt, T eps, int64_t B,
                        int32_t steps, IO* traj, IO* force, int32_t* iters, void* stream, IO* usol = nullptr) {
  if (B < 0 || steps < 0 || !inertia || !mu || !half) return DPLL_EINVAL;
  if (B > 0 && (!x0 || !traj)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  int blocks, lpw;
  if (int rc = rollout_grid(cube_rollout_kernel<T, IO>, B, &blocks, &lpw)) return rc;
  cube_rollout_kernel<T, IO><<<blocks, kLossThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x0, inertia, mu, half, dt, eps, B, steps, traj, force, iters, lpw, usol);
  return cn::launch_status();
}

template <typename T, typename IO>
int launch_elbow_rollout(const IO* x0, const IO* inertia, const IO* mu, const IO* half, const IO* kin, const IO* pts,
                         T dt, T eps, int64_t B, int32_t steps, IO* traj, IO* force, int32_t* iters, void* stream,
                         IO* usol = nullptr) {
  if (B < 0 || steps < 0 || !inertia || !mu || (!half && !pts) || !kin || (pts && steps > 1)) return DPLL_EINVAL;
  if (B > 0 && (!x0 || !traj)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  int blocks, lpw;
  if (int rc = rollout_grid(elbow_rollout_kernel<T, IO>, B, &blocks, &lpw)) return rc;
  elbow_rollout_kernel<T, IO><<<blocks, kLossThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x0, inertia, mu, half, kin, pts, dt, eps, B, steps, traj, force, iters, lpw, usol);
  return cn::launch_status();
}

}  // namespace

extern "C" {

// Cube loss kernel selector for A/B measurements (0 = wavefront, static ranges [default, deterministic];
// 1 = one sample per thread; 2 = wavefront with dynamic sample distribution [not bitwise reproducible]).
// The elbow loss always runs its wavefront kernel.
static int g_loss_variant = 0;
int dpll_set_loss_variant(int variant) {
  if (variant < 0 || variant > 2) return DPLL_EINVAL;
  g_loss_variant = variant;
  return DPLL_OK;
}

int dpll_version(void) { return DPLL_VERSION; }

size_t dpll_workspace_bytes(void) { return cn::kWsBytes; }

int dpll_cube_loss_f64(const double* x, const double* x_plus, const double* weight, const double* inertia,
                       const double* mu_pair, const double* half, double dt, double eps, int64_t B, double* loss,
                       double* force, int32_t* iters, double* grad, double* loss_sum, const int32_t* skip_flag,
                       void* workspace, size_t workspace_bytes, void* stream) {
  return launch_cube_loss<double, double>(g_loss_variant, x, x_plus, weight, inertia, mu_pair, half, nullptr, nullptr, nullptr,
                                  dt, eps, B, loss, force, iters, grad, loss_sum, skip_flag, workspace,
                                  workspace_bytes, stream);
}

int dpll_cube_loss_leaf_f64(const double* x, const double* x_plus, const double* weight, const double* theta,
                            const double* friction, const double* length, double dt, double eps, int64_t B,
                            double* loss, double* force, int32_t* iters, double* grad_leaf, double* loss_sum,
                            const int32_t* skip_flag, void* workspace, size_t workspace_bytes, void* stream) {
  if (!theta) return DPLL_EINVAL;
  return launch_cube_loss<double, double>(g_loss_variant, x, x_plus, weight, nullptr, nullptr, nullptr, theta, friction, length,
                                  dt, eps, B, loss, force, iters, grad_leaf, loss_sum, skip_flag, workspace,
                                  workspace_bytes, stream);
}

int dpll_cube_loss_f32(const float* x, const float* x_plus, const float* weight, const float* inertia,
                       const float* mu_pair, const float* half, float dt, float eps, int64_t B, float* loss,
                       float* force, int32_t* iters, float* grad, float* loss_sum, const int32_t* skip_flag,
                       void* workspace, size_t workspace_bytes, void* stream) {
  return launch_cube_loss<double, float>(g_loss_variant, x, x_plus, weight, inertia, mu_pair, half, nullptr, nullptr, nullptr,
                                 (double)dt, (double)eps, B, loss, force, iters, grad, loss_sum, skip_flag, workspace,
                                 workspace_bytes, stream);
}

int dpll_cube_loss_leaf_f32(const float* x, const float* x_plus, const float* weight, const float* theta,
                            const float* friction, const float* length, float dt, float eps, int64_t B, float* loss,
                            float* force, int32_t* iters, float* grad_leaf, float* loss_sum, const int32_t* skip_flag,
                            void* workspace, size_t workspace_bytes, void* stream) {
  if (!theta) return DPLL_EINVAL;
  return launch_cube_loss<double, float>(g_loss_variant, x, x_plus, weight, nullptr, nullptr, nullptr, theta, friction,
                                         length, (double)dt, (double)eps, B, loss, force, iters, grad_leaf, loss_sum,
                                         skip_flag, workspace, workspace_bytes, stream);
}

int dpll_cube_loss_leaf_dp_f64(const double* x, int64_t x_row_stride, const double* x_plus, int64_t xp_row_stride,
                               const double* theta, const double* friction, const double* length, double dt, double eps,
                               int64_t B, int32_t flags, void* comm, const double* u_init, double* u_out, double* loss,
                               int32_t* iters, double* sums, double* means, double* local, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (!theta || (!sums && !means)) return DPLL_EINVAL;
  return launch_cube_loss<double, double>(g_loss_variant, x, x_plus, nullptr, nullptr, nullptr, nullptr, theta, friction, length,
                                          dt, eps, B, loss, nullptr, iters, nullptr, nullptr, nullptr, workspace,
                                          workspace_bytes, stream, flags,
                                          static_cast<cn::CommDev*>(dpll_comm_device_state(comm)), sums, means, local,
                                          x_row_stride, xp_row_stride, u_init, u_out);
}

int dpll_cube_loss_leaf_dp_f32(const float* x, int64_t x_row_stride, const float* x_plus, int64_t xp_row_stride,
                               const float* theta, const float* friction, const float* length, float dt, float eps,
                               int64_t B, int32_t flags, void* comm, const float* u_init, float* u_out, float* loss,
                               int32_t* iters, float* sums, float* means, float* local, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (!theta || (!sums && !means)) return DPLL_EINVAL;
  return launch_cube_loss<double, float>(g_loss_variant, x, x_plus, nullptr, nullptr, nullptr, nullptr, theta, friction, length,
                                         (double)dt, (double)eps, B, loss, nullptr, iters, nullptr, nullptr, nullptr,
                                         workspace, workspace_bytes, stream, flags,
                                         static_cast<cn::CommDev*>(dpll_comm_device_state(comm)), sums, means, local,
                                         x_row_stride, xp_row_stride, u_init, u_out);
}

int dpll_cube_rollout_f64(const double* x0, const double* inertia, const double* mu_pair, const double* half,
                          double dt, double eps, int64_t B, int32_t steps, double* traj, double* force,
                          int32_t* iters, void* stream) {
  return launch_cube_rollout<double, double>(x0, inertia, mu_pair, half, dt, eps, B, steps, traj, force, iters, stream);
}

int dpll_cube_rollout_saved_f64(const double* x0, const double* inertia, const double* mu_pair, const double* half,
                                double dt, double eps, int64_t B, int32_t steps, double* traj, double* usol,
                                void* stream) {
  if (B > 0 && steps > 0 && !usol) return DPLL_EINVAL;
  return launch_cube_rollout<double, double>(x0, inertia, mu_pair, half, dt, eps, B, steps, traj, nullptr, nullptr, stream,
                                             usol);
}

int dpll_cube_rollout_f32(const float* x0, const float* inertia, const float* mu_pair, const float* half, float dt,
                          float eps, int64_t B, int32_t steps, float* traj, float* force, int32_t* iters,
                          void* stream) {
  return launch_cube_rollout<double, float>(x0, inertia, mu_pair, half, (double)dt, (double)eps, B, steps, traj, force,
                                            iters, stream);
}

int dpll_body_loss_pts_f64(const double* x, const double* x_plus, const double* weight, const double* inertia,
                           const double* mu_pair, const double* pts, int32_t n_contacts, double dt, double eps, int64_t B,
                           int32_t flags, double* loss, double* force, double* grad_pts, int32_t* iters, double* grad,
                           double* loss_sum, const int32_t* skip_flag, void* workspace, size_t workspace_bytes,
                           void* stream) {
  if (B < 0 || !inertia || !mu_pair || n_contacts < 1 || n_contacts > DPLL_CUBE_NC) return DPLL_EINVAL;
  if (B > 0 && (!x || !x_plus || !pts)) return DPLL_EINVAL;
  const bool want_red = grad || loss_sum;
  const bool dynamic = (flags & DPLL_LOSS_DYNAMIC) != 0;
  if ((want_red || dynamic) && !cn::workspace_ok(workspace, workspace_bytes)) return DPLL_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double* partials = want_red ? static_cast<double*>(workspace) : nullptr;
  // the box's wavefront launch, witness-point instance: the points travel in `half`, grad_pts in `u_out`, n_contacts
  // in the upper bits of `want_grad` (see the kernel)
  int rows;
  if (int rc = launch_cube_wf<double, double, true>(dynamic, flags, x, x_plus, weight, inertia, mu_pair, pts, dt, eps, B,
                                                    loss, force, iters, partials, (grad ? 1 : 0) | (n_contacts << 1),
                                                    skip_flag, workspace, workspace_bytes, st, 13, 13, nullptr, grad_pts,
                                                    &rows))
    return rc;
  if (!want_red) return DPLL_OK;
  reduce_partials_kernel<double, double, kNAcc, 11><<<1, 32 * kNAcc, 0, st>>>(partials, rows, grad, loss_sum, skip_flag);
  return cn::launch_status();
}

int dpll_body_loss_pts_warm_f64(const double* x, const double* x_plus, const double* weight, const double* inertia,
                                const double* mu_pair, const double* pts, int32_t n_contacts, double dt, double eps,
                                int64_t B, int32_t flags, double* loss, double* force, double* grad_pts, int32_t* iters,
                                double* grad, double* loss_sum, const int32_t* skip_flag, const double* u_init,
                                double* u_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!u_init && !u_out)      // exactly what dpll_body_loss_pts_f64 launches
    return dpll_body_loss_pts_f64(x, x_plus, weight, inertia, mu_pair, pts, n_contacts, dt, eps, B, flags, loss, force,
                                  grad_pts, iters, grad, loss_sum, skip_flag, workspace, workspace_bytes, stream);
  if (B < 0 || !inertia || !mu_pair || n_contacts < 1 || n_contacts > DPLL_CUBE_NC) return DPLL_EINVAL;
  if (B > 0 && (!x || !x_plus || !pts)) return DPLL_EINVAL;
  const bool want_red = grad || loss_sum;
  const bool dynamic = (flags & DPLL_LOSS_DYNAMIC) != 0;
  if ((want_red || dynamic) && !cn::workspace_ok(workspace, workspace_bytes)) return DPLL_EWORKSPACE;
  if (B == 0 && !want_red) return DPLL_OK;      // nothing to write: an empty warm call launches nothing
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double* partials = want_red ? static_cast<double*>(workspace) : nullptr;
  // the grid and instance policy of launch_cube_wf
  const size_t smem = sizeof(WfWarpPool<double>) * kWfWarps;
  cudaError_t ea = cudaFuncSetAttribute(body_loss_pts_warm_kernel<kWfUnr>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)smem);
  if (ea == cudaSuccess)
    ea = cudaFuncSetAttribute(body_loss_pts_warm_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (ea != cudaSuccess) return (int)ea;
  int blocks;
  int64_t cap;
  if (int rc = cn::resident_blocks(body_loss_pts_warm_kernel<kWfUnr>, kWfWarps * 32, smem,
                                   (B + kWfWarps * kWfMinPerWarp - 1) / (kWfWarps * kWfMinPerWarp), kMaxBlocks,
                                   &blocks, &cap))
    return rc;
  unsigned long long* dyn = nullptr;
  if (dynamic)
    if (int rc = cn::dynamic_counter(workspace, st, &dyn)) return rc;
  const bool small = B <= cap * kWfWarps * 320;
  auto kernel = small ? body_loss_pts_warm_kernel<4> : body_loss_pts_warm_kernel<kWfUnr>;
  kernel<<<blocks, kWfWarps * 32, smem, st>>>(x, x_plus, weight, inertia, mu_pair, pts, n_contacts, dt, eps, B, loss, force,
                                              grad_pts, iters, partials, grad ? 1 : 0, skip_flag, dyn, u_init, u_out);
  if (int rc = cn::launch_status()) return rc;
  if (!want_red) return DPLL_OK;
  reduce_partials_kernel<double, double, kNAcc, 11><<<1, 32 * kNAcc, 0, st>>>(partials, blocks, grad, loss_sum, skip_flag);
  return cn::launch_status();
}

int dpll_body_step_pts_f64(const double* x, const double* inertia, const double* mu_pair, const double* pts,
                           int32_t n_contacts, double dt, double eps, int64_t B, double* x_next, double* force,
                           void* stream) {
  if (B < 0 || !inertia || !mu_pair || n_contacts < 1 || n_contacts > DPLL_CUBE_NC) return DPLL_EINVAL;
  if (B > 0 && (!x || !pts || !x_next)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  body_pts_step_kernel<double, double><<<cn::grid_for(B, kLossThreads), kLossThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x, inertia, mu_pair, pts, n_contacts, dt, eps, B, x_next, force);
  return cn::launch_status();
}

int dpll_cube_terms_f64(const double* q, const double* v, const double* inertia, const double* mu_pair,
                        const double* half, int64_t B, double* M, double* J, double* phi, double* acc, double* delassus,
                        void* stream) {
  if (B < 0 || !inertia || !mu_pair || !half) return DPLL_EINVAL;
  if (B > 0 && (!q || !v || !M || !J || !phi || !acc)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  cube_terms_kernel<double, double><<<cn::grid_for(B, kLossThreads), kLossThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      q, v, inertia, mu_pair, half, B, M, J, phi, acc, delassus);
  return cn::launch_status();
}

int dpll_elbow_terms_f64(const double* q, const double* v, const double* inertia, const double* mu_pair,
                         const double* half, const double* kin, int64_t B, double* M, double* J, double* phi, double* acc,
                         double* delassus, void* stream) {
  if (B < 0 || !inertia || !mu_pair || !half || !kin) return DPLL_EINVAL;
  if (B > 0 && (!q || !v || !M || !J || !phi || !acc)) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  elbow_terms_kernel<double, double><<<cn::grid_for(B, 64), 64, 0, static_cast<cudaStream_t>(stream)>>>(
      q, v, inertia, mu_pair, half, kin, B, M, J, phi, acc, delassus);
  return cn::launch_status();
}

int dpll_elbow_rollout_f64(const double* x0, const double* inertia, const double* mu_pair, const double* half,
                           const double* kin, const double* pts, double dt, double eps, int64_t B, int32_t steps, double* traj,
                           double* force, int32_t* iters, void* stream) {
  return launch_elbow_rollout<double, double>(x0, inertia, mu_pair, half, kin, pts, dt, eps, B, steps, traj, force, iters,
                                              stream);
}

int dpll_elbow_rollout_saved_f64(const double* x0, const double* inertia, const double* mu_pair, const double* half,
                                 const double* kin, const double* pts, double dt, double eps, int64_t B, int32_t steps,
                                 double* traj, double* usol, void* stream) {
  if (B > 0 && steps > 0 && !usol) return DPLL_EINVAL;
  return launch_elbow_rollout<double, double>(x0, inertia, mu_pair, half, kin, pts, dt, eps, B, steps, traj, nullptr, nullptr,
                                              stream, usol);
}

int dpll_elbow_rollout_f32(const float* x0, const float* inertia, const float* mu_pair, const float* half,
                           const float* kin, const float* pts, float dt, float eps, int64_t B, int32_t steps, float* traj, float* force,
                           int32_t* iters, void* stream) {
  return launch_elbow_rollout<double, float>(x0, inertia, mu_pair, half, kin, pts, (double)dt, (double)eps, B, steps, traj,
                                             force, iters, stream);
}

int dpll_fma_peak_f64(double* out, int32_t blocks, int64_t iters, void* stream) {
  if (!out || blocks <= 0 || iters < 0) return DPLL_EINVAL;
  fma_peak_kernel<double><<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(out, iters);
  return cn::launch_status();
}

int dpll_fma_peak_f32(float* out, int32_t blocks, int64_t iters, void* stream) {
  if (!out || blocks <= 0 || iters < 0) return DPLL_EINVAL;
  fma_peak_kernel<float><<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(out, iters);
  return cn::launch_status();
}

}  // extern "C"
