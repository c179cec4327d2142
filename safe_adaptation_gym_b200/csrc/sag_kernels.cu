// sag_kernels.cu -- CUDA kernels (sm_100a) + the C ABI declared in include/sag_b200.h.
//
// The step is two kernels (DESIGN.md 5): k_step_free, one thread per environment over the whole batch (every environment
// in which nothing moves: closed-form path, with an exact overlap pre-test where something is within reach; it appends
// the others to a work list), and k_step_coop, the work list with ONE WARP per environment, the lanes splitting the
// collision phases / row set-up / floor rows / lidar pass and the contact solver's working set in shared memory
// (the scalar one-thread-per-environment contact path lives on in the observe kernels).  Resets run one warp per environment
// too (k_reset).  State is SoA / environment-minor so that every global access of a batch warp is one contiguous 256-byte
// (fp64) segment; observation tiles (lidar bins are accumulated in them) live in shared memory and are written out row by
// row.  No tensor cores: nothing here is a dense contraction.  The per-environment logic is in sag_core.cuh; every kernel
// is templated on the robot model.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <new>

#include "../../include/sag_b200.h"
#include "sag_core.cuh"
#include "sag_layout.h"

using namespace sag;

namespace {

constexpr int kBS = 128;          // environments (threads) per CTA
constexpr int kTileStride = kBS + 1;
template <class RB>
struct TileCfg {
  static constexpr int kObs = RB::kObsDim;
  static constexpr size_t kTileBytes = (sizeof(float) * kObs * kTileStride + 15) / 16 * 16;
  static constexpr size_t kSmemBytes = kTileBytes + sizeof(Scratch) * (kBS / 32);  // > 48 KB: opt-in dynamic shared memory
};

thread_local char g_err[512] = "";
// pinned output blocks handed out by sag_host_alloc_outputs (single-copy layout); process-wide, cleared by sag_host_free
void* g_packed_blocks[64];
bool is_packed_block(const void* p) {
  for (int k = 0; k < 64; ++k) if (g_packed_blocks[k] == p && p) return true;
  return false;
}

int fail(const char* what, cudaError_t ce = cudaSuccess) {
  if (ce != cudaSuccess) snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(ce));
  else snprintf(g_err, sizeof(g_err), "%s", what);
  return 1;
}
#define CK(call)                                   \
  do {                                             \
    cudaError_t ce_ = (call);                      \
    if (ce_ != cudaSuccess) return fail(#call, ce_); \
  } while (0)

// every entry point runs on the handle's device and leaves the caller's current device as it found it
struct DevGuard {
  int prev, want;
  explicit DevGuard(int d) : prev(-1), want(d) { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; if (prev != d) cudaSetDevice(d); }
  ~DevGuard() { if (prev >= 0 && prev != want) cudaSetDevice(prev); }
};

struct Handle {
  Dev D;
  int device;
  void* slab;
  size_t slab_bytes;
  void* field_ptr[SAG_NUM_FIELDS];
  size_t field_bytes[SAG_NUM_FIELDS];
  double *sret, *scost, *sn;  // per-env finished-episode statistics (under the env's current task)
  double* stats_acc;          // [SAG_NUM_TASKS + SAG_MAX_CUSTOM_TASKS][3]: statistics folded away when environments changed task
  CustomTable custom_h;       // host copy of the user-defined task table (sag_define_task; the kernels read the slab's)
  CustomTable* custom_d;      // the slab's table
  int32_t* next_task;         // [stride] SAG_F_NEXT_TASK: task queued for the next reset (-1 = none); k_reset consumes it
  int* err_h;                 // mapped pinned int[4]: sticky error words written by the kernels (sag_error_flags)
  int32_t* ids_d;             // staging for sag_set_tasks_host
  uint8_t* mask_d;            // staging for sag_reset_host
  // device staging for the host-buffer API
  float* act_d;
  float* obs_d;
  double* rew_d;
  uint8_t *cost_d, *done_d;
  cudaStream_t own_stream;
  cudaStream_t copy_stream;          // host-buffer API: bulk device-to-host copies that overlap the busy kernel
  cudaEvent_t ev_free, ev_copied;   // host-buffer API: batch kernel done, bulk copy done
  unsigned long long launches;  // kernels launched on behalf of this handle (sag_launch_count)
  int busy_grid;  // CTAs of k_step_coop: resident CTAs per SM x SMs
};

// coalesced write-out of the CTA's observation tile: tile[k][t] -> out[(e0 + t) * kObs + k]
template <int kObs>
__device__ __forceinline__ void write_tile(const float* tile, float* out, int e0, int n) {
  int cnt = min(kBS, n - e0) * kObs;
  float* dst = out + (size_t)e0 * kObs;
  for (int i = threadIdx.x; i < cnt; i += kBS) {
    int t = i / kObs, k = i - t * kObs;
    dst[i] = tile[k * kTileStride + t];
  }
}

// vectorised variant: 16-byte stores, 4 tile reads each (kObs is a multiple of 4; e0 a multiple of kBS, so rows are
// 16-byte aligned).  Writes every row of the CTA, including columns the caller did not fill.
template <int kObs>
__device__ __forceinline__ void write_tile4(const float* tile, float* out, int e0, int n) {
  static_assert(kObs % 4 == 0, "observation rows are written as float4");
  constexpr int kQ = kObs / 4;
  const int cnt = min(kBS, n - e0) * kQ;
  float4* dst = reinterpret_cast<float4*>(out + (size_t)e0 * kObs);
  for (int j = threadIdx.x; j < cnt; j += kBS) {
    const int t = j / kQ, q = j - t * kQ;
    const float* src = tile + (4 * q) * kTileStride + t;
    dst[j] = make_float4(src[0], src[kTileStride], src[2 * kTileStride], src[3 * kTileStride]);
  }
}

// per-warp write-out of up to 32 observation rows (tile column = lane; e < 0: no row)
template <int kObs>
__device__ __forceinline__ void write_rows(const float* tile, int tstride, float* out, int e) {
  const int lane = threadIdx.x & 31;
#pragma unroll 4
  for (int r = 0; r < 32; ++r) {
    const int er = __shfl_sync(0xffffffffu, e, r);
    if (er < 0) continue;
    float* dst = out + (size_t)er * kObs;
    const float* src = tile + r;
    for (int k = lane; k < kObs; k += 32) dst[k] = src[k * tstride];
  }
}

// ---- the step: two kernels --------------------------------------------------------------------
// k_step_free: one thread per environment over the whole batch.  Every environment in which nothing moves takes the
//   contact-free closed-form path: the quiet ones (nothing within reach for the whole step: 88-100 % under a random
//   policy) without any test, the others with the exact overlap / tendon pre-test in front of every substep.  An
//   environment with a moving body or a sticky physics error, and one whose pre-test fires (nothing has been stored at
//   that point), is appended to the work list and left untouched.
// k_step_coop: the work list, ONE WARP per environment (sag_core.cuh "warp-cooperative variants").  Keeping the contact
//   code out of the batch kernel is what keeps that one at <= 128 registers and free of divergence.

// The work list of a step: D.worklist[0 .. counts[0]).  Two counter sets are used alternately, selected on the device by
// the step epoch (D.epoch[0], in the slab): a step's batch kernel appends to set epoch & 1 and clears the other set for
// the next step, and the last CTA of its cooperative kernel to finish advances the epoch.  Once the batch kernel is
// done the other set is zero, so the kernels after it read the length as the sum of both sets, without the epoch.
// Nothing the host does between steps selects a set, so a step recorded in a CUDA graph behaves on every replay like a
// step issued anew, with no memset node per step.

// What a step kernel does with a step's outputs.  kOutStep: sag_step -- the observation, reward, cost and done.  The
// other two are the steps of sag_evaluate_actions: the epilogue adds the weighted reward and cost into the horizon's
// sums (sag_core.cuh: eval_accumulate) instead of storing them, and only the last step of the horizon (kOutAccumObs)
// builds and writes the observation; the ones before it (kOutAccum) skip the lidar, the sensors and the tile write-out.
constexpr int kOutStep = 0, kOutAccum = 1, kOutAccumObs = 2;

// __launch_bounds__(kBS, 4): 4 CTAs / SM (<= 128 registers) so that the whole 65,536-env point batch is one wave.  The car's
// contact-free step carries the two wheel-row pairs of its friction solve through ten substeps x ten sweeps: it needs
// the registers more than the occupancy (32,768 envs are 7 warps / SM), so it gets 2 CTAs / SM and no spills.
template <class RB, int Out = kOutStep>
__global__ void __launch_bounds__(kBS, RB::kKind == 1 ? 2 : 4) k_step_free(Dev D, const float* __restrict__ act, float* __restrict__ obs,
                                                    double* __restrict__ reward, double* __restrict__ reward2,
                                                    uint8_t* __restrict__ cost, uint8_t* __restrict__ done, EvalAcc A) {
  constexpr int kObs = RB::kObsDim;
  constexpr bool Obs = Out != kOutAccum;  // kOutAccum: no tile in shared memory
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* tile = reinterpret_cast<float*>(smem_raw);  // [kObs][kTileStride]
  const int e = blockIdx.x * kBS + threadIdx.x;
  const int lane = threadIdx.x & 31;
  if (blockIdx.x == 0 && threadIdx.x < 4) D.counts[8 * ((*D.epoch & 1u) ^ 1u) + threadIdx.x] = 0;
  bool run = false, pretest = false;
  if (e < D.n) {
    RB R;
    if constexpr (RB::kCustom) load_robot(D, e, spec_for(D, D.task[e], false, true), R);
    else load_robot(D, e, task_spec(D.task[e]), R);
    const unsigned char fl = D.flags[e];
    run = !(fl & F_PHYS_ERROR) && D.movmask[e] == 0 && D.num_gremlins == 0;  // (a welded gremlin is a constraint row in every pass)
    pretest = !env_is_quiet(D.clear[e], R);
  }
  bool bail = false;
  if (run) {
    float2 a = reinterpret_cast<const float2*>(act)[e];
    double rew[2];
    unsigned char c, d;
    bail = env_step<kStepNear, RB, Obs>(0u, nullptr, D, e, a.x, a.y, tile + threadIdx.x, kTileStride, rew, &c, &d, pretest) != 0;
    if (!bail) {
      if constexpr (Out == kOutStep) {
        reward[e] = rew[0];
        if (reward2) { reward2[2 * e] = rew[0]; reward2[2 * e + 1] = rew[1]; }
        cost[e] = c;
        done[e] = d;
      } else {
        eval_accumulate(A, e, rew, c, d);
      }
    }
  }
  // work list append, one atomic per warp
  const bool busy = e < D.n && (!run || bail);
  const unsigned m = __ballot_sync(0xffffffffu, busy);
  if (m) {
    int base = 0;
    if (lane == 0) base = atomicAdd(&D.counts[8 * (*D.epoch & 1u)], __popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (busy) D.worklist[base + __popc(m & ((1u << lane) - 1u))] = e;
  }
  // all kBS rows of the CTA in one coalesced sweep.  The columns of the work-list environments hold stale shared memory:
  // their rows are rewritten by the cooperative kernel, which always runs after this one on the same stream.
  if constexpr (Obs) {
    __syncthreads();
    write_tile4<kObs>(tile, obs, blockIdx.x * kBS, D.n);
  }
}

// k_step_coop: the work list with ONE WARP per environment (sag_core.cuh "warp-cooperative variants"): the lanes run the
// step's scalar code redundantly on the warp's shared-memory working set and split the collision phases, the overlap
// pre-test, the row set-up and the lidar pass between them.  A contact environment's step is a long dependent chain; what
// bounds this kernel is that chain's latency, not throughput, so the lanes are spent on shortening it and the register
// budget (<= 128) on keeping every work-list environment of the step resident at once (16 warps / SM).
constexpr int kCoopWarps = 16;  // warps (= environments in flight) per CTA; 16 = one CTA per SM at 128 registers
template <class RB>
struct CoopCfg {
  static constexpr int kObs = RB::kObsDim;
  static constexpr size_t kTileBytes = (sizeof(float) * kObs + 15) / 16 * 16;
  static constexpr size_t kPerWarp = kTileBytes + (sizeof(Scratch) + 15) / 16 * 16;
  static constexpr size_t kSmemBytes = kPerWarp * kCoopWarps;
};

template <class RB, int Out = kOutStep>
__global__ void __launch_bounds__(32 * kCoopWarps, 1) k_step_coop(const __grid_constant__ Dev D, const float* __restrict__ act,
                                                              float* __restrict__ obs, double* __restrict__ reward,
                                                              double* __restrict__ reward2, uint8_t* __restrict__ cost,
                                                              uint8_t* __restrict__ done, EvalAcc A) {
  constexpr bool Obs = Out != kOutAccum;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* mine = smem_raw + (size_t)warp * CoopCfg<RB>::kPerWarp;
  float* tile = reinterpret_cast<float*>(mine);
  Scratch* big = reinterpret_cast<Scratch*>(mine + CoopCfg<RB>::kTileBytes);
  // launched with programmatic stream serialization where possible (Ops::step_coop): the grid may be resident before the
  // preceding kernel has finished; everything that kernel wrote is visible after this call (no-op otherwise)
  cudaGridDependencySynchronize();
  const int count = D.counts[0] + D.counts[8];  // the other set was cleared by the batch kernel
  // Static assignment, entries strided over the CTAs so that a short list spreads over all SMs (one environment per SM
  // up to 148 entries: no two chains share a scheduler or an instruction cache before they have to); every warp of the
  // CTA runs the same number of rounds, which the phase alignment (sag_core.cuh: coop_align) relies on.
  const int per_round = gridDim.x * kCoopWarps;
  for (int base = 0; base < count; base += per_round) {
    const int i = base + (warp * gridDim.x + blockIdx.x);
    if (i >= count) { coop_idle_step<RB>(); continue; }
    const int e = D.worklist[i];
#if defined(SAG_TIMING)
    if (lane == 0) { atomicAdd(&D.dbg[15], 1ull); big->tsum[0] = big->tsum[1] = big->tsum[2] = 0ull; }
    __syncwarp();
    long long clk_ = clock64();
#endif
    float2 a = reinterpret_cast<const float2*>(act)[e];
    double rew[2];
    unsigned char c, d;
    env_step<kStepCoop, RB, Obs>(0xffffffffu, big, D, e, a.x, a.y, tile, 1, rew, &c, &d);
#if defined(SAG_TIMING)
    if (lane == 0) {
      const unsigned long long tot = (unsigned long long)(clock64() - clk_);
      atomicAdd(&D.dbg[14], tot);
      // slowest environment of the interval: total cycles in the high bits so that one atomicMax keeps its section sums
      const unsigned long long key = (tot << 40) | ((big->tsum[2] >> 10) << 20) | (big->tsum[0] >> 10);
      atomicMax(&D.dbg[16], key);
      atomicMax(&D.dbg[17], (tot << 40) | (big->tsum[1] >> 10));
    }
#endif
    __syncwarp();
    if (lane == 0) {
      if constexpr (Out == kOutStep) {
        reward[e] = rew[0];
        if (reward2) { reward2[2 * e] = rew[0]; reward2[2 * e + 1] = rew[1]; }
        cost[e] = c;
        done[e] = d;
      } else {
        eval_accumulate(A, e, rew, c, d);
      }
    }
    if constexpr (Obs) {
      float* dst = obs + (size_t)e * CoopCfg<RB>::kObs;
      for (int k = lane; k < CoopCfg<RB>::kObs; k += 32) dst[k] = tile[k];
    }
    __syncwarp();
  }
  // The last CTA to finish advances the step epoch for the next step's batch kernel (which runs after this kernel) and
  // re-arms the counter: one atomic per CTA, no launch
  if (threadIdx.x == 0 && atomicAdd(&D.epoch[1], 1u) == gridDim.x - 1) {
    D.epoch[1] = 0u;
    atomicAdd(&D.epoch[0], 1u);
  }
}

template <class RB>
__global__ void __launch_bounds__(kBS) k_observe(Dev D, float* __restrict__ obs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* tile = reinterpret_cast<float*>(smem_raw);
  Scratch* scratch = reinterpret_cast<Scratch*>(smem_raw + TileCfg<RB>::kTileBytes);
  const int e0 = blockIdx.x * kBS, e = e0 + threadIdx.x;
  const unsigned wmask = __ballot_sync(0xffffffffu, e < D.n);
  if (e < D.n) env_observe<RB>(wmask, &scratch[threadIdx.x >> 5], D, e, tile + threadIdx.x, kTileStride);
  __syncthreads();
  write_tile<RB::kObsDim>(tile, obs, e0, D.n);
}

// synthetic actions of sag_rollout: U(-1, 1) from Philox stream 2, counter = the environment's step count
__global__ void __launch_bounds__(256) k_rollout_actions(Dev D, float* __restrict__ act) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= D.n) return;
  Rng rng = {rng_key(D), D.gid_base + (uint32_t)e, D.episode[e]};
  double u1, u2;
  rng.pair(2u, (uint32_t)D.nstep[e], u1, u2);
  reinterpret_cast<float2*>(act)[e] = make_float2((float)(2.0 * u1 - 1.0), (float)(2.0 * u2 - 1.0));
}

// env.reset for the selected environments, ONE WARP per environment that is reset (sag_core.cuh: env_reset_coop -- 8
// placement candidates x 4 check lanes per round, the first valid draw wins: exactly the sequence of world.py:191-217).
// A CTA of four warps looks after `gpc` consecutive environments (4 for small batches: one per warp; 32 for large ones):
// every warp finds the selected ones with one coalesced read + ballot and takes every fourth of them, so that a sparse
// reset (auto-reset of the few environments that expired in this step) costs one layout's latency and a whole-batch reset
// keeps every SM full of warps.
// Statistics: an episode counts when it FINISHED (time limit or done: the NEEDS_RESET flag), under the task it ran with;
// a manual reset of an unfinished episode is not an episode.
// Next task: an environment with a task queued in next_task[e] takes it at this reset, whatever the reset path, and
// starts a fresh Task instance of it (sag_core.cuh: take_next_task; its statistics are folded into `acc` under the old
// task first).  The others reset as the call asks.
// obs != nullptr: the environments that were reset get the first observation of their new episode written into their
// row (the others' rows are left alone) and was_reset[e] = 1 / 0 tells the caller which (auto-reset, env.py).
constexpr int kResetWarps = 4;
template <class RB>
struct ResetCfg {
  static constexpr size_t kRowBytes = (sizeof(float) * RB::kObsDim + 15) / 16 * 16;
  static constexpr size_t kPlaceBytes = 3 * 32 * sizeof(double);
  static constexpr size_t kPerWarp = kPlaceBytes + kRowBytes + (sizeof(Scratch) + 15) / 16 * 16;
  static constexpr size_t kSmemBytes = kPerWarp * kResetWarps;
};
template <class RB, bool WithObs>
__global__ void __launch_bounds__(32 * kResetWarps) k_reset(Dev D, const uint8_t* __restrict__ mask, int only_flagged, int new_task,
                                                            double* sret, double* scost, double* sn, double* acc,
                                                            int* next_task, float* __restrict__ obs,
                                                            uint8_t* __restrict__ was_reset, int gpc) {
  // gpc: environments per CTA (4 .. 32): small batches get one warp per environment, large ones eight per warp
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* mine = smem_raw + (size_t)warp * (WithObs ? ResetCfg<RB>::kPerWarp : ResetCfg<RB>::kPlaceBytes);
  double* px = reinterpret_cast<double*>(mine);
  double* py = px + 32;
  double* pk = py + 32;
  float* row = reinterpret_cast<float*>(mine + ResetCfg<RB>::kPlaceBytes);
  Scratch* scratch = reinterpret_cast<Scratch*>(mine + ResetCfg<RB>::kPlaceBytes + ResetCfg<RB>::kRowBytes);
  const int e_l = blockIdx.x * gpc + lane;  // this lane looks at environment e_l of the CTA's gpc
  bool doit = lane < gpc && e_l < D.n;
  unsigned char fl_l = 0;
  if (doit) fl_l = D.flags[e_l];
  if (doit && mask && !mask[e_l]) doit = false;
  if (doit && only_flagged && !(fl_l & F_NEEDS_RESET)) doit = false;
  if (warp == 0 && lane < gpc && e_l < D.n && was_reset) was_reset[e_l] = doit ? 1 : 0;
  unsigned todo = __ballot_sync(0xffffffffu, doit);
  int rank = 0;
  for (; todo; todo &= todo - 1, ++rank) {
    if ((rank & (kResetWarps - 1)) != warp) continue;
    const int e = blockIdx.x * gpc + (__ffs((int)todo) - 1);
    const unsigned char fl = D.flags[e];
    const unsigned episode = D.episode[e] + 1u;
    int fresh = new_task != 0;
    if (lane == 0) {
      if ((fl & F_NEEDS_RESET) && D.nstep[e] > 0) { sret[e] += D.epret[e]; scost[e] += D.epcost[e]; sn[e] += 1.0; }
      fresh = take_next_task(D, e, next_task, sret, scost, sn, acc, fresh != 0, num_task_ids(D, RB::kCustom));
    }
    fresh = __shfl_sync(0xffffffffu, fresh, 0);
    __syncwarp();  // lane 0's writes (a new D.task[e]) are seen by the whole warp
#if defined(__CUDA_ARCH__)
    env_reset_coop<RB>(D, e, episode, fresh != 0, px, py, pk);
#endif
    if (lane == 0 && (D.flags[e] & F_RESAMPLE_FAILED)) D.errflags[0] = 1;
    if constexpr (WithObs) {
      if (lane == 0) env_observe<RB>(1u, scratch, D, e, row, 1);
      __syncwarp();
      float* dst = obs + (size_t)e * RB::kObsDim;
      for (int k = lane; k < RB::kObsDim; k += 32) dst[k] = row[k];
      __syncwarp();
    }
  }
}

// env.set_task: statistics gathered under the old task are folded into the per-task accumulator first (so that they
// are not re-labelled), including an episode that has finished but has not been reset yet; ids are validated; queued
// next tasks are dropped.
// nids: the handle's task ids (SAG_NUM_TASKS, or more in k_set_tasks_custom)
__device__ __forceinline__ void set_task_of(const Dev& D, int e, const int32_t* __restrict__ ids, double* sret, double* scost,
                                            double* sn, double* acc, int* next_task, int nids) {
  const int old = D.task[e];
  double r = sret[e], c = scost[e], k = sn[e];
  if ((D.flags[e] & F_NEEDS_RESET) && D.nstep[e] > 0) { r += D.epret[e]; c += D.epcost[e]; k += 1.0; D.nstep[e] = 0; }
  if (k != 0.0 && old >= 0 && old < nids) { atomicAdd(acc + 3 * old, r); atomicAdd(acc + 3 * old + 1, c); atomicAdd(acc + 3 * old + 2, k); }
  sret[e] = 0.0; scost[e] = 0.0; sn[e] = 0.0;
  int id = ids[e];
  if (id < 0 || id >= nids) { id = SAG_T_GO_TO_GOAL; D.errflags[1] = 1; }
  D.task[e] = id;
  next_task[e] = -1;
}
__global__ void k_set_tasks(Dev D, const int32_t* __restrict__ ids, double* sret, double* scost, double* sn, double* acc,
                            int* next_task) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= D.n) return;
  set_task_of(D, e, ids, sret, scost, sn, acc, next_task, SAG_NUM_TASKS);
}
// handles with user-defined tasks: their ids are valid too
__global__ void k_set_tasks_custom(Dev D, const int32_t* __restrict__ ids, double* sret, double* scost, double* sn,
                                   double* acc, int* next_task) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= D.n) return;
  set_task_of(D, e, ids, sret, scost, sn, acc, next_task, num_task_ids(D, true));
}

// sag_copy_envs: environment states gathered column by column.  The fields are SoA and environment-minor, so the
// threads run over (chunk of field rows, destination) with the destination fastest: the stores of a warp are one
// contiguous segment per row, and the loads are too for contiguous sources, or a broadcast for K copies of one source.
// A chunk is up to kCopyRows rows of one field; each thread issues all its loads before its stores.  Memory-bound: no
// arithmetic besides the pair rule (sag_core.cuh: copy_env_source).  The destination's statistics are settled by
// k_copy_envs_fold, launched before it on the same stream: it reads the destination's flags, step count, episode return
// and cost and task id, which k_copy_envs overwrites from other chunks.
constexpr int kCopyRows = 8, kCopyThreads = 256;
struct CopyFields {
  char* dst[SAG_NUM_FIELDS];
  const char* src[SAG_NUM_FIELDS];
  int rows[SAG_NUM_FIELDS], elem[SAG_NUM_FIELDS];
};
constexpr int copy_chunks() {
  int c = 0;
  for (int f = 0; f < SAG_NUM_FIELDS; ++f) c += (kFieldShape[f].rows + kCopyRows - 1) / kCopyRows;
  return c;
}

template <class T>
__device__ __forceinline__ void copy_rows(char* dst, const char* src, int r0, int nr, int dst_stride, int src_stride,
                                          int j, int s) {
  const T* sp = reinterpret_cast<const T*>(src) + (size_t)r0 * src_stride + s;
  T* dp = reinterpret_cast<T*>(dst) + (size_t)r0 * dst_stride + j;
  T v[kCopyRows];
#pragma unroll
  for (int k = 0; k < kCopyRows; ++k) if (k < nr) v[k] = sp[(size_t)k * src_stride];
#pragma unroll
  for (int k = 0; k < kCopyRows; ++k) if (k < nr) dp[(size_t)k * dst_stride] = v[k];
}

// one thread per destination: records bad pairs and settles the statistics of the destinations that will be replaced
__global__ void k_copy_envs_fold(Dev D, const int32_t* __restrict__ src_of_dst, int n_src, int same_handle, double* sret,
                                 double* scost, double* sn, double* acc) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < D.n) copy_env_source(D, src_of_dst, j, n_src, same_handle != 0, true, sret, scost, sn, acc);
}
__global__ void k_copy_envs_fold_custom(Dev D, const int32_t* __restrict__ src_of_dst, int n_src, int same_handle,
                                        double* sret, double* scost, double* sn, double* acc) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < D.n) copy_env_source(D, src_of_dst, j, n_src, same_handle != 0, true, sret, scost, sn, acc, num_task_ids(D, true));
}

__global__ void __launch_bounds__(kCopyThreads) k_copy_envs(Dev D, CopyFields F, const int32_t* __restrict__ src_of_dst,
                                                            int n_src, int src_stride, int same_handle) {
  const int j = blockIdx.x * kCopyThreads + threadIdx.x;
  if (j >= D.n) return;
  int f = 0, c = blockIdx.y;
  for (; f < SAG_NUM_FIELDS - 1; ++f) {
    const int nc = (F.rows[f] + kCopyRows - 1) / kCopyRows;
    if (c < nc) break;
    c -= nc;
  }
  const int r0 = c * kCopyRows, nr = min(kCopyRows, F.rows[f] - r0);
  const int s = copy_env_source(D, src_of_dst, j, n_src, same_handle != 0, false, nullptr, nullptr, nullptr, nullptr);
  if (s < 0) return;
  if (F.elem[f] == 8) copy_rows<unsigned long long>(F.dst[f], F.src[f], r0, nr, D.stride, src_stride, j, s);
  else if (F.elem[f] == 4) copy_rows<unsigned>(F.dst[f], F.src[f], r0, nr, D.stride, src_stride, j, s);
  else copy_rows<unsigned char>(F.dst[f], F.src[f], r0, nr, D.stride, src_stride, j, s);
}

// per-task statistic reduction: out[task][3] += (sum return, sum cost, episodes) of finished episodes
__global__ void k_task_stats(Dev D, const double* sret, const double* scost, const double* sn, double* out) {
  __shared__ double acc[SAG_NUM_TASKS][3];
  for (int i = threadIdx.x; i < SAG_NUM_TASKS * 3; i += blockDim.x) (&acc[0][0])[i] = 0.0;
  __syncthreads();
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < D.n; e += gridDim.x * blockDim.x) {
    int t = D.task[e];
    if (sn[e] != 0.0) { atomicAdd(&acc[t][0], sret[e]); atomicAdd(&acc[t][1], scost[e]); atomicAdd(&acc[t][2], sn[e]); }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < SAG_NUM_TASKS * 3; i += blockDim.x)
    if ((&acc[0][0])[i] != 0.0) atomicAdd(out + i, (&acc[0][0])[i]);
}
// the same with a row for every id a handle with user-defined tasks can have; out has sag_num_task_ids rows, and a row
// beyond them is never non-zero (every environment's task id is below that count)
__global__ void k_task_stats_custom(Dev D, const double* sret, const double* scost, const double* sn, double* out) {
  constexpr int kRows = SAG_NUM_TASKS + SAG_MAX_CUSTOM_TASKS;
  __shared__ double acc[kRows][3];
  for (int i = threadIdx.x; i < kRows * 3; i += blockDim.x) (&acc[0][0])[i] = 0.0;
  __syncthreads();
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < D.n; e += gridDim.x * blockDim.x) {
    int t = D.task[e];
    if (sn[e] != 0.0) { atomicAdd(&acc[t][0], sret[e]); atomicAdd(&acc[t][1], scost[e]); atomicAdd(&acc[t][2], sn[e]); }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kRows * 3; i += blockDim.x)
    if ((&acc[0][0])[i] != 0.0) atomicAdd(out + i, (&acc[0][0])[i]);
}

// ------------------------------------------------------------------------------------------------
// stand-alone streaming kernels (SoA env-minor inputs, one thread per environment)
// ------------------------------------------------------------------------------------------------
constexpr int kLidarTileStride = kBS + 1;

__global__ void __launch_bounds__(kBS) k_lidar(const double* __restrict__ robot, const double* __restrict__ obj_xy,
                                               const uint8_t* __restrict__ group, int n, int nslots, float* __restrict__ out) {
  __shared__ float tile[48 * kLidarTileStride];
  const int e0 = blockIdx.x * kBS, e = e0 + threadIdx.x;
  if (e < n) {
    float* bins = tile + threadIdx.x;
#pragma unroll
    for (int k = 0; k < 48; ++k) bins[k * kLidarTileStride] = 0.0f;
    double rx = robot[e], ry = robot[(size_t)n + e], yaw = robot[2 * (size_t)n + e];
    double sn, cs;
    sag_sincos(yaw, &sn, &cs);
    const double* oxp = obj_xy + e;
    const double* oyp = obj_xy + (size_t)nslots * n + e;
    const uint8_t* gp = group + e;
    // four objects per trip: the loads and the four sqrt / atan2 chains are independent, the shared-memory bin
    // updates (which the compiler must keep in order) come last.  Pointers are bumped by n per object (no 64-bit
    // multiply per access).
    int s = 0;
    for (; s + 4 <= nslots; s += 4) {
      int g[4];
      double wx[4], wy[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        g[k] = *gp; wx[k] = *oxp - rx; wy[k] = *oyp - ry;
        gp += n; oxp += n; oyp += n;
      }
      LidarHit H[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) H[k] = lidar_eval(wx[k], wy[k], cs, sn);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (g[k] == 0) continue;
        int off = g[k] == 1 ? 0 : (g[k] == 3 ? 16 : 32);
        lidar_apply(H[k], bins + off * kLidarTileStride, kLidarTileStride);
      }
    }
    for (; s < nslots; ++s) {
      int g = *gp;
      double px = *oxp, py = *oyp;
      gp += n; oxp += n; oyp += n;
      if (g == 0) continue;
      int off = g == 1 ? 0 : (g == 3 ? 16 : 32);
      lidar_accum(rx, ry, cs, sn, px, py, bins + off * kLidarTileStride, kLidarTileStride);
    }
  }
  __syncthreads();
  int cnt = min(kBS, n - e0) * 48;
  float* dst = out + (size_t)e0 * 48;
  for (int i = threadIdx.x; i < cnt; i += kBS) {
    int t = i / 48, k = i - t * 48;
    dst[i] = tile[k * kLidarTileStride + t];
  }
}

// NH > 0: hazard count known at compile time -> all 2*NH loads of a thread are issued before the first use (HBM-bound
// streaming kernel: memory-level parallelism is what matters); NH == 0: run-time count.
template <int NH>
__global__ void __launch_bounds__(256) k_cost(const double* __restrict__ robot_xy, const float* __restrict__ hazard_xy,
                                              const uint8_t* __restrict__ contact, int n, int nh, double hazard_size,
                                              uint8_t* __restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const float* hx = hazard_xy + e;
  const float* hy = hazard_xy + (size_t)nh * n + e;
  bool hit;
  if (NH > 0) {
    float fx[NH > 0 ? NH : 1], fy[NH > 0 ? NH : 1];
#pragma unroll
    for (int s = 0; s < NH; ++s) { fx[s] = hx[(size_t)s * n]; fy[s] = hy[(size_t)s * n]; }
    const double rx = robot_xy[e], ry = robot_xy[(size_t)n + e];
    hit = contact[e] != 0;                                           // world.py:146
#pragma unroll
    for (int s = 0; s < NH; ++s) {                                   // world.py:148-153
      double dx = rx - (double)fx[s], dy = ry - (double)fy[s];
      hit = hit | hazard_hit(dx * dx + dy * dy, hazard_size);        // == (sqrt(d2) <= size), sqrt only near the boundary
    }
  } else {
    const double rx = robot_xy[e], ry = robot_xy[(size_t)n + e];
    hit = contact[e] != 0;
    for (int s = 0; s < nh; ++s) {
      double dx = rx - (double)hx[(size_t)s * n], dy = ry - (double)hy[(size_t)s * n];
      hit = hit | hazard_hit(dx * dx + dy * dy, hazard_size);
    }
  }
  out[e] = hit ? 1 : 0;                                              // world.py:155
}

// Host-buffer API: copies the rows of this step's busy environments (both work-list segments) from the device output
// arrays into MAPPED pinned host buffers, one warp per row (240 / 288 contiguous bytes: full PCIe write bursts).
template <int kObs>
__global__ void __launch_bounds__(128) k_fixup_host(const __grid_constant__ Dev D, const float* __restrict__ obs,
                                                    const double* __restrict__ reward, const uint8_t* __restrict__ cost,
                                                    const uint8_t* __restrict__ done, float* __restrict__ obs_h,
                                                    double* __restrict__ reward_h, uint8_t* __restrict__ cost_h,
                                                    uint8_t* __restrict__ done_h) {
  const int lane = threadIdx.x & 31, nw = gridDim.x * 4;
  const int count = D.counts[0] + D.counts[8];  // the step that just ran (the other set is zero)
  for (int i = blockIdx.x * 4 + (threadIdx.x >> 5); i < count; i += nw) {
    const int e = D.worklist[i];
    const float* src = obs + (size_t)e * kObs;
    float* dst = obs_h + (size_t)e * kObs;
    for (int k = lane; k < kObs; k += 32) dst[k] = src[k];
    if (lane == 0) { reward_h[e] = reward[e]; cost_h[e] = cost[e]; done_h[e] = done[e]; }
  }
}

// env.step's return values as FRESH arrays in one launch (the host mirror hands out copies by default, like the reference's
// numpy arrays): obs rows as float4, reward (1 or 2 columns), cost as float32 (world.py:155 returns a float), done as bool
// bytes, bound.  Five separate framework copies / casts cost ~6 us of stream time each.
__global__ void __launch_bounds__(256) k_export_outputs(int n, int obs_quads, int reward_cols, const float4* __restrict__ obs,
                                                        const double* __restrict__ reward, const uint8_t* __restrict__ cost,
                                                        const uint8_t* __restrict__ done, const double* __restrict__ bound,
                                                        float4* __restrict__ obs_out, double* __restrict__ reward_out,
                                                        float* __restrict__ cost_out, uint8_t* __restrict__ done_out,
                                                        double* __restrict__ bound_out) {
  const size_t total = (size_t)n * obs_quads;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    obs_out[i] = obs[i];
    if (i < (size_t)n) {
      for (int k = 0; k < reward_cols; ++k) reward_out[i * reward_cols + k] = reward[i * reward_cols + k];
      cost_out[i] = (float)cost[i];
      done_out[i] = done[i] ? 1 : 0;
      if (bound_out) bound_out[i] = bound[i];
    }
  }
}

static inline int grid_for(int n) { return (n + kBS - 1) / kBS; }

// host-side launchers, one set per robot model
template <class RB>
struct Ops {
  static cudaError_t setup(Handle* H) {
    cudaError_t ce = cudaFuncSetAttribute(k_observe<RB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TileCfg<RB>::kSmemBytes);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute(k_reset<RB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ResetCfg<RB>::kSmemBytes);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute(k_step_coop<RB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CoopCfg<RB>::kSmemBytes);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute(k_step_coop<RB, kOutAccum>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CoopCfg<RB>::kSmemBytes);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute(k_step_coop<RB, kOutAccumObs>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CoopCfg<RB>::kSmemBytes);
    if (ce != cudaSuccess) return ce;
    // Local memory: the observation and auto-reset kernels carry the scalar contact path (stack frames of ~1.6 KB
    // per thread, above the default 1 KB limit), so the driver would re-size its local-memory pool whenever one of them
    // follows a run of step kernels -- a device-wide stall of tens to hundreds of milliseconds on the first env.reset()
    // after an episode (measured).  Raising the stack limit once to the largest frame keeps the pool at that size.
    {
      size_t need = 0;
      cudaFuncAttributes fa;
      if (cudaFuncGetAttributes(&fa, k_observe<RB>) == cudaSuccess && fa.localSizeBytes > need) need = fa.localSizeBytes;
      if (cudaFuncGetAttributes(&fa, k_reset<RB, true>) == cudaSuccess && fa.localSizeBytes > need) need = fa.localSizeBytes;
      need = (need + 255) / 256 * 256;
      size_t cur = 0;
      if (cudaDeviceGetLimit(&cur, cudaLimitStackSize) == cudaSuccess && cur < need) cudaDeviceSetLimit(cudaLimitStackSize, need);
      cudaGetLastError();
    }
    int sms = 148, per_sm = 1;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, H->device);
    ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_step_coop<RB>, 32 * kCoopWarps, CoopCfg<RB>::kSmemBytes);
    H->busy_grid = sms * (per_sm > 0 ? per_sm : 1);
    return ce;
  }
  static cudaError_t step(Handle* H, const float* act, float* obs, double* reward, double* reward2, uint8_t* cost, uint8_t* done,
                          cudaStream_t s) {
    cudaError_t ce = step_free(H, act, obs, reward, reward2, cost, done, s);
    if (ce != cudaSuccess) return ce;
    return step_coop(H, act, obs, reward, reward2, cost, done, s);
  }
  template <int Out = kOutStep>
  static cudaError_t step_free(Handle* H, const float* act, float* obs, double* reward, double* reward2, uint8_t* cost,
                               uint8_t* done, cudaStream_t s, const EvalAcc& A = EvalAcc{}) {
    // this step's counter set is zero already (cleared by the previous step's batch kernel, which saves a memset node per
    // step) and the kernels find it from the step epoch on the device; steps of one handle must be stream-ordered
    const size_t smem = Out == kOutAccum ? 0 : TileCfg<RB>::kTileBytes;
    k_step_free<RB, Out><<<grid_for(H->D.n), kBS, smem, s>>>(H->D, act, obs, reward, reward2, cost, done, A);
    ++H->launches;
    return cudaGetLastError();
  }
  // rows of the busy environments -> mapped host buffers (after the bulk copy that carried the quiet rows)
  static cudaError_t fixup_host(Handle* H, const float* obs, const double* reward, const uint8_t* cost, const uint8_t* done,
                                float* obs_h, double* reward_h, uint8_t* cost_h, uint8_t* done_h, cudaStream_t s) {
    k_fixup_host<RB::kObsDim><<<H->busy_grid, 128, 0, s>>>(H->D, obs, reward, cost, done, obs_h, reward_h, cost_h, done_h);
    ++H->launches;
    return cudaGetLastError();
  }
  template <int Out = kOutStep>
  static cudaError_t step_coop(Handle* H, const float* act, float* obs, double* reward, double* reward2, uint8_t* cost, uint8_t* done,
                               cudaStream_t s, const EvalAcc& A = EvalAcc{}) {
    ++H->launches;
    const int need = (H->D.n + kCoopWarps - 1) / kCoopWarps;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(need < H->busy_grid ? need : H->busy_grid);
    cfg.blockDim = dim3(32 * kCoopWarps);
    cfg.dynamicSmemBytes = CoopCfg<RB>::kSmemBytes;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;  // hides this launch's latency behind the previous kernel's tail
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, k_step_coop<RB, Out>, H->D, act, obs, reward, reward2, cost, done, A);
  }
  // sag_evaluate_actions: H x (k_step_free + k_step_coop) with the accumulating epilogue, the observation on the last
  // step only.  The weights are formed here, left to right in float64, and passed by value.
  static cudaError_t evaluate(Handle* H, int h_steps, const float* act, double discount, float* obs, double* ret, int ret_cols,
                              double* cost, int32_t* length, cudaStream_t s) {
    double w = 1.0;
    for (int h = 0; h < h_steps; ++h) {
      const EvalAcc A = {ret, cost, length, w, ret_cols, h == 0, h == h_steps - 1};
      const float* a = act + (size_t)h * H->D.n * 2;
      cudaError_t ce;
      if (h < h_steps - 1) {
        ce = step_free<kOutAccum>(H, a, nullptr, nullptr, nullptr, nullptr, nullptr, s, A);
        if (ce == cudaSuccess) ce = step_coop<kOutAccum>(H, a, nullptr, nullptr, nullptr, nullptr, nullptr, s, A);
      } else {
        ce = step_free<kOutAccumObs>(H, a, obs, nullptr, nullptr, nullptr, nullptr, s, A);
        if (ce == cudaSuccess) ce = step_coop<kOutAccumObs>(H, a, obs, nullptr, nullptr, nullptr, nullptr, s, A);
      }
      if (ce != cudaSuccess) return ce;
      w *= discount;
    }
    return cudaSuccess;
  }
  static cudaError_t observe(Handle* H, float* obs, cudaStream_t s) {
    k_observe<RB><<<grid_for(H->D.n), kBS, TileCfg<RB>::kSmemBytes, s>>>(H->D, obs);
    ++H->launches;
    return cudaGetLastError();
  }
  static cudaError_t rollout(Handle* H, int k_steps, float* obs, double* reward, uint8_t* cost, uint8_t* done, cudaStream_t s) {
    // K x (action kernel + the two step kernels): the same path as sag_step, so a rollout runs at the step's speed (a
    // single-launch scalar form, one thread per environment with the contact solver inline, was 3x slower at BASELINE
    // batch sizes).  Outputs of the last step are returned.
    float* o = obs ? obs : H->obs_d;
    double* r = reward ? reward : H->rew_d;
    uint8_t* c = cost ? cost : H->cost_d;
    uint8_t* d = done ? done : H->done_d;
    for (int k = 0; k < k_steps; ++k) {
      k_rollout_actions<<<(H->D.n + 255) / 256, 256, 0, s>>>(H->D, H->act_d);
      ++H->launches;
      cudaError_t ce = step(H, H->act_d, o, r, nullptr, c, d, s);
      if (ce != cudaSuccess) return ce;
    }
    return cudaGetLastError();
  }
  static cudaError_t reset(Handle* H, const uint8_t* mask, int only_flagged, int new_task, float* obs, uint8_t* was_reset, cudaStream_t s) {
    // environments per CTA of four warps: one per warp while that still fills the GPU, eight per warp for large batches
    const int gpc = H->D.n <= 8192 ? kResetWarps : (H->D.n <= 16384 ? 2 * kResetWarps : (H->D.n <= 32768 ? 4 * kResetWarps : 32));
    const int grid = (H->D.n + gpc - 1) / gpc;
    ++H->launches;
    if (obs && (mask || only_flagged)) {  // selective reset: the first observation of the new episodes is written by the same kernel
      k_reset<RB, true><<<grid, 32 * kResetWarps, ResetCfg<RB>::kSmemBytes, s>>>(H->D, mask, only_flagged, new_task, H->sret, H->scost, H->sn, H->stats_acc, H->next_task, obs, was_reset, gpc);
      return cudaGetLastError();
    }
    k_reset<RB, false><<<grid, 32 * kResetWarps, ResetCfg<RB>::kPlaceBytes * kResetWarps, s>>>(H->D, mask, only_flagged, new_task, H->sret, H->scost, H->sn, H->stats_acc, H->next_task, nullptr, was_reset, gpc);
    cudaError_t ce = cudaGetLastError();
    if (ce == cudaSuccess && obs) ce = observe(H, obs, s);  // whole-batch reset: one thread per environment is the faster observation pass
    return ce;
  }
};

// one set of kernels per robot model; environments with gremlins (SagConfig.num_gremlins > 0) use the *G instantiations,
// handles with user-defined tasks (sag_define_task) the *C ones
#define SAG_DISPATCH(H, call)                                                                                       \
  ((H)->custom_h.count > 0                                                                                          \
       ? ((H)->D.robot == SAG_ROBOT_CAR ? ((H)->D.num_gremlins > 0 ? Ops<CarRobotGC>::call : Ops<CarRobotC>::call)    \
                                        : ((H)->D.num_gremlins > 0 ? Ops<PointRobotGC>::call : Ops<PointRobotC>::call)) \
       : ((H)->D.robot == SAG_ROBOT_CAR ? ((H)->D.num_gremlins > 0 ? Ops<CarRobotG>::call : Ops<CarRobot>::call)      \
                                        : ((H)->D.num_gremlins > 0 ? Ops<PointRobotG>::call : Ops<PointRobot>::call)))

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

const char* sag_last_error(void) { return g_err; }
int sag_abi_version(void) { return SAG_ABI_VERSION; }

void sag_default_config(SagConfig* c) { default_config(c); }

int sag_create(const SagConfig* cfg, int device, void** handle) {
  if (!cfg || !handle) return fail("sag_create: null argument");
  if (cfg->n_envs <= 0) return fail("sag_create: n_envs must be positive");
  if (cfg->robot != SAG_ROBOT_POINT && cfg->robot != SAG_ROBOT_CAR) return fail("sag_create: robot must be point (0) or car (1)");
  if (cfg->num_gremlins < 0 || cfg->num_gremlins > SAG_MAX_GREMLINS) return fail("sag_create: num_gremlins must be in [0, SAG_MAX_GREMLINS]");
  DevGuard guard(device);
  CK(cudaGetLastError());
  Handle* H = new (std::nothrow) Handle();
  if (!H) return fail("sag_create: out of host memory");
  memset(H, 0, sizeof(*H));
  H->device = device;
  Dev& D = H->D;
  dev_from_config(D, *cfg);
  {
    cudaError_t ce = SAG_DISPATCH(H, setup(H));
    if (ce != cudaSuccess) { delete H; return fail("sag_create: kernel setup", ce); }
  }
  const int obs_dim = D.robot == SAG_ROBOT_CAR ? SAG_OBS_CAR : SAG_OBS_POINT;
  SlabLayout LY = slab_layout(D.n, D.stride, obs_dim);
  cudaError_t ce = cudaMalloc(&H->slab, LY.total);
  if (ce != cudaSuccess) { delete H; return fail("sag_create: cudaMalloc", ce); }
  H->slab_bytes = LY.total;
  ce = cudaMemset(H->slab, 0, LY.total);
  if (ce != cudaSuccess) { cudaFree(H->slab); delete H; return fail("sag_create: cudaMemset", ce); }
  char* base = (char*)H->slab;
  const size_t st = (size_t)D.stride;
  slab_bind(D, LY, base);
  for (int f = 0; f < SAG_NUM_FIELDS; ++f) { H->field_ptr[f] = base + LY.off[f]; H->field_bytes[f] = LY.bytes[f]; }
  H->sret = (double*)(base + LY.stats_off); H->scost = H->sret + st; H->sn = H->sret + 2 * st;
  H->act_d = (float*)(base + LY.act_off); H->obs_d = (float*)(base + LY.obs_off); H->rew_d = (double*)(base + LY.rew_off);
  H->cost_d = (uint8_t*)(base + LY.cost_off); H->done_d = (uint8_t*)(base + LY.done_off);
  // episode counters start at 0xFFFFFFFF so that the first reset is episode 0
  ce = cudaMemset(D.episode, 0xFF, st * sizeof(unsigned));
  if (ce == cudaSuccess) ce = cudaMemcpy(D.key, &cfg->seed, sizeof(*D.key), cudaMemcpyHostToDevice);
  H->custom_d = (CustomTable*)(base + LY.custom_off);  // (zeroed with the slab: no task defined)
  if (ce == cudaSuccess) ce = cudaMemcpy(D.counts + kCustomTablePtr, &H->custom_d, sizeof(H->custom_d), cudaMemcpyHostToDevice);
  H->stats_acc = (double*)(base + LY.acc_off);
  H->ids_d = (int32_t*)(base + LY.ids_off); H->mask_d = (uint8_t*)(base + LY.mask_off);
  H->next_task = (int32_t*)H->field_ptr[SAG_F_NEXT_TASK];
  if (ce == cudaSuccess) ce = cudaMemset(H->next_task, 0xFF, st * sizeof(int32_t));  // -1: no task queued
  if (ce == cudaSuccess) ce = cudaHostAlloc((void**)&H->err_h, 4 * sizeof(int), cudaHostAllocMapped);
  if (ce == cudaSuccess) { memset(H->err_h, 0, 4 * sizeof(int)); ce = cudaHostGetDevicePointer((void**)&D.errflags, H->err_h, 0); }
  if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&H->own_stream, cudaStreamNonBlocking);
  if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&H->copy_stream, cudaStreamNonBlocking);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&H->ev_free, cudaEventDisableTiming);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&H->ev_copied, cudaEventDisableTiming);
  if (ce != cudaSuccess) { cudaFree(H->slab); delete H; return fail("sag_create: init", ce); }
  *handle = H;
  return 0;
}

int sag_destroy(void* handle) {
  Handle* H = (Handle*)handle;
  if (!H) return 0;
  DevGuard guard(H->device);
  cudaDeviceSynchronize();
  if (H->err_h) cudaFreeHost(H->err_h);
  if (H->own_stream) cudaStreamDestroy(H->own_stream);
  if (H->copy_stream) cudaStreamDestroy(H->copy_stream);
  if (H->ev_free) cudaEventDestroy(H->ev_free);
  if (H->ev_copied) cudaEventDestroy(H->ev_copied);
  cudaFree(H->slab);
  delete H;
  return 0;
}

// SAG_TIMING builds: section clocks of the cooperative kernel (16 x u64, host buffer); zeroed after the read
int sag_debug_read(void* handle, unsigned long long* out16) {
  Handle* H = (Handle*)handle;
  if (!H || !out16) return fail("sag_debug_read: null argument");
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out16, H->D.dbg, 18 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  CK(cudaMemset(H->D.dbg, 0, 18 * sizeof(unsigned long long)));
  return 0;
}
unsigned long long sag_launch_count(void* handle) { return handle ? ((Handle*)handle)->launches : 0ull; }
int sag_stride(void* handle) { return ((Handle*)handle)->D.stride; }
int sag_obs_dim(void* handle) { return ((Handle*)handle)->D.robot == SAG_ROBOT_CAR ? SAG_OBS_CAR : SAG_OBS_POINT; }
size_t sag_field_bytes(void* handle, int field) {
  if (field < 0 || field >= SAG_NUM_FIELDS) return 0;
  return ((Handle*)handle)->field_bytes[field];
}

static int launch_set_tasks(Handle* H, const int32_t* ids, cudaStream_t s) {
  auto k = H->custom_h.count > 0 ? k_set_tasks_custom : k_set_tasks;
  k<<<(H->D.n + 255) / 256, 256, 0, s>>>(H->D, ids, H->sret, H->scost, H->sn, H->stats_acc, H->next_task);
  ++H->launches;
  CK(cudaGetLastError());
  return 0;
}

int sag_set_tasks(void* handle, const int32_t* ids, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !ids) return fail("sag_set_tasks: null argument");
  DevGuard guard(H->device);
  return launch_set_tasks(H, ids, (cudaStream_t)stream);
}

int sag_num_task_ids(void* handle) { return handle ? SAG_NUM_TASKS + ((Handle*)handle)->custom_h.count : SAG_NUM_TASKS; }

int sag_define_task(void* handle, const SagTaskDef* def, int32_t* task_id) {
  Handle* H = (Handle*)handle;
  if (!H || !def || !task_id) return fail("sag_define_task: null argument");
  if (const char* what = task_def_error(*def, H->D.num_gremlins)) {
    snprintf(g_err, sizeof(g_err), "sag_define_task: %s", what);
    return 1;
  }
  if (H->custom_h.count >= SAG_MAX_CUSTOM_TASKS) return fail("sag_define_task: SAG_MAX_CUSTOM_TASKS tasks are defined already");
  DevGuard guard(H->device);
  CK(cudaDeviceSynchronize());  // ordered after everything issued earlier; the kernels read the table from the slab
  if (H->custom_h.count == 0) {  // the first definition switches the handle to the *C kernel set
    Handle T = *H;
    T.custom_h.count = 1;
    CK(SAG_DISPATCH(&T, setup(&T)));
    H->busy_grid = T.busy_grid;
  }
  CustomTable next = H->custom_h;
  next.t[next.count] = custom_task(*def);
  ++next.count;
  CK(cudaMemcpy(H->custom_d, &next, sizeof(next), cudaMemcpyHostToDevice));
  H->custom_h = next;
  *task_id = SAG_NUM_TASKS + next.count - 1;
  return 0;
}

int sag_set_tasks_host(void* handle, const int32_t* ids_host) {
  Handle* H = (Handle*)handle;
  if (!H || !ids_host) return fail("sag_set_tasks_host: null argument");
  const int nids = sag_num_task_ids(H);
  for (int e = 0; e < H->D.n; ++e)
    if (ids_host[e] < 0 || ids_host[e] >= nids) return fail("sag_set_tasks_host: task id out of range [0, sag_num_task_ids)");
  DevGuard guard(H->device);
  CK(cudaDeviceSynchronize());  // the host API is ordered after everything issued through the stream API
  CK(cudaMemcpyAsync(H->ids_d, ids_host, (size_t)H->D.n * sizeof(int32_t), cudaMemcpyHostToDevice, H->own_stream));
  if (launch_set_tasks(H, H->ids_d, H->own_stream)) return 1;
  CK(cudaStreamSynchronize(H->own_stream));
  return 0;
}

int sag_set_next_tasks(void* handle, const int32_t* ids, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !ids) return fail("sag_set_next_tasks: null argument");
  DevGuard guard(H->device);
  // the ids are checked where they are consumed (k_reset), like ids written with sag_write_field
  CK(cudaMemcpyAsync(H->next_task, ids, (size_t)H->D.n * sizeof(int32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int sag_set_next_tasks_host(void* handle, const int32_t* ids_host) {
  Handle* H = (Handle*)handle;
  if (!H || !ids_host) return fail("sag_set_next_tasks_host: null argument");
  const int nids = sag_num_task_ids(H);
  for (int e = 0; e < H->D.n; ++e)
    if (ids_host[e] < -1 || ids_host[e] >= nids)
      return fail("sag_set_next_tasks_host: task id out of range [-1, sag_num_task_ids)");
  DevGuard guard(H->device);
  CK(cudaDeviceSynchronize());  // the host API is ordered after everything issued through the stream API
  CK(cudaMemcpyAsync(H->next_task, ids_host, (size_t)H->D.n * sizeof(int32_t), cudaMemcpyHostToDevice, H->own_stream));
  CK(cudaStreamSynchronize(H->own_stream));
  return 0;
}

int sag_bound(void* handle, double* bound, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !bound) return fail("sag_bound: null argument");
  DevGuard guard(H->device);
  CK(cudaMemcpyAsync(bound, H->D.bound, (size_t)H->D.n * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

static int copy_envs_check(const Handle* D, const Handle* S, const char* who) {
  if (!D || !S) { snprintf(g_err, sizeof(g_err), "%s: null handle", who); return 1; }
  if (D->device != S->device) { snprintf(g_err, sizeof(g_err), "%s: the handles are on different devices", who); return 1; }
  if (const char* what = copy_incompatibility(D->D, S->D, &D->custom_h, &S->custom_h)) {
    snprintf(g_err, sizeof(g_err), "%s: the handles differ in %s", who, what);
    return 1;
  }
  return 0;
}

static int launch_copy_envs(Handle* H, const Handle* S, const int32_t* src_of_dst, cudaStream_t s) {
  CopyFields F;
  for (int f = 0; f < SAG_NUM_FIELDS; ++f) {
    F.dst[f] = (char*)H->field_ptr[f]; F.src[f] = (const char*)S->field_ptr[f];
    F.rows[f] = kFieldShape[f].rows; F.elem[f] = kFieldShape[f].elem;
  }
  const int blocks = (H->D.n + kCopyThreads - 1) / kCopyThreads;
  auto fold = H->custom_h.count > 0 ? k_copy_envs_fold_custom : k_copy_envs_fold;
  fold<<<blocks, kCopyThreads, 0, s>>>(H->D, src_of_dst, S->D.n, H == S, H->sret, H->scost, H->sn, H->stats_acc);
  ++H->launches;
  CK(cudaGetLastError());
  k_copy_envs<<<dim3(blocks, copy_chunks()), kCopyThreads, 0, s>>>(H->D, F, src_of_dst, S->D.n, S->D.stride, H == S);
  ++H->launches;
  CK(cudaGetLastError());
  return 0;
}

int sag_copy_envs(void* dst, void* src, const int32_t* src_of_dst, void* stream) {
  Handle *H = (Handle*)dst, *S = (Handle*)src;
  if (!src_of_dst) return fail("sag_copy_envs: null argument");
  if (copy_envs_check(H, S, "sag_copy_envs")) return 1;
  DevGuard guard(H->device);
  // the pairs are checked in the kernel (copy_env_source): bad ones are not applied and set SAG_ERR_BAD_ENV_INDEX
  return launch_copy_envs(H, S, src_of_dst, (cudaStream_t)stream);
}

int sag_copy_envs_host(void* dst, void* src, const int32_t* src_of_dst_host) {
  Handle *H = (Handle*)dst, *S = (Handle*)src;
  if (!src_of_dst_host) return fail("sag_copy_envs_host: null argument");
  if (copy_envs_check(H, S, "sag_copy_envs_host")) return 1;
  if (const char* what = copy_index_error(src_of_dst_host, H->D.n, S->D.n, H == S)) {
    snprintf(g_err, sizeof(g_err), "sag_copy_envs_host: %s", what);
    return 1;
  }
  DevGuard guard(H->device);
  CK(cudaDeviceSynchronize());  // the host API is ordered after everything issued through the stream API
  CK(cudaMemcpyAsync(H->ids_d, src_of_dst_host, (size_t)H->D.n * sizeof(int32_t), cudaMemcpyHostToDevice, H->own_stream));
  if (launch_copy_envs(H, S, H->ids_d, H->own_stream)) return 1;
  CK(cudaStreamSynchronize(H->own_stream));
  return 0;
}

int sag_bound_host(void* handle, double* bound_host) {
  Handle* H = (Handle*)handle;
  if (!H || !bound_host) return fail("sag_bound_host: null argument");
  DevGuard guard(H->device);
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(bound_host, H->D.bound, (size_t)H->D.n * sizeof(double), cudaMemcpyDeviceToHost));
  return 0;
}

int sag_error_flags(void* handle, int clear) {
  Handle* H = (Handle*)handle;
  if (!H) return 0;
  int w = 0;
  if (H->err_h[0]) w |= SAG_FLAG_RESAMPLE_FAILED;
  if (H->err_h[1]) w |= SAG_ERR_BAD_TASK_ID;
  if (H->err_h[2]) w |= SAG_ERR_BAD_ENV_INDEX;
  if (clear) { H->err_h[0] = 0; H->err_h[1] = 0; H->err_h[2] = 0; }
  return w;
}

int sag_seed(void* handle, uint64_t seed) {
  Handle* H = (Handle*)handle;
  if (!H) return fail("sag_seed: null handle");
  DevGuard guard(H->device);
  CK(cudaDeviceSynchronize());
  // the key lives in the slab, so that kernels recorded in a CUDA graph draw from the new key on their next replay
  H->D.seed = seed;
  CK(cudaMemcpyAsync(H->D.key, &seed, sizeof(seed), cudaMemcpyHostToDevice, H->own_stream));
  CK(cudaMemsetAsync(H->D.episode, 0xFF, (size_t)H->D.stride * sizeof(unsigned), H->own_stream));
  CK(cudaStreamSynchronize(H->own_stream));
  return 0;
}

int sag_reset(void* handle, const uint8_t* mask, int only_flagged, int new_task, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H) return fail("sag_reset: null handle");
  DevGuard guard(H->device);
  CK(SAG_DISPATCH(H, reset(H, mask, only_flagged, new_task, nullptr, nullptr, (cudaStream_t)stream)));
  return 0;
}

int sag_reset_obs(void* handle, const uint8_t* mask, int only_flagged, int new_task, float* obs, uint8_t* was_reset, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !obs) return fail("sag_reset_obs: null argument");
  DevGuard guard(H->device);
  CK(SAG_DISPATCH(H, reset(H, mask, only_flagged, new_task, obs, was_reset, (cudaStream_t)stream)));
  return 0;
}

int sag_reset_host(void* handle, const uint8_t* mask_h, int only_flagged, int new_task, float* obs_h) {
  Handle* H = (Handle*)handle;
  if (!H) return fail("sag_reset_host: null handle");
  DevGuard guard(H->device);
  cudaStream_t s = H->own_stream;
  CK(cudaDeviceSynchronize());  // the host API is ordered after everything issued through the stream API
  const uint8_t* m = nullptr;
  if (mask_h) { CK(cudaMemcpyAsync(H->mask_d, mask_h, (size_t)H->D.n, cudaMemcpyHostToDevice, s)); m = H->mask_d; }
  CK(SAG_DISPATCH(H, reset(H, m, only_flagged, new_task, nullptr, nullptr, s)));
  if (obs_h) {
    CK(SAG_DISPATCH(H, observe(H, H->obs_d, s)));
    CK(cudaMemcpyAsync(obs_h, H->obs_d, (size_t)H->D.n * (size_t)sag_obs_dim(H) * sizeof(float), cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  if (H->err_h[0]) return fail("sag_reset_host: failed to generate a layout (ResamplingError, world.py:189); see sag_error_flags");
  return 0;
}

int sag_step(void* handle, const float* act, float* obs, double* reward, double* reward2, uint8_t* cost, uint8_t* done,
             void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !act || !obs || !reward || !cost || !done) return fail("sag_step: null argument");
  DevGuard guard(H->device);
  CK(SAG_DISPATCH(H, step(H, act, obs, reward, reward2, cost, done, (cudaStream_t)stream)));
  return 0;
}

int sag_evaluate_actions(void* handle, int h_steps, const float* act, double discount, float* obs, double* ret, int ret_cols,
                         double* cost, int32_t* length, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !act || !obs || !ret || !cost || !length || h_steps <= 0 || (ret_cols != 1 && ret_cols != 2))
    return fail("sag_evaluate_actions: bad argument");
  DevGuard guard(H->device);
  CK(SAG_DISPATCH(H, evaluate(H, h_steps, act, discount, obs, ret, ret_cols, cost, length, (cudaStream_t)stream)));
  return 0;
}

int sag_export_outputs(void* handle, const float* obs, const double* reward, int reward_cols, const uint8_t* cost, const uint8_t* done,
                       const double* bound, float* obs_out, double* reward_out, float* cost_out, uint8_t* done_out, double* bound_out,
                       void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !obs || !reward || !cost || !done || !obs_out || !reward_out || !cost_out || !done_out || (reward_cols != 1 && reward_cols != 2) ||
      (bound_out && !bound))
    return fail("sag_export_outputs: bad argument");
  DevGuard guard(H->device);
  const int quads = sag_obs_dim(H) / 4;
  const size_t total = (size_t)H->D.n * quads;
  int grid = (int)((total + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  k_export_outputs<<<grid, 256, 0, (cudaStream_t)stream>>>(H->D.n, quads, reward_cols, (const float4*)obs, reward, cost, done, bound,
                                                          (float4*)obs_out, reward_out, cost_out, done_out, bound_out);
  ++H->launches;
  CK(cudaGetLastError());
  return 0;
}

int sag_observe(void* handle, float* obs, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !obs) return fail("sag_observe: null argument");
  DevGuard guard(H->device);
  CK(SAG_DISPATCH(H, observe(H, obs, (cudaStream_t)stream)));
  return 0;
}

int sag_rollout(void* handle, int k_steps, float* obs, double* reward, uint8_t* cost, uint8_t* done, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || k_steps <= 0) return fail("sag_rollout: bad argument");
  DevGuard guard(H->device);
  CK(SAG_DISPATCH(H, rollout(H, k_steps, obs, reward, cost, done, (cudaStream_t)stream)));
  return 0;
}

// device-visible alias of a pinned (page-locked, mapped) host pointer, or nullptr for pageable memory
static void* mapped_alias(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (a.type != cudaMemoryTypeHost || !a.devicePointer) return nullptr;
  return a.devicePointer;
}

int sag_step_host(void* handle, const float* act_h, float* obs_h, double* reward_h, uint8_t* cost_h, uint8_t* done_h) {
  Handle* H = (Handle*)handle;
  if (!H || !act_h || !obs_h || !reward_h || !cost_h || !done_h) return fail("sag_step_host: null argument");
  DevGuard guard(H->device);
  cudaStream_t s = H->own_stream;
  const size_t n = (size_t)H->D.n, od = (size_t)sag_obs_dim(H);
#if defined(SAG_E2E_TIMING)  // tuning builds: where does an end-to-end step spend its time?  (events on the handle's two streams)
  static cudaEvent_t te[6];
  static double tacc[6];
  static int tcnt = 0;
  if (!te[0]) for (int i = 0; i < 6; ++i) cudaEventCreate(&te[i]);
  struct timespec w0, w1;
  clock_gettime(CLOCK_MONOTONIC, &w0);
  cudaEventRecord(te[0], s);
#endif
  CK(cudaMemcpyAsync(H->act_d, act_h, n * 2 * sizeof(float), cudaMemcpyHostToDevice, s));
#if defined(SAG_E2E_TIMING)
  cudaEventRecord(te[1], s);
#endif
  float* obs_m = (float*)mapped_alias(obs_h);
  double* rew_m = (double*)mapped_alias(reward_h);
  uint8_t *cost_m = (uint8_t*)mapped_alias(cost_h), *done_m = (uint8_t*)mapped_alias(done_h);
  // (Storing the outputs straight into the mapped buffers from the kernels -- no copy engine, no fix-up -- was measured and
  // lost: SM writes over PCIe sustain ~29 GB/s against the copy engine's ~56, e2e 1.56e8 -> 1.15e8.)
  if (obs_m && rew_m && cost_m && done_m) {
    // Pinned output buffers: the bulk device-to-host copy starts as soon as the quiet kernel is done and runs under the
    // busy kernel; the rows the busy kernel produced (5-30 % of them) follow as direct writes into the mapped buffers.
    // The copy of the observation rows (16 MB: the long pole of the step at PCIe speed) starts when the batch kernel is
    // done and runs under the contact kernel.  (Launching the batch kernel in chunks so that copies could start earlier
    // was measured and lost: the kernel's duration is the latency of one thread's step, not throughput, so every chunk
    // costs as much as the whole batch -- e2e 1.51e8 -> 1.27e8.)
    cudaStream_t c = H->copy_stream;
    // (Reading the actions straight from the pinned host buffer in the kernels instead of copying them first: no difference,
    // 1.556e8 either way.  A split copy -- head of the observation rows under the contact kernel, tail + reward / cost / done after it so that
    // the fix-up runs under the tail, split point adapted from the previous step's timings -- was measured and lost by 1-5 %:
    // the contact kernel's duration varies by +-20 us from step to step, and a copy engine that waits costs more than the
    // 27 us fix-up it hides.)
    CK(SAG_DISPATCH(H, step_free(H, H->act_d, H->obs_d, H->rew_d, nullptr, H->cost_d, H->done_d, s)));
    CK(cudaEventRecord(H->ev_free, s));
    CK(cudaStreamWaitEvent(c, H->ev_free, 0));
    CK(cudaMemcpyAsync(obs_h, H->obs_d, n * od * sizeof(float), cudaMemcpyDeviceToHost, c));
    bool packed = is_packed_block(obs_h);  // a block from sag_host_alloc_outputs, used as handed out
    packed = packed && (char*)reward_h - (char*)obs_h == (char*)H->rew_d - (char*)H->obs_d &&
             (char*)cost_h - (char*)obs_h == (char*)H->cost_d - (char*)H->obs_d &&
             (char*)done_h - (char*)obs_h == (char*)H->done_d - (char*)H->obs_d;
    if (packed) {  // buffers from sag_host_alloc_outputs: reward, cost and done in one copy
      CK(cudaMemcpyAsync(reward_h, H->rew_d, (size_t)((char*)H->done_d - (char*)H->rew_d) + n, cudaMemcpyDeviceToHost, c));
    } else {
      CK(cudaMemcpyAsync(reward_h, H->rew_d, n * sizeof(double), cudaMemcpyDeviceToHost, c));
      CK(cudaMemcpyAsync(cost_h, H->cost_d, n, cudaMemcpyDeviceToHost, c));
      CK(cudaMemcpyAsync(done_h, H->done_d, n, cudaMemcpyDeviceToHost, c));
    }
    CK(cudaEventRecord(H->ev_copied, c));
#if defined(SAG_E2E_TIMING)
    cudaEventRecord(te[3], c);   // bulk copy done
    cudaEventRecord(te[2], s);   // batch kernel done (the copy stream waited for the same point)
#endif
    CK(SAG_DISPATCH(H, step_coop(H, H->act_d, H->obs_d, H->rew_d, nullptr, H->cost_d, H->done_d, s)));
#if defined(SAG_E2E_TIMING)
    cudaEventRecord(te[4], s);   // contact kernel done
#endif
    CK(cudaStreamWaitEvent(s, H->ev_copied, 0));
    CK(SAG_DISPATCH(H, fixup_host(H, H->obs_d, H->rew_d, H->cost_d, H->done_d, obs_m, rew_m, cost_m, done_m, s)));
#if defined(SAG_E2E_TIMING)
    cudaEventRecord(te[5], s);
#endif
    CK(cudaStreamSynchronize(s));
#if defined(SAG_E2E_TIMING)
    clock_gettime(CLOCK_MONOTONIC, &w1);
    {
      float ms;
      for (int i = 1; i < 6; ++i) { cudaEventElapsedTime(&ms, te[0], te[i]); tacc[i] += ms; }
      tacc[0] += 1e3 * (double)(w1.tv_sec - w0.tv_sec) + 1e-6 * (double)(w1.tv_nsec - w0.tv_nsec);
      if (++tcnt % 40 == 0) {
        fprintf(stderr, "sag_step_host (avg of 40, ms since the first enqueue): h2d done %.3f, batch kernel done %.3f, bulk copy done %.3f, contact kernel done %.3f, fix-up done %.3f | wall %.3f\n",
                tacc[1] / 40, tacc[2] / 40, tacc[3] / 40, tacc[4] / 40, tacc[5] / 40, tacc[0] / 40);
        for (int i = 0; i < 6; ++i) tacc[i] = 0.0;
      }
    }
#endif
    return 0;
  }
  CK(SAG_DISPATCH(H, step(H, H->act_d, H->obs_d, H->rew_d, nullptr, H->cost_d, H->done_d, s)));
  CK(cudaMemcpyAsync(obs_h, H->obs_d, n * od * sizeof(float), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(reward_h, H->rew_d, n * sizeof(double), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(cost_h, H->cost_d, n, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(done_h, H->done_d, n, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}

int sag_observe_host(void* handle, float* obs_h) {
  Handle* H = (Handle*)handle;
  if (!H || !obs_h) return fail("sag_observe_host: null argument");
  DevGuard guard(H->device);
  cudaStream_t s = H->own_stream;
  CK(cudaDeviceSynchronize());  // the host API is ordered after everything issued through the stream API
  CK(SAG_DISPATCH(H, observe(H, H->obs_d, s)));
  CK(cudaMemcpyAsync(obs_h, H->obs_d, (size_t)H->D.n * (size_t)sag_obs_dim(H) * sizeof(float), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}

// One pinned block laid out like the handle's device staging area (obs, reward, cost, done at the same relative offsets):
// sag_step_host then moves all four outputs with ONE device-to-host copy.  Free with sag_host_free(*obs_h).
int sag_host_alloc_outputs(void* handle, float** obs_h, double** reward_h, uint8_t** cost_h, uint8_t** done_h) {
  Handle* H = (Handle*)handle;
  if (!H || !obs_h || !reward_h || !cost_h || !done_h) return fail("sag_host_alloc_outputs: null argument");
  DevGuard guard(H->device);
  const size_t span = (size_t)((char*)H->done_d - (char*)H->obs_d) + (size_t)H->D.n;
  char* p = nullptr;
  CK(cudaHostAlloc((void**)&p, span, cudaHostAllocDefault));
  memset(p, 0, span);
  for (int k = 0; k < 64; ++k) if (!g_packed_blocks[k]) { g_packed_blocks[k] = p; break; }
  *obs_h = (float*)p;
  *reward_h = (double*)(p + ((char*)H->rew_d - (char*)H->obs_d));
  *cost_h = (uint8_t*)(p + ((char*)H->cost_d - (char*)H->obs_d));
  *done_h = (uint8_t*)(p + ((char*)H->done_d - (char*)H->obs_d));
  return 0;
}

// Measurement helper (tools/probe_d2h.py, bench.py): `reps` back-to-back device -> pinned-host copies of `bytes` bytes on the
// handle's device, with the same allocation and copy calls sag_step_host uses; returns the elapsed seconds.
int sag_probe_d2h(void* handle, size_t bytes, int reps, double* seconds) {
  Handle* H = (Handle*)handle;
  if (!H || !seconds || bytes == 0 || reps <= 0) return fail("sag_probe_d2h: bad argument");
  DevGuard guard(H->device);
  if (bytes > H->slab_bytes) bytes = H->slab_bytes;
  void* p = nullptr;
  CK(cudaHostAlloc(&p, bytes, cudaHostAllocDefault));
  memset(p, 0, bytes);
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  cudaStream_t s = H->copy_stream;
  CK(cudaDeviceSynchronize());
  for (int i = 0; i < 3; ++i) CK(cudaMemcpyAsync(p, H->slab, bytes, cudaMemcpyDeviceToHost, s));
  CK(cudaEventRecord(e0, s));
  for (int i = 0; i < reps; ++i) CK(cudaMemcpyAsync(p, H->slab, bytes, cudaMemcpyDeviceToHost, s));
  CK(cudaEventRecord(e1, s));
  CK(cudaStreamSynchronize(s));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, e0, e1));
  *seconds = 1e-3 * (double)ms;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFreeHost(p);
  return 0;
}

void* sag_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { fail("sag_host_alloc: cudaHostAlloc failed"); return nullptr; }
  return p;
}
void sag_host_free(void* p) {
  if (!p) return;
  for (int k = 0; k < 64; ++k) if (g_packed_blocks[k] == p) g_packed_blocks[k] = nullptr;
  cudaFreeHost(p);
}

int sag_read_field(void* handle, int field, void* dst, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !dst || field < 0 || field >= SAG_NUM_FIELDS) return fail("sag_read_field: bad argument");
  DevGuard guard(H->device);
  CK(cudaMemcpyAsync(dst, H->field_ptr[field], H->field_bytes[field], cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}
int sag_write_field(void* handle, int field, const void* src, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !src || field < 0 || field >= SAG_NUM_FIELDS) return fail("sag_write_field: bad argument");
  DevGuard guard(H->device);
  CK(cudaMemcpyAsync(H->field_ptr[field], src, H->field_bytes[field], cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  // The step's shortcuts read the clearance and moving mask cached in TASK_F64 / TASK_I32: rebuild them from the state
  // just written (k_observe, into the staging buffer no caller sees).  On a state the kernels left, this rewrites the
  // same values.  The queued next task is read by the resets only.
  if (field != SAG_F_NEXT_TASK) CK(SAG_DISPATCH(H, observe(H, H->obs_d, (cudaStream_t)stream)));
  return 0;
}

int sag_task_stats(void* handle, double* out, int reset, void* stream) {
  Handle* H = (Handle*)handle;
  if (!H || !out) return fail("sag_task_stats: null argument");
  DevGuard guard(H->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t rows = (size_t)sag_num_task_ids(H);
  CK(cudaMemcpyAsync(out, H->stats_acc, rows * 3 * sizeof(double), cudaMemcpyDeviceToDevice, s));
  if (H->custom_h.count > 0) k_task_stats_custom<<<148, 256, 0, s>>>(H->D, H->sret, H->scost, H->sn, out);
  else k_task_stats<<<148, 256, 0, s>>>(H->D, H->sret, H->scost, H->sn, out);
  ++H->launches;
  CK(cudaGetLastError());
  if (reset) {
    CK(cudaMemsetAsync(H->sret, 0, 3 * (size_t)H->D.stride * sizeof(double), s));
    CK(cudaMemsetAsync(H->stats_acc, 0, rows * 3 * sizeof(double), s));
  }
  return 0;
}

int sag_lidar(const double* robot, const double* obj_xy, const uint8_t* group, int n, int nslots, float* out, void* stream) {
  if (!robot || !obj_xy || !group || !out || n <= 0 || nslots < 0) return fail("sag_lidar: bad argument");
  k_lidar<<<grid_for(n), kBS, 0, (cudaStream_t)stream>>>(robot, obj_xy, group, n, nslots, out);
  CK(cudaGetLastError());
  return 0;
}

int sag_cost(const double* robot_xy, const float* hazard_xy, const uint8_t* contact, int n, int nh, double hazard_size,
             uint8_t* out, void* stream) {
  if (!robot_xy || !hazard_xy || !contact || !out || n <= 0 || nh < 0) return fail("sag_cost: bad argument");
  if (nh == 9) k_cost<9><<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(robot_xy, hazard_xy, contact, n, nh, hazard_size, out);
  else k_cost<0><<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(robot_xy, hazard_xy, contact, n, nh, hazard_size, out);
  CK(cudaGetLastError());
  return 0;
}

}  // extern "C"
