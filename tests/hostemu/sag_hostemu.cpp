// sag_hostemu.cpp -- TEST INFRASTRUCTURE ONLY (never loaded by the product package).
//
// Compiles the per-environment kernel body (safe_adaptation_gym_b200/csrc/sag_core.cuh) with g++ and
// drives it with the same CTA/tile structure as sag_kernels.cu, behind the same C ABI symbols, with
// "device" pointers being host pointers.  It lets the GPU-less build container check the kernel body
// against the oracle (tests/test_hostemu_parity.py); on the B200 box the same tests run on the real
// library (tests/test_gpu_parity.py).  The product (safe_adaptation_gym_b200/_abi.py) loads only
// csrc/libsag_b200.so and raises if it is missing.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "../../include/sag_b200.h"
#include "../../safe_adaptation_gym_b200/csrc/sag_core.cuh"
#include "../../safe_adaptation_gym_b200/csrc/sag_layout.h"

#ifdef SAG_PROFILE
long* sag_prof_ptr = nullptr;
extern "C" void sag_prof_set(long* p) { sag_prof_ptr = p; }
#endif

using namespace sag;

namespace {
constexpr int kBS = 128, kTileStride = kBS + 1, kObsMax = SAG_OBS_CAR;
char g_err[512] = "";
int fail(const char* w) { snprintf(g_err, sizeof(g_err), "%s", w); return 1; }
struct Handle {
  Dev D;
  char* slab;
  SlabLayout LY;
  double *sret, *scost, *sn, *stats_acc;
  int err[4];
};
void write_tile(const float* tile, float* out, int e0, int n, int kObs) {
  int cnt = (n - e0 < kBS ? n - e0 : kBS) * kObs;
  float* dst = out + (size_t)e0 * kObs;
  for (int i = 0; i < cnt; ++i) { int t = i / kObs, k = i - t * kObs; dst[i] = tile[k * kTileStride + t]; }
}
int obs_dim_of(const Dev& D) { return D.robot == SAG_ROBOT_CAR ? SAG_OBS_CAR : SAG_OBS_POINT; }

template <class RB>
void do_reset(Handle* H, const uint8_t* mask, int only_flagged, int new_task, float* obs, uint8_t* was_reset) {
  Dev& D = H->D;
  static float tile[kObsMax * kTileStride];
  static Scratch scratch;
  for (int e = 0; e < D.n; ++e) {
    bool doit = true;
    if (mask && !mask[e]) doit = false;
    if (doit && only_flagged && !(D.flags[e] & F_NEEDS_RESET)) doit = false;
    if (was_reset) was_reset[e] = doit ? 1 : 0;
    if (!doit) continue;
    if ((D.flags[e] & F_NEEDS_RESET) && D.nstep[e] > 0) { H->sret[e] += D.epret[e]; H->scost[e] += D.epcost[e]; H->sn[e] += 1.0; }
    env_reset<RB>(D, e, D.episode[e] + 1u, new_task != 0);
    if (D.flags[e] & F_RESAMPLE_FAILED) D.errflags[0] = 1;
    if (obs) {
      env_observe<RB>(1u, &scratch, D, e, tile, kTileStride);
      for (int k = 0; k < RB::kObsDim; ++k) obs[(size_t)e * RB::kObsDim + k] = tile[k * kTileStride];
    }
  }
}
template <class RB>
void do_step(Handle* H, const float* act, float* obs, double* reward, double* reward2, uint8_t* cost, uint8_t* done) {
  Dev& D = H->D;
  static float tile[kObsMax * kTileStride];
  static Scratch scratch;
  for (int e0 = 0; e0 < D.n; e0 += kBS) {
    for (int t = 0; t < kBS && e0 + t < D.n; ++t) {
      int e = e0 + t; double rew[2]; unsigned char c, d;
      // same dispatch as the CUDA kernels (sag_kernels.cu: k_step_free, then the work list): environments in which nothing
      // moves take the contact-free path, with the exact pre-tests unless they are quiet; one whose pre-test fires has
      // stored nothing and is stepped again by the contact path (the scalar one here, the cooperative one on the GPU)
      bool run = false, pretest = false;
      {
        RB R;
        load_robot(D, e, task_spec(D.task[e]), R);
        run = !(D.flags[e] & F_PHYS_ERROR) && D.movmask[e] == 0 && D.num_gremlins == 0;
        pretest = !env_is_quiet(D.clear[e], R);
      }
      bool bail = true;
      if (run) bail = env_step<kStepNear, RB>(1u, nullptr, D, e, act[2 * e], act[2 * e + 1], tile + t, kTileStride, rew, &c, &d, pretest) != 0;
      if (bail) env_step<kStepFull, RB>(1u, &scratch, D, e, act[2 * e], act[2 * e + 1], tile + t, kTileStride, rew, &c, &d);
      reward[e] = rew[0];
      if (reward2) { reward2[2 * e] = rew[0]; reward2[2 * e + 1] = rew[1]; }
      cost[e] = c; done[e] = d;
    }
    write_tile(tile, obs, e0, D.n, RB::kObsDim);
  }
}
template <class RB>
void do_observe(Handle* H, float* obs) {
  Dev& D = H->D;
  static float tile[kObsMax * kTileStride];
  static Scratch scratch;
  for (int e0 = 0; e0 < D.n; e0 += kBS) {
    for (int t = 0; t < kBS && e0 + t < D.n; ++t) env_observe<RB>(1u, &scratch, D, e0 + t, tile + t, kTileStride);
    write_tile(tile, obs, e0, D.n, RB::kObsDim);
  }
}
// sag_write_field: the clearance and moving mask that the step's dispatch reads, rebuilt as k_observe rebuilds them; the
// observation is dropped
template <class RB>
void do_refresh(Handle* H) {
  static float tile[kObsMax * kTileStride];
  static Scratch scratch;
  for (int e = 0; e < H->D.n; ++e) env_observe<RB>(1u, &scratch, H->D, e, tile, kTileStride);
}
template <class RB>
void do_rollout(Handle* H, int k_steps, float* obs, double* reward, uint8_t* cost, uint8_t* done) {
  Dev& D = H->D;
  static float tile[kObsMax * kTileStride];
  static Scratch scratch;
  for (int e0 = 0; e0 < D.n; e0 += kBS) {
    for (int t = 0; t < kBS && e0 + t < D.n; ++t) {
      int e = e0 + t; double rew[2] = {0, 0}; unsigned char c = 0, d = 0;
      Rng rng = {D.seed, D.gid_base + (uint32_t)e, D.episode[e]};
      uint32_t base = (uint32_t)D.nstep[e];
      for (int k = 0; k < k_steps; ++k) {
        double u1, u2; rng.pair(2u, base + (uint32_t)k, u1, u2);
        env_step<kStepFull, RB>(1u, &scratch, D, e, (float)(2.0 * u1 - 1.0), (float)(2.0 * u2 - 1.0), tile + t, kTileStride, rew, &c, &d);
      }
      if (reward) reward[e] = rew[0];
      if (cost) cost[e] = c;
      if (done) done[e] = d;
    }
    if (obs) write_tile(tile, obs, e0, D.n, RB::kObsDim);
  }
}
}  // namespace

// one instantiation per robot model; environments with gremlins use the *G variants (as SAG_DISPATCH in sag_kernels.cu)
#define HOSTEMU_DISPATCH(H, fn, args)                                                                  \
  do {                                                                                                 \
    if ((H)->D.robot == SAG_ROBOT_CAR) { if ((H)->D.num_gremlins > 0) fn<CarRobotG> args; else fn<CarRobot> args; } \
    else { if ((H)->D.num_gremlins > 0) fn<PointRobotG> args; else fn<PointRobot> args; }              \
  } while (0)

extern "C" {
const char* sag_last_error(void) { return g_err; }
int sag_abi_version(void) { return SAG_ABI_VERSION; }
void sag_default_config(SagConfig* c) { default_config(c); }
int sag_create(const SagConfig* cfg, int device, void** handle) {
  (void)device;
  if (!cfg || !handle || cfg->n_envs <= 0) return fail("sag_create: bad argument");
  Handle* H = new Handle();
  memset(H, 0, sizeof(*H));
  dev_from_config(H->D, *cfg);
  H->LY = slab_layout(H->D.n, H->D.stride, obs_dim_of(H->D));
  H->slab = (char*)calloc(1, H->LY.total);
  slab_bind(H->D, H->LY, H->slab);
  size_t st = H->D.stride;
  H->sret = (double*)(H->slab + H->LY.stats_off); H->scost = H->sret + st; H->sn = H->sret + 2 * st;
  H->stats_acc = (double*)(H->slab + H->LY.acc_off);
  H->D.errflags = H->err;
  memset(H->D.episode, 0xFF, st * sizeof(unsigned));
  *handle = H;
  return 0;
}
int sag_destroy(void* h) { Handle* H = (Handle*)h; if (H) { free(H->slab); delete H; } return 0; }
unsigned long long sag_launch_count(void* h) { (void)h; return 0ull; }
int sag_debug_read(void* h, unsigned long long* out16) { (void)h; memset(out16, 0, 18 * sizeof(unsigned long long)); return 0; }
int sag_stride(void* h) { return ((Handle*)h)->D.stride; }
int sag_obs_dim(void* h) { return obs_dim_of(((Handle*)h)->D); }
size_t sag_field_bytes(void* h, int f) { return (f < 0 || f >= SAG_NUM_FIELDS) ? 0 : ((Handle*)h)->LY.bytes[f]; }
int sag_set_tasks(void* h, const int32_t* ids, void* s) {
  (void)s; Handle* H = (Handle*)h; Dev& D = H->D;
  for (int e = 0; e < D.n; ++e) {  // same logic as k_set_tasks
    const int old = D.task[e];
    double r = H->sret[e], c = H->scost[e], k = H->sn[e];
    if ((D.flags[e] & F_NEEDS_RESET) && D.nstep[e] > 0) { r += D.epret[e]; c += D.epcost[e]; k += 1.0; D.nstep[e] = 0; }
    if (k != 0.0 && old >= 0 && old < SAG_NUM_TASKS) { H->stats_acc[3 * old] += r; H->stats_acc[3 * old + 1] += c; H->stats_acc[3 * old + 2] += k; }
    H->sret[e] = H->scost[e] = H->sn[e] = 0.0;
    int id = ids[e];
    if (id < 0 || id >= SAG_NUM_TASKS) { id = SAG_T_GO_TO_GOAL; D.errflags[1] = 1; }
    D.task[e] = id;
  }
  return 0;
}
int sag_error_flags(void* h, int clear) {
  Handle* H = (Handle*)h;
  int w = (H->err[0] ? SAG_FLAG_RESAMPLE_FAILED : 0) | (H->err[1] ? SAG_ERR_BAD_TASK_ID : 0);
  if (clear) H->err[0] = H->err[1] = 0;
  return w;
}
int sag_seed(void* h, uint64_t seed) { Handle* H = (Handle*)h; H->D.seed = seed; memset(H->D.episode, 0xFF, (size_t)H->D.stride * sizeof(unsigned)); return 0; }
int sag_reset(void* h, const uint8_t* mask, int only_flagged, int new_task, void* s) {
  (void)s; Handle* H = (Handle*)h;
  HOSTEMU_DISPATCH(H, do_reset, (H, mask, only_flagged, new_task, nullptr, nullptr));
  return 0;
}
int sag_reset_obs(void* h, const uint8_t* mask, int only_flagged, int new_task, float* obs, uint8_t* was_reset, void* s) {
  (void)s; Handle* H = (Handle*)h;
  HOSTEMU_DISPATCH(H, do_reset, (H, mask, only_flagged, new_task, obs, was_reset));
  return 0;
}
int sag_step(void* h, const float* act, float* obs, double* reward, double* reward2, uint8_t* cost, uint8_t* done, void* s) {
  (void)s; Handle* H = (Handle*)h;
  HOSTEMU_DISPATCH(H, do_step, (H, act, obs, reward, reward2, cost, done));
  return 0;
}
int sag_observe(void* h, float* obs, void* s) {
  (void)s; Handle* H = (Handle*)h;
  HOSTEMU_DISPATCH(H, do_observe, (H, obs));
  return 0;
}
int sag_export_outputs(void* h, const float* obs, const double* reward, int reward_cols, const uint8_t* cost, const uint8_t* done,
                       const double* bound, float* obs_out, double* reward_out, float* cost_out, uint8_t* done_out, double* bound_out,
                       void* s) {
  (void)s; Handle* H = (Handle*)h;
  const int n = H->D.n, od = obs_dim_of(H->D);
  memcpy(obs_out, obs, (size_t)n * od * sizeof(float));
  memcpy(reward_out, reward, (size_t)n * reward_cols * sizeof(double));
  for (int e = 0; e < n; ++e) { cost_out[e] = (float)cost[e]; done_out[e] = done[e] ? 1 : 0; if (bound_out) bound_out[e] = bound[e]; }
  return 0;
}
int sag_rollout(void* h, int k_steps, float* obs, double* reward, uint8_t* cost, uint8_t* done, void* s) {
  (void)s; Handle* H = (Handle*)h;
  HOSTEMU_DISPATCH(H, do_rollout, (H, k_steps, obs, reward, cost, done));
  return 0;
}
int sag_read_field(void* h, int f, void* dst, void* s) { (void)s; Handle* H = (Handle*)h; memcpy(dst, H->slab + H->LY.off[f], H->LY.bytes[f]); return 0; }
int sag_write_field(void* h, int f, const void* src, void* s) {
  (void)s; Handle* H = (Handle*)h;
  memcpy(H->slab + H->LY.off[f], src, H->LY.bytes[f]);
  if (f != SAG_F_NEXT_TASK) HOSTEMU_DISPATCH(H, do_refresh, (H));
  return 0;
}
int sag_task_stats(void* h, double* out, int reset, void* s) {
  (void)s; Handle* H = (Handle*)h; Dev& D = H->D;
  memcpy(out, H->stats_acc, SAG_NUM_TASKS * 3 * sizeof(double));
  for (int e = 0; e < D.n; ++e) { int t = D.task[e]; out[3 * t] += H->sret[e]; out[3 * t + 1] += H->scost[e]; out[3 * t + 2] += H->sn[e]; }
  if (reset) { memset(H->sret, 0, 3 * (size_t)D.stride * sizeof(double)); memset(H->stats_acc, 0, SAG_NUM_TASKS * 3 * sizeof(double)); }
  return 0;
}
int sag_lidar(const double* robot, const double* obj_xy, const uint8_t* group, int n, int nslots, float* out, void* s) {
  (void)s;
  for (int e = 0; e < n; ++e) {
    float bins[48]; for (int k = 0; k < 48; ++k) bins[k] = 0.f;
    double sn, cs; sag_sincos(robot[2 * (size_t)n + e], &sn, &cs);
    for (int sl = 0; sl < nslots; ++sl) {
      int g = group[(size_t)sl * n + e]; if (!g) continue;
      int off = g == 1 ? 0 : (g == 3 ? 16 : 32);
      lidar_accum(robot[e], robot[(size_t)n + e], cs, sn, obj_xy[(size_t)sl * n + e], obj_xy[((size_t)nslots + sl) * n + e], bins + off, 1);
    }
    memcpy(out + (size_t)e * 48, bins, sizeof(bins));
  }
  return 0;
}
int sag_cost(const double* robot_xy, const float* hazard_xy, const uint8_t* contact, int n, int nh, double hazard_size, uint8_t* out, void* s) {
  (void)s;
  for (int e = 0; e < n; ++e) {
    bool hit = contact[e] != 0;
    for (int k = 0; k < nh; ++k) {
      double dx = robot_xy[e] - (double)hazard_xy[(size_t)k * n + e], dy = robot_xy[(size_t)n + e] - (double)hazard_xy[((size_t)nh + k) * n + e];
      if (sqrt(dx * dx + dy * dy) <= hazard_size) hit = true;
    }
    out[e] = hit;
  }
  return 0;
}
}
