// sag_core.cuh -- per-environment step / reset / observe logic of the B200 path.
//
// One CUDA thread owns one environment.  All state is SoA, environment-minor (field[slot][env]),
// so every load/store in here is coalesced across the 32 environments of a warp.  The functions are
// __host__ __device__ so that tests/hostemu can compile the very same body with g++ and compare it
// with the oracle on the GPU-less build container; the product only ever launches them from
// sag_kernels.cu on the device.
//
// Reference lines cited as file:line are relative to lasgroup/safe-adaptation-gym.
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/sag_detmath.h"

#if defined(__CUDACC__)
#define SAG_DEV_CONST __device__
#define SAG_HD __host__ __device__ __forceinline__
#define SAG_HD_NOINLINE __host__ __device__ __noinline__
#else
#define SAG_DEV_CONST
#define SAG_HD inline
#define SAG_HD_NOINLINE
#endif

#if defined(SAG_PROFILE) && !defined(__CUDACC__)
extern long* sag_prof_ptr;  // tests/hostemu instrumentation: per-env work counters [n][16]
#define SAG_PROF(e, i, n) do { if (sag_prof_ptr) sag_prof_ptr[(size_t)(e) * 16 + (i)] += (n); } while (0)
#define SAG_PROF_MAX(e, i, n) do { if (sag_prof_ptr && sag_prof_ptr[(size_t)(e) * 16 + (i)] < (n)) sag_prof_ptr[(size_t)(e) * 16 + (i)] = (n); } while (0)
#else
#define SAG_PROF(e, i, n) do { } while (0)
#define SAG_PROF_MAX(e, i, n) do { } while (0)
#endif

// SAG_TIMING (tuning builds only): the cooperative kernel accumulates clock64() intervals per section into D.dbg[16]
#if defined(SAG_TIMING) && defined(__CUDA_ARCH__)
#define SAG_CLK_DECL long long clk_ = clock64()
#define SAG_CLK_RESET do { clk_ = clock64(); } while (0)
#define SAG_CLK(i) do { long long now_ = clock64(); if ((threadIdx.x & 31) == 0) atomicAdd(&D.dbg[i], (unsigned long long)(now_ - clk_)); clk_ = now_; } while (0)
// same, and the interval is also added to this environment's own section sum g (0 detect, 1 setup, 2 pgs) in the warp's Scratch
#define SAG_CLKG(i, g, Sref) do { long long now_ = clock64(); if ((threadIdx.x & 31) == 0) { atomicAdd(&D.dbg[i], (unsigned long long)(now_ - clk_)); (Sref).tsum[g] += (unsigned long long)(now_ - clk_); } clk_ = now_; } while (0)
#else
#define SAG_CLK_DECL do { } while (0)
#define SAG_CLK_RESET do { } while (0)
#define SAG_CLK(i) do { } while (0)
#define SAG_CLKG(i, g, Sref) do { } while (0)
#endif

namespace sag {

// ------------------------------------------------------------------------------------------------
// constants (assets/xmls/point.xml, primitive_objects.py, tasks/*.py; SURVEY Appendix A)
// ------------------------------------------------------------------------------------------------
constexpr double kPi = 3.14159265358979323846;
constexpr double kTwoPi = 2.0 * kPi;
constexpr double kGrav = 9.81;
constexpr double kPtH = 0.004;          // point.xml:3
constexpr int kPtNsub = 5;              // safe_adaptation_gym.py:17
constexpr double kPtR = 0.1;            // point.xml:18
constexpr double kPtArrowOff = 0.1;     // point.xml:19
constexpr double kPtArrowH = 0.05;      // point.xml:19
constexpr double kPtForceLim = 0.05;    // point.xml:7-8
constexpr double kPtGearX = 0.3;        // point.xml:36
constexpr double kPtGearZ = 0.3;        // point.xml:37
constexpr double kPtDampXY = 0.01;      // point.xml:15-16
constexpr double kPtDampZ = 0.005;      // point.xml:17
constexpr double kPtZ = 0.1;            // point.xml:13
constexpr double kGoalZ = 0.16;         // primitive_objects.py:140
constexpr double kGoalSize = 0.3;       // go_to_goal.py:12
constexpr double kGoalKeepout = 0.4;    // go_to_goal.py:13
constexpr double kButtonSize = 0.1;     // press_buttons.py:15
constexpr double kButtonsKeepout = 0.2; // press_buttons.py:14
constexpr int kButtonDelay = 5;         // press_buttons.py:17
constexpr double kBoxSize = 0.2;        // push_box.py:12
constexpr double kBoxDensity = 0.001;   // push_box.py:15
constexpr double kVaseDensity = 0.001;  // consts.py:21
constexpr double kLidarMax = 5.0;       // safe_adaptation_gym.py:23
constexpr int kLidarBins = 16;          // safe_adaptation_gym.py:22
constexpr double kTendonMax = kBoxSize * 3.75;  // haul_box.py:25
// MuJoCo default soft-constraint parameters [EXT]
constexpr double kSolTc = 0.02, kImpD0 = 0.9, kImpDmax = 0.95, kImpWidth = 0.001;
constexpr double kMu = 1.0;
// roll_rod.py:11-40 / dribble_ball.py:11-38 (oracle obj_mass / obj_geom carry the per-line citations)
constexpr double kBallR = 0.14, kBallDensity = kBoxDensity / 2.0, kBallSolTc = 0.018, kBallSolDr = 0.2;
constexpr double kBallRoll = 0.05, kBallSpin = 0.003;
constexpr double kRodR = 0.08, kRodHalf = 0.3, kRodDensity = kBoxDensity / 2.0, kRodRoll = 0.05;
constexpr double kPrioMu = 1.2;  // ball / rod geoms have priority 1: their sliding friction wins the mix
constexpr int kSweeps = 10;
constexpr double kPgsTol = 1e-8;
constexpr double kSleepV = 1e-8;
constexpr int kMaxObj = 32;
constexpr int kMaxCon = 16;
constexpr int kMaxGremlins = 4;           // each one adds two weld rows to the solver's row table
constexpr double kWeldSolTc = 0.02, kWeldSolDr = 1.5;  // primitive_objects.py:80-82: <weld solref=".02 1.5"/>
constexpr double kHotMargin = 0.05;     // scheduling only: clearance below which an env is planned as "hot"
constexpr double kRobotReach = 0.16;    // >= |hinge -> far arrow corner| = hypot(0.15, 0.05)

// point robot mass properties (MuJoCo uniform-density rule, density 1, point.xml:5,18-19)
constexpr double kPtMs = 4.0 / 3.0 * kPi * kPtR * kPtR * kPtR;
constexpr double kPtMa = 8.0 * kPtArrowH * kPtArrowH * kPtArrowH;
constexpr double kPtM = kPtMs + kPtMa;
constexpr double kPtMc = kPtMa * kPtArrowOff;
constexpr double kPtIo = 0.4 * kPtMs * kPtR * kPtR + kPtMa * (8.0 * kPtArrowH * kPtArrowH) / 12.0 + kPtMa * kPtArrowOff * kPtArrowOff;

enum ObjKind : int { K_NONE = 0, K_HAZARD, K_VASE, K_GREMLIN, K_PILLAR, K_GOAL, K_BUTTON, K_BOX, K_ROD, K_BALL };
enum Task : int {
  T_CATCH_GOAL = 0, T_COLLECT, T_DRIBBLE_BALL, T_GO_TO_GOAL, T_GO_TO_GOAL_DAMPING, T_GO_TO_GOAL_MOTOR, T_GO_TO_GOAL_SCARCE,
  T_HAUL_BOX, T_PRESS_BUTTONS, T_PRESS_BUTTONS_SCARCE, T_PUSH_BOX, T_PUSH_BOX_SCARCE, T_ROLL_ROD, T_UNSUPERVISED, T_COUNT
};
enum Flags : unsigned char { F_PHYS_ERROR = 1, F_RESAMPLE_FAILED = 2, F_NEEDS_RESET = 4 };

// per-task descriptor (tasks/*.py; SURVEY Appendix C, corrected: Collect inherits PressButtons.obstacles)
struct TaskSpec {
  int nh, nv, ng, np;   // hazards, vases, gremlins, pillars
  int kind;             // 0 goal, 1 buttons, 2 goal + box
  int nbuttons;
  int box_kind;
  double extent, button_rect, box_keepout, box_rect;
  double damp_xy, gear_x;
};

SAG_HD TaskSpec task_spec(int t) {
  TaskSpec s = {9, 10, 0, 1, 0, 0, 0, 2.0, 0.0, 0.0, 0.0, kPtDampXY, kPtGearX};
  switch (t) {
    case T_COLLECT: s = {6, 8, 0, 0, 1, 6, 0, 2.25, 1.5, 0.0, 0.0, kPtDampXY, kPtGearX}; break;
    case T_PRESS_BUTTONS: s = {6, 8, 0, 0, 1, 4, 0, 2.0, 1.35, 0.0, 0.0, kPtDampXY, kPtGearX}; break;
    case T_PRESS_BUTTONS_SCARCE: s = {6, 8, 0, 0, 1, 4, 0, 2.0, 1.75, 0.0, 0.0, kPtDampXY, kPtGearX}; break;
    case T_HAUL_BOX: case T_PUSH_BOX: s = {2, 3, 0, 1, 2, 0, K_BOX, 1.75, 0.0, 0.5, 0.0, kPtDampXY, kPtGearX}; break;
    case T_PUSH_BOX_SCARCE: s = {2, 3, 0, 1, 2, 0, K_BOX, 1.75, 0.0, 0.55, 2.25, kPtDampXY, kPtGearX}; break;
    case T_ROLL_ROD: s = {2, 3, 0, 1, 2, 0, K_ROD, 1.75, 0.0, 0.7, 0.0, kPtDampXY, kPtGearX}; break;
    case T_DRIBBLE_BALL: s = {2, 3, 0, 1, 2, 0, K_BALL, 1.75, 0.0, 0.2, 0.0, kPtDampXY, kPtGearX}; break;
    case T_UNSUPERVISED: s = {5, 6, 0, 1, 0, 0, 0, 2.0, 0.0, 0.0, 0.0, kPtDampXY, kPtGearX}; break;
    case T_GO_TO_GOAL_DAMPING: s.damp_xy = kPtDampXY * 0.1; break;   // go_to_goal_damping.py:12-17
    case T_GO_TO_GOAL_MOTOR: s.gear_x = kPtGearX * 10.0; break;      // go_to_goal_motor.py:12-16
    default: break;
  }
  return s;
}

// User-defined tasks (sag_define_task): ids T_COUNT, T_COUNT + 1, ... of a handle.  An entry is the base task's
// descriptor with the user's obstacle counts (nh, nv, ng, np) and placement extents (x_min, y_min, x_max, y_max); `base`
// is the registry id whose reward, goal / button / box logic and dynamics variant the task keeps.  The table lives in
// the handle's slab (custom_table); only the *C instantiations read it.
constexpr int kMaxCustomTasks = 16;
struct CustomTask {
  TaskSpec sp;
  int base;
  double ext[4];
};
struct CustomTable {
  int count;
  CustomTask t[kMaxCustomTasks];
};

// task descriptor of an environment of this handle: the task's table entry + the handle's gremlin count
struct Dev;
SAG_HD TaskSpec spec_for(const Dev& D, int t, bool gremlins);

// slot layout = placement order without the robot (world.py:83-90): hazards, vases, gremlins, pillars, task objects
struct Slots {
  int h0, v0, g0, p0, t0, n;  // first slot of each kind, total
  int goal, box, btn0, nbtn;
};
SAG_HD Slots make_slots(const TaskSpec& s) {
  Slots L;
  L.h0 = 0; L.v0 = s.nh; L.g0 = L.v0 + s.nv; L.p0 = L.g0 + s.ng; L.t0 = L.p0 + s.np;
  L.goal = L.box = L.btn0 = -1; L.nbtn = 0;
  if (s.kind == 0) { L.goal = L.t0; L.n = L.t0 + 1; }
  else if (s.kind == 1) { L.btn0 = L.t0; L.nbtn = s.nbuttons; L.n = L.t0 + s.nbuttons; }
  else { L.goal = L.t0; L.box = L.t0 + 1; L.n = L.t0 + 2; }
  return L;
}
SAG_HD int slot_kind(const TaskSpec& s, const Slots& L, int k) {
  if (k < L.v0) return K_HAZARD;
  if (k < L.g0) return K_VASE;
  if (k < L.p0) return K_GREMLIN;
  if (k < L.t0) return K_PILLAR;
  if (k == L.goal) return K_GOAL;
  if (k == L.box) return s.box_kind;
  return K_BUTTON;
}

// ------------------------------------------------------------------------------------------------
// device-resident state (SoA, env-minor) + config.  Passed by value to every kernel.
// ------------------------------------------------------------------------------------------------
struct Dev {
  int n, stride, nslots, robot;
  // World.DEFAULT (world.py:17-34), keepouts already max'ed with sizes (world.py:60-66)
  double action_noise, placements_margin, robot_keepout;
  double hazards_size, vases_size, pillars_size, gremlins_size;
  double k_hazard, k_vase, k_gremlin, k_pillar;
  double max_bound, ctrl_range_scale;
  int random_bound;
  // Philox key.  Kernels read it from the slab (*key): sag_seed may change it after kernels have been recorded in a CUDA
  // graph, and a replayed kernel sees only device memory, not a new by-value argument.  `seed` is the by-value copy
  // that a host build of this code reads (the host emulation of the tests, which has no slab on a device).
  unsigned long long seed;
  unsigned long long* key;
  unsigned gid_base;
  int max_layout_draws, max_episode_steps;
  int num_gremlins;        // Task.obstacles[2] of a user-defined task (task.py:70); 0 in every shipped task
  double gremlins_travel;  // world.py:28
  // robot
  double *rx, *ry, *ryaw, *rvx, *rvy, *rw;
  double *ctrl0, *ctrl1;
  double *cscale0, *cscale1, *bound;  // per Task instance: ctrl-range scale per actuator, constraint bound (world.py:72-78)
  double* rext;  // car extras [6][stride]: wheel rates (2), castor ball-joint quaternion (4)
  // gremlins [2 + 3 * kMaxGremlins][stride]: mocap position seen by the last kinematics pass (2), spawn x, y, yaw per gremlin
  double* grem;
  // objects [slot][env]
  double *ox, *oy, *oyaw, *ovx, *ovy, *ow;
  // task / bookkeeping
  int* task;
  double *last0, *last1;
  int *gbtn, *bstate, *btimer, *amask;
  double *cgcur, *cgnext, *cgox, *cgoy;
  int* cgtimer;
  int* movmask;  // bit s: movable object s has a non-zero velocity (derived state, rebuilt by env_observe)
  // work list of the environments with a contact or a moving body in the current step (k_step_free -> k_step_coop)
  int* worklist;
  int* counts;             // [2][8]: two counter sets used by alternate steps; counts[8 * (*epoch & 1)] is this step's
  unsigned* epoch;         // [0] step epoch, advanced by the contact kernel's last CTA; [1] CTAs of that kernel that have
                           // finished (sag_kernels.cu: k_step_free, k_step_coop)
  unsigned long long* dbg; // [16] section clocks of SAG_TIMING builds
  int* errflags;           // [4] sticky error words the host can read without a synchronisation (mapped pinned memory):
                           // [0] a layout / goal could not be sampled (ResamplingError), [1] task id out of range,
                           // [2] a bad sag_copy_envs pair
  double *time, *clear;
  unsigned *ctr, *episode;
  int* nstep;
  double *epret, *epcost;
  unsigned char* flags;
};

// the user-defined task table of a handle: at the end of the slab, its address in the scheduling block at
// D.counts + kCustomTablePtr (sag_layout.h: slab_bind); read by the *C instantiations only
constexpr int kCustomTablePtr = 56;
SAG_HD const CustomTable& custom_table(const Dev& D) {
  return **reinterpret_cast<const CustomTable* const*>(D.counts + kCustomTablePtr);
}

// gremlins = RB::kGremlins: in the default instantiations the count is the compile-time constant 0 of the task table
SAG_HD TaskSpec spec_for(const Dev& D, int t, bool gremlins) { TaskSpec s = task_spec(t); if (gremlins) s.ng = D.num_gremlins; return s; }
// custom = RB::kCustom: the *C instantiations look ids >= T_COUNT up in the handle's table (whose gremlin count is the
// handle's); the others never see such an id and compile to the registry lookup alone
SAG_HD TaskSpec spec_for(const Dev& D, int t, bool gremlins, bool custom) {
  if (custom && t >= T_COUNT) return custom_table(D).t[t - T_COUNT].sp;
  return spec_for(D, t, gremlins);
}
// the registry id whose logic an environment with task id t runs (Ctx::task)
SAG_HD int logic_task(const Dev& D, int t, bool custom) { return custom && t >= T_COUNT ? custom_table(D).t[t - T_COUNT].base : t; }
// the ids a handle accepts: the registry's, and with custom (RB::kCustom) the defined ones
SAG_HD int num_task_ids(const Dev& D, bool custom) { return custom ? T_COUNT + custom_table(D).count : T_COUNT; }
SAG_HD size_t oidx(const Dev& D, int slot, int e) { return (size_t)slot * D.stride + e; }

// View of ONE environment's object arrays: field[slot * stride].  Global memory: pointers offset by the environment
// index, stride = D.stride (coalesced across the environments of a warp).  The cooperative kernel stages the arrays in
// the warp's shared-memory working set for the duration of a step (stride 1).
struct ObjView { double *x, *y, *yaw, *vx, *vy, *w; int stride; };
SAG_HD ObjView global_objects(const Dev& D, int e) {
  ObjView O = {D.ox + e, D.oy + e, D.oyaw + e, D.ovx + e, D.ovy + e, D.ow + e, D.stride};
  return O;
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10, counter = (ctr, episode, global env id, stream), key = seed
// ------------------------------------------------------------------------------------------------
SAG_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// The key an Rng draws with.  In kernels it is a pointer, loaded at every draw: holding the 64-bit key itself through a
// step added spills to k_step_free, while the pointer (into the slab, or to a caller's local copy) is an argument the
// compiler can reload.  A host build holds the key by value (Dev::seed).
#if defined(__CUDA_ARCH__)
typedef const unsigned long long* RngKey;
SAG_HD RngKey rng_key(const Dev& D) { return D.key; }
SAG_HD RngKey rng_key_of(const unsigned long long& k) { return &k; }
SAG_HD uint64_t rng_key_value(RngKey k) { return *k; }
#else
typedef unsigned long long RngKey;
SAG_HD RngKey rng_key(const Dev& D) { return D.seed; }
SAG_HD RngKey rng_key_of(const unsigned long long& k) { return k; }
SAG_HD uint64_t rng_key_value(RngKey k) { return k; }
#endif
struct Rng {
  RngKey seed;
  uint32_t gid, episode;
  SAG_HD void pair(uint32_t stream, uint32_t ctr, double& u1, double& u2) const {
    uint32_t r[4];
    const uint64_t key = rng_key_value(seed);
    philox4x32_10(ctr, episode, gid, stream, (uint32_t)key, (uint32_t)(key >> 32), r);
    u1 = ((double)(r[0] >> 5) * 67108864.0 + (double)(r[1] >> 6)) * (1.0 / 9007199254740992.0);
    u2 = ((double)(r[2] >> 5) * 67108864.0 + (double)(r[3] >> 6)) * (1.0 / 9007199254740992.0);
  }
};

// ------------------------------------------------------------------------------------------------
// planar collision primitives (MuJoCo contact convention [EXT]: signed dist, normal geom1->geom2,
// point at the midpoint; listed when dist <= 0)
// ------------------------------------------------------------------------------------------------
struct Geom { int is_box; double cx, cy, c, s, hx, hy, r; };
struct Hit { double nx, ny, px, py, dist; };

SAG_HD int hit_circle_circle(const Geom& A, const Geom& B, Hit* o) {
  double dx = B.cx - A.cx, dy = B.cy - A.cy;
  double len = sqrt(dx * dx + dy * dy);
  double dist = len - A.r - B.r;
  if (dist > 0.0) return 0;
  double nx = 1.0, ny = 0.0;
  if (len > 1e-14) { nx = dx / len; ny = dy / len; }
  o->nx = nx; o->ny = ny;
  o->px = A.cx + nx * (A.r + 0.5 * dist);
  o->py = A.cy + ny * (A.r + 0.5 * dist);
  o->dist = dist;
  return 1;
}

SAG_HD int hit_circle_box(const Geom& Cc, const Geom& B, bool circle_is_a, Hit* o) {
  double rx = Cc.cx - B.cx, ry = Cc.cy - B.cy;
  double lx = rx * B.c + ry * B.s, ly = -rx * B.s + ry * B.c;
  double qx = lx < -B.hx ? -B.hx : (lx > B.hx ? B.hx : lx);
  double qy = ly < -B.hy ? -B.hy : (ly > B.hy ? B.hy : ly);
  double nlx, nly, dist;
  if (qx == lx && qy == ly) {
    double penx = B.hx - fabs(lx), peny = B.hy - fabs(ly);
    if (penx <= peny) { nlx = lx >= 0.0 ? 1.0 : -1.0; nly = 0.0; qx = nlx * B.hx; dist = -penx - Cc.r; }
    else { nlx = 0.0; nly = ly >= 0.0 ? 1.0 : -1.0; qy = nly * B.hy; dist = -peny - Cc.r; }
  } else {
    double ex = lx - qx, ey = ly - qy;
    double len = sqrt(ex * ex + ey * ey);
    dist = len - Cc.r;
    if (dist > 0.0) return 0;
    nlx = ex / len; nly = ey / len;
  }
  double nwx = nlx * B.c - nly * B.s, nwy = nlx * B.s + nly * B.c;
  double pbx = B.cx + qx * B.c - qy * B.s, pby = B.cy + qx * B.s + qy * B.c;
  double pcx = Cc.cx - nwx * Cc.r, pcy = Cc.cy - nwy * Cc.r;
  o->px = 0.5 * (pbx + pcx); o->py = 0.5 * (pby + pcy); o->dist = dist;
  if (circle_is_a) { o->nx = -nwx; o->ny = -nwy; } else { o->nx = nwx; o->ny = nwy; }
  return 1;
}

SAG_HD int hit_box_box_body(const Geom& A, const Geom& B, Hit* o);
// out of line for the scalar paths (several call sites); the cooperative kernel's single narrow-phase site inlines the body
SAG_HD_NOINLINE int hit_box_box(const Geom& A, const Geom& B, Hit* o) { return hit_box_box_body(A, B, o); }
SAG_HD int hit_box_box_body(const Geom& A, const Geom& B, Hit* o) {
  double dx = B.cx - A.cx, dy = B.cy - A.cy;
  double best = -1e300, bsign = 1.0, bux = 0.0, buy = 0.0;
  int bi = -1;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    double ux = k == 0 ? A.c : (k == 1 ? -A.s : (k == 2 ? B.c : -B.s));
    double uy = k == 0 ? A.s : (k == 1 ? A.c : (k == 2 ? B.s : B.c));
    double dp = dx * ux + dy * uy;
    double ra = A.hx * fabs(A.c * ux + A.s * uy) + A.hy * fabs(-A.s * ux + A.c * uy);
    double rb = B.hx * fabs(B.c * ux + B.s * uy) + B.hy * fabs(-B.s * ux + B.c * uy);
    double sep = fabs(dp) - (ra + rb);
    if (sep > 0.0) return 0;
    if (sep > best) { best = sep; bi = k; bsign = dp >= 0.0 ? 1.0 : -1.0; bux = ux; buy = uy; }
  }
  bool ref_is_a = bi < 2;
  const Geom& R = ref_is_a ? A : B;
  const Geom& I = ref_is_a ? B : A;
  double Nx = ref_is_a ? bsign * bux : -bsign * bux, Ny = ref_is_a ? bsign * buy : -bsign * buy;
  int ref_axis = bi & 1;
  double hn = ref_axis == 0 ? R.hx : R.hy, ht = ref_axis == 0 ? R.hy : R.hx;
  double Tx = -Ny, Ty = Nx;
  double nlx = Nx * I.c + Ny * I.s, nly = -Nx * I.s + Ny * I.c;
  double v1x, v1y, v2x, v2y;
  if (fabs(nlx) >= fabs(nly)) { double sx = nlx > 0.0 ? -1.0 : 1.0; v1x = sx * I.hx; v1y = -I.hy; v2x = sx * I.hx; v2y = I.hy; }
  else { double sy = nly > 0.0 ? -1.0 : 1.0; v1x = -I.hx; v1y = sy * I.hy; v2x = I.hx; v2y = sy * I.hy; }
  double w1x = I.cx + v1x * I.c - v1y * I.s - R.cx, w1y = I.cy + v1x * I.s + v1y * I.c - R.cy;
  double w2x = I.cx + v2x * I.c - v2y * I.s - R.cx, w2y = I.cy + v2x * I.s + v2y * I.c - R.cy;
  double n1 = w1x * Nx + w1y * Ny, t1 = w1x * Tx + w1y * Ty;
  double n2 = w2x * Nx + w2y * Ny, t2 = w2x * Tx + w2y * Ty;
  double lo = 0.0, hi = 1.0, dt = t2 - t1;
  if (t1 > ht && t2 > ht) return 0;
  if (t1 < -ht && t2 < -ht) return 0;
  if (dt != 0.0) {
    if (t1 > ht) { double s = (ht - t1) / dt; if (s > lo) lo = s; }
    if (t2 > ht) { double s = (ht - t1) / dt; if (s < hi) hi = s; }
    if (t1 < -ht) { double s = (-ht - t1) / dt; if (s > lo) lo = s; }
    if (t2 < -ht) { double s = (-ht - t1) / dt; if (s < hi) hi = s; }
  }
  if (lo > hi) return 0;
  int n = 0;
  int npts = (hi - lo) > 1e-12 ? 2 : 1;
  for (int k = 0; k < npts; ++k) {
    double s = k == 0 ? lo : hi;
    double pn = n1 + s * (n2 - n1), pt = t1 + s * dt;
    double sep = pn - hn;
    if (sep > 0.0) continue;
    Hit& c = o[n];
    c.px = R.cx + pn * Nx + pt * Tx - 0.5 * sep * Nx;
    c.py = R.cy + pn * Ny + pt * Ty - 0.5 * sep * Ny;
    if (ref_is_a) { c.nx = Nx; c.ny = Ny; } else { c.nx = -Nx; c.ny = -Ny; }
    c.dist = sep;
    ++n;
  }
  return n;
}

SAG_HD int collide(const Geom& A, const Geom& B, Hit* o) {
  if (!A.is_box && !B.is_box) return hit_circle_circle(A, B, o);
  if (!A.is_box) return hit_circle_box(A, B, true, o);
  if (!B.is_box) return hit_circle_box(B, A, false, o);
  return hit_box_box(A, B, o);
}
SAG_HD int collide_inl(const Geom& A, const Geom& B, Hit* o) {
  if (!A.is_box && !B.is_box) return hit_circle_circle(A, B, o);
  if (!A.is_box) return hit_circle_box(A, B, true, o);
  if (!B.is_box) return hit_circle_box(B, A, false, o);
  return hit_box_box_body(A, B, o);
}

// Overlap predicates: the first stage of the hit_* routines above with the same arithmetic, so "no overlap" here
// implies that the full narrow phase would list no contact (the converse may fail for box-box: conservative).
SAG_HD bool overlap_circle_circle(const Geom& A, const Geom& B) {
  double dx = B.cx - A.cx, dy = B.cy - A.cy;
  double len = sqrt(dx * dx + dy * dy);
  double dist = len - A.r - B.r;
  return !(dist > 0.0);
}
SAG_HD bool overlap_circle_box(const Geom& Cc, const Geom& B) {
  double rx = Cc.cx - B.cx, ry = Cc.cy - B.cy;
  double lx = rx * B.c + ry * B.s, ly = -rx * B.s + ry * B.c;
  double qx = lx < -B.hx ? -B.hx : (lx > B.hx ? B.hx : lx);
  double qy = ly < -B.hy ? -B.hy : (ly > B.hy ? B.hy : ly);
  if (qx == lx && qy == ly) return true;
  double ex = lx - qx, ey = ly - qy;
  double len = sqrt(ex * ex + ey * ey);
  double dist = len - Cc.r;
  return !(dist > 0.0);
}
SAG_HD bool overlap_box_box(const Geom& A, const Geom& B) {
  double dx = B.cx - A.cx, dy = B.cy - A.cy;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    double ux = k == 0 ? A.c : (k == 1 ? -A.s : (k == 2 ? B.c : -B.s));
    double uy = k == 0 ? A.s : (k == 1 ? A.c : (k == 2 ? B.s : B.c));
    double dp = dx * ux + dy * uy;
    double ra = A.hx * fabs(A.c * ux + A.s * uy) + A.hy * fabs(-A.s * ux + A.c * uy);
    double rb = B.hx * fabs(B.c * ux + B.s * uy) + B.hy * fabs(-B.s * ux + B.c * uy);
    double sep = fabs(dp) - (ra + rb);
    if (sep > 0.0) return false;
  }
  return true;
}
SAG_HD bool overlap(const Geom& A, const Geom& B) {
  if (!A.is_box && !B.is_box) return overlap_circle_circle(A, B);
  if (!A.is_box) return overlap_circle_box(A, B);
  if (!B.is_box) return overlap_circle_box(B, A);
  return overlap_box_box(A, B);
}

SAG_HD bool kind_collidable(int k) { return k == K_VASE || k == K_GREMLIN || k == K_PILLAR || k == K_BUTTON || k >= K_BOX; }
SAG_HD bool kind_movable(int k) { return k == K_VASE || k == K_GREMLIN || k >= K_BOX; }
SAG_HD int kind_nparts(int k) { return k == K_BOX ? 5 : (kind_collidable(k) ? 1 : 0); }
// bounding radius about the body centre (for the broad phase); select chain, no jump table
SAG_HD double kind_bound(const Dev& D, int k) {
  return k == K_VASE ? D.vases_size * 1.4142135623730951 + 1e-9
       : k == K_PILLAR ? D.pillars_size
       : k == K_BUTTON ? kButtonSize
       : k == K_BOX ? kBoxSize * 1.5 * 1.4142135623730951 + 1e-9
       : k == K_BALL ? kBallR
       : k == K_ROD ? 0.31048349392520047 + 1e-9  // sqrt(kRodR^2 + kRodHalf^2)
       : k == K_GREMLIN ? D.gremlins_size * 1.4142135623730951 + 1e-9 : 0.0;
}
// Planar inertia and floor interaction of a movable body (oracle obj_mass): m translational mass (ball: rolling
// effective mass 7/5 m), iz about the vertical, flin / ftor bounds of the floor friction force (disc) and torque, bfl
// damping rate of the floor rows.  The rod is anisotropic: body x rolls (3/2 m, resistance roll / r * N), body y slides
// (m, mu N), each with its own row.
struct BodyPar { double m, iz, flin, ftor, bfl, mx, my, fx, fy; };
SAG_HD BodyPar kind_body(const Dev& D, int k) {
  BodyPar b;
  b.mx = b.my = b.fx = b.fy = 0.0;
  b.bfl = 2.0 / (kImpDmax * kSolTc);
  if (k == K_BOX) {
    const double d = kBoxSize, wd = kBoxSize / 2;
    const double m0 = 8.0 * d * d * d * kBoxDensity, mc = 8.0 * wd * wd * d * kBoxDensity;
    b.m = m0 + 4.0 * mc;
    b.iz = m0 * (2.0 / 3.0) * d * d + 4.0 * (mc * (2.0 / 3.0) * wd * wd + mc * (2.0 * d * d));
    b.flin = kMu * b.m * kGrav;
    b.ftor = b.flin * (1.5 * d);
  } else if (k == K_BALL) {
    const double m0 = (4.0 / 3.0) * kPi * kBallR * kBallR * kBallR * kBallDensity;
    b.m = 1.4 * m0;
    b.iz = 0.4 * m0 * kBallR * kBallR;
    b.flin = kBallRoll * m0 * kGrav / kBallR;
    b.ftor = kBallSpin * m0 * kGrav;
    b.bfl = 2.0 / (kImpDmax * kBallSolTc);
  } else if (k == K_ROD) {
    const double m0 = kPi * kRodR * kRodR * (2.0 * kRodHalf) * kRodDensity;
    b.m = m0; b.mx = 1.5 * m0; b.my = m0;
    b.iz = m0 * (3.0 * kRodR * kRodR + 4.0 * kRodHalf * kRodHalf) / 12.0;
    b.fx = kRodRoll * m0 * kGrav / kRodR; b.fy = kPrioMu * m0 * kGrav;
    b.flin = b.fy;
    b.ftor = kPrioMu * m0 * kGrav * kRodHalf;
  } else {
    double s = k == K_VASE ? D.vases_size : D.gremlins_size;
    b.m = 8.0 * s * s * s * kVaseDensity;
    b.iz = b.m * (2.0 / 3.0) * s * s;
    b.flin = kMu * b.m * kGrav;
    b.ftor = b.flin * (s * sqrt(2.0));
  }
  return b;
}

SAG_HD void obj_geom(const Dev& D, int kind, int part, double x, double y, double c, double s, Geom& g) {
  g.c = c; g.s = s; g.cx = x; g.cy = y; g.r = 0.0; g.hx = g.hy = 0.0; g.is_box = 0;
  if (kind == K_VASE) { g.is_box = 1; g.hx = g.hy = D.vases_size; }
  else if (kind == K_PILLAR) { g.r = D.pillars_size; }
  else if (kind == K_BUTTON) { g.r = kButtonSize; }
  else if (kind == K_GREMLIN) { g.is_box = 1; g.hx = g.hy = D.gremlins_size; }
  else if (kind == K_BOX) {
    g.is_box = 1;
    if (part == 0) { g.hx = g.hy = kBoxSize; }
    else {
      double sx = (part == 1 || part == 3) ? 1.0 : -1.0, sy = (part <= 2) ? 1.0 : -1.0;
      double ox = sx * kBoxSize, oy = sy * kBoxSize;
      g.hx = g.hy = kBoxSize / 2;
      g.cx = x + ox * c - oy * s; g.cy = y + ox * s + oy * c;
    }
  }
  else if (kind == K_BALL) { g.r = kBallR; }
  else if (kind == K_ROD) { g.is_box = 1; g.hx = kRodR; g.hy = kRodHalf; }
}

// ------------------------------------------------------------------------------------------------
// point robot (point.xml): generalised coordinates (x, y, yaw) in the world frame.
// M = [[a,0,p],[0,a,q],[p,q,I]] with p = -mc sin(yaw), q = mc cos(yaw).  Both slide joints share one
// damping value, so p^2 + q^2 = (mc)^2 and the Schur complement I - (mc)^2 / a is a constant of the
// model: the 3x3 solve needs no division per substep.
// ------------------------------------------------------------------------------------------------
struct PtConst { double ia0, is0, iah, ish; };  // 1/a and 1/schur for M (forward dynamics) and M + hD (Euler)

SAG_HD PtConst pt_const(double damp_xy, double h) {
  PtConst K;
  K.ia0 = 1.0 / (kPtM + 0.0 * damp_xy);
  K.is0 = 1.0 / ((kPtIo + 0.0 * kPtDampZ) - kPtMc * kPtMc * K.ia0);
  K.iah = 1.0 / (kPtM + h * damp_xy);
  K.ish = 1.0 / ((kPtIo + h * kPtDampZ) - kPtMc * kPtMc * K.iah);
  return K;
}
SAG_HD void pt_solve(double p, double q, double ia, double is, const double* f, double* out) {
  double al = (f[2] - (p * f[0] + q * f[1]) * ia) * is;
  out[0] = (f[0] - p * al) * ia;
  out[1] = (f[1] - q * al) * ia;
  out[2] = al;
}
SAG_HD double clampd(double x, double lo, double hi) { return x < lo ? lo : (x > hi ? hi : x); }

// ---- car (car.xml): reduced planar differential-drive model, DESIGN.md 4.  Mirrors oracle car_params().
constexpr double kCarH = 0.008;          // car.xml:3
constexpr int kCarNsub = 10;             // safe_adaptation_gym.py:18
constexpr double kCarForceLim = 0.02;    // car.xml:7
constexpr double kCarWheelR = 0.05;      // car.xml:5
constexpr double kCarWheelDamp = 0.001;  // car.xml:6
constexpr double kCarArmature = 0.00025; // car.xml:22,26
constexpr double kCarDensity = 5.0;      // car.xml:5
constexpr int kCarNGeom = 8;
struct CarGeomTab { double v[kCarNGeom][5]; double hz[5]; };
// body-frame x, y, half-x, half-y | radius (car.xml:16-31; wheels are x-axis cylinders -> footprints); box half heights
constexpr CarGeomTab kCarGeomC = {{{0.0, 0.0, 0.1, 0.1, 0.0}, {0.0, 0.15, 0.1, 0.01, 0.0}, {0.0, 0.125, 0.01, 0.025, 0.0},
                                  {0.0, -0.165, 0.05, 0.01, 0.0}, {0.0, -0.13, 0.05, 0.03, 0.0}, {-0.13, 0.1, 0.025, 0.05, 0.0},
                                  {0.13, 0.1, 0.025, 0.05, 0.0}, {0.0, -0.1, 0.0, 0.0, 0.05}},
                                 {0.05, 0.05, 0.03, 0.05, 0.01}};
SAG_DEV_CONST constexpr CarGeomTab kCarGeom = kCarGeomC;  // run-time indexed copy (device memory under nvcc)
struct CarModel { double M, mcx, mcy, Io, Iw, nwheel, nrear; };
constexpr CarModel car_model() {
  CarModel c = {0, 0, 0, 0, 0, 0, 0};
  double M = 0.0, mx = 0.0, my = 0.0, Io = 0.0;
  for (int g = 0; g < 5; ++g) {
    double hx = kCarGeomC.v[g][2], hy = kCarGeomC.v[g][3], hz = kCarGeomC.hz[g];
    double m = 8.0 * hx * hy * hz * kCarDensity;
    double x = kCarGeomC.v[g][0], y = kCarGeomC.v[g][1];
    M += m; mx += m * x; my += m * y;
    Io += m * (4.0 * hx * hx + 4.0 * hy * hy) / 12.0 + m * (x * x + y * y);
  }
  double mw = kPi * kCarWheelR * kCarWheelR * 0.05 * kCarDensity;
  for (int g = 5; g < 7; ++g) {
    double x = kCarGeomC.v[g][0], y = kCarGeomC.v[g][1];
    M += mw; mx += mw * x; my += mw * y;
    Io += mw * (3.0 * kCarWheelR * kCarWheelR + 0.05 * 0.05) / 12.0 + mw * (x * x + y * y);
  }
  double mb = 4.0 / 3.0 * kPi * kCarWheelR * kCarWheelR * kCarWheelR * kCarDensity;
  {
    double x = kCarGeomC.v[7][0], y = kCarGeomC.v[7][1];
    M += mb; mx += mb * x; my += mb * y;
    Io += 0.4 * mb * kCarWheelR * kCarWheelR + mb * (x * x + y * y);
  }
  c.M = M; c.mcx = mx; c.mcy = my; c.Io = Io;
  c.Iw = 0.5 * mw * kCarWheelR * kCarWheelR + kCarArmature;
  double yc = my / M;
  c.nrear = M * kGrav * (0.1 - yc) / 0.2;
  c.nwheel = (M * kGrav - c.nrear) / 2.0;
  return c;
}
constexpr CarModel kCar = car_model();

struct PointRobot {
  static constexpr int kKind = 0, kNGeom = 2, kNsub = kPtNsub, kObsDim = 60;
  static constexpr bool kGremlins = false;  // the gremlin code paths exist only in the *G instantiations (below)
  static constexpr bool kCustom = false;    // the user-defined task table is read only by the *C instantiations (below)
  static constexpr double kH = kPtH, kReach = kRobotReach;
  double q[3], v[3];
  double ctrl[2];
  double damp_xy, gear_x;
  SAG_HD void pq(double sn, double cs, double& p, double& qq) const { p = -kPtMc * sn; qq = kPtMc * cs; }
  SAG_HD PtConst consts(double h) const { return pt_const(damp_xy, h); }
  // qfrc_smooth = actuation + passive - bias  (SURVEY Appendix A.1 / B.2-3 [EXT])
  SAG_HD void smooth(double sn, double cs, double* f) const {
    double w = v[2];
    double fx = clampd(ctrl[0], -kPtForceLim, kPtForceLim);
    double fz = clampd(ctrl[1] - kPtGearZ * w, -kPtForceLim, kPtForceLim);
    f[0] = gear_x * fx * cs - damp_xy * v[0] + kPtMc * w * w * cs;
    f[1] = gear_x * fx * sn - damp_xy * v[1] + kPtMc * w * w * sn;
    f[2] = kPtGearZ * fz - kPtDampZ * w;
  }
  SAG_HD void geom(int part, double sn, double cs, Geom& g) const {
    g.c = cs; g.s = sn;
    if (part == 0) { g.is_box = 0; g.cx = q[0]; g.cy = q[1]; g.r = kPtR; g.hx = g.hy = 0.0; }
    else { g.is_box = 1; g.cx = q[0] + kPtArrowOff * cs; g.cy = q[1] + kPtArrowOff * sn; g.hx = g.hy = kPtArrowH; g.r = 0.0; }
  }
  SAG_HD void com_offset(double& cx, double& cy) const { cx = kPtMc / kPtM; cy = 0.0; }
  // conservative bound on how far any robot geom can travel during one env step (DESIGN.md 5)
  SAG_HD double travel_bound() const {
    const double tstep = kPtNsub * kPtH;
    double speed = sqrt(v[0] * v[0] + v[1] * v[1]), wabs = fabs(v[2]);
    double alpha_max = 750.0 + 200.0 * wabs, wmax = wabs + alpha_max * tstep;
    double a_bound = 2.0 * (gear_x * kPtForceLim + damp_xy * speed) / kPtM + (kPtMc / kPtM) * (alpha_max + wmax * wmax);
    return tstep * speed + tstep * tstep * a_bound + 1e-3;
  }
};

struct CarRobot {
  static constexpr int kKind = 1, kNGeom = kCarNGeom, kNsub = kCarNsub, kObsDim = 72;
  static constexpr bool kGremlins = false;
  static constexpr bool kCustom = false;
  static constexpr double kH = kCarH, kReach = 0.22;  // >= farthest footprint corner (wheel: hypot(0.155, 0.15))
  double q[3], v[3];
  double ctrl[2];
  double damp_xy, gear_x;  // unused (kept so that shared code can copy them)
  double wheel[2];         // wheel spin rates
  double cq[4];            // castor ball-joint quaternion
  SAG_HD void pq(double sn, double cs, double& p, double& qq) const { p = -(kCar.mcx * sn + kCar.mcy * cs); qq = kCar.mcx * cs - kCar.mcy * sn; }
  SAG_HD PtConst consts(double) const {  // free joint: no damping, so M + hD = M
    PtConst K;
    K.ia0 = 1.0 / kCar.M;
    K.is0 = 1.0 / (kCar.Io - (kCar.mcx * kCar.mcx + kCar.mcy * kCar.mcy) * K.ia0);
    K.iah = K.ia0; K.ish = K.is0;
    return K;
  }
  SAG_HD void smooth(double sn, double cs, double* f) const {  // centripetal bias of the COM offset only
    double w = v[2];
    f[0] = w * w * (kCar.mcx * cs - kCar.mcy * sn);
    f[1] = w * w * (kCar.mcx * sn + kCar.mcy * cs);
    f[2] = 0.0;
  }
  SAG_HD double wheel_smooth(int i) const {  // motor (gear 1, forcerange +-0.02) - joint damping
    return clampd(ctrl[i], -kCarForceLim, kCarForceLim) - kCarWheelDamp * wheel[i];
  }
  SAG_HD void geom(int part, double sn, double cs, Geom& g) const {
    const double* G = kCarGeom.v[part];
    g.c = cs; g.s = sn;
    g.cx = q[0] + G[0] * cs - G[1] * sn; g.cy = q[1] + G[0] * sn + G[1] * cs;
    g.is_box = G[4] == 0.0; g.hx = G[2]; g.hy = G[3]; g.r = G[4];
  }
  SAG_HD void com_offset(double& cx, double& cy) const { cx = kCar.mcx / kCar.M; cy = kCar.mcy / kCar.M; }
  SAG_HD double travel_bound() const {  // traction-limited: |a| <= 2 mu g covers drive + contact pushes
    const double tstep = kCarNsub * kCarH;
    double speed = sqrt(v[0] * v[0] + v[1] * v[1]);
    return tstep * speed + tstep * tstep * (2.0 * kMu * kGrav) + 1e-3;
  }
  // castor ball (car.xml:29-32), ideal rolling: joint angular velocity in the child frame (mjSENS_BALLANGVEL [EXT])
  SAG_HD void castor_angvel(double sn, double cs, double* wc) const {
    double bx = 0.0, by = -0.1;
    double rx = bx * cs - by * sn, ry = bx * sn + by * cs;
    double vx = v[0] - v[2] * ry, vy = v[1] + v[2] * rx;
    double wx = -vy / kCarWheelR, wy = vx / kCarWheelR;
    double px = wx * cs + wy * sn, py = -wx * sn + wy * cs, pz = 0.0;
    double w = cq[0], x = -cq[1], y = -cq[2], z = -cq[3];
    double tx = 2.0 * (y * pz - z * py), ty = 2.0 * (z * px - x * pz), tz = 2.0 * (x * py - y * px);
    wc[0] = px + w * tx + (y * tz - z * ty);
    wc[1] = py + w * ty + (z * tx - x * tz);
    wc[2] = pz + w * tz + (x * ty - y * tx);
  }
};

// Environments with gremlins (Task.obstacles[2] > 0: no task of the reference's registry) run the same code instantiated
// with kGremlins = true; the default instantiations carry none of the weld / mocap code.
struct PointRobotG : PointRobot { static constexpr bool kGremlins = true; };
struct CarRobotG : CarRobot { static constexpr bool kGremlins = true; };
// Handles with user-defined tasks (sag_define_task) run the same code instantiated with kCustom = true: the task
// descriptor of an id >= T_COUNT comes from the handle's table (spec_for), and free placements take the task's
// rectangle.  The default instantiations carry none of it.
struct PointRobotC : PointRobot { static constexpr bool kCustom = true; };
struct CarRobotC : CarRobot { static constexpr bool kCustom = true; };
struct PointRobotGC : PointRobotG { static constexpr bool kCustom = true; };
struct CarRobotGC : CarRobotG { static constexpr bool kCustom = true; };

SAG_HD bool bad_val(double x) { return !(fabs(x) <= 1e10); }

SAG_HD double impedance(double r) {
  double x = fabs(r) / kImpWidth;
  if (x > 1.0) x = 1.0;
  double y = x < 0.5 ? 2.0 * x * x : 1.0 - 2.0 * (1.0 - x) * (1.0 - x);
  return kImpD0 + y * (kImpDmax - kImpD0);
}

// ------------------------------------------------------------------------------------------------
// contact pass (slow path; only taken by environments with something within reach or in motion):
// collision detection in the oracle's canonical order, soft-constraint rows, projected Gauss-Seidel,
// optional integration of the movable bodies.  Work is proportional to the objects actually involved.
// ------------------------------------------------------------------------------------------------
struct Con { int ba, bb; double nx, ny, px, py, dist; };  // ba/bb: -1 static, 0 robot, 1 + slot movable object
struct Row {  // one contact (normal k=0, tangent k=1), the tendon limit (k=0 only) or one car wheel (longitudinal, lateral)
  int ba, bb;                 // indices into Scratch::acc (-1 static, 0 robot, 1 + compact body id, NB + 1 + wheel)
  int type, nk;               // type 0 contact / tendon, 1 equality (weld: bilateral), 2 wheel-floor friction pair (disc bound);
                              // nk scalar rows in this entry: 2, or 1 (tendon, weld yaw)
  double bound;               // type 2: mu * N
  double ja[2][3], jb[2][3];  // Jacobian rows w.r.t. body a / b
  double wa[2][3], wb[2][3];  // M^-1 J^T, precomputed
  double aref[2], R[2], inv[2], f[2];
};
constexpr int kMaxBodies = 8;  // movable bodies with constraint rows in one forward pass

// Constants of the contact solver that depend on the configuration and the task only (oracle obj_mass + the reciprocals
// forward_dynamics takes of them): evaluated once per environment step, not once per forward pass.
struct SolveConsts {
  double vim, vii, bim, bii;                          // 1 / mass, 1 / inertia: vase, task body (push box / rod / ball)
  double v_inv_lin, v_inv_tor, b_inv_lin, b_inv_tor;  // 1 / (A + R) of the floor-friction rows
  double vflin, vftor, vbfl, bflin, bftor, bbfl;      // floor-friction bounds, damping rate of the floor rows
  double rix, riy, bfx, bfy;                          // rod: 1 / mx, 1 / my, per-axis bounds
  double gim, gii, g_inv_lin, g_inv_tor, gflin, gftor, gbfl;  // gremlins (their size is a config value of its own)
};

// Working set of the contact solver of ONE environment, kept in shared memory (local memory would put every access
// of this latency-bound code on an L2 / DRAM round trip).
struct Scratch {
  static constexpr int kCon = kMaxCon, kBodies = kMaxBodies;
  Con con[kMaxCon];
  Row rows[kMaxCon + 3];         // + tendon + two car wheels
  double acc[kMaxBodies + 3][3]; // robot, bodies, two car wheels (1 DoF each, in [.][0])
  double ffl[kMaxBodies][3];
  double bv[kMaxBodies][3];      // velocities of the bodies in the table (read once per pass)
  int bslot[kMaxBodies];
  SolveConsts Q;                 // cooperative kernel: this environment's constants (scalar paths keep them in registers)
  double obj[6][kMaxObj];        // cooperative kernel: the environment's object arrays for the duration of a step (ObjView)
  static constexpr int kItems = 96;
  double sc[2][kMaxObj];         // cooperative kernel: sin / cos of the objects' yaw, valid where scvalid has the slot's bit
  unsigned scvalid, pad_;
  int items[kItems];             // cooperative kernel: flattened part pairs of the object-pair narrow phase
#if defined(SAG_TIMING)
  unsigned long long tsum[4];    // this environment's section clocks (tuning builds)
#endif
};

// env_step / end_of_step modes:
// kStepFull: the full scalar path (one thread = one environment, contact solver included);
// kStepCoop: warp-cooperative (one warp = one environment, device only);
// kStepNear: the contact-free path (no contact code), with (run-time flag `pretest`) the exact overlap / tendon pre-test in
// front of every substep and of the final forward pass -- for environments that have something within reach but
// (usually) touch nothing; the step is abandoned (return 1, nothing written that the full path would not write
// identically) as soon as a robot geom overlaps an object or the tendon is taut, and the environment is handed to the
// contact path.  With pretest == false it is the quiet path.
constexpr int kStepFull = 0, kStepCoop = 1, kStepNear = 2;

struct Ctx {  // per-thread view of one environment
  const Dev& D;
  int e;
  TaskSpec sp;
  Slots L;
  int task;
  ObjView O;
};
SAG_HD size_t oix(const Ctx& C, int slot) { return (size_t)slot * C.O.stride; }

struct Phys {
  double fc[3];    // generalised constraint force on the robot
  double qacc[3];  // robot acceleration M^-1 (fsmooth + fc)
  unsigned touch;  // bit s: a robot geom is in contact (dist <= 0) with object slot s
  unsigned mov;    // bit s: movable body s has a non-zero velocity (after integration, if any)
  int err;
  double wtau[2];  // car: constraint torque on the wheels
};

SAG_HD double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
SAG_HD int ctz32(unsigned m) {
#if defined(__CUDA_ARCH__)
  return __ffs((int)m) - 1;
#else
  return __builtin_ctz(m);
#endif
}

// ---- car wheel-floor friction rows (always present for the car; oracle forward_dynamics "car:" block) ----------
// Reduced model: level chassis, static normal loads; per wheel a longitudinal slip row (chassis point velocity along the
// rolling direction + r * wheel rate) and a lateral slip row, jointly bounded by mu * N.
SAG_HD void wheel_row_setup(const CarRobot& R, int i, double sn, double cs, double p, double q, const PtConst& K, int wheel_body, Row& r) {
  const double iw = 1.0 / kCar.Iw;
  const double bdamp = 2.0 / (kImpDmax * kSolTc), rr0 = (1.0 - kImpD0) / kImpD0;
  double bx = i == 0 ? -0.1 : 0.1, by = 0.1;
  double rx = bx * cs - by * sn, ry = bx * sn + by * cs;
  r.type = 2; r.nk = 2; r.bound = kMu * kCar.nwheel;
  r.ba = 0; r.bb = wheel_body;
  r.ja[0][0] = -sn; r.ja[0][1] = cs; r.ja[0][2] = rx * cs - ry * -sn;
  r.jb[0][0] = kCarWheelR; r.jb[0][1] = 0.0; r.jb[0][2] = 0.0;
  r.ja[1][0] = cs; r.ja[1][1] = sn; r.ja[1][2] = rx * sn - ry * cs;
  r.jb[1][0] = 0.0; r.jb[1][1] = 0.0; r.jb[1][2] = 0.0;
  const double vb[3] = {R.wheel[i], 0.0, 0.0};
  for (int k = 0; k < 2; ++k) {
    double diag = 0.0, vel = 0.0;
    pt_solve(p, q, K.ia0, K.is0, r.ja[k], r.wa[k]);
    diag += dot3(r.ja[k], r.wa[k]); vel += dot3(r.ja[k], R.v);
    r.wb[k][0] = r.wb[k][1] = r.wb[k][2] = 0.0;
    if (k == 0) { r.wb[k][0] = r.jb[k][0] * iw; diag += dot3(r.jb[k], r.wb[k]); vel += dot3(r.jb[k], vb); }
    r.R[k] = rr0 * diag;
    r.inv[k] = 1.0 / (diag + r.R[k]);
    r.aref[k] = -bdamp * vel;
    r.f[k] = 0.0;
  }
}
// one Gauss-Seidel visit of a wheel row pair: both slip rows, then projection onto the friction disc
SAG_HD void wheel_row_update(Row& r, double* accR_, double* accW_, double& sdf, double& sf) {
  const double fo0 = r.f[0], fo1 = r.f[1];
  // chassis / wheel accelerations in registers for the visit (accR_ / accW_ may be shared memory); the wheel has one DoF
  double accR[3] = {accR_[0], accR_[1], accR_[2]}, accW[3] = {accW_[0], accW_[1], accW_[2]};
  for (int k = 0; k < 2; ++k) {
    double a = dot3(r.ja[k], accR);
    if (k == 0) a += dot3(r.jb[k], accW);
    double fn = r.f[k] - (a - r.aref[k] + r.R[k] * r.f[k]) * r.inv[k];
    double df = fn - r.f[k];
    r.f[k] = fn;
    if (df != 0.0) {
      accR[0] += r.wa[k][0] * df; accR[1] += r.wa[k][1] * df; accR[2] += r.wa[k][2] * df;
      if (k == 0) { accW[0] += r.wb[k][0] * df; accW[1] += r.wb[k][1] * df; accW[2] += r.wb[k][2] * df; }
    }
  }
  double nf = sqrt(r.f[0] * r.f[0] + r.f[1] * r.f[1]);
  if (nf > r.bound) {
    double sc = r.bound / nf;
    for (int k = 0; k < 2; ++k) {
      double g = r.f[k] * sc, df = g - r.f[k];
      r.f[k] = g;
      if (df != 0.0) {
        accR[0] += r.wa[k][0] * df; accR[1] += r.wa[k][1] * df; accR[2] += r.wa[k][2] * df;
        if (k == 0) { accW[0] += r.wb[k][0] * df; accW[1] += r.wb[k][1] * df; accW[2] += r.wb[k][2] * df; }
      }
    }
  }
  accR_[0] = accR[0]; accR_[1] = accR[1]; accR_[2] = accR[2];
  accW_[0] = accW[0]; accW_[1] = accW[1]; accW_[2] = accW[2];
  sdf += fabs(r.f[0] - fo0) + fabs(r.f[1] - fo1); sf += fabs(r.f[0]) + fabs(r.f[1]);
}
// the car's forward dynamics when nothing else constrains it: just the two wheel row pairs (registers only)
struct CarFree { double qacc[3], fc[3], wtau[2]; };
SAG_HD void car_free_solve(const CarRobot& R, double sn, double cs, const PtConst& K, const double* fs, CarFree& F) {
  double p, q;
  R.pq(sn, cs, p, q);
  const double iw = 1.0 / kCar.Iw;
  double accR[3], accW[2][3];
  pt_solve(p, q, K.ia0, K.is0, fs, accR);
  Row rows[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    accW[i][0] = R.wheel_smooth(i) * iw; accW[i][1] = accW[i][2] = 0.0;
    wheel_row_setup(R, i, sn, cs, p, q, K, 0, rows[i]);
  }
  for (int it = 0; it < kSweeps; ++it) {
    double sdf = 0.0, sf = 0.0;
#pragma unroll
    for (int i = 0; i < 2; ++i) wheel_row_update(rows[i], accR, accW[i], sdf, sf);
    if (sdf <= kPgsTol * sf) break;
  }
  F.qacc[0] = accR[0]; F.qacc[1] = accR[1]; F.qacc[2] = accR[2];
  F.fc[0] = F.fc[1] = F.fc[2] = 0.0;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    for (int k = 0; k < 2; ++k) for (int d = 0; d < 3; ++d) F.fc[d] += rows[i].ja[k][d] * rows[i].f[k];
    F.wtau[i] = rows[i].jb[0][0] * rows[i].f[0];
  }
}

// ------------------------------------------------------------------------------------------------
// Warp-cooperative variants (device only).  In the cooperative busy kernel ONE WARP owns one environment: all 32
// lanes execute the step's scalar code redundantly (same registers, warp-uniform control flow, identical stores), and
// the sections below split their independent work items over the lanes: the broad and narrow collision phases (one
// slot / one pair / one geom pair per lane, results appended in the scalar code's canonical order by warp prefix sums),
// the overlap pre-test and the lidar pass (one object per lane, bins reduced with shared-memory max).  Every item is
// computed by the same arithmetic as in the scalar path, so results are bit-identical (tests/test_gpu_parity.py runs
// the oracle against this path).
// ------------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
// Phase alignment of the cooperative kernel's warps: every warp of the CTA arrives at a barrier at
// the top of each substep and before the end-of-step pass, so that the 16 environments of an SM walk through the same
// code at the same time and share its instruction-cache lines instead of evicting each other's.  A warp without an
// environment executes the same number of barriers (coop_idle_step).
__device__ __forceinline__ void coop_align() {
#if defined(__CUDA_ARCH__)
  asm volatile("bar.sync 0;" ::: "memory");
#endif
}
template <class RB>
__device__ __forceinline__ void coop_idle_step() {
#pragma unroll 1
  for (int k = 0; k <= RB::kNsub; ++k) coop_align();
}

#endif
#if defined(__CUDA_ARCH__)
constexpr unsigned kFullWarp = 0xffffffffu;
__device__ __forceinline__ int coop_lane() { return threadIdx.x & 31; }
// ordered append: lane order = canonical order; n in {0, 1, 2} hits per lane
__device__ __forceinline__ bool coop_append(Con* con, int cap, int& ncon, bool& overflow, int n, const Hit* hits, int ba, int bb) {
  const int lane = coop_lane();
  const unsigned m1 = __ballot_sync(kFullWarp, n >= 1), m2 = __ballot_sync(kFullWarp, n >= 2);
  const unsigned lower = (1u << lane) - 1u;
  const int off = ncon + __popc(m1 & lower) + __popc(m2 & lower);
  for (int k = 0; k < n; ++k) {
    const int idx = off + k;
    if (idx < cap) {
      Con& c = con[idx];
      c.ba = ba; c.bb = bb;
      c.nx = hits[k].nx; c.ny = hits[k].ny; c.px = hits[k].px; c.py = hits[k].py; c.dist = hits[k].dist;
    }
  }
  const int tot = ncon + __popc(m1) + __popc(m2);
  if (tot > cap) { overflow = true; ncon = cap; } else ncon = tot;
  return n > 0 && off < cap;  // this lane's first hit is in the list
}

// Both collision phases of contact_pass, lane-parallel.  Same outputs: con[0..ncon) in canonical order, overflow, touch,
// active.  (Scalar semantics on overflow: the list stops growing at the capacity, touch / active keep accumulating.)
//   broad phases: lane <-> object slot.  Phase 1 tests every collidable slot against the robot's reach; phase 2 tests, for
//     every awake / robot-touched movable body a, all slots against a in one step and records the near pairs as bit rows
//     pm[j] = {i < j} held by lane j, so that walking j upwards and the bits of pm[j] upwards is the canonical pair order.
//   narrow phase: ONE copy of the collide() code; each trip hands up to 32 geom pairs to the lanes -- phase 1: (robot geom,
//     object part) items of all near objects in slot order (only the push box has more than one part and it is the last
//     slot); phase 2: the part pairs of ALL near object pairs, flattened into the warp's item list in canonical order (a
//     multi-contact cluster -- the environments that set the kernel's duration -- is then one trip, not one per pair).
//     Hits are appended in lane order (= canonical order).  sin / cos of an object's yaw are cached per slot until the
//     object is integrated again (Scratch::sc, scvalid).
template <class RB>
__device__ __forceinline__ void detect_coop(const Ctx& C, const RB& R, double sn, double cs, unsigned mov, Scratch& S,
                                         int& ncon_out, bool& overflow_out, unsigned& touch_out, unsigned& active_out) {
  const Dev& D = C.D;
  const int lane = coop_lane();
  constexpr int cap = Scratch::kCon;
  Con* con = S.con;
  SAG_CLK_DECL;
  int ncon = 0;
  bool overflow = false;
  unsigned touch = 0, active = mov;
  // ---- this lane's slot
  int kind_l = K_NONE;
  bool coll_l = false;
  double x_l = 0.0, y_l = 0.0, bound_l = 0.0;
  if (lane >= C.L.v0 && lane < C.L.n) {
    kind_l = slot_kind(C.sp, C.L, lane);
    coll_l = kind_collidable(kind_l);
    if (coll_l) { size_t i = oix(C, lane); x_l = C.O.x[i]; y_l = C.O.y[i]; bound_l = kind_bound(D, kind_l); }
  }
  const unsigned collm = __ballot_sync(kFullWarp, coll_l);
  // ---- phase 1 broad phase
  bool near1 = false;
  if (coll_l) {
    double dx = x_l - R.q[0], dy = y_l - R.q[1], reach = RB::kReach + bound_l;
    near1 = !(dx * dx + dy * dy > reach * reach);
  }
  const unsigned near1m = __ballot_sync(kFullWarp, near1);
  const unsigned boxbit = (C.sp.box_kind == K_BOX) ? (1u << C.L.box) : 0u;  // the only multi-part object; always the last slot
  const unsigned near_single = near1m & ~boxbit;
  const int n_single = __popc(near_single) * RB::kNGeom;
  const int total1 = n_single + ((near1m & boxbit) ? RB::kNGeom * 5 : 0);
  SAG_CLK(2);
  // ---- narrow phase trips
  int base = 0, total = total1, phase = total1 > 0 ? 0 : 1;
  bool pairs_built = false, sequential = false;
  unsigned pm = 0, jm = 0, pmj = 0;
  int pj = -1;
  for (;;) {
    // -- next trip: per-lane item (geom A of body ia / part pa, geom B of slot sb / part pb); ia < 0: robot geom pa
    bool have = false;
    int ia = -1, pa = 0, sb = 0, pb = 0;
    if (phase == 0) {
      if (base >= total) { phase = 1; continue; }
      const int t = base + lane;
      base += 32;
      if (t < total) {
        have = true;
        if (t < n_single) { const int rank = t / RB::kNGeom; pa = t - rank * RB::kNGeom; sb = (int)__fns(near_single, 0, rank + 1); pb = 0; }
        else { const int u = t - n_single; pa = u / 5; pb = u - pa * 5; sb = C.L.box; }
      }
    } else {
      if (!pairs_built) {
        pairs_built = true;
        if (!active) break;
        // phase 2 broad phase: one body a at a time against all slots
        for (unsigned am = active & collm; am; am &= am - 1) {
          const int a = __ffs((int)am) - 1;
          const size_t ia_ = oix(C, a);
          const double xa = C.O.x[ia_], ya = C.O.y[ia_], ba = kind_bound(D, slot_kind(C.sp, C.L, a));
          bool nearp = false;
          if (coll_l && lane != a) {
            // canonical operands: (x_j - x_i) with i < j; the squares and the sum of the bounds do not depend on the order
            double dx = lane > a ? x_l - xa : xa - x_l, dy = lane > a ? y_l - ya : ya - y_l;
            double reach = lane > a ? bound_l + ba : ba + bound_l;
            nearp = !(dx * dx + dy * dy > reach * reach);
          }
          if (nearp && lane > a) pm |= 1u << a;
          const unsigned below = __ballot_sync(kFullWarp, nearp && lane < a);
          if (lane == a) pm |= below;
        }
        jm = __ballot_sync(kFullWarp, pm != 0);
        if (!jm) { SAG_CLK(12); break; }
        // flatten the part pairs of all near pairs into S.items, canonical order: j ascending (lane order), i ascending,
        // part of i outer, part of j inner.  Only the push box has parts, and as the last slot it can only be a j.
        const int npl = ((boxbit >> lane) & 1u) ? 5 : 1;
        const int cnt = __popc(pm) * npl;
        int incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(kFullWarp, incl, d); if (lane >= d) incl += v; }
        total = __shfl_sync(kFullWarp, incl, 31);
        base = 0;
        if (total <= Scratch::kItems) {
          int off = incl - cnt;
          for (unsigned m = pm; m; m &= m - 1) {
            const int i = __ffs((int)m) - 1;
            for (int b = 0; b < npl; ++b) S.items[off++] = i | (lane << 8) | (b << 16);
          }
          __syncwarp();
        } else sequential = true;  // more near part pairs than the list holds (a heap of bodies): one pair per trip
        SAG_CLK(12);
      }
      if (!sequential) {
        if (base >= total) break;
        const int t = base + lane;
        base += 32;
        if (t < total) { const int it = S.items[t]; have = true; ia = it & 0xff; sb = (it >> 8) & 0xff; pa = 0; pb = it >> 16; }
      } else {
        if (!pmj) {
          if (!jm) break;
          pj = __ffs((int)jm) - 1;
          jm &= jm - 1;
          pmj = __shfl_sync(kFullWarp, pm, pj);
        }
        const int pi = __ffs((int)pmj) - 1;
        pmj &= pmj - 1;
        const int npj = kind_nparts(slot_kind(C.sp, C.L, pj)), items = kind_nparts(slot_kind(C.sp, C.L, pi)) * npj;
        if (lane < items) { have = true; ia = pi; pa = lane / npj; sb = pj; pb = lane - pa * npj; }
      }
    }
    // -- narrow phase of this trip
    Hit hits[2];
    int n = 0;
    bool mvb = false, mva = false;
    unsigned newsc = 0;  // slots whose sin / cos this lane has just computed and cached
    if (have) {
      Geom ga, gb;
      const int kb = slot_kind(C.sp, C.L, sb);
      mvb = kind_movable(kb);
      {
        const size_t i = oix(C, sb);
        double oc = 1.0, os = 0.0;
        if (mvb) {
          if ((S.scvalid >> sb) & 1u) { os = S.sc[0][sb]; oc = S.sc[1][sb]; }
          else { sag_sincos(C.O.yaw[i], &os, &oc); S.sc[0][sb] = os; S.sc[1][sb] = oc; newsc |= 1u << sb; }
        }
        obj_geom(D, kb, pb, C.O.x[i], C.O.y[i], oc, os, gb);
      }
      if (ia < 0) R.geom(pa, sn, cs, ga);
      else {
        const int ka = slot_kind(C.sp, C.L, ia);
        mva = kind_movable(ka);
        const size_t i = oix(C, ia);
        double oc = 1.0, os = 0.0;
        if (mva) {
          if ((S.scvalid >> ia) & 1u) { os = S.sc[0][ia]; oc = S.sc[1][ia]; }
          else { sag_sincos(C.O.yaw[i], &os, &oc); S.sc[0][ia] = os; S.sc[1][ia] = oc; newsc |= 1u << ia; }
        }
        obj_geom(D, ka, pa, C.O.x[i], C.O.y[i], oc, os, ga);
      }
      n = collide_inl(ga, gb, hits);
    }
    const bool stored = coop_append(con, cap, ncon, overflow, n, hits, ia < 0 ? 0 : (mva ? 1 + ia : -1), mvb ? 1 + sb : -1);
    newsc = __reduce_or_sync(kFullWarp, newsc);
    if (newsc) { __syncwarp(); S.scvalid |= newsc; __syncwarp(); }  // every lane stores the same word
    if (phase == 0) {
      touch |= __reduce_or_sync(kFullWarp, stored ? 1u << sb : 0u);
      active |= __reduce_or_sync(kFullWarp, (n && mvb) ? 1u << sb : 0u);
      SAG_CLK(11);
    } else {
      SAG_CLK(13);
    }
  }
  __syncwarp();
  ncon_out = ncon; overflow_out = overflow; touch_out = touch; active_out = active;
}

template <class RB>
__device__ __forceinline__ bool robot_overlaps_any_coop(const Ctx& C, const RB& R, double sn, double cs) {
  const Dev& D = C.D;
  const int s = C.L.v0 + coop_lane();
  bool hit = false;
  if (s < C.L.n) {
    const int kind = slot_kind(C.sp, C.L, s);
    if (kind_collidable(kind)) {
      size_t i = oix(C, s);
      double x = C.O.x[i], y = C.O.y[i];
      double dx = x - R.q[0], dy = y - R.q[1], reach = RB::kReach + kind_bound(D, kind);
      if (!(dx * dx + dy * dy > reach * reach)) {
        double oc = 1.0, os = 0.0;
        if (kind_movable(kind)) sag_sincos(C.O.yaw[i], &os, &oc);
        for (int pt = 0; pt < kind_nparts(kind) && !hit; ++pt) {
          Geom go;
          obj_geom(D, kind, pt, x, y, oc, os, go);
          for (int rg = 0; rg < RB::kNGeom; ++rg) {
            Geom grg;
            R.geom(rg, sn, cs, grg);
            if (overlap(grg, go)) { hit = true; break; }
          }
        }
      }
    }
  }
  return __any_sync(kFullWarp, hit);
}
#endif  // __CUDA_ARCH__

// HaulBox tendon (haul_box.py:21-30): robot site <-> box site, length limited to kTendonMax; taut when dist < 0
template <class RB>
SAG_HD bool tendon_taut(const Ctx& C, const RB& R, double& tdx, double& tdy, double& tlen, double& tdist) {
  size_t ib = oix(C, C.L.box);
  tdx = C.O.x[ib] - R.q[0]; tdy = C.O.y[ib] - R.q[1];
  double dz = kBoxSize - kPtZ;
  tlen = sqrt(tdx * tdx + tdy * tdy + dz * dz);
  tdist = kTendonMax - tlen;
  return tdist < 0.0;
}

SAG_HD void solve_consts(const Dev& D, const TaskSpec& sp, SolveConsts& Q, bool gremlins) {
  const int bkind = sp.box_kind;
  const BodyPar VP = kind_body(D, K_VASE), BP = kind_body(D, bkind ? bkind : K_BOX);
  const double rr = (1.0 - kImpD0) / kImpD0;
  Q.vim = 1.0 / VP.m; Q.vii = 1.0 / VP.iz; Q.bim = 1.0 / BP.m; Q.bii = 1.0 / BP.iz;
  Q.v_inv_lin = 1.0 / (Q.vim + rr * Q.vim); Q.v_inv_tor = 1.0 / (Q.vii + rr * Q.vii);
  Q.b_inv_lin = 1.0 / (Q.bim + rr * Q.bim); Q.b_inv_tor = 1.0 / (Q.bii + rr * Q.bii);
  Q.vflin = VP.flin; Q.vftor = VP.ftor; Q.vbfl = VP.bfl; Q.bflin = BP.flin; Q.bftor = BP.ftor; Q.bbfl = BP.bfl;
  Q.rix = Q.riy = 0.0;
  if (bkind == K_ROD) { Q.rix = 1.0 / BP.mx; Q.riy = 1.0 / BP.my; }
  Q.bfx = BP.fx; Q.bfy = BP.fy;
  if (gremlins) {
    const BodyPar GP = kind_body(D, K_GREMLIN);
    Q.gim = 1.0 / GP.m; Q.gii = 1.0 / GP.iz;
    Q.g_inv_lin = 1.0 / (Q.gim + rr * Q.gim); Q.g_inv_tor = 1.0 / (Q.gii + rr * Q.gii);
    Q.gflin = GP.flin; Q.gftor = GP.ftor; Q.gbfl = GP.bfl;
  }
}

template <class RB, bool Coop>
SAG_HD void contact_pass_body(const Ctx& C, const RB& R, double sn, double cs, const PtConst& K, const double* fs,
                              unsigned mov, bool integrate, double h, Scratch& S, const SolveConsts& Q, Phys& P, const double* mocap);
// scalar paths: one out-of-line copy; the cooperative kernel inlines the body at its single call site (env_step), so
// that the environment's registers need not travel through local memory
template <class RB, bool Coop>
SAG_HD_NOINLINE void contact_pass(const Ctx& C, const RB& R, double sn, double cs, const PtConst& K, const double* fs,
                                  unsigned mov, bool integrate, double h, Scratch& S, const SolveConsts& Q, Phys& P, const double* mocap) {
  contact_pass_body<RB, Coop>(C, R, sn, cs, K, fs, mov, integrate, h, S, Q, P, mocap);
}
template <class RB, bool Coop>
SAG_HD void contact_pass_body(const Ctx& C, const RB& R, double sn, double cs, const PtConst& K, const double* fs,
                              unsigned mov, bool integrate, double h, Scratch& S, const SolveConsts& Q, Phys& P, const double* mocap) {
  constexpr int kCapCon = Scratch::kCon, kCapBodies = Scratch::kBodies;
  const Dev& D = C.D;
  const int e = C.e;
  double p, q;
  R.pq(sn, cs, p, q);
  Con* con = S.con;
  int ncon = 0;
  unsigned active = mov, touch = 0;
  bool overflow = false;
  P.err = 0;
  constexpr bool kCarRobot = RB::kKind == 1;
  SAG_PROF(e, 0, 1);
  SAG_CLK_DECL;
  if constexpr (Coop) {
#if defined(__CUDA_ARCH__)
    detect_coop<RB>(C, R, sn, cs, mov, S, ncon, overflow, touch, active);
#if defined(SAG_TIMING)
    { long long now_ = clock64(); if ((threadIdx.x & 31) == 0) S.tsum[0] += (unsigned long long)(now_ - clk_); }
#endif
#endif
  } else {
  Hit hits[2];
  // ---- phase 1: robot geoms vs objects, slot order
  for (int s = C.L.v0; s < C.L.n; ++s) {
    int kind = slot_kind(C.sp, C.L, s);
    if (!kind_collidable(kind)) continue;
    size_t i = oix(C, s);
    double x = C.O.x[i], y = C.O.y[i];
    double dx = x - R.q[0], dy = y - R.q[1], reach = RB::kReach + kind_bound(D, kind);
    if (dx * dx + dy * dy > reach * reach) continue;
    bool mvb = kind_movable(kind);
    double oc = 1.0, os = 0.0;
    if (mvb) sag_sincos(C.O.yaw[i], &os, &oc);
    for (int rg = 0; rg < RB::kNGeom; ++rg) {
      Geom grg;
      R.geom(rg, sn, cs, grg);
      for (int pt = 0; pt < kind_nparts(kind); ++pt) {
        Geom go;
        obj_geom(D, kind, pt, x, y, oc, os, go);
        int n = collide(grg, go, hits);
        SAG_PROF(e, 1, 1);
        for (int k = 0; k < n; ++k) {
          if (ncon >= kCapCon) { overflow = true; break; }
          Con& c = con[ncon++];
          c.ba = 0; c.bb = mvb ? 1 + s : -1;
          c.nx = hits[k].nx; c.ny = hits[k].ny; c.px = hits[k].px; c.py = hits[k].py; c.dist = hits[k].dist;
          touch |= 1u << s;  // robot_contacts() sees the contacts that made it into the list (mujoco_bridge.py:177-191)
        }
        if (n && mvb) active |= 1u << s;
      }
    }
  }
  // ---- phase 2: object pairs (j ascending, i < j ascending) with at least one awake / robot-touched movable body
  if (active) {
    for (int j = C.L.v0; j < C.L.n; ++j) {
      int kj = slot_kind(C.sp, C.L, j);
      if (!kind_collidable(kj)) continue;
      bool aj = (active >> j) & 1u;
      unsigned cand = aj ? ((1u << j) - 1u) : (active & ((1u << j) - 1u));
      cand &= ~((1u << C.L.v0) - 1u);
      if (!cand) continue;
      size_t ij = oix(C, j);
      double xj = C.O.x[ij], yj = C.O.y[ij], bj = kind_bound(D, kj);
      bool mj = kind_movable(kj);
      double cj = 1.0, sj = 0.0;
      bool have_j = false;
      for (unsigned cm = cand; cm; cm &= cm - 1) {
        int i = ctz32(cm);
        int ki = slot_kind(C.sp, C.L, i);
        if (!kind_collidable(ki)) continue;
        size_t ii = oix(C, i);
        double xi = C.O.x[ii], yi = C.O.y[ii];
        double dx = xj - xi, dy = yj - yi, reach = bj + kind_bound(D, ki);
        SAG_PROF(e, 6, 1);
        if (dx * dx + dy * dy > reach * reach) continue;
        bool mi = kind_movable(ki);
        double ci = 1.0, si = 0.0;
        if (mi) sag_sincos(C.O.yaw[ii], &si, &ci);
        if (mj && !have_j) { sag_sincos(C.O.yaw[ij], &sj, &cj); have_j = true; }
        for (int pi = 0; pi < kind_nparts(ki); ++pi) {
          Geom gi;
          obj_geom(D, ki, pi, xi, yi, ci, si, gi);
          for (int pj = 0; pj < kind_nparts(kj); ++pj) {
            Geom gj;
            obj_geom(D, kj, pj, xj, yj, cj, sj, gj);
            int n = collide(gi, gj, hits);
            SAG_PROF(e, 1, 1);
            for (int k = 0; k < n; ++k) {
              if (ncon >= kCapCon) { overflow = true; break; }
              Con& c = con[ncon++];
              c.ba = mi ? 1 + i : -1; c.bb = mj ? 1 + j : -1;
              c.nx = hits[k].nx; c.ny = hits[k].ny; c.px = hits[k].px; c.py = hits[k].py; c.dist = hits[k].dist;
            }
          }
        }
      }
    }
  }
  }
  P.touch = touch;
  P.mov = mov;
  if constexpr (Coop) SAG_CLK_RESET;
  SAG_PROF(e, 2, ncon);
  P.fc[0] = P.fc[1] = P.fc[2] = 0.0;
  P.wtau[0] = P.wtau[1] = 0.0;
  // ---- which constraint rows exist?
  unsigned touched = 0;
  bool any_row = false;
  for (int i = 0; i < ncon; ++i) {
    const Con& c = con[i];
    if (!(c.dist < 0.0) || (c.ba < 0 && c.bb < 0)) continue;
    // bit 31 marks an active row where no registry task has a movable body in slot 31; a user-defined task can have
    // its box there (*C instantiations: a flag of its own)
    if constexpr (RB::kCustom) any_row = true;
    else touched |= 0x80000000u;
    if (c.ba > 0) touched |= 1u << (c.ba - 1);
    if (c.bb > 0) touched |= 1u << (c.bb - 1);
  }
  if constexpr (!RB::kCustom) {
    any_row = (touched & 0x80000000u) != 0;
    touched &= 0x7fffffffu;
  }
  int nactive = 0;  // contact rows (counted only where weld rows share the row table)
  if constexpr (RB::kGremlins) for (int i = 0; i < ncon; ++i) { const Con& c = con[i]; if (c.dist < 0.0 && !(c.ba < 0 && c.bb < 0)) ++nactive; }
  double tdx = 0.0, tdy = 0.0, tlen = 0.0, tdist = 0.0;
  bool tendon = false;
  if (C.task == T_HAUL_BOX) {  // tendon length limit, haul_box.py:21-30
    tendon = tendon_taut(C, R, tdx, tdy, tlen, tdist);
    if (tendon) touched |= 1u << C.L.box;
  }
  // gremlins: welded to their mocap bodies (primitive_objects.py:79-82), so always in the body table
  const int ng = RB::kGremlins ? C.sp.ng : 0;
  if (ng > 0) touched |= ((1u << ng) - 1u) << C.L.g0;
  // the row table holds kMaxCon + 3 entries; with weld rows in it the active contacts may not fit: a PhysicsError
  if ((RB::kKind == 1 ? 2 : 0) + nactive + (tendon ? 1 : 0) + 2 * ng > kMaxCon + 3) overflow = true;
  double racc[3];
  pt_solve(p, q, K.ia0, K.is0, fs, racc);
  P.qacc[0] = racc[0]; P.qacc[1] = racc[1]; P.qacc[2] = racc[2];
  const unsigned fl = touched | mov;  // floor-friction bodies: awake or touched, slot order
  // capacity limits: a PhysicsError; no constraint forces, no object motion in this pass
  int nb = 0;
  for (unsigned m = fl; m; m &= m - 1) ++nb;
  if (nb > kCapBodies) overflow = true;
  if (overflow) P.err = 1;
  if (!kCarRobot) {
    if (overflow) return;
    if (!any_row && !tendon && mov == 0 && ng == 0) return;  // nothing to solve, nothing to move
  }
  // ---- body table: compact ids in slot order, velocities read once
  nb = 0;
  if (!overflow) for (unsigned m = fl; m; m &= m - 1) {
    const int s = ctz32(m);
    size_t i = oix(C, s);
    S.bslot[nb] = s;
    S.bv[nb][0] = C.O.vx[i]; S.bv[nb][1] = C.O.vy[i]; S.bv[nb][2] = C.O.w[i];
    ++nb;
  }
  auto cid = [&](int slot) { int k = 0; while (S.bslot[k] != slot) ++k; return k; };
  const int bkind = C.sp.box_kind;  // kind of the task's movable body: push box, rod or ball (0: none)
  const bool rod = bkind == K_ROD;
  double rc = 1.0, rs = 0.0, rma = 0.0, rmb = 0.0, rmc = 0.0;  // rod: R diag(1/mx, 1/my) R^T
  if (rod) {
    sag_sincos(C.O.yaw[oix(C, C.L.box)], &rs, &rc);
    rma = Q.rix * rc * rc + Q.riy * rs * rs; rmb = (Q.rix - Q.riy) * rc * rs; rmc = Q.rix * rs * rs + Q.riy * rc * rc;
  }
  // body < 0 static, 0 robot, 1 + slot movable
  auto minv = [&](int body, const double* j, double* o) {
    if (body == 0) { pt_solve(p, q, K.ia0, K.is0, j, o); return; }
    const bool isb = body - 1 == C.L.box;
    if (isb && rod) { o[0] = rma * j[0] + rmb * j[1]; o[1] = rmb * j[0] + rmc * j[1]; o[2] = j[2] * Q.bii; return; }
    const bool isg = RB::kGremlins && body - 1 >= C.L.g0 && body - 1 < C.L.p0;
    double im = isb ? Q.bim : (isg ? Q.gim : Q.vim), ii = isb ? Q.bii : (isg ? Q.gii : Q.vii);
    o[0] = j[0] * im; o[1] = j[1] * im; o[2] = j[2] * ii;
  };
  auto bvel = [&](int body, double* v) {
    if (body == 0) { v[0] = R.v[0]; v[1] = R.v[1]; v[2] = R.v[2]; }
    else { size_t i = oix(C, body - 1); v[0] = C.O.vx[i]; v[1] = C.O.vy[i]; v[2] = C.O.w[i]; }
  };
  auto bpos = [&](int body, double* o) {
    if (body == 0) { o[0] = R.q[0]; o[1] = R.q[1]; }
    else { size_t i = oix(C, body - 1); o[0] = C.O.x[i]; o[1] = C.O.y[i]; }
  };
  Row* rows = S.rows;
  int nrow = 0, tendon_row = -1;
  const double bdamp = 2.0 / (kImpDmax * kSolTc);
  const double kbase = 1.0 / (kImpDmax * kImpDmax * kSolTc * kSolTc);
  double (*acc)[3] = S.acc;
  constexpr int kWheelBody = kCapBodies + 1;  // acc index of the left wheel
  if constexpr (kCarRobot) {
    const double iw = 1.0 / kCar.Iw;
    for (int i = 0; i < 2; ++i) {
      acc[kWheelBody + i][0] = R.wheel_smooth(i) * iw; acc[kWheelBody + i][1] = acc[kWheelBody + i][2] = 0.0;
      wheel_row_setup(R, i, sn, cs, p, q, K, kWheelBody + i, rows[nrow++]);
    }
  }
  if (overflow) { ncon = 0; tendon = false; }  // car: the wheel rows are still solved, nothing else
  const int nweld = overflow ? 0 : ng;
  (void)nweld;
  if constexpr (Coop) SAG_CLKG(8, 1, S);
  // one row pair per active contact, in contact order.  Cooperative mode: contact i is set up by lane i (ncon <= 16),
  // the row index is the rank of the contact among the active ones.
  int i_begin = 0, i_end = ncon, my_row = 0;
  (void)my_row;
#if defined(__CUDA_ARCH__)
  if constexpr (Coop) {
    __syncwarp();
    const int lane = coop_lane();
    bool act = false;
    if (lane < ncon) { const Con& c = con[lane]; act = c.dist < 0.0 && !(c.ba < 0 && c.bb < 0); }
    const unsigned am = __ballot_sync(kFullWarp, act);
    my_row = nrow + __popc(am & ((1u << lane) - 1u));
    nrow += __popc(am);
    i_begin = act ? lane : 0; i_end = act ? lane + 1 : 0;
  }
#endif
  for (int i = i_begin; i < i_end; ++i) {
    const Con c = con[i];
    if (!(c.dist < 0.0)) continue;
    if (c.ba < 0 && c.bb < 0) continue;
    Row& r = Coop ? rows[my_row] : rows[nrow++];
    r.type = 0; r.nk = 2; r.bound = kMu;  // contact rows: friction coefficient of the pair
    double cb = bdamp, ck = kbase;
    if (bkind > K_BOX && (c.ba - 1 == C.L.box || c.bb - 1 == C.L.box)) {  // priority-1 geom: its friction / solref
      r.bound = kPrioMu;
      if (bkind == K_BALL) {
        cb = 2.0 / (kImpDmax * kBallSolTc);
        ck = 1.0 / (kImpDmax * kImpDmax * kBallSolTc * kBallSolTc * kBallSolDr * kBallSolDr);
      }
    }
    r.ba = c.ba > 0 ? 1 + cid(c.ba - 1) : c.ba; r.bb = c.bb > 0 ? 1 + cid(c.bb - 1) : c.bb;
    double tx = -c.ny, ty = c.nx;
    double pa[2] = {0, 0}, pb[2] = {0, 0}, va[3] = {0, 0, 0}, vb[3] = {0, 0, 0};
    if (c.ba >= 0) { bpos(c.ba, pa); bvel(c.ba, va); }
    if (c.bb >= 0) { bpos(c.bb, pb); bvel(c.bb, vb); }
    double rax = c.px - pa[0], ray = c.py - pa[1], rbx = c.px - pb[0], rby = c.py - pb[1];
    r.ja[0][0] = -c.nx; r.ja[0][1] = -c.ny; r.ja[0][2] = -(rax * c.ny - ray * c.nx);
    r.jb[0][0] = c.nx; r.jb[0][1] = c.ny; r.jb[0][2] = rbx * c.ny - rby * c.nx;
    r.ja[1][0] = -tx; r.ja[1][1] = -ty; r.ja[1][2] = -(rax * ty - ray * tx);
    r.jb[1][0] = tx; r.jb[1][1] = ty; r.jb[1][2] = rbx * ty - rby * tx;
    double d = impedance(c.dist);
    for (int k = 0; k < 2; ++k) {
      double diag = 0.0, vel = 0.0;
      if (c.ba >= 0) { minv(c.ba, r.ja[k], r.wa[k]); diag += dot3(r.ja[k], r.wa[k]); vel += dot3(r.ja[k], va); }
      if (c.bb >= 0) { minv(c.bb, r.jb[k], r.wb[k]); diag += dot3(r.jb[k], r.wb[k]); vel += dot3(r.jb[k], vb); }
      r.R[k] = (1.0 - d) / d * diag;
      r.inv[k] = 1.0 / (diag + r.R[k]);
      r.aref[k] = -cb * vel - (k == 0 ? d * ck * c.dist : 0.0);
      r.f[k] = 0.0;
    }
  }
#if defined(__CUDA_ARCH__)
  if constexpr (Coop) __syncwarp();
#endif
  if (tendon) {
    Row& r = rows[nrow]; tendon_row = nrow++;
    r.type = 0; r.nk = 1; r.bound = 0.0;
    const int bbox = 1 + C.L.box;
    r.ba = 0; r.bb = 1 + cid(C.L.box);
    r.ja[0][0] = tdx / tlen; r.ja[0][1] = tdy / tlen; r.ja[0][2] = 0.0;
    r.jb[0][0] = -tdx / tlen; r.jb[0][1] = -tdy / tlen; r.jb[0][2] = 0.0;
    double va[3], vb[3], diag = 0.0;
    bvel(0, va); bvel(bbox, vb);
    minv(0, r.ja[0], r.wa[0]); diag += dot3(r.ja[0], r.wa[0]);
    minv(bbox, r.jb[0], r.wb[0]); diag += dot3(r.jb[0], r.wb[0]);
    double d = impedance(tdist);
    r.R[0] = (1.0 - d) / d * diag;
    r.inv[0] = 1.0 / (diag + r.R[0]);
    r.aref[0] = -bdamp * (dot3(r.ja[0], va) + dot3(r.jb[0], vb)) - d * kbase * tdist;
    r.f[0] = 0.0;
  }
  // gremlin welds (primitive_objects.py:79-82, world.py:157-165): soft equality between the gremlin and its mocap body,
  // target = spawn pose + mocap position [EXT], solref (0.02, 1.5), default solimp.  Planar reduction: one bilateral
  // row pair (x, y) and one bilateral row (yaw) per gremlin, the impedance of a row from its own residual.
  if constexpr (RB::kGremlins)
  for (int g = 0; g < nweld; ++g) {
    const int s = C.L.g0 + g;
    const size_t i = oix(C, s);
    const double wbd = 2.0 / (kImpDmax * kWeldSolTc);
    const double wkk = 1.0 / (kImpDmax * kImpDmax * kWeldSolTc * kWeldSolTc * kWeldSolDr * kWeldSolDr);
    const double* sp0 = D.grem + (size_t)(2 + 3 * g) * D.stride + e;
    const double res[3] = {C.O.x[i] - (sp0[0] + mocap[0]), C.O.y[i] - (sp0[D.stride] + mocap[1]), C.O.yaw[i] - sp0[2 * (size_t)D.stride]};
    const double vb[3] = {C.O.vx[i], C.O.vy[i], C.O.w[i]};
    const int body = 1 + cid(s);
    for (int part = 0; part < 2; ++part) {
      Row& r = rows[nrow++];
      r.type = 1; r.nk = part == 0 ? 2 : 1; r.bound = 0.0;
      r.ba = -1; r.bb = body;
      for (int k = 0; k < 2; ++k) for (int d = 0; d < 3; ++d) { r.ja[k][d] = 0.0; r.jb[k][d] = 0.0; r.wa[k][d] = 0.0; r.wb[k][d] = 0.0; }
      if (part == 0) { r.jb[0][0] = 1.0; r.jb[1][1] = 1.0; } else r.jb[0][2] = 1.0;
      for (int k = 0; k < 2; ++k) { r.aref[k] = 0.0; r.R[k] = 0.0; r.inv[k] = 0.0; r.f[k] = 0.0; }
      for (int k = 0; k < r.nk; ++k) {
        const double resid = part == 0 ? res[k] : res[2];
        minv(1 + s, r.jb[k], r.wb[k]);
        const double diag = dot3(r.jb[k], r.wb[k]), d = impedance(resid);
        r.R[k] = (1.0 - d) / d * diag;
        r.inv[k] = 1.0 / (diag + r.R[k]);
        r.aref[k] = -wbd * dot3(r.jb[k], vb) - d * wkk * resid;
      }
    }
  }
  // body accelerations: acc[0] = robot, acc[1 + compact id] = movable object
  double (*ffl)[3] = S.ffl;
  acc[0][0] = racc[0]; acc[0][1] = racc[1]; acc[0][2] = racc[2];
  for (int b = 0; b < nb; ++b) { acc[1 + b][0] = acc[1 + b][1] = acc[1 + b][2] = 0.0; ffl[b][0] = ffl[b][1] = ffl[b][2] = 0.0; }
  const double rr = (1.0 - kImpD0) / kImpD0;
  SAG_PROF(e, 9, nrow); SAG_PROF(e, 10, nb); SAG_PROF(e, 11, any_row ? 1 : 0);
  SAG_PROF_MAX(e, 12, ncon); SAG_PROF_MAX(e, 13, nb); SAG_PROF_MAX(e, 14, nrow);
  { int oo = 0; for (int i = 0; i < ncon; ++i) if (con[i].ba != 0) oo = 1; SAG_PROF_MAX(e, 15, oo); (void)oo; }
  if constexpr (Coop) SAG_CLKG(3, 1, S);
  // Projected Gauss-Seidel; stops after kSweeps sweeps or when a sweep changes the forces by < kPgsTol (relative, L1).
  // The row visits are strictly sequential; in the cooperative kernel all lanes run them redundantly on the warp's
  // shared-memory working set (broadcast reads, identical stores).  Every visit first stages ALL the constants it needs in
  // registers (one batch of loads, one wait) -- the compiler cannot hoist shared-memory loads over the visit's own stores.
  // The floor-friction visits of different bodies touch disjoint state, so the cooperative kernel runs them one body per
  // lane; their contributions to the running sums are then added in body order, as the sequential sweep does.
  auto floor_visit = [&](int b, double& tdf, double& tf) {
    SAG_PROF(e, 5, 1);
    const bool isb = S.bslot[b] == C.L.box;
    const bool isg = RB::kGremlins && S.bslot[b] >= C.L.g0 && S.bslot[b] < C.L.p0;
    const double Al = isb ? Q.bim : (isg ? Q.gim : Q.vim), At = isb ? Q.bii : (isg ? Q.gii : Q.vii);
    const double inv_lin = isb ? Q.b_inv_lin : (isg ? Q.g_inv_lin : Q.v_inv_lin), inv_tor = isb ? Q.b_inv_tor : (isg ? Q.g_inv_tor : Q.v_inv_tor);
    const double flin = isb ? Q.bflin : (isg ? Q.gflin : Q.vflin), ftor = isb ? Q.bftor : (isg ? Q.gftor : Q.vftor);
    const double bfl = isb ? Q.bbfl : (isg ? Q.gbfl : Q.vbfl);
    const double vx = S.bv[b][0], vy = S.bv[b][1], w = S.bv[b][2];
    double* acs = acc[1 + b];
    double* flb = ffl[b];
    const double fl0 = flb[0], fl1 = flb[1], fl2 = flb[2];
    double ac[3] = {acs[0], acs[1], acs[2]};  // registers for the visit, stored back at the end
    double f0, f1, d0, d1;
    if (isb && rod) {  // one row across the axis (rolling, body x) and one along it (sliding, body y), clamped separately
      const double inv_x = 1.0 / (Q.rix + rr * Q.rix), inv_y = 1.0 / (Q.riy + rr * Q.riy);
      double au = ac[0] * rc + ac[1] * rs, aw = -ac[0] * rs + ac[1] * rc;
      double vu = vx * rc + vy * rs, vw = -vx * rs + vy * rc;
      f0 = fl0 - (au + bfl * vu + rr * Q.rix * fl0) * inv_x;
      f1 = fl1 - (aw + bfl * vw + rr * Q.riy * fl1) * inv_y;
      f0 = clampd(f0, -Q.bfx, Q.bfx); f1 = clampd(f1, -Q.bfy, Q.bfy);
      d0 = f0 - fl0; d1 = f1 - fl1;
      double du = d0 * Q.rix, dw = d1 * Q.riy;
      ac[0] += du * rc - dw * rs; ac[1] += du * rs + dw * rc;
    } else {
      f0 = fl0 - (ac[0] + bfl * vx + rr * Al * fl0) * inv_lin;
      f1 = fl1 - (ac[1] + bfl * vy + rr * Al * fl1) * inv_lin;
      double nf = sqrt(f0 * f0 + f1 * f1);
      if (nf > flin) { double sc = flin / nf; f0 *= sc; f1 *= sc; }
      d0 = f0 - fl0; d1 = f1 - fl1;
      ac[0] += d0 * Al; ac[1] += d1 * Al;
    }
    double f2 = fl2 - (ac[2] + bfl * w + rr * At * fl2) * inv_tor;
    f2 = clampd(f2, -ftor, ftor);
    double d2 = f2 - fl2;
    ac[2] += d2 * At;
    flb[0] = f0; flb[1] = f1; flb[2] = f2;
    acs[0] = ac[0]; acs[1] = ac[1]; acs[2] = ac[2];
    tdf = fabs(d0) + fabs(d1) + fabs(d2); tf = fabs(f0) + fabs(f1) + fabs(f2);
  };
#pragma unroll 1
  for (int it = 0; it < kSweeps; ++it) {
    double sdf = 0.0, sf = 0.0;
    SAG_PROF(e, 8, 1);
#pragma unroll 1
    for (int i = 0; i < nrow; ++i) {
      Row& r = rows[i];
      if (kCarRobot && r.type == 2) {
        // the wheel visit on a register copy of the row: one batch of loads instead of a reload after every store to r.f
        Row Lr;
        Lr.bound = r.bound;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
#pragma unroll
          for (int d = 0; d < 3; ++d) { Lr.ja[k][d] = r.ja[k][d]; Lr.jb[k][d] = r.jb[k][d]; Lr.wa[k][d] = r.wa[k][d]; Lr.wb[k][d] = r.wb[k][d]; }
          Lr.aref[k] = r.aref[k]; Lr.R[k] = r.R[k]; Lr.inv[k] = r.inv[k]; Lr.f[k] = r.f[k];
        }
        wheel_row_update(Lr, acc[0], acc[r.bb], sdf, sf);
        r.f[0] = Lr.f[0]; r.f[1] = Lr.f[1];
        continue;
      }
      // one visit of a contact row pair (normal, tangent) or of the tendon row (one row)
      const int ba = r.ba, bb = r.bb, nk = RB::kGremlins ? r.nk : ((i == tendon_row) ? 1 : 2);
      const bool bilateral = RB::kGremlins && r.type == 1;
      const double bound = r.bound;
      double ja[2][3], jb[2][3], wa[2][3], wb[2][3], aref[2], Rk[2], inv[2], f[2];
#pragma unroll
      for (int k = 0; k < 2; ++k) {
#pragma unroll
        for (int d = 0; d < 3; ++d) { ja[k][d] = r.ja[k][d]; jb[k][d] = r.jb[k][d]; wa[k][d] = r.wa[k][d]; wb[k][d] = r.wb[k][d]; }
        aref[k] = r.aref[k]; Rk[k] = r.R[k]; inv[k] = r.inv[k]; f[k] = r.f[k];
      }
      double aa[3] = {0.0, 0.0, 0.0}, ab[3] = {0.0, 0.0, 0.0};
      if (ba >= 0) { aa[0] = acc[ba][0]; aa[1] = acc[ba][1]; aa[2] = acc[ba][2]; }
      if (bb >= 0) { ab[0] = acc[bb][0]; ab[1] = acc[bb][1]; ab[2] = acc[bb][2]; }
      bool changed = false;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (k >= nk) break;
        SAG_PROF(e, 4, 1);
        double a = 0.0;
        if (ba >= 0) a += dot3(ja[k], aa);
        if (bb >= 0) a += dot3(jb[k], ab);
        const double fo = f[k];
        double fn = fo - (a - aref[k] + Rk[k] * fo) * inv[k];
        if (bilateral) { }  // equality row: no projection
        else if (k == 0) { if (fn < 0.0) fn = 0.0; }
        else { double lim = bound * f[0]; fn = clampd(fn, -lim, lim); }
        double df = fn - fo;
        f[k] = fn;
        sdf += fabs(df); sf += fabs(fn);
        if (df != 0.0) {
          changed = true;
          if (ba >= 0) { aa[0] += wa[k][0] * df; aa[1] += wa[k][1] * df; aa[2] += wa[k][2] * df; }
          if (bb >= 0) { ab[0] += wb[k][0] * df; ab[1] += wb[k][1] * df; ab[2] += wb[k][2] * df; }
        }
      }
      r.f[0] = f[0];
      if (nk == 2) r.f[1] = f[1];
      if (changed) {
        if (ba >= 0) { acc[ba][0] = aa[0]; acc[ba][1] = aa[1]; acc[ba][2] = aa[2]; }
        if (bb >= 0) { acc[bb][0] = ab[0]; acc[bb][1] = ab[1]; acc[bb][2] = ab[2]; }
      }
    }
    // floor-friction rows of every body in the table
    bool floors_done = false;
#if defined(__CUDA_ARCH__)
    if constexpr (Coop) {
      floors_done = true;
      __syncwarp();
      const int b = coop_lane();
      double tdf = 0.0, tf = 0.0;
      if (b < nb) floor_visit(b, tdf, tf);
      __syncwarp();
      for (int k = 0; k < nb; ++k) { sdf += __shfl_sync(kFullWarp, tdf, k); sf += __shfl_sync(kFullWarp, tf, k); }
    }
#endif
    if (!floors_done) {
#pragma unroll 1
      for (int b = 0; b < nb; ++b) {
        double tdf, tf;
        floor_visit(b, tdf, tf);
        sdf += tdf; sf += tf;
      }
    }
    if (sdf <= kPgsTol * sf) break;
  }
  if constexpr (Coop) SAG_CLKG(4, 2, S);
  P.qacc[0] = acc[0][0]; P.qacc[1] = acc[0][1]; P.qacc[2] = acc[0][2];
  for (int i = 0; i < nrow; ++i) {
    const Row& r = rows[i];
    int nk = RB::kGremlins ? r.nk : ((i == tendon_row) ? 1 : 2);
    for (int k = 0; k < nk; ++k) {
      if (r.ba == 0) for (int d = 0; d < 3; ++d) P.fc[d] += r.ja[k][d] * r.f[k];
      if (r.bb == 0) for (int d = 0; d < 3; ++d) P.fc[d] += r.jb[k][d] * r.f[k];
    }
    if (kCarRobot && r.type == 2) P.wtau[r.bb - kWheelBody] = r.jb[0][0] * r.f[0];
  }
  if (!integrate || overflow) return;
  // ---- semi-implicit Euler for the awake / touched movable bodies (free joints: no damping)
  if constexpr (Coop) {
#if defined(__CUDA_ARCH__)
    // one body per lane (read-modify-write of global state: must not be replicated); mov / err combined by ballots
    __syncwarp();
    const int b = coop_lane();
    bool moving = false, bad = false;
    int sb = 0;
    if (b < nb) {
      sb = S.bslot[b];
      size_t i = oix(C, sb);
      double vx = S.bv[b][0], vy = S.bv[b][1], w = S.bv[b][2];
      bool tch = (touched >> sb) & 1u;
      vx += h * acc[1 + b][0]; vy += h * acc[1 + b][1]; w += h * acc[1 + b][2];
      if (!tch && vx * vx + vy * vy < kSleepV * kSleepV && fabs(w) < kSleepV) { vx = vy = w = 0.0; }
      double x = C.O.x[i] + h * vx, y = C.O.y[i] + h * vy, yaw = C.O.yaw[i] + h * w;
      C.O.vx[i] = vx; C.O.vy[i] = vy; C.O.w[i] = w; C.O.x[i] = x; C.O.y[i] = y; C.O.yaw[i] = yaw;
      moving = vx != 0.0 || vy != 0.0 || w != 0.0;
      bad = bad_val(x) || bad_val(y) || bad_val(vx) || bad_val(vy) || bad_val(w);
    }
    const unsigned handled = __reduce_or_sync(kFullWarp, b < nb ? 1u << sb : 0u);
    const unsigned nowmov = __reduce_or_sync(kFullWarp, moving ? 1u << sb : 0u);
    P.mov = (P.mov & ~handled) | nowmov;
    S.scvalid &= ~handled;  // their yaw has changed (every lane stores the same word)
    if (__any_sync(kFullWarp, bad)) P.err = 1;
    __syncwarp();
    SAG_CLK(5);
#endif
  } else
  for (int b = 0; b < nb; ++b) {
    const int s = S.bslot[b];
    size_t i = oix(C, s);
    double vx = S.bv[b][0], vy = S.bv[b][1], w = S.bv[b][2];
    bool tch = (touched >> s) & 1u;
    vx += h * acc[1 + b][0]; vy += h * acc[1 + b][1]; w += h * acc[1 + b][2];
    if (!tch && vx * vx + vy * vy < kSleepV * kSleepV && fabs(w) < kSleepV) { vx = vy = w = 0.0; }
    double x = C.O.x[i] + h * vx, y = C.O.y[i] + h * vy, yaw = C.O.yaw[i] + h * w;
    C.O.vx[i] = vx; C.O.vy[i] = vy; C.O.w[i] = w; C.O.x[i] = x; C.O.y[i] = y; C.O.yaw[i] = yaw;
    if (vx != 0.0 || vy != 0.0 || w != 0.0) P.mov |= 1u << s; else P.mov &= ~(1u << s);
    if (bad_val(x) || bad_val(y) || bad_val(vx) || bad_val(vy) || bad_val(w)) P.err = 1;
  }
}

// Cheap exact pre-test run by every non-quiet lane in parallel: does any robot geom overlap any object geom?
// (same broad phase and first-stage arithmetic as contact_pass phase 1, so a `false` here means phase 1 lists nothing)
template <class RB>
SAG_HD bool robot_overlaps_any(const Ctx& C, const RB& R, double sn, double cs) {
  const Dev& D = C.D;
  for (int s = C.L.v0; s < C.L.n; ++s) {
    int kind = slot_kind(C.sp, C.L, s);
    if (!kind_collidable(kind)) continue;
    size_t i = oix(C, s);
    double x = C.O.x[i], y = C.O.y[i];
    double dx = x - R.q[0], dy = y - R.q[1], reach = RB::kReach + kind_bound(D, kind);
    if (dx * dx + dy * dy > reach * reach) continue;
    double oc = 1.0, os = 0.0;
    if (kind_movable(kind)) sag_sincos(C.O.yaw[i], &os, &oc);
    for (int pt = 0; pt < kind_nparts(kind); ++pt) {
      Geom go;
      obj_geom(D, kind, pt, x, y, oc, os, go);
      for (int rg = 0; rg < RB::kNGeom; ++rg) {
        Geom grg;
        R.geom(rg, sn, cs, grg);
        if (overlap(grg, go)) return true;
      }
    }
  }
  return false;
}

// The same pre-test restricted to candidate slots.  `cand` must contain every collidable slot whose centre can come within
// reach + bound of the robot during the step (near_candidates below); the others fail the broad test above anyway.
template <class RB>
SAG_HD bool robot_overlaps_masked(const Ctx& C, const RB& R, double sn, double cs, unsigned cand) {
  const Dev& D = C.D;
  for (unsigned m = cand; m; m &= m - 1) {
    const int s = ctz32(m);
    const int kind = slot_kind(C.sp, C.L, s);
    size_t i = oix(C, s);
    double x = C.O.x[i], y = C.O.y[i];
    double dx = x - R.q[0], dy = y - R.q[1], reach = RB::kReach + kind_bound(D, kind);
    if (dx * dx + dy * dy > reach * reach) continue;
    double oc = 1.0, os = 0.0;
    if (kind_movable(kind)) sag_sincos(C.O.yaw[i], &os, &oc);
    for (int pt = 0; pt < kind_nparts(kind); ++pt) {
      Geom go;
      obj_geom(D, kind, pt, x, y, oc, os, go);
      for (int rg = 0; rg < RB::kNGeom; ++rg) {
        Geom grg;
        R.geom(rg, sn, cs, grg);
        if (overlap(grg, go)) return true;
      }
    }
  }
  return false;
}
// collidable slots within reach + bound + travel of the robot at the start of a contact-free step: nothing moves but the
// robot, and it moves by less than `travel` (RB::travel_bound, conservative) before the step ends
template <class RB>
SAG_HD unsigned near_candidates(const Ctx& C, const RB& R, double travel) {
  const Dev& D = C.D;
  unsigned cand = 0;
  for (int s = C.L.v0; s < C.L.n; ++s) {
    const int kind = slot_kind(C.sp, C.L, s);
    if (!kind_collidable(kind)) continue;
    size_t i = oix(C, s);
    double dx = C.O.x[i] - R.q[0], dy = C.O.y[i] - R.q[1], reach = RB::kReach + kind_bound(D, kind) + travel;
    if (!(dx * dx + dy * dy > reach * reach)) cand |= 1u << s;
  }
  return cand;
}

// Contact path of a warp of the scalar (one thread = one environment) kernels: the lanes that need it take turns on the
// warp's Scratch.  `wmask` = lanes of this warp that own an environment (all of them call this together).  On the host
// there is a single lane.
template <class RB>
SAG_HD void warp_contact_pass(unsigned wmask, bool need, const Ctx& C, const RB& R, double sn, double cs, const PtConst& K,
                              const double* fs, unsigned mov, bool integrate, double h, Scratch* S, const SolveConsts& Q, Phys& P,
                              const double* mocap) {
#if defined(__CUDA_ARCH__)
  unsigned todo = __ballot_sync(wmask, need);
  const int lane = threadIdx.x & 31;
  while (todo) {
    const int turn = __ffs((int)todo) - 1;
    todo &= todo - 1;
    if (lane == turn) contact_pass<RB, false>(C, R, sn, cs, K, fs, mov, integrate, h, *S, Q, P, mocap);
    __syncwarp(wmask);
  }
#else
  (void)wmask;
  if (need) contact_pass<RB, false>(C, R, sn, cs, K, fs, mov, integrate, h, *S, Q, P, mocap);
#endif
}

// ------------------------------------------------------------------------------------------------
// lidar (safe_adaptation_gym.py:174-223): one object -> (bin, centre, next, previous) contributions.
// Bins live in the CTA's shared-memory observation tile (stride = tile row length).
// ------------------------------------------------------------------------------------------------
struct LidarHit { int bin; float s0, sp, sm; };

SAG_HD LidarHit lidar_eval(double wx, double wy, double cs, double sn) {
  double ex = SAG_FMA(wx, cs, wy * sn), ey = SAG_FMA(wy, cs, -(wx * sn));  // :197-202 ego frame
  double dist = sqrt(SAG_FMA(ex, ex, ey * ey));                             // :209
  int bin;
  double alias;
  sag_lidar_bin16(ex, ey, &bin, &alias);                                    // :210-213,216 (folded form, sag_detmath.h)
  double sensor = kLidarMax - dist;                                         // :214
  if (sensor < 0.0) sensor = 0.0;
  sensor *= 1.0 / kLidarMax;
  LidarHit H;
  H.bin = bin;
  H.s0 = (float)sensor; H.sp = (float)(alias * sensor); H.sm = (float)((1.0 - alias) * sensor);
  return H;
}
SAG_HD void lidar_apply(const LidarHit& H, float* bins, int bstride) {
  int b0 = H.bin & (kLidarBins - 1), bp = (H.bin + 1) & (kLidarBins - 1), bm = (H.bin + kLidarBins - 1) & (kLidarBins - 1);
#if defined(__CUDA_ARCH__)
  // bins live in shared memory: a max without return value instead of load / compare / store, so the thread does not
  // wait for the round trip.  Values are >= 0 or tiny negatives / -0 that must not be stored, and for those the signed
  // integer order of the float bits is the float order (bins start at +0).
  atomicMax(reinterpret_cast<int*>(bins + b0 * bstride), __float_as_int(H.s0));   // :215
  atomicMax(reinterpret_cast<int*>(bins + bp * bstride), __float_as_int(H.sp));   // :221
  atomicMax(reinterpret_cast<int*>(bins + bm * bstride), __float_as_int(H.sm));   // :222
#else
  if (H.s0 > bins[b0 * bstride]) bins[b0 * bstride] = H.s0;   // :215
  if (H.sp > bins[bp * bstride]) bins[bp * bstride] = H.sp;   // :221
  if (H.sm > bins[bm * bstride]) bins[bm * bstride] = H.sm;   // :222
#endif
}
SAG_HD void lidar_accum(double rx, double ry, double cs, double sn, double px, double py, float* bins, int bstride) {
  LidarHit H = lidar_eval(px - rx, py - ry, cs, sn);
  lidar_apply(H, bins, bstride);
}

// lidar group of a slot (consts.py:13-16; press_buttons.py:78-91; collect.py:34,44-45)
SAG_HD int slot_group(const Ctx& C, int s, int kind, int gbtn, int bstate, int amask) {
  if (kind == K_GOAL) return 2;
  if (kind == K_BUTTON) {
    int i = s - C.L.btn0;
    if (C.task == T_COLLECT) return ((amask >> i) & 1) ? 2 : 0;
    if (bstate == 0) return 0;
    return i == gbtn ? 2 : 3;
  }
  if (kind == K_BOX || kind == K_ROD || kind == K_BALL) return 3;
  return 1;
}

// sqrt(d2) < thr, evaluated exactly: the root is only taken when d2 is within 1e-6 (relative) of thr^2 -- outside that
// band the comparison of the squares decides, far beyond the rounding error of either side
SAG_HD bool sqrt_less(double d2, double thr) {
  const double lo = thr * 0.999999, hi = thr * 1.000001;
  if (d2 < lo * lo) return true;
  if (d2 > hi * hi) return false;
  return sqrt(d2) < thr;
}

// ------------------------------------------------------------------------------------------------
// goal resampling (go_to_goal.py:59-80): the rectangle grows x1.01 after every failed draw
// ------------------------------------------------------------------------------------------------
SAG_HD int resample_goal(const Ctx& C, const Rng& rng, uint32_t stream, uint32_t& ctr, double rx, double ry, double& gx, double& gy) {
  const Dev& D = C.D;
  double rect[4] = {-1.5, -1.5, 1.5, 1.5};
  for (int j = 0; j < 500000; ++j) {
    double u1, u2;
    rng.pair(stream, ctr++, u1, u2);
    double xmin = rect[0] + kGoalKeepout, ymin = rect[1] + kGoalKeepout, xmax = rect[2] - kGoalKeepout, ymax = rect[3] - kGoalKeepout;
    double x = xmin + (xmax - xmin) * u1, y = ymin + (ymax - ymin) * u2;
    bool valid = true;
    { double dx = x - rx, dy = y - ry; if (sqrt_less(dx * dx + dy * dy, D.robot_keepout + kGoalKeepout)) valid = false; }
    for (int s = 0; valid && s < C.L.n; ++s) {
      if (s == C.L.goal) continue;
      int kind = slot_kind(C.sp, C.L, s);
      double ko = kind == K_HAZARD ? D.k_hazard : kind == K_VASE ? D.k_vase : kind == K_GREMLIN ? D.k_gremlin
                : kind == K_PILLAR ? D.k_pillar : kind == K_BUTTON ? kButtonsKeepout : C.sp.box_keepout;
      size_t i = oix(C, s);
      double dx = x - C.O.x[i], dy = y - C.O.y[i];
      if (sqrt_less(dx * dx + dy * dy, ko + kGoalKeepout)) valid = false;
    }
    if (valid) { gx = x; gy = y; return 0; }
#pragma unroll
    for (int k = 0; k < 4; ++k) rect[k] = rect[k] * 1.01;
  }
  return 1;
}

SAG_HD double dist2d(double ax, double ay, double bx, double by) { double dx = ax - bx, dy = ay - by; return sqrt(dx * dx + dy * dy); }

// per-env task scalars kept in registers during a step
struct TaskState {
  double last0, last1;
  int gbtn, bstate, btimer, amask;
  double cgcur, cgnext, cgox, cgoy;
  int cgtimer;
  uint32_t ctr;
};

SAG_HD void load_task_state(const Dev& D, int e, TaskState& T) {
  T.last0 = D.last0[e]; T.last1 = D.last1[e];
  T.gbtn = D.gbtn[e]; T.bstate = D.bstate[e]; T.btimer = D.btimer[e]; T.amask = D.amask[e];
  T.cgcur = D.cgcur[e]; T.cgnext = D.cgnext[e]; T.cgox = D.cgox[e]; T.cgoy = D.cgoy[e]; T.cgtimer = D.cgtimer[e];
  T.ctr = D.ctr[e];
}
SAG_HD void store_task_state(const Dev& D, int e, const TaskState& T) {
  D.last0[e] = T.last0; D.last1[e] = T.last1;
  D.gbtn[e] = T.gbtn; D.bstate[e] = T.bstate; D.btimer[e] = T.btimer; D.amask[e] = T.amask;
  D.cgcur[e] = T.cgcur; D.cgnext[e] = T.cgnext; D.cgox[e] = T.cgox; D.cgoy[e] = T.cgoy; D.cgtimer[e] = T.cgtimer;
  D.ctr[e] = T.ctr;
}

template <class RB>
SAG_HD void sample_goal_button(const Ctx& C, const Rng& rng, uint32_t stream, uint32_t& ctr, const RB& R, TaskState& T) {
  double u1, u2;  // press_buttons.py:70-76
  rng.pair(stream, ctr++, u1, u2);
  int k = (int)(u1 * C.L.nbtn);
  if (k >= C.L.nbtn) k = C.L.nbtn - 1;
  T.gbtn = k;
  T.btimer = kButtonDelay;
  size_t i = oix(C, C.L.btn0 + k);
  T.last0 = dist2d(R.q[0], R.q[1], C.O.x[i], C.O.y[i]);
}

// task.reset(): go_to_goal.py:50-57, push_box.py:94-100, press_buttons.py:65-68, collect.py:41-47, catch_goal.py:36-40
template <class RB>
SAG_HD int task_reset(const Ctx& C, const Rng& rng, uint32_t stream, uint32_t& ctr, const RB& R, TaskState& T) {
  const Dev& D = C.D;
  if (C.sp.kind == 1) {
    if (C.task == T_COLLECT) T.amask = (1 << C.L.nbtn) - 1;
    else sample_goal_button(C, rng, stream, ctr, R, T);
    return 0;
  }
  double gx, gy;
  if (resample_goal(C, rng, stream, ctr, R.q[0], R.q[1], gx, gy)) return 1;
  size_t ig = oix(C, C.L.goal);
  C.O.x[ig] = gx; C.O.y[ig] = gy;
  T.last0 = dist2d(R.q[0], R.q[1], gx, gy);
  if (C.task == T_CATCH_GOAL) { T.cgox = gx; T.cgoy = gy; }
  if (C.sp.kind == 2) {
    size_t ib = oix(C, C.L.box);
    double bx = C.O.x[ib], by = C.O.y[ib];
    T.last1 = dist2d(gx, gy, bx, by);
    T.last0 = dist2d(R.q[0], R.q[1], bx, by);
  }
  return 0;
}

// task.compute_reward family (SURVEY Appendix C); touch = robot contact bitmask from the forward pass
template <class RB>
SAG_HD int compute_reward(const Ctx& C, const Rng& rng, const RB& R, TaskState& T, unsigned touch, double* reward) {
  const Dev& D = C.D;
  reward[0] = reward[1] = 0.0;
  if (C.sp.kind == 0) {  // go_to_goal.py:31-45
    size_t ig = oix(C, C.L.goal);
    double dx = R.q[0] - C.O.x[ig], dy = R.q[1] - C.O.y[ig], dz = kPtZ - kGoalZ;
    double distance = sqrt(dx * dx + dy * dy + dz * dz);
    double r = T.last0 - distance;
    if (C.task == T_GO_TO_GOAL_SCARCE) r = ((distance >= 0.0 && distance <= kGoalSize * 1.5) ? 1.0 : 0.0) * r;
    T.last0 = distance;
    if (distance <= kGoalSize) {
      if (task_reset(C, rng, 1u, T.ctr, R, T)) return 1;
      r += 1.0;
    }
    if (C.task == T_UNSUPERVISED) {  // unsupervised.py:48-67
      double cx, cy;
      R.com_offset(cx, cy);
      double cs = sag_cos(R.q[2]), sn = sag_sin(R.q[2]);
      double ox = cx * cs - cy * sn, oy = cx * sn + cy * cs;
      double x = R.q[0] + ox, y = R.q[1] + oy;
      double u = R.v[0] - R.v[2] * oy, v = R.v[1] + R.v[2] * ox;
      double radius = sqrt(x * x + y * y);
      reward[0] = (((-u * y + v * x) / radius) / (1.0 + fabs(radius - 1.5))) * 1e-1;
      reward[1] = r;
    } else reward[0] = r;
    return 0;
  }
  if (C.sp.kind == 1 && C.task == T_COLLECT) {  // collect.py:24-39
    if (!T.amask) T.amask = (1 << C.L.nbtn) - 1;
    for (int i = 0; i < C.L.nbtn; ++i) {
      if (!((T.amask >> i) & 1)) continue;
      if ((touch >> (C.L.btn0 + i)) & 1u) { reward[0] += 1.0; T.amask &= ~(1 << i); break; }
    }
    return 0;
  }
  if (C.sp.kind == 1) {  // press_buttons.py:42-63, press_buttons_scarce.py:22-55
    size_t ib = oix(C, C.L.btn0 + T.gbtn);
    double d = dist2d(R.q[0], R.q[1], C.O.x[ib], C.O.y[ib]);
    double r = C.task == T_PRESS_BUTTONS_SCARCE ? 0.0 : T.last0 - d;
    T.last0 = d;
    if ((touch >> (C.L.btn0 + T.gbtn)) & 1u) {
      r += 1.0;
      sample_goal_button(C, rng, 1u, T.ctr, R, T);
      T.bstate = 0;
    }
    if (T.bstate == 0) {
      if (T.btimer != 0) T.btimer = T.btimer - 1 > 0 ? T.btimer - 1 : 0;
      else { T.bstate = 1; T.btimer = kButtonDelay; }
    }
    reward[0] = r;
    return 0;
  }
  // push_box.py:74-92, push_box_scarce.py:22-50, haul_box.py:34-48
  size_t ig = oix(C, C.L.goal), ib = oix(C, C.L.box);
  double bx = C.O.x[ib], by = C.O.y[ib];
  double r = 0.0;
  if (C.task != T_HAUL_BOX) {
    double bd = dist2d(R.q[0], R.q[1], bx, by);
    double sh = T.last0 - bd;
    if (C.task == T_PUSH_BOX_SCARCE) sh = ((bd >= 0.0 && bd <= kGoalSize * 1.70) ? 1.0 : 0.0) * sh;
    r += sh;
    T.last0 = bd;
  }
  double bg = dist2d(bx, by, C.O.x[ig], C.O.y[ig]);
  r += T.last1 - bg;
  T.last1 = bg;
  if (bg <= kGoalSize) {
    if (task_reset(C, rng, 1u, T.ctr, R, T)) return 1;
    r += 1.0;
  }
  reward[0] = r;
  return 0;
}

// CatchGoal.set_mocaps, catch_goal.py:20-31
SAG_HD void set_mocaps(const Ctx& C, const Rng& rng, TaskState& T, double time) {
  if (C.task != T_CATCH_GOAL) return;
  T.cgtimer = T.cgtimer - 1 > 0 ? T.cgtimer - 1 : 0;
  if (T.cgtimer == 0) {
    T.cgcur = T.cgnext;
    double u1, u2;
    rng.pair(1u, T.ctr++, u1, u2);
    T.cgnext = 0.2 + (1.0 - 0.2) * u1;
    T.cgtimer = 10;
  }
  double progress = (10 - T.cgtimer) / 10.0;
  double radius = progress * (T.cgnext - T.cgcur) + T.cgcur;
  size_t ig = oix(C, C.L.goal);
  C.O.x[ig] = T.cgox + sag_sin(time) * radius;
  C.O.y[ig] = T.cgoy + sag_cos(time) * radius;
}

// ------------------------------------------------------------------------------------------------
// end-of-step: forward() (contacts, qacc) -> reward -> cost -> observation, fused into two passes over the
// objects (obstacle kinds before the reward, task objects after it because the reward may move the goal or
// change button groups).  obs_s: this env's column of the CTA's shared-memory tile (stride ostride).
// ------------------------------------------------------------------------------------------------
struct EndOut { double rew[2]; double cost; double clear; unsigned mov, touch; int err; int resample_failed; int bail; };

SAG_HD bool hazard_hit(double d2, double size) {  // world.py:151-152: ||robot_xy - hazard_xy|| <= size, exactly
  double lo = size * 0.999, hi = size * 1.001;
  if (d2 > hi * hi) return false;
  if (d2 < lo * lo) return true;
  return sqrt(d2) <= size;
}

#if defined(__CUDA_ARCH__)
__device__ __forceinline__ double coop_min(double v) {
#pragma unroll
  for (int d = 16; d; d >>= 1) v = fmin(v, __shfl_xor_sync(kFullWarp, v, d));
  return v;
}
// max into a shared-memory bin; lidar values are >= 0 or tiny negatives / -0 that must not be stored, and for those
// the signed-integer order of the float bits is the float order
__device__ __forceinline__ void coop_lidar_apply(const LidarHit& H, float* bins, int bstride) {
  int b0 = H.bin & (kLidarBins - 1), bp = (H.bin + 1) & (kLidarBins - 1), bm = (H.bin + kLidarBins - 1) & (kLidarBins - 1);
  atomicMax(reinterpret_cast<int*>(bins + b0 * bstride), __float_as_int(H.s0));
  atomicMax(reinterpret_cast<int*>(bins + bp * bstride), __float_as_int(H.sp));
  atomicMax(reinterpret_cast<int*>(bins + bm * bstride), __float_as_int(H.sm));
}
// pass A of end_of_step with one object per lane: obstacle lidar (Obs), hazard flag, min squared distances per kind
template <class RB, bool Obs = true>
__device__ __forceinline__ void pass_a_coop(const Ctx& C, const RB& R, double cs, double sn, float* obs_s, int ostride, bool& hz,
                                            double& d2v, double& d2p, double& d2b, double& d2x) {
  const Dev& D = C.D;
  const int s = coop_lane();
  __syncwarp();  // the zeroed bins are visible
  bool hzl = false;
  double lv = 1e300, lp = 1e300, lb = 1e300, lx = 1e300;
  if (s < C.L.n) {
    size_t i = oix(C, s);
    double wx = C.O.x[i] - R.q[0], wy = C.O.y[i] - R.q[1];
    double d2 = wx * wx + wy * wy;
    if (s < C.L.t0) {
      if (s < C.L.v0) hzl = hazard_hit(d2, D.hazards_size);
      else if (s < C.L.p0) lv = d2;
      else lp = d2;
      if constexpr (Obs) coop_lidar_apply(lidar_eval(wx, wy, cs, sn), obs_s, ostride);
    } else {
      int kind = slot_kind(C.sp, C.L, s);
      if (kind_collidable(kind)) { if (kind == K_BUTTON) lb = d2; else lx = d2; }
    }
  }
  hz = __any_sync(kFullWarp, hzl);
  d2v = coop_min(lv); d2p = coop_min(lp); d2b = coop_min(lb); d2x = coop_min(lx);
  __syncwarp();
}
#endif

// Obs = false (sag_evaluate_actions' steps before the last): no observation.  obs_s is not touched -- no zeroing, no
// lidar, no pass B, no sensors -- and everything that feeds the state, the reward, the cost or the clearance is computed
// as with Obs = true, in the same order.
template <int Mode, class RB, bool Obs = true>
SAG_HD void end_of_step(unsigned wmask, Scratch* S, const SolveConsts& Q, const Ctx& C, const RB& R, TaskState& T, const Rng& rng, const PtConst& K,
                        unsigned mov, bool phys_err, const double* qacc_err, bool with_reward, float* obs_s, int ostride, EndOut& O,
                        const Phys* Pfwd = nullptr, unsigned cand = 0xffffffffu, const double* mocap = nullptr) {
  constexpr bool Coop = Mode == kStepCoop, Near = Mode == kStepNear;
  const Dev& D = C.D;
  const int e = C.e;
  O.bail = 0;
  SAG_CLK_DECL;
  double sn, cs;
  sag_sincos(R.q[2], &sn, &cs);
  if constexpr (Obs) for (int k = 0; k < 48; ++k) obs_s[k * ostride] = 0.0f;
  // ---- pass A: hazards / vases / gremlins / pillars -> obstacle lidar, hazard cost, clearance
  bool hz = false;
  double d2v = 1e300, d2p = 1e300, d2b = 1e300, d2x = 1e300;  // min squared centre distance per collidable kind
  if constexpr (Coop) {
#if defined(__CUDA_ARCH__)
    pass_a_coop<RB, Obs>(C, R, cs, sn, obs_s, ostride, hz, d2v, d2p, d2b, d2x);
#endif
  } else {
  if constexpr (!Obs) {  // the distances and the hazard flag alone
    for (int s = 0; s < C.L.t0; ++s) {
      size_t i = oix(C, s);
      double wx = C.O.x[i] - R.q[0], wy = C.O.y[i] - R.q[1];
      double d2 = wx * wx + wy * wy;
      if (s < C.L.v0) hz = hz || hazard_hit(d2, D.hazards_size);
      else if (s < C.L.p0) { if (d2 < d2v) d2v = d2; }
      else { if (d2 < d2p) d2p = d2; }
    }
  } else
  // obstacle slots [0, t0) in trips of three: loads and the sqrt / atan2 chains of a trip are independent, the
  // shared-memory bin updates come last (the compiler has to keep those in order)
  for (int s0 = 0; s0 < C.L.t0; s0 += 3) {
    double wx[3], wy[3];
    bool on[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      int s = s0 + k;
      on[k] = s < C.L.t0;
      size_t i = oix(C, on[k] ? s : s0);
      wx[k] = C.O.x[i] - R.q[0]; wy[k] = C.O.y[i] - R.q[1];
    }
    LidarHit H[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) H[k] = lidar_eval(wx[k], wy[k], cs, sn);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      if (!on[k]) continue;
      int s = s0 + k;
      double d2 = wx[k] * wx[k] + wy[k] * wy[k];
      if (s < C.L.v0) hz = hz || hazard_hit(d2, D.hazards_size);
      else if (s < C.L.p0) { if (d2 < d2v) d2v = d2; }
      else { if (d2 < d2p) d2p = d2; }
      lidar_apply(H[k], obs_s, ostride);
    }
  }
  for (int s = C.L.t0; s < C.L.n; ++s) {  // collidable task objects: buttons, push box
    int kind = slot_kind(C.sp, C.L, s);
    if (!kind_collidable(kind)) continue;
    size_t i = oix(C, s);
    double wx = C.O.x[i] - R.q[0], wy = C.O.y[i] - R.q[1];
    double d2 = wx * wx + wy * wy;
    if (kind == K_BUTTON) { if (d2 < d2b) d2b = d2; } else { if (d2 < d2x) d2x = d2; }
  }
  }
  double clear = 1e30;
  if (d2v < 1e299) clear = fmin(clear, sqrt(d2v) - (RB::kReach + kind_bound(D, K_VASE)));
  if (d2p < 1e299) clear = fmin(clear, sqrt(d2p) - (RB::kReach + kind_bound(D, K_PILLAR)));
  if (d2b < 1e299) clear = fmin(clear, sqrt(d2b) - (RB::kReach + kind_bound(D, K_BUTTON)));
  if (d2x < 1e299) clear = fmin(clear, sqrt(d2x) - (RB::kReach + kind_bound(D, C.sp.box_kind)));
  // HaulBox: the tendon's slack bounds the clearance too (a slack tendon adds no constraint row: haul_box.py:21-30)
  bool taut = false;
  if (C.task == T_HAUL_BOX) {
    double tdx, tdy, tlen, tdist;
    taut = tendon_taut(C, R, tdx, tdy, tlen, tdist);
    clear = fmin(clear, tdist);
  }
  // ---- forward(): contacts + acceleration at the final state (safe_adaptation_gym.py:76)
  double fs[3], qacc[3];
  R.smooth(sn, cs, fs);
  unsigned touch = 0;
  O.err = 0;
  Phys P;
  P.err = 0; P.touch = 0;
  bool need = false;
  if constexpr (Near) {  // forward() at the final state would list a contact: not a contact-free step after all
    if (!(clear > 0.0) && (taut || robot_overlaps_masked(C, R, sn, cs, cand))) { O.bail = 1; return; }
  }
  // A PhysicsError in physics.step returns the observation at once (safe_adaptation_gym.py:73-75): no forward(), the
  // accelerometer shows the last substep's acceleration, no reward / cost evaluation.
  const bool skip_forward = phys_err && qacc_err != nullptr;
  if (Pfwd) {  // cooperative kernel: the forward pass has been evaluated as the last trip of env_step's pass loop
    P = *Pfwd;
  } else {
  if (!Near && !skip_forward) {  // (a quiet step ends with positive clearance: no contact is possible)
    const bool always = RB::kGremlins && C.sp.ng > 0;  // a welded gremlin is a constraint row in every pass
    const bool near_ = !(clear > 0.0 && mov == 0) || always;
    if constexpr (Coop) {
#if defined(__CUDA_ARCH__)
      need = near_ && (always || mov != 0 || taut || robot_overlaps_any_coop(C, R, sn, cs));
#endif
    } else {
      need = near_ && (always || mov != 0 || taut || robot_overlaps_any(C, R, sn, cs));
    }
  }
  if (skip_forward) {
    P.qacc[0] = qacc_err[0]; P.qacc[1] = qacc_err[1]; P.qacc[2] = qacc_err[2];
  } else if (!need) {
    if constexpr (RB::kKind == 1) { CarFree F; car_free_solve(R, sn, cs, K, fs, F); P.qacc[0] = F.qacc[0]; P.qacc[1] = F.qacc[1]; P.qacc[2] = F.qacc[2]; }
    else { double p, q; R.pq(sn, cs, p, q); pt_solve(p, q, K.ia0, K.is0, fs, P.qacc); }
  }
  if constexpr (Coop) {
    SAG_CLK(7);
    if (need) contact_pass<RB, true>(C, R, sn, cs, K, fs, mov, false, 0.0, *S, Q, P, mocap);
    SAG_CLK_RESET;
  } else if (!Near) {
    warp_contact_pass(wmask, need, C, R, sn, cs, K, fs, mov, false, 0.0, S, Q, P, mocap);
  }
  }
  qacc[0] = P.qacc[0]; qacc[1] = P.qacc[1]; qacc[2] = P.qacc[2];
  touch = P.touch;
  O.err = P.err;
  if (mov != 0 || (RB::kGremlins && C.sp.ng > 0)) clear = -1.0;
  O.clear = clear;
  O.mov = mov;
  O.touch = touch;
  // ---- reward (may resample the goal / change button groups) and cost
  O.rew[0] = O.rew[1] = 0.0; O.cost = 0.0; O.resample_failed = 0;
  if (with_reward) {
    if (phys_err) { O.rew[0] = -10.0; }                                     // :73-75 (an error raised by forward() itself,
                                                                            // O.err, is sticky and takes this path next step)
    else {
      if (compute_reward(C, rng, R, T, touch, O.rew)) O.resample_failed = 1;  // :77
      unsigned obstacle_mask = C.L.t0 >= 32 ? 0xffffffffu : ((1u << C.L.t0) - 1u);
      O.cost = (hz || (touch & obstacle_mask)) ? 1.0 : 0.0;                  // :78, world.py:144-155
    }
  }
  if constexpr (!Obs) {
    if constexpr (Coop) SAG_CLK(9);
    return;
  }
  // ---- pass B: task objects -> objects / goal lidar (safe_adaptation_gym.py:133-139, world.py:219-231)
  if constexpr (Coop) {
#if defined(__CUDA_ARCH__)
    __syncwarp();
    const int s = C.L.t0 + coop_lane();
    if (s < C.L.n) {
      int kind = slot_kind(C.sp, C.L, s);
      int g = slot_group(C, s, kind, T.gbtn, T.bstate, T.amask);
      if (g != 0) {
        size_t i = oix(C, s);
        int off = g == 1 ? 0 : (g == 3 ? 16 : 32);
        coop_lidar_apply(lidar_eval(C.O.x[i] - R.q[0], C.O.y[i] - R.q[1], cs, sn), obs_s + off * ostride, ostride);
      }
    }
    __syncwarp();
#endif
  } else
  for (int s = C.L.t0; s < C.L.n; ++s) {
    int kind = slot_kind(C.sp, C.L, s);
    int g = slot_group(C, s, kind, T.gbtn, T.bstate, T.amask);
    if (g == 0) continue;
    size_t i = oix(C, s);
    int off = g == 1 ? 0 : (g == 3 ? 16 : 32);
    lidar_apply(lidar_eval(C.O.x[i] - R.q[0], C.O.y[i] - R.q[1], cs, sn), obs_s + off * ostride, ostride);
  }
  // ---- sensors (safe_adaptation_gym.py:225-237; semantics SURVEY App. B.6 [EXT])
  float* o = obs_s + 48 * ostride;
  o[0 * ostride] = (float)(qacc[0] * cs + qacc[1] * sn);    // accelerometer
  o[1 * ostride] = (float)(-qacc[0] * sn + qacc[1] * cs);
  o[2 * ostride] = (float)kGrav;
  o[3 * ostride] = (float)(R.v[0] * cs + R.v[1] * sn);      // velocimeter
  o[4 * ostride] = (float)(-R.v[0] * sn + R.v[1] * cs);
  o[5 * ostride] = 0.0f;
  o[6 * ostride] = 0.0f; o[7 * ostride] = 0.0f; o[8 * ostride] = (float)R.v[2];  // gyro
  o[9 * ostride] = (float)(-0.5 * sn); o[10 * ostride] = (float)(-0.5 * cs); o[11 * ostride] = 0.0f;  // magnetometer
  if constexpr (RB::kKind == 1) {  // ballangvel_rear (3), quat2mat(ballquat_rear).ravel() (9): safe_adaptation_gym.py:228-236
    double wc[3];
    R.castor_angvel(sn, cs, wc);
    o[12 * ostride] = (float)wc[0]; o[13 * ostride] = (float)wc[1]; o[14 * ostride] = (float)wc[2];
    const double w = R.cq[0], x = R.cq[1], y = R.cq[2], z = R.cq[3];
    o[15 * ostride] = (float)(w * w + x * x - y * y - z * z); o[16 * ostride] = (float)(2.0 * (x * y - w * z)); o[17 * ostride] = (float)(2.0 * (x * z + w * y));
    o[18 * ostride] = (float)(2.0 * (x * y + w * z)); o[19 * ostride] = (float)(w * w - x * x + y * y - z * z); o[20 * ostride] = (float)(2.0 * (y * z - w * x));
    o[21 * ostride] = (float)(2.0 * (x * z - w * y)); o[22 * ostride] = (float)(2.0 * (y * z + w * x)); o[23 * ostride] = (float)(w * w - x * x - y * y + z * z);
  }
  if constexpr (Coop) SAG_CLK(9);
}

template <class RB>
SAG_HD void load_robot(const Dev& D, int e, const TaskSpec& sp, RB& R) {
  R.q[0] = D.rx[e]; R.q[1] = D.ry[e]; R.q[2] = D.ryaw[e];
  R.v[0] = D.rvx[e]; R.v[1] = D.rvy[e]; R.v[2] = D.rw[e];
  R.ctrl[0] = D.ctrl0[e]; R.ctrl[1] = D.ctrl1[e];
  R.damp_xy = sp.damp_xy; R.gear_x = sp.gear_x;
  if constexpr (RB::kKind == 1) {
    R.wheel[0] = D.rext[e]; R.wheel[1] = D.rext[(size_t)D.stride + e];
    for (int k = 0; k < 4; ++k) R.cq[k] = D.rext[(size_t)(2 + k) * D.stride + e];
  }
}
template <class RB>
SAG_HD void store_robot(const Dev& D, int e, const RB& R) {
  D.rx[e] = R.q[0]; D.ry[e] = R.q[1]; D.ryaw[e] = R.q[2];
  D.rvx[e] = R.v[0]; D.rvy[e] = R.v[1]; D.rw[e] = R.v[2];
  D.ctrl0[e] = R.ctrl[0]; D.ctrl1[e] = R.ctrl[1];
  if constexpr (RB::kKind == 1) {
    D.rext[e] = R.wheel[0]; D.rext[(size_t)D.stride + e] = R.wheel[1];
    for (int k = 0; k < 4; ++k) D.rext[(size_t)(2 + k) * D.stride + e] = R.cq[k];
  }
}

// "Quiet" environment: nothing can come within reach of the robot during the coming step and nothing is moving
// (clearance cached by the previous end-of-step pass; -1 when a body moves or a tendon exists).  The bound on the
// travel of the hinge point during one step is conservative (DESIGN.md 5).
template <class RB>
SAG_HD bool env_is_quiet(double clear, const RB& R) { return clear > R.travel_bound(); }

// ------------------------------------------------------------------------------------------------
// SafeAdaptationGym.step for one environment (safe_adaptation_gym.py:56-83)
// ------------------------------------------------------------------------------------------------
// Obs = false: the step without its observation (end_of_step); obs_s is not touched
template <int Mode, class RB, bool Obs = true>
SAG_HD int env_step(unsigned wmask, Scratch* S, const Dev& D, int e, float a0, float a1, float* obs_s, int ostride, double* reward2,
                     unsigned char* cost, unsigned char* done, bool pretest = true) {
  constexpr bool Coop = Mode == kStepCoop, Near = Mode == kStepNear;
  SAG_CLK_DECL;
  Ctx C = {D, e, spec_for(D, D.task[e], RB::kGremlins, RB::kCustom), Slots(), logic_task(D, D.task[e], RB::kCustom),
           global_objects(D, e)};
  C.L = make_slots(C.sp);
#if defined(__CUDA_ARCH__)
  if constexpr (Coop) {  // stage the object arrays in the warp's working set, one slot per lane; written back at the end
    const int s = coop_lane();
    if (s < C.L.n) {
      const size_t i = oix(C, s);
      S->obj[0][s] = C.O.x[i]; S->obj[1][s] = C.O.y[i]; S->obj[2][s] = C.O.yaw[i];
      S->obj[3][s] = C.O.vx[i]; S->obj[4][s] = C.O.vy[i]; S->obj[5][s] = C.O.w[i];
    }
    C.O.x = S->obj[0]; C.O.y = S->obj[1]; C.O.yaw = S->obj[2]; C.O.vx = S->obj[3]; C.O.vy = S->obj[4]; C.O.w = S->obj[5];
    C.O.stride = 1;
    S->scvalid = 0u;
    __syncwarp();
  }
#endif
  RB R;
  load_robot(D, e, C.sp, R);
  TaskState T;
  load_task_state(D, e, T);
  Rng rng = {rng_key(D), D.gid_base + (uint32_t)e, D.episode[e]};
  double time = D.time[e];
  unsigned mov = (unsigned)D.movmask[e];
  const double h = RB::kH;
  const PtConst K = R.consts(h);
  // constants of the contact solver: the cooperative kernel keeps them in the warp's shared-memory working set (every
  // lane writes the same values), the scalar path in registers / local memory; the contact-free modes need none
  SolveConsts Qloc;
  if constexpr (Mode == kStepFull) solve_consts(D, C.sp, Qloc, RB::kGremlins);
  if constexpr (Coop) solve_consts(D, C.sp, S->Q, RB::kGremlins);
  const SolveConsts& Q = Coop ? S->Q : Qloc;
  const bool tendon_task = C.task == T_HAUL_BOX;
  unsigned cand = 0;  // contact-free modes with pre-tests: the slots the robot can reach during this step
  if constexpr (Near) { if (pretest) cand = near_candidates(C, R, R.travel_bound()); }
  // action noise + clip (:58-67)
  double act0 = (double)a0, act1 = (double)a1;
  if (D.action_noise != 0.0) {
    double u1, u2;
    rng.pair(1u, T.ctr++, u1, u2);
    double rad = sqrt(-2.0 * sag_log(1.0 - u1));
    double ns, nc;
    sag_sincos(kTwoPi * u2, &ns, &nc);
    act0 += D.action_noise * (rad * nc);
    act1 += D.action_noise * (rad * ns);
  }
  // np.clip = min(max(a, lo), hi) (:66-67), then MuJoCo's ctrl clamp; they differ only for an inverted range, which a
  // Cauchy-scaled ctrlrange can be (world.py:72-73, mujoco_bridge.py:164-166).  Uniform branch: off in World.DEFAULT.
  if (D.ctrl_range_scale != 0.0) {
    const double sc0 = D.cscale0[e], sc1 = D.cscale1[e];
    const double lo0 = -1.0 * sc0, hi0 = 1.0 * sc0, lo1 = -1.0 * sc1, hi1 = 1.0 * sc1;
    double t0 = act0 > lo0 ? act0 : lo0, t1 = act1 > lo1 ? act1 : lo1;
    t0 = t0 < hi0 ? t0 : hi0; t1 = t1 < hi1 ? t1 : hi1;
    R.ctrl[0] = clampd(t0, lo0, hi0);
    R.ctrl[1] = clampd(t1, lo1, hi1);
  } else {
    R.ctrl[0] = clampd(act0, -1.0, 1.0);
    R.ctrl[1] = clampd(act1, -1.0, 1.0);
  }
  set_mocaps(C, rng, T, time);  // :71
  // World.set_mocaps (world.py:157-165): every gremlin's mocap body goes to travel * (sin t, cos t).  The first substep of
  // physics.step still sees the position of the previous kinematics pass (SURVEY App. B.1); from the second on, the new one.
  const bool gremlins = RB::kGremlins && C.sp.ng > 0;
  double moc_old[2] = {0.0, 0.0}, moc_new[2] = {0.0, 0.0};
  if (gremlins) {
    moc_old[0] = D.grem[e]; moc_old[1] = D.grem[(size_t)D.stride + e];
    moc_new[0] = sag_sin(time) * D.gremlins_travel; moc_new[1] = sag_cos(time) * D.gremlins_travel;
  }
  // physics.step(nstep) (:72).  "Quiet" envs (nothing within reach for the whole step, nothing moving) skip
  // contact detection; the bound on the hinge point's travel is conservative (DESIGN.md 5).
  unsigned char fl = D.flags[e];
  int err = (fl & F_PHYS_ERROR) ? 1 : 0;  // a physics error is sticky until the env is reset
  const bool quiet = Near ? true : env_is_quiet(D.clear[e], R);  // (gremlin environments keep clear = -1)
  (void)Coop;
  SAG_PROF(e, 7, quiet ? 0 : 1);
  double qacc_err[3] = {0.0, 0.0, 0.0};
  if constexpr (Coop) SAG_CLK(0);
  // Cooperative kernel: the final forward() (safe_adaptation_gym.py:76) runs as one more trip of this loop -- without
  // integration -- so that the contact pass has a single call site and is inlined there.  Its `need` is the one
  // end_of_step would compute: clear > 0 (nothing within reach, tendon slack) implies no overlap and a slack tendon.
  Phys Pfwd;
  Pfwd.qacc[0] = Pfwd.qacc[1] = Pfwd.qacc[2] = 0.0; Pfwd.touch = 0; Pfwd.err = 0; Pfwd.mov = mov;
  constexpr int kTrips = Coop ? RB::kNsub + 1 : RB::kNsub;
#pragma unroll 1
  for (int k = 0; k < kTrips; ++k) {
#if defined(__CUDA_ARCH__)
    if constexpr (Coop) coop_align();
#endif
    const bool fwd = Coop && k == RB::kNsub;
    if (fwd && err) { Pfwd.qacc[0] = qacc_err[0]; Pfwd.qacc[1] = qacc_err[1]; Pfwd.qacc[2] = qacc_err[2]; break; }  // :73-75, no forward()
    double sn, cs, fs[3], fc[3] = {0.0, 0.0, 0.0}, wtau[2] = {0.0, 0.0}, rhs[3], a[3], p, q;
    sag_sincos(R.q[2], &sn, &cs);
    R.pq(sn, cs, p, q);
    R.smooth(sn, cs, fs);
    bool need = false;
    bool taut = false;
    if (tendon_task && (fwd || (Near ? pretest : !quiet))) {
      double tdx, tdy, tlen, tdist;
      taut = tendon_taut(C, R, tdx, tdy, tlen, tdist);
    }
    if constexpr (Coop) {
#if defined(__CUDA_ARCH__)
      need = (fwd || !quiet) && (gremlins || mov != 0 || taut || robot_overlaps_any_coop(C, R, sn, cs));
#endif
    } else if (!Near) {
      need = !quiet && (gremlins || mov != 0 || taut || robot_overlaps_any(C, R, sn, cs));
    }
    if constexpr (Near) {
      if (pretest && (taut || robot_overlaps_masked(C, R, sn, cs, cand))) return 1;
    }
    SAG_PROF(e, 3, need ? 1 : 0);
    double subq[3] = {0.0, 0.0, 0.0};  // this substep's forward-dynamics acceleration, if a solve produced one
    if constexpr (RB::kKind == 1) {  // car: the wheel-floor friction rows are always there
      if (!need) {
        CarFree F;
        car_free_solve(R, sn, cs, K, fs, F);
        fc[0] = F.fc[0]; fc[1] = F.fc[1]; fc[2] = F.fc[2]; wtau[0] = F.wtau[0]; wtau[1] = F.wtau[1];
        subq[0] = F.qacc[0]; subq[1] = F.qacc[1]; subq[2] = F.qacc[2];
      }
    }
    if (!Near) {
      Phys P;
      P.fc[0] = fc[0]; P.fc[1] = fc[1]; P.fc[2] = fc[2]; P.wtau[0] = wtau[0]; P.wtau[1] = wtau[1];
      P.mov = mov; P.err = 0;
      if constexpr (Coop) {
        SAG_CLK(1);
        if (need) contact_pass_body<RB, true>(C, R, sn, cs, K, fs, mov, !fwd, h, *S, Q, P, k == 0 ? moc_old : moc_new);
        SAG_CLK_RESET;
        if (fwd) {  // forward(): acceleration + contacts at the final state, nothing is integrated
          if (need) { Pfwd = P; }
          else {
            if (RB::kKind == 1) { Pfwd.qacc[0] = subq[0]; Pfwd.qacc[1] = subq[1]; Pfwd.qacc[2] = subq[2]; }
            else pt_solve(p, q, K.ia0, K.is0, fs, Pfwd.qacc);
            Pfwd.touch = 0; Pfwd.err = 0;
          }
          break;
        }
      } else {
        warp_contact_pass(wmask, need, C, R, sn, cs, K, fs, mov, true, h, S, Q, P, k == 0 ? moc_old : moc_new);
      }
      fc[0] = P.fc[0]; fc[1] = P.fc[1]; fc[2] = P.fc[2]; wtau[0] = P.wtau[0]; wtau[1] = P.wtau[1];
      mov = P.mov;
      if (P.err) err = 1;
      if (need) { subq[0] = P.qacc[0]; subq[1] = P.qacc[1]; subq[2] = P.qacc[2]; }
    }
    rhs[0] = fs[0] + fc[0]; rhs[1] = fs[1] + fc[1]; rhs[2] = fs[2] + fc[2];
    pt_solve(p, q, K.iah, K.ish, rhs, a);   // (M + hD) a = f: implicit joint damping
#pragma unroll
    for (int d = 0; d < 3; ++d) R.v[d] += h * a[d];
#pragma unroll
    for (int d = 0; d < 3; ++d) R.q[d] += h * R.v[d];
    if constexpr (RB::kKind == 1) {  // wheels (implicit joint damping) and castor quaternion (mju_quatIntegrate [EXT])
      for (int i = 0; i < 2; ++i) {
        double al = (R.wheel_smooth(i) + wtau[i]) / (kCar.Iw + h * kCarWheelDamp);
        R.wheel[i] += h * al;
        if (bad_val(R.wheel[i])) err = 1;
      }
      double sn2, cs2, wc[3];
      sag_sincos(R.q[2], &sn2, &cs2);
      R.castor_angvel(sn2, cs2, wc);
      double wn = sqrt(wc[0] * wc[0] + wc[1] * wc[1] + wc[2] * wc[2]);
      if (wn > 0.0) {
        double sh, ch;
        sag_sincos(0.5 * h * wn, &sh, &ch);
        double ax = wc[0] / wn * sh, ay = wc[1] / wn * sh, az = wc[2] / wn * sh;
        double qa = R.cq[0], qb = R.cq[1], qc = R.cq[2], qd = R.cq[3];
        double q0 = qa * ch - qb * ax - qc * ay - qd * az;
        double q1 = qa * ax + qb * ch + qc * az - qd * ay;
        double q2 = qa * ay - qb * az + qc * ch + qd * ax;
        double q3 = qa * az + qb * ay - qc * ax + qd * ch;
        double nq = sqrt(q0 * q0 + q1 * q1 + q2 * q2 + q3 * q3);
        R.cq[0] = q0 / nq; R.cq[1] = q1 / nq; R.cq[2] = q2 / nq; R.cq[3] = q3 / nq;
      }
    }
#pragma unroll
    for (int d = 0; d < 3; ++d) if (bad_val(R.q[d]) || bad_val(R.v[d]) || bad_val(a[d])) err = 1;
    if (err) {  // PhysicsError: the observation will show the acceleration of the last forward-dynamics pass of step()
      if (RB::kKind == 0 && !need) pt_solve(p, q, K.ia0, K.is0, fs, subq);
      qacc_err[0] = subq[0]; qacc_err[1] = subq[1]; qacc_err[2] = subq[2];
    }
    time += h;
    if constexpr (Coop) SAG_CLK(6);
  }
  EndOut O;
  end_of_step<Mode, RB, Obs>(wmask, S, Q, C, R, T, rng, K, mov, err != 0, qacc_err, true, obs_s, ostride, O, Coop ? &Pfwd : nullptr, cand, moc_new);
  if constexpr (Coop) SAG_CLK_RESET;
  if constexpr (Near) { if (O.bail) return 1; }
  unsigned char dn = 0;
  if (err) { dn = 1; fl |= F_PHYS_ERROR; }
  if (O.err) fl |= F_PHYS_ERROR;
  if (O.resample_failed) { fl |= F_RESAMPLE_FAILED; D.errflags[0] = 1; }
  // bookkeeping (cooperative mode: read-modify-write of global state by one lane only)
  bool writer = true;
#if defined(__CUDA_ARCH__)
  if constexpr (Coop) {
    __syncwarp();
    writer = coop_lane() == 0;
    const int s = coop_lane();  // objects back to global memory (hazards never change)
    if (s >= C.L.v0 && s < C.L.n) {
      const ObjView G = global_objects(D, e);
      const size_t i = (size_t)s * G.stride;
      G.x[i] = S->obj[0][s]; G.y[i] = S->obj[1][s]; G.yaw[i] = S->obj[2][s];
      G.vx[i] = S->obj[3][s]; G.vy[i] = S->obj[4][s]; G.w[i] = S->obj[5][s];
    }
  }
#endif
  if (writer) {
    int ns = D.nstep[e] + 1;
    if (D.max_episode_steps > 0 && ns >= D.max_episode_steps) fl |= F_NEEDS_RESET;
    if (dn) fl |= F_NEEDS_RESET;
    D.nstep[e] = ns;
    D.epret[e] += O.rew[0];
    D.epcost[e] += O.cost;
    D.flags[e] = fl;
    D.time[e] = time;
    D.clear[e] = O.clear;
    D.movmask[e] = (int)O.mov;
    if (gremlins) { D.grem[e] = moc_new[0]; D.grem[(size_t)D.stride + e] = moc_new[1]; }
    store_robot(D, e, R);
    store_task_state(D, e, T);
  }
  reward2[0] = O.rew[0]; reward2[1] = O.rew[1];
  *cost = (unsigned char)(O.cost > 0.0);
  *done = dn;
  if constexpr (Coop) SAG_CLK(10);
  return 0;
}

// ------------------------------------------------------------------------------------------------
// sag_evaluate_actions: return, cost and length over a horizon of H steps, accumulated by the step kernels where a step
// stores reward / cost / done.  Every environment is finished by exactly one kernel per step, so nothing races.
//   L_e = min(H, 1 + first step that reported done); ret += w_h r_h and cost += w_h c_h for h < L_e, each product
//   rounded before the sum (no FMA), in step order.
// Step 0 writes the accumulators (0 + w_0 r_0: a sum that starts at zero) instead of reading them, so no memset is
// needed.  While an environment still counts, its length holds minus the steps counted so far; a done, or the last
// step, stores the final (positive) length.
// ------------------------------------------------------------------------------------------------
struct EvalAcc {
  double* ret;      // [n] or [n][2] (Unsupervised's pair)
  double* cost;     // [n]
  int32_t* length;  // [n]
  double w;         // this step's weight
  int cols, first, last;
};

SAG_HD double mul_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  return a * b;  // (the host build has -ffp-contract=off)
#endif
}
SAG_HD double add_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}

SAG_HD void eval_accumulate(const EvalAcc& A, int e, const double* rew, unsigned char c, unsigned char d) {
  if (!A.first && A.length[e] >= 0) return;  // ended by a done at an earlier step
  const int k = A.first ? 1 : 1 - A.length[e];
  if (A.cols == 2) {
    A.ret[2 * e] = add_rn(A.first ? 0.0 : A.ret[2 * e], mul_rn(A.w, rew[0]));
    A.ret[2 * e + 1] = add_rn(A.first ? 0.0 : A.ret[2 * e + 1], mul_rn(A.w, rew[1]));
  } else {
    A.ret[e] = add_rn(A.first ? 0.0 : A.ret[e], mul_rn(A.w, rew[0]));
  }
  A.cost[e] = add_rn(A.first ? 0.0 : A.cost[e], mul_rn(A.w, c ? 1.0 : 0.0));
  A.length[e] = (d || A.last) ? k : -k;
}

// observation at the current state (reset return value / refresh after state injection)
template <class RB>
SAG_HD void env_observe(unsigned wmask, Scratch* S, const Dev& D, int e, float* obs_s, int ostride) {
  Ctx C = {D, e, spec_for(D, D.task[e], RB::kGremlins, RB::kCustom), Slots(), logic_task(D, D.task[e], RB::kCustom),
           global_objects(D, e)};
  C.L = make_slots(C.sp);
  RB R;
  load_robot(D, e, C.sp, R);
  TaskState T;
  load_task_state(D, e, T);
  Rng rng = {rng_key(D), D.gid_base + (uint32_t)e, D.episode[e]};
  const PtConst K = R.consts(RB::kH);
  unsigned mov = 0;  // rebuilt from the velocities: state may have been injected
  for (int s = C.L.v0; s < C.L.n; ++s) {
    if (!kind_movable(slot_kind(C.sp, C.L, s))) continue;
    size_t i = oix(C, s);
    if (C.O.vx[i] != 0.0 || C.O.vy[i] != 0.0 || C.O.w[i] != 0.0) mov |= 1u << s;
  }
  SolveConsts Q;
  solve_consts(D, C.sp, Q, RB::kGremlins);
  EndOut O;
  double moc[2] = {0.0, 0.0};
  if (RB::kGremlins && C.sp.ng > 0) { moc[0] = D.grem[e]; moc[1] = D.grem[(size_t)D.stride + e]; }
  end_of_step<kStepFull, RB>(wmask, S, Q, C, R, T, rng, K, mov, false, nullptr, false, obs_s, ostride, O, nullptr, 0xffffffffu, moc);
  D.clear[e] = O.clear;
  D.movmask[e] = (int)mov;
}

// ------------------------------------------------------------------------------------------------
// reset: layout rejection sampling (world.py:172-217, utils.py:22-70), yaw draws (world.py:108-137),
// fresh physics (mujoco_bridge.py:170-175), task.reset (world.py:167-170)
// ------------------------------------------------------------------------------------------------
// the placement extents (x_min, y_min, x_max, y_max) of a user-defined task; a registry id keeps (-e, -e, e, e)
SAG_HD void custom_extents(const Dev& D, int t, double* rect) {
  if (t < T_COUNT) return;
  const double* x = custom_table(D).t[t - T_COUNT].ext;
  rect[0] = x[0]; rect[1] = x[1]; rect[2] = x[2]; rect[3] = x[3];
}

SAG_HD double slot_keepout(const Dev& D, const TaskSpec& sp, int kind) {
  return kind == K_HAZARD ? D.k_hazard : kind == K_VASE ? D.k_vase : kind == K_GREMLIN ? D.k_gremlin
       : kind == K_PILLAR ? D.k_pillar : kind == K_GOAL ? kGoalKeepout : kind == K_BUTTON ? kButtonsKeepout : sp.box_keepout;
}

// The per-environment "next task" slot (SAG_F_NEXT_TASK, -1 = none), consumed by the next reset of environment e, whatever
// the reset path.  Called by k_reset (lane 0 of the warp that resets e) and by the host emulation's reset, after the
// finished episode has been credited to the per-environment statistics.  A queued task: the statistics gathered under
// the old task are folded into the per-task accumulator `acc` (as k_set_tasks does), e takes the new task id and is
// reset as a fresh Task instance even if the id is unchanged.  An id outside [0, nids) is not applied: the slot is
// cleared and SAG_ERR_BAD_TASK_ID recorded.  nids: the handle's ids (num_task_ids).  Returns whether e is reset as a
// fresh Task instance.
SAG_HD bool take_next_task(const Dev& D, int e, int* next_task, double* sret, double* scost, double* sn, double* acc,
                           bool new_task, int nids = T_COUNT) {
  const int id = next_task[e];
  if (id == -1) return new_task;
  next_task[e] = -1;
  if (id < 0 || id >= nids) { D.errflags[1] = 1; return new_task; }
  const int old = D.task[e];
  if (sn[e] != 0.0 && old >= 0 && old < nids) {
#if defined(__CUDA_ARCH__)
    atomicAdd(acc + 3 * old, sret[e]); atomicAdd(acc + 3 * old + 1, scost[e]); atomicAdd(acc + 3 * old + 2, sn[e]);
#else
    acc[3 * old] += sret[e]; acc[3 * old + 1] += scost[e]; acc[3 * old + 2] += sn[e];
#endif
  }
  sret[e] = 0.0; scost[e] = 0.0; sn[e] = 0.0;
  D.task[e] = id;
  return true;
}

// sag_copy_envs, the rule for destination j of the destination handle D: returns the source environment whose state j
// takes, or -1 when j is left untouched.  -1 in src_of_dst[j] and the no-op j <- j leave j alone.  A pair is bad, and
// not applied, when its index is outside [-1, n_src) or, within one handle, when its source is itself overwritten by the
// call (src_of_dst[s] not in {-1, s}): read from the index array alone, so every thread decides alike.  With `fold`
// (k_copy_envs_fold, one thread per destination, before any field is overwritten; the host emulation's loop), a bad
// pair records SAG_ERR_BAD_ENV_INDEX, and for an applied one j's statistics are settled as a reset or k_set_tasks
// settles them before j's state is replaced: an episode that has finished (NEEDS_RESET, nstep > 0) but has not been
// reset yet is credited, then j's finished-episode statistics are folded into the per-task accumulator `acc` under j's
// OLD task and cleared, so that they are not credited to the copied task.  An unfinished episode of j is dropped.
SAG_HD int copy_env_source(const Dev& D, const int32_t* src_of_dst, int j, int n_src, bool same_handle, bool fold,
                           double* sret, double* scost, double* sn, double* acc, int nids = T_COUNT) {
  const int s = src_of_dst[j];
  if (s == -1 || (same_handle && s == j)) return -1;
  bool bad = s < -1 || s >= n_src;
  if (!bad && same_handle) {
    const int t = src_of_dst[s];
    bad = t != -1 && t != s;
  }
  if (bad) {
    if (fold) D.errflags[2] = 1;
    return -1;
  }
  if (fold) {
    const int old = D.task[j];
    double r = sret[j], c = scost[j], k = sn[j];
    if ((D.flags[j] & F_NEEDS_RESET) && D.nstep[j] > 0) { r += D.epret[j]; c += D.epcost[j]; k += 1.0; }
    if (k != 0.0 && old >= 0 && old < nids) {
#if defined(__CUDA_ARCH__)
      atomicAdd(acc + 3 * old, r); atomicAdd(acc + 3 * old + 1, c); atomicAdd(acc + 3 * old + 2, k);
#else
      acc[3 * old] += r; acc[3 * old + 1] += c; acc[3 * old + 2] += k;
#endif
    }
    sret[j] = 0.0; scost[j] = 0.0; sn[j] = 0.0;
  }
  return s;
}

// The fresh episode after placement, shared by env_reset and env_reset_coop: the robot at rest at (x, y, yaw) and the
// task state of environment C.e.  For a fresh Task instance (new_task) it makes the per-instance draws of World.__init__
// (world.py:72-78): Task.ctrl_scale, standard Cauchy per actuator (task.py:85-89), and Task.constraint_bound
// (task.py:91-94), on Philox stream 3, Cauchy by inversion; and it resets the task state (catch_goal.py:12-18,
// press_buttons.py:20-24, collect.py:15-16).  Returns the Task instance's ctrl scales and bound: the fresh draws, which
// the caller stores, when new_task, the stored ones otherwise.
struct TaskDraws { double cscale[2], bound; };
template <class RB>
SAG_HD TaskDraws fresh_episode(const Dev& D, const Ctx& C, const Rng& rng, double x, double y, double yaw, bool new_task,
                               RB& R, TaskState& T) {
  const int e = C.e;
  R.q[0] = x; R.q[1] = y; R.q[2] = yaw; R.v[0] = R.v[1] = R.v[2] = 0.0; R.ctrl[0] = R.ctrl[1] = 0.0;
  if constexpr (RB::kKind == 1) { R.wheel[0] = R.wheel[1] = 0.0; R.cq[0] = 1.0; R.cq[1] = R.cq[2] = R.cq[3] = 0.0; }
  R.damp_xy = C.sp.damp_xy; R.gear_x = C.sp.gear_x;
  load_task_state(D, e, T);
  TaskDraws d;
  if (new_task) {
    double u[2];
    rng.pair(3u, 0u, u[0], u[1]);
    for (int k = 0; k < 2; ++k) {
      double tn, tc;
      sag_sincos(kPi * (u[k] - 0.5), &tn, &tc);
      d.cscale[k] = (tn / tc) * D.ctrl_range_scale + 1.0;
    }
    rng.pair(3u, 1u, u[0], u[1]);
    d.bound = D.random_bound ? 0.0 + (D.max_bound - 0.0) * u[0] : D.max_bound;
  } else {
    d.cscale[0] = D.cscale0[e]; d.cscale[1] = D.cscale1[e]; d.bound = D.bound[e];
  }
  if (D.ctrl_range_scale != 0.0) {  // MuJoCo clamps the zero control of a fresh physics into an inverted range, too
    R.ctrl[0] = clampd(0.0, -1.0 * d.cscale[0], 1.0 * d.cscale[0]); R.ctrl[1] = clampd(0.0, -1.0 * d.cscale[1], 1.0 * d.cscale[1]);
  }
  if (new_task) {
    T.cgcur = 1.0; T.cgnext = 0.2; T.cgtimer = 0; T.bstate = 1; T.btimer = kButtonDelay; T.gbtn = 0;
    T.amask = C.task == T_COLLECT ? (1 << C.L.nbtn) - 1 : 0; T.cgox = T.cgoy = 0.0; T.last0 = T.last1 = 0.0;
  }
  return d;
}

template <class RB>
SAG_HD_NOINLINE void env_reset(const Dev& D, int e, uint32_t episode, bool new_task) {
  Ctx C = {D, e, spec_for(D, D.task[e], RB::kGremlins, RB::kCustom), Slots(), logic_task(D, D.task[e], RB::kCustom),
           global_objects(D, e)};
  C.L = make_slots(C.sp);
  const unsigned long long key = rng_key_value(rng_key(D));  // once per layout: the rejection sampler draws in a loop
  Rng rng = {rng_key_of(key), D.gid_base + (uint32_t)e, episode};
  uint32_t ctr = 0;
  long draws_left = D.max_layout_draws > 0 ? D.max_layout_draws : (1L << 22);
  unsigned char fl = 0;
  double rxy[2] = {0.0, 0.0};
  bool ok = false;
  const double ext = C.sp.extent;
  double rect[4] = {-ext, -ext, ext, ext};  // free placements (*C instantiations: a user-defined task's own extents)
  if constexpr (RB::kCustom) custom_extents(D, D.task[e], rect);
  // the placed bodies' positions and keepout + margin, thread-private (the rejection loop below reads them ~10^3 times)
  double px[kMaxObj], py[kMaxObj], pk[kMaxObj];
  for (int j = 0; j < kMaxObj; ++j) { px[j] = 0.0; py[j] = 0.0; pk[j] = 0.0; }
  for (int j = 0; j < C.L.n; ++j) pk[j] = slot_keepout(D, C.sp, slot_kind(C.sp, C.L, j)) + D.placements_margin;
  const double rk = D.robot_keepout + D.placements_margin;
  for (int attempt = 0; attempt < 10000 && !ok && draws_left >= 0; ++attempt) {
    bool failed = false;
    for (int idx = -1; idx < C.L.n && !failed; ++idx) {
      int kind = idx < 0 ? K_NONE : slot_kind(C.sp, C.L, idx);
      double keepout = idx < 0 ? D.robot_keepout : slot_keepout(D, C.sp, kind);
      double half = ext;  // free placement in the task extents
      bool free_xy = true;
      if (kind == K_GOAL) { half = 1.5; free_xy = false; }
      else if (kind == K_BUTTON) { half = C.sp.button_rect; free_xy = false; }
      else if ((kind == K_BOX || kind == K_ROD || kind == K_BALL) && C.sp.box_rect > 0.0) { half = C.sp.box_rect; free_xy = false; }
      double xmin = -half + keepout, xmax = half - keepout, ymin = xmin, ymax = xmax;
      if constexpr (RB::kCustom) {
        if (free_xy) { xmin = rect[0] + keepout; ymin = rect[1] + keepout; xmax = rect[2] - keepout; ymax = rect[3] - keepout; }
      }
      bool placed = false;
      double x = 0.0, y = 0.0;
      for (int k = 0; k < 1000; ++k) {
        if (--draws_left < 0) { failed = true; break; }
        double u1, u2;
        rng.pair(0u, ctr++, u1, u2);
        x = xmin + (xmax - xmin) * u1; y = ymin + (ymax - ymin) * u2;
        bool valid = true;
        if (idx >= 0) {
          double dx = x - rxy[0], dy = y - rxy[1];
          if (sqrt_less(dx * dx + dy * dy, rk + keepout)) valid = false;
          for (int j = 0; valid && j < idx; ++j) {
            double ex = x - px[j], ey = y - py[j];
            if (sqrt_less(ex * ex + ey * ey, pk[j] + keepout)) valid = false;
          }
        }
        if (valid) { placed = true; break; }
      }
      if (!placed) { failed = true; break; }
      if (idx < 0) { rxy[0] = x; rxy[1] = y; }
      else { px[idx] = x; py[idx] = y; }
    }
    if (!failed) ok = true;
  }
  for (int j = 0; j < C.L.n; ++j) { size_t i = oix(C, j); C.O.x[i] = px[j]; C.O.y[i] = py[j]; }
  if (!ok) fl |= F_RESAMPLE_FAILED;
  // yaw draws in the reference's order
  double u1, u2;
  rng.pair(0u, ctr++, u1, u2);
  double robot_rot = kTwoPi * u1;
  for (int s = 0; s < C.L.t0; ++s) {
    rng.pair(0u, ctr++, u1, u2);
    size_t i = oix(C, s);
    C.O.yaw[i] = kTwoPi * u1; C.O.vx[i] = 0.0; C.O.vy[i] = 0.0; C.O.w[i] = 0.0;
  }
  for (int s = C.L.t0; s < C.L.n; ++s) { size_t i = oix(C, s); C.O.yaw[i] = 0.0; C.O.vx[i] = 0.0; C.O.vy[i] = 0.0; C.O.w[i] = 0.0; }
  if (C.task == T_HAUL_BOX) { size_t ib = oix(C, C.L.box); C.O.x[ib] = rxy[0] + kBoxSize * 3.0; C.O.y[ib] = rxy[1]; }
  if (C.sp.kind == 0 || C.sp.kind == 2) { rng.pair(0u, ctr++, u1, u2); C.O.yaw[oix(C, C.L.goal)] = kTwoPi * u1; }
  if (C.sp.kind == 2 && C.sp.box_kind == K_BOX) { rng.pair(0u, ctr++, u1, u2); C.O.yaw[oix(C, C.L.box)] = kTwoPi * u1; }
  if (C.sp.kind == 1) for (int i = 0; i < C.L.nbtn; ++i) { rng.pair(0u, ctr++, u1, u2); C.O.yaw[oix(C, C.L.btn0 + i)] = kTwoPi * u1; }
  RB R;
  TaskState T;
  const TaskDraws td = fresh_episode(D, C, rng, rxy[0], rxy[1], robot_rot, new_task, R, T);
  if (new_task) { D.cscale0[e] = td.cscale[0]; D.cscale1[e] = td.cscale[1]; D.bound[e] = td.bound; }
  if (ok && task_reset(C, rng, 0u, ctr, R, T)) fl |= F_RESAMPLE_FAILED;
  T.ctr = 0;
  store_robot(D, e, R);
  store_task_state(D, e, T);
  D.episode[e] = episode; D.nstep[e] = 0; D.time[e] = 0.0; D.epret[e] = 0.0; D.epcost[e] = 0.0; D.flags[e] = fl;
  // clearance of the fresh layout (same definition as end_of_step's; scheduling hint only: without it the first step
  // after a reset would send the whole batch down the contact path)
  double clear = 1e30;
  for (int s = C.L.v0; s < C.L.n; ++s) {
    const int kind = slot_kind(C.sp, C.L, s);
    if (!kind_collidable(kind)) continue;
    size_t i = oix(C, s);
    double dx = C.O.x[i] - R.q[0], dy = C.O.y[i] - R.q[1];
    clear = fmin(clear, sqrt(dx * dx + dy * dy) - (RB::kReach + kind_bound(D, kind)));
  }
  if (C.task == T_HAUL_BOX) {
    double tdx, tdy, tlen, tdist;
    tendon_taut(C, R, tdx, tdy, tlen, tdist);
    clear = fmin(clear, tdist);
  }
  if (RB::kGremlins && C.sp.ng > 0) {  // gremlins: weld anchor = spawn pose, mocap bodies at the world origin; never a quiet environment
    clear = -1.0;
    D.grem[e] = 0.0; D.grem[(size_t)D.stride + e] = 0.0;
    for (int g = 0; g < C.sp.ng; ++g) {
      const size_t i = oix(C, C.L.g0 + g);
      double* sp0 = D.grem + (size_t)(2 + 3 * g) * D.stride + e;
      sp0[0] = C.O.x[i]; sp0[D.stride] = C.O.y[i]; sp0[2 * (size_t)D.stride] = C.O.yaw[i];
    }
  }
  D.clear[e] = clear;
  D.movmask[e] = 0;
}


// ------------------------------------------------------------------------------------------------
// Warp-cooperative reset (device only): ONE WARP resets one environment.  The rejection samplers (world.py:191-217,
// go_to_goal.py:59-80) draw candidate k from Philox counter ctr + k, so a round of candidates is a set of independent
// draws: a round evaluates 8 candidates, the validity checks of one candidate split over 4 lanes (lane = 4 * candidate +
// group; under the reference's keepouts the first valid draw is among the first eight 94 % of the time), and a ballot
// picks the FIRST valid one -- the very draw the sequential sampler would have stopped at; the counter advances by exactly
// the draws it would have used (per-object limit of 1000 draws and the layout's draw budget included).  Same arithmetic
// per candidate, so layouts are bit-identical to env_reset / the oracle (tests/test_gpu_parity.py).  px / py / pk: 32
// doubles each of the warp's shared memory (positions placed so far, keepout + margin per slot).
// ------------------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
constexpr int kResetCand = 8;  // candidates per round; lane = 4 * candidate + check group
// index of the first candidate (< window) none of whose four lanes raised `bad`, or -1
__device__ __forceinline__ int coop_first_valid(bool bad, int window) {
  const unsigned mb = __ballot_sync(kFullWarp, bad);
  const unsigned t = mb | (mb >> 1) | (mb >> 2) | (mb >> 3);   // bit 4c: some lane of candidate c said bad
  const unsigned wmask = window >= kResetCand ? 0x11111111u : (((1u << (4 * window)) - 1u) & 0x11111111u);
  const unsigned okm = ~t & wmask;
  return okm ? ((__ffs((int)okm) - 1) >> 2) : -1;
}
__device__ __forceinline__ int resample_goal_coop(const Ctx& C, const Rng& rng, uint32_t stream, uint32_t& ctr, double rx, double ry,
                                                  double& gx, double& gy) {
  const Dev& D = C.D;
  const int lane = coop_lane();
  const int cand = lane >> 2, grp = lane & 3;  // 8 candidates per round, the checks of one candidate split over 4 lanes
  double base[4] = {-1.5, -1.5, 1.5, 1.5};  // the rectangle after the failed draws so far (x1.01 per failure, go_to_goal.py:76-79)
  int used = 0;
  const int kMaxDraws = 500000;
  while (used < kMaxDraws) {
    const int window = min(kResetCand, kMaxDraws - used);
    double rect[4] = {base[0], base[1], base[2], base[3]};
    for (int t = 0; t < cand; ++t) {
#pragma unroll
      for (int k = 0; k < 4; ++k) rect[k] = rect[k] * 1.01;
    }
    double u1, u2;
    rng.pair(stream, ctr + (uint32_t)cand, u1, u2);
    double xmin = rect[0] + kGoalKeepout, ymin = rect[1] + kGoalKeepout, xmax = rect[2] - kGoalKeepout, ymax = rect[3] - kGoalKeepout;
    double x = xmin + (xmax - xmin) * u1, y = ymin + (ymax - ymin) * u2;
    bool bad = false;
    if (grp == 0) { double dx = x - rx, dy = y - ry; if (sqrt_less(dx * dx + dy * dy, D.robot_keepout + kGoalKeepout)) bad = true; }
    for (int s = grp; s < C.L.n; s += 4) {
      if (s == C.L.goal) continue;
      int kind = slot_kind(C.sp, C.L, s);
      double ko = kind == K_HAZARD ? D.k_hazard : kind == K_VASE ? D.k_vase : kind == K_GREMLIN ? D.k_gremlin
                : kind == K_PILLAR ? D.k_pillar : kind == K_BUTTON ? kButtonsKeepout : C.sp.box_keepout;
      size_t i = oix(C, s);
      double dx = x - C.O.x[i], dy = y - C.O.y[i];
      if (sqrt_less(dx * dx + dy * dy, ko + kGoalKeepout)) bad = true;
    }
    const int first = coop_first_valid(bad, window);
    if (first >= 0) {
      gx = __shfl_sync(kFullWarp, x, first * 4); gy = __shfl_sync(kFullWarp, y, first * 4);
      ctr += (uint32_t)(first + 1);
      return 0;
    }
    ctr += (uint32_t)window; used += window;
    for (int t = 0; t < window; ++t) {
#pragma unroll
      for (int k = 0; k < 4; ++k) base[k] = base[k] * 1.01;
    }
  }
  return 1;
}

// task.reset() with the cooperative goal sampler (otherwise task_reset above, run redundantly by every lane)
template <class RB>
__device__ __forceinline__ int task_reset_coop(const Ctx& C, const Rng& rng, uint32_t stream, uint32_t& ctr, const RB& R, TaskState& T) {
  if (C.sp.kind == 1) {
    if (C.task == T_COLLECT) T.amask = (1 << C.L.nbtn) - 1;
    else sample_goal_button(C, rng, stream, ctr, R, T);
    return 0;
  }
  double gx = 0.0, gy = 0.0;
  if (resample_goal_coop(C, rng, stream, ctr, R.q[0], R.q[1], gx, gy)) return 1;
  size_t ig = oix(C, C.L.goal);
  __syncwarp();
  if (coop_lane() == 0) { C.O.x[ig] = gx; C.O.y[ig] = gy; }
  __syncwarp();
  T.last0 = dist2d(R.q[0], R.q[1], gx, gy);
  if (C.task == T_CATCH_GOAL) { T.cgox = gx; T.cgoy = gy; }
  if (C.sp.kind == 2) {
    size_t ib = oix(C, C.L.box);
    double bx = C.O.x[ib], by = C.O.y[ib];
    T.last1 = dist2d(gx, gy, bx, by);
    T.last0 = dist2d(R.q[0], R.q[1], bx, by);
  }
  return 0;
}

template <class RB>
__device__ __noinline__ void env_reset_coop(const Dev& D, int e, uint32_t episode, bool new_task, double* px, double* py, double* pk) {
  const int lane = coop_lane();
  const int cand = lane >> 2, grp = lane & 3;  // 8 placement candidates per round, each checked by 4 lanes
  Ctx C = {D, e, spec_for(D, D.task[e], RB::kGremlins, RB::kCustom), Slots(), logic_task(D, D.task[e], RB::kCustom),
           global_objects(D, e)};
  C.L = make_slots(C.sp);
  const ObjView G = C.O;
  const unsigned long long key = rng_key_value(rng_key(D));  // once per layout: the rejection sampler draws in a loop
  Rng rng = {rng_key_of(key), D.gid_base + (uint32_t)e, episode};
  uint32_t ctr = 0;
  long draws_left = D.max_layout_draws > 0 ? D.max_layout_draws : (1L << 22);
  unsigned char fl = 0;
  double rxy[2] = {0.0, 0.0};
  bool ok = false;
  const double ext = C.sp.extent;
  double rect[4] = {-ext, -ext, ext, ext};
  if constexpr (RB::kCustom) custom_extents(D, D.task[e], rect);
  px[lane] = 0.0; py[lane] = 0.0;
  pk[lane] = lane < C.L.n ? slot_keepout(D, C.sp, slot_kind(C.sp, C.L, lane)) + D.placements_margin : 0.0;
  __syncwarp();
  const double rk = D.robot_keepout + D.placements_margin;
  for (int attempt = 0; attempt < 10000 && !ok && draws_left >= 0; ++attempt) {
    bool failed = false;
    for (int idx = -1; idx < C.L.n && !failed; ++idx) {
      int kind = idx < 0 ? K_NONE : slot_kind(C.sp, C.L, idx);
      double keepout = idx < 0 ? D.robot_keepout : slot_keepout(D, C.sp, kind);
      double half = ext;
      bool free_xy = true;
      if (kind == K_GOAL) { half = 1.5; free_xy = false; }
      else if (kind == K_BUTTON) { half = C.sp.button_rect; free_xy = false; }
      else if ((kind == K_BOX || kind == K_ROD || kind == K_BALL) && C.sp.box_rect > 0.0) { half = C.sp.box_rect; free_xy = false; }
      double xmin = -half + keepout, xmax = half - keepout, ymin = xmin, ymax = xmax;
      if constexpr (RB::kCustom) {
        if (free_xy) { xmin = rect[0] + keepout; ymin = rect[1] + keepout; xmax = rect[2] - keepout; ymax = rect[3] - keepout; }
      }
      bool placed = false;
      double x = 0.0, y = 0.0;
      int used = 0;  // draws spent on this object (limit 1000, world.py:209)
      while (used < 1000) {
        if (draws_left <= 0) { draws_left = -1; failed = true; break; }  // the layout's draw budget is spent
        int window = 1000 - used;
        if (window > kResetCand) window = kResetCand;
        if ((long)window > draws_left) window = (int)draws_left;
        double u1, u2;
        rng.pair(0u, ctr + (uint32_t)cand, u1, u2);
        const double cx = xmin + (xmax - xmin) * u1, cy = ymin + (ymax - ymin) * u2;
        bool bad = false;
        if (idx >= 0) {
          if (grp == 0) { double dx = cx - rxy[0], dy = cy - rxy[1]; if (sqrt_less(dx * dx + dy * dy, rk + keepout)) bad = true; }
          for (int j = grp; j < idx; j += 4) {
            double ex = cx - px[j], ey = cy - py[j];
            if (sqrt_less(ex * ex + ey * ey, pk[j] + keepout)) bad = true;
          }
        }
        const int first = coop_first_valid(bad, window);
        if (first >= 0) {
          x = __shfl_sync(kFullWarp, cx, first * 4); y = __shfl_sync(kFullWarp, cy, first * 4);
          ctr += (uint32_t)(first + 1); draws_left -= first + 1; used += first + 1;
          placed = true;
          break;
        }
        ctr += (uint32_t)window; draws_left -= window; used += window;
      }
      if (!placed) { failed = true; break; }
      if (idx < 0) { rxy[0] = x; rxy[1] = y; }
      else {
        __syncwarp();
        if (lane == 0) { px[idx] = x; py[idx] = y; }
        __syncwarp();
      }
    }
    if (!failed) ok = true;
  }
  if (!ok) fl |= F_RESAMPLE_FAILED;
  if (C.task == T_HAUL_BOX) {  // haul_box.py:17-18: the box is put next to the robot whatever was sampled for it
    __syncwarp();
    if (lane == 0) { px[C.L.box] = rxy[0] + kBoxSize * 3.0; py[C.L.box] = rxy[1]; }
  }
  __syncwarp();
  // yaw draws in the reference's order (world.py:115-136): robot, obstacle slots [0, t0), then goal / box / buttons.  Draw d
  // of that list is counter ctr + d; the lane of a slot evaluates the slot's own draw.
  const int n_extra = (C.sp.kind == 0 ? 1 : C.sp.kind == 2 ? (C.sp.box_kind == K_BOX ? 2 : 1) : C.L.nbtn);
  const int n_yaw = 1 + C.L.t0 + n_extra;
  double robot_rot, yaw_l = 0.0;
  {
    double u1, u2;
    rng.pair(0u, ctr, u1, u2);
    robot_rot = kTwoPi * u1;
    int d = -1;  // this lane's slot: which draw?
    if (lane < C.L.t0) d = 1 + lane;
    else if (lane < C.L.n) {
      if (C.sp.kind == 1) d = 1 + C.L.t0 + (lane - C.L.btn0);
      else if (lane == C.L.goal) d = 1 + C.L.t0;
      else if (lane == C.L.box && C.sp.box_kind == K_BOX) d = 2 + C.L.t0;
    }
    if (d >= 0) { rng.pair(0u, ctr + (uint32_t)d, u1, u2); yaw_l = kTwoPi * u1; }
  }
  ctr += (uint32_t)n_yaw;
  if (lane < C.L.n) {
    const size_t i = (size_t)lane * G.stride;
    G.x[i] = px[lane]; G.y[i] = py[lane]; G.yaw[i] = yaw_l; G.vx[i] = 0.0; G.vy[i] = 0.0; G.w[i] = 0.0;
  }
  // from here on the object positions are read from the warp's shared memory (task_reset, clearance)
  C.O.x = px; C.O.y = py; C.O.stride = 1;
  RB R;
  TaskState T;
  const TaskDraws td = fresh_episode(D, C, rng, rxy[0], rxy[1], robot_rot, new_task, R, T);
  if (new_task && lane == 0) { D.cscale0[e] = td.cscale[0]; D.cscale1[e] = td.cscale[1]; D.bound[e] = td.bound; }
  if (ok && task_reset_coop(C, rng, 0u, ctr, R, T)) fl |= F_RESAMPLE_FAILED;
  T.ctr = 0;
  __syncwarp();
  // clearance of the fresh layout, one slot per lane (a min: the order of the operands does not matter)
  double cl = 1e30;
  if (lane >= C.L.v0 && lane < C.L.n) {
    const int kind = slot_kind(C.sp, C.L, lane);
    if (kind_collidable(kind)) {
      double dx = px[lane] - R.q[0], dy = py[lane] - R.q[1];
      cl = sqrt(dx * dx + dy * dy) - (RB::kReach + kind_bound(D, kind));
    }
  }
  double clear = fmin(1e30, coop_min(cl));
  if (C.task == T_HAUL_BOX) {
    double tdx, tdy, tlen, tdist;
    tendon_taut(C, R, tdx, tdy, tlen, tdist);
    clear = fmin(clear, tdist);
  }
  if (RB::kGremlins && C.sp.ng > 0) {
    clear = -1.0;
    if (lane == 0) { D.grem[e] = 0.0; D.grem[(size_t)D.stride + e] = 0.0; }
    if (lane >= C.L.g0 && lane < C.L.p0) {
      double* sp0 = D.grem + (size_t)(2 + 3 * (lane - C.L.g0)) * D.stride + e;
      sp0[0] = px[lane]; sp0[D.stride] = py[lane]; sp0[2 * (size_t)D.stride] = yaw_l;
    }
  }
  if (lane == 0) {
    if (C.L.goal >= 0) { const size_t ig = (size_t)C.L.goal * G.stride; G.x[ig] = px[C.L.goal]; G.y[ig] = py[C.L.goal]; }
    store_robot(D, e, R);
    store_task_state(D, e, T);
    D.episode[e] = episode; D.nstep[e] = 0; D.time[e] = 0.0; D.epret[e] = 0.0; D.epcost[e] = 0.0; D.flags[e] = fl;
    D.clear[e] = clear;
    D.movmask[e] = 0;
  }
  __syncwarp();
}
#endif  // __CUDA_ARCH__

}  // namespace sag
