// sag_layout.h -- host-side carving of the single state slab into the SoA arrays of sag::Dev, and the configuration defaults.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <string.h>

#include "../../include/sag_b200.h"
#include "sag_core.cuh"

namespace sag {

// sag_default_config: World.DEFAULT (world.py:17-34), one environment, the point robot
inline void default_config(SagConfig* c) {
  memset(c, 0, sizeof(*c));
  c->n_envs = 1; c->robot = SAG_ROBOT_POINT; c->seed = 666;
  c->placements_margin = 0.0; c->robot_keepout = 0.4;
  c->hazards_size = 0.2; c->vases_size = 0.1; c->pillars_size = 0.2; c->gremlins_size = 0.1;
  c->hazards_keepout = 0.18; c->gremlins_keepout = 0.4; c->vases_keepout = 0.15; c->pillars_keepout = 0.3;
  c->gremlins_travel = 0.35; c->robot_ctrl_range_scale = 0.0; c->action_noise = 0.01; c->max_bound = 25.0;
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct SlabLayout {
  size_t off[SAG_NUM_FIELDS], bytes[SAG_NUM_FIELDS];
  size_t stats_off, sched_off, act_off, obs_off, rew_off, cost_off, done_off, acc_off, ids_off, mask_off, custom_off, total;
};

// The per-environment shape of every state field: rows of `elem`-byte elements, each row `stride` elements long
// (field[row][env]).  The one list of the fields: the slab is carved from it, and sag_copy_envs copies every row it
// names, so a field added here is carried by a copy without touching the kernel.
struct FieldShape { int rows, elem; };
constexpr FieldShape kFieldShape[SAG_NUM_FIELDS] = {
    {6, 8},                          // SAG_F_ROBOT
    {6 * SAG_MAX_SLOTS, 8},          // SAG_F_OBJECTS
    {15, 8},                         // SAG_F_TASK_F64
    {10, 4},                         // SAG_F_TASK_I32
    {1, 1},                          // SAG_F_FLAGS
    {6, 8},                          // SAG_F_ROBOT_EXT
    {2 + 3 * SAG_MAX_GREMLINS, 8},   // SAG_F_GREMLINS
    {1, 4},                          // SAG_F_NEXT_TASK: not bound into Dev, the reset kernels take it as an argument
};

inline SlabLayout slab_layout(int n, int stride, int obs_dim) {
  SlabLayout L;
  const size_t st = (size_t)stride;
  for (int f = 0; f < SAG_NUM_FIELDS; ++f) L.bytes[f] = (size_t)kFieldShape[f].rows * kFieldShape[f].elem * st;
  size_t total = 0;
  for (int f = 0; f < SAG_NUM_FIELDS; ++f) { L.off[f] = total; total += align_up(L.bytes[f], 256); }
  L.stats_off = total; total += align_up(3 * st * sizeof(double), 256);
  L.sched_off = total; total += align_up((3 * st + 96) * sizeof(int32_t), 256);
  L.act_off = total; total += align_up((size_t)n * 2 * sizeof(float), 256);
  L.obs_off = total; total += align_up((size_t)n * obs_dim * sizeof(float), 256);
  L.rew_off = total; total += align_up((size_t)n * sizeof(double), 256);
  L.cost_off = total; total += align_up((size_t)n, 256);
  L.done_off = total; total += align_up((size_t)n, 256);
  L.acc_off = total; total += align_up((SAG_NUM_TASKS + SAG_MAX_CUSTOM_TASKS) * 3 * sizeof(double), 256);
  L.ids_off = total; total += align_up((size_t)n * sizeof(int32_t), 256);
  L.mask_off = total; total += align_up((size_t)n, 256);
  L.custom_off = total; total += align_up(sizeof(CustomTable), 256);
  L.total = total;
  return L;
}

inline void slab_bind(Dev& D, const SlabLayout& L, char* base) {
  const size_t st = (size_t)D.stride;
  double* r = (double*)(base + L.off[SAG_F_ROBOT]);
  D.rx = r; D.ry = r + st; D.ryaw = r + 2 * st; D.rvx = r + 3 * st; D.rvy = r + 4 * st; D.rw = r + 5 * st;
  double* o = (double*)(base + L.off[SAG_F_OBJECTS]);
  const size_t os = (size_t)SAG_MAX_SLOTS * st;
  D.ox = o; D.oy = o + os; D.oyaw = o + 2 * os; D.ovx = o + 3 * os; D.ovy = o + 4 * os; D.ow = o + 5 * os;
  double* t = (double*)(base + L.off[SAG_F_TASK_F64]);
  D.last0 = t; D.last1 = t + st; D.cgcur = t + 2 * st; D.cgnext = t + 3 * st; D.cgox = t + 4 * st; D.cgoy = t + 5 * st;
  D.time = t + 6 * st; D.clear = t + 7 * st; D.epret = t + 8 * st; D.epcost = t + 9 * st; D.ctrl0 = t + 10 * st; D.ctrl1 = t + 11 * st;
  D.cscale0 = t + 12 * st; D.cscale1 = t + 13 * st; D.bound = t + 14 * st;
  int32_t* ii = (int32_t*)(base + L.off[SAG_F_TASK_I32]);
  D.task = ii; D.gbtn = ii + st; D.bstate = ii + 2 * st; D.btimer = ii + 3 * st; D.amask = ii + 4 * st; D.cgtimer = ii + 5 * st;
  D.nstep = ii + 6 * st; D.ctr = (unsigned*)(ii + 7 * st); D.episode = (unsigned*)(ii + 8 * st); D.movmask = ii + 9 * st;
  D.flags = (unsigned char*)(base + L.off[SAG_F_FLAGS]);
  D.rext = (double*)(base + L.off[SAG_F_ROBOT_EXT]);
  D.grem = (double*)(base + L.off[SAG_F_GREMLINS]);
  int32_t* sc = (int32_t*)(base + L.sched_off);
  // the block after the work list is 96 ints: two counter sets (16), 18 x u64 (36), the step epoch and the contact
  // kernel's finished-CTA counter (2), the Philox key (u64; 8-byte aligned: the block starts 256-aligned and 3 * st is a
  // multiple of 96), the address of the user-defined task table (custom_table; 8-byte aligned too)
  D.worklist = sc; D.counts = sc + 3 * st;
  D.dbg = (unsigned long long*)(sc + 3 * st + 16);
  D.epoch = (unsigned*)(sc + 3 * st + 52);
  D.key = (unsigned long long*)(sc + 3 * st + 54);
#if !defined(__CUDACC__)
  // a host build (the host emulation of the tests) stores the table's address here; the library copies it to the device
  *reinterpret_cast<CustomTable**>(sc + 3 * st + kCustomTablePtr) = reinterpret_cast<CustomTable*>(base + L.custom_off);
#endif
}

inline void dev_from_config(Dev& D, const SagConfig& c) {
  D.n = c.n_envs;
  D.stride = (int)align_up((size_t)c.n_envs, 32);
  D.nslots = SAG_MAX_SLOTS;
  D.robot = c.robot;
  D.action_noise = c.action_noise; D.placements_margin = c.placements_margin; D.robot_keepout = c.robot_keepout;
  D.hazards_size = c.hazards_size; D.vases_size = c.vases_size; D.pillars_size = c.pillars_size; D.gremlins_size = c.gremlins_size;
  D.k_hazard = c.hazards_keepout < c.hazards_size ? c.hazards_size : c.hazards_keepout;  // world.py:60-66
  D.k_vase = c.vases_keepout < c.vases_size ? c.vases_size : c.vases_keepout;
  D.k_gremlin = c.gremlins_keepout < c.gremlins_size ? c.gremlins_size : c.gremlins_keepout;
  D.k_pillar = c.pillars_keepout < c.pillars_size ? c.pillars_size : c.pillars_keepout;
  D.max_bound = c.max_bound; D.ctrl_range_scale = c.robot_ctrl_range_scale; D.random_bound = c.random_bound;
  D.seed = c.seed; D.gid_base = c.env_id_base;  // (the library also writes the key into the slab: sag_create)
  D.max_layout_draws = c.max_layout_draws; D.max_episode_steps = c.max_episode_steps;
  D.num_gremlins = c.num_gremlins; D.gremlins_travel = c.gremlins_travel;
}

// sag_copy_envs: the two handles must have defined the same tasks in the same order (the ids are part of the state)
inline bool custom_tables_differ(const CustomTable& a, const CustomTable& b) {
  if (a.count != b.count) return true;
  for (int i = 0; i < a.count; ++i) {
    const CustomTask &x = a.t[i], &y = b.t[i];
    if (x.base != y.base || x.sp.nh != y.sp.nh || x.sp.nv != y.sp.nv || x.sp.ng != y.sp.ng || x.sp.np != y.sp.np) return true;
    for (int k = 0; k < 4; ++k) if (x.ext[k] != y.ext[k]) return true;
  }
  return false;
}

// sag_copy_envs: two handles whose environments can exchange states -- every configuration value that the layout
// samplers or the step read from Dev, except the Philox key, the global ids and the per-handle budgets (n_envs,
// max_episode_steps, max_layout_draws, action_noise).  Returns the first difference, or nullptr.
// ta / tb: host copies of the handles' user-defined task tables, which must be equal (the ids are part of the state).
inline const char* copy_incompatibility(const Dev& a, const Dev& b, const CustomTable* ta = nullptr,
                                        const CustomTable* tb = nullptr) {
  if (ta && tb && custom_tables_differ(*ta, *tb)) return "user-defined tasks";
  if (a.robot != b.robot) return "robot";
  if (a.num_gremlins != b.num_gremlins) return "num_gremlins";
  if (a.hazards_size != b.hazards_size || a.vases_size != b.vases_size || a.pillars_size != b.pillars_size ||
      a.gremlins_size != b.gremlins_size)
    return "object size";
  if (a.k_hazard != b.k_hazard || a.k_vase != b.k_vase || a.k_gremlin != b.k_gremlin || a.k_pillar != b.k_pillar)
    return "keepout";
  if (a.placements_margin != b.placements_margin) return "placements_margin";
  if (a.robot_keepout != b.robot_keepout) return "robot_keepout";
  if (a.gremlins_travel != b.gremlins_travel) return "gremlins_travel";
  if (a.ctrl_range_scale != b.ctrl_range_scale) return "robot_ctrl_range_scale";
  if (a.random_bound != b.random_bound) return "random_bound";
  if (a.max_bound != b.max_bound) return "max_bound";
  return nullptr;
}

static_assert(SAG_MAX_CUSTOM_TASKS == kMaxCustomTasks, "the ABI's and the kernels' custom-task capacity");

// sag_define_task: the definition's errors, or nullptr.  `base` must be a registry id.
inline const char* task_def_error(const SagTaskDef& d, int num_gremlins) {
  if (d.base_task < 0 || d.base_task >= SAG_NUM_TASKS) return "base_task must be a registry task id [0, SAG_NUM_TASKS)";
  for (int k = 0; k < 4; ++k) if (d.obstacles[k] < 0) return "obstacle counts must be >= 0";
  if (d.obstacles[2] != num_gremlins) return "obstacles[2] (gremlins) must equal the handle's num_gremlins";
  const TaskSpec b = task_spec(d.base_task);
  const int task_objects = b.kind == 0 ? 1 : b.kind == 1 ? b.nbuttons : 2;
  if ((long)d.obstacles[0] + d.obstacles[1] + d.obstacles[2] + d.obstacles[3] + task_objects > SAG_MAX_SLOTS)
    return "hazards + vases + gremlins + pillars + the base task's objects exceed SAG_MAX_SLOTS";
  const double* x = d.placement_extents;
  if (!(x[0] < x[2]) || !(x[1] < x[3])) return "placement_extents need x_min < x_max and y_min < y_max";
  return nullptr;
}

// the table entry of a valid definition: the base's descriptor with the definition's counts and extents
inline CustomTask custom_task(const SagTaskDef& d) {
  CustomTask c;
  memset(&c, 0, sizeof(c));
  c.sp = task_spec(d.base_task);
  c.sp.nh = d.obstacles[0]; c.sp.nv = d.obstacles[1]; c.sp.ng = d.obstacles[2]; c.sp.np = d.obstacles[3];
  c.base = d.base_task;
  for (int k = 0; k < 4; ++k) c.ext[k] = d.placement_extents[k];
  return c;
}

// sag_copy_envs_host: the checks the device path makes per pair (copy_env_source), for a whole host index array, so
// that a bad array fails the call instead of being reported afterwards.  Returns nullptr or the message.
inline const char* copy_index_error(const int32_t* src_of_dst, int n_dst, int n_src, bool same_handle) {
  for (int j = 0; j < n_dst; ++j) {
    const int s = src_of_dst[j];
    if (s < -1 || s >= n_src) return "source index out of range [-1, source n_envs)";
    if (same_handle && s >= 0 && s != j && src_of_dst[s] != -1 && src_of_dst[s] != s)
      return "a source environment is itself overwritten by the same call";
  }
  return nullptr;
}

}  // namespace sag
