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
  size_t stats_off, sched_off, act_off, obs_off, rew_off, cost_off, done_off, acc_off, ids_off, mask_off, total;
};

inline SlabLayout slab_layout(int n, int stride, int obs_dim) {
  SlabLayout L;
  const size_t st = (size_t)stride;
  L.bytes[SAG_F_ROBOT] = 6 * st * sizeof(double);
  L.bytes[SAG_F_OBJECTS] = 6 * (size_t)SAG_MAX_SLOTS * st * sizeof(double);
  L.bytes[SAG_F_TASK_F64] = 15 * st * sizeof(double);
  L.bytes[SAG_F_TASK_I32] = 10 * st * sizeof(int32_t);
  L.bytes[SAG_F_FLAGS] = st;
  L.bytes[SAG_F_ROBOT_EXT] = 6 * st * sizeof(double);
  L.bytes[SAG_F_GREMLINS] = (2 + 3 * (size_t)SAG_MAX_GREMLINS) * st * sizeof(double);
  size_t total = 0;
  for (int f = 0; f < SAG_NUM_FIELDS; ++f) { L.off[f] = total; total += align_up(L.bytes[f], 256); }
  L.stats_off = total; total += align_up(3 * st * sizeof(double), 256);
  L.sched_off = total; total += align_up((3 * st + 96) * sizeof(int32_t), 256);
  L.act_off = total; total += align_up((size_t)n * 2 * sizeof(float), 256);
  L.obs_off = total; total += align_up((size_t)n * obs_dim * sizeof(float), 256);
  L.rew_off = total; total += align_up((size_t)n * sizeof(double), 256);
  L.cost_off = total; total += align_up((size_t)n, 256);
  L.done_off = total; total += align_up((size_t)n, 256);
  L.acc_off = total; total += align_up(SAG_NUM_TASKS * 3 * sizeof(double), 256);
  L.ids_off = total; total += align_up((size_t)n * sizeof(int32_t), 256);
  L.mask_off = total; total += align_up((size_t)n, 256);
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
  // multiple of 96)
  D.worklist = sc; D.counts = sc + 3 * st;
  D.dbg = (unsigned long long*)(sc + 3 * st + 16);
  D.epoch = (unsigned*)(sc + 3 * st + 52);
  D.key = (unsigned long long*)(sc + 3 * st + 54);
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

}  // namespace sag
