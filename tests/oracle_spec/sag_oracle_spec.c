/* sag_oracle_spec.c -- TEST INFRASTRUCTURE ONLY: the CPU oracle (oracle/sag_oracle.c, compiled unchanged as part of
 * this file) plus orc_env_create_spec, an oracle environment built from an explicit task descriptor: a registry task
 * (the base: reward, goal / button / box logic, dynamics variant) with its own obstacle counts and placement extents,
 * as a user-defined Task subclass overriding Task.obstacles and Task.placement_extents (task.py:14-98) builds it.
 * tests/test_custom_tasks.py compares the library's user-defined tasks against it. */
#define orc_env_reset orc_env_reset_registry
#define orc_env_destroy orc_env_destroy_registry
#include "../../oracle/sag_oracle.c"
#undef orc_env_reset
#undef orc_env_destroy

/* world.py:53-102: an obstacle slot of the given type, keepout = max(keepout, size) (world.py:60-66) */
static orc_obj obstacle_slot(const orc_config* c, int type) {
  orc_obj o;
  memset(&o, 0, sizeof(o));
  o.type = type; o.group = ORC_GROUP_OBSTACLES;
  switch (type) {
    case ORC_HAZARD: o.keepout = c->hazards_keepout < c->hazards_size ? c->hazards_size : c->hazards_keepout; break;
    case ORC_VASE: o.keepout = c->vases_keepout < c->vases_size ? c->vases_size : c->vases_keepout; break;
    case ORC_GREMLIN: o.keepout = c->gremlins_keepout < c->gremlins_size ? c->gremlins_size : c->gremlins_keepout; break;
    default: o.keepout = c->pillars_keepout < c->pillars_size ? c->pillars_size : c->pillars_keepout; break;
  }
  return o;
}

/* the slots of a descriptor: the registry task's slots (setup_slots) with the obstacles re-laid and the extents replaced */
static void apply_spec(orc_env* e, const int obstacles[4], const double extents[4]) {
  const task_spec* t = &TASKS[e->task];
  const int base_t0 = t->obstacles[0] + t->obstacles[1] + obstacles[2] + t->obstacles[3];
  const int ntask = e->nobj - base_t0;
  const int t0 = obstacles[0] + obstacles[1] + obstacles[2] + obstacles[3];
  orc_obj task_obj[ORC_MAX_OBJ];
  int has_rect[ORC_MAX_OBJ];
  double rect[ORC_MAX_OBJ][4];
  for (int i = 0; i < ntask; ++i) {
    task_obj[i] = e->obj[base_t0 + i]; has_rect[i] = e->has_rect[base_t0 + i];
    memcpy(rect[i], e->rect[base_t0 + i], sizeof(rect[i]));
  }
  static const int kinds[4] = {ORC_HAZARD, ORC_VASE, ORC_GREMLIN, ORC_PILLAR};
  int n = 0;
  for (int k = 0; k < 4; ++k)
    for (int i = 0; i < obstacles[k]; ++i) { e->obj[n] = obstacle_slot(&e->cfg, kinds[k]); e->has_rect[n] = 0; ++n; }
  for (int i = 0; i < ntask; ++i, ++n) { e->obj[n] = task_obj[i]; e->has_rect[n] = has_rect[i]; memcpy(e->rect[n], rect[i], sizeof(rect[i])); }
  e->nobj = n;
  const int shift = t0 - base_t0;
  if (e->goal_slot >= 0) e->goal_slot += shift;
  if (e->box_slot >= 0) e->box_slot += shift;
  if (e->first_button >= 0) e->first_button += shift;
  if (e->tendon_slot >= 0) e->tendon_slot += shift;
  for (int k = 0; k < 4; ++k) e->extents[k] = extents[k];
}

/* the descriptors of the environments made by orc_env_create_spec (removed by orc_env_destroy) */
typedef struct { orc_env* e; int obstacles[4]; double extents[4]; } spec_entry;
static spec_entry* g_specs;
static int g_nspecs, g_capspecs;
static pthread_mutex_t g_specs_lock = PTHREAD_MUTEX_INITIALIZER;
static const spec_entry* spec_of(const orc_env* e) {
  const spec_entry* r = NULL;
  pthread_mutex_lock(&g_specs_lock);
  for (int i = 0; i < g_nspecs; ++i) if (g_specs[i].e == e) { r = &g_specs[i]; break; }
  pthread_mutex_unlock(&g_specs_lock);
  return r;
}

/* orc_env_reset (sag_oracle.c) with the descriptor's slots after setup_slots */
static int spec_env_reset(orc_env* e, uint32_t episode, const spec_entry* sp) {
  const task_spec* t = &TASKS[e->task];
  e->episode = episode; e->ctr[0] = e->ctr[1] = e->ctr[2] = 0;
  setup_slots(e);
  apply_spec(e, sp->obstacles, sp->extents);  /* the only change: the descriptor's slots and extents */
  /* World.__init__, world.py:72-78: Task.ctrl_scale (standard Cauchy per actuator, task.py:85-89) and
   * Task.constraint_bound (U(0, max_bound), task.py:91-94) are drawn once per Task instance and cached on it, so they
   * survive env.reset() and change with env.set_task / reset(options={'task': ...}).  Philox stream 3; Cauchy by
   * inversion tan(pi (u - 1/2)).  Not drawn in replay mode (the golden harness injects the reference's ranges). */
  if (e->new_task) {
    e->new_task = 0;
    if (!e->replay_mode) {
      double u[2];
      orc_philox_uniform2(e->seed, 0u, episode, e->gid, 3u, u);
      for (int k = 0; k < 2; ++k) {
        double sn, cs;
        sag_sincos(PI_D * (u[k] - 0.5), &sn, &cs);
        double sc = (sn / cs) * e->cfg.robot_ctrl_range_scale + 1.0;
        e->ctrl_lo[k] = -1.0 * sc; e->ctrl_hi[k] = 1.0 * sc;         /* mujoco_bridge.py:164-166 */
      }
      orc_philox_uniform2(e->seed, 1u, episode, e->gid, 3u, u);
      e->bound = e->cfg.random_bound ? 0.0 + (e->cfg.max_bound - 0.0) * u[0] : e->cfg.max_bound;
    }
  }
  e->draws_left = e->cfg.max_layout_draws > 0 ? e->cfg.max_layout_draws : (1L << 22);
  /* World._generate_new_layout, world.py:172-189 (10000 attempts; the extents-growth fallback is
   * broken in the reference -- quirk D12 -- and is treated as ResamplingError) */
  double rxy[2] = {0, 0};
  int ok = 0;
  for (int a = 0; a < 10000; ++a) { int r = sample_layout(e, rxy); if (r < 0) break; if (r) { ok = 1; break; } }
  if (!ok) return 1;
  /* World._build_world_config, world.py:108-137: yaw draws */
  e->robot_rot = TWO_PI * rng_single(e, 0);                /* :115, utils.py:11-13 */
  for (int s = 0; s < e->nobj; ++s) {
    int ty = e->obj[s].type;
    if (ty == ORC_HAZARD || ty == ORC_VASE || ty == ORC_GREMLIN || ty == ORC_PILLAR) e->obj[s].yaw = TWO_PI * rng_single(e, 0);
  }
  if (e->task == ORC_T_HAUL_BOX) {                         /* haul_box.py:17-18, quirk D16 */
    e->obj[e->box_slot].x = rxy[0] + BOX_SIZE * 3.0; e->obj[e->box_slot].y = rxy[1];
  }
  if (t->kind == 0 || t->kind == 2) e->obj[e->goal_slot].yaw = TWO_PI * rng_single(e, 0); /* go_to_goal.py:26-27 */
  if (t->kind == 2 && t->box_type == ORC_BOX) e->obj[e->box_slot].yaw = TWO_PI * rng_single(e, 0); /* push_box.py:35 */
  if (t->kind == 1) for (int i = 0; i < e->nbuttons; ++i) e->obj[e->first_button + i].yaw = TWO_PI * rng_single(e, 0); /* press_buttons.py:35 */
  /* MujocoBridge.rebuild: fresh physics, mujoco_bridge.py:170-175 */
  e->q[0] = rxy[0]; e->q[1] = rxy[1]; e->q[2] = e->robot_rot;
  e->v[0] = e->v[1] = e->v[2] = 0.0; e->ctrl[0] = e->ctrl[1] = 0.0;
  e->wheel_w[0] = e->wheel_w[1] = 0.0; e->cq[0] = 1.0; e->cq[1] = e->cq[2] = e->cq[3] = 0.0;
  e->time = 0.0; e->error = 0;
  /* gremlins: weld anchor = spawn pose; the mocap bodies start at the world origin (primitive_objects.py:24-31,71-77) */
  e->mocap_pos[0] = e->mocap_pos[1] = e->mocap_kin[0] = e->mocap_kin[1] = 0.0;
  for (int s = 0; s < e->nobj; ++s) { e->gspawn[s][0] = e->obj[s].x; e->gspawn[s][1] = e->obj[s].y; e->gspawn[s][2] = e->obj[s].yaw; }
  orc_phys_forward(e);
  /* World.reset -> task.reset, world.py:167-170 */
  if (task_reset(e, 0)) return 1;
  orc_phys_forward(e);
  return 0;
}

int orc_env_reset(orc_env* e, uint32_t episode) {
  const spec_entry* sp = spec_of(e);
  return sp ? spec_env_reset(e, episode, sp) : orc_env_reset_registry(e, episode);
}

void orc_env_destroy(orc_env* e) {
  pthread_mutex_lock(&g_specs_lock);
  for (int i = 0; i < g_nspecs; ++i) if (g_specs[i].e == e) { g_specs[i] = g_specs[--g_nspecs]; break; }
  pthread_mutex_unlock(&g_specs_lock);
  orc_env_destroy_registry(e);
}

/* obstacles = {hazards, vases, gremlins, pillars}; extents = {x_min, y_min, x_max, y_max}.  NULL if the slots do not
 * fit.  The gremlin count is obstacles[2] (cfg->num_gremlins is ignored). */
orc_env* orc_env_create_spec(int robot, int base_task, const int obstacles[4], const double extents[4], const orc_config* cfg) {
  orc_config c;
  if (cfg) c = *cfg; else orc_default_config(&c);
  c.num_gremlins = obstacles[2];
  orc_env* e = orc_env_create(robot, base_task, &c);
  const task_spec* t = &TASKS[base_task];
  const int ntask = e->nobj - (t->obstacles[0] + t->obstacles[1] + obstacles[2] + t->obstacles[3]);
  if (obstacles[0] + obstacles[1] + obstacles[2] + obstacles[3] + ntask > ORC_MAX_OBJ) { orc_env_destroy(e); return NULL; }
  apply_spec(e, obstacles, extents);
  pthread_mutex_lock(&g_specs_lock);
  if (g_nspecs == g_capspecs) {
    g_capspecs = g_capspecs ? 2 * g_capspecs : 64;
    g_specs = (spec_entry*)realloc(g_specs, (size_t)g_capspecs * sizeof(spec_entry));
  }
  spec_entry* s = &g_specs[g_nspecs++];
  s->e = e;
  memcpy(s->obstacles, obstacles, sizeof(s->obstacles));
  memcpy(s->extents, extents, sizeof(s->extents));
  pthread_mutex_unlock(&g_specs_lock);
  return e;
}
