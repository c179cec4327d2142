/*
 * sag_b200.h -- C ABI of the B200-native batched safe-adaptation-gym hot path.
 *
 * Drop-in boundary.  In the reference the only door from the environment / world / task code to the
 * simulator is the Python class MujocoBridge (safe_adaptation_gym/mujoco_bridge.py:15-280) and the env
 * methods built on it (safe_adaptation_gym/safe_adaptation_gym.py:56-107).  This library replaces that
 * whole per-step path (dynamics -> reward / goal logic -> cost -> pseudo-lidar observation, plus layout
 * rejection sampling at reset) for N environments at once.  Each entry point below names the reference
 * interface it stands in for.  INTEGRATION.md shows the ctypes stub a reference maintainer would add.
 *
 * Conventions: extern "C", plain pointers and sizes, no C++ / torch types.  Every call returns an int
 * status (0 = ok); sag_last_error() gives the message of the last failure on the calling thread.
 * Launches are asynchronous on the caller's cudaStream_t (passed as void*).  The caller owns all I/O
 * buffers; the library owns the handle's internal SoA state.  A handle is not thread-safe; several handles (on one or
 * several devices) may coexist in a process: every entry point switches to the handle's device and restores the
 * caller's.  The *_host entry points are synchronous and ordered after everything issued earlier on the device; the
 * stream entry points are ordered by the caller's stream.
 *
 * CUDA graphs.  These stream entry points may be recorded in a CUDA graph (stream capture) and the graph replayed any
 * number of times: sag_step, sag_reset_obs / sag_reset with a mask or only_flagged != 0, sag_export_outputs,
 * sag_observe, sag_rollout, sag_read_field / sag_write_field, sag_task_stats, sag_set_next_tasks, sag_bound,
 * sag_copy_envs and sag_evaluate_actions.  A replay
 * behaves exactly like issuing the same calls again: everything the kernels read that can change after sag_create (the
 * work-list counter sets and the step epoch that selects them, the Philox key, the task ids, the queued next tasks)
 * lives in the handle's device memory, so sag_seed and sag_set_tasks issued between replays are seen by the graph.  The
 * *_host entry points, sag_seed, sag_set_tasks_host, sag_set_next_tasks_host, sag_bound_host, sag_copy_envs_host,
 * sag_create / sag_destroy, sag_define_task
 * and sag_probe_d2h synchronise and must not be called while a capture is open.  The first sag_define_task of a handle
 * switches it to the kernel set that reads the user-defined task table, so a graph captured before it must be captured
 * again.  sag_launch_count counts host-side enqueues only: replays do not add to it.  Conditions recorded by replayed
 * kernels are read with sag_error_flags as usual.
 */
#ifndef SAG_B200_H
#define SAG_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAG_ABI_VERSION 3
#define SAG_LIDAR_BINS 16   /* safe_adaptation_gym.py:22 */
#define SAG_OBS_POINT 60    /* 3*16 lidar + 12 sensor floats, safe_adaptation_gym.py:120-139,225-237 */
#define SAG_OBS_CAR 72      /* + ballangvel_rear (3) + quat2mat(ballquat_rear) (9), car.xml:37-38 */
#define SAG_MAX_SLOTS 32
#define SAG_MAX_GREMLINS 4
#define SAG_MAX_CUSTOM_TASKS 16  /* user-defined tasks per handle (sag_define_task) */

enum { SAG_ROBOT_POINT = 0, SAG_ROBOT_CAR = 1 };
/* task ids: alphabetical registry order of the reference, benchmark/__init__.py:16-20 */
enum {
  SAG_T_CATCH_GOAL = 0, SAG_T_COLLECT, SAG_T_DRIBBLE_BALL, SAG_T_GO_TO_GOAL, SAG_T_GO_TO_GOAL_DAMPING,
  SAG_T_GO_TO_GOAL_MOTOR, SAG_T_GO_TO_GOAL_SCARCE, SAG_T_HAUL_BOX, SAG_T_PRESS_BUTTONS,
  SAG_T_PRESS_BUTTONS_SCARCE, SAG_T_PUSH_BOX, SAG_T_PUSH_BOX_SCARCE, SAG_T_ROLL_ROD, SAG_T_UNSUPERVISED,
  SAG_NUM_TASKS
};
/* per-env flag bits (sag_read_field(SAG_F_FLAGS)) */
enum { SAG_FLAG_PHYSICS_ERROR = 1, SAG_FLAG_RESAMPLE_FAILED = 2, SAG_FLAG_NEEDS_RESET = 4 };
/* additional bits of sag_error_flags() */
enum { SAG_ERR_BAD_TASK_ID = 8, SAG_ERR_BAD_ENV_INDEX = 16 };

/* World.DEFAULT (world.py:17-34) + batching parameters.  POD, copied at sag_create. */
typedef struct SagConfig {
  int32_t n_envs;             /* environments on this device */
  int32_t robot;              /* SAG_ROBOT_* */
  uint64_t seed;              /* Philox key */
  uint32_t env_id_base;       /* global id of env 0 (multi-GPU sharding: results do not depend on the GPU count) */
  int32_t max_episode_steps;  /* 0 = never flag NEEDS_RESET on step count (reference behaviour) */
  int32_t max_layout_draws;   /* draw budget of one layout rejection sampling; 0 = 1<<22 */
  int32_t random_bound;       /* world.py:33,75-78: constraint bound ~ U(0, max_bound) per Task instance instead of max_bound */
  double placements_margin, robot_keepout;
  double hazards_size, vases_size, pillars_size, gremlins_size;
  double hazards_keepout, gremlins_keepout, vases_keepout, pillars_keepout;
  double gremlins_travel, robot_ctrl_range_scale, action_noise, max_bound;
  int32_t num_gremlins;       /* Task.obstacles[2] (task.py:70) of a user-defined task: gremlins per environment, 0 .. SAG_MAX_GREMLINS.
                                 Every task of the reference's registry has 0; world.py:157-165, primitive_objects.py:57-86 */
  int32_t reserved_;
} SagConfig;

/* state fields for injection / extraction (parity tests, checkpointing).  All arrays are SoA,
 * environment-minor with element stride sag_stride(h):  field[k][env].  Together with the Philox key and the global
 * environment id they are the complete state of an environment: sag_copy_envs copies every row of every field. */
enum {
  SAG_F_ROBOT = 0,    /* double [6][stride]: x, y, yaw, vx, vy, w */
  SAG_F_OBJECTS = 1,  /* double [6][SAG_MAX_SLOTS][stride]: x, y, yaw, vx, vy, w per object slot */
  SAG_F_TASK_F64 = 2, /* double [15][stride]: last0,last1,cg_cur,cg_next,cg_ox,cg_oy,time,clearance,ep_return,ep_cost,ctrl0,ctrl1,
                         ctrl_scale0,ctrl_scale1 (world.py:72-73),bound (world.py:75-78) */
  SAG_F_TASK_I32 = 3, /* int32 [10][stride]: task, goal_button, btn_state, btn_timer, active_mask, cg_timer, n_step, step_ctr, episode,
                         moving_mask (derived; rebuilt by sag_observe after an injection) */
  SAG_F_FLAGS = 4,    /* uint8 [stride] */
  SAG_F_ROBOT_EXT = 5,/* double [6][stride]: car only -- wheel rates (2), castor ball-joint quaternion w,x,y,z (4) */
  SAG_F_GREMLINS = 6, /* double [2 + 3 * SAG_MAX_GREMLINS][stride]: mocap position of the last kinematics pass (x, y), then the weld
                         anchor (spawn x, y, yaw) of each gremlin */
  SAG_F_NEXT_TASK = 7,/* int32 [stride]: task queued for the environment's next reset, -1 = none (sag_set_next_tasks) */
  SAG_NUM_FIELDS
};

const char* sag_last_error(void);
int sag_abi_version(void);
void sag_default_config(SagConfig* cfg); /* world.py:17-34 defaults */

/* lifetime.  replaces SafeAdaptationGym.__init__ + MujocoBridge.__init__ (safe_adaptation_gym.py:30-54).
 * Side effect on the device: cudaLimitStackSize is raised (never lowered) to the largest stack frame of the library's kernels
 * (about 1.7 KB), so that the driver does not re-size its local-memory pool -- a device-wide stall of tens to hundreds of
 * milliseconds -- whenever an observation / auto-reset kernel follows a run of step kernels. */
int sag_create(const SagConfig* cfg, int device, void** handle);
int sag_destroy(void* handle);
int sag_stride(void* handle);
int sag_obs_dim(void* handle);
size_t sag_field_bytes(void* handle, int field);
/* number of CUDA kernels launched on behalf of this handle so far (bench.py's gpu_launches is a difference of two reads) */
unsigned long long sag_launch_count(void* handle);
/* tuning hook: section clocks of the contact kernel, 18 x u64 into a HOST buffer, zeroed after the read.  All zero
 * unless the library was built with -DSAG_TIMING (tools/late_phase.py). */
int sag_debug_read(void* handle, unsigned long long* out18_host);

/* env.set_task (safe_adaptation_gym.py:165-168): task_ids is a DEVICE int32[n_envs] array.  Statistics gathered under
 * the previous task are folded into the per-task totals first.  An id outside [0, sag_num_task_ids) is replaced by
 * SAG_T_GO_TO_GOAL and reported through sag_error_flags (SAG_ERR_BAD_TASK_ID). */
int sag_set_tasks(void* handle, const int32_t* task_ids_dev, void* stream);
/* same with a HOST int32[n_envs] array (validated: out-of-range ids fail the call); synchronous.  sag_set_tasks and
 * sag_set_tasks_host also clear every environment's queued next task. */
int sag_set_tasks_host(void* handle, const int32_t* task_ids_host);
/* Task switches at episode boundaries, per environment.  Every environment has a "next task" slot (SAG_F_NEXT_TASK,
 * -1 = none) that its next reset consumes, whichever path resets it: the auto-reset of sag_reset_obs(only_flagged = 1),
 * sag_reset / sag_reset_obs with or without a mask, sag_reset_host.  At that reset the environment (1) credits a
 * finished episode to the task it ran under, as every reset does, (2) folds its statistics into the per-task totals
 * under that old task, as sag_set_tasks does, (3) takes the queued id and clears the slot to -1, and (4) is reset as a
 * fresh Task instance of the new task (as with new_task != 0, for this environment only, even if the id is unchanged):
 * new ctrl-range scale and bound draws, new task state.  Environments with no task queued reset as the call asks.  A
 * queued id outside [0, sag_num_task_ids) is not applied: the slot is cleared and SAG_ERR_BAD_TASK_ID is reported through
 * sag_error_flags.
 * sag_set_next_tasks replaces every environment's slot from a DEVICE int32[n_envs] array (-1 = none); stream-ordered. */
int sag_set_next_tasks(void* handle, const int32_t* task_ids_dev, void* stream);
/* same with a HOST int32[n_envs] array (validated: an id outside [-1, sag_num_task_ids) fails the call); synchronous */
int sag_set_next_tasks_host(void* handle, const int32_t* task_ids_host);
/* info['bound'] (safe_adaptation_gym.py:79, world.py:75-78): DEVICE double[n_envs] constraint bound of every
 * environment's current Task instance; stream-ordered.  After task switches with SagConfig.random_bound this is how a
 * caller's bound buffer follows the new draws. */
int sag_bound(void* handle, double* bound_dev, void* stream);
/* same into a HOST double[n_envs] buffer; synchronous */
int sag_bound_host(void* handle, double* bound_host);
/* Sticky error conditions recorded by the kernels since the last call with clear != 0, readable WITHOUT synchronising
 * (the kernels write them into mapped host memory): SAG_FLAG_RESAMPLE_FAILED -- a layout (world.py:189) or a goal
 * (go_to_goal.py:80) could not be sampled, i.e. the reference would have raised ResamplingError out of reset / step;
 * SAG_ERR_BAD_TASK_ID; SAG_ERR_BAD_ENV_INDEX (sag_copy_envs).  A condition raised by a kernel that is still running
 * shows up in a later call. */
int sag_error_flags(void* handle, int clear);

/* Copy environment states, within one handle or from another handle of the same device (lookahead from the live
 * state, resets to chosen states).  src_of_dst holds one int32 per destination environment: every environment j of
 * `dst` with src_of_dst[j] = s >= 0 takes the complete state of environment s of `src` (src may be dst); -1 leaves j
 * untouched.  A gather: a destination never receives two sources, and one source may go to many destinations.
 *  - Copied: every row of every SAG_F_* field (robot, objects, task_f64, task_i32, flags, robot_ext, gremlins,
 *    next_task), bit for bit, also rows the robot model does not use.  The derived values (moving mask, clearance) come
 *    with them, so no sag_observe is needed.  So do the episode number and the in-step draw counter: with the same seed
 *    and an env_id_base that gives the copy the source's global id, the copy replays the source exactly (goal and
 *    button resamples, auto-resets, queued task switches); with another global id it follows the source until its
 *    first in-step draw.  The running return and cost (task_f64 rows 8-9) come too: the copy's episode is credited in
 *    full to dst when it finishes.
 *  - Not copied (they belong to the handle or the slot): the Philox key and the global id, so the copy draws from dst's
 *    streams; the finished-episode statistics; the work list, counter sets and step epoch; the error words.
 *  - Statistics: before its state is replaced, the destination is settled as a reset settles it: an episode that has
 *    finished (time limit or done) but has not been reset yet is credited to its OLD task, an unfinished one is dropped
 *    and not counted.  Its finished-episode statistics are then folded into dst's per-task totals under its OLD task
 *    and cleared (the rule of sag_set_tasks), so that sag_task_stats does not credit them to the copied task.
 *  - Aliasing: a pair j <- s with s != j is applied only if s is not itself overwritten by the call, i.e. src_of_dst[s]
 *    is -1 or s (dst == src only); j <- j does nothing.  Decided from the read-only index array: race-free, deterministic.
 *  - Compatibility: the call fails (nothing enqueued) unless both handles are on the same device and agree in robot,
 *    num_gremlins, every object size and (effective) keepout, placements_margin, robot_keepout, gremlins_travel,
 *    robot_ctrl_range_scale, random_bound and max_bound.  They may differ in n_envs, seed, env_id_base,
 *    max_episode_steps, max_layout_draws and action_noise.
 * sag_copy_envs: src_of_dst_dev is a DEVICE int32[dst n_envs] array; stream-ordered.  A pair whose index is outside
 * [-1, src n_envs) or that breaks the aliasing rule is not applied and SAG_ERR_BAD_ENV_INDEX is reported through
 * dst's sag_error_flags. */
int sag_copy_envs(void* dst, void* src, const int32_t* src_of_dst_dev, void* stream);
/* same with a HOST int32[dst n_envs] array (validated: an index out of range or a pair that breaks the aliasing rule
 * fails the call); synchronous */
int sag_copy_envs_host(void* dst, void* src, const int32_t* src_of_dst_host);

/* env.seed (safe_adaptation_gym.py:113-118): new Philox key; per-env episode counters restart */
int sag_seed(void* handle, uint64_t seed);

/* env.reset / _build_world (safe_adaptation_gym.py:85-107,170-172): layout rejection sampling
 * (world.py:172-217), yaw draws (world.py:108-137), fresh physics (mujoco_bridge.py:170-175), task.reset.
 * mask_dev: DEVICE uint8[n_envs] or NULL (= all).  only_flagged != 0 resets only envs whose NEEDS_RESET
 * flag is set (auto-reset).  new_task != 0 re-initialises task-instance state (a new Task object).
 * episode numbers are incremented per env (safe_adaptation_gym.py:97-100 `self._seed += 1`). */
int sag_reset(void* handle, const uint8_t* mask_dev, int only_flagged, int new_task, void* stream);
/* same, and the environments that were reset get the first observation of their new episode written into their row of
 * obs_dev (float[n][obs_dim]; other rows untouched); was_reset_dev (uint8[n], may be NULL) tells which.  This is the
 * auto-reset call of a vectorised wrapper: sag_step, then sag_reset_obs(only_flagged = 1) on the same buffers. */
int sag_reset_obs(void* handle, const uint8_t* mask_dev, int only_flagged, int new_task, float* obs_dev, uint8_t* was_reset_dev,
                  void* stream);
/* env.reset with HOST buffers: mask_host uint8[n] or NULL, obs_host float[n][obs_dim] or NULL (= env.observation of the
 * new episodes).  Synchronous, ordered after all earlier work of the device; fails when a layout could not be sampled. */
int sag_reset_host(void* handle, const uint8_t* mask_host, int only_flagged, int new_task, float* obs_host);

/* env.step (safe_adaptation_gym.py:56-83).  DEVICE buffers: act float[n][2]; obs float[n][obs_dim];
 * reward double[n]; reward2 double[n][2] or NULL (Unsupervised's 2-vector, unsupervised.py:66);
 * cost uint8[n] (world.py:155 binary); done uint8[n]. */
int sag_step(void* handle, const float* act, float* obs, double* reward, double* reward2, uint8_t* cost, uint8_t* done,
             void* stream);
/* env.observation (safe_adaptation_gym.py:120-131) at the current state; also refreshes internal caches
 * after sag_write_field. */
int sag_observe(void* handle, float* obs, void* stream);
/* same as sag_step with HOST buffers: H2D, kernels, D2H, sync; returns when the outputs are in the host buffers.
 * Page-locked buffers (sag_host_alloc, cudaHostRegister, torch pin_memory) take the overlapped path: the bulk copy runs
 * under the contact kernel and that kernel's rows follow as writes into the mapped buffers.  Steps of one handle must be
 * issued in order (one stream, or externally ordered streams): consecutive steps alternate two work-list counter sets,
 * selected by a step epoch in device memory. */
int sag_step_host(void* handle, const float* act_h, float* obs_h, double* reward_h, uint8_t* cost_h, uint8_t* done_h);
int sag_observe_host(void* handle, float* obs_h);
void* sag_host_alloc(size_t bytes);
/* measurement helper: `reps` back-to-back device -> pinned-host copies of `bytes` bytes with the allocation and copy calls of
 * sag_step_host; *seconds = elapsed time (CUDA events).  The host ceiling bench.py reports e2e against. */
int sag_probe_d2h(void* handle, size_t bytes, int reps, double* seconds);
/* the four output buffers of sag_step_host as ONE pinned block laid out like the library's device staging area, so that
 * a step needs a single device-to-host copy; free with sag_host_free(*obs_h) */
int sag_host_alloc_outputs(void* handle, float** obs_h, double** reward_h, uint8_t** cost_h, uint8_t** done_h);
void sag_host_free(void* p);

/* Score a horizon of actions: h_steps >= 1 steps with act[h] (DEVICE float[h_steps][n][2]), enqueued in one call:
 * h_steps x (the two step kernels).  Every environment takes all h_steps steps, exactly as h_steps sag_step calls with
 * act[0], act[1], ... would take them: afterwards every SAG_F_* field, the statistics and the Philox draw counters are
 * bit-identical to theirs (sag_step does not reset; neither does this call, also with a time limit).  Outputs, DEVICE:
 *   obs     float[n][obs_dim]: the observation of the last step (bit-identical to the last sag_step's);
 *   ret     double[n] (ret_cols = 1) or double[n][2] (ret_cols = 2, Unsupervised's pair, as sag_step's reward2);
 *   cost    double[n];  length  int32[n].
 * With w_0 = 1, w_{h+1} = w_h * discount (float64, formed on the host left to right) and L_e = min(h_steps, 1 + the
 * first step at which environment e reported done -- a physics error):
 *   ret[e] = sum over h < L_e of w_h * reward_h[e], cost[e] = the same with the binary step cost, length[e] = L_e,
 * each product rounded before it is added, summed in step order from zero.  With discount = 1 that is the sum a loop
 * `ret += reward` over sag_step calls forms, stopped at the first done.  Steps after L_e still run but do not count.
 * Only the last step builds the observation: the steps before it skip the lidar, the sensors and the observation
 * write-out.  Stream-ordered; may be recorded in a CUDA graph (h_steps and discount are fixed by the capture). */
int sag_evaluate_actions(void* handle, int h_steps, const float* act, double discount, float* obs, double* ret, int ret_cols,
                         double* cost, int32_t* length, void* stream);

/* The outputs of a step as fresh arrays in one launch (device pointers): obs rows, reward (reward_cols = 1, or 2 for the
 * Unsupervised task's pair), cost as float32 -- the reference returns float(cost > 0.), world.py:155 --, done as bool bytes,
 * and (bound_out != NULL) info['bound'].  What the reference's step() returns are new numpy arrays
 * (safe_adaptation_gym.py:80-83); the Python mirror hands out copies through this call. */
int sag_export_outputs(void* handle, const float* obs, const double* reward, int reward_cols, const uint8_t* cost, const uint8_t* done,
                       const double* bound, float* obs_out, double* reward_out, float* cost_out, uint8_t* done_out, double* bound_out,
                       void* stream);

/* K steps with on-device Philox U(-1,1) actions (stream 2, counter = the environment's step count), enqueued in one call:
 * K x (action kernel + the two step kernels); benchmark helper.  Writes the last step's obs/reward/cost/done (any may be
 * NULL). */
int sag_rollout(void* handle, int k_steps, float* obs, double* reward, uint8_t* cost, uint8_t* done, void* stream);

/* state injection / extraction; buffers are DEVICE pointers of sag_field_bytes(field) bytes */
int sag_read_field(void* handle, int field, void* dst_dev, void* stream);
int sag_write_field(void* handle, int field, const void* src_dev, void* stream);
/* User-defined tasks (a subclass of a registry task that overrides Task.obstacles and Task.placement_extents,
 * task.py:14-98).  base_task is the registry id whose reward, goal / button / box logic, dynamics variant and
 * goal / button / box rectangles the task keeps; obstacles = {hazards, vases, gremlins, pillars}; placement_extents =
 * {x_min, y_min, x_max, y_max}: free placements draw x in [x_min + k, x_max - k] and y in [y_min + k, y_max - k] for an
 * object of keepout k. */
typedef struct SagTaskDef {
  int32_t base_task;
  int32_t obstacles[4];
  double placement_extents[4];
} SagTaskDef;
/* Define a task on this handle; synchronous.  *task_id receives SAG_NUM_TASKS, SAG_NUM_TASKS + 1, ... in order of
 * definition.  Fails (nothing defined) unless base_task is a registry id, every count is >= 0, obstacles[2] equals
 * SagConfig.num_gremlins, hazards + vases + gremlins + pillars + the base's task objects <= SAG_MAX_SLOTS,
 * x_min < x_max, y_min < y_max, and fewer than SAG_MAX_CUSTOM_TASKS tasks are defined.  Once a handle has a definition,
 * sag_task_stats writes sag_num_task_ids rows, and sag_set_tasks*, sag_set_next_tasks* and the queued-task rule accept
 * ids below sag_num_task_ids (SAG_ERR_BAD_TASK_ID covers the ids outside it).  A layout that cannot be sampled is
 * reported at reset as for registry tasks (SAG_FLAG_RESAMPLE_FAILED). */
int sag_define_task(void* handle, const SagTaskDef* def, int32_t* task_id);
/* SAG_NUM_TASKS + the number of tasks defined on this handle */
int sag_num_task_ids(void* handle);

/* per-task statistics of the episodes that FINISHED (time limit or done) since the last call with reset != 0, under the
 * task they ran with: DEVICE double out[sag_num_task_ids(handle)][3] = {sum of episode returns, sum of episode costs, number of
 * episodes} (the buffer NCCL all-reduces).  Episodes cut short by a manual reset / set_task are not counted. */
int sag_task_stats(void* handle, double* out_dev, int reset, void* stream);

/* stand-alone streaming kernels on caller-provided SoA buffers (roofline evidence; SURVEY 8d)
 * lidar: SafeAdaptationGym._lidar x3 (safe_adaptation_gym.py:133-139,174-223)
 *   robot double[3][n] (x,y,yaw); obj_xy double[2][nslots][n]; group uint8[nslots][n] (0 skip,1,2,3);
 *   out float[n][48] = obstacles, objects, goal */
int sag_lidar(const double* robot, const double* obj_xy, const uint8_t* group, int n, int nslots, float* out, void* stream);
/* cost: World.compute_cost (world.py:144-155)
 *   robot_xy double[2][n]; hazard_xy float[2][nh][n]; contact uint8[n] (robot-obstacle contact flag); out uint8[n] */
int sag_cost(const double* robot_xy, const float* hazard_xy, const uint8_t* contact, int n, int nh, double hazard_size,
             uint8_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif
