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
/* additional bit of sag_error_flags() */
enum { SAG_ERR_BAD_TASK_ID = 8 };

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
 * environment-minor with element stride sag_stride(h):  field[k][env]. */
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
 * the previous task are folded into the per-task totals first.  An id outside [0, SAG_NUM_TASKS) is replaced by
 * SAG_T_GO_TO_GOAL and reported through sag_error_flags (SAG_ERR_BAD_TASK_ID). */
int sag_set_tasks(void* handle, const int32_t* task_ids_dev, void* stream);
/* same with a HOST int32[n_envs] array (validated: out-of-range ids fail the call); synchronous */
int sag_set_tasks_host(void* handle, const int32_t* task_ids_host);
/* info['bound'] (safe_adaptation_gym.py:79, world.py:75-78): HOST double[n_envs] constraint bound of every environment's
 * current Task instance; synchronous */
int sag_bound_host(void* handle, double* bound_host);
/* Sticky error conditions recorded by the kernels since the last call with clear != 0, readable WITHOUT synchronising
 * (the kernels write them into mapped host memory): SAG_FLAG_RESAMPLE_FAILED -- a layout (world.py:189) or a goal
 * (go_to_goal.py:80) could not be sampled, i.e. the reference would have raised ResamplingError out of reset / step;
 * SAG_ERR_BAD_TASK_ID.  A condition raised by a kernel that is still running shows up in a later call. */
int sag_error_flags(void* handle, int clear);

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
 * issued in order (one stream, or externally ordered streams): consecutive steps alternate two work-list counter sets. */
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
/* per-task statistics of the episodes that FINISHED (time limit or done) since the last call with reset != 0, under the
 * task they ran with: DEVICE double out[SAG_NUM_TASKS][3] = {sum of episode returns, sum of episode costs, number of
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
