// sag_hostemu_custom.cpp -- TEST INFRASTRUCTURE ONLY (never loaded by the product package).
//
// The host emulation with sag_evaluate_actions (sag_hostemu_evaluate.cpp and the files it includes, compiled unchanged
// as part of this file) plus the user-defined tasks of the CUDA library: tests/test_custom_tasks.py runs its cases on
// the CPU against it.  The additions mirror sag_kernels.cu:
//   - every handle runs the *C instantiations (sag_core.cuh: PointRobotC, ...), the ones the library switches a handle
//     to at its first sag_define_task; for registry ids they compute what the default ones compute;
//   - the emulation's contact-free dispatch loads the robot with spec_for, as k_step_free of the *C instantiations;
//   - the queued-task rule (take_next_task), the copy settlement (copy_env_source), sag_set_tasks*, sag_set_next_tasks_host
//     and sag_task_stats follow sag_num_task_ids, and the copy compatibility check compares the task tables;
//   - sag_define_task / sag_num_task_ids, as declared in include/sag_b200.h, with the library's validation
//     (task_def_error) and table entry (custom_task, sag_layout.h), written to the table in the slab.
#include "../../include/sag_b200.h"
#include "../../safe_adaptation_gym_b200/csrc/sag_core.cuh"
#include "../../safe_adaptation_gym_b200/csrc/sag_layout.h"

#define PointRobot PointRobotC
#define PointRobotG PointRobotGC
#define CarRobot CarRobotC
#define CarRobotG CarRobotGC
#define load_robot(D, e, sp, R) sag::load_robot(D, e, sag::spec_for(D, (D).task[e], false, true), R)
#define take_next_task(D, e, slots, r, c, n, acc, fresh) \
  sag::take_next_task(D, e, slots, r, c, n, acc, fresh, sag::num_task_ids(D, true))
#define copy_env_source(D, idx, j, n_src, same, fold, r, c, n, acc) \
  sag::copy_env_source(D, idx, j, n_src, same, fold, r, c, n, acc, sag::num_task_ids(D, true))
#define copy_incompatibility(a, b) sag::copy_incompatibility(a, b, &sag::custom_table(a), &sag::custom_table(b))
// the id bound of the emulation's sag_set_tasks, sag_set_next_tasks_host and sag_task_stats (each has its handle in H)
#define SAG_NUM_TASKS (sag_num_task_ids(H))
#include "sag_hostemu_evaluate.cpp"
#undef SAG_NUM_TASKS

extern "C" {
int sag_num_task_ids(void* h) { return h ? num_task_ids(((Handle*)h)->D, true) : (int)SAG_NUM_TASKS; }
int sag_define_task(void* h, const SagTaskDef* def, int32_t* task_id) {
  Handle* H = (Handle*)h;
  if (!H || !def || !task_id) return fail("sag_define_task: null argument");
  if (const char* what = task_def_error(*def, H->D.num_gremlins)) {
    snprintf(g_err, sizeof(g_err), "sag_define_task: %s", what);
    return 1;
  }
  CustomTable& T = const_cast<CustomTable&>(custom_table(H->D));
  if (T.count >= SAG_MAX_CUSTOM_TASKS) return fail("sag_define_task: SAG_MAX_CUSTOM_TASKS tasks are defined already");
  T.t[T.count] = custom_task(*def);
  *task_id = SAG_NUM_TASKS + T.count;
  ++T.count;
  return 0;
}
}
