// sag_hostemu_next_task.cpp -- TEST INFRASTRUCTURE ONLY (never loaded by the product package).
//
// The host emulation of sag_hostemu.cpp (the kernel body compiled with g++ behind the C ABI) with the per-environment
// "next task" slot (SAG_F_NEXT_TASK) of the CUDA library: tests/test_task_switch.py runs the task-switch cases on the
// CPU against it.  sag_hostemu.cpp is compiled unchanged as part of this file; the names below are redirected to the
// additions, which mirror sag_kernels.cu:
//   - every reset goes through take_next_task (sag_core.cuh), the helper k_reset calls from the lane that resets an
//     environment, before env_reset -- the same code the GPU runs, after the same crediting of a finished episode;
//   - sag_create fills the slots with -1 (no task queued), sag_set_tasks clears them;
//   - sag_set_next_tasks / sag_set_next_tasks_host / sag_bound, as declared in include/sag_b200.h.
#include "../../include/sag_b200.h"
#include "../../safe_adaptation_gym_b200/csrc/sag_core.cuh"
#include "../../safe_adaptation_gym_b200/csrc/sag_layout.h"

namespace sag {
template <class RB>
void reset_taking_next_task(const Dev& D, int e, uint32_t episode, bool new_task);
}

#define env_reset reset_taking_next_task
#define sag_create sag_create_without_slots
#define sag_set_tasks sag_set_tasks_keeping_slots
#include "sag_hostemu.cpp"
#undef env_reset
#undef sag_create
#undef sag_set_tasks

namespace {
int32_t* next_task_slots(Handle* H) { return (int32_t*)(H->slab + H->LY.off[SAG_F_NEXT_TASK]); }
}  // namespace

namespace sag {
// do_reset of sag_hostemu.cpp passes H->D, the first member of its Handle
template <class RB>
void reset_taking_next_task(const Dev& D, int e, uint32_t episode, bool new_task) {
  Handle* H = reinterpret_cast<Handle*>(const_cast<Dev*>(&D));
  const bool fresh = take_next_task(D, e, next_task_slots(H), H->sret, H->scost, H->sn, H->stats_acc, new_task);
  env_reset<RB>(D, e, episode, fresh);
}
}  // namespace sag

extern "C" {
int sag_create(const SagConfig* cfg, int device, void** handle) {
  const int rc = sag_create_without_slots(cfg, device, handle);
  if (rc == 0) {
    Handle* H = (Handle*)*handle;
    memset(next_task_slots(H), 0xFF, (size_t)H->D.stride * sizeof(int32_t));  // -1: no task queued
  }
  return rc;
}
int sag_set_tasks(void* h, const int32_t* ids, void* s) {
  const int rc = sag_set_tasks_keeping_slots(h, ids, s);
  Handle* H = (Handle*)h;
  memset(next_task_slots(H), 0xFF, (size_t)H->D.stride * sizeof(int32_t));
  return rc;
}
int sag_set_next_tasks(void* h, const int32_t* ids, void* s) {
  (void)s; Handle* H = (Handle*)h;
  memcpy(next_task_slots(H), ids, (size_t)H->D.n * sizeof(int32_t));
  return 0;
}
int sag_set_next_tasks_host(void* h, const int32_t* ids) {
  Handle* H = (Handle*)h;
  for (int e = 0; e < H->D.n; ++e)
    if (ids[e] < -1 || ids[e] >= SAG_NUM_TASKS) return fail("sag_set_next_tasks_host: task id out of range [-1, SAG_NUM_TASKS)");
  return sag_set_next_tasks(h, ids, nullptr);
}
int sag_bound(void* h, double* bound, void* s) {
  (void)s; Handle* H = (Handle*)h;
  memcpy(bound, H->D.bound, (size_t)H->D.n * sizeof(double));
  return 0;
}
}
