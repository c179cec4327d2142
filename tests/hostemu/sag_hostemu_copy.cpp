// sag_hostemu_copy.cpp -- TEST INFRASTRUCTURE ONLY (never loaded by the product package).
//
// The host emulation with the next-task slot (sag_hostemu_next_task.cpp, compiled unchanged as part of this file) plus
// the environment copies of the CUDA library: tests/test_copy_envs.py runs its cases on the CPU against it.  The
// additions mirror sag_kernels.cu:
//   - sag_copy_envs / sag_copy_envs_host, as declared in include/sag_b200.h: the same compatibility check
//     (copy_incompatibility) and host-index validation (copy_index_error) as the library, and per destination the pair
//     rule and statistics settlement of copy_env_source (sag_core.cuh) -- the code k_copy_envs_fold runs -- before
//     every row of every field (kFieldShape, sag_layout.h) is copied;
//   - SAG_ERR_BAD_ENV_INDEX in sag_error_flags (error word 2, as in the library).
#define sag_error_flags sag_error_flags_without_index
#include "sag_hostemu_next_task.cpp"
#undef sag_error_flags

namespace {
int copy_check(Handle* H, Handle* S, const char* who) {
  if (!H || !S) { snprintf(g_err, sizeof(g_err), "%s: null handle", who); return 1; }
  if (const char* what = copy_incompatibility(H->D, S->D)) {
    snprintf(g_err, sizeof(g_err), "%s: the handles differ in %s", who, what);
    return 1;
  }
  return 0;
}
}  // namespace

extern "C" {
int sag_error_flags(void* h, int clear) {
  Handle* H = (Handle*)h;
  const int w = sag_error_flags_without_index(h, clear) | (H->err[2] ? SAG_ERR_BAD_ENV_INDEX : 0);
  if (clear) H->err[2] = 0;
  return w;
}
int sag_copy_envs(void* dst, void* src, const int32_t* src_of_dst, void* s) {
  (void)s;
  Handle *H = (Handle*)dst, *S = (Handle*)src;
  if (!src_of_dst) return fail("sag_copy_envs: null argument");
  if (copy_check(H, S, "sag_copy_envs")) return 1;
  const size_t dst_st = H->D.stride, src_st = S->D.stride;
  // Sources are never destinations of the same call (the pair rule), so the order of the destinations does not matter.
  for (int j = 0; j < H->D.n; ++j) {
    const int e = copy_env_source(H->D, src_of_dst, j, S->D.n, H == S, true, H->sret, H->scost, H->sn, H->stats_acc);
    if (e < 0) continue;
    for (int f = 0; f < SAG_NUM_FIELDS; ++f) {
      const int elem = kFieldShape[f].elem;
      char* d = H->slab + H->LY.off[f];
      const char* o = S->slab + S->LY.off[f];
      for (int r = 0; r < kFieldShape[f].rows; ++r)
        memcpy(d + (r * dst_st + j) * elem, o + (r * src_st + e) * elem, elem);
    }
  }
  return 0;
}
int sag_copy_envs_host(void* dst, void* src, const int32_t* src_of_dst) {
  Handle *H = (Handle*)dst, *S = (Handle*)src;
  if (!src_of_dst) return fail("sag_copy_envs_host: null argument");
  if (copy_check(H, S, "sag_copy_envs_host")) return 1;
  if (const char* what = copy_index_error(src_of_dst, H->D.n, S->D.n, H == S)) {
    snprintf(g_err, sizeof(g_err), "sag_copy_envs_host: %s", what);
    return 1;
  }
  return sag_copy_envs(dst, src, src_of_dst, nullptr);
}
}
