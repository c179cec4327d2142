// sag_hostemu_evaluate.cpp -- TEST INFRASTRUCTURE ONLY (never loaded by the product package).
//
// The host emulation with the environment copies (sag_hostemu_copy.cpp, compiled unchanged as part of this file) plus
// sag_evaluate_actions of the CUDA library: tests/test_evaluate_actions.py runs its small cases on the CPU against it.
// The addition mirrors sag_kernels.cu (Ops::evaluate): H steps, each with the dispatch of do_step (the contact-free
// path, and the full path where its pre-test bails), the observation-free env_step instantiations (Obs = false) before
// the last step, and eval_accumulate (sag_core.cuh) where a step stores its reward, cost and done.
#include "sag_hostemu_copy.cpp"

namespace {
template <class RB, bool Obs>
void eval_step(Handle* H, const float* act, float* obs, const EvalAcc& A) {
  Dev& D = H->D;
  static float tile[kObsMax * kTileStride];
  static Scratch scratch;
  for (int e0 = 0; e0 < D.n; e0 += kBS) {
    for (int t = 0; t < kBS && e0 + t < D.n; ++t) {
      const int e = e0 + t;
      double rew[2];
      unsigned char c, d;
      bool run = false, pretest = false;
      {
        RB R;
        load_robot(D, e, task_spec(D.task[e]), R);
        run = !(D.flags[e] & F_PHYS_ERROR) && D.movmask[e] == 0 && D.num_gremlins == 0;
        pretest = !env_is_quiet(D.clear[e], R);
      }
      bool bail = true;
      if (run) bail = env_step<kStepNear, RB, Obs>(1u, nullptr, D, e, act[2 * e], act[2 * e + 1], tile + t, kTileStride, rew, &c, &d, pretest) != 0;
      if (bail) env_step<kStepFull, RB, Obs>(1u, &scratch, D, e, act[2 * e], act[2 * e + 1], tile + t, kTileStride, rew, &c, &d);
      eval_accumulate(A, e, rew, c, d);
    }
    if (Obs) write_tile(tile, obs, e0, D.n, RB::kObsDim);
  }
}

template <class RB>
void do_evaluate(Handle* H, int h_steps, const float* act, double discount, float* obs, double* ret, int ret_cols,
                 double* cost, int32_t* length) {
  double w = 1.0;
  for (int h = 0; h < h_steps; ++h) {
    const EvalAcc A = {ret, cost, length, w, ret_cols, h == 0, h == h_steps - 1};
    const float* a = act + (size_t)h * H->D.n * 2;
    if (h < h_steps - 1) eval_step<RB, false>(H, a, nullptr, A);
    else eval_step<RB, true>(H, a, obs, A);
    w *= discount;
  }
}
}  // namespace

extern "C" {
int sag_evaluate_actions(void* h, int h_steps, const float* act, double discount, float* obs, double* ret, int ret_cols,
                         double* cost, int32_t* length, void* s) {
  (void)s;
  Handle* H = (Handle*)h;
  if (!H || !act || !obs || !ret || !cost || !length || h_steps <= 0 || (ret_cols != 1 && ret_cols != 2))
    return fail("sag_evaluate_actions: bad argument");
  HOSTEMU_DISPATCH(H, do_evaluate, (H, h_steps, act, discount, obs, ret, ret_cols, cost, length));
  return 0;
}
}
