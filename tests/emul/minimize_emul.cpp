// TEST-ONLY host build of the loop control of ms_ctx_minimize (ms_minimize.cuh).
//
// The control kernel k_min_control runs ms_min_step in one thread; this file exposes the SAME function to Python, so
// the no-GPU test tier can let it drive the emulated device (tests/fake_device.py) action by action and compare the
// action sequence, the step sizes, the history and the result with the host loop of DeviceMinimizer.  Built with
// -ffp-contract=off, like the device code's explicitly rounded operations.  Nothing under membrane_solver_b200/ loads
// it.
#include <cstring>

#include "../../membrane_solver_b200/csrc/ms_minimize.cuh"

using namespace ms;

extern "C" {

int emul_min_state_bytes() { return int(sizeof(MinState)); }
int emul_min_opts_bytes() { return int(sizeof(MinOpts)); }

// cg_valid: the emulated context holds a committed conjugate-gradient pair
void emul_min_init(MinState* s, double step_size, int32_t cg_iter, int32_t cg_have_history, int32_t cg_valid,
                   int32_t n_steps) {
  std::memset(s, 0, sizeof(*s));
  s->step_size = step_size;
  s->cg_iter = cg_iter;
  s->cg_have_history = cg_have_history ? 1 : 0;
  s->cg_valid = cg_valid ? 1 : 0;
  s->n_steps = n_steps;
  s->pc = PC_START;
  s->proj_active = -1;
  s->last_ran_a = -1;
}

// one call of the control kernel: sc (16 scalars), ls4 (line_search_stats), ok (normal_change_ok) of the last action
int emul_min_step(const MinOpts* o, MinState* s, const double* sc, const double* ls4, int32_t ok, double* hist,
                  int32_t hist_cap) {
  MinInput in;
  in.sc = sc;
  for (int k = 0; k < 4; ++k) in.ls[k] = ls4[k];
  in.ok = ok;
  return ms_min_step(*o, *s, in, hist, hist_cap, 0, 0);
}

// what the action launches read from the state: alpha (trial), -lambda (Newton step), the restart flag
void emul_min_args(const MinState* s, double* alpha, double* neg_lam, int32_t* cg_restart) {
  *alpha = s->alpha;
  *neg_lam = s->neg_lam;
  *cg_restart = s->cg_restart;
}

// d3 = {step_size, energy, grad_norm}; i9 = {cg_iter, cg_have_history, iterations, terminated_early, step_success,
// has_grad_norm, n_hist, n_trials, n_evals}
void emul_min_result(const MinState* s, double* d3, int32_t* i9) {
  d3[0] = s->step_size;
  d3[1] = s->res_energy;
  d3[2] = s->res_grad_norm;
  const int32_t v[9] = {s->cg_iter, s->cg_have_history, s->res_iterations, s->res_terminated_early, s->res_step_success,
                        s->res_has_grad_norm, s->n_hist, s->n_trials, s->n_evals};
  std::memcpy(i9, v, sizeof(v));
}

// the four values of ms_ctx_line_search_stats from the reduction words and the scalars
void emul_min_ls_stats(const unsigned long long* bits, const double* sc, int32_t nf, double* out4) {
  ms_min_ls_stats(bits, sc, nf, out4);
}

}  // extern "C"
