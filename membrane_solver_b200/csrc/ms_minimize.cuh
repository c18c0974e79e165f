// Loop control of the device-resident minimiser (ms_ctx_minimize): DeviceMinimizer.minimize, _line_search, _enforce
// and _total of runtime/device_minimizer.py restated as a state machine, shared by the control kernel (one thread)
// and the test-only host emulator (tests/emul/minimize_emul.cpp).
//
// ms_min_advance() takes the state and the scalars of the action that just ran and returns the next action; the
// device runs that action's launches and calls it again.  The decisions are those of the Python loop bit for bit:
//   - every floating-point expression is the Python one, operation for operation, in Python's evaluation order and
//     never contracted (mn_mul / mn_add / ... round each operation on the device; the host build uses
//     -ffp-contract=off);
//   - min(a, b) / max(a, b) are Python's builtins (the first argument wins unless the second is strictly smaller /
//     larger), so a NaN argument resolves as it does there, and every comparison with a NaN is false;
//   - <g,g> ** 0.5 is the correctly rounded square root.
#pragma once

#include <stdint.h>

#include "../../include/ms_b200.h"
#include "ms_math.cuh"

namespace ms {

#ifdef __CUDA_ARCH__
MS_HD double mn_mul(double a, double b) { return __dmul_rn(a, b); }
MS_HD double mn_div(double a, double b) { return __ddiv_rn(a, b); }
MS_HD double mn_add(double a, double b) { return __dadd_rn(a, b); }
MS_HD double mn_sub(double a, double b) { return __dsub_rn(a, b); }
MS_HD double mn_sqrt(double a) { return __dsqrt_rn(a); }
MS_HD double mn_bits(uint64_t u) { return __longlong_as_double((long long)u); }
#else
MS_HD double mn_mul(double a, double b) { return a * b; }
MS_HD double mn_div(double a, double b) { return a / b; }
MS_HD double mn_add(double a, double b) { return a + b; }
MS_HD double mn_sub(double a, double b) { return a - b; }
MS_HD double mn_sqrt(double a) { return __builtin_sqrt(a); }
MS_HD double mn_bits(uint64_t u) {
  double d;
  __builtin_memcpy(&d, &u, 8);
  return d;
}
#endif
MS_HD double mn_abs(double a) { return a < 0.0 ? -a : (a == 0.0 ? 0.0 : a); }
MS_HD double py_min(double a, double b) { return b < a ? b : a; }  // Python's min(a, b)
MS_HD double py_max(double a, double b) { return b > a ? b : a; }  // Python's max(a, b)

// Actions: each is one fixed sequence of launches (ms_capi.cu, minimize_action) or one call of the Python loop.
enum MinAction : int32_t {
  MN_EVAL_GRAD = 0,      // energy_and_gradient(): evaluation with the projected, fixed-masked gradient
  MN_DIRECTION = 1,      // direction_from_gradient(-1), or cg_direction(restart) + cg_commit
  MN_STATS = 2,          // line_search_stats()
  MN_EVAL_ENERGY = 3,    // energy(): energy-only evaluation at the positions
  MN_MAKE_TRIAL = 4,     // make_trial(alpha)
  MN_GUARD = 5,          // normal_change_ok(0.5)
  MN_ENF_EVAL_POS = 6,   // _enforce: volume evaluation with gradient at the positions ...
  MN_ENF_EVAL_TRIAL = 7, // ... or at the trial positions
  MN_ENF_AXPY_POS = 8,   // _enforce: axpy(target, MS_ARR_VOLGRAD, -lambda, skip_fixed)
  MN_ENF_AXPY_TRIAL = 9,
  MN_EVAL_TRIAL = 10,    // energy(trial=True)
  MN_ACCEPT = 11,        // accept_trial()
  MN_DRIFT_EVAL = 12,    // volume-only evaluation of the drift check
  MN_DONE = 13,
  MN_ACTIONS = 13,       // actions that run launches
};

// Options: the DeviceMinimizer fields the loop reads (checked by ms_min_valid).
using MinOpts = ms_minimize_opts;

// Program counter of the loop (labels of the Python code that are not actions).
enum MinPc : int32_t {
  PC_START = 0, PC_LOOP, PC_AFTER_GRAD, PC_AFTER_DIR, PC_AFTER_STATS1, PC_LS_E0, PC_LS_STATS, PC_TRIAL, PC_AFTER_MAKE,
  PC_AFTER_GUARD, PC_PRE_EVAL, PC_EVAL_TRIAL, PC_AFTER_TRIAL, PC_LS_FAIL, PC_AFTER_LS, PC_AFTER_DRIFT, PC_DRIFT_DONE,
  PC_NEXT, PC_FINAL, PC_FINAL_E, PC_FINAL_DONE, PC_ZERO_EXIT, PC_ENF, PC_ENF_AFTER, PC_DONE,
};

// The state: in/out fields first (the caller's step size and conjugate-gradient memory), then the loop's locals and
// the result.  Plain data, the same layout on both sides.
struct MinState {
  double step_size;
  int32_t cg_iter, cg_have_history;
  int32_t n_steps;
  int32_t pc, i, zero_steps, success, t;   // t: line-search trial index
  int32_t enf_left, enf_trial, enf_ret;    // _enforce: iterations left, target (0 positions / 1 trial), return label
  int32_t cg_restart;                      // read by the direction launch
  int32_t cg_valid;                        // the context holds a committed direction / gradient pair (ms_ctx_cg_direction
                                           // restarts without one, whatever the caller's history flag says)
  int32_t ls_ok;                           // result of the line search
  int32_t proj_active;                     // the gradient's projection is still deferred (host mirror ms_ctx::proj)
  int32_t last_ran_a;                      // the last evaluation ran pass A (host mirror ms_ctx::ran_pass_a)
  int32_t n_accepted;
  double energy, energy0, alpha, alpha_max, step_in, min_edge, max_dir_norm, g_dot_d, safe_limit, neg_lam;
  double ls_step, ls_energy;
  // result (the dict DeviceMinimizer.minimize returns) and counters
  double res_energy, res_grad_norm;
  int32_t res_iterations, res_terminated_early, res_step_success, res_has_grad_norm;
  int32_t n_hist, n_trials, n_evals, n_actions, n_guards, n_guard_rejects, last_action;
};

// Input of ms_min_advance: the scalar vector after an evaluation, line_search_stats' four values after MN_STATS,
// normal_change_ok's answer after MN_GUARD.
struct MinInput {
  const double* sc;  // MS_SC_COUNT doubles
  double ls[4];
  int32_t ok;
};

// the four values of ms_ctx_line_search_stats from the reduction words and the scalar vector
MS_HD void ms_min_ls_stats(const unsigned long long* bits, const double* sc, int32_t nf, double* out4) {
  const double e2 = mn_bits(bits[0]), d2 = mn_bits(bits[1]);
  out4[0] = (nf > 0 && e2 < 1.0e299) ? mn_sqrt(e2) : 0.0;
  out4[1] = mn_sqrt(d2);
  out4[2] = sc[9];   // MS_SC_G_GC: <gradient, direction>
  out4[3] = sc[8];   // MS_SC_G_G
}

MS_HD bool ms_min_valid(const MinOpts& o) {
  const uint32_t mods = 1u | 2u | 4u | 8u;  // surface, volume, bending, tilt (bending-tilt and smoothness: leaflet paths)
  if (o.modules & ~mods) return false;
  if (o.volume_mode < -1 || o.volume_mode > 1) return false;
  if (o.stepper < 0 || o.stepper > 1) return false;
  if (o.max_iter < 0 || o.max_iter > (1 << 20) || o.max_zero_steps < 0 || o.restart_interval < 1) return false;
  if (o.flags & ~3u) return false;
  return true;
}

// _total(res)
MS_HD double ms_min_total(const MinOpts& o, const double* sc) {
  double e = 0.0;
  if (o.modules & 1u) e = mn_add(e, sc[0]);  // e_surface
  if (o.modules & 4u) e = mn_add(e, sc[3]);  // e_bending
  if (o.modules & 8u) e = mn_add(e, sc[4]);  // e_tilt
  if (o.volume_mode == 1) {
    const double d = mn_sub(sc[2], o.v_target);
    e = mn_add(e, mn_mul(mn_mul(mn_mul(0.5, o.k_vol), d), d));
  }
  return e;
}

MS_HD double mn_inf() { return mn_bits(0x7ff0000000000000ull); }
MS_HD double mn_nan() { return mn_bits(0x7ff8000000000000ull); }

// Advance from the state after the last action (its results in `in`) to the next action.  hist receives
// (i, accepted energy, step size in, success) per line search, at most hist_cap rows (n_hist counts them all).
MS_HD int32_t ms_min_advance(const MinOpts& o, MinState& s, const MinInput& in, double* hist, int32_t hist_cap) {
  const bool cg = o.stepper == 1;
  for (;;) {
    switch (s.pc) {
      case PC_START:
        s.zero_steps = 0;
        s.success = 1;
        s.energy = mn_nan();
        s.i = 0;
        s.n_hist = s.n_trials = s.n_evals = s.n_actions = s.n_guards = s.n_guard_rejects = s.n_accepted = 0;
        if (o.enforce_volume && s.n_steps > 0) {  // minimizer.py:1223-1226
          s.enf_trial = 0; s.enf_left = 12; s.enf_ret = PC_LOOP; s.pc = PC_ENF;
        } else {
          s.pc = PC_LOOP;
        }
        break;
      case PC_LOOP:
        if (s.i < s.n_steps) { s.pc = PC_AFTER_GRAD; return MN_EVAL_GRAD; }
        s.pc = PC_FINAL;
        break;
      case PC_AFTER_GRAD:
        s.energy = ms_min_total(o, in.sc);
        if (cg) {
          s.cg_restart = (!s.cg_have_history) || (s.cg_iter % o.restart_interval == 0) || !s.cg_valid;
          s.cg_valid = 1;  // the direction action commits gradient and direction
        }
        s.pc = PC_AFTER_DIR;
        return MN_DIRECTION;
      case PC_AFTER_DIR:
        s.pc = PC_AFTER_STATS1;
        return MN_STATS;
      case PC_AFTER_STATS1: {
        const double grad_norm = mn_sqrt(in.ls[3]);
        if (grad_norm < o.tol) {
          s.res_energy = s.energy; s.res_iterations = s.i + 1; s.res_terminated_early = 1; s.res_step_success = 1;
          s.res_has_grad_norm = 1; s.res_grad_norm = grad_norm;
          s.pc = PC_DONE;
          return MN_DONE;
        }
        s.step_in = s.step_size;
        s.pc = PC_LS_E0;
        return MN_EVAL_ENERGY;
      }
      case PC_LS_E0:
        s.energy0 = ms_min_total(o, in.sc);
        s.pc = PC_LS_STATS;
        return MN_STATS;
      case PC_LS_STATS: {
        s.min_edge = in.ls[0]; s.max_dir_norm = in.ls[1]; s.g_dot_d = in.ls[2];
        s.safe_limit = s.min_edge > 0 ? mn_mul(0.3, s.min_edge) : mn_inf();
        if (s.g_dot_d >= 0.0) {
          s.ls_ok = 0; s.ls_step = s.step_in; s.ls_energy = s.energy0;
          s.pc = PC_AFTER_LS;
          break;
        }
        s.alpha = s.step_in;
        if (o.edge_fraction > 0.0 && s.min_edge > 0.0 && s.max_dir_norm > 0.0)
          s.alpha = py_min(s.alpha, mn_div(mn_mul(o.edge_fraction, s.min_edge), s.max_dir_norm));
        s.alpha_max = mn_mul(o.alpha_max_factor, s.step_in);
        s.t = 0;
        s.pc = PC_TRIAL;
        break;
      }
      case PC_TRIAL:
        if (s.t < o.max_iter) { s.n_trials++; s.pc = PC_AFTER_MAKE; return MN_MAKE_TRIAL; }
        s.pc = PC_LS_FAIL;
        break;
      case PC_AFTER_MAKE:
        if (!(mn_mul(s.alpha, s.max_dir_norm) < s.safe_limit)) { s.n_guards++; s.pc = PC_AFTER_GUARD; return MN_GUARD; }
        s.pc = PC_PRE_EVAL;
        break;
      case PC_AFTER_GUARD:
        if (!in.ok) {
          s.n_guard_rejects++;
          s.alpha = mn_mul(s.alpha, o.beta);
          if (s.alpha < 1e-8) { s.pc = PC_LS_FAIL; break; }
          s.t++;
          s.pc = PC_TRIAL;
          break;
        }
        s.pc = PC_PRE_EVAL;
        break;
      case PC_PRE_EVAL:
        if (o.enforce_volume && o.projection_during) {
          s.enf_trial = 1; s.enf_left = 3; s.enf_ret = PC_EVAL_TRIAL; s.pc = PC_ENF;
        } else {
          s.pc = PC_EVAL_TRIAL;
        }
        break;
      case PC_EVAL_TRIAL:
        s.pc = PC_AFTER_TRIAL;
        return MN_EVAL_TRIAL;
      case PC_AFTER_TRIAL: {
        const double te = ms_min_total(o, in.sc);
        if (te <= mn_add(s.energy0, mn_mul(mn_mul(o.c, s.alpha), s.g_dot_d))) {
          s.ls_ok = 1; s.ls_step = py_min(mn_mul(s.alpha, o.gamma), s.alpha_max); s.ls_energy = te;
          s.n_accepted++;
          s.pc = PC_AFTER_LS;
          return MN_ACCEPT;
        }
        s.alpha = mn_mul(s.alpha, o.beta);
        if (s.alpha < 1e-8) { s.pc = PC_LS_FAIL; break; }
        s.t++;
        s.pc = PC_TRIAL;
        break;
      }
      case PC_LS_FAIL: {
        const double reduced = py_max(mn_mul(s.alpha, o.beta), 0.0);
        s.ls_ok = 0; s.ls_step = py_max(reduced, mn_mul(s.step_in, o.beta)); s.ls_energy = s.energy0;
        s.pc = PC_AFTER_LS;
        break;
      }
      case PC_AFTER_LS:
        s.success = s.ls_ok;
        s.step_size = s.ls_step;
        if (s.n_hist < hist_cap && hist) {
          double* h = hist + 4 * int64_t(s.n_hist);
          h[0] = double(s.i); h[1] = s.ls_energy; h[2] = s.step_in; h[3] = s.ls_ok ? 1.0 : 0.0;
        }
        s.n_hist++;
        if (cg) {
          if (s.success) { s.cg_have_history = 1; s.cg_iter++; }
          else { s.cg_have_history = 0; s.cg_iter = 0; }
        }
        if (!s.success) {
          if (s.step_size <= o.step_size_floor) {
            s.zero_steps++;
            if (s.zero_steps >= o.max_zero_steps) { s.pc = PC_ZERO_EXIT; return MN_EVAL_ENERGY; }
          } else {
            s.zero_steps = 0;
          }
          s.pc = PC_NEXT;
        } else {
          s.zero_steps = 0;
          if (o.enforce_volume && o.volume_mode == 0 && !o.projection_during) { s.pc = PC_AFTER_DRIFT; return MN_DRIFT_EVAL; }
          s.pc = PC_NEXT;
        }
        break;
      case PC_AFTER_DRIFT: {
        const double drift = mn_div(mn_abs(mn_sub(in.sc[2], o.v_target)), py_max(mn_abs(o.v_target), 1.0));
        if (drift > o.volume_tolerance) {
          s.enf_trial = 0; s.enf_left = 12; s.enf_ret = PC_DRIFT_DONE; s.pc = PC_ENF;
        } else {
          s.pc = PC_NEXT;
        }
        break;
      }
      case PC_DRIFT_DONE:
        s.cg_have_history = 0;
        s.cg_iter = 0;
        s.pc = PC_NEXT;
        break;
      case PC_NEXT:
        s.i++;
        s.pc = PC_LOOP;
        break;
      case PC_FINAL:
        if (o.enforce_volume) {  // minimizer.py:1518-1521, also when n_steps == 0
          s.enf_trial = 0; s.enf_left = 12; s.enf_ret = PC_FINAL_E; s.pc = PC_ENF;
        } else {
          s.pc = PC_FINAL_E;
        }
        break;
      case PC_FINAL_E:
        s.pc = PC_FINAL_DONE;
        return MN_EVAL_ENERGY;
      case PC_FINAL_DONE:
        s.res_energy = ms_min_total(o, in.sc); s.res_iterations = s.n_steps; s.res_terminated_early = 0;
        s.res_step_success = s.success; s.res_has_grad_norm = 0;
        s.pc = PC_DONE;
        return MN_DONE;
      case PC_ZERO_EXIT:
        s.res_energy = ms_min_total(o, in.sc); s.res_iterations = s.i + 1; s.res_terminated_early = 1;
        s.res_step_success = 0; s.res_has_grad_norm = 0;
        s.pc = PC_DONE;
        return MN_DONE;
      case PC_ENF:
        if (s.enf_left > 0) {
          s.enf_left--;
          s.pc = PC_ENF_AFTER;
          return s.enf_trial ? MN_ENF_EVAL_TRIAL : MN_ENF_EVAL_POS;
        }
        s.pc = s.enf_ret;
        break;
      case PC_ENF_AFTER: {
        const double delta = mn_sub(in.sc[2], o.v_target);
        if (mn_abs(delta) < 1e-12) { s.pc = s.enf_ret; break; }
        s.neg_lam = -mn_div(delta, mn_add(in.sc[10], 1e-12));  // MS_SC_GC_GC
        s.pc = PC_ENF;
        return s.enf_trial ? MN_ENF_AXPY_TRIAL : MN_ENF_AXPY_POS;
      }
      default:
        s.pc = PC_DONE;
        return MN_DONE;
    }
  }
}

// ms_min_advance plus the bookkeeping of the host mirrors: evaluations counted, the deferred projection's state after
// the action (proj_grad: the projection an MN_EVAL_GRAD leaves pending; a conjugate-gradient direction applies it in
// place; a volume evaluation with gradient drops it) and whether the last evaluation ran pass A.
MS_HD int32_t ms_min_step(const MinOpts& o, MinState& s, const MinInput& in, double* hist, int32_t hist_cap,
                          int32_t proj_grad, int32_t ran_a_grad) {
  const int32_t act = ms_min_advance(o, s, in, hist, hist_cap);
  switch (act) {
    case MN_EVAL_GRAD: s.n_evals++; s.proj_active = proj_grad; s.last_ran_a = ran_a_grad; break;
    case MN_DIRECTION: if (o.stepper == 1) s.proj_active = 0; break;
    case MN_EVAL_ENERGY: case MN_EVAL_TRIAL: case MN_DRIFT_EVAL: s.n_evals++; s.last_ran_a = 1; break;
    case MN_ENF_EVAL_POS: case MN_ENF_EVAL_TRIAL: s.n_evals++; s.proj_active = 0; s.last_ran_a = 0; break;
    default: break;
  }
  if (act != MN_DONE) s.n_actions++;
  s.last_action = act;
  return act;
}

}  // namespace ms
