// Batched lock-step L-BFGS + BackTracking(order=2): the caller of the hot path (SURVEY.md section 8f rank 1).
//
// Restates, per GP, exactly what the reference hands every GP to
//     GaussianProcesses.optimize!(gp, LBFGS(linesearch = BackTracking(order=2)), Optim.Options(time_limit=10.))
//     (examples/maximal_coordinates/CPnoise.jl:41 and every other experiment file)
// i.e. Optim 1.4.1 LBFGS(m=10, InitialStatic(alpha=1), scaleinvH0=true) + LineSearches 7.1.1 BackTracking
// (SURVEY.md appendix A.4/A.5; same state machine as oracle/lbfgs_oracle.py), but for B GPs at once:
// every round issues ONE mixed pass through gprb_eval_mixed - a value-only evaluation for each GP inside a line
// search and a value+gradient evaluation for each GP that accepted a step in the previous round.  Per GP the
// sequence of evaluations is exactly the scalar algorithm's; only the batching across GPs differs.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <functional>
#include <limits>
#include <vector>

#include "common.cuh"

namespace gprb {

// objective(theta[B*P], mode[B] (0 skip / 1 value / 2 value+gradient), retry[B], f[B], g[B*P], pending[B]) -> rc ;
// f = -mll (+Inf on failure), g = -dmll for the mode-2 GPs.  pending[b] = 1: the evaluation of GP b is not finished
// (its factorisation needs another make_posdef! jitter) - the caller re-submits it with retry[b] = 1 and the same
// theta in its next pass, next to the other GPs' new evaluations, instead of stalling the whole batch on it.
using Objective = std::function<int(const double*, const uint8_t*, const uint8_t*, double*, double*, uint8_t*)>;

struct GpState {
  std::vector<double> x, g, g_prev, s, dx, x_trial;
  std::vector<double> dx_hist, dg_hist, rho;  // ring buffers [m][P], [m]
  double fx = 0, f_prev = 0, phi0 = 0, dphi0 = 0, a1 = 1, a2 = 1, phi1 = 0;
  int pseudo_iteration = 0, iteration = 0, f_calls = 0, fg_calls = 0;
  int iterfinite = 0, ls_iter = 0;
  bool ls_prefinite = true;  // still in the "halve until finite" pre-loop
  enum Phase { NEED_DIR, IN_LS, NEED_GRAD, DONE } phase = NEED_DIR;
  bool converged = false, ls_failed = false;
  double vclock = 0.0;  // per-GP virtual clock (opts.cost_value / cost_grad), compared with opts.time_limit
};

static double dot(const double* a, const double* b, int n) {
  double s = 0;
  for (int i = 0; i < n; ++i) s += a[i] * b[i];
  return s;
}
// maximum(abs, g) with Julia's semantics: NaN if any entry is NaN (fmax would drop it and report a failed gradient as 0)
static double inf_norm(const std::vector<double>& v) {
  double m = 0;
  for (double e : v) {
    if (isnan(e)) return NAN;
    m = fmax(m, fabs(e));
  }
  return m;
}

// Optim.twoloop! (scaleinvH0 = true, no preconditioner): s = -H g
static void twoloop(GpState& st, int m, int P) {
  const int lower = st.pseudo_iteration - m, upper = st.pseudo_iteration - 1;
  std::vector<double> q(st.g), alpha(m, 0.0);
  for (int index = upper; index >= lower; --index) {
    if (index < 1) continue;
    const int i = (index - 1) % m;
    alpha[i] = st.rho[i] * dot(&st.dx_hist[(size_t)i * P], q.data(), P);
    for (int p = 0; p < P; ++p) q[p] -= alpha[i] * st.dg_hist[(size_t)i * P + p];
  }
  if (st.pseudo_iteration > 1) {
    const int i = (upper - 1) % m;
    const double* dxi = &st.dx_hist[(size_t)i * P];
    const double* dgi = &st.dg_hist[(size_t)i * P];
    const double scaling = dot(dxi, dgi, P) / dot(dgi, dgi, P);
    for (int p = 0; p < P; ++p) st.s[p] = scaling * q[p];
  } else {
    st.s = q;
  }
  for (int index = lower; index <= upper; ++index) {
    if (index < 1) continue;
    const int i = (index - 1) % m;
    const double beta = st.rho[i] * dot(&st.dg_hist[(size_t)i * P], st.s.data(), P);
    for (int p = 0; p < P; ++p) st.s[p] += st.dx_hist[(size_t)i * P + p] * (alpha[i] - beta);
  }
  for (int p = 0; p < P; ++p) st.s[p] = -st.s[p];
}

int batched_lbfgs(int B, int P, double* theta_inout, const gprb_lbfgs_opts& o, const Objective& obj,
                  gprb_opt_result* results) {
  const int m = o.m > 0 ? o.m : 10;
  const int iterfinite_max = 52;  // ceil(-log2(eps(Float64)))
  const auto t0 = std::chrono::steady_clock::now();
  std::vector<GpState> S(B);
  std::vector<double> theta((size_t)B * P), f(B), g((size_t)B * P);
  std::vector<uint8_t> act(B, 2);
  memcpy(theta.data(), theta_inout, sizeof(double) * B * P);
  std::vector<uint8_t> retry(B, 0), pending(B, 0);
  // evaluate `act` for everyone, looping until no GP has a retry pending (initial and final evaluations)
  auto eval_all = [&]() -> int {
    std::vector<uint8_t> cur(act), rt(B, 0), pd(B, 0);
    for (;;) {
      int r = obj(theta.data(), cur.data(), rt.data(), f.data(), g.data(), pd.data());
      if (r) return r;
      bool any = false;
      for (int b = 0; b < B; ++b) { cur[b] = pd[b] ? cur[b] : 0; rt[b] = pd[b]; any = any || pd[b]; }
      if (!any) return 0;
    }
  };
  int rc = eval_all();
  if (rc) return rc;
  for (int b = 0; b < B; ++b) {
    GpState& st = S[b];
    st.x.assign(theta.begin() + (size_t)b * P, theta.begin() + (size_t)(b + 1) * P);
    st.g.assign(g.begin() + (size_t)b * P, g.begin() + (size_t)(b + 1) * P);
    st.g_prev.assign(P, 0.0); st.s.assign(P, 0.0); st.dx.assign(P, 0.0); st.x_trial.assign(P, 0.0);
    st.dx_hist.assign((size_t)m * P, 0.0); st.dg_hist.assign((size_t)m * P, 0.0); st.rho.assign(m, 0.0);
    st.fx = f[b];
    st.fg_calls = 1;
    st.vclock = o.cost_grad;
    bool finite = isfinite(st.fx);
    for (double e : st.g) finite = finite && isfinite(e);
    if (!finite) st.phase = GpState::DONE;                                              // nothing to optimise from
    else if (inf_norm(st.g) <= o.g_abstol) { st.phase = GpState::DONE; st.converged = true; }  // initial_convergence
    else if (o.iterations <= 0) st.phase = GpState::DONE;
  }

  auto set_trial = [&](GpState& st, double a) {
    for (int p = 0; p < P; ++p) st.x_trial[p] = st.x[p] + a * st.s[p];
  };
  bool timed_out = false;
  for (;;) {
    // ---- 1. search directions for GPs starting an iteration (update_state! up to the line search): host only
    for (int b = 0; b < B; ++b) {
      GpState& st = S[b];
      if (st.phase != GpState::NEED_DIR) continue;
      st.iteration++;
      st.pseudo_iteration++;
      twoloop(st, m, P);
      st.g_prev = st.g;
      st.dphi0 = dot(st.g.data(), st.s.data(), P);
      if (st.dphi0 >= 0.0) {  // reset_search_direction!
        st.pseudo_iteration = 1;
        for (int p = 0; p < P; ++p) st.s[p] = -st.g[p];
        st.dphi0 = dot(st.g.data(), st.s.data(), P);
      }
      st.phi0 = st.fx;
      st.a1 = st.a2 = 1.0;  // InitialStatic(alpha = 1)
      st.iterfinite = 0; st.ls_iter = 0; st.ls_prefinite = true;
      set_trial(st, st.a2);
      st.phase = GpState::IN_LS;
    }
    // ---- 2. ONE mixed pass: value-only at the trial point of every GP inside a line search, value+gradient at the
    //         accepted point of every GP that left its line search in the previous round (update_g!)
    int nact = 0;
    for (int b = 0; b < B; ++b) {
      GpState& st = S[b];
      act[b] = st.phase == GpState::IN_LS ? 1 : st.phase == GpState::NEED_GRAD ? 2 : 0;
      if (act[b] == 1) memcpy(&theta[(size_t)b * P], st.x_trial.data(), sizeof(double) * P);
      else if (act[b] == 2)
        for (int p = 0; p < P; ++p) theta[(size_t)b * P + p] = st.x[p] + st.dx[p];
      nact += act[b] != 0;
    }
    if (nact == 0) break;
    const auto tr0 = std::chrono::steady_clock::now();
    if ((rc = obj(theta.data(), act.data(), retry.data(), f.data(), g.data(), pending.data()))) return rc;
    for (int b = 0; b < B; ++b) {  // unfinished evaluations ride along with the next round
      retry[b] = pending[b];
      if (pending[b]) act[b] = 0;
    }
    if (getenv("GPRB200_LBFGS_TRACE")) {  // per-round trace: GPs in the value-only / value+gradient sets and the round time
      int nv = 0, ng = 0, np = 0;
      for (int b = 0; b < B; ++b) { nv += act[b] == 1; ng += act[b] == 2; np += pending[b]; }
      fprintf(stderr, "lbfgs round: value %d grad %d retry-pending %d  %.2f ms\n", nv, ng, np,
              1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - tr0).count());
    }
    // wall-clock form of time_limit (whole batch); with evaluation costs set the limit is per GP on its virtual clock
    const bool vtime = o.cost_value > 0.0 || o.cost_grad > 0.0;
    if (!vtime && o.time_limit > 0 && std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > o.time_limit)
      timed_out = true;
    for (int b = 0; b < B; ++b) {
      GpState& st = S[b];
      if (act[b] == 1) {
        st.f_calls++;
        st.vclock += o.cost_value;
        st.phi1 = f[b];
        // BackTracking: "halve until finite" pre-loop
        if (st.ls_prefinite && !isfinite(st.phi1) && st.iterfinite < iterfinite_max) {
          st.iterfinite++;
          st.a1 = st.a2;
          st.a2 = st.a1 / 2.0;
          set_trial(st, st.a2);
          continue;
        }
        st.ls_prefinite = false;
        if (st.phi1 > st.phi0 + o.c_1 * st.a2 * st.dphi0) {  // sufficient decrease violated (false for NaN)
          st.ls_iter++;
          if (st.ls_iter > o.ls_iterations) {  // LineSearchException: step applied, optimisation of this GP aborts
            for (int p = 0; p < P; ++p) st.x[p] += st.a2 * st.s[p];
            st.ls_failed = true;
            st.phase = GpState::DONE;
            continue;
          }
          const double denom = 2.0 * (st.phi1 - st.phi0 - st.dphi0 * st.a2);
          double a_tmp = denom != 0.0 ? -(st.dphi0 * st.a2 * st.a2) / denom : NAN;
          st.a1 = st.a2;
          const double hi = st.a2 * o.rho_hi, lo = st.a2 * o.rho_lo;
          a_tmp = isnan(a_tmp) ? hi : fmin(a_tmp, hi);  // NaNMath.min / max
          st.a2 = isnan(a_tmp) ? lo : fmax(a_tmp, lo);
          set_trial(st, st.a2);
          continue;
        }
        // accepted: the gradient at the new point is requested in the next round
        for (int p = 0; p < P; ++p) st.dx[p] = st.a2 * st.s[p];
        st.f_prev = st.fx;
        st.phase = GpState::NEED_GRAD;
      } else if (act[b] == 2) {
        st.fg_calls++;
        st.vclock += o.cost_grad;
        const double fnew = f[b];
        const double* gnew = &g[(size_t)b * P];
        bool gfinite = true;
        double dxmax = 0.0;
        for (int p = 0; p < P; ++p) {
          gfinite = gfinite && isfinite(gnew[p]);
          dxmax = fmax(dxmax, fabs(theta[(size_t)b * P + p] - st.x[p]));
        }
        // assess_convergence: x/f tolerances are 0 => only exact stalls; g_abstol on the inf-norm (NaN never converges)
        double gmax = 0.0;
        for (int p = 0; p < P; ++p) gmax = isnan(gnew[p]) ? NAN : fmax(gmax, fabs(gnew[p]));
        const bool x_conv = dxmax <= 0.0, f_conv = fabs(fnew - st.f_prev) <= 0.0, g_conv = gmax <= o.g_abstol;
        // Optim: f_increased (f_x > f_x_previous, e.g. +Inf from a re-evaluation that failed) stops the run when
        // allow_f_increases = false (the default) and pick_best_x hands back the PREVIOUS point; a non-finite gradient
        // ends it too ("Terminated early due to NaN in gradient").  Either way this GP keeps its last good x, f, g.
        if (fnew > st.f_prev || !gfinite || !isfinite(fnew)) {
          st.converged = x_conv || f_conv || g_conv;
          st.phase = GpState::DONE;
          continue;
        }
        for (int p = 0; p < P; ++p) {
          st.x[p] = theta[(size_t)b * P + p];
          st.g[p] = gnew[p];
        }
        st.fx = fnew;
        if (x_conv || f_conv || g_conv) { st.converged = true; st.phase = GpState::DONE; continue; }
        // update_h!
        double denom = 0.0;
        std::vector<double> dg(P);
        for (int p = 0; p < P; ++p) { dg[p] = st.g[p] - st.g_prev[p]; denom += st.dx[p] * dg[p]; }
        const double rho_it = denom == 0.0 ? INFINITY : 1.0 / denom;
        if (isinf(rho_it)) {
          st.pseudo_iteration = 0;
        } else {
          const int idx = (st.pseudo_iteration - 1) % m;
          memcpy(&st.dx_hist[(size_t)idx * P], st.dx.data(), sizeof(double) * P);
          memcpy(&st.dg_hist[(size_t)idx * P], dg.data(), sizeof(double) * P);
          st.rho[idx] = rho_it;
        }
        st.phase = GpState::NEED_DIR;
        if (st.iteration >= o.iterations) st.phase = GpState::DONE;
        if (o.max_evals > 0 && st.f_calls + st.fg_calls >= o.max_evals) st.phase = GpState::DONE;
        if (vtime && o.time_limit > 0 && st.vclock > o.time_limit) st.phase = GpState::DONE;  // this GP's own 10 s are up
      }
    }
    if (timed_out) {  // Optim checks the time limit once per iteration: GPs keep their last accepted x
      for (int b = 0; b < B; ++b) {
        GpState& st = S[b];
        if (st.phase == GpState::NEED_GRAD) {  // the line search just accepted x + dx (f known): the step is not discarded
          for (int p = 0; p < P; ++p) st.x[p] += st.dx[p];
          st.fx = st.phi1;
        }
        st.phase = GpState::DONE;
      }
      break;
    }
  }
  // ---- write the minimiser back and leave the device state evaluated there (optimize! -> update_target!).
  // The state is left WITH the inverse (a value+gradient evaluation): for a GP that stopped right after a gradient
  // evaluation - the normal case - that state is still resident and the evaluation costs nothing (state reuse); for the
  // others it is one extra inverse + gradient per GP, and in return the reference's next call, predict_y(gp, obs) with
  // one test column (examples/utils/predictdynamics.jl:13), always finds V = L^-T resident (0.11 ms instead of 0.7 ms).
  // mll is bit-identical either way (same factorisation).
  for (int b = 0; b < B; ++b) {
    memcpy(&theta[(size_t)b * P], S[b].x.data(), sizeof(double) * P);
    act[b] = 2;
  }
  if ((rc = eval_all())) return rc;
  memcpy(theta_inout, theta.data(), sizeof(double) * B * P);
  for (int b = 0; b < B; ++b) {
    gprb_opt_result& r = results[b];
    r.mll = -f[b];
    r.g_norm = inf_norm(S[b].g);
    r.iterations = S[b].iteration;
    r.f_calls = S[b].f_calls;
    r.fg_calls = S[b].fg_calls;
    r.converged = S[b].converged;
    r.ls_failed = S[b].ls_failed;
    r.info = 0;
  }
  return 0;
}

}  // namespace gprb

using namespace gprb;

extern "C" {

void gprb_lbfgs_default_opts(gprb_lbfgs_opts* o) {
  if (!o) return;
  o->m = 10; o->iterations = 1000; o->max_evals = 0; o->ls_iterations = 1000;
  o->g_abstol = 1e-8; o->time_limit = 0.0; o->c_1 = 1e-4; o->rho_hi = 0.5; o->rho_lo = 0.1;
  o->cost_value = 0.0; o->cost_grad = 0.0;
}

int gprb_optimize(gprb_batch* b, double* theta_inout, const gprb_lbfgs_opts* opts, gprb_opt_result* results) {
  GPRB_REQUIRE(b && theta_inout && results, "gprb_optimize: NULL argument");
  if (int rc = refuse_while_predicting(b, "gprb_optimize")) return rc;
  gprb_lbfgs_opts o;
  if (opts) o = *opts; else gprb_lbfgs_default_opts(&o);
  const int B = b->B, P = b->P;
  std::vector<double> mll(B), grad((size_t)B * P);
  std::vector<int32_t> info(B, 0), last_info(B, 0);
  // get_optim_target: objective = -mll, gradient = -dmll, +Inf when the evaluation fails (info < 0)
  Objective obj = [&](const double* theta, const uint8_t* mode, const uint8_t* retry, double* f, double* g, uint8_t* pending) -> int {
    int rc = eval_pass_host(b, theta, mode, retry, mll.data(), grad.data(), info.data(), pending);
    if (rc) return rc;
    for (int i = 0; i < B; ++i) {
      if (!mode[i] || pending[i]) continue;
      last_info[i] = info[i];
      f[i] = info[i] < 0 ? INFINITY : -mll[i];
      if (mode[i] == 2)
        for (int p = 0; p < P; ++p) g[(size_t)i * P + p] = info[i] < 0 ? NAN : -grad[(size_t)i * P + p];
    }
    return 0;
  };
  int rc = batched_lbfgs(B, P, theta_inout, o, obj, results);
  if (rc) return rc;
  for (int i = 0; i < B; ++i) results[i].info = last_info[i];
  return GPRB_OK;
}

// Host-only self test of the batched state machine on an analytic objective (no GPU): B copies of the
// P-dimensional Rosenbrock function, +Inf outside the box |x_i| <= bound (exercises the halve-until-finite loop).
// Used by tests/test_lbfgs_cpu.py to compare against oracle/lbfgs_oracle.py trajectory by trajectory.
int gprb_lbfgs_selftest(int32_t B, int32_t P, double* theta_inout, const gprb_lbfgs_opts* opts, double bound,
                        gprb_opt_result* results) {
  GPRB_REQUIRE(theta_inout && results && B > 0 && P > 1, "gprb_lbfgs_selftest: bad argument");
  gprb_lbfgs_opts o;
  if (opts) o = *opts; else gprb_lbfgs_default_opts(&o);
  Objective obj = [&](const double* theta, const uint8_t* mode, const uint8_t*, double* f, double* gout, uint8_t* pending) -> int {
    for (int b = 0; b < B; ++b) {
      pending[b] = 0;
      if (!mode[b]) continue;
      double* g = mode[b] == 2 ? gout : nullptr;
      const double* x = theta + (size_t)b * P;
      bool inside = true;
      for (int p = 0; p < P; ++p) inside = inside && fabs(x[p]) <= bound;
      if (!inside) {
        f[b] = INFINITY;
        if (g) for (int p = 0; p < P; ++p) g[(size_t)b * P + p] = NAN;
        continue;
      }
      double s = 0;
      if (g) for (int p = 0; p < P; ++p) g[(size_t)b * P + p] = 0.0;
      for (int p = 0; p + 1 < P; ++p) {
        const double t1 = x[p + 1] - x[p] * x[p], t2 = 1.0 - x[p];
        s += 100.0 * t1 * t1 + t2 * t2;
        if (g) {
          g[(size_t)b * P + p] += -400.0 * x[p] * t1 - 2.0 * t2;
          g[(size_t)b * P + p + 1] += 200.0 * t1;
        }
      }
      f[b] = s;
    }
    return 0;
  };
  int rc = batched_lbfgs(B, P, theta_inout, o, obj, results);
  for (int b = 0; b < B && !rc; ++b) results[b].mll = -results[b].mll;  // report f, not -f
  return rc;
}

}  // extern "C"
