// Host-side launch sequence of one solver.run() over a batch (shared by solver.cu and the test-only host
// emulation).  Mirrors the loop structure of aligator::SolverProxDDPTpl::run (fulldynamic_talos.py:393-397).
// Kernels run over COMPACTED instance lists so that the cost of late linesearch rounds / late iterations is
// proportional to the number of instances still working, not to the batch.
#pragma once
#include "solver_core.cuh"
#include <type_traits>

namespace mpcdev {

// f(std::integral_constant<int, KIND>{}) for the runtime model kind: the one place where a kind becomes the template argument
// of KindTraits and of the kernels
template <class F> auto dispatch_kind(int kind, F &&f) {
  switch (kind) {
  case MPC_KIND_FULL: return f(std::integral_constant<int, MPC_KIND_FULL>{});
  case MPC_KIND_KINO: return f(std::integral_constant<int, MPC_KIND_KINO>{});
  default: return f(std::integral_constant<int, MPC_KIND_CENT>{});
  }
}

// Backend: reset_counters(), eval(deriv, list, n), decide_eval(list, n, next_eval), riccati(list, n), apply_step(list, n),
//          decide_ls(list, n, ls_out, next_eval), rollout_ls(list, n, next_eval), read_counters(int[4])
// first / count: the sub-batch [first, first + count) of instances this call advances (the first pass takes its list from the
// identity list written by the run prologue; later passes use the compacted lists the decide kernels build)
template <class Backend> int run_loop(Backend &be, const Ws &w, int max_iters, const SolverConst &sc, int first = 0, int count = -1) {
  int launches = 0, n_eval = (count < 0) ? w.B : count, cur = 0;
  const int guard = max_iters + sc.max_al_iters + 2;
  for (int pass = 0; pass < guard && n_eval > 0; pass++) {
    int32_t *L = eval_list(w, cur) + (pass == 0 ? first : 0), *Lnext = eval_list(w, cur + 1);
    be.reset_counters();
    be.eval(true, L, n_eval); be.decide_eval(L, n_eval, Lnext); be.riccati(L, n_eval);
    int c[4] = {0, 0, 0, 0};
    if (sc.rollout == 1) { // ROLLOUT_NONLINEAR: rollout and the whole linesearch of every instance in ONE kernel
      be.rollout_ls(L, n_eval, Lnext);
      launches += 4;
      be.read_counters(c);
      n_eval = c[2];
      cur ^= 1;
      continue;
    }
    be.apply_step(L, n_eval); be.eval(false, L, n_eval); be.decide_ls(L, n_eval, ls_list(w, 0), Lnext);
    launches += 6;
    be.read_counters(c);
    int n_ls = c[0];
    for (int r = 0; n_ls > 0 && r <= sc.ls_max_steps; r++) {
      int32_t *Lin = ls_list(w, r), *Lout = ls_list(w, r + 1);
      be.apply_step(Lin, n_ls); be.eval(false, Lin, n_ls); be.decide_ls(Lin, n_ls, Lout, Lnext);
      launches += 3;
      be.read_counters(c);
      n_ls = c[0];
    }
    n_eval = c[2];
    cur ^= 1;
  }
  return launches;
}

// one instance's solve summary as the C-ABI returns it
inline mpc_info_t info_of(const InstState &s) {
  mpc_info_t o;
  o.prim_infeas = s.prim_infeas; o.dual_infeas = s.dual_infeas; o.traj_cost = s.traj_cost; o.merit = s.merit; o.mu = s.mu; o.alpha = s.alpha;
  o.ls_evals = s.ls_evals; o.pad_ = 0; o.num_iters = s.num_iters; o.al_iters = s.al_iters; o.conv = s.conv; o.status = s.status;
  return o;
}

} // namespace mpcdev
