"""Batched iLQR on the device (DESIGN.md §4g): a Gauss-Newton shooting solver for the tracking cost of `TrackingCost`, every
scenario of a batch solved at once.

One iteration per scenario b, around the current trajectory (xbar, taubar):
  1. the step Jacobians at nodes 0..N-1 (`step_rk4_jvp`);
  2. the Riccati feedback gains of the Gauss-Newton model, with mu_b added to the torque curvature (`riccati_gains`);
  3. the closed-loop cost of every step length in `alphas` (`ilqr_costs`);
  4. alpha_b = the candidate with the smallest cost strictly below J_b (the earlier entry on a tie; NaN never wins), else 0;
  5. the closed-loop rollout with alpha_b, which also gives the cost's gradient and curvature planes (`feedback_rollout`);
  6. mu_b / 10 (floored at mu_min) on an accepted step, mu_b * 10 on a rejection; mu_b > mu_max is "stalled";
  7. converged when an accepted step lowers J_b by less than tol J_b + atol, or when the feedforward is negligible,
     max_k |k_k|_inf <= ktol (1 + |taubar|_inf).
A scenario that has converged, stalled or started non-finite keeps alpha_b = 0, which reproduces its trajectory bit for bit, so its
result depends on its own data only.  The loop synchronises once per iteration, for the all-done check.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

RUNNING, CONVERGED, MAX_ITERATIONS, STALLED, NONFINITE = 0, 1, 2, 3, 4
STATUS_NAMES = {RUNNING: "running", CONVERGED: "converged", MAX_ITERATIONS: "max_iterations", STALLED: "stalled", NONFINITE: "nonfinite"}


@dataclass
class TrackingCost:
    """The tracking cost of include/mpcf.h (mpcf_track_cost).  Device float64 tensors, None = zero (or, for bound_table, absent):
    x_ref [3n, (N+1)*B], tau_ref [n, N*B], weight vectors wx [3n], wu [n], wN [3n], bound_table [N, n, 2] = (lb, ub) (as built by
    ocp.f0_bound_table, step_bound_table or switch_off_bound_table).  Per scenario:
      J = sum_{k<N} 1/2 |x_k - x_ref_k|^2_wx + 1/2 |tau_k - tau_ref_k|^2_wu + rho_tau/2 |(lb_k - tau_k)+|^2 + rho_tau/2 |(tau_k - ub_k)+|^2
          + rho_f/2 |(f_k - f_max)+|^2  +  1/2 |x_N - x_ref_N|^2_wN + rho_f/2 |(f_N - f_max)+|^2"""
    x_ref: torch.Tensor | None = None
    tau_ref: torch.Tensor | None = None
    wx: torch.Tensor | None = None
    wu: torch.Tensor | None = None
    wN: torch.Tensor | None = None
    bound_table: torch.Tensor | None = None
    rho_tau: float = 0.0
    f_max: float = math.inf
    rho_f: float = 0.0


@dataclass
class ILQRResult:
    x: torch.Tensor        # [3n, (N+1)*B]
    tau: torch.Tensor      # [n, N*B]
    J: torch.Tensor        # [B]
    iters: torch.Tensor    # [B] int64: iterations until the scenario stopped
    status: torch.Tensor   # [B] int64: CONVERGED, MAX_ITERATIONS, STALLED or NONFINITE
    history: torch.Tensor  # [iterations + 1, B]: J before the first iteration and after each


def select_alpha(Jc: torch.Tensor, Jbar: torch.Tensor, alphas) -> tuple[torch.Tensor, torch.Tensor]:
    """The step-length rule: Jc [na, B] candidate costs, Jbar [B] current costs.  Per scenario the candidate with the smallest cost
    strictly below Jbar wins (NaN never: NaN < Jbar is false); on a tie the earlier entry of `alphas`.  Returns (alpha [B], accepted
    [B] bool); alpha = 0 where no candidate is below Jbar."""
    a = torch.as_tensor([float(v) for v in alphas], dtype=Jc.dtype, device=Jc.device)
    ok = Jc < Jbar[None, :]
    masked = torch.where(ok, Jc, torch.full_like(Jc, math.inf))
    idx = torch.argmin(masked, dim=0)  # the first of equal minima
    accepted = ok.any(dim=0)
    return torch.where(accepted, a[idx], torch.zeros_like(Jbar)), accepted


def solve_ilqr(ev, x0, tau_init, N: int, dt: float, cost: TrackingCost, *, alphas=tuple(0.5 ** i for i in range(8)), iters: int = 100,
               mu0: float = 1e-8, mu_min: float = 1e-12, mu_max: float = 1e10, tol: float = 1e-10, atol: float = 0.0,
               ktol: float = 1e-10) -> ILQRResult:
    """Gauss-Newton iLQR of B scenarios: x0 [3n, B] (the (q, qd, f) rows), tau_init [n, N*B] node-major.  `ev` is a
    BatchEvaluator; n <= 16 (the Riccati entry's limit).  See the module docstring for one iteration."""
    n, N = ev.n, int(N)
    B = x0.shape[1]
    U = N * B
    alphas = tuple(float(a) for a in alphas)
    x, tau, J, dv = ev.feedback_rollout(cost, x0, tau_init.contiguous(), N, dt, derivatives=True)
    f64 = dict(dtype=torch.float64, device=x.device)
    mu = torch.full((B,), float(mu0), **f64)
    status = torch.where(torch.isfinite(J), RUNNING, NONFINITE).to(torch.int64)
    count = torch.zeros(B, dtype=torch.int64, device=x.device)
    history = [J]
    for _ in range(int(iters)):
        if not bool((status == RUNNING).any()):  # the one synchronisation of an iteration
            break
        run = status == RUNNING
        # 1. step Jacobians at nodes 0..N-1 of the current trajectory
        xs = [x[r * n:(r + 1) * n, :U].contiguous() for r in range(3)]
        jac = ev.step_rk4_jvp(xs[0], xs[1], tau, xs[2], dt)[3]
        # 2. gains of the Gauss-Newton model, mu_b on the torque curvature
        wu = (dv["wu"].view(n, N, B) + mu).view(n, U)
        K = ev.riccati_gains(jac, B, N, wx=dv["wx"], wu=wu, gx=dv["gx"], gu=dv["gu"], wN=dv["wN"], gN=dv["gN"])
        del jac
        kff = K[:, 3 * n].reshape(n * N, B).abs().amax(dim=0)
        small = kff <= ktol * (1.0 + tau.view(n * N, B).abs().amax(dim=0))
        # 3. + 4. line search over the candidates and the per-scenario choice
        Jc = ev.ilqr_costs(cost, x0, x, tau, K, alphas, N, dt)
        alpha, accepted = select_alpha(Jc, J, alphas)
        live = run & ~small
        alpha = torch.where(live, alpha, torch.zeros_like(alpha))
        accepted = accepted & live
        # 5. accept pass
        xn, taun, Jn, dv = ev.feedback_rollout(cost, x0, tau, N, dt, xbar=x, K=K, alpha=alpha, derivatives=True)
        # 6. + 7. Levenberg update and the stopping tests
        conv = (run & small) | (accepted & (J - Jn < tol * J + atol))
        mu = torch.where(live, torch.where(accepted, torch.clamp(mu / 10.0, min=mu_min), mu * 10.0), mu)
        stalled = live & ~accepted & (mu > mu_max)
        count = count + run.to(torch.int64)
        status = torch.where(conv, CONVERGED, torch.where(stalled, STALLED, status))
        x, tau, J = xn, taun, Jn
        history.append(J)
    status = torch.where(status == RUNNING, MAX_ITERATIONS, status)
    return ILQRResult(x=x, tau=tau, J=J, iters=count, status=status, history=torch.stack(history))
