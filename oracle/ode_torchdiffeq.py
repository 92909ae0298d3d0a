"""ORACLE (test infrastructure, not product code) -- torchdiffeq's `rk4` and adaptive `dopri5` solvers, and the CFM
sampler with them.

Reference call site: cfm_superresolution.py:243
    trajectory = torchdiffeq.odeint(ode_fn, y0, t, atol=atol, rtol=rtol, method=torchdiffeq_ode_method)
torchdiffeq (pyproject.toml:14 `torchdiffeq>=0.2.3`) is NOT installed offline, so this file restates its published
`rk4` (fixed_grid.py: rk4_alt_step_func, the 3/8 rule, its last stage at the grid point t1; euler / midpoint stay in
model.odeint_fixed) and `dopri5` (torchdiffeq/_impl/dopri5.py, rk_common.py, misc.py, interp.py):
  * Dormand-Prince stages with FSAL (7 stages, 6 new field evaluations per attempted step); the error estimate uses
    Shampine's embedded weights (`C_ERROR`), not the classic b_hat.
  * state tensors keep their dtype; times are promoted to fp64; inside a step t0, dt and t0 + dt are cast to the state's
    dtype, stages with c = 1 sit at t0 + dt, and the field receives `t.to(y.dtype)`.
  * initial step: Hairer's heuristic with order - 1 = 4 (exponent 1/5), no clamp to the span.
  * error ratio = rms over the WHOLE state tensor of err / (atol + rtol * max(|y0|, |y1|)); accept when <= 1;
    dt_next = dt * min(10, max(0.9 / ratio^(1/5), dfactor)), dfactor = 1 when ratio < 1 and 0.2 otherwise; dt * 10 when
    ratio == 0.
  * the solver steps while the last accepted step ends before the requested time (so the last step overshoots) and
    every output time is the quartic dense output of the step that covers it.  Output times never shorten a step, so
    the final state does not depend on the interior points of t.
A batch tensor is ONE problem: one shared step sequence, one norm over every clip (what the reference's `sample()` does
with B > 1).

PARITY UNPINNED against torchdiffeq itself: without the package no golden can be generated.  What the tests pin instead
(tests/test_ode_methods_cpu.py): rk4 against a hand expansion of the 3/8 rule and its convergence order; for dopri5 the
embedded weights against the Runge-Kutta order conditions, the dense output exact on a quartic solution, the solution
against scipy's DOP853 at 1e-12 on a closed-form problem and on Van der Pol, and independence of the final state from the
interior output times.
"""
from __future__ import annotations

from typing import Callable, Tuple

import torch

from . import model

# torchdiffeq's _DORMAND_PRINCE_SHAMPINE_TABLEAU (alpha, beta, c_error) and DPS_C_MID, as its own float expressions
# (the solution row is the last beta row: FSAL)
ALPHA = [1 / 5, 3 / 10, 4 / 5, 8 / 9, 1., 1.]
BETA = [[1 / 5], [3 / 40, 9 / 40], [44 / 45, -56 / 15, 32 / 9], [19372 / 6561, -25360 / 2187, 64448 / 6561, -212 / 729],
        [9017 / 3168, -355 / 33, 46732 / 5247, 49 / 176, -5103 / 18656],
        [35 / 384, 0, 500 / 1113, 125 / 192, -2187 / 6784, 11 / 84]]
C_ERROR = [35 / 384 - 1951 / 21600, 0, 500 / 1113 - 22642 / 50085, 125 / 192 - 451 / 720, -2187 / 6784 - -12231 / 42400,
           11 / 84 - 649 / 6300, -1. / 60.]
C_MID = [6025192743 / 30085553152 / 2, 0, 51252292925 / 65400821598 / 2, -2691868925 / 45128329728 / 2,
         187940372067 / 1594534317056 / 2, -1776094331 / 19743644256 / 2, 11237099 / 235043384 / 2]


def _rms(x: torch.Tensor) -> torch.Tensor:
    return x.abs().pow(2).mean().sqrt()


def odeint_dopri5(fn: Callable, y0: torch.Tensor, t: torch.Tensor, *, atol: float, rtol: float,
                  max_steps: int = 10000) -> Tuple[torch.Tensor, dict]:
    """Solution at every time of t ([len(t), *y0.shape], like torchdiffeq.odeint) and the solve's step statistics."""
    dt_, dty = torch.float64, y0.dtype
    t = t.to(dt_)
    beta = [torch.tensor(r, dtype=dty) for r in BETA]
    c_err = torch.tensor(C_ERROR, dtype=dty)
    mid = torch.tensor(C_MID, dtype=dty)
    atol_t, rtol_t = torch.tensor(atol, dtype=dt_), torch.tensor(rtol, dtype=dt_)
    f = lambda tt, yy: fn(tt.to(yy.dtype), yy)

    f0 = f(t[0], y0)
    nfe = 1
    # _select_initial_step(order = 5 - 1)
    scale = atol_t + torch.abs(y0) * rtol_t
    d0, d1 = _rms(y0 / scale), _rms(f0 / scale)
    h0 = torch.tensor(1e-6, dtype=dty) if (d0 < 1e-5 or d1 < 1e-5) else 0.01 * d0 / d1
    f1 = f(t[0] + h0, y0 + h0 * f0)
    nfe += 1
    d2 = torch.abs(_rms((f1 - f0) / scale) / h0)
    if d1 <= 1e-15 and d2 <= 1e-15:
        h1 = torch.max(torch.tensor(1e-6, dtype=dty), h0 * 1e-3)
    else:
        h1 = (0.01 / max(d1, d2)) ** (1.0 / 5.0)
    dt = torch.min(100 * h0, h1).to(dt_)

    y, fy, tcur = y0, f0, t[0]
    interp, step_t0, step_t1 = None, t[0], t[0]
    n_steps = n_acc = 0
    sol = [y0]
    for tn in t[1:]:
        while tn > step_t1:
            if n_steps >= max_steps:
                raise RuntimeError(f"adaptive solve did not reach t_end in {max_steps} steps (t = {float(step_t1)})")
            t1 = tcur + dt
            t0s, dts, t1s = tcur.to(dty), dt.to(dty), t1.to(dty)
            k = [fy]
            for i in range(6):
                ti = t1s if ALPHA[i] == 1.0 else t0s + ALPHA[i] * dts
                yi = y + sum(kk * (w * dts) for kk, w in zip(k, beta[i]))
                k.append(fn(ti, yi))
            nfe += 6
            y1, f1 = yi, k[6]
            err = sum(kk * (w * dts) for kk, w in zip(k, c_err))
            ratio = _rms(err / (atol_t + rtol_t * torch.max(y.abs(), y1.abs()))).to(dt_)
            n_steps += 1
            if ratio <= 1:
                n_acc += 1
                y_mid = y + sum(kk * (w * dts) for kk, w in zip(k, mid))
                interp = [y, dts * fy, dts * (f1 - 4 * fy) - 11 * y - 5 * y1 + 16 * y_mid,
                          dts * (5 * fy - 3 * f1) + 18 * y + 14 * y1 - 32 * y_mid,
                          2 * dts * (f1 - fy) - 8 * (y1 + y) + 16 * y_mid]
                step_t0, step_t1 = tcur, t1
                tcur, y, fy = t1, y1, f1
            # _optimal_step_size
            if ratio == 0:
                dt = dt * 10.0
            else:
                dfactor = 1.0 if ratio < 1 else 0.2
                dt = dt * torch.min(torch.tensor(10.0, dtype=dt_),
                                    torch.max(0.9 / ratio ** (1.0 / 5.0), torch.tensor(dfactor, dtype=dt_)))
        x = ((tn - step_t0) / (step_t1 - step_t0)).to(dty)
        total, xp = interp[0] + x * interp[1], x
        for coef in interp[2:]:
            xp = xp * x
            total = total + xp * coef
        sol.append(total)
    return torch.stack(sol), {"n_steps": n_steps, "n_accepted": n_acc, "n_f_evals": nfe}


def odeint_rk4(fn: Callable, y0: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    """Final state of torchdiffeq's fixed-grid `rk4` on grid t (rk4_alt_step_func: the 3/8 rule, not classic RK4)."""
    y = y0
    for i in range(len(t) - 1):
        t0, t1 = t[i], t[i + 1]
        dt = t1 - t0
        k1 = fn(t0, y)
        k2 = fn(t0 + dt * (1 / 3), y + dt * k1 * (1 / 3))
        k3 = fn(t0 + dt * (2 / 3), y + dt * (k2 - k1 * (1 / 3)))
        k4 = fn(t1, y + dt * (k1 - k2 + k3))
        y = y + (k1 + 3 * (k2 + k3) + k4) * dt * 0.125
    return y


def cfm_sample_mel(sd, cond_mel, eps, *, steps, ode_method, cfm_method, sigma, cond_scale=1.0, atol=1e-5, rtol=1e-5,
                   depth=2, heads=16):
    """model.cfm_sample_mel (the reference's `sample()` up to `sampled`, without mel_pp) for every torchdiffeq method built
    here.  dopri5 solves the batch as one problem (one step sequence, one error norm over all clips), exactly as the
    reference's `sample()` does with B > 1."""
    y0 = model.cfm_prior(cond_mel, eps, cfm_method, sigma)
    t = torch.linspace(0, 1, steps + 1)
    fn = lambda tt, yy: model.vector_field_cfg(sd, yy, cond_mel, tt, cond_scale=cond_scale, depth=depth, heads=heads)
    if ode_method == "rk4":
        return odeint_rk4(fn, y0, t)
    if ode_method == "dopri5":
        return odeint_dopri5(fn, y0, t, atol=atol, rtol=rtol)[0][-1]
    return model.odeint_fixed(fn, y0, t, ode_method)
