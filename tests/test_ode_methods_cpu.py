"""CPU suite for torchdiffeq's `rk4` and `dopri5` (`torchdiffeq_ode_method`): torchdiffeq is absent offline, so the
restatements (oracle/ode_torchdiffeq.py) and the product's host-side pieces
(flowhigh_b200/rk.py) are pinned against mathematics and scipy instead of goldens."""
import math

import numpy as np
import pytest
import torch

from flowhigh_b200 import rk
from oracle import model, ode_torchdiffeq as otd
from util import golden_weights, load_golden

f64 = torch.float64


# ------------------------------------------------------------------ rk4 (fixed grid)
def test_rk4_is_the_three_eighths_rule():
    """y' = y^2 + t^3: one step against a hand expansion of the 3/8 rule (bit for bit) and away from classic RK4."""
    fn = lambda t, y: y * y + t ** 3
    y0, h = torch.tensor([0.7], dtype=f64), 0.3
    t = torch.tensor([0.0, h], dtype=f64)
    k1 = fn(t[0], y0)
    k2 = fn(t[0] + h * (1 / 3), y0 + h * k1 * (1 / 3))
    k3 = fn(t[0] + h * (2 / 3), y0 + h * (k2 - k1 * (1 / 3)))
    k4 = fn(t[1], y0 + h * (k1 - k2 + k3))
    want = y0 + (k1 + 3 * (k2 + k3) + k4) * h * 0.125
    got = otd.odeint_rk4(fn, y0, t)
    assert torch.equal(got, want)
    c1 = fn(0.0, y0)
    c2 = fn(h / 2, y0 + h / 2 * c1)
    c3 = fn(h / 2, y0 + h / 2 * c2)
    c4 = fn(h, y0 + h * c3)
    classic = y0 + h / 6 * (c1 + 2 * c2 + 2 * c3 + c4)
    assert float((got - classic).abs()) > 1e-6


def test_rk4_converges_with_order_four():
    A = torch.tensor([[-0.5, 3.0], [-3.0, -0.2]], dtype=f64)
    y0 = torch.tensor([[1.0, -0.5]], dtype=f64)
    fn = lambda t, y: y @ A.T + torch.cos(2 * t) * torch.tensor([1.0, 0.0], dtype=f64)
    fine = otd.odeint_rk4(fn, y0, torch.linspace(0, 1, 2049, dtype=f64))
    errs = [float((otd.odeint_rk4(fn, y0, torch.linspace(0, 1, n + 1, dtype=f64)) - fine).abs().max())
            for n in (8, 16, 32)]
    orders = [math.log2(errs[i] / errs[i + 1]) for i in range(2)]
    assert all(3.7 <= o <= 4.3 for o in orders), (errs, orders)


# ------------------------------------------------------------------ dopri5 constants and dense output
def test_dopri5_constants_match_torchdiffeq_restatement_and_order_conditions():
    assert tuple(otd.C_ERROR) == rk.DPS_C_ERROR and tuple(otd.C_MID) == rk.DPS_C_MID
    for row_o, row_p in zip(otd.BETA, rk.DOPRI5.a[1:]):
        assert np.abs(np.array(row_o) - np.array(row_p)).max() <= 1e-16
    # b_hat = b - c_error is a 4th-order solution: e = c_error satisfies every condition through order 4
    A = np.zeros((7, 7))
    for i, r in enumerate(rk.DOPRI5.a):
        A[i, :len(r)] = r
    c, e = np.array(rk.DOPRI5.c), np.array(rk.DPS_C_ERROR)
    conds = [e.sum(), e @ c, e @ c ** 2, e @ (A @ c), e @ c ** 3, (e * c) @ (A @ c), e @ (A @ c ** 2), e @ (A @ (A @ c))]
    assert max(abs(x) for x in conds) <= 1e-15
    assert abs(e @ c ** 4) > 1e-5  # and not a 5th-order one


def test_dopri5_dense_output_reproduces_a_quartic():
    """y' = 4 t^3 has the quartic solution t^4: the oracle's interpolated interior points are exact, and the product's
    dense-output weights give the oracle's interpolant."""
    fn = lambda t, y: 4 * t ** 3 * torch.ones_like(y)
    t = torch.linspace(0, 1, 7, dtype=f64)
    y, st = otd.odeint_dopri5(fn, torch.zeros(1, dtype=f64), t, atol=1e-6, rtol=1e-6)
    assert float((y[:, 0] - t ** 4).abs().max()) <= 1e-12 and st["n_steps"] >= 2
    # one step from t0 = 0.3 with dt = 0.5: dense output at every theta against the exact quartic
    t0, dt = 0.3, 0.5
    k = [4 * (t0 + ci * dt) ** 3 for ci in rk.DOPRI5.c]
    for x in (0.0, 0.25, 0.4, 0.8, 1.0):
        w = rk.dopri5_dense_weights(x, dt)
        assert abs(t0 ** 4 + sum(wi * ki for wi, ki in zip(w, k)) - (t0 + x * dt) ** 4) <= 1e-12


def test_controller_follows_torchdiffeq_rules():
    ctl = rk.TorchdiffeqController(atol=1e-5, rtol=1e-5)
    for ratio in (0.0, 1e-9, 0.3, 0.999, 1.0, 1.7, 1e6):
        if ratio == 0.0:
            want = 10.0
        else:
            want = min(10.0, max(0.9 / ratio ** 0.2, 1.0 if ratio < 1 else 0.2))
        assert ctl.next_dt(0.125, ratio) == pytest.approx(0.125 * want, rel=1e-15)
        assert ctl.accept(ratio) == (ratio <= 1.0)
    assert ctl.next_dt(0.125, 0.9) == 0.125  # 0.9 / 0.9^0.2 < 1: no shrinking after a good step
    assert ctl.initial_dt(1.0, 1e-6) == 1e-6 and ctl.initial_dt(2.0, 4.0) == pytest.approx(0.005)
    assert ctl.initial_dt_refine(0.5, 0.01, 0.02) == pytest.approx((0.01 / 0.02) ** 0.2)  # no clamp to a span of 1
    assert ctl.initial_dt_refine(0.002, 0.01, 1e-3) == pytest.approx(0.2)


@pytest.mark.parametrize("name", ["bosh3", "fehlberg2", "adaptive_heun", "dopri8", "explicit_adams", "implicit_adams",
                                  "fixed_adams", "scipy_solver", "heun3", "rk45"])
def test_unsupported_methods_raise(name):
    with pytest.raises(ValueError, match="euler|midpoint|rk4|dopri5"):
        rk.check_torchdiffeq_method(name)
    with pytest.raises(ValueError):
        otd.cfm_sample_mel({}, torch.zeros(1, 2, 256), torch.zeros(1, 2, 256), steps=2, ode_method=name,
                           cfm_method="basic_cfm", sigma=0.0)


def test_built_methods_pass_the_check():
    for name in ("euler", "midpoint", "rk4", "dopri5"):
        rk.check_torchdiffeq_method(name)


# ------------------------------------------------------------------ dopri5 against scipy
def test_dopri5_meets_tolerance_on_closed_form():
    from scipy.integrate import solve_ivp
    tol = 1e-6
    A = np.array([[-0.5, 6.0], [-6.0, -0.3]])
    y0 = np.array([1.0, 0.5])
    At = torch.tensor(A)
    fn = lambda t, y: y @ At.T
    y, st = otd.odeint_dopri5(fn, torch.tensor(y0)[None], torch.linspace(0, 1, 2, dtype=f64), atol=tol, rtol=tol)
    tight = solve_ivp(lambda t, y: A @ y, (0.0, 1.0), y0, method="DOP853", atol=1e-12, rtol=1e-12).y[:, -1]
    assert np.abs(y[-1, 0].numpy() - tight).max() <= 20 * tol
    assert st["n_f_evals"] == 2 + 6 * st["n_steps"] and st["n_accepted"] <= st["n_steps"]


def test_dopri5_meets_tolerance_on_van_der_pol():
    from scipy.integrate import solve_ivp
    tol = 1e-6

    def vdp(t, y):
        return np.array([y[1], 2.0 * (1.0 - y[0] ** 2) * y[1] - y[0]])
    y0 = np.array([2.0, 0.0])
    tight = solve_ivp(vdp, (0.0, 3.0), y0, method="DOP853", atol=1e-12, rtol=1e-12).y[:, -1]
    fn = lambda t, y: torch.stack([y[0, 1], 2.0 * (1.0 - y[0, 0] ** 2) * y[0, 1] - y[0, 0]])[None]
    y, st = otd.odeint_dopri5(fn, torch.tensor(y0)[None], torch.linspace(0, 3, 2, dtype=f64), atol=tol, rtol=tol)
    print(f"dopri5 Van der Pol tol {tol:g}: err {np.abs(y[-1, 0].numpy() - tight).max():.3g} in {st['n_steps']} steps")
    assert np.abs(y[-1, 0].numpy() - tight).max() <= 20 * tol


def test_dopri5_joint_and_per_instance_norms_differ():
    """Two instances of very different scale: solved as one problem they share one step sequence (torchdiffeq on a
    batch tensor), solved apart each has its own -- both scopes are real and give different results."""
    A = torch.tensor([[-0.5, 6.0], [-6.0, -0.3]], dtype=f64)
    fn = lambda t, y: y @ A.T
    y0 = torch.tensor([[1.0, 0.5], [40.0, -30.0]], dtype=f64)
    t = torch.linspace(0, 1, 2, dtype=f64)
    joint, stj = otd.odeint_dopri5(fn, y0, t, atol=1e-4, rtol=1e-4)
    apart = [otd.odeint_dopri5(fn, y0[b: b + 1], t, atol=1e-4, rtol=1e-4) for b in range(2)]
    sep = torch.cat([a[0][-1] for a in apart])
    assert not torch.equal(joint[-1], sep)
    assert stj["n_steps"] not in [a[1]["n_steps"] for a in apart] or not torch.equal(joint[-1, 0], sep[0])


# ------------------------------------------------------------------ the FLowHigh field
def _field_problem(n=16):
    g = load_golden("gen_basic_midpoint")
    sd, _ = golden_weights(g)
    cond = torch.from_numpy(np.ascontiguousarray(g["ref_cond_mel"]))[:, :n].contiguous()
    eps = torch.from_numpy(np.ascontiguousarray(g["eps"])).reshape(1, -1, 256)[:, :n].contiguous()
    return sd, cond, eps


def test_dopri5_final_state_does_not_depend_on_time_steps():
    sd, cond, eps = _field_problem()
    kw = dict(ode_method="dopri5", cfm_method="basic_cfm", sigma=0.0, atol=1e-3, rtol=1e-3)
    a = otd.cfm_sample_mel(sd, cond, eps, steps=1, **kw)
    b = otd.cfm_sample_mel(sd, cond, eps, steps=4, **kw)
    assert torch.equal(a, b)


def test_rk4_field_solve_beats_midpoint_against_fine_grid():
    """On the reference-pinned FLowHigh field (fp64), 4 rk4 steps are closer to a 64-step rk4 solve than 8 midpoint
    steps (same 16 NFEs), and dopri5 at 1e-6 is closer still."""
    sd, cond, eps = _field_problem(12)
    sd = {k: v.double() if v.is_floating_point() else v for k, v in sd.items()}
    fn = lambda t, y: model.vector_field(sd, y, cond.double(), t.double())
    y0 = eps.double()
    grid = lambda n: torch.linspace(0, 1, n + 1, dtype=f64)
    fine = otd.odeint_rk4(fn, y0, grid(64))
    e_rk4 = float((otd.odeint_rk4(fn, y0, grid(4)) - fine).abs().max())
    e_mid = float((model.odeint_fixed(fn, y0, grid(8), "midpoint") - fine).abs().max())
    yd, st = otd.odeint_dopri5(fn, y0, grid(1), atol=1e-6, rtol=1e-6)
    e_dp = float((yd[-1] - fine).abs().max())
    print(f"vs 64-step rk4: 4 rk4 steps {e_rk4:.3g}, 8 midpoint steps {e_mid:.3g}, dopri5 1e-6 {e_dp:.3g} ({st})")
    assert e_dp < 0.2 * e_rk4 < 0.2 * e_mid
