"""Embedded Runge-Kutta pairs and the integral step-size controller of the adaptive sampler
(`use_torchode=True`; reference call site cfm_superresolution.py:259-276: `to.Tsit5` / `to.Dopri5` stepped by
`to.IntegralController(atol, rtol)` inside `to.AutoDiffAdjoint`), and torchdiffeq's `dopri5` controller and dense output
(`torchdiffeq_ode_method='dopri5'`, call site cfm_superresolution.py:243; bottom of this file).

Host-side control only: the stage combinations and the scaled error norm run on the GPU (`fh_rk_lincomb_f32`,
`fh_rk_scaled_sumsq_f32`); one 8-byte read per attempted step brings the error ratio back for the accept / reject decision.
torchode 1.0.0 is not installable offline, so the controller follows its published description (PID controller with
(p, i, d) = (0, 1, 0), safety 0.9, factor range [0.2, 10], rms norm, Hairer's initial step) -- see DESIGN.md section 2.
"""
from __future__ import annotations

from dataclasses import dataclass
from fractions import Fraction as Fr
from typing import List, Sequence


@dataclass(frozen=True)
class Tableau:
    name: str
    order: int                 # convergence order k of the propagated solution (controller exponent 1 / k)
    c: Sequence[float]         # stage times
    a: Sequence[Sequence[float]]  # a[s] = weights of k_0 .. k_{s-1} for stage s; a[6] is also the solution row (FSAL)
    e: Sequence[float]         # error-estimate weights b - b_hat


def _f(rows):
    return [[float(x) for x in r] for r in rows]


TSIT5 = Tableau(
    "tsit5", 5,
    (0.0, 0.161, 0.327, 0.9, 0.9800255409045097, 1.0, 1.0),
    ((),
     (0.161,),
     (-0.008480655492356989, 0.335480655492357),
     (2.8971530571054935, -6.359448489975075, 4.3622954328695815),
     (5.325864828439257, -11.748883564062828, 7.4955393428898365, -0.09249506636175525),
     (5.86145544294642, -12.92096931784711, 8.159367898576159, -0.071584973281401, -0.028269050394068383),
     (0.09646076681806523, 0.01, 0.4798896504144996, 1.379008574103742, -3.290069515436081, 2.324710524099774)),
    (-0.00178001105222577714, -0.0008164344596567469, 0.007880878010261995, -0.1447110071732629,
     0.5823571654525552, -0.45808210592918697, 1.0 / 66.0),
)

_DP_A = [[], [Fr(1, 5)], [Fr(3, 40), Fr(9, 40)], [Fr(44, 45), Fr(-56, 15), Fr(32, 9)],
         [Fr(19372, 6561), Fr(-25360, 2187), Fr(64448, 6561), Fr(-212, 729)],
         [Fr(9017, 3168), Fr(-355, 33), Fr(46732, 5247), Fr(49, 176), Fr(-5103, 18656)],
         [Fr(35, 384), Fr(0), Fr(500, 1113), Fr(125, 192), Fr(-2187, 6784), Fr(11, 84)]]
_DP_BHAT = [Fr(5179, 57600), Fr(0), Fr(7571, 16695), Fr(393, 640), Fr(-92097, 339200), Fr(187, 2100), Fr(1, 40)]
DOPRI5 = Tableau(
    "dopri5", 5,
    (0.0, 0.2, 0.3, 0.8, 8.0 / 9.0, 1.0, 1.0),
    tuple(tuple(float(x) for x in r) for r in _DP_A),
    tuple(float(b - bh) for b, bh in zip(_DP_A[6] + [Fr(0)], _DP_BHAT)),
)

TABLEAUX = {"tsit5": TSIT5, "dopri5": DOPRI5}


def resolve(klass) -> Tableau:
    """`torchode_method_klass` as the reference passes it (a class such as torchode.Tsit5), a name, or None (Tsit5,
    the reference default, flowhighsr.py:31)."""
    if klass is None:
        return TSIT5
    name = klass if isinstance(klass, str) else getattr(klass, "__name__", type(klass).__name__)
    tab = TABLEAUX.get(str(name).lower())
    if tab is None:
        raise NotImplementedError(f"torchode step method {name!r}: only Tsit5 and Dopri5 are built")
    return tab


@dataclass
class IntegralController:
    atol: float
    rtol: float
    order: int
    safety: float = 0.9
    factor_min: float = 0.2
    factor_max: float = 10.0

    def accept(self, ratio: float) -> bool:
        return ratio < 1.0

    def next_dt(self, dt: float, ratio: float) -> float:
        if ratio == 0.0:
            return dt * self.factor_max
        return dt * min(self.factor_max, max(self.factor_min, self.safety * ratio ** (-1.0 / self.order)))

    def initial_dt(self, d0: float, d1: float, span: float) -> float:
        h0 = 1e-6 if (d0 < 1e-5 or d1 < 1e-5) else 0.01 * d0 / d1
        return min(h0, span)

    def initial_dt_refine(self, h0: float, d1: float, d2: float, span: float) -> float:
        if d1 <= 1e-15 and d2 <= 1e-15:
            h1 = max(1e-6, h0 * 1e-3)
        else:
            h1 = (0.01 / max(d1, d2)) ** (1.0 / (self.order + 1))
        return min(100.0 * h0, h1, span)


# ---------------------------------------------------------------------------------------------------------------------
# torchdiffeq's `odeint(..., method=...)` (reference call site cfm_superresolution.py:243).  Fixed-grid methods step
# exactly on `t = linspace(0, 1, steps + 1)`; `dopri5` is adaptive and ignores the interior points of `t` except to
# interpolate there.
TORCHDIFFEQ_METHODS = ("euler", "midpoint", "rk4", "dopri5")


def check_torchdiffeq_method(name: str) -> None:
    """Raises ValueError for a torchdiffeq method name this package has not built (bosh3, fehlberg2, adaptive_heun,
    dopri8, the Adams methods, scipy_solver)."""
    if name not in TORCHDIFFEQ_METHODS:
        raise ValueError(f"unsupported ODE method {name!r} ({'|'.join(TORCHDIFFEQ_METHODS)})")


# torchdiffeq's `dopri5` is the Dormand-Prince pair (the `DOPRI5` stages above) with Shampine's embedded 4th-order
# weights for the error estimate -- not the b_hat of `DOPRI5.e` -- and a quartic dense output through y_mid.  The values
# are torchdiffeq's own float expressions (dopri5.py), so they round the same way.
DPS_C_ERROR = (35 / 384 - 1951 / 21600, 0.0, 500 / 1113 - 22642 / 50085, 125 / 192 - 451 / 720,
               -2187 / 6784 - -12231 / 42400, 11 / 84 - 649 / 6300, -1. / 60.)
DPS_C_MID = (6025192743 / 30085553152 / 2, 0.0, 51252292925 / 65400821598 / 2, -2691868925 / 45128329728 / 2,
             187940372067 / 1594534317056 / 2, -1776094331 / 19743644256 / 2, 11237099 / 235043384 / 2)


def dopri5_dense_weights(x: float, dt: float) -> List[float]:
    """Weights w of torchdiffeq's dense output of one accepted dopri5 step at theta = x in [0, 1]:
    y(t0 + x dt) = y0 + sum_i w_i k_i over the 7 stages k_0 (= f0) .. k_6 (= f1, FSAL).  torchdiffeq evaluates
    y0 + x d + x^2 c + x^3 b + x^4 a with d = dt f0, c = dt (f1 - 4 f0) - 11 y0 - 5 y1 + 16 y_mid,
    b = dt (5 f0 - 3 f1) + 18 y0 + 14 y1 - 32 y_mid, a = 2 dt (f1 - f0) - 8 (y1 + y0) + 16 y_mid, where
    y1 = y0 + dt sum b_i k_i and y_mid = y0 + dt sum DPS_C_MID_i k_i; the y0 terms cancel, leaving one linear combination."""
    b = list(DOPRI5.a[6]) + [0.0]
    w = []
    for i in range(7):
        f0, f1 = float(i == 0), float(i == 6)
        c = f1 - 4.0 * f0 - 5.0 * b[i] + 16.0 * DPS_C_MID[i]
        bb = 5.0 * f0 - 3.0 * f1 + 14.0 * b[i] - 32.0 * DPS_C_MID[i]
        a = 2.0 * (f1 - f0) - 8.0 * b[i] + 16.0 * DPS_C_MID[i]
        w.append(dt * (x * f0 + x ** 2 * c + x ** 3 * bb + x ** 4 * a))
    return w


@dataclass
class TorchdiffeqController:
    """Step-size rules of torchdiffeq's adaptive Runge-Kutta solvers (rk_common.py / misc.py): accept when the rms error
    ratio is <= 1; next dt = dt * min(ifactor, max(safety / ratio^(1/order), dfactor)) with dfactor = 1 after a ratio
    below 1 (no shrinking after a good step) and 0.2 otherwise, dt * ifactor when the ratio is 0; no clamp to the span
    (the last step overshoots the end and the result is interpolated).  Initial step: Hairer's heuristic with exponent
    1 / order (torchdiffeq passes order - 1 and raises to 1 / (order' + 1)), and no clamp either."""
    atol: float
    rtol: float
    order: int = 5
    safety: float = 0.9
    ifactor: float = 10.0
    dfactor: float = 0.2

    def accept(self, ratio: float) -> bool:
        return ratio <= 1.0

    def next_dt(self, dt: float, ratio: float) -> float:
        if ratio == 0.0:
            return dt * self.ifactor
        dfactor = 1.0 if ratio < 1.0 else self.dfactor
        return dt * min(self.ifactor, max(self.safety / ratio ** (1.0 / self.order), dfactor))

    def initial_dt(self, d0: float, d1: float) -> float:
        return 1e-6 if (d0 < 1e-5 or d1 < 1e-5) else 0.01 * d0 / d1

    def initial_dt_refine(self, h0: float, d1: float, d2: float) -> float:
        if d1 <= 1e-15 and d2 <= 1e-15:
            h1 = max(1e-6, h0 * 1e-3)
        else:
            h1 = (0.01 / max(d1, d2)) ** (1.0 / self.order)
        return min(100.0 * h0, h1)
