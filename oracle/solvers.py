"""Oracle restatement of the third-party solvers the reference calls (TEST INFRASTRUCTURE ONLY).

PARITY UNPINNED: torchdiffeq / torchsde are not vendored by the reference, not pinned and not
installed here.  What follows restates their published algorithms (torchdiffeq 0.2.x, torchsde 0.2.x)
from the call sites' point of view:

  * ``odeint(func, y0, t)``                /root/reference/scripts/xor_ode.py:114, parity_ode.py:233,
                                           plotting_results.py:131, bifurcation_ode.py:163,210
  * ``sdeint(sde, y0, ts, names=, method=)``  /root/reference/scripts/wta_ode.py:174,200

Algorithms restated
  * fixed grid ``rk4``: the 3/8-rule step (torchdiffeq ``rk4_alt_step_func``) on the grid ``t``, outputs by
    linear interpolation (exact at grid points);
  * adaptive ``dopri5``: Dormand-Prince 5(4) with FSAL, Hairer initial step, RMS error ratio over the whole
    state tensor, step controller (safety .9, ifactor 10, dfactor .2), 4th-order dense output through y_mid;
    time kept in float64, state in the dtype of y0, coefficients cast to the dtype of y0;
  * ``odeint_adjoint``: continuous adjoint, augmented state integrated backwards between output times;
  * torchsde integrate loop with the Euler-Maruyama step, fixed step and step-doubling adaptive;
  * torchsde ``method='srk'`` for scalar / diagonal noise: Roessler's SRI2 scheme ("SRID2" tableau, strong order
    1.5) driven by the Brownian increment W and the space-time Levy area U = int (W_r - W_s) dr of every step --
    what every committed sdeint call of the reference names (scripts/wta_ode.py:174,200,
    plotting_results.py:391,506,594), fixed step and step-doubling adaptive (scripts/parity_ode.py:234).

``tests/test_oracle_selfcheck.py`` anchors them (order conditions, convergence order, analytic solutions).
All functions take ``func(t, y)`` with y of shape (B, D); the reference modules are used with B = 1.
"""
from __future__ import annotations

import math
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch

# ----------------------------------------------------------------------------------------------------------------
# Dormand-Prince 5(4) tableau (Shampine's dense-output variant used by torchdiffeq).
# ----------------------------------------------------------------------------------------------------------------
DP_ALPHA = [1 / 5, 3 / 10, 4 / 5, 8 / 9, 1.0, 1.0]
DP_BETA = [
    [1 / 5],
    [3 / 40, 9 / 40],
    [44 / 45, -56 / 15, 32 / 9],
    [19372 / 6561, -25360 / 2187, 64448 / 6561, -212 / 729],
    [9017 / 3168, -355 / 33, 46732 / 5247, 49 / 176, -5103 / 18656],
    [35 / 384, 0.0, 500 / 1113, 125 / 192, -2187 / 6784, 11 / 84],
]
DP_C_SOL = [35 / 384, 0.0, 500 / 1113, 125 / 192, -2187 / 6784, 11 / 84, 0.0]
DP_C_ERR = [
    35 / 384 - 1951 / 21600,
    0.0,
    500 / 1113 - 22642 / 50085,
    125 / 192 - 451 / 720,
    -2187 / 6784 - -12231 / 42400,
    11 / 84 - 649 / 6300,
    -1.0 / 60.0,
]
DP_C_MID = [
    6025192743 / 30085553152 / 2, 0.0, 51252292925 / 65400821598 / 2, -2691868925 / 45128329728 / 2,
    187940372067 / 1594534317056 / 2, -1776094331 / 19743644256 / 2, 11237099 / 235043384 / 2,
]

ONE_THIRD = 1.0 / 3.0
TWO_THIRDS = 2.0 / 3.0


def _rms(x: torch.Tensor) -> torch.Tensor:
    return x.abs().pow(2).mean().sqrt()


def _call(func, t, y):
    """torchdiffeq wraps func so that t is cast to y.dtype before every call."""
    return func(torch.as_tensor(t).to(y.dtype), y)


# ----------------------------------------------------------------------------------------------------------------
# Fixed-grid RK4 (3/8 rule)
# ----------------------------------------------------------------------------------------------------------------
def rk4_38_step(func, t0, dt, t1, y0, f0=None):
    """One 3/8-rule step; returns (dy, f0).  Operation order as in torchdiffeq's ``rk4_alt_step_func``."""
    k1 = _call(func, t0, y0) if f0 is None else f0
    k2 = _call(func, t0 + dt * ONE_THIRD, y0 + dt * k1 * ONE_THIRD)
    k3 = _call(func, t0 + dt * TWO_THIRDS, y0 + dt * (k2 - k1 * ONE_THIRD))
    k4 = _call(func, t1, y0 + dt * (k1 - k2 + k3))
    return (k1 + 3 * (k2 + k3) + k4) * dt * 0.125, k1


def odeint_rk4(func, y0: torch.Tensor, t: torch.Tensor, step_size: Optional[float] = None) -> torch.Tensor:
    """Fixed grid solve.  Without ``step_size`` the grid is ``t`` itself."""
    if step_size is None:
        grid = t
    else:
        n = int(math.ceil(float((t[-1] - t[0]) / step_size + 1)))
        grid = torch.arange(0, n, dtype=t.dtype) * step_size + t[0]
        grid[-1] = t[-1] if grid[-1] > t[-1] else grid[-1]
        if grid[-1] != t[-1]:
            grid = torch.cat([grid, t[-1:]])
    sol = [y0]
    j = 1
    y = y0
    for i in range(len(grid) - 1):
        t0, t1 = grid[i], grid[i + 1]
        dt = t1 - t0
        dy, _ = rk4_38_step(func, t0, dt, t1, y)
        y1 = y + dy
        while j < len(t) and t1 >= t[j]:
            if t[j] == t0:
                sol.append(y)
            elif t[j] == t1:
                sol.append(y1)
            else:
                sol.append(y + (t[j] - t0) / (t1 - t0) * (y1 - y))
            j += 1
        y = y1
    return torch.stack(sol, dim=0)


# ----------------------------------------------------------------------------------------------------------------
# dopri5
# ----------------------------------------------------------------------------------------------------------------
def _initial_step(func, t0, y0, order, rtol, atol, f0):
    dtype = y0.dtype
    scale = atol + torch.abs(y0) * rtol
    d0 = _rms(y0 / scale).abs()
    d1 = _rms(f0 / scale).abs()
    if d0 < 1e-5 or d1 < 1e-5:
        h0 = torch.tensor(1e-6, dtype=dtype)
    else:
        h0 = 0.01 * d0 / d1
    h0 = h0.abs()
    y1 = y0 + h0 * f0
    f1 = _call(func, t0 + h0, y1)
    d2 = torch.abs(_rms((f1 - f0) / scale) / h0)
    if d1 <= 1e-15 and d2 <= 1e-15:
        h1 = torch.max(torch.tensor(1e-6, dtype=dtype), h0 * 1e-3)
    else:
        h1 = (0.01 / max(d1, d2)) ** (1.0 / float(order + 1))
    h1 = h1.abs()
    return torch.min(100 * h0, h1).to(t0.dtype)


def _dp_step(func, y0, f0, t0, dt, t1, alpha, beta, c_err):
    """Six stages; returns y1, f1, error estimate, k (..., 7)."""
    t0c = t0.to(y0.dtype)
    dtc = dt.to(y0.dtype)
    ks = [f0]
    yi = y0
    for i in range(6):
        ti = t1 if DP_ALPHA[i] == 1.0 else t0c + alpha[i] * dtc
        kmat = torch.stack(ks, dim=-1)
        yi = y0 + kmat.matmul(beta[i] * dtc).view_as(f0)
        ks.append(_call(func, ti, yi))
    k = torch.stack(ks, dim=-1)
    y1 = yi                                   # FSAL: c_sol == last beta row + [0]
    f1 = ks[-1]
    err = k.matmul(dtc * c_err)
    return y1, f1, err, k


def _dense_coeffs(y0, y1, k, dt, c_mid):
    dtc = dt.to(y0.dtype)
    y_mid = y0 + k.matmul(dtc * c_mid).view_as(y0)
    f0 = k[..., 0]
    f1 = k[..., -1]
    a = 2 * dtc * (f1 - f0) - 8 * (y1 + y0) + 16 * y_mid
    b = dtc * (5 * f0 - 3 * f1) + 18 * y0 + 14 * y1 - 32 * y_mid
    c = dtc * (f1 - 4 * f0) - 11 * y0 - 5 * y1 + 16 * y_mid
    d = dtc * f0
    e = y0
    return [e, d, c, b, a]


def _dense_poly(coeffs, x):
    """The dense-output quartic at abscissa x = (t - t0) / (t1 - t0)."""
    total = coeffs[0] + x * coeffs[1]
    xp = x
    for c in coeffs[2:]:
        xp = xp * x
        total = total + xp * c
    return total


def _dense_eval(coeffs, t0, t1, t):
    return _dense_poly(coeffs, ((t - t0) / (t1 - t0)).to(coeffs[0].dtype))


def _dp_tableau(dtype):
    cast = lambda v: torch.tensor(v, dtype=torch.float64).to(dtype)
    return cast(DP_ALPHA), [cast(b) for b in DP_BETA], cast(DP_C_ERR), cast(DP_C_MID)


def dopri5_step(func, y0: torch.Tensor, t0, dt, f0: Optional[torch.Tensor] = None):
    """One Dormand-Prince step of size dt from (t0, y0), state in y0's dtype, time in float64 -- the step odeint_dopri5
    takes.  f0 = func(t0, y0) unless given (FSAL).  Returns (y1, f1, err, coeffs): the solution, its slope, the embedded
    error estimate and the dense-output coefficients (evaluate with ``dense_output``).  Started from a recorded state it
    checks one step of a solver in isolation."""
    alpha, beta, c_err, c_mid = _dp_tableau(y0.dtype)
    t0 = torch.as_tensor(t0, dtype=torch.float64)
    dt = torch.as_tensor(dt, dtype=torch.float64)
    if f0 is None:
        f0 = _call(func, t0, y0)
    y1, f1, err, k = _dp_step(func, y0, f0, t0, dt, t0 + dt, alpha, beta, c_err)
    return y1, f1, err, _dense_coeffs(y0, y1, k, dt, c_mid)


def dense_output(coeffs, x) -> torch.Tensor:
    """The dense output of a step (coefficients from dopri5_step) at abscissa x in [0, 1]."""
    return _dense_poly(coeffs, torch.as_tensor(x, dtype=torch.float64).to(coeffs[0].dtype))


def dopri5_error_ratio(y0, y1, err, rtol: float, atol: float) -> torch.Tensor:
    """torchdiffeq's RMS error ratio of a step (accepted iff <= 1)."""
    return _rms(err / (atol + rtol * torch.max(y0.abs(), y1.abs()))).abs()


def dopri5_replay(func, y0: torch.Tensor, t0, dt, n_accept: int, out_step, out_x) -> torch.Tensor:
    """Differentiable replay of a recorded dopri5 solve of one trial group: accepted step n starts at t0[n] with size
    dt[n] (chained from y0 with the FSAL slope, as the solver chains them); output j >= 1 is the dense output of step
    out_step[j] at abscissa out_x[j], row 0 is y0.  The record fixes the discrete map, so autograd through the replay
    gives the exact gradient of the computation a discrete adjoint differentiates, free of step-controller noise.  The
    abscissae are taken as recorded (a float32 record is replayed at its float32 x)."""
    T = len(out_step)
    sol = [y0]
    y, f = y0, None
    j = 1
    for n in range(int(n_accept)):
        y1, f1, _, coeffs = dopri5_step(func, y, float(t0[n]), float(dt[n]), f)
        while j < T and int(out_step[j]) == n:
            sol.append(dense_output(coeffs, float(out_x[j])))
            j += 1
        y, f = y1, f1
    if j != T:
        raise ValueError(f"record places output {j} in no replayed step (out_step {int(out_step[j])}, n_accept {int(n_accept)})")
    return torch.stack(sol, dim=0)


def odeint_dopri5(func, y0: torch.Tensor, t: torch.Tensor, rtol: float = 1e-7, atol: float = 1e-9,
                  safety: float = 0.9, ifactor: float = 10.0, dfactor: float = 0.2,
                  max_num_steps: int = 2 ** 31 - 1, stats: Optional[Dict] = None,
                  record: Optional[Dict] = None) -> torch.Tensor:
    """Adaptive solve of ONE trial group (the error norm is taken over the whole tensor y).  ``record`` (a dict) receives
    the accepted steps in the layout of include/odecol.h's dopri5 record: ``t0`` / ``dt`` (float64, one entry per
    accepted step) and, for every output j >= 1, ``out_step[j]`` (the accepted step it lies in) and ``out_x[j]`` (its
    dense-output abscissa); entry 0 of both is 0.  ``dopri5_replay`` recomputes the solve from it."""
    dtype = y0.dtype
    alpha, beta, c_err, c_mid = _dp_tableau(dtype)

    t64 = t.to(torch.float64)
    f0 = _call(func, t64[0], y0)
    dt = _initial_step(func, t64[0], y0, 4, rtol, atol, f0)
    st_y, st_f, st_t0, st_t1, st_dt = y0, f0, t64[0], t64[0], dt
    coeffs = [y0] * 5
    n_acc = n_rej = 0
    sol = [y0]
    rec_t0, rec_dt, out_step, out_x = [], [], [0], [0.0]
    for i in range(1, len(t64)):
        next_t = t64[i]
        n_steps = 0
        while next_t > st_t1:
            assert n_steps < max_num_steps
            y_, f_, t0_, dt_ = st_y, st_f, st_t1, st_dt
            t1_ = t0_ + dt_
            assert t0_ + dt_ > t0_, "underflow in dt"
            assert torch.isfinite(y_).all(), "non-finite state"
            y1, f1, err, k = _dp_step(func, y_, f_, t0_, dt_, t1_, alpha, beta, c_err)
            tol = atol + rtol * torch.max(y_.abs(), y1.abs())
            ratio = _rms(err / tol).abs()
            accept = bool(ratio <= 1)
            if accept:
                coeffs = _dense_coeffs(y_, y1, k, dt_, c_mid)
                st_y, st_f, st_t0, st_t1 = y1, f1, t0_, t1_
                rec_t0.append(float(t0_))
                rec_dt.append(float(dt_))
                n_acc += 1
            else:
                st_t0 = t0_
                n_rej += 1
            with torch.no_grad():
                r64 = ratio.detach().to(torch.float64)
                if r64 == 0:
                    st_dt = dt_ * ifactor
                else:
                    df = 1.0 if r64 < 1 else dfactor
                    fac = min(ifactor, max(safety / float(r64) ** 0.2, df))
                    st_dt = dt_ * fac
            n_steps += 1
        sol.append(_dense_eval(coeffs, st_t0, st_t1, next_t))
        out_step.append(n_acc - 1)
        out_x.append(float((next_t - st_t0) / (st_t1 - st_t0)))
    if stats is not None:
        stats["n_accept"] = n_acc
        stats["n_reject"] = n_rej
    if record is not None:
        record.update(t0=rec_t0, dt=rec_dt, out_step=out_step, out_x=out_x)
    return torch.stack(sol, dim=0)


def odeint(func, y0, t, *, rtol=1e-7, atol=1e-9, method=None, options=None, stats=None):
    """torchdiffeq.odeint signature subset; default method dopri5 (what the reference scripts get)."""
    method = method or "dopri5"
    options = options or {}
    if method == "rk4":
        return odeint_rk4(func, y0, t, step_size=options.get("step_size"))
    if method == "dopri5":
        return odeint_dopri5(func, y0, t, rtol=rtol, atol=atol, stats=stats, **options)
    raise ValueError(f"oracle restates rk4 and dopri5 only, not {method!r}")


# ----------------------------------------------------------------------------------------------------------------
# torchsde integrate loop + Euler-Maruyama
# ----------------------------------------------------------------------------------------------------------------
class TabulatedBrownian:
    """Deterministic Brownian source for bit-parity tests: the k-th call returns row k of ``increments``
    (shape (steps, B, 1)); torchsde only needs ``__call__(t0, t1)`` and ``.shape``."""

    def __init__(self, increments: torch.Tensor):
        self.increments = increments
        self.shape = tuple(increments.shape[1:])
        self.k = 0

    def __call__(self, t0, t1):
        out = self.increments[self.k]
        self.k += 1
        return out


def _em_step(sde, bm, t0, t1, y0):
    dt = t1 - t0
    dW = bm(t0, t1)                                  # (B, 1)
    f = sde.forward(t0, y0)
    g = sde.diffusion(t0, y0)                        # (B, D, 1) scalar noise
    return y0 + f * dt + (g * dW.unsqueeze(-2)).sum(-1)


def adaptive_update(err: float, step: float, prev_ratio: Optional[float], safety=0.9, facmin=0.2, facmax=1.4):
    if err > 1:
        pfactor, ifactor = 0.0, 1 / 1.5
    else:
        pfactor, ifactor = 0.13, 1 / 4.5
    ratio = safety / err if err > 0 else math.inf       # torchsde divides tensors: a zero error gives an infinite ratio
    if prev_ratio is None:
        prev_ratio = ratio
    factor = ratio ** ifactor * (ratio / prev_ratio) ** pfactor
    if err <= 1:
        prev_ratio = ratio
        facmin = 1.0
    factor = min(facmax, max(facmin, factor))
    return step * factor, prev_ratio


def sdeint_euler(sde, y0: torch.Tensor, ts: torch.Tensor, bm, dt: float = 1e-3, adaptive: bool = False,
                 rtol: float = 1e-5, atol: float = 1e-4, dt_min: float = 1e-5, stats: Optional[Dict] = None,
                 trace: Optional[List] = None):
    """torchsde ``BaseSDESolver.integrate`` with the Euler step.  Times stay in ts.dtype (float32 in the
    reference).  ``bm`` is any callable (t0, t1) -> (B, 1) increment (see TabulatedBrownian).  For the adaptive
    controller bm must be a consistent path (W(a,c) = W(a,b) + W(b,c)), e.g. oracle.brownian.VirtualBrownianTree.
    ``trace`` (a list, adaptive mode) receives one tuple (t0, t1, err, accepted) per attempted step, so a caller can
    check which regime the controller ran in."""
    step = dt
    prev_t = curr_t = ts[0]
    prev_y = curr_y = y0
    ys = [y0]
    prev_ratio = None
    n_acc = n_rej = 0
    for out_t in ts[1:]:
        while curr_t < out_t:
            next_t = torch.minimum(curr_t + step, ts[-1])
            if adaptive:
                y_full = _em_step(sde, bm, curr_t, next_t, curr_y)
                mid_t = 0.5 * (curr_t + next_t)
                y_mid = _em_step(sde, bm, curr_t, mid_t, curr_y)
                y_half = _em_step(sde, bm, mid_t, next_t, y_mid)
                with torch.no_grad():
                    tol = atol + rtol * torch.max(y_full.abs(), y_half.abs())
                    err = float(_rms((y_full - y_half) / tol))
                    step, prev_ratio = adaptive_update(err, step, prev_ratio)
                if step < dt_min:
                    step = dt_min
                    prev_ratio = None
                accepted = err <= 1 or step <= dt_min
                if trace is not None:
                    trace.append((float(curr_t), float(next_t), err, accepted))
                if accepted:
                    prev_t, prev_y = curr_t, curr_y
                    curr_t, curr_y = next_t, y_half
                    n_acc += 1
                else:
                    n_rej += 1
            else:
                prev_t, prev_y = curr_t, curr_y
                curr_y = _em_step(sde, bm, curr_t, next_t, curr_y)
                curr_t = next_t
                n_acc += 1
        # torchsde interp.linear_interp: two-sided weights (exactly curr_y when out_t == curr_t)
        span = curr_t - prev_t
        ys.append((curr_t - out_t) / span * prev_y + (out_t - prev_t) / span * curr_y)
    if stats is not None:
        stats["n_accept"] = n_acc
        stats["n_reject"] = n_rej
    return torch.stack(ys, dim=0)


def em_step_schedule(ts: torch.Tensor, dt: float) -> List[Tuple[float, float]]:
    """The (t0, t1) pairs the fixed-step loop visits, in ts.dtype arithmetic (data-independent)."""
    out = []
    curr = ts[0]
    for out_t in ts[1:]:
        while curr < out_t:
            nxt = torch.minimum(curr + dt, ts[-1])
            out.append((float(curr), float(nxt)))
            curr = nxt
    return out


# ----------------------------------------------------------------------------------------------------------------
# torchsde method='srk' (diagonal / scalar noise): Roessler SRI2, tableau "SRID2" [memory: torchsde 0.2.x
# _core/methods/srk.py::diagonal_or_scalar_step and _core/methods/tableaus/srid2.py; Roessler 2010, table 5.3 SRI2W1]
# ----------------------------------------------------------------------------------------------------------------
SRID2_STAGES = 4
SRID2_C0 = (0, 1, 1 / 2, 0)
SRID2_C1 = (0, 1 / 4, 1, 1 / 4)
SRID2_A0 = ((), (1,), (1 / 4, 1 / 4), (0, 0, 0))
SRID2_A1 = ((), (1 / 4,), (1, 0), (0, 0, 1 / 4))
SRID2_B0 = ((), (0,), (1, 1 / 2), (0, 0, 0))
SRID2_B1 = ((), (-1 / 2,), (1, 0), (2, -1, 1 / 2))
SRID2_ALPHA = (1 / 6, 1 / 6, 2 / 3, 0)
SRID2_BETA1 = (-1, 4 / 3, 2 / 3, 0)
SRID2_BETA2 = (1, -4 / 3, 1 / 3, 0)
SRID2_BETA3 = (2, -4 / 3, -2 / 3, 0)
SRID2_BETA4 = (-2, 5 / 3, -2 / 3, 1)


class TabulatedBrownianU(TabulatedBrownian):
    """Deterministic (W, U) source: call k returns rows k of ``increments`` and ``levy_u`` (both (steps, B, 1));
    U is torchsde's space-time Levy area of the step, U = int_{t0}^{t1} (W_r - W_{t0}) dr, U | W ~ N(h W / 2, h^3 / 12)."""

    def __init__(self, increments: torch.Tensor, levy_u: torch.Tensor):
        super().__init__(increments)
        self.levy_u = levy_u

    def __call__(self, t0, t1, return_U=False):
        k = self.k
        w = super().__call__(t0, t1)
        return (w, self.levy_u[k]) if return_U else w


def sample_w_u(n_steps: int, B: int, h: float, generator: torch.Generator):
    """Joint draw of (W, U) for steps of size h: W = sqrt(h) z1, U = h W / 2 + sqrt(h^3 / 12) z2."""
    z = torch.randn(2, n_steps, B, 1, generator=generator)
    w = math.sqrt(h) * z[0]
    return w, 0.5 * h * w + math.sqrt(h ** 3 / 12.0) * z[1]


def _srk_step(sde, bm, t0, t1, y0):
    dt = t1 - t0
    rdt = 1 / dt
    sqrt_dt = torch.sqrt(dt) if torch.is_tensor(dt) else math.sqrt(dt)
    I_k, I_k0 = bm(t0, t1, return_U=True)            # (B, 1) each: broadcast over the state for scalar noise
    I_kk = (I_k ** 2 - dt) / 2
    I_kkk = (I_k ** 3 - 3 * dt * I_k) / 6
    y1 = y0
    H0, H1 = [], []
    for s in range(SRID2_STAGES):
        H0s, H1s = y0, y0
        for j in range(s):
            f = sde.forward(t0 + SRID2_C0[j] * dt, H0[j])
            g = sde.diffusion(t0 + SRID2_C1[j] * dt, H1[j])
            g = g.squeeze(2) if g.dim() == 3 else g
            H0s = H0s + SRID2_A0[s][j] * f * dt + SRID2_B0[s][j] * g * I_k0 * rdt
            H1s = H1s + SRID2_A1[s][j] * f * dt + SRID2_B1[s][j] * g * sqrt_dt
        H0.append(H0s)
        H1.append(H1s)
        f = sde.forward(t0 + SRID2_C0[s] * dt, H0s)
        g_weight = (SRID2_BETA1[s] * I_k + SRID2_BETA2[s] * I_kk / sqrt_dt + SRID2_BETA3[s] * I_k0 * rdt
                    + SRID2_BETA4[s] * I_kkk * rdt)
        g = sde.diffusion(t0 + SRID2_C1[s] * dt, H1s)
        g = g.squeeze(2) if g.dim() == 3 else g
        y1 = y1 + SRID2_ALPHA[s] * f * dt + g * g_weight            # g_prod for diagonal / scalar noise
    return y1


def sdeint_srk(sde, y0: torch.Tensor, ts: torch.Tensor, bm, dt: float = 1e-3, adaptive: bool = False, rtol: float = 1e-5,
               atol: float = 1e-4, dt_min: float = 1e-5, stats: Optional[Dict] = None):
    """torchsde ``sdeint(..., method='srk')``: the integrate loop of sdeint_euler with the SRI2 step, fixed step or
    step-doubling adaptive (``adaptive=True``: what /root/reference/scripts/parity_ode.py:234 names).
    ``bm(t0, t1, return_U=True)`` -> (W, U), each (B, 1) (see TabulatedBrownianU); the adaptive controller needs a source
    whose (W, U) are consistent on sub-intervals (a Brownian interval / tree, not a table)."""
    step = dt
    prev_t = curr_t = ts[0]
    prev_y = curr_y = y0
    ys = [y0]
    prev_ratio = None
    n_acc = n_rej = 0
    for out_t in ts[1:]:
        while curr_t < out_t:
            next_t = torch.minimum(curr_t + step, ts[-1])
            if adaptive:
                y_full = _srk_step(sde, bm, curr_t, next_t, curr_y)
                mid_t = 0.5 * (curr_t + next_t)
                y_mid = _srk_step(sde, bm, curr_t, mid_t, curr_y)
                y_half = _srk_step(sde, bm, mid_t, next_t, y_mid)
                with torch.no_grad():
                    tol = atol + rtol * torch.max(y_full.abs(), y_half.abs())
                    err = float(_rms((y_full - y_half) / tol))
                    step, prev_ratio = adaptive_update(err, step, prev_ratio)
                if step < dt_min:
                    step = dt_min
                    prev_ratio = None
                if err <= 1 or step <= dt_min:
                    prev_t, prev_y = curr_t, curr_y
                    curr_t, curr_y = next_t, y_half
                    n_acc += 1
                else:
                    n_rej += 1
            else:
                prev_t, prev_y = curr_t, curr_y
                curr_y = _srk_step(sde, bm, curr_t, next_t, curr_y)
                curr_t = next_t
                n_acc += 1
        span = curr_t - prev_t
        ys.append((curr_t - out_t) / span * prev_y + (out_t - prev_t) / span * curr_y)
    if stats is not None:
        stats["n_accept"] = n_acc
        stats["n_reject"] = n_rej
    return torch.stack(ys, dim=0)
