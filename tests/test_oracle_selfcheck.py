"""Self-checks that anchor the restated third-party solvers (oracle/solvers.py).  torchdiffeq / torchsde are not
installable offline, so these stand in for their own test-suites: tableau order conditions, empirical convergence
order, analytic solutions, controller behaviour."""
import math

import numpy as np
import pytest
import torch

from oracle import solvers as S


def test_dopri5_tableau_order_conditions():
    b = np.array(S.DP_C_SOL)
    c = np.array([0.0] + S.DP_ALPHA)
    A = np.zeros((7, 7))
    for i, row in enumerate(S.DP_BETA):
        A[i + 1, :len(row)] = row
    assert abs(b.sum() - 1) < 1e-15
    assert np.allclose(A.sum(1), c, atol=1e-15)                 # row sums
    assert abs(b @ c - 1 / 2) < 1e-15
    assert abs(b @ c ** 2 - 1 / 3) < 1e-15
    assert abs(b @ (A @ c) - 1 / 6) < 1e-15
    assert abs(b @ c ** 3 - 1 / 4) < 1e-15
    assert abs(b @ c ** 4 - 1 / 5) < 1e-14
    e = np.array(S.DP_C_ERR)
    assert abs(e.sum()) < 1e-15                                 # the survey's 50085-vs-50001 typo fails this
    assert abs(e @ c) < 1e-15 and abs(e @ c ** 2) < 1e-15 and abs(e @ c ** 3) < 1e-15
    assert np.allclose(S.DP_BETA[-1] + [0.0], S.DP_C_SOL)       # FSAL
    m = np.array(S.DP_C_MID)
    assert abs(m.sum() - 0.5) < 1e-12                           # y_mid is the solution at t0 + h/2


def _lin(lmbda):
    return lambda t, y: lmbda * y


def test_rk4_38_is_fourth_order():
    y0 = torch.ones(1, 1, dtype=torch.float64)
    errs = []
    for n in (20, 40, 80):
        t = torch.linspace(0, 1, n + 1, dtype=torch.float64)
        y = S.odeint_rk4(_lin(-2.0), y0, t)
        errs.append(abs(float(y[-1]) - math.exp(-2.0)))
    orders = [math.log2(errs[i] / errs[i + 1]) for i in range(2)]
    assert all(3.8 < o < 4.3 for o in orders), orders


def test_rk4_outputs_by_linear_interpolation_between_grid_points():
    y0 = torch.ones(1, 1, dtype=torch.float64)
    t = torch.tensor([0.0, 0.25, 1.0], dtype=torch.float64)
    coarse = S.odeint_rk4(_lin(-1.0), y0, t, step_size=0.5)
    grid = S.odeint_rk4(_lin(-1.0), y0, torch.tensor([0.0, 0.5, 1.0], dtype=torch.float64))
    assert torch.allclose(coarse[1], 0.5 * (grid[0] + grid[1]))
    assert torch.allclose(coarse[2], grid[2])


def test_dopri5_meets_tolerance_and_dense_output_is_accurate():
    y0 = torch.tensor([[1.0, 0.0]], dtype=torch.float64)

    def osc(t, y):
        return torch.stack((y[..., 1], -y[..., 0]), dim=-1)

    t = torch.linspace(0, 6.0, 61, dtype=torch.float64)
    st = {}
    y = S.odeint_dopri5(osc, y0, t, rtol=1e-8, atol=1e-10, stats=st)
    exact = torch.stack((torch.cos(t), -torch.sin(t)), dim=-1)
    assert float((y[:, 0] - exact).abs().max()) < 2e-7
    assert st["n_accept"] < 200 and st["n_reject"] < st["n_accept"]


def test_dopri5_step_count_scales_with_tolerance():
    y0 = torch.ones(1, 1, dtype=torch.float64)
    t = torch.tensor([0.0, 5.0], dtype=torch.float64)
    counts = []
    for tol in (1e-4, 1e-6, 1e-8):
        st = {}
        S.odeint_dopri5(_lin(-1.0), y0, t, rtol=tol, atol=tol * 1e-2, stats=st)
        counts.append(st["n_accept"])
    assert counts[0] < counts[1] < counts[2]
    # a 5th-order controller: 100x tighter tolerance -> about 100^(1/5) = 2.5x the steps
    assert 1.5 < counts[2] / counts[1] < 4.0


class _OU:
    noise_type, sde_type = "scalar", "ito"

    def __init__(self, theta, sigma):
        self.theta, self.sigma = theta, sigma

    def forward(self, t, y):
        return -self.theta * y

    def diffusion(self, t, y):
        return torch.full_like(y, self.sigma).unsqueeze(-1)


def test_em_schedule_and_exact_recursion():
    ts = torch.linspace(0, 0.1, 11)
    sched = S.em_step_schedule(ts, 0.01)
    assert len(sched) in (10, 11) and abs(sched[-1][1] - 0.1) < 1e-7
    g = torch.Generator().manual_seed(0)
    dW = torch.randn(len(sched), 3, 1, generator=g) * 0.1
    sde = _OU(2.0, 0.5)
    y0 = torch.ones(3, 1)
    ys = S.sdeint_euler(sde, y0, ts, S.TabulatedBrownian(dW), dt=0.01)
    y = y0.clone()
    for k, (a, b) in enumerate(sched):                          # hand recursion
        y = y + (-2.0 * y) * (b - a) + 0.5 * dW[k]
    assert torch.allclose(ys[-1], y, atol=1e-6)


def test_em_ou_moments():
    torch.manual_seed(0)
    theta, sigma, T = 1.5, 0.8, 1.0
    ts = torch.linspace(0, T, 11)
    sched = S.em_step_schedule(ts, 0.005)
    B = 4000
    dW = torch.randn(len(sched), B, 1) * math.sqrt(0.005)
    ys = S.sdeint_euler(_OU(theta, sigma), torch.ones(B, 1), ts, S.TabulatedBrownian(dW), dt=0.005)
    mean, var = float(ys[-1].mean()), float(ys[-1].var())
    assert abs(mean - math.exp(-theta * T)) < 0.03
    assert abs(var - sigma ** 2 / (2 * theta) * (1 - math.exp(-2 * theta * T))) < 0.02


def test_adaptive_controller_limits():
    # error above 1 shrinks the step by at most 5x, error below 1 never shrinks and grows by at most 1.4x
    s, _ = S.adaptive_update(1e6, 1.0, None)
    assert abs(s - 0.2) < 1e-12
    s, r = S.adaptive_update(1e-9, 1.0, None)
    assert abs(s - 1.4) < 1e-12 and r == 0.9 / 1e-9
    s, _ = S.adaptive_update(0.95, 1.0, None)
    assert s == 1.0


class _PiecewiseLinearPath:
    """A consistent Brownian path for the adaptive loop: W linear between the points of a fine random walk."""
    shape = (1, 1)

    def __init__(self, span, n, seed):
        g = torch.Generator().manual_seed(seed)
        self.t = torch.linspace(0.0, span, n + 1, dtype=torch.float64)
        self.w = torch.cat((torch.zeros(1), torch.randn(n, generator=g).double().cumsum(0) * math.sqrt(span / n)))

    def _at(self, t):
        return float(np.interp(float(t), self.t.numpy(), self.w.numpy()))

    def __call__(self, t0, t1):
        return torch.tensor([[self._at(t1) - self._at(t0)]], dtype=torch.float32)


@pytest.mark.parametrize("rtol,atol", [(1e-3, 1e-3), (1e-12, 1e-12)], ids=["controlled", "at_dt_min"])
def test_adaptive_euler_trace_records_the_attempts_and_changes_no_result(rtol, atol):
    ts = torch.linspace(0.0, 0.5, 6)
    y0 = torch.tensor([[1.0], [-0.5]])
    bm = _PiecewiseLinearPath(0.5, 4096, seed=3)
    kw = dict(dt=0.05, adaptive=True, rtol=rtol, atol=atol, dt_min=5e-3)
    st_a, st_b, trace = {}, {}, []
    ya = S.sdeint_euler(_OU(2.0, 0.7), y0, ts, bm, stats=st_a, **kw)
    yb = S.sdeint_euler(_OU(2.0, 0.7), y0, ts, bm, stats=st_b, trace=trace, **kw)
    assert torch.equal(ya, yb) and st_a == st_b
    assert len(trace) == st_a["n_accept"] + st_a["n_reject"] and sum(a for *_, a in trace) == st_a["n_accept"]
    assert st_a["n_reject"] > 0
    # accepted attempts tile [ts[0], ts[-1]]; a rejected one restarts from the same t0
    t_cur = float(ts[0])
    for t0, t1, err, accepted in trace:
        assert t0 == t_cur and t1 > t0 and err >= 0
        assert accepted or err > 1
        if accepted:
            t_cur = t1
    assert t_cur == float(ts[-1])


# ---------------------------------------------------------------------------------------------------------------
# torchsde method='srk' (SRI2 / "SRID2" tableau) restatement
# ---------------------------------------------------------------------------------------------------------------
def test_srid2_tableau_order_conditions():
    # Roessler 2010, conditions for strong order 1.5 (m = 1): the ones that pin the tableau's rows
    al, b1, b2, b3, b4 = (np.array(x, dtype=float) for x in (S.SRID2_ALPHA, S.SRID2_BETA1, S.SRID2_BETA2, S.SRID2_BETA3, S.SRID2_BETA4))
    full = lambda rows: np.array([list(r) + [0.0] * (4 - len(r)) for r in rows])
    A0, A1, B0, B1 = (full(x) for x in (S.SRID2_A0, S.SRID2_A1, S.SRID2_B0, S.SRID2_B1))
    e = np.ones(4)
    assert abs(al.sum() - 1) < 1e-15 and abs(b1.sum() - 1) < 1e-15
    assert abs(b2.sum()) < 1e-15 and abs(b3.sum()) < 1e-15 and abs(b4.sum()) < 1e-15
    assert np.allclose(A0 @ e, S.SRID2_C0) and np.allclose(A1 @ e, S.SRID2_C1)
    assert abs(al @ (A0 @ e) - 0.5) < 1e-15                 # deterministic order 2
    assert abs(al @ (B0 @ e) - 1.0) < 1e-15                 # drift sees the space-time integral once
    assert abs(al @ (B0 @ e) ** 2 - 1.5) < 1e-15
    assert abs(b1 @ (B1 @ e)) < 1e-15 and abs(b2 @ (B1 @ e) - 1.0) < 1e-15
    assert abs(b3 @ (B1 @ e)) < 1e-15 and abs(b4 @ (B1 @ e)) < 1e-15
    assert abs(b1 @ (A1 @ e) - 1.0) < 1e-15 and abs(b3 @ (A1 @ e) + 1.0) < 1e-15
    assert abs(b2 @ (A1 @ e)) < 1e-15 and abs(b4 @ (A1 @ e)) < 1e-15      # NB not the full set; the empirical
    # strong-order test below is the anchor


class _Logistic:
    """dy = y (1 - y) dt + sigma dW (additive), a nonlinear drift for convergence-order checks."""
    noise_type, sde_type = "scalar", "ito"

    def __init__(self, sigma):
        self.sigma = sigma

    def forward(self, t, y):
        return y * (1 - y)

    def diffusion(self, t, y):
        return torch.full_like(y, self.sigma).unsqueeze(-1)


def test_srk_without_noise_is_third_order():
    errs = []
    for n in (10, 20, 40):
        ts = torch.linspace(0, 2, 2, dtype=torch.float64)
        z = torch.zeros(n + 2, 1, 1, dtype=torch.float64)
        y = S.sdeint_srk(_Logistic(0.0), torch.full((1, 1), 0.1, dtype=torch.float64), ts, S.TabulatedBrownianU(z, z), dt=2.0 / n)
        exact = 0.1 * math.exp(2) / (1 + 0.1 * (math.exp(2) - 1))
        errs.append(abs(float(y[-1]) - exact))
    assert 6.5 < errs[0] / errs[1] < 9.5 and 6.5 < errs[1] / errs[2] < 9.5, errs


def _coarsen(w, u, delta, factor):
    """(W, U) of steps of size delta -> steps of size factor * delta on the same Brownian path."""
    n = w.shape[0] // factor
    w = w[:n * factor].reshape(n, factor, *w.shape[1:])
    u = u[:n * factor].reshape(n, factor, *u.shape[1:])
    before = torch.cumsum(w, dim=1) - w                      # W(t_i) - W(t_0) at the start of each fine step
    return w.sum(1), (u + delta * before).sum(1)


def test_srk_strong_order_on_a_shared_brownian_path():
    g = torch.Generator().manual_seed(3)
    n_fine, B, T = 256, 2000, 1.0
    delta = T / n_fine
    w, u = S.sample_w_u(n_fine, B, delta, g)
    w, u = w.double(), u.double()
    ts = torch.tensor([0.0, T], dtype=torch.float64)
    y0 = torch.full((B, 1), 0.3, dtype=torch.float64)
    sde = _Logistic(0.4)
    ref = S.sdeint_srk(sde, y0, ts, S.TabulatedBrownianU(w, u), dt=delta)[-1]
    errs, errs_em = [], []
    for factor in (16, 32):
        wc, uc = _coarsen(w, u, delta, factor)
        y = S.sdeint_srk(sde, y0, ts, S.TabulatedBrownianU(wc, uc), dt=delta * factor)[-1]
        errs.append(float((y - ref).abs().mean()))
        ye = S.sdeint_euler(sde, y0, ts, S.TabulatedBrownian(wc), dt=delta * factor)[-1]
        errs_em.append(float((ye - ref).abs().mean()))
    ratio, ratio_em = errs[1] / errs[0], errs_em[1] / errs_em[0]
    # strong order 1.5 -> 2^1.5 = 2.83 per halving; Euler-Maruyama (additive noise, order 1) -> 2
    assert 2.45 < ratio < 3.3, (errs, ratio)
    assert 1.7 < ratio_em < 2.3 and errs[0] < 0.2 * errs_em[0], (errs_em, errs)


# ---------------------------------------------------------------------------------------------------------------
# independent third-party anchor that IS installed: scipy's Dormand-Prince (scipy.integrate.RK45)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rtol,atol", [(1e-7, 1e-9), (1e-4, 1e-6)], ids=["reference_defaults", "loose"])
def test_dopri5_replay_of_the_record_reproduces_the_solve_and_its_gradients(rtol, atol):
    """The record of odeint_dopri5 (accepted t0 / dt, output step and abscissa) fixes the discrete map: replaying it in
    float64 gives the solver's outputs and autograd's gradients (y0, W, U, bias) through its adaptive solve."""
    from oracle import rhs as orhs
    from oracle.column_model import LinearForm
    rng = np.random.default_rng(5)
    N, n_in, T = 8, 3, 25
    lf = LinearForm(W=rng.standard_normal((N, N)) * 0.04, U=rng.standard_normal((N, n_in)) * 0.02, bias=rng.random(N) * 0.3,
                    kappa=rng.random(N) * 1.5, sigma=np.zeros(3 * N), tau_s=5e-4, tau_m=0.02, tau_a=10.0, resistance=80.0)
    kt = np.array([-1e-4, 6e-4, 1.1e-3, 2e-3])
    ku = rng.random((1, 4, n_in)) * 20
    t = torch.linspace(0, 2.4e-3, T, dtype=torch.float64)
    y0 = torch.tensor(np.concatenate((rng.random(N) * 8 - 10, rng.random(N), rng.random(N) * 3))[None])
    wgt = torch.tensor(rng.standard_normal((T, 1, 3 * N)))
    runs = []
    for replay in (False, True):
        ode = orhs.UnifiedColumnODE(lf, kt, ku, dtype=torch.float64, requires_grad=True)
        y0g = y0.clone().requires_grad_(True)
        if replay:
            y = S.dopri5_replay(ode, y0g, rec["t0"], rec["dt"], st["n_accept"], rec["out_step"], rec["out_x"])
        else:
            rec, st = {}, {}
            y = S.odeint_dopri5(ode, y0g, t, rtol=rtol, atol=atol, stats=st, record=rec)
        (y * wgt).sum().backward()
        runs.append([y.detach(), y0g.grad, ode.W.grad, ode.U.grad, ode.bias.grad])
    n = st["n_accept"]
    assert len(rec["t0"]) == len(rec["dt"]) == n and len(rec["out_step"]) == len(rec["out_x"]) == T
    assert all(rec["t0"][i + 1] == rec["t0"][i] + rec["dt"][i] for i in range(n - 1))
    steps = np.array(rec["out_step"][1:])
    assert np.all(np.diff(steps) >= 0) and steps[-1] == n - 1 and all(0 < x <= 1 for x in rec["out_x"][1:])
    errs = [float((a - b).abs().max() / b.abs().max()) for a, b in zip(runs[1], runs[0])]
    print(f"\n[oracle dopri5 replay rtol {rtol:g}] {n} accepted steps; trajectory / dy0 / dW / dU / dbias {errs}")
    assert max(errs) < 1e-13
    if rtol == 1e-7:
        assert np.any(np.diff(steps) > 1)                      # steps with no output inside
    else:
        assert np.any(np.diff(steps) == 0)                     # several outputs inside one step


def test_dopri5_tableau_equals_scipy_rk45():
    from scipy.integrate._ivp.rk import RK45
    A = np.asarray(RK45.A)                       # (6, 5): stage rows 0..5 (row 0 empty)
    for i, row in enumerate(S.DP_BETA[:5]):      # our rows 0..4 are scipy's rows 1..5
        assert np.allclose(A[i + 1, :len(row)], row, rtol=0, atol=1e-16), i
    assert np.allclose(RK45.C[1:], S.DP_ALPHA[:5], rtol=0, atol=1e-16)
    assert np.allclose(RK45.B, S.DP_C_SOL[:6], rtol=0, atol=1e-16)       # 5th-order weights = the FSAL row
    assert np.allclose(S.DP_BETA[5], S.DP_C_SOL[:6], rtol=0, atol=1e-16)
    # scipy's E uses the classic 4th-order weights (5179/57600, ...), torchdiffeq's c_error Shampine's (1951/21600, ...):
    # both embedded estimators point along the same direction, torchdiffeq's is exactly -2/3 of scipy's
    assert np.allclose(np.asarray(RK45.E), -1.5 * np.asarray(S.DP_C_ERR), rtol=0, atol=1e-15)


def test_dopri5_and_rk4_agree_with_scipy_on_the_column_model(cfg, golden):
    # the reference-generated golden rk4 trajectory (WTA, dt = 1e-4) against scipy's adaptive RK45 / DOP853 at tight
    # tolerance in float64 on the oracle's right-hand side: the restated fixed-step solver integrates the same ODE
    from scipy.integrate import solve_ivp
    from helpers import oracle_form, stim_table
    from oracle import rhs as orhs
    g = golden["wta"]
    lf = oracle_form("wta", cfg, g)
    tv = g["time_vec"].astype(np.float64)
    ode = orhs.UnifiedColumnODE(lf, tv, stim_table("wta", g["stim"]), dtype=torch.float64)
    T = 900                                       # through the stimulus onset (knot at T/3) and well into the response

    def f(t, y):
        with torch.no_grad():
            return ode.forward(torch.tensor(t, dtype=torch.float64), torch.tensor(y)[None])[0].numpy()

    sol = solve_ivp(f, (tv[0], tv[T]), np.zeros(48), method="DOP853", rtol=1e-10, atol=1e-12, t_eval=tv[[300, 600, T]],
                    max_step=float(tv[1] - tv[0]) * 4)
    assert sol.success
    ref = g["rk4_traj"][[300, 600, T], 0].astype(np.float64)
    err = np.abs(sol.y.T - ref).max() / np.abs(ref).max()
    assert err < 5e-5, err                        # fp32 rk4 at dt = 1e-4 vs converged float64 solution


def test_levy_area_bridge_matches_the_conditional_law():
    """The midpoint bisection of the Levy-area-consistent Brownian tree (csrc/odecol_common.cuh): conditional on (W, H) of an
    interval of length h, the half-interval variables (W1, H1, W2, H2) must have mean (W/2 + 3H/2, H/4, W/2 - 3H/2, H/4) and
    the covariance generated by Z ~ N(0, h/16), N ~ N(0, h/12) through W1 = .. + Z, H1 = .. - Z/2 + N/2, W2 = .. - Z,
    H2 = .. - Z/2 - N/2.  Checked against Gaussian conditioning of the four underlying variables (W1, U1, W2, U2)."""
    import numpy as np
    for h in (1.0, 0.037):
        g = h / 2
        C1 = np.array([[g, g * g / 2], [g * g / 2, g ** 3 / 3]])                 # cov of (W, U = int W) on a half
        C = np.zeros((4, 4)); C[:2, :2] = C1; C[2:, 2:] = C1
        A = np.array([[1, 0, 1, 0], [g, 1, 0, 1]])                               # W = W1 + W2;  U = U1 + U2 + g W1
        A_WH = np.array([A[0], A[1] / h - A[0] / 2])                             # H = U / h - W / 2
        Sg = A_WH @ C @ A_WH.T
        assert np.allclose(Sg, np.diag([h, h / 12]))                             # H ~ N(0, h / 12), independent of W
        K = C @ A_WH.T @ np.linalg.inv(Sg)
        Cc = C - K @ A_WH @ C
        Tm = np.array([[1, 0, 0, 0], [-0.5, 1 / g, 0, 0], [0, 0, 1, 0], [0, 0, -0.5, 1 / g]])     # (W1, H1, W2, H2)
        assert np.allclose(Tm @ K, [[0.5, 1.5], [0, 0.25], [0.5, -1.5], [0, 0.25]])
        Bm = np.array([[1, 0], [-0.5, 0.5], [-1, 0], [-0.5, -0.5]])
        assert np.allclose(Tm @ Cc @ Tm.T, Bm @ np.diag([h / 16, h / 12]) @ Bm.T)
