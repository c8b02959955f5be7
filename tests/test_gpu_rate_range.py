"""The transfer function φ(x) = x_nom / (1 - exp(z)) (x = V - A, x_nom = 48 x - 981, z = 80 tanh(-0.0089 x_nom / 80)) and its
derivative across the whole firing-rate range, through every code site that evaluates them, against float64.

The other kernel-versus-oracle tests run in φ's exponential tail, where it is tiny and nearly linear.  Here:

  * a probe reads φ and φ′ off one step of every solver, forward and reverse, with the state frozen (τ_m = τ_a = 1e6,
    W_aug = 0) so that every stage evaluates φ at x₀ = V₀: over x ∈ [-80, 200] (both clamps of the fast tanh), densely
    over the knee, and in the band around the removable pole at x = 981/48 where 1 - exp(z) cancels;
  * solver tests start from states spread over φ's steep range with strong coupling, and assert that the float64
    oracle trajectory really visits the clamp, the knee and the range beyond the pole.

The float64 truth of the probe is `phi_dphi_exact`: the same function written as R(u) B(v) / d, a product of two smooth
factors (u / tanh u and v / (1 - exp(-v))) with series where their quotients would cancel, so that it holds at and
around the pole where the oracle's own formula returns NaN or loses digits."""
import math
import os

import numpy as np
import pytest
import torch

import odecol
from helpers import check_dopri5_against_replay, ext_problem, sheet_oracle_form, to_device
from oracle import rhs as orhs, solvers as S
from oracle.column_model import LinearForm

DEV = "cuda"
D = 0.0089
POLE = 981.0 / 48.0                     # exactly representable: 20.4375
CLAMP_LO, CLAMP_HI = -54.4, 95.3        # tanh_small clamps its argument beyond these (|x_nom| > 3595)
RATE_FLOOR = 1e-6                       # Hz: below it the bars are absolute (1e-9 Hz)
_ORACLE_PHI = orhs.phi


# ----------------------------------------------------------------------------------------------------------------------
# float64 truth
# ----------------------------------------------------------------------------------------------------------------------
def phi_dphi_exact(x):
    """φ(x) and φ′(x) in float64 without cancellation: φ = R(u) B(v) / d with u = d x_nom / 80, v = 80 tanh u = -z,
    R(u) = u / tanh u and B(v) = v / (1 - exp(-v)); both factors by their series near zero.  Finite at the pole
    (φ = 1/d = 112.36 Hz, φ′ = 24)."""
    x = torch.as_tensor(x, dtype=torch.float64)
    xn = 48.0 * x - 981.0
    u = D * xn / 80.0
    t = torch.tanh(u)
    v = 80.0 * t
    su = u.abs() < 1e-3
    u2 = u * u
    R = torch.where(su, 1 + u2 / 3 - u2 * u2 / 45, u / t)
    dR = torch.where(su, 2 * u / 3 - 4 * u * u2 / 45, (t - u * (1 - t * t)) / (t * t))
    sv = v.abs() < 1e-2
    q = -torch.expm1(-v)
    v2 = v * v
    B = torch.where(sv, 1 + v / 2 + v2 / 12 - v2 * v2 / 720 + v2 * v2 * v2 / 30240, v / q)
    dB = torch.where(sv, 0.5 + v / 6 - v * v2 / 180 + v * v2 * v2 / 5040, (q - v * torch.exp(-v)) / (q * q))
    r = R * B / D
    dr = 48.0 * (dR * B / 80.0 + R * dB * (1 - t * t))
    return r, dr


class _PhiExact(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        r, dr = phi_dphi_exact(x)
        ctx.save_for_backward(dr)
        return r

    @staticmethod
    def backward(ctx, g):
        (dr,) = ctx.saved_tensors
        return g * dr


class _PhiScaledSlope(torch.autograd.Function):
    """oracle.rhs.phi with its derivative multiplied by `scale` (what a reverse kernel with a slightly wrong φ′ computes)."""
    @staticmethod
    def forward(ctx, x, scale):
        with torch.enable_grad():
            xd = x.detach().requires_grad_(True)
            r = _ORACLE_PHI(xd)
            (dr,) = torch.autograd.grad(r.sum(), xd)
        ctx.save_for_backward(dr)
        ctx.scale = scale
        return r.detach()

    @staticmethod
    def backward(ctx, g):
        (dr,) = ctx.saved_tensors
        return g * dr * ctx.scale, None


def test_exact_phi_matches_the_oracle_formula_and_high_precision_at_the_pole():
    """The probe's truth: equal to the oracle's float64 φ and autograd φ′ where that formula is well conditioned, and to
    50-digit arithmetic in the pole band and at the pole itself."""
    import mpmath as mp
    x = torch.cat((torch.linspace(-80, 200, 2001, dtype=torch.float64), torch.linspace(0, 19, 500, dtype=torch.float64)))
    x = x[(x - POLE).abs() > 0.5]
    r, dr = phi_dphi_exact(x)
    xr = x.clone().requires_grad_(True)
    ro = _ORACLE_PHI(xr)
    (dro,) = torch.autograd.grad(ro.sum(), xr)
    assert float(((r - ro.detach()).abs() / ro.detach()).max()) < 1e-12
    assert float(((dr - dro).abs() / dro).max()) < 1e-10

    mp.mp.dps = 50
    def phi_mp(xx):
        xn = 48 * xx - 981
        if xn == 0:
            return 1 / mp.mpf("0.0089")
        z = 80 * mp.tanh(-mp.mpf("0.0089") * xn / 80)
        return xn / (1 - mp.exp(z))
    pts = [POLE] + [POLE + s * k * 2.0 ** -19 for k in (1, 2, 7, 64) for s in (1, -1)] + \
          [POLE + s * 10.0 ** e for e in (-6, -4, -3, -2, -1, 0) for s in (1, -1)] + [-80.0, -30.0, 5.0, 19.0, 60.0, 200.0]
    r, dr = phi_dphi_exact(torch.tensor(pts, dtype=torch.float64))
    for i, p in enumerate(pts):
        xm = mp.mpf(p)
        rm = phi_mp(xm)
        drm = mp.diff(phi_mp, xm) if p != POLE else mp.mpf(24)
        assert abs(float(r[i]) / float(rm) - 1) < 1e-13, (p, float(r[i]), float(rm))
        assert abs(float(dr[i]) / float(drm) - 1) < 1e-9, (p, float(dr[i]), float(drm))


# ----------------------------------------------------------------------------------------------------------------------
# 1. the probe
# ----------------------------------------------------------------------------------------------------------------------
PN, PB = 16, 4096                       # 4096 trials x 16 populations: the batch that selects tiny_tc / k_rk4_bwd_small<40, true>
H = 1e-4


def _probe_points():
    """65,536 float32 abscissae: the pole band (pole +- k ulp, k = 1..64, and +- 1e-6 .. 1e-1 log-spaced), the knee (0..20)
    and a grid over [-80, 200] that reaches both clamps of the fast tanh."""
    p32 = np.float32(POLE)
    ulp = np.spacing(p32)
    k = np.arange(1, 65, dtype=np.float32)
    band = np.concatenate((p32 + k * ulp, p32 - k * ulp))
    off = np.logspace(-6, -1, 1200)
    band = np.concatenate((band, (POLE + off).astype(np.float32), (POLE - off).astype(np.float32)))
    band = band[band != p32]
    knee = np.linspace(0.0, 20.0, 16384, dtype=np.float32)
    rest = PB * PN - len(band) - len(knee)
    grid = np.linspace(-80.0, 200.0, rest, dtype=np.float32)
    x = np.concatenate((band, knee, grid)).astype(np.float32)
    assert len(x) == PB * PN
    np.random.default_rng(0).shuffle(x)             # every band in every trial tile and lane
    return x.reshape(PB, PN)


def _bands(x):
    x = np.asarray(x, dtype=np.float64)
    return {"clamp": (x < CLAMP_LO) | (x > CLAMP_HI),
            "tail": (x >= CLAMP_LO) & (x < 0),
            "knee": (x >= 0) & (x < POLE - 0.1),
            "pole band": np.abs(x - POLE) <= 0.1,
            "beyond": (x > POLE + 0.1) & (x <= CLAMP_HI)}


def _probe_form():
    N = PN
    return LinearForm(W=np.zeros((N, N), np.float32), U=np.zeros((N, 1), np.float32), bias=np.zeros(N, np.float32),
                      kappa=np.zeros(N, np.float32), sigma=np.zeros(3 * N, np.float32), tau_s=1.0, tau_m=1e6, tau_a=1e6,
                      resistance=1.0)


def _probe_problem(ext, B, flags=0, sde=False):
    N = PN
    return ext.Problem(torch.zeros(N, 20, device=DEV), torch.zeros(N, device=DEV),
                       torch.zeros(3 * N, device=DEV) if sde else None, torch.tensor([0.0, H], dtype=torch.float32, device=DEV),
                       torch.zeros(B, 2, 1, device=DEV), 1, B, 1.0, 1e6, 1e6, 1.0, flags)


def _y0(x):
    x = torch.as_tensor(x, dtype=torch.float32)
    return torch.cat((x, torch.zeros_like(x), torch.zeros_like(x)), 1)


def _oracle_probe(method, x, records=None):
    """F(t1) and dF(t1)/dV0 of the float64 oracle's solve with the exact φ (x: (B, N) float32 abscissae)."""
    N, B = PN, x.shape[0]
    lf = _probe_form()
    ode = orhs.UnifiedColumnODE(lf, np.array([0.0, H], np.float32), np.zeros((B, 2, 1), np.float32), dtype=torch.float64,
                                requires_grad=False)
    ts = torch.tensor([0.0, H], dtype=torch.float32)
    old = orhs.phi
    orhs.phi = _PhiExact.apply
    try:
        y0 = _y0(x).double().requires_grad_(True)
        if method == "rk4":
            y = S.odeint_rk4(ode, y0, ts.double())
        elif method == "euler":
            y = S.sdeint_euler(ode, y0, ts, S.TabulatedBrownian(torch.zeros(1, B, 1, dtype=torch.float64)), dt=H)
        elif method == "srk":
            z = torch.zeros(1, B, 1, dtype=torch.float64)
            y = S.sdeint_srk(ode, y0, ts, S.TabulatedBrownianU(z, z), dt=H)
        else:                                   # dopri5: replay of the recorded steps, trials with one record together
            rt0, rdt, ost, oxs, na = records
            groups = {}
            for b in range(B):
                n = int(na[b])
                key = (rt0[b, :n].tobytes(), rdt[b, :n].tobytes(), ost[b].tobytes(), oxs[b].tobytes())
                groups.setdefault(key, []).append(b)
            y = torch.zeros(2, B, 3 * N, dtype=torch.float64)
            for idx in groups.values():
                b = idx[0]
                n = int(na[b])
                yr = S.dopri5_replay(ode.select_trials(torch.tensor(idx)), y0[idx], rt0[b, :n], rdt[b, :n], n, ost[b], oxs[b])
                y = y.index_put((torch.tensor([0, 1])[:, None], torch.tensor(idx)[None]), yr)
        (g,) = torch.autograd.grad(y[-1, :, 2 * N:].sum(), y0)
    finally:
        orhs.phi = old
    return y[-1, :, 2 * N:].detach(), g[:, :N]


def _judge(site, fast, fp16_rate, x, F, gV, Fo, gVo, failures, report):
    """Point-by-point errors of φ = F / c and φ′ = gV / c' (c, c' the solver's factors from the oracle solve) against
    float64, with the bars of the site's arithmetic, relative where the rate is above 1e-6 Hz and 1e-9 Hz absolute below.

    Fast path: FP32 accuracy, 5e-6 for φ and 2e-5 for φ′.  Where the elementwise A / F update reads the rate back from its
    FP16 operand pair (xh + xl / 2048, fp16_rate), the pair's absolute resolution 2^-35 Hz is added to φ's bar: it is the
    format's, not φ's.
    Reference arithmetic: its own float32 conditioning, 4e-6 + 8 ulp κ max(1, |z|) for φ and 2e-5 + 8 ulp κ² max(1, |z|)
    for φ′, κ = e / |1 - e| with e = exp(z) (the cancellation in 1 - e), |z| because exp turns a relative rounding error
    of z into |z| times as much in e."""
    x64 = torch.as_tensor(np.asarray(x, dtype=np.float64)).reshape(-1)
    r, dr = phi_dphi_exact(x64)
    z = 80.0 * torch.tanh(-D * (48.0 * x64 - 981.0) / 80.0)
    e = torch.exp(z)
    kap = e / (1 - e).abs()
    cond = kap * z.abs().clamp_min(1.0)
    live = r > RATE_FLOOR
    rows = {}
    for name, val, ref, truth, rel_bar in (
            ("phi", F, Fo, r, (5e-6 + (2.0 ** -35 if fp16_rate else 0.0) / r) if fast else 4e-6 + 8 * 2.0 ** -24 * cond),
            ("dphi", gV, gVo, dr, (2e-5 + 0 * kap) if fast else 2e-5 + 8 * 2.0 ** -24 * kap * cond)):
        if val is None:
            continue
        est = val.double().cpu().reshape(-1) * (truth / ref.reshape(-1))        # the kernel's φ (φ′) at x
        err_abs = (est - truth).abs()
        err_rel = err_abs / truth
        bad = torch.where(live, err_rel > rel_bar, err_abs > 1e-9) | ~torch.isfinite(est)
        for bname, m in _bands(x64.numpy()).items():
            mt = torch.as_tensor(m)
            rel = err_rel[mt & live]
            absl = err_abs[mt & ~live]
            rows.setdefault(bname, {})[name] = (float(rel.max()) if rel.numel() else 0.0, float(absl.max()) if absl.numel() else 0.0)
        if bad.any():
            i = torch.nonzero(bad)[:5, 0]
            failures.append(f"{site} {name}: {int(bad.sum())} points over the bar, e.g. x = {x64[i].tolist()} "
                            f"est {est[i].tolist()} truth {truth[i].tolist()}")
    line = f"  {site:<34}" + "  ".join(
        f"{b}: " + " ".join(f"{n} {v[0]:.1e}" + (f"/abs {v[1]:.0e}" if v[1] else "") for n, v in d.items())
        for b, d in rows.items())
    report.append(line)


def _run_site(ext, site, x, pole=False):
    """(F(t1), dF(t1)/dV0 or None, fast path?, dopri5 record or None) of one code site on the abscissae x (B, N)."""
    N, B = PN, x.shape[0]
    y0 = _y0(x).to(DEV)
    ts = torch.tensor([0.0, H], dtype=torch.float32, device=DEV)
    sel = torch.arange(2 * N, 3 * N, dtype=torch.int32, device=DEV)
    gy = torch.zeros(2, B, N, device=DEV)
    gy[1] = 1.0
    zeros = torch.zeros(1, B, device=DEV)
    if site in ("rhs", "drift_staged"):
        prob = _probe_problem(ext, B)
        f = (ext.rhs if site == "rhs" else ext.drift_staged)(prob, torch.zeros(B, device=DEV), y0)
        return f[:, 2 * N:] * H, None, site == "drift_staged", None           # F(t1) ~ h phi: same scale as the solves
    if site.startswith("rk4"):
        flags = ext.FLAG_FORCE_TENSOR if "tensor" in site else 0
        if site == "rk4 on-chip (chunks < 4096)":
            chunks = [(lo, min(B, lo + 1500)) for lo in range(0, B, 1500)]
        else:
            chunks = [(0, B)]
        Fs, gs = [], []
        for lo, hi in chunks:
            prob = _probe_problem(ext, hi - lo, flags)
            if flags == 0:
                assert prob.kernel_family(ext.OP_RK4_FWD) == 0
                assert (prob.workspace_bytes(ext.OP_RK4_FWD, 2, 0) > 0) == (hi - lo >= 4096)
            if "ckpt" in site:
                assert ext.rk4_ckpt_bytes(prob, 2) > 0
                y, ck = ext.rk4_fwd_ckpt(prob, ts, y0[lo:hi].contiguous(), sel)
                g0, _ = ext.rk4_bwd_ckpt(prob, ts, ck, gy[:, lo:hi].contiguous(), sel)
                Fs.append(y[-1]); gs.append(g0[:, :N])
            else:
                y = ext.rk4_fwd(prob, ts, y0[lo:hi].contiguous(), 1)
                g0, _ = ext.rk4_bwd(prob, ts, y, gy[:, lo:hi].contiguous(), sel)
                Fs.append(y[-1, :, 2 * N:]); gs.append(g0[:, :N])
        fast = site in ("rk4 tiny_tc + bwd<40,true>",) or "tensor" in site
        return torch.cat(Fs, 0), torch.cat(gs, 0), fast, None
    staged = "staged" in site
    prob = _probe_problem(ext, B, ext.FLAG_FORCE_STAGED if staged else 0, sde=True)
    if site.startswith("euler"):
        assert prob.kernel_family(ext.OP_EM_FWD) == (1 if staged else 0)
        y, _, _, st, ys = ext.em_fwd(prob, ts, y0, zeros, 0, 0, H, False, 0.0, 0.0, 0.0, 1)
        g0, _ = ext.em_bwd(prob, ts, ys, gy, sel, H)
    elif site.startswith("srk"):
        assert prob.kernel_family(ext.OP_SRK_FWD) == (1 if staged else 0)
        y, st, ys = ext.srk_fwd(prob, ts, y0, zeros, zeros, 0, 0, H, 1)
        g0, _ = ext.srk_bwd(prob, ts, ys, zeros, zeros, 0, 0, gy, sel, H)
    else:
        assert prob.kernel_family(ext.OP_DOPRI5_FWD) == (1 if staged else 0)
        y, na, nr, st, rec_y, rec_t0, rec_dt, out_step, out_x = ext.dopri5_fwd_record(prob, ts, y0, 1e-7, 1e-9, 4_000_000, 64)
        g0, _ = ext.dopri5_bwd(prob, 2, rec_y, rec_t0, rec_dt, out_step, out_x, na, gy, sel)
        rec = (rec_t0.cpu().numpy(), rec_dt.cpu().numpy(), out_step.cpu().numpy(), out_x.cpu().numpy(), na.cpu().numpy())
        if not pole:
            assert int(st.abs().sum()) == 0
        return y[-1, :, 2 * N:], g0[:, :N], staged, rec
    if not pole:
        assert int(st.abs().sum()) == 0
    return y[-1, :, 2 * N:], g0[:, :N], staged, None


PROBE_SITES = [
    # reference arithmetic (phi / phi_dphi)
    "rhs", "rk4 on-chip (chunks < 4096)", "euler on-chip", "srk on-chip", "dopri5 on-chip",
    # fast path (phi_fast / phi_dphi_fast)
    "drift_staged", "rk4 tiny_tc + bwd<40,true>", "rk4 tensor ckpt persistent", "rk4 tensor ckpt per-stage",
    "rk4 tensor recompute", "euler staged", "srk staged", "dopri5 staged",
]


def _oracle_method(site):
    return "rk4" if site.startswith("rk4") or site in ("rhs", "drift_staged") else site.split()[0]


@pytest.mark.gpu
def test_transfer_function_probe_through_every_code_site():
    """φ (from F(t1)) and φ′ (from dF(t1)/dV0) of every code site, point by point against float64, over the whole
    firing-rate range and the pole band; then each site at the pole exactly, in a solve of its own."""
    ext = odecol._native.ext()
    x = _probe_points()
    xp = np.full((PB, PN), np.float32(POLE))
    truth = {}
    failures, report = [], []
    old = os.environ.get("ODECOL_PERSISTENT")
    pole_line = []
    try:
        for site in PROBE_SITES:
            os.environ["ODECOL_PERSISTENT"] = "0" if site == "rk4 tensor ckpt per-stage" else "1"
            F, gV, fast, rec = _run_site(ext, site, x)
            torch.cuda.synchronize()
            method = _oracle_method(site)
            if method == "dopri5":
                Fo, gVo = _oracle_probe(method, x, rec)
            else:
                if method not in truth:
                    truth[method] = _oracle_probe(method, x)
                Fo, gVo = truth[method]
            if site in ("rhs", "drift_staged"):
                Fo = torch.as_tensor(phi_dphi_exact(x.astype(np.float64))[0]) * H
            _judge(site, fast, site in ("euler staged", "srk staged"), x, F.cpu(), None if gV is None else gV.cpu(), Fo, gVo, failures, report)
            # ---- the pole exactly
            Fp, gVp, _, _ = _run_site(ext, site, xp, pole=True)
            r0, dr0 = phi_dphi_exact(np.float64(x[0, 0]))
            Fp = Fp.cpu().double() * (r0 / Fo[0, 0])                            # F / c: the site's φ at the pole
            if gVp is not None:
                gVp = gVp.cpu().double() * (dr0 / gVo[0, 0])
            if fast:
                ok = bool(torch.isfinite(Fp).all()) and float((Fp - 1 / D).abs().max()) <= 5e-6 / D
                if gVp is not None:
                    ok = ok and bool(torch.isfinite(gVp).all()) and float((gVp - 24).abs().max()) <= 2e-5 * 24
            else:
                ok = bool(torch.isnan(Fp).all())
            pole_line.append(f"{site}: {float(Fp.reshape(-1)[0]):.7g}" +
                             ("" if gVp is None else f" / {float(gVp.reshape(-1)[0]):.7g}"))
            if not ok:
                failures.append(f"{site} at the pole: phi {Fp.reshape(-1)[:3].tolist()} "
                                f"dphi {None if gVp is None else gVp.reshape(-1)[:3].tolist()}")
    finally:
        if old is None:
            os.environ.pop("ODECOL_PERSISTENT", None)
        else:
            os.environ["ODECOL_PERSISTENT"] = old
    print("\n[phi probe] worst relative error per site and band (rates above 1e-6 Hz; abs = worst absolute error below)")
    print("\n".join(report))
    print("[phi probe] phi / dphi at x = 981/48 exactly (limits 112.36 Hz, 24 Hz/mV): " + "; ".join(pole_line))
    assert not failures, "\n".join(failures)


# ----------------------------------------------------------------------------------------------------------------------
# 2. solvers through φ's steep range, against the oracle's autograd
# ----------------------------------------------------------------------------------------------------------------------
TRAJ_BAR, GRAD_BAR = 1e-5, 5e-5
POLE_MARGIN = 6.0        # start states this far from the pole; a window of T <= 12 steps moves x by a few mV at most


class _phi_patch:
    """oracle.rhs.phi replaced for one oracle solve: `xs` collects every argument (every stage evaluation), `slope`
    scales φ′ (the oracle as a reverse kernel with a slightly wrong φ′ would compute it)."""

    def __init__(self, slope=None):
        self.slope, self.xs = slope, []

    def _phi(self, x):
        self.xs.append(x.detach().reshape(-1).double())
        return _ORACLE_PHI(x) if self.slope is None else _PhiScaledSlope.apply(x, self.slope)

    def __enter__(self):
        orhs.phi = self._phi
        return self

    def __exit__(self, *exc):
        orhs.phi = _ORACLE_PHI


def assert_spread(xs, label):
    """Preconditions on the oracle solve: populations in the clamp of the fast tanh, on the knee and beyond the pole;
    every rate finite and within FP16 range; no stage evaluation within 0.05 of the pole (the probe owns that band)."""
    x = torch.cat(xs)
    r = _ORACLE_PHI(x)
    assert bool(torch.isfinite(r).all()) and float(r.max()) < 6.5e4, (label, float(r.max()))
    assert bool((x < -54).any()) and bool(((x > 0) & (x < 20.4)).any()) and bool((x > 20.44).any()), label
    gap = float((x - POLE).abs().min())
    assert gap >= 0.05, (label, gap)
    return gap


def _spread_states(rng, B, N, margin=POLE_MARGIN):
    V = rng.uniform(-60, 40, (B, N))
    A = rng.uniform(0, 15, (B, N))
    x = V - A
    near = np.abs(x - POLE) < margin
    V = np.where(near, V + np.sign(x - POLE + 1e-9) * 2 * margin, V)
    F = rng.uniform(0, 3, (B, N))
    return np.concatenate((V, A, F), 1).astype(np.float32)


def _spread_problem(N, n_in, B, K, seed, T=12):
    """`_problem` of test_gpu_random_problems with start states over φ's range and coupling strong enough that the rates
    of hundreds of Hz feed back (a few mV per window)."""
    rng = np.random.default_rng(seed)
    W = (rng.standard_normal((N, N)) * 1.2 / math.sqrt(N)).astype(np.float32)
    U = (rng.standard_normal((N, n_in)) * 0.05).astype(np.float32)
    bias = (rng.random(N) * 0.3).astype(np.float32)
    kappa = (rng.random(N) * 1.5).astype(np.float32)
    lf = LinearForm(W=W, U=U, bias=bias, kappa=kappa, sigma=(rng.random(3 * N) * 3.0).astype(np.float32), tau_s=5e-4,
                    tau_m=0.02, tau_a=10.0, resistance=80.0)
    tv = np.linspace(0, (T - 1) * 1e-4, T, dtype=np.float32)
    kt = np.unique(np.sort(rng.random(K).astype(np.float32)) * tv[-1] * 1.2 - 0.1 * tv[-1])
    while len(kt) < K:
        kt = np.unique(np.append(kt, kt[-1] + 1e-4 * (1 + len(kt))).astype(np.float32))
    ku = (rng.random((B, K, n_in)) * 20).astype(np.float32)
    return lf, tv, kt, ku, _spread_states(rng, B, N)


def _oracle(lf, kt, ku, y0, tv, wgt, method="rk4", sel=None, bm=None, dt=None, dtype=torch.float32, slope=None):
    """Oracle solve + autograd of sum(wgt * y[..., sel]): (y, grad y0, grad W_aug = [W | U | bias], stage abscissae)."""
    ode = orhs.UnifiedColumnODE(lf, kt, ku, dtype=dtype, requires_grad=True)
    y0o = torch.as_tensor(y0).to(dtype).clone().requires_grad_(True)
    tvt = torch.as_tensor(tv)
    with _phi_patch(slope) as rec:
        if method == "rk4":
            yo = S.odeint_rk4(ode, y0o, tvt.to(dtype))
        elif method == "euler":
            yo = S.sdeint_euler(ode, y0o, tvt, S.TabulatedBrownian(bm[0].to(dtype)), dt=dt)
        else:
            yo = S.sdeint_srk(ode, y0o, tvt, S.TabulatedBrownianU(bm[0].to(dtype), bm[1].to(dtype)), dt=dt)
        ys = yo if sel is None else yo[..., sel]
        (ys * wgt.to(dtype)).sum().backward()
    gW = torch.cat((ode.W.grad, ode.U.grad, ode.bias.grad[:, None]), 1)
    return ys.detach(), y0o.grad, gW, rec.xs


def _relmax(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def _worst_trial(y, yo):
    y, yo = y.double(), yo.double()
    return float(((y - yo).abs().amax(dim=(0, 2)) / yo.abs().amax(dim=(0, 2)).clamp_min(1e-6)).max())


RK4_SHAPES = [(16, 4, 3, 3), (40, 8, 4, 3), (72, 10, 2, 3), (120, 7, 3, 4)]       # K_aug 21 / 49 / 83 / 128: KP = 40 / 64 / 96 / 128
SDE_SHAPES = [(16, 4, 3, 3), (120, 7, 3, 4)]
SDE_DT = 2.5e-4


def _rk4_case(shape):
    N, n_in, B, K = shape
    lf, tv, kt, ku, y0 = _spread_problem(N, n_in, B, K, seed=N * 13 + n_in)
    wgt = torch.randn(len(tv), B, 3 * N, generator=torch.Generator().manual_seed(N))
    return lf, tv, kt, ku, y0, wgt


def _sde_case(shape, method):
    lf, tv, kt, ku, y0, wgt = _rk4_case(shape)
    n_steps = len(S.em_step_schedule(torch.tensor(tv), SDE_DT))
    W, U = S.sample_w_u(n_steps, y0.shape[0], SDE_DT, torch.Generator().manual_seed(shape[0] + 5))
    return lf, tv, kt, ku, y0, wgt, (W, U)


@pytest.mark.gpu
@pytest.mark.parametrize("family", [0, "tensor"])
@pytest.mark.parametrize("shape", RK4_SHAPES, ids=lambda s: "N%d_in%d_B%d_K%d" % s)
def test_rk4_through_the_steep_range(shape, family):
    N, n_in, B, K = shape
    lf, tv, kt, ku, y0, wgt = _rk4_case(shape)
    yo, gy0o, gWo, xs = _oracle(lf, kt, ku, y0, tv, wgt)
    gap = assert_spread(xs, shape)
    ext = odecol._native.ext()
    prob = ext_problem(ext, lf, kt, ku, {0: 0, "tensor": ext.FLAG_FORCE_TENSOR}[family])
    assert prob.kernel_family(ext.OP_RK4_FWD) == {0: 0, "tensor": 2}[family]
    t_dev = torch.tensor(tv).to(DEV)
    y = ext.rk4_fwd(prob, t_dev, torch.tensor(y0).to(DEV), 1)
    gy0, gW = ext.rk4_bwd(prob, t_dev, y, wgt.to(DEV).contiguous(), None)
    y, gy0, gW = y.cpu(), gy0.cpu(), gW.cpu()[:, :N + n_in + 1]
    et, e0, eW, wt = _relmax(y, yo), _relmax(gy0, gy0o), _relmax(gW, gWo), _worst_trial(y, yo)
    print(f"\n[rk4 steep range {shape} family {family}] pole gap {gap:.2f}  trajectory {et:.1e} (worst trial {wt:.1e})  "
          f"grad y0 {e0:.1e}  grad W_aug {eW:.1e}")
    assert et < TRAJ_BAR and e0 < GRAD_BAR and eW < GRAD_BAR and wt < 2e-5


@pytest.mark.gpu
@pytest.mark.parametrize("family", [0, "staged"])
@pytest.mark.parametrize("method", ["euler", "srk"])
@pytest.mark.parametrize("shape", SDE_SHAPES, ids=lambda s: "N%d_in%d_B%d_K%d" % s)
def test_sde_solvers_through_the_steep_range(shape, method, family):
    N, n_in, B, K = shape
    lf, tv, kt, ku, y0, wgt, (W, U) = _sde_case(shape, method)
    yo, gy0o, gWo, xs = _oracle(lf, kt, ku, y0, tv, wgt, method, bm=(W, U), dt=SDE_DT)
    gap = assert_spread(xs, shape)
    ext = odecol._native.ext()
    flags = {0: 0, "staged": ext.FLAG_FORCE_STAGED}[family]
    W_aug = torch.zeros(N, (N + n_in + 1 + 3) // 4 * 4)
    W_aug[:, :N] = torch.tensor(lf.W); W_aug[:, N:N + n_in] = torch.tensor(lf.U); W_aug[:, N + n_in] = torch.tensor(lf.bias)
    prob = ext.Problem(W_aug.to(DEV), torch.tensor(lf.kappa).to(DEV), torch.tensor(lf.sigma).to(DEV), torch.tensor(kt).to(DEV),
                       torch.tensor(ku).to(DEV), n_in, B, lf.tau_s, lf.tau_m, lf.tau_a, lf.resistance, flags)
    assert prob.kernel_family({"euler": ext.OP_EM_FWD, "srk": ext.OP_SRK_FWD}[method]) == (1 if family else 0)
    t_dev, y0d = torch.tensor(tv).to(DEV), torch.tensor(y0).to(DEV)
    n_steps = W.shape[0]
    Wd, Ud = W[:, :, 0].contiguous().to(DEV), U[:, :, 0].contiguous().to(DEV)
    if method == "srk":
        y, st, ysteps = ext.srk_fwd(prob, t_dev, y0d, Wd, Ud, 0, 0, SDE_DT, n_steps)
        gy0, gW = ext.srk_bwd(prob, t_dev, ysteps, Wd, Ud, 0, 0, wgt.to(DEV).contiguous(), None, SDE_DT)
    else:
        y, _, _, st, ysteps = ext.em_fwd(prob, t_dev, y0d, Wd, 0, 0, SDE_DT, False, 0.0, 0.0, 0.0, n_steps)
        gy0, gW = ext.em_bwd(prob, t_dev, ysteps, wgt.to(DEV).contiguous(), None, SDE_DT)
    assert int(st.abs().sum()) == 0
    y, gy0, gW = y.cpu(), gy0.cpu(), gW.cpu()[:, :N + n_in + 1]
    et, e0, eW, wt = _relmax(y, yo), _relmax(gy0, gy0o), _relmax(gW, gWo), _worst_trial(y, yo)
    print(f"\n[{method} steep range {shape} family {family}] pole gap {gap:.2f}  trajectory {et:.1e} (worst trial {wt:.1e})  "
          f"grad y0 {e0:.1e}  grad W_aug {eW:.1e}")
    assert et < TRAJ_BAR and e0 < GRAD_BAR and eW < GRAD_BAR and wt < 2e-5


def _moderate_weights(N, seed):
    """Recurrent weights of the coupling strength of `_spread_problem`.  The reference networks' own (entries up to ~500)
    move x by hundreds of mV per step from spread start states: every window would sweep populations through the pole
    band and past the FP16 range, which is the probe's subject, not these tests'."""
    return torch.randn(N, N, generator=torch.Generator().manual_seed(seed)) * (1.2 / math.sqrt(N))


def _wta_case(cfg, B=4097, T=12, seed=11):
    """The --workload small network (ColumnAreaWTA, N = 16) at 4097 trials: an odd count, so the packed last warp is half
    empty and the last 128-trial CTA of the trial-major kernel is ragged; spread start states, moderate recurrent
    weights.  The module's background drive moves x by up to 8 mV per window, hence the wider margin around the pole."""
    from oracle import column_model as cm
    torch.manual_seed(0)
    net = odecol.ColumnAreaWTA(cfg, "mt")
    with torch.no_grad():
        net.recurrent_weights.copy_(_moderate_weights(16, seed))
    gen = torch.Generator().manual_seed(seed)
    amp = torch.zeros(B, 16)
    a = torch.rand(B, 2, generator=gen) * 30.0
    amp[:, 2] = amp[:, 3] = a[:, 0]; amp[:, 10] = amp[:, 11] = a[:, 1]
    tv = torch.linspace(0.0, (T - 1) * 1e-4, T)
    kt, ku = odecol.step_knots(3e-4, 7e-4, float(tv[-1]), amp, 1e-4)
    y0 = torch.tensor(_spread_states(np.random.default_rng(seed), B, 16, margin=10.0))
    lf = cm.wta_linear_form(cfg, net.recurrent_weights.detach().numpy())
    return net, lf, kt, ku, tv, y0


WTA_SEL = [0, 8, 16, 24]                 # V and A of both columns' L2/3e: the bench's read-out


def _wta_oracle(lf, kt, ku, tv, y0, dtype=torch.float32, slope=None):
    """Oracle of odeint(components=WTA_SEL) + huber_rate_loss(target 0.5).backward()."""
    ode = orhs.UnifiedColumnODE(lf, kt.numpy(), ku.numpy(), dtype=dtype, requires_grad=True)
    y0o = y0.to(dtype).clone().requires_grad_(True)
    with _phi_patch(slope) as rec:
        yo = S.odeint_rk4(ode, y0o, tv.to(dtype))[..., WTA_SEL]
        n_stage = len(rec.xs)
        rate = orhs.phi(yo[..., :2] - yo[..., 2:])
        torch.nn.functional.smooth_l1_loss(rate, torch.full_like(rate, 0.5), beta=1.0).backward()
    return yo.detach(), y0o.grad, ode.W.grad, rec.xs[:n_stage]


@pytest.mark.gpu
def test_smallest_networks_at_large_batch_through_the_steep_range(cfg):
    """tiny_tc forward + the register-resident reverse kernel <40, true> with a component selection and the fused read-out
    loss, as bench.py --workload small runs them, against the oracle's autograd."""
    net, lf, kt, ku, tv, y0 = _wta_case(cfg)
    yo, gy0o, gWo, xs = _wta_oracle(lf, kt, ku, tv, y0)
    gap = assert_spread(xs, "wta")
    net = to_device(net, DEV)
    net.time_vec, net.stim = kt.to(DEV), ku.to(DEV)
    y0p = y0.to(DEV).requires_grad_(True)
    y = odecol.odeint(net, y0p, tv.to(DEV), method="rk4", components=torch.tensor(WTA_SEL, device=DEV))
    odecol.huber_rate_loss(y, torch.full((1, 1, 2), 0.5, device=DEV), 1).backward()
    torch.cuda.synchronize()
    yc = y.detach().cpu()
    et = max(_relmax(yc[..., :2], yo[..., :2]), _relmax(yc[..., 2:], yo[..., 2:]))
    e0, eW, wt = _relmax(y0p.grad.cpu(), gy0o), _relmax(net.recurrent_weights.grad.cpu(), gWo), _worst_trial(yc, yo)
    print(f"\n[WTA 4097 trials, steep range] pole gap {gap:.2f}  trajectory {et:.1e} (worst trial {wt:.1e})  grad y0 {e0:.1e}  "
          f"grad W {eW:.1e}")
    assert et < TRAJ_BAR and e0 < GRAD_BAR and eW < GRAD_BAR and wt < 2e-5


def _c4_case(cfg, B=4790, T=10, seed=21, device=DEV):
    cols, N = 64, 512
    sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=0, device=device)
    with torch.no_grad():
        sheet.recurrent_weights.copy_(_moderate_weights(N, seed))
    gen = torch.Generator().manual_seed(seed)
    amp = torch.rand(B, cols, generator=gen) * 30.0
    t_end = (T - 1) * 1e-4
    kt, ku = odecol.step_knots(0.3 * t_end, 0.7 * t_end, t_end, amp, 1e-4)
    sheet.set_knots(kt.to(device), ku.to(device))
    tv = torch.linspace(0.0, t_end, T)
    y0 = torch.tensor(_spread_states(np.random.default_rng(seed), B, N, margin=10.0))
    sel = list(range(0, N, 8)) + list(range(N, 2 * N, 8)) + [2 * N, 2 * N + 129, 3 * N - 1]
    wgt = torch.randn(T, B, len(sel), generator=gen)
    return sheet, sheet_oracle_form(sheet), kt, ku, tv, y0, sel, wgt


@pytest.mark.gpu
def test_c4_shape_through_the_steep_range(cfg):
    """N = 512, B = 4790, T = 10: checkpoint mode with the persistent FP16 forward solve, the benched path."""
    sheet, lf, kt, ku, tv, y0, sel, wgt = _c4_case(cfg)
    yo, gy0o, gWo, xs = [], [], 0, []
    for lo in range(0, y0.shape[0], 512):                     # trials are independent: the oracle chunk by chunk
        hi = min(y0.shape[0], lo + 512)
        a, b, c, d = _oracle(lf, kt.numpy(), ku[lo:hi].numpy(), y0[lo:hi], tv, wgt[:, lo:hi], sel=sel)
        yo.append(a); gy0o.append(b); gWo = gWo + c; xs += d
    yo, gy0o = torch.cat(yo, 1), torch.cat(gy0o, 0)
    gap = assert_spread(xs, "C4")
    y0p = y0.to(DEV).requires_grad_(True)
    yp = odecol.odeint(sheet, y0p, tv.to(DEV), method="rk4", components=sel, options={"checkpoint": True})
    assert "Ckpt" in type(yp.grad_fn).__name__
    (yp * wgt.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    N, nV = 512, 64
    ypc = yp.detach().cpu()
    et = max(_relmax(ypc[..., sl], yo[..., sl]) for sl in (slice(0, nV), slice(nV, 2 * nV), slice(2 * nV, None)))
    e0, eW, eU = _relmax(y0p.grad.cpu(), gy0o), _relmax(sheet.recurrent_weights.grad.cpu(), gWo[:, :N]), \
        _relmax(sheet.input_weights.grad.cpu(), gWo[:, N:N + 64])
    wt = _worst_trial(ypc, yo)
    print(f"\n[C4 shape, steep range] pole gap {gap:.2f}  trajectory {et:.1e} (worst trial {wt:.1e})  dy0 {e0:.1e}  dW {eW:.1e}  "
          f"dU {eU:.1e}")
    assert et < TRAJ_BAR and e0 < GRAD_BAR and eW < GRAD_BAR and eU < GRAD_BAR and wt < 2e-5


@pytest.mark.gpu
@pytest.mark.parametrize("family", [0, "staged"])
def test_dopri5_through_the_steep_range(family):
    """dopri5 record and discrete adjoint against a float64 replay of the recorded steps; the range preconditions are
    asserted on the oracle's rk4 solve of the same problem and window."""
    shape = (40, 8, 4, 3)
    lf, tv, kt, ku, y0, wgt = _rk4_case(shape)
    gap = assert_spread(_oracle(lf, kt, ku, y0, tv, wgt)[3], shape)
    ext = odecol._native.ext()
    prob = ext_problem(ext, lf, kt, ku, {0: 0, "staged": ext.FLAG_FORCE_STAGED}[family])
    assert prob.kernel_family(ext.OP_DOPRI5_FWD) == (1 if family else 0)
    print(f"\n[dopri5 steep range, pole gap {gap:.2f}]", end="")
    check_dopri5_against_replay(ext, prob, lf, kt, ku, y0, tv, 1e-7, 1e-9, f"steep range {family}", seed=3)


def test_solver_tests_of_the_steep_range_see_phi_prime(cfg):
    """Without a GPU: scaling φ′ by 1.01 in the float64 oracle moves dy0 and dW_aug of every steep-range problem by at
    least 20x the gradient bar (the tail-bound problems of the older tests move by 1-6x)."""
    moved = {}
    for shape in RK4_SHAPES:
        lf, tv, kt, ku, y0, wgt = _rk4_case(shape)
        runs = [_oracle(lf, kt, ku, y0, tv, wgt, dtype=torch.float64, slope=s)[1:3] for s in (None, 1.01)]
        moved[f"rk4 {shape}"] = runs
    for shape in SDE_SHAPES:
        for m in ("euler", "srk"):
            lf, tv, kt, ku, y0, wgt, bm = _sde_case(shape, m)
            runs = [_oracle(lf, kt, ku, y0, tv, wgt, m, bm=bm, dt=SDE_DT, dtype=torch.float64, slope=s)[1:3] for s in (None, 1.01)]
            moved[f"{m} {shape}"] = runs
    _, lf, kt, ku, tv, y0 = _wta_case(cfg)
    moved["wta 4097"] = [_wta_oracle(lf, kt, ku, tv, y0, torch.float64, s)[1:3] for s in (None, 1.01)]
    _, lf, kt, ku, tv, y0, sel, wgt = _c4_case(cfg, B=256, device="cpu")          # the C4 sheet, its first 256 trials
    moved["C4 (256 trials)"] = [_oracle(lf, kt.numpy(), ku.numpy(), y0, tv, wgt, sel=sel, dtype=torch.float64, slope=s)[1:3]
                                for s in (None, 1.01)]
    lines = []
    for k, ((g0, gW), (g0s, gWs)) in moved.items():
        d0, dW = _relmax(g0s, g0), _relmax(gWs, gW)
        lines.append(f"  {k}: dy0 {d0:.1e}  dW_aug {dW:.1e}")
        assert d0 >= 20 * GRAD_BAR and dW >= 20 * GRAD_BAR, (k, d0, dW)
    print("\n[phi' x 1.01 in the float64 oracle]\n" + "\n".join(lines))
