"""Adaptive Euler-Maruyama held to float32 rounding, in the two regimes where the step controller's decisions cannot flip.

torchsde's controller multiplies the step by a factor clamped to [0.2, 1.4] (to [1, 1.4] after an accepted step).  Where
the unclamped factor sits far beyond a clamp, the last bits of the drift cannot change a decision, so the float32
kernels and the float64 oracle (oracle.solvers.sdeint_euler, one trial at a time on the kernels' virtual Brownian tree)
must walk the SAME steps, and their outputs must agree to float32 rounding:

  * grow:   loose tolerances -- every attempt is accepted and the step grows by exactly 1.4 each time;
  * ladder: tolerances near zero -- every error is above 20, so the step shrinks by exactly 0.2: from dt = 1e-3 the
            1e-3 and 2e-4 attempts are rejected, the 4e-5 attempt is accepted (its successor would fall below dt_min)
            and every later step runs at dt_min.  This is the rejection path: the operand of f(t_cur, y) must survive
            a rejected attempt, and the next attempt's Brownian increments are drawn relative to W(t_cur).

Each case checks its regime from the oracle's trace first (a failed premise is reported as such, not as a tolerance
error).  Every case has per-trial noise amplitudes (one trial without noise), a nonzero seed and trial offset; the
staged cases also have per-trial lateral gains.  The same sweep split into two shards must give the same bits."""
import dataclasses
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import odecol
from helpers import TreeBrownian, sheet_oracle_form
from oracle import rhs as orhs, solvers as S
from oracle.column_model import LinearForm

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

f32 = lambda x: float(np.float32(x))          # the kernels take dt, dt_min and the tolerances as float32
#                rtol        atol        dt          dt_min      window
REGIMES = {"grow": (f32(1.0), f32(1e3), f32(1e-5), f32(1e-6), 1.2e-3),
           "ladder": (f32(1e-12), f32(1e-12), f32(1e-3), f32(1e-5), 3e-4)}
SEED, TRIAL_OFFSET = 1234, 17


def _unclamped_factors(trace):
    """torchsde's step factor before its clamp, for every attempt of a trace (adaptive_update without min / max)."""
    out, prev = [], None
    for _, _, err, _ in trace:
        ratio = 0.9 / err if err > 0 else np.inf
        if err > 1:
            out.append(ratio ** (1 / 1.5))
        else:
            out.append(ratio ** (1 / 4.5) * (ratio / (ratio if prev is None else prev)) ** 0.13)
            prev = ratio
    return out


def _check_premise(regime, traces, dt, dt_min):
    for b, tr in enumerate(traces):
        errs = [e for _, _, e, _ in tr]
        if regime == "grow":
            fac = _unclamped_factors(tr)
            assert all(a for *_, a in tr) and min(fac) >= 1.4 * 1.1, \
                f"premise of the grow regime fails for trial {b}: unclamped factors down to {min(fac):.3f}, errors up to {max(errs):.2e}"
        else:
            # the last attempt ends the solve at dt_min, accepted whatever its error (it may be a sliver of a step)
            assert min(errs[:-1]) >= 20, f"premise of the ladder regime fails for trial {b}: an error of {min(errs[:-1]):.2e} < 20"
            hs = [t1 - t0 for t0, t1, _, _ in tr]
            assert [a for *_, a in tr[:3]] == [False, False, True] and all(a for *_, a in tr[3:]), \
                f"ladder regime: trial {b} did not reject exactly its first two attempts"
            assert abs(hs[2] - dt * 0.04) < 1e-9 and all(abs(h - dt_min) < 1e-9 for h in hs[3:-1]), (b, hs[:5])


def _oracle(lf_of_trial, kt, ku, ts, y0, regime, trials):
    """sdeint_euler(adaptive=True) per trial in float64 (times in float32 as torchsde keeps them), with its trace."""
    rtol, atol, dt, dt_min, _ = REGIMES[regime]
    ys, na, nr, traces = [], [], [], []
    for b in range(trials):
        ode = orhs.UnifiedColumnODE(lf_of_trial(b), kt, ku[b:b + 1], dtype=torch.float64)
        st, tr = {}, []
        bm = TreeBrownian(SEED, TRIAL_OFFSET + b, ts[0], ts[-1])
        with torch.no_grad():
            ys.append(S.sdeint_euler(ode, y0[b:b + 1].double(), ts, bm, dt=dt, adaptive=True, rtol=rtol, atol=atol,
                                     dt_min=dt_min, stats=st, trace=tr))
        na.append(st["n_accept"]); nr.append(st["n_reject"]); traces.append(tr)
    _check_premise(regime, traces, dt, dt_min)
    return torch.cat(ys, 1), np.array(na), np.array(nr)


def _compare(label, yp, na, nr, status, yo, nao, nro):
    N = yo.shape[-1] // 3
    assert int(np.abs(status).sum()) == 0, status
    errs = np.array([[float((yp[:, b, c * N:(c + 1) * N].double() - yo[:, b, c * N:(c + 1) * N]).abs().max()) /
                      float(yo[:, b, c * N:(c + 1) * N].abs().max().clamp_min(1e-30)) for c in range(3)] for b in range(yo.shape[1])])
    print(f"\n[adaptive EM {label}] accepted {na.tolist()} (oracle {nao.tolist()}), rejected {nr.tolist()} (oracle {nro.tolist()}); "
          f"worst V/A/F over trials {errs[:, 0].max():.1e} {errs[:, 1].max():.1e} {errs[:, 2].max():.1e}")
    assert np.array_equal(na, nao) and np.array_equal(nr, nro)
    assert errs.max() < 1e-5, errs


def _noise_scales(B, gen):
    sc = torch.rand(B, generator=gen) * 2.0
    sc[1] = 0.0
    return sc


# ----------------------------------------------------------------------------------------------------------------------
# on-chip family: a random problem, through the extension
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("regime", list(REGIMES))
def test_on_chip_adaptive_em_walks_the_oracle_steps(regime):
    N, n_in, B, K = 120, 7, 5, 4
    rng = np.random.default_rng(5)
    lf = LinearForm(W=(rng.standard_normal((N, N)) * 0.04).astype(np.float32), U=(rng.standard_normal((N, n_in)) * 0.02).astype(np.float32),
                    bias=(rng.random(N) * 0.3).astype(np.float32), kappa=(rng.random(N) * 1.5).astype(np.float32),
                    sigma=(rng.random(3 * N) * 3.0).astype(np.float32), tau_s=5e-4, tau_m=0.02, tau_a=10.0, resistance=80.0)
    t_end = REGIMES[regime][4]
    ts = torch.linspace(0.0, t_end, 5)
    kt = np.array([0.0, 0.3, 0.6, 1.2], dtype=np.float32) * t_end           # the stimulus changes inside the window
    ku = (rng.random((B, K, n_in)) * 20).astype(np.float32)
    y0 = torch.tensor(np.concatenate((rng.random((B, N)) * 8 - 10, rng.random((B, N)), rng.random((B, N)) * 3), 1), dtype=torch.float32)
    sc = _noise_scales(B, torch.Generator().manual_seed(6))
    yo, nao, nro = _oracle(lambda b: dataclasses.replace(lf, sigma=lf.sigma * float(sc[b])), kt, ku, ts, y0, regime, B)
    ext = odecol._native.ext()
    W_aug = torch.zeros(N, (N + n_in + 1 + 3) // 4 * 4)
    W_aug[:, :N] = torch.tensor(lf.W); W_aug[:, N:N + n_in] = torch.tensor(lf.U); W_aug[:, N + n_in] = torch.tensor(lf.bias)
    prob = ext.Problem(W_aug.to(DEV), torch.tensor(lf.kappa).to(DEV), torch.tensor(lf.sigma).to(DEV), torch.tensor(kt).to(DEV),
                       torch.tensor(ku).to(DEV), n_in, B, lf.tau_s, lf.tau_m, lf.tau_a, lf.resistance, 0)
    prob.set_sigma_scale(sc.to(DEV))
    assert prob.kernel_family(ext.OP_EM_FWD) == 0
    rtol, atol, dt, dt_min, _ = REGIMES[regime]
    y, na, nr, st, _ = ext.em_fwd(prob, ts.to(DEV), y0.to(DEV), None, SEED, TRIAL_OFFSET, dt, True, rtol, atol, dt_min, 0)
    _compare(f"on-chip N={N} {regime}", y.cpu(), na.cpu().numpy(), nr.cpu().numpy(), st.cpu().numpy(), yo, nao, nro)


# ----------------------------------------------------------------------------------------------------------------------
# staged family: column sheets through the public sdeint, with the sweep's per-member lateral gain
# ----------------------------------------------------------------------------------------------------------------------
def _sheet_case(cfg, cols, B, regime):
    sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=cols, device=DEV, sigma_v=4.0)
    N = 8 * cols
    t_end = REGIMES[regime][4]
    gen = torch.Generator().manual_seed(cols + B)
    amp = torch.rand(B, cols, generator=gen) * 25
    kt, ku = odecol.step_knots(0.2 * t_end, 0.6 * t_end, 2 * t_end, amp, 0.1 * t_end)
    sheet.set_knots(kt.to(DEV), ku.to(DEV))
    ts = torch.linspace(0.0, t_end, 5)
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 4 - 6, torch.rand(B, N, generator=gen) * 0.5, torch.rand(B, N, generator=gen)), 1)
    sc = _noise_scales(B, gen)
    gain = torch.rand(B, generator=gen) * 1.5 + 0.5
    gain[0] = 1.0
    return sheet, kt, ku, ts, y0, sc, gain


def _sheet_oracle(sheet, kt, ku, ts, y0, sc, gain, regime):
    lf = sheet_oracle_form(sheet)
    W_lat = sheet.lateral_split()[0].detach().cpu().numpy()
    W_loc = lf.W - W_lat
    return _oracle(lambda b: dataclasses.replace(lf, W=W_loc + float(gain[b]) * W_lat, sigma=lf.sigma * float(sc[b])),
                   kt.numpy(), ku.numpy(), ts, y0, regime, y0.shape[0])


def _sheet_solve(sheet, ts, y0, sc, gain, regime, trial_offset=TRIAL_OFFSET):
    rtol, atol, dt, dt_min, _ = REGIMES[regime]
    st = {}
    with torch.no_grad():
        y = odecol.sdeint(sheet, y0.to(DEV), ts.to(DEV), method="euler", dt=dt, adaptive=True, rtol=rtol, atol=atol,
                          dt_min=dt_min, seed=SEED, trial_offset=trial_offset, stats=st,
                          options={"sigma_scale": sc, "lateral_gain": gain})
    return y.cpu(), st["n_accept"].cpu().numpy(), st["n_reject"].cpu().numpy(), st["status"].cpu().numpy()


@pytest.mark.parametrize("regime", list(REGIMES))
@pytest.mark.parametrize("cols", [32, 128], ids=["N256", "N1024"])
def test_staged_adaptive_em_walks_the_oracle_steps(cfg, cols, regime):
    """FP16 operand pairs (the default); N = 1024 runs the chunked contraction (K_aug = 1153)."""
    sheet, kt, ku, ts, y0, sc, gain = _sheet_case(cfg, cols, 5, regime)
    yo, nao, nro = _sheet_oracle(sheet, kt, ku, ts, y0, sc, gain, regime)
    _compare(f"staged N={8 * cols} {regime}", *_sheet_solve(sheet, ts, y0, sc, gain, regime), yo, nao, nro)


_TF32_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
import odecol
a = torch.load(sys.argv[2])
cfg = odecol.load_config(sys.argv[1] + "/config/model.toml")
sheet = odecol.SyntheticColumnSheet(cfg, a["cols"], seed=a["cols"], device="cuda", sigma_v=4.0)
sheet.set_knots(a["kt"].cuda(), a["ku"].cuda())
st = {}
with torch.no_grad():
    y = odecol.sdeint(sheet, a["y0"].cuda(), a["ts"].cuda(), method="euler", dt=a["dt"], adaptive=True, rtol=a["rtol"], atol=a["atol"],
                      dt_min=a["dt_min"], seed=a["seed"], trial_offset=a["trial_offset"], stats=st,
                      options={"sigma_scale": a["sc"], "lateral_gain": a["gain"]})
torch.save({"y": y.cpu(), **{k: v.cpu() for k, v in st.items()}}, sys.argv[3])
"""


@pytest.mark.parametrize("regime", list(REGIMES))
def test_staged_adaptive_em_in_tf32_pairs_walks_the_oracle_steps(cfg, regime, tmp_path):
    """The same N = 1024 sweep with ODECOL_EM16=0 (TF32 operand pairs); the switch is read once per process."""
    cols = 128
    sheet, kt, ku, ts, y0, sc, gain = _sheet_case(cfg, cols, 5, regime)
    yo, nao, nro = _sheet_oracle(sheet, kt, ku, ts, y0, sc, gain, regime)
    rtol, atol, dt, dt_min, _ = REGIMES[regime]
    torch.save(dict(cols=cols, kt=kt, ku=ku, ts=ts, y0=y0, sc=sc, gain=gain, rtol=rtol, atol=atol, dt=dt, dt_min=dt_min,
                    seed=SEED, trial_offset=TRIAL_OFFSET), tmp_path / "in.pt")
    subprocess.run([sys.executable, "-c", _TF32_SCRIPT, ROOT, str(tmp_path / "in.pt"), str(tmp_path / "out.pt")],
                   env=dict(os.environ, ODECOL_EM16="0"), check=True, timeout=600)
    r = torch.load(tmp_path / "out.pt")
    _compare(f"staged N={8 * cols} TF32 pairs {regime}", r["y"], r["n_accept"].numpy(), r["n_reject"].numpy(),
             r["status"].numpy(), yo, nao, nro)


# ----------------------------------------------------------------------------------------------------------------------
# sharding: sdeint promises that results do not depend on it
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [40, 400])
def test_sharded_sweep_gives_the_bits_of_the_whole_batch(cfg, B):
    """The C5 sweep's settings (rtol 1e-5, atol 1e-4, dt 1e-3, per-member noise amplitude and lateral gain) at N = 1024:
    the batch in one call, and again as two shards with trial_offset = lo and their slices of every per-trial input, must
    give the same counts and bit-identical outputs.  At B = 40 every call tiles its trials 16 to a tile; at B = 400 the
    whole batch runs 32-trial tiles and its shards 16-trial tiles (stage_tc.cuh: pick_tile_n), so the contraction's
    per-element sums must not depend on the trial-tile width either."""
    cols = 128
    N = 8 * cols
    sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=9, device=DEV)
    gen = torch.Generator().manual_seed(B)
    amp = torch.rand(B, cols, generator=gen) * 25
    kt, ku = odecol.step_knots(1e-3, 3e-3, 6e-3, amp, 1e-4)
    ts = torch.linspace(0.0, 4e-3, 5)
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 4 - 6, torch.rand(B, N, generator=gen) * 0.5, torch.rand(B, N, generator=gen)), 1)
    sc = torch.rand(B, generator=gen) * 2.0
    gain = torch.rand(B, generator=gen) * 1.5 + 0.5

    def solve(lo, hi):
        sheet.set_knots(kt.to(DEV), ku[lo:hi].to(DEV))
        st = {}
        with torch.no_grad():
            y = odecol.sdeint(sheet, y0[lo:hi].to(DEV), ts.to(DEV), method="euler", dt=1e-3, adaptive=True, rtol=1e-5, atol=1e-4,
                              seed=SEED, trial_offset=lo, stats=st, options={"sigma_scale": sc[lo:hi], "lateral_gain": gain[lo:hi]})
        return y.cpu(), st["n_accept"].cpu(), st["n_reject"].cpu()

    y, na, nr = solve(0, B)
    parts = [solve(0, B // 2), solve(B // 2, B)]
    ys, nas, nrs = (torch.cat(x, d) for x, d in zip(zip(*parts), (1, 0, 0)))
    n_diff = int((ys != y).any(dim=(0, 2)).sum())
    print(f"\n[sharded sweep B={B}] accepted {int(na.min())}..{int(na.max())}, rejected {int(nr.min())}..{int(nr.max())}; "
          f"trials whose outputs differ from the whole batch: {n_diff}, largest difference {float((ys - y).abs().max()):.1e}")
    assert torch.equal(nas, na) and torch.equal(nrs, nr)
    assert torch.equal(ys, y)
