"""Oracle parity on the paths bench.py actually runs (VERDICT round 1, items 1a-1c):

  * C4: rk4 forward + exact discrete adjoint at N = 512, n_in = 64 (K_aug = 577, four population tiles), batches large enough
    that the persistent tcgen05 kernels own SEVERAL (population tile, trial tile) pairs per CTA and more tiles than SMs --
    the cross-CTA `done[nt]` counter protocol of stage_tc_persist.cu / k_tc_bwd_chain -- in checkpoint and recompute mode,
    persistent and per-stage launches, with and without an F component in the selection;
  * C5: the adaptive Euler-Maruyama controller (on-chip and staged) against oracle.solvers.sdeint_euler(adaptive=True)
    trial by trial (torchsde controls the step of each solve on its own), first without noise, then on the SAME
    Brownian path (odecol_brownian_query exposes the virtual tree the kernels draw from);
  * C5: one drift evaluation at N = 8192 (K_aug = 9217: chunked accumulation, grouped tile order, 64 population tiles)
    against the float64 oracle right-hand side -- in TF32 pairs through odecol_drift_staged, and in the FP16 pairs the
    sweep runs, with and without the per-member lateral gain, through one noiseless sdeint step.
"""
import os

import numpy as np
import pytest
import torch

import odecol
from oracle import rhs as orhs, solvers as S
from helpers import XOR_DICT, TreeBrownian, oracle_form, product_network, sheet_oracle_form

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _scale(a):
    return float(a.abs().max().clamp_min(1e-30))


def _relmax(a, b):
    return float((a - b).abs().max()) / _scale(b)


# ----------------------------------------------------------------------------------------------------------------------
# C4 shape
# ----------------------------------------------------------------------------------------------------------------------
def _c4_problem(cfg, B, T, seed, amp_scale=30.0):
    cols, N = 64, 512
    sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=0, device=DEV)
    gen = torch.Generator().manual_seed(seed)
    amp = torch.rand(B, cols, generator=gen) * amp_scale
    dt = 1e-4
    t_end = (T - 1) * dt
    kt, ku = odecol.step_knots(0.3 * t_end, 0.7 * t_end, t_end, amp, dt)       # stimulus switches on and off inside the window
    sheet.set_knots(kt.to(DEV), ku.to(DEV))
    tv = torch.linspace(0.0, t_end, T)
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 6 - 8, torch.rand(B, N, generator=gen),
                    torch.rand(B, N, generator=gen) * 2), 1)
    return sheet, kt, ku, tv, y0, gen


def _oracle_rk4_grads(lf, kt, ku, tv, y0, sel, wgt, chunk=256):
    """Oracle rk4 + autograd, trial chunk by trial chunk (trials are independent; dW, dU, dbias add up)."""
    B = y0.shape[0]
    traj, gy0 = [], []
    gW = gU = gb = None
    for lo in range(0, B, chunk):
        hi = min(B, lo + chunk)
        ode = orhs.UnifiedColumnODE(lf, kt.numpy(), ku[lo:hi].numpy(), requires_grad=True)
        y0c = y0[lo:hi].clone().requires_grad_(True)
        yo = S.odeint_rk4(ode, y0c, tv)
        ys = yo[:, :, sel]
        (ys * wgt[:, lo:hi]).sum().backward()
        traj.append(ys.detach())
        gy0.append(y0c.grad)
        gW = ode.W.grad if gW is None else gW + ode.W.grad
        gU = ode.U.grad if gU is None else gU + ode.U.grad
        gb = ode.bias.grad if gb is None else gb + ode.bias.grad
    return torch.cat(traj, 1), torch.cat(gy0, 0), gW, gU, gb


C4_CASES = [
    # B,    T,  checkpoint, persistent, with_F
    (4790, 10, True, "1", False),        # TN = 80: 240 tiles on 148 CTAs (92 CTAs own two), ragged last trial tile
    (4790, 10, True, "1", True),
    (4790, 10, False, "1", False),       # recompute mode: trajectory + three recomputed contractions per reverse step
    (4790, 10, True, "0", False),        # one launch per stage instead of the cooperative kernels
    (8192, 6, True, "1", False),         # the benched batch: TN = 112, 296 tiles = exactly two per CTA
    (4790, 10, True, "1:nofuse", False), # dW as a launch of its own (ODECOL_FUSE_DW=0) instead of the chain's fifth phase
]


@pytest.mark.parametrize("B,T,ckpt,persistent,with_f", C4_CASES,
                         ids=lambda v: str(v))
def test_rk4_adjoint_at_the_benchmarked_shape(cfg, B, T, ckpt, persistent, with_f):
    sheet, kt, ku, tv, y0, gen = _c4_problem(cfg, B, T, seed=B + T)
    N = 512
    sel = list(range(0, N, 8)) + list(range(N, 2 * N, 8)) + [3, 130, 257, 511, N + 1, N + 300]     # the bench's read-out + strays
    if with_f:
        sel += [2 * N, 2 * N + 129, 3 * N - 1]
    wgt = torch.randn(T, B, len(sel), generator=gen)
    lf = sheet_oracle_form(sheet)
    tro, gy0o, gWo, gUo, gbo = _oracle_rk4_grads(lf, kt, ku, tv, y0, sel, wgt)

    old = os.environ.get("ODECOL_PERSISTENT")
    persistent, _, variant = persistent.partition(":")
    os.environ["ODECOL_PERSISTENT"] = persistent
    if variant == "nofuse":
        os.environ["ODECOL_FUSE_DW"] = "0"
    try:
        y0p = y0.to(DEV).requires_grad_(True)
        yp = odecol.odeint(sheet, y0p, tv.to(DEV), method="rk4", components=sel, options={"checkpoint": ckpt})
        assert ("Ckpt" in type(yp.grad_fn).__name__) == ckpt
        (yp * wgt.to(DEV)).sum().backward()
        torch.cuda.synchronize()
    finally:
        os.environ.pop("ODECOL_FUSE_DW", None)
        if old is None:
            os.environ.pop("ODECOL_PERSISTENT", None)
        else:
            os.environ["ODECOL_PERSISTENT"] = old
    nV = len([c for c in sel if c < N])
    nA = len([c for c in sel if N <= c < 2 * N])
    ypc = yp.detach().cpu()
    blocks = {"V": slice(0, nV), "A": slice(nV, nV + nA)}
    if with_f:
        blocks["F"] = slice(nV + nA, len(sel))
    et = max(_relmax(ypc[:, :, sl], tro[:, :, sl]) for sl in blocks.values())
    e0 = _relmax(y0p.grad.cpu(), gy0o)
    eW = _relmax(sheet.recurrent_weights.grad.cpu(), gWo)
    eU = _relmax(sheet.input_weights.grad.cpu(), gUo)
    print(f"\n[C4 shape B={B} T={T} ckpt={ckpt} persistent={persistent} F={with_f}] trajectory {et:.1e}  dy0 {e0:.1e}  "
          f"dW {eW:.1e}  dU {eU:.1e}")
    assert et < 1e-5 and e0 < 5e-5 and eW < 5e-5 and eU < 5e-5
    # worst single trial (a mis-addressed trial tile would hide in a max over the whole batch only if it were tiny)
    per_trial = (ypc - tro).abs().amax(dim=(0, 2)) / tro.abs().amax(dim=(0, 2)).clamp_min(1e-6)
    assert float(per_trial.max()) < 2e-5, int(per_trial.argmax())


_FALLBACK_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
import odecol
cfg = odecol.load_config(sys.argv[1] + "/config/model.toml")
B, T, N, cols = 300, 6, 512, 64
sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=0, device="cuda")
gen = torch.Generator().manual_seed(77)
amp = torch.rand(B, cols, generator=gen) * 30.0
t_end = (T - 1) * 1e-4
kt, ku = odecol.step_knots(0.3 * t_end, 0.7 * t_end, t_end, amp, 1e-4)
sheet.set_knots(kt.cuda(), ku.cuda())
tv = torch.linspace(0.0, t_end, T).cuda()
y0 = torch.cat((torch.rand(B, N, generator=gen) * 6 - 8, torch.rand(B, N, generator=gen), torch.rand(B, N, generator=gen) * 2), 1)
hot = torch.rand(B, N, generator=gen) < 0.01
y0[:, :N][hot] = float(sys.argv[3])          # phi(1400 - A) = 6.6e4: beyond what the FP16 operand planes hold
sel = list(range(0, N, 8)) + list(range(N, 2 * N, 8))
y0p = y0.cuda().requires_grad_(True)
y = odecol.odeint(sheet, y0p, tv, method="rk4", components=sel, options={"checkpoint": True, "deterministic": True})
y.square().sum().backward()
torch.save({"y": y.detach().cpu(), "dy0": y0p.grad.cpu(), "dW": sheet.recurrent_weights.grad.cpu()}, sys.argv[2])
"""


def test_rk4_forward_repeats_in_tf32_when_fp16_cannot_hold_the_operand(tmp_path):
    """The persistent forward kernel keeps its operands as FP16 pairs; a firing rate of 66 kHz (V - A = 1400) does not fit.
    The kernels raise a device flag and the launch sequence repeats the solve in the TF32 format (stage_tc_persist.cu,
    a kernel that returns at once when the flag is clear).  The repeated solve IS the TF32 solve: the result must be
    bit-identical to a run with ODECOL_FWD16=0 -- and with ordinary rates the two formats must differ (or the 16-bit
    kernel is not what ran)."""
    import subprocess
    import sys

    def run(fwd16, v_hot):
        out = tmp_path / f"r_{fwd16}_{int(v_hot)}.pt"
        env = dict(os.environ, ODECOL_FWD16=fwd16)
        subprocess.run([sys.executable, "-c", _FALLBACK_SCRIPT, ROOT, str(out), str(v_hot)], env=env, check=True, timeout=600)
        return torch.load(out)

    a, b = run("1", 1400.0), run("0", 1400.0)
    assert torch.isfinite(a["y"]).all()
    for k in ("y", "dy0", "dW"):
        assert torch.equal(a[k], b[k]), k
    c, d = run("1", 4.0), run("0", 4.0)                      # V = 4: rates of a few Hz, the 16-bit format holds everything
    assert not torch.equal(c["y"], d["y"])
    assert float((c["y"] - d["y"]).abs().max()) <= 2e-6 * float(d["y"].abs().max())


_EM_RETRY_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
import odecol
cfg = odecol.load_config(sys.argv[1] + "/config/model.toml")
B, cols = 5, 32
N = 8 * cols
sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=0, device="cuda")
gen = torch.Generator().manual_seed(5)
amp = torch.rand(B, cols, generator=gen) * 30.0
kt, ku = odecol.step_knots(0.002, 0.006, 0.01, amp, 1e-3)
sheet.set_knots(kt.cuda(), ku.cuda())
ts = torch.linspace(0.0, 0.01, 6).cuda()
y0 = torch.cat((torch.rand(B, N, generator=gen) * 6 - 8, torch.rand(B, N, generator=gen), torch.rand(B, N, generator=gen) * 2), 1)
y0[:, 3] = float(sys.argv[3])
adaptive = sys.argv[4] == "1"
with torch.no_grad():
    y = odecol.sdeint(sheet, y0.cuda(), ts, method="euler", dt=1e-3 if adaptive else 1e-4, adaptive=adaptive, rtol=1e-4, atol=1e-3, dt_min=1e-5, seed=3,
                      options={"sigma_scale": torch.full((B,), 0.1)})
torch.save(y.cpu(), sys.argv[2])
"""


@pytest.mark.parametrize("adaptive", ["0", "1"])
def test_staged_euler_maruyama_repeats_in_tf32_when_fp16_cannot_hold_the_operand(tmp_path, adaptive):
    """The drift contractions of the staged Euler-Maruyama solvers read FP16 pairs; the host reads the overflow flag at its
    polls and repeats the solve in the TF32 format.  Same criterion as for the rk4 forward kernel above."""
    import subprocess
    import sys

    def run(em16, v_hot):
        out = tmp_path / f"e_{em16}_{int(v_hot)}.pt"
        env = dict(os.environ, ODECOL_EM16=em16)
        subprocess.run([sys.executable, "-c", _EM_RETRY_SCRIPT, ROOT, str(out), str(v_hot), adaptive], env=env, check=True, timeout=600)
        return torch.load(out)

    a, b = run("1", 1400.0), run("0", 1400.0)
    assert torch.isfinite(a).all() and torch.equal(a, b)
    c, d = run("1", 4.0), run("0", 4.0)
    assert not torch.equal(c, d)
    assert float((c - d).abs().max()) <= (2e-4 if adaptive == "1" else 2e-6) * float(d.abs().max())


_DP_SRK_RETRY_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
import odecol
cfg = odecol.load_config(sys.argv[1] + "/config/model.toml")
B, cols = 5, 32
N = 8 * cols
sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=0, device="cuda")
gen = torch.Generator().manual_seed(5)
amp = torch.rand(B, cols, generator=gen) * 30.0
kt, ku = odecol.step_knots(0.002, 0.006, 0.01, amp, 1e-3)
sheet.set_knots(kt.cuda(), ku.cuda())
ts = torch.linspace(0.0, 0.01, 6).cuda()
y0 = torch.cat((torch.rand(B, N, generator=gen) * 6 - 8, torch.rand(B, N, generator=gen), torch.rand(B, N, generator=gen) * 2), 1)
out = {}
for tag, v_hot in (("hot", 1400.0), ("plain", 4.0)):
    y0[:, 3] = v_hot
    st = {}
    with torch.no_grad():
        out["dopri5_" + tag] = odecol.odeint(sheet, y0.cuda(), ts, rtol=1e-5, atol=1e-6, stats=st).cpu()      # N = 256: staged family
        out["srk_" + tag] = odecol.sdeint(sheet, y0.cuda(), ts, method="srk", dt=1e-4, seed=3,
                                          options={"sigma_scale": torch.full((B,), 0.1)}).cpu()
    out["n_accept_" + tag] = st["n_accept"].cpu()
torch.save(out, sys.argv[2])
"""


def test_staged_dopri5_and_srk_repeat_in_tf32_when_fp16_cannot_hold_the_operand(tmp_path):
    """The drift contractions of the staged srk forward solve and of the forward-only staged dopri5 solve (no record: training
    keeps TF32 pairs) read FP16 pairs as well (stage_em.cu: dopri5_fwd_impl, srk_fwd_impl); same overflow protocol and same
    criterion as for Euler-Maruyama above."""
    import subprocess
    import sys

    def run(f16):
        out = tmp_path / f"d_{f16}.pt"
        env = dict(os.environ, ODECOL_DP16=f16, ODECOL_SRK16=f16)
        subprocess.run([sys.executable, "-c", _DP_SRK_RETRY_SCRIPT, ROOT, str(out)], env=env, check=True, timeout=600)
        return torch.load(out)

    a, b = run("1"), run("0")
    for k in ("dopri5_hot", "srk_hot", "n_accept_hot"):
        assert torch.isfinite(a[k].float()).all() and torch.equal(a[k], b[k]), k
    for k, bar in (("dopri5_plain", 5e-4), ("srk_plain", 1e-5)):        # srk: 100 noisy steps, F components of a few hundred
        assert not torch.equal(a[k], b[k]), k
        assert float((a[k] - b[k]).abs().max()) <= bar * float(b[k].abs().max()), k
    assert float((a["n_accept_plain"] - b["n_accept_plain"]).abs().max()) <= 2


# ----------------------------------------------------------------------------------------------------------------------
# adaptive Euler-Maruyama vs the oracle's step-doubling loop
# ----------------------------------------------------------------------------------------------------------------------
class _NoBrownian:
    shape = (1, 1)

    def __call__(self, t0, t1):
        return torch.zeros(1, 1)


def _oracle_adaptive(lf, kt, ku, ts, y0, sigma_scale, bms, rtol, atol, dt, dt_min):
    """One adaptive solve per trial, as the reference runs them (B = 1 per sdeint call)."""
    ys, na, nr = [], [], []
    for b in range(y0.shape[0]):
        lfb = lf
        if sigma_scale is not None:
            import dataclasses
            lfb = dataclasses.replace(lf, sigma=(lf.sigma * float(sigma_scale[b])).astype(np.float32))
        ode = orhs.UnifiedColumnODE(lfb, kt.numpy(), ku[b:b + 1].numpy() if ku.shape[0] > 1 else ku.numpy())
        st = {}
        with torch.no_grad():
            y = S.sdeint_euler(ode, y0[b:b + 1], ts, bms[b], dt=dt, adaptive=True, rtol=rtol, atol=atol, dt_min=dt_min, stats=st)
        ys.append(y)
        na.append(st["n_accept"]); nr.append(st["n_reject"])
    return torch.cat(ys, 1), np.array(na), np.array(nr)


def _adaptive_case(kind, cfg, golden):
    gen = torch.Generator().manual_seed(11)
    if kind == "xor":                                         # on-chip family, the reference's XOR network
        net = product_network("xor", cfg, golden["xor"], DEV)
        lf = oracle_form("xor", cfg, golden["xor"])
        B, N = 4, 24
        amp = torch.tensor([[20.0, 0.0], [0.0, 20.0], [20.0, 20.0], [0.0, 0.0]])
        u = torch.zeros(B, 2, 16)
        u[:, 0, 2] = u[:, 0, 3] = amp[:, 0]; u[:, 1, 10] = u[:, 1, 11] = amp[:, 1]
        kt = torch.tensor([0.0, 0.01, 0.0101, 1.0])
        ku = torch.stack((torch.zeros(B, 32), torch.zeros(B, 32), u.reshape(B, 32), u.reshape(B, 32)), 1)
        net.time_vec, net.stim = kt.to(DEV), ku.reshape(B, 4, 2, 16).to(DEV)
        ts = torch.linspace(0.0, 0.06, 7)
        options = {}
    else:                                                     # staged family: 32-column sheet, N = 256
        net = odecol.SyntheticColumnSheet(cfg, 32, seed=3, device=DEV, sigma_v=4.0)
        lf = sheet_oracle_form(net)
        B, N = 3, 256
        amp = torch.rand(B, 32, generator=gen) * 25
        kt, ku = odecol.step_knots(1e-3, 5e-3, 8e-3, amp, 1e-4)
        net.set_knots(kt.to(DEV), ku.to(DEV))
        ts = torch.linspace(0.0, 6e-3, 5)
        options = {}
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 4 - 6, torch.rand(B, N, generator=gen) * 0.5,
                    torch.rand(B, N, generator=gen)), 1)
    return net, lf, kt, ku, ts, y0, B, options


@pytest.mark.parametrize("noise", [False, True], ids=["deterministic", "same_brownian_path"])
@pytest.mark.parametrize("kind", ["xor", "sheet256"])
def test_adaptive_euler_maruyama_matches_the_oracle_controller(kind, noise, cfg, golden):
    """What can and cannot agree.  torchsde's error estimate is the difference of the full step and the two half steps, two
    nearly equal float32 states: at rtol 1e-5 / atol 1e-4 (about 30 float32 ulps of a state of magnitude 10) the last-ulp
    differences between any two float32 implementations of phi (torch's tanh / exp on the CPU, tanhf / expf or the fast
    path on the GPU) move the estimate by ~1 %, the step factor by a few 1e-3, and the two solvers walk slightly different
    -- equally valid -- time grids from the first steps on (the reference run on another machine would, too).  Their
    results then differ at the level of the solve's own discretisation error, not of float32 rounding.  Hence:
      * a SHORT solve (~20 attempts): accept / reject counts within one step, and without noise V and A within 2e-5
        (F, whose filter has |1 - h / tau_s| ~ 1 at these steps, within 5e-4);
      * the LONG solve: accepted / rejected counts per trial +-3 without noise, 3 % / 20 % with noise (the Brownian
        increments make the estimate rough), outputs within 5e-4 / 1e-3, and without noise the product must be as close to a
        converged float64 solution as the oracle is -- the criterion that a wrong controller cannot meet."""
    net, lf, kt, ku, ts, y0, B, options = _adaptive_case(kind, cfg, golden)
    ts = torch.linspace(0.0, float(ts[-1]), 61 if kind == "xor" else 13)
    rtol, atol, dt, dt_min = 1e-5, 1e-4, 1e-3, 1e-5
    seed, trial_offset = 77, 5
    sc = torch.tensor([0.0] * B) if not noise else torch.tensor([0.05, 0.1, 0.2, 0.15][:B])
    N = y0.shape[1] // 3
    blk = lambda a, c: a[..., c * N:(c + 1) * N]

    def both(tgrid):
        bms = [(TreeBrownian(seed, trial_offset + b, tgrid[0], tgrid[-1]) if noise else _NoBrownian()) for b in range(B)]
        yo_, nao_, nro_ = _oracle_adaptive(lf, kt, ku, tgrid, y0, sc.numpy(), bms, rtol, atol, dt, dt_min)
        st_ = {}
        with torch.no_grad():
            yp_ = odecol.sdeint(net, y0.to(DEV), tgrid.to(DEV), method="euler", dt=dt, adaptive=True, rtol=rtol, atol=atol,
                                dt_min=dt_min, seed=seed, trial_offset=trial_offset, stats=st_,
                                options=dict(options, sigma_scale=sc))
        torch.cuda.synchronize()
        assert int(st_["status"].abs().sum()) == 0
        return yp_.cpu(), yo_, st_["n_accept"].cpu().numpy(), st_["n_reject"].cpu().numpy(), nao_, nro_

    # ---- short solve
    yp, yo, na, nr, nao, nro = both(torch.linspace(0.0, 3e-4, 3))
    errs = [_relmax(blk(yp, c), blk(yo, c)) for c in range(3)]
    print(f"\n[adaptive EM {kind} noise={noise}] short solve: accepted {na.tolist()} vs oracle {nao.tolist()}, rejected {nr.tolist()} vs "
          f"{nro.tolist()}; V/A/F {errs[0]:.1e} {errs[1]:.1e} {errs[2]:.1e}")
    assert np.all(np.abs(na - nao) <= 1) and np.all(np.abs(nr - nro) <= 1) and int((na + nr).min()) >= 3
    if not noise:
        assert max(errs[:2]) < 2e-5 and errs[2] < 5e-4
    # ---- long solve
    yp, yo, na, nr, nao, nro = both(ts)
    errs = [_relmax(blk(yp, c), blk(yo, c)) for c in range(3)]
    print(f"[adaptive EM {kind} noise={noise}] accepted {na.tolist()} vs oracle {nao.tolist()}; rejected {nr.tolist()} vs "
          f"{nro.tolist()}; outputs V/A/F {errs[0]:.1e} {errs[1]:.1e} {errs[2]:.1e}")
    assert nao.min() > 10                                        # the controller really ran (not parked at one step)
    if noise:
        # rejections are the small, noisy count: an attempt whose error estimate sits at the tolerance flips with the last bits
        # of the drift (TF32 pairs: 43 rejections on one sheet trial, FP16 pairs: 50, oracle: 42 -- same accepted steps +-1 %)
        assert np.all(np.abs(na - nao) <= 0.03 * nao + 2) and np.all(np.abs(nr - nro) <= 0.2 * nro + 3)
        assert max(errs) < 1e-3
    else:
        assert np.all(np.abs(na - nao) <= 3) and np.all(np.abs(nr - nro) <= 3)
        assert max(errs) < 5e-4
        # converged solution: float64 Euler with a step far below what the controller picks
        ode64 = orhs.UnifiedColumnODE(lf, kt.numpy(), ku.numpy(), dtype=torch.float64)
        with torch.no_grad():
            yt = S.sdeint_euler(ode64, y0.double(), ts.double(), lambda a, b: torch.zeros(B, 1, dtype=torch.float64), dt=2e-6)
        for c in range(3):
            ep, eo = _relmax(blk(yp.double(), c), blk(yt, c)), _relmax(blk(yo.double(), c), blk(yt, c))
            print(f"    block {c}: distance to the converged solution: product {ep:.2e}, oracle {eo:.2e}")
            assert ep < 1.25 * eo + 2e-5


# ----------------------------------------------------------------------------------------------------------------------
# C5: one drift evaluation at N = 8192
# ----------------------------------------------------------------------------------------------------------------------
def test_c5_drift_evaluation_matches_the_float64_oracle(cfg):
    cols, N, B = 1024, 8192, 300
    sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=0, device=DEV)
    gen = torch.Generator().manual_seed(5)
    amp = torch.rand(B, cols, generator=gen) * 30.0
    kt = torch.tensor([0.0, 1.0])
    ku = torch.stack((amp, amp * 0.5), 1)                        # a ramp: the lookup interpolates
    tq = torch.rand(B, generator=gen)
    y = torch.cat((torch.rand(B, N, generator=gen) * 10 - 8, torch.rand(B, N, generator=gen) * 2,
                   torch.rand(B, N, generator=gen) * 3), 1)
    ext = odecol._native.ext()
    lfp = sheet.export_linear_form()
    prob = ext.Problem(lfp.W_aug.detach().contiguous(), lfp.kappa.contiguous(), lfp.sigma.contiguous(), kt.to(DEV), ku.to(DEV),
                       lfp.n_in, B, lfp.tau_s, lfp.tau_m, lfp.tau_a, lfp.resistance, 0)
    f = ext.drift_staged(prob, tq.to(DEV), y.to(DEV)).cpu()
    torch.cuda.synchronize()
    ode = orhs.UnifiedColumnODE(sheet_oracle_form(sheet), kt.numpy(), ku.numpy(), dtype=torch.float64)
    fo = ode.forward(tq.double(), y.double())
    # error scale of the V slope: the contraction's sum |w||r| times tau_s R / tau_m, plus |V| / tau_m
    r = orhs.phi(y[:, :N].double() - y[:, N:2 * N].double())
    s = orhs.interp_knots(tq.double(), ode.knot_t, ode.knot_u)
    mag = (r.abs() @ ode.W.abs().T + s.abs() @ ode.U.abs().T + ode.bias.abs()) * float(ode.tau_s * ode.R / ode.tau_m) \
        + y[:, :N].double().abs() / float(ode.tau_m)
    eV = float(((f[:, :N].double() - fo[:, :N]).abs() / mag).max())
    eA = _relmax(f[:, N:2 * N].double(), fo[:, N:2 * N]); eF = _relmax(f[:, 2 * N:].double(), fo[:, 2 * N:])
    print(f"\n[C5 drift N={N} B={B}] dV err / (sum|w||r| scale) {eV:.2e}; dA {eA:.1e}; dF {eF:.1e}; "
          f"dV rel to max|dV| {_relmax(f[:, :N].double(), fo[:, :N]):.1e}")
    assert eV < 4e-6 and eA < 2e-6 and eF < 2e-6


@pytest.mark.parametrize("gain", [False, True], ids=["plain", "lateral_gain"])
@pytest.mark.parametrize("cols,B", [(1024, 300), (125, 37)], ids=["N8192", "N1000"])
def test_c5_sweep_drift_in_fp16_pairs_matches_the_float64_oracle(cfg, cols, B, gain):
    """The drift the C5 sweep runs: FP16 operand pairs (ODECOL_EM16, on by default), chunked contraction (K_aug = 9217 /
    1126), per-member lateral gain -- reached through the public sdeint.  One Euler-Maruyama step of h = 1 without noise
    writes y[1] = y0 + f rounded once, so y[1] - y0 is the drift to ~1e-7.  N = 8192 with B = 300 leaves the last trial tile
    ragged; N = 1000 pads the last population tile.  The stimulus ramp's knots straddle t = 0, where the step evaluates."""
    N = 8 * cols
    sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=0, device=DEV)
    gen = torch.Generator().manual_seed(cols + int(gain))
    amp = torch.rand(B, cols, generator=gen) * 30.0
    kt = torch.tensor([-0.25, 0.75])
    ku = torch.stack((amp, amp * 0.5), 1)
    sheet.set_knots(kt.to(DEV), ku.to(DEV))
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 10 - 8, torch.rand(B, N, generator=gen) * 2,
                    torch.rand(B, N, generator=gen) * 3), 1).to(DEV)
    g = torch.ones(B, dtype=torch.float64)
    options = {}
    if gain:
        g = torch.rand(B, generator=gen).double() + 0.5
        g[B // 3] = 1.0
        options = {"lateral_gain": g.float()}
    with torch.no_grad():
        ys = odecol.sdeint(sheet, y0, torch.tensor([0.0, 1.0], device=DEV), bm=torch.zeros(1, B), method="euler", dt=1.0,
                           options=dict(options))
        # the same inputs through odecol_drift_staged, which evaluates in TF32 pairs
        from ode_column_b200.solvers import _Setup
        setup = _Setup(sheet, y0, torch.tensor([0.0, 1.0], device=DEV), None)
        if gain:
            setup.set_lateral_gain(sheet, options["lateral_gain"])
        f32 = odecol._native.ext().drift_staged(setup.problem(setup.lf.W_aug), torch.zeros(B, device=DEV), y0)
        y1_tf32 = y0 + f32
    torch.cuda.synchronize()
    assert torch.equal(ys[0], y0)
    f = ys[1].double() - y0.double()
    # float64 oracle (on the device, as plain torch): g_b (W_lat r) + W_loc (*) r + U s + bias
    lf = sheet_oracle_form(sheet)
    W_lat, W_loc = (x.detach().double() for x in sheet.lateral_split())
    U, bias = torch.tensor(lf.U, dtype=torch.float64, device=DEV), torch.tensor(lf.bias, dtype=torch.float64, device=DEV)
    kappa = torch.tensor(lf.kappa, dtype=torch.float64, device=DEV)
    yd = y0.double()
    V, A, F = yd[:, :N], yd[:, N:2 * N], yd[:, 2 * N:]
    r = orhs.phi(V - A)
    s = orhs.interp_knots(torch.tensor(0.0, dtype=torch.float64), kt.double(), ku.double()).to(DEV)
    gd = g.to(DEV)[:, None]
    loc = lambda W8, x: torch.einsum("cpj,bcj->bcp", W8.reshape(cols, 8, 8), x.reshape(B, cols, 8)).reshape(B, N)
    cur = gd * (r @ W_lat.T) + loc(W_loc, r) + s @ U.T + bias
    c = lf.tau_s * lf.resistance / lf.tau_m
    fo = torch.cat(((cur * lf.tau_s * lf.resistance - V) / lf.tau_m, (kappa * r - A) / lf.tau_a, (r - F) / lf.tau_s), 1)
    mag = (gd * (r.abs() @ W_lat.abs().T) + loc(W_loc.abs(), r.abs()) + s.abs() @ U.abs().T + bias.abs()) * c + V.abs() / lf.tau_m
    eV = float(((f[:, :N] - fo[:, :N]).abs() / mag).max())
    eA, eF = _relmax(f[:, N:2 * N], fo[:, N:2 * N]), _relmax(f[:, 2 * N:], fo[:, 2 * N:])
    d16 = float((ys[1] - y1_tf32).abs().max()) / _scale(fo)
    print(f"\n[C5 sweep drift, FP16 pairs, N={N} B={B} gain={gain}] dV err / (sum|w||r| scale) {eV:.2e}; dA {eA:.1e}; "
          f"dF {eF:.1e}; FP16 vs TF32 pairs {d16:.1e} of max|f|")
    assert eV < 4e-6 and eA < 2e-6 and eF < 2e-6
    assert not torch.equal(ys[1], y1_tf32)                     # the FP16 contraction is the one that ran


# ----------------------------------------------------------------------------------------------------------------------
# C5: the per-member global lateral gain (third sweep axis)
# ----------------------------------------------------------------------------------------------------------------------
def test_lateral_gain_sweep_axis_matches_per_member_networks(cfg):
    """options['lateral_gain']: trial b integrates the sheet whose between-column weights are gain[b] times the module's.
    Oracle: one network per member with W = W_local + gain[b] * W_lateral, Euler-Maruyama on supplied increments."""
    import dataclasses
    sheet = odecol.SyntheticColumnSheet(cfg, 32, seed=4, device=DEV, sigma_v=3.0)
    B, N, T = 5, 256, 17
    gen = torch.Generator().manual_seed(21)
    gain = torch.tensor([0.25, 0.5, 1.0, 2.0, 3.5])
    amp = torch.rand(B, 32, generator=gen) * 25
    kt, ku = odecol.step_knots(5e-4, 2.5e-3, 4e-3, amp, 1e-4)
    sheet.set_knots(kt.to(DEV), ku.to(DEV))
    ts = torch.linspace(0.0, 3.2e-3, T)
    dt = 2e-4
    n_steps = len(S.em_step_schedule(ts, dt))
    W_inc = torch.randn(n_steps, B, 1, generator=gen) * dt ** 0.5
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 4 - 6, torch.rand(B, N, generator=gen) * 0.5, torch.rand(B, N, generator=gen)), 1)
    lf = sheet_oracle_form(sheet)
    W_lat, W_loc = (x.detach().cpu() for x in sheet.lateral_split())
    W_loc_dense = torch.tensor(lf.W) - W_lat
    assert float((W_loc_dense.reshape(32, 8, 32, 8)[torch.arange(32), :, torch.arange(32), :].reshape(N, 8) - W_loc).abs().max()) == 0
    ys = []
    for b in range(B):
        lfb = dataclasses.replace(lf, W=(W_loc_dense + float(gain[b]) * W_lat).numpy())
        ode = orhs.UnifiedColumnODE(lfb, kt.numpy(), ku[b:b + 1].numpy())
        with torch.no_grad():
            ys.append(S.sdeint_euler(ode, y0[b:b + 1], ts, S.TabulatedBrownian(W_inc[:, b:b + 1]), dt=dt))
    yo = torch.cat(ys, 1)
    with torch.no_grad():
        yp = odecol.sdeint(sheet, y0.to(DEV), ts.to(DEV), bm=W_inc[:, :, 0], method="euler", dt=dt,
                           options={"lateral_gain": gain}).cpu()
        yp1 = odecol.sdeint(sheet, y0.to(DEV), ts.to(DEV), bm=W_inc[:, :, 0], method="euler", dt=dt, options={"family": "staged"}).cpu()
    errs = [_relmax(yp[..., c * N:(c + 1) * N], yo[..., c * N:(c + 1) * N]) for c in range(3)]
    print(f"\n[lateral gain sweep, N={N}] V/A/F vs per-member oracle networks {errs[0]:.1e} {errs[1]:.1e} {errs[2]:.1e}; "
          f"gain 1 member vs the plain solve {_relmax(yp[:, 2], yp1[:, 2]):.1e}; gain 0.25 vs 3.5 differ by {_relmax(yp[:, 0, :N], yp[:, 4, :N]):.2f}")
    assert max(errs) < 1e-5
    assert _relmax(yp[:, 2], yp1[:, 2]) < 2e-6            # gain 1 reproduces the unsplit network
    # adaptive mode takes the gain too, and refuses what it cannot honour
    st = {}
    with torch.no_grad():
        ya = odecol.sdeint(sheet, y0.to(DEV), ts.to(DEV), method="euler", adaptive=True, seed=3, stats=st,
                           options={"lateral_gain": gain, "sigma_scale": torch.full((B,), 0.1)})
    assert torch.isfinite(ya).all() and int(st["n_accept"].min()) > 3
    with torch.no_grad():
        with pytest.raises(ValueError):
            odecol.sdeint(sheet, y0.to(DEV), ts.to(DEV), method="euler", options={"lateral_gain": torch.zeros(B)})
        with pytest.raises(NotImplementedError):
            odecol.sdeint(sheet, y0.to(DEV), ts.to(DEV), method="srk", options={"lateral_gain": gain})
    with pytest.raises(NotImplementedError):                  # a sweep feature: no reverse sweep through the gain
        odecol.sdeint(sheet, y0.to(DEV), ts.to(DEV), method="euler", options={"lateral_gain": gain})


# ----------------------------------------------------------------------------------------------------------------------
# dopri5 + loss.backward() beyond the on-chip family (the reference's default training path, scripts/xor_ode.py:114,177)
# ----------------------------------------------------------------------------------------------------------------------
def test_staged_dopri5_adjoint_matches_oracle_autograd(cfg):
    """N = 256 sheet: odeint(default method).backward() through the staged reverse sweep against autograd through the
    oracle's dopri5 (one solve per trial: torchdiffeq controls the step over the whole tensor of a B = 1 solve)."""
    sheet = odecol.SyntheticColumnSheet(cfg, 32, seed=6, device=DEV)
    B, N, T = 4, 256, 9
    gen = torch.Generator().manual_seed(31)
    amp = torch.rand(B, 32, generator=gen) * 25
    amp[3] *= 0.1                                              # a quiet trial: fewer accepted steps than the others
    kt, ku = odecol.step_knots(2e-3, 8e-3, 1.2e-2, amp, 5e-4)
    sheet.set_knots(kt.to(DEV), ku.to(DEV))
    tv = torch.linspace(0.0, 1e-2, T)
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 4 - 6, torch.rand(B, N, generator=gen) * 0.5, torch.rand(B, N, generator=gen)), 1)
    sel = list(range(0, N, 8)) + [N + 8 * k for k in range(32)] + [2 * N + 5]
    wgt = torch.randn(T, B, len(sel), generator=gen)
    rtol, atol = 1e-6, 1e-8
    lf = sheet_oracle_form(sheet)
    gW = gU = None
    trs, g0s, nacc_o = [], [], []
    for b in range(B):
        ode = orhs.UnifiedColumnODE(lf, kt.numpy(), ku[b:b + 1].numpy(), requires_grad=True)
        y0o = y0[b:b + 1].clone().requires_grad_(True)
        st = {}
        yo = S.odeint_dopri5(ode, y0o, tv, rtol=rtol, atol=atol, stats=st)
        (yo[:, :, sel] * wgt[:, b:b + 1]).sum().backward()
        trs.append(yo[:, :, sel].detach()); g0s.append(y0o.grad); nacc_o.append(st["n_accept"])
        gW = ode.W.grad if gW is None else gW + ode.W.grad
        gU = ode.U.grad if gU is None else gU + ode.U.grad
    tro, g0o = torch.cat(trs, 1), torch.cat(g0s, 0)
    y0p = y0.to(DEV).requires_grad_(True)
    stp = {}
    yp = odecol.odeint(sheet, y0p, tv.to(DEV), rtol=rtol, atol=atol, components=sel, stats=stp)
    (yp * wgt.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    et = _relmax(yp.detach().cpu(), tro)
    e0, eW, eU = _relmax(y0p.grad.cpu(), g0o), _relmax(sheet.recurrent_weights.grad.cpu(), gW), _relmax(sheet.input_weights.grad.cpu(), gU)
    print(f"\n[staged dopri5 adjoint N={N}] accepted {stp['n_accept'].tolist()} vs oracle {nacc_o}; trajectory {et:.1e}  dy0 {e0:.1e}  "
          f"dW {eW:.1e}  dU {eU:.1e}")
    assert np.all(np.abs(stp["n_accept"].cpu().numpy() - np.array(nacc_o)) <= 0.1 * np.array(nacc_o) + 2)
    assert et < 2e-4 and e0 < 1e-3 and eW < 1e-3 and eU < 1e-3     # two rtol = 1e-6 solves on step sequences that differ by one step
    assert len(set(stp["n_accept"].tolist())) > 1              # trials really ran different numbers of rounds


# ----------------------------------------------------------------------------------------------------------------------
# adaptive srk (the reference's "avoid the artefacts" option, scripts/parity_ode.py:234) on the Levy-area-consistent tree
# ----------------------------------------------------------------------------------------------------------------------
class _LevyTreeBrownian:
    """bm(t0, t1, return_U=True) for the oracle from odecol_brownian_levy_query: the path the adaptive srk kernel sees."""

    def __init__(self, seed, trial, t_begin, t_end):
        self.ext = odecol._native.ext()
        self.seed, self.trial, self.t_begin, self.t_end = seed, trial, float(t_begin), float(t_end)
        self.shape = (1, 1)

    def __call__(self, t0, t1, return_U=False):
        q = torch.tensor([float(t0), float(t1)], dtype=torch.float32, device=DEV)
        w, iw = (x.cpu() for x in self.ext.brownian_levy_query(self.seed, self.trial, 1, self.t_begin, self.t_end, q))
        W = (w[1] - w[0]).float().reshape(1, 1)
        if not return_U:
            return W
        h = float(q[1].cpu()) - float(q[0].cpu())
        return W, (iw[1] - iw[0] - h * w[0]).float().reshape(1, 1)


def test_levy_tree_gives_w_and_u_with_the_right_law_and_is_consistent():
    ext = odecol._native.ext()
    B, span = 20000, 0.8
    # consistency on sub-intervals is exact by construction (cumulative W and int W): check the law of (W, U) of steps
    for a, b in ((0.0, 0.8), (0.1, 0.1007), (0.3, 0.55), (0.7999, 0.8)):
        q = torch.tensor([a, b], dtype=torch.float32, device=DEV)
        w, iw = ext.brownian_levy_query(11, 0, B, 0.0, span, q)
        h = float(q[1] - q[0])
        W = (w[1] - w[0]).cpu().numpy()
        U = (iw[1] - iw[0] - h * w[0]).cpu().numpy()
        vW, vU, cWU = W.var(), U.var(), np.mean(W * U)
        print(f"\n[levy tree] step [{a}, {b}]: var W / h {vW / h:.3f}, var U / (h^3/3) {vU / (h ** 3 / 3):.3f}, cov / (h^2/2) {cWU / (h * h / 2):.3f}, "
              f"means {W.mean() / h ** 0.5:+.3f} {U.mean() / h ** 1.5:+.3f}")
        assert abs(vW / h - 1) < 0.04 and abs(vU / (h ** 3 / 3) - 1) < 0.05 and abs(cWU / (h * h / 2) - 1) < 0.05
        assert abs(W.mean()) < 0.03 * h ** 0.5 and abs(U.mean()) < 0.03 * h ** 1.5
    # chaining: U(a, c) = U(a, b) + U(b, c) + (c - b) W(a, b), W additive
    q = torch.tensor([0.2, 0.2004, 0.2011], dtype=torch.float32, device=DEV)
    w, iw = (x.cpu().double() for x in ext.brownian_levy_query(11, 0, 64, 0.0, span, q))
    t = q.cpu().double()
    Ust = lambda i, j: iw[j] - iw[i] - (t[j] - t[i]) * w[i]
    assert float((Ust(0, 2) - (Ust(0, 1) + Ust(1, 2) + (t[2] - t[1]) * (w[1] - w[0]))).abs().max()) < 1e-12
    # different trials and seeds are different paths; the same key reproduces
    w2, _ = ext.brownian_levy_query(11, 0, 64, 0.0, span, q)
    w3, _ = ext.brownian_levy_query(12, 0, 64, 0.0, span, q)
    assert torch.equal(w2.cpu().double(), w) and not torch.equal(w3.cpu().double(), w)


@pytest.mark.parametrize("noise", [False, True], ids=["deterministic", "same_brownian_path"])
def test_adaptive_srk_matches_the_oracle(noise, cfg, golden):
    """sdeint(method='srk', adaptive=True) on the parity network (the call of scripts/parity_ode.py:234) against the
    oracle's step-doubling srk on the same Levy tree, trial by trial; criteria as for adaptive Euler-Maruyama."""
    net = product_network("parity", cfg, golden["parity"], DEV)
    lf = oracle_form("parity", cfg, golden["parity"])
    B, N = 3, 104
    gen = torch.Generator().manual_seed(17)
    kt = torch.tensor([0.0, 0.005, 0.0051, 1.0])
    amp = torch.tensor([[15.0, 0, 15.0, 0], [0, 15.0, 15.0, 15.0], [15.0, 15.0, 15.0, 15.0]])
    ku = torch.stack((torch.zeros(B, 4), torch.zeros(B, 4), amp, amp), 1)
    net.time_vec, net.stim = kt.to(DEV), ku.to(DEV)
    ts = torch.linspace(0.0, 0.03, 16)
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 4 - 6, torch.rand(B, N, generator=gen) * 0.5, torch.rand(B, N, generator=gen)), 1)
    rtol, atol, dt, dt_min = 1e-5, 1e-4, 1e-3, 1e-5
    seed, off = 5, 40
    sc = torch.tensor([0.0] * B) if not noise else torch.tensor([0.02, 0.05, 0.1])
    import dataclasses
    ys, nao, nro = [], [], []
    for b in range(B):
        lfb = dataclasses.replace(lf, sigma=(lf.sigma * float(sc[b])).astype(np.float32))
        ode = orhs.UnifiedColumnODE(lfb, kt.numpy(), ku[b:b + 1].numpy())
        so = {}
        with torch.no_grad():
            ys.append(S.sdeint_srk(ode, y0[b:b + 1], ts, _LevyTreeBrownian(seed, off + b, ts[0], ts[-1]), dt=dt, adaptive=True,
                                   rtol=rtol, atol=atol, dt_min=dt_min, stats=so))
        nao.append(so["n_accept"]); nro.append(so["n_reject"])
    yo, nao, nro = torch.cat(ys, 1), np.array(nao), np.array(nro)
    st = {}
    with torch.no_grad():
        yp = odecol.sdeint(net, y0.to(DEV), ts.to(DEV), method="srk", dt=dt, adaptive=True, rtol=rtol, atol=atol, dt_min=dt_min,
                           seed=seed, trial_offset=off, stats=st, options={"sigma_scale": sc}).cpu()
    na, nr = st["n_accept"].cpu().numpy(), st["n_reject"].cpu().numpy()
    blk = lambda a, c: a[..., c * N:(c + 1) * N]
    errs = [_relmax(blk(yp, c), blk(yo, c)) for c in range(3)]
    print(f"\n[adaptive srk parity noise={noise}] accepted {na.tolist()} vs oracle {nao.tolist()}; rejected {nr.tolist()} vs {nro.tolist()}; "
          f"outputs V/A/F {errs[0]:.1e} {errs[1]:.1e} {errs[2]:.1e}")
    assert nao.min() > 10
    assert np.all(np.abs(na - nao) <= 0.05 * nao + 3) and np.all(np.abs(nr - nro) <= 0.2 * nro + 3)
    if noise:
        # outputs are LINEAR interpolations between the solver states around each output time (torchsde), so two step
        # sequences on the same path differ by the path's excursion inside a step: ~ sigma sqrt(h) per component
        h_mean = float(ts[-1]) / float(nao.min())
        sig = torch.tensor(lf.sigma) * float(sc.max())
        for c in range(3):
            bound = 3.0 * float(blk(sig, c).max()) * h_mean ** 0.5 / _scale(blk(yo, c)) + 1e-3
            assert errs[c] < bound, (c, errs[c], bound)
    else:
        assert max(errs) < 5e-4
        ode64 = orhs.UnifiedColumnODE(lf, kt.numpy(), ku.numpy(), dtype=torch.float64)
        with torch.no_grad():
            yt = S.odeint_rk4(ode64, y0.double(), torch.linspace(0.0, 0.03, 15 * 400 + 1, dtype=torch.float64))[::400]
        for c in range(3):
            ep, eo = _relmax(blk(yp.double(), c), blk(yt, c)), _relmax(blk(yo.double(), c), blk(yt, c))
            print(f"    block {c}: distance to the converged solution: product {ep:.2e}, oracle {eo:.2e}")
            assert ep < 1.25 * eo + 2e-5
    # larger networks have no fused adaptive srk
    sheet = odecol.SyntheticColumnSheet(cfg, 32, seed=1, device=DEV)
    sheet.set_knots(torch.tensor([0.0, 1.0], device=DEV), torch.zeros(1, 2, 32, device=DEV))
    with torch.no_grad(), pytest.raises(NotImplementedError):
        odecol.sdeint(sheet, torch.zeros(1, 768, device=DEV), ts.to(DEV), method="srk", adaptive=True)


def test_tensor_family_gradients_are_bit_reproducible(cfg):
    """options={'deterministic': True}: the reverse sweep reduces dW_aug over trials in a fixed order (per-split copies
    summed at the end) instead of float atomics: two runs give identical bits."""
    sheet, kt, ku, tv, y0, gen = _c4_problem(cfg, 600, 8, seed=3)
    sel = list(range(0, 512, 8)) + list(range(512, 1024, 8))
    wgt = torch.randn(8, 600, len(sel), generator=gen).to(DEV)
    grads = []
    for _ in range(2):
        sheet.zero_grad()
        y0p = y0.to(DEV).requires_grad_(True)
        yp = odecol.odeint(sheet, y0p, tv.to(DEV), method="rk4", components=sel, options={"deterministic": True})
        (yp * wgt).sum().backward()
        grads.append((y0p.grad.clone(), sheet.recurrent_weights.grad.clone(), sheet.input_weights.grad.clone()))
    assert all(torch.equal(a, b) for a, b in zip(*grads))


def test_large_batch_rk4_of_the_parity_network_runs_on_the_tensor_cores(cfg, golden):
    """From 4096 trials the rk4 solve of a network that fits the on-chip family (N = 104) is routed to the tensor family
    (1.9x - 3.4x faster there, csrc/abi.cu::use_small_rk4): same results -- trajectories and gradients of every trial
    against the oracle, and against the on-chip kernels on a slice of the batch."""
    net = product_network("parity", cfg, golden["parity"], DEV)
    lf = oracle_form("parity", cfg, golden["parity"])
    B, N, T = 4100, 104, 12
    gen = torch.Generator().manual_seed(9)
    tv = torch.linspace(0.0, 1.1e-3, T)
    kt = torch.tensor([0.0, 3e-4, 4e-4, 1.0])
    amp = (torch.rand(B, 4, generator=gen) > 0.5).float() * 15.0
    ku = torch.stack((torch.zeros(B, 4), torch.zeros(B, 4), amp, amp), 1)
    net.time_vec, net.stim = kt.to(DEV), ku.to(DEV)
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 6 - 8, torch.rand(B, N, generator=gen), torch.rand(B, N, generator=gen)), 1)
    sel = list(range(96, 104)) + list(range(N + 96, N + 104)) + [5, N + 50, 2 * N + 7]
    wgt = torch.randn(T, B, len(sel), generator=gen)
    tro, g0o, gWo, gUo, _ = _oracle_rk4_grads(lf, kt, ku, tv, y0, sel, wgt, chunk=1025)
    ext = odecol._native.ext()
    from ode_column_b200.solvers import _Setup
    setup = _Setup(net, y0.to(DEV), tv.to(DEV), None)
    assert setup.problem(setup.lf.W_aug).kernel_family(ext.OP_RK4_FWD) == 2
    y0p = y0.to(DEV).requires_grad_(True)
    yp = odecol.odeint(net, y0p, tv.to(DEV), method="rk4", components=sel)
    assert "Ckpt" in type(yp.grad_fn).__name__
    (yp * wgt.to(DEV)).sum().backward()
    lfp = net.export_linear_form()
    g_aug = torch.autograd.grad(lfp.W_aug, [p for p in net.parameters() if p.requires_grad], torch.ones_like(lfp.W_aug), allow_unused=True)
    et = _relmax(yp.detach().cpu(), tro)
    e0 = _relmax(y0p.grad.cpu(), g0o)
    # parameter gradients through the oracle's dW, dU mapped onto the module's parameters by the same autograd graph
    net2 = product_network("parity", cfg, golden["parity"], DEV)
    net2.time_vec, net2.stim = net.time_vec, net.stim
    lf2 = net2.export_linear_form()
    gaug = torch.zeros_like(lf2.W_aug)
    gaug[:, :N] = gWo.to(DEV); gaug[:, N:N + 4] = gUo.to(DEV)
    lf2.W_aug.backward(gaug)
    errs = []
    for (n1, p1), (n2, p2) in zip(net.named_parameters(), net2.named_parameters()):
        if p1.grad is not None and p2.grad is not None and float(p2.grad.abs().max()) > 0:
            errs.append((n1, _relmax(p1.grad.cpu(), p2.grad.cpu())))
    print(f"\n[parity network, B={B}, tensor family] trajectory {et:.1e}  dy0 {e0:.1e}  parameter gradients "
          f"{[(n, f'{e:.1e}') for n, e in errs]}")
    assert et < 1e-5 and e0 < 5e-5 and all(e < 5e-5 for _, e in errs) and len(errs) >= 3
    # the same trials through the on-chip kernels (a batch below the threshold)
    with torch.no_grad():
        ys = odecol.odeint(net_slice(net, slice(0, 64)), y0[:64].to(DEV), tv.to(DEV), method="rk4", components=sel)
    assert _relmax(ys.cpu(), yp.detach().cpu()[:, :64]) < 5e-6


def net_slice(net, sl):
    import copy
    other = copy.copy(net)
    other.stim = net.stim[sl]
    return other
