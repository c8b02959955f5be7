"""Differential test on problem shapes the reference networks do not reach: every register-tile size of the on-chip
family (KP = 40 / 64 / 96 / 128), two trials per warp with and without it, more stimulus channels than lanes (the
uncached knot path), ragged batches -- rk4 forward and reverse through the extension, against the CPU oracle's autograd;
and the same problems forced through the tensor family.  dopri5 is judged against a float64 replay of
the steps its record holds (the oracle's adaptive solve takes another step sequence)."""
import numpy as np
import pytest
import torch

import odecol
from helpers import check_dopri5_against_replay, ext_problem
from oracle import rhs as orhs, solvers as S
from oracle.column_model import LinearForm

pytestmark = pytest.mark.gpu
DEV = "cuda"

#           N  n_in  B  K
SHAPES = [(8, 1, 3, 2), (16, 16, 5, 4), (16, 20, 3, 3), (8, 40, 2, 3), (40, 8, 4, 5), (72, 10, 2, 3), (120, 7, 3, 4),
          (24, 32, 1, 6)]


def _problem(N, n_in, B, K, seed):
    rng = np.random.default_rng(seed)
    W = (rng.standard_normal((N, N)) * 0.04).astype(np.float32)
    U = (rng.standard_normal((N, n_in)) * 0.02).astype(np.float32)
    bias = (rng.random(N) * 0.3).astype(np.float32)
    kappa = (rng.random(N) * 1.5).astype(np.float32)
    lf = LinearForm(W=W, U=U, bias=bias, kappa=kappa, sigma=np.zeros(3 * N, np.float32), tau_s=5e-4, tau_m=0.02, tau_a=10.0,
                    resistance=80.0)
    T = 48
    tv = np.linspace(0, (T - 1) * 1e-4, T, dtype=np.float32)
    kt = np.sort(rng.random(K).astype(np.float32)) * tv[-1] * 1.2 - 0.1 * tv[-1]      # knots partly outside the solve window
    kt = np.unique(kt)
    while len(kt) < K:
        kt = np.unique(np.append(kt, kt[-1] + 1e-4 * (1 + len(kt))).astype(np.float32))
    ku = (rng.random((B, K, n_in)) * 20).astype(np.float32)
    y0 = np.concatenate((rng.random((B, N)) * 8 - 10, rng.random((B, N)), rng.random((B, N)) * 3), 1).astype(np.float32)
    return lf, tv, kt, ku, y0


@pytest.mark.parametrize("family", [0, "tensor"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "N%d_in%d_B%d_K%d" % s)
def test_rk4_forward_and_reverse_on_random_problems(shape, family):
    N, n_in, B, K = shape
    lf, tv, kt, ku, y0 = _problem(N, n_in, B, K, seed=N * 1000 + n_in)
    ext = odecol._native.ext()
    # oracle
    ode = orhs.UnifiedColumnODE(lf, kt, ku, requires_grad=True)
    y0o = torch.tensor(y0, requires_grad=True)
    yo = S.odeint_rk4(ode, y0o, torch.tensor(tv))
    gen = torch.Generator().manual_seed(N)
    wgt = torch.randn(yo.shape, generator=gen)
    (yo * wgt).sum().backward()
    assert torch.isfinite(yo).all() and float(yo[..., :N].abs().max()) < 200
    # product, through the extension (arbitrary W_aug, not one of the module classes)
    ld = (N + n_in + 1 + 3) // 4 * 4
    W_aug = torch.zeros(N, ld)
    W_aug[:, :N] = torch.tensor(lf.W); W_aug[:, N:N + n_in] = torch.tensor(lf.U); W_aug[:, N + n_in] = torch.tensor(lf.bias)
    flags = {0: 0, "tensor": ext.FLAG_FORCE_TENSOR}[family]
    prob = ext.Problem(W_aug.to(DEV), torch.tensor(lf.kappa).to(DEV), None, torch.tensor(kt).to(DEV), torch.tensor(ku).to(DEV),
                       n_in, B, lf.tau_s, lf.tau_m, lf.tau_a, lf.resistance, flags)
    assert prob.kernel_family(ext.OP_RK4_FWD) == {0: 0, "tensor": 2}[family]
    t_dev = torch.tensor(tv).to(DEV)
    y = ext.rk4_fwd(prob, t_dev, torch.tensor(y0).to(DEV), 1)
    gy0, gW = ext.rk4_bwd(prob, t_dev, y, wgt.to(DEV).contiguous(), None)
    scale = lambda a: float(a.abs().max().clamp_min(1e-30))
    et = float((y.cpu() - yo.detach()).abs().max()) / scale(yo.detach())
    e0 = float((gy0.cpu() - y0o.grad).abs().max()) / scale(y0o.grad)
    gWo = torch.cat((ode.W.grad, ode.U.grad, ode.bias.grad[:, None]), 1)
    eW = float((gW.cpu()[:, :N + n_in + 1] - gWo).abs().max()) / scale(gWo)
    print(f"\n[{shape} family {family}] trajectory {et:.1e}  grad y0 {e0:.1e}  grad W_aug {eW:.1e}")
    assert et < 1e-5 and e0 < 5e-5 and eW < 5e-5
    assert float(gW.cpu()[:, N + n_in + 1:].abs().max()) == 0 if ld > N + n_in + 1 else True     # padding columns stay zero


#             rtol  atol  output grid: points over the 4.7 ms window
DP_GRIDS = {"defaults": (1e-7, 1e-9, 48),       # the reference's tolerances: several steps between outputs, steps without one
            "loose_dense": (1e-4, 1e-6, 189),   # several outputs inside one step (the dense-output adjoint)
            "T2": (1e-7, 1e-9, 2)}              # one output at the end


@pytest.mark.parametrize("grid", list(DP_GRIDS))
@pytest.mark.parametrize("family", [0, "staged"])
@pytest.mark.parametrize("shape", [(8, 1, 3, 2), (16, 20, 5, 3), (8, 40, 2, 3), (40, 8, 4, 5), (72, 10, 2, 3), (120, 7, 3, 4)],
                         ids=lambda s: "N%d_in%d_B%d_K%d" % s)
def test_dopri5_record_and_adjoint_against_a_float64_replay(shape, family, grid):
    """dopri5 record / reverse sweep on every on-chip tile size (KP = 40 / 64 / 96 / 128), more stimulus channels than
    lanes, ragged batches, and the same problems through the staged family, against a float64 replay of the recorded
    steps.  The last trial is quiet (stimulus x 0.1, F starting at its rest value, so no fast transient): trials accept
    different numbers of steps, so the staged reverse sweep runs ragged rounds, some with first steps and some without."""
    N, n_in, B, K = shape
    rtol, atol, T = DP_GRIDS[grid]
    lf, tv, kt, ku, y0 = _problem(N, n_in, B, K, seed=N * 31 + n_in)
    ku[-1] *= 0.1
    y0[-1, 2 * N:] = orhs.phi(torch.tensor(y0[-1, :N] - y0[-1, N:2 * N])).numpy()
    tv = np.linspace(0, tv[-1], T, dtype=np.float32)
    ext = odecol._native.ext()
    flags = {0: 0, "staged": ext.FLAG_FORCE_STAGED}[family]
    prob = ext_problem(ext, lf, kt, ku, flags)
    assert prob.kernel_family(ext.OP_DOPRI5_FWD) == {0: 0, "staged": 1}[family]
    _, na, _, out_step, _ = check_dopri5_against_replay(ext, prob, lf, kt, ku, y0, tv, rtol, atol, f"{shape} {family} {grid}",
                                                        controller=grid == "loose_dense", seed=N)
    assert len(set(na.tolist())) > 1                          # ragged rounds in the staged reverse sweep
    steps = out_step[:, 1:]
    if grid == "defaults":
        assert (np.diff(steps, axis=1) > 1).any()             # accepted steps that hold no output
    if grid == "loose_dense":
        assert (np.diff(steps, axis=1) == 0).any()            # several outputs inside one step


@pytest.mark.parametrize("method", ["srk", "euler"])
@pytest.mark.parametrize("shape", [(8, 1, 3, 2), (16, 20, 3, 3), (8, 40, 2, 3), (72, 10, 2, 3), (120, 7, 3, 4)],
                         ids=lambda s: "N%d_in%d_B%d_K%d" % s)
def test_sde_solvers_on_random_problems(shape, method):
    """srk / Euler-Maruyama with supplied increments: forward + reverse sweep on the on-chip AND the staged family."""
    N, n_in, B, K = shape
    lf, tv, kt, ku, y0 = _problem(N, n_in, B, K, seed=N * 77 + n_in)
    lf.sigma[:] = np.random.default_rng(N).random(3 * N).astype(np.float32) * 3.0
    ext = odecol._native.ext()
    tvt = torch.tensor(tv)
    dt = 2.5e-4                                             # 2.5 grid intervals per solver step: interpolated outputs
    n_steps = len(S.em_step_schedule(tvt, dt))
    gen = torch.Generator().manual_seed(N + 5)
    W, U = S.sample_w_u(n_steps, B, dt, gen)
    ode = orhs.UnifiedColumnODE(lf, kt, ku, requires_grad=True)
    y0o = torch.tensor(y0, requires_grad=True)
    if method == "srk":
        yo = S.sdeint_srk(ode, y0o, tvt, S.TabulatedBrownianU(W, U), dt=dt)
    else:
        yo = S.sdeint_euler(ode, y0o, tvt, S.TabulatedBrownian(W), dt=dt)
    wgt = torch.randn(yo.shape, generator=gen)
    (yo * wgt).sum().backward()
    ld = (N + n_in + 1 + 3) // 4 * 4
    W_aug = torch.zeros(N, ld)
    W_aug[:, :N] = torch.tensor(lf.W); W_aug[:, N:N + n_in] = torch.tensor(lf.U); W_aug[:, N + n_in] = torch.tensor(lf.bias)
    mk = lambda flags: ext.Problem(W_aug.to(DEV), torch.tensor(lf.kappa).to(DEV), torch.tensor(lf.sigma).to(DEV),
                                   torch.tensor(kt).to(DEV), torch.tensor(ku).to(DEV), n_in, B, lf.tau_s, lf.tau_m, lf.tau_a,
                                   lf.resistance, flags)
    t_dev, y0d = tvt.to(DEV), torch.tensor(y0).to(DEV)
    Wd, Ud = W[:, :, 0].contiguous().to(DEV), U[:, :, 0].contiguous().to(DEV)
    scale = lambda a: float(a.abs().max().clamp_min(1e-30))
    gWo = torch.cat((ode.W.grad, ode.U.grad, ode.bias.grad[:, None]), 1)
    if method == "srk":
        y, st, ysteps = ext.srk_fwd(mk(0), t_dev, y0d, Wd, Ud, 0, 0, dt, n_steps)
        gy0, gW = ext.srk_bwd(mk(0), t_dev, ysteps, Wd, Ud, 0, 0, wgt.to(DEV).contiguous(), None, dt)
        ys, _, yss = ext.srk_fwd(mk(ext.FLAG_FORCE_STAGED), t_dev, y0d, Wd, Ud, 0, 0, dt, n_steps)
        gy0s, gWs = ext.srk_bwd(mk(ext.FLAG_FORCE_STAGED), t_dev, yss, Wd, Ud, 0, 0, wgt.to(DEV).contiguous(), None, dt)
    else:
        y, _, _, st, ysteps = ext.em_fwd(mk(0), t_dev, y0d, Wd, 0, 0, dt, False, 0.0, 0.0, 0.0, n_steps)
        gy0, gW = ext.em_bwd(mk(0), t_dev, ysteps, wgt.to(DEV).contiguous(), None, dt)
        ys, _, _, _, yss = ext.em_fwd(mk(ext.FLAG_FORCE_STAGED), t_dev, y0d, Wd, 0, 0, dt, False, 0.0, 0.0, 0.0, n_steps)
        gy0s, gWs = ext.em_bwd(mk(ext.FLAG_FORCE_STAGED), t_dev, yss, wgt.to(DEV).contiguous(), None, dt)
    et = float((y.cpu() - yo.detach()).abs().max()) / scale(yo.detach())
    es = float((ys.cpu() - yo.detach()).abs().max()) / scale(yo.detach())
    e0 = float((gy0.cpu() - y0o.grad).abs().max()) / scale(y0o.grad)
    eW = float((gW.cpu()[:, :N + n_in + 1] - gWo).abs().max()) / scale(gWo)
    e0s = float((gy0s.cpu() - y0o.grad).abs().max()) / scale(y0o.grad)
    eWs = float((gWs.cpu()[:, :N + n_in + 1] - gWo).abs().max()) / scale(gWo)
    print(f"\n[{method} {shape}] trajectory on-chip {et:.1e} staged {es:.1e}  grad y0 {e0:.1e} / staged {e0s:.1e}  "
          f"grad W_aug {eW:.1e} / staged {eWs:.1e}")
    assert int(st.abs().sum()) == 0
    assert et < 1e-5 and es < 2e-5 and e0 < 5e-5 and eW < 5e-5 and e0s < 5e-5 and eWs < 5e-5


@pytest.mark.parametrize("method,cols", [pytest.param(m, c, id=m if c == 32 else f"{m}-N1024") for c in (32, 128) for m in ("srk", "euler")])
def test_large_network_sde_gradients_through_the_public_api(method, cols):
    """N = 256 (two population tiles, beyond the on-chip family) and N = 1024 (K_aug = 1153: chunked contractions in the
    FP16 forward solve and in the reverse sweep's VJP): sdeint(...).backward() through the staged reverse sweep against
    the oracle's autograd, with the sheet module (W, U trainable) and a component selection."""
    import os
    cfg = odecol.load_config(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "config", "model.toml"))
    sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=1, device=DEV, sigma_v=2.0)
    B, T, N = 3, 21, 8 * cols
    gen = torch.Generator().manual_seed(4)
    amp = torch.rand(B, cols, generator=gen) * 20
    kt, ku = odecol.step_knots(5e-4, 1.5e-3, 2e-3, amp, 1e-4)
    sheet.set_knots(kt.to(DEV), ku.to(DEV))
    tv = torch.linspace(0, 2e-3, T)
    dt = 2.5e-4
    n_steps = len(S.em_step_schedule(tv, dt))
    W, U = S.sample_w_u(n_steps, B, dt, gen)
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 6 - 8, torch.rand(B, N, generator=gen), torch.rand(B, N, generator=gen)), 1)
    sel = [0, 9, N - 1, N + 17, 2 * N + 3]
    wgt = torch.randn(T, B, len(sel), generator=gen)
    # oracle on the sheet's linear form
    lfp = sheet.export_linear_form()
    Wa = lfp.W_aug.detach().cpu().numpy()
    lf = LinearForm(W=Wa[:, :N], U=Wa[:, N:N + cols], bias=Wa[:, N + cols], kappa=lfp.kappa.cpu().numpy(), sigma=lfp.sigma.cpu().numpy(),
                    tau_s=lfp.tau_s, tau_m=lfp.tau_m, tau_a=lfp.tau_a, resistance=lfp.resistance)
    ode = orhs.UnifiedColumnODE(lf, kt.numpy(), ku.numpy(), requires_grad=True)
    y0o = y0.clone().requires_grad_(True)
    if method == "srk":
        yo = S.sdeint_srk(ode, y0o, tv, S.TabulatedBrownianU(W, U), dt=dt)
    else:
        yo = S.sdeint_euler(ode, y0o, tv, S.TabulatedBrownian(W), dt=dt)
    (yo[:, :, sel] * wgt).sum().backward()
    # product
    y0p = y0.to(DEV).requires_grad_(True)
    bm = (W, U) if method == "srk" else W
    yp = odecol.sdeint(sheet, y0p, tv.to(DEV), bm=bm, method=method, dt=dt, components=sel)
    (yp * wgt.to(DEV)).sum().backward()
    scale = lambda a: float(a.abs().max().clamp_min(1e-30))
    et = float((yp.detach().cpu() - yo[:, :, sel].detach()).abs().max()) / scale(yo[:, :, sel].detach())
    e0 = float((y0p.grad.cpu() - y0o.grad).abs().max()) / scale(y0o.grad)
    eW = float((sheet.recurrent_weights.grad.cpu() - ode.W.grad).abs().max()) / scale(ode.W.grad)
    eU = float((sheet.input_weights.grad.cpu() - ode.U.grad).abs().max()) / scale(ode.U.grad)
    print(f"\n[{method} N={N}] trajectory {et:.1e}  grad y0 {e0:.1e}  grad W {eW:.1e}  grad U {eU:.1e}")
    assert et < 1e-5 and e0 < 5e-5 and eW < 5e-5 and eU < 5e-5


def test_rk4_and_adjoint_on_a_long_contraction():
    """N = 1024 (K = 1153 > 768): the contraction accumulates in chunks (two accumulator sets drained into FP32 registers),
    forward and reverse sweep run one launch per stage; against the oracle's autograd."""
    import os
    cfg = odecol.load_config(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "config", "model.toml"))
    cols, N, B, T = 128, 1024, 3, 7
    sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=2, device=DEV)
    gen = torch.Generator().manual_seed(8)
    amp = torch.rand(B, cols, generator=gen) * 20
    kt, ku = odecol.step_knots(1e-4, 4e-4, 6e-4, amp, 1e-4)
    sheet.set_knots(kt.to(DEV), ku.to(DEV))
    tv = torch.linspace(0, 6e-4, T)
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 6 - 8, torch.rand(B, N, generator=gen), torch.rand(B, N, generator=gen)), 1)
    sel = list(range(0, N, 64)) + [N + 5, 2 * N + 9]
    wgt = torch.randn(T, B, len(sel), generator=gen)
    lfp = sheet.export_linear_form()
    Wa = lfp.W_aug.detach().cpu().numpy()
    lf = LinearForm(W=Wa[:, :N], U=Wa[:, N:N + cols], bias=Wa[:, N + cols], kappa=lfp.kappa.cpu().numpy(), sigma=lfp.sigma.cpu().numpy(),
                    tau_s=lfp.tau_s, tau_m=lfp.tau_m, tau_a=lfp.tau_a, resistance=lfp.resistance)
    ode = orhs.UnifiedColumnODE(lf, kt.numpy(), ku.numpy(), requires_grad=True)
    y0o = y0.clone().requires_grad_(True)
    yo = S.odeint_rk4(ode, y0o, tv)
    (yo[:, :, sel] * wgt).sum().backward()
    y0p = y0.to(DEV).requires_grad_(True)
    yp = odecol.odeint(sheet, y0p, tv.to(DEV), method="rk4", components=sel)
    assert "Ckpt" not in type(yp.grad_fn).__name__            # checkpoint mode belongs to the persistent kernel (K <= 768)
    (yp * wgt.to(DEV)).sum().backward()
    scale = lambda a: float(a.abs().max().clamp_min(1e-30))
    et = float((yp.detach().cpu() - yo[:, :, sel].detach()).abs().max()) / scale(yo[:, :, sel].detach())
    e0 = float((y0p.grad.cpu() - y0o.grad).abs().max()) / scale(y0o.grad)
    eW = float((sheet.recurrent_weights.grad.cpu() - ode.W.grad).abs().max()) / scale(ode.W.grad)
    print(f"\n[rk4 N=1024, chunked contraction] trajectory {et:.1e}  grad y0 {e0:.1e}  grad W {eW:.1e}")
    assert et < 1e-5 and e0 < 5e-5 and eW < 5e-5


@pytest.mark.parametrize("hot", [False, True], ids=["ordinary", "beyond_fp16"])
@pytest.mark.parametrize("shape", [(16, 16, 1), (8, 3, 1), (12, 16, 3), (16, 5, 2)], ids=lambda s: "N%d_in%d_every%d" % s)
def test_tensor_core_path_of_the_smallest_networks_matches_the_on_chip_kernel(shape, hot):
    """From 4096 trials on, rk4 forward solves of networks with N <= 16, n_in <= 16 run with the trials on the M axis of the
    tensor core (csrc/tiny_tc.cu, FP16 pairs).  The same trials in batches below the threshold run the on-chip kernel: the
    two must agree to float32 rounding (ragged last CTA, padded populations / channels, subsampled outputs) -- and be
    IDENTICAL when a rate does not fit FP16, because the launch sequence then repeats the solve with the on-chip kernel."""
    N, n_in, every = shape
    B, K = 4100, 4
    lf, tv, kt, ku, y0 = _problem(N, n_in, B, K, seed=7 * N + n_in)
    if hot:
        y0[::37, 3] = 1400.0                                   # phi(1400 - A) = 6.6e4
    ext = odecol._native.ext()
    ld = (N + n_in + 1 + 3) // 4 * 4
    W_aug = torch.zeros(N, ld)
    W_aug[:, :N] = torch.tensor(lf.W); W_aug[:, N:N + n_in] = torch.tensor(lf.U); W_aug[:, N + n_in] = torch.tensor(lf.bias)
    t_dev = torch.tensor(tv).to(DEV)

    gen = torch.Generator().manual_seed(3)
    n_rows = (len(tv) - 2) // every + 2 if every > 1 else len(tv)
    wgt = torch.randn(n_rows, B, 3 * N, generator=gen).to(DEV)
    grads = []

    def solve(lo, hi):
        prob = ext.Problem(W_aug.to(DEV), torch.tensor(lf.kappa).to(DEV), None, torch.tensor(kt).to(DEV),
                           torch.tensor(ku[lo:hi]).contiguous().to(DEV), n_in, hi - lo, lf.tau_s, lf.tau_m, lf.tau_a, lf.resistance, 0)
        assert prob.kernel_family(ext.OP_RK4_FWD) == 0
        assert (prob.workspace_bytes(ext.OP_RK4_FWD, len(tv), 0) > 0) == (hi - lo >= 4096)
        y = ext.rk4_fwd(prob, t_dev, torch.tensor(y0[lo:hi]).to(DEV), every)
        if every == 1 and not hot:                             # the on-chip reverse sweep on top of either forward solve
            grads.append(ext.rk4_bwd(prob, t_dev, y, wgt[:, lo:hi].contiguous(), None))
        return y

    big = solve(0, B)
    g_big = grads.pop() if grads else None
    ref = torch.cat([solve(lo, min(B, lo + 1500)) for lo in range(0, B, 1500)], 1)
    torch.cuda.synchronize()
    if g_big is not None:
        gy_ref = torch.cat([g[0] for g in grads], 0)
        gW_ref = sum(g[1] for g in grads)
        e0 = float((g_big[0] - gy_ref).abs().max() / gy_ref.abs().max())
        eW = float((g_big[1] - gW_ref).abs().max() / gW_ref.abs().max())
        print(f"\n[tiny tensor-core path {shape}] reverse sweep on its trajectory vs on the on-chip one: dy0 {e0:.1e}  dW {eW:.1e}")
        assert e0 < 2e-5 and eW < 2e-5
    assert big.shape == ref.shape and torch.isfinite(ref).all()
    if hot:
        assert torch.equal(big, ref)
        return
    errs = [float((big[..., c * N:(c + 1) * N] - ref[..., c * N:(c + 1) * N]).abs().max() / ref[..., c * N:(c + 1) * N].abs().max())
            for c in range(3)]
    print(f"\n[tiny tensor-core path {shape}] V/A/F vs the on-chip kernel {errs[0]:.1e} {errs[1]:.1e} {errs[2]:.1e}")
    assert not torch.equal(big, ref)                           # it is the other kernel that ran
    assert max(errs) < 5e-6
