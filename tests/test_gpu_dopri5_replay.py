"""dopri5 beyond the random problems: the staged family on column sheets (N = 256; N = 200, not a multiple of the
128-row population tile; N = 1024, whose contractions accumulate in chunks) against a float64 replay of the recorded steps; the public odeint entry point on the same
computation at any record capacity; inputs the dopri5 path must reject (a time grid that is not strictly increasing)
and repeated read-out components, which every solver must treat as torch.index_select does."""
import numpy as np
import pytest
import torch

import odecol
from helpers import check_dopri5_against_replay, ext_problem, product_network, sheet_oracle_form
from oracle import rhs as orhs

pytestmark = pytest.mark.gpu
DEV = "cuda"

#                rtol  atol  output grid: points over the 2 ms window
SHEET_GRIDS = {"defaults": (1e-7, 1e-9, 21),       # several steps between outputs, steps without one
               "loose_dense": (1e-4, 1e-6, 161),   # several outputs inside one step
               "T2": (1e-7, 1e-9, 2)}


def _sheet(cfg, cols, B, seed):
    """A column sheet with an on/off stimulus; the last trial is quiet (stimulus x 0.1, F starting at its rest value) and
    accepts fewer steps."""
    sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=seed, device=DEV)
    gen = torch.Generator().manual_seed(seed)
    amp = torch.rand(B, cols, generator=gen) * 25
    amp[-1] *= 0.1
    kt, ku = odecol.step_knots(5e-4, 1.5e-3, 2e-3, amp, 1e-4)
    sheet.set_knots(kt.to(DEV), ku.to(DEV))
    N = sheet.export_linear_form().N
    y0 = torch.cat((torch.rand(B, N, generator=gen) * 4 - 6, torch.rand(B, N, generator=gen) * 0.5, torch.rand(B, N, generator=gen)), 1)
    y0[-1, 2 * N:] = orhs.phi(y0[-1, :N] - y0[-1, N:2 * N])
    return sheet, kt, ku, y0, gen


@pytest.mark.parametrize("cols,grid", [pytest.param(c, g, id=f"N{8 * c}-{g}") for g in SHEET_GRIDS for c in (32, 25)] +
                         [pytest.param(128, "defaults", id="N1024-defaults")])      # K_aug = 1153: chunked contractions
def test_staged_dopri5_on_column_sheets_against_a_float64_replay(cfg, cols, grid):
    rtol, atol, T = SHEET_GRIDS[grid]
    sheet, kt, ku, y0, _ = _sheet(cfg, cols, 3, seed=cols)
    ext = odecol._native.ext()
    lf = sheet_oracle_form(sheet)
    prob = ext_problem(ext, lf, kt.numpy(), ku.numpy())
    assert prob.kernel_family(ext.OP_DOPRI5_FWD) == 1
    tv = np.linspace(0, 2e-3, T, dtype=np.float32)
    _, na, _, out_step, _ = check_dopri5_against_replay(ext, prob, lf, kt.numpy(), ku.numpy(), y0.numpy(), tv, rtol, atol,
                                                        f"sheet N={lf.n} {grid}", controller=grid == "loose_dense", seed=cols)
    assert len(set(na.tolist())) > 1                          # ragged rounds: first steps fall into different rounds
    steps = out_step[:, 1:]
    if grid == "defaults":
        assert (np.diff(steps, axis=1) > 1).any()
    if grid == "loose_dense":
        assert (np.diff(steps, axis=1) == 0).any()


@pytest.mark.parametrize("family", [None, "staged"], ids=["on_chip", "staged"])
def test_dopri5_through_odeint_is_the_replayed_computation_at_any_record_capacity(cfg, family):
    """odeint(default method) + backward() on a sheet runs exactly the record / reverse sweep the replay checks; a record
    too small for a trial stops it with status 2 at the capacity, and odeint(options={'record_capacity': 8}) grows the
    record until every trial fits, with the same outputs and gradients."""
    sheet, kt, ku, y0, gen = _sheet(cfg, 4, 3, seed=7)                     # N = 32
    N, T = 32, 21
    tv = torch.linspace(0, 2e-3, T)
    rtol, atol = 1e-5, 1e-7
    sel = [0, 5, N + 3, 2 * N + 7]
    wgt = torch.randn(T, 3, len(sel), generator=gen)
    ext = odecol._native.ext()
    setup = odecol.solvers._Setup(sheet, y0.to(DEV), tv.to(DEV), family)
    prob = setup.problem(setup.lf.W_aug)
    assert prob.kernel_family(ext.OP_DOPRI5_FWD) == (0 if family is None else 1)
    y_ext, na, _, _, rec = check_dopri5_against_replay(ext, prob, sheet_oracle_form(sheet), kt.numpy(), ku.numpy(), y0.numpy(),
                                                       tv.numpy(), rtol, atol, f"odeint sheet N={N} {family}", controller=True)
    gy0_ext, _ = ext.dopri5_bwd(prob, T, *rec, wgt.to(DEV).contiguous(), torch.tensor(sel, dtype=torch.int32, device=DEV))
    # extension level: a record of 8 steps stops every trial that needs more at 8 accepted steps with status 2
    _, na8, _, st8 = [v.cpu() for v in ext.dopri5_fwd_record(prob, tv.to(DEV), y0.to(DEV), rtol, atol, 4_000_000, 8)[:4]]
    full = na > 8
    assert bool(full.any())
    assert (na8[full] == 8).all() and (st8[full] == 2).all() and (st8[~full] == 0).all() and torch.equal(na8[~full], na[~full])
    runs = []
    for cap in (None, 8):
        sheet.zero_grad()
        y0g = y0.to(DEV).requires_grad_(True)
        st = {}
        y = odecol.odeint(sheet, y0g, tv.to(DEV), rtol=rtol, atol=atol, components=sel, stats=st,
                          options={"family": family, "record_capacity": cap})
        (y * wgt.to(DEV)).sum().backward()
        runs.append((y.detach().cpu(), y0g.grad.cpu(), sheet.recurrent_weights.grad.cpu().clone(), st["n_accept"].cpu()))
    (y_a, g_a, w_a, na_a), (y_b, g_b, w_b, na_b) = runs
    eW = float((w_b - w_a).abs().max() / w_a.abs().max())
    print(f"\n[odeint dopri5 {family}] record capacity 8 vs default: grad W {eW:.1e}")
    assert torch.equal(y_a.double(), y_ext[:, :, sel]) and torch.equal(na_a, na) and torch.equal(g_a, gy0_ext.cpu())
    assert torch.equal(y_b, y_a) and torch.equal(na_b, na_a) and torch.equal(g_b, g_a)
    assert eW < 1e-6                                          # float atomics over trials in grad_W


def test_dopri5_rejects_a_time_grid_that_is_not_strictly_increasing(cfg, golden):
    """torchdiffeq rejects such a grid.  Unchecked, the on-chip kernel emits NaN at a repeated time (0 / 0 abscissa) and
    the staged one y0: the two families would disagree."""
    net = product_network("xor", cfg, golden["xor"], DEV)
    net.stim = torch.tensor(golden["xor"]["stims"]).to(DEV)[:2]
    y0 = torch.zeros(2, 72, device=DEV)
    ts = net.time_vec[:20].clone()
    for bad in (torch.cat((ts[:1], ts)), torch.flip(ts, (0,))):
        for family in (None, "staged"):
            with torch.no_grad(), pytest.raises(ValueError, match="strictly increasing"):
                odecol.odeint(net, y0, bad, options={"family": family})
            with pytest.raises(ValueError, match="strictly increasing"):
                odecol.odeint(net, y0.clone().requires_grad_(True), bad, options={"family": family})


@pytest.mark.parametrize("solver", ["rk4_on_chip", "rk4_tensor", "dopri5_on_chip", "dopri5_staged"])
def test_repeated_components_get_the_summed_gradient(cfg, golden, solver):
    """A loss on components [c, c, d] with weights (w1, w2, w3) is the loss on [c, d] with weights (w1 + w2, w3): the same
    outputs in every copy of c and the same gradients, as torch.index_select gives."""
    method, family = {"rk4_on_chip": ("rk4", None), "rk4_tensor": ("rk4", "tensor"), "dopri5_on_chip": ("dopri5", None),
                      "dopri5_staged": ("dopri5", "staged")}[solver]
    net = product_network("xor", cfg, golden["xor"], DEV)
    net.stim = torch.tensor(golden["xor"]["stims"]).to(DEV)[:4]
    gen = torch.Generator().manual_seed(2)
    y0 = (torch.rand(4, 72, generator=gen) * 2).to(DEV)
    ts = net.time_vec[:60]
    c, d = 17, 24 + 5
    wgt = torch.randn(60, 4, 3, generator=gen).to(DEV)
    runs = []
    for comps, w in (([c, c, d], wgt), ([c, d], torch.stack((wgt[..., 0] + wgt[..., 1], wgt[..., 2]), -1))):
        net.zero_grad()
        y0g = y0.clone().requires_grad_(True)
        y = odecol.odeint(net, y0g, ts, method=method, rtol=1e-5, atol=1e-7, components=comps, options={"family": family})
        (y * w).sum().backward()
        grads = [p.grad.detach().clone() for p in net.parameters() if p.grad is not None]
        runs.append((y.detach(), y0g.grad.detach(), grads))
    (y3, g3, p3), (y2, g2, p2) = runs
    assert torch.equal(y3[..., 0], y3[..., 1]) and torch.equal(y3[..., 1:], y2)
    assert len(p3) == len(p2) > 0
    e0 = float((g3 - g2).abs().max() / g2.abs().max())
    eW = max(float((a - b).abs().max() / b.abs().max().clamp_min(1e-30)) for a, b in zip(p3, p2))
    print(f"\n[{solver} components [c, c, d] vs [c, d]] grad y0 {e0:.1e}  grad params {eW:.1e}")
    assert e0 < 1e-6 and eW < 1e-6
