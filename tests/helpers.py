"""Shared builders for the tests: product networks loaded with the golden (reference-generated) parameters, and the
oracle's unified form of the same networks."""
import numpy as np
import torch

import odecol
from oracle import column_model as cm

XOR_DICT = {"nr_areas": 2, "areas": ["mt", "mt"], "nr_columns_per_area": [2, 1], "nr_input_units": 2}
PARITY_DICT = {"nr_areas": 3, "areas": ["mt"] * 3, "nr_columns_per_area": [8, 4, 1], "nr_input_units": 4}


def product_network(name, cfg, g, device="cpu"):
    """Product module carrying exactly the reference's seed-0 parameters (copied from the golden file)."""
    torch.manual_seed(0)
    if name == "wta":
        net = odecol.ColumnAreaWTA(cfg, "mt")
        with torch.no_grad():
            net.recurrent_weights.copy_(torch.tensor(g["recurrent_weights"]))
    elif name == "xor":
        net = odecol.ColumnNetworkXOR(cfg, XOR_DICT)
        with torch.no_grad():
            for a in "01":
                for i in range(2):
                    net.feedforward_target_weights[a][i].copy_(torch.tensor(g[f"ffw_{a}_{i}"]))
    elif name == "parity":
        net = odecol.ColumnNetwork(cfg, PARITY_DICT, torch.device("cpu"))
        with torch.no_grad():
            for k in "012":
                net.areas[k].lateral_weights.copy_(torch.tensor(g[f"lateral_{k}"]))
            for k in "12":
                net.areas[k].feedforward_weights.copy_(torch.tensor(g[f"feedforward_{k}"]))
            net.areas["0"].input_weights.copy_(torch.tensor(g["input_weights"]))
            net.output_weights.copy_(torch.tensor(g["output_weights"]))
    else:
        raise KeyError(name)
    net.time_vec = torch.tensor(g["time_vec"])
    return to_device(net, device)


def to_device(net, device):
    """Module.to() plus the plain-tensor attributes the reference keeps outside buffers."""
    net = net.to(device)
    mods = [net] + list(net.modules())
    for m in mods:
        for k, v in list(vars(m).items()):
            if torch.is_tensor(v) and not isinstance(v, torch.nn.Parameter):
                setattr(m, k, v.to(device))
    return net


def oracle_form(name, cfg, g):
    if name == "wta":
        return cm.wta_linear_form(cfg, g["recurrent_weights"])
    if name == "xor":
        return cm.xor_linear_form(cfg, [[g["ffw_0_0"], g["ffw_0_1"]], [g["ffw_1_0"], g["ffw_1_1"]]])
    if name == "parity":
        return cm.parity_linear_form(cfg, [g[f"lateral_{k}"] for k in range(3)],
                                     {1: g["feedforward_1"], 2: g["feedforward_2"]}, g["input_weights"])
    raise KeyError(name)


def stim_table(name, stim):
    """Reference-shaped stimulus -> (B, T, n_in) channel table (B = leading batch if present)."""
    s = torch.as_tensor(stim)
    if name == "xor":
        if s.dim() == 3:
            s = s[None]
        return s.reshape(s.shape[0], s.shape[1], -1)
    if s.dim() == 2:
        s = s[None]
    return s


def block_errs(a, b):
    """Norm-relative error of the V, A and F blocks (SURVEY.md section 7: elementwise relative error is meaningless
    at zero crossings of V)."""
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    n = a.shape[-1] // 3
    out = []
    for c in range(3):
        x, y = a[..., c * n:(c + 1) * n], b[..., c * n:(c + 1) * n]
        out.append(float((x - y).abs().max() / y.abs().max().clamp_min(1e-30)))
    return out


def rel_err(a, b):
    return max(block_errs(a, b))


def ext_problem(ext, lf, kt, ku, flags=0, device="cuda"):
    """Extension-level problem of an oracle LinearForm (W_aug = [W | U | bias], rows padded to a multiple of 4) with the
    stimulus knots kt (K,) and ku (B, K, n_in)."""
    N, n_in = lf.n, lf.n_in
    W_aug = torch.zeros(N, (N + n_in + 1 + 3) // 4 * 4)
    W_aug[:, :N] = torch.as_tensor(lf.W); W_aug[:, N:N + n_in] = torch.as_tensor(lf.U); W_aug[:, N + n_in] = torch.as_tensor(lf.bias)
    return ext.Problem(W_aug.to(device), torch.as_tensor(lf.kappa, dtype=torch.float32).to(device), None,
                       torch.as_tensor(kt, dtype=torch.float32).to(device), torch.as_tensor(ku, dtype=torch.float32).contiguous().to(device),
                       n_in, ku.shape[0], lf.tau_s, lf.tau_m, lf.tau_a, lf.resistance, flags)


class TreeBrownian:
    """bm(t0, t1) for the oracle, reading the virtual Brownian tree of ONE trial through odecol_brownian_query -- the
    path the kernels integrate against.  shape = (1, 1) like a torchsde Brownian object for one scalar-noise solve."""

    def __init__(self, seed, trial, t_begin, t_end, device="cuda"):
        self.ext = odecol._native.ext()
        self.seed, self.trial, self.t_begin, self.t_end = seed, trial, float(t_begin), float(t_end)
        self.device = device
        self.shape = (1, 1)

    def __call__(self, t0, t1):
        q = torch.tensor([float(t0), float(t1)], dtype=torch.float32, device=self.device)
        w = self.ext.brownian_query(self.seed, self.trial, 1, self.t_begin, self.t_end, q).cpu()
        return (w[1] - w[0]).reshape(1, 1)


def dopri5_controller_factor(ratio):
    """torchdiffeq's step factor after an ACCEPTED step with error ratio r: min(10, max(0.9 r^-1/5, 1))."""
    return 10.0 if ratio == 0 else min(10.0, max(0.9 * ratio ** -0.2, 1.0))


def check_dopri5_against_replay(ext, prob, lf, kt, ku, y0, tv, rtol, atol, label, controller=False, seed=0,
                                traj_bar=1e-5, grad_bar=5e-5, device="cuda"):
    """dopri5_fwd_record / dopri5_bwd of one problem against a float64 replay of the recorded steps (oracle
    dopri5_replay): the record contract exactly, every accepted step and its dense outputs from the recorded start state,
    the chained trajectory, and the discrete adjoint (dense grad_y, a selection without F, one with F) against autograd
    through the replay.  controller=True also checks the accept decisions and the step-size sequence (loose tolerances
    only: at 1e-7 the error ratio of a float32 solve is rounding noise).  Prints every figure; returns the kernel's y,
    n_accept, n_reject, out_step (on the host) and the record (rec_y, rec_t0, rec_dt, out_step, out_x, n_accept on the
    device, the arguments of dopri5_bwd)."""
    from oracle import rhs as orhs, solvers as S
    N, T, B = lf.n, len(tv), y0.shape[0]
    n3, Kaug = 3 * N, N + lf.n_in + 1
    t_dev = torch.as_tensor(tv, dtype=torch.float32).to(device)
    y, na, nr, st, rec_y, rec_t0, rec_dt, out_step, out_x = ext.dopri5_fwd_record(
        prob, t_dev, torch.as_tensor(y0, dtype=torch.float32).to(device), rtol, atol, 4_000_000, 4096)
    rec_dev = (rec_y, rec_t0, rec_dt, out_step, out_x, na)
    y, na, nr, st = y.cpu().double(), na.cpu(), nr.cpu(), st.cpu()
    ry, rt0, rdt, ost, oxs = rec_y.cpu().double(), rec_t0.cpu().numpy(), rec_dt.cpu().numpy(), out_step.cpu().numpy(), out_x.cpu().numpy()
    assert int(st.abs().sum()) == 0, st
    t64 = np.asarray(tv, dtype=np.float32).astype(np.float64)
    scale = torch.stack([y[..., c * N:(c + 1) * N].abs().max() for c in range(3)])      # per block: V, A, F
    blk = lambda d: (torch.stack([d[..., c * N:(c + 1) * N].abs().max() for c in range(3)]) / scale).max().item()

    gen = torch.Generator().manual_seed(seed)
    sels = {"dense": None,
            "VA": [0, N - 1, N + 1, N + N // 2, N // 2],
            "VF": [2 * N, 1, 3 * N - 1, N + 2, 2 * N + N // 3]}
    wgts = {k: torch.randn(T, B, n3 if s is None else len(s), generator=gen, dtype=torch.float64) for k, s in sels.items()}
    ode = orhs.UnifiedColumnODE(lf, kt, ku, dtype=torch.float64, requires_grad=True)
    params = [ode.W, ode.U, ode.bias]
    g_y0 = {k: torch.zeros(B, n3, dtype=torch.float64) for k in sels}
    g_W = {k: torch.zeros(N, Kaug, dtype=torch.float64) for k in sels}
    e_step = e_dense = e_traj = 0.0
    r_max, fac_dev, n_broken = 0.0, 0.0, []
    for b in range(B):
        n = int(na[b])
        t0s, dts, os_, ox = rt0[b, :n], rdt[b, :n], ost[b], oxs[b]
        # ---- record contract (exact)
        assert t0s[0] == t64[0], (label, b)
        assert np.array_equal(t0s[1:], t0s[:-1] + dts[:-1]), (label, b)
        assert t0s[-1] < t64[-1] <= t0s[-1] + dts[-1], (label, b)
        o, x = os_[1:], ox[1:]
        assert (o >= 0).all() and (o < n).all() and (np.diff(o) >= 0).all() and o[-1] == n - 1, (label, b, o)
        assert (x > 0).all() and (x <= 1).all(), (label, b, x)
        x_exp = ((t64[1:] - t0s[o]) / ((t0s[o] + dts[o]) - t0s[o])).astype(np.float32)   # both families: (t_j - t0) / (t1 - t0)
        assert np.array_equal(x, x_exp), (label, b, np.abs(x - x_exp).max())
        ode_b = ode.select_trials(slice(b, b + 1))
        # ---- every accepted step from its recorded start state, its dense outputs, its error ratio
        ratios = []
        with torch.no_grad():
            for m in range(n):
                ym = ry[m, b][None]
                y1, _, err, coeffs = S.dopri5_step(ode_b, ym, t0s[m], dts[m])
                if m + 1 < n:
                    e_step = max(e_step, blk(y1[0] - ry[m + 1, b]))
                for j in np.nonzero(os_[1:] == m)[0] + 1:
                    e_dense = max(e_dense, blk(S.dense_output(coeffs, float(ox[j]))[0] - y[j, b]))
                ratios.append(float(S.dopri5_error_ratio(ym, y1, err, rtol, atol)))
        if controller:
            r_max = max(r_max, max(ratios))
            obs = dts[1:] / dts[:-1]
            fac = np.array([dopri5_controller_factor(r) for r in ratios[:-1]])
            dev = np.abs(obs / fac - 1)
            broken = int((dev > 1e-3).sum())            # a rejected attempt in between breaks the relation
            n_broken.append(broken)
            fac_dev = max(fac_dev, float(dev[dev <= 1e-3].max()) if (dev <= 1e-3).any() else 0.0)
            assert broken <= int(nr[b]), (label, b, broken, int(nr[b]), dev)
        # ---- chained float64 replay with autograd
        y0g = torch.as_tensor(y0[b:b + 1], dtype=torch.float64).clone().requires_grad_(True)
        yr = S.dopri5_replay(ode_b, y0g, t0s, dts, n, os_, ox)
        e_traj = max(e_traj, blk(yr[:, 0].detach() - y[:, b]))
        for k, s in sels.items():
            ys = yr[:, 0] if s is None else yr[:, 0, s]
            g = torch.autograd.grad((ys * wgts[k][:, b]).sum(), [y0g] + params, retain_graph=True)
            g_y0[k][b] = g[0][0]
            g_W[k] += torch.cat((g[1], g[2], g[3][:, None]), 1)
    if controller:
        assert r_max <= 1 + 1e-2, (label, r_max)
    # ---- discrete adjoint of the kernels
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    e_g = {}
    for k, s in sels.items():
        sel = None if s is None else torch.tensor(s, dtype=torch.int32, device=device)
        gy0, gW = ext.dopri5_bwd(prob, T, *rec_dev, wgts[k].float().to(device).contiguous(), sel)
        gy0, gW = gy0.cpu().double(), gW.cpu().double()
        e_g[k] = (rel(gy0, g_y0[k]), rel(gW[:, :Kaug], g_W[k]))
        assert gW.shape[1] == Kaug or float(gW[:, Kaug:].abs().max()) == 0.0, (label, k)     # padding columns stay zero
    fig = dict(step=e_step, dense=e_dense, traj=e_traj, grads=e_g, ratio_max=r_max, factor_dev=fac_dev)
    print(f"\n[dopri5 replay {label}] accepted {na.tolist()} rejected {nr.tolist()}; one step {e_step:.1e}  dense output "
          f"{e_dense:.1e}  trajectory {e_traj:.1e}; grad y0 / W_aug " +
          "  ".join(f"{k} {a:.1e} / {w:.1e}" for k, (a, w) in e_g.items()) +
          (f"; controller: max ratio {r_max:.6f}, factor deviation {fac_dev:.1e}, broken transitions {n_broken}" if controller else ""))
    assert e_step < traj_bar and e_dense < traj_bar and e_traj < traj_bar, (label, fig)
    assert all(a < grad_bar and w < grad_bar for a, w in e_g.values()), (label, fig)
    return y, na, nr, ost, rec_dev


def sheet_oracle_form(sheet):
    """Oracle LinearForm of a product SyntheticColumnSheet (its W_aug split back into W | U | bias)."""
    from oracle.column_model import LinearForm
    lfp = sheet.export_linear_form()
    n, n_in = lfp.N, lfp.n_in
    Wa = lfp.W_aug.detach().cpu().numpy()
    return LinearForm(W=Wa[:, :n], U=Wa[:, n:n + n_in], bias=Wa[:, n + n_in], kappa=lfp.kappa.cpu().numpy(),
                      sigma=lfp.sigma.cpu().numpy(), tau_s=lfp.tau_s, tau_m=lfp.tau_m, tau_a=lfp.tau_a,
                      resistance=lfp.resistance)
