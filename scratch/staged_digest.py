"""Seeded digest of the staged (N > 128) Euler-Maruyama, srk and dopri5 solvers and of drift_staged: outputs, statistics,
y_steps, gradients and launch counts, for A/B checks of host-side changes that must not change results.

  python scratch/staged_digest.py run OUT.npz               one digest with the library of this tree
  python scratch/staged_digest.py compare A.npz B.npz [C.npz]   every entry bit-identical, except grad_W_aug of the
                                                            reverse sweeps (float atomics): A vs C must stay within A vs B
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def run(out_path):
    import odecol
    from odecol import solvers as SV
    cfg = odecol.load_config(os.path.join(ROOT, "config", "model.toml"))
    ext = odecol._native.ext()
    out = {}

    def put(name, *tensors):
        for i, t in enumerate(tensors):
            out[f"{name}/{i}"] = t.detach().cpu().numpy()
        out[f"{name}/launches"] = np.array([ext.last_launch_count()])

    for cols in (32, 64):
        N, B, T = 8 * cols, 37, 11
        sheet = odecol.SyntheticColumnSheet(cfg, cols, seed=1, device="cuda", sigma_v=3.0)
        gen = torch.Generator().manual_seed(cols)
        amp = torch.rand(B, cols, generator=gen) * 25
        kt, ku = odecol.step_knots(5e-4, 2.5e-3, 4e-3, amp, 1e-4)
        sheet.set_knots(kt.cuda(), ku.cuda())
        ts = torch.linspace(0.0, 4e-3, T).cuda()
        y0 = torch.cat((torch.rand(B, N, generator=gen) * 4 - 6, torch.rand(B, N, generator=gen) * 0.5,
                        torch.rand(B, N, generator=gen)), 1).cuda()
        hot = y0.clone()
        hot[:, 3] = 1400.0                   # a rate FP16 cannot hold: the 16-bit solves repeat in TF32
        dt = 2e-4
        gain = torch.linspace(0.25, 3.0, B)
        scale = torch.linspace(0.0, 2.0, B)

        def setup(y, sigma_scale=None, lateral_gain=None):
            s = SV._Setup(sheet, y, ts, "staged")
            if sigma_scale is not None:
                s.sigma_scale = sigma_scale.cuda()
            if lateral_gain is not None:
                s.set_lateral_gain(sheet, lateral_gain)
            return s, s.problem(s.lf.W_aug)

        su, prob = setup(y0)
        n_steps = int(ext.em_num_steps(ts.cpu(), dt))
        dW = torch.randn(n_steps, B, generator=gen).cuda() * dt ** 0.5
        dU = torch.randn(n_steps, B, generator=gen).cuda() * dt ** 1.5
        g = torch.randn(T, B, 3 * N, generator=gen).cuda()
        p = f"N{N}"
        with torch.no_grad():
            # Euler-Maruyama, fixed step
            put(f"{p}/em_philox", *ext.em_fwd(prob, su.t, y0, None, 7, 3, dt, False, 0.0, 0.0, 0.0, 0)[:4])
            put(f"{p}/em_table", *ext.em_fwd(prob, su.t, y0, dW, 7, 0, dt, False, 0.0, 0.0, 0.0, 0)[:4])
            y, na, nr, st, ys = ext.em_fwd(prob, su.t, y0, None, 7, 0, dt, False, 0.0, 0.0, 0.0, n_steps)
            put(f"{p}/em_train", y, na, nr, st, ys)
            put(f"{p}/em_bwd", *ext.em_bwd(prob, su.t, ys, g, None, dt))
            _, prob_s = setup(y0, sigma_scale=scale)
            put(f"{p}/em_sigma_scale", *ext.em_fwd(prob_s, su.t, y0, None, 7, 0, dt, False, 0.0, 0.0, 0.0, 0)[:4])
            _, prob_g = setup(y0, lateral_gain=gain)
            put(f"{p}/em_gain", *ext.em_fwd(prob_g, su.t, y0, dW, 7, 0, dt, False, 0.0, 0.0, 0.0, 0)[:4])
            # Euler-Maruyama, adaptive
            put(f"{p}/em_adaptive", *ext.em_fwd(prob_s, su.t, y0, None, 7, 0, 1e-3, True, 1e-4, 1e-3, 1e-5, 0)[:4])
            _, prob_gs = setup(y0, sigma_scale=scale, lateral_gain=gain)
            put(f"{p}/em_adaptive_gain", *ext.em_fwd(prob_gs, su.t, y0, None, 7, 0, 1e-3, True, 1e-4, 1e-3, 1e-5, 0)[:4])
            # srk, forward and reverse sweep
            y, st, ys = ext.srk_fwd(prob, su.t, y0, None, None, 7, 0, dt, n_steps)
            put(f"{p}/srk_philox", y, st, ys)
            put(f"{p}/srk_philox_bwd", *ext.srk_bwd(prob, su.t, ys, None, None, 7, 0, g, None, dt))
            y, st, ys = ext.srk_fwd(prob, su.t, y0, dW, dU, 7, 0, dt, n_steps)
            put(f"{p}/srk_table", y, st, ys)
            put(f"{p}/srk_table_bwd", *ext.srk_bwd(prob, su.t, ys, dW, dU, 7, 0, g, None, dt))
            # dopri5: forward only, and with a record plus its reverse sweep
            put(f"{p}/dopri5", *ext.dopri5_fwd(prob, su.t, y0, 1e-5, 1e-6, 100000))
            rec = ext.dopri5_fwd_record(prob, su.t, y0, 1e-5, 1e-6, 100000, 512)
            put(f"{p}/dopri5_record", *rec)
            rec_y, rec_t0, rec_dt, out_step, out_x, na = rec[4], rec[5], rec[6], rec[7], rec[8], rec[1]
            put(f"{p}/dopri5_bwd", *ext.dopri5_bwd(prob, T, rec_y, rec_t0, rec_dt, out_step, out_x, na, g, None))
            # one drift evaluation, per-trial times
            tt = torch.linspace(0.0, 4e-3, B).cuda()
            put(f"{p}/drift", ext.drift_staged(prob, tt, y0))
            put(f"{p}/drift_gain", ext.drift_staged(prob_g, tt, y0))
            # the three FP16 -> TF32 repeats
            _, prob_h = setup(hot, sigma_scale=torch.full((B,), 0.1))
            put(f"{p}/em_hot", *ext.em_fwd(prob_h, su.t, hot, None, 7, 0, dt, False, 0.0, 0.0, 0.0, 0)[:4])
            put(f"{p}/em_adaptive_hot", *ext.em_fwd(prob_h, su.t, hot, None, 7, 0, 1e-3, True, 1e-4, 1e-3, 1e-5, 0)[:4])
            put(f"{p}/srk_hot", *ext.srk_fwd(prob_h, su.t, hot, None, None, 7, 0, dt, 0)[:2])
            put(f"{p}/dopri5_hot", *ext.dopri5_fwd(prob_h, su.t, hot, 1e-5, 1e-6, 100000))
        torch.cuda.synchronize()
    np.savez(out_path, **out)
    print(f"{len(out)} entries -> {out_path}")


def compare(a_path, b_path, c_path=None):
    a, b = np.load(a_path), np.load(b_path)
    c = np.load(c_path) if c_path else None
    assert sorted(a.files) == sorted(b.files), "different entries"
    bad = 0
    for k in sorted(a.files):
        x, y = a[k], b[k]
        # grad_W_aug of the staged reverse sweeps is accumulated with float atomics: not bitwise reproducible
        atomic = k.endswith("_bwd/1")
        same = x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))
        if same:
            continue
        if atomic:
            d = float(np.abs(x - y).max())
            ref = float(np.abs(x - c[k]).max()) if c is not None else float("nan")
            print(f"{k}: max |a - b| = {d:.3e} (|a| max {float(np.abs(x).max()):.3e}); max |a - c| = {ref:.3e}")
            if c is not None and d > 2 * ref:
                bad += 1
            continue
        bad += 1
        print(f"{k}: DIFFERS (max abs {float(np.abs(x.astype(np.float64) - y.astype(np.float64)).max()):.3e})")
    print(f"{len(a.files)} entries, {bad} mismatches")
    return bad


if __name__ == "__main__":
    if sys.argv[1] == "run":
        run(sys.argv[2])
    else:
        sys.exit(1 if compare(*sys.argv[2:]) else 0)
