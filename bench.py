#!/usr/bin/env python
"""Headline benchmark: population-steps/s of the fused column-ODE solver, forward + adjoint (BASELINE.json metric).

Workload (BASELINE.json configs[3], SURVEY.md section 8d "C4"): synthetic 64-column network (N = 512 populations, dense
W), rk4 (3/8 rule) on T = 1500 grid points (dt = 1e-4), 8192 trials per GPU (65,536 at 8 GPUs, weak scaling), per-trial
three-phase stimuli, Huber loss on the L2/3e rates over the whole trajectory, exact discrete adjoint -> dW_aug, and for
N > 1 one NCCL all-reduce of the parameter gradients per step.  One "step" = one such forward + adjoint pass.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA, one process per GPU under torchrun)
  python bench.py --impl reference [...]                          the CPU path (oracle port, all host threads), same metric
  python bench.py [...] --dump-outputs DIR                        also write the last timed step's outputs as DIR/<name>.npy

Prints ONE JSON line (rank 0).  See DESIGN.md section "Measurement" for how every field is computed.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "population_steps_per_sec_fwd_adjoint"
UNIT = "population-steps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--columns", type=int, default=64)
    ap.add_argument("--trials-per-gpu", type=int, default=8192)
    ap.add_argument("--time-points", type=int, default=1500)
    ap.add_argument("--dt", type=float, default=1e-4)
    ap.add_argument("--cpu-trials", type=int, default=1024, help="trials of the bounded CPU sample")
    ap.add_argument("--cpu-time-points", type=int, default=81, help="grid points of the bounded CPU sample (a few seconds of CPU work per pass, ~10 GB of autograd state)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--family", default=None, help="force a kernel family (staged, tensor)")
    ap.add_argument("--workload", default="c4", choices=["c4", "c5", "small", "configs"],
                    help="c4 (default, the headline): N=512 rk4 forward+adjoint; c5: N=8192 adaptive Euler-Maruyama sweep; "
                         "small: the reference's own WTA / parity networks at large batch (persistent on-chip family); "
                         "configs: BASELINE.json configs[0..2] as the scripts run them (latency, next to the CPU oracle)")
    ap.add_argument("--small-trials", type=int, default=65536, help="trials per GPU of the small workload (WTA; parity uses a quarter)")
    ap.add_argument("--c5-columns", type=int, default=1024)
    ap.add_argument("--c5-trials", type=int, default=8192, help="sweep members in total (strong scaling over GPUs)")
    ap.add_argument("--c5-horizon", type=float, default=0.004, help="simulated seconds per step of the c5 workload")
    ap.add_argument("--c5-no-gain", action="store_true", help="c5 without the lateral-gain sweep axis (the round-1 workload)")
    ap.add_argument("--no-secondary", action="store_true", help="c4: skip the compact C5 measurement embedded as `secondary`")
    ap.add_argument("--trials-total", type=int, default=0,
                    help="c4: total trials of the job (strong scaling): every rank integrates trials-total / gpus trials per step in "
                         "chunks of --trials-per-gpu, accumulating dW; 65536 = the literal BASELINE.json configs[3] batch at any N")
    ap.add_argument("--integrate-f", action="store_true",
                    help="c4: also select the F (synaptic) component of the read-out populations, so that the solve integrates and "
                         "returns F as torchdiffeq would (default: F feeds nothing back and no loss reads it, so the kernels skip it)")
    ap.add_argument("--parity-trials", type=int, default=8, help="trials of the in-bench oracle parity check (0 = skip)")
    ap.add_argument("--parity-steps", type=int, default=40)
    ap.add_argument("--probe-trials", type=int, default=1024, help="global trials of the sharding-invariance probe (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="c4: after the timed steps, write what the last timed step returned (loss, parameter gradients, a seeded "
                         "sample of the trajectory) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c4"):
        ap.error("--dump-outputs is implemented for the c4 workload of --impl ours")
    return args


# ----------------------------------------------------------------------------------------------------------------------
# workload construction (shared by both arms; everything seeded, nothing read from disk but config/model.toml)
# ----------------------------------------------------------------------------------------------------------------------
def make_stimulus(torch, B, columns, T, dt, trial0, device):
    """Three-phase stimulus (off / on / off, thirds of the window) with per-trial, per-column amplitudes U(0, 30) Hz,
    as knots; the draw of a chunk of trials is seeded by the GLOBAL index of its first trial, so a rank's chunk is the same
    whatever else runs (the sharding-invariance `probe` uses probe_amplitudes: one draw for the whole job, sliced)."""
    import odecol
    g = torch.Generator(device="cpu").manual_seed(1000 + trial0)
    amp = torch.rand(B, columns, generator=g) * 30.0
    t_end = T * dt
    grid = t_end / (T - 1)
    on, off = (T // 3) * grid, (2 * (T // 3)) * grid
    kt, ku = odecol.step_knots(on, off, t_end, amp, grid)
    return kt.to(device), ku.to(device), amp


def probe_amplitudes(torch, n_trials, columns):
    """Stimulus amplitudes of the sharding-invariance probe: ONE draw for the global trials [0, n_trials); ranks slice it."""
    g = torch.Generator(device="cpu").manual_seed(4242)
    return torch.rand(n_trials, columns, generator=g) * 30.0


def loss_components(torch, columns, with_f=False):
    n = 8 * columns
    v = torch.arange(columns) * 8                       # L2/3e of every column: V and A components
    if with_f:                                          # --integrate-f: their F components ride along (the loss ignores them)
        return torch.cat((v, v + n, v + 2 * n)).to(torch.int64)
    return torch.cat((v, v + n)).to(torch.int64)


def huber_on_rates(torch, odecol, sel_traj, target, columns):
    """Huber loss on the L2/3e firing rates over the whole trajectory.  On the GPU arm this is the product's fused
    read-out (one kernel: loss + gradient w.r.t. the trajectory); the CPU arms evaluate the same expression in torch."""
    if sel_traj.shape[2] == 3 * columns:                # --integrate-f: V, A, F selected; the read-out takes V and A
        sel_traj = sel_traj[:, :, :2 * columns]
    if sel_traj.is_cuda:
        return odecol.huber_rate_loss(sel_traj, target, pops_per_group=1)
    rate = odecol.compute_firing_rate(sel_traj[:, :, :columns] - sel_traj[:, :, columns:])
    return torch.nn.functional.smooth_l1_loss(rate, target.expand_as(rate), beta=1.0)


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
def cpu_sample(args, threads=None):
    """The oracle port of the SAME workload on the host cores: batched unified form (torch CPU), restated rk4, autograd
    backward.  Bounded sample: --cpu-trials trials x (--cpu-time-points - 1) steps of the N = 8*columns network."""
    import torch
    import odecol
    from oracle import rhs as orhs, solvers as S
    from oracle.column_model import LinearForm
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    cfg = odecol.load_config(os.path.join(ROOT, "config", "model.toml"))
    sheet = odecol.SyntheticColumnSheet(cfg, args.columns, seed=0)
    n = 8 * args.columns
    lfp = sheet.export_linear_form()
    Wa = lfp.W_aug.detach().numpy()
    lf = LinearForm(W=Wa[:, :n], U=Wa[:, n:n + args.columns], bias=Wa[:, n + args.columns], kappa=lfp.kappa.numpy(),
                    sigma=lfp.sigma.numpy(), tau_s=lfp.tau_s, tau_m=lfp.tau_m, tau_a=lfp.tau_a, resistance=lfp.resistance)
    B, T = args.cpu_trials, args.cpu_time_points
    kt, ku, _ = make_stimulus(torch, B, args.columns, args.time_points, args.dt, 0, "cpu")
    tv = torch.linspace(0.0, args.time_points * args.dt, args.time_points)[:T]
    sel = loss_components(torch, args.columns)
    target = torch.full((1, 1, args.columns), 0.5)

    def one_pass():
        ode = orhs.UnifiedColumnODE(lf, kt, ku, requires_grad=True)
        y = S.odeint_rk4(ode, torch.zeros(B, 3 * n), tv)
        loss = huber_on_rates(torch, odecol, y[:, :, sel], target, args.columns)
        loss.backward()
        return float(loss.detach())

    def literal_loop(n_trials=2, steps=20):
        """The reference's own execution model (scripts/xor_ode.py:104-117, parity_ode.py:223-236): ONE trial per solve, a
        Python loop over trials, one thread -- here with the oracle's unified-form module standing in for the reference
        classes (they cannot build a 64-column network in reasonable time).  Returns population-steps/s."""
        torch.set_num_threads(1)
        t0 = time.perf_counter()
        for b in range(n_trials):
            ode = orhs.UnifiedColumnODE(lf, kt, ku[b:b + 1], requires_grad=True)
            y = S.odeint_rk4(ode, torch.zeros(1, 3 * n), tv[:steps + 1])
            huber_on_rates(torch, odecol, y[:, :, sel], target, args.columns).backward()
        el = time.perf_counter() - t0
        torch.set_num_threads(threads)
        return n * n_trials * steps / el

    one_pass.literal_loop = literal_loop
    return one_pass, n * B * (T - 1), threads, f"{B} trials x {T - 1} rk4 steps, N={n}, forward + autograd backward"


def run_reference(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    one_pass, pop_steps, threads, sample = cpu_sample(args)
    for _ in range(min(args.warmup, 1)):
        one_pass()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_pass()
    el = time.perf_counter() - t0
    value = pop_steps * args.steps / el
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "note": "reference CPU path = oracle port (the reference is pure "
                   "Python driving third-party solvers that are not installable offline); bounded sample per step"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def workload_name(args):
    name = _workload_name(args)
    return name + ("; F of the read-out populations selected, so F is integrated and returned" if args.integrate_f else "")


def _workload_name(args):
    if args.trials_total:
        return (f"C4: synthetic {args.columns}-column network (N={8 * args.columns}), rk4 forward + discrete adjoint dW, "
                f"T={args.time_points} grid points, {args.trials_total} trials in the job ({args.trials_total // args.gpus} per GPU, "
                f"chunks of {args.trials_per_gpu})")
    return (f"C4: synthetic {args.columns}-column network (N={8 * args.columns}), rk4 forward + discrete adjoint dW, "
            f"T={args.time_points} grid points, {args.trials_per_gpu} trials/GPU (x{args.gpus} GPUs = {args.trials_per_gpu * args.gpus})")



# ----------------------------------------------------------------------------------------------------------------------
def parity_block(torch, odecol, net, args, kt, ku_local, tv, sel, dev, options):
    """The timed configuration checked against the CPU oracle inside the bench run (rank 0): the SAME network, batch,
    tiling and code path (persistent tcgen05 forward in checkpoint mode, reverse sweep) on a window of --parity-steps
    grid steps straddling the stimulus onset, with a seeded linear loss on the first --parity-trials trials only -- so
    trajectory and dW_aug of those trials are comparable with oracle.solvers.odeint_rk4 + autograd on them alone."""
    from oracle import rhs as orhs, solvers as S
    from oracle.column_model import LinearForm
    nb, steps = args.parity_trials, args.parity_steps
    columns, n = args.columns, 8 * args.columns
    B = ku_local.shape[0]
    j0 = max(0, args.time_points // 3 - steps // 2)
    tvp = tv[j0:j0 + steps + 1].contiguous()
    g = torch.Generator(device="cpu").manual_seed(99)
    y0 = torch.zeros(B, 3 * n)
    y0[:nb] = torch.cat((torch.rand(nb, n, generator=g) * 6 - 8, torch.rand(nb, n, generator=g), torch.rand(nb, n, generator=g)), 1)
    wgt = torch.zeros(steps + 1, B, sel.numel())
    wgt[:, :nb] = torch.randn(steps + 1, nb, sel.numel(), generator=g)
    params = [net.recurrent_weights, net.input_weights]
    for p in params:
        p.grad = None
    net.set_knots(kt.to(dev), ku_local.to(dev))
    y0d = y0.to(dev).requires_grad_(True)
    traj = odecol.odeint(net, y0d, tvp, method="rk4", components=sel, options=options)
    ckpt_mode = "Ckpt" in type(traj.grad_fn).__name__
    (traj * wgt.to(dev)).sum().backward()
    torch.cuda.synchronize()
    lfp = net.export_linear_form()
    Wa = lfp.W_aug.detach().cpu().numpy()
    lf = LinearForm(W=Wa[:, :n], U=Wa[:, n:n + columns], bias=Wa[:, n + columns], kappa=lfp.kappa.cpu().numpy(),
                    sigma=lfp.sigma.cpu().numpy(), tau_s=lfp.tau_s, tau_m=lfp.tau_m, tau_a=lfp.tau_a, resistance=lfp.resistance)
    ode = orhs.UnifiedColumnODE(lf, kt.cpu().numpy(), ku_local[:nb].cpu().numpy(), requires_grad=True)
    y0o = y0[:nb].clone().requires_grad_(True)
    yo = S.odeint_rk4(ode, y0o, tvp.cpu())
    selc = sel.cpu()
    (yo[:, :, selc] * wgt[:, :nb]).sum().backward()
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    out = {"trials": nb, "steps": steps, "window_start_index": j0, "batch": B, "checkpoint_mode": ckpt_mode,
           "y_sel_rel_err": rel(traj.detach().cpu()[:, :nb], yo[:, :, selc].detach()),
           "dy0_rel_err": rel(y0d.grad.cpu()[:nb], y0o.grad),
           "dW_rel_err": rel(net.recurrent_weights.grad.cpu(), ode.W.grad),
           "dU_rel_err": rel(net.input_weights.grad.cpu(), ode.U.grad),
           "against": "oracle.solvers.odeint_rk4 + torch autograd (CPU, fp32), same inputs", "bar": "1e-5 trajectory, 5e-5 gradients"}
    out["ok"] = bool(out["y_sel_rel_err"] < 1e-5 and out["dy0_rel_err"] < 5e-5 and out["dW_rel_err"] < 5e-5 and out["dU_rel_err"] < 5e-5)
    for p in params:
        p.grad = None
    return out


def probe_block(torch, dist, odecol, net, args, tv, sel, dev, options, rank, world):
    """Sharding invariance on hardware: the global trials [0, --probe-trials) are split over the ranks (amplitudes and loss
    weights keyed by the GLOBAL trial index), every rank runs forward + adjoint on its share, loss and dW are all-reduced.
    The printed checksums must agree between the N = 1, 2, 4, 8 lines (to float32 summation order)."""
    P, steps = args.probe_trials, args.parity_steps
    columns, n = args.columns, 8 * args.columns
    lo, hi = odecol.distributed.shard_bounds(P, rank, world)
    amp = probe_amplitudes(torch, P, columns)[lo:hi]
    T, dt = args.time_points, args.dt
    t_end = T * dt
    grid = t_end / (T - 1)
    kt, ku = odecol.step_knots((T // 3) * grid, (2 * (T // 3)) * grid, t_end, amp, grid)
    j0 = max(0, T // 3 - steps // 2)
    tvp = tv[j0:j0 + steps + 1].contiguous()
    g = torch.Generator(device="cpu").manual_seed(4243)
    wgt = torch.randn(P, steps + 1, sel.numel(), generator=g)[lo:hi].permute(1, 0, 2).contiguous().to(dev)
    params = [net.recurrent_weights, net.input_weights]
    for p in params:
        p.grad = None
    net.set_knots(kt.to(dev), ku.to(dev))
    traj = odecol.odeint(net, torch.zeros(hi - lo, 3 * n, device=dev), tvp, method="rk4", components=sel, options=options)
    loss = (traj * wgt).sum()
    loss.backward()
    loss = loss.detach().double()
    if world > 1:
        odecol.distributed.allreduce_gradients(params)
        dist.all_reduce(loss)
    gW = net.recurrent_weights.grad.double()
    pos = torch.arange(gW.numel(), device=dev, dtype=torch.float64).reshape(gW.shape)
    out = {"trials": P, "steps": steps, "loss": float(loss), "dW_sum": float(gW.sum()), "dW_abs_sum": float(gW.abs().sum()),
           "dW_weighted_sum": float((gW * torch.cos(pos)).sum()), "dU_abs_sum": float(net.input_weights.grad.double().abs().sum())}
    for p in params:
        p.grad = None
    return out


def dump_outputs(torch, out_dir, loss, net, traj, budget=48 << 20):
    """What the last timed step handed its caller, as float32 .npy files in out_dir: the loss, the gradients of both
    parameters and the trajectory of the selected components (T, trials, components) of the step's last chunk.  The
    trajectory (6 GB at the default shape) is sampled: a fixed, seeded set of at most 32 trials, every time point while the
    sample fits `budget` bytes, every k-th otherwise.  Loss and trajectory repeat bit for bit from run to run; the gradients
    are reduced over trials with float atomics (odeint's options['deterministic'] is off here, as in the timed steps), so
    two runs of one build differ in their last bits (5e-7 relative on a B200): compare them with a float32 tolerance."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    T, B, S = traj.shape
    k = max(1, min(32, B, budget // (4 * T * S)))
    trials = torch.randperm(B, generator=torch.Generator(device="cpu").manual_seed(0))[:k].sort().values
    every = -(-4 * T * S * k // budget)
    out = {"loss": loss, "grad_recurrent_weights": net.recurrent_weights.grad, "grad_input_weights": net.input_weights.grad,
           "trajectory_sample": traj[::every, trials.to(traj.device)]}
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.detach().float().cpu().numpy())

# ----------------------------------------------------------------------------------------------------------------------
def init_nccl(torch, dist, dev):
    """One process per GPU over NCCL.  NCCL writes its version banner to STDOUT when the first communicator is created
    (NCCL_DEBUG=VERSION / WARN on some boxes); stdout carries the ONE JSON line of the contract, so file descriptor 1
    points at stderr while the communicator comes up."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group("nccl", device_id=dev)
        warm = torch.zeros(1, device=dev)
        dist.all_reduce(warm)
        torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import odecol

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_nccl(torch, dist, dev)
    ext = odecol._native.ext()

    cfg = odecol.load_config(os.path.join(ROOT, "config", "model.toml"))
    columns, B, T = args.columns, args.trials_per_gpu, args.time_points
    n = 8 * columns
    net = odecol.SyntheticColumnSheet(cfg, columns, seed=0, device=dev)
    params = [net.recurrent_weights, net.input_weights]
    # default: weak scaling, one chunk of B trials per rank and step.  --trials-total: the job's batch is fixed and every
    # rank walks its share in chunks of B trials per step, dW accumulating over the chunks (strong scaling)
    chunks = 1
    if args.trials_total:
        if args.trials_total % (world * B):
            raise SystemExit("--trials-total must be a multiple of gpus x trials-per-gpu")
        chunks = args.trials_total // (world * B)
    trial0 = rank * B * chunks
    stim = [make_stimulus(torch, B, columns, T, args.dt, trial0 + c * B, "cpu") for c in range(chunks)]
    kt, ku = stim[0][0], stim[0][1]
    tv = torch.linspace(0.0, T * args.dt, T, device=dev)
    sel = loss_components(torch, columns, args.integrate_f).to(dev)
    target = torch.full((1, 1, columns), 0.5, device=dev)
    y0_host = torch.zeros(B, 3 * n).pin_memory()
    ku_hosts = [st[1].pin_memory() for st in stim]
    ku_host = ku_hosts[0]
    kt_dev = kt.to(dev)
    options = {"family": args.family} if args.family else None
    launches = {"n": 0}

    def step(from_host: bool):
        """One forward + adjoint pass through the public API.  from_host: inputs come from pinned host memory and the
        loss + dW go back to the host inside the pass (the e2e leg)."""
        for p in params:
            p.grad = None
        step.traj = None
        total = None
        for c in range(chunks):
            if from_host:
                y0 = y0_host.to(dev, non_blocking=True)
                ku_d = ku_hosts[c].to(dev, non_blocking=True)
            else:
                y0, ku_d = step.y0_dev, step.ku_devs[c]
            net.set_knots(kt_dev, ku_d)
            traj = odecol.odeint(net, y0, tv, method="rk4", components=sel, options=options)
            launches["n"] += ext.last_launch_count()
            loss = huber_on_rates(torch, odecol, traj, target, columns)
            launches["n"] += ext.last_launch_count()
            loss.backward()
            launches["n"] += ext.last_launch_count()
            total = loss.detach() if total is None else total + loss.detach()
            if step.keep_traj and c == chunks - 1:
                step.traj = traj.detach()
            del traj, loss
        total = total / chunks
        if world > 1:
            odecol.distributed.allreduce_gradients(params)
            dist.all_reduce(total)
            total = total / world                  # mean over the job's trials (equal shares per rank)
        if from_host:
            return total.cpu(), net.recurrent_weights.grad.cpu()
        return total, None

    step.y0_dev = y0_host.to(dev)
    step.ku_devs = [k.to(dev) for k in ku_hosts]
    step.ku_dev = step.ku_devs[0]
    step.keep_traj = False                               # the timed steps keep their last trajectory for --dump-outputs

    def timed(n_steps, from_host):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(n_steps):
            out = step(from_host)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms) / 1e3, out

    for _ in range(args.warmup):
        step(False)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches["n"] = 0
    step.keep_traj = bool(args.dump_outputs)
    sec, (loss, _) = timed(args.steps, False)
    n_launch = launches["n"]
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, loss, net, step.traj)
    step.keep_traj, step.traj = False, None
    pop_steps_job = n * B * chunks * world * (T - 1)
    value = pop_steps_job * args.steps / sec

    # where one pass spends its time (one extra, untimed-for-the-metric pass with events between the phases)
    net.set_knots(kt_dev, step.ku_dev)
    phases = None
    for _ in range(2):                                   # best of two passes per phase
        for p in params:
            p.grad = None
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        torch.cuda.synchronize()
        ev[0].record()
        traj = odecol.odeint(net, step.y0_dev, tv, method="rk4", components=sel, options=options)
        ev[1].record()
        loss_p = huber_on_rates(torch, odecol, traj, target, columns)
        ev[2].record()
        loss_p.backward()
        ev[3].record()
        torch.cuda.synchronize()
        cur = {"forward_ms": ev[0].elapsed_time(ev[1]), "loss_ms": ev[1].elapsed_time(ev[2]),
               "loss_backward_plus_adjoint_ms": ev[2].elapsed_time(ev[3])}
        phases = cur if phases is None else {k: min(v, phases[k]) for k, v in cur.items()}
        ckpt_mode = bool(traj.grad_fn is not None and "Ckpt" in type(traj.grad_fn).__name__)
        del traj, loss_p
    phases["checkpoint_mode"] = ckpt_mode

    # e2e leg: same pass, inputs from pinned host memory, loss and dW read back every step
    step(True)
    e2e_steps = max(1, args.steps)
    sec_e2e, (loss_h, gW_h) = timed(e2e_steps, True)
    e2e_value = pop_steps_job * e2e_steps / sec_e2e
    h2d = (y0_host.numel() * 4 + ku_host.numel() * 4) * chunks
    d2h = gW_h.numel() * 4 + 4

    # roofline of the dominant kernel (the fused forward stage contraction): forward-only solve, CUDA events around it
    net.set_knots(kt_dev, step.ku_dev)
    with torch.no_grad():
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        odecol.odeint(net, step.y0_dev, tv, method="rk4", components=sel, options=options)
        e1.record()
        torch.cuda.synchronize()
        fwd_sec = e0.elapsed_time(e1) / 1e3
        fwd_launches = ext.last_launch_count()
    kaug = n + columns + 1
    flops_per_launch = 2.0 * n * kaug * B                       # algorithmic: one W_aug . r_aug contraction of all trials
    stage_launches = 4 * (T - 1)
    avg_launch = fwd_sec / stage_launches
    achieved_tflops = flops_per_launch / avg_launch / 1e12
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    bf16 = peaks.get("bf16_tflops_sustained", 1400.0)
    # operand format of the persistent forward kernel: FP16 pairs, three kind::f16 products per K step (default), or the TF32
    # split, three kind::tf32 products at half the rate (ODECOL_FWD16=0); either keeps float32 accuracy
    fmt16 = os.environ.get("ODECOL_FWD16", "1") != "0"
    tensor_peak = bf16 / 3.0 if fmt16 else bf16 / 2.0 / 3.0
    tf32_peak = bf16 / 2.0 / 3.0
    sm_max = peaks.get("sm_max_mhz", 1965.0)
    ffma_peak = 148 * 128 * 2 * sm_max * 1e6 / 1e12
    family = net_family(ext, odecol, net, step.y0_dev, tv, args)
    # DRAM bytes per stage pass from the committed ncu --set full capture of this kernel on this workload shape
    traffic, traffic_src = None, None
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        if rec.get("populations") == n and rec.get("trials") == B:
            traffic, traffic_src = rec["dram_bytes_per_stage_pass"], rec["source"]
    except (OSError, KeyError, ValueError):
        pass
    # the same pass seen from HBM: algorithmic bytes of the stage epilogues (DESIGN.md section 2: 20 / 24 / 28 / 36 bytes per
    # population and trial for stages 1..4) + the next operand written and read once (two FP16 or two TF32 planes)
    kpa = (kaug + 63) // 64 * 64 if fmt16 else (kaug + 31) // 32 * 32
    op_bytes = 4.0 if fmt16 else 8.0
    hbm_bytes = (20 + 24 + 28 + 36) / 4.0 * n * B + op_bytes * n * B + op_bytes * kpa * B
    hbm_peak = peaks.get("hbm_gbs", 6457.0)
    # what crosses the L2 <-> SM ports: every 128-population tile re-reads its trial tile and every trial tile re-reads the
    # W_aug tile (both planes), plus the bookkeeping bytes above
    l2_bytes = (n // 128) * B * kpa * op_bytes + ((B + 111) // 112) * n * kpa * op_bytes + hbm_bytes
    roofline = {
        "bound": "tensor",
        "kernel": "k_tc_rk4_fwd_persistent, per RK stage pass (fused W_aug.r_aug contraction + stage epilogue; one "
                  "cooperative launch runs all 4(T-1) passes, 'launch' below = one stage pass)",
        "achieved": achieved_tflops, "peak": tensor_peak, "unit": "TFLOP/s", "frac": achieved_tflops / tensor_peak,
        "traffic": traffic,
        "peak_source": (("measured bf16_tflops_sustained (FP16 runs at the BF16 rate) /3 (hi/lo FP16 pairs: three products) "
                         if fmt16 else "measured bf16_tflops_sustained/2 (TF32) /3 (3xTF32 split) ") + "from MEASURED_PEAKS.json"
                        if peaks else "fallback 1.4 PFLOP/s bf16 sustained / products"),
        "operand_format": "fp16 pairs (x = xh + xl/2048), 3 kind::f16 products" if fmt16 else "tf32 pairs, 3 kind::tf32 products",
        "frac_of_3xtf32_peak": achieved_tflops / tf32_peak,
        "flops_per_launch": flops_per_launch, "avg_launch_ms": 1e3 * avg_launch, "kernel_family": family,
        "fp32_ffma_peak_tflops": ffma_peak, "frac_of_fp32_ffma_peak": achieved_tflops / ffma_peak,
        "forward_only_pop_steps_per_sec": n * B * (T - 1) / fwd_sec,
        "traffic_source": traffic_src,
        "hbm_view": {"algorithmic_bytes_per_launch": hbm_bytes, "achieved_gbs": hbm_bytes / avg_launch / 1e9,
                     "peak_gbs": hbm_peak, "frac": hbm_bytes / avg_launch / 1e9 / hbm_peak},
        # what binds at N=512 (DESIGN.md section 5): every byte of operand tile and of bookkeeping crosses the L2 <-> SM
        # ports, whose full-chip throughput is ~6300 B/cycle (B300_MICROARCH.md, LTS cap)
        "l2_view": {"bytes_per_launch": l2_bytes, "achieved_gbs": l2_bytes / avg_launch / 1e9,
                    "cap_gbs": 6300.0 * sm_max * 1e6 / 1e9, "frac": l2_bytes / avg_launch / (6300.0 * sm_max * 1e6)},
    }

    # correctness inside the bench run: oracle parity of the timed configuration (rank 0) and the sharding-invariance probe
    parity = None
    if rank == 0 and args.parity_trials > 0:
        parity = parity_block(torch, odecol, net, args, kt, ku, tv, sel, dev, options)
    probe = None
    if args.probe_trials > 0:
        probe = probe_block(torch, dist, odecol, net, args, tv, sel, dev, options, rank, world)

    # BASELINE.json configs[4] next to the headline: one short adaptive Euler-Maruyama sweep at N = 8192 (strong scaling)
    secondary = None
    if not args.no_secondary:
        del net
        step.ku_devs = step.ku_dev = step.y0_dev = None
        torch.cuda.empty_cache()
        sec_line = c5_measure(args, torch, dist, odecol, dev, rank, world, 1, 1, args.c5_horizon)
        secondary = {k: sec_line[k] for k in ("metric", "value", "unit", "scaling", "ms_per_step", "config", "gpu_launches",
                                               "attempted_steps_per_member", "accepted_steps_per_member", "rounds_per_solve",
                                               "all_members_finite")}
        secondary["roofline"] = {k: sec_line["roofline"][k] for k in ("bound", "kernel", "achieved", "peak", "unit", "frac")}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        one_pass, ps, threads, sample = cpu_sample(args)
        one_pass()
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            one_pass()
        cpu = {"value": ps * reps / (time.perf_counter() - t0), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
               "note": "batched unified-form port on all host threads (BASELINE.md's 'strong CPU'), not the reference's B = 1 loop",
               "literal_trial_loop": {"value": one_pass.literal_loop(), "unit": UNIT, "cores": 1,
                                      "sample": "2 trials x 20 rk4 steps, ONE trial per solve in a Python loop (the reference's "
                                                "execution model), forward + autograd backward, extrapolates linearly in trials"}}

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * sec / args.steps, "higher_is_better": True, "scaling": "strong" if args.trials_total else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args), "populations": n, "trials_per_gpu": B * chunks, "time_points": T,
                       "solver": "rk4 (3/8 rule) + exact discrete adjoint", "l2": "working set larger than L2: 126 GB of per-step checkpoints (or the 75 GB trajectory) stream through HBM every pass",
                       "parallelism": f"trial-parallel x{world}, allreduce(dW) per step" if world > 1 else "single GPU"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps},
            "gpu_launches": n_launch,
            "roofline": roofline,
            "phases": phases,
            "cpu_baseline": cpu,
            "loss": float(loss),
            "parity": parity,
            "probe": probe,
            "secondary": secondary,
        }))
    if world > 1:
        dist.destroy_process_group()


def c5_measure(args, torch, dist, odecol, dev, rank, world, steps, warmup, horizon):
    """BASELINE.json configs[4] (SURVEY.md 8d C5): 1,024-column network (N = 8192, dense W on the tensor cores), sweep of
    8192 members differing in stimulus amplitude, noise amplitude (sigma in [0, 20]) and global lateral gain (0.5 .. 1.5),
    stochastic adaptive Euler-Maruyama (rtol 1e-5, atol 1e-4, dt 1e-3, dt_min 1e-5, in-kernel Philox seed 0), members
    sharded over the GPUs (strong scaling, no collective).  One step = one solve over `horizon` simulated seconds; the unit
    is one population advanced by one ATTEMPTED step.  Returns the fields of the JSON line (rank 0 prints)."""
    ext = odecol._native.ext()
    cfg = odecol.load_config(os.path.join(ROOT, "config", "model.toml"))
    cols, n = args.c5_columns, 8 * args.c5_columns
    lo, hi = odecol.distributed.shard_bounds(args.c5_trials, rank, world)
    B = hi - lo
    net = odecol.SyntheticColumnSheet(cfg, cols, seed=0, device=dev)
    g = torch.Generator(device="cpu").manual_seed(2000)
    amp = (torch.rand(args.c5_trials, 1, generator=g) * 30.0)[lo:hi].expand(B, cols).contiguous()
    # second sweep axis: the noise amplitude, sigma in [0, 20] (SyntheticColumnSheet carries sigma_V = 10)
    sigma_scale = (torch.rand(args.c5_trials, generator=g) * 2.0)[lo:hi].contiguous().to(dev)
    # third sweep axis: the global lateral gain, 0.5 .. 1.5 times the network's between-column weights
    lateral_gain = (0.5 + torch.rand(args.c5_trials, generator=g))[lo:hi].contiguous().to(dev)
    kt = torch.tensor([0.0, 1.0], device=dev)
    ku = torch.stack((amp, amp), dim=1).to(dev)                  # constant stimulus, per-member amplitude
    net.set_knots(kt, ku)
    y0 = torch.zeros(B, 3 * n, device=dev)
    sweep = {"sigma_scale": sigma_scale}
    if not args.c5_no_gain:
        sweep["lateral_gain"] = lateral_gain

    def step(h):
        st = {}
        ts = torch.linspace(0.0, h, 3, device=dev)
        with torch.no_grad():
            y = odecol.sdeint(net, y0, ts, method="euler", dt=1e-3, adaptive=True, rtol=1e-5, atol=1e-4, dt_min=1e-5,
                              seed=0, trial_offset=lo, stats=st, options=dict(sweep))
        return y, st, ext.last_launch_count()

    for _ in range(warmup):
        step(min(horizon, 2e-4))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    attempts = torch.zeros((), device=dev, dtype=torch.float64)
    accepted = torch.zeros((), device=dev, dtype=torch.float64)
    launches = 0
    for _ in range(steps):
        y, st, nl = step(horizon)
        attempts += (st["n_accept"] + st["n_reject"]).double().sum()
        accepted += st["n_accept"].double().sum()
        launches += nl
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    rounds_t = (st["n_accept"] + st["n_reject"]).max().double()
    finite = torch.isfinite(y[-1]).all().double()
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(attempts)
        dist.all_reduce(accepted)
        dist.all_reduce(rounds_t, op=dist.ReduceOp.MAX)
        dist.all_reduce(finite, op=dist.ReduceOp.MIN)
    clocks = sampler.stop() if rank == 0 else None
    sec = float(ms) / 1e3
    rounds = int(rounds_t)
    value = n * float(attempts) / sec
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    # operand format of the drift contraction: FP16 pairs (three kind::f16 products per K step, default) or the TF32 split
    # (ODECOL_EM16=0: three kind::tf32 products at half the rate); float32 accuracy either way
    em16 = os.environ.get("ODECOL_EM16", "1") != "0"
    tensor_peak = peaks.get("bf16_tflops_sustained", 1400.0) / (3.0 if em16 else 6.0)
    kaug = n + cols + 1
    # DRAM bytes of one drift evaluation from the committed ncu --set full capture of this kernel on this workload shape
    traffic, traffic_src = None, None
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "r1_traffic_c5.json")))
        if rec.get("populations") == n and rec.get("trials") == B and world == 1:
            traffic, traffic_src = rec["dram_bytes_per_drift_evaluation"], rec["source"]
    except (OSError, KeyError, ValueError):
        pass
    # two drift evaluations per round, all resident members (max over ranks of the rounds: the slowest rank sets the time)
    achieved = 2.0 * n * kaug * B * 2 * rounds * steps / sec / 1e12 if rounds else 0.0
    del net, y0, y
    torch.cuda.empty_cache()
    return {
        "metric": "population_steps_per_sec_adaptive_em", "value": value, "unit": "population-steps/s (attempted steps)",
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * sec / steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"C5: synthetic {cols}-column network (N={n}), sweep of {args.c5_trials} members (stimulus amplitude, "
                   f"sigma in [0, 20]" + ("" if args.c5_no_gain else ", global lateral gain in [0.5, 1.5]") + "), adaptive "
                   f"Euler-Maruyama (rtol 1e-5, atol 1e-4, dt 1e-3, dt_min 1e-5, Philox seed 0), {horizon}s horizon",
                   "l2": "W_aug hi+lo (539 MB) larger than L2"},
        "clocks": clocks, "gpu_launches": launches,
        "attempted_steps_per_member": float(attempts) / steps / args.c5_trials,
        "accepted_steps_per_member": float(accepted) / steps / args.c5_trials, "rounds_per_solve": rounds,
        "all_members_finite": bool(finite > 0),
        "roofline": {"bound": "tensor", "kernel": "k_tc_contract<RhsEpi> (tcgen05 drift evaluation, " +
                               ("FP16 pairs: 3 kind::f16 products)" if em16 else "TF32 pairs: 3 kind::tf32 products)"),
                     "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s", "frac": achieved / tensor_peak,
                     "frac_of_3xtf32_peak": achieved / (peaks.get("bf16_tflops_sustained", 1400.0) / 6.0),
                     "traffic": traffic, "traffic_source": traffic_src,
                     "note": "lower bound: the elementwise stepping kernels are inside the timed region; per rank at N > 1"},
    }


def run_c5(args):
    import torch
    import torch.distributed as dist
    import odecol
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_nccl(torch, dist, dev)
    line = c5_measure(args, torch, dist, odecol, dev, rank, world, args.steps, args.warmup, args.c5_horizon)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_small(args):
    """The reference's own networks (BASELINE.json configs[0..2] sizes: WTA N=16, parity N=104) at large batch on the
    persistent on-chip kernel family: one CTA integrates one trial through the whole time loop.  Reports, per case,
    population-steps/s and the fraction of min(HBM with the (T,B,3N) trajectory materialised, FP32 FFMA) -- SURVEY.md 8d."""
    import torch
    import odecol
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    ext = odecol._native.ext()
    cfg = odecol.load_config(os.path.join(ROOT, "config", "model.toml"))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6457.0)
    ffma_peak = 148 * 128 * 2 * peaks.get("sm_max_mhz", 1965.0) * 1e6 / 1e12
    torch.manual_seed(0)

    def move(net):
        net = net.to(dev)
        for m in [net] + list(net.modules()):
            for k, v in list(vars(m).items()):
                if torch.is_tensor(v) and not isinstance(v, torch.nn.Parameter):
                    setattr(m, k, v.to(dev))
        return net

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3 / reps

    cases = {}
    sampler = ClockSampler(local)
    sampler.start()
    launches = 0
    for name in ("wta", "parity"):
        if name == "wta":
            net = move(odecol.ColumnAreaWTA(cfg, "mt"))
            N, n_in, T, dt, B = 16, 16, 1500, 1e-4, args.small_trials
            amp = torch.zeros(B, 16)
            g = torch.Generator().manual_seed(3000)
            a = torch.rand(B, 2, generator=g) * 30.0
            amp[:, 2] = amp[:, 3] = a[:, 0]; amp[:, 10] = amp[:, 11] = a[:, 1]
            read = torch.tensor([0, 8])                                   # L2/3e of both columns
        else:
            nd = {"nr_areas": 3, "areas": ["mt"] * 3, "nr_columns_per_area": [8, 4, 1], "nr_input_units": 4}
            net = move(odecol.ColumnNetwork(cfg, nd, torch.device("cpu")))
            N, n_in, T, dt, B = 104, 4, 1000, 1e-3, max(1, args.small_trials // 4)
            g = torch.Generator().manual_seed(3001)
            amp = (torch.rand(B, 4, generator=g) > 0.5).float() * 15.0
            read = torch.tensor([96])                                     # L2/3e of the output column
        t_end = T * dt
        grid = t_end / (T - 1)
        kt, ku = odecol.step_knots((T // 3) * grid, (2 * (T // 3)) * grid, t_end, amp, grid)
        net.time_vec, net.stim = kt.to(dev), (ku.to(dev) if name == "wta" else ku.to(dev))
        tv = torch.linspace(0.0, t_end, T, device=dev)
        y0 = torch.zeros(B, 3 * N, device=dev)
        sel = torch.cat((read, read + N)).to(dev)
        target = torch.full((1, 1, len(read)), 0.5, device=dev)
        params = [p for p in net.parameters() if p.requires_grad]
        kaug = N + n_in + 1
        res = {"populations": N, "trials": B, "time_points": T}

        opts = {"family": args.family} if args.family else None

        def fwd():
            with torch.no_grad():
                return odecol.odeint(net, y0, tv, method="rk4", options=opts)

        def fwd_adj():
            for p in params:
                p.grad = None
            y = odecol.odeint(net, y0, tv, method="rk4", components=sel, options=opts)
            odecol.huber_rate_loss(y, target, 1).backward()

        sec = timed(fwd, args.steps)
        launches += ext.last_launch_count() * (args.steps + 1)
        ps = N * B * (T - 1) / sec
        flops = 4 * (2 * kaug + 24) + 48                                  # per population-step (SURVEY 8d)
        res["rk4_forward"] = {"pop_steps_per_sec": ps, "ms": 1e3 * sec,
                              "hbm_gbs_trajectory": 12.0 * ps / 1e9, "hbm_frac": 12.0 * ps / 1e9 / hbm_peak,
                              "fp32_tflops": flops * ps / 1e12, "fp32_frac": flops * ps / 1e12 / ffma_peak}
        sec = timed(fwd_adj, args.steps)
        ps = N * B * (T - 1) / sec
        res["rk4_forward_adjoint"] = {"pop_steps_per_sec": ps, "ms": 1e3 * sec}
        if name == "wta":
            def srk():
                for p in params:
                    p.grad = None
                y = odecol.sdeint(net, y0, tv, method="srk", dt=1e-3, seed=0, components=sel,
                                  options={"sigma_scale": torch.full((B,), 0.1)})
                odecol.huber_rate_loss(y, target, 1).backward()
            sec = timed(srk, args.steps)
            n_steps = ext.em_num_steps(tv.cpu(), 1e-3)
            res["srk_forward_adjoint"] = {"pop_steps_per_sec": N * B * n_steps / sec, "ms": 1e3 * sec, "solver_steps": n_steps}
        cases[name] = res
        del net
        torch.cuda.empty_cache()
    clocks = sampler.stop()
    w = cases["wta"]
    bound = min(("hbm", w["rk4_forward"]["hbm_frac"]), ("fp32", w["rk4_forward"]["fp32_frac"]), key=lambda kv: -kv[1])
    print(json.dumps({
        "metric": METRIC, "value": w["rk4_forward_adjoint"]["pop_steps_per_sec"], "unit": UNIT, "n_gpus": 1,
        "steps": args.steps, "warmup": 1, "ms_per_step": w["rk4_forward_adjoint"]["ms"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "small: reference WTA network (N=16, T=1500) and parity network (N=104, T=1000) at large "
                               "batch, persistent on-chip family (whole time loop in one launch; WTA forward: 128 trials per CTA on the tensor core)",
                   "l2": "trajectories (18.9 GB / 20.4 GB) larger than L2"},
        "clocks": clocks, "gpu_launches": launches, "cases": cases,
        "roofline": {"bound": "hbm", "kernel": "k_rk4_fwd_tiny (WTA from 4096 trials: trials on the M axis of tcgen05, FP16 pairs; k_rk4_fwd_small<40> below that or with ODECOL_TINY_TC=0); full (T,B,3N) trajectory written: 12 B per population-step",
                     "achieved": w["rk4_forward"]["hbm_gbs_trajectory"], "peak": hbm_peak, "unit": "GB/s",
                     "frac": w["rk4_forward"]["hbm_frac"], "traffic": None,
                     "fp32_view": {"achieved_tflops": w["rk4_forward"]["fp32_tflops"], "peak_tflops": ffma_peak,
                                   "frac": w["rk4_forward"]["fp32_frac"]}, "binding": bound[0]},
    }))


def run_configs(args):
    """BASELINE.json configs[0..2] exactly as the reference scripts run them -- C1: WTA network, one trial, 1500 grid points
    (rk4 forward + Huber-loss backward, and the scripts' sdeint srk call); C2: XOR network, dopri5 (rtol 1e-7, atol 1e-9)
    with discrete-adjoint training, the four input patterns; C3: parity network, Euler-Maruyama dt 1e-3 with one
    Brownian path shared by the four patterns.  Latency-bound by construction (1..4 trials); reported as wall time per
    solve next to the CPU oracle driving the same solve trial by trial (torch CPU, one thread -- the reference's loop)."""
    import torch
    import odecol
    from oracle import column_model as cm, rhs as orhs, solvers as S, stimuli
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    ext = odecol._native.ext()
    cfg = odecol.load_config(os.path.join(ROOT, "config", "model.toml"))

    def move(net):
        net = net.to(dev)
        for m in [net] + list(net.modules()):
            for k, v in list(vars(m).items()):
                if torch.is_tensor(v) and not isinstance(v, torch.nn.Parameter):
                    setattr(m, k, v.to(dev))
        return net

    def gpu_ms(fn, reps=5):
        fn(); fn()
        out = []
        for _ in range(reps):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1))
        return statistics.median(out)

    def cpu_ms(fn):
        torch.set_num_threads(1)
        t0 = time.perf_counter(); fn()
        return 1e3 * (time.perf_counter() - t0)

    cases = {}
    launches = 0
    # ---- C1
    torch.manual_seed(0)
    net = odecol.ColumnAreaWTA(cfg, "mt")
    tv = stimuli.time_vec(1500, 1e-4)
    stim = stimuli.wta_stimulus(tv, (20.0, 30.0))
    target = torch.linspace(0, 1, 1500).reshape(1, 1500, 1).repeat(1, 1, 2) * torch.tensor([0.6, 0.3])
    lf = cm.wta_linear_form(cfg, net.recurrent_weights.detach().numpy())
    def c1_cpu():
        ode = orhs.UnifiedColumnODE(lf, tv, stim[None], requires_grad=True)
        y = S.odeint_rk4(ode, torch.zeros(1, 48), tv)
        r = orhs.phi(y[:, 0, :16] - y[:, 0, 16:32])
        torch.nn.functional.smooth_l1_loss(torch.stack((r[:, 0], r[:, 8]), 1)[None], target).backward()
    def c1_cpu_srk():
        ode = orhs.UnifiedColumnODE(lf, tv, stim[None])
        n = len(S.em_step_schedule(tv, 1e-3))
        W, U = S.sample_w_u(n, 1, 1e-3, torch.Generator().manual_seed(0))
        with torch.no_grad():
            S.sdeint_srk(ode, torch.zeros(1, 48), tv, S.TabulatedBrownianU(0.1 * W, 0.1 * U), dt=1e-3)
    netd = move(net)
    netd.time_vec, netd.stim = tv.to(dev), stim.to(dev)
    y0 = torch.zeros(1, 48, device=dev)
    tgt = target.to(dev)
    def c1_gpu():
        netd.zero_grad()
        y = odecol.odeint(netd, y0, netd.time_vec, method="rk4")
        odecol.huber_loss_wta(y.unsqueeze(0), tgt, netd).backward()
    def c1_gpu_srk():
        with torch.no_grad():
            odecol.sdeint(netd, y0, netd.time_vec, names={"drift": "forward", "diffusion": "diffusion"}, method="srk", seed=0,
                          options={"sigma_scale": [0.1]})
    cases["C1 wta rk4 forward+backward (1 trial, 1499 steps)"] = {"gpu_ms": gpu_ms(c1_gpu), "cpu_oracle_ms": cpu_ms(c1_cpu)}
    cases["C1 wta sdeint srk forward (1 trial, 150 steps, 1500 outputs)"] = {"gpu_ms": gpu_ms(c1_gpu_srk), "cpu_oracle_ms": cpu_ms(c1_cpu_srk)}
    # ---- C2
    torch.manual_seed(0)
    nd = {"nr_areas": 2, "areas": ["mt", "mt"], "nr_columns_per_area": [2, 1], "nr_input_units": 2}
    net = odecol.ColumnNetworkXOR(cfg, nd)
    tv = stimuli.time_vec(1000, 1e-3)
    stims = torch.stack([stimuli.xor_stimulus(tv, c) for c in stimuli.XOR_CONDITIONS])
    ffw = [[p.detach().numpy() for p in net.feedforward_target_weights[a]] for a in "01"]
    lf = cm.xor_linear_form(cfg, ffw)
    def c2_cpu():                                          # one of the four patterns; the loop is linear in the trial count
        ode = orhs.UnifiedColumnODE(lf, tv, stims[1:2].reshape(1, 1000, 32), requires_grad=True)
        y = S.odeint_dopri5(ode, torch.zeros(1, 72), tv)
        orhs.phi(y[-1, :, 16:24] - y[-1, :, 40:48])[:, 0].sum().backward()
    netd = move(net)
    netd.time_vec, netd.stim = tv.to(dev), stims.to(dev)
    y0x = torch.zeros(4, 72, device=dev)
    st = {}
    def c2_gpu():
        netd.zero_grad()
        y = odecol.odeint(netd, y0x, netd.time_vec, stats=st)
        odecol.xor_readout(y, netd).sum().backward()
    g2 = gpu_ms(c2_gpu, reps=3)
    cases["C2 xor dopri5 forward+adjoint (4 patterns, rtol 1e-7 atol 1e-9)"] = {
        "gpu_ms": g2, "cpu_oracle_ms": 4.0 * cpu_ms(c2_cpu), "cpu_note": "one pattern timed, x4",
        "accepted_steps_per_trial": [int(v) for v in st["n_accept"].tolist()]}
    # ---- C3
    torch.manual_seed(0)
    nd = {"nr_areas": 3, "areas": ["mt"] * 3, "nr_columns_per_area": [8, 4, 1], "nr_input_units": 4}
    net = odecol.ColumnNetwork(cfg, nd, torch.device("cpu"))
    stims = torch.stack([stimuli.parity_stimulus(tv, p) for p in stimuli.PARITY_PATTERNS])
    lf = cm.parity_linear_form(cfg, [net.areas[k].lateral_weights.detach().numpy() for k in "012"],
                               {1: net.areas["1"].feedforward_weights.detach().numpy(), 2: net.areas["2"].feedforward_weights.detach().numpy()},
                               net.areas["0"].input_weights.detach().numpy())
    nst = len(S.em_step_schedule(tv, 1e-3))
    dW = torch.randn(nst, 1, 1, generator=torch.Generator().manual_seed(1234)) * math.sqrt(1e-3)
    def c3_cpu():
        with torch.no_grad():
            for b in range(4):
                ode = orhs.UnifiedColumnODE(lf, tv, stims[b:b + 1])
                S.sdeint_euler(ode, torch.zeros(1, 312), tv, S.TabulatedBrownian(dW), dt=1e-3)
    netd = move(net)
    netd.time_vec, netd.stim = tv.to(dev), stims.to(dev)
    y0p = torch.zeros(4, 312, device=dev)
    dWd = dW[:, :, 0].to(dev)
    def c3_gpu():
        with torch.no_grad():
            odecol.sdeint(netd, y0p, netd.time_vec, bm=dWd, method="euler", dt=1e-3)
    cases["C3 parity Euler-Maruyama, shared Brownian path (4 patterns, 1000 steps)"] = {"gpu_ms": gpu_ms(c3_gpu), "cpu_oracle_ms": cpu_ms(c3_cpu)}
    launches = ext.last_launch_count()
    for v in cases.values():
        v["speedup_vs_cpu_oracle"] = v["cpu_oracle_ms"] / v["gpu_ms"]
    c1 = cases["C1 wta rk4 forward+backward (1 trial, 1499 steps)"]
    print(json.dumps({
        "metric": METRIC, "value": 16 * 1499 / (c1["gpu_ms"] / 1e3), "unit": UNIT, "n_gpus": 1, "steps": 5, "warmup": 2,
        "ms_per_step": c1["gpu_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "configs: BASELINE.json configs[0..2] as the reference scripts run them (1..4 trials, latency bound); "
                               "value = C1 (WTA, rk4 forward + backward, one trial)", "l2": "working sets of a few hundred kB"},
        "gpu_launches": launches, "cases": cases,
        "cpu_baseline": {"value": 16 * 1499 / (c1["cpu_oracle_ms"] / 1e3), "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": "the same C1 solve, oracle rk4 + autograd, one trial"},
    }))


def net_family(ext, odecol, net, y0, tv, args):
    from ode_column_b200.solvers import _Setup
    setup = _Setup(net, y0, tv, args.family)
    fam = setup.problem(setup.lf.W_aug).kernel_family(ext.OP_RK4_FWD)
    return {0: "persistent on-chip (FP32 FFMA)", 1: "staged FP32-FFMA", 2: "staged tcgen05, split operands (FP16 pairs forward / TF32 pairs reverse)"}.get(fam, str(fam))


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "c5":
        run_c5(args)
    elif args.workload == "small":
        run_small(args)
    elif args.workload == "configs":
        run_configs(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
