"""odeint / odeint_adjoint / sdeint-compatible entry points that run FUSED on the GPU.

They keep the call shapes of the third-party functions the reference uses

    torchdiffeq.odeint(func, y0, t, *, rtol=1e-7, atol=1e-9, method=None, options=None, event_fn=None)
        call sites: reference scripts/xor_ode.py:114, scripts/parity_ode.py:233, scripts/plotting_results.py:131
    torchsde.sdeint(sde, y0, ts, bm=None, method=None, dt=1e-3, adaptive=False, rtol=1e-5, atol=1e-4, dt_min=1e-5,
                    options=None, names=None, ...)
        call sites: reference scripts/wta_ode.py:174,200

but ``func`` / ``sde`` must be one of this package's column networks (anything with ``export_linear_form()`` and
``stimulus_channels()``): the whole time loop then runs inside the sm_100a kernels behind ``include/odecol.h``.
There is no generic-function path, no CPU path and no multi-backend dispatch -- other inputs raise.

Batching: where the reference loops over trials with B = 1 solves, pass y0 of shape (B, 3N) and a stimulus with a
leading trial dimension; the result is (T, B, 3N).

Gradients: ``method='rk4'``, ``method='dopri5'`` and fixed-step Euler-Maruyama are differentiable w.r.t. every module parameter that enters
W_aug = [W | U | bias] and w.r.t. y0, through hand-written exact discrete adjoints (what ``loss.backward()`` through
the reference's unrolled solver computes).
"""
from __future__ import annotations

from typing import Callable, Dict, Optional, Sequence, Union

import torch

from . import _native
from .stimulus import compress_knots

_DEFAULT_MAX_STEPS = 4_000_000


class _nvtx:
    """NVTX range around a fused solve / reverse sweep (shows up in ncu / nsys timelines; a few hundred nanoseconds when
    no profiler is attached).  The reference has no tracing of its own (SURVEY.md section 5)."""

    def __init__(self, name: str):
        self.name = name

    def __enter__(self):
        torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *exc):
        torch.cuda.nvtx.range_pop()
        return False


def _require_linear_form(func):
    if not (hasattr(func, "export_linear_form") and hasattr(func, "stimulus_channels")):
        raise TypeError(
            "odecol solvers integrate column networks exposing export_linear_form()/stimulus_channels(); got "
            f"{type(func).__name__}. There is no generic-function or CPU fallback.")


class _Setup:
    """Everything a solve needs besides the differentiable tensors (kept out of autograd's way)."""

    def __init__(self, func, y0: torch.Tensor, t: torch.Tensor, family: Optional[str], deterministic: Optional[bool] = None):
        _require_linear_form(func)
        if not y0.is_cuda:
            raise RuntimeError("odecol: y0 must live on a CUDA device (no CPU path); move the module and state to cuda")
        if y0.dim() != 2:
            raise ValueError("odecol: y0 must be (B, 3N)")
        self.ext = _native.ext()
        dev = y0.device
        self.lf = func.export_linear_form()
        if y0.shape[1] != 3 * self.lf.N:
            raise ValueError(f"odecol: y0 has {y0.shape[1]} components, the network needs {3 * self.lf.N}")
        self.B = y0.shape[0]
        self.t = t.detach().to(device=dev, dtype=torch.float32).contiguous()
        table = func.stimulus_channels().detach().to(device=dev, dtype=torch.float32)
        if table.shape[0] not in (1, self.B):
            raise ValueError(f"odecol: stimulus has {table.shape[0]} trials, y0 has {self.B}")
        time_vec = func.time_vec.detach().to(device=dev, dtype=torch.float32)
        self.knot_t, self.knot_u = compress_knots(time_vec, table)
        if family not in (None, "staged", "tensor"):
            raise ValueError("odecol: options['family'] must be None, 'staged' or 'tensor' (both skip the on-chip family)")
        self.flags = {None: 0, "staged": self.ext.FLAG_FORCE_STAGED, "tensor": self.ext.FLAG_FORCE_TENSOR}[family]
        # bit-reproducible gradients on request, or whenever torch itself is asked for deterministic algorithms
        if deterministic if deterministic is not None else torch.are_deterministic_algorithms_enabled():
            self.flags |= self.ext.FLAG_DETERMINISTIC
        self.kappa = self.lf.kappa.detach().to(dev, torch.float32).contiguous()
        self.sigma = self.lf.sigma.detach().to(dev, torch.float32).contiguous()
        self.sigma_scale = None       # (B,) per-trial factor on sigma, set by sdeint(options={'sigma_scale': ...})
        self.lateral_gain = None      # (B,) per-trial gain on the between-column recurrent input (sweeps), with
        self.W_local = None           # (N, 8) the within-column weights that stay unscaled

    def set_lateral_gain(self, func, gain):
        """Per-trial global lateral gain (the third axis of BASELINE.json configs[4]'s sweep): trial b integrates the network
        whose between-column weights are gain[b] times the module's.  The module says which weights those are."""
        if not hasattr(func, "lateral_split"):
            raise TypeError(f"odecol: options['lateral_gain'] needs a network with lateral_split(); {type(func).__name__} has none")
        g = torch.as_tensor(gain, dtype=torch.float32).to(self.kappa.device).reshape(-1).contiguous()
        if g.numel() != self.B:
            raise ValueError(f"odecol: options['lateral_gain'] needs {self.B} entries (one per trial), got {g.numel()}")
        if not bool((g > 0).all()):
            raise ValueError("odecol: options['lateral_gain'] must be positive")
        W_lat, W_loc = func.lateral_split()
        lf = self.lf
        n = lf.N
        W_aug = torch.cat((W_lat.detach().to(torch.float32), lf.W_aug.detach()[:, n:]), dim=1).contiguous()
        self.lf = type(lf)(W_aug=W_aug, kappa=lf.kappa, sigma=lf.sigma, n_in=lf.n_in, tau_s=lf.tau_s, tau_m=lf.tau_m,
                           tau_a=lf.tau_a, resistance=lf.resistance)
        self.lateral_gain, self.W_local = g, W_loc.detach().to(torch.float32).contiguous()
        if not (self.flags & (self.ext.FLAG_FORCE_STAGED | self.ext.FLAG_FORCE_TENSOR)):
            self.flags |= self.ext.FLAG_FORCE_STAGED      # the gain lives in the staged Euler-Maruyama kernels

    def problem(self, W_aug: torch.Tensor):
        lf = self.lf
        prob = self.ext.Problem(W_aug.detach().to(torch.float32).contiguous(), self.kappa, self.sigma, self.knot_t,
                                self.knot_u, lf.n_in, self.B, lf.tau_s, lf.tau_m, lf.tau_a, lf.resistance, self.flags)
        if self.sigma_scale is not None:
            prob.set_sigma_scale(self.sigma_scale)
        if self.lateral_gain is not None:
            prob.set_lateral_gain(self.lateral_gain, self.W_local)
        return prob


_STATUS_NAMES = {1: "state became non-finite", 2: "step budget (max_num_steps) exhausted", 3: "step size underflow"}


def _check_status(status: torch.Tensor, options: dict, what: str):
    """torchdiffeq / torchsde raise when a solve fails (max_num_steps exceeded, dt underflow); the kernels report a
    per-trial status and fill the remaining output rows with NaN, so the default is to raise here too.
    ``options={'check_status': False}`` skips the check (and the device synchronisation it costs)."""
    if not options.get("check_status", True) or status is None or status.numel() == 0:
        return
    if bool((status != 0).any()):
        bad = torch.nonzero(status != 0).flatten()[:8].tolist()
        codes = [int(status[b]) for b in bad]
        raise RuntimeError(f"odecol: {what} failed for trial(s) {bad} (first of {int((status != 0).sum())}): " +
                           "; ".join(f"trial {b}: {_STATUS_NAMES.get(c, c)}" for b, c in zip(bad, codes)) +
                           " -- pass options={'check_status': False} and stats={} to inspect the partial result")


def _sel_tensors(components, N3, device):
    """(sel_long, sel_i32, inverse) of a component selection.  The kernels map each state component to one column of
    grad_y (include/odecol.h), so they get the distinct components; when some repeat, ``_expand`` rebuilds the requested
    columns outside the autograd Functions and autograd sums the gradients of the copies, as torch.index_select does."""
    if components is None:
        return None, None, None
    idx = torch.as_tensor(components, dtype=torch.int64).flatten().cpu()
    if idx.numel() == 0 or int(idx.min()) < 0 or int(idx.max()) >= N3:
        raise ValueError("odecol: components out of range")
    inverse = None
    uniq, inv = torch.unique(idx, return_inverse=True)
    if uniq.numel() < idx.numel():
        idx, inverse = uniq, inv.to(device)
    idx = idx.to(device)
    return idx, idx.to(torch.int32).contiguous(), inverse


def _expand(y, inverse):
    return y if inverse is None else y.index_select(2, inverse)


class _RK4Function(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y0, W_aug, setup: _Setup, sel_long, sel_i32):
        prob = setup.problem(W_aug)
        with _nvtx("odecol.rk4_fwd"):
            y = setup.ext.rk4_fwd(prob, setup.t, y0.detach().to(torch.float32).contiguous(), 1)
        ctx.setup, ctx.prob, ctx.sel_i32 = setup, prob, sel_i32
        ctx.save_for_backward(y)
        return y if sel_long is None else y.index_select(2, sel_long)

    @staticmethod
    def backward(ctx, grad):
        (y,) = ctx.saved_tensors
        with _nvtx("odecol.rk4_bwd"):
            gy0, gW = ctx.setup.ext.rk4_bwd(ctx.prob, ctx.setup.t, y, grad.to(torch.float32).contiguous(), ctx.sel_i32)
        return gy0, gW, None, None, None


def _ckpt_fits(nbytes: int, device) -> bool:
    """Checkpoint mode trades memory for three contractions per reverse step; use it when the buffer fits in what the
    device has free plus what the caching allocator already holds unused, with headroom for the loss graph."""
    free, _total = torch.cuda.mem_get_info(device)
    cached = torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device)
    return nbytes <= 0.85 * (free + cached)


class _RK4CkptFunction(torch.autograd.Function):
    """rk4 on a component selection in checkpoint mode (include/odecol.h: odecol_rk4_fwd_ckpt / odecol_rk4_bwd_ckpt)."""

    @staticmethod
    def forward(ctx, y0, W_aug, setup: _Setup, sel_i32):
        prob = setup.problem(W_aug)
        with _nvtx("odecol.rk4_fwd_ckpt"):
            y_sel, ckpt = setup.ext.rk4_fwd_ckpt(prob, setup.t, y0.detach().to(torch.float32).contiguous(), sel_i32)
        ctx.setup, ctx.prob, ctx.sel_i32 = setup, prob, sel_i32
        ctx.save_for_backward(ckpt)
        return y_sel

    @staticmethod
    def backward(ctx, grad):
        (ckpt,) = ctx.saved_tensors
        with _nvtx("odecol.rk4_bwd_ckpt"):
            gy0, gW = ctx.setup.ext.rk4_bwd_ckpt(ctx.prob, ctx.setup.t, ckpt, grad.to(torch.float32).contiguous(), ctx.sel_i32)
        return gy0, gW, None, None


class _EMFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y0, W_aug, setup: _Setup, dW, seed, trial_offset, dt, n_steps, sel_long, sel_i32, stats):
        prob = setup.problem(W_aug)
        need_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        y, na, nr, st, ysteps = setup.ext.em_fwd(prob, setup.t, y0.detach().to(torch.float32).contiguous(), dW, seed,
                                                 trial_offset, dt, False, 0.0, 0.0, 0.0, n_steps if need_grad else 0)
        if stats is not None:
            stats.update(n_accept=na, n_reject=nr, status=st)
        ctx.setup, ctx.prob, ctx.sel_i32, ctx.dt = setup, prob, sel_i32, dt
        ctx.save_for_backward(ysteps)
        return y if sel_long is None else y.index_select(2, sel_long)

    @staticmethod
    def backward(ctx, grad):
        (ysteps,) = ctx.saved_tensors
        gy0, gW = ctx.setup.ext.em_bwd(ctx.prob, ctx.setup.t, ysteps, grad.to(torch.float32).contiguous(), ctx.sel_i32, ctx.dt)
        return (gy0, gW) + (None,) * 9


class _SRKFunction(torch.autograd.Function):
    """torchsde method='srk' (SRI2, fixed step) and its discrete adjoint (include/odecol.h: odecol_srk_fwd / _bwd)."""

    @staticmethod
    def forward(ctx, y0, W_aug, setup: _Setup, dW, dU, seed, trial_offset, dt, n_steps, sel_long, sel_i32, stats):
        prob = setup.problem(W_aug)
        need_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        y, st, ysteps = setup.ext.srk_fwd(prob, setup.t, y0.detach().to(torch.float32).contiguous(), dW, dU, seed,
                                          trial_offset, dt, n_steps if need_grad else 0)
        if stats is not None:
            stats.update(status=st)
        ctx.setup, ctx.prob, ctx.sel_i32, ctx.dt = setup, prob, sel_i32, dt
        ctx.noise = (dW, dU, seed, trial_offset)
        ctx.save_for_backward(ysteps)
        return y if sel_long is None else y.index_select(2, sel_long)

    @staticmethod
    def backward(ctx, grad):
        (ysteps,) = ctx.saved_tensors
        dW, dU, seed, trial_offset = ctx.noise
        gy0, gW = ctx.setup.ext.srk_bwd(ctx.prob, ctx.setup.t, ysteps, dW, dU, seed, trial_offset,
                                        grad.to(torch.float32).contiguous(), ctx.sel_i32, ctx.dt)
        return (gy0, gW) + (None,) * 10


def odeint(func, y0, t, *, rtol=1e-7, atol=1e-9, method=None, options=None, event_fn=None,
           components=None, stats: Optional[Dict] = None):
    """Fused replacement of ``torchdiffeq.odeint``.  ``method``: None/'dopri5' (adaptive, per-trial control, the
    default the reference scripts get) or 'rk4' (3/8 rule on the grid ``t``); both for every network size, both
    differentiable (exact discrete adjoints).  Extras beyond torchdiffeq:
    ``components`` restricts the returned trajectory to those state components (T, B, len(components));
    ``stats`` (a dict) receives per-trial n_accept / n_reject / status tensors; ``options['family']='staged'`` (or
    ``'tensor'``, the same) forces the global-state kernel family, for rk4 the tcgen05 tensor family,
    ``options['max_num_steps']`` bounds dopri5, ``options['deterministic']=True`` (default:
    ``torch.are_deterministic_algorithms_enabled()``) makes the tensor family's rk4 gradients bit-reproducible (fixed-order
    reduction over trials instead of float atomics, about 2 % slower)."""
    if event_fn is not None:
        raise NotImplementedError("odecol: event handling is not part of the fused path")
    options = dict(options or {})
    method = method or "dopri5"
    setup = _Setup(func, y0, t, options.pop("family", None), options.pop("deterministic", None))
    sel_long, sel_i32, inverse = _sel_tensors(components, 3 * setup.lf.N, y0.device)
    if method == "rk4":
        if options.get("step_size") is not None:
            raise NotImplementedError("odecol rk4 integrates on the grid `t` (the reference passes no step_size)")
        ckpt = options.get("checkpoint", "auto")      # 'auto' | True | False
        needs_grad = torch.is_grad_enabled() and (y0.requires_grad or setup.lf.W_aug.requires_grad)
        if sel_i32 is not None and needs_grad and ckpt is not False:
            nbytes = setup.ext.rk4_ckpt_bytes(setup.problem(setup.lf.W_aug), setup.t.numel())
            if nbytes > 0 and (ckpt is True or _ckpt_fits(nbytes, y0.device)):
                return _expand(_RK4CkptFunction.apply(y0, setup.lf.W_aug, setup, sel_i32), inverse)
            if ckpt is True:
                raise RuntimeError("odecol: checkpoint mode is not available for this problem (tensor family only)")
        return _expand(_RK4Function.apply(y0, setup.lf.W_aug, setup, sel_long, sel_i32), inverse)
    if method == "dopri5":
        # torchdiffeq rejects such a grid; the kernels would emit NaN (on-chip) or y0 (staged) at a repeated time
        if setup.t.numel() > 1 and not bool((setup.t[1:] > setup.t[:-1]).all()):
            raise ValueError("odecol: dopri5 needs a strictly increasing time grid t")
        if torch.is_grad_enabled() and (y0.requires_grad or setup.lf.W_aug.requires_grad):
            from .dopri5_adjoint import dopri5_with_grad   # discrete adjoint through the accepted steps (both families)
            return _expand(dopri5_with_grad(setup, y0, rtol, atol, options, sel_long, sel_i32, stats), inverse)
        prob = setup.problem(setup.lf.W_aug)
        y, na, nr, st = setup.ext.dopri5_fwd(prob, setup.t, y0.detach().to(torch.float32).contiguous(), float(rtol),
                                             float(atol), int(options.get("max_num_steps", _DEFAULT_MAX_STEPS)))
        if stats is not None:
            stats.update(n_accept=na, n_reject=nr, status=st)
        _check_status(st, options, "dopri5")
        return y if sel_long is None else _expand(y.index_select(2, sel_long), inverse)
    raise ValueError(f"odecol: method {method!r} is not fused (have 'rk4', 'dopri5')")


def odeint_adjoint(func, y0, t, *, rtol=1e-7, atol=1e-9, method=None, options=None, event_fn=None,
                   adjoint_rtol=None, adjoint_atol=None, adjoint_method=None, adjoint_options=None,
                   adjoint_params=None, components=None, stats=None):
    """Signature of ``torchdiffeq.odeint_adjoint`` (imported but never called by the reference).  The fused solvers
    already run their backward pass inside a kernel from O(T) saved states, so this is ``odeint``; the adjoint_*
    arguments are accepted for compatibility."""
    return odeint(func, y0, t, rtol=rtol, atol=atol, method=method, options=options, event_fn=event_fn,
                  components=components, stats=stats)


def _tabulate_bm(bm, ts_cpu: torch.Tensor, dt: float, B: int, device, with_u: bool = False):
    """Increments of a torchsde-style Brownian object along the fixed-step schedule (float32 time loop); with_u also
    tabulates the space-time Levy areas ``bm(t0, t1, return_U=True)`` hands to the srk scheme."""
    out, out_u = [], []
    curr = ts_cpu[0].clone()
    t_end = ts_cpu[-1]
    row = lambda v: (lambda w: w.expand(B) if w.numel() == 1 else w)(torch.as_tensor(v, dtype=torch.float32).reshape(-1))
    for out_t in ts_cpu[1:]:
        while curr < out_t:
            nxt = torch.minimum(curr + dt, t_end)
            if with_u:
                w, u = bm(curr, nxt, return_U=True)
                out_u.append(row(u))
            else:
                w = bm(curr, nxt)
            out.append(row(w))
            curr = nxt
    W = torch.stack(out).to(device).contiguous()
    return (W, torch.stack(out_u).to(device).contiguous()) if with_u else W


def _increment_table(x, n_steps: int, B: int, device) -> torch.Tensor:
    x = x.detach().to(device, torch.float32).reshape(x.shape[0], -1)
    if x.shape[1] == 1 and B > 1:
        x = x.expand(-1, B)
    if x.shape != (n_steps, B):
        raise ValueError(f"odecol: need Brownian increments of shape ({n_steps}, {B}), got {tuple(x.shape)}")
    return x.contiguous()


def sdeint(sde, y0, ts, bm=None, method=None, dt=1e-3, adaptive=False, rtol=1e-5, atol=1e-4, dt_min=1e-5,
           options=None, names=None, logqp=False, extra=False, extra_solver_state=None,
           seed: Optional[int] = None, trial_offset: int = 0, components=None, stats: Optional[Dict] = None):
    """Fused replacement of ``torchsde.sdeint`` for scalar-noise Ito SDEs: ``method='euler'`` (Euler-Maruyama) and
    ``method='srk'`` (Roessler SRI2 with torchsde's SRID2 tableau -- what the reference scripts name; also torchsde's
    default for this noise type, so ``method=None`` selects it).

    ``bm``: None -> in-kernel Philox4x32-10 noise keyed by (seed, trial_offset + trial index); a tensor (n_steps, B)
    or (n_steps, B, 1) of increments in step order (bit-parity mode, fixed step) -- for 'srk' a pair ``(W, U)`` of such
    tensors, U the space-time Levy area of each step; or a torchsde-style callable ``bm(t0, t1)`` /
    ``bm(t0, t1, return_U=True)``, tabulated along the step schedule.  ``adaptive=True`` uses step doubling with
    torchsde's controller, per trial, on a virtual Brownian tree (Philox only): 'euler' for every network size, 'srk' (on
    a Levy-area-consistent tree) for the on-chip family.
    ``seed``: None -> a fresh key from torch's global generator on every call (independent paths per call, as torchsde's
    fresh BrownianInterval gives; ``torch.manual_seed`` reproduces a run); an int fixes the paths.  ``trial_offset``: the
    GLOBAL index of this call's first trial.  A job sharded over ranks or chunks passes ONE seed everywhere and
    ``trial_offset = lo`` of its block (``distributed.shard_bounds``): trial t then sees the same Brownian path wherever
    it runs, and results do not depend on the sharding -- with one exception: when a firing rate of some trial does not
    fit the FP16 operand pairs of the staged solvers, they repeat the whole call in TF32 pairs, so that trial's batch mates
    change in the last bits.
    ``options['sigma_scale']``: (B,) per-trial factor on the diffusion -- the noise-amplitude axis of a parameter sweep
    (trial b integrates with g = sigma_scale[b] * diffusion); ``options['lateral_gain']``: (B,) positive per-trial gain on
    the between-column recurrent weights (networks with ``lateral_split()``, e.g. ``SyntheticColumnSheet``; Euler-Maruyama,
    under ``torch.no_grad()``) -- the lateral-gain axis of the same sweep; ``options['family']`` as in ``odeint``."""
    if logqp or extra or extra_solver_state is not None:
        raise NotImplementedError("odecol: logqp / extra solver state are not part of the fused path")
    method = method or "srk"
    if method not in ("euler", "srk"):
        raise NotImplementedError(f"odecol: sdeint method {method!r} is not fused (have 'euler', 'srk')")
    if getattr(sde, "noise_type", "scalar") != "scalar" or getattr(sde, "sde_type", "ito") != "ito":
        raise ValueError("odecol: only scalar-noise Ito SDEs (what the reference declares) are supported")
    options = dict(options or {})
    sigma_scale = options.pop("sigma_scale", None)
    lateral_gain = options.pop("lateral_gain", None)
    setup = _Setup(sde, y0, ts, options.pop("family", None))
    if lateral_gain is not None:
        if method != "euler":
            raise NotImplementedError("odecol: options['lateral_gain'] is fused for method='euler' (fixed step and adaptive)")
        if torch.is_grad_enabled() and (y0.requires_grad or setup.lf.W_aug.requires_grad):
            raise NotImplementedError("odecol: options['lateral_gain'] is a forward (sweep) feature; wrap the call in torch.no_grad()")
        setup.set_lateral_gain(sde, lateral_gain)
    if sigma_scale is not None:
        sc = torch.as_tensor(sigma_scale, dtype=torch.float32).to(y0.device).reshape(-1).contiguous()
        if sc.numel() != setup.B:
            raise ValueError(f"odecol: options['sigma_scale'] needs {setup.B} entries (one per trial), got {sc.numel()}")
        setup.sigma_scale = sc
    sel_long, sel_i32, inverse = _sel_tensors(components, 3 * setup.lf.N, y0.device)
    ext = setup.ext
    if seed is None:
        # torchsde builds a fresh BrownianInterval (new entropy) per call: draw a new key from torch's global generator, so
        # successive calls see independent paths and torch.manual_seed still reproduces a run
        seed = int(torch.randint(0, 2 ** 62, (), dtype=torch.int64).item())
    dt = float(dt)
    if adaptive:
        if bm is not None:
            raise NotImplementedError("odecol: adaptive stepping draws from the in-kernel Brownian tree; pass bm=None")
        prob = setup.problem(setup.lf.W_aug)
        if method == "srk":
            if prob.kernel_family(ext.OP_SRK_FWD) != 0:
                raise NotImplementedError("odecol: adaptive srk is fused for the on-chip family (N <= 128, the reference's "
                                          "networks); larger networks: method='euler' with adaptive=True, or fixed-step srk")
            y, na, nr, st = ext.srk_fwd_adaptive(prob, setup.t, y0.detach().to(torch.float32).contiguous(), seed, int(trial_offset),
                                                 dt, float(rtol), float(atol), float(dt_min))
            if stats is not None:
                stats.update(n_accept=na, n_reject=nr, status=st)
            _check_status(st, options, "adaptive srk")
            return y if sel_long is None else _expand(y.index_select(2, sel_long), inverse)
        y, na, nr, st, _ = ext.em_fwd(prob, setup.t, y0.detach().to(torch.float32).contiguous(), None, seed,
                                      int(trial_offset), dt, True, float(rtol), float(atol), float(dt_min), 0)
        if stats is not None:
            stats.update(n_accept=na, n_reject=nr, status=st)
        _check_status(st, options, "adaptive Euler-Maruyama")
        return y if sel_long is None else _expand(y.index_select(2, sel_long), inverse)
    ts_cpu = setup.t.cpu()
    n_steps = int(ext.em_num_steps(ts_cpu, dt))
    if method == "srk":
        dW = dU = None
        if bm is not None:
            if isinstance(bm, (tuple, list)) and len(bm) == 2 and all(torch.is_tensor(x) for x in bm):
                dW, dU = (_increment_table(x, n_steps, setup.B, y0.device) for x in bm)
            elif torch.is_tensor(bm):
                raise ValueError("odecol: method='srk' needs the pair (W, U) of increment tables, or a callable bm")
            else:
                dW, dU = _tabulate_bm(bm, ts_cpu, dt, setup.B, y0.device, with_u=True)
                if dW.shape != (n_steps, setup.B):
                    raise ValueError(f"odecol: bm produced increments of shape {tuple(dW.shape)}")
        return _expand(_SRKFunction.apply(y0, setup.lf.W_aug, setup, dW, dU, seed, int(trial_offset), dt, n_steps, sel_long,
                                          sel_i32, stats), inverse)
    dW = None
    if bm is not None:
        if torch.is_tensor(bm):
            dW = _increment_table(bm, n_steps, setup.B, y0.device)
        else:
            dW = _tabulate_bm(bm, ts_cpu, dt, setup.B, y0.device)
            if dW.shape != (n_steps, setup.B):
                raise ValueError(f"odecol: bm produced increments of shape {tuple(dW.shape)}")
    return _expand(_EMFunction.apply(y0, setup.lf.W_aug, setup, dW, seed, int(trial_offset), dt, n_steps, sel_long, sel_i32, stats),
                   inverse)


def sdeint_adjoint(sde, y0, ts, bm=None, method=None, adjoint_method=None, dt=1e-3, adaptive=False, adjoint_adaptive=False,
                   rtol=1e-5, adjoint_rtol=1e-5, atol=1e-4, adjoint_atol=1e-4, dt_min=1e-5, options=None,
                   adjoint_options=None, adjoint_params=None, names=None, logqp=False, extra=False,
                   extra_solver_state=None, **kwargs):
    """Signature of ``torchsde.sdeint_adjoint`` (imported but never called by the reference scripts,
    scripts/wta_ode.py:9, xor_ode.py:2, parity_ode.py:10).  The fused solvers already run their backward pass inside a
    kernel from the saved solver states, so this is ``sdeint``; the adjoint_* arguments are accepted for compatibility."""
    return sdeint(sde, y0, ts, bm=bm, method=method, dt=dt, adaptive=adaptive, rtol=rtol, atol=atol, dt_min=dt_min,
                  options=options, names=names, logqp=logqp, extra=extra, extra_solver_state=extra_solver_state, **kwargs)
