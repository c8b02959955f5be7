"""The C-ABI shared library loads without a GPU and exports every symbol include/odecol.h declares."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "ode-column_b200", "lib", "libodecol.so")


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(LIB):
        import importlib.util
        spec = importlib.util.spec_from_file_location("odecol_build", os.path.join(ROOT, "ode-column_b200", "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build()
    return ctypes.CDLL(LIB)


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "odecol.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(odecol_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported(lib):
    names = declared_symbols()
    assert len(names) >= 12
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/odecol.h but not exported"


def test_version_and_strerror(lib):
    assert lib.odecol_abi_version() == 3
    lib.odecol_strerror.restype = ctypes.c_char_p
    assert lib.odecol_strerror(0) == b"ok"
    assert b"workspace" in lib.odecol_strerror(-4)


def test_null_problem_is_rejected_without_touching_the_gpu(lib):
    lib.odecol_rk4_fwd.restype = ctypes.c_int
    rc = lib.odecol_rk4_fwd(None, None, 4, None, None, 1, None, ctypes.c_size_t(0), None)
    assert rc == -1


def test_em_num_steps_matches_oracle_schedule(lib):
    from oracle import solvers, stimuli
    lib.odecol_em_num_steps.restype = ctypes.c_int64
    lib.odecol_em_num_steps.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_float]
    for T, dt_grid, dt in ((1500, 1e-4, 1e-3), (1000, 1e-3, 1e-3), (1000, 1e-3, 2.5e-4), (37, 0.01, 0.003)):
        ts = stimuli.time_vec(T, dt_grid).contiguous()
        n = lib.odecol_em_num_steps(ts.data_ptr(), T, dt)
        assert n == len(solvers.em_step_schedule(ts, dt))


def test_torch_extension_imports_without_gpu():
    import odecol
    e = odecol._native.ext()
    assert e.abi_version() == 3
    with pytest.raises(RuntimeError):
        # CPU tensors are refused: there is no CPU path
        e.Problem(torch.zeros(8, 12), torch.zeros(8), None, torch.zeros(2), torch.zeros(1, 2, 1), 1, 1, 5e-4, 0.02, 10.0, 80.0, 0)


# ---------------------------------------------------------------------------------------------------------------
# argument validation happens before anything touches the GPU: error codes, never a crash (edge cases: empty batch,
# single grid point, ragged / misaligned buffers, inconsistent optional tables)
# ---------------------------------------------------------------------------------------------------------------
class _Problem(ctypes.Structure):
    _fields_ = [("N", ctypes.c_int32), ("n_in", ctypes.c_int32), ("B", ctypes.c_int32), ("K", ctypes.c_int32),
                ("ld_w", ctypes.c_int32), ("flags", ctypes.c_int32), ("W_aug", ctypes.c_void_p),
                ("kappa", ctypes.c_void_p), ("sigma", ctypes.c_void_p), ("knot_t", ctypes.c_void_p),
                ("knot_u", ctypes.c_void_p), ("knot_stride_b", ctypes.c_int64), ("tau_s", ctypes.c_float),
                ("tau_m", ctypes.c_float), ("tau_a", ctypes.c_float), ("resistance", ctypes.c_float),
                ("sigma_scale", ctypes.c_void_p), ("lat_gain", ctypes.c_void_p), ("W_local", ctypes.c_void_p)]


def _problem(**kw):
    fake = 0x7F0000001000                      # never dereferenced on the host; 16-byte aligned
    base = dict(N=16, n_in=16, B=4, K=6, ld_w=36, flags=0, W_aug=fake, kappa=fake, sigma=None, knot_t=fake, knot_u=fake,
                knot_stride_b=96, tau_s=5e-4, tau_m=0.02, tau_a=10.0, resistance=80.0, sigma_scale=None, lat_gain=None, W_local=None)
    base.update(kw)
    return _Problem(**base)


def test_struct_layout_matches_the_header(lib):
    # 6 int32, 5 pointers, int64, 4 floats, 1 pointer (ABI v2), 2 pointers (ABI v3) -- what a cgo / ctypes binding sees
    assert ctypes.sizeof(_Problem) == 6 * 4 + 5 * 8 + 8 + 4 * 4 + 8 + 2 * 8
    hdr = open(os.path.join(ROOT, "include", "odecol.h")).read()
    body = hdr[hdr.index("typedef struct odecol_problem {"):hdr.index("} odecol_problem;")]
    names = re.findall(r"\b(?:int32_t|int64_t|float|const float\*)\s+([a-z_A-Z, ]+);", re.sub(r"/\*.*?\*/", "", body, flags=re.S))
    flat = [n.strip() for group in names for n in group.split(",")]
    assert flat == [f[0] for f in _Problem._fields_]


def test_shape_and_pointer_validation_without_a_gpu(lib):
    E_NULL, E_SHAPE, E_UNSUPPORTED, E_WORKSPACE, E_ALIGN = -1, -2, -3, -4, -6
    fake = ctypes.c_void_p(0x7F0000002000)
    rk4 = lib.odecol_rk4_fwd
    rk4.restype = ctypes.c_int
    rk4.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                    ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    call = lambda p, T=10, every=1, y0=fake: rk4(ctypes.byref(p), fake, T, y0, fake, every, None, 0, None)
    assert call(_problem(B=0)) == E_SHAPE                      # empty batch
    assert call(_problem(N=0)) == E_SHAPE
    assert call(_problem(K=1)) == E_SHAPE                      # a stimulus needs two knots
    assert call(_problem(ld_w=32)) == E_SHAPE                  # row shorter than N + n_in + 1
    assert call(_problem(ld_w=35)) == E_SHAPE                  # not a multiple of 4
    assert call(_problem(W_aug=0x7F0000001004)) == E_ALIGN
    assert call(_problem(kappa=None)) == E_NULL
    assert call(_problem(), T=1) == E_SHAPE                    # a single grid point is not a solve
    assert call(_problem(), every=0) == E_SHAPE
    assert call(_problem(), y0=None) == E_NULL
    assert call(_problem(lat_gain=0x7F0000003000)) == E_UNSUPPORTED   # the lateral-gain axis exists in the staged EM path only
    # srk: increments come as a (W, U) pair or not at all; only the on-chip family implements it
    srk = lib.odecol_srk_fwd
    srk.restype = ctypes.c_int
    srk.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                    ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p,
                    ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    p = _problem()
    assert srk(ctypes.byref(p), fake, 10, fake, fake, fake, None, 0, 0, 1e-3, None, None, None, 0, None) == E_NULL
    assert srk(ctypes.byref(p), fake, 10, fake, fake, None, None, 0, 0, 0.0, None, None, None, 0, None) == E_SHAPE
    big = _problem(N=512, n_in=64, ld_w=580)
    # beyond the on-chip family the staged solver takes over: it wants its workspace (with or without a state record)
    assert srk(ctypes.byref(big), fake, 10, fake, fake, None, None, 0, 0, 1e-3, None, None, None, 0, None) == E_WORKSPACE
    assert srk(ctypes.byref(big), fake, 10, fake, fake, None, None, 0, 0, 1e-3, None, fake, None, 0, None) == E_WORKSPACE
    # reverse sweeps insist on their workspace and on a sane component selection
    bwd = lib.odecol_em_bwd
    bwd.restype = ctypes.c_int
    bwd.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                    ctypes.c_void_p, ctypes.c_int32, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                    ctypes.c_size_t, ctypes.c_void_p]
    assert bwd(ctypes.byref(p), fake, 10, fake, 9, fake, None, 48, 1e-3, fake, fake, None, 0, None) == E_WORKSPACE
    assert bwd(ctypes.byref(p), fake, 10, fake, 9, fake, None, 49, 1e-3, fake, fake, None, 0, None) == E_SHAPE
    assert bwd(ctypes.byref(p), fake, 10, fake, 0, fake, None, 48, 1e-3, fake, fake, None, 0, None) == E_SHAPE
    assert bwd(ctypes.byref(big), fake, 10, fake, 9, fake, None, 3 * 512, 1e-3, fake, fake, None, 0, None) == E_WORKSPACE   # staged sweep
    # generators / read-outs
    ww = lib.odecol_ww_generate
    ww.restype = ctypes.c_int
    ww.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                   ctypes.c_double, ctypes.c_uint64, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]
    assert ww(fake, None, 0, 5001, 10, 1500, 0.0, 0, 0, fake, None) == E_SHAPE
    assert ww(fake, None, 4, 5001, 10, 1502, 0.0, 0, 0, fake, None) == E_SHAPE      # more rows than recorded updates
    assert ww(None, None, 4, 5001, 10, 1500, 0.0, 0, 0, fake, None) == E_NULL
    hub = lib.odecol_huber_rate_loss
    hub.restype = ctypes.c_int
    hub.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p,
                    ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p,
                    ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    assert hub(fake, 10, 4, 2, 0, None, fake, 0, 0, 0, 1.0, fake, fake, fake, 8, None) == E_SHAPE
    assert hub(fake, 10, 4, 2, 1, None, fake, 0, 0, 0, 0.0, fake, fake, fake, 8, None) == E_SHAPE
    assert hub(fake, 10, 4, 2, 1, None, fake, 0, 0, 0, 1.0, fake, fake, None, 0, None) == E_WORKSPACE
    # round-2 entry points: window read-out, Brownian queries, adaptive srk, the dopri5 record / reverse pair, the staged drift
    win = lib.odecol_window_rate_l1_loss
    win.restype = ctypes.c_int
    win.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p,
                    ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                    ctypes.c_size_t, ctypes.c_void_p]
    assert win(fake, 100, 4, 8, 101, None, fake, fake, fake, fake, fake, fake, 8, None) == E_SHAPE      # window longer than the solve
    assert win(fake, 100, 4, 8, 0, None, fake, fake, fake, fake, fake, fake, 8, None) == E_SHAPE
    assert win(fake, 100, 4, 8, 100, None, fake, fake, fake, fake, None, fake, 8, None) == E_NULL        # grad_w is not optional
    assert win(fake, 100, 4, 8, 100, None, fake, fake, fake, fake, fake, None, 0, None) == E_WORKSPACE
    for name in ("odecol_brownian_query", "odecol_brownian_levy_query"):
        fn = getattr(lib, name)
        fn.restype = ctypes.c_int
        extra = [ctypes.c_void_p] if name.endswith("levy_query") else []
        fn.argtypes = [ctypes.c_uint64, ctypes.c_int64, ctypes.c_int32, ctypes.c_float, ctypes.c_float, ctypes.c_void_p,
                       ctypes.c_int32, ctypes.c_void_p] + extra + [ctypes.c_void_p]
        tail = [fake] * len(extra) + [None]
        assert fn(0, 0, 4, 0.0, 0.0, fake, 3, fake, *tail) == E_SHAPE                # empty span
        assert fn(0, 0, 0, 0.0, 1.0, fake, 3, fake, *tail) == E_SHAPE
        assert fn(0, 0, 4, 0.0, 1.0, None, 3, fake, *tail) == E_NULL
    asrk = lib.odecol_srk_fwd_adaptive
    asrk.restype = ctypes.c_int
    asrk.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                     ctypes.c_int64, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_void_p,
                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    assert asrk(ctypes.byref(big), fake, 10, fake, fake, 0, 0, 1e-3, 1e-5, 1e-4, 1e-5, None, None, None, None, 0, None) == E_UNSUPPORTED
    assert asrk(ctypes.byref(p), fake, 10, fake, fake, 0, 0, 1e-3, 1e-5, 1e-4, 0.0, None, None, None, None, 0, None) == E_SHAPE
    assert asrk(ctypes.byref(p), fake, 10, None, fake, 0, 0, 1e-3, 1e-5, 1e-4, 1e-5, None, None, None, None, 0, None) == E_NULL
    rec = lib.odecol_dopri5_fwd_record
    rec.restype = ctypes.c_int
    rec.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_float,
                    ctypes.c_float, ctypes.c_int32] + [ctypes.c_void_p] * 8 + [ctypes.c_int32, ctypes.c_void_p, ctypes.c_size_t,
                                                                            ctypes.c_void_p]
    assert rec(ctypes.byref(big), fake, 10, fake, fake, 1e-7, 1e-9, 100, fake, fake, fake, fake, fake, fake, fake, fake, 64,
               None, 0, None) == E_WORKSPACE                                            # staged record pass wants its workspace
    assert rec(ctypes.byref(big), fake, 10, fake, fake, 1e-7, 1e-9, 100, fake, fake, fake, fake, fake, fake, fake, fake, 0,
               None, 0, None) == E_SHAPE
    dbw = lib.odecol_dopri5_bwd
    dbw.restype = ctypes.c_int
    dbw.argtypes = [ctypes.c_void_p, ctypes.c_int32] + [ctypes.c_void_p] * 5 + [ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p,
                                                                                ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p,
                                                                                ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t,
                                                                                ctypes.c_void_p]
    assert dbw(ctypes.byref(big), 10, fake, fake, fake, fake, fake, 64, fake, fake, None, 3 * 512, fake, fake, None, 0, None) == E_WORKSPACE
    drift = lib.odecol_drift_staged
    drift.restype = ctypes.c_int
    drift.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    assert drift(ctypes.byref(big), fake, fake, fake, None, 0, None) == E_WORKSPACE
    assert drift(ctypes.byref(big), fake, None, fake, None, 0, None) == E_NULL
    # bookkeeping helpers answer without a device
    wsb = lib.odecol_workspace_bytes
    wsb.restype = ctypes.c_size_t
    wsb.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int32, ctypes.c_int64]
    assert wsb(ctypes.byref(p), 1, 1500, 0) == 0                 # on-chip family: no workspace
    assert wsb(ctypes.byref(p), 7, 1500, 150) > 0                # srk reverse sweep: the step schedule
    assert wsb(ctypes.byref(_problem(B=0)), 1, 1500, 0) == 0
    assert wsb(ctypes.byref(big), 8, 100, 0) > wsb(ctypes.byref(big), 3, 100, 0) > 0      # dopri5 reverse / forward, staged family
    gain = _problem(N=512, n_in=64, ld_w=580, lat_gain=0x7F0000003000)
    assert wsb(ctypes.byref(gain), 4, 3, 0) > wsb(ctypes.byref(big), 4, 3, 0)              # lateral-gain sweeps: two more planes
    fam = lib.odecol_kernel_family
    fam.restype = ctypes.c_int
    fam.argtypes = [ctypes.c_void_p, ctypes.c_int]
    assert fam(ctypes.byref(p), 1) == 0 and fam(ctypes.byref(big), 1) == 2 and fam(ctypes.byref(_problem(N=0)), 1) == -1
    assert fam(ctypes.byref(_problem(N=160, n_in=20, ld_w=184)), 1) == 2            # beyond the on-chip family: tensor cores
    assert fam(ctypes.byref(_problem(N=160, n_in=20, ld_w=184, flags=1)), 1) == 2   # ... whichever staged family is forced
    assert fam(ctypes.byref(_problem(N=162, n_in=20, ld_w=184)), 1) == 2            # N not a multiple of 4: unsupported there
    # the parity network (N = 104) fits the on-chip family, but from 4096 trials its rk4 runs on the tensor cores; the adaptive
    # and stochastic solvers stay on chip, and so do the small networks at any batch size
    par = dict(N=104, n_in=4, ld_w=112)
    assert fam(ctypes.byref(_problem(B=4095, **par)), 1) == 0 and fam(ctypes.byref(_problem(B=4096, **par)), 1) == 2
    assert fam(ctypes.byref(_problem(B=4096, **par)), 2) == 2 and fam(ctypes.byref(_problem(B=4096, **par)), 3) == 0
    assert fam(ctypes.byref(_problem(B=65536)), 1) == 0
    assert wsb(ctypes.byref(_problem(B=4096, **par)), 1, 100, 0) > 0 and wsb(ctypes.byref(_problem(B=4095, **par)), 1, 100, 0) == 0


def test_error_codes_become_python_exceptions_not_crashes():
    # regression: the message of a failing entry point used to be assembled with an ostream << int, which crashed
    # inside the extension module (every error code was a segmentation fault); CPU-testable through check_code
    import odecol
    e = odecol._native.ext()
    e.check_code(0)
    for code, text in ((-1, "NULL"), (-2, "out of range"), (-3, "no kernel"), (-4, "workspace"), (-5, "CUDA"), (-6, "aligned")):
        with pytest.raises(RuntimeError, match=text) as ei:
            e.check_code(code)
        assert f"({code})" in str(ei.value) and "self-test" in str(ei.value)
