"""The Riemann-solver plugin seam on the GPU: the KPP solver of examples/user_rp/rp_kpp.cuh
(the reference's apps/kpp links rpn2_kpp.f + rpt2_dummy.f through RP_SOURCE)."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "examples"))


def _hits(a, b, p):
    return np.floor((b - p) / (2 * np.pi)) >= np.ceil((a - p) / (2 * np.pi))


def _kpp_numpy(ixy, ul, ur):
    """The formulas of rp_kpp.cuh in numpy."""
    a, b = np.minimum(ul, ur), np.maximum(ul, ur)
    if ixy == 1:
        fl, fr = np.sin(ul), np.sin(ur)
        smax = np.where(_hits(a, b, 0.0), 1.0, np.maximum(np.cos(a), np.cos(b)))
        smin = np.where(_hits(a, b, np.pi), -1.0, np.minimum(np.cos(a), np.cos(b)))
    else:
        fl, fr = np.cos(ul), np.cos(ur)
        smax = np.where(_hits(a, b, 1.5 * np.pi), 1.0, np.maximum(-np.sin(a), -np.sin(b)))
        smin = np.where(_hits(a, b, 0.5 * np.pi), -1.0, np.minimum(-np.sin(a), -np.sin(b)))
    with np.errstate(invalid="ignore", divide="ignore"):
        um = np.where(smax > smin, (smax * ur - smin * ul - (fr - fl)) / (smax - smin), ul)
    w1, w2 = um - ul, ur - um
    amdq = np.minimum(smin, 0) * w1 + np.minimum(smax, 0) * w2
    apdq = np.maximum(smin, 0) * w1 + np.maximum(smax, 0) * w2
    return np.stack([w1, w2]), np.stack([smin, smax]), amdq, apdq, fl, fr


@pytest.mark.parametrize("ixy", [1, 2])
def test_user_solver_pointwise_contract(ixy):
    """solver.rp as a callable, the reference's Python contract (doc/rp.rst): waves, speeds and
    fluctuations of the compiled-in user solver against the same formulas in numpy; the waves sum
    to the jump and the fluctuations to the flux difference (HLL is conservative)."""
    import torch
    import pyclaw
    import kpp
    rs = kpp.kpp_solver_descriptor(pyclaw)
    rng = np.random.RandomState(ixy)
    n = 5000
    ul, ur = rng.uniform(0, 4 * np.pi, n), rng.uniform(0, 4 * np.pi, n)
    ur[:200] = ul[:200]
    ql = torch.as_tensor(ul[None, :], device="cuda")
    qr = torch.as_tensor(ur[None, :], device="cuda")
    wave, s, amdq, apdq = [t.cpu().numpy() for t in rs(ql, qr, None, None, {}, ixy=ixy)]
    w_np, s_np, am_np, ap_np, fl, fr = _kpp_numpy(ixy, ul, ur)
    assert np.abs(wave[0] - w_np).max() < 1e-12 and np.abs(s - s_np).max() < 1e-14
    assert np.abs(amdq[0] - am_np).max() < 1e-12 and np.abs(apdq[0] - ap_np).max() < 1e-12
    assert np.abs(wave[0].sum(axis=0) - (ur - ul)).max() < 1e-13
    assert np.abs(amdq[0] + apdq[0] - (fr - fl)).max() < 1e-12


@pytest.mark.parametrize("solver_type", ["classic", "sharpclaw"])
def test_kpp_application_runs_on_the_user_solver(solver_type):
    import kpp
    c = kpp.kpp(solver_type=solver_type, mx=80, my=80, tfinal=0.4, nout=2)
    q0 = np.asarray(c.frames[0].q)
    q = np.asarray(c.frames[-1].q)
    assert np.isfinite(q).all() and c.frames[-1].t == 0.4
    # scalar conservation law, outflow boundaries not reached by t = 0.4: mass is conserved
    assert abs(q.sum() - q0.sum()) < 1e-9 * abs(q0.sum())
    # the solution stays (essentially) inside the initial range [pi/4, 3.5 pi]
    assert q.min() > 0.25 * np.pi - 0.05 and q.max() < 3.5 * np.pi + 0.05
    # and it did something: the rotating-wave structure has developed
    assert np.abs(q - q0).max() > 1.0


def test_user_solver_equals_builtin_when_it_is_the_same_solver():
    """A user header that restates a built-in solver (2-D advection) gives bit-identical runs."""
    import pyclaw
    hdr = os.path.join(ROOT, "examples", "user_rp", "rp_advection_user.cuh")
    rs = pyclaw.riemann.from_header(hdr, name="advuser", meqn=1, mwaves=1, ndims=(2,), param_names=["u", "v"])

    def run(rp):
        x = pyclaw.Dimension('x', 0.0, 1.0, 64)
        y = pyclaw.Dimension('y', 0.0, 1.0, 48)
        state = pyclaw.State(pyclaw.Grid([x, y]), 1)
        state.aux_global.update(u=0.7, v=-0.4)
        X, Y = np.meshgrid(state.grid.x.center, state.grid.y.center, indexing="ij")
        state.q[0] = np.exp(-60 * ((X - 0.4) ** 2 + (Y - 0.6) ** 2))
        solver = pyclaw.ClawSolver2D()
        solver.rp = rp
        solver.mwaves = 1
        solver.limiters = [4]
        solver.dim_split = False
        solver.order_trans = 2
        for i in range(2):
            solver.bc_lower[i] = solver.bc_upper[i] = pyclaw.BC.periodic
        claw = pyclaw.Controller()
        claw.tfinal, claw.nout, claw.keep_copy, claw.output_format = 0.3, 1, True, None
        claw.solution, claw.solver = pyclaw.Solution(state), solver
        claw.run()
        return np.asarray(claw.frames[-1].q)
    assert np.array_equal(run(rs), run(pyclaw.riemann.advection))


USER_PATHS = ["step1", "step2ds_1", "step2ds_2", "sharpclaw1d_f32", "sharpclaw1d_old", "sharpclaw2d_f32",
              "sharpclaw2d_old", "rp_solve", "rp_transverse"]


@pytest.mark.parametrize("path", USER_PATHS)
def test_user_paths_equal_builtin_advection(path):
    """Each 1-D / 2-D user-solver entry of the C ABI (classic 1-D step, dimensionally split sweeps,
    SharpClaw stage in both WENO literal readings, pointwise normal and transverse solves) on the
    advection header gives bit-identical results to the built-in advection solver."""
    import ctypes
    import pyclaw
    from pyclaw_b200 import _lib
    hdr = os.path.join(ROOT, "examples", "user_rp", "rp_advection_user.cuh")
    rs = pyclaw.riemann.from_header(hdr, name="advuser", meqn=1, mwaves=1, ndims=(1, 2), param_names=["u", "v"])
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)
    params = [0.7, -0.4]
    mx, my, mbc = 300, 70, 3
    dx, dy, dt = 1.0 / mx, 1.0 / my, 0.4 / mx
    rng = np.random.RandomState(len(path))
    ndim = 1 if path in ("step1", "sharpclaw1d_f32", "sharpclaw1d_old") else 2
    pad = (1, mx + 2 * mbc) if ndim == 1 else (1, mx + 2 * mbc, my + 2 * mbc)
    q = np.asfortranarray(rng.uniform(-1, 1, pad))
    n = 5000
    ql, qr, asdq = (np.ascontiguousarray(rng.uniform(-1, 1, (1, n))) for _ in range(3))

    def run(rp_id):
        out = []
        cfl = ctypes.c_double()
        if path == "step1" or path.startswith("step2ds"):
            P = _lib.make_problem(ndim, 1, 1, mbc, mx, my if ndim == 2 else 1, dx, dy, rp_id, params,
                                  [1, 2, -1, 0, 0, 0, 0], [4])
            qn = q.copy("F")
            if path == "step1":
                _lib.call("clawb200_step1_host", ctypes.byref(P), ptr(qn), None, dt, ctypes.byref(cfl))
            else:
                _lib.call("clawb200_step2ds_host", ctypes.byref(P), ptr(q), ptr(qn), None, dt, int(path[-1]),
                          ctypes.byref(cfl))
            out = [qn, cfl.value]
        elif path.startswith("sharpclaw"):
            variant = _lib.WENO_PYWENO_F32 if path.endswith("f32") else _lib.WENO_OLD
            P = _lib.make_problem(ndim, 1, 1, mbc, mx, my if ndim == 2 else 1, dx, dy, rp_id, params,
                                  weno_variant=variant)
            dq = np.zeros_like(q, order="F")
            _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), ptr(q), ptr(dq), None, dt, ctypes.byref(cfl))
            out = [dq, cfl.value]
        elif path == "rp_solve":
            for nd, ixy in ((1, 1), (2, 1), (2, 2)):
                P = _lib.make_problem(nd, 1, 1, 2, 8, 8, 1.0, 1.0, rp_id, params)
                wave, s, amdq, apdq = (np.zeros((1, n)) for _ in range(4))
                _lib.call("clawb200_rp_solve_host", ctypes.byref(P), ixy, n, ptr(ql), ptr(qr), None, None,
                          ptr(wave), ptr(s), ptr(amdq), ptr(apdq))
                out += [wave, s, amdq, apdq]
        else:
            P = _lib.make_problem(2, 1, 1, 2, 8, 8, 1.0, 1.0, rp_id, params)
            for ixy in (1, 2):
                for imp in (1, 2):
                    bm, bp = np.zeros((1, n)), np.zeros((1, n))
                    _lib.call("clawb200_rp_transverse_host", ctypes.byref(P), ixy, n, ptr(ql), ptr(qr), imp,
                              ptr(asdq), ptr(bm), ptr(bp))
                    out += [bm, bp]
        return out

    builtin = run(_lib.RP_ADVECTION)
    prev = _lib.set_variant(rs._variant())
    try:
        user = run(_lib.RP_USER)
    finally:
        _lib.set_variant(prev)
    assert len(user) == len(builtin)
    for a, b in zip(builtin, user):
        assert np.array_equal(a, b), path
    # not vacuous: the step moved the solution, dq and the fluctuations are not zero
    assert np.abs(builtin[0] - (q if path.startswith("step") else 0.0)).max() > 1e-3
