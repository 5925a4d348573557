"""The 3-D f-wave path (step3.cuh with the sign(s) lead factor, sharpclaw3.cuh) for the f-wave transport
solver vc_advection_fwave_3d (aux = {u, v, w} per cell): the device against the CPU restatement oracle3d
bit for bit (split, unsplit, pointwise, SharpClaw), the user header rp_fwave3d_user.cuh against the
built-in solver, periodic conservation, the fma build, the transport3d application and its convergence,
and the argument checks."""
import ctypes
import os
import sys

import numpy as np
import pytest

import oracle3d as o3
from pyclaw_b200 import _lib

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FW = o3.RP_ADVECTION3D_VC_FWAVE
ERR_INVALID, ERR_UNSUPPORTED = -1, -2  # CLAWB200_ERR_*
SHAPES = [(9, 7, 5), (130, 6, 4), (20, 33, 17), (5, 4, 70)]
D = (0.02, 0.025, 0.03)


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _fields(pad, seed, nq=1):
    """Random q and a random velocity field with sign changes everywhere, blocks at rest and a block in
    which neighbouring cells have opposite velocities (s == 0 at their interfaces)."""
    rng = np.random.RandomState(seed)
    q = np.asfortranarray(rng.uniform(-1, 1, (nq,) + pad))
    aux = rng.uniform(-1.5, 1.5, (3,) + pad)
    aux[:, :3, :3, :] = 0.0
    blk = aux[:, -4:, -4:, :]
    sign = (-1.0) ** (np.indices(blk.shape[1:]).sum(0))
    aux[:, -4:, -4:, :] = 0.75 * sign
    return q, np.asfortranarray(aux)


def _step_host(fn, P, mz, q, aux, dt, idir=None):
    qn = np.zeros_like(q, order="F")
    cfl = ctypes.c_double()
    args = [ctypes.byref(P), mz, D[2], _ptr(q), _ptr(qn), _ptr(aux), dt] + ([idir] if idir else [])
    _lib.call(fn, *(args + [ctypes.byref(cfl)]))
    return qn, cfl.value


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("lim", [4, 0, 2])
def test_step3ds_vs_oracle(shape, lim):
    mx, my, mz = shape
    mbc = 2
    pad = (mx + 2 * mbc, my + 2 * mbc, mz + 2 * mbc)
    q, aux = _fields(pad, mx + 10 * my + lim)
    method = [1, 1 if lim == 0 else 2, -1, 0, 0, 0, 3]
    P = _lib.make_problem(3, 1, 1, mbc, mx, my, D[0], D[1], FW, [], method, [lim], maux=3)
    dt = 0.004
    for idir in (1, 2, 3):
        qn_o = q.copy("F")
        cfl_o = o3.step3ds(FW, [], mbc, mx, my, mz, q, qn_o, *D, dt, method, [lim], idir, aux=aux)
        qn_g, cfl_g = _step_host("clawb200_step3ds_host", P, mz, q, aux, dt, idir)
        assert np.array_equal(qn_g, qn_o), (idir, np.abs(qn_g - qn_o).max())
        assert cfl_g == cfl_o and cfl_o > 0.05
        assert np.abs(qn_o - q).max() > 1e-3


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("order,trans,lim", [(2, 22, 4), (2, 21, 2), (2, 20, 3), (2, 11, 4), (1, 10, 0), (2, 0, 1)])
def test_step3_unsplit_vs_oracle(shape, order, trans, lim):
    mx, my, mz = shape
    mbc = 2
    pad = (mx + 2 * mbc, my + 2 * mbc, mz + 2 * mbc)
    q, aux = _fields(pad, mx + 10 * my + trans)
    method = [1, order, trans, 0, 0, 0, 3]
    P = _lib.make_problem(3, 1, 1, mbc, mx, my, D[0], D[1], FW, [], method, [lim], maux=3)
    dt = 0.004
    qn_o = q.copy("F")
    cfl_o = o3.step3(FW, [], mbc, mx, my, mz, q, qn_o, *D, dt, method, [lim], aux=aux)
    qn_g, cfl_g = _step_host("clawb200_step3_host", P, mz, q, aux, dt)
    inner = (slice(None),) + (slice(mbc, -mbc),) * 3
    assert np.array_equal(qn_g[inner], qn_o[inner]), np.abs(qn_g[inner] - qn_o[inner]).max()
    assert cfl_g == cfl_o and cfl_o > 0.05
    assert np.abs(qn_o[inner] - q[inner]).max() > 1e-3


def test_rp_solve_vs_oracle():
    import torch
    from pyclaw_b200 import riemann
    n = 4000
    rng = np.random.RandomState(7)
    ql, qr = rng.uniform(-1, 1, (1, n)), rng.uniform(-1, 1, (1, n))
    auxl, auxr = rng.uniform(-2, 2, (3, n)), rng.uniform(-2, 2, (3, n))
    auxr[:, :500] = -auxl[:, :500]          # s == 0
    auxl[:, 500:600] = auxr[:, 500:600] = 0.0
    rs = riemann.vc_advection_fwave_3d
    dev = lambda a: torch.tensor(a, device='cuda')
    for ixyz in (1, 2, 3):
        ref = o3.rp_point_aux(FW, [], ixyz, 1, ql, qr, auxl, auxr)
        out = rs(dev(ql), dev(qr), dev(auxl), dev(auxr), ixy=ixyz)
        for a, b in zip(out, ref):
            assert np.array_equal(a.cpu().numpy(), b), ixyz
        amdq, apdq = out[2].cpu().numpy(), out[3].cpu().numpy()
        assert np.array_equal(amdq + apdq, auxr[ixyz - 1] * qr - auxl[ixyz - 1] * ql)


# ---- SharpClaw ----------------------------------------------------------------------------------
VARIANTS = {"f32": o3.WENO_PYWENO_F32, "f64": o3.WENO_PYWENO_F64, "old": o3.WENO_OLD, "tvd2": o3.RECON_TVD2}


def _device_dq(P, mz, q, aux, dt):
    dq = np.zeros_like(q, order="F")
    cfl = ctypes.c_double()
    _lib.call("clawb200_sharpclaw_dq3_host", ctypes.byref(P), mz, D[2], _ptr(q), _ptr(dq), _ptr(aux), dt,
              ctypes.byref(cfl))
    return dq, cfl.value


@pytest.mark.parametrize("shape", SHAPES + [(260, 40, 40)])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_sharpclaw_dq3_vs_oracle(variant, shape):
    mx, my, mz = shape
    mbc = 3
    pad = tuple(n + 2 * mbc for n in shape)
    q, aux = _fields(pad, sum(shape) + len(variant))
    v = VARIANTS[variant]
    dt = 0.004
    dq_o, cfl_o = o3.sc_flux3(FW, [], 1, mbc, mx, my, mz, q, *D, dt, v, aux=aux, mthlim=[4])
    P = _lib.make_problem(3, 1, 1, mbc, mx, my, D[0], D[1], FW, [], [1, 2, 0, 0, 0, 0, 3], [4], maux=3,
                          weno_variant=v)
    dq_g, cfl_g = _device_dq(P, mz, q, aux, dt)
    assert np.array_equal(dq_g, dq_o), np.abs(dq_g - dq_o).max()
    assert cfl_g == cfl_o and cfl_o > 0.05
    assert np.abs(dq_o).max() > 1e-3


# ---- the user header restates the built-in solver ----------------------------------------------
def _user_fwave3d():
    import pyclaw
    hdr = os.path.join(ROOT, "examples", "user_rp", "rp_fwave3d_user.cuh")
    return pyclaw.riemann.from_header(hdr, meqn=1, mwaves=1, maux=3, ndims=(3,), fwave=True)


def test_user_header_equals_builtin():
    """Split, unsplit (all six method(3) settings) and the SharpClaw dq: the user header is the built-in
    solver bit for bit, so a user's FWAVE = true header gets the sign(s) correction of the f-wave step."""
    rs = _user_fwave3d()
    dt = 0.004
    for mx, my, mz in ((9, 7, 5), (130, 6, 4), (5, 4, 70)):
        pad2 = (mx + 4, my + 4, mz + 4)
        q, aux = _fields(pad2, mx)
        cases = [("clawb200_step3ds_host", [1, 2, -1, 0, 0, 0, 3], idir) for idir in (1, 2, 3)]
        cases += [("clawb200_step3_host", [1, 1 if t in (0, 10) else 2, t, 0, 0, 0, 3], None)
                  for t in (0, 10, 11, 20, 21, 22)]
        for fn, method, idir in cases:
            res = []
            for variant, rp_id in (("strict", FW), (rs._variant(), _lib.RP_USER)):
                _lib.set_variant(variant)
                P = _lib.make_problem(3, 1, 1, 2, mx, my, D[0], D[1], rp_id, [], method, [4], maux=3)
                res.append(_step_host(fn, P, mz, q, aux, dt, idir))
            _lib.set_variant("strict")
            assert np.array_equal(res[0][0], res[1][0]) and res[0][1] == res[1][1], (fn, method, idir)
            assert np.abs(res[0][0] - q).max() > 1e-3
        q3, aux3 = _fields((mx + 6, my + 6, mz + 6), mx + 1)
        for v in VARIANTS.values():
            res = []
            for variant, rp_id in (("strict", FW), (rs._variant(), _lib.RP_USER)):
                _lib.set_variant(variant)
                P = _lib.make_problem(3, 1, 1, 3, mx, my, D[0], D[1], rp_id, [], [1, 2, 0, 0, 0, 0, 3], [4], maux=3,
                                      weno_variant=v)
                res.append(_device_dq(P, mz, q3, aux3, dt))
            _lib.set_variant("strict")
            assert np.array_equal(res[0][0], res[1][0]) and res[0][1] == res[1][1], v


# ---- runs through import pyclaw: conservation and the fma build -------------------------------
def _periodic_field(n, seed):
    """a random periodic, divergent velocity field with sign changes, and random positive q"""
    rng = np.random.RandomState(seed)
    x = (np.arange(n) + 0.5) / n
    X, Y, Z = np.meshgrid(x, x, x, indexing='ij')
    ph = rng.uniform(0, 2 * np.pi, 6)
    aux = np.stack([np.sin(2 * np.pi * X + ph[0]) * np.cos(2 * np.pi * Z + ph[1]),
                    0.8 * np.cos(2 * np.pi * Y + ph[2]) + 0.3 * np.sin(2 * np.pi * X + ph[3]),
                    0.6 * np.sin(2 * np.pi * (X + Y + Z) + ph[4])]) + rng.uniform(-0.2, 0.2, (3, n, n, n))
    q0 = np.asfortranarray(rng.uniform(0.5, 1.5, (1, n, n, n)))
    return q0, np.asfortranarray(aux)


def _run(q0, aux, nsteps, dt, solver_type='classic', dim_split=False, limiters=4, arithmetic='strict', rp=None):
    import pyclaw
    mx, my, mz = q0.shape[1:]
    if solver_type == 'sharpclaw':
        solver = pyclaw.SharpClawSolver3D()
        solver.time_integrator = 'SSP104'
        solver.cfl_desired, solver.cfl_max = 0.8, 0.9
    else:
        solver = pyclaw.ClawSolver3D()
        solver.dim_split = dim_split
        solver.limiters = limiters
    solver.rp = rp or pyclaw.riemann.vc_advection_fwave_3d
    solver.fwave = True
    solver.mwaves = 1
    solver.arithmetic = arithmetic
    solver.dt_variable, solver.dt_initial = False, dt
    for i in range(3):
        solver.bc_lower[i] = solver.bc_upper[i] = pyclaw.BC.periodic
        solver.aux_bc_lower[i] = solver.aux_bc_upper[i] = pyclaw.BC.periodic
    grid = pyclaw.Grid([pyclaw.Dimension('x', 0.0, 1.0, mx), pyclaw.Dimension('y', 0.0, 1.0, my),
                        pyclaw.Dimension('z', 0.0, 1.0, mz)])
    state = pyclaw.State(grid, 1, 3)
    state.aux = aux
    state.q[...] = q0
    claw = pyclaw.Controller()
    claw.keep_copy, claw.output_format = True, None
    claw.solution, claw.solver = pyclaw.Solution(state), solver
    claw.tfinal, claw.nout = nsteps * dt, 1
    claw.run()
    return np.asarray(claw.frames[-1].q)


# The split step sweeps one ghost layer of slices only (step3ds.f), so with a limiter the two periodic
# boundaries see different neighbours (tests/test_gpu_3d_solvers.py): it is checked without limiters.
@pytest.mark.parametrize("kind", ["unsplit", "split", "sharpclaw"])
def test_periodic_conservation_and_fma_build(kind):
    n = 20
    q0, aux = _periodic_field(n, 3)
    kw = dict(unsplit=dict(), split=dict(dim_split=True, limiters=0), sharpclaw=dict(solver_type='sharpclaw'))[kind]
    qs = _run(q0, aux, 40, 0.4 / n, **kw)
    assert abs(qs.sum() - q0.sum()) <= 1e-13 * np.abs(q0).sum(), abs(qs.sum() - q0.sum()) / np.abs(q0).sum()
    assert np.abs(qs - q0).max() > 1e-2
    qf = _run(q0, aux, 40, 0.4 / n, arithmetic='fma', **kw)
    dev = np.abs(qf - qs).max() / np.abs(qs).max()
    print("%s: fma vs strict relative L-inf %.3g" % (kind, dev))
    assert dev <= 1e-12


def test_user_header_runs_equal_builtin_through_pyclaw():
    n = 12
    q0, aux = _periodic_field(n, 4)
    rs = _user_fwave3d()
    for kw in (dict(), dict(dim_split=True), dict(solver_type='sharpclaw')):
        a = _run(q0, aux, 6, 0.4 / n, **kw)
        b = _run(q0, aux, 6, 0.4 / n, rp=rs, **kw)
        assert np.array_equal(a, b), kw


# ---- the application ---------------------------------------------------------------------------
def _apps():
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    import apps
    return apps


# Measured on a B200 (L1 error at t = T, 32^3 -> 64^3): classic split 2.57, classic unsplit 4.73, SharpClaw
# 2.20.  The classic f-wave correction 0.5 sign(s) (1 - |s| dt/dx) fwave makes the interface flux the
# average of the two cell fluxes (second order).  SharpClaw's flux at an interface is the upwind cell's
# velocity times the reconstructed edge value, u_i q(x_i+1/2): with cell-centred velocities that is off by
# u' dx / 2 * q, a first-order truncation error however accurate WENO5 is, so its ratio tends to 2.
@pytest.mark.parametrize("solver_type,dim_split,ratio", [("classic", True, 2.5), ("classic", False, 2.5),
                                                         ("sharpclaw", True, 2.0)])
def test_transport3d_returns_to_its_initial_data(solver_type, dim_split, ratio):
    """The flow reverses at t = T / 2: at t = T the error against the initial data falls from 32^3 to 64^3
    (by 2.5x for the classic steps, 2x for SharpClaw), and the periodic box conserves q."""
    apps = _apps()
    err = []
    for n in (32, 64):
        c = apps.transport3d(mx=n, my=n, mz=n, dim_split=dim_split, solver_type=solver_type)
        q0, q = np.asarray(c.frames[0].q), np.asarray(c.frames[-1].q)
        assert c.frames[-1].t == pytest.approx(1.0) and np.isfinite(q).all()
        tol = 1e-9 if (dim_split and solver_type == 'classic') else 1e-12
        assert abs(q.sum() - q0.sum()) <= tol * np.abs(q0).sum()
        mid = np.asarray(c.frames[5].q)
        assert np.abs(mid - q0).max() > 0.2            # the bell is well deformed at t = T / 2
        err.append(np.abs(q - q0).sum() / n ** 3)
    print("transport3d %s dim_split=%s: L1 error 32^3 %.4g, 64^3 %.4g, ratio %.3f"
          % (solver_type, dim_split, err[0], err[1], err[0] / err[1]))
    assert err[0] / err[1] >= ratio


def test_transport3d_sharpclaw_unsplit_flag_runs():
    """SharpClaw has no split / unsplit choice; dim_split=False gives the same run."""
    apps = _apps()
    a = np.asarray(apps.transport3d(mx=16, my=16, mz=16, tfinal=0.2, solver_type='sharpclaw').frames[-1].q)
    b = np.asarray(apps.transport3d(mx=16, my=16, mz=16, tfinal=0.2, solver_type='sharpclaw',
                                    dim_split=False).frames[-1].q)
    assert np.array_equal(a, b) and np.isfinite(a).all()


# ---- argument checks --------------------------------------------------------------------------
def test_argument_checks():
    lib = _lib.load()
    q = np.zeros((1, 12, 12, 12), order="F")
    qn = np.zeros_like(q)
    aux = np.zeros((4, 12, 12, 12), order="F")
    cfl = ctypes.c_double()

    def rcs(maux, with_aux, mcapa=0):
        method = [1, 2, 22, 0, 0, mcapa, maux]
        a = _ptr(aux) if with_aux else None
        P = _lib.make_problem(3, 1, 1, 2, 8, 8, 0.1, 0.1, FW, [], method, [4], maux=maux)
        r1 = lib.clawb200_step3_host(ctypes.byref(P), 8, 0.1, _ptr(q), _ptr(qn), a, 0.01, ctypes.byref(cfl))
        method[2] = -1
        P = _lib.make_problem(3, 1, 1, 2, 8, 8, 0.1, 0.1, FW, [], method, [4], maux=maux)
        r2 = lib.clawb200_step3ds_host(ctypes.byref(P), 8, 0.1, _ptr(q), _ptr(qn), a, 0.01, 1, ctypes.byref(cfl))
        method[2] = 0
        P = _lib.make_problem(3, 1, 1, 3, 6, 6, 0.1, 0.1, FW, [], method, [4], maux=maux)
        r3 = lib.clawb200_sharpclaw_dq3_host(ctypes.byref(P), 6, 0.1, _ptr(q), _ptr(qn), a, 0.01, ctypes.byref(cfl))
        return r1, r2, r3
    assert rcs(3, False) == (ERR_INVALID,) * 3
    assert b"{u, v, w}" in lib.clawb200_last_error()
    assert rcs(2, True) == (ERR_INVALID,) * 3
    assert rcs(4, True, mcapa=4) == (ERR_UNSUPPORTED,) * 3
    assert rcs(3, True) == (0, 0, 0)
    P = _lib.make_problem(3, 1, 2, 2, 8, 8, 0.1, 0.1, FW, [], [1, 2, 22, 0, 0, 0, 3], [4, 4], maux=3)
    with pytest.raises(_lib.ClawB200Error, match="meqn/mwaves"):
        _lib.call("clawb200_step3_host", ctypes.byref(P), 8, 0.1, _ptr(q), _ptr(qn), _ptr(aux), 0.01, ctypes.byref(cfl))
