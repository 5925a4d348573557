"""Shallow water over bathymetry (``pyclaw.riemann.shallow_bathymetry_fwave``, RpShallowBathyFwave in
csrc/rp.cuh) on the GPU.

1. Parity: the strict build against the CPU oracle (oracle_bathy/claw_oracle_bathy.c), bit for bit:
   the pointwise solve, step1, step2ds in both directions, step2 for method(3) = 0, 1, 2, and whole runs
   through ``import pyclaw`` against ``OracleSolver`` with a variable time step and a rejected step.
2. Physics: a lake at rest stays at rest (both builds, split and unsplit), LeVeque's perturbed steady
   state over a bump leaves the water ahead of the waves untouched, the closed basin conserves mass, a
   flat-bottom dam break is as accurate as the Roe solver, and y-invariant 2-D data is the 1-D run.
3. The fma build: one call of each kernel family within 1e-13 of the oracle.
4. Two ranks equal one (tests/mp_bathymetry_check.py)."""
import contextlib
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import problems
import oracle_bathy as ob
from oracle import pyclaw_oracle as po
from pyclaw_b200 import _lib

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "examples"))

G, DRY = 9.81, 1e-3
RP = _lib.RP_SHALLOW_BATHY_FWAVE
PARAMS = [G, DRY]


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


@contextlib.contextmanager
def _variant(name):
    prev = _lib.set_variant(name)
    try:
        yield
    finally:
        _lib.set_variant(prev)


def _data(shape, seed, dry=False):
    """Moving water over a rough bottom (padded arrays); with dry=True a few cells hold less than
    dry_tolerance, some of them exactly nothing."""
    rng = np.random.RandomState(seed)
    ndim = len(shape)
    q = np.empty((ndim + 1,) + tuple(shape), order="F")
    h = rng.uniform(0.3, 2.0, shape)
    if dry:
        d = rng.uniform(0, 1, shape) < 0.05
        h[d] = rng.uniform(0.0, DRY, d.sum())
        h[rng.uniform(0, 1, shape) < 0.01] = 0.0
    q[0] = h
    for m in range(1, ndim + 1):
        q[m] = h * rng.uniform(-1.5, 1.5, shape)
    aux = np.asfortranarray(rng.uniform(-0.5, 0.5, (1,) + tuple(shape)))
    return q, aux


# =============================================================================================
# 1. parity with the oracle
# =============================================================================================
def _rp_solve(ndim, ixy, ql, qr, al, ar):
    meqn, n = ql.shape
    mw = ndim + 1
    P = _lib.make_problem(ndim, meqn, mw, 2, 8, 8, 1.0, 1.0, RP, PARAMS, maux=1)
    wave, s = np.zeros((meqn, mw, n)), np.zeros((mw, n))
    amdq, apdq = np.zeros((meqn, n)), np.zeros((meqn, n))
    c = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    ql, qr, al, ar = c(ql), c(qr), c(al), c(ar)
    _lib.call("clawb200_rp_solve_host", ctypes.byref(P), ixy, n, _ptr(ql), _ptr(qr), _ptr(al), _ptr(ar),
              _ptr(wave), _ptr(s), _ptr(amdq), _ptr(apdq))
    return wave, s, amdq, apdq


def _point_states(ndim, n, seed):
    q, aux = _data((2 * n,), seed, dry=True)
    rng = np.random.RandomState(seed)
    ql, qr = q[:, :n].copy(), q[:, n:].copy()
    if ndim == 2:
        ql = np.vstack([ql, ql[1:] * rng.uniform(-1, 1, n)])
        qr = np.vstack([qr, qr[1:] * rng.uniform(-1, 1, n)])
    k = n // 8
    ql[0, :k] = qr[0, :k] = 0.0                                 # dry on both sides
    ql[1:, k:2 * k] = qr[1:, k:2 * k] = 0.0                     # water at rest
    qr[0, k:2 * k] = ql[0, k:2 * k] + aux[0, :k] - aux[0, n:n + k]   # ... and a lake at rest
    return ql, qr, aux[:, :n].copy(), aux[:, n:].copy()


@pytest.mark.parametrize("ndim,ixy", [(1, 1), (2, 1), (2, 2)])
def test_pointwise_solve_vs_oracle(ndim, ixy):
    n = 5000
    ql, qr, al, ar = _point_states(ndim, n, 3 + ixy)
    got = _rp_solve(ndim, ixy, ql, qr, al, ar)
    want = ob.rp_point(PARAMS, 0 if ndim == 1 else ixy, ndim + 1, ql, qr, al, ar)
    for g, w in zip(got, want):
        assert np.array_equal(g, w), np.abs(g - w).max()
    assert np.isfinite(got[2]).all() and np.abs(got[2]).max() > 0.1


def test_pointwise_transverse_needs_an_aux_free_solver():
    n = 16
    P = _lib.make_problem(2, 3, 3, 2, 8, 8, 1.0, 1.0, RP, PARAMS, maux=1)
    q = np.ones((3, n))
    with pytest.raises(_lib.ClawB200Error):
        _lib.call("clawb200_rp_transverse_host", ctypes.byref(P), 1, n, _ptr(q), _ptr(q), 1, _ptr(q),
                  _ptr(q.copy()), _ptr(q.copy()))


@pytest.mark.parametrize("mx", [7, 130, 1001])
@pytest.mark.parametrize("order,lim", [(1, [0, 0]), (2, [4, 4]), (2, [1, 3])])
@pytest.mark.parametrize("dry", [False, True])
def test_step1_vs_oracle(mx, order, lim, dry):
    mbc = 2
    dx, dt = 0.01, 0.0012
    method = [1, order, 0, 0, 0, 0, 1]
    q, aux = _data((mx + 2 * mbc,), seed=mx + order + dry, dry=dry)
    P = _lib.make_problem(1, 2, 2, mbc, mx, 1, dx, 1.0, RP, PARAMS, method, lim, maux=1)
    q_o = q.copy("F")
    cfl_o = ob.step1(PARAMS, mbc, mx, q_o, aux, dx, dt, method, lim)
    q_g = q.copy("F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_step1_host", ctypes.byref(P), _ptr(q_g), _ptr(aux), dt, ctypes.byref(cfl_g))
    assert 0.1 < cfl_o < 2.0 and np.isfinite(q_o).all()
    assert np.array_equal(q_g[:, mbc:-mbc], q_o[:, mbc:-mbc]), np.abs(q_g - q_o)[:, mbc:-mbc].max()
    assert cfl_g.value == cfl_o


SHAPES = [(37, 29), (130, 70), (9, 140)]
LIMS = [[4, 4, 4], [1, 2, 3], [0, 0, 0]]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("order,lim", [(1, LIMS[2]), (2, LIMS[0]), (2, LIMS[1])])
def test_step2ds_vs_oracle(shape, order, lim):
    mx, my = shape
    mbc = 2
    dx, dy, dt = 0.02, 0.025, 0.002
    method = [1, order, -1, 0, 0, 0, 1]
    q, aux = _data((mx + 2 * mbc, my + 2 * mbc), seed=mx + order, dry=(order == 2))
    P = _lib.make_problem(2, 3, 3, mbc, mx, my, dx, dy, RP, PARAMS, method, lim, maux=1)
    cfl_g = ctypes.c_double()
    for ids in (1, 2):
        qn_o = q.copy("F")
        cfl_o = ob.step2ds(PARAMS, mbc, mx, my, q, qn_o, aux, dx, dy, dt, method, lim, ids)
        qn_g = q.copy("F")
        _lib.call("clawb200_step2ds_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), _ptr(aux), dt, ids,
                  ctypes.byref(cfl_g))
        assert 0.1 < cfl_o < 2.0 and np.isfinite(qn_o).all()
        assert np.array_equal(qn_g, qn_o), (ids, np.abs(qn_g - qn_o).max())
        assert cfl_g.value == cfl_o


@pytest.mark.parametrize("shape", SHAPES + [(251, 9)])
@pytest.mark.parametrize("trans", [0, 1, 2])
@pytest.mark.parametrize("lim", [0, 1])
def test_step2_vs_oracle(shape, trans, lim):
    mx, my = shape
    mbc = 2
    dx, dy, dt = 0.02, 0.025, 0.002
    method = [1, 2, trans, 0, 0, 0, 1]
    q, aux = _data((mx + 2 * mbc, my + 2 * mbc), seed=mx + 10 * trans + lim, dry=(lim == 1))
    P = _lib.make_problem(2, 3, 3, mbc, mx, my, dx, dy, RP, PARAMS, method, LIMS[lim], maux=1)
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    qn_o = q.copy("F")
    cfl_o = ob.step2(PARAMS, mbc, mx, my, q, qn_o, aux, dx, dy, dt, method, LIMS[lim])
    qn_g = q.copy("F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), _ptr(aux), dt, ctypes.byref(cfl_g))
    assert 0.1 < cfl_o < 2.0 and np.isfinite(qn_o[inner]).all()
    assert np.array_equal(qn_g[inner], qn_o[inner]), np.abs(qn_g[inner] - qn_o[inner]).max()
    assert cfl_g.value == cfl_o


def test_argument_checks():
    mbc, mx, my = 2, 20, 12
    cfl = ctypes.c_double()
    q, aux = _data((mx + 4, my + 4), seed=1)
    q1, aux1 = _data((mx + 4,), seed=1)
    step2 = lambda P, a: _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(q.copy("F")),
                                   None if a is None else _ptr(a), 0.001, ctypes.byref(cfl))
    P = _lib.make_problem(2, 3, 3, mbc, mx, my, 0.1, 0.1, RP, PARAMS, [1, 2, 2, 0, 0, 0, 1], [4] * 3, maux=1)
    with pytest.raises(_lib.ClawB200Error, match="aux"):
        step2(P, None)
    with pytest.raises(_lib.ClawB200Error, match="aux"):
        step2(_lib.make_problem(2, 3, 3, mbc, mx, my, 0.1, 0.1, RP, PARAMS, [1, 2, 2, 0, 0, 0, 0], [4] * 3), aux)
    with pytest.raises(_lib.ClawB200Error, match="capacity"):
        step2(_lib.make_problem(2, 3, 3, mbc, mx, my, 0.1, 0.1, RP, PARAMS, [1, 2, 2, 0, 0, 1, 1], [4] * 3, maux=1),
              aux)
    with pytest.raises(_lib.ClawB200Error, match="dry_tolerance"):
        step2(_lib.make_problem(2, 3, 3, mbc, mx, my, 0.1, 0.1, RP, [G, -1.0], [1, 2, 2, 0, 0, 0, 1], [4] * 3, maux=1),
              aux)
    with pytest.raises(_lib.ClawB200Error, match="meqn"):
        step2(_lib.make_problem(2, 3, 2, mbc, mx, my, 0.1, 0.1, RP, PARAMS, [1, 2, 2, 0, 0, 0, 1], [4] * 2, maux=1),
              aux)
    P1 = _lib.make_problem(1, 2, 2, mbc, mx, 1, 0.1, 1.0, RP, PARAMS, [1, 2, 0, 0, 0, 0, 1], [4, 4], maux=1)
    with pytest.raises(_lib.ClawB200Error, match="aux"):
        _lib.call("clawb200_step1_host", ctypes.byref(P1), _ptr(q1), None, 0.001, ctypes.byref(cfl))
    # SharpClaw: the stage kernel is not compiled for this solver
    P1.mbc = 3
    with pytest.raises(_lib.ClawB200Error):
        q3 = np.zeros((2, mx + 6), order="F")
        _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P1), _ptr(q3), _ptr(q3.copy("F")),
                  _ptr(np.zeros((1, mx + 6), order="F")), 0.001, ctypes.byref(cfl))


def test_sharpclaw_refuses_the_solver():
    import pyclaw
    solver = pyclaw.SharpClawSolver1D()
    solver.rp = pyclaw.riemann.shallow_bathymetry_fwave
    solver.fwave, solver.mwaves = True, 2
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.outflow
    solver.aux_bc_lower[0] = solver.aux_bc_upper[0] = pyclaw.BC.outflow
    state = pyclaw.State(pyclaw.Grid(pyclaw.Dimension('x', 0., 1., 50)), 2, 1)
    state.aux_global['grav'] = G
    state.q[0, :] = 1.0
    with pytest.raises(NotImplementedError, match="balanced"):
        solver.setup(pyclaw.Solution(state))


def _pyclaw_run(pyclaw, ndim, q0, aux, d, lower, tfinal, nout, bc, dim_split=True, order_trans=2,
                dt_initial=None, dt_variable=True, arithmetic='strict', rp=None, limiters=4):
    solver = pyclaw.ClawSolver1D() if ndim == 1 else pyclaw.ClawSolver2D()
    solver.rp = rp or pyclaw.riemann.shallow_bathymetry_fwave
    solver.fwave = solver.rp.fwave
    solver.mwaves, solver.limiters = ndim + 1, limiters
    solver.cfl_max, solver.cfl_desired = 1.0, 0.9
    solver.arithmetic = arithmetic
    if ndim == 2:
        solver.dim_split, solver.order_trans = dim_split, order_trans
    for i in range(ndim):
        solver.bc_lower[i] = solver.bc_upper[i] = bc[i]
        solver.aux_bc_lower[i] = solver.aux_bc_upper[i] = bc[i]
    n = q0.shape[1:]
    dims = [pyclaw.Dimension('xy'[i], lower[i], lower[i] + d[i] * n[i], n[i]) for i in range(ndim)]
    state = pyclaw.State(pyclaw.Grid(dims), ndim + 1, 0 if aux is None else 1)
    state.aux_global['grav'] = G
    if aux is not None:
        state.aux = aux
    state.q[...] = q0
    solver.dt_initial = dt_initial if dt_initial is not None else 0.1 * min(d)
    solver.dt_variable = dt_variable
    claw = pyclaw.Controller()
    claw.keep_copy, claw.output_format, claw.tfinal, claw.nout = True, None, tfinal, nout
    claw.solution, claw.solver = pyclaw.Solution(state), solver
    claw.run()
    return claw


def _oracle_run(ndim, q0, aux, d, tfinal, nout, bc, dim_split=True, order_trans=2, dt_initial=None, dt_variable=True):
    s = ob.OracleSolver(ndim, PARAMS)
    s.limiters = 4
    s.cfl_max, s.cfl_desired = 1.0, 0.9
    s.bc_lower = s.bc_upper = list(bc)
    s.aux_bc_lower = s.aux_bc_upper = list(bc)
    s.dim_split, s.order_trans = dim_split, order_trans
    s.dt_initial = dt_initial if dt_initial is not None else 0.1 * min(d)
    s.dt_variable = dt_variable
    frames = s.run(q0, aux, list(d), tfinal, nout)
    return frames, s


def _bump_profile(x):
    return np.where(np.abs(x - 0.5) < 0.1, 0.25 * (np.cos(10 * np.pi * (x - 0.5)) + 1.0), 0.0)


def test_run_1d_vs_oracle_with_a_rejected_step():
    import pyclaw
    mx = 160
    x = (np.arange(mx) + 0.5) / mx
    b = _bump_profile(x)
    q0 = np.zeros((2, mx), order="F")
    q0[0] = 1.0 + 0.2 * np.exp(-200 * (x - 0.25) ** 2) - b
    q0[1] = 0.3 * q0[0]
    aux = np.asfortranarray(b[None])
    # dt_initial = 2 dx / sqrt(g): the first step runs at Courant number ~2 and is rejected
    dt0 = 2.0 / mx / np.sqrt(G)
    frames, s = _oracle_run(1, q0, aux, [1.0 / mx], 0.3, 3, [po.BC_OUTFLOW], dt_initial=dt0)
    assert s.total['rejected'] >= 1
    claw = _pyclaw_run(pyclaw, 1, q0, aux, [1.0 / mx], [0.0], 0.3, 3, [pyclaw.BC.outflow], dt_initial=dt0)
    for fg, fo in zip(claw.frames, frames):
        assert np.array_equal(np.asarray(fg.q), fo)
    assert np.abs(frames[-1] - q0).max() > 0.05


@pytest.mark.parametrize("dim_split,order_trans", [(True, 1), (False, 0), (False, 1), (False, 2)])
def test_run_2d_vs_oracle(dim_split, order_trans):
    import pyclaw
    mx, my = 40, 36
    d = [2.0 / mx, 2.0 / my]
    Y, X = np.meshgrid(-1 + (np.arange(my) + 0.5) * d[1], -1 + (np.arange(mx) + 0.5) * d[0])
    b = -1.0 + 0.8 * np.exp(-((X - 0.25) ** 2 + Y ** 2) / 0.2 ** 2)
    q0 = np.zeros((3, mx, my), order="F")
    q0[0] = 0.1 * np.exp(-((X + 0.5) ** 2 + Y ** 2) / 0.1 ** 2) - b
    q0[1] = 0.2 * q0[0]
    q0[2] = -0.1 * q0[0]
    aux = np.asfortranarray(b[None])
    dt0 = 2.0 * d[0] / np.sqrt(G)                     # rejected first step, as above
    bc = [po.BC_REFLECTING, po.BC_OUTFLOW]
    frames, s = _oracle_run(2, q0, aux, d, 0.15, 2, bc, dim_split, order_trans, dt_initial=dt0)
    assert s.total['rejected'] >= 1
    claw = _pyclaw_run(pyclaw, 2, q0, aux, d, [-1.0, -1.0], 0.15, 2, [pyclaw.BC.reflecting, pyclaw.BC.outflow],
                       dim_split, order_trans, dt_initial=dt0)
    for fg, fo in zip(claw.frames, frames):
        assert np.array_equal(np.asarray(fg.q), fo), np.abs(np.asarray(fg.q) - fo).max()
    assert np.abs(frames[-1] - q0).max() > 0.01


# =============================================================================================
# 2. physics
# =============================================================================================
@pytest.mark.parametrize("arithmetic", ["strict", "fma"])
@pytest.mark.parametrize("ndim,dim_split,order_trans", [(1, True, 0), (2, True, 1), (2, False, 0), (2, False, 1),
                                                        (2, False, 2)])
def test_lake_at_rest_stays_at_rest(arithmetic, ndim, dim_split, order_trans):
    import pyclaw
    shape = (64,) if ndim == 1 else (48, 40)
    b = -1.0 + 0.6 * problems.smooth_state("advection", shape, seed=3)[0]
    eta0 = 0.25
    q0 = np.zeros((ndim + 1,) + shape, order="F")
    q0[0] = eta0 - b
    d = [2.0 / n for n in shape]
    dt = 0.4 * min(d) / np.sqrt(G * 1.25)
    claw = _pyclaw_run(pyclaw, ndim, q0, np.asfortranarray(b[None]), d, [-1.0] * ndim, 200 * dt, 1,
                       [pyclaw.BC.reflecting] * ndim, dim_split, order_trans, dt_initial=dt, dt_variable=False,
                       arithmetic=arithmetic)
    assert claw.solver.status['numsteps'] == 200
    q = np.asarray(claw.frames[-1].q)
    assert np.abs(q[0] + b - eta0).max() <= 1e-12
    assert np.abs(q[1:]).max() <= 1e-12


def test_bump1d_leaves_the_water_ahead_of_the_waves_at_rest():
    import apps
    claw = apps.bump1d(mx=200, tfinal=0.1)
    x = np.asarray(claw.solution.state.grid.x.center)
    q = np.asarray(claw.frames[-1].q)
    b = np.asarray(claw.solution.state.aux)[0]
    eta = q[0] + b
    # the fastest wave, sqrt(g (1 + eps)) ~ 3.13, leaves 0.2 at t = 0 and is short of x = 0.52 at t = 0.1
    ahead = x > 0.6
    assert np.abs(eta[ahead] - 1.0).max() <= 1e-13 and np.abs(q[1, ahead]).max() <= 1e-13
    assert np.abs(eta - 1.0).max() > 1e-4                 # the pulse is there
    assert abs(claw.frames[-1].t - 0.1) < 1e-14


@pytest.mark.parametrize("dim_split", [True, False])
def test_seamount2d_conserves_mass(dim_split):
    import apps
    claw = apps.seamount2d(mx=80, my=80, tfinal=0.4, dim_split=dim_split)
    q0, q1 = np.asarray(claw.frames[0].q), np.asarray(claw.frames[-1].q)
    assert np.isfinite(q1).all() and np.abs(q1[1]).max() > 1e-3
    assert abs(q1[0].sum() - q0[0].sum()) <= 1e-12 * q0[0].sum()
    assert q1[0].min() > 0.1


def _dam_break_exact(hl, hr, x, t):
    from scipy.optimize import brentq
    f = lambda hm: 2 * (np.sqrt(G * hl) - np.sqrt(G * hm)) - (hm - hr) * np.sqrt(0.5 * G * (1 / hm + 1 / hr))
    hm = brentq(f, hr, hl, xtol=1e-15)
    um = 2 * (np.sqrt(G * hl) - np.sqrt(G * hm))
    sh = hm * um / (hm - hr)
    cl, cm = np.sqrt(G * hl), np.sqrt(G * hm)
    xi = x / t
    return np.where(xi < -cl, hl, np.where(xi < um - cm, ((2 * cl - xi) / 3) ** 2 / G, np.where(xi < sh, hm, hr)))


def test_flat_bottom_dam_break_is_as_accurate_as_roe():
    import pyclaw
    mx = 400
    dx = 10.0 / mx
    x = -5 + (np.arange(mx) + 0.5) * dx
    q0 = np.zeros((2, mx), order="F")
    q0[0] = np.where(x <= 0, 3.0, 1.0)
    exact = _dam_break_exact(3.0, 1.0, x, 0.5)
    err = {}
    for name, rp, aux in (("roe", pyclaw.riemann.shallow_roe_with_efix, None),
                          ("bathy", pyclaw.riemann.shallow_bathymetry_fwave, np.zeros((1, mx), order="F"))):
        claw = _pyclaw_run(pyclaw, 1, q0, aux, [dx], [-5.0], 0.5, 1, [pyclaw.BC.outflow], rp=rp, dt_initial=0.01)
        err[name] = np.abs(np.asarray(claw.frames[-1].q)[0] - exact).sum() * dx
    print("dam break L1(h): %s" % err)
    assert err["bathy"] <= 1.5 * err["roe"] and err["bathy"] < 0.05


@pytest.mark.parametrize("dim_split", [True, False])
def test_y_invariant_2d_data_is_the_1d_run(dim_split):
    import pyclaw
    mx, my = 200, 6
    dx = 1.0 / mx
    x = (np.arange(mx) + 0.5) * dx
    b = _bump_profile(x)
    h = 1.0 + 0.1 * np.exp(-300 * (x - 0.3) ** 2) - b
    hu = 0.2 * h
    dt = 0.5 * dx / 4.0
    q1 = np.asfortranarray(np.stack([h, hu]))
    c1 = _pyclaw_run(pyclaw, 1, q1, np.asfortranarray(b[None]), [dx], [0.0], 60 * dt, 1, [pyclaw.BC.outflow],
                     dt_initial=dt, dt_variable=False)
    q2 = np.zeros((3, mx, my), order="F")
    q2[0], q2[1] = h[:, None], hu[:, None]
    aux2 = np.asfortranarray(np.broadcast_to(b[None, :, None], (1, mx, my)))
    c2 = _pyclaw_run(pyclaw, 2, q2, aux2, [dx, dx], [0.0, 0.0], 60 * dt, 1, [pyclaw.BC.outflow, pyclaw.BC.periodic],
                     dim_split, 2, dt_initial=dt, dt_variable=False)
    r1, r2 = np.asarray(c1.frames[-1].q), np.asarray(c2.frames[-1].q)
    assert np.abs(r1 - q1).max() > 1e-3
    assert np.abs(r2[2]).max() <= 1e-12
    for j in range(my):
        assert np.abs(r2[:2, :, j] - r1).max() <= 1e-12


# =============================================================================================
# 3. the fma build: one call of each kernel family against the oracle
# =============================================================================================
def _fma_close(got, ref, tol=1e-13):
    for m in range(ref.shape[0]):
        sc = max(np.abs(ref[m]).max(), 1e-300)
        assert np.abs(got[m] - ref[m]).max() <= tol * sc, (m, np.abs(got[m] - ref[m]).max() / sc)


def test_fma_build_each_kernel_family():
    with _variant("fma"):
        for ndim, ixy in ((1, 1), (2, 1), (2, 2)):
            ql, qr, al, ar = _point_states(ndim, 2000, 90 + ixy)
            got = _rp_solve(ndim, ixy, ql, qr, al, ar)
            want = ob.rp_point(PARAMS, 0 if ndim == 1 else ixy, ndim + 1, ql, qr, al, ar)
            for g, w in zip(got, want):
                _fma_close(g.reshape(g.shape[0], -1), w.reshape(w.shape[0], -1))
        mbc, mx, my = 2, 130, 70
        dx, dy, dt = 0.02, 0.025, 0.002
        cfl = ctypes.c_double()
        q, aux = _data((mx + 2 * mbc,), seed=7)
        method = [1, 2, 0, 0, 0, 0, 1]
        P = _lib.make_problem(1, 2, 2, mbc, mx, 1, dx, 1.0, RP, PARAMS, method, [4, 4], maux=1)
        q_o, q_g = q.copy("F"), q.copy("F")
        ob.step1(PARAMS, mbc, mx, q_o, aux, dx, dt, method, [4, 4])
        _lib.call("clawb200_step1_host", ctypes.byref(P), _ptr(q_g), _ptr(aux), dt, ctypes.byref(cfl))
        _fma_close(q_g[:, mbc:-mbc], q_o[:, mbc:-mbc])
        q, aux = _data((mx + 2 * mbc, my + 2 * mbc), seed=8)
        inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
        for trans in (-1, 0, 1, 2):
            method = [1, 2, trans, 0, 0, 0, 1]
            P = _lib.make_problem(2, 3, 3, mbc, mx, my, dx, dy, RP, PARAMS, method, [4, 4, 4], maux=1)
            for ids in ((1, 2) if trans < 0 else (0,)):
                qn_o, qn_g = q.copy("F"), q.copy("F")
                if trans < 0:
                    ob.step2ds(PARAMS, mbc, mx, my, q, qn_o, aux, dx, dy, dt, method, [4, 4, 4], ids)
                    _lib.call("clawb200_step2ds_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), _ptr(aux), dt, ids,
                              ctypes.byref(cfl))
                else:
                    ob.step2(PARAMS, mbc, mx, my, q, qn_o, aux, dx, dy, dt, method, [4, 4, 4])
                    _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), _ptr(aux), dt,
                              ctypes.byref(cfl))
                _fma_close(qn_g[inner], qn_o[inner])


# =============================================================================================
# 4. two ranks
# =============================================================================================
def test_seamount2d_two_ranks_equal_one():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29519", os.path.join(HERE, "mp_bathymetry_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    sys.stdout.write(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
