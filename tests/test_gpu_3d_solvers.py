"""The 3-D classic steps for solvers other than vc-acoustics: 3-D advection and 3-D Euler through the
generic kernels (step3.cuh) against the oracle bit for bit, a user 3-D solver (RpUser3) that restates
vc-acoustics against the built-in one, exact transport, the 1-D anchor of the Euler solver,
conservation, the fma build and the euler3d / advection3d applications."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle3d as o3
from oracle import pyclaw_oracle as po
from pyclaw_b200 import _lib

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
G, G1 = 1.4, 0.4
SOLVERS = {"advection": (o3.RP_ADVECTION3D, [0.7, -0.45, 0.3], 1, 1),
           "euler": (o3.RP_EULER3D, [G, G1], 5, 3)}
SHAPES = [(9, 7, 5), (130, 6, 4), (20, 33, 17), (5, 4, 70)]


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _state(name, pad, seed):
    """Random states with jumps in every component; positive density and pressure for Euler."""
    rng = np.random.RandomState(seed)
    if name == "advection":
        return np.asfortranarray(rng.uniform(-1, 1, (1,) + pad))
    rho = rng.uniform(0.5, 2.0, pad)
    u = rng.uniform(-1.0, 1.0, (3,) + pad)
    p = rng.uniform(0.5, 2.0, pad)
    return np.asfortranarray(np.concatenate([rho[None], rho * u, (p / G1 + 0.5 * rho * (u * u).sum(0))[None]]))


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("lim", [[4, 4, 4], [0, 0, 0], [2, 3, 1]])
@pytest.mark.parametrize("name", ["advection", "euler"])
def test_step3ds_vs_oracle(name, shape, lim):
    rp_id, params, meqn, mw = SOLVERS[name]
    mx, my, mz = shape
    mbc = 2
    dx, dy, dz, dt = 0.02, 0.025, 0.03, 0.002
    pad = (mx + 2 * mbc, my + 2 * mbc, mz + 2 * mbc)
    q = _state(name, pad, mx + 10 * my + lim[0])
    lim = lim[:mw]
    order = 1 if lim[0] == 0 else 2
    method = [1, order, -1, 0, 0, 0, 0]
    P = _lib.make_problem(3, meqn, mw, mbc, mx, my, dx, dy, rp_id, params, method, lim)
    cfl_g = ctypes.c_double()
    for idir in (1, 2, 3):
        qn_o = q.copy("F")
        cfl_o = o3.step3ds(rp_id, params, mbc, mx, my, mz, q, qn_o, dx, dy, dz, dt, method, lim, idir)
        qn_g = np.zeros_like(q, order="F")
        _lib.call("clawb200_step3ds_host", ctypes.byref(P), mz, dz, _ptr(q), _ptr(qn_g), None, dt, idir,
                  ctypes.byref(cfl_g))
        assert np.array_equal(qn_g, qn_o), (idir, np.abs(qn_g - qn_o).max())
        assert cfl_g.value == cfl_o and cfl_o > 0.01
        assert np.abs(qn_o - q).max() > 1e-3


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("order,trans,lim", [(2, 22, [4, 4, 4]), (2, 21, [4, 2, 3]), (2, 20, [2, 3, 1]),
                                             (2, 11, [4, 4, 4]), (1, 11, [0, 0, 0]), (1, 10, [0, 0, 0]),
                                             (2, 10, [1, 0, 4]), (2, 0, [4, 4, 4])])
@pytest.mark.parametrize("name", ["advection", "euler"])
def test_step3_unsplit_vs_oracle(name, shape, order, trans, lim):
    rp_id, params, meqn, mw = SOLVERS[name]
    mx, my, mz = shape
    mbc = 2
    dx, dy, dz, dt = 0.02, 0.025, 0.03, 0.002
    pad = (mx + 2 * mbc, my + 2 * mbc, mz + 2 * mbc)
    q = _state(name, pad, mx + 10 * my + order + trans)
    lim = lim[:mw]
    method = [1, order, trans, 0, 0, 0, 0]
    P = _lib.make_problem(3, meqn, mw, mbc, mx, my, dx, dy, rp_id, params, method, lim)
    assert _lib.load().clawb200_step3_scratch_doubles(ctypes.byref(P)) == 14 * meqn * P.mstride
    qn_o = q.copy("F")
    cfl_o = o3.step3(rp_id, params, mbc, mx, my, mz, q, qn_o, dx, dy, dz, dt, method, lim)
    qn_g = np.zeros_like(q, order="F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_step3_host", ctypes.byref(P), mz, dz, _ptr(q), _ptr(qn_g), None, dt, ctypes.byref(cfl_g))
    inner = (slice(None),) + (slice(mbc, -mbc),) * 3
    assert np.array_equal(qn_g[inner], qn_o[inner]), np.abs(qn_g[inner] - qn_o[inner]).max()
    assert cfl_g.value == cfl_o and cfl_o > 0.01
    assert np.abs(qn_o[inner] - q[inner]).max() > 1e-3


@pytest.mark.parametrize("name", ["advection", "euler"])
def test_rp_solve_3d_vs_oracle(name):
    import torch
    from pyclaw_b200 import riemann
    rp_id, params, meqn, mw = SOLVERS[name]
    n = 3000
    ql = _state(name, (n,), 1).reshape(meqn, n)
    qr = _state(name, (n,), 2).reshape(meqn, n)
    qr[:, :100] = ql[:, :100]
    rs = riemann.advection_3d if name == "advection" else riemann.euler_3d
    ag = dict(zip(rs.param_names, params))
    for ixyz in (1, 2, 3):
        wo, so, amo, apo = o3.rp_point(rp_id, params, ixyz, mw, ql, qr)
        out = rs(torch.tensor(ql, device='cuda'), torch.tensor(qr, device='cuda'), aux_global=ag, ixy=ixyz)
        for a, b in zip(out, (wo, so, amo, apo)):
            assert np.array_equal(a.cpu().numpy(), b), ixyz


def test_step3_argument_checks_new_solvers():
    q = np.zeros((5, 12, 12, 12), order="F")
    cfl = ctypes.c_double()
    P = _lib.make_problem(3, 4, 3, 2, 8, 8, 0.1, 0.1, o3.RP_EULER3D, [G, G1], [1, 2, 22, 0, 0, 0, 0], [4, 4, 4])
    with pytest.raises(_lib.ClawB200Error, match="meqn/mwaves"):
        _lib.call("clawb200_step3_host", ctypes.byref(P), 8, 0.1, _ptr(q), _ptr(q.copy("F")), None, 0.01, ctypes.byref(cfl))
    P = _lib.make_problem(3, 5, 3, 2, 8, 8, 0.1, 0.1, po.RP_EULER1D, [G, G1], [1, 2, 22, 0, 0, 0, 0], [4, 4, 4])
    with pytest.raises(_lib.ClawB200Error, match="no 3-D version"):
        _lib.call("clawb200_step3_host", ctypes.byref(P), 8, 0.1, _ptr(q), _ptr(q.copy("F")), None, 0.01, ctypes.byref(cfl))


# ---- the user seam in 3-D: vc-acoustics restated as RpUser3 -----------------------------------
def _user_acoustics3d():
    import pyclaw
    hdr = os.path.join(ROOT, "examples", "user_rp", "rp_acoustics3d_user.cuh")
    return pyclaw.riemann.from_header(hdr, meqn=4, mwaves=2, maux=2, ndims=(3,))


def test_user_rp3_equals_builtin_through_the_c_abi():
    rs = _user_acoustics3d()
    mbc = 2
    dx, dy, dz, dt = 0.02, 0.025, 0.03, 0.004
    for mx, my, mz in ((9, 7, 5), (130, 6, 4), (5, 4, 70)):
        rng = np.random.RandomState(mx)
        pad = (mx + 2 * mbc, my + 2 * mbc, mz + 2 * mbc)
        q = np.asfortranarray(rng.uniform(-1, 1, (4,) + pad))
        aux = np.asfortranarray(np.stack([rng.choice([1.0, 2.0, 3.5], pad), rng.choice([1.0, 2.0], pad)]))
        cases = [("clawb200_step3ds_host", [1, 2, -1, 0, 0, 0, 2], idir) for idir in (1, 2, 3)]
        cases += [("clawb200_step3_host", [1, 1 if t in (0, 10) else 2, t, 0, 0, 0, 2], None)
                  for t in (0, 10, 11, 20, 21, 22)]
        for fn, method, idir in cases:
            res = []
            for variant, rp_id in (("strict", po.RP_ACOUSTICS3D_VC), (rs._variant(), _lib.RP_USER)):
                _lib.set_variant(variant)
                P = _lib.make_problem(3, 4, 2, mbc, mx, my, dx, dy, rp_id, [], method, [4, 4], maux=2)
                qn = np.zeros_like(q, order="F")
                cfl = ctypes.c_double()
                args = [ctypes.byref(P), mz, dz, _ptr(q), _ptr(qn), _ptr(aux), dt] + ([idir] if idir else [])
                _lib.call(fn, *(args + [ctypes.byref(cfl)]))
                res.append((qn, cfl.value))
            _lib.set_variant("strict")
            assert np.array_equal(res[0][0], res[1][0]) and res[0][1] == res[1][1], (fn, method, idir)
            assert np.abs(res[0][0] - q).max() > 1e-3


def test_user_rp3_reproduces_the_pressure_3d_golden():
    """The reference's heterogeneous unsplit 3-D acoustics test (30^3, order_trans = 22, t = 2) on
    the user header through ``import pyclaw`` reproduces golden/pressure_3D.txt as the built-in
    solver does."""
    import pyclaw
    rs = _user_acoustics3d()
    mx = my = mz = 30
    solver = pyclaw.ClawSolver3D()
    solver.rp = rs
    for i in range(3):
        solver.bc_lower[i] = solver.aux_bc_lower[i] = pyclaw.BC.reflecting
        solver.bc_upper[i] = solver.aux_bc_upper[i] = pyclaw.BC.periodic
    solver.dim_split = False
    solver.mwaves, solver.limiters = 2, pyclaw.limiters.tvd.MC
    grid = pyclaw.Grid([pyclaw.Dimension('x', -1.0, 1.0, mx), pyclaw.Dimension('y', -1.0, 1.0, my),
                        pyclaw.Dimension('z', -1.0, 1.0, mz)])
    state = pyclaw.State(grid, 4, 2)
    grid.compute_c_center()
    X, Y, Z = grid._c_center
    aux = np.empty((2, mx, my, mz), order='F')
    aux[0] = 1.0 * (X < 0.) + 2.0 * (X >= 0.)
    aux[1] = 1.0 * (X < 0.) + 2.0 * (X >= 0.)
    state.aux = aux
    r = np.sqrt((X + 0.5) ** 2 + Y ** 2 + Z ** 2)
    q0 = np.zeros((4, mx, my, mz), order='F')
    q0[0] = (np.abs(r - 0.3) <= 0.1) * (1. + np.cos(np.pi * (r - 0.3) / 0.1))
    state.q[...] = q0
    claw = pyclaw.Controller()
    claw.keep_copy, claw.output_format = True, None
    claw.solution, claw.solver = pyclaw.Solution(state), solver
    claw.tfinal, claw.nout = 2.0, 10
    claw.run()
    pfinal = np.asarray(claw.frames[claw.nout].q)[0].reshape(-1)
    gold = np.loadtxt(os.path.join(HERE, "golden", "pressure_3D.txt"))
    assert np.linalg.norm(pfinal - gold) < 1e-13 and np.abs(pfinal - gold).max() < 1e-14


# ---- runs through import pyclaw ---------------------------------------------------------------
def _run3d(rp, q0, params, bc, dt, nsteps, dim_split, order_trans=22, arithmetic='strict', d=(1.0, 1.0, 1.0),
           limiters=4, cfl_max=1.0):
    import pyclaw
    meqn, mx, my, mz = q0.shape
    solver = pyclaw.ClawSolver3D()
    solver.rp = rp
    solver.arithmetic = arithmetic
    solver.dim_split = dim_split
    solver.order_trans = order_trans
    solver.mwaves = rp.nwaves(3)
    solver.limiters = limiters
    solver.dt_variable = False
    solver.dt_initial = dt
    solver.cfl_max, solver.cfl_desired = cfl_max, 0.9 * cfl_max
    for i in range(3):
        solver.bc_lower[i] = solver.bc_upper[i] = bc
    grid = pyclaw.Grid([pyclaw.Dimension('x', 0.0, d[0], mx), pyclaw.Dimension('y', 0.0, d[1], my),
                        pyclaw.Dimension('z', 0.0, d[2], mz)])
    state = pyclaw.State(grid, meqn)
    state.aux_global.update(params)
    state.q[...] = q0
    claw = pyclaw.Controller()
    claw.keep_copy, claw.output_format = True, None
    claw.solution, claw.solver = pyclaw.Solution(state), solver
    claw.tfinal, claw.nout = nsteps * dt, nsteps
    claw.run()
    return [np.asarray(f.q) for f in claw.frames]


@pytest.mark.parametrize("dim_split", [True, False])
@pytest.mark.parametrize("axis", [0, 1, 2])
def test_advection3d_exact_one_cell_shift(axis, dim_split):
    """u dt / dx = 1 with dyadic data: every step is an exact one-cell shift along the axis."""
    import pyclaw
    n = 16
    vel = [0.0, 0.0, 0.0]
    vel[axis] = 1.0
    rng = np.random.RandomState(axis)
    q0 = np.asfortranarray(rng.randint(-8, 9, (1, n, n, n)) / 8.0)
    frames = _run3d(pyclaw.riemann.advection_3d, q0, dict(u=vel[0], v=vel[1], w=vel[2]), pyclaw.BC.periodic,
                    1.0 / n, 4, dim_split)
    for k, qk in enumerate(frames):
        assert np.array_equal(qk, np.roll(q0, k, axis=1 + axis)), k


def _sod3d(n, axis, m=6):
    shape = [m, m, m]
    shape[axis] = n
    x = (np.arange(n) + 0.5) / n
    sh = [1, 1, 1]
    sh[axis] = n
    rho = np.where(x < 0.5, 1.0, 0.125).reshape(sh) * np.ones(shape)
    p = np.where(x < 0.5, 1.0, 0.1).reshape(sh) * np.ones(shape)
    q = np.zeros((5,) + tuple(shape), order='F')
    q[0], q[4] = rho, p / G1
    return q


def test_euler3d_sod_against_the_1d_solver():
    """A Sod tube along x, y and z in turn, uniform across: 20 split steps agree with ClawSolver1D +
    euler_with_efix to 1e-12 relative; the unsplit solver's three orientations agree with each other."""
    import pyclaw
    n, dt = 64, 2.0 ** -9
    solver = pyclaw.ClawSolver1D()
    solver.rp = pyclaw.riemann.euler_with_efix
    solver.mwaves, solver.limiters = 3, 4
    solver.dt_variable, solver.dt_initial = False, dt
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.outflow
    state = pyclaw.State(pyclaw.Grid(pyclaw.Dimension('x', 0.0, 1.0, n)), 3)
    state.aux_global.update(gamma=G, gamma1=G1)
    q3 = _sod3d(n, 0)
    state.q[...] = q3[[0, 1, 4], :, 0, 0]
    claw = pyclaw.Controller()
    claw.keep_copy, claw.output_format = True, None
    claw.solution, claw.solver = pyclaw.Solution(state), solver
    claw.tfinal, claw.nout = 20 * dt, 1
    claw.run()
    ref = np.asarray(claw.frames[-1].q)
    assert np.abs(ref - q3[[0, 1, 4], :, 0, 0]).max() > 0.1
    unsplit = []
    for axis in range(3):
        q0 = _sod3d(n, axis)
        for dim_split in (True, False):
            q = _run3d(pyclaw.riemann.euler_3d, q0, dict(gamma=G, gamma1=G1), pyclaw.BC.outflow, dt, 20,
                       dim_split, d=tuple(1.0 if a == axis else 6.0 / n for a in range(3)))[-1]
            line = np.moveaxis(q, 1 + axis, 1)[:, :, 2, 3][[0, 1 + axis, 4]]
            if dim_split:
                assert np.abs(line - ref).max() <= 1e-12 * np.abs(ref).max(), (axis, np.abs(line - ref).max())
            else:
                unsplit.append(line)
            # uniform across the tube: no transverse momentum (in the unsplit step the transverse
            # increments of neighbouring slices cancel up to rounding)
            tr = [m for m in (1, 2, 3) if m != 1 + axis]
            assert np.abs(q[tr]).max() <= (0.0 if dim_split else 1e-15 * np.abs(q).max())
    for line in unsplit[1:]:
        assert np.abs(line - unsplit[0]).max() <= 1e-12 * np.abs(unsplit[0]).max()
    assert np.abs(unsplit[0] - ref).max() < 1e-2


def _smooth_euler(n, seed=0):
    x = (np.arange(n) + 0.5) / n
    X, Y, Z = np.meshgrid(x, x, x, indexing='ij')
    rng = np.random.RandomState(seed)
    ph = rng.uniform(0, 2 * np.pi, 6)
    rho = 1.0 + 0.2 * np.sin(2 * np.pi * X + ph[0]) * np.cos(2 * np.pi * Y + ph[1])
    u = 0.3 * np.sin(2 * np.pi * Y + ph[2])
    v = 0.2 * np.cos(2 * np.pi * Z + ph[3])
    w = 0.25 * np.sin(2 * np.pi * X + ph[4])
    p = 1.0 + 0.1 * np.cos(2 * np.pi * (X + Y + Z) + ph[5])
    return np.asfortranarray(np.stack([rho, rho * u, rho * v, rho * w, p / G1 + 0.5 * rho * (u * u + v * v + w * w)]))


# The split step sweeps one ghost layer of slices only (step3ds.f: j = 0..my+1 in an x-sweep), so in
# the next sweep the limiter at a periodic boundary sees a swept neighbour on one side and an unswept
# second ghost layer on the other: with limiters the split step conserves up to that difference
# (~1e-6 relative over 50 steps here), exactly what the oracle computes.  Without limiters every flux
# depends on the two cells of its interface only and the sums are fixed to rounding.
@pytest.mark.parametrize("dim_split", [True, False])
def test_euler3d_periodic_conservation_and_fma_build(dim_split):
    import pyclaw
    n = 24
    q0 = _smooth_euler(n)
    run = lambda ar: _run3d(pyclaw.riemann.euler_3d, q0, dict(gamma=G, gamma1=G1), pyclaw.BC.periodic,
                            0.2 / n, 50, dim_split, arithmetic=ar, limiters=0 if dim_split else 4)[-1]
    qs = run('strict')
    for m in range(5):
        scale = np.abs(q0[m]).sum()
        assert abs(qs[m].sum() - q0[m].sum()) <= 1e-12 * scale, m
    assert np.abs(qs - q0).max() > 1e-2
    qf = run('fma')
    assert np.abs(qf - qs).max() <= 1e-12 * np.abs(qs).max()


# ---- the applications -------------------------------------------------------------------------
def _apps():
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    import apps
    return apps


@pytest.mark.parametrize("dim_split", [True, False])
def test_euler3d_app(dim_split):
    apps = _apps()
    c = apps.euler3d(mx=24, my=20, mz=16, tfinal=0.05, dim_split=dim_split)
    q0, q = np.asarray(c.frames[0].q), np.asarray(c.frames[-1].q)
    assert c.frames[-1].t == 0.05 and np.isfinite(q).all() and q[0].min() > 0
    for m in (0, 4):   # reflecting walls conserve mass and energy
        assert abs(q[m].sum() - q0[m].sum()) <= 1e-12 * abs(q0[m].sum()), m
    assert np.abs(q - q0).max() > 0.1


@pytest.mark.parametrize("dim_split", [True, False])
def test_advection3d_app(dim_split):
    apps = _apps()
    c = apps.advection3d(mx=20, my=16, mz=12, tfinal=0.25, dim_split=dim_split)
    q0, q = np.asarray(c.frames[0].q), np.asarray(c.frames[-1].q)
    assert c.frames[-1].t == 0.25 and np.isfinite(q).all()
    # periodic box: the unsplit step conserves to rounding, the limited split step up to its
    # one-ghost-layer sweeps (see test_euler3d_periodic_conservation_and_fma_build)
    assert abs(q.sum() - q0.sum()) <= (1e-9 if dim_split else 1e-12) * np.abs(q0).sum()
    assert np.abs(q - q0).max() > 0.05


def test_euler3d_app_two_ranks_equal_one():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.join(HERE, "mp_euler3d_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    sys.stdout.write(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
