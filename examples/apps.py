#!/usr/bin/env python
"""The reference's applications (``/apps`` and ``/test`` of the PyClaw snapshot) as functions over
``import pyclaw`` -- the scripts a PyClaw user would bring along, at their original settings
unless sizes are passed.  Each returns the Controller after ``run()`` (frames kept in memory).

    python examples/apps.py shockbubble mx=640 my=160
    python -m torch.distributed.run --nproc-per-node 8 examples/apps.py shockbubble mx=4096 my=1024 petsc=1

Problem definitions follow the reference scripts cited in each docstring; see
tests/test_gpu_golden.py for the versions that are checked against golden data.
"""
import sys

import numpy as np


def _pc(petsc):
    if petsc:
        import petclaw as pyclaw
    else:
        import pyclaw
    return pyclaw


def _run(pyclaw, solver, state, tfinal, nout, outdir=None):
    claw = pyclaw.Controller()
    claw.keep_copy = True
    claw.output_format = None if outdir is None else 'ascii'
    if outdir is not None:
        claw.outdir = outdir
    claw.tfinal, claw.nout = tfinal, nout
    claw.solution, claw.solver = pyclaw.Solution(state), solver
    claw.status = claw.run()
    return claw


def acoustics1d(mx=100, solver_type='classic', weno_order=5, petsc=False, tfinal=1.0, outdir=None):
    """apps/acoustics/1d/homogeneous/acoustics.py"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver1D() if solver_type == 'classic' else pyclaw.SharpClawSolver1D()
    if solver_type != 'classic':
        solver.weno_order = weno_order
    solver.mwaves, solver.limiters = 2, [4, 4]
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.periodic
    grid = pyclaw.Grid(pyclaw.Dimension('x', 0.0, 1.0, mx))
    state = pyclaw.State(grid, 2)
    state.aux_global.update(rho=1.0, bulk=1.0, zz=1.0, cc=1.0)
    xc = grid.x.center
    state.q[0, :] = np.exp(-100 * (xc - 0.75) ** 2)
    state.q[1, :] = 0.
    solver.dt_initial = grid.d[0] * 0.1
    return _run(pyclaw, solver, state, tfinal, 5, outdir)


def acoustics2d(mx=100, my=100, solver_type='classic', dim_split=True, petsc=False, tfinal=0.12, outdir=None):
    """apps/acoustics/2d/homogeneous/acoustics.py"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver2D() if solver_type == 'classic' else pyclaw.SharpClawSolver2D()
    solver.mwaves, solver.limiters = 2, [4, 4]
    solver.cfl_max, solver.cfl_desired = 0.5, 0.45
    if solver_type == 'classic':
        solver.dim_split, solver.order_trans = dim_split, 2
    for i in range(2):
        solver.bc_lower[i] = solver.bc_upper[i] = pyclaw.BC.outflow
    grid = pyclaw.Grid([pyclaw.Dimension('x', -1.0, 1.0, mx), pyclaw.Dimension('y', -1.0, 1.0, my)])
    state = pyclaw.State(grid, 3)
    state.aux_global.update(rho=1.0, bulk=4.0, zz=2.0, cc=2.0)
    Y, X = np.meshgrid(grid.y.center, grid.x.center)
    r = np.sqrt(X ** 2 + Y ** 2)
    state.q[0, :, :] = (np.abs(r - 0.5) <= 0.2) * (1. + np.cos(np.pi * (r - 0.5) / 0.2))
    solver.dt_initial = np.min(grid.d) / 2.0 * solver.cfl_desired
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def vc_acoustics2d(mx=200, my=200, petsc=False, tfinal=0.6, outdir=None):
    """apps/acoustics/2d/variable/acoustics.py: two materials, interface at x = 0"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver2D()
    solver.rp = pyclaw.riemann.vc_acoustics
    solver.mwaves, solver.limiters = 2, pyclaw.limiters.tvd.MC
    solver.dim_split, solver.order_trans = False, 2
    solver.bc_lower[0], solver.bc_upper[0] = pyclaw.BC.reflecting, pyclaw.BC.outflow
    solver.bc_lower[1], solver.bc_upper[1] = pyclaw.BC.reflecting, pyclaw.BC.outflow
    solver.aux_bc_lower[0], solver.aux_bc_upper[0] = pyclaw.BC.reflecting, pyclaw.BC.outflow
    solver.aux_bc_lower[1], solver.aux_bc_upper[1] = pyclaw.BC.reflecting, pyclaw.BC.outflow
    grid = pyclaw.Grid([pyclaw.Dimension('x', -1.0, 1.0, mx), pyclaw.Dimension('y', -1.0, 1.0, my)])
    state = pyclaw.State(grid, 3, 2)
    Y, X = np.meshgrid(grid.y.center, grid.x.center)
    aux = np.empty((2,) + X.shape, order='F')
    aux[0] = 4.0 * (X < 0.) + 1.0 * (X >= 0.)       # density
    aux[1] = 1.0 * (X < 0.) + 2.0 * (X >= 0.)       # sound speed
    state.aux = aux
    r = np.sqrt((X + 0.5) ** 2 + (Y - 0.) ** 2)
    state.q[0, :, :] = (np.abs(r - 0.3) <= 0.1) * (1. + np.cos(np.pi * (r - 0.3) / 0.1))
    solver.dt_initial = 0.1 * grid.d[0]
    return _run(pyclaw, solver, state, tfinal, 6, outdir)


def shockbubble(mx=160, my=40, petsc=False, tfinal=0.2, outdir=None):
    """apps/euler/2d/shockbubble/shockbubble.py (without the axisymmetric source term)"""
    pyclaw = _pc(petsc)
    gamma, gamma1 = 1.4, 0.4
    pinf = 5.
    rinf = (gamma1 + pinf * (gamma + 1.)) / ((gamma + 1.) + gamma1 * pinf)
    vinf = 1. / np.sqrt(gamma) * (pinf - 1.) / np.sqrt(0.5 * ((gamma + 1.) / gamma) * pinf + 0.5 * gamma1 / gamma)
    einf = 0.5 * rinf * vinf ** 2 + pinf / gamma1

    def incoming_shock(state, dim, t, qbc, mbc):
        if dim.nstart == 0:
            qbc[0, :mbc], qbc[1, :mbc], qbc[2, :mbc] = rinf, rinf * vinf, 0.
            qbc[3, :mbc], qbc[4, :mbc] = einf, 0.

    solver = pyclaw.ClawSolver2D()
    solver.mwaves, solver.limiters = 5, [4, 4, 4, 4, 2]
    solver.cfl_max, solver.cfl_desired = 0.5, 0.45
    solver.dim_split, solver.order_trans = False, 2
    solver.dt_initial = 0.005 * 160.0 / mx
    solver.user_bc_lower = incoming_shock
    solver.bc_lower[0], solver.bc_upper[0] = pyclaw.BC.custom, pyclaw.BC.outflow
    solver.bc_lower[1], solver.bc_upper[1] = pyclaw.BC.reflecting, pyclaw.BC.outflow
    grid = pyclaw.Grid([pyclaw.Dimension('x', 0.0, 2.0, mx), pyclaw.Dimension('y', 0.0, 0.5, my)])
    state = pyclaw.State(grid, 5)
    state.aux_global.update(gamma=gamma, gamma1=gamma1)
    Y, X = np.meshgrid(grid.y.center, grid.x.center)
    r = np.sqrt((X - 0.5) ** 2 + Y ** 2)
    state.q[0, :, :] = 0.1 * (r <= 0.2) + 1. * (r > 0.2)
    state.q[1, :, :] = 0.
    state.q[2, :, :] = 0.
    state.q[3, :, :] = 1. / gamma1
    state.q[4, :, :] = 1. * (r <= 0.2)
    return _run(pyclaw, solver, state, tfinal, 4, outdir)


def shallow1d(mx=500, solver_type='classic', ic='dam-break', petsc=False, tfinal=2.0, outdir=None):
    """apps/shallow/1d/shallow1D.py"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver1D() if solver_type == 'classic' else pyclaw.SharpClawSolver1D()
    solver.mwaves, solver.limiters = 2, pyclaw.limiters.tvd.vanleer
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.outflow
    grid = pyclaw.Grid(pyclaw.Dimension('x', -5.0, 5.0, mx))
    state = pyclaw.State(grid, 2)
    state.aux_global['grav'] = 1.0
    xc = grid.x.center
    hl, ul, hr, ur = (3., 0., 1., 0.) if ic == 'dam-break' else (1., 1., 1., -1.)
    state.q[0, :] = hl * (xc <= 0.) + hr * (xc > 0.)
    state.q[1, :] = hl * ul * (xc <= 0.) + hr * ur * (xc > 0.)
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def shallow2d(mx=150, my=150, solver_type='classic', petsc=False, tfinal=2.5, outdir=None):
    """apps/shallow/2d/shallow2D.py: radial dam break"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver2D() if solver_type == 'classic' else pyclaw.SharpClawSolver2D()
    solver.mwaves, solver.limiters = 3, pyclaw.limiters.tvd.MC
    if solver_type == 'classic':
        solver.dim_split = True
    else:
        solver.time_integrator, solver.cfl_max, solver.cfl_desired = 'SSP33', 0.6, 0.5
    solver.bc_lower[0], solver.bc_upper[0] = pyclaw.BC.outflow, pyclaw.BC.reflecting
    solver.bc_lower[1], solver.bc_upper[1] = pyclaw.BC.outflow, pyclaw.BC.reflecting
    grid = pyclaw.Grid([pyclaw.Dimension('x', -2.5, 2.5, mx), pyclaw.Dimension('y', -2.5, 2.5, my)])
    state = pyclaw.State(grid, 3)
    state.aux_global['grav'] = 1.0
    Y, X = np.meshgrid(grid.y.center, grid.x.center)
    r = np.sqrt(X ** 2 + Y ** 2)
    state.q[0, :, :] = 2.0 * (r <= 0.5) + 1.0 * (r > 0.5)
    state.q[1, :, :] = 0.
    state.q[2, :, :] = 0.
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def shallow_sphere(mx=40, my=20, petsc=False, tfinal=10.0, outdir=None):
    """apps/shallow-sphere/shallow_4_Rossby_Haurwitz_wave.py"""
    pyclaw = _pc(petsc)
    from pyclaw_b200.apps import shallow_sphere as app
    state, solver = app.setup(pyclaw, mx, my)
    solver.dt_initial = 0.1 * state.grid.d[0] / 4.0
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def stegoton(cells_per_layer=6, layers=100, solver_type='classic', petsc=False, tfinal=50.0, outdir=None):
    """apps/elasticity/1d/stegoton/stegoton.py: nonlinear elasticity in a layered medium"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver1D() if solver_type == 'classic' else pyclaw.SharpClawSolver1D()
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.periodic
    solver.aux_bc_lower[0] = solver.aux_bc_upper[0] = pyclaw.BC.periodic
    solver.fwave, solver.mwaves = True, 2
    solver.max_steps = 5000000
    xupper = float(layers)
    grid = pyclaw.Grid(pyclaw.Dimension('x', 0.0, xupper, layers * cells_per_layer))
    state = pyclaw.State(grid, 2)
    xc = grid.x.center
    xfrac = xc - np.floor(xc)
    aux = np.empty((3, len(xc)), order='F')
    aux[0] = 1.0 * (xfrac < 0.5) + 4.0 * (xfrac >= 0.5)       # density
    aux[1] = 1.0 * (xfrac < 0.5) + 4.0 * (xfrac >= 0.5)       # bulk modulus
    aux[2] = 0.
    state.aux = aux
    sigma = np.exp(-((xc - xupper / 2.) / 10.) ** 2.)
    state.q[0, :] = np.log(sigma + 1.) / aux[1]
    state.q[1, :] = 0.
    return _run(pyclaw, solver, state, tfinal, 5, outdir)


def psystem(cells_per_layer=20, petsc=False, tfinal=2.0, outdir=None):
    """test/psystem/psystem.py: 2-D p-system in a checkerboard medium (f-waves, unsplit)"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver2D()
    solver.mwaves, solver.limiters = 2, pyclaw.limiters.tvd.superbee
    for i in range(2):
        solver.bc_lower[i] = solver.aux_bc_lower[i] = pyclaw.BC.reflecting
        solver.bc_upper[i] = solver.aux_bc_upper[i] = pyclaw.BC.outflow
    solver.fwave, solver.dim_split = True, False
    solver.cfl_max, solver.cfl_desired = 1.0, 0.9
    n = int(5 * cells_per_layer)
    grid = pyclaw.Grid([pyclaw.Dimension('x', 0.25, 5.25, n), pyclaw.Dimension('y', 0.25, 5.25, n)])
    state = pyclaw.State(grid, 3, 4)
    x, y = grid.x.center, grid.y.center
    yy, xx = np.meshgrid(y - np.floor(y), x - np.floor(x))
    same = (xx <= 0.5) * (yy <= 0.5) + (xx > 0.5) * (yy > 0.5)
    aux = np.empty((4, len(x), len(y)), order='F')
    aux[0] = 1. * same + 4. * (1 - same)
    aux[1] = 1. * same + 4. * (1 - same)
    aux[2] = 2.                                               # exponential stress law
    Y, X = np.meshgrid(y, x)
    s = 5. * np.exp(-(X - 0.25) ** 2 / 10. - (Y - 0.25) ** 2 / 10.)
    eps0 = np.log(s + 1.) / aux[1]
    aux[3] = eps0
    state.aux = aux
    state.q[0, :, :] = eps0
    state.q[1, :, :] = 0.
    state.q[2, :, :] = 0.

    def keep_strain_copy(solver, solution):                  # the script's b4step
        st = solution.states[0]
        st.aux[3, :, :] = st.q[0, :, :]
        solver.apply_aux_bcs(st)
    solver.start_step = keep_strain_copy
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def bump1d(mx=200, petsc=False, tfinal=0.7, eps=1e-3, outdir=None):
    """Shallow water over a bump (pyclaw.riemann.shallow_bathymetry_fwave): LeVeque's perturbed steady
    state (J. Comput. Phys. 146, 1998, sec. 5).  Bottom b = 0.25 (cos(10 pi (x - 0.5)) + 1) for
    |x - 0.5| < 0.1, else 0, on [0, 1]; the lake at rest eta = h + b = 1 carries a pulse eta = 1 + eps
    on 0.1 < x < 0.2; g = 9.81, outflow boundaries.  The well-balanced solver keeps the undisturbed
    water exactly at rest while the pulse crosses the bump."""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver1D()
    solver.rp = pyclaw.riemann.shallow_bathymetry_fwave
    solver.fwave = True
    solver.mwaves, solver.limiters = 2, pyclaw.limiters.tvd.MC
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.outflow
    solver.aux_bc_lower[0] = solver.aux_bc_upper[0] = pyclaw.BC.outflow
    grid = pyclaw.Grid(pyclaw.Dimension('x', 0.0, 1.0, mx))
    state = pyclaw.State(grid, 2, 1)
    state.aux_global['grav'] = 9.81
    xc = grid.x.center
    b = np.where(np.abs(xc - 0.5) < 0.1, 0.25 * (np.cos(10 * np.pi * (xc - 0.5)) + 1.0), 0.0)
    state.aux[0, :] = b
    state.q[0, :] = 1.0 + eps * ((xc > 0.1) & (xc < 0.2)) - b
    state.q[1, :] = 0.
    solver.dt_initial = 0.2 * grid.d[0]
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def seamount2d(mx=200, my=200, dim_split=True, petsc=False, tfinal=1.0, outdir=None):
    """Shallow water over bathymetry in a closed basin (pyclaw.riemann.shallow_bathymetry_fwave): a
    Gaussian hump on the surface west of a Gaussian seamount, reflecting walls on [-1, 1]^2, g = 9.81.
    The bottom rises from b = -1 to b = -0.2 at the seamount's top (0.25, 0), so h >= 0.2 everywhere.
    dim_split=False runs the unsplit step with transverse corrections (order_trans = 2)."""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver2D()
    solver.rp = pyclaw.riemann.shallow_bathymetry_fwave
    solver.fwave = True
    solver.mwaves, solver.limiters = 3, pyclaw.limiters.tvd.MC
    solver.dim_split, solver.order_trans = bool(dim_split), 2
    for i in range(2):
        solver.bc_lower[i] = solver.bc_upper[i] = pyclaw.BC.reflecting
        solver.aux_bc_lower[i] = solver.aux_bc_upper[i] = pyclaw.BC.reflecting
    grid = pyclaw.Grid([pyclaw.Dimension('x', -1.0, 1.0, mx), pyclaw.Dimension('y', -1.0, 1.0, my)])
    state = pyclaw.State(grid, 3, 1)
    state.aux_global['grav'] = 9.81
    Y, X = np.meshgrid(grid.y.center, grid.x.center)
    b = -1.0 + 0.8 * np.exp(-((X - 0.25) ** 2 + Y ** 2) / 0.2 ** 2)
    state.aux[0, :, :] = b
    state.q[0, :, :] = 0.1 * np.exp(-((X + 0.5) ** 2 + Y ** 2) / 0.1 ** 2) - b
    state.q[1, :, :] = 0.
    state.q[2, :, :] = 0.
    solver.dt_initial = 0.2 * min(grid.d)
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def acoustics3d(mx=256, my=4, mz=4, petsc=False, tfinal=2.0, outdir=None, test='hom', upper_bc=None):
    """test/acoustics/3d/acoustics.py: 'hom' (homogeneous medium, dimensional splitting, periodic) or
    'het' (impedance and sound speed double at x = 0, unsplit with order_trans = 22, reflecting lower
    boundaries; the reference runs it at 30^3 against test/pressure_3D.txt)"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver3D()
    for i in range(3):
        solver.bc_lower[i] = solver.bc_upper[i] = pyclaw.BC.periodic
        solver.aux_bc_lower[i] = solver.aux_bc_upper[i] = pyclaw.BC.periodic
    solver.dim_split, solver.mwaves, solver.limiters = True, 2, pyclaw.limiters.tvd.MC
    zr = cr = 1.0
    if test == 'het':
        solver.dim_split = False
        for i in range(3):
            solver.bc_lower[i] = solver.aux_bc_lower[i] = pyclaw.BC.reflecting
            # the reference's script keeps the upper boundaries periodic next to reflecting lower ones;
            # a slab partition (like the reference's DMDA, petclaw/state.py:205-208) cannot wrap one
            # side of the partitioned dimension only: upper_bc overrides
            if upper_bc is not None:
                solver.bc_upper[i] = solver.aux_bc_upper[i] = upper_bc
        zr = cr = 2.0
    grid = pyclaw.Grid([pyclaw.Dimension('x', -1.0, 1.0, mx), pyclaw.Dimension('y', -1.0, 1.0, my),
                        pyclaw.Dimension('z', -1.0, 1.0, mz)])
    state = pyclaw.State(grid, 4, 2)
    grid.compute_c_center()
    X, Y, Z = grid._c_center
    aux = np.empty((2,) + X.shape, order='F')
    aux[0] = 1.0 * (X < 0.) + zr * (X >= 0.)
    aux[1] = 1.0 * (X < 0.) + cr * (X >= 0.)
    state.aux = aux
    q0 = np.zeros((4,) + X.shape, order='F')
    if test == 'het':
        r = np.sqrt((X + 0.5) ** 2 + Y ** 2 + Z ** 2)
        q0[0] = (np.abs(r - 0.3) <= 0.1) * (1. + np.cos(np.pi * (r - 0.3) / 0.1))
    else:
        r = np.abs(X + 0.5)
        q0[0] = (r <= 0.2) * (1. + np.cos(np.pi * r / 0.2))
    state.q[...] = q0
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def burgers(mx=500, solver_type='classic', petsc=False, tfinal=0.5, outdir=None):
    """apps/burgers/1d/burgers1D.py"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver1D() if solver_type == 'classic' else pyclaw.SharpClawSolver1D()
    solver.rp = pyclaw.riemann.burgers
    solver.mwaves, solver.limiters = 1, pyclaw.limiters.tvd.vanleer
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.periodic
    grid = pyclaw.Grid(pyclaw.Dimension('x', 0.0, 1.0, mx))
    state = pyclaw.State(grid, 1)
    xc = grid.x.center
    state.q[0, :] = np.sin(np.pi * 2 * xc) + 0.50
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def wcblast(mx=500, solver_type='classic', petsc=False, tfinal=0.038, outdir=None):
    """apps/euler/1d/wcblast/wcblast.py: Woodward-Colella interacting blast waves"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver1D() if solver_type == 'classic' else pyclaw.SharpClawSolver1D()
    solver.mwaves, solver.limiters = 3, 4
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.reflecting
    grid = pyclaw.Grid([pyclaw.Dimension('x', 0.0, 1.0, mx)])
    state = pyclaw.State(grid, 3)
    state.aux_global.update(gamma=1.4, gamma1=0.4)
    x = grid.x.center
    state.q[0, :] = 1.
    state.q[1, :] = 0.
    state.q[2, :] = ((x < 0.1) * 1.e3 + (0.1 <= x) * (x < 0.9) * 1.e-2 + (0.9 <= x) * 1.e2) / 0.4
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def vc_advection1d(mx=100, petsc=False, tfinal=1.0, outdir=None):
    """apps/advection/1d/variable/variable_coefficient_advection.py"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver1D()
    solver.rp = pyclaw.riemann.advection_color
    solver.mwaves, solver.limiters = 1, pyclaw.limiters.tvd.MC
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.periodic
    solver.aux_bc_lower[0] = solver.aux_bc_upper[0] = pyclaw.BC.periodic
    grid = pyclaw.Grid(pyclaw.Dimension('x', 0.0, 1.0, mx))
    state = pyclaw.State(grid, 1, 1)
    xc = grid.x.center
    state.aux[0, :] = np.sin(2. * np.pi * xc) + 2
    state.q[0, :] = np.exp(-200. * (xc - 0.25) ** 2) + 1.0 * (xc > 0.6) * (xc < 0.8)
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def annulus(mx=40, my=120, petsc=False, tfinal=1.0, outdir=None):
    """apps/advection/2d/annulus/advection_annulus.py: solid-body rotation on a polar grid
    (edge velocities from a stream function, capacity function = cell area ratio)"""
    pyclaw = _pc(petsc)
    solver = pyclaw.ClawSolver2D()
    solver.rp = pyclaw.riemann.vc_advection
    solver.mwaves, solver.limiters = 1, pyclaw.limiters.tvd.vanleer
    solver.dim_split, solver.order_trans = False, 2
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.outflow
    solver.bc_lower[1] = solver.bc_upper[1] = pyclaw.BC.periodic
    solver.aux_bc_lower[0] = solver.aux_bc_upper[0] = pyclaw.BC.custom
    solver.aux_bc_lower[1] = solver.aux_bc_upper[1] = pyclaw.BC.periodic
    rlo, rhi = 0.2, 1.0
    grid = pyclaw.Grid([pyclaw.Dimension('r', rlo, rhi, mx), pyclaw.Dimension('t', 0.0, 2 * np.pi, my)])
    dr, dth = grid.d
    mbc = solver.mbc
    stream = lambda xp, yp: np.pi * (xp ** 2 + yp ** 2)

    def edge_data(i0, i1, j0, j1):
        """aux for cells i0..i1-1, j0..j1-1 (0-based, may lie outside the grid)"""
        re = rlo + dr * np.arange(i0, i1 + 1)
        te = dth * np.arange(j0, j1 + 1)
        T, R = np.meshgrid(te, re)
        X, Y = R * np.cos(T), R * np.sin(T)
        a = np.empty((3, i1 - i0, j1 - j0), order='F')
        a[0] = (stream(X[:-1, 1:], Y[:-1, 1:]) - stream(X[:-1, :-1], Y[:-1, :-1])) / dth
        a[1] = -(stream(X[1:, :-1], Y[1:, :-1]) - stream(X[:-1, :-1], Y[:-1, :-1])) / dr
        area = 0.5 * np.abs((X[1:, 1:] - X[:-1, :-1]) * (Y[:-1, 1:] - Y[1:, :-1]) -
                            (X[:-1, 1:] - X[1:, :-1]) * (Y[1:, 1:] - Y[:-1, :-1]))
        a[2] = area / (dr * dth)
        return a

    state = pyclaw.State(grid, 1, 3)
    j0, j1 = grid.dimensions[1].nstart, grid.dimensions[1].nend
    state.aux = edge_data(0, mx, j0, j1)
    state.mcapa = 2
    import torch
    lo = torch.as_tensor(edge_data(-mbc, 0, j0 - mbc, j1 + mbc).transpose(0, 2, 1).copy(), device=state.device).permute(0, 2, 1)
    hi = torch.as_tensor(edge_data(mx, mx + mbc, j0 - mbc, j1 + mbc).transpose(0, 2, 1).copy(), device=state.device).permute(0, 2, 1)

    def aux_lower(state, dim, t, auxbc, mbc):
        auxbc[:, :mbc, :] = lo

    def aux_upper(state, dim, t, auxbc, mbc):
        auxbc[:, -mbc:, :] = hi
    solver.user_aux_bc_lower, solver.user_aux_bc_upper = aux_lower, aux_upper
    rc = rlo + dr * (np.arange(mx) + 0.5)
    tc = dth * (np.arange(j0, j1) + 0.5)
    T, R = np.meshgrid(tc, rc)
    X, Y = R * np.cos(T), R * np.sin(T)
    state.q[0, :, :] = np.exp(-40. * ((X + 0.4) ** 2 + Y ** 2)) + np.exp(-40. * ((X - 0.5) ** 2 + (Y - 0.3) ** 2))
    solver.dt_initial = 0.1
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def _solver3d(pyclaw, solver_type, dim_split):
    """ClawSolver3D (dimensional splitting or the unsplit step), or SharpClawSolver3D (WENO5, SSP104).
    SharpClaw's 3-D Courant number is the largest of the three directions, not their sum, so the
    SharpClaw variant runs at cfl_desired = 0.8, cfl_max = 0.9: three directions at 0.8 add up to the
    2.4 that SSP104 allows in one dimension."""
    if solver_type == 'sharpclaw':
        solver = pyclaw.SharpClawSolver3D()
        solver.cfl_desired, solver.cfl_max = 0.8, 0.9
        return solver
    if solver_type != 'classic':
        raise ValueError("solver_type must be 'classic' or 'sharpclaw'")
    solver = pyclaw.ClawSolver3D()
    solver.dim_split = dim_split
    return solver


def euler3d(mx=64, my=64, mz=64, petsc=False, tfinal=0.1, dim_split=True, outdir=None, solver_type='classic'):
    """3-D Euler equations (Roe solver with entropy fix, pyclaw.riemann.euler_3d): a spherical blast
    wave in the unit box with reflecting walls.  Gas at rest, rho = 1; pressure 10 inside the sphere
    of radius 0.2 around the centre, 0.1 outside.  dim_split=False runs the unsplit step with
    transverse corrections (order_trans = 22); solver_type='sharpclaw' runs SharpClawSolver3D."""
    pyclaw = _pc(petsc)
    solver = _solver3d(pyclaw, solver_type, dim_split)
    solver.rp = pyclaw.riemann.euler_3d
    solver.mwaves, solver.limiters = 3, pyclaw.limiters.tvd.MC
    for i in range(3):
        solver.bc_lower[i] = solver.bc_upper[i] = pyclaw.BC.reflecting
    grid = pyclaw.Grid([pyclaw.Dimension('x', 0.0, 1.0, mx), pyclaw.Dimension('y', 0.0, 1.0, my),
                        pyclaw.Dimension('z', 0.0, 1.0, mz)])
    state = pyclaw.State(grid, 5)
    gamma = 1.4
    state.aux_global.update(gamma=gamma, gamma1=gamma - 1.0)
    grid.compute_c_center()
    X, Y, Z = grid._c_center
    r = np.sqrt((X - 0.5) ** 2 + (Y - 0.5) ** 2 + (Z - 0.5) ** 2)
    p = np.where(r <= 0.2, 10.0, 0.1)
    q0 = np.zeros((5,) + X.shape, order='F')
    q0[0] = 1.0
    q0[4] = p / (gamma - 1.0)
    state.q[...] = q0
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def advection3d(mx=32, my=32, mz=32, petsc=False, tfinal=1.0, dim_split=True, u=1.0, v=0.5, w=0.25, outdir=None,
                solver_type='classic'):
    """3-D constant-coefficient advection (pyclaw.riemann.advection_3d) of a Gaussian in the
    periodic unit box with velocity (u, v, w); solver_type='sharpclaw' runs SharpClawSolver3D."""
    pyclaw = _pc(petsc)
    solver = _solver3d(pyclaw, solver_type, dim_split)
    solver.rp = pyclaw.riemann.advection_3d
    solver.mwaves, solver.limiters = 1, pyclaw.limiters.tvd.MC
    for i in range(3):
        solver.bc_lower[i] = solver.bc_upper[i] = pyclaw.BC.periodic
    grid = pyclaw.Grid([pyclaw.Dimension('x', 0.0, 1.0, mx), pyclaw.Dimension('y', 0.0, 1.0, my),
                        pyclaw.Dimension('z', 0.0, 1.0, mz)])
    state = pyclaw.State(grid, 1)
    state.aux_global.update(u=u, v=v, w=w)
    grid.compute_c_center()
    X, Y, Z = grid._c_center
    state.q[0] = np.exp(-50.0 * ((X - 0.5) ** 2 + (Y - 0.5) ** 2 + (Z - 0.5) ** 2))
    return _run(pyclaw, solver, state, tfinal, 10, outdir)


def deformation_field(X, Y, Z):
    """LeVeque's 3-D deformation flow on the unit cube (divergence free, zero normal velocity on the faces)"""
    s2 = lambda a: np.sin(np.pi * a) ** 2
    s = lambda a: np.sin(2 * np.pi * a)
    return np.stack([2 * s2(X) * s(Y) * s(Z), -s(X) * s2(Y) * s(Z), -s(X) * s(Y) * s2(Z)])


def transport3d(mx=32, my=32, mz=32, petsc=False, period=1.0, tfinal=None, dim_split=True, outdir=None,
                solver_type='classic'):
    """Conservative transport q_t + div(u q) = 0 of a cosine bell in LeVeque's 3-D deformation field on the
    periodic unit cube (pyclaw.riemann.vc_advection_fwave_3d, solver.fwave = True).  A start_step hook
    scales the field by cos(pi t / period), evaluated at the middle of each step, and rewrites state.aux
    (ghost cells included): the flow reverses, so at t = period (the default tfinal) the exact solution
    is the initial data again.  dim_split / solver_type select the split or unsplit classic step or
    SharpClawSolver3D."""
    pyclaw = _pc(petsc)
    import torch
    solver = _solver3d(pyclaw, solver_type, dim_split)
    solver.rp = pyclaw.riemann.vc_advection_fwave_3d
    solver.fwave = True
    solver.mwaves, solver.limiters = 1, pyclaw.limiters.tvd.MC
    for i in range(3):
        solver.bc_lower[i] = solver.bc_upper[i] = pyclaw.BC.periodic
        solver.aux_bc_lower[i] = solver.aux_bc_upper[i] = pyclaw.BC.periodic
    grid = pyclaw.Grid([pyclaw.Dimension('x', 0.0, 1.0, mx), pyclaw.Dimension('y', 0.0, 1.0, my),
                        pyclaw.Dimension('z', 0.0, 1.0, mz)])
    state = pyclaw.State(grid, 1, 3)
    grid.compute_c_center()
    X, Y, Z = grid._c_center
    aux0 = deformation_field(X, Y, Z)
    state.aux = aux0
    r = np.sqrt((X - 0.35) ** 2 + (Y - 0.35) ** 2 + (Z - 0.35) ** 2)
    state.q[0] = 0.5 * (1.0 + np.cos(np.pi * np.minimum(r / 0.2, 1.0)))
    field = torch.as_tensor(np.ascontiguousarray(aux0), device=state.aux.device)

    def reverse_flow(solver, solution):                      # the script's b4step
        st = solution.states[0]
        st.aux[...] = field * float(np.cos(np.pi * (solution.t + 0.5 * solver.dt) / period))
        solver.apply_aux_bcs(st)
    solver.start_step = reverse_flow
    return _run(pyclaw, solver, state, period if tfinal is None else tfinal, 10, outdir)


APPS = {f.__name__: f for f in (acoustics1d, acoustics2d, vc_acoustics2d, shockbubble, shallow1d, shallow2d,
                                shallow_sphere, stegoton, psystem, bump1d, seamount2d, acoustics3d, burgers,
                                wcblast, vc_advection1d, annulus, euler3d, advection3d, transport3d)}


def main(argv):
    if len(argv) < 2 or argv[1] not in APPS:
        print("usage: apps.py <%s> [key=value ...]" % "|".join(sorted(APPS)))
        return 2
    kwargs = {}
    for a in argv[2:]:
        k, v = a.split('=', 1)
        try:
            v = int(v)
        except ValueError:
            try:
                v = float(v)
            except ValueError:
                pass
        kwargs[k] = v
    claw = APPS[argv[1]](**kwargs)
    q = np.asarray(claw.frames[-1].q)
    print("%s: %d steps in the last output interval, t = %g, q range [%g, %g]"
          % (argv[1], claw.status['numsteps'], claw.frames[-1].t, q.min(), q.max()))
    return 0


if __name__ == "__main__":
    import os
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.exit(main(sys.argv))
