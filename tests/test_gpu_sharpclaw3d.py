"""SharpClaw in 3-D (clawb200_sharpclaw_stage3, SharpClawSolver3D): the device dq against the CPU
restatement oracle3d.sc_flux3 bit for bit, the stage modes, whole runs against the oracle driver, the user
3-D header, the 1-D anchor, conservation, the fma build, the applications, the dq_src path, two ranks and
the argument checks."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle3d as o3
from pyclaw_b200 import _lib

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
G, G1 = 1.4, 0.4
MBC = 3
ERR_INVALID, ERR_UNSUPPORTED = -1, -2  # CLAWB200_ERR_*
SOLVERS = {"advection": (o3.RP_ADVECTION3D, [0.7, -0.45, 0.3], 1, 1, 0),
           "euler": (o3.RP_EULER3D, [G, G1], 5, 3, 0),
           "acoustics": (o3.RP_ACOUSTICS3D_VC, [], 4, 2, 2)}
VARIANTS = {"f32": o3.WENO_PYWENO_F32, "f64": o3.WENO_PYWENO_F64, "old": o3.WENO_OLD, "tvd2": o3.RECON_TVD2}
LIMS = {1: [4], 2: [1, 3], 4: [1, 2, 3, 4], 5: [1, 2, 3, 4, 5]}  # tvd2: a limiter per component
SHAPES = [(9, 7, 5), (130, 6, 4), (20, 33, 17), (5, 4, 70)]
BIG = (260, 40, 40)  # several CTAs along x, several row chunks (kernel A) and k-chunks (kernel B)


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _fields(name, pad, seed):
    rng = np.random.RandomState(seed)
    aux = None
    if name == "advection":
        q = rng.uniform(-1, 1, (1,) + pad)
    elif name == "acoustics":
        q = rng.uniform(-1, 1, (4,) + pad)
        rho, c = rng.choice([1.0, 3.0], pad), rng.choice([1.0, 0.5], pad)
        aux = np.asfortranarray(np.stack([rho * c, c]))
    else:
        rho = rng.uniform(0.5, 2.0, pad)
        u = rng.uniform(-1.0, 1.0, (3,) + pad)
        p = rng.uniform(0.5, 2.0, pad)
        q = np.concatenate([rho[None], rho * u, (p / G1 + 0.5 * rho * (u * u).sum(0))[None]])
    return np.asfortranarray(q), aux


def _problem(name, variant, mx, my, maux=None):
    rp_id, params, meqn, mw, ma = SOLVERS[name]
    lim = LIMS[meqn]
    P = _lib.make_problem(3, meqn, mw, MBC, mx, my, 0.02, 0.025, rp_id, params, [1, 2, 0, 0, 0, 0, ma],
                          lim[:mw] if variant != o3.RECON_TVD2 else lim, maux=ma if maux is None else maux,
                          weno_variant=variant)
    return P, lim


def _device_dq(name, variant, shape, q, aux, dt):
    mx, my, mz = shape
    P, _ = _problem(name, variant, mx, my)
    dq = np.zeros_like(q, order="F")
    cfl = ctypes.c_double()
    _lib.call("clawb200_sharpclaw_dq3_host", ctypes.byref(P), mz, 0.03, _ptr(q), _ptr(dq),
              None if aux is None else _ptr(aux), dt, ctypes.byref(cfl))
    return dq, cfl.value


def _oracle_dq(name, variant, shape, q, aux, dt):
    rp_id, params, meqn, mw, _ = SOLVERS[name]
    return o3.sc_flux3(rp_id, params, mw, MBC, *shape, q, 0.02, 0.025, 0.03, dt, variant, aux=aux,
                       mthlim=LIMS[meqn])


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("name", list(SOLVERS))
def test_dq3_vs_oracle(name, variant, shape):
    pad = tuple(n + 2 * MBC for n in shape)
    q, aux = _fields(name, pad, sum(shape) + len(variant))
    v = VARIANTS[variant]
    dt = 0.004
    dq_o, cfl_o = _oracle_dq(name, v, shape, q, aux, dt)
    dq_g, cfl_g = _device_dq(name, v, shape, q, aux, dt)
    assert np.array_equal(dq_g, dq_o), np.abs(dq_g - dq_o).max()
    assert cfl_g == cfl_o and cfl_o > 0.01
    assert np.abs(dq_o).max() > 1e-3


@pytest.mark.parametrize("name,variant", [("advection", "f32"), ("euler", "f64"), ("acoustics", "tvd2"),
                                          ("euler", "old")])
def test_dq3_vs_oracle_many_ctas(name, variant):
    pad = tuple(n + 2 * MBC for n in BIG)
    q, aux = _fields(name, pad, 5)
    v = VARIANTS[variant]
    dq_o, cfl_o = _oracle_dq(name, v, BIG, q, aux, 0.004)
    dq_g, cfl_g = _device_dq(name, v, BIG, q, aux, 0.004)
    assert np.array_equal(dq_g, dq_o) and cfl_g == cfl_o


# ---- stage modes on device buffers ------------------------------------------------------------
@pytest.mark.parametrize("name", ["euler", "acoustics"])
def test_stage3_modes(name):
    import torch
    shape = (20, 33, 17)
    mx, my, mz = shape
    pad = tuple(n + 2 * MBC for n in shape)
    q, aux = _fields(name, pad, 11)
    qa = _fields(name, pad, 12)[0]
    dt = 0.004
    dq_o, cfl_o = _oracle_dq(name, o3.WENO_PYWENO_F32, shape, q, aux, dt)
    P, _ = _problem(name, o3.WENO_PYWENO_F32, mx, my)
    # device layout: q[m][k][j][i] with pitch = mx + 2 mbc (the Fortran array's memory order per component)
    dev = lambda a: torch.tensor(np.ascontiguousarray(np.transpose(a, (0, 3, 2, 1))), device='cuda')
    host = lambda t: np.asfortranarray(np.transpose(t.cpu().numpy(), (0, 3, 2, 1)))
    P.pitch, P.mstride = pad[0], pad[0] * pad[1] * pad[2]
    P.maux = 0 if aux is None else 2
    qd, qad = dev(q), dev(qa)
    auxd = None if aux is None else dev(aux)
    inner = (slice(None),) + (slice(MBC, -MBC),) * 3
    cfl = torch.zeros(1, dtype=torch.float64, device='cuda')
    dqt = torch.tensor(dq_o)
    qt, qat = torch.tensor(q), torch.tensor(qa)
    sixth = torch.full((), 6.0, dtype=torch.float64)
    expect = {(0, 1.0): qt + dqt, (0, 6.0): qt + torch.div(dqt, sixth),
              (1, 1.0): 0.75 * qat + 0.25 * (qt + dqt), (2, 1.0): (qat + 0.6 * qt) + 0.1 * dqt}
    ca_cb = {0: (0.0, 0.0), 1: (0.75, 0.25), 2: (0.6, 0.1)}
    for (mode, div), exp in expect.items():
        out = torch.zeros_like(qd)
        cfl.zero_()
        ca, cb = ca_cb[mode]
        _lib.call("clawb200_sharpclaw_stage3", ctypes.byref(P), mz, 0.03, ctypes.c_void_p(qd.data_ptr()),
                  ctypes.c_void_p(qad.data_ptr()) if mode in (1, 2) else None, ctypes.c_void_p(out.data_ptr()), None,
                  None if auxd is None else ctypes.c_void_p(auxd.data_ptr()), dt, mode, ca, cb, div,
                  ctypes.c_void_p(cfl.data_ptr()), None)
        torch.cuda.synchronize()
        got = host(out)
        assert np.array_equal(got[inner], exp.numpy()[inner]), (mode, div)
        assert cfl.item() == cfl_o
    # mode 3 with dq_out, and a stage that writes out and dq_out at once
    for mode in (3, 0):
        dqd = torch.zeros_like(qd)
        out = torch.zeros_like(qd)
        _lib.call("clawb200_sharpclaw_stage3", ctypes.byref(P), mz, 0.03, ctypes.c_void_p(qd.data_ptr()), None,
                  ctypes.c_void_p(out.data_ptr()) if mode == 0 else None, ctypes.c_void_p(dqd.data_ptr()),
                  None if auxd is None else ctypes.c_void_p(auxd.data_ptr()), dt, mode, 0.0, 0.0, 1.0,
                  ctypes.c_void_p(cfl.data_ptr()), None)
        torch.cuda.synchronize()
        assert np.array_equal(host(dqd), dq_o)
        if mode == 0:
            assert np.array_equal(host(out)[inner], (qt + dqt).numpy()[inner])


# ---- whole runs through import pyclaw ---------------------------------------------------------
def _blast(n):
    x = (np.arange(n) + 0.5) / n
    X, Y, Z = np.meshgrid(x, x, x, indexing='ij')
    r = np.sqrt((X - 0.4) ** 2 + (Y - 0.5) ** 2 + (Z - 0.55) ** 2)
    q = np.zeros((5, n, n, n), order='F')
    q[0] = 1.0 + 0.5 * (r < 0.25)
    q[1] = 0.2 * q[0]
    q[4] = np.where(r < 0.25, 5.0, 0.5) / G1 + 0.5 * q[1] ** 2 / q[0]
    return q


def _run_sc3(rp, q0, params, bc, tfinal, nout, ti='SSP104', dt=None, lim_type=2, arithmetic='strict', shape=None,
             cfl=(0.8, 0.9), dt_initial=0.01, dq_src=None, aux=None, limiters=None):
    import pyclaw
    meqn = q0.shape[0]
    mx, my, mz = q0.shape[1:]
    solver = pyclaw.SharpClawSolver3D()
    solver.rp = rp
    solver.arithmetic = arithmetic
    solver.time_integrator = ti
    solver.lim_type = lim_type
    solver.mwaves = rp.nwaves(3)
    if limiters is not None:
        solver.limiters = limiters
    solver.cfl_desired, solver.cfl_max = cfl
    solver.dq_src = dq_src
    if dt is not None:
        solver.dt_variable, solver.dt_initial = False, dt
    else:
        solver.dt_initial = dt_initial
    for i in range(3):
        solver.bc_lower[i] = solver.bc_upper[i] = bc
        solver.aux_bc_lower[i] = solver.aux_bc_upper[i] = bc
    L = shape or (1.0, 1.0, 1.0)
    grid = pyclaw.Grid([pyclaw.Dimension('x', 0.0, L[0], mx), pyclaw.Dimension('y', 0.0, L[1], my),
                        pyclaw.Dimension('z', 0.0, L[2], mz)])
    state = pyclaw.State(grid, meqn, 0 if aux is None else aux.shape[0])
    state.aux_global.update(params)
    if aux is not None:
        state.aux = aux
    state.q[...] = q0
    claw = pyclaw.Controller()
    claw.keep_copy, claw.output_format = True, None
    claw.solution, claw.solver = pyclaw.Solution(state), solver
    claw.tfinal, claw.nout = tfinal, nout
    claw.run()
    return claw


@pytest.mark.parametrize("ti", ["SSP33", "SSP104"])
def test_euler_run_vs_oracle_driver(ti):
    """Variable dt with a rejected first step (dt_initial far above the Courant limit): the run through
    import pyclaw equals the oracle driver bit for bit, frames, step counts and rejections."""
    import pyclaw
    from oracle import pyclaw_oracle as po
    n = 14
    q0 = _blast(n)
    claw = _run_sc3(pyclaw.riemann.euler_3d, q0, dict(gamma=G, gamma1=G1), pyclaw.BC.reflecting, 0.06, 2, ti=ti,
                    dt_initial=0.2)
    s = o3.sharpclaw3d_solver(o3.RP_EULER3D, [G, G1], 3)
    s.time_integrator = ti
    s.cfl_desired, s.cfl_max = 0.8, 0.9
    s.dt_initial = 0.2
    s.bc_lower = s.bc_upper = [po.BC_REFLECTING] * 3
    frames = s.run(q0, None, [1.0 / n] * 3, 0.06, 2)
    assert s.total["rejected"] >= 1 and s.total["numsteps"] >= 4
    for fg, fo in zip(claw.frames, frames):
        assert np.array_equal(np.asarray(fg.q), fo)
    assert np.abs(frames[-1] - q0).max() > 0.05


def _user_acoustics3d():
    import pyclaw
    hdr = os.path.join(ROOT, "examples", "user_rp", "rp_acoustics3d_user.cuh")
    return pyclaw.riemann.from_header(hdr, meqn=4, mwaves=2, maux=2, ndims=(3,))


def test_user_header_equals_builtin_and_oracle():
    """vc-acoustics from the user header equals the built-in vc_acoustics_3d in a SharpClaw 3-D run, and
    both equal the oracle driver."""
    import pyclaw
    from oracle import pyclaw_oracle as po
    n = 12
    x = (np.arange(n) + 0.5) / n
    X, Y, Z = np.meshgrid(x, x, x, indexing='ij')
    r = np.sqrt((X - 0.3) ** 2 + (Y - 0.5) ** 2 + (Z - 0.5) ** 2)
    q0 = np.zeros((4, n, n, n), order='F')
    q0[0] = np.exp(-40 * r * r)
    aux = np.asfortranarray(np.stack([np.where(X < 0.5, 1.0, 3.0), np.where(X < 0.5, 1.0, 0.5)]))
    res = [np.asarray(_run_sc3(rp, q0, {}, pyclaw.BC.periodic, 0.1, 1, aux=aux).frames[-1].q)
           for rp in (pyclaw.riemann.vc_acoustics_3d, _user_acoustics3d())]
    assert np.array_equal(res[0], res[1])
    s = o3.sharpclaw3d_solver(o3.RP_ACOUSTICS3D_VC, [], 2)
    s.cfl_desired, s.cfl_max = 0.8, 0.9
    s.dt_initial = 0.01
    s.bc_lower = s.bc_upper = s.aux_bc_lower = s.aux_bc_upper = [po.BC_PERIODIC] * 3
    assert np.array_equal(s.run(q0, aux, [1.0 / n] * 3, 0.1, 1)[-1], res[0])
    assert np.abs(res[0] - q0).max() > 1e-2


def test_sod_against_sharpclaw1d():
    """A Sod tube along x, y and z with euler_3d agrees with SharpClawSolver1D + euler_with_efix to 1e-12
    relative (fixed dt, so that round-off in the transverse directions cannot move the time step; measured on a
    B200: 0 along each axis)."""
    import pyclaw
    n, dt, nsteps = 48, 2.0 ** -9, 12
    solver = pyclaw.SharpClawSolver1D()
    solver.rp = pyclaw.riemann.euler_with_efix
    solver.mwaves = 3
    solver.dt_variable, solver.dt_initial = False, dt
    solver.bc_lower[0] = solver.bc_upper[0] = pyclaw.BC.outflow
    state = pyclaw.State(pyclaw.Grid(pyclaw.Dimension('x', 0.0, 1.0, n)), 3)
    state.aux_global.update(gamma=G, gamma1=G1)
    x = (np.arange(n) + 0.5) / n
    rho, p = np.where(x < 0.5, 1.0, 0.125), np.where(x < 0.5, 1.0, 0.1)
    state.q[0], state.q[1], state.q[2] = rho, 0.0, p / G1
    claw = pyclaw.Controller()
    claw.keep_copy, claw.output_format = True, None
    claw.solution, claw.solver = pyclaw.Solution(state), solver
    claw.tfinal, claw.nout = nsteps * dt, 1
    claw.run()
    ref = np.asarray(claw.frames[-1].q)
    m = 4
    for axis in range(3):
        shape = [m, m, m]
        shape[axis] = n
        sh = [1, 1, 1]
        sh[axis] = n
        q0 = np.zeros((5,) + tuple(shape), order='F')
        q0[0] = rho.reshape(sh) * np.ones(shape)
        q0[4] = (p / G1).reshape(sh) * np.ones(shape)
        L = tuple(1.0 if a == axis else float(m) / n for a in range(3))
        q = np.asarray(_run_sc3(pyclaw.riemann.euler_3d, q0, dict(gamma=G, gamma1=G1), pyclaw.BC.outflow,
                                nsteps * dt, 1, dt=dt, shape=L, cfl=(2.45, 2.5)).frames[-1].q)
        line = np.moveaxis(q, 1 + axis, 1)[:, :, 1, 2][[0, 1 + axis, 4]]
        err = np.abs(line - ref).max() / np.abs(ref).max()
        print("Sod along axis %d: relative L-inf deviation from SharpClawSolver1D %.3g" % (axis, err))
        assert err <= 1e-12, (axis, err)


def _smooth_euler(n, seed=0):
    x = (np.arange(n) + 0.5) / n
    X, Y, Z = np.meshgrid(x, x, x, indexing='ij')
    ph = np.random.RandomState(seed).uniform(0, 2 * np.pi, 6)
    rho = 1.0 + 0.2 * np.sin(2 * np.pi * X + ph[0]) * np.cos(2 * np.pi * Y + ph[1])
    u = 0.3 * np.sin(2 * np.pi * Y + ph[2])
    v = 0.2 * np.cos(2 * np.pi * Z + ph[3])
    w = 0.25 * np.sin(2 * np.pi * X + ph[4])
    p = 1.0 + 0.1 * np.cos(2 * np.pi * (X + Y + Z) + ph[5])
    return np.asfortranarray(np.stack([rho, rho * u, rho * v, rho * w, p / G1 + 0.5 * rho * (u * u + v * v + w * w)]))


def test_periodic_conservation_and_fma_build():
    """Periodic box, 24 fixed steps: advection and Euler conserve every component to 1e-12 relative.
    The fma build against the strict one on the smooth Euler run: measured 1.1e-13 relative L-inf (B200),
    hence the bound 1e-12."""
    import pyclaw
    n = 16
    q0 = _smooth_euler(n)
    run = lambda ar: np.asarray(_run_sc3(pyclaw.riemann.euler_3d, q0, dict(gamma=G, gamma1=G1), pyclaw.BC.periodic,
                                         24 * 0.01, 1, dt=0.01, arithmetic=ar).frames[-1].q)
    qs = run('strict')
    for m in range(5):
        assert abs(qs[m].sum() - q0[m].sum()) <= 1e-12 * np.abs(q0[m]).sum(), m
    assert np.abs(qs - q0).max() > 1e-2
    qf = run('fma')
    dev = np.abs(qf - qs).max() / np.abs(qs).max()
    print("fma vs strict, smooth Euler 16^3, 24 SSP104 steps: relative L-inf %.3g" % dev)
    assert dev <= 1e-12
    a0 = np.asfortranarray(np.random.RandomState(1).uniform(-1, 1, (1, n, n, n)))
    qa = np.asarray(_run_sc3(pyclaw.riemann.advection_3d, a0, dict(u=0.7, v=-0.45, w=0.3), pyclaw.BC.periodic,
                             24 * 0.01, 1, dt=0.01).frames[-1].q)
    assert abs(qa.sum() - a0.sum()) <= 1e-12 * np.abs(a0).sum()
    assert np.abs(qa - a0).max() > 1e-2


def test_dq_src_unfused_equals_fused():
    """With a dq_src hook the stages run unfused (dq materialised, combined with torch); with a hook that
    adds zero the result equals the fused run."""
    import pyclaw
    import torch
    n = 12
    q0 = _smooth_euler(n, 3)
    calls = []

    def zero_src(solver, state, dt):
        calls.append(dt)
        return torch.zeros_like(state.q)
    kw = dict(ti='SSP104', dt=0.01)
    fused = np.asarray(_run_sc3(pyclaw.riemann.euler_3d, q0, dict(gamma=G, gamma1=G1), pyclaw.BC.periodic, 0.05, 1,
                                **kw).frames[-1].q)
    unfused = np.asarray(_run_sc3(pyclaw.riemann.euler_3d, q0, dict(gamma=G, gamma1=G1), pyclaw.BC.periodic, 0.05,
                                  1, dq_src=zero_src, **kw).frames[-1].q)
    assert len(calls) == 50
    assert np.array_equal(fused, unfused)


def test_lim_types_run():
    """lim_type 3 (hand-written weno5) with Euler; lim_type 1 (tvd2 reads a limiter per COMPONENT, so it
    needs meqn <= mwaves, as in 1-D / 2-D) with advection: both equal the oracle driver bit for bit."""
    import pyclaw
    from oracle import pyclaw_oracle as po
    cases = [(3, pyclaw.riemann.euler_3d, o3.RP_EULER3D, [G, G1], dict(gamma=G, gamma1=G1), _smooth_euler(10, 4), [1]),
             (1, pyclaw.riemann.advection_3d, o3.RP_ADVECTION3D, [0.7, -0.45, 0.3], dict(u=0.7, v=-0.45, w=0.3),
              np.asfortranarray(np.random.RandomState(2).uniform(-1, 1, (1, 10, 10, 10))), [2])]
    for lim_type, rp, rp_id, params, ag, q0, lim in cases:
        claw = _run_sc3(rp, q0, ag, pyclaw.BC.periodic, 0.05, 1, lim_type=lim_type, limiters=lim)
        q = np.asarray(claw.frames[-1].q)
        s = o3.sharpclaw3d_solver(rp_id, params, rp.nwaves(3))
        s.lim_type, s.limiters = lim_type, lim
        s.cfl_desired, s.cfl_max = 0.8, 0.9
        s.dt_initial = 0.01
        s.bc_lower = s.bc_upper = [po.BC_PERIODIC] * 3
        assert np.array_equal(s.run(q0, None, [0.1] * 3, 0.05, 1)[-1], q), lim_type
        assert np.isfinite(q).all() and np.abs(q - q0).max() > 1e-3


# ---- applications -----------------------------------------------------------------------------
def _apps():
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    import apps
    return apps


def test_euler3d_app_sharpclaw():
    c = _apps().euler3d(mx=20, my=18, mz=16, tfinal=0.03, solver_type='sharpclaw')
    q0, q = np.asarray(c.frames[0].q), np.asarray(c.frames[-1].q)
    assert c.frames[-1].t == pytest.approx(0.03) and np.isfinite(q).all()
    p = G1 * (q[4] - 0.5 * (q[1] ** 2 + q[2] ** 2 + q[3] ** 2) / q[0])
    assert q[0].min() > 0 and p.min() > 0
    assert np.abs(q - q0).max() > 0.1


def test_advection3d_app_sharpclaw():
    c = _apps().advection3d(mx=16, my=14, mz=12, tfinal=0.2, solver_type='sharpclaw')
    q0, q = np.asarray(c.frames[0].q), np.asarray(c.frames[-1].q)
    assert np.isfinite(q).all()
    assert abs(q.sum() - q0.sum()) <= 1e-12 * np.abs(q0).sum()
    assert np.abs(q - q0).max() > 0.05


def test_sharpclaw3d_two_ranks_equal_one():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29519", os.path.join(HERE, "mp_sharpclaw3d_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    sys.stdout.write(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


# ---- argument checks --------------------------------------------------------------------------
def test_argument_checks():
    q = np.zeros((5, 14, 14, 14), order="F")
    dq = np.zeros_like(q)
    cfl = ctypes.c_double()
    stage = _lib.load().clawb200_sharpclaw_stage
    stage3 = _lib.load().clawb200_sharpclaw_stage3

    def err(fn, P, *a):
        return fn(ctypes.byref(P), *a)
    nul = ctypes.c_void_p(0)
    buf = ctypes.c_void_p(16)  # never dereferenced: every call below fails its checks first
    for rp_id, meqn, mw, params in ((o3.RP_EULER3D, 5, 3, [G, G1]), (2, 1, 1, [1.0, 0.5]), (1, 4, 2, [1, 1, 1, 1])):
        P = _lib.make_problem(3, meqn, mw, 3, 8, 8, 0.1, 0.1, rp_id, params, [1, 2, 0, 0, 0, 0, 0], [1] * mw)
        rc = err(stage, P, buf, nul, ctypes.c_void_p(32), nul, nul, 0.01, 0, 0.0, 0.0, 1.0, ctypes.c_void_p(64), nul)
        assert rc == ERR_INVALID and b"clawb200_sharpclaw_stage3" in _lib.load().clawb200_last_error()
    P = _lib.make_problem(2, 5, 3, 3, 8, 8, 0.1, 0.1, o3.RP_EULER3D, [G, G1], [1, 2, 0, 0, 0, 0, 0], [1, 1, 1])
    assert err(stage3, P, 8, 0.1, buf, nul, ctypes.c_void_p(32), nul, nul, 0.01, 0, 0.0, 0.0, 1.0,
               ctypes.c_void_p(64), nul) == ERR_INVALID
    P = _lib.make_problem(3, 5, 3, 2, 8, 8, 0.1, 0.1, o3.RP_EULER3D, [G, G1], [1, 2, 0, 0, 0, 0, 0], [1, 1, 1])
    with pytest.raises(_lib.ClawB200Error, match="mbc >= 3"):
        _lib.call("clawb200_sharpclaw_dq3_host", ctypes.byref(P), 8, 0.1, _ptr(q), _ptr(dq), None, 0.01,
                  ctypes.byref(cfl))
    P = _lib.make_problem(3, 5, 3, 3, 8, 8, 0.1, 0.1, o3.RP_EULER3D, [G, G1], [1, 2, 0, 0, 0, 0, 0], [1, 1, 1],
                          weno_variant=_lib.WENO_TABLES)
    assert err(stage3, P, 8, 0.1, buf, nul, ctypes.c_void_p(32), nul, nul, 0.01, 0, 0.0, 0.0, 1.0,
               ctypes.c_void_p(64), nul) == ERR_UNSUPPORTED
    P = _lib.make_problem(3, 5, 3, 3, 8, 8, 0.1, 0.1, o3.RP_EULER3D, [G, G1], [1, 2, 0, 0, 0, 1, 1], [1, 1, 1],
                          maux=1)
    assert err(stage3, P, 8, 0.1, buf, nul, ctypes.c_void_p(32), nul, ctypes.c_void_p(48), 0.01, 0, 0.0, 0.0, 1.0,
               ctypes.c_void_p(64), nul) == ERR_UNSUPPORTED
    P = _lib.make_problem(3, 5, 3, 3, 8, 8, 0.1, 0.1, o3.RP_EULER3D, [G, G1], [1, 2, 0, 0, 0, 0, 0], [1, 1, 1])
    # the x/y partial of dq lives in out or dq_out: qa must be a third buffer
    assert err(stage3, P, 8, 0.1, buf, ctypes.c_void_p(32), ctypes.c_void_p(32), nul, nul, 0.01, 1, 0.5, 0.5, 1.0,
               ctypes.c_void_p(64), nul) == ERR_INVALID
