"""
Kernel-level parity: the CUDA sweeps, called through the C ABI's host-pointer entry
points (the f2py-shaped signatures of include/clawb200.h), against the CPU oracle on the
same seeded inputs.  Everything here is float64 and must agree BIT FOR BIT.
"""
import ctypes

import numpy as np
import pytest

import problems
from oracle import pyclaw_oracle as po
from pyclaw_b200 import _lib

pytestmark = pytest.mark.gpu

RPS = {
    # name: (rp_id, params, meqn(2d), mwaves, limiters)
    "acoustics": (1, [1.0, 4.0, 2.0, 2.0], 3, 2, [4, 4]),
    "advection": (2, [0.7, -0.4], 1, 1, [3]),
    "euler": (3, [1.4, 0.4], 5, 5, [4, 4, 4, 4, 2]),
    "shallow": (4, [1.0], 3, 3, [4, 1, 2]),
}


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _random_padded(rp, mx, my, mbc, seed, smooth=False):
    shape = (mx + 2 * mbc, my + 2 * mbc) if my else (mx + 2 * mbc,)
    q = (problems.smooth_state if smooth else problems.random_state)(rp, shape, seed)
    return q


@pytest.mark.parametrize("rp", ["acoustics", "advection", "euler", "shallow"])
@pytest.mark.parametrize("shape", [(37, 29), (130, 70), (251, 9)])
@pytest.mark.parametrize("order", [1, 2])
def test_step2ds(rp, shape, order):
    rp_id, params, meqn, mwaves, lim = RPS[rp]
    mx, my = shape
    mbc = 2
    dx, dy, dt = 0.01, 0.013, 0.0011
    method = [1, order, -1, 0, 0, 0, 0]
    q = _random_padded(rp, mx, my, mbc, seed=mx + order)
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, method, lim)
    for ids in (1, 2):
        qn_o = q.copy("F")
        cfl_o = po.step2ds(rp_id, params, mbc, mx, my, q, qn_o, None, dx, dy, dt, method, lim, ids)
        qn_g = q.copy("F")
        cfl_g = ctypes.c_double()
        _lib.call("clawb200_step2ds_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), None, dt, ids,
                  ctypes.byref(cfl_g))
        # the GPU sweep updates exactly the cells the Fortran updates
        assert np.array_equal(qn_g, qn_o), (rp, ids, np.abs(qn_g - qn_o).max())
        assert cfl_g.value == cfl_o


@pytest.mark.parametrize("rp", ["acoustics", "advection", "euler", "shallow"])
@pytest.mark.parametrize("shape", [(37, 29), (130, 70), (9, 251)])
@pytest.mark.parametrize("order,trans", [(2, 2), (2, 1), (1, 1), (2, 0)])
@pytest.mark.parametrize("mode", [0, 1])
def test_step2_unsplit(rp, shape, order, trans, mode):
    """mode 0: the single-pass kernel (fused.cuh) for acoustics / advection / shallow water, the
    two sweep kernels for Euler; mode 1: the two sweep kernels for every solver."""
    rp_id, params, meqn, mwaves, lim = RPS[rp]
    mx, my = shape
    mbc = 2
    dx, dy, dt = 0.01, 0.013, 0.0011
    method = [1, order, trans, 0, 0, 0, 0]
    q = _random_padded(rp, mx, my, mbc, seed=my + trans)
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, method, lim)
    P.step2_mode = mode
    qn_o = q.copy("F")
    cfl_o = po.step2(rp_id, params, mbc, mx, my, q, qn_o, None, dx, dy, dt, method, lim)
    qn_g = q.copy("F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), None, dt,
              ctypes.byref(cfl_g))
    # only interior cells are defined output (clawpack.py:555 keeps qbc[:,mbc:-mbc,mbc:-mbc])
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    assert np.array_equal(qn_g[inner], qn_o[inner]), (rp, np.abs(qn_g[inner] - qn_o[inner]).max())
    assert cfl_g.value == cfl_o


def test_step2_mode_2_needs_a_single_pass_kernel():
    """problem.step2_mode = 2 asks for the single-pass kernel: compiled for acoustics, not for Euler."""
    mx, my, mbc = 20, 12, 2
    for rp, ok in (("acoustics", True), ("euler", False)):
        rp_id, params, meqn, mwaves, lim = RPS[rp]
        q = _random_padded(rp, mx, my, mbc, seed=3)
        P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, 0.01, 0.01, rp_id, params, [1, 2, 2, 0, 0, 0, 0], lim)
        P.step2_mode = 2
        qn, cfl = q.copy("F"), ctypes.c_double()
        args = (ctypes.byref(P), _ptr(q), _ptr(qn), None, 0.001, ctypes.byref(cfl))
        if ok:
            _lib.call("clawb200_step2_host", *args)
            assert _lib.load().clawb200_step2_launches(ctypes.byref(P)) == 1 and cfl.value > 0
        else:
            with pytest.raises(_lib.ClawB200Error, match="single-pass"):
                _lib.call("clawb200_step2_host", *args)
    P.step2_mode = 7
    with pytest.raises(_lib.ClawB200Error, match="step2_mode"):
        _lib.call("clawb200_step2_host", *args)


@pytest.mark.parametrize("rp", ["acoustics", "advection"])
@pytest.mark.parametrize("mx", [5, 100, 800, 1001])
@pytest.mark.parametrize("order", [1, 2])
def test_step1(rp, mx, order):
    rp_id, params, _, mwaves, lim = RPS[rp]
    meqn = 2 if rp == "acoustics" else 1
    params = [1.0, 1.0, 1.0, 1.0] if rp == "acoustics" else params
    mbc = 2
    dx, dt = 1.0 / mx, 0.4 / mx
    method = [1, order, 0, 0, 0, 0, 0]
    q = _random_padded(rp, mx, 0, mbc, seed=mx)
    P = _lib.make_problem(1, meqn, mwaves, mbc, mx, 1, dx, 1.0, rp_id, params, method, lim)
    q_o = q.copy("F")
    cfl_o = po.step1(rp_id, params, mbc, mx, q_o, None, dx, dt, method, lim)
    q_g = q.copy("F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_step1_host", ctypes.byref(P), _ptr(q_g), None, dt, ctypes.byref(cfl_g))
    assert np.array_equal(q_g[:, mbc:-mbc], q_o[:, mbc:-mbc])
    assert cfl_g.value == cfl_o


@pytest.mark.parametrize("rp", ["acoustics", "advection", "euler", "shallow"])
@pytest.mark.parametrize("shape", [(37, 29), (130, 70), (9, 140)])
@pytest.mark.parametrize("variant", [0, 1, 2])
def test_sharpclaw_dq2(rp, shape, variant):
    rp_id, params, meqn, mwaves, _ = RPS[rp]
    mx, my = shape
    mbc = 3
    dx, dy, dt = 0.01, 0.013, 0.0011
    q = _random_padded(rp, mx, my, mbc, seed=mx + variant, smooth=True)
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, weno_variant=variant)
    dq_o, cfl_o = po.sc_flux2(rp_id, params, mwaves, mbc, mx, my, q, dx, dy, dt, variant)
    dq_g = np.zeros_like(q, order="F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), None, dt,
              ctypes.byref(cfl_g))
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    assert not np.isnan(dq_o).any()
    assert np.array_equal(dq_g[inner], dq_o[inner]), (rp, np.abs(dq_g[inner] - dq_o[inner]).max())
    assert cfl_g.value == cfl_o


@pytest.mark.parametrize("rp", ["acoustics", "advection"])
@pytest.mark.parametrize("mx", [7, 100, 1001])
@pytest.mark.parametrize("variant", [0, 1, 2])
def test_sharpclaw_dq1(rp, mx, variant):
    rp_id, params, _, mwaves, _ = RPS[rp]
    meqn = 2 if rp == "acoustics" else 1
    params = [1.0, 1.0, 1.0, 1.0] if rp == "acoustics" else params
    mbc = 3
    dx, dt = 1.0 / mx, 0.4 / mx
    q = _random_padded(rp, mx, 0, mbc, seed=mx)
    P = _lib.make_problem(1, meqn, mwaves, mbc, mx, 1, dx, 1.0, rp_id, params, weno_variant=variant)
    dq_o, cfl_o = po.sc_flux1(rp_id, params, mwaves, mbc, mx, q, dx, dt, variant)
    dq_g = np.zeros_like(q, order="F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), None, dt,
              ctypes.byref(cfl_g))
    assert np.array_equal(dq_g[:, mbc:-mbc], dq_o[:, mbc:-mbc])
    assert cfl_g.value == cfl_o


def test_errors_are_reported_not_fatal():
    P = _lib.make_problem(2, 5, 5, 2, 16, 16, 0.1, 0.1, 3, [1.4, 0.4], [1, 2, 2, 0, 0, 1, 1], [4] * 5)
    q = np.zeros((5, 20, 20), order="F")
    cfl = ctypes.c_double()
    with pytest.raises(_lib.ClawB200Error):
        _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(q.copy("F")), None, 0.1,
                  ctypes.byref(cfl))
    P2 = _lib.make_problem(2, 4, 5, 2, 16, 16, 0.1, 0.1, 3, [1.4, 0.4], None, [4] * 5)
    with pytest.raises(_lib.ClawB200Error):
        _lib.call("clawb200_step2_host", ctypes.byref(P2), _ptr(q), _ptr(q.copy("F")), None, 0.1,
                  ctypes.byref(cfl))


def test_f2py_shaped_modules():
    """INTEGRATION.md path B: the f2py call signatures of classic2 / sharpclaw2."""
    from pyclaw_b200 import f2py_shim
    mx, my, mbc = 50, 41, 2
    dx, dy, dt = 0.01, 0.013, 0.0011
    q = _random_padded("euler", mx, my, mbc, seed=11)
    method, lim = [1, 2, 2, 0, 0, 0, 0], [4, 4, 4, 4, 2]
    classic2 = f2py_shim.classic2('euler_5wave')
    classic2.cparam.gamma, classic2.cparam.gamma1 = 1.4, 0.4
    qnew = q.copy('F')
    out, cfl = classic2.step2(max(mx, my), mbc, mx, my, q, qnew, None, dx, dy, dt, method, lim)
    assert out is qnew
    qo = q.copy('F')
    cfl_o = po.step2(3, [1.4, 0.4], mbc, mx, my, q, qo, None, dx, dy, dt, method, lim)
    assert np.array_equal(qnew[:, mbc:-mbc, mbc:-mbc], qo[:, mbc:-mbc, mbc:-mbc]) and cfl == cfl_o
    # dimensional splitting exactly as clawpack.py:538-548 calls it (second call aliased)
    method[2] = -1
    qnew = q.copy('F')
    qq, cx = classic2.step2ds(max(mx, my), mbc, mx, my, q, qnew, None, dx, dy, dt, method, lim, None, None, None, None, 1)
    qq, cy = classic2.step2ds(max(mx, my), mbc, mx, my, qq, qq, None, dx, dy, dt, method, lim, None, None, None, None, 2)
    qo = q.copy('F')
    ox = po.step2ds(3, [1.4, 0.4], mbc, mx, my, q, qo, None, dx, dy, dt, method, lim, 1)
    oy = po.step2ds(3, [1.4, 0.4], mbc, mx, my, qo, qo, None, dx, dy, dt, method, lim, 2)
    assert np.array_equal(qq, qo) and max(cx, cy) == max(ox, oy)
    q3 = _random_padded("shallow", mx, my, 3, seed=2, smooth=True)
    sharpclaw2 = f2py_shim.sharpclaw2('shallow_roe_with_efix')
    sharpclaw2.cparam.grav = 1.0
    dq, cfl = sharpclaw2.flux2(q3, None, dt, 0.0, 3, max(mx, my), mx, my, dx=dx, dy=dy)
    dqo, cflo = po.sc_flux2(4, [1.0], 3, 3, mx, my, q3, dx, dy, dt, 0)
    assert np.array_equal(dq[:, 3:-3, 3:-3], dqo[:, 3:-3, 3:-3]) and cfl == cflo
    with pytest.raises(ValueError):
        classic2.step2(max(mx, my), mbc, mx, my, np.ascontiguousarray(q), qnew, None, dx, dy, dt, method, lim)
    # an aux-dependent solver through the same signatures, and the three aliased classic3 calls
    rng = np.random.RandomState(5)
    pad = (mx + 2 * mbc, my + 2 * mbc)
    qa = _random_padded("acoustics", mx, my, mbc, seed=4)
    aux = np.asfortranarray(np.stack([rng.choice([1.0, 4.0], pad), rng.choice([1.0, 2.0], pad)]))
    vc = f2py_shim.classic2('vc_acoustics')
    m2 = [1, 2, 2, 0, 0, 0, 2]
    qn = qa.copy('F')
    _, cfl = vc.step2(max(mx, my), mbc, mx, my, qa, qn, aux, dx, dy, dt, m2, [4, 4])
    qo = qa.copy('F')
    cfl_o = po.step2(po.RP_VC_ACOUSTICS, [], mbc, mx, my, qa, qo, aux, dx, dy, dt, m2, [4, 4])
    assert np.array_equal(qn[:, mbc:-mbc, mbc:-mbc], qo[:, mbc:-mbc, mbc:-mbc]) and cfl == cfl_o
    mz, dz = 6, 0.02
    pad3 = (mx + 2 * mbc, 9 + 2 * mbc, mz + 2 * mbc)
    q3d = np.asfortranarray(rng.uniform(-1, 1, (4,) + pad3))
    a3d = np.asfortranarray(np.stack([rng.choice([1.0, 2.0], pad3), rng.choice([1.0, 2.0], pad3)]))
    classic3 = f2py_shim.classic3()
    m3 = [1, 2, -1, 0, 0, 0, 2]
    qg, qo = q3d.copy('F'), q3d.copy('F')
    qg, c1 = classic3.step3ds(mx, mbc, mx, 9, mz, q3d, qg, a3d, dx, dy, dz, dt, m3, [4, 4], None, None, None, None, 1)
    qg, c2 = classic3.step3ds(mx, mbc, mx, 9, mz, qg, qg, a3d, dx, dy, dz, dt, m3, [4, 4], None, None, None, None, 2)
    qg, c3 = classic3.step3ds(mx, mbc, mx, 9, mz, qg, qg, a3d, dx, dy, dz, dt, m3, [4, 4], None, None, None, None, 3)
    o = 0.0
    for idir in (1, 2, 3):
        qold = qo.copy('F')
        o = max(o, po.step3ds(po.RP_ACOUSTICS3D_VC, [], mbc, mx, 9, mz, qold, qo, a3d, dx, dy, dz, dt, m3, [4, 4], idir))
    assert np.array_equal(qg, qo) and max(c1, c2, c3) == o


@pytest.mark.parametrize("rp", ["acoustics", "advection", "euler", "shallow"])
@pytest.mark.parametrize("shape", [(37, 29), (130, 70)])
@pytest.mark.parametrize("trans", [-1, 0, 1, 2])
def test_capacity_function(rp, shape, trans):
    """mcapa > 0: dtdx1d = dtdx/capa and the /capa update forms of step2.f:145-152,227-234
    and step2ds.f:152-156,228-232."""
    rp_id, params, meqn, mwaves, lim = RPS[rp]
    mx, my = shape
    mbc = 2
    dx, dy, dt = 0.01, 0.013, 0.0011
    method = [1, 2, trans, 0, 0, 1, 1]
    q = _random_padded(rp, mx, my, mbc, seed=mx + trans)
    rng = np.random.RandomState(7)
    aux = np.asfortranarray(rng.uniform(0.5, 1.5, (1, mx + 2 * mbc, my + 2 * mbc)))
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, method, lim, maux=1)
    cfl_g = ctypes.c_double()
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    if trans < 0:
        for ids in (1, 2):
            qn_o = q.copy("F")
            cfl_o = po.step2ds(rp_id, params, mbc, mx, my, q, qn_o, aux, dx, dy, dt, method, lim, ids)
            qn_g = q.copy("F")
            _lib.call("clawb200_step2ds_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), _ptr(aux), dt, ids,
                      ctypes.byref(cfl_g))
            assert np.array_equal(qn_g, qn_o), (ids, np.abs(qn_g - qn_o).max())
            assert cfl_g.value == cfl_o
    else:
        qn_o = q.copy("F")
        cfl_o = po.step2(rp_id, params, mbc, mx, my, q, qn_o, aux, dx, dy, dt, method, lim)
        qn_g = q.copy("F")
        _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), _ptr(aux), dt,
                  ctypes.byref(cfl_g))
        assert np.array_equal(qn_g[inner], qn_o[inner]), np.abs(qn_g[inner] - qn_o[inner]).max()
        assert cfl_g.value == cfl_o


@pytest.mark.parametrize("shape", [(40, 20), (128, 64)])
def test_shallow_sphere_step(shape):
    """rpn2/rpt2_shallow_sphere + step2qcor on the Rossby-Haurwitz data (16 aux, capa)."""
    mx, my = shape
    mbc = 2
    pb = problems.sphere_problem(mx, my)
    dx, dy = pb["d"]
    aux = pb["auxbc_full"]
    qbc = np.zeros((4, mx + 2 * mbc, my + 2 * mbc), order="F")
    qbc[:, mbc:-mbc, mbc:-mbc] = pb["q"]
    po.fill_bcs(qbc, mbc, [po.BC_PERIODIC, po.BC_CUSTOM], [po.BC_PERIODIC, po.BC_CUSTOM],
                problems.sphere_qbc_lower_y, problems.sphere_qbc_upper_y)
    method, lim = [1, 2, 2, 0, 0, 1, 16], [4, 4, 4]
    dt = 0.4 * dx / 4.0
    qn_o = qbc.copy("F")
    cfl_o = po.step2(po.RP_SPHERE, pb["params"], mbc, mx, my, qbc, qn_o, aux, dx, dy, dt, method, lim)
    P = _lib.make_problem(2, 4, 3, mbc, mx, my, dx, dy, _lib.RP_SPHERE, pb["params"], method, lim, maux=16)
    qn_g = qbc.copy("F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(qbc), _ptr(qn_g), _ptr(aux), dt, ctypes.byref(cfl_g))
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    assert not np.isnan(qn_o).any() and cfl_o > 0
    assert np.array_equal(qn_g[inner], qn_o[inner]), np.abs(qn_g[inner] - qn_o[inner]).max()
    assert cfl_g.value == cfl_o


@pytest.mark.parametrize("rp", ["acoustics", "euler"])
def test_host_slab_pipeline(rp):
    """Tall grids go through the slab pipeline of the host entry points (upload / sweeps /
    download overlapped); results must equal the oracle's single pass bit for bit.  Every slab
    partition, the scratch and the host threads are tested in test_gpu_host_pipeline.py."""
    rp_id, params, meqn, mwaves, lim = RPS[rp]
    mx, my, mbc = 24, 1500, 2
    dx, dy, dt = 0.01, 0.013, 0.0011
    q = _random_padded(rp, mx, my, mbc, seed=3)
    cfl_g = ctypes.c_double()
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    # unsplit
    method = [1, 2, 2, 0, 0, 0, 0]
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, method, lim)
    qn_o = q.copy("F")
    cfl_o = po.step2(rp_id, params, mbc, mx, my, q, qn_o, None, dx, dy, dt, method, lim)
    qn_g = q.copy("F")
    _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), None, dt, ctypes.byref(cfl_g))
    assert np.array_equal(qn_g[inner], qn_o[inner]) and cfl_g.value == cfl_o
    assert np.array_equal(qn_g[:, :, :mbc], q[:, :, :mbc])          # ghost rows untouched
    # dimensional splitting, second call aliased as in clawpack.py:543-544
    method = [1, 2, -1, 0, 0, 0, 0]
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, method, lim)
    qo = q.copy("F")
    ox = po.step2ds(rp_id, params, mbc, mx, my, q, qo, None, dx, dy, dt, method, lim, 1)
    oy = po.step2ds(rp_id, params, mbc, mx, my, qo, qo, None, dx, dy, dt, method, lim, 2)
    qg = q.copy("F")
    cx, cy = ctypes.c_double(), ctypes.c_double()
    _lib.call("clawb200_step2ds_host", ctypes.byref(P), _ptr(q), _ptr(qg), None, dt, 1, ctypes.byref(cx))
    _lib.call("clawb200_step2ds_host", ctypes.byref(P), _ptr(qg), _ptr(qg), None, dt, 2, ctypes.byref(cy))
    assert np.array_equal(qg, qo) and (cx.value, cy.value) == (ox, oy)


@pytest.mark.parametrize("shape", [(1, 1), (2, 3), (4, 4), (125, 64), (126, 65), (124, 63), (250, 128),
                                   (251, 129), (127, 1), (1, 130), (376, 5)])
def test_tile_boundary_shapes(shape):
    """Grid sizes at and around the CTA column tiles (125 / 126 columns) and degenerate grids:
    classic unsplit + dim-split (Euler) and SharpClaw (shallow).  All of them run at 8-row strips;
    the taller strips of large grids are tested in test_gpu_strip_heights.py."""
    mx, my = shape
    dx, dy, dt = 0.01, 0.013, 0.0011
    cfl_g = ctypes.c_double()
    # classic
    mbc = 2
    rp_id, params, meqn, mwaves, lim = RPS["euler"]
    q = _random_padded("euler", mx, my, mbc, seed=mx * 7 + my)
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    method = [1, 2, 2, 0, 0, 0, 0]
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, method, lim)
    qn_o = q.copy("F")
    cfl_o = po.step2(rp_id, params, mbc, mx, my, q, qn_o, None, dx, dy, dt, method, lim)
    qn_g = q.copy("F")
    _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), None, dt, ctypes.byref(cfl_g))
    assert np.array_equal(qn_g[inner], qn_o[inner]) and cfl_g.value == cfl_o
    method = [1, 2, -1, 0, 0, 0, 0]
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, method, lim)
    for ids in (1, 2):
        qn_o = q.copy("F")
        cfl_o = po.step2ds(rp_id, params, mbc, mx, my, q, qn_o, None, dx, dy, dt, method, lim, ids)
        qn_g = q.copy("F")
        _lib.call("clawb200_step2ds_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), None, dt, ids, ctypes.byref(cfl_g))
        assert np.array_equal(qn_g, qn_o) and cfl_g.value == cfl_o
    # sharpclaw
    mbc = 3
    rp_id, params, meqn, mwaves, _ = RPS["shallow"]
    q = _random_padded("shallow", mx, my, mbc, seed=mx + my, smooth=(mx > 3 and my > 3))
    if mx <= 3 or my <= 3:
        q = np.asfortranarray(0.9 + 0.2 * q / np.abs(q).max())   # keep tiny grids admissible
        q[1:] *= 0.1
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, weno_variant=0)
    dq_o, cfl_o = po.sc_flux2(rp_id, params, mwaves, mbc, mx, my, q, dx, dy, dt, 0)
    dq_g = np.zeros_like(q, order="F")
    _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), None, dt, ctypes.byref(cfl_g))
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    assert not np.isnan(dq_o).any()
    assert np.array_equal(dq_g[inner], dq_o[inner]) and cfl_g.value == cfl_o


def test_extreme_magnitudes_take_the_exact_path():
    """Values far outside the fast division / sqrt windows (arith.cuh) must fall back to the
    IEEE operators and still agree bit for bit: acoustics scaled by 1e-290 and 1e+250."""
    rp_id, params, meqn, mwaves, lim = RPS["acoustics"]
    mx, my, mbc = 40, 33, 2
    dx, dy, dt = 0.01, 0.013, 0.0011
    method = [1, 2, 2, 0, 0, 0, 0]
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, method, lim)
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    for scale in (1e-290, 1e-160, 1e250):
        q = np.asfortranarray(_random_padded("acoustics", mx, my, mbc, seed=5) * scale)
        q[:, 10:20, 10:20] = 0.0                      # exact zeros: zero numerators and 0/0 limiter skips
        qn_o = q.copy("F")
        cfl_o = po.step2(rp_id, params, mbc, mx, my, q, qn_o, None, dx, dy, dt, method, lim)
        qn_g = q.copy("F")
        cfl_g = ctypes.c_double()
        _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), None, dt, ctypes.byref(cfl_g))
        assert np.array_equal(qn_g[inner], qn_o[inner], equal_nan=True), scale
        assert cfl_g.value == cfl_o


# ---------------------------------------------------------------------------
# f-wave solvers (classic1fw / classic2fw of the reference: step1fw.f, flux2fw.f)
# ---------------------------------------------------------------------------
def _elastic_data(shape, seed, law, ndim):
    """Strain / momentum and a layered medium; law 1 = linear, 2 = exponential stress."""
    rng = np.random.RandomState(seed)
    meqn = ndim + 1
    q = np.asfortranarray(rng.uniform(-0.3, 0.3, (meqn,) + tuple(shape)))
    q[0] = rng.uniform(0.0, 0.4, shape)
    if ndim == 1:
        aux = np.empty((3,) + tuple(shape), order="F")
        aux[0] = rng.choice([1.0, 4.0], shape)
        aux[1] = rng.choice([1.0, 4.0], shape)
        aux[2] = 0.0
    else:
        aux = np.empty((4,) + tuple(shape), order="F")
        aux[0] = rng.choice([1.0, 4.0], shape)
        aux[1] = rng.choice([1.0, 4.0], shape)
        aux[2] = float(law) if law in (1, 2) else rng.choice([1.0, 2.0], shape)
        aux[3] = q[0] + rng.uniform(-0.01, 0.01, shape)      # the app's stale copy of eps
    return q, aux


def _close(a, b, law):
    if law == 1:
        return np.array_equal(a, b)          # no exp(): bit for bit
    # exp() comes from the CUDA math library on one side and libm on the other (<= 1 ulp each)
    return np.allclose(a, b, rtol=1e-13, atol=1e-15)


@pytest.mark.parametrize("law", [1, 2])
@pytest.mark.parametrize("mx", [6, 130, 1001])
@pytest.mark.parametrize("order,lim", [(1, [0, 0]), (2, [4, 4]), (2, [2, 1])])
def test_step1_fwave_elasticity(law, mx, order, lim):
    mbc = 2
    dx, dt = 1.0 / 6, 0.3 / 6
    method = [1, order, 0, 0, 0, 0, 3]
    q, aux = _elastic_data((mx + 2 * mbc,), seed=mx + law, law=law, ndim=1)
    P = _lib.make_problem(1, 2, 2, mbc, mx, 1, dx, 1.0, po.RP_NEL_FWAVE, [float(law)], method, lim, maux=3)
    q_o = q.copy("F")
    cfl_o = po.step1(po.RP_NEL_FWAVE, [float(law)], mbc, mx, q_o, aux, dx, dt, method, lim)
    q_g = q.copy("F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_step1_host", ctypes.byref(P), _ptr(q_g), _ptr(aux), dt, ctypes.byref(cfl_g))
    assert 0.05 < cfl_o < 2.0 and not np.isnan(q_o).any()
    assert _close(q_g[:, mbc:-mbc], q_o[:, mbc:-mbc], law)
    assert _close(np.array(cfl_g.value), np.array(cfl_o), law)
    # the f-wave correction differs from the wave one: same solver through the wave formula
    # would not reproduce this (guards against silently using |s| instead of sign(s))
    if order == 2:
        q1 = q.copy("F")
        po.step1(po.RP_NEL_FWAVE, [float(law)], mbc, mx, q1, aux, dx, dt, [1, 1, 0, 0, 0, 0, 3], lim)
        assert np.abs(q1 - q_o).max() > 1e-6


@pytest.mark.parametrize("law", [1, 2, 0])
@pytest.mark.parametrize("shape", [(37, 29), (130, 70), (9, 140)])
@pytest.mark.parametrize("order,trans", [(2, 2), (2, 1), (1, 0), (2, -1)])
def test_step2_fwave_psystem(law, shape, order, trans):
    mx, my = shape
    mbc = 2
    dx, dy, dt = 0.05, 0.04, 0.008
    method = [1, order, trans, 0, 0, 0, 4]
    lim = [2, 2]
    q, aux = _elastic_data((mx + 2 * mbc, my + 2 * mbc), seed=mx + trans + law, law=law, ndim=2)
    P = _lib.make_problem(2, 3, 2, mbc, mx, my, dx, dy, po.RP_PSYSTEM, [], method, lim, maux=4)
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    cfl_g = ctypes.c_double()
    if trans >= 0:
        qn_o = q.copy("F")
        cfl_o = po.step2(po.RP_PSYSTEM, [], mbc, mx, my, q, qn_o, aux, dx, dy, dt, method, lim)
        qn_g = q.copy("F")
        _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), _ptr(aux), dt, ctypes.byref(cfl_g))
        assert 0.05 < cfl_o < 2.0 and not np.isnan(qn_o[inner]).any()
        assert _close(qn_g[inner], qn_o[inner], law), np.abs(qn_g[inner] - qn_o[inner]).max()
        assert _close(np.array(cfl_g.value), np.array(cfl_o), law)
    else:
        for ids in (1, 2):
            qn_o = q.copy("F")
            cfl_o = po.step2ds(po.RP_PSYSTEM, [], mbc, mx, my, q, qn_o, aux, dx, dy, dt, method, lim, ids)
            qn_g = q.copy("F")
            _lib.call("clawb200_step2ds_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), _ptr(aux), dt, ids,
                      ctypes.byref(cfl_g))
            assert _close(qn_g, qn_o, law), np.abs(qn_g - qn_o).max()
            assert _close(np.array(cfl_g.value), np.array(cfl_o), law)


def test_fwave_solver_argument_checks():
    mbc, mx = 2, 20
    q, aux = _elastic_data((mx + 2 * mbc,), seed=1, law=1, ndim=1)
    cfl = ctypes.c_double()
    P = _lib.make_problem(1, 2, 2, mbc, mx, 1, 0.1, 1.0, po.RP_NEL_FWAVE, [1.0], [1, 2, 0, 0, 0, 0, 3], [4, 4], maux=3)
    with pytest.raises(_lib.ClawB200Error, match="aux"):
        _lib.call("clawb200_step1_host", ctypes.byref(P), _ptr(q), None, 0.01, ctypes.byref(cfl))
    P = _lib.make_problem(2, 3, 2, mbc, mx, 8, 0.1, 0.1, po.RP_PSYSTEM, [], [1, 2, 2, 0, 0, 0, 3], [4, 4], maux=3)
    q2 = np.zeros((3, mx + 4, 12), order="F")
    a2 = np.ones((3, mx + 4, 12), order="F")
    with pytest.raises(_lib.ClawB200Error, match="aux"):
        _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q2), _ptr(q2.copy("F")), _ptr(a2), 0.01, ctypes.byref(cfl))


@pytest.mark.parametrize("rp", ["acoustics", "advection"])
@pytest.mark.parametrize("mx", [7, 300, 1001])
@pytest.mark.parametrize("order", [1, 2])
def test_step1_capacity_function(rp, mx, order):
    """step1.f:62-73: dtdx(i) = dt / (dx * aux(mcapa, i)); mcapa is the second aux component."""
    rp_id, params, _, mwaves, lim = RPS[rp]
    meqn = 2 if rp == "acoustics" else 1
    params = [1.0, 1.0, 1.0, 1.0] if rp == "acoustics" else params
    mbc = 2
    dx, dt = 1.0 / mx, 0.3 / mx
    method = [1, order, 0, 0, 0, 2, 2]
    q = _random_padded(rp, mx, 0, mbc, seed=mx)
    aux = np.asfortranarray(np.random.RandomState(mx).uniform(0.5, 1.5, (2, mx + 2 * mbc)))
    P = _lib.make_problem(1, meqn, mwaves, mbc, mx, 1, dx, 1.0, rp_id, params, method, lim, maux=2)
    q_o = q.copy("F")
    cfl_o = po.step1(rp_id, params, mbc, mx, q_o, aux, dx, dt, method, lim)
    q_g = q.copy("F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_step1_host", ctypes.byref(P), _ptr(q_g), _ptr(aux), dt, ctypes.byref(cfl_g))
    assert np.array_equal(q_g[:, mbc:-mbc], q_o[:, mbc:-mbc])
    assert cfl_g.value == cfl_o
    # and it is not the uniform-grid result
    q_u = q.copy("F")
    po.step1(rp_id, params, mbc, mx, q_u, None, dx, dt, [1, order, 0, 0, 0, 0, 0], lim)
    assert np.abs(q_u - q_o)[:, mbc:-mbc].max() > 1e-4


@pytest.mark.parametrize("rp", ["acoustics", "advection"])
@pytest.mark.parametrize("variant", [0, 2])
def test_sharpclaw_capacity_function(rp, variant):
    """flux1.f90:59-63: dtdx = dt / (dx(ixy) * aux(mcapa, :)) in both sweep directions."""
    rp_id, params, meqn2, mwaves, _ = RPS[rp]
    mbc = 3
    dt = 0.0011
    rng = np.random.RandomState(11)
    cfl_g = ctypes.c_double()
    # 2-D
    for mx, my in ((37, 29), (130, 70)):
        dx, dy = 0.01, 0.013
        q = _random_padded(rp, mx, my, mbc, seed=mx + variant, smooth=True)
        aux = np.asfortranarray(rng.uniform(0.5, 1.5, (2, mx + 2 * mbc, my + 2 * mbc)))
        method = [1, 2, 0, 0, 0, 2, 2]
        P = _lib.make_problem(2, meqn2, mwaves, mbc, mx, my, dx, dy, rp_id, params, method=method,
                              maux=2, weno_variant=variant)
        dq_o, cfl_o = po.sc_flux2(rp_id, params, mwaves, mbc, mx, my, q, dx, dy, dt, variant, auxbc=aux, mcapa=2)
        dq_g = np.zeros_like(q, order="F")
        _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), _ptr(aux), dt,
                  ctypes.byref(cfl_g))
        inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
        assert np.array_equal(dq_g[inner], dq_o[inner]) and cfl_g.value == cfl_o
        dq_u, _ = po.sc_flux2(rp_id, params, mwaves, mbc, mx, my, q, dx, dy, dt, variant)
        assert np.abs(dq_u - dq_o)[inner].max() > 1e-4
    # 1-D
    meqn = 2 if rp == "acoustics" else 1
    params1 = [1.0, 1.0, 1.0, 1.0] if rp == "acoustics" else params
    for mx in (9, 500):
        dx = 1.0 / mx
        q = _random_padded(rp, mx, 0, mbc, seed=mx, smooth=True)
        aux = np.asfortranarray(rng.uniform(0.5, 1.5, (2, mx + 2 * mbc)))
        P = _lib.make_problem(1, meqn, mwaves, mbc, mx, 1, dx, 1.0, rp_id, params1, method=[1, 2, 0, 0, 0, 1, 2],
                              maux=2, weno_variant=variant)
        dq_o, cfl_o = po.sc_flux1(rp_id, params1, mwaves, mbc, mx, q, dx, dt, variant, auxbc=aux, mcapa=1)
        dq_g = np.zeros_like(q, order="F")
        _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), _ptr(aux), dt,
                  ctypes.byref(cfl_g))
        assert np.array_equal(dq_g[:, mbc:-mbc], dq_o[:, mbc:-mbc]) and cfl_g.value == cfl_o


# ---------------------------------------------------------------------------
# 1-D shallow water (rp1_shallow_roe_with_efix; apps/shallow/1d)
# ---------------------------------------------------------------------------
def _shallow1d_data(mx, mbc, seed, smooth):
    q2 = _random_padded("shallow", mx, 0, mbc, seed=seed, smooth=smooth)   # (3, n): h, hu, hv
    return np.asfortranarray(q2[:2])


@pytest.mark.parametrize("mx", [5, 100, 1001])
@pytest.mark.parametrize("order,lim", [(1, [0, 0]), (2, [4, 4]), (2, [1, 3])])
def test_step1_shallow(mx, order, lim):
    mbc = 2
    dx, dt = 1.0 / mx, 0.1 / mx
    method = [1, order, 0, 0, 0, 0, 0]
    q = _shallow1d_data(mx, mbc, mx, False)
    P = _lib.make_problem(1, 2, 2, mbc, mx, 1, dx, 1.0, 4, [1.0], method, lim)
    q_o = q.copy("F")
    cfl_o = po.step1(4, [1.0], mbc, mx, q_o, None, dx, dt, method, lim)
    q_g = q.copy("F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_step1_host", ctypes.byref(P), _ptr(q_g), None, dt, ctypes.byref(cfl_g))
    assert not np.isnan(q_o).any() and cfl_o > 0.05
    assert np.array_equal(q_g[:, mbc:-mbc], q_o[:, mbc:-mbc])
    assert cfl_g.value == cfl_o


@pytest.mark.parametrize("mx", [9, 500])
@pytest.mark.parametrize("variant", [0, 1, 2])
def test_sharpclaw_dq1_shallow(mx, variant):
    mbc = 3
    dx, dt = 1.0 / mx, 0.1 / mx
    q = _shallow1d_data(mx, mbc, mx + variant, True)
    P = _lib.make_problem(1, 2, 2, mbc, mx, 1, dx, 1.0, 4, [1.0], weno_variant=variant)
    dq_o, cfl_o = po.sc_flux1(4, [1.0], 2, mbc, mx, q, dx, dt, variant)
    dq_g = np.zeros_like(q, order="F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), None, dt, ctypes.byref(cfl_g))
    assert not np.isnan(dq_o).any()
    assert np.array_equal(dq_g[:, mbc:-mbc], dq_o[:, mbc:-mbc]) and cfl_g.value == cfl_o


def test_limiter_id_range():
    """philim.f:19 is a computed GO TO: ids 1..5 select minmod, superbee, van Leer, MC and
    Beam-Warming; any other positive id falls through to minmod."""
    rp_id, params, meqn, mwaves, _ = RPS["acoustics"]
    mx, my, mbc = 60, 21, 2
    dx, dy, dt = 0.01, 0.013, 0.0011
    method = [1, 2, 2, 0, 0, 0, 0]
    q = _random_padded("acoustics", mx, my, mbc, seed=3)
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    out = {}
    for lim in ([5, 3], [9, 23], [1, 1]):
        P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, method, lim)
        qn_o = q.copy("F")
        po.step2(rp_id, params, mbc, mx, my, q, qn_o, None, dx, dy, dt, method, lim)
        qn_g = q.copy("F")
        cfl_g = ctypes.c_double()
        _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), None, dt, ctypes.byref(cfl_g))
        assert np.array_equal(qn_g[inner], qn_o[inner]), lim
        out[tuple(lim)] = qn_g[inner].copy()
    assert np.array_equal(out[(9, 23)], out[(1, 1)])
    assert not np.array_equal(out[(5, 3)], out[(1, 1)])


# ---------------------------------------------------------------------------
# WENO of order 7 .. 17 (weno.f90:104-2425), 1-D, table driven
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("order", [7, 9, 11, 13, 15, 17])
@pytest.mark.parametrize("rp", ["acoustics", "advection", "shallow"])
@pytest.mark.parametrize("literals", ["f32", "f64"])
def test_sharpclaw_high_order_weno(order, rp, literals):
    from pyclaw_b200.weno_tables import tables
    k = (order + 1) // 2
    mbc = k
    rp_id, params, _, mwaves, _ = RPS[rp]
    meqn = {"acoustics": 2, "advection": 1, "shallow": 2}[rp]
    mwaves = {"acoustics": 2, "advection": 1, "shallow": 2}[rp]
    params = [1.0, 1.0, 1.0, 1.0] if rp == "acoustics" else params
    tab = tables(k, literals)
    po.set_weno_tables(tab)
    packed = _lib.pack_weno_tables(tab)   # host table: the *_host entry point uploads it
    for mx in (11, 300):
        dx, dt = 1.0 / mx, 0.1 / mx
        q = _shallow1d_data(mx, mbc, mx + order, True) if rp == "shallow" else \
            _random_padded(rp, mx, 0, mbc, seed=mx + order, smooth=True)
        P = _lib.make_problem(1, meqn, mwaves, mbc, mx, 1, dx, 1.0, rp_id, params, weno_variant=_lib.WENO_TABLES)
        P.weno_k, P.weno_tab = k, packed.ctypes.data
        dq_o, cfl_o = po.sc_flux1(rp_id, params, mwaves, mbc, mx, q, dx, dt, po.WENO_TABLES)
        dq_g = np.zeros_like(q, order="F")
        cfl_g = ctypes.c_double()
        _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), None, dt, ctypes.byref(cfl_g))
        assert not np.isnan(dq_o).any()
        assert np.array_equal(dq_g[:, mbc:-mbc], dq_o[:, mbc:-mbc]), np.abs(dq_g - dq_o)[:, mbc:-mbc].max()
        assert cfl_g.value == cfl_o
    # too few ghost cells for the stencil are refused
    P2 = _lib.make_problem(1, meqn, mwaves, mbc - 1, 20, 1, 0.1, 1.0, rp_id, params, weno_variant=_lib.WENO_TABLES)
    P2.weno_k, P2.weno_tab = k, packed.ctypes.data
    q2 = np.zeros((meqn, 20 + 2 * (mbc - 1)), order="F")
    with pytest.raises(_lib.ClawB200Error, match="mbc"):
        _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P2), _ptr(q2), _ptr(q2.copy("F")), None, 0.01, ctypes.byref(cfl_g))


@pytest.mark.parametrize("order", [7, 11, 17])
@pytest.mark.parametrize("rp", ["acoustics", "advection", "shallow", "euler"])
def test_sharpclaw_high_order_weno_2d(order, rp):
    """flux2.f90 over weno7 .. weno17: 2-D, both sweep directions."""
    from pyclaw_b200.weno_tables import tables
    k = (order + 1) // 2
    mbc = k
    rp_id, params, meqn, mwaves, _ = RPS[rp]
    tab = tables(k, 'f32')
    po.set_weno_tables(tab)
    packed = _lib.pack_weno_tables(tab)   # host table: the *_host entry point uploads it
    cfl_g = ctypes.c_double()
    for mx, my in ((37, 29), (130, 70), (5, 140)):
        dx, dy, dt = 0.01, 0.013, 0.0011
        q = _random_padded(rp, mx, my, mbc, seed=mx + order, smooth=True)
        P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, weno_variant=_lib.WENO_TABLES)
        P.weno_k, P.weno_tab = k, packed.ctypes.data
        dq_o, cfl_o = po.sc_flux2(rp_id, params, mwaves, mbc, mx, my, q, dx, dy, dt, po.WENO_TABLES)
        dq_g = np.zeros_like(q, order="F")
        _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), None, dt, ctypes.byref(cfl_g))
        inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
        assert not np.isnan(dq_o).any()
        assert np.array_equal(dq_g[inner], dq_o[inner]), np.abs(dq_g - dq_o)[inner].max()
        assert cfl_g.value == cfl_o


# ---------------------------------------------------------------------------
# Further solvers of the reference's applications (external sources, parity unpinned):
# variable-coefficient acoustics / colour equation, Burgers, 1-D Euler.
# ---------------------------------------------------------------------------
def _euler1d_data(n, seed, smooth):
    q5 = (problems.smooth_state if smooth else problems.random_state)("euler", (n,), seed)   # rho, mx, my, E, tracer
    rho, mom, e = q5[0], q5[1], q5[3] - 0.5 * q5[2] ** 2 / q5[0]
    return np.asfortranarray(np.stack([rho, mom, e]))


@pytest.mark.parametrize("rp", ["burgers", "color", "euler1d"])
@pytest.mark.parametrize("mx", [7, 300, 1001])
@pytest.mark.parametrize("order,limid", [(1, 0), (2, 4), (2, 2)])
def test_step1_more_solvers(rp, mx, order, limid):
    mbc = 2
    dx, dt = 1.0 / mx, 0.15 / mx
    rng = np.random.RandomState(mx)
    aux, maux = None, 0
    if rp == "burgers":
        rp_id, params, meqn, mwaves = po.RP_BURGERS, [], 1, 1
        q = np.asfortranarray(rng.uniform(-1.0, 1.0, (1, mx + 2 * mbc)))
    elif rp == "color":
        rp_id, params, meqn, mwaves = po.RP_ADVECTION_COLOR, [], 1, 1
        q = np.asfortranarray(rng.uniform(0.0, 1.0, (1, mx + 2 * mbc)))
        aux, maux = np.asfortranarray(rng.uniform(-1.5, 2.5, (1, mx + 2 * mbc))), 1
    else:
        rp_id, params, meqn, mwaves = po.RP_EULER1D, [1.4, 0.4], 3, 3
        q = _euler1d_data(mx + 2 * mbc, mx, False)
    lim = [limid] * mwaves
    method = [1, order, 0, 0, 0, 0, maux]
    P = _lib.make_problem(1, meqn, mwaves, mbc, mx, 1, dx, 1.0, rp_id, params, method, lim, maux=maux)
    q_o = q.copy("F")
    cfl_o = po.step1(rp_id, params, mbc, mx, q_o, aux, dx, dt, method, lim)
    q_g = q.copy("F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_step1_host", ctypes.byref(P), _ptr(q_g), None if aux is None else _ptr(aux), dt,
              ctypes.byref(cfl_g))
    assert not np.isnan(q_o).any() and cfl_o > 0.01
    assert np.array_equal(q_g[:, mbc:-mbc], q_o[:, mbc:-mbc]), np.abs(q_g - q_o)[:, mbc:-mbc].max()
    assert cfl_g.value == cfl_o


@pytest.mark.parametrize("rp", ["burgers", "euler1d"])
@pytest.mark.parametrize("variant", [0, 2])
def test_sharpclaw_dq1_more_solvers(rp, variant):
    mbc = 3
    for mx in (9, 400):
        dx, dt = 1.0 / mx, 0.1 / mx
        if rp == "burgers":
            rp_id, params, meqn, mwaves = po.RP_BURGERS, [], 1, 1
            q = np.asfortranarray(problems.smooth_state("advection", (mx + 2 * mbc,), seed=mx) * 2.0 - 1.0)
        else:
            rp_id, params, meqn, mwaves = po.RP_EULER1D, [1.4, 0.4], 3, 3
            q = _euler1d_data(mx + 2 * mbc, mx, True)
        P = _lib.make_problem(1, meqn, mwaves, mbc, mx, 1, dx, 1.0, rp_id, params, weno_variant=variant)
        dq_o, cfl_o = po.sc_flux1(rp_id, params, mwaves, mbc, mx, q, dx, dt, variant)
        dq_g = np.zeros_like(q, order="F")
        cfl_g = ctypes.c_double()
        _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), None, dt, ctypes.byref(cfl_g))
        assert not np.isnan(dq_o).any()
        assert np.array_equal(dq_g[:, mbc:-mbc], dq_o[:, mbc:-mbc]) and cfl_g.value == cfl_o


@pytest.mark.parametrize("rp", ["vc_acoustics", "vc_advection", "vc_advection_capa"])
@pytest.mark.parametrize("shape", [(37, 29), (130, 70)])
@pytest.mark.parametrize("trans", [-1, 0, 1, 2])
def test_step2_variable_coefficient_solvers(rp, shape, trans):
    mx, my = shape
    mbc = 2
    dx, dy, dt = 0.01, 0.013, 0.0011
    rng = np.random.RandomState(mx + trans)
    pad = (mx + 2 * mbc, my + 2 * mbc)
    mcapa = 0
    if rp == "vc_acoustics":
        rp_id, meqn, mwaves, lim = po.RP_VC_ACOUSTICS, 3, 2, [4, 4]
        q = _random_padded("acoustics", mx, my, mbc, seed=mx)
        aux = np.asfortranarray(np.stack([rng.choice([1.0, 4.0], pad), rng.choice([1.0, 0.5, 2.0], pad)]))
    else:
        rp_id, meqn, mwaves, lim = po.RP_VC_ADVECTION, 1, 1, [4]
        q = _random_padded("advection", mx, my, mbc, seed=mx)
        comps = [rng.uniform(-1.0, 1.5, pad), rng.uniform(-1.2, 0.8, pad)]
        if rp.endswith("capa"):
            comps.append(rng.uniform(0.5, 1.5, pad))
            mcapa = 3
        aux = np.asfortranarray(np.stack(comps))
    maux = aux.shape[0]
    method = [1, 2, trans, 0, 0, mcapa, maux]
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, [], method, lim, maux=maux)
    cfl_g = ctypes.c_double()
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    if trans < 0:
        for ids in (1, 2):
            qn_o = q.copy("F")
            cfl_o = po.step2ds(rp_id, [], mbc, mx, my, q, qn_o, aux, dx, dy, dt, method, lim, ids)
            qn_g = q.copy("F")
            _lib.call("clawb200_step2ds_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), _ptr(aux), dt, ids, ctypes.byref(cfl_g))
            assert np.array_equal(qn_g, qn_o), (ids, np.abs(qn_g - qn_o).max())
            assert cfl_g.value == cfl_o
    else:
        qn_o = q.copy("F")
        cfl_o = po.step2(rp_id, [], mbc, mx, my, q, qn_o, aux, dx, dy, dt, method, lim)
        qn_g = q.copy("F")
        _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(q), _ptr(qn_g), _ptr(aux), dt, ctypes.byref(cfl_g))
        assert np.array_equal(qn_g[inner], qn_o[inner]), np.abs(qn_g[inner] - qn_o[inner]).max()
        assert cfl_g.value == cfl_o and cfl_o > 0.01


@pytest.mark.parametrize("rp", ["nel", "color1d", "psystem", "vc_acoustics", "vc_advection"])
@pytest.mark.parametrize("variant", [0, 2])
def test_sharpclaw_with_aux_dependent_solvers(rp, variant):
    """flux1.f90:128,177-186: the interface solve sees aux(i-1), aux(i), the in-cell solve aux(i)
    on both sides."""
    mbc, dt = 3, 0.0011
    rng = np.random.RandomState(17)
    cfl_g = ctypes.c_double()
    if rp in ("nel", "color1d"):
        for mx in (9, 400):
            dx = 1.0 / mx
            n = mx + 2 * mbc
            if rp == "nel":
                rp_id, params, meqn, mwaves = po.RP_NEL_FWAVE, [1.0], 2, 2
                q, aux = _elastic_data((n,), seed=mx, law=1, ndim=1)
                q = np.asfortranarray(problems.smooth_state("acoustics", (n,), seed=mx) * 0.2)
            else:
                rp_id, params, meqn, mwaves = po.RP_ADVECTION_COLOR, [], 1, 1
                q = problems.smooth_state("advection", (n,), seed=mx)
                aux = np.asfortranarray(rng.uniform(-1.0, 2.0, (1, n)))
            maux = aux.shape[0]
            P = _lib.make_problem(1, meqn, mwaves, mbc, mx, 1, dx, 1.0, rp_id, params, method=[1, 2, 0, 0, 0, 0, maux],
                                  maux=maux, weno_variant=variant)
            dq_o, cfl_o = po.sc_flux1(rp_id, params, mwaves, mbc, mx, q, dx, dt, variant, auxbc=aux, mcapa=0)
            dq_g = np.zeros_like(q, order="F")
            _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), _ptr(aux), dt, ctypes.byref(cfl_g))
            assert not np.isnan(dq_o).any() and np.abs(dq_o).max() > 1e-6
            assert np.array_equal(dq_g[:, mbc:-mbc], dq_o[:, mbc:-mbc]) and cfl_g.value == cfl_o
        return
    for mx, my in ((37, 29), (130, 70)):
        dx, dy = 0.01, 0.013
        pad = (mx + 2 * mbc, my + 2 * mbc)
        if rp == "psystem":
            rp_id, meqn, mwaves = po.RP_PSYSTEM, 3, 2
            _, aux = _elastic_data(pad, seed=mx, law=1, ndim=2)
            q = np.asfortranarray(problems.smooth_state("acoustics", pad, seed=mx) * 0.2)
        elif rp == "vc_acoustics":
            rp_id, meqn, mwaves = po.RP_VC_ACOUSTICS, 3, 2
            q = problems.smooth_state("acoustics", pad, seed=mx)
            aux = np.asfortranarray(np.stack([rng.choice([1.0, 4.0], pad), rng.choice([1.0, 2.0], pad)]))
        else:
            rp_id, meqn, mwaves = po.RP_VC_ADVECTION, 1, 1
            q = problems.smooth_state("advection", pad, seed=mx)
            aux = np.asfortranarray(np.stack([rng.uniform(-1.0, 1.5, pad), rng.uniform(-1.2, 0.8, pad)]))
        maux = aux.shape[0]
        P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, [], method=[1, 2, 0, 0, 0, 0, maux],
                              maux=maux, weno_variant=variant)
        dq_o, cfl_o = po.sc_flux2(rp_id, [], mwaves, mbc, mx, my, q, dx, dy, dt, variant, auxbc=aux, mcapa=0)
        dq_g = np.zeros_like(q, order="F")
        _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), _ptr(aux), dt, ctypes.byref(cfl_g))
        inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
        assert not np.isnan(dq_o).any() and np.abs(dq_o).max() > 1e-6
        assert np.array_equal(dq_g[inner], dq_o[inner]), np.abs(dq_g - dq_o)[inner].max()
        assert cfl_g.value == cfl_o


@pytest.mark.parametrize("ndim", [1, 2, 3])
def test_boundary_fills_match_the_reference_order(ndim):
    """qbc_lower / qbc_upper (solver.py:384-452) for every combination of outflow / periodic /
    reflecting per side, filled dimension by dimension (lower, then upper): corner ghost cells
    depend on that order.  Device kernels vs the numpy restatement, all ghost cells compared."""
    import itertools
    import torch
    rng = np.random.RandomState(ndim)
    mbc = 2
    n = {1: (11,), 2: (7, 5), 3: (5, 4, 6)}[ndim]
    meqn = ndim + 1
    pad = tuple(m + 2 * mbc for m in n)
    q0 = np.asfortranarray(rng.uniform(-1, 1, (meqn,) + pad))
    mz = n[2] if ndim == 3 else 1
    nx, ny = pad[0], (pad[1] if ndim > 1 else 1)
    mstride = int(np.prod(pad))
    P = _lib.make_problem(ndim, meqn, 1, mbc, n[0], n[1] if ndim > 1 else 1, 0.1, 0.1, 2, [1.0, 1.0],
                          pitch=nx, mstride=mstride)
    kinds = [po.BC_OUTFLOW, po.BC_PERIODIC, po.BC_REFLECTING]
    combos = list(itertools.product(kinds, repeat=2))
    for trial in range(12):
        lower = [combos[rng.randint(len(combos))][0] for _ in range(ndim)]
        upper = [combos[rng.randint(len(combos))][1] for _ in range(ndim)]
        ref = q0.copy("F")
        po.fill_bcs(ref, mbc, lower, upper)
        # device layout: [m][k][j][i]
        dev = torch.as_tensor(np.ascontiguousarray(q0.transpose([0] + list(range(ndim, 0, -1)))), device="cuda")
        for idim in range(ndim):
            for side, bcs in ((0, lower), (1, upper)):
                negate = idim + 1 if bcs[idim] == po.BC_REFLECTING else -1
                if ndim == 3:
                    _lib.call("clawb200_bc_fill3", ctypes.byref(P), mz, ctypes.c_void_p(dev.data_ptr()), meqn, idim, side,
                              bcs[idim], negate, None)
                else:
                    _lib.call("clawb200_bc_fill", ctypes.byref(P), ctypes.c_void_p(dev.data_ptr()), meqn, idim, side,
                              bcs[idim], negate, None)
        torch.cuda.synchronize()
        got = dev.cpu().numpy().transpose([0] + list(range(ndim, 0, -1)))
        assert np.array_equal(got, ref), (ndim, lower, upper)


def test_halo_pack_unpack_and_layout_converters():
    """clawb200_halo_pack / unpack (DMDA globalToLocal's replacement for a C caller) and the
    AoS <-> SoA converters of the host entry points."""
    import torch
    rng = np.random.RandomState(4)
    meqn, mx, my, mbc = 3, 37, 21, 2
    nx, ny = mx + 2 * mbc, my + 2 * mbc
    P = _lib.make_problem(2, meqn, 2, mbc, mx, my, 0.1, 0.1, 1, [1.0, 4.0, 2.0, 2.0])
    soa = torch.as_tensor(rng.uniform(-1, 1, (meqn, ny, nx)), device="cuda")
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())
    # rows mbc .. 2 mbc - 1 (what a lower neighbour needs) into a contiguous buffer and back
    buf = torch.zeros((meqn, mbc, nx), dtype=torch.float64, device="cuda")
    _lib.call("clawb200_halo_pack", ctypes.byref(P), ptr(soa), meqn, mbc, mbc, ptr(buf), None)
    assert torch.equal(buf, soa[:, mbc:2 * mbc, :])
    dst = torch.zeros_like(soa)
    _lib.call("clawb200_halo_unpack", ctypes.byref(P), ptr(dst), meqn, ny - mbc, mbc, ptr(buf), None)
    assert torch.equal(dst[:, ny - mbc:, :], soa[:, mbc:2 * mbc, :]) and float(dst[:, :ny - mbc].abs().max()) == 0.0
    # Fortran-ordered q(m, i, j) (component fastest) <-> device [m][j][i]
    host = np.asfortranarray(rng.uniform(-1, 1, (meqn, nx, ny)))
    aos = torch.as_tensor(host.ravel(order="F").copy(), device="cuda")
    out = torch.zeros((meqn, ny, nx), dtype=torch.float64, device="cuda")
    _lib.call("clawb200_aos_to_soa", ptr(aos), ptr(out), meqn, nx, ny, nx * ny, nx, None)
    assert np.array_equal(out.cpu().numpy(), host.transpose(0, 2, 1))
    back = torch.zeros_like(aos)
    _lib.call("clawb200_soa_to_aos", ptr(out), ptr(back), meqn, nx, ny, nx * ny, nx, None)
    assert torch.equal(back, aos)


# ---------------------------------------------------------------------------
# lim_type = 1: second-order TVD reconstruction (reconstruct.f90:568-625, flux1.f90:79-83)
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("rp", ["advection", "euler", "shallow"])
@pytest.mark.parametrize("lim", [1, 2, 3, 4, 5])
def test_sharpclaw_tvd2_dq2(rp, lim):
    rp_id, params, meqn, mwaves, _ = RPS[rp]
    mx, my, mbc = 70, 45, 3
    dx, dy, dt = 0.01, 0.013, 0.0011
    # smooth data without flat patches: with van Leer (3) a zero jump gives r = 0/0 and the
    # reference itself returns NaN there
    q = _random_padded(rp, mx, my, mbc, seed=mx + lim, smooth=True)
    mthlim = [lim] * mwaves
    po.set_tvd_limiters(mthlim)
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, mthlim=mthlim,
                          weno_variant=_lib.RECON_TVD2)
    dq_o, cfl_o = po.sc_flux2(rp_id, params, mwaves, mbc, mx, my, q, dx, dy, dt, po.RECON_TVD2)
    dq_g = np.zeros_like(q, order="F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), None, dt,
              ctypes.byref(cfl_g))
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    assert np.isfinite(dq_o[inner]).all()
    assert np.array_equal(dq_g[inner], dq_o[inner]), (rp, lim, np.abs(dq_g[inner] - dq_o[inner]).max())
    assert cfl_g.value == cfl_o


@pytest.mark.parametrize("lim", [1, 2, 4, 5])
def test_sharpclaw_tvd2_dq1_flat_regions(lim):
    """1-D, data with constant stretches: dqm = 0 gives r = +-Inf or NaN, and gfortran's MIN / MAX
    drop the NaN (the limited slope is multiplied by dqm = 0 afterwards)."""
    rp_id, params, _, mwaves, _ = RPS["acoustics"]
    params = [1.0, 1.0, 1.0, 1.0]
    mx, mbc = 300, 3
    dx, dt = 1.0 / mx, 0.4 / mx
    q = _random_padded("acoustics", mx, 0, mbc, seed=lim)
    q[:, 40:90] = q[:, 40:41]
    q[0, 150:] = 0.25
    mthlim = [lim, lim]
    po.set_tvd_limiters(mthlim)
    P = _lib.make_problem(1, 2, mwaves, mbc, mx, 1, dx, 1.0, rp_id, params, mthlim=mthlim,
                          weno_variant=_lib.RECON_TVD2)
    dq_o, cfl_o = po.sc_flux1(rp_id, params, mwaves, mbc, mx, q, dx, dt, po.RECON_TVD2)
    dq_g = np.zeros_like(q, order="F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g), None, dt,
              ctypes.byref(cfl_g))
    assert np.isfinite(dq_o[:, mbc:-mbc]).all()
    assert np.array_equal(dq_g[:, mbc:-mbc], dq_o[:, mbc:-mbc])
    assert cfl_g.value == cfl_o


# ---------------------------------------------------------------------------
# char_decomp = 1: wave-based WENO5 (reconstruct.f90:393-565, flux1.f90:95-105), 1-D
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("rp", ["acoustics", "advection", "shallow", "burgers", "euler1d", "elastic_fwave"])
@pytest.mark.parametrize("mx", [9, 130, 1001])
def test_sharpclaw_wave_based_weno_dq1(rp, mx):
    mbc = 3
    dx, dt = 1.0 / mx, 0.1 / mx
    aux, maux = None, 0
    variant = _lib.RECON_WENO_WAVE
    rng = np.random.RandomState(mx)
    if rp == "acoustics":
        rp_id, params, meqn, mwaves = 1, [1.0, 1.0, 1.0, 1.0], 2, 2
        q = _random_padded(rp, mx, 0, mbc, seed=mx, smooth=True)
    elif rp == "advection":
        rp_id, params, meqn, mwaves = 2, [0.7, -0.4], 1, 1
        q = _random_padded(rp, mx, 0, mbc, seed=mx, smooth=True)
        q[:, mx // 2:mx // 2 + 9] = q[:, mx // 2:mx // 2 + 1]    # a flat patch: wnorm2 <= 1e-14 branch
    elif rp == "shallow":
        rp_id, params, meqn, mwaves = 4, [1.0], 2, 2
        q = _shallow1d_data(mx, mbc, mx, True)
    elif rp == "burgers":
        rp_id, params, meqn, mwaves = po.RP_BURGERS, [], 1, 1
        q = _random_padded("advection", mx, 0, mbc, seed=mx, smooth=True) - 0.4
    elif rp == "euler1d":
        rp_id, params, meqn, mwaves = po.RP_EULER1D, [1.4, 0.4], 3, 3
        q = _euler1d_data(mx + 2 * mbc, mx, True)
    else:  # the stegoton's f-wave solver with the linear stress law: weno5_fwave
        rp_id, params, meqn, mwaves = po.RP_NEL_FWAVE, [1.0], 2, 2
        variant = _lib.RECON_WENO_FWAVE
        q = np.asfortranarray(0.1 * _random_padded("acoustics", mx, 0, mbc, seed=mx, smooth=True))
        aux, maux = np.asfortranarray(np.stack([rng.uniform(1.0, 4.0, mx + 2 * mbc), rng.uniform(1.0, 4.0, mx + 2 * mbc),
                                                np.zeros(mx + 2 * mbc)])), 3
    method = [1, 2, 0, 0, 0, 0, maux]
    P = _lib.make_problem(1, meqn, mwaves, mbc, mx, 1, dx, 1.0, rp_id, params, method=method, maux=maux,
                          weno_variant=variant)
    dq_o, cfl_o = po.sc_flux1(rp_id, params, mwaves, mbc, mx, q, dx, dt, variant, auxbc=aux)
    dq_g = np.zeros_like(q, order="F")
    cfl_g = ctypes.c_double()
    _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(dq_g),
              _ptr(aux) if aux is not None else None, dt, ctypes.byref(cfl_g))
    assert np.isfinite(dq_o[:, mbc:-mbc]).all()
    assert np.array_equal(dq_g[:, mbc:-mbc], dq_o[:, mbc:-mbc]), np.abs(dq_g - dq_o)[:, mbc:-mbc].max()
    assert cfl_g.value == cfl_o


def test_sharpclaw_wave_based_weno_is_1d_only():
    P = _lib.make_problem(2, 3, 2, 3, 16, 16, 0.1, 0.1, 1, [1.0, 4.0, 2.0, 2.0], weno_variant=_lib.RECON_WENO_WAVE)
    q = np.zeros((3, 22, 22), order="F")
    with pytest.raises(_lib.ClawB200Error, match="1-D only"):
        _lib.call("clawb200_sharpclaw_dq_host", ctypes.byref(P), _ptr(q), _ptr(q.copy("F")), None, 0.01,
                  ctypes.byref(ctypes.c_double()))
