"""The CPU restatement of SharpClaw in 3-D (oracle3d.sc_flux3, DESIGN.md §1) against oracle/:

- every routine oracle3d copies from oracle/claw_oracle.c (the reconstructions weno5_pyweno with f32 and
  f64 literals, weno5_old and tvd2, flux1, rpn3_vc_acoustics) is pinned bit for bit through the existing
  SharpClaw entries of oracle/: oracle3d.sc_flux1 slices against oracle_sc_flux1 (advection, Euler) and,
  accumulated over a 2-D field, against oracle_sc_flux2_capa (vc-acoustics with aux, directions 1 and 2;
  direction 3 is direction 2 with the transverse velocities swapped);
- 1-D anchors: on data that varies along one axis only, sc_flux3 equals oracle.sc_flux1 applied slice by
  slice along that axis, for x, y and z;
- SharpClawSolver3D.setup rejects the variants that are not built in 3-D."""
import numpy as np
import pytest

import oracle3d as o3
from oracle import pyclaw_oracle as po

G, G1 = 1.4, 0.4
VARIANTS = [o3.WENO_PYWENO_F32, o3.WENO_PYWENO_F64, o3.WENO_OLD, o3.RECON_TVD2]


def euler_slice(rng, n, mu):
    """A random 3-D Euler slice with only the normal momentum (component mu) non-zero."""
    rho = rng.uniform(0.5, 2.0, n)
    u = rng.uniform(-1.0, 1.0, n)
    p = rng.uniform(0.5, 2.0, n)
    q = np.zeros((5, n), order="F")
    q[0], q[mu], q[4] = rho, rho * u, p / G1 + 0.5 * rho * u * u
    return q


# ---------------------------------------------------------------------------------------------
# copied routines, bit for bit against oracle/
# ---------------------------------------------------------------------------------------------
def _vc_fields(rng, shape):
    q = np.asfortranarray(rng.uniform(-1, 1, (4,) + shape))
    rho = np.where(rng.rand(*shape) < 0.5, 1.0, 3.0)
    c = np.where(rng.rand(*shape) < 0.5, 1.0, 0.5)
    return q, np.asfortranarray(np.stack([rho * c, c]))


@pytest.mark.parametrize("variant", VARIANTS)
def test_vc_acoustics_xy_slices_equal_oracle_flux2(variant):
    """rpn3_vc_acoustics in directions 1 and 2, the reconstructions and flux1 with aux: oracle3d.sc_flux1
    over the x- and y-slices of a 2-D field, accumulated as flux2.f90 does (the ghost slices add to the ghost
    cells too), equals the 2-D flux2 of oracle/ (oracle_sc_flux2_capa with aux and no capacity function) bit
    for bit, dq and Courant number."""
    rng = np.random.RandomState(20 + variant)
    mbc, mx, my = 3, 23, 17
    q, aux = _vc_fields(rng, (mx + 2 * mbc, my + 2 * mbc))
    lim = [1, 2, 3, 5]
    dx, dy, dt = 0.1, 0.12, 0.03
    po.set_tvd_limiters(lim)
    ref, cfl_ref = po.sc_flux2(po.RP_ACOUSTICS3D_VC, [], 2, mbc, mx, my, q, dx, dy, dt, variant, auxbc=aux, mcapa=0)
    dq = np.zeros_like(q, order="F")
    cfl = 0.0
    for j in range(my + 2):  # Fortran j = 0 .. my+1 at offset j + mbc - 1
        jj = j + mbc - 1
        d1, c1 = o3.sc_flux1(o3.RP_ACOUSTICS3D_VC, [], 2, mbc, mx, q[:, :, jj], dx, dt, 1, variant,
                             aux1d=aux[:, :, jj], mthlim=lim)
        cfl = max(cfl, c1)
        dq[:, mbc:mbc + mx, jj] = dq[:, mbc:mbc + mx, jj] + d1[:, mbc:mbc + mx]
    for i in range(mx + 2):
        ii = i + mbc - 1
        d2, c2 = o3.sc_flux1(o3.RP_ACOUSTICS3D_VC, [], 2, mbc, my, q[:, ii, :], dy, dt, 2, variant,
                             aux1d=aux[:, ii, :], mthlim=lim)
        cfl = max(cfl, c2)
        dq[:, ii, mbc:mbc + my] = dq[:, ii, mbc:mbc + my] + d2[:, mbc:mbc + my]
    assert np.array_equal(dq, ref) and cfl == cfl_ref
    assert np.abs(dq).max() > 0


@pytest.mark.parametrize("variant", VARIANTS)
def test_vc_acoustics_z_slice_is_the_y_slice_with_swapped_velocities(variant):
    """Direction 3 of rpn3_vc_acoustics reads and writes components 0 and 3 where direction 2 uses 0 and 2,
    and the reconstructions are component-wise: a z-slice equals the y-slice with v and w (and their tvd2
    limiters) swapped, bit for bit.  With the test above this pins direction 3 as well."""
    rng = np.random.RandomState(40 + variant)
    mbc, mx = 3, 23
    q, aux = _vc_fields(rng, (mx + 2 * mbc,))
    lim = [1, 2, 3, 5]
    swap = [0, 1, 3, 2]
    d2, c2 = o3.sc_flux1(o3.RP_ACOUSTICS3D_VC, [], 2, mbc, mx, q, 0.1, 0.03, 2, variant, aux1d=aux, mthlim=lim)
    d3, c3 = o3.sc_flux1(o3.RP_ACOUSTICS3D_VC, [], 2, mbc, mx, np.asfortranarray(q[swap]), 0.1, 0.03, 3, variant,
                         aux1d=aux, mthlim=[lim[m] for m in swap])
    assert np.array_equal(d3[swap], d2) and c3 == c2
    assert np.abs(d2[2]).max() > 0


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("ixyz", [1, 2, 3])
def test_advection_slice_equals_oracle(variant, ixyz):
    """3-D advection along ixyz equals rp1_advection of oracle/ (oracle_sc_flux1) with that velocity, bit
    for bit."""
    rng = np.random.RandomState(7 * ixyz + variant)
    mbc, mx = 3, 31
    q = np.asfortranarray(rng.uniform(-1, 1, (1, mx + 2 * mbc)))
    vel = [0.7, -0.45, 0.3]
    dq3, cfl3 = o3.sc_flux1(o3.RP_ADVECTION3D, vel, 1, mbc, mx, q, 0.1, 0.05, ixyz, variant, mthlim=[4])
    po.set_tvd_limiters([4])
    dq1, cfl1 = po.sc_flux1(po.RP_ADVECTION, [vel[ixyz - 1]], 1, mbc, mx, q, 0.1, 0.05, variant)
    assert np.array_equal(dq3, dq1) and cfl3 == cfl1


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("ixyz", [1, 2, 3])
def test_euler_slice_equals_oracle_1d(variant, ixyz):
    """3-D Euler with zero transverse momentum equals rp1_euler_with_efix of oracle/ (oracle_sc_flux1), bit
    for bit."""
    rng = np.random.RandomState(3 * ixyz + variant)
    mbc, mx = 3, 27
    q = euler_slice(rng, mx + 2 * mbc, ixyz)
    lim3 = [2, 1, 1, 1, 3]
    lim3[ixyz] = 4
    dq3, cfl3 = o3.sc_flux1(o3.RP_EULER3D, [G, G1], 3, mbc, mx, q, 0.1, 0.02, ixyz, variant, mthlim=lim3)
    q1 = np.asfortranarray(q[[0, ixyz, 4]])
    po.set_tvd_limiters([2, 4, 3])
    dq1, cfl1 = po.sc_flux1(po.RP_EULER1D, [G, G1], 3, mbc, mx, q1, 0.1, 0.02, variant)
    assert np.array_equal(dq3[[0, ixyz, 4]], dq1) and cfl3 == cfl1
    assert not np.any(np.delete(dq3, [0, ixyz, 4], axis=0))


# ---------------------------------------------------------------------------------------------
# 1-D anchors of sc_flux3
# ---------------------------------------------------------------------------------------------
def _embed(q1d, axis, shape):
    """q1d [meqn, n_axis] broadcast to a 3-D field [meqn, *shape] that varies along `axis` only."""
    view = [1, 1, 1]
    view[axis] = q1d.shape[1]
    q = np.broadcast_to(q1d.reshape((q1d.shape[0],) + tuple(view)), (q1d.shape[0],) + tuple(shape))
    return np.asfortranarray(q)


def _anchor(rp_id, params, mwaves, q1d, rp1_id, params1, comps, axis, variant):
    mbc, n = 3, q1d.shape[1] - 6
    dims = [5, 4, 6]
    dims[axis] = n
    shape = [d + 2 * mbc for d in dims]
    d = [0.1, 0.12, 0.09]
    dt = 0.02
    q = _embed(q1d, axis, shape)
    dq, cfl = o3.sc_flux3(rp_id, params, mwaves, mbc, *dims, q, *d, dt, variant)
    ref, cfl1 = po.sc_flux1(rp1_id, params1, mwaves, mbc, n, np.asfortranarray(q1d[comps]), d[axis], dt, variant)
    sl = [slice(mbc, -mbc)] * 3
    got = np.moveaxis(dq[(slice(None),) + tuple(sl)], axis + 1, 1)  # [meqn, n, a, b]
    exp = ref[:, mbc:-mbc][:, :, None, None]
    err = np.abs(got[comps] - exp).max() / np.abs(exp).max()
    return err, cfl, cfl1


@pytest.mark.parametrize("variant", [o3.WENO_PYWENO_F32, o3.WENO_PYWENO_F64])
@pytest.mark.parametrize("axis", [0, 1, 2])
def test_advection_anchor(variant, axis):
    """Advection with the velocity along one axis: exactly the 1-D dq (measured: 0), same Courant number."""
    rng = np.random.RandomState(axis)
    q1d = np.asfortranarray(rng.uniform(-1, 1, (1, 20 + 6)))
    vel = [0.0, 0.0, 0.0]
    vel[axis] = 0.7
    err, cfl, cfl1 = _anchor(o3.RP_ADVECTION3D, vel, 1, q1d, po.RP_ADVECTION, [0.7], [0], axis, variant)
    assert err == 0.0
    assert cfl == cfl1


@pytest.mark.parametrize("variant", [o3.WENO_PYWENO_F32, o3.WENO_PYWENO_F64])
@pytest.mark.parametrize("axis", [0, 1, 2])
def test_euler_sod_anchor(variant, axis):
    """A Sod tube along one axis (v = w = 0) agrees with the 1-D Euler dq to 1e-12 relative L-inf.  The
    transverse reconstructions of constant data are not exactly constant, so the transverse directions
    could add round-off (measured: 0 with both literal readings)."""
    n = 24
    x = np.arange(n + 6)
    rho = np.where(x < (n + 6) // 2, 1.0, 0.125)
    p = np.where(x < (n + 6) // 2, 1.0, 0.1)
    q1d = np.zeros((5, n + 6), order="F")
    q1d[0], q1d[4] = rho, p / G1
    q1d[axis + 1] = 0.0
    err, _, _ = _anchor(o3.RP_EULER3D, [G, G1], 3, q1d, po.RP_EULER1D, [G, G1], [0, axis + 1, 4], axis, variant)
    assert err <= 1e-12


def test_sc_flux3_rejects_unsupported():
    q = np.asfortranarray(np.ones((1, 8, 8, 8)))
    with pytest.raises(ValueError):
        o3.sc_flux3(o3.RP_ADVECTION3D, [1, 0, 0], 1, 3, 2, 2, 2, q, 1, 1, 1, 0.1, 3)  # weno tables
    with pytest.raises(ValueError):
        o3.sc_flux3(o3.RP_ACOUSTICS3D_VC, [], 2, 3, 2, 2, 2, np.asfortranarray(np.ones((4, 8, 8, 8))), 1, 1, 1, 0.1, 0)


# ---------------------------------------------------------------------------------------------
# SharpClawSolver3D: variants that are not built in 3-D
# ---------------------------------------------------------------------------------------------
def _solution_3d(maux=0):
    import pyclaw
    x, y, z = (pyclaw.Dimension(0.0, 1.0, 6, name=nm) for nm in "xyz")
    s = pyclaw.State(pyclaw.Grid([x, y, z]), 5, maux, device='cpu')
    return pyclaw.Solution(s)


@pytest.mark.parametrize("attr,value", [("weno_order", 7), ("char_decomp", 1), ("mcapa", 0)])
def test_sharpclaw3d_setup_rejects(attr, value):
    import pyclaw
    solver = pyclaw.SharpClawSolver3D()
    solver.rp = pyclaw.riemann.euler_3d
    sol = _solution_3d(maux=1 if attr == "mcapa" else 0)
    if attr == "mcapa":
        sol.state.mcapa = value
    else:
        setattr(solver, attr, value)
    with pytest.raises(NotImplementedError, match="SharpClawSolver3D"):
        solver.setup(sol)


def test_sharpclaw3d_exported():
    import pyclaw
    import petclaw
    assert pyclaw.SharpClawSolver3D is petclaw.SharpClawSolver3D
    assert pyclaw.SharpClawSolver3D().ndim == 3
