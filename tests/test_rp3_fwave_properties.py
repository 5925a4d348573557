"""The CPU restatement of the 3-D f-wave transport solver (oracle3d: rpn3 / rpt3 / rptt3 of
vc_advection_fwave_3d, aux = {u, v, w} per cell) against the formulas that define it, and the 3-D
f-wave step (flux3 with the sign(s) lead factor of flux2fw.f) against the 3-D advection solver at
constant velocity, in every method(3) setting and for limiters 0-4."""
import numpy as np
import pytest

import oracle3d as o3

FW = o3.RP_ADVECTION3D_VC_FWAVE
MBC = 2


def _dir(ixyz, icoor):
    return (ixyz - 1 + icoor - 1) % 3 + 1


def fwave_states(n, seed):
    """q and cell velocities of both signs, with blocks where the velocity changes sign across the
    interface, where s = (ul + ur) / 2 is exactly 0 (ur = -ul, and ul = ur = 0) and where ql == qr."""
    rng = np.random.RandomState(seed)
    ql, qr = rng.uniform(-1, 1, (1, n)), rng.uniform(-1, 1, (1, n))
    auxl, auxr = rng.uniform(-2, 2, (3, n)), rng.uniform(-2, 2, (3, n))
    k = n // 8
    auxr[:, k:2 * k] = -auxl[:, k:2 * k]                       # s == 0, fwave != 0
    auxl[:, 2 * k:3 * k] = auxr[:, 2 * k:3 * k] = 0.0           # no motion at all
    auxl[:, 3 * k:4 * k] = np.abs(auxl[:, 3 * k:4 * k])         # sign change across the interface
    auxr[:, 3 * k:4 * k] = -np.abs(auxr[:, 3 * k:4 * k])
    qr[:, 4 * k:5 * k] = ql[:, 4 * k:5 * k]
    return ql, qr, auxl, auxr


def check_normal(solve, ixyz, ql, qr, auxl, auxr):
    """wave == amdq + apdq == fwave == ur*qr - ul*ql bit for bit, s = 0.5*(ul + ur), and the f-wave goes
    whole to the side s points to (half to each side when s == 0)."""
    wave, s, amdq, apdq = solve(ixyz, ql, qr, auxl, auxr)
    d = _dir(ixyz, 1) - 1
    ul, ur = auxl[d], auxr[d]
    fwave = ur * qr[0] - ul * ql[0]
    sp = 0.5 * (ul + ur)
    assert np.array_equal(wave[0, 0], fwave)
    assert np.array_equal(s[0], sp)
    assert np.array_equal(amdq[0] + apdq[0], fwave)
    assert np.array_equal(amdq[0], np.where(sp < 0, fwave, np.where(sp > 0, 0.0, 0.5 * fwave)))
    assert np.array_equal(apdq[0], np.where(sp > 0, fwave, np.where(sp < 0, 0.0, 0.5 * fwave)))


def check_transverse(transverse, ixyz, aux9, asdq):
    """rpt3 splits at the lower / upper edge of the cell asdq enters; rptt3 (impt = 1 / 2) along the
    line one cell down / up in the other transverse direction."""
    for icoor in (2, 3):
        v = aux9[_dir(ixyz, icoor) - 1]
        for impt in (0, 1, 2):
            off = -1 if impt == 1 else 1
            e0 = off if (impt and icoor == 3) else 0
            f0 = off if (impt and icoor == 2) else 0
            de, df = (1, 0) if icoor == 2 else (0, 1)
            line = [v[1 + e0 + k * de, 1 + f0 + k * df] for k in (-1, 0, 1)]
            bm_x = np.minimum(0.5 * (line[0] + line[1]), 0.0) * asdq[0]
            bp_x = np.maximum(0.5 * (line[1] + line[2]), 0.0) * asdq[0]
            for imp in (1, 2):
                bm, bp = transverse(ixyz, icoor, imp, impt, aux9, asdq)
                assert np.array_equal(bm[0], bm_x), (ixyz, icoor, imp, impt)
                assert np.array_equal(bp[0], bp_x), (ixyz, icoor, imp, impt)


def _solve(ixyz, ql, qr, auxl, auxr):
    return o3.rp_point_aux(FW, [], ixyz, 1, ql, qr, auxl, auxr)


def _transverse(ixyz, icoor, imp, impt, aux9, asdq):
    return o3.rp3_transverse_aux(FW, [], ixyz, icoor, imp, impt, aux9, asdq)


@pytest.mark.parametrize("ixyz", [1, 2, 3])
def test_oracle_fwave3_normal_solve(ixyz):
    ql, qr, auxl, auxr = fwave_states(4096, ixyz)
    check_normal(_solve, ixyz, ql, qr, auxl, auxr)
    sp = 0.5 * (auxl + auxr)[ixyz - 1]
    assert (sp > 0).any() and (sp < 0).any() and (sp == 0).sum() >= 1024


@pytest.mark.parametrize("ixyz", [1, 2, 3])
def test_oracle_fwave3_transverse_splits(ixyz):
    rng = np.random.RandomState(10 + ixyz)
    n = 2048
    aux9 = rng.uniform(-2, 2, (3, 3, 3, n))
    asdq = rng.uniform(-1, 1, (1, n))
    check_transverse(_transverse, ixyz, aux9, asdq)


@pytest.mark.parametrize("vel", [(0.7, -0.45, 0.3), (-1.25, 0.5, -0.75), (0.0, 2.0, -0.5)])
def test_oracle_fwave3_constant_velocity_split_is_exact(vel):
    """With the same velocity in every cell, bm + bp == v * asdq in both transverse directions."""
    rng = np.random.RandomState(3)
    n = 1024
    aux9 = np.empty((3, 3, 3, n))
    for ma in range(3):
        aux9[ma] = vel[ma]
    asdq = rng.uniform(-1, 1, (1, n))
    for ixyz in (1, 2, 3):
        for icoor in (2, 3):
            vt = vel[_dir(ixyz, icoor) - 1]
            for imp, impt in ((1, 0), (2, 0), (1, 1), (2, 2)):
                bm, bp = _transverse(ixyz, icoor, imp, impt, aux9, asdq)
                assert np.array_equal(bm + bp, vt * asdq)


# ---- the 3-D f-wave step against advection_3d at constant velocity ------------------------------
SHAPE = (7, 6, 5)
# (method(3), order, limiter): every method(3) setting with limiters 0-4 at second order, and first order
CASES = [(t, 2, lim) for t in (-1, 0, 10, 11, 20, 21, 22) for lim in range(5)] + [(t, 1, 0) for t in (-1, 0, 10, 11)]


def _pad(shape):
    return tuple(n + 2 * MBC for n in shape)


def _const_aux(vel, pad):
    aux = np.empty((3,) + pad, order="F")
    for ma in range(3):
        aux[ma] = vel[ma]
    return aux


def _steps(rp_id, params, q, aux, trans, order, lim, d=(0.1, 0.125, 0.15), dt=0.02):
    mx, my, mz = (n - 2 * MBC for n in q.shape[1:])
    method = [1, order, trans, 0, 0, 0, 3 if aux is not None else 0]
    out = []
    if trans < 0:
        for idir in (1, 2, 3):
            qn = q.copy("F")
            cfl = o3.step3ds(rp_id, params, MBC, mx, my, mz, q, qn, *d, dt, method, [lim], idir, aux=aux)
            out.append((qn, cfl))
    else:
        qn = q.copy("F")
        cfl = o3.step3(rp_id, params, MBC, mx, my, mz, q, qn, *d, dt, method, [lim], aux=aux)
        out.append((qn, cfl))
    return out


@pytest.mark.parametrize("trans,order,lim", CASES)
@pytest.mark.parametrize("vel", [(0.7, -0.45, 0.3), (-0.6, 0.8, -0.35)])
def test_fwave3_step_equals_advection3d_at_constant_velocity(vel, trans, order, lim):
    """u*qr - u*ql and u*(qr - ql) round differently, so the two agree to 1e-13 relative, not bit for bit."""
    pad = _pad(SHAPE)
    rng = np.random.RandomState(lim + 7 * max(trans, 0))
    q = np.asfortranarray(rng.uniform(-1, 1, (1,) + pad))
    fw = _steps(FW, [], q, _const_aux(vel, pad), trans, order, lim)
    ad = _steps(o3.RP_ADVECTION3D, list(vel), q, None, trans, order, lim)
    inner = (slice(None),) + (slice(MBC, -MBC),) * 3
    for (qf, cf), (qa, ca) in zip(fw, ad):
        assert np.abs(qf[inner] - qa[inner]).max() <= 1e-13 * np.abs(qa[inner]).max()
        assert abs(cf - ca) <= 1e-15 * ca and ca > 0.03
        assert np.abs(qa[inner] - q[inner]).max() > 1e-2


def _periodic(qi):
    return np.asfortranarray(np.pad(qi, ((0, 0),) + ((MBC, MBC),) * 3, mode="wrap"))


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_fwave3_one_cell_shift(axis):
    """u = 1 along one axis, dt = dx, dyadic data: one split sweep, and one unsplit step with full
    transverse corrections, are exact one-cell shifts."""
    n = 8
    rng = np.random.RandomState(axis)
    qi = rng.randint(-8, 9, (1, n, n, n)) / 8.0
    q = _periodic(qi)
    vel = [0.0, 0.0, 0.0]
    vel[axis] = 1.0
    aux = _const_aux(vel, q.shape[1:])
    inner = (slice(None),) + (slice(MBC, -MBC),) * 3
    qn = q.copy("F")
    o3.step3ds(FW, [], MBC, n, n, n, q, qn, 1.0 / n, 1.0 / n, 1.0 / n, 1.0 / n, [1, 2, -1, 0, 0, 0, 3], [4],
               axis + 1, aux=aux)
    assert np.array_equal(qn[inner], np.roll(qi, 1, axis=1 + axis))
    qn = q.copy("F")
    o3.step3(FW, [], MBC, n, n, n, q, qn, 1.0 / n, 1.0 / n, 1.0 / n, 1.0 / n, [1, 2, 22, 0, 0, 0, 3], [4], aux=aux)
    assert np.array_equal(qn[inner], np.roll(qi, 1, axis=1 + axis))


def test_fwave3_step_conserves_in_a_periodic_box():
    """A divergent random velocity field: the unsplit f-wave step keeps the sum of q to rounding."""
    n = 8
    rng = np.random.RandomState(5)
    q = _periodic(rng.uniform(0, 1, (1, n, n, n)))
    aux = _periodic(rng.uniform(-1, 1, (3, n, n, n)))
    qn = q.copy("F")
    o3.step3(FW, [], MBC, n, n, n, q, qn, 0.1, 0.1, 0.1, 0.02, [1, 2, 22, 0, 0, 0, 3], [4], aux=aux)
    inner = (slice(None),) + (slice(MBC, -MBC),) * 3
    assert abs(qn[inner].sum() - q[inner].sum()) <= 1e-13 * np.abs(q[inner]).sum()
    assert np.abs(qn[inner] - q[inner]).max() > 1e-3


def test_fwave3_step_needs_aux():
    q = np.zeros((1,) + _pad(SHAPE), order="F")
    with pytest.raises(ValueError):
        o3.step3(FW, [], MBC, *SHAPE, q, q.copy("F"), 0.1, 0.1, 0.1, 0.01, [1, 2, 22, 0, 0, 0, 0], [4])
    with pytest.raises(ValueError):
        o3.step3ds(FW, [], MBC, *SHAPE, q, q.copy("F"), 0.1, 0.1, 0.1, 0.01, [1, 2, -1, 0, 0, 0, 2], [4], 1,
                   aux=np.zeros((2,) + _pad(SHAPE), order="F"))


def test_fwave3_checks_detect_a_wrong_solver():
    """The checks are not vacuous: a speed off by 1e-6, an f-wave split by the wrong sign, rpt3 in the
    wrong direction and rptt3 on the wrong side all fail them."""
    ql, qr, auxl, auxr = fwave_states(512, 9)

    def bad_speed(ixyz, *a):
        w, s, am, ap = _solve(ixyz, *a)
        return w, s + 1e-6, am, ap

    def swapped(ixyz, *a):
        w, s, am, ap = _solve(ixyz, *a)
        return w, s, ap, am
    check_normal(_solve, 1, ql, qr, auxl, auxr)
    for bad in (bad_speed, swapped):
        with pytest.raises(AssertionError):
            check_normal(bad, 1, ql, qr, auxl, auxr)
    rng = np.random.RandomState(1)
    aux9, asdq = rng.uniform(-2, 2, (3, 3, 3, 256)), rng.uniform(-1, 1, (1, 256))
    wrong_dir = lambda ixyz, icoor, imp, impt, a, q: _transverse(ixyz, 5 - icoor, imp, impt, a, q)
    wrong_side = lambda ixyz, icoor, imp, impt, a, q: _transverse(ixyz, icoor, imp, (3 - impt) if impt else 0, a, q)
    for bad in (wrong_dir, wrong_side):
        with pytest.raises(AssertionError):
            check_transverse(bad, 1, aux9, asdq)
