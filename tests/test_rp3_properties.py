"""The CPU restatements of the 3-D Riemann solvers (oracle3d: rpn3 / rpt3 / rptt3 of 3-D advection and
3-D Euler) against the properties that define them (tests/rp_properties.py), in each of the three
sweep directions, and the restated 3-D Euler step against its 1-D anchor (rp1_euler_with_efix in
oracle/).  Neither solver reads aux data, so rptt3 is the same split as rpt3."""
import numpy as np
import pytest

import rp_properties as rpp
import oracle3d as o3
from oracle import pyclaw_oracle as po

G, G1 = rpp.GAMMA, rpp.GAMMA1
EULER = [G, G1]


def euler3_states(n, seed):
    """Random states with jumps in every component (positive density and pressure), a block of
    identical states, a block at rest and a transonic rarefaction in x (entropy fix active)."""
    rng = np.random.RandomState(seed)

    def one():
        rho = rng.uniform(0.1, 3.0, n)
        u = rng.uniform(-3.0, 3.0, (3, n))
        p = rng.uniform(0.1, 4.0, n)
        return np.vstack([rho, rho * u, p / G1 + 0.5 * rho * (u * u).sum(0)])
    ql, qr = one(), one()
    k = n // 8
    qr[:, :k] = ql[:, :k]
    ql[1:4, k:2 * k] = 0.0
    qr[1:4, k:2 * k] = 0.0
    sl = slice(2 * k, 3 * k)
    c = np.sqrt(G)
    for q, un in ((ql, 0.5 * c), (qr, 1.8 * c)):
        q[0, sl], q[1:4, sl] = 1.0, 0.0
        q[1, sl] = un
        q[4, sl] = 1.0 / G1 + 0.5 * un * un
    return ql, qr, sl


def euler3_flux(q, d):
    rho, mom, e = q[0], q[1:4], q[4]
    u = mom / rho
    p = G1 * (e - 0.5 * rho * (u * u).sum(0))
    un = u[d - 1]
    f = np.vstack([rho * un, mom * un, (e + p) * un])
    f[d] += p
    return f


def euler3_roe(ql, qr):
    sl, sr = np.sqrt(ql[0]), np.sqrt(qr[0])
    pl = G1 * (ql[4] - 0.5 * (ql[1:4] ** 2).sum(0) / ql[0])
    pr = G1 * (qr[4] - 0.5 * (qr[1:4] ** 2).sum(0) / qr[0])
    u = (ql[1:4] / sl + qr[1:4] / sr) / (sl + sr)
    H = ((ql[4] + pl) / sl + (qr[4] + pr) / sr) / (sl + sr)
    return u, H


def euler3_jacobian(u, H, d):
    """d f_d / d q of the 3-D Euler equations, shape [n, 5, 5]."""
    n = u.shape[1]
    q2 = (u * u).sum(0)
    A = np.zeros((n, 5, 5))
    a = d                      # the momentum of direction d
    ud = u[d - 1]
    A[:, 0, a] = 1.0
    for k in range(1, 4):
        uk = u[k - 1]
        A[:, k, 0] = -uk * ud
        A[:, k, k] += ud
        A[:, k, a] += uk
    A[:, a, 0] += 0.5 * G1 * q2
    for k in range(1, 4):
        A[:, a, k] -= G1 * u[k - 1]
    A[:, a, 4] = G1
    A[:, 4, 0] = ud * (0.5 * G1 * q2 - H)
    for k in range(1, 4):
        A[:, 4, k] = -G1 * ud * u[k - 1]
    A[:, 4, a] += H
    A[:, 4, 4] = G * ud
    return A


def _dir(ixyz, icoor):
    return (ixyz - 1 + icoor - 1) % 3 + 1


def _check_euler3_normal(solve, ixyz, ql, qr):
    u, H = euler3_roe(ql, qr)
    return rpp.check_normal("euler3", solve, ixyz, ql, qr, euler3_flux, lambda d: euler3_jacobian(u, H, d))


def _check_euler3_transverse(transverse, ixyz, ql, qr, asdq):
    """T and U for rpt3 (= rptt3) in both transverse directions of the sweep ixyz."""
    u, H = euler3_roe(ql, qr)
    a = np.sqrt(G1 * (H - 0.5 * (u * u).sum(0)))
    for icoor in (2, 3):
        d = _dir(ixyz, icoor)
        B = euler3_jacobian(u, H, d)
        Bm, Bp = rpp._split(B, [u[d - 1] - a, u[d - 1], u[d - 1] + a])
        want, wm, wp = (np.einsum('nij,jn->in', X, asdq) for X in (B, Bm, Bp))
        sc = rpp._scale(want)
        bm, bp = transverse(ixyz, icoor, ql, qr, asdq)
        errT = np.abs(bm + bp - want).max() / sc
        assert errT < 1e-10, "euler3 ixyz=%d icoor=%d: bm + bp != B asdq (%g)" % (ixyz, icoor, errT)
        errU = max(np.abs(bm - wm).max(), np.abs(bp - wp).max()) / sc
        assert errU < 1e-8, "euler3 ixyz=%d icoor=%d: wrong split (%g)" % (ixyz, icoor, errU)


def _solve(rp_id, params, mw):
    return lambda ixyz, ql, qr: o3.rp_point(rp_id, params, ixyz, mw, ql, qr)


def _transverse(rp_id, params):
    return lambda ixyz, icoor, ql, qr, asdq: o3.rp3_transverse(rp_id, params, ixyz, icoor, ql, qr, asdq)


@pytest.mark.parametrize("ixyz", [1, 2, 3])
def test_oracle_euler3_satisfies_its_defining_properties(ixyz):
    ql, qr, sl = euler3_states(2048, 11)
    if ixyz != 1:   # the transonic block along the sweep direction
        for q in (ql, qr):
            q[[1, ixyz], sl] = q[[ixyz, 1], sl]
    wave, s, amdq, apdq = _check_euler3_normal(_solve(o3.RP_EULER3D, EULER, 3), ixyz, ql, qr)
    assert np.abs(amdq[0, sl]).min() > 0 and np.abs(apdq[0, sl]).min() > 0   # entropy fix acted
    rng = np.random.RandomState(5 + ixyz)
    _check_euler3_transverse(_transverse(o3.RP_EULER3D, EULER), ixyz, ql, qr, rng.uniform(-1, 1, ql.shape))
    _check_euler3_transverse(_transverse(o3.RP_EULER3D, EULER), ixyz, ql, qr, amdq)


def test_oracle_euler3_reduces_to_the_1d_solver():
    """With v = w = 0 the normal solve is rp1_euler_with_efix on (rho, rho u, E), bit for bit."""
    ql, qr, sl = euler3_states(1024, 3)
    for ixyz in (1, 2, 3):
        l, r = ql.copy(), qr.copy()
        for q in (l, r):
            un = q[1].copy()
            q[1:4] = 0.0
            q[ixyz] = un
        w3, s3, am3, ap3 = o3.rp_point(o3.RP_EULER3D, EULER, ixyz, 3, l, r)
        l1, r1 = l[[0, ixyz, 4]], r[[0, ixyz, 4]]
        w1, s1, am1, ap1 = po.rp_point(po.RP_EULER1D, EULER, 0, 3, l1, r1)
        assert np.array_equal(s3, s1)
        assert np.array_equal(am3[[0, ixyz, 4]], am1) and np.array_equal(ap3[[0, ixyz, 4]], ap1)
        assert np.array_equal(w3[[0, ixyz, 4]], w1)


@pytest.mark.parametrize("uvw", [(0.7, -0.4, 0.25), (-0.3, 0.9, -1.1)])
def test_oracle_advection3_exact_formulas(uvw):
    rng = np.random.RandomState(2)
    n = 512
    ql, qr, asdq = rng.uniform(-1, 1, (1, n)), rng.uniform(-1, 1, (1, n)), rng.uniform(-1, 1, (1, n))
    for ixyz in (1, 2, 3):
        wave, s, amdq, apdq = o3.rp_point(o3.RP_ADVECTION3D, list(uvw), ixyz, 1, ql, qr)
        sp = uvw[ixyz - 1]
        assert np.array_equal(wave[:, 0], qr - ql) and np.all(s == sp)
        assert np.array_equal(amdq, min(sp, 0.0) * (qr - ql)) and np.array_equal(apdq, max(sp, 0.0) * (qr - ql))
        for icoor in (2, 3):
            st = uvw[_dir(ixyz, icoor) - 1]
            bm, bp = o3.rp3_transverse(o3.RP_ADVECTION3D, list(uvw), ixyz, icoor, ql, qr, asdq)
            assert np.array_equal(bm, min(st, 0.0) * asdq) and np.array_equal(bp, max(st, 0.0) * asdq)


def test_euler3_checks_detect_a_wrong_solver():
    """The checks are not vacuous: a wave speed off by 1e-6, or rpt3 splitting in the wrong
    direction, fails them."""
    ql, qr, sl = euler3_states(256, 4)
    good = _solve(o3.RP_EULER3D, EULER, 3)

    def bad_speed(ixyz, l, r):
        w, s, am, ap = good(ixyz, l, r)
        s = s.copy()
        s[2] += 1e-6
        return w, s, am, ap
    _check_euler3_normal(good, 1, ql, qr)
    with pytest.raises(AssertionError):
        _check_euler3_normal(bad_speed, 1, ql, qr)
    tg = _transverse(o3.RP_EULER3D, EULER)
    wrong_dir = lambda ixyz, icoor, l, r, a: tg(ixyz, 5 - icoor, l, r, a)
    asdq = np.random.RandomState(0).uniform(-1, 1, ql.shape)
    with pytest.raises(AssertionError):
        _check_euler3_transverse(wrong_dir, 1, ql, qr, asdq)


def _sod(n, d, mbc):
    """A Sod tube along direction d (0, 1, 2) of an n x 4 x 3 (permuted) box, ghost cells included."""
    shape = [4 + 2 * mbc, 5 + 2 * mbc, 3 + 2 * mbc]
    shape[d] = n + 2 * mbc
    x = (np.arange(shape[d]) - mbc + 0.5) / n
    left = x < 0.5
    rho = np.where(left, 1.0, 0.125)
    p = np.where(left, 1.0, 0.1)
    q = np.zeros((5,) + tuple(shape), order="F")
    sh = [1, 1, 1]
    sh[d] = -1
    q[0] = rho.reshape(sh)
    q[4] = (p / G1).reshape(sh)
    return np.asfortranarray(q)


def test_oracle_euler3_split_sod_equals_the_1d_solver():
    """A Sod tube along x, y and z: the oracle's dimensionally split 3-D step agrees with the 1-D step
    (rp1_euler_with_efix) on the tube to 1e-12 relative over 5 steps (step1.f and step3ds.f sum the
    same increments in a different order)."""
    mbc, n, dt, dx = 2, 40, 0.01, 1.0 / 40
    method = [1, 2, -1, 0, 0, 0, 0]
    lim = [4, 4, 4]
    q1 = np.asfortranarray(_sod(n, 0, mbc)[[0, 1, 4], :, mbc, mbc])
    qs1 = [q1.copy("F")]
    for _ in range(5):
        q = qs1[-1].copy("F")
        q[:, :mbc], q[:, -mbc:] = q[:, mbc:mbc + 1], q[:, -mbc - 1:-mbc]
        po.step1(po.RP_EULER1D, EULER, mbc, n, q, None, dx, dt, [1, 2, 0, 0, 0, 0, 0], lim)
        qs1.append(q)
    for d in range(3):
        q = _sod(n, d, mbc)
        mx, my, mz = (np.array(q.shape[1:]) - 2 * mbc)
        for _ in range(5):
            # outflow ghost cells (zero-order extrapolation) in every direction
            for ax in range(1, 4):
                sl = [slice(None)] * 4
                for g in range(mbc):
                    sl[ax] = g
                    src = list(sl); src[ax] = mbc
                    q[tuple(sl)] = q[tuple(src)]
                    sl[ax] = q.shape[ax] - 1 - g
                    src[ax] = q.shape[ax] - 1 - mbc
                    q[tuple(sl)] = q[tuple(src)]
            for idir in (1, 2, 3):
                qn = q.copy("F")
                o3.step3ds(o3.RP_EULER3D, EULER, mbc, mx, my, mz, q, qn, dx, dx, dx, dt, method, lim, idir)
                q = qn
        line = [slice(None), mbc + 1, mbc + 1, mbc + 1]
        line[1 + d] = slice(mbc, -mbc)
        got = q[tuple(line)][[0, 1 + d, 4]]
        ref = qs1[-1][:, mbc:-mbc]
        assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max(), (d, np.abs(got - ref).max())
        assert np.abs(ref - qs1[0][:, mbc:-mbc]).max() > 0.1
