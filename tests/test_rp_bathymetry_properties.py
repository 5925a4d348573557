"""The shallow-water-over-bathymetry f-wave solver (``shallow_bathymetry_fwave``) of the CPU oracle against
the properties that define it, on seeded random states:

  C  sum_p Z_p = amdq + apdq = f(q_r) - f(q_l) + (0, g (h_l + h_r) (b_r - b_l) / 2 [, 0])
     (the bathymetry source is folded into the flux jump)
  L  a lake at rest (u = v = 0, h + b constant) gives fluctuations of round-off size (well balanced)
  D  an interface dry on both sides gives exact zeros; one dry side stays finite
  E  Einfeldt speeds: s1 <= u^ - c^ and s3 >= u^ + c^
  R  the ixy = 2 solve of data with hu and hv swapped is the ixy = 1 solve, bit for bit
  T  the transverse split is B(q^) asdq split into its down- and up-going parts (rp_properties)

The CUDA kernels are held to this oracle bit for bit in tests/test_gpu_bathymetry.py."""
import numpy as np
import pytest

import rp_properties as rpp
import oracle_bathy as ob

G = 9.81
DRY = 1e-3


def _solve(ixy, ql, qr, bl, br, dry=DRY):
    mw = 2 if ixy == 0 else 3
    return ob.rp_point([G, dry], ixy, mw, ql, qr, bl[None], br[None])


def _transverse(ixy, ql, qr, bl, br, imp, asdq):
    return ob.rp_point([G, DRY], ixy, 3, ql, qr, bl[None], br[None], imp, asdq)


def _states(ndim, n, seed):
    rng = np.random.RandomState(seed)

    def one():
        h = rng.uniform(0.1, 3.0, n)
        q = [h, h * rng.uniform(-3.0, 3.0, n)]
        if ndim == 2:
            q.append(h * rng.uniform(-3.0, 3.0, n))
        return np.stack(q)
    ql, qr = one(), one()
    bl, br = rng.uniform(-2.0, 1.0, n), rng.uniform(-2.0, 1.0, n)
    k = n // 8
    qr[:, :k] = ql[:, :k]                 # no jump in q, a step in b
    ql[1:, k:2 * k] = 0.0                 # water at rest on both sides
    qr[1:, k:2 * k] = 0.0
    return ql, qr, bl, br


def _velocity(q, m, dry=DRY):
    return np.where(q[0] > dry, q[m] / np.where(q[0] > dry, q[0], 1.0), 0.0)


def _flux(q, mu, dry=DRY):
    """f in the direction of component mu (1 or 2), with the solver's dry-cell velocity rule."""
    un = _velocity(q, mu, dry)
    f = q * un
    f[0] = q[mu]
    f[mu] = q[mu] * un + 0.5 * G * q[0] * q[0]
    return f


def _roe(ql, qr):
    sl, sr = np.sqrt(np.maximum(ql[0], 0.0)), np.sqrt(np.maximum(qr[0], 0.0))
    u = [(sl * _velocity(ql, m) + sr * _velocity(qr, m)) / (sl + sr) for m in range(1, ql.shape[0])]
    c2 = 0.5 * G * (np.maximum(ql[0], 0.0) + np.maximum(qr[0], 0.0))
    return u, c2


CASES = [(0, 1), (1, 2), (2, 2)]     # (ixy, ndim); ixy = 0: the 1-D solver


@pytest.mark.parametrize("ixy,ndim", CASES)
def test_fluctuations_are_the_flux_jump_plus_the_bathymetry_source(ixy, ndim):
    ql, qr, bl, br = _states(ndim, 4096, 1 + ixy)
    wave, s, amdq, apdq = _solve(ixy, ql, qr, bl, br)
    mu = 2 if ixy == 2 else 1
    want = _flux(qr, mu) - _flux(ql, mu)
    want[mu] += 0.5 * G * (ql[0] + qr[0]) * (br - bl)
    sc = np.abs(want).max(axis=0) + np.abs(_flux(qr, mu)).max(axis=0) + np.abs(_flux(ql, mu)).max(axis=0)
    assert np.all(np.abs(wave.sum(axis=1) - want) <= 1e-12 * sc)
    assert np.all(np.abs(amdq + apdq - want) <= 1e-12 * sc)
    # amdq / apdq are the f-waves sorted by the sign of their speed
    assert np.array_equal(amdq, np.einsum('mwn,wn->mn', wave, (s < 0) + 0.5 * (s == 0)))
    assert np.array_equal(apdq, np.einsum('mwn,wn->mn', wave, (s > 0) + 0.5 * (s == 0)))
    # f-waves are eigenvectors of the Roe matrix: Z_p proportional to (1, s_p, v) for p = 1, 3
    for p in (0, wave.shape[1] - 1):
        assert np.allclose(wave[mu, p], s[p] * wave[0, p], rtol=1e-14, atol=0)


@pytest.mark.parametrize("ixy,ndim", CASES)
def test_lake_at_rest_gives_round_off(ixy, ndim):
    rng = np.random.RandomState(11 + ixy)
    n = 4096
    eta = rng.uniform(-1.0, 2.0)
    hl, hr = rng.uniform(0.01, 3.0, n), rng.uniform(0.01, 3.0, n)
    ql = np.zeros((ndim + 1, n))
    qr = np.zeros((ndim + 1, n))
    ql[0], qr[0] = hl, hr
    bl, br = eta - hl, eta - hr
    wave, s, amdq, apdq = _solve(ixy, ql, qr, bl, br)
    bound = 1e-13 * G * max(hl.max(), hr.max()) ** 2
    assert np.abs(amdq).max() <= bound and np.abs(apdq).max() <= bound
    assert np.abs(wave).max() <= bound
    # a bathymetry source alone (the same data with the bottom made flat) is not at rest
    _, _, am, ap = _solve(ixy, ql, qr, np.zeros(n), np.zeros(n))
    assert np.abs(am).max() > 1.0


@pytest.mark.parametrize("ixy,ndim", CASES)
def test_dry_interfaces(ixy, ndim):
    rng = np.random.RandomState(21 + ixy)
    n = 1024
    ql, qr, bl, br = _states(ndim, n, 31 + ixy)
    # both sides dry: h in [0, dry_tolerance] with arbitrary momentum, including exact zeros
    ld, rd = ql.copy(), qr.copy()
    ld[0] = rng.uniform(0.0, DRY, n)
    rd[0] = rng.uniform(0.0, DRY, n)
    ld[0, :8] = 0.0
    rd[0, 4:12] = 0.0
    rd[0, -4:] = DRY
    wave, s, amdq, apdq = _solve(ixy, ld, rd, bl, br)
    for a in (wave, s, amdq, apdq):
        assert np.array_equal(a, np.zeros_like(a)) and not np.signbit(a).any()
    if ixy:
        bm, bp = _transverse(ixy, ld, rd, bl, br, 1, rng.uniform(-1, 1, ld.shape))
        assert np.array_equal(bm, np.zeros_like(bm)) and np.array_equal(bp, np.zeros_like(bp))
    # one side dry (a shoreline next to a wet cell): finite, and still C
    mu = 2 if ixy == 2 else 1
    for side in (0, 1):
        l, r = ql.copy(), qr.copy()
        (l if side == 0 else r)[0] = rng.uniform(0.0, DRY, n)
        (l if side == 0 else r)[0, :16] = 0.0
        wave, s, amdq, apdq = _solve(ixy, l, r, bl, br)
        for a in (wave, s, amdq, apdq):
            assert np.isfinite(a).all()
        want = _flux(r, mu) - _flux(l, mu)
        want[mu] += 0.5 * G * (l[0] + r[0]) * (br - bl)
        sc = np.abs(want).max(axis=0) + np.abs(_flux(r, mu)).max(axis=0) + np.abs(_flux(l, mu)).max(axis=0)
        assert np.all(np.abs(amdq + apdq - want) <= 1e-12 * sc)


@pytest.mark.parametrize("ixy,ndim", CASES)
def test_einfeldt_speeds_bound_the_roe_speeds(ixy, ndim):
    ql, qr, bl, br = _states(ndim, 4096, 41 + ixy)
    wave, s, amdq, apdq = _solve(ixy, ql, qr, bl, br)
    (u, *rest), c2 = _roe(ql, qr)
    un = rest[0] if ixy == 2 else u
    c = np.sqrt(c2)
    tol = 1e-14 * (np.abs(un) + c)
    assert np.all(s[0] <= un - c + tol) and np.all(s[-1] >= un + c - tol)
    assert np.all(s[0] <= _velocity(ql, 2 if ixy == 2 else 1) - np.sqrt(G * ql[0]) + tol)
    assert np.all(s[-1] >= _velocity(qr, 2 if ixy == 2 else 1) + np.sqrt(G * qr[0]) - tol)
    if ndim == 2:
        assert np.allclose(s[1], un, rtol=1e-15, atol=0)


def test_y_solve_of_swapped_data_is_the_x_solve():
    ql, qr, bl, br = _states(2, 4096, 51)
    sw = [0, 2, 1]
    w1, s1, am1, ap1 = _solve(1, ql, qr, bl, br)
    w2, s2, am2, ap2 = _solve(2, ql[sw], qr[sw], bl, br)
    assert np.array_equal(w2, w1[sw]) and np.array_equal(s2, s1)
    assert np.array_equal(am2, am1[sw]) and np.array_equal(ap2, ap1[sw])
    rng = np.random.RandomState(5)
    asdq = rng.uniform(-1, 1, ql.shape)
    for imp in (1, 2):
        bm1, bp1 = _transverse(1, ql, qr, bl, br, imp, asdq)
        bm2, bp2 = _transverse(2, ql[sw], qr[sw], bl, br, imp, asdq[sw])
        assert np.array_equal(bm2, bm1[sw]) and np.array_equal(bp2, bp1[sw])


@pytest.mark.parametrize("ixy", [1, 2])
def test_transverse_split(ixy):
    ql, qr, bl, br = _states(2, 2048, 61 + ixy)
    (u, v), c2 = _roe(ql, qr)
    jac = lambda d: rpp.shallow_jacobian(u, v, c2, d)
    c = np.sqrt(c2)
    eig = lambda d: [(u if d == 1 else v) - c, (u if d == 1 else v), (u if d == 1 else v) + c]
    transverse = lambda ixy_, l, r, imp, asdq: _transverse(ixy_, l, r, bl, br, imp, asdq)
    rng = np.random.RandomState(71 + ixy)
    rpp.check_transverse("shallow_bathymetry", transverse, ixy, ql, qr, rng.uniform(-1, 1, ql.shape), jac, eig)
    _, _, amdq, apdq = _solve(ixy, ql, qr, bl, br)
    rpp.check_transverse("shallow_bathymetry", transverse, ixy, ql, qr, apdq, jac, eig)


def test_descriptor_and_solver_choice():
    from pyclaw_b200 import riemann
    rs = riemann.shallow_bathymetry_fwave
    assert riemann.resolve("shallow_bathymetry_fwave", {}, 2) is rs
    assert rs.fwave and rs.maux == 1 and rs.ndims == (1, 2)
    assert rs.meqn(1) == rs.nwaves(1) == 2 and rs.meqn(2) == rs.nwaves(2) == 3
    assert rs.params({"grav": 9.81}) == [9.81, 1e-3]
    assert rs.params({"grav": 1.0, "dry_tolerance": 0.0}) == [1.0, 0.0]
    # scripts that set only grav keep the flat-bottom Roe solver
    assert riemann._infer({"grav": 1.0}, 2, False) is riemann.shallow_roe_with_efix
