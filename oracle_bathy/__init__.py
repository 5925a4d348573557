"""CPU restatement of the classic steps with the shallow-water-over-bathymetry f-wave solver
(``shallow_bathymetry_fwave``) -- TEST INFRASTRUCTURE ONLY (never imported by pyclaw_b200/).  ctypes driver of
oracle_bathy/liboracle_bathy.so (claw_oracle_bathy.c), with the array conventions of oracle/pyclaw_oracle.py:
Fortran-ordered q[m, i(, j)], aux[0] = b.  ``OracleSolver`` is oracle/pyclaw_oracle.py's driver (boundary
conditions, variable dt, rejected steps, outputs) with this library's steps."""
import ctypes
import os
import subprocess

import numpy as np

from oracle import pyclaw_oracle as po

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

RP_SHALLOW_BATHY_FWAVE = 17   # shallow water over bathymetry, f-waves: aux = {b}; params {grav, dry_tolerance}

_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)


def build():
    """Compile oracle_bathy/liboracle_bathy.so with the committed Makefile."""
    subprocess.check_call(["make", "-s", "-C", _HERE])


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "liboracle_bathy.so")
        if not os.path.exists(path):
            build()
        L = ctypes.CDLL(path)
        d, i = ctypes.c_double, ctypes.c_int
        L.oracle_bathy_step1.restype = d
        L.oracle_bathy_step1.argtypes = [_dp, i, i, i, i, i, _dp, _dp, d, d, _ip, _ip]
        L.oracle_bathy_step2ds.restype = d
        L.oracle_bathy_step2ds.argtypes = [_dp, i, i, i, i, i, i, i, _dp, _dp, _dp, d, d, d, _ip, _ip, i]
        L.oracle_bathy_step2.restype = d
        L.oracle_bathy_step2.argtypes = [_dp, i, i, i, i, i, i, i, _dp, _dp, _dp, d, d, d, _ip, _ip]
        L.oracle_bathy_rp_point.restype = None
        L.oracle_bathy_rp_point.argtypes = [_dp, i, i, i, ctypes.c_longlong, _dp, _dp, i, _dp, _dp, _dp, _dp, _dp,
                                            _dp, i, _dp, _dp, _dp]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(_dp)


def _params(p):
    out = np.zeros(8)
    out[: len(p)] = p
    return out


def _ints(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _no_capa(method):
    if method[5] != 0:
        raise ValueError("the bathymetry solver has no capacity-function form")


def rp_point(rp_params, ixy, mwaves, ql, qr, aux_l, aux_r, imp=0, asdq=None):
    """The solver on n independent interfaces: ql, qr [meqn, n] (left / right state), aux_l, aux_r [maux, n].
    Returns (wave[meqn, mwaves, n], s[mwaves, n], amdq, apdq), or (bmasdq, bpasdq) of the transverse solve
    at the Roe averages of the same interfaces when ``asdq`` is given.  ixy = 0: the 1-D solver."""
    c = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    ql, qr, aux_l, aux_r = c(ql), c(qr), c(aux_l), c(aux_r)
    meqn, n = ql.shape
    maux = aux_l.shape[0]
    assert aux_l.shape == aux_r.shape == (maux, n)
    null = ctypes.cast(None, _dp)
    p = _p(_params(rp_params))
    if asdq is None:
        wave, s = np.zeros((meqn, mwaves, n)), np.zeros((mwaves, n))
        amdq, apdq = np.zeros((meqn, n)), np.zeros((meqn, n))
        lib().oracle_bathy_rp_point(p, ixy, meqn, mwaves, n, _p(ql), _p(qr), maux, _p(aux_l), _p(aux_r), _p(wave),
                                    _p(s), _p(amdq), _p(apdq), 0, null, null, null)
        return wave, s, amdq, apdq
    asdq = c(asdq)
    bm, bp = np.zeros((meqn, n)), np.zeros((meqn, n))
    lib().oracle_bathy_rp_point(p, ixy, meqn, mwaves, n, _p(ql), _p(qr), maux, _p(aux_l), _p(aux_r), null, null,
                                null, null, imp, _p(asdq), _p(bm), _p(bp))
    return bm, bp


def step1(rp_params, mbc, mx, qbc, auxbc, dx, dt, method, mthlim):
    """classic1.step1 (with step1fw.f's correction): updates qbc in place, returns cfl."""
    _no_capa(method)
    assert qbc.flags["F_CONTIGUOUS"] and auxbc.flags["F_CONTIGUOUS"]
    mthlim = _ints(mthlim)
    return lib().oracle_bathy_step1(_p(_params(rp_params)), qbc.shape[0], len(mthlim), mbc, auxbc.shape[0], mx,
                                    _p(qbc), _p(auxbc), dx, dt, _ints(method).ctypes.data_as(_ip),
                                    mthlim.ctypes.data_as(_ip))


def step2ds(rp_params, mbc, mx, my, qold, qnew, auxbc, dx, dy, dt, method, mthlim, ids):
    _no_capa(method)
    assert qold.flags["F_CONTIGUOUS"] and qnew.flags["F_CONTIGUOUS"] and auxbc.flags["F_CONTIGUOUS"]
    mthlim = _ints(mthlim)
    return lib().oracle_bathy_step2ds(_p(_params(rp_params)), max(mx, my), qold.shape[0], len(mthlim),
                                      auxbc.shape[0], mbc, mx, my, _p(qold), _p(qnew), _p(auxbc), dx, dy, dt,
                                      _ints(method).ctypes.data_as(_ip), mthlim.ctypes.data_as(_ip), ids)


def step2(rp_params, mbc, mx, my, qold, qnew, auxbc, dx, dy, dt, method, mthlim):
    _no_capa(method)
    assert qold.flags["F_CONTIGUOUS"] and qnew.flags["F_CONTIGUOUS"] and auxbc.flags["F_CONTIGUOUS"]
    mthlim = _ints(mthlim)
    return lib().oracle_bathy_step2(_p(_params(rp_params)), max(mx, my), qold.shape[0], len(mthlim),
                                    auxbc.shape[0], mbc, mx, my, _p(qold), _p(qnew), _p(auxbc), dx, dy, dt,
                                    _ints(method).ctypes.data_as(_ip), mthlim.ctypes.data_as(_ip))


class OracleSolver(po.OracleSolver):
    """The classic 1-D / 2-D solver of oracle/pyclaw_oracle.py (clawpack.py:114-165, 299-324, 510-555) with
    this library's steps: ``OracleSolver(ndim, rp_params)``."""

    def __init__(self, ndim, rp_params):
        super().__init__("classic", ndim, RP_SHALLOW_BATHY_FWAVE, rp_params, ndim + 1)

    def _hyperbolic_classic(self, state):
        self._bcs(state["q"], state["t"])
        mbc = self.mbc
        if self.ndim == 1:
            cfl = step1(self.rp_params, mbc, self.n[0], self.qbc, self.auxbc, self.d[0], self.dt, self.method,
                        self.mthlim)
        else:
            mx, my = self.n
            dx, dy = self.d
            qnew = self.qbc
            qold = qnew.copy("F")
            if self.dim_split:
                cx = step2ds(self.rp_params, mbc, mx, my, qold, qnew, self.auxbc, dx, dy, self.dt, self.method,
                             self.mthlim, 1)
                cy = step2ds(self.rp_params, mbc, mx, my, qnew, qnew, self.auxbc, dx, dy, self.dt, self.method,
                             self.mthlim, 2)
                cfl = max(cx, cy)
            else:
                cfl = step2(self.rp_params, mbc, mx, my, qold, qnew, self.auxbc, dx, dy, self.dt, self.method,
                            self.mthlim)
        self.cfl = cfl
        state["q"] = self.qbc[(slice(None),) + (slice(mbc, -mbc),) * self.ndim].copy("F")
