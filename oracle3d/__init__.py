"""CPU restatement of the 3-D classic steps for the aux-free 3-D solvers -- TEST INFRASTRUCTURE ONLY
(never imported by pyclaw_b200/).  ctypes driver of oracle3d/liboracle3d.so (claw_oracle3d.c), with
the array conventions of oracle/pyclaw_oracle.py: Fortran-ordered q[m, i, j, k]."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

RP_ADVECTION3D, RP_EULER3D = 14, 15  # 3-D advection {u, v, w}; 3-D Euler, Roe + entropy fix {gamma, gamma1}

_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)


def build():
    """Compile oracle3d/liboracle3d.so with the committed Makefile."""
    subprocess.check_call(["make", "-s", "-C", _HERE])


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "liboracle3d.so")
        if not os.path.exists(path):
            build()
        L = ctypes.CDLL(path)
        d, i = ctypes.c_double, ctypes.c_int
        L.oracle3d_step3ds.restype = d
        L.oracle3d_step3ds.argtypes = [i, _dp, i, i, i, i, i, i, _dp, _dp, d, d, d, d, _ip, _ip, i]
        L.oracle3d_step3.restype = d
        L.oracle3d_step3.argtypes = [i, _dp, i, i, i, i, i, i, _dp, _dp, d, d, d, d, _ip, _ip]
        L.oracle3d_rp_point.restype = None
        L.oracle3d_rp_point.argtypes = [i, _dp, i, i, i, ctypes.c_longlong, _dp, _dp, _dp, _dp, _dp, _dp, i, _dp,
                                        _dp, _dp]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(_dp)


def _params(p):
    out = np.zeros(8)
    out[: len(p)] = p
    return out


def _check(cfl):
    if cfl < 0:
        raise ValueError("oracle3d: unsupported solver or capacity function")
    return cfl


def step3ds(rp_id, rp_params, mbc, mx, my, mz, qold, qnew, dx, dy, dz, dt, method, mthlim, idir):
    """classic3.step3ds: one directional sweep (idir = 1, 2, 3); qnew (== qold on entry) updated in place."""
    method = np.ascontiguousarray(method, dtype=np.int32)
    mthlim = np.ascontiguousarray(mthlim, dtype=np.int32)
    assert qold.flags["F_CONTIGUOUS"] and qnew.flags["F_CONTIGUOUS"]
    return _check(lib().oracle3d_step3ds(rp_id, _p(_params(rp_params)), qold.shape[0], len(mthlim), mbc, mx, my, mz,
                                         _p(qold), _p(qnew), dx, dy, dz, dt, method.ctypes.data_as(_ip),
                                         mthlim.ctypes.data_as(_ip), idir))


def step3(rp_id, rp_params, mbc, mx, my, mz, qold, qnew, dx, dy, dz, dt, method, mthlim):
    """classic3.step3 (step3.f + flux3.f with rpt3 / rptt3); qnew (== qold on entry) updated in place."""
    method = np.ascontiguousarray(method, dtype=np.int32)
    mthlim = np.ascontiguousarray(mthlim, dtype=np.int32)
    assert qold.flags["F_CONTIGUOUS"] and qnew.flags["F_CONTIGUOUS"]
    return _check(lib().oracle3d_step3(rp_id, _p(_params(rp_params)), qold.shape[0], len(mthlim), mbc, mx, my, mz,
                                       _p(qold), _p(qnew), dx, dy, dz, dt, method.ctypes.data_as(_ip),
                                       mthlim.ctypes.data_as(_ip)))


def rp_point(rp_id, rp_params, ixyz, mwaves, ql, qr):
    """rpn3 on n interfaces ql | qr ([meqn, n]): (wave[meqn, mwaves, n], s[mwaves, n], amdq, apdq)."""
    ql = np.ascontiguousarray(ql, dtype=np.float64)
    qr = np.ascontiguousarray(qr, dtype=np.float64)
    meqn, n = ql.shape
    wave, s = np.zeros((meqn, mwaves, n)), np.zeros((mwaves, n))
    amdq, apdq = np.zeros((meqn, n)), np.zeros((meqn, n))
    null = ctypes.cast(None, _dp)
    lib().oracle3d_rp_point(rp_id, _p(_params(rp_params)), ixyz, meqn, mwaves, n, _p(ql), _p(qr), _p(wave), _p(s),
                            _p(amdq), _p(apdq), 0, null, null, null)
    return wave, s, amdq, apdq


def rp3_transverse(rp_id, rp_params, ixyz, icoor, ql, qr, asdq):
    """rpt3 (= rptt3 for these solvers, which read no aux data) on n interfaces ql | qr: asdq split in
    direction icoor = 2 | 3 of the sweep ixyz.  Returns (bm, bp)."""
    ql = np.ascontiguousarray(ql, dtype=np.float64)
    qr = np.ascontiguousarray(qr, dtype=np.float64)
    asdq = np.ascontiguousarray(asdq, dtype=np.float64)
    meqn, n = ql.shape
    bm, bp = np.zeros((meqn, n)), np.zeros((meqn, n))
    null = ctypes.cast(None, _dp)
    lib().oracle3d_rp_point(rp_id, _p(_params(rp_params)), ixyz, meqn, 1, n, _p(ql), _p(qr), null, null, null, null,
                            icoor, _p(asdq), _p(bm), _p(bp))
    return bm, bp
