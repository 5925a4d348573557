"""CPU restatement of the 3-D classic steps for the 3-D solvers other than vc-acoustics and of SharpClaw in
3-D (flux3, sc_flux3) -- TEST INFRASTRUCTURE ONLY (never imported by pyclaw_b200/).  ctypes driver of
oracle3d/liboracle3d.so (claw_oracle3d.c), with the array conventions of oracle/pyclaw_oracle.py:
Fortran-ordered q[m, i, j, k]."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

RP_ADVECTION3D, RP_EULER3D = 14, 15  # 3-D advection {u, v, w}; 3-D Euler, Roe + entropy fix {gamma, gamma1}
RP_ACOUSTICS3D_VC = 8                # 3-D acoustics, aux = {impedance, sound speed} (SharpClaw only here)
RP_ADVECTION3D_VC_FWAVE = 16         # 3-D f-wave transport, aux = {u, v, w} per cell
WENO_PYWENO_F32, WENO_PYWENO_F64, WENO_OLD, RECON_TVD2 = 0, 1, 2, 4  # as oracle/pyclaw_oracle.py

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
        L.oracle3d_step3ds_aux.restype = d
        L.oracle3d_step3ds_aux.argtypes = [i, _dp, i, i, i, i, i, i, _dp, _dp, _dp, i, d, d, d, d, _ip, _ip, i]
        L.oracle3d_step3_aux.restype = d
        L.oracle3d_step3_aux.argtypes = [i, _dp, i, i, i, i, i, i, _dp, _dp, _dp, i, d, d, d, d, _ip, _ip]
        L.oracle3d_rp_point_aux.restype = None
        L.oracle3d_rp_point_aux.argtypes = [i, _dp, i, i, i, i, ctypes.c_longlong, _dp, _dp, _dp, _dp, _dp, _dp, _dp,
                                            _dp, i, i, i, _dp, _dp, _dp, _dp]
        L.oracle3d_sc_flux1.restype = d
        L.oracle3d_sc_flux1.argtypes = [i, _dp, i, i, i, i, i, _dp, _dp, _dp, d, d, i, i, _ip]
        L.oracle3d_sc_flux3.restype = d
        L.oracle3d_sc_flux3.argtypes = [i, _dp, i, i, i, i, i, i, i, _dp, _dp, _dp, d, d, d, d, i, _ip]
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


def _aux(aux):
    """(pointer, maux) of an optional aux array [maux, mx+2mbc, my+2mbc, mz+2mbc] (Fortran order)"""
    if aux is None:
        return ctypes.cast(None, _dp), 0
    assert aux.flags["F_CONTIGUOUS"] and aux.dtype == np.float64
    return _p(aux), aux.shape[0]


def step3ds(rp_id, rp_params, mbc, mx, my, mz, qold, qnew, dx, dy, dz, dt, method, mthlim, idir, aux=None):
    """classic3.step3ds: one directional sweep (idir = 1, 2, 3); qnew (== qold on entry) updated in place.
    aux [maux, ...] (Fortran order, ghost cells filled) for the solvers that read aux data."""
    method = np.ascontiguousarray(method, dtype=np.int32)
    mthlim = np.ascontiguousarray(mthlim, dtype=np.int32)
    assert qold.flags["F_CONTIGUOUS"] and qnew.flags["F_CONTIGUOUS"]
    a, maux = _aux(aux)
    return _check(lib().oracle3d_step3ds_aux(rp_id, _p(_params(rp_params)), qold.shape[0], len(mthlim), mbc, mx, my,
                                             mz, _p(qold), _p(qnew), a, maux, dx, dy, dz, dt,
                                             method.ctypes.data_as(_ip), mthlim.ctypes.data_as(_ip), idir))


def step3(rp_id, rp_params, mbc, mx, my, mz, qold, qnew, dx, dy, dz, dt, method, mthlim, aux=None):
    """classic3.step3 (step3.f + flux3.f with rpt3 / rptt3); qnew (== qold on entry) updated in place.
    aux [maux, ...] (Fortran order, ghost cells filled) for the solvers that read aux data."""
    method = np.ascontiguousarray(method, dtype=np.int32)
    mthlim = np.ascontiguousarray(mthlim, dtype=np.int32)
    assert qold.flags["F_CONTIGUOUS"] and qnew.flags["F_CONTIGUOUS"]
    a, maux = _aux(aux)
    return _check(lib().oracle3d_step3_aux(rp_id, _p(_params(rp_params)), qold.shape[0], len(mthlim), mbc, mx, my, mz,
                                           _p(qold), _p(qnew), a, maux, dx, dy, dz, dt, method.ctypes.data_as(_ip),
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


def rp_point_aux(rp_id, rp_params, ixyz, mwaves, ql, qr, auxl, auxr):
    """rpn3 of a solver with aux data on n interfaces ql | qr ([meqn, n]); auxl / auxr [maux, n] are the
    cells left / right of each interface.  Returns (wave[meqn, mwaves, n], s[mwaves, n], amdq, apdq)."""
    ql, qr = (np.ascontiguousarray(a, dtype=np.float64) for a in (ql, qr))
    auxl, auxr = (np.ascontiguousarray(a, dtype=np.float64) for a in (auxl, auxr))
    meqn, n = ql.shape
    wave, s = np.zeros((meqn, mwaves, n)), np.zeros((mwaves, n))
    amdq, apdq = np.zeros((meqn, n)), np.zeros((meqn, n))
    null = ctypes.cast(None, _dp)
    lib().oracle3d_rp_point_aux(rp_id, _p(_params(rp_params)), ixyz, meqn, mwaves, auxl.shape[0], n, _p(ql), _p(qr),
                                _p(auxl), _p(auxr), _p(wave), _p(s), _p(amdq), _p(apdq), 0, 0, 0, null, null, null, null)
    return wave, s, amdq, apdq


def rp3_transverse_aux(rp_id, rp_params, ixyz, icoor, imp, impt, aux9, asdq):
    """rpt3 (impt = 0) or rptt3 (impt = 1, 2) of a solver with aux data on n fluctuations asdq [meqn, n]
    entering a cell on side imp = 1 | 2 of their interface: aux9 [maux, 3, 3, n] holds the 3x3 cells around
    that cell, [ma, e+1, f+1] at the offset e / f in the y-like / z-like direction.  Returns (bm, bp)."""
    asdq = np.ascontiguousarray(asdq, dtype=np.float64)
    aux9 = np.ascontiguousarray(aux9, dtype=np.float64)
    meqn, n = asdq.shape
    bm, bp = np.zeros((meqn, n)), np.zeros((meqn, n))
    null = ctypes.cast(None, _dp)
    q = np.zeros((meqn, n))
    lib().oracle3d_rp_point_aux(rp_id, _p(_params(rp_params)), ixyz, meqn, 1, aux9.shape[0], n, _p(q), _p(q), null,
                                null, null, null, null, null, icoor, imp, impt, _p(aux9), _p(asdq), _p(bm), _p(bp))
    return bm, bp


def _mthlim8(mthlim, meqn):
    """tvd2 limiter per COMPONENT (reconstruct.f90:568-625): one entry is repeated, as solver.limiters"""
    lim = list(mthlim) if mthlim is not None else [1]
    if len(lim) == 1:
        lim = lim * meqn
    out = np.zeros(8, dtype=np.int32)
    out[: len(lim)] = lim
    return out


def sc_flux1(rp_id, rp_params, mwaves, mbc, mx, q1d, dx, dt, ixyz, weno_variant, aux1d=None, mthlim=None):
    """flux1 on one slice in direction ixyz = 1, 2, 3: q1d [meqn, mx+2mbc], aux1d [maux, mx+2mbc] or None.
    Returns (dq1d, cfl)."""
    q1d = np.asfortranarray(q1d, dtype=np.float64)
    dq = np.zeros_like(q1d, order="F")
    null = ctypes.cast(None, _dp)
    maux = 0 if aux1d is None else aux1d.shape[0]
    a = null if aux1d is None else _p(np.asfortranarray(aux1d, dtype=np.float64))
    lim = _mthlim8(mthlim, q1d.shape[0])
    cfl = lib().oracle3d_sc_flux1(rp_id, _p(_params(rp_params)), q1d.shape[0], mwaves, maux, mbc, mx, _p(q1d), a,
                                  _p(dq), dx, dt, ixyz, weno_variant, lim.ctypes.data_as(_ip))
    return dq, _check(cfl)


def sc_flux3(rp_id, rp_params, mwaves, mbc, mx, my, mz, q, dx, dy, dz, dt, weno_variant, aux=None, mthlim=None):
    """SharpClaw's dq in 3-D (DESIGN.md §1): q [meqn, mx+2mbc, my+2mbc, mz+2mbc] with ghost cells filled,
    aux [maux, ...] or None.  Returns (dq, cfl); dq is zero outside the interior."""
    assert q.flags["F_CONTIGUOUS"]
    dq = np.zeros_like(q, order="F")
    null = ctypes.cast(None, _dp)
    maux = 0 if aux is None else aux.shape[0]
    a = null if aux is None else _p(np.asfortranarray(aux, dtype=np.float64))
    lim = _mthlim8(mthlim, q.shape[0])
    cfl = lib().oracle3d_sc_flux3(rp_id, _p(_params(rp_params)), q.shape[0], mwaves, maux, mbc, mx, my, mz, _p(q), a,
                                  _p(dq), dx, dy, dz, dt, weno_variant, lim.ctypes.data_as(_ip))
    return dq, _check(cfl)


def sharpclaw3d_solver(rp_id, rp_params, mwaves):
    """oracle/pyclaw_oracle.py's OracleSolver (kind 'sharpclaw': time integrators, boundary conditions,
    variable dt with rejected steps, solver.py:602-717) with the 3-D dq of sc_flux3.  lim_type 1 / 2 / 3
    select tvd2 / PyWENO weno5 (weno_variant, f32 by default) / the hand-written weno5."""
    import sys
    sys.path.insert(0, os.path.dirname(_HERE))
    from oracle import pyclaw_oracle as po

    class SharpClaw3D(po.OracleSolver):
        def _dq(self, q, t):
            self._bcs(q, t)
            mbc = self.mbc
            variant = {1: RECON_TVD2, 3: WENO_OLD}.get(self.lim_type, self.weno_variant)
            mx, my, mz = self.n
            dq, cfl = sc_flux3(self.rp_id, self.rp_params, self.mwaves, mbc, mx, my, mz, self.qbc, self.d[0],
                               self.d[1], self.d[2], self.dt, variant, aux=self.auxbc, mthlim=self.limiters)
            self.cfl = cfl
            if cfl > self.cfl_max:
                raise po._CFLError()
            return po._interior(dq, mbc)

        def setup(self, q, aux, d):
            lim_type = self.lim_type
            self.lim_type = 2  # the base class would set the 1-D / 2-D oracle's global tvd2 limiters
            super().setup(q, aux, d)
            self.lim_type = lim_type

    return SharpClaw3D("sharpclaw", 3, rp_id, rp_params, mwaves)
