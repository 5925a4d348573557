"""Riemann-solver descriptors.

The reference bakes the Riemann solver into classic2.so / sharpclaw2.so at link time
(RP_SOURCE in each application's Makefile, e.g. apps/euler/2d/shockbubble/Makefile:3), so
its scripts never name the solver in Python.  Here ``solver.rp`` may be set to one of
these descriptors (or its name); if it is left unset the solver is inferred from the
keys of ``state.aux_global`` (the cparam common block the script fills).
"""
from .._lib import (RP_ACOUSTICS, RP_ADVECTION, RP_EULER5, RP_SHALLOW, RP_SPHERE, RP_NEL_FWAVE,
                    RP_PSYSTEM, RP_ACOUSTICS3D_VC, RP_VC_ACOUSTICS, RP_BURGERS, RP_ADVECTION_COLOR,
                    RP_VC_ADVECTION, RP_EULER1D, RP_ADVECTION3D, RP_EULER3D,
                    RP_ADVECTION3D_VC_FWAVE, RP_SHALLOW_BATHY_FWAVE)


class RiemannSolver(object):
    def __init__(self, name, rp_id, meqn, mwaves, param_names, ndims, optional=(), defaults=None,
                 fwave=False, maux=0):
        self.name, self.rp_id, self.param_names, self.ndims = name, rp_id, param_names, ndims
        self._meqn = meqn
        self._mwaves = mwaves
        self.mwaves = self.nwaves(max(ndims))
        self.optional = set(optional)
        self.defaults = dict(defaults or {})
        self.fwave = fwave      # returns f-waves: pairs with the classic*fw modules (clawpack.py:222)
        self.maux = maux        # aux components the solver reads
        self.lib = None         # user-supplied solvers: {arithmetic: path of the library variant}

    def __call__(self, q_l, q_r, aux_l=None, aux_r=None, aux_global=None, ixy=1):
        """The reference's Python Riemann-solver contract (doc/rp.rst:7-62, clawpack.py:349):
        ``wave, s, amdq, apdq = rp(q_l, q_r, aux_l, aux_r, aux_global)`` on arrays of interfaces,
        evaluated by the CUDA solver that the sweeps inline (ixy = 1, 2, 3 for a 3-D solver).  q_l, q_r: [meqn, n] CUDA tensors
        (left / right state of each interface); returns CUDA tensors wave[meqn, mwaves, n],
        s[mwaves, n], amdq[meqn, n], apdq[meqn, n].  aux_l, aux_r: [maux, n] or None."""
        import ctypes
        import torch
        from .. import _lib
        ndim = 2 if 2 in self.ndims else (1 if 1 in self.ndims else 3)
        q_l = q_l.contiguous().to(torch.float64)
        q_r = q_r.contiguous().to(torch.float64)
        meqn, n = q_l.shape
        mw = self.nwaves(ndim)
        maux = 0 if aux_l is None else aux_l.shape[0]
        if aux_l is not None:
            aux_l, aux_r = aux_l.contiguous().to(torch.float64), aux_r.contiguous().to(torch.float64)
        P = _lib.make_problem(ndim, meqn, mw, 2, 8, 8, 1.0, 1.0, self.rp_id, self.params(aux_global or {}), maux=maux)
        wave = torch.empty((meqn, mw, n), dtype=torch.float64, device=q_l.device)
        s = torch.empty((mw, n), dtype=torch.float64, device=q_l.device)
        amdq, apdq = torch.empty_like(q_l), torch.empty_like(q_l)
        ptr = lambda t: ctypes.c_void_p(t.data_ptr())
        prev = _lib.set_variant(self._variant()) if self.lib else None
        try:
            _lib.call("clawb200_rp_solve", ctypes.byref(P), ixy, n, ptr(q_l), ptr(q_r),
                      ptr(aux_l) if aux_l is not None else None, ptr(aux_r) if aux_r is not None else None, ptr(wave), ptr(s),
                      ptr(amdq), ptr(apdq), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        finally:
            if prev is not None:
                _lib.set_variant(prev)
        return wave, s, amdq, apdq

    def _variant(self, arithmetic='strict'):
        """Name under which the library variant holding a user-supplied solver is registered."""
        from .. import _lib
        base = 'fma' if arithmetic == 'fma' else 'strict'
        if base not in self.lib:
            from ..build import build_user
            self.lib[base] = build_user(self.header, self.name, fma=(base == 'fma'), ndims=self.ndims)
        key = 'user:%s:%s' % (self.name, base)
        _lib.LIB_PATHS[key] = self.lib[base]
        return key

    def meqn(self, ndim):
        return self._meqn(ndim) if callable(self._meqn) else self._meqn

    def nwaves(self, ndim):
        return self._mwaves(ndim) if callable(self._mwaves) else self._mwaves

    def params(self, aux_global):
        missing = [k for k in self.param_names if k not in aux_global and k not in self.optional]
        if missing:
            # state.py:154-158: every cparam variable must be present in aux_global
            raise Exception("Some required value(s) in the cparam common block in the Riemann "
                            "solver have not been set in aux_global: %s" % missing)
        return [float(aux_global.get(k, self.defaults.get(k, 0.0))) for k in self.param_names]

    def __repr__(self):
        return "<riemann %s>" % self.name


acoustics = RiemannSolver("acoustics", RP_ACOUSTICS, lambda ndim: ndim + 1, 2, ["rho", "bulk", "cc", "zz"], (1, 2))
advection = RiemannSolver("advection", RP_ADVECTION, 1, 1, ["u", "v"], (1, 2), optional=["v"])
euler_5wave = RiemannSolver("euler_5wave", RP_EULER5, 5, 5, ["gamma", "gamma1"], (2,))
shallow_roe_with_efix = RiemannSolver("shallow_roe_with_efix", RP_SHALLOW, lambda ndim: ndim + 1,
                                      lambda ndim: ndim + 1, ["grav"], (1, 2))

# shallow water on the sphere (apps/shallow-sphere): `g` is the reference's common /sw/ g;
# dxcom / dycom (common /comxyt/) default to the grid spacing
shallow_sphere = RiemannSolver("shallow_sphere", RP_SPHERE, 4, 3, ["g", "dxcom", "dycom"], (2,),
                               optional=["dxcom", "dycom"])

# f-wave solvers (solver.fwave = True).  Stress law 1: sigma = K eps; 2: sigma = exp(K eps) - 1.
#   1-D: aux = {rho, K}     (apps/elasticity/1d/stegoton/stegoton.py:17-27), law from
#        aux_global['stress_law'] (default 2, the stegoton's)
#   2-D: aux = {rho, E, stress law, copy of eps}   (test/psystem/psystem.py:35-86)
nonlinear_elasticity_fwave = RiemannSolver("nonlinear_elasticity_fwave", RP_NEL_FWAVE, 2, 2, ["stress_law"],
                                           (1,), optional=["stress_law"], defaults={"stress_law": 2.0},
                                           fwave=True, maux=2)
psystem = RiemannSolver("psystem", RP_PSYSTEM, 3, 2, [], (2,), fwave=True, maux=4)
# shallow water over bathymetry (1-D, 2-D), well balanced: aux = {b}, the bottom elevation (surface
# eta = h + b); cells with h <= dry_tolerance have zero velocity.  Classic solvers only.
shallow_bathymetry_fwave = RiemannSolver("shallow_bathymetry_fwave", RP_SHALLOW_BATHY_FWAVE, lambda ndim: ndim + 1,
                                         lambda ndim: ndim + 1, ["grav", "dry_tolerance"], (1, 2),
                                         optional=["dry_tolerance"], defaults={"dry_tolerance": 1e-3},
                                         fwave=True, maux=1)

# 3-D acoustics in a heterogeneous medium (test/acoustics/3d): aux = {impedance, sound speed}
vc_acoustics_3d = RiemannSolver("vc_acoustics_3d", RP_ACOUSTICS3D_VC, 4, 2, [], (3,), maux=2)
# 3-D constant-coefficient advection and 3-D Euler (Roe + entropy fix; q = rho, rho u, rho v, rho w, E)
advection_3d = RiemannSolver("advection_3d", RP_ADVECTION3D, 1, 1, ["u", "v", "w"], (3,))
euler_3d = RiemannSolver("euler_3d", RP_EULER3D, 5, 3, ["gamma", "gamma1"], (3,))
# 3-D conservative transport q_t + (u q)_x + (v q)_y + (w q)_z = 0 in a cell-centred velocity field,
# aux = {u, v, w}; an f-wave solver (solver.fwave = True): conserves q for any velocity field
vc_advection_fwave_3d = RiemannSolver("vc_advection_fwave_3d", RP_ADVECTION3D_VC_FWAVE, 1, 1, [], (3,), fwave=True,
                                      maux=3)

# further solvers of the reference's applications (set solver.rp to use them)
vc_acoustics = RiemannSolver("vc_acoustics", RP_VC_ACOUSTICS, 3, 2, [], (2,), maux=2)          # aux {rho, c}
burgers = RiemannSolver("burgers", RP_BURGERS, 1, 1, [], (1,))
advection_color = RiemannSolver("advection_color", RP_ADVECTION_COLOR, 1, 1, [], (1,), maux=1)  # aux {u}
vc_advection = RiemannSolver("vc_advection", RP_VC_ADVECTION, 1, 1, [], (2,), maux=2)           # aux {u, v[, capa]}
euler_with_efix = RiemannSolver("euler_with_efix", RP_EULER1D, 3, 3, ["gamma", "gamma1"], (1,))

def from_header(header, name=None, meqn=1, mwaves=1, ndims=(2,), param_names=(), optional=(), defaults=None,
                fwave=False, maux=0, build=True):
    """A user-supplied Riemann solver: ``header`` defines ``template <int IXY> struct RpUser`` with the
    interface of the solvers in pyclaw_b200/csrc/rp.cuh (examples/user_rp/rp_kpp.cuh) and, when
    ``ndims`` contains 3, ``template <int IXYZ> struct RpUser3`` with the 3-D interface (rpn3 / rpt3 /
    rptt3; examples/user_rp/rp_acoustics3d_user.cuh).  It is
    compiled into a variant of the library (pyclaw_b200.build.build_user; nvcc must be on PATH
    unless the variant was built before) and returned as a descriptor for ``solver.rp``.

    This is the reference's plugin seam -- the rpn2 / rpt2 Fortran files an application's Makefile
    names in RP_SOURCE (Makefile.rules:1-26) -- with the solver named in Python instead of in a
    Makefile.  ``param_names``: the aux_global entries handed to the solver as P.p[0..7] (the
    cparam common block); meqn / mwaves / maux must agree with the header's constants (the
    library checks them at the first call)."""
    import os
    from .. import _lib
    from ..build import build_user, user_lib_path
    header = os.path.abspath(header)
    name = name or os.path.splitext(os.path.basename(header))[0]
    rs = RiemannSolver(name, _lib.RP_USER, meqn, mwaves, list(param_names), tuple(ndims), optional=optional,
                       defaults=defaults, fwave=fwave, maux=maux)
    rs.header = header
    rs.lib = {}
    if build:
        rs.lib['strict'] = build_user(header, name, ndims=rs.ndims)
    elif os.path.exists(user_lib_path(name)):
        rs.lib['strict'] = user_lib_path(name)
    else:
        raise Exception("library variant %s has not been built" % user_lib_path(name))
    return rs


_BY_NAME = {s.name: s for s in (vc_acoustics, burgers, advection_color, vc_advection, euler_with_efix,
                                vc_acoustics_3d, advection_3d, euler_3d, vc_advection_fwave_3d,
                                acoustics, advection, euler_5wave, shallow_roe_with_efix, shallow_sphere,
                                nonlinear_elasticity_fwave, psystem, shallow_bathymetry_fwave)}
_BY_NAME.update({"euler": euler_5wave, "shallow": shallow_roe_with_efix})


class _Module(object):
    """Mimics ``riemann.rp_acoustics.rp_acoustics_1d`` style access."""

    def __init__(self, solver, names):
        self.mwaves = solver.mwaves
        for n in names:
            setattr(self, n, solver)


rp_acoustics = _Module(acoustics, ["rp_acoustics_1d", "rp_acoustics_2d"])
rp_advection = _Module(advection, ["rp_advection_1d", "rp_advection_2d"])
rp_euler = _Module(euler_5wave, ["rp_euler_5wave_2d"])
rp_shallow = _Module(shallow_roe_with_efix, ["rp_shallow_roe_with_efix_2d"])


def resolve(rp, aux_global, ndim, fwave=False):
    if isinstance(rp, RiemannSolver):
        return rp
    if isinstance(rp, str):
        if rp not in _BY_NAME:
            raise Exception("Unknown Riemann solver %r" % rp)
        return _BY_NAME[rp]
    if rp is not None:
        raise NotImplementedError("Python Riemann solvers are not supported: there is no CPU "
                                  "path; set solver.rp to a pyclaw.riemann descriptor")
    found = _infer(aux_global, ndim, fwave)
    # The reference binds the solver at link time (RP_SOURCE in the application's Makefile); a
    # guess from the cparam names must be visible, so that a script whose aux_global happens to
    # match another physics does not run the wrong solver silently.
    import logging
    logging.getLogger('evolve').warning(
        "solver.rp is not set: using Riemann solver %r inferred from aux_global keys %s "
        "(set solver.rp = pyclaw.riemann.<name> to choose explicitly)", found.name, sorted(aux_global.keys()))
    return found


def _infer(aux_global, ndim, fwave):
    if ndim == 3:
        return vc_acoustics_3d       # the only 3-D solver the reference's applications link
    if fwave:
        # the only f-wave solvers the reference's applications link (stegoton, psystem)
        return nonlinear_elasticity_fwave if ndim == 1 else psystem
    keys = set(aux_global.keys())
    if {"rho", "bulk", "cc", "zz"} <= keys:
        return acoustics
    if {"gamma", "gamma1"} <= keys:
        return euler_with_efix if ndim == 1 else euler_5wave
    if "grav" in keys:
        return shallow_roe_with_efix
    if "u" in keys:
        return advection
    raise Exception("Cannot infer the Riemann solver from aux_global keys %s; set solver.rp" % sorted(keys))
