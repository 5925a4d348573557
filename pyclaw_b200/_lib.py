"""ctypes binding of libclawb200.so (include/clawb200.h).

There is deliberately no fallback: if the CUDA library is missing or a call fails,
an exception is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CLAWB200_LIB selects another build of the same library (kernel tuning experiments)
LIB_PATH = os.environ.get("CLAWB200_LIB") or os.path.join(_HERE, "csrc", "libclawb200.so")
# Arithmetic variants: two builds of the same sources (pyclaw_b200/build.py).  'strict' is the
# parity build (-fmad=false, bit for bit against the oracle); 'fma' lets nvcc contract a*b+c.
LIB_PATHS = {"strict": LIB_PATH, "fma": os.path.join(_HERE, "csrc", "libclawb200_fma.so")}

MAXWAVES = 8
RP_ACOUSTICS, RP_ADVECTION, RP_EULER5, RP_SHALLOW, RP_SPHERE = 1, 2, 3, 4, 5
RP_NEL_FWAVE, RP_PSYSTEM, RP_ACOUSTICS3D_VC = 6, 7, 8
RP_VC_ACOUSTICS, RP_BURGERS, RP_ADVECTION_COLOR, RP_VC_ADVECTION, RP_EULER1D = 9, 10, 11, 12, 13
RP_ADVECTION3D, RP_EULER3D, RP_ADVECTION3D_VC_FWAVE = 14, 15, 16
RP_SHALLOW_BATHY_FWAVE = 17
RP_USER = 100   # a solver compiled in from a user header (riemann.from_header)
WENO_PYWENO_F32, WENO_PYWENO_F64, WENO_OLD, WENO_TABLES, RECON_TVD2 = 0, 1, 2, 3, 4
RECON_WENO_WAVE, RECON_WENO_FWAVE = 5, 6
STAGE_AXPY, STAGE_CONVEX, STAGE_FINAL104, STAGE_DQ_ONLY = 0, 1, 2, 3
# clawb200_arith_probe: policies and operations
ARITH_FAST, ARITH_FAST_FZ, ARITH_EXACT, ARITH_GUARDED, ARITH_GUARDED_FZ = 0, 1, 2, 3, 4
(ARITH_RCP, ARITH_RCP_NC, ARITH_DIV_RCP, ARITH_DIV, ARITH_DIV_NZ, ARITH_SQRT, ARITH_SQRT_RCP, ARITH_SQRT_RCPS,
 ARITH_SQRT_RCP2S) = range(9)


class ClawB200Error(RuntimeError):
    pass


class Problem(ctypes.Structure):
    """struct clawb200_problem"""
    _fields_ = [
        ("ndim", ctypes.c_int), ("meqn", ctypes.c_int), ("mwaves", ctypes.c_int),
        ("maux", ctypes.c_int), ("mbc", ctypes.c_int),
        ("mx", ctypes.c_int), ("my", ctypes.c_int),
        ("dx", ctypes.c_double), ("dy", ctypes.c_double),
        ("method", ctypes.c_int * 7),
        ("mthlim", ctypes.c_int * MAXWAVES),
        ("rp_id", ctypes.c_int),
        ("rp_params", ctypes.c_double * 8),
        ("mstride", ctypes.c_longlong),
        ("pitch", ctypes.c_int),
        ("weno_variant", ctypes.c_int),
        ("dt_dev", ctypes.c_void_p),
        ("weno_k", ctypes.c_int),
        ("weno_tab", ctypes.c_void_p),
        ("step2_mode", ctypes.c_int),
    ]


def make_problem(ndim, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, rp_params, method=None,
                 mthlim=None, maux=0, pitch=None, mstride=None, weno_variant=WENO_PYWENO_F32):
    p = Problem()
    p.ndim, p.meqn, p.mwaves, p.maux, p.mbc = ndim, meqn, mwaves, maux, mbc
    p.mx, p.my = mx, (my if ndim > 1 else 1)
    p.dx, p.dy = dx, (dy if ndim > 1 else 1.0)
    method = list(method) if method is not None else [1, 2, 0, 0, 0, 0, maux]
    for i in range(7):
        p.method[i] = int(method[i])
    mthlim = list(mthlim) if mthlim is not None else [0] * mwaves
    for i in range(MAXWAVES):
        p.mthlim[i] = int(mthlim[i]) if i < len(mthlim) else 0
    p.rp_id = rp_id
    for i in range(8):
        p.rp_params[i] = float(rp_params[i]) if i < len(rp_params) else 0.0
    nx = mx + 2 * mbc
    ny = (my + 2 * mbc) if ndim > 1 else 1
    p.pitch = nx if pitch is None else pitch
    p.mstride = p.pitch * ny if mstride is None else mstride
    p.weno_variant = weno_variant
    p.dt_dev = None
    p.weno_k = 0
    p.weno_tab = None
    p.step2_mode = 0
    return p


def pack_weno_tables(tab):
    """Coefficient tables of pyclaw_b200.weno_tables.tables() in the layout the kernels read
    (clawb200_pack_weno_tables): a float64 numpy array the caller keeps alive / uploads."""
    import numpy as np
    L = load()
    out = np.zeros(L.clawb200_weno_table_doubles(), dtype=np.float64)
    arr = [np.ascontiguousarray(tab[k], dtype=np.float64) for k in ('S', 'CL', 'CR', 'WL', 'WR')]
    call("clawb200_pack_weno_tables", int(tab['k']), *[ctypes.c_void_p(a.ctypes.data) for a in arr],
         float(tab['eps']), ctypes.c_void_p(out.ctypes.data))
    return out


_libs = {}
_active = "strict"
_vp, _dp, _i, _d = ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_double
_pp = ctypes.POINTER(Problem)
_dref = ctypes.POINTER(ctypes.c_double)

# name -> argtypes ; every function returns int
SIGNATURES = {
    "clawb200_cfl_reset": [_dp, _vp],
    "clawb200_step1": [_pp, _dp, _dp, _dp, _d, _dp, _vp],
    "clawb200_step2ds": [_pp, _dp, _dp, _dp, _d, _i, _dp, _vp],
    "clawb200_step2": [_pp, _dp, _dp, _dp, _d, _dp, _vp],
    "clawb200_step2_parts": [_pp, _dp, _dp, _dp, _d, _i, _dp, _vp],
    "clawb200_step2_rows": [_pp, _dp, _dp, _dp, _d, _i, _i, _dp, _vp],
    "clawb200_sharpclaw_stage": [_pp, _dp, _dp, _dp, _dp, _dp, _d, _i, _d, _d, _d, _dp, _vp],
    "clawb200_sharpclaw_stage3": [_pp, _i, _d, _dp, _dp, _dp, _dp, _dp, _d, _i, _d, _d, _d, _dp, _vp],
    "clawb200_ssp104_combine": [_dp, _dp, _dp, ctypes.c_longlong, _vp],
    "clawb200_sphere_src2": [_pp, _dp, _dp, _d, _vp],
    "clawb200_bc_fill": [_pp, _dp, _i, _i, _i, _i, _i, _vp],
    "clawb200_aos_to_soa": [_dp, _dp, _i, _i, _i, ctypes.c_longlong, _i, _vp],
    "clawb200_soa_to_aos": [_dp, _dp, _i, _i, _i, ctypes.c_longlong, _i, _vp],
    "clawb200_halo_pack": [_pp, _dp, _i, _i, _i, _dp, _vp],
    "clawb200_halo_unpack": [_pp, _dp, _i, _i, _i, _dp, _vp],
    "clawb200_step1_host": [_pp, _dp, _dp, _d, _dref],
    "clawb200_step2ds_host": [_pp, _dp, _dp, _dp, _d, _i, _dref],
    "clawb200_step2_host": [_pp, _dp, _dp, _dp, _d, _dref],
    "clawb200_sharpclaw_dq_host": [_pp, _dp, _dp, _dp, _d, _dref],
    "clawb200_sharpclaw_dq3_host": [_pp, _i, _d, _dp, _dp, _dp, _d, _dref],
    "clawb200_pack_weno_tables": [_i, _dp, _dp, _dp, _dp, _dp, _d, _dp],
    "clawb200_step3ds": [_pp, _i, _d, _dp, _dp, _dp, _d, _i, _dp, _vp],
    "clawb200_bc_fill3": [_pp, _i, _dp, _i, _i, _i, _i, _i, _vp],
    "clawb200_step3ds_host": [_pp, _i, _d, _dp, _dp, _dp, _d, _i, _dref],
    "clawb200_step3": [_pp, _i, _d, _dp, _dp, _dp, _d, _dp, _dp, _vp],
    "clawb200_step3_host": [_pp, _i, _d, _dp, _dp, _dp, _d, _dref],
    "clawb200_release_host_scratch": [],
    "clawb200_rp_solve": [_pp, _i, ctypes.c_longlong, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _vp],
    "clawb200_rp_transverse": [_pp, _i, ctypes.c_longlong, _dp, _dp, _i, _dp, _dp, _dp, _vp],
    "clawb200_rp_solve_host": [_pp, _i, ctypes.c_longlong, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp],
    "clawb200_rp_transverse_host": [_pp, _i, ctypes.c_longlong, _dp, _dp, _i, _dp, _dp, _dp],
    "clawb200_arith_probe": [_i, _i, ctypes.c_longlong, _dp, _dp, _dp, _vp],
}


def set_variant(name):
    """Select the build that `call` dispatches to ('strict' | 'fma'); returns the previous one.
    Solvers set it from ``solver.arithmetic`` at the start of every step."""
    global _active
    if name not in LIB_PATHS:
        raise ClawB200Error("unknown arithmetic variant %r (expected 'strict' or 'fma')" % (name,))
    prev, _active = _active, name
    return prev


def load(variant=None):
    """Load the CUDA library; raises if it has not been built (no CPU fallback)."""
    variant = variant or _active
    if variant not in _libs:
        path = LIB_PATHS[variant]
        if not os.path.exists(path):
            raise ClawB200Error(
                "%s is missing (%s): build it with `python -m pyclaw_b200.build%s`; "
                "pyclaw_b200 has no CPU fallback" % (os.path.basename(path), path,
                                                     " --fma" if variant == "fma" else ""))
        L = ctypes.CDLL(path)
        L.clawb200_version.restype = ctypes.c_int
        L.clawb200_weno_table_doubles.restype = ctypes.c_int
        L.clawb200_step2_launches.restype = ctypes.c_int
        L.clawb200_step2_launches.argtypes = [_pp]
        L.clawb200_step3_scratch_doubles.restype = ctypes.c_longlong
        L.clawb200_step3_scratch_doubles.argtypes = [_pp]
        L.clawb200_last_error.restype = ctypes.c_char_p
        for name, args in SIGNATURES.items():
            f = getattr(L, name)
            f.restype = ctypes.c_int
            f.argtypes = args
        _libs[variant] = L
    return _libs[variant]


def check(rc):
    if rc != 0:
        raise ClawB200Error("clawb200 error %d: %s" % (rc, load().clawb200_last_error().decode()))


def call(name, *args):
    check(getattr(load(), name)(*args))
