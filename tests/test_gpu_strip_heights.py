"""
The streaming kernels at the strip heights that large grids run on.

Every 2-D streaming kernel (the x- and y-engines of the classic sweeps, the single-pass unsplit
step, the SharpClaw 2-D stage and the SharpClaw 3-D x/y and z kernels) walks a strip of
``rows_per_cta`` rows, and ``pick_rows`` (pyclaw_b200/csrc/launch.cuh) picks that height at run time
from the number of column CTAs times the number of strips: 8 rows on the grids of the other kernel
tests, 16 to 128 on grids above 1024^2.  The height depends on the number of strips, not on the
grid's area, so tall narrow grids reach every height with few cells.

Each case builds its grid from the Python copy of the launch geometry below, asserts the strip
height and the rows of the last strip that each of its launches gets (one row, h - 1 rows, a full
strip), calls the device entry points directly (the host entry points cut grids without aux into
slabs of 8-row strips) on torch CUDA tensors in the [m][j][i] / [m][k][j][i] layout, and compares
interior cells and the Courant number with the CPU oracle bit for bit.  The fma build is held to the
bounds of test_gpu_fma_build.py.
"""
import ctypes
import os

import numpy as np
import pytest

import problems
from oracle import pyclaw_oracle as po
from pyclaw_b200 import _lib

NTHREADS = max(2, os.cpu_count() or 2)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# =============================================================================================
# The launch geometry, restated.  If pick_rows or a tile width changes, this copy changes with it.
# =============================================================================================
XNT = 128  # x-engine threads per CTA, launch.cuh:64
YNT = 128  # y-engine threads per CTA, launch.cuh:65
FNT = 128  # single-pass kernel threads per CTA, sweep_fused.cu:5
SNT = 128  # SharpClaw stage threads per CTA, sharpclaw.cuh:517


def pick_rows(nrows, ncol_ctas, tall=True):
    """launch.cuh:113-124"""
    if tall and ncol_ctas * ((nrows + 127) // 128) >= 148 * 28:
        return 128
    h = 64
    while h > 8 and ncol_ctas * ((nrows + h - 1) // h) < 148 * 4:
        h //= 2
    return h


def ctas_x(mx):
    """x-engine, unsplit and step2ds: XNT - 3 columns per CTA (clawb200.cu:202, :368)"""
    return (mx + XNT - 4) // (XNT - 3)


def ctas_y(mx):
    """y-engine, unsplit: YNT - 2 columns per CTA (clawb200.cu:372)"""
    return (mx + YNT - 3) // (YNT - 2)


def ctas_y_ds(mx, mbc):
    """y-engine, step2ds: YNT columns of the padded row per CTA (clawb200.cu:207)"""
    return (mx + 2 * mbc + YNT - 1) // YNT


def ctas_fused(mx):
    """single-pass kernel: FNT - 4 columns per CTA (sweep_fused.cu:10-17)"""
    return (mx + FNT - 5) // (FNT - 4)


def ctas_sc(mx):
    """SharpClaw stage, 2-D and the 3-D x/y kernel per plane: SNT - 2 columns per CTA (sharpclaw.cuh:536-541,
    sharpclaw.cu:43-47, sharpclaw3.cuh:114-122)"""
    return (mx + SNT - 3) // (SNT - 2)


def ctas_sc3_z(mx, my):
    """SharpClaw 3-D z kernel: one thread per (i, j) column of the grid plus one ghost layer
    (sharpclaw3.cuh:132-135)"""
    return min(-(-(mx + 2) * (my + 2) // SNT), 1 << 24)


def strip(nrows, ncol_ctas, tall=True):
    """(strip height, rows in the last strip) of a launch over nrows rows"""
    h = pick_rows(nrows, ncol_ctas, tall)
    return h, nrows - (nrows - 1) // h * h


def rows_for(h, last, ncol_ctas):
    """The fewest rows at which ncol_ctas column CTAs get h-row strips, the last one `last` rows tall:
    pick_rows takes h once ncol_ctas * strips reaches 148 * 4 (148 * 28 for 128 rows)."""
    strips = -(-148 * (28 if h == 128 else 4) // ncol_ctas)
    return (strips - 1) * h + last


def step2_strips(mx, nrows, single_pass):
    if single_pass:
        return {"single-pass": strip(nrows, ctas_fused(mx))}
    return {"x": strip(nrows, ctas_x(mx)), "y": strip(nrows, ctas_y(mx))}


def step2ds_strips(mx, my, mbc, ids):
    if ids == 1:   # every padded row
        return {"x": strip(my + 2 * mbc, ctas_x(mx))}
    return {"y": strip(my, ctas_y_ds(mx, mbc))}


# A shape is (mx, h, last): the narrow grids have one column CTA in every kernel (mx = 5, and mx = 3
# for the 128-row strips, which need 530 k rows); mx = 251 has three x-engine / single-pass tiles,
# the last one partial, and two y-engine / SharpClaw tiles.  Rows come from the kernel with the
# fewest column CTAs; the others then get the same height.
def _last(h, i):
    return (1, h - 1, h)[i % 3]


def full_shapes(i, tall128=True):
    """every narrow shape, each height at mx = 251 and (classic) 128 rows, the last-strip sizes rotating with i"""
    s = [(5, h, last) for h in (16, 32, 64) for last in (1, h - 1, h)] + [(251, h, _last(h, i + k)) for k, h in enumerate((16, 32, 64))]
    return s + ([(3, 128, _last(128, i))] if tall128 else [])


def light_shapes(i, tall128=True):
    """one narrow shape per height, one mx = 251 shape and (classic) one 128-row shape, rotating with i"""
    s = [(5, h, _last(h, i + k)) for k, h in enumerate((16, 32, 64))]
    h = (16, 32, 64)[i % 3]
    s.append((251, h, _last(h, i + 1)))
    return s + ([(3, 128, _last(128, i + 2))] if tall128 else [])


def _nrows(mx, h, last):
    ctas = 1 if mx < 124 else min(ctas_x(mx), ctas_y(mx), ctas_fused(mx), ctas_sc(mx))
    return rows_for(h, last, ctas)


def _id(shape):
    return "%dx%d-last%d" % shape


# =============================================================================================
# The geometry copy on its own (no GPU)
# =============================================================================================
def test_geometry_copy_gives_the_known_heights():
    """The heights of square grids (8 rows up to 1024^2, 32 at 2048^2, 64 at 4096^2, 128 at 8192^2 and
    64 for SharpClaw there), and the first row count of each height on one column CTA."""
    for n, classic, sc in ((1024, 8, 8), (2048, 32, 32), (4096, 64, 64), (8192, 128, 64)):
        assert pick_rows(n, ctas_x(n)) == classic and pick_rows(n, ctas_y(n)) == classic
        assert pick_rows(n, ctas_fused(n)) == classic and pick_rows(n, ctas_sc(n), False) == sc
    assert [rows_for(h, 1, 1) for h in (16, 32, 64, 128)] == [9457, 18913, 37825, 530305]
    assert rows_for(64, 1, 3) == 12609 and rows_for(64, 1, 2) == 18881
    for h in (16, 32, 64, 128):
        assert pick_rows(rows_for(h, 1, 1) - 1, 1) == h // 2


def _coverage():
    """(kernel, h, last) of every launch the parametrised cases below make."""
    out = set()
    for i, (name, mode, *_rest) in enumerate(UNSPLIT):
        for mx, h, last in UNSPLIT_SHAPES[i]:
            fused = mode == 0 and name in SINGLE_PASS and not _rest[0]
            for k, v in step2_strips(mx, _nrows(mx, h, last), fused).items():
                out.add(("unsplit " + k, v))
    for i, (name, mbc) in enumerate(DS):
        for mx, h, last in DS_SHAPES[i]:
            n = _nrows(mx, h, last)
            for ids in (1, 2):
                for k, v in step2ds_strips(mx, n - 2 * mbc if ids == 1 else n, mbc, ids).items():
                    out.add(("step2ds " + k, v))
    for shapes in SC2_SHAPES:
        for mx, h, last in shapes:
            out.add(("sharpclaw2", strip(_nrows(mx, h, last), ctas_sc(mx), False)))
    for name in SC3_SOLVERS:
        for shape, _ in SC3_XY + SC3_Z:
            for k, v in sc3_strips(*shape).items():
                out.add(("sharpclaw3 " + k, v))
    return out


def test_matrix_covers_every_height_and_last_strip():
    """Every kernel at every height it can take, each with a last strip of one row, h - 1 rows and h rows."""
    cov = _coverage()
    need = {("unsplit x", 128), ("unsplit y", 128), ("unsplit single-pass", 128), ("step2ds x", 128),
            ("step2ds y", 128)}
    for k in ("unsplit x", "unsplit y", "unsplit single-pass", "step2ds x", "step2ds y", "sharpclaw2",
              "sharpclaw3 xy", "sharpclaw3 z"):
        need |= {(k, h) for h in (16, 32, 64)}
    for k, h in need:
        for last in (1, h - 1, h):
            assert (k, (h, last)) in cov, (k, h, last)


# =============================================================================================
# Device harness
# =============================================================================================
def _axes(ndim):
    return (0,) + tuple(range(ndim - 1, 0, -1))


def _dev(a):
    """Fortran-ordered q[m, i, j(, k)] -> a CUDA tensor [m][(k)][j][i]"""
    import torch
    return torch.from_numpy(np.ascontiguousarray(np.transpose(a, _axes(a.ndim)))).cuda()


def _host(t):
    """the inverse of _dev (a view in the oracle's index order)"""
    a = t.cpu().numpy()
    return np.transpose(a, _axes(a.ndim))


def _vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _cfl_dev():
    import torch
    return torch.zeros(1, dtype=torch.float64, device="cuda")


def _inner(mbc, ndim=2):
    return (slice(None),) + (slice(mbc, -mbc),) * ndim


def _same(got, ref, what):
    for m in range(ref.shape[0]):
        if not np.array_equal(got[m], ref[m]):
            d = np.abs(got[m] - ref[m])
            raise AssertionError("%s: component %d differs, max |diff| = %g at %s"
                                 % (what, m, np.nanmax(d), np.unravel_index(np.nanargmax(d), d.shape)))


# =============================================================================================
# Classic solvers: data and oracles
# =============================================================================================
# name: (rp_id, params, meqn, mwaves, limiters, (dx, dy, dt))
CLASSIC = {
    "acoustics": (1, [1.0, 4.0, 2.0, 2.0], 3, 2, [4, 4], (0.01, 0.013, 0.0011)),
    "advection": (2, [0.7, -0.4], 1, 1, [3], (0.01, 0.013, 0.0011)),
    "euler": (3, [1.4, 0.4], 5, 5, [4, 4, 4, 4, 2], (0.01, 0.013, 0.0011)),
    "shallow": (4, [1.0], 3, 3, [4, 1, 2], (0.01, 0.013, 0.0011)),
    "vc_acoustics": (po.RP_VC_ACOUSTICS, [], 3, 2, [4, 4], (0.01, 0.013, 0.0011)),
    "vc_advection": (po.RP_VC_ADVECTION, [], 1, 1, [4], (0.01, 0.013, 0.0011)),
    "psystem": (po.RP_PSYSTEM, [], 3, 2, [2, 2], (0.05, 0.04, 0.008)),
    "bathymetry": (_lib.RP_SHALLOW_BATHY_FWAVE, [9.81, 1e-3], 3, 3, [4, 4, 4], (0.05, 0.04, 0.002)),
}
SINGLE_PASS = ("acoustics", "advection", "shallow")


def _classic_data(name, mx, my, mbc, seed, capa):
    """(q, aux, method[5], method[6]) on the padded grid; capa appends a capacity function to aux."""
    pad = (mx + 2 * mbc, my + 2 * mbc)
    rng = np.random.RandomState(seed)
    aux = None
    if name in ("acoustics", "advection", "euler", "shallow"):
        q = problems.random_state(name, pad, seed)
    elif name == "vc_acoustics":
        q = problems.random_state("acoustics", pad, seed)
        aux = np.stack([rng.choice([1.0, 4.0], pad), rng.choice([1.0, 0.5, 2.0], pad)])
    elif name == "vc_advection":
        q = problems.random_state("advection", pad, seed)
        aux = np.stack([rng.uniform(-1.0, 1.5, pad), rng.uniform(-1.2, 0.8, pad)])
    elif name == "psystem":
        from test_gpu_kernels import _elastic_data
        q, aux = _elastic_data(pad, seed=seed, law=1, ndim=2)
    else:
        from test_gpu_bathymetry import _data
        q, aux = _data(pad, seed)
    if capa:
        c = rng.uniform(0.5, 1.5, (1,) + pad)
        aux = c if aux is None else np.concatenate([aux, c])
    mcapa = aux.shape[0] if capa else 0
    return q, (None if aux is None else np.asfortranarray(aux)), mcapa, (0 if aux is None else aux.shape[0])


def _oracle_step2(name, mbc, mx, my, q, aux, method):
    rp_id, params, _, _, lim, (dx, dy, dt) = CLASSIC[name]
    qn = q.copy("F")
    if name == "bathymetry":
        import oracle_bathy as ob
        cfl = ob.step2(params, mbc, mx, my, q, qn, aux, dx, dy, dt, method, lim)
    else:
        cfl = po.step2_slabs(rp_id, params, mbc, mx, my, q, qn, aux, dx, dy, dt, method, lim, NTHREADS, False)
    return qn, cfl


def _oracle_step2ds(name, mbc, mx, my, q, aux, method, ids):
    rp_id, params, _, _, lim, (dx, dy, dt) = CLASSIC[name]
    qn = q.copy("F")
    if name == "bathymetry":
        import oracle_bathy as ob
        cfl = ob.step2ds(params, mbc, mx, my, q, qn, aux, dx, dy, dt, method, lim, ids)
    else:
        cfl = po.step2ds(rp_id, params, mbc, mx, my, q, qn, aux, dx, dy, dt, method, lim, ids)
    return qn, cfl


def _problem(name, mbc, mx, my, method, maux, rp_id=None):
    rid, params, meqn, mwaves, lim, (dx, dy, _) = CLASSIC[name]
    return _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rid if rp_id is None else rp_id, params, method,
                             lim, maux=maux)


def _device_step2(P, q, aux, dt, rows=None):
    """clawb200_step2 on device buffers, or clawb200_step2_rows over the given row ranges into one output"""
    qd, auxd, cfl = _dev(q), (None if aux is None else _dev(aux)), _cfl_dev()
    qn = qd.clone()
    if rows is None:
        _lib.call("clawb200_step2", ctypes.byref(P), _vp(qd), _vp(qn), _vp(auxd), dt, _vp(cfl), None)
    else:
        for jlo, jhi in rows:
            _lib.call("clawb200_step2_rows", ctypes.byref(P), _vp(qd), _vp(qn), _vp(auxd), dt, jlo, jhi, _vp(cfl), None)
    return _host(qn), cfl.item()


def _device_step2ds(P, q, aux, dt, ids):
    qd, auxd, cfl = _dev(q), (None if aux is None else _dev(aux)), _cfl_dev()
    qn = qd.clone()
    _lib.call("clawb200_step2ds", ctypes.byref(P), _vp(qd), _vp(qn), _vp(auxd), dt, ids, _vp(cfl), None)
    return _host(qn), cfl.item()


# =============================================================================================
# Unsplit step (trans = 2 unless stated): the two sweep kernels (step2_mode = 1), the capacity form,
# the single-pass kernel (step2_mode = 0) and the other transverse / order settings
# =============================================================================================
# (solver, step2_mode, capacity function, order, trans)
UNSPLIT = ([(name, 1, False, 2, 2) for name in CLASSIC] +
           [(name, 0, False, 2, 2) for name in SINGLE_PASS] +
           [(name, 1, True, 2, 2) for name in ("acoustics", "shallow", "vc_advection")] +
           [(name, 1, False, o, t) for name in ("euler", "shallow") for o, t in ((2, 1), (1, 2))])
UNSPLIT_SHAPES = [full_shapes(i) if not capa and o == 2 and t == 2 else light_shapes(i)
                  for i, (_, _, capa, o, t) in enumerate(UNSPLIT)]
UNSPLIT_CASES = [pytest.param(*fam, s, id="%s-mode%d%s-o%dt%d-%s" % (fam[0], fam[1], "-capa" if fam[2] else "",
                                                                      fam[3], fam[4], _id(s)))
                 for fam, shapes in zip(UNSPLIT, UNSPLIT_SHAPES) for s in shapes]


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode,capa,order,trans,shape", UNSPLIT_CASES)
def test_unsplit_step(name, mode, capa, order, trans, shape):
    mx, h, last = shape
    mbc = 2
    my = _nrows(mx, h, last)
    fused = mode == 0 and not capa
    assert set(step2_strips(mx, my, fused).values()) == {(h, last)}
    q, aux, mcapa, maux = _classic_data(name, mx, my, mbc, my + mx + order + trans, capa)
    method = [1, order, trans, 0, 0, mcapa, maux]
    qn_o, cfl_o = _oracle_step2(name, mbc, mx, my, q, aux, method)
    assert 0.0 < cfl_o and np.isfinite(qn_o[_inner(mbc)]).all()
    P = _problem(name, mbc, mx, my, method, maux)
    P.step2_mode = mode
    assert _lib.load().clawb200_step2_launches(ctypes.byref(P)) == (1 if fused else 2)
    qn_g, cfl_g = _device_step2(P, q, aux, CLASSIC[name][5][2])
    _same(qn_g[_inner(mbc)], qn_o[_inner(mbc)], "step2 %s %dx%d" % (name, mx, my))
    assert cfl_g == cfl_o


# =============================================================================================
# Dimensional splitting: both sweeps of step2ds, at mbc = 2 and (Euler, shallow water) mbc = 3
# =============================================================================================
DS = [(name, 2) for name in CLASSIC] + [("euler", 3), ("shallow", 3)]
DS_SHAPES = [light_shapes(i) for i in range(len(DS))]
DS_CASES = [pytest.param(name, mbc, s, id="%s-mbc%d-%s" % (name, mbc, _id(s)))
            for (name, mbc), shapes in zip(DS, DS_SHAPES) for s in shapes]


@pytest.mark.gpu
@pytest.mark.parametrize("name,mbc,shape", DS_CASES)
def test_step2ds(name, mbc, shape):
    """The shape's rows are the rows each sweep walks: my + 2 mbc padded rows for the x-sweeps, my for
    the y-sweeps."""
    mx, h, last = shape
    n = _nrows(mx, h, last)
    for ids in (1, 2):
        my = n - 2 * mbc if ids == 1 else n
        assert set(step2ds_strips(mx, my, mbc, ids).values()) == {(h, last)}
        q, aux, _, maux = _classic_data(name, mx, my, mbc, n + ids, False)
        method = [1, 2, -1, 0, 0, 0, maux]
        qn_o, cfl_o = _oracle_step2ds(name, mbc, mx, my, q, aux, method, ids)
        assert 0.0 < cfl_o
        P = _problem(name, mbc, mx, my, method, maux)
        qn_g, cfl_g = _device_step2ds(P, q, aux, CLASSIC[name][5][2], ids)
        # the sweep updates exactly the cells the oracle updates and copies the others
        _same(qn_g, qn_o, "step2ds %s ids=%d %dx%d" % (name, ids, mx, my))
        assert cfl_g == cfl_o


# =============================================================================================
# step2_rows in the overlapped multi-GPU decomposition (clawpack.py:233-244)
# =============================================================================================
ROWS = [("euler", 1), ("acoustics", 0), ("vc_acoustics", 1)]
ROWS_CASES = [pytest.param(name, mode, s, id="%s-mode%d-%s" % (name, mode, _id(s)))
              for i, (name, mode) in enumerate(ROWS) for s in light_shapes(i + 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode,shape", ROWS_CASES)
def test_step2_rows_overlapped_decomposition(name, mode, shape):
    """The interior rows 1 + mbc .. my - mbc, then the mbc boundary rows at each edge, into one output:
    the oracle's full step.  No strip of the interior launch starts at row 1."""
    mx, h, last = shape
    mbc = 2
    my = _nrows(mx, h, last) + 2 * mbc
    fused = mode == 0
    assert set(step2_strips(mx, my - 2 * mbc, fused).values()) == {(h, last)}
    q, aux, _, maux = _classic_data(name, mx, my, mbc, my + 3, False)
    method = [1, 2, 2, 0, 0, 0, maux]
    qn_o, cfl_o = _oracle_step2(name, mbc, mx, my, q, aux, method)
    P = _problem(name, mbc, mx, my, method, maux)
    P.step2_mode = mode
    qn_g, cfl_g = _device_step2(P, q, aux, CLASSIC[name][5][2],
                                rows=[(1 + mbc, my - mbc), (1, mbc), (my - mbc + 1, my)])
    _same(qn_g[_inner(mbc)], qn_o[_inner(mbc)], "step2_rows %s %dx%d" % (name, mx, my))
    assert cfl_g == cfl_o


# =============================================================================================
# Shallow water on the sphere: 16 aux components, capacity function, the four-row aux ring and the
# L1 prefetch of row k + 2
# =============================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(5, 64, 1), (5, 64, 63), (3, 128, 128)], ids=_id)
def test_sphere_step(shape):
    mx, h, last = shape
    mbc = 2
    my = _nrows(mx, h, last)
    assert set(step2_strips(mx, my, False).values()) == {(h, last)}
    pb = problems.sphere_problem(mx, my)
    dx, dy = pb["d"]
    aux = pb["auxbc_full"]
    qbc = np.zeros((4, mx + 2 * mbc, my + 2 * mbc), order="F")
    qbc[_inner(mbc)] = pb["q"]
    del pb
    po.fill_bcs(qbc, mbc, [po.BC_PERIODIC, po.BC_CUSTOM], [po.BC_PERIODIC, po.BC_CUSTOM],
                problems.sphere_qbc_lower_y, problems.sphere_qbc_upper_y)
    method, lim = [1, 2, 2, 0, 0, 1, 16], [4, 4, 4]
    dt = 0.01 * min(dx, dy)
    qn_o = qbc.copy("F")
    cfl_o = po.step2_slabs(po.RP_SPHERE, [problems.SPHERE_G], mbc, mx, my, qbc, qn_o, aux, dx, dy, dt, method, lim,
                           NTHREADS, False)
    assert 0.0 < cfl_o < 1.0 and np.isfinite(qn_o[_inner(mbc)]).all()
    P = _lib.make_problem(2, 4, 3, mbc, mx, my, dx, dy, _lib.RP_SPHERE, [problems.SPHERE_G], method, lim, maux=16)
    qn_g, cfl_g = _device_step2(P, qbc, aux, dt)
    _same(qn_g[_inner(mbc)], qn_o[_inner(mbc)], "sphere %dx%d" % (mx, my))
    assert cfl_g == cfl_o


# =============================================================================================
# A user Riemann solver (examples/user_rp/rp_advection_user.cuh) at 64-row strips
# =============================================================================================
@pytest.mark.gpu
def test_user_solver_at_tall_strips():
    """The header restates the built-in advection solver: the unsplit step and both step2ds sweeps
    equal the built-in solver and the oracle bit for bit."""
    import pyclaw
    hdr = os.path.join(ROOT, "examples", "user_rp", "rp_advection_user.cuh")
    rs = pyclaw.riemann.from_header(hdr, name="advuser", meqn=1, mwaves=1, ndims=(1, 2), param_names=["u", "v"])
    mx, h, last = 5, 64, 63
    mbc = 2
    my = _nrows(mx, h, last)
    assert set(step2_strips(mx, my, False).values()) == {(h, last)}
    assert step2ds_strips(mx, my, mbc, 2) == {"y": (h, last)}
    dt = CLASSIC["advection"][5][2]
    q, _, _, _ = _classic_data("advection", mx, my, mbc, 17, False)
    for method, ids in (([1, 2, 2, 0, 0, 0, 0], None), ([1, 2, -1, 0, 0, 0, 0], 1), ([1, 2, -1, 0, 0, 0, 0], 2)):
        out = []
        for rp_id, variant in ((_lib.RP_ADVECTION, "strict"), (_lib.RP_USER, rs._variant())):
            prev = _lib.set_variant(variant)
            try:
                P = _problem("advection", mbc, mx, my, method, 0, rp_id=rp_id)
                P.step2_mode = 1
                out.append(_device_step2(P, q, None, dt) if ids is None else _device_step2ds(P, q, None, dt, ids))
            finally:
                _lib.set_variant(prev)
        if ids is None:
            ref, cfl_o = _oracle_step2("advection", mbc, mx, my, q, None, method)
            sl = _inner(mbc)
        else:
            ref, cfl_o = _oracle_step2ds("advection", mbc, mx, my, q, None, method, ids)
            sl = (slice(None),) * 3
        for got, cfl_g in out:
            _same(got[sl], ref[sl], "user advection %s" % (ids,))
            assert cfl_g == cfl_o
        assert np.abs(ref[sl] - q[sl]).max() > 1e-3


# =============================================================================================
# SharpClaw 2-D stage
# =============================================================================================
# (solver, reconstruction, aux kind): aux kind "vc" reads {impedance, sound speed}, "capa" is a
# capacity function (aux component 2)
SC2 = ([(name, v, None) for name in ("acoustics", "euler", "shallow") for v in (0, 1, 2)] +
       [("euler", "tvd2", None), ("acoustics", "weno7", None), ("shallow", "weno11", None),
        ("vc_acoustics", 0, "vc"), ("acoustics", 0, "capa"), ("advection", 2, "capa")])
SC2_SHAPES = [full_shapes(i, tall128=False)[:9] + [full_shapes(i, tall128=False)[9 + i % 3]]
              for i in range(len(SC2))]
SC2_CASES = [pytest.param(*fam, s, id="%s-%s%s-%s" % (fam[0], fam[1], "-" + fam[2] if fam[2] else "", _id(s)))
             for fam, shapes in zip(SC2, SC2_SHAPES) for s in shapes]
SC_RPS = {"acoustics": (1, [1.0, 4.0, 2.0, 2.0], 3, 2), "advection": (2, [0.7, -0.4], 1, 1),
          "euler": (3, [1.4, 0.4], 5, 5), "shallow": (4, [1.0], 3, 3), "vc_acoustics": (po.RP_VC_ACOUSTICS, [], 3, 2)}


@pytest.mark.gpu
@pytest.mark.parametrize("name,recon,auxkind,shape", SC2_CASES)
def test_sharpclaw_stage2(name, recon, auxkind, shape):
    """DQ_ONLY with dq_out, then one combining stage mode (rotating with the shape) against the same dq."""
    import torch
    mx, h, last = shape
    my = _nrows(mx, h, last)
    assert strip(my, ctas_sc(mx), False) == (h, last)
    rp_id, params, meqn, mwaves = SC_RPS[name]
    dx, dy, dt = 0.01, 0.013, 0.0011
    seed = my + mx + len(str(recon))
    variant, mbc, mthlim, tab_dev = recon, 3, None, None
    if recon == "tvd2":
        variant, mthlim = po.RECON_TVD2, [1, 2, 4, 5, 4][:meqn]
        po.set_tvd_limiters(mthlim)
    elif isinstance(recon, str):          # weno7 / weno11: the table-driven kernel
        from pyclaw_b200.weno_tables import tables
        k = (int(recon[4:]) + 1) // 2
        variant, mbc = po.WENO_TABLES, k
        tab = tables(k, "f32")
        po.set_weno_tables(tab)
        tab_dev = torch.from_numpy(_lib.pack_weno_tables(tab)).cuda()
    pad = (mx + 2 * mbc, my + 2 * mbc)
    q = problems.smooth_state("acoustics" if name == "vc_acoustics" else name, pad, seed)
    aux, maux, mcapa = None, 0, 0
    rng = np.random.RandomState(seed)
    if auxkind == "vc":
        aux = np.asfortranarray(np.stack([rng.choice([1.0, 4.0], pad), rng.choice([1.0, 2.0], pad)]))
        maux = 2
    elif auxkind == "capa":
        aux = np.asfortranarray(rng.uniform(0.5, 1.5, (2,) + pad))
        maux, mcapa = 2, 2
    if aux is not None:
        dq_o, cfl_o = po.sc_flux2(rp_id, params, mwaves, mbc, mx, my, q, dx, dy, dt, variant, auxbc=aux, mcapa=mcapa)
    else:
        dq_o, cfl_o = po.sc_flux2(rp_id, params, mwaves, mbc, mx, my, q, dx, dy, dt, variant, NTHREADS)
    inner = _inner(mbc)
    assert np.isfinite(dq_o[inner]).all() and np.abs(dq_o[inner]).max() > 1e-6 and cfl_o > 0
    P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, method=[1, 2, 0, 0, 0, mcapa, maux],
                          mthlim=mthlim, maux=maux, weno_variant=variant)
    if tab_dev is not None:
        P.weno_k, P.weno_tab = mbc, tab_dev.data_ptr()
    qd, auxd = _dev(q), (None if aux is None else _dev(aux))
    cfl = _cfl_dev()
    dqd = torch.zeros_like(qd)
    _lib.call("clawb200_sharpclaw_stage", ctypes.byref(P), _vp(qd), None, None, _vp(dqd), _vp(auxd), dt,
              _lib.STAGE_DQ_ONLY, 0.0, 0.0, 1.0, _vp(cfl), None)
    _same(_host(dqd)[inner], dq_o[inner], "sharpclaw dq %s %s %dx%d" % (name, recon, mx, my))
    assert cfl.item() == cfl_o
    # one combining mode, out = f(q, qa, dq)
    mode = (_lib.STAGE_AXPY, _lib.STAGE_CONVEX, _lib.STAGE_FINAL104)[(my + mx) % 3]
    qa = problems.smooth_state("acoustics" if name == "vc_acoustics" else name, pad, seed + 1)
    ca, cb, div = {0: (0.0, 0.0, 6.0), 1: (0.75, 0.25, 1.0), 2: (0.6, 0.1, 1.0)}[mode]
    expect = {0: lambda: q + dq_o / div, 1: lambda: ca * qa + cb * (q + dq_o), 2: lambda: (qa + ca * q) + cb * dq_o}[mode]()
    qad, out = _dev(qa), torch.zeros_like(qd)
    cfl.zero_()
    _lib.call("clawb200_sharpclaw_stage", ctypes.byref(P), _vp(qd), _vp(qad), _vp(out), None, _vp(auxd), dt, mode,
              ca, cb, div, _vp(cfl), None)
    _same(_host(out)[inner], expect[inner], "sharpclaw stage mode %d %s %s" % (mode, name, recon))
    assert cfl.item() == cfl_o


# =============================================================================================
# SharpClaw 3-D stage: the x/y kernel (plane by plane) and the z kernel
# =============================================================================================
def sc3_strips(mx, my, mz):
    return {"xy": strip(my, ctas_sc(mx) * (mz + 2), False), "z": strip(mz, ctas_sc3_z(mx, my), False)}


# ((mx, my, mz), (kernel, h, last)): the x/y kernel needs tall y with mx = 5, mz = 6 (eight planes of
# one CTA), the z kernel tall z with mx = my = 3 (one CTA of (i, j) columns)
SC3_XY = [((5, rows_for(h, last, 8), 6), ("xy", h, last)) for h in (16, 32, 64) for last in (1, h - 1, h)]
SC3_Z = [((3, 3, rows_for(h, last, 1)), ("z", h, last)) for h in (16, 32, 64) for last in (1, h - 1, h)]
SC3_SOLVERS = ["advection", "euler", "acoustics", "fwave"]


def _sc3_cases():
    out = []
    for i, name in enumerate(SC3_SOLVERS):
        shapes = SC3_XY + SC3_Z
        if name in ("euler", "acoustics"):
            # the larger z grids (3.1 M cells) on the one-component solvers only
            shapes = [s for s in shapes if s[1][0] == "xy" or s[1][1] < 64 or s[1][2] == _last(64, i)]
        out += [pytest.param(name, shape, exp, id="%s-%s%d-last%d" % ((name,) + exp)) for shape, exp in shapes]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name,shape,expect", _sc3_cases())
def test_sharpclaw_stage3(name, shape, expect):
    import torch
    import oracle3d as o3
    mx, my, mz = shape
    kern, h, last = expect
    assert sc3_strips(mx, my, mz)[kern] == (h, last)
    mbc = 3
    pad = tuple(n + 2 * mbc for n in shape)
    rng = np.random.RandomState(sum(shape))
    aux = None
    if name == "advection":
        rp_id, params, meqn, mwaves, lim = o3.RP_ADVECTION3D, [0.7, -0.45, 0.3], 1, 1, [4]
        q = rng.uniform(-1, 1, (1,) + pad)
    elif name == "fwave":
        rp_id, params, meqn, mwaves, lim = o3.RP_ADVECTION3D_VC_FWAVE, [], 1, 1, [4]
        q = rng.uniform(-1, 1, (1,) + pad)
        aux = np.asfortranarray(rng.uniform(-1.5, 1.5, (3,) + pad))
    elif name == "acoustics":
        rp_id, params, meqn, mwaves, lim = o3.RP_ACOUSTICS3D_VC, [], 4, 2, [1, 2, 3, 4]
        q = rng.uniform(-1, 1, (4,) + pad)
        rho, c = rng.choice([1.0, 3.0], pad), rng.choice([1.0, 0.5], pad)
        aux = np.asfortranarray(np.stack([rho * c, c]))
    else:
        rp_id, params, meqn, mwaves, lim = o3.RP_EULER3D, [1.4, 0.4], 5, 3, [1, 2, 3, 4, 5]
        # milder than white noise over [0.5, 2]: on millions of cells WENO5 overshoots of that data
        # reach negative pressures, and the oracle's dq has NaNs
        rho = rng.uniform(0.8, 1.25, pad)
        u = rng.uniform(-0.5, 0.5, (3,) + pad)
        p = rng.uniform(0.8, 1.25, pad)
        q = np.concatenate([rho[None], rho * u, (p / 0.4 + 0.5 * rho * (u * u).sum(0))[None]])
        del rho, u, p
    q = np.asfortranarray(q)
    maux = 0 if aux is None else aux.shape[0]
    dx, dy, dz, dt = 0.02, 0.025, 0.03, 0.004
    variant = (o3.WENO_PYWENO_F32, o3.WENO_PYWENO_F64, o3.WENO_OLD)[(mx + my + mz) % 3]
    dq_o, cfl_o = o3.sc_flux3(rp_id, params, mwaves, mbc, mx, my, mz, q, dx, dy, dz, dt, variant, aux=aux, mthlim=lim)
    assert np.isfinite(dq_o).all() and cfl_o > 0.01 and np.abs(dq_o).max() > 1e-3
    P = _lib.make_problem(3, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, [1, 2, 0, 0, 0, 0, maux], lim[:mwaves],
                          maux=maux, weno_variant=variant)
    P.pitch, P.mstride = pad[0], pad[0] * pad[1] * pad[2]
    qd, auxd = _dev(q), (None if aux is None else _dev(aux))
    cfl = _cfl_dev()
    inner = _inner(mbc, 3)
    # DQ_ONLY into dq_out, then the SSP104 final combination into out with the x/y partial in dq_out
    dqd = torch.zeros_like(qd)
    _lib.call("clawb200_sharpclaw_stage3", ctypes.byref(P), mz, dz, _vp(qd), None, None, _vp(dqd), _vp(auxd), dt,
              _lib.STAGE_DQ_ONLY, 0.0, 0.0, 1.0, _vp(cfl), None)
    _same(_host(dqd)[inner], dq_o[inner], "sharpclaw3 dq %s %s" % (name, shape))
    assert cfl.item() == cfl_o
    del dqd
    qa = np.asfortranarray(q[:, ::-1])
    qad, out, part = _dev(qa), torch.zeros_like(qd), torch.zeros_like(qd)
    cfl.zero_()
    _lib.call("clawb200_sharpclaw_stage3", ctypes.byref(P), mz, dz, _vp(qd), _vp(qad), _vp(out), _vp(part), _vp(auxd),
              dt, _lib.STAGE_FINAL104, 0.6, 0.1, 1.0, _vp(cfl), None)
    _same(_host(out)[inner], ((qa + 0.6 * q) + 0.1 * dq_o)[inner], "sharpclaw3 stage %s %s" % (name, shape))
    assert cfl.item() == cfl_o


# =============================================================================================
# The fma build at 64- and 128-row strips
# =============================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("kernel,shape", [("sweeps", (5, 64, 1)), ("sweeps", (3, 128, 127)),
                                          ("single-pass", (251, 64, 64)), ("single-pass", (3, 128, 1)),
                                          ("sharpclaw", (5, 64, 63)), ("sharpclaw", (251, 64, 1))],
                         ids=lambda v: v if isinstance(v, str) else _id(v))
def test_fma_build_at_tall_strips(kernel, shape):
    """The unsplit step (Euler, two sweep kernels), the single-pass kernel (shallow water) and the
    SharpClaw 2-D stage (shallow water, WENO5 f32) on the fma build, within test_gpu_fma_build's bounds.

    The SharpClaw dq of a tall narrow grid is smooth along y apart from 1 % noise, and its WENO weights
    turn last-bit differences into a larger share of dq than on the square grids of test_gpu_fma_build
    (measured on a B200: 1.2e-13 of max |dq|).  As there for ill-conditioned data, it is held to twice
    the strict build's own response to a 1-ulp change of its input, or 1e-13, whichever is larger."""
    import torch
    from test_gpu_fma_build import TOL, _close
    mx, h, last = shape
    name = "euler" if kernel == "sweeps" else "shallow"
    my = _nrows(mx, h, last)
    tol = TOL
    if kernel == "sharpclaw":
        assert strip(my, ctas_sc(mx), False) == (h, last)
        rp_id, params, meqn, mwaves = SC_RPS[name]
        mbc, dx, dy, dt = 3, 0.01, 0.013, 0.0011
        q = problems.smooth_state(name, (mx + 2 * mbc, my + 2 * mbc), my)
        ref, cfl_o = po.sc_flux2(rp_id, params, mwaves, mbc, mx, my, q, dx, dy, dt, 0, NTHREADS)
        P = _lib.make_problem(2, meqn, mwaves, mbc, mx, my, dx, dy, rp_id, params, weno_variant=0)

        def dq(variant, qh):
            prev = _lib.set_variant(variant)
            try:
                qd, cfl = _dev(qh), _cfl_dev()
                dqd = torch.zeros_like(qd)
                _lib.call("clawb200_sharpclaw_stage", ctypes.byref(P), _vp(qd), None, None, _vp(dqd), None, dt,
                          _lib.STAGE_DQ_ONLY, 0.0, 0.0, 1.0, _vp(cfl), None)
                return _host(dqd), cfl.item()
            finally:
                _lib.set_variant(prev)
        qp = q.copy("F")
        qp[:, ::2, ::2] *= 1.0 + 2.0 ** -52
        pert, _ = dq("strict", qp)
        cond = _close("sharpclaw strict, 1-ulp input perturbation %dx%d" % (mx, my), pert[_inner(mbc)],
                      ref[_inner(mbc)], tol=np.inf)
        tol = max(TOL, 2.0 * cond)
        got, cfl_g = dq("fma", q)
    else:
        fused = kernel == "single-pass"
        assert set(step2_strips(mx, my, fused).values()) == {(h, last)}
        mbc = 2
        q, _, _, _ = _classic_data(name, mx, my, mbc, my, False)
        method = [1, 2, 2, 0, 0, 0, 0]
        ref, cfl_o = _oracle_step2(name, mbc, mx, my, q, None, method)
        P = _problem(name, mbc, mx, my, method, 0)
        P.step2_mode = 0 if fused else 1
        prev = _lib.set_variant("fma")
        try:
            assert _lib.load().clawb200_step2_launches(ctypes.byref(P)) == (1 if fused else 2)
            got, cfl_g = _device_step2(P, q, None, CLASSIC[name][5][2])
        finally:
            _lib.set_variant(prev)
    inner = _inner(mbc)
    _close("%s %dx%d" % (kernel, mx, my), got[inner], ref[inner], cfl_g, cfl_o, tol=tol)


# =============================================================================================
# Whole runs through import pyclaw on a tall narrow grid: CUDA-graph replay and the BC kernels
# =============================================================================================
def _tall_state(pyclaw, q0, d):
    x = pyclaw.Dimension('x', 0.0, d[0] * q0.shape[1], q0.shape[1])
    y = pyclaw.Dimension('y', 0.0, d[1] * q0.shape[2], q0.shape[2])
    state = pyclaw.State(pyclaw.Grid([x, y]), q0.shape[0])
    state.q[...] = q0
    return state


def _controller(pyclaw, state, solver, tfinal):
    claw = pyclaw.Controller()
    claw.tfinal, claw.nout, claw.keep_copy, claw.output_format = tfinal, 1, True, None
    claw.solution, claw.solver = pyclaw.Solution(state), solver
    claw.run()
    return np.asarray(claw.frames[-1].q)


@pytest.mark.gpu
def test_classic_euler_unsplit_run_on_a_tall_grid():
    import pyclaw
    mx, h, last = 5, 64, 63
    my = _nrows(mx, h, last)
    assert set(step2_strips(mx, my, False).values()) == {(h, last)}
    q0 = problems.smooth_state("euler", (mx, my), seed=3)
    d = [0.01, 0.013]
    tfinal = 0.02
    state = _tall_state(pyclaw, q0, d)
    state.aux_global.update(gamma=1.4, gamma1=0.4)
    solver = pyclaw.ClawSolver2D()
    solver.mwaves = 5
    solver.limiters = [4, 4, 4, 4, 2]
    solver.dim_split, solver.order_trans = False, 2
    solver.cfl_max, solver.cfl_desired = 0.5, 0.45
    solver.dt_initial = 0.002
    solver.bc_lower[0], solver.bc_upper[0] = pyclaw.BC.outflow, pyclaw.BC.reflecting
    solver.bc_lower[1] = solver.bc_upper[1] = pyclaw.BC.periodic
    assert solver.use_cuda_graph
    got = _controller(pyclaw, state, solver, tfinal)
    s = po.OracleSolver("classic", 2, po.RP_EULER5, [1.4, 0.4], 5)
    s.limiters = [4, 4, 4, 4, 2]
    s.dim_split, s.order_trans = False, 2
    s.cfl_max, s.cfl_desired = 0.5, 0.45
    s.dt_initial = 0.002
    s.bc_lower, s.bc_upper = [po.BC_OUTFLOW, po.BC_PERIODIC], [po.BC_REFLECTING, po.BC_PERIODIC]
    s.nthreads = NTHREADS
    ref = s.run(q0, None, d, tfinal, 1)[-1]
    assert s.total["numsteps"] >= 3 and np.isfinite(ref).all()
    _same(got, ref, "ClawSolver2D Euler %dx%d" % (mx, my))


@pytest.mark.gpu
def test_sharpclaw_shallow_ssp104_run_on_a_tall_grid():
    import pyclaw
    mx, h, last = 5, 64, 1
    my = _nrows(mx, h, last)
    assert strip(my, ctas_sc(mx), False) == (h, last)
    q0 = problems.smooth_state("shallow", (mx, my), seed=4)
    q0[1:] *= 0.25        # subcritical flow: |u|, |v| <= 0.4 < sqrt(g h)
    d = [0.01, 0.013]
    tfinal = 0.03
    state = _tall_state(pyclaw, q0, d)
    state.aux_global['grav'] = 1.0
    solver = pyclaw.SharpClawSolver2D()
    solver.mwaves = 3
    solver.time_integrator = 'SSP104'
    solver.cfl_max, solver.cfl_desired = 1.3, 1.2
    solver.dt_initial = 0.005
    solver.bc_lower[0], solver.bc_upper[0] = pyclaw.BC.outflow, pyclaw.BC.reflecting
    solver.bc_lower[1] = solver.bc_upper[1] = pyclaw.BC.periodic
    got = _controller(pyclaw, state, solver, tfinal)
    s = po.OracleSolver("sharpclaw", 2, po.RP_SHALLOW, [1.0], 3)
    s.time_integrator = "SSP104"
    s.cfl_max, s.cfl_desired = 1.3, 1.2
    s.dt_initial = 0.005
    s.bc_lower, s.bc_upper = [po.BC_OUTFLOW, po.BC_PERIODIC], [po.BC_REFLECTING, po.BC_PERIODIC]
    s.nthreads = NTHREADS
    ref = s.run(q0, None, d, tfinal, 1)[-1]
    assert s.total["numsteps"] >= 3 and np.isfinite(ref).all()
    _same(got, ref, "SharpClawSolver2D SSP104 %dx%d" % (mx, my))
