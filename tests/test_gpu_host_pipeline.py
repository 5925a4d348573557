"""
The slab pipeline of the host-array entry points, at every slab partition.

clawb200_step2_host and clawb200_step2ds_host take the reference's Fortran-ordered host arrays (the
f2py-shaped calls of INTEGRATION.md path B, pyclaw_b200/f2py_shim.py, and bench.py's e2e figure).
A grid with my >= 1024, no aux, no capacity function and not the sphere solver is not swept in one
piece: host_pipeline (pyclaw_b200/csrc/clawb200.cu) cuts its output rows into slabs of about 128 rows
and uploads, sweeps and downloads each slab as a stand-alone padded problem on three streams.  The
result must equal the single pass bit for bit at every size.

The partition is restated below.  The CPU tests check that every slab of every height up to 70 000
rows is a valid padded problem and that the slabs tile the output rows.  The GPU tests compare the
entry points with the CPU oracle, Courant number included, at the heights where the partition's
arithmetic has its edges: the last height of the direct path and the first pipelined one, slabs that
divide evenly, the heights at which a partition into slabs of ceil(rows / nslab) rows plus a remainder
leaves a last x-sweep slab of 1, 2, 2 mbc or 2 mbc + 1 rows (the pipeline cut such slabs once; a slab
of 2 mbc rows or fewer has no interior row and its x-sweep ran into the next component), and
my = 16384.  Before each pipelined call, one call of the same entry point on a NaN grid of the same
shape leaves NaN in every slab buffer and in the Courant slot, so that a read outside a slab shows
up as NaN rather than as a stale but plausible value.
"""
import ctypes
import threading

import numpy as np
import pytest

import problems
from oracle import pyclaw_oracle as po
from pyclaw_b200 import _lib
from test_gpu_kernels import RPS

# =============================================================================================
# The partition, restated.  If host_pipeline changes, this copy changes with it.
# =============================================================================================
SLAB_ROWS = 128          # clawb200.cu:864
PIPELINE_MIN_MY = 1024   # clawb200.cu:995, :1021 (and no aux, no capacity function, not the sphere)


def partition(mode, my, mbc):
    """host_pipeline, clawb200.cu:859-892, for an array of heights my: one row per height, one column
    per slab k < the largest nslab (`live` marks the slabs a height has).  mode 0 = step2_host,
    1 = step2ds_host ids 1 (x-sweeps over every padded row), 2 = ids 2.  Rows are 0-based padded
    rows: slab k reads the host rows [in0, in1) and writes back [r0, r1); its problem has P.my = `my`
    and P.mstride = nx * `rows`; each slab buffer holds `nmax_rows` padded rows."""
    my = np.atleast_1d(np.asarray(my, dtype=np.int64))[:, None]
    out0 = np.zeros_like(my) if mode == 1 else np.full_like(my, mbc)
    out1 = my + 2 * mbc if mode == 1 else my + mbc
    halo = 0 if mode == 1 else mbc
    nout = out1 - out0
    nslab = np.maximum(1, -(-nout // SLAB_ROWS))
    k = np.arange(int(nslab.max()))[None, :]
    r0, r1 = out0 + k * nout // nslab, out0 + (k + 1) * nout // nslab
    in0, in1 = r0 - halo, r1 + halo
    return dict(out0=out0[:, 0], out1=out1[:, 0], halo=halo, nslab=nslab[:, 0], live=k < nslab,
                r0=r0, r1=r1, in0=in0, in1=in1, my=(in1 - in0 - 2 * mbc) if mode == 1 else r1 - r0,
                rows=in1 - in0, nmax_rows=(-(-nout // nslab) + 2 * mbc)[:, 0])


def slabs(mode, my, mbc):
    """[(r0, r1, in0, in1, P.my, P.mstride / nx)] of one height"""
    p = partition(mode, my, mbc)
    return [tuple(int(p[f][0, k]) for f in ("r0", "r1", "in0", "in1", "my", "rows")) for k in range(p["nslab"][0])]


def ceil_last_rows(nout):
    """Rows of the last slab when nout rows are cut into slabs of ceil(nout / nslab) rows from the
    top and the last slab takes the remainder: the heights at which this leaves a mode-1 slab of
    2 mbc rows or fewer are the heights the GPU cases below single out."""
    nslab = -(-nout // SLAB_ROWS)
    return nout - (nslab - 1) * -(-nout // nslab)


def case_heights(mbc):
    """The heights the GPU cases run, by class."""
    def first(pred):
        my = PIPELINE_MIN_MY
        while not pred(my):
            my += 1
        return my
    h = {"direct": PIPELINE_MIN_MY - 1, "first": PIPELINE_MIN_MY,
         "full-x": first(lambda my: my > PIPELINE_MIN_MY and (my + 2 * mbc) % SLAB_ROWS == 0)}
    for last in (1, 2, 2 * mbc, 2 * mbc + 1):
        h["ceil-last%d" % last] = first(lambda my: ceil_last_rows(my + 2 * mbc) == last)
    h["16384"] = 16384
    return h


# =============================================================================================
# The partition copy on its own (no GPU)
# =============================================================================================
def test_partition_copy_gives_the_known_partitions():
    """1500 rows (test_host_slab_pipeline) in 12 slabs of 125, and 8192^2 (bench.py's e2e) in 64 of 128."""
    p = partition(0, 1500, 2)
    assert p["nslab"][0] == 12 and p["nmax_rows"][0] == 129
    assert [s[:2] for s in slabs(0, 1500, 2)] == [(2 + 125 * k, 2 + 125 * (k + 1)) for k in range(12)]
    p = partition(0, 8192, 2)
    assert p["nslab"][0] == 64 and p["nmax_rows"][0] == 132
    assert slabs(0, 8192, 2) == [(2 + 128 * k, 130 + 128 * k, 128 * k, 132 + 128 * k, 128, 132) for k in range(64)]
    # the x-sweep of 16384 rows: 16388 padded rows in 129 slabs of 127 or 128 rows
    s = slabs(1, 16384, 2)
    assert len(s) == 129 and {r1 - r0 for r0, r1, *_ in s} == {127, 128} and s[-1][1] == 16388


@pytest.mark.parametrize("mbc", [2, 3, 4])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_every_slab_is_a_valid_padded_problem(mode, mbc):
    """Every height the pipeline takes up to 70 000 rows: each slab has P.my >= 1 and as many rows as
    P.my plus its ghost rows, reads inside the padded grid, fits the slab buffers, has 64 .. 128 output
    rows, and the slabs tile the output rows exactly once."""
    for lo in range(PIPELINE_MIN_MY, 70000, 2048):
        my = np.arange(lo, min(lo + 2048, 70000))
        p = partition(mode, my, mbc)
        live = p["live"]
        ny = (my + 2 * mbc)[:, None]
        n = p["r1"] - p["r0"]
        assert (p["my"][live] >= 1).all()
        assert (p["rows"] == p["my"] + 2 * mbc)[live].all()
        assert ((p["in0"] >= 0) & (p["in1"] <= ny))[live].all()
        assert (p["rows"] <= p["nmax_rows"][:, None])[live].all()
        assert ((n >= 64) & (n <= SLAB_ROWS))[live].all()
        # tiling: the first slab starts at out0, each next one where the previous one ends, the last
        # one ends at out1
        assert (p["r0"][:, 0] == p["out0"]).all()
        nxt = live[:, 1:]
        assert (p["r0"][:, 1:] == p["r1"][:, :-1])[nxt].all()
        assert (p["r1"][np.arange(len(my)), p["nslab"] - 1] == p["out1"]).all()


def test_ceil_partition_heights():
    """The heights at which slabs of ceil(rows / nslab) rows leave a last x-sweep slab without an interior
    row: the first one for each mbc and how many there are below 70 000 rows for mbc = 2 and 3."""
    my = np.arange(PIPELINE_MIN_MY, 70000)
    short = {mbc: my[ceil_last_rows(my + 2 * mbc) <= 2 * mbc] for mbc in (2, 3, 4)}
    assert [int(short[mbc][0]) for mbc in (2, 3, 4)] == [15872, 15616, 15360]
    assert len(short[2]) + len(short[3]) == 4221
    assert 16384 in short[2]


# The GPU matrix.  Narrow grids keep every case cheap (mx = 3 or 5, one column tile of every kernel);
# a few cases run mx = 251, which has two or three.  The order rotates over the heights of a solver.
WIDE_DS = {("euler", 2, "first"), ("acoustics", 2, "ceil-last1"), ("shallow", 3, "full-x")}
WIDE_UNSPLIT = {("euler", 3, "first"), ("shallow", 2, "ceil-last2")}
ORDER_TRANS = [(2, 2), (1, 1), (2, 1), (1, 2)]


def _cases(wide, unsplit):
    out = []
    for mbc in (2, 3):
        for i, (cls, my) in enumerate(case_heights(mbc).items()):
            for j, name in enumerate(RPS):
                mx = 251 if (name, mbc, cls) in wide else (3, 5)[(i + j) % 2]
                order, trans = ORDER_TRANS[(i + j + mbc) % 4]
                out.append(pytest.param(name, mbc, cls, my, mx, order, *((trans,) if unsplit else ()),
                                        id="%s-mbc%d-%s-%dx%d-o%d%s" % (name, mbc, cls, mx, my, order,
                                                                      "t%d" % trans if unsplit else "")))
    return out


DS_CASES = _cases(WIDE_DS, False)
UNSPLIT_CASES = _cases(WIDE_UNSPLIT, True)


def test_gpu_matrix_covers_every_class():
    """For mbc = 2 and 3, every solver of RPS in step2ds_host and step2_host, each at both orders and at
    every class of height: the last direct height, the first pipelined one, all slabs of 128 rows in
    each mode, a ceil-partition last slab of 1, 2, 2 mbc and 2 mbc + 1 x-sweep rows, and 16384."""
    for cases, modes in ((DS_CASES, (1, 2)), (UNSPLIT_CASES, (0,))):
        for mbc in (2, 3):
            for name in RPS:
                mine = [c.values for c in cases if c.values[0] == name and c.values[1] == mbc]
                heights = [v[3] for v in mine]
                assert {v[5] for v in mine} == {1, 2}
                assert PIPELINE_MIN_MY - 1 in heights and PIPELINE_MIN_MY in heights and 16384 in heights
                for last in (1, 2, 2 * mbc, 2 * mbc + 1):
                    assert any(ceil_last_rows(my + 2 * mbc) == last for my in heights), (name, mbc, last)
                for mode in modes:
                    assert any({s[1] - s[0] for s in slabs(mode, my, mbc)} == {SLAB_ROWS}
                               for my in heights if my >= PIPELINE_MIN_MY), (name, mbc, mode)
            if modes == (0,):
                assert {v[6] for v in (c.values for c in cases) if v[1] == mbc} == {1, 2}
    assert {c.values[4] for c in DS_CASES} == {3, 5, 251} and {c.values[4] for c in UNSPLIT_CASES} == {3, 5, 251}


# =============================================================================================
# Device harness
# =============================================================================================
DX, DY, DT = 0.01, 0.013, 0.0011


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _problem(name, mbc, mx, my, method):
    rp_id, params, meqn, mwaves, lim = RPS[name]
    return _lib.make_problem(2, meqn, mwaves, mbc, mx, my, DX, DY, rp_id, params, method, lim)


def _poison(P, shape, ids=None):
    """One call of the same entry point on a NaN grid of the same shape: it leaves NaN in every slab
    buffer (or, below 1024 rows, in the direct path's buffers) and in the Courant slot."""
    nan = np.full(shape, np.nan, order="F")
    _call(P, nan, nan, ids)


def _call(P, qold, qnew, ids=None):
    """step2ds_host (ids 1 or 2) or step2_host (ids None); qnew may be qold"""
    cfl = ctypes.c_double()
    if ids is None:
        _lib.call("clawb200_step2_host", ctypes.byref(P), _ptr(qold), _ptr(qnew), None, DT, ctypes.byref(cfl))
    else:
        _lib.call("clawb200_step2ds_host", ctypes.byref(P), _ptr(qold), _ptr(qnew), None, DT, ids, ctypes.byref(cfl))
    return cfl.value


def _oracle(name, mbc, mx, my, q, method, ids=None, qnew=None):
    rp_id, params, _, _, lim = RPS[name]
    qn = q.copy("F") if qnew is None else qnew
    if ids is None:
        cfl = po.step2(rp_id, params, mbc, mx, my, q, qn, None, DX, DY, DT, method, lim)
    else:
        cfl = po.step2ds(rp_id, params, mbc, mx, my, q, qn, None, DX, DY, DT, method, lim, ids)
    return qn, cfl


def _rows(js):
    js = [int(j) for j in js]
    return "%s (%d rows)" % (js if len(js) <= 8 else js[:4] + ["..."] + js[-4:], len(js))


def _check(what, got, ref, cfl_g, cfl_o, mbc, j0=0):
    """Bit for bit, Courant number included; the message names each component that differs and its
    rows as Fortran j (1 .. my interior).  j0 is the padded row of got[:, :, 0]."""
    bad = []
    for m in range(ref.shape[0]):
        eq = (got[m] == ref[m]).all(axis=0)
        if not eq.all():
            d = np.abs(got[m] - ref[m])
            bad.append("component %d differs in rows j = %s, max |diff| %g, %d NaN"
                       % (m, _rows(np.nonzero(~eq)[0] + j0 - mbc + 1), np.nanmax(d), np.isnan(d).sum()))
    if cfl_g != cfl_o:
        bad.append("Courant number %r, oracle %r" % (cfl_g, cfl_o))
    assert not bad, "%s: %s" % (what, "; ".join(bad))


def _data(name, mbc, mx, my, seed):
    return problems.random_state(name, (mx + 2 * mbc, my + 2 * mbc), seed)


# =============================================================================================
# Parity with the oracle at every class of height
# =============================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("name,mbc,cls,my,mx,order", DS_CASES)
def test_step2ds_host(name, mbc, cls, my, mx, order):
    """ids 1 and ids 2, each with qnew a copy of qold and with qnew the same array as qold, then the
    reference's pair (clawpack.py:538-548): x-sweeps into a copy, y-sweeps aliased.  Whole arrays."""
    method = [1, order, -1, 0, 0, 0, 0]
    q = _data(name, mbc, mx, my, seed=my + mx + order)
    P = _problem(name, mbc, mx, my, method)
    what = "step2ds_host %s mbc=%d %dx%d order %d" % (name, mbc, mx, my, order)
    ref = {}
    for ids in (1, 2):
        ref[ids] = _oracle(name, mbc, mx, my, q, method, ids)
        for alias in (False, True):
            _poison(P, q.shape, ids)
            qn = q.copy("F")
            cfl = _call(P, qn if alias else q, qn, ids)
            _check("%s ids=%d%s" % (what, ids, " aliased" if alias else ""), qn, ref[ids][0], cfl, ref[ids][1], mbc)
    qo = ref[1][0].copy("F")
    oy = _oracle(name, mbc, mx, my, qo, method, 2, qnew=qo)[1]
    _poison(P, q.shape, 1)
    qg = q.copy("F")
    cx = _call(P, q, qg, 1)
    _poison(P, q.shape, 2)
    cy = _call(P, qg, qg, 2)
    _check(what + " x then aliased y", qg, qo, (cx, cy), (ref[1][1], oy), mbc)


@pytest.mark.gpu
@pytest.mark.parametrize("name,mbc,cls,my,mx,order,trans", UNSPLIT_CASES)
def test_step2_host(name, mbc, cls, my, mx, order, trans):
    """Interior cells against the oracle; the ghost rows keep their input (qnew == qold on entry)."""
    method = [1, order, trans, 0, 0, 0, 0]
    q = _data(name, mbc, mx, my, seed=my + mx + trans)
    P = _problem(name, mbc, mx, my, method)
    qn_o, cfl_o = _oracle(name, mbc, mx, my, q, method)
    _poison(P, q.shape)
    qn = q.copy("F")
    cfl = _call(P, q, qn)
    what = "step2_host %s mbc=%d %dx%d order %d trans %d" % (name, mbc, mx, my, order, trans)
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    _check(what, qn[inner], qn_o[inner], cfl, cfl_o, mbc, mbc)
    ghost = np.r_[0:mbc, my + mbc:my + 2 * mbc]
    assert np.array_equal(qn[:, :, ghost], q[:, :, ghost]), what + ": ghost rows changed"


# =============================================================================================
# Scratch: the first call after a release, growth, reuse, and two host threads
# =============================================================================================
@pytest.mark.gpu
def test_first_call_after_releasing_the_scratch():
    mbc, mx, my = 2, 5, 16384
    method = [1, 2, -1, 0, 0, 0, 0]
    q = _data("euler", mbc, mx, my, seed=7)
    P = _problem("euler", mbc, mx, my, method)
    qn_o, cfl_o = _oracle("euler", mbc, mx, my, q, method, 1)
    _lib.call("clawb200_release_host_scratch")
    qn = q.copy("F")
    cfl = _call(P, q, qn, 1)
    _check("step2ds_host ids=1 after release", qn, qn_o, cfl, cfl_o, mbc)


def _job(name, mbc, mx, my, ids, seed):
    """one host call: (problem, qold, ids, seed)"""
    method = [1, 2, -1 if ids else 2, 0, 0, 0, 0]
    return _problem(name, mbc, mx, my, method), _data(name, mbc, mx, my, seed), ids


def _run(job):
    P, q, ids = job
    qn = q.copy("F")
    return qn, _call(P, q, qn, ids)


@pytest.mark.gpu
def test_scratch_grows_and_is_reused():
    """Small (direct path), tall (pipelined), small again, then wider than before on the direct path
    (HostScratch grows) and in the pipeline (the slab buffers grow): each call equals the same call
    made on freshly released scratch, and the oracle."""
    seq = [(5, 100), (5, 16384), (5, 100), (600, 900), (251, 1100)]
    jobs = [_job("euler", 2, mx, my, ids, seed=mx + my) for mx, my in seq for ids in (1, 2, None)]
    fresh = []
    for job in jobs:
        _lib.call("clawb200_release_host_scratch")
        fresh.append(_run(job))
    _lib.call("clawb200_release_host_scratch")
    for job, (qf, cf) in zip(jobs, fresh):
        P, q, ids = job
        qn, cfl = _run(job)
        what = "euler %dx%d ids=%s" % (P.mx, P.my, ids)
        assert np.array_equal(qn, qf) and cfl == cf, what + ": differs from the call on fresh scratch"
        method = list(P.method)
        qn_o, cfl_o = _oracle("euler", 2, P.mx, P.my, q, method, ids)
        sl = (slice(None),) * 3 if ids else (slice(None), slice(2, -2), slice(2, -2))
        _check(what, qn[sl], qn_o[sl], cfl, cfl_o, 2, 0 if ids else 2)


@pytest.mark.gpu
def test_two_host_threads():
    """The host scratch, streams and events are per thread (clawb200.cu:740, :846) and ctypes drops the
    GIL during a call: two threads of ten pipelined calls each on different grids give the results
    of the same calls made one after the other."""
    kinds = (1, 2, None)
    jobs = [[_job("euler", 2, 5, 1024 + 389 * i, kinds[i % 3], seed=i) for i in range(10)],
            [_job("shallow", 3, 3, 2000 + 1237 * i, kinds[(i + 1) % 3], seed=50 + i) for i in range(10)]]
    serial = [[_run(j) for j in js] for js in jobs]
    out = [[None] * len(js) for js in jobs]
    errors = []

    def worker(t):
        try:
            for i, job in enumerate(jobs[t]):
                out[t][i] = _run(job)
        except BaseException as e:   # re-raised in the main thread
            errors.append(e)
        finally:
            _lib.call("clawb200_release_host_scratch")

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(len(jobs))]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    for t, js in enumerate(jobs):
        for i, ((qs, cs), (qt, ct)) in enumerate(zip(serial[t], out[t])):
            assert np.array_equal(qs, qt) and cs == ct, "thread %d call %d (my = %d)" % (t, i, js[i][0].my)


# =============================================================================================
# Through f2py_shim, and on the fma build
# =============================================================================================
@pytest.mark.gpu
def test_f2py_shim_classic2_at_16384_rows():
    """classic2('euler_5wave') called as clawpack.py calls it: step2ds x-sweeps, then y-sweeps with
    qold and qnew the same array (clawpack.py:538-548), and step2."""
    from pyclaw_b200 import f2py_shim
    mx, my, mbc = 5, 16384, 2
    lim = RPS["euler"][4]
    q = _data("euler", mbc, mx, my, seed=13)
    classic2 = f2py_shim.classic2('euler_5wave')
    classic2.cparam.gamma, classic2.cparam.gamma1 = 1.4, 0.4
    method = [1, 2, -1, 0, 0, 0, 0]
    qnew = q.copy('F')
    qq, cx = classic2.step2ds(max(mx, my), mbc, mx, my, q, qnew, None, DX, DY, DT, method, lim, None, None, None, None, 1)
    qq, cy = classic2.step2ds(max(mx, my), mbc, mx, my, qq, qq, None, DX, DY, DT, method, lim, None, None, None, None, 2)
    qo, ox = _oracle("euler", mbc, mx, my, q, method, 1)
    oy = _oracle("euler", mbc, mx, my, qo, method, 2, qnew=qo)[1]
    _check("classic2.step2ds x then y", qq, qo, (cx, cy), (ox, oy), mbc)
    method = [1, 2, 2, 0, 0, 0, 0]
    qnew = q.copy('F')
    out, cfl = classic2.step2(max(mx, my), mbc, mx, my, q, qnew, None, DX, DY, DT, method, lim)
    assert out is qnew
    qn_o, cfl_o = _oracle("euler", mbc, mx, my, q, method)
    inner = (slice(None), slice(mbc, -mbc), slice(mbc, -mbc))
    _check("classic2.step2", qnew[inner], qn_o[inner], cfl, cfl_o, mbc, mbc)


@pytest.fixture
def fma():
    """Runs the test on the fma build and restores the previous variant afterwards (test_gpu_fma_build.py)."""
    import test_gpu_fma_build as tfb
    with tfb._variant("fma"):
        yield tfb


@pytest.mark.gpu
def test_fma_x_sweeps_at_16384_rows(fma):
    """The fma build through the pipeline: within test_gpu_fma_build.py's 1e-13 of max |q| per component."""
    mbc, mx, my = 2, 5, 16384
    method = [1, 2, -1, 0, 0, 0, 0]
    q = _data("euler", mbc, mx, my, seed=21)
    P = _problem("euler", mbc, mx, my, method)
    qn_o, cfl_o = _oracle("euler", mbc, mx, my, q, method, 1)
    _poison(P, q.shape, 1)
    qn = q.copy("F")
    cfl = _call(P, q, qn, 1)
    fma._close("step2ds_host euler ids=1 5x16384", qn, qn_o, cfl, cfl_o)


# =============================================================================================
# The component stride
# =============================================================================================
@pytest.mark.gpu
def test_component_stride_smaller_than_the_padded_field_is_refused():
    """A 2-D problem whose mstride is below pitch * (my + 2 mbc) would alias the last padded rows of
    one component with the first of the next: every 2-D device entry point refuses it.  A 1-D problem
    keeps mstride = nx."""
    import torch
    mx, my = 20, 12
    for mbc, pitch in ((2, None), (3, 31)):
        P = _problem("acoustics", mbc, mx, my, [1, 2, 2, 0, 0, 0, 0])
        if pitch:
            P.pitch = pitch
        full = P.pitch * (my + 2 * mbc)
        q = torch.zeros(3 * full, dtype=torch.float64, device="cuda")
        qn, cfl = torch.zeros_like(q), torch.zeros(1, dtype=torch.float64, device="cuda")
        v = [ctypes.c_void_p(t.data_ptr()) for t in (q, qn, cfl)]
        calls = [("clawb200_step2", v[0], v[1], None, DT, v[2], None),
                 ("clawb200_step2_rows", v[0], v[1], None, DT, 1, my, v[2], None),
                 ("clawb200_step2ds", v[0], v[1], None, DT, 1, v[2], None),
                 ("clawb200_step2ds", v[0], v[1], None, DT, 2, v[2], None)]
        if mbc == 3:
            calls.append(("clawb200_sharpclaw_stage", v[0], None, None, v[1], None, DT, _lib.STAGE_DQ_ONLY,
                          0.0, 0.0, 1.0, v[2], None))
        for fn, *args in calls:
            P.method[2] = -1 if fn == "clawb200_step2ds" else 2
            P.mstride = full - 1
            with pytest.raises(_lib.ClawB200Error, match="mstride"):
                _lib.call(fn, ctypes.byref(P), *args)
            P.mstride = full
            _lib.call(fn, ctypes.byref(P), *args)
        torch.cuda.synchronize()
    P1 = _lib.make_problem(1, 2, 2, 2, mx, 1, DX, 1.0, 1, [1.0, 1.0, 1.0, 1.0], [1, 2, 0, 0, 0, 0, 0], [4, 4])
    assert P1.mstride == mx + 4
    q1 = torch.ones(2 * (mx + 4), dtype=torch.float64, device="cuda")
    q1n = q1.clone()
    _lib.call("clawb200_step1", ctypes.byref(P1), ctypes.c_void_p(q1.data_ptr()), ctypes.c_void_p(q1n.data_ptr()),
              None, DT, ctypes.c_void_p(cfl.data_ptr()), None)
    torch.cuda.synchronize()
