"""Time the 3-D classic steps of every built-in 3-D solver on the GPU.

    python profiles/time3d_solvers.py [--sizes 128,256] [--steps 10] [--solvers a,b] [--parent path/to/libclawb200.so]

For each 3-D solver (vc_acoustics_3d, advection_3d, euler_3d, vc_advection_fwave_3d; --solvers picks some)
and each algorithm (dimensional
splitting: three step3ds sweeps; unsplit: step3 with order_trans = 22) at n^3 cells: ms per step
(CUDA events around `steps` steps after 2 warm-up steps, strict build) and cell-updates per second.
Every working set exceeds the 126 MB L2 except the advection split step at 128^3 (three 18 MB
arrays), which runs largely from L2.

With --parent (another build of the library, e.g. the parent commit's, whose vc-acoustics steps
ran specialised kernels), the vc-acoustics steps at 256^3 -- split and unsplit -- are timed with
this tree's build and with that one, alternating the builds in one process, 5 repeats each.
The card's name and power limit are read in the same run and printed with the numbers.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def setup(torch, _lib, name, n, method):
    from pyclaw_b200 import riemann
    rs = {"vc_acoustics_3d": riemann.vc_acoustics_3d, "advection_3d": riemann.advection_3d,
          "euler_3d": riemann.euler_3d, "vc_advection_fwave_3d": riemann.vc_advection_fwave_3d}[name]
    mbc = 2
    nx = ny = nz = n + 2 * mbc
    meqn, mw = rs.meqn(3), rs.nwaves(3)
    params = {"advection_3d": [1.0, 0.5, 0.25], "euler_3d": [1.4, 0.4]}.get(name, [])
    P = _lib.make_problem(3, meqn, mw, mbc, n, n, 1.0 / n, 1.0 / n, rs.rp_id, params, method, [4] * mw,
                          maux=rs.maux, pitch=nx, mstride=nx * ny * nz)
    g = torch.Generator(device='cuda').manual_seed(0)
    q = torch.rand((meqn, nz, ny, nx), dtype=torch.float64, device='cuda', generator=g)
    if name == "euler_3d":
        q[0] += 1.0
        q[1:4] -= 0.5
        q[4] = 2.5 + 0.5 * (q[1:4] ** 2).sum(0) / q[0]
    aux = None
    if name == "vc_advection_fwave_3d":   # cell velocities of both signs
        aux = 2.0 * torch.rand((rs.maux, nz, ny, nx), dtype=torch.float64, device='cuda', generator=g) - 1.0
    elif rs.maux:
        aux = 1.0 + torch.randint(0, 2, (rs.maux, nz, ny, nx), device='cuda', generator=g).to(torch.float64)
    return rs, P, q, aux


def time_step(torch, _lib, variant, rp_id, name, n, dim_split, steps):
    _lib.set_variant(variant)
    method = [1, 2, -1 if dim_split else 22, 0, 0, 0, 0]
    rs, P, q, aux = setup(torch, _lib, name, n, method)
    P.rp_id = rp_id
    qn = torch.empty_like(q)
    qm = torch.empty_like(q)
    cfl = torch.zeros(1, dtype=torch.float64, device='cuda')
    ptr = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    dt = 0.3 / n
    scratch = None
    if not dim_split:
        scratch = torch.empty(_lib.load().clawb200_step3_scratch_doubles(ctypes.byref(P)), dtype=torch.float64,
                              device='cuda')

    def step():
        if dim_split:
            for idir, (a, b) in zip((1, 2, 3), ((q, qn), (qn, qm), (qm, qn))):
                _lib.call("clawb200_step3ds", ctypes.byref(P), n, 1.0 / n, ptr(a), ptr(b), ptr(aux), dt, idir,
                          ptr(cfl), st)
        else:
            _lib.call("clawb200_step3", ctypes.byref(P), n, 1.0 / n, ptr(q), ptr(qn), ptr(aux), dt, ptr(scratch),
                      ptr(cfl), st)
    for _ in range(2):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    assert torch.isfinite(qn).all()
    del scratch, q, qn, qm, aux
    torch.cuda.empty_cache()
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="128,256")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--parent", default=None, help="another build of libclawb200.so to compare with")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--solvers", default="vc_acoustics_3d,advection_3d,euler_3d,vc_advection_fwave_3d")
    args = ap.parse_args()
    import torch
    from pyclaw_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to time")
    dev = card()
    print("card: %s" % dev, flush=True)
    ids = {"vc_acoustics_3d": _lib.RP_ACOUSTICS3D_VC, "advection_3d": _lib.RP_ADVECTION3D, "euler_3d": _lib.RP_EULER3D,
           "vc_advection_fwave_3d": _lib.RP_ADVECTION3D_VC_FWAVE}
    for n in [int(s) for s in args.sizes.split(",")]:
        for name in args.solvers.split(","):
            for dim_split in (True, False):
                ms = time_step(torch, _lib, "strict", ids[name], name, n, dim_split, args.steps)
                r = dict(solver=name, n=n, algorithm="split" if dim_split else "unsplit22", ms_per_step=round(ms, 3),
                         cell_updates_per_s=n ** 3 / (ms * 1e-3), card=dev)
                print(json.dumps(r), flush=True)
    if not args.parent:
        return
    _lib.LIB_PATHS["parent"] = os.path.abspath(args.parent)
    for dim_split in (True, False):
        ab = {"this tree": [], "parent": []}
        for rep in range(args.repeats):
            for label, variant in (("this tree", "strict"), ("parent", "parent")):
                ab[label].append(time_step(torch, _lib, variant, _lib.RP_ACOUSTICS3D_VC, "vc_acoustics_3d", 256,
                                           dim_split, args.steps))
        for label, ts in ab.items():
            med = sorted(ts)[len(ts) // 2]
            print(json.dumps(dict(ab="vc_acoustics_3d %s 256^3" % ("split" if dim_split else "unsplit22"), build=label,
                                  ms=[round(t, 3) for t in ts], median_ms=round(med, 3), card=dev)), flush=True)
    _lib.set_variant("strict")


if __name__ == "__main__":
    main()
