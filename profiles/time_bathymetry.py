"""Time the 2-D classic step of the shallow-water-over-bathymetry solver beside the flat-bottom Roe solver.

    python profiles/time_bathymetry.py [--n 8192] [--steps 20] [--out profiles/time_bathymetry.json]

For shallow_bathymetry_fwave and shallow_roe_with_efix, the strict and the fma build, and two
algorithms (unsplit step2 with order_trans = 2: the x-sweep and y-sweep kernels; dimensional splitting:
two step2ds sweeps), at n^2 cells: ms per step from CUDA events around `steps` steps after 3 warm-up
steps, and cell-updates per second.  At 8192^2 one array of q is 1.6 GB, far above the 126 MB L2.  The
Roe solver's unsplit step runs the single-pass kernel (fused.cuh) unless --two-pass is given; the
bathymetry solver has no single-pass kernel (it reads aux), so its unsplit step is always two sweeps.
The card's name and power limit are read in the same run and printed and stored with the numbers.
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


def time_step(torch, _lib, variant, solver, n, dim_split, steps, two_pass):
    _lib.set_variant(variant)
    bathy = solver == "shallow_bathymetry_fwave"
    mbc = 2
    nx = n + 2 * mbc
    rp_id = _lib.RP_SHALLOW_BATHY_FWAVE if bathy else _lib.RP_SHALLOW
    params = [9.81, 1e-3] if bathy else [9.81]
    method = [1, 2, -1 if dim_split else 2, 0, 0, 0, 1 if bathy else 0]
    dx = 1.0 / n
    P = _lib.make_problem(2, 3, 3, mbc, n, n, dx, dx, rp_id, params, method, [4, 4, 4], maux=1 if bathy else 0,
                          pitch=nx, mstride=nx * nx)
    P.step2_mode = 1 if two_pass else 0
    # smooth bottom and surface, velocities of both signs up to ~1 (Froude numbers up to ~0.4)
    x = torch.linspace(0.0, 1.0, nx, dtype=torch.float64, device='cuda')
    sx, cy = torch.sin(6.2832 * 3 * x), torch.cos(6.2832 * 2 * x)
    b = -1.0 + 0.3 * torch.outer(cy, sx)
    q = torch.empty((3, nx, nx), dtype=torch.float64, device='cuda')
    q[0] = 0.05 * torch.outer(sx, cy) - b
    q[1] = q[0] * torch.outer(cy, cy)
    q[2] = -q[0] * torch.outer(sx, sx)
    aux = b[None].contiguous() if bathy else None
    qn, qm = torch.empty_like(q), torch.empty_like(q)
    cfl = torch.zeros(1, dtype=torch.float64, device='cuda')
    ptr = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    dt = 0.2 * dx

    def step():
        if dim_split:
            _lib.call("clawb200_step2ds", ctypes.byref(P), ptr(q), ptr(qn), ptr(aux), dt, 1, ptr(cfl), st)
            _lib.call("clawb200_step2ds", ctypes.byref(P), ptr(qn), ptr(qm), ptr(aux), dt, 2, ptr(cfl), st)
        else:
            _lib.call("clawb200_step2", ctypes.byref(P), ptr(q), ptr(qn), ptr(aux), dt, ptr(cfl), st)
    for _ in range(3):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    assert torch.isfinite(qm if dim_split else qn).all()
    launches = 2 if dim_split else _lib.load().clawb200_step2_launches(ctypes.byref(P))
    del q, qn, qm, aux, b
    torch.cuda.empty_cache()
    return ms, launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--two-pass", action="store_true", help="run the Roe solver's unsplit step as two sweeps too")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_bathymetry.json"))
    args = ap.parse_args()
    if args.steps < 20:
        raise SystemExit("--steps must be at least 20")
    import torch
    from pyclaw_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to time")
    dev = card()
    print("card (name, power limit): %s" % dev, flush=True)
    rows = []
    print("%-26s %-7s %-10s %9s %12s %9s" % ("solver", "build", "algorithm", "ms/step", "Gcell-upd/s", "launches"))
    for dim_split in (False, True):
        for variant in ("strict", "fma"):
            for solver in ("shallow_bathymetry_fwave", "shallow_roe_with_efix"):
                ms, launches = time_step(torch, _lib, variant, solver, args.n, dim_split, args.steps, args.two_pass)
                r = dict(solver=solver, build=variant, algorithm="split" if dim_split else "unsplit2", n=args.n,
                         steps=args.steps, ms_per_step=round(ms, 3), cell_updates_per_s=args.n ** 2 / (ms * 1e-3),
                         launches_per_step=launches, card=dev)
                rows.append(r)
                print("%-26s %-7s %-10s %9.3f %12.3f %9d" % (solver, variant, r["algorithm"], ms,
                                                             r["cell_updates_per_s"] / 1e9, launches), flush=True)
    _lib.set_variant("strict")
    with open(args.out, "w") as f:
        json.dump(dict(card=dev, n=args.n, steps=args.steps, rows=rows), f, indent=1)
    print("wrote %s" % args.out)


if __name__ == "__main__":
    main()
