"""Time the 3-D SharpClaw stage of every built-in 3-D solver on the GPU.

    python profiles/time3d_sharpclaw.py [--sizes 128,256] [--stages 20] [--steps 5] [--solvers a,b]
                                        [--parent DIR --bench-reps 3]

For each 3-D solver (vc_acoustics_3d, advection_3d, euler_3d, vc_advection_fwave_3d; --solvers picks some)
at n^3 cells, strict build, PyWENO weno5
with f32 literals:
  - ms per RK stage (clawb200_sharpclaw_stage3, mode 0): CUDA events around `stages` stages after 3
    warm-up stages;
  - kernel A (sc2d_kernel: x and y, plane by plane) and kernel B (sc3d_z_kernel: z) separately, from a
    torch.profiler capture of the same stages in a run of its own;
  - ms per SSP104 step through SharpClawSolver3D.step (10 stages, the SSP104 combination, periodic
    boundary fills and the Courant-number read), CUDA events around `steps` steps after one warm-up step;
  - cell-updates per second = n^3 / (time per step).
At 256^3 every working set (q, out, aux: 134-671 MB) is above the 126 MB L2.

With --parent DIR (a built checkout of another commit), `python bench.py --workload shallow` is run in
DIR and in this tree, alternating, --bench-reps times each, to show the 2-D SharpClaw path unchanged.
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


PARAMS = {"advection_3d": dict(u=1.0, v=0.5, w=0.25), "euler_3d": dict(gamma=1.4, gamma1=0.4), "vc_acoustics_3d": {},
          "vc_advection_fwave_3d": {}}


def make(torch, name, n):
    import pyclaw
    rs = getattr(pyclaw.riemann, name)
    solver = pyclaw.SharpClawSolver3D()
    solver.rp = rs
    solver.fwave = rs.fwave
    solver.mwaves = rs.nwaves(3)
    solver.dt_variable, solver.dt_initial = False, 0.3 / n
    solver.cfl_desired, solver.cfl_max = 0.8, 10.0
    for i in range(3):
        solver.bc_lower[i] = solver.bc_upper[i] = pyclaw.BC.periodic
        solver.aux_bc_lower[i] = solver.aux_bc_upper[i] = pyclaw.BC.periodic
    grid = pyclaw.Grid([pyclaw.Dimension(nm, 0.0, 1.0, n) for nm in 'xyz'])
    meqn = rs.meqn(3)
    state = pyclaw.State(grid, meqn, rs.maux)
    state.aux_global.update(PARAMS[name])
    g = torch.Generator(device='cuda').manual_seed(0)
    q = torch.rand((meqn, n, n, n), dtype=torch.float64, device='cuda', generator=g)
    if name == "euler_3d":
        q[0] += 1.0
        q[1:4] -= 0.5
        q[4] = 2.5 + 0.5 * (q[1:4] ** 2).sum(0) / q[0]
    state.q = q
    if name == "vc_advection_fwave_3d":   # cell velocities of both signs
        state.aux = 2.0 * torch.rand((rs.maux, n, n, n), dtype=torch.float64, device='cuda', generator=g) - 1.0
    elif rs.maux:
        state.aux = 1.0 + torch.randint(0, 2, (rs.maux, n, n, n), device='cuda', generator=g).to(torch.float64)
    sol = pyclaw.Solution(state)
    solver.setup(sol)
    solver.dt = solver.dt_initial
    return solver, sol


def time_stages(torch, solver, state, stages, profile=False):
    from pyclaw_b200.solver import _ptr
    F = state._q
    q0, out = F.cur, F.get_spare()
    solver._bcs_on(state, q0)
    run = lambda: solver._stage(q0, None, out, 0, 0.0, 0.0, 1.0, 0)
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    if profile:
        from torch.profiler import profile as prof, ProfilerActivity
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            for _ in range(stages):
                run()
            torch.cuda.synchronize()
        tot = {"A": 0.0, "B": 0.0}
        for e in p.key_averages():
            key = "A" if "sc2d_kernel" in e.key else ("B" if "sc3d_z_kernel" in e.key else None)
            if key:
                tot[key] += e.device_time_total / 1e3 / stages  # us -> ms per stage
        F.put_spare(out)
        return tot
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(stages):
        run()
    e1.record()
    torch.cuda.synchronize()
    F.put_spare(out)
    return e0.elapsed_time(e1) / stages


def time_steps(torch, solver, sol, steps):
    solver.step(sol)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        solver.step(sol)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def bench_ab(parent, reps):
    """bench.py --workload shallow in the parent checkout and in this tree, alternating."""
    res = {"parent": [], "this": []}
    for _ in range(reps):
        for key, d in (("parent", parent), ("this", ROOT)):
            r = subprocess.run([sys.executable, "bench.py", "--workload", "shallow", "--gpus", "1"], cwd=d,
                               capture_output=True, text=True)
            line = [l for l in r.stdout.splitlines() if l.startswith("{")]
            res[key].append(json.loads(line[-1]) if line else {"error": r.stderr[-500:]})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="128,256")
    ap.add_argument("--stages", type=int, default=20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--parent", default=None)
    ap.add_argument("--bench-reps", type=int, default=3)
    ap.add_argument("--solvers", default="vc_acoustics_3d,advection_3d,euler_3d,vc_advection_fwave_3d")
    args = ap.parse_args()
    import torch
    print("card: %s" % card(), flush=True)
    rows = []
    for n in [int(s) for s in args.sizes.split(",")]:
        for name in args.solvers.split(","):
            solver, sol = make(torch, name, n)
            st = sol.states[0]
            ms_stage = time_stages(torch, solver, st, args.stages)
            kern = time_stages(torch, solver, st, args.stages, profile=True)
            ms_step = time_steps(torch, solver, sol, args.steps)
            row = dict(solver=name, n=n, ms_per_stage=ms_stage, ms_kernel_A=kern["A"], ms_kernel_B=kern["B"],
                       ms_kernels_A_plus_B=kern["A"] + kern["B"], ms_per_ssp104_step=ms_step,
                       cell_updates_per_s=n ** 3 / (ms_step * 1e-3))
            rows.append(row)
            print(json.dumps(row), flush=True)
            del solver, sol, st
            torch.cuda.empty_cache()
    if args.parent:
        print(json.dumps({"bench_shallow_ab": bench_ab(args.parent, args.bench_reps)}), flush=True)
    print("card: %s" % card(), flush=True)


if __name__ == "__main__":
    main()
