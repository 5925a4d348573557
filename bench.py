#!/usr/bin/env python
"""
bench.py -- cell-updates/s (float64) of the finite-volume time step on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference]
                    [--dump-outputs DIR]

N > 1 is launched by the driver with torch.distributed.run (one rank per GPU); the grid
is then N y-slabs of the per-GPU size (weak scaling) with NCCL halo exchange and an
all-reduce(MAX) of the Courant number.  Rank 0 prints ONE JSON line.

Workloads (BASELINE.json `configs`):
  euler      (default) 2-D Euler 5-wave Roe, ClawSolver2D unsplit + transverse, 8192^2 per GPU
  acoustics  2-D acoustics, ClawSolver2D unsplit + transverse rpt2, 4096^2
  shallow    2-D shallow water, SharpClawSolver2D WENO5 + SSP33, 8192^2 per GPU
A "step" is one full time step through the public API (solver.evolve_to_time(solution)):
boundary conditions, sweeps, Courant-number reduction and the 8-byte read-back that the
dt controller needs.  `value` counts accepted steps only.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GAMMA, GAMMA1 = 1.4, 0.4

WORKLOADS = {
    # name: per-GPU grid, meqn, algorithmic bytes per cell-step (SURVEY.md 8(d))
    "euler": dict(n=8192, meqn=5, mwaves=5, balg=80, label="euler5_roe_unsplit_8192x8192_per_gpu"),
    "acoustics": dict(n=4096, meqn=3, mwaves=2, balg=48, label="acoustics_unsplit_rpt2_4096x4096_per_gpu"),
    "shallow": dict(n=8192, meqn=3, mwaves=3, balg=192, label="shallow_sharpclaw_weno5_ssp33_8192x8192_per_gpu"),
    # config 5: shallow water on the sphere, 4096 x 2048 per GPU (n = cells in y; x has 2n)
    "sphere": dict(n=2048, meqn=4, mwaves=3, balg=192, label="shallow_sphere_rossby_haurwitz_4096x2048_per_gpu"),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


# --------------------------------------------------------------------------------------
# problem set-up through the PyClaw API
# --------------------------------------------------------------------------------------
def shock_state(pinf=5.):
    rinf = (GAMMA1 + pinf * (GAMMA + 1.)) / ((GAMMA + 1.) + GAMMA1 * pinf)
    vinf = 1. / np.sqrt(GAMMA) * (pinf - 1.) / np.sqrt(0.5 * ((GAMMA + 1.) / GAMMA) * pinf + 0.5 * GAMMA1 / GAMMA)
    einf = 0.5 * rinf * vinf ** 2 + pinf / GAMMA1
    return rinf, vinf, einf


def build_problem(pyclaw, workload, n, nranks, torch):
    """Synthetic data of the BASELINE shapes: analytic initial conditions evaluated on the
    device (no RNG), n x n cells per GPU, n x (n*nranks) globally."""
    if workload == "euler":
        # test/euler/2d/shockbubble.py scaled up: bubble of light gas, shock entering from
        # the left ghost cells; source term off (kernel metric)
        x = pyclaw.Dimension('x', 0.0, 2.0, n)
        y = pyclaw.Dimension('y', 0.0, 2.0 * nranks, n * nranks)
        state = pyclaw.State(pyclaw.Grid([x, y]), 5)
        state.aux_global['gamma'] = GAMMA
        state.aux_global['gamma1'] = GAMMA1
        xc = torch.as_tensor(state.grid.x.center, device=state.device)
        yc = torch.as_tensor(state.grid.y.center, device=state.device)
        r = torch.sqrt((xc[:, None] - 0.5) ** 2 + (yc[None, :] - 0.0) ** 2)
        inside = (r <= 0.2).to(torch.float64)
        q = state.q
        q[0] = 0.1 * inside + 1.0 * (1.0 - inside)
        q[1] = 0.
        q[2] = 0.
        q[3] = 1.0 / GAMMA1
        q[4] = inside
        solver = pyclaw.ClawSolver2D()
        solver.mwaves = 5
        solver.limiters = [4, 4, 4, 4, 2]
        solver.dim_split = False
        solver.order_trans = 2
        solver.cfl_max, solver.cfl_desired = 0.5, 0.45
        rinf, vinf, einf = shock_state()

        def shockbc(state, dim, t, qbc, mbc):
            if dim.nstart == 0:
                qbc[0, :mbc] = rinf
                qbc[1, :mbc] = rinf * vinf
                qbc[2, :mbc] = 0.
                qbc[3, :mbc] = einf
                qbc[4, :mbc] = 0.
        solver.user_bc_lower = shockbc
        solver.bc_lower[0] = pyclaw.BC.custom
        solver.bc_upper[0] = pyclaw.BC.outflow
        solver.bc_lower[1] = pyclaw.BC.reflecting
        solver.bc_upper[1] = pyclaw.BC.outflow
        solver.dt_initial = 0.1 * state.grid.d[0]
    elif workload == "acoustics":
        x = pyclaw.Dimension('x', -1.0, 1.0, n)
        y = pyclaw.Dimension('y', -1.0, -1.0 + 2.0 * nranks, n * nranks)
        state = pyclaw.State(pyclaw.Grid([x, y]), 3)
        rho, bulk = 1.0, 4.0
        cc = np.sqrt(bulk / rho)
        state.aux_global.update(rho=rho, bulk=bulk, zz=rho * cc, cc=cc)
        xc = torch.as_tensor(state.grid.x.center, device=state.device)
        yc = torch.as_tensor(state.grid.y.center, device=state.device)
        r = torch.sqrt(xc[:, None] ** 2 + yc[None, :] ** 2)
        width = 0.2
        q = state.q
        q[0] = (torch.abs(r - 0.5) <= width) * (1. + torch.cos(np.pi * (r - 0.5) / width))
        q[1] = 0.
        q[2] = 0.
        solver = pyclaw.ClawSolver2D()
        solver.mwaves = 2
        solver.limiters = [4, 4]
        solver.dim_split = False
        solver.order_trans = 2
        for i in range(2):
            solver.bc_lower[i] = solver.bc_upper[i] = pyclaw.BC.outflow
        solver.dt_initial = 0.5 * state.grid.d[0] / cc
    elif workload == "shallow":
        x = pyclaw.Dimension('x', -2.5, 2.5, n)
        y = pyclaw.Dimension('y', -2.5, -2.5 + 5.0 * nranks, n * nranks)
        state = pyclaw.State(pyclaw.Grid([x, y]), 3)
        state.aux_global['grav'] = 1.0
        xc = torch.as_tensor(state.grid.x.center, device=state.device)
        yc = torch.as_tensor(state.grid.y.center, device=state.device)
        r = torch.sqrt(xc[:, None] ** 2 + yc[None, :] ** 2)
        inside = (r <= 0.5).to(torch.float64)
        q = state.q
        q[0] = 2.0 * inside + 1.0 * (1.0 - inside)
        q[1] = 0.
        q[2] = 0.
        solver = pyclaw.SharpClawSolver2D()
        solver.mwaves = 3
        solver.time_integrator = 'SSP33'
        solver.cfl_max, solver.cfl_desired = 0.6, 0.5
        solver.bc_lower[0] = solver.bc_lower[1] = pyclaw.BC.outflow
        solver.bc_upper[0] = solver.bc_upper[1] = pyclaw.BC.reflecting
        solver.dt_initial = 0.2 * state.grid.d[0]
    elif workload == "sphere":
        # apps/shallow-sphere: 16 aux, capacity function, pole-fold custom BCs, Strang src2
        from pyclaw_b200.apps import shallow_sphere as app
        state, solver = app.setup(pyclaw, mx=2 * n, my=n * nranks)
        solver.dt_initial = 0.1 * state.grid.d[0] / 4.0
    else:
        raise SystemExit("unknown workload %s" % workload)
    return state, solver


DUMP_CELLS = 1 << 20   # cells kept per field by --dump-outputs: 5 x 2^20 float64 = 40 MB for Euler


def dump_outputs(outdir, solution, solver):
    """Write what the caller of solver.evolve_to_time holds after the last timed step, as float64
    .npy files: q (all cells, or on a larger grid the same DUMP_CELLS cells drawn by
    numpy.random.default_rng(0), shape [meqn, cells]), t, and the step's cflmax / dtmin / dtmax."""
    import torch
    os.makedirs(outdir, exist_ok=True)
    q = solution.state.q.as_subclass(torch.Tensor)   # [m, i, j]
    meqn, cells = q.shape[0], q[0].numel()
    if cells > DUMP_CELLS:
        flat = np.sort(np.random.default_rng(0).choice(cells, DUMP_CELLS, replace=False))
        idx = [torch.as_tensor(a, device=q.device) for a in np.unravel_index(flat, q.shape[1:])]
        q = q[(slice(None),) + tuple(idx)]
    np.save(os.path.join(outdir, "q.npy"), q.reshape(meqn, -1).cpu().numpy())
    for name, v in (("t", solution.t), ("cflmax", solver.status["cflmax"]),
                    ("dtmin", solver.status["dtmin"]), ("dtmax", solver.status["dtmax"])):
        np.save(os.path.join(outdir, name + ".npy"), np.array([v], dtype=np.float64))


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md): NVML every
    20 ms when the bindings load, else the recipe's nvidia-smi query every 200 ms."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self._halt = index, [], threading.Event()
        self.reasons, self.smax, self.source = set(), None, "nvidia-smi"
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.smax = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            pynvml.nvmlDeviceGetClockInfo(self._h, pynvml.NVML_CLOCK_SM)
            self._nvml, self.source = pynvml, "nvml"
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        self.samples.append(int(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
        try:
            get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
            r = int(get(self._h))
            for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
                              ("hw_thermal_slowdown", 0x40)):
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True,
                             timeout=5).stdout.strip()
        if not out:
            return
        f = [x.strip() for x in out.split(",")]
        if f[0].replace('.', '').isdigit():
            self.samples.append(int(float(f[0])))
        if self.smax is None and f[1].replace('.', '').isdigit():
            self.smax = int(float(f[1]))
        for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
            if v.lower().startswith("active"):
                self.reasons.add(name)

    def run(self):
        while not self._halt.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._halt.wait(0.02 if self._nvml is not None else 0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm = sorted(self.samples)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.smax,
                "reasons": sorted(self.reasons), "samples": len(sm), "source": self.source}


# --------------------------------------------------------------------------------------
# CPU legs: the oracle (strict-IEEE C restatement of the reference's Fortran path) on the
# host cores.  This is the only place bench.py touches oracle/.
# --------------------------------------------------------------------------------------
def cpu_problem(workload, n):
    import problems
    if workload == "euler":
        pb = problems.shockbubble(n, n, xupper=2.0, yupper=2.0)
        rp, params, lim = 3, [GAMMA, GAMMA1], [4, 4, 4, 4, 2]
    elif workload == "acoustics":
        pb = problems.acoustics2d(n, n)
        rp, params, lim = 1, pb["params"], [4, 4]
    else:
        pb = problems.shallow2d(n, n)
        rp, params, lim = 4, [1.0], [4, 4, 4]
    return pb, rp, params, lim


def cpu_step_fn(workload, n, nthreads):
    """Returns (fn, cells) where fn() advances one full time step on an n x n sample."""
    from oracle import pyclaw_oracle as po
    pb, rp, params, lim = cpu_problem(workload, n)
    q = pb["q"]
    dx, dy = pb["d"]
    if workload == "shallow":
        mbc = 3
        s = po.OracleSolver("sharpclaw", 2, rp, params, 3)
        s.time_integrator = "SSP33"
        s.bc_lower = [po.BC_OUTFLOW] * 2
        s.bc_upper = [po.BC_REFLECTING] * 2
        s.nthreads = nthreads
        s.setup(q, None, [dx, dy])
        s.dt = 0.2 * dx
        st = {"q": q.copy("F"), "t": 0.0}

        def fn():
            s.step(st)
    else:
        s = po.OracleSolver("classic", 2, rp, params, len(lim))
        s.limiters = lim
        s.dim_split = False
        s.order_trans = 2
        s.bc_lower = [po.BC_OUTFLOW] * 2
        s.bc_upper = [po.BC_OUTFLOW] * 2
        s.nthreads = max(nthreads, 2)  # slab driver (nthreads=1 would take the serial path; same result)
        if nthreads == 1:
            s.nthreads = 1
        s.setup(q, None, [dx, dy])
        s.dt = 0.1 * dx
        st = {"q": q.copy("F"), "t": 0.0}

        def fn():
            s._hyperbolic_classic(st)
    return fn, n * n


def time_cpu(workload, n, nthreads, budget_s):
    fn, cells = cpu_step_fn(workload, n, nthreads)
    fn()  # warm
    t0 = time.perf_counter()
    k = 0
    while True:
        fn()
        k += 1
        el = time.perf_counter() - t0
        if el > budget_s or k >= 50:
            break
    return cells * k / el, k, el


def run_reference(args, rank):
    if rank != 0:
        return
    ncores = os.cpu_count() or 1
    wl = WORKLOADS[args.workload]
    n = 2048 if args.workload != "shallow" else 1024
    fn, cells = cpu_step_fn(args.workload, n, ncores)
    for _ in range(args.warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    el = time.perf_counter() - t0
    value = cells * args.steps / el
    # the reference's Fortran is serial: the same port on ONE core, bounded sample
    v1, k1, el1 = time_cpu(args.workload, 512, 1, 4.0)
    single = {"value": v1, "unit": "cell-updates/s", "cores": 1,
              "sample": "%d steps on a 512x512 sample in %.1f s" % (k1, el1)}
    sample = "%dx%d sample of the workload, %d host threads (y-slabs), oracle C port of step2/flux2/rpn2/rpt2" % (n, n, ncores)
    line = {
        "impl": "reference", "metric": "cell-updates/s", "value": value, "unit": "cell-updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["label"], "sample": sample},
        "cpu_baseline": {"value": value, "unit": "cell-updates/s", "cores": ncores, "kind": "port",
                         "sample": sample, "single_core": single},
        "e2e": {"value": value, "unit": "cell-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def check_partition_parity(rank, world, torch, dist):
    """Strong-scaling comparison on a small grid: the same global problem on `world` slabs and on
    one GPU (rank 0), np.array_equal on q and equal step counts.  Returns a dict on rank 0."""
    import mp_partition_check as mp
    import problems
    import petclaw
    import pyclaw
    mx, my = 160, 16 * world
    pb = problems.shockbubble(mx, my)
    qs = problems.smooth_state("shallow", (mx, my), seed=5)
    cases = [("euler_unsplit", "euler", pb["q"], dict(dim_split=False, order_trans=2)),
             ("euler_dimsplit", "euler", pb["q"], dict(dim_split=True)),
             ("shallow_sharpclaw_ssp33", "shallow", qs, dict(time_integrator="SSP33"))]
    res = {"ranks": world, "grid": [mx, my], "cases": {}}
    ok = True
    for name, kind, q0, opts in cases:
        qp, nsteps = mp.run(petclaw, kind, q0, None, mx, my, opts)
        if rank == 0:
            qser, nser = mp.run(pyclaw, kind, q0, None, mx, my, opts)
            same = bool(np.array_equal(qp, qser) and nsteps == nser and np.isfinite(qser).all())
            res["cases"][name] = {"bit_identical": same, "steps": int(nsteps)}
            ok = ok and same
        dist.barrier()
    res["ok"] = ok
    return res if rank == 0 else None


# --------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="euler", choices=sorted(WORKLOADS))  # sphere: no --impl reference arm
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=0, help="override the per-GPU grid size (debug)")
    ap.add_argument("--perturb", action="store_true", help="(default now) time the developed field")
    ap.add_argument("--quiescent", action="store_true",
                    help="time the application's own initial data only (mostly at rest) instead of the developed field")
    ap.add_argument("--arithmetic", default="auto", choices=["auto", "strict", "fma"],
                    help="library build: strict IEEE (bit-exact parity build) or fma (FMA contraction + "
                         "1.5-ulp division).  auto = the fastest build that meets north_star's 1e-12 "
                         "relative tolerance on that workload (profiles/README.md, table 'fma vs strict'): "
                         "fma for the classic sweeps, strict for SharpClaw")
    ap.add_argument("--no-parity", action="store_true", help="skip the N > 1 partition-parity check")
    ap.add_argument("--no-other-build", action="store_true", help="skip timing the other arithmetic build")
    ap.add_argument("--no-other-workloads", action="store_true",
                    help="skip the short runs of the other BASELINE configurations")
    ap.add_argument("--no-quiescent-leg", action="store_true", help="skip timing the application's own (quiescent) field")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer e2e leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the solution they computed to DIR/<name>.npy "
                         "(rank 0's slab at N > 1) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU solution: it needs --impl ours")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        import petclaw as pyclaw
        pyclaw.init("nccl")
    else:
        import pyclaw
    from pyclaw_b200 import _lib

    wl = WORKLOADS[args.workload]
    n = args.n or wl["n"]
    cells_per_rank = n * n if args.workload != "sphere" else 2 * n * n
    # measured relative L-infinity of the fma build against the strict one over the reference's
    # own test runs (profiles/fma_study.py -> profiles/r2/fma_study_r2i.json)
    FMA_ERR = {"euler": 5.1e-14, "acoustics": 6.3e-16, "sphere": 1.5e-13, "shallow": 1.0e-11}
    if args.arithmetic == "auto":
        args.arithmetic = "fma" if FMA_ERR[args.workload] <= 1e-12 else "strict"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- partition parity (N > 1): the slab-partitioned run against the single-GPU run, bit for
    # bit, on a small grid, before anything is timed (the reference compares its 6-rank run with
    # the serial golden file, test/test_examples.py:264-277) ------------------------------------
    partition_parity = None
    if world > 1 and not args.no_parity:
        partition_parity = check_partition_parity(rank, world, torch, dist)

    def timed_run(field, steps, warmup, sample_clocks, arithmetic=None, workload=None):
        """Set the problem up, let dt settle, time `steps` calls of solver.evolve_to_time."""
        workload = workload or args.workload
        wn = (args.n if workload == args.workload and args.n else WORKLOADS[workload]["n"])
        wcells = wn * wn if workload != "sphere" else 2 * wn * wn
        state, solver = build_problem(pyclaw, workload, wn, world, torch)
        solver.arithmetic = arithmetic or args.arithmetic
        if field == "developed" and workload in ("euler", "shallow"):
            # A smooth velocity field over the whole domain (SURVEY 8(d)): every interface has
            # non-zero jumps in every wave family, so the limiter, the entropy fix and the
            # transverse solves do their full work everywhere.  The initial data of the reference's
            # application alone leaves > 99 % of an 8192^2 grid at rest for the first few hundred
            # steps (zero waves: the limiter is skipped, the entropy fix exits early).
            xc = torch.as_tensor(state.grid.x.center, device=state.device)
            yc = torch.as_tensor(state.grid.y.center, device=state.device)
            bump = torch.sin(2 * np.pi * xc)[:, None] * torch.sin(2 * np.pi * yc)[None, :]
            rho = state.q[0].clone()
            state.q[1] = rho * 0.3 * bump
            state.q[2] = -rho * 0.2 * bump
            if workload == "euler":
                state.q[3] = state.q[3] + 0.5 * (state.q[1] ** 2 + state.q[2] ** 2) / rho
        solution = pyclaw.Solution(state)
        solver.setup(solution)
        solver.dt = solver.dt_initial
        solver.max_steps = 10 ** 9
        for _ in range(warmup):
            solver.evolve_to_time(solution)
        sampler = ClockSampler(local) if (sample_clocks and rank == 0) else None
        if sampler:
            sampler.start()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        accepted = 0
        ev0.record()
        for _ in range(steps):
            st = solver.evolve_to_time(solution)
            accepted += st['numsteps']
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        clocks = sampler.stop() if sampler else None
        if world > 1:
            tmax = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            ms = float(tmax.item())
            acc = torch.tensor([accepted], dtype=torch.float64, device="cuda")
            dist.all_reduce(acc, op=dist.ReduceOp.MIN)
            accepted = int(acc.item())
        value = wcells * world * accepted / (ms * 1e-3)
        return dict(value=value, ms=ms, accepted=accepted, clocks=clocks, state=state, solver=solver,
                    solution=solution)

    # The headline field: for the workloads whose application data is mostly at rest (Euler
    # shock-bubble, shallow-water dam break) the timed field is the developed one; the
    # application's own initial data is timed next to it and reported as config.quiescent_value.
    has_quiescent = args.workload in ("euler", "shallow")
    field = "developed" if (has_quiescent and not args.quiescent) else "application"
    quiescent = None
    if has_quiescent and field == "developed" and not args.no_quiescent_leg:
        rq = timed_run("application", min(args.steps, 10), max(args.warmup, 3), False)
        quiescent = {"value": rq["value"], "ms_per_step": rq["ms"] / min(args.steps, 10),
                     "what": "the application's own initial data (>99% of the cells at rest)"}
        del rq
        torch.cuda.empty_cache()
    # ---- the other BASELINE configurations, short runs, so that the driver's one line carries a
    # measured number for every config (configs[1] acoustics is a 1-GPU configuration) ----------
    others = None
    if args.workload == "euler" and not args.no_other_workloads and not args.n:
        others = {}
        for w in ("acoustics", "shallow", "sphere"):
            if w == "acoustics" and world > 1:
                continue
            ar = "fma" if FMA_ERR[w] <= 1e-12 else "strict"
            ksteps = 10 if w == "acoustics" else 5
            r = timed_run("developed" if w == "shallow" else "application", ksteps, 3, False, arithmetic=ar, workload=w)
            others[w] = {"workload": WORKLOADS[w]["label"], "value": r["value"], "unit": "cell-updates/s",
                         "ms_per_step": r["ms"] / ksteps, "steps": ksteps, "arithmetic": ar,
                         "field": "developed" if w == "shallow" else "application",
                         "step_frac_of_hbm_roofline": r["value"] / world * WORKLOADS[w]["balg"] / 1e9 / peaks()[0]}
            del r
            torch.cuda.empty_cache()
    other_build = None
    if not args.no_other_build:
        ob = "strict" if args.arithmetic == "fma" else "fma"
        ro = timed_run(field, min(args.steps, 10), max(args.warmup, 3), False, arithmetic=ob)
        other_build = {"arithmetic": ob, "value": ro["value"], "ms_per_step": ro["ms"] / min(args.steps, 10),
                       "field": field}
        del ro
        torch.cuda.empty_cache()
    run = timed_run(field, args.steps, max(args.warmup, 3), True)
    value, ms, accepted, clocks = run["value"], run["ms"], run["accepted"], run["clocks"]
    state, solver, solution = run["state"], run["solver"], run["solution"]
    if args.dump_outputs and rank == 0:
        # before the e2e leg below, which steps this solution further
        dump_outputs(args.dump_outputs, solution, solver)
    _lib.set_variant(args.arithmetic)

    # ---- e2e at N > 1: every rank uploads its slab from pinned host memory, takes one step
    # through the petclaw API (halo exchange + CFL all-reduce included) and downloads the result
    e2e_multi = None
    if world > 1 and not args.no_e2e:
        F = state._q
        host_in = torch.empty(F.cur.shape, dtype=torch.float64).pin_memory()
        host_out = torch.empty(F.cur.shape, dtype=torch.float64).pin_memory()
        host_in.copy_(F.cur)
        k = 3
        for it in range(k + 1):
            if it == 1:
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                acc_e = 0
            state._q.cur.copy_(host_in, non_blocking=True)
            st = solver.evolve_to_time(solution)
            host_out.copy_(state._q.cur, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            if it >= 1:
                acc_e += st['numsteps']
        e1.record()
        barrier()
        ems = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(ems, op=dist.ReduceOp.MAX)
        acc_t = torch.tensor([acc_e], dtype=torch.float64, device="cuda")
        dist.all_reduce(acc_t, op=dist.ReduceOp.MIN)
        nbytes = host_in.numel() * 8
        e2e_multi = {"value": cells_per_rank * world * float(acc_t.item()) / (float(ems.item()) * 1e-3),
                     "unit": "cell-updates/s", "h2d_bytes_per_step": nbytes * world,
                     "d2h_bytes_per_step": (nbytes + 8) * world, "steps": k,
                     "what": "per rank and step: pinned host slab -> H2D -> solver.evolve_to_time through the "
                             "petclaw API (NCCL halo exchange, CFL all-reduce) -> D2H of the new slab; "
                             "device-timed, max over ranks"}
        del host_in, host_out

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peak, peak_kind = peaks()
    # ---- per-kernel timing of the dominant kernel (CUDA events on the launch stream) ----
    roofline = None
    P = ctypes.byref(solver._problem)
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    F = state._q
    halo, solver._halo = solver._halo, None   # rank-local from here on: no collectives
    solver.apply_q_bcs(state)
    solver._halo = halo
    scratch = F.get_spare()
    kern = {}
    if args.workload in ("euler", "acoustics", "sphere"):
        scratch.copy_(F.cur)
        auxp = ptr(state._aux.cur) if state._aux is not None else None
        auxb = 16 * 8 if args.workload == "sphere" else 0   # each launch also streams the aux array once
        launches_per_step = _lib.load().clawb200_step2_launches(P)
        if launches_per_step == 1:
            # single-pass kernel (fused.cuh): both sweep families in one walk, q read once, written once
            parts = (("fused_step2_kernel", 3, 2 * wl["meqn"] * 8 + auxb),)
        else:
            parts = (("xsweep_kernel<TRANS>", 1, 2 * wl["meqn"] * 8 + auxb),
                     ("ysweep_kernel<TRANS>", 2, 3 * wl["meqn"] * 8 + auxb))
        for name, part, bytes_per_cell in parts:
            for rep in range(2):
                _lib.call("clawb200_step2_parts", P, ptr(F.cur), ptr(scratch), auxp, float(solver.dt), part,
                          ptr(solver._cfl_dev), stream)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 5
            e0.record()
            for rep in range(reps):
                _lib.call("clawb200_step2_parts", P, ptr(F.cur), ptr(scratch), auxp, float(solver.dt), part,
                          ptr(solver._cfl_dev), stream)
            e1.record()
            torch.cuda.synchronize()
            kern[name] = (e0.elapsed_time(e1) / reps, bytes_per_cell)
    else:
        launches_per_step = 3
        for rep in range(2):
            solver._stage(F.cur, None, scratch, 0, 0, 0, 1.0, 0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record()
        for rep in range(reps):
            solver._stage(F.cur, None, scratch, 0, 0, 0, 1.0, 0)
        e1.record()
        torch.cuda.synchronize()
        kern["sc2d_kernel"] = (e0.elapsed_time(e1) / reps, 2 * wl["meqn"] * 8)
    F.put_spare(scratch)
    dom = max(kern, key=lambda k: kern[k][0])
    kms, bpc = kern[dom]
    achieved = bpc * cells_per_rank / (kms * 1e-3) / 1e9
    traffic = None
    fp64 = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            prof = json.load(f)
            tr = prof.get(args.workload, {}).get(dom)
            if tr:  # measured DRAM bytes per cell per launch (ncu), scaled to this launch's cells
                traffic = tr["bytes_per_cell"] * cells_per_rank
            ipc = (tr or {}).get("fp64_inst_per_cell", {}).get(args.arithmetic)
            if ipc:
                # the resource that actually binds (DESIGN.md section 4): FP64-pipe instructions the
                # kernel executes (ncu count for this arithmetic build, developed field) per second,
                # against the FP64 issue rate measured on this GPU type by scratch/fp64_peak.cu
                rate = ipc * cells_per_rank / (kms * 1e-3)
                fp64 = {"achieved": rate / 1e12, "peak": prof["_fp64_peak_inst_per_s"] / 1e12,
                        "unit": "T FP64 inst/s", "frac": rate / prof["_fp64_peak_inst_per_s"],
                        "inst_per_cell_per_launch": ipc}
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_kind": peak_kind,
                "kernel_ms": kms, "algorithmic_bytes_per_cell_per_launch": bpc,
                "all_kernels_ms": {k: v[0] for k, v in kern.items()},
                "step_frac": value / world * wl["balg"] / 1e9 / peak,
                "step_algorithmic_bytes_per_cell": wl["balg"], "fp64_pipe": fp64}

    # ---- e2e: the f2py-shaped C ABI call with HOST buffers (H2D + kernels + D2H timed) ----
    e2e = None
    if not args.no_e2e and world > 1:
        e2e = e2e_multi
    elif not args.no_e2e and args.workload in ("euler", "acoustics"):
        mbc = solver.mbc
        nx = n + 2 * mbc
        host_in = torch.empty((nx, nx, wl["meqn"]), dtype=torch.float64).pin_memory()
        host_out = torch.empty((nx, nx, wl["meqn"]), dtype=torch.float64).pin_memory()
        # Fortran-ordered q(m,i,j) == C-ordered [j][i][m]
        host_in.copy_(F.cur.permute(1, 2, 0))
        from pyclaw_b200._lib import make_problem
        Ph = make_problem(2, wl["meqn"], wl["mwaves"], mbc, n, n, state.grid.d[0], state.grid.d[1],
                          solver._rp.rp_id, solver._rp.params(state.aux_global), solver.method, solver.mthlim)
        cflv = ctypes.c_double()
        hp = lambda t: ctypes.c_void_p(t.data_ptr())
        _lib.call("clawb200_step2_host", ctypes.byref(Ph), hp(host_in), hp(host_out), None, float(solver.dt),
                  ctypes.byref(cflv))
        k = 3
        t0 = time.perf_counter()
        for _ in range(k):
            _lib.call("clawb200_step2_host", ctypes.byref(Ph), hp(host_in), hp(host_out), None, float(solver.dt),
                      ctypes.byref(cflv))
        el = time.perf_counter() - t0
        nbytes = host_in.numel() * 8
        e2e = {"value": cells_per_rank * k / el, "unit": "cell-updates/s", "h2d_bytes_per_step": nbytes,
               "d2h_bytes_per_step": nbytes + 8, "steps": k,
               "what": "clawb200_step2_host (the f2py-shaped call): pinned host qold -> H2D -> layout kernel -> sweeps -> layout kernel -> D2H qnew every step, as a 3-stream pipeline of 128-row slabs",
               "resident_api": {"value": value, "unit": "cell-updates/s",
                                "what": "solver.evolve_to_time through the pyclaw API, q resident in HBM, "
                                        "8-byte CFL read back per step"}}
        del host_in, host_out
    elif not args.no_e2e:
        # no f2py-shaped host entry point exists for a whole SharpClaw / sphere step: upload the
        # padded field from pinned host memory, one step through the API, download the result
        host_in = torch.empty(F.cur.shape, dtype=torch.float64).pin_memory()
        host_out = torch.empty(F.cur.shape, dtype=torch.float64).pin_memory()
        host_in.copy_(F.cur)
        k, acc_e = 3, 0
        for it in range(k + 1):
            if it == 1:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
            state._q.cur.copy_(host_in, non_blocking=True)
            st = solver.evolve_to_time(solution)
            host_out.copy_(state._q.cur, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            if it >= 1:
                acc_e += st['numsteps']
        el = time.perf_counter() - t0
        nbytes = host_in.numel() * 8
        e2e = {"value": cells_per_rank * acc_e / el, "unit": "cell-updates/s", "h2d_bytes_per_step": nbytes,
               "d2h_bytes_per_step": nbytes + 8 * 3, "steps": k,
               "what": "pinned host q -> H2D -> solver.evolve_to_time through the pyclaw API -> D2H of the new q, every step"}
        del host_in, host_out

    # ---- CPU baseline on a bounded sample (rank 0, N = 1 only) ------------------------
    cpu = None
    if not args.no_cpu and world == 1 and args.workload != "sphere":
        ncores = os.cpu_count() or 1
        ncpu = 1024
        v, k, el = time_cpu(args.workload, ncpu, ncores, 12.0)
        cpu = {"value": v, "unit": "cell-updates/s", "cores": ncores, "kind": "port",
               "sample": "%d steps on a %dx%d sample of the workload in %.1f s, y-slab threads over the oracle C port" % (k, ncpu, ncpu, el)}
        # the reference's Fortran is serial: the same port on one core (SURVEY section 8d)
        v1, k1, el1 = time_cpu(args.workload, 512, 1, 4.0)
        cpu["single_core"] = {"value": v1, "unit": "cell-updates/s", "cores": 1,
                              "sample": "%d steps on a 512x512 sample in %.1f s" % (k1, el1)}

    bc_launches = sum(1 for b in solver.bc_lower + solver.bc_upper if b in (1, 2, 3))
    # kernels of libclawb200.so per accepted step: boundary fills + sweeps (classic), or
    # per Runge-Kutta stage: boundary fills + one fused stage kernel (SharpClaw SSP33)
    if args.workload == "shallow":
        per_step_launches = 3 * (bc_launches + 1)
    elif world > 1:
        # overlapped halo path: x-BC fills run twice, the sweeps as interior + 2 boundary ranges
        per_step_launches = 2 * bc_launches + 3 * launches_per_step
    else:
        per_step_launches = bc_launches + launches_per_step
    line = {
        "metric": "cell-updates/s", "value": value, "unit": "cell-updates/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": wl["label"], "cells_per_gpu": cells_per_rank, "accepted_steps": accepted,
                   "l2": "inputs larger than L2 (%.1f GB per field)" % (cells_per_rank * wl["meqn"] * 8 / 1e9),
                   "parallelism": "y-slabs x%d" % world,
                   "arithmetic": args.arithmetic,
                   "arithmetic_note": (("strict IEEE build, -fmad=false: bit for bit against the oracle" +
                                        ("; the fma build differs by 1.0e-11 over the reference-style test run of this "
                                         "workload, the strict build on input moved by one unit in the last place by 1.5e-11 "
                                         "(profiles/r2/fma_study_r2i.json): the run's own conditioning is above 1e-12"
                                         if args.workload == "shallow" else "")) if args.arithmetic == "strict"
                                       else "fma build (-fmad=true, quotients within 1.5 ulp): relative L-inf %.1e against the "
                                            "strict build over the reference's own test run of this workload; north_star asks 1e-12"
                                            % FMA_ERR[args.workload]),
                   "fma_rel_linf_vs_strict": FMA_ERR[args.workload],
                   "other_build": other_build,
                   "field": field, "quiescent_value": quiescent["value"] if quiescent else None,
                   "quiescent": quiescent},
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "e2e": e2e,
        "gpu_launches": args.steps * per_step_launches,
        "other_workloads": others,
    }
    if world > 1:
        line["partition_parity"] = partition_parity
        line["ranks"] = world
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
