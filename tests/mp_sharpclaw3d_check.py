"""Run under torchrun with 2 ranks (one GPU each): the euler3d application with SharpClawSolver3D
(z-slab partition, mbc = 3 halos) must equal the single-GPU run bit for bit."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))


def main():
    import petclaw
    import apps
    rank, world = petclaw.init('nccl')
    kw = dict(mx=20, my=16, mz=8 * world, tfinal=0.02, solver_type='sharpclaw')
    cp = apps.euler3d(petsc=True, **kw)
    st = cp.frames[-1].state
    qp = np.asarray(st._partition.gather_interior(st))
    ok = True
    if rank == 0:
        qs = np.asarray(apps.euler3d(petsc=False, **kw).frames[-1].q)
        ok = np.array_equal(qp, qs) and np.isfinite(qs).all()
        print("euler3d sharpclaw: %d ranks, bit-identical=%s maxdiff=%g" % (world, ok, np.abs(qp - qs).max()),
              flush=True)
    flag = torch.tensor([1.0 if ok else 0.0], device='cuda')
    dist.broadcast(flag, 0)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
