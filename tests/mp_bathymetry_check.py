"""Run under torchrun with 2 ranks (one GPU each): the seamount2d application (shallow water over
bathymetry, y-slab partition, aux halo exchange) must equal the single-GPU run bit for bit, split and
unsplit."""
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
    ok = True
    for dim_split in (True, False):
        kw = dict(mx=48, my=24 * world, tfinal=0.1, dim_split=dim_split)
        cp = apps.seamount2d(petsc=True, **kw)
        st = cp.frames[-1].state
        qp = np.asarray(st._partition.gather_interior(st))
        if rank == 0:
            qs = np.asarray(apps.seamount2d(petsc=False, **kw).frames[-1].q)
            same = np.array_equal(qp, qs) and np.isfinite(qs).all()
            print("seamount2d dim_split=%s: %d ranks, bit-identical=%s maxdiff=%g"
                  % (dim_split, world, same, np.abs(qp - qs).max()), flush=True)
            ok &= same
    flag = torch.tensor([1.0 if ok else 0.0], device='cuda')
    dist.broadcast(flag, 0)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
