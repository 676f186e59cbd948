"""Micro-benchmark of the cut-face halo exchange (update_overlaps across GPUs): time per pamg_update_overlaps call
on the c5 partition (256 parents per GPU, n_split 8).  torchrun --nproc-per-node N tools/halo_microbench.py"""
import os
import sys

import numpy as np
import torch.distributed as dist

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from pamg_pkg import pamg  # noqa: E402


def main():
    dist.init_process_group(backend="gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    local = int(os.environ.get("LOCAL_RANK", rank))
    kp, n = 4, 8
    mesh = pamg.Mesh.synthetic(kp, world)
    per = 4 ** kp
    pf = np.arange(world + 1, dtype=np.int32) * per
    params = pamg.default_params(n_split=n, multi_levels=1, u_x=0.9, u_y=0.3)
    g = pamg.SemiImplicitIterative(params, mesh, device=local, nparts=world, part_first=pf, my_part=rank)
    ids = [pamg.get_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    g.comm_init(ids[0], world, rank)
    g.fill(pamg.TNONLIN, 1, 1.0)
    for what, fn in (("update_overlaps", lambda: g.update_overlaps(1)), ("jacobi_sweep", lambda: g.smoother(1, pamg.JACOBI, 1))):
        for _ in range(20):
            fn()
        g.sync(); dist.barrier()
        g.event_record(0)
        reps = 200
        for _ in range(reps):
            fn()
        g.event_record(1)
        g.sync(); dist.barrier()
        ms = g.elapsed_ms(0, 1) / reps
        allms = [None] * world
        dist.all_gather_object(allms, ms)
        if rank == 0:
            print(f"{what}: {max(allms) * 1e3:.1f} us per call (PAMG_P2P={os.environ.get('PAMG_P2P', '1')}, ranks {world})", flush=True)
    g.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
