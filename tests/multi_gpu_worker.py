"""Rank worker for tests/test_gpu_multi.py: each rank owns one block of parents on its own GPU; after Jacobi
sweeps, a residual evaluation and a V-cycle solve the gathered field must equal the single-GPU run."""
import os
import sys

import numpy as np
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from pamg_pkg import pamg  # noqa: E402


def main():
    dist.init_process_group(backend="gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    local = int(os.environ.get("LOCAL_RANK", rank))
    kp, n = 2, 6
    mesh = pamg.Mesh.synthetic(kp, world)
    per = 4 ** kp
    pf = np.arange(world + 1, dtype=np.int32) * per
    # PAMG_TEST_THETA != 1: the told values of the cut faces travel too (old-time branch of get_RHS, exchange_told)
    params = pamg.default_params(n_split=n, multi_levels=n, u_x=0.9, u_y=0.3, theta=float(os.environ.get("PAMG_TEST_THETA", "1.0")))
    g = pamg.SemiImplicitIterative(params, mesh, device=local, nparts=world, part_first=pf, my_part=rank)
    ids = [pamg.get_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    g.comm_init(ids[0], world, rank)
    rng = np.random.Generator(np.random.MT19937(4242))
    C = 4 ** n
    T = rng.random((mesh.U, C, 3)); Told = rng.random((mesh.U, C, 3))
    sl = slice(rank * per, (rank + 1) * per)
    g.upload(pamg.TNONLIN, 1, T[sl]); g.copy(1, pamg.TNEW, pamg.TNONLIN); g.upload(pamg.TOLD, 1, Told[sl])
    g.smoother(1, pamg.JACOBI, 3)
    g.smoother(1, pamg.GAUSS_SEIDEL, 2)
    g.copy(1, pamg.TNEW, pamg.TNONLIN)
    g.update_overlaps(1)
    l2, linf = g.get_residual(1)
    mine = g.download(pamg.TNONLIN, 1)
    cyc, hist = g.vcycle_solve(solver=pamg.GAUSS_SEIDEL, max_cycles=40, tol=1e-8)
    sol = g.download(pamg.TNONLIN, 1)
    parts = [None] * world
    dist.all_gather_object(parts, (mine, sol, l2, linf, cyc))
    ok = True
    if rank == 0:
        ref = pamg.SemiImplicitIterative(params, mesh, device=local)
        ref.upload(pamg.TNONLIN, 1, T); ref.copy(1, pamg.TNEW, pamg.TNONLIN); ref.upload(pamg.TOLD, 1, Told)
        ref.smoother(1, pamg.JACOBI, 3)
        ref.smoother(1, pamg.GAUSS_SEIDEL, 2)
        ref.copy(1, pamg.TNEW, pamg.TNONLIN)
        ref.update_overlaps(1)
        rl2, rlinf = ref.get_residual(1)
        full = ref.download(pamg.TNONLIN, 1)
        rcyc, rhist = ref.vcycle_solve(solver=pamg.GAUSS_SEIDEL, max_cycles=40, tol=1e-8)
        rsol = ref.download(pamg.TNONLIN, 1)
        got = np.concatenate([p[0] for p in parts]); gsol = np.concatenate([p[1] for p in parts])
        e1 = np.linalg.norm(got - full) / np.linalg.norm(full)
        e2 = np.max(np.abs(gsol - rsol))
        ok = (e1 <= 1e-13 and abs(parts[0][2] - rl2) <= 1e-12 * rl2 and abs(parts[0][3] - rlinf) <= 1e-12 * rlinf
              and parts[0][4] == rcyc and e2 <= 1e-10)
        print("MULTI_OK" if ok else "MULTI_FAIL", e1, e2, parts[0][2], rl2, parts[0][4], rcyc, flush=True)
    dist.barrier()
    g.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
