#!/usr/bin/env python
"""Block Jacobi against the flow-ordered block Gauss-Seidel preconditioner (pamg_implicit_set_precond) for one implicit time
step (pamg_implicit_step, ntime = nits = 1, tol 1e-10) on the synthetic meshes 4^11 and 4^12: CFL 1, 4, 16, 64 and 256, pure
advection and a small diffusion (cell Peclet number 10), the uniform velocity u = (0.9, 0.3) and the rotating field of
tools/unstr_bench.py.  The two preconditioners alternate in the same process, 3 rounds each; the fastest round is reported.
Per case: solve ms (device events around the step, host synchronisations included), Krylov iterations and relative residual
for both; ms per sweep application, the number of flow levels, us per level and lagged edges; the host set-up of the levels
(mask kernel + download, pamg_flow_levels, upload).  Prints one JSON line with the card's name and power limit.

    python tools/precond_bench.py [--kp 11,12] [--cfl 1,4,16,64,256] [--rounds 3] [--max-iters 1000]"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("p-a_multigrids_b200")


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:      # the numbers still print; the card is then unknown
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kp", default="11,12")
    ap.add_argument("--cfl", default="1,4,16,64,256")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--max-iters", type=int, default=1000)
    args = ap.parse_args()
    if pkg.device_count() < 1:
        raise SystemExit("precond_bench needs a CUDA device")
    out = {"card": card(), "tol": 1e-10, "max_iters": args.max_iters, "rounds": args.rounds, "cases": []}
    for kp in (int(k) for k in args.kp.split(",")):
        um = pkg.Mesh.synthetic(kp, 1)
        E = um.U
        g = pkg.SemiImplicitIterative(pkg.default_params(), pkg.Mesh.synthetic(0, 1))
        g.set_unstructured(um)
        X = um.X
        area = 0.5 * np.abs((X[:, 0, 0] - X[:, 2, 0]) * (X[:, 1, 1] - X[:, 2, 1]) - (X[:, 0, 1] - X[:, 2, 1]) * (X[:, 1, 0] - X[:, 2, 0]))
        h = float(np.sqrt(area.min()))
        c = X.reshape(-1, 2).mean(axis=0)
        rot = np.stack([-(X[:, :, 1] - c[1]), X[:, :, 0] - c[0]], axis=2)
        cx = X.mean(axis=1)
        L = float(X.max() - X.min())
        r2 = (cx[:, 0] - c[0]) ** 2 + (cx[:, 1] - c[1]) ** 2
        T0 = np.repeat(np.exp(-r2 / (0.1 * L) ** 2)[:, None], 3, axis=1)
        for vel in ("uniform", "rotating"):
            g.set_velocity(rot if vel == "rotating" else None)
            umax = float(np.hypot(0.9, 0.3)) if vel == "uniform" else float(np.abs(rot).max())
            for kdiff in (0.0, 0.1 * umax * h):
                for cfl in (float(v) for v in args.cfl.split(",")):
                    dt = cfl * h / umax
                    case = {"elements": E, "velocity": vel, "k": kdiff, "cfl": cfl, "dt": dt}
                    g.implicit_assemble(dt, 0.9, 0.3, use_dir=True, k=kdiff)
                    g.implicit_set_precond("flow_gs")
                    level, nlevels, lagged = g.implicit_flow_levels()     # built here (or kept from the last case)
                    sweep_ms, setup = g.implicit_flow_time(5)
                    case.update({"nlevels": nlevels, "lagged": lagged, "sweep_ms": sweep_ms,
                                 "us_per_level": 1e3 * sweep_ms / nlevels,
                                 "setup_ms": {"mask": setup[0], "levels": setup[1], "upload": setup[2]}})
                    res = {p: [] for p in ("block_jacobi", "flow_gs")}
                    for _ in range(args.rounds):
                        for p in ("block_jacobi", "flow_gs"):
                            g.implicit_set_precond(p)
                            g._ck(g.L.pamg_unstr_upload(g.h, T0))
                            it = C.c_int(0); rr = C.c_double(0.0)
                            g.sync(); g.event_record(8)
                            g._ck(g.L.pamg_implicit_step(g.h, 1, 1, 1e-10, args.max_iters, C.byref(it), C.byref(rr)))
                            g.event_record(9); g.sync()
                            res[p].append((g.elapsed_ms(8, 9), it.value, rr.value))
                    for p, runs in res.items():
                        ms = [r[0] for r in runs]
                        case[p] = {"solve_ms": min(ms), "spread": max(ms) / min(ms), "iters": runs[0][1],
                                   "relres": runs[0][2]}
                    case["flow_over_jacobi"] = case["flow_gs"]["solve_ms"] / case["block_jacobi"]["solve_ms"]
                    out["cases"].append(case)
                    print(json.dumps(case), file=sys.stderr, flush=True)
        g.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
