#!/usr/bin/env python
"""Times the unstructured front-end kernels alone at HBM scale (4^PAMG_BENCH_UNSTR_KP triangles, default 4^12 = 16.7 M):
k_unstr_explicit (144 B/element), k_assemble_bsr (456 B/element, with and without the diffusion blocks), k_bsr_spmv
(352 B/element).  With PAMG_BENCH_UNSTR_FIELD=1 (default) the explicit step and both assemblies are also timed with a
rotating nodal velocity field u_ele (pamg_unstr_set_velocity; +48 B/element read: explicit 192 B, assembly 120 B read +
384 B written, +24 B with the diffusion blocks), the uniform and the field runs alternating so that both see the same
machine.  Prints one JSON line with the card's name and power limit.  PAMG_LIB selects an A/B build (tools/ab_build.sh)."""
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
    kp = int(os.environ.get("PAMG_BENCH_UNSTR_KP", "12"))
    with_field = os.environ.get("PAMG_BENCH_UNSTR_FIELD", "1") != "0"
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        peak = 6555.2
    um = pkg.Mesh.synthetic(kp, 1)
    g = pkg.SemiImplicitIterative(pkg.default_params(n_split=1, multi_levels=1, u_x=0.9, u_y=0.3, dt=1e-3), pkg.Mesh.synthetic(1, 1))
    g.set_unstructured(um)
    E = um.U
    T0 = np.random.Generator(np.random.MT19937(7)).random((E, 3))
    g._ck(g.L.pamg_unstr_upload(g.h, T0))
    out = {"elements": E, "card": card(), "peak_gbs": peak,
           "lib": os.path.basename(pkg.pamg.LIB_PATH) if hasattr(pkg, "pamg") else ""}
    c = um.X.reshape(-1, 2).mean(axis=0)
    rot = np.stack([-(um.X[:, :, 1] - c[1]), um.X[:, :, 0] - c[0]], axis=2) if with_field else None

    def timed(fn, reps, warm=2):
        for _ in range(warm):
            fn()
        g.sync()
        g.event_record(8)
        for _ in range(reps):
            fn()
        g.event_record(9)
        g.sync()
        return g.elapsed_ms(8, 9) / reps

    area = 0.5 * np.abs((um.X[:, 0, 0] - um.X[:, 2, 0]) * (um.X[:, 1, 1] - um.X[:, 2, 1])
                        - (um.X[:, 0, 1] - um.X[:, 2, 1]) * (um.X[:, 1, 0] - um.X[:, 2, 0]))
    dt_i = 4.0 * float(np.sqrt(area.min()))
    # (name, bytes per element uniform, bytes per element with the field, call)
    cases = [("explicit", 144.0, 192.0, lambda: g._ck(g.L.pamg_explicit_step(g.h, 1e-6, 0.9, 0.3, 0.0, 1, 10, 10, 0, 0)), 3, 10.0),
             ("assemble", 456.0, 504.0, lambda: g.implicit_assemble(dt_i, 0.9, 0.3, use_dir=True), 10, 1.0),
             ("assemble_diff", 480.0, 528.0, lambda: g.implicit_assemble(dt_i, 0.9, 0.3, use_dir=True, k=1.0), 10, 1.0)]
    rounds = 3 if with_field else 1
    for name, b_u, b_f, fn, reps, per in cases:
        tu, tf = [], []
        for _ in range(rounds):
            g.set_velocity(None)
            tu.append(timed(fn, reps) / per)
            if with_field:
                g.set_velocity(rot)
                tf.append(timed(fn, reps) / per)
        t = min(tu)
        out[name + "_ms"] = t; out[name + "_frac"] = b_u * E / (t * 1e-3) / 1e9 / peak
        out[name + "_ns_per_elem"] = t * 1e6 / E
        if with_field:
            t = min(tf)
            out[name + "_field_ms"] = t; out[name + "_field_frac"] = b_f * E / (t * 1e-3) / 1e9 / peak
            out[name + "_field_ns_per_elem"] = t * 1e6 / E
            out[name + "_field_over_uniform"] = min(tf) / min(tu)
            out[name + "_spread"] = [max(tu) / min(tu), max(tf) / min(tf)]
    out["bytes_per_elem"] = {n: [b_u, b_f] for n, b_u, b_f, *_ in cases}
    g.set_velocity(None)
    g.implicit_assemble(dt_i, 0.9, 0.3, use_dir=True)
    t = g.implicit_spmv_ms(20)
    out["spmv_ms"] = t; out["spmv_frac"] = 352.0 * E / (t * 1e-3) / 1e9 / peak
    print(json.dumps(out))
    g.close()


if __name__ == "__main__":
    main()
