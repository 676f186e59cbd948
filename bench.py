#!/usr/bin/env python
"""bench.py -- DG DOF-updates/s of the smoother sweep (and V-cycle time to 1e-8) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--scaling weak|strong] [--workload c5|c4] [--impl reference]
    torchrun --nproc-per-node N ... bench.py --gpus N --steps K --warmup W      (N > 1: one process per GPU)
    python bench.py --gpus N --single-process                                   (N > 1: one host thread drives N GPUs)
    python bench.py ... --dump-outputs DIR      (DIR/tnonlin.npy: the smoothed field of the last timed step, seeded sample)

Workload (BASELINE.json configs[4], SURVEY 8(d) "c5"): synthetic semi-structured triangle mesh, kp = 4 (256 parents per
super-triangle), n_split = 8 -> 16 777 216 P1 DG elements = 50.3 M DOFs.  Weak scaling (default): every GPU holds one
super-triangle (N GPUs = N super-triangles coupled through ordinary parent faces).  Strong scaling: ONE super-triangle
(c5, or c4 = n_split 7 with 4 194 304 elements) is cut into N contiguous blocks of parents.
One step = one call of the reference's `smoother` (transport_tri_semi.F90:543-722) on level 1: n_smooth = 4 Jacobi
sweeps, each with its update_overlaps.  Fields (403 MB each at c5) are far larger than the 126 MB L2, so no flush is
needed between timed iterations.  After the timed regions one more sweep from a seeded field is checked against the
CPU oracle on the parents along the GPU cuts (`parity_check`): the run exits non-zero if the cut-face strips are not
bit-exact or the swept field differs.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the benchmark leaves the source tree untouched (it may be read-only)

KP, NSMOOTH = 4, 4
DUMP_VALUES = 1 << 22                # float64 values --dump-outputs writes per run (32 MB)
NSPLIT_OF = {"c5": 8, "c4": 7}
BYTES_PER_DOF_JACOBI = 24.0      # read T, read b, write T' (SURVEY 8(d))
METRIC = "DG DOF-updates/s per smoother sweep"
UNIT = "DOF-updates/s"


KERNEL_NAMES = {
    "win": "k_element_win2<JACOBI,face> (ring of 8 field tiles in shared memory via 1-D TMA, all neighbours from the ring, "
           "producer warp + named barriers; the producer warp also writes the next sweep's halo strips)",
    "tma1d": "k_element_tma<JACOBI,face> (pipelined 1-D TMA tiles, vertical neighbour by global load)",
    "direct2": "k_element_direct2<JACOBI,face>",
}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def bind_to_gpu_numa(gpu):
    """Pin this rank to the CPUs of the NUMA node its GPU hangs off BEFORE any pinned host buffer is allocated: the pages are
    then local to that node and the PCIe copies of the end-to-end arm do not cross the socket interconnect (with N ranks on
    one box the unpinned default made every rank's copies share one memory path).  Returns what was done, for the JSON line."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(gpu), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bus = bus[-12:]                                   # sysfs: 0000:xx:yy.z (nvidia-smi prints an 8-digit domain)
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return {"numa_node": None, "note": "single NUMA node (sysfs reports -1)"}
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if not use:
            return {"numa_node": node, "note": "no CPU of that node is in this process's affinity mask"}
        os.sched_setaffinity(0, use)
        return {"numa_node": node, "cpus_bound": len(use)}
    except Exception as e:     # noqa: BLE001 - best effort, the run goes on unbound
        return {"numa_node": None, "note": f"not bound: {type(e).__name__}"}


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def lines(self):
        try:
            with open(self.f.name) as f:
                return sum(1 for _ in f)
        except OSError:
            return 0

    def wait_first_sample(self, timeout=5.0):
        """nvidia-smi needs a few hundred ms to start: block until it has written a sample, return the line count."""
        if self.p is None:
            return 0
        t0 = time.time()
        while self.lines() == 0 and time.time() - t0 < timeout:
            time.sleep(0.05)
        return self.lines()

    def stop(self, skip=0):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for i, line in enumerate(self.f):
            if i < skip:
                continue            # samples taken before the timed region (warm-up)
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        self.f.close()
        os.unlink(self.f.name)
        if sm:
            out["sm_mhz"] = float(np.median(sm)); out["sm_max_mhz"] = float(max(mx)); out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


def oracle_api():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_api as orc       # CPU oracle: the checker (parity_check) and the cpu_baseline / --impl reference legs
    return orc


def cpu_smoother_rate(orc, nsplit, kp, threads, sweeps):
    """DOF-updates/s of the oracle's smoother (Jacobi, face block on) on 4**kp parents x 4**nsplit children."""
    mesh = orc.synthetic_mesh(kp, 1)
    p = orc.intended_params(nsplit, 1, dt=1e-3, u=(0.9, 0.3))
    s = orc.Semi(p, mesh["X"], mesh["neig"], mesh["fneig"], mesh["dir"])
    rng = np.random.Generator(np.random.MT19937(20221))
    s.field(orc.TNONLIN)[:] = rng.random(s.field(orc.TNONLIN).shape)
    s.field(orc.TOLD)[:] = rng.random(s.field(orc.TOLD).shape)
    orc.lib().orc_semi_set_threads(threads)
    t0 = time.perf_counter()
    s.smooth(1, 1, sweeps)
    dt = time.perf_counter() - t0
    ndof = s.field(orc.TNEW).size
    del s
    return ndof * sweeps / dt, ndof, dt


def workload_config(n, nsplit, scaling, single_process=False):
    per = 4 ** (KP + nsplit)
    name = "c5" if nsplit == 8 else "c4"
    who = ("one process drives all GPUs (pamg_create_multi), " if single_process else "") if n > 1 else ""
    if scaling == "strong":
        size = f"{per} elements ({3 * per / 1e6:.1f}M DOFs) in TOTAL, cut into {n} contiguous blocks of parents"
    else:
        size = f"{per} elements ({3 * per / 1e6:.1f}M DOFs) per GPU"
    return {"workload": f"{name}: synthetic semi-structured triangles, kp={KP} (256 parents) x n_split={nsplit} = {size}; "
                        f"smoother = {NSMOOTH} Jacobi sweeps + update_overlaps on level 1",
            "elements_per_gpu": per if scaling == "weak" else per // n, "n_split": nsplit,
            "parents_per_gpu": 4 ** KP if scaling == "weak" else 4 ** KP // n,
            "n_smooth": NSMOOTH, "face_terms": 1, "velocity": [0.9, 0.3], "dt": 1e-3, "k": 1.0, "omega": 0.8,
            "parallelism": f"parent-partition x{n}, {who}cut-face values stored straight into the peer GPU's memory over NVLink by "
                           "the producer warps of the sweep kernels (flagged words, unpack launch between sweeps), norms "
                           "all-reduced, small coarse levels agglomerated on GPU 0",
            "l2_policy": "inputs larger than L2 (403 MB per field at c5)"}


def run_reference(args, rank):
    """Reference arm: the reference's own CPU algorithm (C++ restatement; the Fortran cannot be compiled here) on the host
    cores, all threads, same metric / config.  Loads nothing of the product: the mesh comes from the oracle side too."""
    if rank != 0:
        return
    orc = oracle_api()
    nsplit = NSPLIT_OF[args.workload]
    cores = os.cpu_count() or 1
    # calibrate on 16 parents, then pick the sample so that the whole run stays within ~2 minutes
    rate, _, _ = cpu_smoother_rate(orc, nsplit, 2, cores, 1)
    total = args.steps + args.warmup
    kp = KP
    while kp > 1 and (3 * 4 ** (kp + nsplit) * NSMOOTH * total) / rate > 120.0:
        kp -= 1
    mesh = orc.synthetic_mesh(kp, 1)
    p = orc.intended_params(nsplit, 1, dt=1e-3, u=(0.9, 0.3))
    s = orc.Semi(p, mesh["X"], mesh["neig"], mesh["fneig"], mesh["dir"])
    rng = np.random.Generator(np.random.MT19937(20221))
    s.field(orc.TNONLIN)[:] = rng.random(s.field(orc.TNONLIN).shape)
    s.field(orc.TOLD)[:] = rng.random(s.field(orc.TOLD).shape)
    orc.lib().orc_semi_set_threads(cores)
    for _ in range(args.warmup):
        s.smooth(1, 1, NSMOOTH)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        s.smooth(1, 1, NSMOOTH)
    dt = time.perf_counter() - t0
    ndof = s.field(orc.TNEW).size
    value = ndof * NSMOOTH * args.steps / dt
    sample = f"{4 ** kp} of 256 parents x 4^{nsplit} children ({ndof} DOFs), {NSMOOTH} Jacobi sweeps per step"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus, nsplit, args.scaling),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference Fortran cannot be compiled in this image (no Fortran compiler); this is the fp64 C++ "
                "restatement of its algorithm (oracle/), OpenMP over parents",
    }
    print(json.dumps(line), flush=True)


def seeded_parent_field(gids, C_children, seed):
    """field values that depend only on the GLOBAL parent number, so every rank (and the oracle) generates the same ones"""
    out = np.empty((len(gids), C_children, 3))
    for i, g in enumerate(gids):
        out[i] = np.random.Generator(np.random.MT19937(seed + int(g))).random((C_children, 3))
    return out


def dump_sample(field, nvalues):
    """The whole field when it has at most nvalues entries, else the entries at a fixed, seeded set of flat indices
    (sorted, depending only on the field size), so that two builds can be compared value for value."""
    flat = field.reshape(-1)
    if flat.size <= nvalues:
        return flat.copy()
    keep = np.zeros(flat.size, bool)
    keep[np.random.Generator(np.random.MT19937(4242)).integers(0, flat.size, nvalues)] = True
    return flat[keep]


def parity_check(pkg, orc, g, mesh, first, U_local, nsplit, gather, part_first, nshare):
    """One Jacobi sweep from a seeded field: the parents along the GPU cuts (or the first 8 parents on one GPU) and their
    halo strips against the CPU oracle run on those parents plus all their neighbours."""
    C_ch = 4 ** nsplit
    local = np.arange(first, first + U_local)
    T = seeded_parent_field(local, C_ch, 777)
    Told = seeded_parent_field(local, C_ch, 999)
    g.upload(pkg.TNONLIN, 1, T); g.copy(1, pkg.TNEW, pkg.TNONLIN); g.upload(pkg.TOLD, 1, Told)
    g.update_overlaps(1)
    strips = g.overlap(1)                                    # [U_local][3][S][3] of the start field (received over NVLink on cut faces)
    g.smoother(1, pkg.JACOBI, 1)
    after = g.download(pkg.TNONLIN, 1)
    nb = mesh.neig[local] - 1                               # 0-based global neighbours, -1 = domain boundary
    owner = np.searchsorted(part_first, np.arange(mesh.U), side="right") - 1
    cut = np.any((nb >= 0) & (owner[np.maximum(nb, 0)] != owner[local][:, None]), axis=1)
    check = local[cut] if cut.any() else local[:8]
    sub = sorted(set(check.tolist()) | set(int(q) for q in nb[check - first].ravel() if q >= 0))
    pos = {gid: i for i, gid in enumerate(sub)}
    sm = pkg.Mesh.from_arrays(mesh.X[sub])                   # same parents in the same order, neighbours rebuilt
    o = orc.Semi(orc.intended_params(nsplit, 1, dt=1e-3, u=(0.9, 0.3)), sm.X, sm.neig, sm.fneig, sm.dir)
    orc.lib().orc_semi_set_threads(max(1, min(os.cpu_count() or 1, 16) // nshare))
    o.field(orc.TNONLIN)[:] = seeded_parent_field(sub, C_ch, 777)
    o.field(orc.TOLD)[:] = seeded_parent_field(sub, C_ch, 999)
    o.field(orc.TNEW)[:] = o.field(orc.TNONLIN)
    o.update_overlaps(1)
    ostrips = o.overlap(1).copy()
    o.smooth(1, 1, 1)
    oafter = o.field(orc.TNONLIN)
    idx_o = np.array([pos[int(gid)] for gid in check])
    idx_g = check - first
    # strips of faces between parents are copies of field values: bit-exact; Dirichlet entries (sin on device vs libm): 1e-13
    interior_face = mesh.neig[check] != 0
    sg, so = strips[idx_g], ostrips[idx_o]
    bit_exact = bool(np.array_equal(sg[interior_face], so[interior_face]))
    dir_ok = bool(np.allclose(sg[~interior_face], so[~interior_face], rtol=0, atol=1e-13))
    num = float(np.linalg.norm(after[idx_g] - oafter[idx_o])); den = float(np.linalg.norm(oafter[idx_o]))
    mine = {"parents_checked": int(len(check)), "cut_parents": int(cut.sum()), "rel_l2": num / den,
            "strips_bit_exact": bit_exact and dir_ok}
    allr = gather(mine)
    return {"ranks": len(allr), "parents_checked": sum(r["parents_checked"] for r in allr),
            "cut_parents": sum(r["cut_parents"] for r in allr), "max_rel_l2": max(r["rel_l2"] for r in allr),
            "strips_bit_exact": all(r["strips_bit_exact"] for r in allr), "tolerance": 1e-12,
            "against": "CPU oracle on the checked parents + all their neighbours, one Jacobi sweep from a seeded field"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="pamg")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--workload", default="c5", choices=["c5", "c4"])
    ap.add_argument("--single-process", action="store_true", help="N > 1 GPUs driven by ONE host thread (pamg_create_multi)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-vcycle", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the other kernels of the path (GS, residual, unstructured)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the level-1 field after the last timed step to DIR/tnonlin.npy (float64; a fixed, seeded "
                         "sample of at most 32 MB; with several ranks one file per rank, tnonlin_rank<R>.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # watchdog: a run that makes no progress for this long dumps every thread's stack and exits instead of holding the box
    wd = int(os.environ.get("PAMG_BENCH_WATCHDOG_S", "900"))
    if wd > 0:
        import faulthandler
        faulthandler.dump_traceback_later(wd, exit=True)
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the CUDA path, not to --impl reference")
        run_reference(args, rank)
        return
    single = args.single_process and world == 1 and args.gpus > 1
    if world != args.gpus and not single:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N > 1 (or pass --single-process)")
    args.warmup = max(args.warmup, 3)
    affinity0 = os.sched_getaffinity(0)
    binding = bind_to_gpu_numa(local) if os.environ.get("PAMG_BENCH_BIND", "1") != "0" else {"numa_node": None, "note": "PAMG_BENCH_BIND=0"}
    nsplit = NSPLIT_OF[args.workload]
    pkg = importlib.import_module("p-a_multigrids_b200")
    if pkg.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    ngpu = args.gpus if single else world        # GPUs of the whole job

    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group(backend="gloo")   # control plane only; the data path is inside libpamg_cuda

    def barrier():
        if dist is not None:
            dist.barrier()

    def allmax(v):
        if dist is None:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather(obj):
        if dist is None:
            return [obj]
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    # ---- set-up: mesh, partition, handle ------------------------------------------------------------
    per = 4 ** KP
    if args.scaling == "weak":
        mesh = pkg.Mesh.synthetic(KP, ngpu)
        part_first = np.arange(ngpu + 1, dtype=np.int32) * per
    else:
        mesh = pkg.Mesh.synthetic(KP, 1)
        part_first = np.array([per * i // ngpu for i in range(ngpu + 1)], dtype=np.int32)
    # (`solver` only matters for pamg_timestep_host, which takes it from the handle like the reference's literal argument;
    # the timed smoother calls pass theirs explicitly)
    params = pkg.default_params(n_split=nsplit, multi_levels=nsplit, n_smooth=NSMOOTH, solver=pkg.GAUSS_SEIDEL,
                                u_x=0.9, u_y=0.3, dt=1e-3)
    if os.environ.get("PAMG_BENCH_FACE") == "0":      # experiment only: volume terms only (HEAD's operator)
        params.face_terms = 0
    if single:
        g = pkg.SemiImplicitIterative(params, mesh, devices=list(range(ngpu)))
        first, U_local = 0, mesh.U
    else:
        g = pkg.SemiImplicitIterative(params, mesh, device=local, nparts=world, part_first=part_first, my_part=rank)
        first, U_local = int(part_first[rank]), int(part_first[rank + 1] - part_first[rank])
    if world > 1:
        # NCCL may print its version banner on stdout; the contract is ONE JSON line there, so park fd 1 on
        # stderr while the communicator is created
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            ids = [pkg.get_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            g.comm_init(ids[0], world, rank)
            g.update_overlaps(1)          # first exchange: channel set-up
            g.sync()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    ndof = g.ndof(1)                     # DOFs this process drives (one GPU, or all of them with --single-process)
    ndof_job = ndof * (world if not single else 1)
    rng = np.random.Generator(np.random.MT19937(20221 + rank))
    pin_in = pkg.PinnedBuffer(ndof)
    pin_out = pkg.PinnedBuffer(ndof)
    pin_in.array[:] = rng.random(ndof)
    g.upload(pkg.TOLD, 1, rng.random(ndof))
    g.upload_ptr(pkg.TNONLIN, 1, pin_in.ptr)
    g.copy(1, pkg.TNEW, pkg.TNONLIN)

    def step():
        g.smoother(1, pkg.JACOBI, NSMOOTH)

    # ---- device-resident timing ----------------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        step()
    g.sync()
    skip = sampler.wait_first_sample() if sampler else 0     # clocks are sampled from here on (timed regions only)
    for _ in range(3):
        step()                                               # the GPU idled while nvidia-smi started: warm again
    g.sync(); barrier()
    g.profile(True)
    l0 = g.launch_count()
    g.sync(); barrier()
    g.event_record(0)
    for _ in range(args.steps):
        step()
    g.event_record(1)
    g.sync(); barrier()
    ms = allmax(g.elapsed_ms(0, 1))
    launches = g.launch_count() - l0
    kern_ms, kern_n = g.profile_read()
    g.profile(False)
    value = ndof_job * NSMOOTH * args.steps / (ms * 1e-3)
    if args.dump_outputs:
        # what a caller of the timed smoother receives: the swept level-1 field (this rank's parents)
        out = dump_sample(g.download(pkg.TNONLIN, 1), DUMP_VALUES // world)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "tnonlin.npy" if world == 1 else f"tnonlin_rank{rank}.npy"), out)

    # ---- end to end through the C ABI with HOST buffers ---------------------------------------------------
    # (a) the headline e2e: one reference-facing smoother call per step with pinned HOST fields - upload of the field,
    #     4 sweeps, download of the result, every step; calls are independent, so the library pipelines the upload of a
    #     step under the download of the previous one
    e2e_steps = max(3, min(args.steps, 20))

    def timed(fn, reps):
        fn(); fn()
        g.sync(); barrier()
        t0 = time.perf_counter()
        g.event_record(2)
        for _ in range(reps):
            fn()
        g.event_record(3)
        g.sync(); barrier()
        dev = allmax(g.elapsed_ms(2, 3))
        wall = allmax((time.perf_counter() - t0) * 1e3)
        return max(dev, wall) / reps      # blocking host copies: take the slower of device and host clocks

    e2e_ms = timed(lambda: g.smooth_host(pkg.JACOBI, NSMOOTH, pin_in.ptr, pin_out.ptr), e2e_steps)
    e2e_value = ndof_job * NSMOOTH / (e2e_ms * 1e-3)
    # (b) the dependent loop of a real driver: the result of a call is the input of the next one, blocking calls
    dep_ms = timed(lambda: g.smoother_host(pkg.JACOBI, NSMOOTH, pin_out.ptr, pin_out.ptr), max(3, e2e_steps // 2))
    clocks = sampler.stop(skip) if sampler else None

    # ---- other kernels of the path: coloured GS sweep (32 B/DOF) and residual + norms (24 B/DOF) -----------
    peak, peak_src = peaks()
    extra = {}
    if not args.no_extras:
        for name, fn, bpd in (("gauss_seidel_sweep", lambda: g.smoother(1, pkg.GAUSS_SEIDEL, 1), 32.0),
                              ("residual_with_norms", lambda: g.get_residual(1), 24.0)):
            for _ in range(3):
                fn()
            g.sync(); barrier()
            g.event_record(6)
            reps = 20
            for _ in range(reps):
                fn()
            g.event_record(7)
            g.sync(); barrier()
            t_ms = allmax(g.elapsed_ms(6, 7)) / reps
            per_gpu = ndof_job / ngpu
            extra[name] = {"ms": t_ms, "dof_updates_per_s": ndof_job / (t_ms * 1e-3),
                           "algorithmic_GBps_per_gpu": bpd * per_gpu / (t_ms * 1e-3) / 1e9, "bytes_per_dof": bpd,
                           "frac": bpd * per_gpu / (t_ms * 1e-3) / 1e9 / peak}
            if name == "gauss_seidel_sweep":
                # SURVEY 8(d): report against 32 B/DOF (two passes re-reading T) AND against the 24 B/DOF Jacobi figure,
                # which is what the one-pass kernel actually moves (T read once, rhs read once, T written once)
                extra[name]["GBps_at_24B_per_dof"] = 24.0 * per_gpu / (t_ms * 1e-3) / 1e9
                extra[name]["frac_at_24B_per_dof"] = 24.0 * per_gpu / (t_ms * 1e-3) / 1e9 / peak
                extra[name]["includes"] = "one k_gs_win2 launch (its producer warp writes the next halo strips)"

    # unstructured front-ends on one GPU: explicit DG step, block-CSR assembly, SpMV, BiCGStab
    if rank == 0 and not args.no_extras and not single:
        kpu = int(os.environ.get("PAMG_BENCH_UNSTR_KP", "11"))      # 4^11 = 4.2M triangles (1.2 GB of matrix blocks): beyond L2
        um = pkg.Mesh.synthetic(kpu, 1)
        g.set_unstructured(um)
        T0 = np.random.Generator(np.random.MT19937(7)).random((um.U, 3))
        g._ck(g.L.pamg_unstr_upload(g.h, T0))
        g._ck(g.L.pamg_explicit_step(g.h, 1e-6, 0.9, 0.3, 0.0, 1, 2, 10, 0, 0))     # warm-up
        g.sync()
        g.event_record(8)
        g._ck(g.L.pamg_explicit_step(g.h, 1e-6, 0.9, 0.3, 0.0, 1, 10, 10, 0, 0))    # one time step of 10 element-loop passes
                                                                                     # (one told copy, 10 kernel launches)
        g.event_record(9)
        g.sync()
        t_ms = g.elapsed_ms(8, 9) / 10.0
        extra["unstr_explicit_pass"] = {"elements": um.U, "ms": t_ms, "dof_updates_per_s": 3 * um.U / (t_ms * 1e-3),
                                        "algorithmic_GBps": 144.0 * um.U / (t_ms * 1e-3) / 1e9, "bytes_per_element": 144.0,
                                        "frac": 144.0 * um.U / (t_ms * 1e-3) / 1e9 / peak}
        area = 0.5 * np.abs((um.X[:, 0, 0] - um.X[:, 2, 0]) * (um.X[:, 1, 1] - um.X[:, 2, 1])
                            - (um.X[:, 0, 1] - um.X[:, 2, 1]) * (um.X[:, 1, 0] - um.X[:, 2, 0]))
        dt_i = 4.0 * float(np.sqrt(area.min()))
        g.implicit_assemble(dt_i, 0.9, 0.3, use_dir=True)                             # warm-up
        g.sync()
        g.event_record(8)
        for _ in range(10):
            g.implicit_assemble(dt_i, 0.9, 0.3, use_dir=True)
        g.event_record(9)
        g.sync()
        t_asm = g.elapsed_ms(8, 9) / 10.0
        g._ck(g.L.pamg_unstr_upload(g.h, T0))
        it = C.c_int(0); rr = C.c_double(0.0)
        g._ck(g.L.pamg_implicit_step(g.h, 1, 1, 1e-10, 400, C.byref(it), C.byref(rr)))   # warm-up
        g._ck(g.L.pamg_unstr_upload(g.h, T0))
        g.sync()
        g.event_record(8)
        g._ck(g.L.pamg_implicit_step(g.h, 1, 1, 1e-10, 400, C.byref(it), C.byref(rr)))
        g.event_record(9)
        g.sync()
        t_solve = g.elapsed_ms(8, 9)
        extra["unstr_implicit"] = {"elements": um.U, "assemble_ms": t_asm,
                                   "assemble_GBps": 456.0 * um.U / (t_asm * 1e-3) / 1e9, "assemble_bytes_per_element": 456.0,
                                   "assemble_frac": 456.0 * um.U / (t_asm * 1e-3) / 1e9 / peak,
                                   "solve_ms": t_solve, "bicgstab_iters": it.value, "relres": rr.value, "cfl": 4.0,
                                   "note": "reference: dense (3E)^2 FINDInv, impossible at this size"}
        if hasattr(g, "implicit_spmv_ms"):
            t_spmv = g.implicit_spmv_ms(20)
            extra["unstr_implicit"].update({"spmv_ms": t_spmv, "spmv_bytes_per_element": 352.0,
                                            "spmv_GBps": 352.0 * um.U / (t_spmv * 1e-3) / 1e9,
                                            "spmv_frac": 352.0 * um.U / (t_spmv * 1e-3) / 1e9 / peak})

    # ---- V-cycle time to 1e-8 (second half of the BASELINE metric) ----------------------------------------
    vc = None
    if not args.no_vcycle:
        gs = {}
        for name, solver in (("jacobi", pkg.JACOBI), ("gauss_seidel", pkg.GAUSS_SEIDEL)):
            for timed_run in (False, True):   # first solve untimed: CUDA-graph capture, channels
                g.fill(pkg.TNONLIN, 1, 0.0)
                g.copy(1, pkg.TNEW, pkg.TNONLIN)
                g.fill(pkg.TOLD, 1, 0.0)
                g.sync(); barrier()
                l1 = g.launch_count()
                g.event_record(4)
                cyc, hist = g.vcycle_solve(solver=solver, nu1=NSMOOTH, nu2=NSMOOTH, ncoarse=15, max_cycles=60, tol=1e-8)
                g.event_record(5)
                g.sync(); barrier()
                if timed_run:
                    gs[name] = {"cycles": cyc, "ms": allmax(g.elapsed_ms(4, 5)), "relres": float(hist[-1] / hist[0]),
                                "launches": g.launch_count() - l1}
        # the reference's call unit: one time step with HOST fields (upload tnew once, told = tnew, GS V-cycles to 1e-8,
        # download once: the body of `do itime`, transport_tri_semi.F90:299-381)
        pin_in.array[:] = 0.0
        g.L.pamg_timestep_host(g.h, pin_in.ptr, pin_out.ptr, 60, 1e-8, None, None)   # warm-up (solver taken from the handle)
        g.sync(); barrier()
        t0 = time.perf_counter()
        cyc_t, rel_t = C.c_int(0), C.c_double(0)
        g._ck(g.L.pamg_timestep_host(g.h, pin_in.ptr, pin_out.ptr, 60, 1e-8, C.byref(cyc_t), C.byref(rel_t)))
        barrier()
        ts_ms = allmax((time.perf_counter() - t0) * 1e3)
        gs["timestep_host"] = {"ms": ts_ms, "cycles": cyc_t.value, "relres": rel_t.value, "solver": "gauss_seidel",
                               "h2d_bytes": 8 * ndof_job, "d2h_bytes": 8 * ndof_job,
                               "what": "upload tnew, told = tnew, V-cycles to 1e-8, download tnew (one `do itime` body)"}
        vc = gs

    # ---- numerical check of the run (cut-face strips + one sweep against the oracle) ----------------------------
    os.sched_setaffinity(0, affinity0)          # the CPU arms (oracle threads are created from here on) may use every core again
    orc = oracle_api()
    pc = parity_check(pkg, orc, g, mesh, first, U_local, nsplit, gather, part_first, world)

    if rank == 0:
        kern_avg_ms = kern_ms / max(kern_n, 1)
        per_gpu_dof = ndof_job / ngpu
        achieved = BYTES_PER_DOF_JACOBI * per_gpu_dof / (kern_avg_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ngpu, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "vcycle_to_1e-8": vc,
            "parity_check": pc,
            "config": workload_config(ngpu, nsplit, args.scaling, single),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 8 * ndof_job, "d2h_bytes_per_step": 8 * ndof_job,
                    "steps": e2e_steps, "ms_per_step": e2e_ms, "host_binding": binding,
                    "what": "pamg_smooth_host: pinned host field up, 4 Jacobi sweeps, result down, every step (independent calls, pipelined)",
                    "dependent_loop": {"ms_per_step": dep_ms, "value": ndof_job * NSMOOTH / (dep_ms * 1e-3),
                                       "what": "pamg_smoother_host, blocking, output of a call = input of the next"}},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "kernel": KERNEL_NAMES.get(os.environ.get("PAMG_KERNEL", "win"), os.environ.get("PAMG_KERNEL")),
                         "kernel_avg_ms": kern_avg_ms,
                         "kernel_launches_timed": kern_n, "algorithmic_bytes_per_launch": BYTES_PER_DOF_JACOBI * per_gpu_dof,
                         "peak_source": peak_src,
                         "whole_step_frac": (BYTES_PER_DOF_JACOBI * per_gpu_dof * NSMOOTH * args.steps / (ms * 1e-3) / 1e9) / peak},
            "clocks": clocks,
            "other_kernels": extra,
        }
        try:   # DRAM bytes of the dominant kernel from the committed ncu --set full capture (per launch)
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                tr = json.load(f)
            if os.environ.get("PAMG_KERNEL", "win") == tr.get("kernel_mode") and args.workload == "c5" and args.scaling == "weak":
                line["roofline"]["traffic"] = tr.get("jacobi_face_dram_bytes_per_launch")
                line["roofline"]["traffic_source"] = tr.get("source")
        except Exception:
            pass
        if not args.no_cpu_baseline:
            cores = len(affinity0) or 1
            v1, nd1, t1 = cpu_smoother_rate(orc, nsplit, 4, 1, 2)       # all 256 parents, 1 thread (serial like the reference)
            vall, nd2, t2 = cpu_smoother_rate(orc, nsplit, 4, cores, 2)  # all 256 parents, all cores
            line["cpu_baseline"] = {
                "value": v1, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": f"256 parents x 4^{nsplit} children ({nd1} DOFs), 2 Jacobi sweeps incl. update_overlaps, {t1:.1f} s",
                "all_cores": {"value": vall, "cores": cores,
                              "sample": f"full 256 parents ({nd2} DOFs), 2 sweeps, {t2:.1f} s, OpenMP over parents"}}
        print(json.dumps(line), flush=True)
    pin_in.free(); pin_out.free()
    g.close()
    ok = pc["strips_bit_exact"] and pc["max_rel_l2"] <= 1e-12
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if not ok:
        sys.stderr.write("parity_check FAILED: %s\n" % json.dumps(pc))
        sys.exit(3)


if __name__ == "__main__":
    main()
