"""The unstructured kernels at streaming sizes: meshes of 1 to 1.2M elements on which every grid-stride loop takes several trips,
grid_sum2 adds more per-CTA partials than a CTA has threads, the plane stride is padded, the last warp is partial and the last
CTA has idle warps.  On each: the block-CSR operator against velocity_field_ref's sparse assembly; the product and both
preconditioners against A_ref x, the inverse diagonal blocks and the block-triangular solve; BiCGStab iterate by iterate
against a numpy restatement of the device recurrence, and its converged answer against the reference operator; the explicit
step and the stabilisation against velocity_field_ref; boundary data over compact lists longer than one trip; and the
batched local inverse over three trips."""
import ctypes as C

import numpy as np
import pytest

import oracle_api as orc
import unstr_boundary_ref as ubr
import velocity_field_ref as vf
from helpers import inlet_open_boundary, random_parent_mesh, rel_l2, rng_field, strip_mesh
from pamg_pkg import pamg
from test_gpu_flow_precond import sweep_reference
from test_host_flow_levels import uniform_mask

pytestmark = pytest.mark.gpu
TPB = 256
CTAS_PER_SM = 8                  # stream_grid and the set-up kernels launch at most nsm * 8 CTAs
UNIFORM = (0.9, 0.3)
SCALE = ["tiny1", "tiny33", "mid", "large"]
OP_TOL, KERNEL_TOL = 1e-13, 1e-12


def sm_count():
    cu = C.CDLL("libcuda.so.1")
    dev, n = C.c_int(0), C.c_int(0)
    assert cu.cuInit(0) == 0 and cu.cuDeviceGet(C.byref(dev), 0) == 0
    assert cu.cuDeviceGetAttribute(C.byref(n), 16, dev) == 0          # CU_DEVICE_ATTRIBUTE_MULTIPROCESSOR_COUNT
    return n.value


@pytest.fixture(scope="module")
def nsm():
    return sm_count()


def padded(E):
    return -(-E // 32) % 2 == 0                                        # plane_stride pads ld past E + 31


@pytest.fixture(scope="module")
def meshes(nsm):
    out = {"tiny1": pamg.Mesh.from_arrays(np.array([[[0.0, 0.0], [1.0, 0.0], [0.2, 0.9]]])),
           "tiny33": pamg.Mesh.from_arrays(strip_mesh(17)[:33]),
           "mid": pamg.Mesh.from_arrays(random_parent_mesh(5, m=185, jitter=0.2)),
           "large": pamg.Mesh.from_arrays(random_parent_mesh(6, m=775, jitter=0.2)),
           "pow2": pamg.Mesh.synthetic(10, 1),
           "strip": pamg.Mesh.from_arrays(strip_mesh(400_001))}
    E = {k: m.U for k, m in out.items()}
    assert E["tiny1"] == 1 and np.all(out["tiny1"].neig == 0)
    assert E["tiny33"] == 33 and padded(33) and np.all((out["tiny33"].neig == 0).any(axis=1))
    for name in ("mid", "large"):
        assert E[name] % 32 == 2 and padded(E[name]), name
    assert -(-E["mid"] // TPB) > TPB                                   # more CTAs than a CTA has threads
    assert E["large"] > 2 * nsm * CTAS_PER_SM * TPB                    # three trips at any occupancy
    assert E["pow2"] == 2 ** 20 and E["pow2"] % 32 == 0
    assert E["strip"] == 800_002 and np.all((out["strip"].neig == 0).any(axis=1))
    assert E["strip"] > nsm * CTAS_PER_SM * TPB
    return out


def handle(mesh):
    g = pamg.SemiImplicitIterative(pamg.default_params(), pamg.Mesh.synthetic(0, 1))
    g.set_unstructured(mesh)
    return g


def random_field(E, seed):
    return np.random.Generator(np.random.MT19937(seed)).uniform(-1.0, 1.0, (E, 3, 2))


def rotating_field(X):
    c = X.reshape(-1, 2).mean(axis=0)
    return np.stack([-(X[:, :, 1] - c[1]), X[:, :, 0] - c[0]], axis=2)


def velocity(mesh, which):
    """(nodal field for the reference, field for set_velocity or None for the uniform path)"""
    if which == "uniform":
        return np.tile(np.array(UNIFORM), (mesh.U, 3, 1)), None
    U = random_field(mesh.U, 11) if which == "field" else rotating_field(mesh.X)
    return U, U


def areas(X):
    return 0.5 * np.abs((X[:, 0, 0] - X[:, 2, 0]) * (X[:, 1, 1] - X[:, 2, 1]) - (X[:, 0, 1] - X[:, 2, 1]) * (X[:, 1, 0] - X[:, 2, 0]))


def locate(err, E, nsm):
    """where the worst element sits relative to the last warp, the last CTA and the first trip of a grid-stride loop"""
    e = int(np.argmax(err))
    tags = [t for t, on in (("last warp", e >= (E - 1) // 32 * 32), ("last CTA", e >= (E - 1) // TPB * TPB),
                            ("past the first trip at any occupancy", e >= nsm * CTAS_PER_SM * TPB)) if on]
    return f"worst element {e} of {E} ({', '.join(tags) or f'below nsm * 8 * TPB = {nsm * CTAS_PER_SM * TPB}'})"


def check(name, kernel, got, ref, tol, nsm):
    E = got.shape[0]
    err = rel_l2(got, ref)
    print(f"MEASURED {kernel} {name} rel-L2 {err:.3e}")
    per = np.abs(np.asarray(got).reshape(E, -1) - np.asarray(ref).reshape(E, -1)).max(axis=1)
    assert err <= tol, f"{kernel} on {name}: rel-L2 {err:.3e} > {tol:g}; {locate(per, E, nsm)}"


# -- 1. the block-CSR operator ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", SCALE + ["pow2"])
@pytest.mark.parametrize("which,k", [("uniform", 0.0), ("uniform", 0.3), ("field", 0.3)])
def test_block_csr_operator(meshes, nsm, name, which, k):
    mesh = meshes[name]
    E = mesh.U
    U, dev = velocity(mesh, which)
    g = handle(mesh)
    g.set_velocity(dev)
    dt = 0.05
    g.implicit_assemble(dt, *UNIFORM, use_dir=True, k=k)
    val, col = g.implicit_bsr()
    A = vf.implicit_matrix(mesh.X, mesh.neig, mesh.fneig, U, dt, k, True, sparse=True)[0].tocoo()
    D = vf.bsr_to_dense(val, col, sparse=True)
    diff = (D - A).tocoo()
    scale = np.abs(A.data).max()
    worst = np.zeros(E)
    np.maximum.at(worst, diff.row // 3, np.abs(diff.data))
    print(f"MEASURED k_assemble_bsr {name} {which} k={k} max-abs/max {worst.max() / scale:.3e}")
    assert worst.max() <= OP_TOL * scale, f"k_assemble_bsr on {name}: {worst.max() / scale:.3e}; {locate(worst, E, nsm)}"
    # a block is stored exactly where the reference couples two elements (and on the diagonal)
    nz = A.data != 0.0
    coupled = np.unique(np.concatenate([(A.row[nz] // 3).astype(np.int64) * E + A.col[nz] // 3, np.arange(E) * (E + 1)]))
    ok = col >= 0
    present = np.unique(np.concatenate([np.nonzero(ok)[0].astype(np.int64) * E + col[ok], np.arange(E) * (E + 1)]))
    assert np.array_equal(coupled, present), f"block pattern on {name}"
    assert np.all(col[:, 0] == np.arange(E))


# -- 2. product and preconditioners -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", SCALE + ["pow2"])
@pytest.mark.parametrize("which", ["uniform", "rotating"])
def test_product_and_preconditioners(meshes, nsm, name, which):
    mesh = meshes[name]
    E = mesh.U
    U, dev = velocity(mesh, which)
    g = handle(mesh)
    g.set_velocity(dev)
    dt = 0.05
    g.implicit_assemble(dt, *UNIFORM, use_dir=True, k=0.0)
    A = vf.implicit_matrix(mesh.X, mesh.neig, mesh.fneig, U, dt, 0.0, True, sparse=True)[0]
    x = rng_field((E, 3), 21) - 0.5
    check(name, "k_bsr_spmv", g.implicit_apply(x), (A @ x.ravel()).reshape(E, 3), KERNEL_TOL, nsm)
    val, col = g.implicit_bsr()
    check(name, "k_block_apply", g.implicit_precond_apply(x), np.einsum("eij,ej->ei", np.linalg.inv(val[:, 0]), x),
          KERNEL_TOL, nsm)
    g.implicit_set_precond("flow_gs")
    level, nlevels, lagged = g.implicit_flow_levels()
    if which == "uniform":
        want, _, nl, lag = pamg.flow_levels(mesh.neig, uniform_mask(mesh, UNIFORM))
        assert np.array_equal(level, want) and (nlevels, lagged) == (nl, lag) and lagged == 0, name
    elif E > 1000:
        assert lagged > 0, name
    ys = [g.implicit_precond_apply(x) for _ in range(3)]
    check(name, "k_flow_sweep", ys[0], sweep_reference(val, col, level, x), KERNEL_TOL, nsm)
    assert np.array_equal(ys[0], ys[1]) and np.array_equal(ys[1], ys[2]), f"k_flow_sweep on {name}: applications differ"


# -- 3. BiCGStab iterate by iterate -------------------------------------------------------------------------------------------
def dinv_blocks(val):
    """the inverse diagonal blocks as k_assemble_bsr forms them (adjugate over the determinant)"""
    d = val[:, 0].reshape(-1, 9)
    c00, c01, c02 = d[:, 4] * d[:, 8] - d[:, 5] * d[:, 7], d[:, 5] * d[:, 6] - d[:, 3] * d[:, 8], d[:, 3] * d[:, 7] - d[:, 4] * d[:, 6]
    i = 1.0 / (d[:, 0] * c00 + d[:, 1] * c01 + d[:, 2] * c02)
    o = np.stack([c00 * i, (d[:, 2] * d[:, 7] - d[:, 1] * d[:, 8]) * i, (d[:, 1] * d[:, 5] - d[:, 2] * d[:, 4]) * i,
                  c01 * i, (d[:, 0] * d[:, 8] - d[:, 2] * d[:, 6]) * i, (d[:, 2] * d[:, 3] - d[:, 0] * d[:, 5]) * i,
                  c02 * i, (d[:, 1] * d[:, 6] - d[:, 0] * d[:, 7]) * i, (d[:, 0] * d[:, 4] - d[:, 1] * d[:, 3]) * i], axis=1)
    return o.reshape(-1, 3, 3)


def bicgstab(A, prec, b, x0, tol, max_iters, keep):
    """The device recurrence (k_kry_init, k_kry_p / k_kry_vec, k_kry_spmv, k_kry_s, k_kry_x) restated: right-preconditioned
    BiCGStab from x0 with rh = r0, rho = alpha = omega = 1, rho_new = (r0, r0), no exit on ||s||, stopped when rr <= tol^2 bb,
    after max_iters iterations or on a breakdown.  Returns ({k: (x_k, sqrt(rr_k / bb))} for k in keep, iterations, x, relres)."""
    x = x0.copy()
    r = b - A @ x
    rh, p, v = r.copy(), np.zeros_like(r), np.zeros_like(r)
    bb, rr = b @ b, r @ r
    rho = alpha = omega = 1.0
    rho_new = rr
    out, it = {}, 0
    while rr > tol * tol * bb and it < max_iters:
        beta = (rho_new / rho) * (alpha / omega)
        p = r + beta * p + (-beta * omega) * v
        y = prec(p)
        v = A @ y
        t0 = rh @ v
        if t0 == 0.0:
            break
        alpha = rho_new / t0
        s = r - alpha * v
        z = prec(s)
        t = A @ z
        tt = t @ t
        omega = (t @ s) / tt if tt > 0.0 else 0.0
        x = x + alpha * y + omega * z
        r = s + (-omega) * t
        rr, rho, rho_new = r @ r, rho_new, rh @ r
        it += 1
        if it in keep:
            out[it] = (x.copy(), np.sqrt(rr / bb))
        if rho_new == 0.0 or omega == 0.0:
            break
    return out, it, x, np.sqrt(rr / bb)


def step(g, T0, tol, max_iters):
    g._ck(g.L.pamg_unstr_upload(g.h, np.ascontiguousarray(T0)))
    it, rr = C.c_int(0), C.c_double(0.0)
    g._ck(g.L.pamg_implicit_step(g.h, 1, 1, tol, max_iters, C.byref(it), C.byref(rr)))
    out = np.empty_like(T0)
    g._ck(g.L.pamg_unstr_download(g.h, out))
    return out, it.value, rr.value


KRYLOV_KS = (1, 2, 15, 16, 17, 33)
KRYLOV_TOL = 1e-11
XK_TOL, RELRES_TOL = 1e-13, 1e-10     # largest measured on a B200: 2.1e-15 and 8.0e-12


@pytest.mark.parametrize("name", SCALE)
@pytest.mark.parametrize("precond", ["block_jacobi", "flow_gs"])
def test_bicgstab_iterate_by_iterate(meshes, nsm, name, precond):
    mesh = meshes[name]
    E = mesh.U
    h = float(np.sqrt(areas(mesh.X).min()))
    dt, kdiff = 4.0 * h / np.hypot(*UNIFORM), 0.1 * h * np.hypot(*UNIFORM)     # CFL 4, cell Peclet number 10
    g = handle(mesh)
    g.implicit_set_precond(precond)
    g.implicit_assemble(dt, *UNIFORM, use_dir=True, k=kdiff)
    val, col = g.implicit_bsr()
    Ad = vf.bsr_to_dense(val, col, sparse=True)                              # the device's operator: only the recurrence differs
    Aref, Mref = vf.implicit_matrix(mesh.X, mesh.neig, mesh.fneig, np.tile(np.array(UNIFORM), (E, 3, 1)), dt, kdiff, True,
                                    sparse=True)
    if precond == "block_jacobi":
        Dinv = dinv_blocks(val)
        prec = lambda w: np.einsum("eij,ej->ei", Dinv, w.reshape(E, 3)).ravel()
    else:
        level = g.implicit_flow_levels()[0]
        prec = lambda w: sweep_reference(val, col, level, w.reshape(E, 3)).ravel()
    T0 = rng_field((E, 3), 31)
    b = Mref @ T0.ravel()
    ref, ref_it, ref_x, ref_rel = bicgstab(Ad, prec, b, T0.ravel(), KRYLOV_TOL, 10_000, set(KRYLOV_KS))
    for k in KRYLOV_KS:
        x, it, rel = step(g, T0, KRYLOV_TOL, k)
        kk = min(k, ref_it)
        want_x, want_rel = ref[kk] if kk in ref else (ref_x, ref_rel)
        assert it == kk, f"BiCGStab ({precond}) on {name}: {it} iterations with max_iters {k}, numpy {kk}"
        check(name, f"BiCGStab-{precond}-x{k}", x, want_x.reshape(E, 3), XK_TOL, nsm)
        print(f"MEASURED BiCGStab-{precond}-relres{k} {name} {abs(rel - want_rel) / max(want_rel, 1e-15):.3e}")
        # (1e-15: a system solved exactly in one iteration leaves a relres of 0 or a few ulp)
        assert abs(rel - want_rel) <= RELRES_TOL * want_rel + 1e-15, (name, precond, k, rel, want_rel)
    if name in ("mid", "large"):
        assert ref_it > 17 or precond == "flow_gs", (name, ref_it)        # block Jacobi needs tens of iterations here
    # to the tolerance: the iteration count, the true residual with the reference operator, and determinism
    runs = [step(g, T0, KRYLOV_TOL, 10_000) for _ in range(2)]
    x, it, rel = runs[0]
    print(f"MEASURED BiCGStab-{precond}-iterations {name} device {it} numpy {ref_it}")
    assert abs(it - ref_it) <= 1 and rel <= KRYLOV_TOL, (name, precond, it, ref_it, rel)
    true = np.linalg.norm(b - Aref @ x.ravel()) / np.linalg.norm(b)
    print(f"MEASURED BiCGStab-{precond}-true-residual {name} {true:.3e}")
    assert true <= 10 * KRYLOV_TOL, (name, precond, true)
    assert np.array_equal(runs[1][0], x) and runs[1][1:] == (it, rel), f"BiCGStab ({precond}) on {name} is not deterministic"


# -- 4. the explicit step -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,which,exact", [(n, w, x) for n in SCALE for w in ("uniform", "field") for x in (False, True)]
                         + [("pow2", "field", True)])
def test_explicit_step(meshes, nsm, name, which, exact):
    mesh = meshes[name]
    U, dev = velocity(mesh, which)
    g = handle(mesh)
    g.set_velocity(dev)
    T0 = rng_field((mesh.U, 3), 41)
    got = g.unstr_explicit(T0, 1e-4, *UNIFORM, ntime=2, nits=2, njac_its=3, t_bc=0.25, exact_minv=exact, use_dir=True)
    ref = vf.explicit_step(mesh.X, mesh.neig, mesh.fneig, U, T0, 1e-4, 2, 2, 3, exact, True, 0.25)
    check(name, f"k_unstr_explicit-{which}-exact{int(exact)}", got, ref, KERNEL_TOL, nsm)


# -- 5. the stabilisation -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["mid", "large"])
@pytest.mark.parametrize("which", ["uniform", "field"])
def test_stabilisation(meshes, nsm, name, which):
    mesh = meshes[name]
    U, dev = velocity(mesh, which)
    g = handle(mesh)
    g.set_velocity(dev)
    T0, Told = rng_field((mesh.U, 3), 51), rng_field((mesh.U, 3), 52)
    dc, st = g.unstr_stab(T0, Told, 1e-3, *UNIFORM)
    dcr, str_ = vf.stab(mesh.X, U, T0, Told, 1e-3)
    check(name, f"k_unstr_stab-diff_coe-{which}", dc, dcr, KERNEL_TOL, nsm)
    check(name, f"k_unstr_stab-stab-{which}", st, str_, KERNEL_TOL, nsm)


# -- 6. boundary data on the strip --------------------------------------------------------------------------------------------
def strip_kinds(mesh):
    """inlet_open_boundary (T = 1 on x = 0, open elsewhere), with kind 0 and kind 1 (random values) on a third each of the
    faces without inflow (walls and outlet)"""
    kind, val = inlet_open_boundary(mesh.X, mesh.neig)
    value = np.repeat(val[:, :, None], 2, axis=2)
    rng = np.random.Generator(np.random.MT19937(61))
    free = kind == 2
    pick = rng.integers(0, 3, kind.shape)
    kind[free & (pick == 0)] = 0
    kind[free & (pick == 1)] = 1
    value[free & (pick == 1)] = rng.uniform(-1.0, 1.0, (int((free & (pick == 1)).sum()), 2))
    bd = mesh.neig == 0
    assert all(((kind == c) & bd).any() for c in (0, 1, 2))
    return kind, value


def test_boundary_data_on_the_strip(meshes, nsm):
    mesh = meshes["strip"]
    E = mesh.U
    u = (1.0, 0.0)
    U = ubr.uniform(E, u)
    kind, value = strip_kinds(mesh)
    g = handle(mesh)
    g.set_unstructured_boundary(kind, value)
    T0 = rng_field((E, 3), 62)
    H = 1.0 / 400_001
    for exact in (False, True):
        got = g.unstr_explicit(T0, 0.1 * H, *u, ntime=2, nits=2, njac_its=3, exact_minv=exact, use_dir=True)
        ref = ubr.explicit_step(mesh.X, mesh.neig, mesh.fneig, U, T0, 0.1 * H, 2, 2, 3, exact, True, kind, value)
        check("strip", f"k_unstr_explicit_bc-exact{int(exact)}", got, ref, KERNEL_TOL, nsm)
    dt, kdiff = 0.5 * H, 0.2 * H                                            # CFL 1/2, k dt / H^2 = 1/10
    x, it, rel = g.unstr_implicit(T0, dt, *u, ntime=1, use_dir=True, k=kdiff, tol=KRYLOV_TOL, max_iters=2000)
    assert rel <= KRYLOV_TOL, (it, rel)
    A, M, bc = ubr.implicit_system(mesh.X, mesh.neig, mesh.fneig, U, dt, kdiff, True, kind, value, sparse=True)
    b = M @ T0.ravel() + bc
    true = np.linalg.norm(b - A @ x.ravel()) / np.linalg.norm(b)
    print(f"MEASURED strip-implicit-true-residual {true:.3e} iterations {it}")
    assert true <= 10 * KRYLOV_TOL, (true, it)
    assert np.linalg.norm(bc) > 1e-3 * np.linalg.norm(M @ T0.ravel())      # the data reach the right-hand side


# -- 7. the batched local inverse over three trips ----------------------------------------------------------------------------
@pytest.mark.parametrize("n", [3, 4, 6])
def test_findinv_multi_trip(nsm, n):
    trip = nsm * CTAS_PER_SM * 128                                          # k_local_minv: 128 threads, one block each
    B = 2 * trip + 5
    rng = np.random.default_rng(70 + n)
    M = rng.random((B, n, n)) + n * np.eye(n)
    rhs = rng.random((B, n))
    singular = np.zeros((n, n))
    pivot = rng.random((n, n)) + n * np.eye(n); pivot[0, 0] = 0.0
    mass = 0.37 / 12 * (np.ones((3, 3)) + np.eye(3)) if n == 3 else pivot
    special = {0: singular, trip - 1: pivot, trip: mass, trip + 1: singular, 2 * trip - 1: mass, 2 * trip: pivot,
               B - 5: pivot, B - 4: singular, B - 3: mass, B - 2: singular, B - 1: pivot}
    for i, blk in special.items():
        M[i] = blk
    g = pamg.SemiImplicitIterative(pamg.default_params(), pamg.Mesh.synthetic(0, 1))
    Minv, x, status = g.findinv(M, rhs)
    regular = np.ones(B, bool); regular[list(special)] = False
    inv = np.linalg.inv(M[regular])
    err = np.abs(Minv[regular] - inv).max(axis=(1, 2)) / np.abs(inv).max(axis=(1, 2))
    print(f"MEASURED k_local_minv<{n}> max-abs/max {err.max():.3e}")
    where = np.nonzero(regular)[0][int(np.argmax(err))]
    assert err.max() <= KERNEL_TOL, f"k_local_minv<{n}>: {err.max():.3e} at block {where} of {B} (trip {trip})"
    assert np.all(status[regular] == 0)
    xr = np.einsum("bij,bj->bi", inv, rhs[regular])
    assert np.abs(x[regular] - xr).max() <= KERNEL_TOL * np.abs(xr).max()
    for i, blk in special.items():
        ref = np.zeros(n * n)
        flag = orc.lib().orc_findinv(np.ascontiguousarray(blk.ravel()), ref, n)
        assert status[i] == flag, (n, i)
        assert np.allclose(Minv[i].ravel(), ref, rtol=1e-12, atol=1e-13), (n, i)
        if flag == 0:
            assert np.allclose(x[i], ref.reshape(n, n) @ rhs[i], rtol=1e-12, atol=1e-13), (n, i)
        else:
            assert np.all(Minv[i] == 0)
