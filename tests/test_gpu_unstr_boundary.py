"""Boundary data on the unstructured front-ends on the device (pamg_unstr_set_boundary): operator, right-hand side, implicit
solve and explicit step against the numpy reference of unstr_boundary_ref with mixed kinds (sin(x+y) / values / open), uniform
and nodal velocities, with and without diffusion and with both preconditioners; a steady linear field kept to 1e-12 at CFL 1
and 64; the reference's erfc boundary layer on the implicit solve, against its gate and the device's semi-structured run;
HEAD kept bit for bit without data; the state rules and refusals."""
import ctypes as C

import numpy as np
import pytest
from scipy.sparse.linalg import spsolve

import unstr_boundary_ref as ubr
import velocity_field_ref as vf
from helpers import probe_p1, rel_l2, rng_field, write_msh
from pamg_pkg import pamg
from test_oracle_unstr_boundary import DT, K, N_SPLIT, NSTEPS, PROBE, PROBE_X, erfc_children

pytestmark = pytest.mark.gpu
UNIFORM = (0.8, -0.35)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def meshes(tmp_path_factory):
    d = tmp_path_factory.mktemp("msh")
    out = {name: pamg.Mesh.read_msh(write_msh(name, str(d / (name + ".msh")))) for name in ["irregular", "900_ele"]}
    out["synthetic"] = pamg.Mesh.synthetic(3, 1)
    return out


def handle(mesh):
    g = pamg.SemiImplicitIterative(pamg.default_params(), pamg.Mesh.synthetic(0, 1))
    g.set_unstructured(mesh)
    return g


def smooth_field(X):
    x, y = X[..., 0], X[..., 1]
    return np.stack([1.0 + 0.3 * np.sin(3.0 * y), 0.5 * np.cos(2.0 * x)], axis=-1)


def strict_outflow(mesh, u):
    """[E,3]: faces with outflow of non-zero flux at both Gauss points (where an open face is allowed)."""
    G = vf.Geometry(mesh.X, mesh.neig, mesh.fneig, True)
    out = np.ones((mesh.U, 3), bool)
    for f in range(3):
        for s in range(2):
            us, _ = G.traces(u, f, s)
            out[:, f] &= np.einsum("ed,ed->e", G.normal[:, f], us) > 0.0
    return out


def mixed_kinds(mesh, u, seed):
    rng = np.random.Generator(np.random.MT19937(seed))
    kind = rng.integers(0, 2, (mesh.U, 3)).astype(np.int32)
    kind[strict_outflow(mesh, u) & (rng.random((mesh.U, 3)) < 0.6)] = 2
    value = rng.uniform(-1.0, 1.0, (mesh.U, 3, 2))
    bd = mesh.neig == 0
    assert ((kind == 2) & bd).any() and ((kind == 0) & bd).any() and ((kind == 1) & bd).any()
    return kind, value


def velocity(mesh, which):
    return ubr.uniform(mesh.U, UNIFORM) if which == "uniform" else smooth_field(mesh.X)


def set_velocity(g, mesh, which):
    g.set_velocity(None if which == "uniform" else smooth_field(mesh.X))


@pytest.mark.parametrize("which", ["uniform", "field"])
@pytest.mark.parametrize("k", [0.0, 0.7])
@pytest.mark.parametrize("precond", ["block_jacobi", "flow_gs"])
def test_device_against_the_numpy_reference(meshes, which, k, precond):
    mesh = meshes["900_ele"]
    E = mesh.U
    u = velocity(mesh, which)
    kind, value = mixed_kinds(mesh, u, 31)
    g = handle(mesh)
    set_velocity(g, mesh, which)
    g.set_unstructured_boundary(kind, value)
    dt = 2e-2
    A, M, b = ubr.implicit_system(mesh.X, mesh.neig, mesh.fneig, u, dt, k, True, kind, value, sparse=True)
    T0 = rng_field((E, 3), 41)
    # two implicit steps against spsolve of the reference system
    T1, it1, rr1 = g.unstr_implicit(T0, dt, UNIFORM[0], UNIFORM[1], ntime=1, use_dir=True, precond=precond, k=k)
    ref1 = spsolve(A.tocsc(), M @ T0.ravel() + b)
    assert rr1 <= 1e-13 and rel_l2(T1.ravel(), ref1) <= 1e-10
    if precond == "flow_gs" and which == "uniform" and k == 0.0:
        assert it1 == 1                                            # pure advection: the sweep is the inverse, data or not
    # the operator: the reference's with the open faces' penalty taken out
    val, col = g.implicit_bsr()
    D = vf.bsr_to_dense(val, col, sparse=True)
    Ad = A.toarray()
    assert np.max(np.abs(D.toarray() - Ad)) <= 1e-13 * np.max(np.abs(Ad))
    # the device's solution satisfies the reference's right-hand side, data included
    assert rel_l2(g.implicit_apply(T1).ravel(), M @ T0.ravel() + b) <= 1e-10
    T2, _, rr2 = g.unstr_implicit(T0, dt, UNIFORM[0], UNIFORM[1], ntime=2, use_dir=True, precond=precond, k=k)
    ref2 = spsolve(A.tocsc(), M @ ref1 + b)
    assert rr2 <= 1e-13 and rel_l2(T2.ravel(), ref2) <= 1e-10
    # explicit steps (no diffusion there): exact local inverse and Jacobi
    if k == 0.0 and precond == "block_jacobi":
        for exact in (True, False):
            got = g.unstr_explicit(T0, 1e-3, UNIFORM[0], UNIFORM[1], ntime=2, nits=2, njac_its=5, exact_minv=exact,
                                   use_dir=True)
            ref = ubr.explicit_step(mesh.X, mesh.neig, mesh.fneig, u, T0, 1e-3, 2, 2, 5, exact, True, kind, value)
            assert rel_l2(got, ref) <= 1e-12


@pytest.mark.parametrize("cfl", [1.0, 64.0])
@pytest.mark.parametrize("precond", ["block_jacobi", "flow_gs"])
def test_steady_linear_field_stays(meshes, cfl, precond):
    def steady(x, y):
        return 1.5 + 0.7 * (UNIFORM[1] * x - UNIFORM[0] * y)
    for name in ["900_ele", "synthetic"]:
        mesh = meshes[name]
        g = handle(mesh)
        g.set_unstructured_boundary(np.ones((mesh.U, 3), np.int32), ubr.face_values(mesh.X, steady))
        G = vf.Geometry(mesh.X, mesh.neig, mesh.fneig, True)
        dt = cfl * float(np.sqrt(2.0 * G.area.mean())) / float(np.hypot(*UNIFORM))
        T0 = steady(mesh.X[..., 0], mesh.X[..., 1])
        T, it, rr = g.unstr_implicit(T0, dt, UNIFORM[0], UNIFORM[1], ntime=3, use_dir=True, precond=precond)
        assert np.max(np.abs(T - T0)) <= 1e-12 * np.max(np.abs(T0)), (name, np.max(np.abs(T - T0)))
        if precond == "flow_gs":
            assert it <= 3                                          # at most one iteration per step
        # started away from it, one flow sweep per step still solves: the data adds no upwind edge
        if precond == "flow_gs":
            _, it2, rr2 = g.unstr_implicit(T0 + 0.1, dt, UNIFORM[0], UNIFORM[1], ntime=2, use_dir=True, precond=precond)
            assert it2 == 2 and rr2 <= 1e-13


def erfc_device_semi(parents, tol=1e-10):
    X, neig, fneig, dirv, kind, val = parents
    mesh = pamg.Mesh.from_arrays(X)
    assert np.array_equal(mesh.neig, neig) and np.array_equal(mesh.fneig, fneig)
    p = pamg.default_params(n_split=N_SPLIT, multi_levels=N_SPLIT, dt=DT, k=K, u_x=1.0, u_y=0.0, source_coef=0.0)
    g = pamg.SemiImplicitIterative(p, mesh, bc_kind=kind, bc_value=val)
    for _ in range(NSTEPS):
        g.copy(1, pamg.TOLD, pamg.TNONLIN)
        cyc, hist = g.vcycle_solve(solver=pamg.GAUSS_SEIDEL, max_cycles=200, tol=tol)
        assert hist[-1] <= max(tol * hist[0], 1e-14)
    T = g.download(pamg.TNONLIN, 1).reshape(-1, 3)
    g.close()
    return T


def test_erfc_boundary_layer_on_the_implicit_solve(tmp_path):
    from test_erfc_boundary_layer import analytical_solution
    parents, (Xc, neig, fneig, kind, val) = erfc_children(tmp_path)
    mesh = pamg.Mesh.from_arrays(Xc)
    E = mesh.U
    assert E == 7680
    g = handle(mesh)
    g.set_unstructured_boundary(kind, val)
    T, it, rr = g.unstr_implicit(np.zeros((E, 3)), DT, 1.0, 0.0, ntime=NSTEPS, use_dir=True, k=K, tol=1e-13,
                                 max_iters=2000)
    assert rr <= 1e-13
    L1 = float(np.mean(np.abs(probe_p1(Xc, T, PROBE) - analytical_solution(PROBE_X))))
    assert L1 <= 0.01, L1
    semi = erfc_device_semi(parents)
    assert rel_l2(T, semi) <= 1e-8, rel_l2(T, semi)
    # a large step with the flow sweep: converges and equals the direct solve (the gate is not asserted at this dt)
    dt, n = 0.02, 5
    Tl, itl, rrl = g.unstr_implicit(np.zeros((E, 3)), dt, 1.0, 0.0, ntime=n, use_dir=True, k=K, tol=1e-13, max_iters=2000,
                                    precond="flow_gs")
    assert rrl <= 1e-13
    ref = ubr.implicit_solve(Xc, neig, fneig, ubr.uniform(E, (1.0, 0.0)), np.zeros((E, 3)), dt, n, K, True, kind, val)
    assert rel_l2(Tl, ref) <= 1e-8, rel_l2(Tl, ref)


@pytest.mark.parametrize("which", ["uniform", "field"])
def test_without_data_is_head_bit_for_bit(meshes, which):
    mesh = meshes["900_ele"]
    E = mesh.U
    T0 = rng_field((E, 3), 51)
    kind, value = mixed_kinds(mesh, velocity(mesh, which), 52)

    def run(setup):
        g = handle(mesh)
        set_velocity(g, mesh, which)
        setup(g)
        out = [g.unstr_explicit(T0, 1e-3, UNIFORM[0], UNIFORM[1], ntime=2, nits=2, njac_its=5, exact_minv=ex, use_dir=True)
               for ex in (True, False)]
        for precond in ("block_jacobi", "flow_gs"):
            out.append(g.unstr_implicit(T0, 2e-2, UNIFORM[0], UNIFORM[1], ntime=2, use_dir=True, k=0.7, precond=precond)[0])
        g.close()
        return out

    def cleared(g):
        g.set_unstructured_boundary(kind, value)
        g.set_unstructured_boundary(None)

    kind1 = np.ones((E, 3), np.int32)                              # kind 1 with zero values
    labels = ["explicit exact", "explicit Jacobi", "implicit block_jacobi", "implicit flow_gs"]
    for lab, a, b, c in zip(labels, run(lambda g: None), run(cleared),
                            run(lambda g: g.set_unstructured_boundary(kind1, np.zeros((E, 3, 2))))):
        assert np.array_equal(a, b), (lab, np.max(np.abs(a - b)))
        assert np.array_equal(a, c), (lab, np.max(np.abs(a - c)))


def test_state_and_refusals(meshes):
    mesh = meshes["irregular"]
    E = mesh.U
    ones = np.ones((E, 3), np.int32)
    # before pamg_set_unstructured
    g0 = pamg.SemiImplicitIterative(pamg.default_params(), pamg.Mesh.synthetic(0, 1))
    assert g0.L.pamg_unstr_set_boundary(g0.h, E, _ptr(ones), None) == pamg.ERR_STATE
    g0.close()
    g = handle(mesh)
    assert g.L.pamg_unstr_set_boundary(g.h, E + 1, _ptr(ones), None) == pamg.ERR_ARG
    bad = ones.copy(); bad[mesh.neig == 0] = 3
    assert g.L.pamg_unstr_set_boundary(g.h, E, _ptr(bad), None) == pamg.ERR_ARG
    inner = ones.copy(); inner[mesh.neig != 0] = 7                    # interior entries are ignored
    assert g.L.pamg_unstr_set_boundary(g.h, E, _ptr(inner), None) == pamg.OK
    # the operator is stale after the call, until the next assembly
    g.implicit_assemble(1e-2, *UNIFORM, use_dir=True)
    g.set_unstructured_boundary(ones, None)
    x = rng_field((E, 3), 61)
    it, rr = np.zeros(1, np.int32), np.zeros(1)
    calls = [lambda: g.L.pamg_implicit_step(g.h, 1, 1, 1e-12, 100, it.ctypes.data_as(C.POINTER(C.c_int)),
                                            rr.ctypes.data_as(C.POINTER(C.c_double))),
             lambda: g.L.pamg_implicit_apply(g.h, x, np.empty_like(x)),
             lambda: g.L.pamg_implicit_get_bsr(g.h, _ptr(np.zeros((E, 4, 9))), None),
             lambda: g.L.pamg_implicit_set_stab(g.h, 1),
             lambda: g.L.pamg_implicit_precond_apply(g.h, x, np.empty_like(x)),
             lambda: g.L.pamg_implicit_flow_levels(g.h, None, None, None)]
    for call in calls:
        assert call() == pamg.ERR_STATE
    g.implicit_assemble(1e-2, *UNIFORM, use_dir=True)
    for call in calls:
        assert call() == pamg.OK
    g.set_unstructured_boundary(None)
    assert calls[1]() == pamg.ERR_STATE
    # an open face with inflow: refused by the assembly (which leaves the operator unassembled) and by the explicit step
    u = ubr.uniform(E, UNIFORM)
    G = vf.Geometry(mesh.X, mesh.neig, mesh.fneig, True)
    c = np.stack([G.sdet[:, f] * (G.normal[:, f] @ np.asarray(UNIFORM)) for f in range(3)], axis=1)
    inflow = (mesh.neig == 0) & (c < 0.0)
    e, f = (int(v[0]) for v in np.nonzero(inflow))
    kind = ones.copy(); kind[e, f] = 2
    g.set_unstructured_boundary(kind, None)
    with pytest.raises(pamg.PamgError) as ei:
        g.implicit_assemble(1e-2, *UNIFORM, use_dir=True)
    assert ei.value.code == pamg.ERR_UNSUPPORTED and f"element {e} " in str(ei.value) and f"face {f + 1} " in str(ei.value)
    assert calls[1]() == pamg.ERR_STATE
    with pytest.raises(pamg.PamgError) as ei:
        g.unstr_explicit(x, 1e-3, *UNIFORM, ntime=1, nits=1, use_dir=True)
    assert ei.value.code == pamg.ERR_UNSUPPORTED
    # the same face open while it is outflow is fine
    g.unstr_explicit(x, 1e-3, -UNIFORM[0], -UNIFORM[1], ntime=1, nits=1, use_dir=True)
    g.implicit_assemble(1e-2, -UNIFORM[0], -UNIFORM[1], use_dir=True)
    # pamg_set_unstructured clears the data: HEAD again
    kind1 = ones.copy()
    g.set_unstructured_boundary(kind1, np.full((E, 3, 2), 0.5))
    g.set_unstructured(mesh)
    h = handle(mesh)
    assert np.array_equal(g.unstr_explicit(x, 1e-3, *UNIFORM, ntime=1, nits=1, use_dir=True),
                          h.unstr_explicit(x, 1e-3, *UNIFORM, ntime=1, nits=1, use_dir=True))
    h.close(); g.close()


def test_multi_device_handle_reaches_part0(meshes):
    mesh = meshes["irregular"]
    E = mesh.U
    g = pamg.SemiImplicitIterative(pamg.default_params(n_split=3, multi_levels=3), pamg.Mesh.synthetic(2, 2), devices=[0, 0])
    g.set_unstructured(mesh)
    u = ubr.uniform(E, UNIFORM)
    kind, value = np.ones((E, 3), np.int32), np.random.Generator(np.random.MT19937(71)).uniform(-1, 1, (E, 3, 2))
    g.set_unstructured_boundary(kind, value)
    T0 = rng_field((E, 3), 72)
    got = g.unstr_explicit(T0, 1e-3, *UNIFORM, ntime=1, nits=2, exact_minv=True, use_dir=True)
    ref = ubr.explicit_step(mesh.X, mesh.neig, mesh.fneig, u, T0, 1e-3, 1, 2, 10, True, True, kind, value)
    assert rel_l2(got, ref) <= 1e-12
    g.close()
