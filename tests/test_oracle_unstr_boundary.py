"""Boundary data on the unstructured front-ends (pamg_unstr_set_boundary): the numpy reference of unstr_boundary_ref pinned
before any device runs.

  * a linear field transported along its level lines is steady: with its own values as data it solves the implicit system
    exactly at any CFL number, which it does not without data on the elements with an inflow face;
  * the explicit step with the exact local inverse moves a linear field by dt u.grad T on every element, boundary ones
    included, once the data is the field itself;
  * the erfc boundary layer (the reference's acceptance case, tests/test_erfc_boundary_layer.py): the whole time loop of the
    semi-structured multigrid path (oracle, V-cycles to 1e-10) equals the unstructured implicit solve on the same children
    taken as an element list, with the same boundary kinds, and meets the reference's L1 gate."""
import os

import numpy as np
import pytest

import oracle_api as orc
import unstr_boundary_ref as ubr
from helpers import child_coordinates, inlet_open_boundary, probe_p1, rel_l2, strip_mesh, write_msh, write_msh_triangles
from pamg_pkg import pamg
from velocity_field_ref import Geometry

UNIFORM = (0.8, -0.35)


def shipped(tmp_path, name="900_ele"):
    m = orc.read_msh(write_msh(name, str(tmp_path / (name + ".msh"))))
    fneig, _ = orc.neig_data(m["neig"], m["dir"])
    return m["X"], m["neig"], fneig


def synthetic():
    m = pamg.Mesh.synthetic(2, 2)
    return m.X, m.neig, m.fneig


def meshes(tmp_path):
    return [shipped(tmp_path), synthetic()]


def steady_field(x, y):
    # u . grad T = 0 for u = UNIFORM: T varies across the flow only
    return 1.5 + 0.7 * (UNIFORM[1] * x - UNIFORM[0] * y)


@pytest.mark.parametrize("cfl", [1.0, 64.0])
def test_steady_linear_field_solves_the_implicit_system_with_its_own_data(tmp_path, cfl):
    for X, neig, fneig in meshes(tmp_path):
        E = X.shape[0]
        u = ubr.uniform(E, UNIFORM)
        G = Geometry(X, neig, fneig, True)
        h = float(np.sqrt(2.0 * G.area.mean()))
        dt = cfl * h / float(np.hypot(*UNIFORM))
        T = steady_field(X[..., 0], X[..., 1]).reshape(-1)
        kind = np.ones((E, 3), np.int32)
        A, M, b = ubr.implicit_system(X, neig, fneig, u, dt, 0.0, True, kind, ubr.face_values(X, steady_field))
        r = A @ T - (M @ T + b)
        assert np.max(np.abs(r)) <= 1e-12 * np.max(np.abs(M @ T)), np.max(np.abs(r))
        sol = np.linalg.solve(A, M @ T + b) if E < 1500 else None
        if sol is not None:
            assert np.max(np.abs(sol - T)) <= 1e-12 * np.max(np.abs(T))
        # without data (HEAD) the rows of elements with an inflow boundary face are not satisfied, the others are
        A0, M0, b0 = ubr.implicit_system(X, neig, fneig, u, dt, 0.0, True)
        assert not b0.any()
        r0 = np.abs(A0 @ T - M0 @ T).reshape(E, 3).max(axis=1)
        bd = (neig == 0).any(axis=1)
        assert np.max(r0[~bd]) <= 1e-12 * np.max(np.abs(M @ T))
        assert np.max(r0[bd]) > 1e-3 * np.max(np.abs(M @ T))


def test_explicit_exact_step_moves_a_linear_field_on_every_element(tmp_path):
    def lin(x, y):
        return 0.3 + 1.1 * x - 0.6 * y
    for X, neig, fneig in meshes(tmp_path):
        E = X.shape[0]
        u = ubr.uniform(E, UNIFORM)
        T = lin(X[..., 0], X[..., 1])
        dt = 1e-2
        drift = dt * (UNIFORM[0] * 1.1 - UNIFORM[1] * 0.6)
        kind = np.ones((E, 3), np.int32)
        out = ubr.explicit_step(X, neig, fneig, u, T, dt, 1, 1, 0, True, True, kind, ubr.face_values(X, lin))
        assert np.max(np.abs(out - (T - drift))) <= 1e-12
        # HEAD: exact only on the elements without a boundary face
        head = ubr.explicit_step(X, neig, fneig, u, T, dt, 1, 1, 0, True, True)
        bd = (neig == 0).any(axis=1)
        assert np.max(np.abs(head - (T - drift))[~bd]) <= 1e-12
        assert np.max(np.abs(head - (T - drift))[bd]) > 1e-3


def test_open_face_with_inflow_is_refused_by_the_reference(tmp_path):
    X, neig, fneig = synthetic()
    E = X.shape[0]
    kind = np.full((E, 3), 2, np.int32)
    with pytest.raises(ValueError):
        ubr.implicit_system(X, neig, fneig, ubr.uniform(E, UNIFORM), 1e-2, 0.0, True, kind)


# ---- the erfc boundary layer: semi-structured == unstructured, whole time loop ---------------------------------------------
N_SPLIT, DT, NSTEPS, K = 4, 2e-3, 50, 2.0
PROBE_X = np.linspace(0.0, 1.0, 202)
PROBE = np.stack([PROBE_X, np.full_like(PROBE_X, 0.0333)], axis=1)


def erfc_children(tmp_path):
    """The strip of test_erfc_boundary_layer: parents (oracle geometry) and its children as an element list with the kinds of
    inlet_open_boundary found on the children directly."""
    X = strip_mesh(15)
    m = orc.read_msh(write_msh_triangles(X, os.path.join(str(tmp_path), "strip.msh")))
    fneig, _ = orc.neig_data(m["neig"], m["dir"])
    kind, val = inlet_open_boundary(m["X"], m["neig"])
    # get_splitting places a vertex shared by several children in the last bits differently per child (and the walls at
    # y = +-1e-18): snapped, the children form a conforming mesh with exact walls (n.u = 0)
    Xc = np.round(child_coordinates(orc, m["X"], N_SPLIT).reshape(-1, 3, 2), 12) + 0.0
    mc = pamg.Mesh.from_arrays(Xc)
    assert int((mc.neig == 0).sum()) == 2 * 15 * 2 ** N_SPLIT + 2 * 2 ** N_SPLIT
    assert np.array_equal(mc.X, Xc)
    ck, cv = inlet_open_boundary(Xc, mc.neig)
    return (m["X"], m["neig"], fneig, m["dir"], kind, val), (Xc, mc.neig, mc.fneig, ck, np.repeat(cv[:, :, None], 2, axis=2))


def semi_oracle_run(parents, tol=1e-10):
    X, neig, fneig, dirv, kind, val = parents
    orc.lib().orc_semi_set_threads(os.cpu_count() or 1)
    p = orc.intended_params(N_SPLIT, N_SPLIT, dt=DT, k=K, u=(1.0, 0.0), source_coef=0.0)
    s = orc.Semi(p, X, neig, fneig, dirv)
    s.set_boundary(kind, val)
    for _ in range(NSTEPS):
        s.field(orc.TOLD)[:] = s.field(orc.TNONLIN)
        cyc, hist = s.vcycle_solve(solver=4, max_cycles=200, tol=tol)
        assert hist[-1] <= tol * hist[0]
    return s.field(orc.TNONLIN).copy()


def test_erfc_semi_structured_equals_unstructured_whole_time_loop(tmp_path):
    from test_erfc_boundary_layer import analytical_solution
    parents, (Xc, neig, fneig, kind, val) = erfc_children(tmp_path)
    semi = semi_oracle_run(parents).reshape(-1, 3)
    E = Xc.shape[0]
    un = ubr.implicit_solve(Xc, neig, fneig, ubr.uniform(E, (1.0, 0.0)), np.zeros((E, 3)), DT, NSTEPS, K, True, kind, val)
    assert rel_l2(un, semi) <= 1e-8, rel_l2(un, semi)
    L1 = float(np.mean(np.abs(probe_p1(Xc, un, PROBE) - analytical_solution(PROBE_X))))
    assert L1 <= 0.01, L1
