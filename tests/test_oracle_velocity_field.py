"""The nodal velocity field u_ele(2,3,E) of the unstructured front-ends on the CPU, in two restatements: the oracle's bodies
with the field (oracle_field/, oracle_field_api) and a vectorised numpy one (velocity_field_ref).  A constant field
reproduces the oracle's uniform entries; the two restatements agree with discontinuous random fields; an affine field
satisfies the exact identities of the scheme; HEAD's single target block per face differs from the per-Gauss-point split
exactly on the faces where the two Gauss points disagree about the upwind side."""
import numpy as np
import pytest

import oracle_api as orc
import oracle_field_api as of
import velocity_field_ref as vf
from helpers import write_msh

MESHES = ["gmsh_100", "irregular", "test_sn2", "untitled8"]


def load(name, tmp_path):
    m = orc.read_msh(write_msh(name, str(tmp_path / (name + ".msh"))))
    fneig, _ = orc.neig_data(m["neig"], m["dir"])
    X = np.ascontiguousarray(m["X"]); neig = np.ascontiguousarray(m["neig"])
    return X, neig, fneig, np.ascontiguousarray(m["dir"])


def all_ccw(X):
    det = (X[:, 1, 0] - X[:, 0, 0]) * (X[:, 2, 1] - X[:, 0, 1]) - (X[:, 2, 0] - X[:, 0, 0]) * (X[:, 1, 1] - X[:, 0, 1])
    return bool(np.all(det > 0))


def rel(a, b):
    return np.linalg.norm(np.ravel(a) - np.ravel(b)) / max(np.linalg.norm(np.ravel(b)), 1e-300)


def rules(X):
    return [1, 0] if all_ccw(X) else [1]


@pytest.mark.parametrize("name", MESHES)
def test_constant_field_equals_the_uniform_oracle(name, tmp_path):
    X, neig, fneig, dirv = load(name, tmp_path)
    E = X.shape[0]
    u = (0.6, -0.35)
    U = np.tile(np.array(u), (E, 3, 1))
    rng = np.random.Generator(np.random.MT19937(11))
    T0, Told = rng.random((E, 3)), rng.random((E, 3))
    dt = 2e-3
    for use_dir in rules(X):
        for exact in (0, 1):
            ref = T0.copy()
            orc.lib().orc_unstr_explicit(E, X, neig, fneig, dirv, u[0], u[1], dt, 2, 2, 10, exact, use_dir, 0.25, ref)
            got = vf.explicit_step(X, neig, fneig, U, T0, dt, 2, 2, 10, exact, use_dir, 0.25)
            assert rel(got, ref) <= 1e-13, (use_dir, exact)
        for k in (0.0, 0.4):
            A = np.zeros((3 * E, 3 * E)); M = np.zeros((3 * E, 3 * E))
            orc.lib().orc_unstr_implicit_assemble_diff(E, X, neig, fneig, u[0], u[1], k, dt, use_dir, A, M)
            Af, Mf = vf.implicit_matrix(X, neig, fneig, U, dt, k, use_dir)
            assert rel(Af, A) <= 1e-13 and rel(Mf, M) <= 1e-13, (use_dir, k)
        ref = T0.copy()
        assert orc.lib().orc_unstr_implicit(E, X, neig, fneig, u[0], u[1], dt, 2, 1, use_dir, ref) == 0
        assert rel(vf.implicit_solve(X, neig, fneig, U, T0, dt, 2, 1, use_dir), ref) <= 1e-13
        ref = T0.copy()
        assert orc.lib().orc_unstr_implicit_stab(E, X, neig, fneig, u[0], u[1], dt, 2, 2, use_dir, ref) == 0
        assert rel(vf.implicit_solve(X, neig, fneig, U, T0, dt, 2, 2, use_dir, with_stab=True), ref) <= 1e-13
    dc, st = np.zeros((E, 3)), np.zeros((E, 9))
    orc.lib().orc_unstr_stab(E, X, T0, Told, u[0], u[1], dt, dc, st)
    dcf, stf = vf.stab(X, U, T0, Told, dt)
    assert rel(dcf, dc) <= 1e-13 and rel(stf, st) <= 1e-13


def affine_case(X):
    """u = (0.3 + 0.5x - 0.2y, -0.4 + 0.1x + 0.7y) (div u = 1.2), T = 1 + 0.3x - 0.6y at the nodes, and div(uT) there."""
    x, y = X[:, :, 0], X[:, :, 1]
    ux, uy = 0.3 + 0.5 * x - 0.2 * y, -0.4 + 0.1 * x + 0.7 * y
    T = 1.0 + 0.3 * x - 0.6 * y
    div = 1.2 * T + 0.3 * ux - 0.6 * uy
    return np.stack([ux, uy], axis=2), T, div


@pytest.mark.parametrize("name", ["irregular", "test_sn2", "split1", "900_ele"])
def test_affine_field_gives_the_exact_divergence(name, tmp_path):
    """Every integrand is exact under the quadratures (quadratic in the volume, cubic on faces) and both traces agree, so
    on elements without a boundary face one exact explicit step is T - dt div(uT) at the nodes and the implicit operator
    applied to T is (M/dt) T + M div(uT) + k A grad(phi_i).grad(T)."""
    X, neig, fneig, _ = load(name, tmp_path)
    E = X.shape[0]
    U, T, div = affine_case(X)
    inner = np.all(neig != 0, axis=1)
    assert inner.sum() > 0
    dt, k = 1e-2, 0.3
    got = vf.explicit_step(X, neig, fneig, U, T, dt, 1, 1, 0, 1, 1)
    assert np.abs(got - (T - dt * div))[inner].max() <= 1e-12 * np.abs(T).max()
    A, Mdt = vf.implicit_matrix(X, neig, fneig, U, dt, k, 1)
    G = vf.Geometry(X, neig, fneig, 1)
    Mloc = (np.ones((3, 3)) + np.eye(3)) / 12.0
    want = np.einsum("ij,ej->ei", Mloc, T / dt + div) * G.area[:, None]
    gT = np.array([0.3, -0.6])
    want += k * G.area[:, None] * (G.grad @ gT)
    AT = (A @ T.reshape(-1)).reshape(E, 3)
    assert np.abs(AT - want)[inner].max() <= 1e-11 * np.abs(want).max()


def random_field(E, seed):
    return np.random.Generator(np.random.MT19937(seed)).uniform(-1.0, 1.0, (E, 3, 2))


@pytest.mark.parametrize("name", MESHES)
def test_field_oracle_with_a_constant_field_is_the_uniform_oracle(name, tmp_path):
    """The oracle's field entries (oracle_field/) filled with (u_x, u_y) against its uniform entries."""
    X, neig, fneig, dirv = load(name, tmp_path)
    E = X.shape[0]
    u = (0.6, -0.35)
    U = np.tile(np.array(u), (E, 3, 1))
    rng = np.random.Generator(np.random.MT19937(17))
    T0, Told = rng.random((E, 3)), rng.random((E, 3))
    dt = 2e-3
    for use_dir in rules(X):
        for exact in (0, 1):
            ref = T0.copy()
            orc.lib().orc_unstr_explicit(E, X, neig, fneig, dirv, u[0], u[1], dt, 2, 2, 10, exact, use_dir, 0.25, ref)
            assert rel(of.explicit(X, neig, fneig, U, T0, dt, 2, 2, 10, exact, use_dir, 0.25), ref) <= 1e-13
        A = np.zeros((3 * E, 3 * E)); M = np.zeros((3 * E, 3 * E))
        orc.lib().orc_unstr_implicit_assemble_diff(E, X, neig, fneig, u[0], u[1], 0.4, dt, use_dir, A, M)
        for literal in (False, True):
            Af, Mf = of.assemble(X, neig, fneig, U, dt, 0.4, use_dir, literal)
            assert rel(Af, A) <= 1e-13 and rel(Mf, M) <= 1e-13, literal
        for with_stab in (False, True):
            ref = T0.copy()
            f = orc.lib().orc_unstr_implicit_stab if with_stab else orc.lib().orc_unstr_implicit
            assert f(E, X, neig, fneig, u[0], u[1], dt, 2, 2, use_dir, ref) == 0
            assert rel(of.implicit(X, neig, fneig, U, T0, dt, 2, 2, use_dir, with_stab), ref) <= 1e-13
    dc, st = np.zeros((E, 3)), np.zeros((E, 9))
    orc.lib().orc_unstr_stab(E, X, T0, Told, u[0], u[1], dt, dc, st)
    dcf, stf = of.stab(X, U, T0, Told, dt)
    assert rel(dcf, dc) <= 1e-13 and rel(stf, st) <= 1e-13


def sign_changes(X, neig, fneig, U):
    """elements with a face (towards a neighbour) whose two Gauss points disagree about the upwind side"""
    G = vf.Geometry(X, neig, fneig, 1)
    mixed = np.zeros(X.shape[0], bool)
    for f in range(3):
        inc = [G.income(f, *G.traces(U, f, s)) for s in range(2)]
        mixed |= (inc[0] != inc[1]) & (neig[:, f] != 0)
    return mixed


@pytest.mark.parametrize("name", ["gmsh_100", "irregular", "test_sn2", "split1"])
def test_numpy_restatement_equals_the_field_oracle_with_discontinuous_fields(name, tmp_path):
    """Random per-node fields: n.u changes sign inside many faces and the two traces of a face differ, so every branch of
    the per-Gauss-point upwinding is taken.  Two independent restatements (vectorised numpy, and the oracle's own bodies
    with the field) agree on every matrix entry, the explicit steps, the stabilisation and the implicit solves."""
    X, neig, fneig, _ = load(name, tmp_path)
    E = X.shape[0]
    U = random_field(E, 21)
    assert sign_changes(X, neig, fneig, U).sum() > 0
    rng = np.random.Generator(np.random.MT19937(22))
    T0, Told = rng.random((E, 3)), rng.random((E, 3))
    dt = 2e-3
    for use_dir in rules(X):
        for exact in (0, 1):
            want = of.explicit(X, neig, fneig, U, T0, dt, 2, 2, 10, exact, use_dir, 0.25)
            assert rel(vf.explicit_step(X, neig, fneig, U, T0, dt, 2, 2, 10, exact, use_dir, 0.25), want) <= 1e-12
        for k in (0.0, 0.4):
            for literal in (False, True):
                A, M = of.assemble(X, neig, fneig, U, dt, k, use_dir, literal)
                An, Mn = vf.implicit_matrix(X, neig, fneig, U, dt, k, use_dir, literal=literal)
                assert np.abs(An - A).max() <= 1e-12 * np.abs(A).max() and rel(Mn, M) <= 1e-12, (k, literal)
                assert np.array_equal(An != 0.0, A != 0.0)
        for with_stab in (False, True):
            want = of.implicit(X, neig, fneig, 0.3 * U, T0, dt, 2, 2, use_dir, with_stab)
            assert rel(vf.implicit_solve(X, neig, fneig, 0.3 * U, T0, dt, 2, 2, use_dir, with_stab), want) <= 1e-12
    dc, st = of.stab(X, U, T0, Told, dt)
    dcn, stn = vf.stab(X, U, T0, Told, dt)
    assert rel(dcn, dc) <= 1e-12 and rel(stn, st) <= 1e-12


@pytest.mark.parametrize("name", MESHES)
def test_oracle_literal_single_target_differs_only_where_the_gauss_points_disagree(name, tmp_path):
    """orc_unstr_implicit_assemble_diff_field(literal_target = 1) is HEAD's rule (one block per face from income(1)); it
    differs from the per-Gauss-point split in the rows of exactly the elements with a face whose Gauss points disagree."""
    X, neig, fneig, _ = load(name, tmp_path)
    E = X.shape[0]
    U = random_field(E, 5)
    As, _ = of.assemble(X, neig, fneig, U, 1e-2, 0.0, True, False)
    Al, _ = of.assemble(X, neig, fneig, U, 1e-2, 0.0, True, True)
    mixed = sign_changes(X, neig, fneig, U)
    assert mixed.sum() > 0
    differs = np.abs(As - Al).reshape(E, 3, -1).max(axis=(1, 2)) > 0.0
    assert np.array_equal(differs, mixed)
