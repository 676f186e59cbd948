"""The nodal velocity field u_ele(2,3,E) on the device (pamg_unstr_set_velocity): the explicit step, the block-CSR operator,
the implicit time loop and the stabilisation against the oracle's field entries (oracle_field_api) with random per-node
fields whose normal component changes sign inside faces - where a dense (3E)^2 oracle is too large, against the numpy
restatement (velocity_field_ref, itself checked against the oracle on the CPU) in block-sparse form; a constant field against the uniform path; the affine identities; the
state rules; and the explicit step at 4^11 triangles."""
import numpy as np
import pytest

import oracle_field_api as of
import velocity_field_ref as vf
from helpers import rel_l2, rng_field, write_msh
from pamg_pkg import pamg

pytestmark = pytest.mark.gpu
TOL = 1e-12
NAMES = ["untitled8192", "irregular", "split1", "900_ele"]
DENSE = ["irregular", "split1", "900_ele"]          # small enough for a dense (3E)^2 operator
SOLVE = ["irregular", "split1"]                     # small enough for the oracle's dense FINDInv solve


@pytest.fixture(scope="module")
def meshes(tmp_path_factory):
    d = tmp_path_factory.mktemp("msh")
    return {name: pamg.Mesh.read_msh(write_msh(name, str(d / (name + ".msh")))) for name in NAMES}


def handle(mesh):
    g = pamg.SemiImplicitIterative(pamg.default_params(), pamg.Mesh.synthetic(0, 1))
    g.set_unstructured(mesh)
    return g


def random_field(E, seed):
    return np.random.Generator(np.random.MT19937(seed)).uniform(-1.0, 1.0, (E, 3, 2))


def rotating_field(X):
    c = X.reshape(-1, 2).mean(axis=0)
    return np.stack([-(X[:, :, 1] - c[1]), X[:, :, 0] - c[0]], axis=2)


@pytest.mark.parametrize("name", NAMES)
def test_explicit_step_with_a_random_field(meshes, name):
    mesh = meshes[name]
    g = handle(mesh)
    U = random_field(mesh.U, 1)
    g.set_velocity(U)
    T0 = rng_field((mesh.U, 3), 3)
    for exact in (0, 1):
        got = g.unstr_explicit(T0, 1e-3, 7.0, -9.0, ntime=3, nits=2, njac_its=10, t_bc=0.25, exact_minv=bool(exact),
                               use_dir=True)
        ref = of.explicit(mesh.X, mesh.neig, mesh.fneig, U, T0, 1e-3, 3, 2, 10, exact, 1, 0.25)
        assert rel_l2(got, ref) <= TOL, exact


@pytest.mark.parametrize("name", NAMES)
def test_stabilisation_with_a_random_field(meshes, name):
    mesh = meshes[name]
    g = handle(mesh)
    U = random_field(mesh.U, 2)
    g.set_velocity(U)
    T0, Told = rng_field((mesh.U, 3), 4), rng_field((mesh.U, 3), 5)
    dc, st = g.unstr_stab(T0, Told, 1e-3, 7.0, -9.0)
    dcr, str_ = of.stab(mesh.X, U, T0, Told, 1e-3)
    assert rel_l2(dc, dcr) <= TOL and rel_l2(st, str_) <= TOL


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("k", [0.0, 0.4])
def test_block_csr_operator_with_a_random_field(meshes, name, k):
    mesh = meshes[name]
    g = handle(mesh)
    U = random_field(mesh.U, 6)
    g.set_velocity(U)
    dt = 0.05
    g.implicit_assemble(dt, 7.0, -9.0, use_dir=True, k=k)
    val, col = g.implicit_bsr()
    E = mesh.U
    if name in DENSE:
        A, _ = of.assemble(mesh.X, mesh.neig, mesh.fneig, U, dt, k, True)
        assert rel_l2(vf.bsr_to_dense(val, col), A) <= TOL
        coupled = np.abs(A).reshape(E, 3, E, 3).max(axis=(1, 3)) > 0.0
    else:                                                        # block by block, without the dense form
        A = vf.implicit_matrix(mesh.X, mesh.neig, mesh.fneig, U, dt, k, True, sparse=True)[0].tocsr()
        D = vf.bsr_to_dense(val, col, sparse=True).tocsr()
        assert np.sqrt(((D - A).multiply(D - A)).sum()) <= TOL * np.sqrt(A.multiply(A).sum())
        Ab = abs(A).tocoo()
        coupled = np.zeros((E, E), bool)
        coupled[Ab.row[Ab.data > 0] // 3, Ab.col[Ab.data > 0] // 3] = True
    # a block is present exactly where the operator couples two elements
    present = np.zeros((E, E), bool)
    for b in range(4):
        ok = col[:, b] >= 0
        present[np.arange(E)[ok], col[ok, b]] = True
    assert np.array_equal(coupled, present | np.eye(E, dtype=bool))


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("with_stab", [False, True])
def test_implicit_time_loop_with_a_random_field(meshes, name, with_stab):
    mesh = meshes[name]
    g = handle(mesh)
    U = 0.3 * random_field(mesh.U, 7)
    g.set_velocity(U)
    T0 = rng_field((mesh.U, 3), 8)
    # a step of at most a tenth of an element per step: with larger steps the discontinuous random field makes the implicit
    # operator of untitled8192's small elements nearly singular (solutions of 1e6 and more, in any solver)
    X = mesh.X
    area = 0.5 * np.abs((X[:, 0, 0] - X[:, 2, 0]) * (X[:, 1, 1] - X[:, 2, 1]) - (X[:, 0, 1] - X[:, 2, 1]) * (X[:, 1, 0] - X[:, 2, 0]))
    dt = min(0.02, 0.1 * np.sqrt(area.min()) / 0.3)
    got, _, relres = g.unstr_implicit(T0, dt, 7.0, -9.0, ntime=2, nits=2, use_dir=True, tol=1e-13, max_iters=2000,
                                      with_stab=with_stab)
    if name in SOLVE:
        ref = of.implicit(mesh.X, mesh.neig, mesh.fneig, U, T0, dt, 2, 2, True, with_stab)
    else:
        ref = vf.implicit_solve(mesh.X, mesh.neig, mesh.fneig, U, T0, dt, 2, 2, True, with_stab=with_stab)
    assert rel_l2(got, ref) <= TOL, relres


@pytest.mark.parametrize("name", NAMES)
def test_constant_field_equals_the_uniform_path(meshes, name):
    mesh = meshes[name]
    u = (0.6, -0.35)
    g, h = handle(mesh), handle(mesh)
    h.set_velocity(np.tile(np.array(u), (mesh.U, 3, 1)))
    T0, Told = rng_field((mesh.U, 3), 9), rng_field((mesh.U, 3), 10)
    for exact in (0, 1):
        a = g.unstr_explicit(T0, 1e-3, u[0], u[1], ntime=2, nits=2, t_bc=0.25, exact_minv=bool(exact), use_dir=True)
        b = h.unstr_explicit(T0, 1e-3, 0.0, 0.0, ntime=2, nits=2, t_bc=0.25, exact_minv=bool(exact), use_dir=True)
        assert rel_l2(b, a) <= 1e-13
    for x, y in zip(g.unstr_stab(T0, Told, 1e-3, u[0], u[1]), h.unstr_stab(T0, Told, 1e-3, 0.0, 0.0)):
        assert rel_l2(y, x) <= 1e-13
    if name in DENSE:
        for k in (0.0, 0.4):
            g.implicit_assemble(0.05, u[0], u[1], use_dir=True, k=k); h.implicit_assemble(0.05, 0.0, 0.0, use_dir=True, k=k)
            (va, ca), (vb, cb) = g.implicit_bsr(), h.implicit_bsr()
            assert rel_l2(vf.bsr_to_dense(vb, cb), vf.bsr_to_dense(va, ca)) <= 1e-13
        a = g.unstr_implicit(T0, 0.02, u[0], u[1], ntime=2, nits=2, use_dir=True, tol=1e-13, with_stab=True)[0]
        b = h.unstr_implicit(T0, 0.02, 0.0, 0.0, ntime=2, nits=2, use_dir=True, tol=1e-13, with_stab=True)[0]
        assert rel_l2(b, a) <= 1e-13


@pytest.mark.parametrize("name", DENSE)
def test_affine_identities_on_the_device(meshes, name):
    mesh = meshes[name]
    X = mesh.X
    x, y = X[:, :, 0], X[:, :, 1]
    ux, uy = 0.3 + 0.5 * x - 0.2 * y, -0.4 + 0.1 * x + 0.7 * y
    T = 1.0 + 0.3 * x - 0.6 * y
    div = 1.2 * T + 0.3 * ux - 0.6 * uy
    inner = np.all(mesh.neig != 0, axis=1)
    g = handle(mesh)
    g.set_velocity(np.stack([ux, uy], axis=2))
    dt, k = 1e-2, 0.3
    got = g.unstr_explicit(T, dt, 0.0, 0.0, ntime=1, nits=1, exact_minv=True, use_dir=True)
    assert np.abs(got - (T - dt * div))[inner].max() <= 1e-12 * np.abs(T).max()
    g.implicit_assemble(dt, 0.0, 0.0, use_dir=True, k=k)
    G = vf.Geometry(X, mesh.neig, mesh.fneig, 1)
    want = np.einsum("ij,ej->ei", (np.ones((3, 3)) + np.eye(3)) / 12.0, T / dt + div) * G.area[:, None]
    want += k * G.area[:, None] * (G.grad @ np.array([0.3, -0.6]))
    AT = g.implicit_apply(T)
    assert np.abs(AT - want)[inner].max() <= 1e-11 * np.abs(want).max()


def test_state_rules(meshes):
    mesh = meshes["irregular"]
    E = mesh.U
    U = random_field(E, 12)
    T0 = rng_field((E, 3), 13)
    g = pamg.SemiImplicitIterative(pamg.default_params(), pamg.Mesh.synthetic(0, 1))
    assert g.L.pamg_unstr_set_velocity(g.h, U.ctypes.data) == pamg.ERR_STATE          # no mesh yet
    g.set_unstructured(mesh)
    fresh = handle(mesh)
    # a cleared field is the uniform path bit for bit
    g.set_velocity(U)
    g.set_velocity(None)
    assert np.array_equal(g.unstr_explicit(T0, 1e-3, 0.6, -0.35), fresh.unstr_explicit(T0, 1e-3, 0.6, -0.35))
    # a field change makes the assembled operator stale until the next assembly
    g.implicit_assemble(0.05, 0.6, -0.35, use_dir=True)
    g.set_velocity(U)
    h = g.h
    assert g.L.pamg_implicit_step(h, 1, 1, 1e-12, 10, None, None) == pamg.ERR_STATE
    assert g.L.pamg_implicit_apply(h, T0, np.empty_like(T0)) == pamg.ERR_STATE
    assert g.L.pamg_implicit_get_bsr(h, np.empty((E, 36)).ctypes.data, None) == pamg.ERR_STATE
    assert g.L.pamg_implicit_set_stab(h, 1) == pamg.ERR_STATE
    g.implicit_assemble(0.05, 0.6, -0.35, use_dir=True)
    A, _ = of.assemble(mesh.X, mesh.neig, mesh.fneig, U, 0.05, 0.0, True)
    assert rel_l2(vf.bsr_to_dense(*g.implicit_bsr()), A) <= TOL
    # set_stab(0) re-assembles with the stored field
    g._ck(g.L.pamg_implicit_set_stab(h, 1)); g._ck(g.L.pamg_implicit_set_stab(h, 0))
    assert rel_l2(vf.bsr_to_dense(*g.implicit_bsr()), A) <= TOL
    # a new mesh clears the field
    g.set_unstructured(mesh)
    assert np.array_equal(g.unstr_explicit(T0, 1e-3, 0.6, -0.35), fresh.unstr_explicit(T0, 1e-3, 0.6, -0.35))


def test_multi_device_handle_reaches_part0(meshes):
    mesh = meshes["irregular"]
    src = pamg.Mesh.synthetic(2, 2)
    g = pamg.SemiImplicitIterative(pamg.default_params(n_split=3, multi_levels=3), src, devices=[0, 0])
    g.set_unstructured(mesh)
    U = random_field(mesh.U, 14)
    g.set_velocity(U)
    T0 = rng_field((mesh.U, 3), 15)
    got = g.unstr_explicit(T0, 1e-3, 0.0, 0.0, ntime=1, nits=2, use_dir=True)
    ref = of.explicit(mesh.X, mesh.neig, mesh.fneig, U, T0, 1e-3, 1, 2, 10, 0, 1)
    assert rel_l2(got, ref) <= TOL


def test_full_size_rotating_field():
    mesh = pamg.Mesh.synthetic(11, 1)                   # 4^11 triangles
    g = handle(mesh)
    U = rotating_field(mesh.X)
    g.set_velocity(U)
    T0 = rng_field((mesh.U, 3), 16)
    got = g.unstr_explicit(T0, 1e-5, 0.0, 0.0, ntime=1, nits=2, njac_its=3, t_bc=0.25, use_dir=True)
    ref = of.explicit(mesh.X, mesh.neig, mesh.fneig, U, T0, 1e-5, 1, 2, 3, 0, 1, 0.25)
    assert rel_l2(got, ref) <= TOL
