"""The flow-ordered block Gauss-Seidel preconditioner of the implicit solve (pamg_implicit_set_precond, k_flow_sweep) on the
device: one application against a numpy block-triangular solve built from the device's own blocks and levels; the device's
upwind graph against the numpy restatement of the inflow rule; pure advection with a uniform velocity solved in one BiCGStab
iteration at any CFL number, equal to the oracle; diffusion and a random nodal field with the stabilisation equal to the
block-Jacobi path and the references; the state rules; and the 4^11 mesh with a rotating field."""
import numpy as np
import pytest

import oracle_api as orc
import oracle_field_api as of
import velocity_field_ref as vf
from helpers import rel_l2, rng_field, write_msh
from pamg_pkg import pamg
from test_host_flow_levels import uniform_mask

pytestmark = pytest.mark.gpu
NAMES = ["split1", "test_sn2", "irregular", "900_ele"]


@pytest.fixture(scope="module")
def meshes(tmp_path_factory):
    d = tmp_path_factory.mktemp("msh")
    out = {name: pamg.Mesh.read_msh(write_msh(name, str(d / (name + ".msh")))) for name in NAMES + ["untitled8192"]}
    out["synthetic8"] = pamg.Mesh.synthetic(8, 1)
    return out


def handle(mesh):
    g = pamg.SemiImplicitIterative(pamg.default_params(), pamg.Mesh.synthetic(0, 1))
    g.set_unstructured(mesh)
    return g


def areas(X):
    return 0.5 * np.abs((X[:, 0, 0] - X[:, 2, 0]) * (X[:, 1, 1] - X[:, 2, 1]) - (X[:, 0, 1] - X[:, 2, 1]) * (X[:, 1, 0] - X[:, 2, 0]))


def random_field(E, seed):
    return np.random.Generator(np.random.MT19937(seed)).uniform(-1.0, 1.0, (E, 3, 2))


def rotating_field(X):
    c = X.reshape(-1, 2).mean(axis=0)
    return np.stack([-(X[:, :, 1] - c[1]), X[:, :, 0] - c[0]], axis=2)


def sweep_reference(val, col, level, x):
    """y = M^-1 x, M = D + the blocks (e, c) with level[c] < level[e], level by level"""
    y = np.zeros_like(x)
    dinv = np.linalg.inv(val[:, 0])
    for lev in range(level.max() + 1):
        es = np.nonzero(level == lev)[0]
        r = x[es].copy()
        for b in range(1, 4):
            c = col[es, b]
            use = (c >= 0) & (level[np.maximum(c, 0)] < lev)
            r[use] -= np.einsum("eij,ej->ei", val[es[use], b], y[c[use]])
        y[es] = np.einsum("eij,ej->ei", dinv[es], r)
    return y


def step(g, T0, ntime, nits, tol, max_iters):
    """pamg_implicit_step on the operator assembled last (with its k), from T0"""
    import ctypes as C
    g._ck(g.L.pamg_unstr_upload(g.h, np.ascontiguousarray(T0)))
    it = C.c_int(0); rr = C.c_double(0.0)
    g._ck(g.L.pamg_implicit_step(g.h, ntime, nits, tol, max_iters, C.byref(it), C.byref(rr)))
    out = np.empty_like(T0)
    g._ck(g.L.pamg_unstr_download(g.h, out))
    return out, it.value, rr.value


@pytest.mark.parametrize("name,case", [("irregular", "uniform"), ("900_ele", "uniform"), ("irregular", "diffusion"),
                                       ("untitled8192", "diffusion"), ("irregular", "field"), ("900_ele", "field"),
                                       ("irregular", "stab"), ("untitled8192", "stab")])
def test_precond_apply_is_the_block_triangular_solve(meshes, name, case):
    mesh = meshes[name]
    E = mesh.U
    g = handle(mesh)
    if case == "field":
        g.set_velocity(random_field(E, 31))
    g.implicit_assemble(0.05, 0.6, -0.35, use_dir=True, k=0.3 if case == "diffusion" else 0.0)
    if case == "stab":
        g.unstr_implicit(rng_field((E, 3), 32), 0.02, 0.6, -0.35, ntime=1, nits=2, use_dir=True, with_stab=True)
    x = rng_field((E, 3), 33)
    val, col = g.implicit_bsr()
    assert rel_l2(g.implicit_precond_apply(x), np.einsum("eij,ej->ei", np.linalg.inv(val[:, 0]), x)) <= 1e-13
    g.implicit_set_precond("flow_gs")
    y = g.implicit_precond_apply(x)
    level, nlevels, lagged = g.implicit_flow_levels()
    assert nlevels == level.max() + 1
    if case == "uniform" or case == "stab":
        assert lagged == 0
    assert rel_l2(y, sweep_reference(val, col, level, x)) <= 1e-13
    assert np.array_equal(g.implicit_precond_apply(x), y)          # bit-identical applications
    if case in ("uniform", "stab"):                                   # M = A: the sweep inverts the operator
        assert rel_l2(g.implicit_apply(y), x) <= 1e-12


@pytest.mark.parametrize("name", NAMES + ["untitled8192", "synthetic8"])
def test_device_levels_follow_the_inflow_rule(meshes, name):
    mesh = meshes[name]
    g = handle(mesh)
    for u in [(0.9, 0.3), (-0.35, 0.8), (1.0, 0.0)]:
        g.implicit_assemble(0.05, u[0], u[1], use_dir=True)
        level, nlevels, lagged = g.implicit_flow_levels()
        want, _, nl, lag = pamg.flow_levels(mesh.neig, uniform_mask(mesh, u))
        assert np.array_equal(level, want) and (nlevels, lagged) == (nl, lag) and lagged == 0, u


def reference_solution(mesh, u, dt, T0, ntime):
    E = mesh.U
    if E <= 100:
        ref = T0.copy()
        assert orc.lib().orc_unstr_implicit(E, mesh.X, mesh.neig, mesh.fneig, u[0], u[1], dt, ntime, 1, 1, ref) == 0
        return ref
    if E <= 1000:
        A = np.zeros((3 * E, 3 * E)); M = np.zeros((3 * E, 3 * E))
        orc.lib().orc_unstr_implicit_assemble(E, mesh.X, mesh.neig, mesh.fneig, u[0], u[1], dt, 1, A, M)
        r = T0.ravel().copy()
        for _ in range(ntime):
            r = np.linalg.solve(A, M @ r)
        return r.reshape(E, 3)
    return vf.implicit_solve(mesh.X, mesh.neig, mesh.fneig, np.tile(np.array(u), (E, 3, 1)), T0, dt, ntime, 1, True)


@pytest.mark.parametrize("name", NAMES + ["synthetic8"])
@pytest.mark.parametrize("cfl", [4, 64, 1000])
def test_pure_advection_in_one_iteration(meshes, name, cfl):
    mesh = meshes[name]
    u = (0.9, 0.3)
    dt = cfl * float(np.sqrt(areas(mesh.X).min())) / np.hypot(*u)
    T0 = rng_field((mesh.U, 3), 34)
    g = handle(mesh)
    got, iters, relres = g.unstr_implicit(T0, dt, u[0], u[1], ntime=1, nits=1, use_dir=True, tol=1e-12, precond="flow_gs")
    assert iters == 1 and relres <= 1e-12
    assert rel_l2(got, reference_solution(mesh, u, dt, T0, 1)) <= 1e-10
    bj, it_bj, rr_bj = g.unstr_implicit(T0, dt, u[0], u[1], ntime=1, nits=1, use_dir=True, tol=1e-12, max_iters=2000)
    if rr_bj <= 1e-12:
        assert rel_l2(got, bj) <= 1e-10 and it_bj >= 1


@pytest.mark.parametrize("name", ["split1", "irregular"])
def test_random_field_with_stabilisation(meshes, name):
    mesh = meshes[name]
    U = 0.3 * random_field(mesh.U, 35)
    T0 = rng_field((mesh.U, 3), 36)
    dt = min(0.02, 0.1 * np.sqrt(areas(mesh.X).min()) / 0.3)
    out = {}
    for prec in ("block_jacobi", "flow_gs"):
        g = handle(mesh)
        g.set_velocity(U)
        out[prec] = g.unstr_implicit(T0, dt, 7.0, -9.0, ntime=2, nits=2, use_dir=True, tol=1e-13, max_iters=2000,
                                     with_stab=True, precond=prec)
    ref = of.implicit(mesh.X, mesh.neig, mesh.fneig, U, T0, dt, 2, 2, True, True)
    assert rel_l2(out["flow_gs"][0], ref) <= 1e-10 and rel_l2(out["flow_gs"][0], out["block_jacobi"][0]) <= 1e-10
    assert out["flow_gs"][1] <= out["block_jacobi"][1]


@pytest.mark.parametrize("name", ["irregular", "900_ele"])
@pytest.mark.parametrize("k", [0.01, 0.3])
def test_diffusion(meshes, name, k):
    mesh = meshes[name]
    E = mesh.U
    u = (0.9, 0.3)
    dt = 16.0 * float(np.sqrt(areas(mesh.X).min())) / np.hypot(*u)
    T0 = rng_field((E, 3), 37)
    A = np.zeros((3 * E, 3 * E)); M = np.zeros((3 * E, 3 * E))
    orc.lib().orc_unstr_implicit_assemble_diff(E, mesh.X, mesh.neig, mesh.fneig, u[0], u[1], k, dt, 1, A, M)
    ref = np.linalg.solve(A, M @ T0.ravel()).reshape(E, 3)
    out = {}
    for prec in ("block_jacobi", "flow_gs"):
        g = handle(mesh)
        g.implicit_set_precond(prec)
        g.implicit_assemble(dt, u[0], u[1], use_dir=True, k=k)
        out[prec] = step(g, T0, 1, 1, 1e-13, 3000)
    assert rel_l2(out["flow_gs"][0], ref) <= 1e-10 and rel_l2(out["flow_gs"][0], out["block_jacobi"][0]) <= 1e-10
    assert out["flow_gs"][1] <= out["block_jacobi"][1]


def test_state_rules(meshes):
    mesh = meshes["irregular"]
    E = mesh.U
    g = pamg.SemiImplicitIterative(pamg.default_params(), pamg.Mesh.synthetic(0, 1))
    assert g.L.pamg_implicit_set_precond(g.h, 1) == pamg.ERR_STATE          # no mesh yet
    assert g.L.pamg_implicit_set_precond(g.h, 7) == pamg.ERR_ARG
    g.set_unstructured(mesh)
    assert g.L.pamg_implicit_set_precond(g.h, 2) == pamg.ERR_ARG
    assert g.L.pamg_implicit_set_precond(g.h, -1) == pamg.ERR_ARG
    with pytest.raises(ValueError):
        g.implicit_set_precond("ilu")
    g.implicit_set_precond("flow_gs")                                        # before assembly
    x = rng_field((E, 3), 38)
    assert g.L.pamg_implicit_precond_apply(g.h, x, np.empty_like(x)) == pamg.ERR_STATE
    assert g.L.pamg_implicit_flow_levels(g.h, None, None, None) == pamg.ERR_STATE
    g.implicit_assemble(0.05, 0.6, -0.35, use_dir=True)
    assert g.implicit_flow_levels()[2] == 0
    # a rotating field: the levels are rebuilt and its cycles are lagged
    g.set_velocity(rotating_field(mesh.X))
    assert g.L.pamg_implicit_flow_levels(g.h, None, None, None) == pamg.ERR_STATE   # stale until the next assembly
    g.implicit_assemble(0.05, 0.0, 0.0, use_dir=True)
    level, nlevels, lagged = g.implicit_flow_levels()
    assert lagged > 0
    val, col = g.implicit_bsr()
    assert rel_l2(g.implicit_precond_apply(x), sweep_reference(val, col, level, x)) <= 1e-13
    # dt and k keep the levels; back to the uniform velocity rebuilds them
    g.implicit_assemble(0.5, 0.0, 0.0, use_dir=True, k=0.2)
    assert np.array_equal(g.implicit_flow_levels()[0], level)
    g.set_velocity(None)
    g.implicit_assemble(0.05, 0.6, -0.35, use_dir=True)
    assert g.implicit_flow_levels()[2] == 0
    # a different uniform velocity rebuilds them too
    a = g.implicit_flow_levels()[0]
    g.implicit_assemble(0.05, -0.6, 0.35, use_dir=True)
    b = g.implicit_flow_levels()[0]
    assert not np.array_equal(a, b) and b.max() == a.max()
    # the choice survives a new mesh
    g.set_unstructured(mesh)
    g.implicit_assemble(0.05, 0.6, -0.35, use_dir=True)
    val, col = g.implicit_bsr()
    assert rel_l2(g.implicit_precond_apply(x), sweep_reference(val, col, g.implicit_flow_levels()[0], x)) <= 1e-13


def test_multi_device_handle_reaches_part0(meshes):
    mesh = meshes["irregular"]
    src = pamg.Mesh.synthetic(2, 2)
    g = pamg.SemiImplicitIterative(pamg.default_params(n_split=3, multi_levels=3), src, devices=[0, 0])
    g.set_unstructured(mesh)
    u = (0.9, 0.3)
    dt = 64.0 * float(np.sqrt(areas(mesh.X).min()))
    T0 = rng_field((mesh.U, 3), 39)
    got, iters, _ = g.unstr_implicit(T0, dt, u[0], u[1], ntime=1, nits=1, use_dir=True, tol=1e-12, precond="flow_gs")
    assert iters == 1 and rel_l2(got, reference_solution(mesh, u, dt, T0, 1)) <= 1e-10
    assert g.implicit_flow_levels()[2] == 0


def test_full_size_rotating_field():
    """4^11 triangles, a rotating field: the true residual of the returned solution is at the tolerance and a bump in the
    middle keeps its mass"""
    um = pamg.Mesh.synthetic(11, 1)
    E = um.U
    g = handle(um)
    g.set_velocity(rotating_field(um.X))
    area = areas(um.X)
    h = float(np.sqrt(area.min()))
    umax = 0.5 * float(um.X.max() - um.X.min())
    dt = 16.0 * h / umax
    cx = um.X.mean(axis=1)
    L = float(um.X.max() - um.X.min())
    r2 = (cx[:, 0] - cx[:, 0].mean()) ** 2 + (cx[:, 1] - cx[:, 1].mean()) ** 2
    T0 = np.repeat(np.exp(-r2 / (0.03 * L) ** 2)[:, None], 3, axis=1)
    got, iters, relres = g.unstr_implicit(T0, dt, 0.0, 0.0, ntime=1, nits=1, use_dir=True, tol=1e-11, max_iters=400,
                                          precond="flow_gs")
    assert relres <= 1e-11 and 0 < iters < 400
    assert g.implicit_flow_levels()[2] > 0
    sT = T0.sum(axis=1)
    b = (area / (12 * dt))[:, None] * (T0 + sT[:, None])
    r = b - g.implicit_apply(got)
    assert np.linalg.norm(r) <= 1e-10 * np.linalg.norm(b)
    mass0 = float(np.sum(area[:, None] / 3.0 * T0)); mass1 = float(np.sum(area[:, None] / 3.0 * got))
    assert abs(mass1 - mass0) <= 1e-9 * abs(mass0)
