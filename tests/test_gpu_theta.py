"""theta != 1 on the device (get_A_x / get_RHS, transport_tri_semi.F90:441-446,457-460) through the C ABI, against the oracle
and against the device's own theta = 1 path.

The weighted spatial terms are folded into the per-parent coefficient tables on the host; the old-time branch of get_RHS is a
residual-mode pass of the level-1 sweep kernel over TOLD with a second table (`add_old_time_terms`, csrc/pamg_api.cu).
Tolerance as everywhere: relative L2 <= 1e-12 per sweep / evaluation."""
import os

import numpy as np
import pytest

import oracle_api as orc
from helpers import rel_l2, rng_field, write_msh
from pamg_pkg import pamg

pytestmark = pytest.mark.gpu
TOL = 1e-12
os.environ.setdefault("PAMG_P2P_TIMEOUT_S", "30")


def make_pair(mesh, n, levels, theta, u=(0.0, 0.0), dt=1e-3):
    op = orc.intended_params(n, levels, dt=dt, u=u)
    op.theta = theta
    gp = pamg.default_params(n_split=n, multi_levels=levels)
    for f in ("face_terms", "literal_source", "transfer", "residual_sign", "halo_rule", "coarse_bc_zero",
              "theta", "dt", "k", "omega", "u_x", "u_y", "source_coef"):
        setattr(gp, f, getattr(op, f))
    return orc.Semi(op, mesh.X, mesh.neig, mesh.fneig, mesh.dir), pamg.SemiImplicitIterative(gp, mesh)


def seed_fields(o, g, seed=20221):
    T, Told = rng_field(g.shape(1), seed), rng_field(g.shape(1), seed + 1)
    o.field(orc.TNONLIN)[:] = T; o.field(orc.TNEW)[:] = T; o.field(orc.TOLD)[:] = Told
    g.upload(pamg.TNONLIN, 1, T); g.copy(1, pamg.TNEW, pamg.TNONLIN); g.upload(pamg.TOLD, 1, Told)


@pytest.fixture(scope="module")
def meshes(tmp_path_factory):
    d = tmp_path_factory.mktemp("msh_theta")
    out = {name: pamg.Mesh.read_msh(write_msh(name, str(d / (name + ".msh")))) for name in ("test_sn2", "split0", "irregular")}
    out["syn"] = pamg.Mesh.synthetic(1, 2)
    return out


# kernel families: n_split <= 3 direct, 4-5 window kernel with a CTA barrier, 6-8 window kernel with a producer warp
CASES = [("test_sn2", 3, 0.5, (0.9, 0.3)), ("irregular", 2, 0.25, (-0.4, 0.7)), ("split0", 5, 0.5, (0.9, 0.3)),
         ("syn", 6, 0.5, (0.9, 0.3)), ("split0", 7, 0.75, (-0.5, 0.8)), ("test_sn2", 4, 0.0, (0.3, -0.2))]


@pytest.mark.parametrize("name,n,theta,u", CASES)
def test_rhs_sweeps_and_residual_match_the_oracle(meshes, name, n, theta, u):
    o, g = make_pair(meshes[name], n, 1, theta, u=u)
    seed_fields(o, g)
    o.build_rhs(); g.get_RHS()
    assert rel_l2(g.download(pamg.RHS), o.field(orc.RHS)) <= TOL
    for sweep in range(2):
        o.smooth(1, 1, 1); g.smoother(1, pamg.JACOBI, 1)
        assert rel_l2(g.download(pamg.TNONLIN), o.field(orc.TNONLIN)) <= TOL, sweep
    o.smooth(1, 4, 1); g.smoother(1, pamg.GAUSS_SEIDEL, 1)
    assert rel_l2(g.download(pamg.TNONLIN), o.field(orc.TNONLIN)) <= TOL
    o.smooth(1, 2, 1); g.smoother(1, pamg.RICHARDSON, 1)
    assert rel_l2(g.download(pamg.TNONLIN), o.field(orc.TNONLIN)) <= TOL
    o.field(orc.TNEW)[:] = o.field(orc.TNONLIN); g.copy(1, pamg.TNEW, pamg.TNONLIN)
    o.update_overlaps(1); g.update_overlaps(1)
    l2o, _ = o.residual(1); l2g, _ = g.get_residual(1)
    assert rel_l2(g.download(pamg.RES), o.field(orc.RES)) <= TOL
    assert abs(l2g - l2o) <= 1e-12 * l2o
    # a new told invalidates the right-hand side: it is rebuilt with the old-time terms of the NEW told
    Told2 = rng_field(g.shape(1), 77)
    o.field(orc.TOLD)[:] = Told2; g.upload(pamg.TOLD, 1, Told2)
    o.smooth(1, 1, 1); g.smoother(1, pamg.JACOBI, 1)
    assert rel_l2(g.download(pamg.TNONLIN), o.field(orc.TNONLIN)) <= TOL


@pytest.mark.parametrize("name,n,theta", [("test_sn2", 3, 0.5), ("syn", 6, 0.25)])
def test_old_time_branch_equals_the_theta_one_path_of_the_device(meshes, name, n, theta):
    """R_th(x, told) = R_1(x, told) - (1 - theta) [R_1(x, x) - R_1(told, told)]: the device against itself, no oracle."""
    mesh = meshes[name]
    kw = dict(n_split=n, multi_levels=1, u_x=0.6, u_y=-0.3, dt=1e-2, k=0.05)
    g1 = pamg.SemiImplicitIterative(pamg.default_params(theta=1.0, **kw), mesh)
    gt = pamg.SemiImplicitIterative(pamg.default_params(theta=theta, **kw), mesh)
    shape = g1.shape(1)
    x, told = rng_field(shape, 3), rng_field(shape, 4)

    def resid(g, a, b):
        g.upload(pamg.TNONLIN, 1, a); g.copy(1, pamg.TNEW, pamg.TNONLIN); g.upload(pamg.TOLD, 1, b)
        g.update_overlaps(1)
        g.get_residual(1)
        return g.download(pamg.RES)
    lhs = resid(gt, x, told)
    rhs = resid(g1, x, told) - (1.0 - theta) * (resid(g1, x, x) - resid(g1, told, told))
    assert rel_l2(lhs, rhs) <= TOL
    g1.close(); gt.close()


@pytest.mark.parametrize("solver", [pamg.JACOBI, pamg.GAUSS_SEIDEL])
def test_crank_nicolson_time_steps_with_vcycles(meshes, solver):
    n, theta = 6, 0.5
    o, g = make_pair(meshes["syn"], n, n, theta, u=(0.9, 0.3))
    orc.lib().orc_semi_set_threads(os.cpu_count() or 1)
    T0 = rng_field(g.shape(1), 11)
    o.field(orc.TNONLIN)[:] = T0; o.field(orc.TNEW)[:] = T0
    g.upload(pamg.TNONLIN, 1, T0); g.copy(1, pamg.TNEW, pamg.TNONLIN)
    for step in range(2):                                   # do itime (:299-381): told = tnew, V-cycles to 1e-8
        o.field(orc.TOLD)[:] = o.field(orc.TNONLIN); o.field(orc.TNEW)[:] = o.field(orc.TNONLIN)
        g.copy(1, pamg.TNEW, pamg.TNONLIN); g.copy(1, pamg.TOLD, pamg.TNEW)
        co, ho = o.vcycle_solve(solver=4 if solver == pamg.GAUSS_SEIDEL else 1, nu1=4, nu2=4, ncoarse=15, max_cycles=40, tol=1e-8)
        cg, hg = g.vcycle_solve(solver=solver, nu1=4, nu2=4, ncoarse=15, max_cycles=40, tol=1e-8)
        assert cg <= 40 and abs(cg - co) <= 1 and hg[-1] <= 1e-8 * hg[0], (step, cg, co)
        k = min(len(hg), len(ho))
        assert np.allclose(hg[:k], ho[:k], rtol=1e-6)
        if cg != co:            # (a residual within rounding of the tolerance: the two runs stop one cycle apart)
            break
        assert rel_l2(g.download(pamg.TNONLIN), o.field(orc.TNONLIN)) <= 1e-9, step


def test_partitioned_mesh_exchanges_the_told_strips():
    """three parts on one device: the told values of the cut faces travel into the neighbours' told strips before the
    old-time pass (exchange_told); result equal to the single handle's"""
    kp, n, theta = 2, 6, 0.5
    mesh = pamg.Mesh.synthetic(kp, 2)
    params = pamg.default_params(n_split=n, multi_levels=n, u_x=0.9, u_y=0.3, theta=theta)
    g = pamg.SemiImplicitIterative(params, mesh, devices=[0, 0, 0])
    ref = pamg.SemiImplicitIterative(params, mesh)
    shape = (mesh.U, 4 ** n, 3)
    T, Told = rng_field(shape, 4242), rng_field(shape, 4243)
    for s in (g, ref):
        s.upload(pamg.TNONLIN, 1, T); s.copy(1, pamg.TNEW, pamg.TNONLIN); s.upload(pamg.TOLD, 1, Told)
        s.get_RHS()
    assert rel_l2(g.download(pamg.RHS, 1), ref.download(pamg.RHS, 1)) <= 1e-14
    for s in (g, ref):
        s.smoother(1, pamg.JACOBI, 3); s.smoother(1, pamg.GAUSS_SEIDEL, 2)
    assert rel_l2(g.download(pamg.TNONLIN, 1), ref.download(pamg.TNONLIN, 1)) <= 1e-14
    for s in (g, ref):
        s.copy(1, pamg.TNEW, pamg.TNONLIN); s.copy(1, pamg.TOLD, pamg.TNEW)
    cg, hg = g.vcycle_solve(solver=pamg.GAUSS_SEIDEL, max_cycles=40, tol=1e-8)
    cr, hr = ref.vcycle_solve(solver=pamg.GAUSS_SEIDEL, max_cycles=40, tol=1e-8)
    assert cg == cr and hg[-1] <= 1e-8 * hg[0]
    np.testing.assert_allclose(hg, hr, rtol=1e-6)
    g.close(); ref.close()
