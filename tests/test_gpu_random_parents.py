"""The semi-structured path on a random parent mesh whose faces take every branch of the halo tables, against the oracle.

The sweep kernels never see a parent face: they read a neighbour's children through host-built tables (hmap, rev, the packed
strip-free descriptor nsrc) and the orientation-folded parent tables, and the branch a face takes is picked by the parent's
gmsh side s, the neighbour's side ns (fNeig) and the reversal flag Dir - 18 combinations.  The shipped meshes hold at most 11.
helpers.random_parent_mesh(2) (32 parents, every triangle in a random vertex order) holds all 18, both orientations and
domain-boundary faces on all three sides (asserted on the CPU in test_host_random_parents.py), and here every kernel family the
dispatcher can select runs on it:

    n_split   Jacobi / Richardson / residual   two-colour GS
    1-3       k_element_direct2                k_gs_small
    4         k_element_win                    k_gs_small
    5         k_element_win                    k_gs_win
    6-8       k_element_win2                   k_gs_win2
    9         k_element_tma                    two in-place k_element_tma<GS> passes

(test_dispatch_selects_the_family_of_each_row checks that table against the kernels actually launched).  Tolerances as in
test_gpu_parity.py: relative L2 <= 1e-12 per sweep and per residual, copies bit-exact, Dirichlet data 4e-16.  A failing
comparison reports the largest error per face class, so the broken branch can be read off the message."""
import os
import re

import numpy as np
import pytest

import oracle_api as orc
from helpers import ALL_FACE_COMBINATIONS, face_combinations, random_parent_mesh, rel_l2, rng_field
from pamg_pkg import pamg
from test_gpu_parity import make_pair, seed_fields

pytestmark = pytest.mark.gpu
TOL = 1e-12
SEED = 2
os.environ.setdefault("PAMG_P2P_TIMEOUT_S", "30")     # a protocol bug must fail the test, not hang the box

VELOCITIES = [(0.9, 0.3), (-0.4, 0.7)]               # upwinding flips between the two across the face classes
N_SPLITS = list(range(1, 10))


def nsweeps(n):
    return 1 if n == 9 else 3                         # n_split 9: 8.4M children, one sweep of each kind bounds the oracle


@pytest.fixture(scope="module")
def mesh():
    m = pamg.Mesh.from_arrays(random_parent_mesh(SEED))
    assert face_combinations(m.neig, m.fneig, m.dir) == ALL_FACE_COMBINATIONS
    orc.lib().orc_semi_set_threads(os.cpu_count() or 1)
    return m


# ----------------------------------------------------------------------------------------------------- per-class errors
def face_class(mesh, u, f):
    if mesh.neig[u, f] == 0:
        return ("boundary", f + 1)
    return (f + 1, int(mesh.fneig[u, f]), int(mesh.dir[u, f]))


def surface_children(n):
    """0-based children of a parent along gmsh sides 1, 2, 3 (surf_ele), shape (3, 2**n)."""
    surf = np.zeros(3 * 2 ** n, np.int32)
    orc.lib().orc_surf_ele(n, surf)
    return surf.reshape(3, 2 ** n) - 1


def class_report(mesh, n, got, ref):
    """max |got - ref| over the children along the parent faces of each (s, ns, dir) class, along each domain-boundary side,
    over the corner children (on two parent faces, so they belong to no single class) and over the children on no parent
    face.  got / ref: fields (U, 4**n, 3) or strips (U, 3, 2**n, 3)."""
    got, ref = np.asarray(got), np.asarray(ref)
    worst = {}
    if got.ndim == 4:                                 # strips: one per parent face
        err = np.abs(got - ref).reshape(mesh.U, 3, -1).max(axis=2)
        for u in range(mesh.U):
            for f in range(3):
                k = face_class(mesh, u, f)
                worst[k] = max(worst.get(k, 0.0), float(err[u, f]))
    else:
        err = np.abs(got - ref).reshape(mesh.U, 4 ** n, -1).max(axis=2)
        surf = surface_children(n)
        faces = np.zeros(4 ** n, np.int32)
        np.add.at(faces, surf.ravel(), 1)
        for name, sel in (("inside", faces == 0), ("corners", faces > 1)):
            worst[name] = float(err[:, sel].max()) if sel.any() else 0.0
        for u in range(mesh.U):
            for f in range(3):
                k = face_class(mesh, u, f)
                own = surf[f][faces[surf[f]] == 1]
                if own.size:
                    worst[k] = max(worst.get(k, 0.0), float(err[u, own].max()))
    return "max |error| per face class: " + ", ".join("%s %.2e" % (k, v) for k, v in sorted(worst.items(), key=str))


def check(mesh, n, got, ref, what, tol=TOL):
    r = rel_l2(got, ref)
    assert r <= tol, "%s: rel-L2 %.3e > %.0e; %s" % (what, r, tol, class_report(mesh, n, got, ref))


def check_strips(mesh, n, got, ref, what):
    interior = mesh.neig != 0
    assert np.array_equal(got[interior], ref[interior]), "%s copies: %s" % (what, class_report(mesh, n, got, ref))
    assert np.allclose(got[~interior], ref[~interior], rtol=0, atol=4e-16), "%s Dirichlet: %s" % (
        what, class_report(mesh, n, got, ref))


def check_residual(mesh, n, o, g):
    o.field(orc.TNEW)[:] = o.field(orc.TNONLIN)
    g.copy(1, pamg.TNEW, pamg.TNONLIN)
    o.update_overlaps(1); g.update_overlaps(1)
    l2o, lio = o.residual(1)
    l2g, lig = g.get_residual(1)
    check(mesh, n, g.download(pamg.RES), o.field(orc.RES), "residual")
    assert abs(l2g - l2o) <= 1e-12 * l2o and abs(lig - lio) <= 1e-12 * lio, (l2g, l2o, lig, lio)
    assert abs(g.get_convergence(1) - o.convergence(1)) <= 1e-12 * max(1.0, abs(lio))


# ----------------------------------------------------------------------------------------------------- every family
@pytest.mark.parametrize("n", N_SPLITS)
@pytest.mark.parametrize("rule", [0, 1])
def test_update_overlaps(mesh, n, rule):
    o, g = make_pair(mesh, n, 1, True, u=VELOCITIES[0], halo_rule=rule)
    seed_fields(o, g)
    o.update_overlaps(1)
    g.update_overlaps(1)
    check_strips(mesh, n, g.overlap(1), o.overlap(1), "strips")
    check_strips(mesh, n, g.overlap(1, old=True), o.overlap(1, old=True), "old-time strips")


@pytest.mark.parametrize("n", N_SPLITS)
@pytest.mark.parametrize("literal_source", [0, 1])
def test_build_rhs(mesh, n, literal_source):
    o, g = make_pair(mesh, n, 1, True, u=VELOCITIES[0], literal_source=literal_source)
    seed_fields(o, g)
    o.build_rhs()
    g.get_RHS()
    check(mesh, n, g.download(pamg.RHS), o.field(orc.RHS), "rhs")


SWEEP_CASES = [(n, u) for n in N_SPLITS for u in VELOCITIES] + [(6, (0.0, 0.0))]


@pytest.mark.parametrize("n,u", SWEEP_CASES)
def test_jacobi_sweeps_and_residual(mesh, n, u):
    o, g = make_pair(mesh, n, 1, True, u=u)
    seed_fields(o, g)
    for sweep in range(nsweeps(n)):
        o.smooth(1, 1, 1)
        g.smoother(1, pamg.JACOBI, 1)
        check(mesh, n, g.download(pamg.TNONLIN), o.field(orc.TNONLIN), "Jacobi sweep %d" % sweep)
        check(mesh, n, g.download(pamg.TNEW), o.field(orc.TNEW), "tnew after Jacobi sweep %d" % sweep)
    check_residual(mesh, n, o, g)


@pytest.mark.parametrize("n,u", SWEEP_CASES)
def test_richardson_sweep(mesh, n, u):
    # (the default omega 0.8: with a tiny omega the update omega * r, and any error in its face terms, would sit far below
    # the tolerance on the iterate)
    o, g = make_pair(mesh, n, 1, True, u=u)
    seed_fields(o, g)
    o.smooth(1, 2, 1)
    g.smoother(1, pamg.RICHARDSON, 1)
    check(mesh, n, g.download(pamg.TNONLIN), o.field(orc.TNONLIN), "Richardson sweep")


@pytest.mark.parametrize("n,u", SWEEP_CASES)
def test_two_colour_gauss_seidel_sweeps(mesh, n, u):
    o, g = make_pair(mesh, n, 1, True, u=u, keep_tnew_gs=1)
    seed_fields(o, g)
    for sweep in range(nsweeps(n)):
        o.smooth(1, 4, 1)                       # the oracle runs the same colouring: down children, then up
        g.smoother(1, pamg.GAUSS_SEIDEL, 1)
        check(mesh, n, g.download(pamg.TNONLIN), o.field(orc.TNONLIN), "GS sweep %d" % sweep)
        check(mesh, n, g.download(pamg.TNEW), o.field(orc.TNEW), "tnew after GS sweep %d" % sweep)


@pytest.mark.parametrize("n", [2, 5, 6, 9])
def test_literal_head_parameters(mesh, n):
    """face_terms = 0, halo_rule = 0 (the checked-in composition): strips by the literal reversal table, the in-place GS
    passes of every level size, Jacobi and the residual."""
    o, g = make_pair(mesh, n, 1, False, u=VELOCITIES[0], keep_tnew_gs=1)
    assert g.params.face_terms == 0 and g.params.halo_rule == 0
    seed_fields(o, g)
    o.update_overlaps(1); g.update_overlaps(1)
    check_strips(mesh, n, g.overlap(1), o.overlap(1), "literal strips")
    for sweep in range(nsweeps(n)):
        o.smooth(1, 1, 1); g.smoother(1, pamg.JACOBI, 1)
        check(mesh, n, g.download(pamg.TNONLIN), o.field(orc.TNONLIN), "literal Jacobi sweep %d" % sweep)
    for sweep in range(nsweeps(n)):
        o.smooth(1, 4, 1); g.smoother(1, pamg.GAUSS_SEIDEL, 1)
        check(mesh, n, g.download(pamg.TNONLIN), o.field(orc.TNONLIN), "literal GS sweep %d" % sweep)
    check_residual(mesh, n, o, g)


# ---------------------------------------------------------------------------------------------- transfers, theta, V-cycle
@pytest.mark.parametrize("transfer", [0, 1])
def test_restrict_and_prolong_every_level(mesh, transfer):
    n = 6
    o, g = make_pair(mesh, n, n, True, u=VELOCITIES[0], transfer=transfer)
    for lvl in range(1, n):
        shape_f, shape_c = g.shape(lvl), g.shape(lvl + 1)
        sf, sc = n - lvl + 1, n - lvl
        R = rng_field(shape_f, 7 + lvl)
        o.field(orc.RES, lvl)[:] = R
        g.upload(pamg.RES, lvl, R)
        o.restrict(lvl); g.restrictor(lvl)
        check(mesh, sc, g.download(pamg.RHS, lvl + 1), o.field(orc.RHS, lvl + 1), "restriction of level %d" % lvl)
        Tf, Tc = rng_field(shape_f, 70 + lvl), rng_field(shape_c, 700 + lvl)
        for fld_o in (orc.TNONLIN, orc.TNEW):
            o.field(fld_o, lvl)[:] = Tf; o.field(fld_o, lvl + 1)[:] = Tc
        g.upload(pamg.TNONLIN, lvl, Tf); g.copy(lvl, pamg.TNEW, pamg.TNONLIN)
        g.upload(pamg.TNONLIN, lvl + 1, Tc); g.copy(lvl + 1, pamg.TNEW, pamg.TNONLIN)
        o.prolong(lvl); g.prolongator(lvl)
        fo, fg = (orc.TNEW, pamg.TNEW) if transfer == 0 else (orc.TNONLIN, pamg.TNONLIN)
        check(mesh, sf, g.download(fg, lvl), o.field(fo, lvl), "prolongation to level %d" % lvl)


@pytest.mark.parametrize("n", [3, 6])
@pytest.mark.parametrize("u", VELOCITIES)
def test_theta_half(mesh, n, u):
    """theta = 1/2: the old-time pass of get_RHS reads ovl_old through every face class."""
    o, g = make_pair(mesh, n, 1, True, u=u, theta=0.5, keep_tnew_gs=1)
    assert g.params.theta == 0.5
    seed_fields(o, g)
    o.build_rhs(); g.get_RHS()
    check(mesh, n, g.download(pamg.RHS), o.field(orc.RHS), "theta 1/2 rhs")
    o.smooth(1, 1, 1); g.smoother(1, pamg.JACOBI, 1)
    check(mesh, n, g.download(pamg.TNONLIN), o.field(orc.TNONLIN), "theta 1/2 Jacobi sweep")
    o.smooth(1, 4, 1); g.smoother(1, pamg.GAUSS_SEIDEL, 1)
    check(mesh, n, g.download(pamg.TNONLIN), o.field(orc.TNONLIN), "theta 1/2 GS sweep")
    check_residual(mesh, n, o, g)


@pytest.mark.parametrize("solver", [pamg.JACOBI, pamg.GAUSS_SEIDEL])
def test_vcycle_to_1e8_matches_oracle(mesh, solver):
    """Also runs the norm-fused Jacobi sweep (k_element_win2<JACOBI, .., NORM>), which only the V-cycle selects."""
    n = 6
    o, g = make_pair(mesh, n, n, True, u=VELOCITIES[0])
    it_o, hist_o = o.vcycle_solve(solver=4 if solver == pamg.GAUSS_SEIDEL else 1, nu1=4, nu2=4, ncoarse=15, max_cycles=40,
                                  tol=1e-8)
    it_g, hist_g = g.vcycle_solve(solver=solver, nu1=4, nu2=4, ncoarse=15, max_cycles=40, tol=1e-8)
    assert it_g <= 40 and abs(it_g - it_o) <= 1, (it_g, it_o)
    assert hist_g[-1] / hist_g[0] <= 1e-8
    m = min(len(hist_o), len(hist_g))
    assert np.allclose(hist_g[:m], hist_o[:m], rtol=1e-6)
    if it_g == it_o:
        sol_o, sol_g = o.field(orc.TNONLIN), g.download(pamg.TNONLIN)
        assert np.max(np.abs(sol_g - sol_o)) <= 1e-10 * max(1.0, np.max(np.abs(sol_o))), class_report(mesh, n, sol_g, sol_o)


# ----------------------------------------------------------------------------------------------------- cut faces
def test_cut_faces_on_three_parts_equal_single_gpu_and_oracle(mesh):
    """devices = [0, 0, 0]: the 32 parents in the blocks the handle cuts (U * i / 3); cut faces go through the exchanged strips,
    so the reversal and node pairing of rev / hmap on cut faces meet every kind of pairing too."""
    n, nparts = 6, 3
    pf = np.array([mesh.U * i // nparts for i in range(nparts + 1)], np.int32)
    revs, classes = set(), set()
    for part in range(nparts):
        plan = pamg.halo_plan(mesh, halo_rule=1, nparts=nparts, part_first=pf, my_part=part)
        rev = plan["rev"].reshape(-1, 3)
        for ul in range(pf[part + 1] - pf[part]):
            u = pf[part] + ul
            for f in range(3):
                q = mesh.neig[u, f]
                if q != 0 and not pf[part] <= q - 1 < pf[part + 1]:
                    revs.add(int(rev[ul, f]))
                    classes.add(face_class(mesh, u, f))
    assert revs == {0, 1} and len(classes) >= 6, (revs, classes)

    u = VELOCITIES[0]
    params = pamg.default_params(n_split=n, multi_levels=n, u_x=u[0], u_y=u[1])
    g = pamg.SemiImplicitIterative(params, mesh, devices=[0] * nparts)
    ref = pamg.SemiImplicitIterative(params, mesh)
    o = orc.Semi(orc.intended_params(n, n, dt=params.dt, u=u), mesh.X, mesh.neig, mesh.fneig, mesh.dir)
    shape = (mesh.U, 4 ** n, 3)
    T, Told = rng_field(shape, 4242), rng_field(shape, 4243)
    for s in (g, ref):
        s.upload(pamg.TNONLIN, 1, T); s.copy(1, pamg.TNEW, pamg.TNONLIN); s.upload(pamg.TOLD, 1, Told)
    o.field(orc.TNONLIN)[:] = T; o.field(orc.TNEW)[:] = T; o.field(orc.TOLD)[:] = Told
    g.update_overlaps(1); ref.update_overlaps(1); o.update_overlaps(1)
    ovg = g.overlap(1)
    assert np.array_equal(ovg, ref.overlap(1)), class_report(mesh, n, ovg, ref.overlap(1))
    assert np.array_equal(g.overlap(1, old=True), ref.overlap(1, old=True))
    check_strips(mesh, n, ovg, o.overlap(1), "strips of the parts")
    for s in (g, ref):
        s.smoother(1, pamg.JACOBI, 3)
        s.smoother(1, pamg.GAUSS_SEIDEL, 2)
    o.smooth(1, 1, 3); o.smooth(1, 4, 2)
    got = g.download(pamg.TNONLIN, 1)
    check(mesh, n, got, ref.download(pamg.TNONLIN, 1), "sweeps: parts against one handle", tol=1e-14)
    check(mesh, n, got, o.field(orc.TNONLIN), "sweeps: parts against the oracle")
    for s in (g, ref):
        s.copy(1, pamg.TNEW, pamg.TNONLIN); s.update_overlaps(1)
    o.field(orc.TNEW)[:] = o.field(orc.TNONLIN); o.update_overlaps(1)
    l2g, lig = g.get_residual(1); l2r, lir = ref.get_residual(1); l2o, lio = o.residual(1)
    assert abs(l2g - l2r) <= 1e-13 * l2r and lig == lir
    assert abs(l2g - l2o) <= 1e-12 * l2o and abs(lig - lio) <= 1e-12 * lio
    res = g.download(pamg.RES, 1)
    check(mesh, n, res, ref.download(pamg.RES, 1), "residual: parts against one handle", tol=1e-14)
    check(mesh, n, res, o.field(orc.RES), "residual: parts against the oracle")
    # one V-cycle solve from zero (graphs per part, coarse levels agglomerated on part 0)
    for s in (g, ref):
        s.fill(pamg.TNONLIN, 1, 0.0); s.copy(1, pamg.TNEW, pamg.TNONLIN); s.fill(pamg.TOLD, 1, 0.0)
    cg, hg = g.vcycle_solve(solver=pamg.GAUSS_SEIDEL, max_cycles=40, tol=1e-8)
    cr, hr = ref.vcycle_solve(solver=pamg.GAUSS_SEIDEL, max_cycles=40, tol=1e-8)
    assert cg == cr and hg[-1] <= 1e-8 * hg[0]
    np.testing.assert_allclose(hg, hr, rtol=1e-6)
    assert np.max(np.abs(g.download(pamg.TNONLIN, 1) - ref.download(pamg.TNONLIN, 1))) <= 1e-10
    g.close(); ref.close()


# ----------------------------------------------------------------------------------------------------- dispatch
SWEEP_FAMILIES = ("k_element_direct2", "k_element_win", "k_element_win2", "k_element_tma", "k_gs_small", "k_gs_win",
                  "k_gs_win2")
DISPATCH_ROWS = [  # n_split, Jacobi / Richardson / residual family, GS family
    (1, "k_element_direct2", "k_gs_small"), (2, "k_element_direct2", "k_gs_small"), (3, "k_element_direct2", "k_gs_small"),
    (4, "k_element_win", "k_gs_small"), (5, "k_element_win", "k_gs_win"),
    (6, "k_element_win2", "k_gs_win2"), (7, "k_element_win2", "k_gs_win2"), (8, "k_element_win2", "k_gs_win2"),
    (9, "k_element_tma", "k_element_tma")]


def kernel_name(name):
    """function name of a launched kernel, from the demangled 'void k_element_win<0, true>(ElemArgs)' or the mangled
    '_Z13k_element_winILi0ELb1EEv8ElemArgs' form of the profiler's event name."""
    m = re.match(r"_ZN?(\d+)", name)
    if m:
        return name[m.end(): m.end() + int(m.group(1))]
    m = re.search(r"([A-Za-z_]\w*)\s*[<(]", name)
    return m.group(1) if m else name


def launched_families(names):
    return {kernel_name(nm) for nm in names} & set(SWEEP_FAMILIES)


def test_dispatch_selects_the_family_of_each_row(mesh):
    """Each row of the table of this module runs under torch.profiler: the sweep kernel launched is the family the row claims.
    Without this, a change of the dispatcher would quietly empty part of the matrix above."""
    from torch.profiler import ProfilerActivity, profile
    for n, elem, gs in DISPATCH_ROWS:
        g = pamg.SemiImplicitIterative(pamg.default_params(n_split=n, multi_levels=1, u_x=0.9, u_y=0.3), mesh)
        shape = g.shape(1)
        g.upload(pamg.TNONLIN, 1, rng_field(shape, 1)); g.copy(1, pamg.TNEW, pamg.TNONLIN)
        g.upload(pamg.TOLD, 1, rng_field(shape, 2))
        g.smoother(1, pamg.JACOBI, 1)               # right-hand side and first strips outside the captures
        g.sync()
        for what, run, want in (("Jacobi", lambda: g.smoother(1, pamg.JACOBI, 1), elem),
                                ("Richardson", lambda: g.smoother(1, pamg.RICHARDSON, 1), elem),
                                ("residual", lambda: g.get_residual(1), elem),
                                ("Gauss-Seidel", lambda: g.smoother(1, pamg.GAUSS_SEIDEL, 1), gs)):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run()
                g.sync()
            names = [e.name for e in prof.events()]
            assert launched_families(names) == {want}, (n, what, sorted(set(names)))
        g.close()
