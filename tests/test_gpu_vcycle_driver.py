"""The V-cycle driver (pamg_vcycle_solve) against the oracle, cycle by cycle.

The kernels are pinned launch by launch elsewhere; this file pins the host-side state of the driver above them: cycle 1 runs
eagerly and later cycles replay CUDA graphs cached per handle (at most 8), each captured for one schedule and one buffer
parity of every level; normalise_parity moves a level back after an odd sweep count; a fused Jacobi solve on a producer level
appends the first pre-sweep of cycle c+1 to cycle c as its norm sweep and takes it back when the solve stops
(undo_norm_sweep); group handles agglomerate the coarse levels on part 0.  Odd sweep counts make the parity of level 1 (and
of the strips of a producer level) alternate from cycle to cycle, so two graphs take turns.

The oracle's cycle depends on the level-1 iterate alone (it zeroes the coarse levels every cycle), so oracle solves of one
cycle each, run back to back, give its state after every cycle c.  The device runs vcycle_solve(max_cycles=c) from the same
zero start on the same handle for c = 1, 2, ..., so warm restarts and graph reuse are part of every comparison.  Tolerances:
the level-1 iterate to relative L2 <= 1e-11, the fields that shrink with the residual to 1e-11 of their norm after the first
cycle (check_state), and |h_gpu[k] - h_oracle[k]| <= 1e-11 h_oracle[0] for the residual history."""
import os

import numpy as np
import pytest

import oracle_api as orc
from helpers import random_parent_mesh, rel_l2, rng_field, write_msh
from pamg_pkg import pamg
from test_gpu_parity import make_pair

pytestmark = pytest.mark.gpu
TOL = 1e-11
VEL = (0.9, 0.3)
os.environ.setdefault("PAMG_P2P_TIMEOUT_S", "30")     # a protocol bug must fail the test, not hang the box

J, R, GS = pamg.JACOBI, pamg.RICHARDSON, pamg.GAUSS_SEIDEL
ORACLE_SOLVER = {J: 1, R: 2, GS: 4}                  # the oracle's solver 4 is the two-colour ordering of the GPU's GS
NAME = {J: "Jacobi", R: "Richardson", GS: "GS"}
# Richardson: omega * (b - A x).  The default omega 0.8 (test_richardson_sweep on the random parents) makes the V-cycle
# diverge by ~1e5 per cycle, which no bound relative to the first residual can follow; at 1e-4 it contracts (residual
# 0.89, 0.80, 0.73 of r0 over three (4,4,15) cycles) and the update is still a tenth of the error
RICHARDSON_OMEGA = 1e-4
# (nu1, nu2, ncoarse): odd and even nu1 + nu2, no pre-sweep left after the fusion (1, 0, 1), no post-sweep, odd ncoarse
SCHEDULES = [(4, 4, 15), (3, 4, 15), (1, 0, 1), (2, 3, 2), (0, 3, 4)]


def ids(v):
    return NAME[v] if isinstance(v, int) else "-".join(map(str, v))


@pytest.fixture(scope="module")
def meshes(tmp_path_factory):
    orc.lib().orc_semi_set_threads(os.cpu_count() or 1)
    d = tmp_path_factory.mktemp("msh")
    return {"random": pamg.Mesh.from_arrays(random_parent_mesh(2)),
            "split0": pamg.Mesh.read_msh(write_msh("split0", str(d / "split0.msh")))}


def make(mesh, n, levels, solver=J, devices=None, handle_solver=None):
    """oracle / device pair with a seeded TOLD (so the right-hand side is not just boundary data)."""
    kw = {"omega": RICHARDSON_OMEGA} if solver == R else {}
    o, g = make_pair(mesh, n, levels, True, u=VEL, **kw)
    if devices is not None or handle_solver is not None:
        p = g.params
        if handle_solver is not None:
            p.solver = handle_solver
        g.close()
        g = pamg.SemiImplicitIterative(p, mesh, devices=devices)
    told = rng_field(g.shape(1), 4711)
    o.field(orc.TOLD)[:] = told
    g.upload(pamg.TOLD, 1, told)
    zero_start(o, g)
    return o, g


def zero_start(o, g):
    o.field(orc.TNONLIN)[:] = 0.0
    o.field(orc.TNEW)[:] = 0.0
    g.fill(pamg.TNONLIN, 1, 0.0)
    g.copy(1, pamg.TNEW, pamg.TNONLIN)


def oracle_solve(o, solver, sched, cycles):
    """cycles of the oracle from its current state; (history, state after each cycle)."""
    hist, states = [], []
    for _ in range(cycles):
        _, h = o.vcycle_solve(solver=ORACLE_SOLVER[solver], nu1=sched[0], nu2=sched[1], ncoarse=sched[2], max_cycles=1,
                              tol=1e-30)
        if not hist:
            hist.append(h[0])
        hist.append(h[1])
        states.append(snapshot(o))
    return np.array(hist), states


def snapshot(o):
    L = o.params.multi_levels
    s = {("TNONLIN", lvl): o.field(orc.TNONLIN, lvl).copy() for lvl in range(1, L + 1)}
    s.update({("RHS", lvl): o.field(orc.RHS, lvl).copy() for lvl in range(2, L + 1)})
    s[("RES", 1)] = o.field(orc.RES, 1).copy()
    s[("TNEW", 1)] = o.field(orc.TNEW, 1).copy()
    return s


FIELD = {"TNONLIN": pamg.TNONLIN, "RHS": pamg.RHS, "RES": pamg.RES, "TNEW": pamg.TNEW}


def check_state(g, ref, what, first=None, levels=None):
    """every field of the oracle snapshot ref on levels <= levels (a group handle holds the levels past the agglomeration
    level on part 0's coarse problem, out of reach of download).  The level-1 iterate is held to TOL relative to its own
    norm.  The level-1 residual, and all the coarse levels hold (restricted residuals and the corrections solved from them),
    shrink with the residual and carry its cancellation: they are held to TOL times their norm in `first`, the oracle's
    state after the first cycle of the same solve.  (Relative to their own norm the errors reached 3.2e-11 for the level-1
    residual and 1.5e-11 for the level-2 right-hand side after four GS cycles, and 4.4e-11 for the level-2 right-hand side
    and 1.2e-11 for the level-2 iterate three cycles into a warm restart.)"""
    for (fld, lvl), want in sorted(ref.items()):
        if levels is not None and lvl > levels:
            continue
        got = g.download(FIELD[fld], lvl)
        if lvl == 1 and fld != "RES":
            r = rel_l2(got, want)
            assert r <= TOL, "%s: level %d %s rel-L2 %.3e > %.0e" % (what, lvl, fld, r, TOL)
        else:
            scale = float(np.linalg.norm((want if first is None else first[(fld, lvl)]).ravel()))
            err = float(np.linalg.norm((got - want).ravel()))
            assert err <= TOL * scale, "%s: level %d %s |error| %.3e > %.0e * %.3e (its norm after cycle 1)" % (
                what, lvl, fld, err, TOL, scale)


def check_hist(hg, ho, what):
    hg, ho = np.asarray(hg), np.asarray(ho)
    assert len(hg) == len(ho), (what, hg, ho)
    err = np.abs(hg - ho)
    k = int(np.argmax(err))
    assert err[k] <= TOL * ho[0], "%s: history entry %d gpu %.17g oracle %.17g" % (what, k, hg[k], ho[k])


def gpu_solve(g, solver, sched, cycles, tol=1e-30):
    return g.vcycle_solve(solver=solver, nu1=sched[0], nu2=sched[1], ncoarse=sched[2], max_cycles=cycles, tol=tol)


def cycle_by_cycle(o, g, solver, sched, cycles, levels=None):
    ho, states = oracle_solve(o, solver, sched, cycles)
    for c in range(1, cycles + 1):
        what = "%s %s cycle %d" % (NAME[solver], sched, c)
        g.fill(pamg.TNONLIN, 1, 0.0)
        g.copy(1, pamg.TNEW, pamg.TNONLIN)
        it, hg = gpu_solve(g, solver, sched, c)
        assert it == c + 1, (what, it)
        check_hist(hg, ho[:c + 1], what)
        check_state(g, states[c - 1], what, states[0], levels)


# ----------------------------------------------------------------------------------------------- a. cycle by cycle
@pytest.mark.parametrize("sched", SCHEDULES, ids=ids)
@pytest.mark.parametrize("solver", [J, R, GS], ids=ids)
def test_cycle_by_cycle_random_parents(meshes, solver, sched):
    """n_split 6: level 1 runs the fused k_element_win2 / k_gs_win2, the coarse levels k_element_win, k_element_direct2
    and k_gs_small."""
    o, g = make(meshes["random"], 6, 6, solver)
    cycle_by_cycle(o, g, solver, sched, 4)
    g.close()


@pytest.mark.parametrize("sched", [(4, 4, 15), (3, 4, 15)], ids=ids)
@pytest.mark.parametrize("solver", [J, GS], ids=ids)
def test_cycle_by_cycle_two_producer_levels(meshes, solver, sched):
    """split0, n_split 7, 3 levels: levels 1 and 2 (s = 7, 6) are both producer levels, the coarsest is s = 5."""
    o, g = make(meshes["split0"], 7, 3, solver)
    cycle_by_cycle(o, g, solver, sched, 4)
    g.close()


@pytest.mark.parametrize("solver", [J, GS], ids=ids)
def test_cycle_by_cycle_tma_level(meshes, solver):
    """split0, n_split 9: level 1 runs k_element_tma (in-place GS passes, no norm fusion)."""
    o, g = make(meshes["split0"], 9, 9, solver)
    cycle_by_cycle(o, g, solver, (3, 4, 15), 3)
    g.close()


# ----------------------------------------------------------------------------------------------- b. replay == eager
@pytest.mark.parametrize("solver,sched", [(J, (4, 4, 15)), (J, (3, 4, 15)), (GS, (3, 4, 15))], ids=ids)
def test_graph_replay_equals_eager(meshes, solver, sched):
    """With profiling on every cycle runs eagerly; the replayed graphs must give the same bits."""
    _, g = make(meshes["random"], 6, 6, solver)
    out = []
    for prof in (True, False, False, True):     # eager, capture, replay of the cached graphs, eager
        g.profile(prof)
        g.fill(pamg.TNONLIN, 1, 0.0)
        g.copy(1, pamg.TNEW, pamg.TNONLIN)
        _, h = gpu_solve(g, solver, sched, 4)
        out.append((h, g.download(pamg.TNONLIN, 1)))
    g.profile(False)
    for h, t in out[1:]:
        assert np.array_equal(h, out[0][0]), (h, out[0][0])
        assert np.array_equal(t, out[0][1])
    g.close()


# ----------------------------------------------------------------------------------------------- c. fused norms
@pytest.mark.parametrize("sched", [(4, 4, 15), (3, 4, 15)], ids=ids)
def test_fused_norms_equal_get_residual(meshes, sched):
    """The norm sweep of a fused Jacobi solve reduces the residual of the iterate it starts from: bit for bit what
    get_residual computes after a solve that stops there."""
    _, g = make(meshes["random"], 6, 6, J)
    _, h4 = gpu_solve(g, J, sched, 4)
    for c in range(1, 5):
        g.fill(pamg.TNONLIN, 1, 0.0)
        g.copy(1, pamg.TNEW, pamg.TNONLIN)
        _, hc = gpu_solve(g, J, sched, c)
        l2, _ = g.get_residual(1)
        assert hc[c] == l2 and h4[c] == l2, (c, hc[c], h4[c], l2)
    g.close()


# ----------------------------------------------------------------------------------------------- d. after a solve
def check_strips_of_own_iterate(o, g, what):
    """The device's level-1 strips after update_overlaps are copies of its own iterate: the oracle fills strips from the
    device's field and they must agree bit for bit on interior faces."""
    keep = o.field(orc.TNONLIN).copy(), o.field(orc.TNEW).copy()
    t = g.download(pamg.TNONLIN, 1)
    o.field(orc.TNONLIN)[:] = t
    o.field(orc.TNEW)[:] = t
    o.update_overlaps(1)
    ref = o.overlap(1).copy()
    o.field(orc.TNONLIN)[:], o.field(orc.TNEW)[:] = keep
    o.update_overlaps(1)
    got = g.overlap(1)
    interior = g.mesh.neig != 0
    assert np.array_equal(got[interior], ref[interior]), "%s: interior strips" % what
    assert np.allclose(got[~interior], ref[~interior], rtol=0, atol=4e-16), "%s: Dirichlet strips" % what


@pytest.mark.parametrize("stop", ["max_cycles", "tol"])
@pytest.mark.parametrize("solver,sched", [(J, (4, 4, 15)), (J, (3, 4, 15)), (GS, (3, 4, 15))], ids=ids)
def test_handle_after_a_solve(meshes, solver, sched, stop):
    """A solve stops after 3 cycles; a sweep, a halo update and a residual evaluation continue from where it stopped, on
    both sides.  The fused solve has taken back its norm sweep (undo_norm_sweep): iterate, field buffer and strip buffer."""
    o, g = make(meshes["random"], 6, 6, solver)
    stop_at = 3
    ho, states = oracle_solve(o, solver, sched, stop_at)
    assert ho[stop_at] < ho[stop_at - 1]
    if stop == "tol":       # halfway (geometric mean) between the relative residuals of cycles 2 and 3: stops after 3
        tol, max_cycles = float(np.sqrt(ho[stop_at - 1] * ho[stop_at]) / ho[0]), 40
    else:
        tol, max_cycles = 1e-30, stop_at
    zero_start(o, g)
    it_o, hist_o = o.vcycle_solve(solver=ORACLE_SOLVER[solver], nu1=sched[0], nu2=sched[1], ncoarse=sched[2],
                                  max_cycles=max_cycles, tol=tol)
    it_g, hist_g = gpu_solve(g, solver, sched, max_cycles, tol)
    assert it_g == it_o == (stop_at if stop == "tol" else stop_at + 1), (it_g, it_o)
    check_hist(hist_g, hist_o, "solve")
    check_state(g, snapshot(o), "after the solve", states[0])
    o.smooth(1, ORACLE_SOLVER[solver], 1)
    g.smoother(1, solver, 1)
    swept = {("TNONLIN", 1): o.field(orc.TNONLIN)}
    if solver != GS:          # (Jacobi: TNEW is the start-of-sweep field on both sides)
        swept[("TNEW", 1)] = o.field(orc.TNEW)
    check_state(g, swept, "sweep after the solve")
    o.field(orc.TNEW)[:] = o.field(orc.TNONLIN)
    g.copy(1, pamg.TNEW, pamg.TNONLIN)
    o.update_overlaps(1)
    g.update_overlaps(1)
    check_strips_of_own_iterate(o, g, "strips after the solve")
    l2o, lio = o.residual(1)
    l2g, lig = g.get_residual(1)
    check_state(g, {("RES", 1): o.field(orc.RES)}, "residual after the solve", states[0])
    r0 = hist_o[0]
    assert abs(l2g - l2o) <= TOL * r0 and abs(lig - lio) <= TOL * r0, (l2g, l2o, lig, lio)
    g.close()


# ----------------------------------------------------------------------------------------------- e. reuse of a handle
def fresh_solve(o, g, solver, sched, cycles, what):
    zero_start(o, g)
    ho, states = oracle_solve(o, solver, sched, cycles)
    _, hg = gpu_solve(g, solver, sched, cycles)
    check_hist(hg, ho, what)
    check_state(g, states[-1], what, states[0])


@pytest.mark.parametrize("solver", [J, GS], ids=ids)
def test_schedules_with_equal_packed_keys(meshes, solver):
    """(4, 4, 130) and (4, 6, 2) packed as ((solver*64 + nu1)*64 + nu2)*64 + ncoarse are the same number, and on n_split 6
    both leave every level with the same buffer parity after cycle 1: a cache keyed that way replays the first schedule's
    graph for the second."""
    o, g = make(meshes["random"], 6, 6, solver)
    for sched in [(4, 4, 130), (4, 6, 2)]:
        fresh_solve(o, g, solver, sched, 3, "%s %s" % (NAME[solver], sched))
    g.close()


def test_more_schedules_than_cached_graphs(meshes):
    """Nine schedules (alternating ones capture two graphs each) evict the first one's graphs; it runs again."""
    scheds = [(J, (4, 4, 15)), (J, (3, 4, 15)), (J, (2, 3, 2)), (J, (1, 0, 1)), (J, (0, 3, 4)), (GS, (4, 4, 15)),
              (GS, (3, 4, 15)), (GS, (2, 3, 2)), (GS, (0, 3, 4))]
    o, g = make(meshes["random"], 6, 6, J)
    for solver, sched in scheds + scheds[:1]:
        fresh_solve(o, g, solver, sched, 3, "%s %s" % (NAME[solver], sched))
    g.close()


def test_solve_sweeps_solve(meshes):
    """A solve, three Jacobi sweeps (odd: the parity of level 1 changes), a solve."""
    sched = (3, 4, 15)
    o, g = make(meshes["random"], 6, 6, J)
    fresh_solve(o, g, J, sched, 3, "first solve")
    o.smooth(1, 1, 3)
    g.smoother(1, J, 3)
    check_state(g, {("TNONLIN", 1): o.field(orc.TNONLIN)}, "sweeps")
    ho, states = oracle_solve(o, J, sched, 3)
    _, hg = gpu_solve(g, J, sched, 3)
    check_hist(hg, ho, "second solve")
    check_state(g, states[-1], "second solve", states[0])
    g.close()


def test_solve_smooth_host_solve(meshes):
    """A solve, pamg_smooth_host (which swaps the level-1 field buffers and drops the cached graphs), a solve."""
    sched = (3, 4, 15)
    o, g = make(meshes["random"], 6, 6, J)
    fresh_solve(o, g, J, sched, 3, "first solve")
    field = rng_field(g.shape(1), 99)
    n = field.size
    src, dst = pamg.PinnedBuffer(n), pamg.PinnedBuffer(n)
    src.array[:] = field.ravel()
    g.smooth_host(J, 3, src.ptr, dst.ptr)
    g.sync()
    o.field(orc.TNONLIN)[:] = field
    o.field(orc.TNEW)[:] = field
    o.smooth(1, 1, 3)
    r = rel_l2(dst.array, o.field(orc.TNONLIN))
    assert r <= TOL, r
    ho, states = oracle_solve(o, J, sched, 3)
    _, hg = gpu_solve(g, J, sched, 3)
    check_hist(hg, ho, "second solve")
    check_state(g, states[-1], "second solve", states[0])
    g.close()
    src.free(); dst.free()


@pytest.mark.parametrize("solver", [J, GS], ids=ids)
def test_timestep_host_steps(meshes, solver):
    """Three time steps of pamg_timestep_host (told = tnew, tnew_nonlin = tnew, V-cycles of the handle's schedule) against
    the oracle doing the same."""
    o, g = make(meshes["random"], 6, 6, solver, handle_solver=solver)
    p = g.params
    sched = (p.n_smooth, p.n_smooth, p.n_coarse_smooth)
    t = rng_field(g.shape(1), 5)
    o.field(orc.TNEW)[:] = t
    for step in range(3):
        o.field(orc.TOLD)[:] = o.field(orc.TNEW)
        o.field(orc.TNONLIN)[:] = o.field(orc.TNEW)
        ho, _ = oracle_solve(o, solver, sched, 3)
        out = np.empty_like(t)
        cyc, rel = g.timestep_host(t, out, max_cycles=3, tol=1e-30)
        assert cyc == 4, cyc
        assert abs(rel - ho[3] / ho[0]) <= TOL, (step, rel, ho[3] / ho[0])
        r = rel_l2(out, o.field(orc.TNONLIN))
        assert r <= TOL, "step %d: rel-L2 %.3e" % (step, r)
        t = out
    g.close()


# ----------------------------------------------------------------------------------------------- f. group handles
@pytest.mark.parametrize("ngpu", [2, 3])
@pytest.mark.parametrize("solver", [J, GS], ids=ids)
def test_cycle_by_cycle_group(meshes, solver, ngpu):
    """devices = [0] * ngpu: halo exchange between the parts, and the coarse levels agglomerated on part 0 from level 2 on
    (32 parents of 4**5 children fit its 2**17 elements), with its gather and scatter inside the graph."""
    o, g = make(meshes["random"], 6, 6, solver, devices=[0] * ngpu)
    cycle_by_cycle(o, g, solver, (3, 4, 15), 4, levels=2)
    g.close()
