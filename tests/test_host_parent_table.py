"""The folded per-parent operator table of the product (host code of libpamg_cuda.so, pamg_parent_table: no GPU needed)
against the level-1 matrix the oracle assembles from residual evaluations.

The sweep kernels never see shape functions or Gauss points: `parent_coefficients` (csrc/pamg_api.cu) folds mass, advection,
diffusion, upwind flux and penalty of a parent into a 3x3 block + 3 neighbour couplings per orientation, a penalty change per
face on the parent boundary and omega/D per face mask.  Here every diagonal block, every coupling to a neighbour child inside
the parent, the total coupling across parent faces and omega/D of every child are compared with the oracle's matrix - for
theta = 1, theta = 1/2 and for the old-time table of get_RHS (theta weight 1 - theta, no mass)."""
import numpy as np
import pytest

import oracle_api as orc
from helpers import random_parent_mesh, rng_field, write_msh
from pamg_pkg import pamg

FACE_NODES = [(0, 2), (2, 1), (1, 0)]        # child faces f1 (1,3), f2 (3,2), f3 (2,1): transport_tri_semi.F90:142-147


def setup(name, n, theta, tmp_path, u=(0.6, -0.3), dt=1e-2, k=0.05):
    mesh = pamg.Mesh.read_msh(write_msh(name, str(tmp_path / (name + ".msh"))))
    op = orc.intended_params(n, 1, dt=dt, k=k, u=u)
    op.theta = theta
    gp = pamg.default_params(n_split=n, multi_levels=1)
    for f in ("face_terms", "literal_source", "transfer", "residual_sign", "halo_rule", "coarse_bc_zero",
              "theta", "dt", "k", "omega", "u_x", "u_y", "source_coef"):
        setattr(gp, f, getattr(op, f))
    return mesh, gp, orc.Semi(op, mesh.X, mesh.neig, mesh.fneig, mesh.dir)


def resid(o, x):
    sh = o.field(orc.TNEW).shape
    o.field(orc.TNEW)[:] = x.reshape(sh); o.field(orc.TNONLIN)[:] = x.reshape(sh); o.field(orc.TOLD)[:] = 0.0
    o.update_overlaps(1)
    o.residual(1)
    return o.field(orc.RES).reshape(-1).copy()


def matrix(o):
    N = int(np.prod(o.field(orc.TNEW).shape))
    b = resid(o, np.zeros(N))
    A = np.zeros((N, N))
    for j in range(N):
        e = np.zeros(N); e[j] = 1.0
        A[:, j] = b - resid(o, e)
    return A, b


def numbering(n):
    C = 4 ** n
    nb = np.zeros((C, 3), np.int32)
    orc.lib().orc_str_neig(n, nb)
    import ctypes
    up = np.zeros(C, bool)
    for e in range(1, C + 1):
        r, p, ori = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        orc.lib().orc_get_str_info(n, e, ctypes.byref(r), ctypes.byref(p), ctypes.byref(ori))
        up[e - 1] = ori.value == 1
    return nb, up


def folded(table, up, mask):
    """3x3 own block, couplings c[3] and omega/D[3] of a child from the 88-entry table."""
    o = 0 if up else 1
    F = table[24 + 16 * o: 24 + 16 * o + 9].reshape(3, 3).copy()
    c = table[24 + 16 * o + 9: 24 + 16 * o + 12].copy()
    for f in range(3):
        if (mask >> f) & 1:
            d = table[56 + f]
            ia, ib = FACE_NODES[f]
            F[ia, ia] += 2 * d; F[ia, ib] += d; F[ib, ia] += d; F[ib, ib] += 2 * d
            c[f] -= d
    return F, c, table[60 + 3 * mask: 60 + 3 * mask + 3]


def check_against_matrix(A, mesh, gp, n, weight, with_mass, wD=None):
    C = 4 ** n
    nb, up = numbering(n)
    scale = np.abs(A).max()
    for u in range(mesh.U):
        t = pamg.parent_table(gp, mesh, u, n, theta_weight=weight, with_mass=with_mass)
        for e in range(C):
            mask = sum(1 << f for f in range(3) if nb[e, f] == 0)
            F, c, w = folded(t, up[e], mask)
            row0 = (u * C + e) * 3
            blk = A[row0:row0 + 3, row0:row0 + 3]
            assert np.abs(blk - F).max() <= 1e-12 * scale, (u, e, mask)
            outside = np.zeros(3)                   # what the rows of this child must hold outside their own parent
            for f in range(3):
                ia, ib = FACE_NODES[f]
                if nb[e, f] != 0:
                    # neighbour child inside the parent: the shared nodes appear reversed on the other side
                    col0 = (u * C + nb[e, f] - 1) * 3
                    want = np.zeros((3, 3))
                    want[ia, ib] = 2 * c[f]; want[ia, ia] = c[f]; want[ib, ib] = c[f]; want[ib, ia] = 2 * c[f]
                    assert np.abs(A[row0:row0 + 3, col0:col0 + 3] - want).max() <= 1e-12 * scale, (u, e, f)
                else:
                    side = (0, 2, 1)[f]             # child face -> gmsh side of the parent
                    if mesh.neig[u, side] != 0:
                        outside[ia] += 3 * c[f]; outside[ib] += 3 * c[f]
            rows = A[row0:row0 + 3]
            got = rows.sum(axis=1) - rows[:, u * C * 3:(u + 1) * C * 3].sum(axis=1)
            assert np.abs(got - outside).max() <= 1e-11 * scale, (u, e, mask)
            if wD is not None:
                assert np.abs(w - wD[row0:row0 + 3]).max() <= 1e-10 * np.abs(w).max(), (u, e, mask)


@pytest.mark.parametrize("name,n", [("test_sn2", 2), ("irregular", 2), ("split0", 3)])
@pytest.mark.parametrize("theta", [1.0, 0.5])
def test_folded_table_equals_the_assembled_operator(name, n, theta, tmp_path):
    mesh, gp, o = setup(name, n, theta, tmp_path)
    A, b = matrix(o)
    # omega / D from one Jacobi sweep: x1 = x0 + (omega / D)(b - A x0)
    sh = o.field(orc.TNEW).shape
    x0 = rng_field(sh, 9).reshape(-1)
    o.field(orc.TNONLIN)[:] = x0.reshape(sh); o.field(orc.TNEW)[:] = x0.reshape(sh); o.field(orc.TOLD)[:] = 0.0
    o.smooth(1, 1, 1)
    wD = (o.field(orc.TNONLIN).reshape(-1) - x0) / (b - A @ x0)
    check_against_matrix(A, mesh, gp, n, theta, True, wD)


def test_old_time_table_is_the_weighted_spatial_operator(tmp_path):
    name, n, theta = "test_sn2", 2, 0.25
    mesh, gp, o1 = setup(name, n, 1.0, tmp_path)
    _, _, o0 = setup(name, n, 0.0, tmp_path)
    A1, _ = matrix(o1)
    A0, _ = matrix(o0)                  # theta = 0: mass / dt only
    check_against_matrix((1.0 - theta) * (A1 - A0), mesh, gp, n, 1.0 - theta, False)


def test_parent_table_argument_errors(tmp_path):
    mesh, gp, _ = setup("test_sn2", 1, 1.0, tmp_path)
    out = np.zeros(88)
    L = pamg.lib()
    import ctypes as C
    assert L.pamg_parent_table(C.byref(gp), mesh.U, mesh.X, mesh.neig, None, mesh.U, 1, 1.0, 1, out) == pamg.ERR_ARG
    assert L.pamg_parent_table(C.byref(gp), mesh.U, mesh.X, mesh.neig, None, -1, 1, 1.0, 1, out) == pamg.ERR_ARG
    assert L.pamg_parent_table(C.byref(gp), mesh.U, mesh.X, mesh.neig, None, 0, 14, 1.0, 1, out) == pamg.ERR_ARG
    # an open boundary face with inflow is refused (the exterior trace would have to follow the interior one)
    kind = np.zeros((mesh.U, 3), np.int32)
    kind[mesh.neig == 0] = 2
    codes = {L.pamg_parent_table(C.byref(gp), mesh.U, mesh.X, mesh.neig, kind.ctypes.data_as(C.c_void_p), u, 1, 1.0, 1, out)
             for u in range(mesh.U)}
    gp.u_x, gp.u_y = 0.7, 0.2
    codes = {L.pamg_parent_table(C.byref(gp), mesh.U, mesh.X, mesh.neig, kind.ctypes.data_as(C.c_void_p), u, 1, 1.0, 1, out)
             for u in range(mesh.U)}
    assert codes == {pamg.OK, pamg.ERR_UNSUPPORTED}


@pytest.mark.parametrize("seed,npts", [(1, 8), (5, 20), pytest.param(2, None, id="permuted-grid-2")])
@pytest.mark.parametrize("theta", [1.0, 0.5])
def test_folded_table_on_random_triangulations_with_mixed_orientation(seed, npts, theta, tmp_path):
    """npts None: the jittered grid with every triangle in a random vertex order (all 18 face pairings)."""
    if npts is None:
        X = random_parent_mesh(seed)
    else:
        from scipy.spatial import Delaunay
        rng = np.random.Generator(np.random.MT19937(seed))
        pts = rng.random((npts, 2))
        simplices = Delaunay(pts).simplices.copy()
        flip = rng.random(len(simplices)) < 0.5
        simplices[flip] = simplices[flip][:, [0, 2, 1]]
        X = pts[simplices]
    mesh = pamg.Mesh.from_arrays(X)
    n = 2
    op = orc.intended_params(n, 1, dt=1e-2, k=0.05, u=(0.6, -0.3))
    op.theta = theta
    gp = pamg.default_params(n_split=n, multi_levels=1)
    for f in ("face_terms", "literal_source", "transfer", "residual_sign", "halo_rule", "coarse_bc_zero",
              "theta", "dt", "k", "omega", "u_x", "u_y", "source_coef"):
        setattr(gp, f, getattr(op, f))
    o = orc.Semi(op, mesh.X, mesh.neig, mesh.fneig, mesh.dir)
    A, _ = matrix(o)
    check_against_matrix(A, mesh, gp, n, theta, True)
