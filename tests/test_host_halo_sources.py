"""Where the sweeps take the exterior values of parent faces from - halo strip entries (hmap) or, strip-free, the neighbour
parent's field (nsrc, decoded by the function the kernels use, behind pamg_halo_sources) - checked on the CPU with a globally
CONTINUOUS nodal field: the exterior value at the node coincident with my face node must equal my own value there.
Independent of both implementations: it only uses that shared nodes have the same coordinates (update_overlaps,
splitting.F90:1255-1391, and the face block's pick of the neighbour trace, transport_tri_semi.F90:629-655)."""
import numpy as np
import pytest

import oracle_api as orc
from helpers import child_coordinates, random_parent_mesh, write_msh
from pamg_pkg import pamg

SIDE_FACE_NODES = [(0, 2), (1, 0), (2, 1)]      # parent gmsh side 1, 2, 3 = child face f1 (1,3), f3 (2,1), f2 (3,2)


def continuous_field(xy):
    x, y = xy[..., 0], xy[..., 1]
    return np.sin(3.0 * x) + np.cos(2.0 * y) + x * y + 0.25


@pytest.mark.parametrize("name", ["test_sn2", "split1", "irregular", "900_ele"])
@pytest.mark.parametrize("rule", [0, 1])
@pytest.mark.parametrize("n", [1, 3])
def test_exterior_values_are_the_neighbours_values_at_the_coincident_nodes(name, rule, n, tmp_path):
    m = pamg.Mesh.read_msh(write_msh(name, str(tmp_path / (name + ".msh"))))
    S = 2 ** n
    T = continuous_field(child_coordinates(orc, m.X, n))                 # (U, C, 3)
    flat = T.reshape(-1)
    surf = np.zeros(3 * S, np.int32)
    orc.lib().orc_surf_ele(n, surf)
    surf = surf.reshape(3, S)
    # the strips as the reference fills them
    p = orc.intended_params(n, 1)
    p.halo_rule = rule
    s = orc.Semi(p, m.X, m.neig, m.fneig, m.dir)
    s.field(orc.TNEW, 1)[:] = T
    s.update_overlaps(1)
    ovl = s.overlap(1)                                                   # (U, 3, S, 3)
    plan = pamg.halo_plan(m, halo_rule=rule)
    src = pamg.halo_sources(m, n, halo_rule=rule)
    hmap = plan["hmap"].reshape(m.U, 3)
    checked = 0
    for u in range(m.U):
        for mf in range(3):
            if m.neig[u, mf] == 0:
                assert np.all(src[u, mf] == -1)                          # Dirichlet data lives in the strip
                continue
            a, b = SIDE_FACE_NODES[mf]
            own = T[u, surf[mf] - 1]                                     # (S, 3): my boundary children along this side
            hm = int(hmap[u, mf])
            # through the strip: entries (hm & 3, hm >> 2) of position p
            assert np.abs(ovl[u, mf, :, hm & 3] - own[:, a]).max() <= 1e-12
            assert np.abs(ovl[u, mf, :, hm >> 2] - own[:, b]).max() <= 1e-12
            # strip-free: straight from the neighbour parent's field
            assert np.all(src[u, mf] >= 0)
            assert np.abs(flat[src[u, mf, :, 0]] - own[:, a]).max() <= 1e-12
            assert np.abs(flat[src[u, mf, :, 1]] - own[:, b]).max() <= 1e-12
            # ... and bit for bit what update_overlaps copied
            assert np.array_equal(flat[src[u, mf, :, 0]], ovl[u, mf, :, hm & 3])
            assert np.array_equal(flat[src[u, mf, :, 1]], ovl[u, mf, :, hm >> 2])
            checked += 1
    assert checked == int((m.neig != 0).sum())


def test_cut_faces_of_a_partition_keep_their_strips():
    m = pamg.Mesh.synthetic(2, 2)
    pf = np.array([0, 10, 32], np.int32)
    n = 2
    for part in (0, 1):
        src = pamg.halo_sources(m, n, nparts=2, part_first=pf, my_part=part)
        first, last = pf[part], pf[part + 1]
        for u in range(first, last):
            for mf in range(3):
                q = m.neig[u, mf]
                local = q != 0 and first <= q - 1 < last
                assert np.all(src[u - first, mf] >= 0) == local and (local or np.all(src[u - first, mf] == -1))
                if local:                                                 # offsets are relative to the part's own field
                    assert src[u - first, mf].max() < (last - first) * 4 ** n * 3


def random_triangles(seed, npts):
    """X[U,3,2]: npts random points with half the triangles flipped by one swap, or (npts None) the jittered grid with every
    triangle in a random vertex order, which holds all 18 (side, neighbour side, Dir) pairings (helpers.random_parent_mesh)."""
    if npts is None:
        return random_parent_mesh(seed)
    from scipy.spatial import Delaunay
    rng = np.random.Generator(np.random.MT19937(seed))
    pts = rng.random((npts, 2))
    simplices = Delaunay(pts).simplices.copy()
    flip = rng.random(len(simplices)) < 0.5
    simplices[flip] = simplices[flip][:, [0, 2, 1]]
    return pts[simplices]


@pytest.mark.parametrize("seed,npts", [(2, 14), (7, 60), pytest.param(2, None, id="permuted-grid-2")])
@pytest.mark.parametrize("rule", [0, 1])
def test_exterior_values_on_random_triangulations_with_mixed_orientation(seed, npts, rule):
    m = pamg.Mesh.from_arrays(random_triangles(seed, npts))
    n = 2
    S = 2 ** n
    T = continuous_field(child_coordinates(orc, m.X, n))
    flat = T.reshape(-1)
    surf = np.zeros(3 * S, np.int32)
    orc.lib().orc_surf_ele(n, surf)
    surf = surf.reshape(3, S)
    src = pamg.halo_sources(m, n, halo_rule=rule)
    # the strips as the reference fills them (its reversal table under halo_rule 0, geometry under 1)
    p = orc.intended_params(n, 1)
    p.halo_rule = rule
    s = orc.Semi(p, m.X, m.neig, m.fneig, m.dir)
    s.field(orc.TNEW, 1)[:] = T
    s.update_overlaps(1)
    ovl = s.overlap(1)
    hmap = pamg.halo_plan(m, halo_rule=rule)["hmap"].reshape(m.U, 3)
    for u in range(m.U):
        for mf in range(3):
            if m.neig[u, mf] == 0:
                continue
            a, b = SIDE_FACE_NODES[mf]
            own = T[u, surf[mf] - 1]
            assert np.abs(flat[src[u, mf, :, 0]] - own[:, a]).max() <= 1e-12
            assert np.abs(flat[src[u, mf, :, 1]] - own[:, b]).max() <= 1e-12
            hm = int(hmap[u, mf])
            assert np.array_equal(flat[src[u, mf, :, 0]], ovl[u, mf, :, hm & 3])
            assert np.array_equal(flat[src[u, mf, :, 1]], ovl[u, mf, :, hm >> 2])
