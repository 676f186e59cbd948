"""The host mesh pipeline of the product (O(N) edge hash, csrc/pamg_mesh.cpp; replaces CheckNeig's all-pairs search and
getNeigDataMesh, Msh2Tri.F90:132-334,454-548,780-963) on RANDOM triangulations against scipy's Delaunay neighbour table and
against the oracle's restatement of the reference search - CPU only.

gmsh side s of a triangle holds the nodes SIDE_NODES[s] = (1,3), (1,2), (2,3) (Msh2Tri.F90:877-901), i.e. it lies opposite
vertex 2, 3, 1; Delaunay.neighbors[:, i] is the neighbour opposite vertex i."""
import numpy as np
import pytest
from scipy.spatial import Delaunay

import oracle_api as orc
from helpers import random_parent_triangulation, write_msh_triangles
from pamg_pkg import pamg

OPPOSITE = [1, 2, 0]                     # gmsh side 1, 2, 3 -> the vertex (0-based) it lies opposite
SIDE_NODES = [(0, 2), (0, 1), (1, 2)]


def triangulation(seed, npts):
    """(pts, simplices, neighbours): npts random points with half the triangles flipped, or (npts None) the permuted jittered
    grid of helpers.random_parent_triangulation, which pairs every gmsh side with every other in both reversal senses."""
    if npts is None:
        return random_parent_triangulation(seed)
    rng = np.random.Generator(np.random.MT19937(seed))
    pts = rng.random((npts, 2))
    tri = Delaunay(pts)
    simplices = tri.simplices.copy()
    flip = rng.random(len(simplices)) < 0.5          # mixed orientation, like the shipped meshes
    simplices[flip] = simplices[flip][:, [0, 2, 1]]
    nbrs = tri.neighbors.copy()
    nbrs[flip] = nbrs[flip][:, [0, 2, 1]]
    return pts, simplices, nbrs


@pytest.mark.parametrize("seed,npts", [(1, 12), (2, 40), (3, 150), (4, 600), pytest.param(2, None, id="permuted-grid-2")])
def test_edge_hash_neighbours_equal_delaunay_and_the_reference_search(seed, npts, tmp_path):
    pts, simplices, nbrs = triangulation(seed, npts)
    X = pts[simplices]
    m = pamg.Mesh.from_arrays(X)
    U = len(simplices)
    assert m.U == U
    for s in range(3):
        assert np.array_equal(m.neig[:, s], nbrs[:, OPPOSITE[s]] + 1)          # 1-based, 0 = domain boundary (Delaunay: -1)
    # fNeig: the side of the neighbour that carries the shared edge
    for u in range(U):
        for s in range(3):
            q = m.neig[u, s]
            if q == 0:
                continue
            ns = m.fneig[u, s] - 1
            mine = {tuple(X[u, i]) for i in SIDE_NODES[s]}
            theirs = {tuple(X[q - 1, i]) for i in SIDE_NODES[ns]}
            assert mine == theirs and m.neig[q - 1, ns] == u + 1
    # the oracle's restatement of ReadMSH + CheckNeig (all pairs) on the same triangles
    if U <= 400:
        o = orc.read_msh(write_msh_triangles(X, str(tmp_path / "rnd.msh")))
        assert np.array_equal(o["X"], m.X) and np.array_equal(o["neig"], m.neig) and np.array_equal(o["dir"], m.dir)
        fneig, _ = orc.neig_data(o["neig"], o["dir"])
        assert np.array_equal(fneig, m.fneig)
