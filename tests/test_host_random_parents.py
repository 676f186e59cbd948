"""The random parent meshes of helpers.random_parent_mesh (jittered grid, Delaunay, every triangle in a random one of the 6
vertex orders) - CPU only.

Which branch of the halo tables and of the in-kernel face conventions a parent face takes depends on my gmsh side s, the
neighbour's side ns (fNeig) and the reversal flag Dir: 18 combinations.  The shipped meshes hold at most 11 of them and meshes
flipped by one fixed swap never pair side 3 with side 3.  The GPU parity tests on these meshes (test_gpu_random_parents.py)
are only as good as the cases the mesh contains, so the coverage is asserted here, where a change of the generator that loses
a case fails instead of quietly shrinking the matrix."""
import numpy as np
import pytest

import oracle_api as orc
from helpers import ALL_FACE_COMBINATIONS, face_combinations, min_angle_deg, random_parent_mesh, write_msh_triangles
from pamg_pkg import pamg

SEEDS = [2, 3]


@pytest.mark.parametrize("seed", SEEDS)
def test_random_parent_mesh_holds_every_face_pairing(seed):
    X = random_parent_mesh(seed)
    assert X.shape == (32, 3, 2)
    assert min_angle_deg(X) >= 15.0
    m = pamg.Mesh.from_arrays(X)
    assert face_combinations(m.neig, m.fneig, m.dir) == ALL_FACE_COMBINATIONS
    # both orientations, each a fair share of the parents
    det = ((X[:, 1, 0] - X[:, 0, 0]) * (X[:, 2, 1] - X[:, 0, 1]) - (X[:, 1, 1] - X[:, 0, 1]) * (X[:, 2, 0] - X[:, 0, 0]))
    assert np.all(np.abs(det) > 0)
    ccw = int((det > 0).sum())
    assert 8 <= ccw <= 24, ccw
    # domain-boundary faces (Dirichlet strips) on every gmsh side
    assert {int(f) + 1 for f in np.nonzero(m.neig == 0)[1]} == {1, 2, 3}
    assert int((m.neig == 0).sum()) == 16                    # the 4 x 4 boundary edges of the unit square


@pytest.mark.parametrize("seed", SEEDS)
def test_product_neighbours_equal_the_reference_reader(seed, tmp_path):
    """Mesh.from_arrays (edge hash) == ReadMSH + CheckNeig + getNeigDataMesh as the oracle restates them, on the same file."""
    X = random_parent_mesh(seed)
    m = pamg.Mesh.from_arrays(X)
    o = orc.read_msh(write_msh_triangles(X, str(tmp_path / "rnd.msh")))
    fneig, _ = orc.neig_data(o["neig"], o["dir"])
    assert np.array_equal(o["X"], m.X)
    assert np.array_equal(o["neig"], m.neig)
    assert np.array_equal(o["dir"], m.dir)
    assert np.array_equal(fneig, m.fneig)
    # and the combinations the oracle sees are the same 18
    assert face_combinations(o["neig"], fneig, o["dir"]) == ALL_FACE_COMBINATIONS


def test_generator_is_deterministic_and_rejects_large_jitter():
    assert np.array_equal(random_parent_mesh(2), random_parent_mesh(2))
    assert not np.array_equal(random_parent_mesh(2), random_parent_mesh(3))
    with pytest.raises(AssertionError):
        random_parent_mesh(2, jitter=0.5)
