"""Flow levels of the upwind graph (pamg_flow_levels, host code of libpamg_cuda.so: no GPU needed), the order of the
flow-ordered block Gauss-Seidel preconditioner of the implicit solve.

The inflow masks here are an independent numpy restatement of the uniform-velocity upwind rule: the sign of n.u on every face,
with n the outward normal found from the coordinates (away from the centroid); a face with n.u = 0 (axis-aligned velocities on
the synthetic meshes) is not inflow.  Acyclic graphs must come out with nothing lagged and the levels of a plain longest-path
search; cyclic masks must follow the documented lowest-index rule."""
import numpy as np
import pytest

from helpers import write_msh
from pamg_pkg import pamg

FACES = [(0, 2), (1, 0), (2, 1)]          # gmsh face f of the unstructured path: nodes (l1, l2)
NAMES = ["untitled8192", "irregular", "split1", "900_ele"]
DIRECTIONS = [(0.9, 0.3), (-0.35, 0.8), (1.0, 0.0), (0.0, -1.0), (-1.0, -1.0)]


@pytest.fixture(scope="module")
def meshes(tmp_path_factory):
    d = tmp_path_factory.mktemp("msh")
    out = {name: pamg.Mesh.read_msh(write_msh(name, str(d / (name + ".msh")))) for name in NAMES}
    for kp in (3, 5):
        out[f"synthetic{kp}"] = pamg.Mesh.synthetic(kp, 1)
    return out


def uniform_mask(mesh, u):
    """bit f of element e: face f has a neighbour and n.u < 0 there (n = outward normal from the coordinates)"""
    X = mesh.X
    cen = X.mean(axis=1)
    mask = np.zeros(mesh.U, np.int32)
    for f, (l1, l2) in enumerate(FACES):
        ex, ey = X[:, l2, 0] - X[:, l1, 0], X[:, l2, 1] - X[:, l1, 1]
        nx, ny = ey, -ex
        mx, my = 0.5 * (X[:, l1, 0] + X[:, l2, 0]) - cen[:, 0], 0.5 * (X[:, l1, 1] + X[:, l2, 1]) - cen[:, 1]
        flip = nx * mx + ny * my < 0.0
        nx, ny = np.where(flip, -nx, nx), np.where(flip, -ny, ny)
        inflow = (nx * u[0] + ny * u[1] < 0.0) & (mesh.neig[:, f] != 0)
        mask |= inflow.astype(np.int32) << f
    return mask


def edges(neig, mask):
    """upwind edges (c, e), 0-based"""
    out = []
    for e in range(len(mask)):
        for f in range(3):
            if (mask[e] >> f) & 1 and neig[e, f] != 0:
                out.append((int(neig[e, f]) - 1, e))
    return out


def longest_path(E, E_list):
    """plain-Python longest upwind path ending at every element (iterative depth-first search, acyclic graphs only)"""
    preds = [[] for _ in range(E)]
    for c, e in E_list:
        preds[e].append(c)
    level = [None] * E
    for s in range(E):
        stack = [s]
        while stack:
            e = stack[-1]
            if level[e] is not None:
                stack.pop()
                continue
            todo = [c for c in preds[e] if level[c] is None]
            if todo:
                stack.extend(todo)
            else:
                level[e] = 1 + max((level[c] for c in preds[e]), default=-1)
                stack.pop()
    return np.array(level, np.int32)


def check_common(neig, mask, level, order, nlevels, lagged):
    E = len(mask)
    assert sorted(order.tolist()) == list(range(E))
    assert np.all(level >= 0) and nlevels == level.max() + 1
    keys = [(int(level[e]), int(e)) for e in order]
    assert keys == sorted(keys)                                  # order sorted by (level, index)
    ed = edges(neig, mask)
    assert lagged == sum(1 for c, e in ed if level[c] >= level[e])
    again = pamg.flow_levels(neig, mask)
    assert np.array_equal(again[0], level) and np.array_equal(again[1], order) and again[2:] == (nlevels, lagged)


def test_face_numbering_of_the_restatement(meshes):
    """the neighbour across face f shares the face's two nodes (the mask above is per gmsh face)"""
    for mesh in meshes.values():
        X = mesh.X
        for f, (l1, l2) in enumerate(FACES):
            has = mesh.neig[:, f] != 0
            q = mesh.neig[has, f] - 1
            for li in (l1, l2):
                d = np.abs(X[q][:, :, None, :] - X[has][:, None, li, :][:, :, None, :]).sum(axis=3).min(axis=1)
                assert np.all(d.min(axis=1) == 0.0)


@pytest.mark.parametrize("u", DIRECTIONS)
def test_uniform_velocity_is_acyclic(meshes, u):
    for name, mesh in meshes.items():
        mask = uniform_mask(mesh, u)
        level, order, nlevels, lagged = pamg.flow_levels(mesh.neig, mask)
        assert lagged == 0, name
        ed = edges(mesh.neig, mask)
        assert all(level[c] < level[e] for c, e in ed), name     # every inflow edge goes upward
        assert np.array_equal(level, longest_path(mesh.U, ed)), name
        check_common(mesh.neig, mask, level, order, nlevels, lagged)


def test_axis_aligned_velocity_leaves_tangential_faces_out(meshes):
    """on the synthetic meshes a horizontal velocity is tangential to the horizontal faces: fewer edges than faces with a
    neighbour, and still no cycle"""
    mesh = meshes["synthetic5"]
    mask = uniform_mask(mesh, (1.0, 0.0))
    inner_faces = int((mesh.neig != 0).sum())
    assert 0 < len(edges(mesh.neig, mask)) < inner_faces // 2
    assert pamg.flow_levels(mesh.neig, mask)[3] == 0


def ring(n, pairs):
    """n elements, face 0 of element e looks at pairs[e] (1-based, 0 = none), every face bit set where a neighbour exists"""
    neig = np.zeros((n, 3), np.int32)
    for e, q in enumerate(pairs):
        neig[e, 0] = q
    mask = (neig[:, 0] != 0).astype(np.int32)
    return neig, mask


def test_two_cycle():
    neig, mask = ring(2, [2, 1])                 # 0 <- 1 and 1 <- 0
    level, order, nlevels, lagged = pamg.flow_levels(neig, mask)
    # the lowest index (0) is taken first, with no levelled upstream neighbour: level 0; 1 follows it
    assert level.tolist() == [0, 1] and order.tolist() == [0, 1] and nlevels == 2 and lagged == 1
    check_common(neig, mask, level, order, nlevels, lagged)


def test_three_cycle_with_a_tail():
    # 3 -> 0 -> 1 -> 2 -> 0 (element e depends on pairs[e]); element 4 depends on 2
    neig = np.zeros((5, 3), np.int32)
    neig[0, 0], neig[0, 1] = 3, 4                 # 0 <- 2 and 0 <- 3
    neig[1, 0] = 1                               # 1 <- 0
    neig[2, 0] = 2                               # 2 <- 1
    neig[4, 2] = 3                               # 4 <- 2
    mask = np.array([3, 1, 1, 0, 4], np.int32)
    level, order, nlevels, lagged = pamg.flow_levels(neig, mask)
    # queue: 3 (no inflow) -> level 0; then stuck: lowest left is 0, levelled upstream {3}: level 1; 1: 2; 2: 3; 4: 4
    assert level.tolist() == [1, 2, 3, 0, 4] and order.tolist() == [3, 0, 1, 2, 4]
    assert nlevels == 5 and lagged == 1           # the edge 2 -> 0
    check_common(neig, mask, level, order, nlevels, lagged)


def rotating_mask(mesh):
    """a rotating velocity, with the upwind choice taken per face from the velocity at the face midpoint"""
    X = mesh.X
    c = X.reshape(-1, 2).mean(axis=0)
    cen = X.mean(axis=1)
    mask = np.zeros(mesh.U, np.int32)
    for f, (l1, l2) in enumerate(FACES):
        mid = 0.5 * (X[:, l1] + X[:, l2])
        ux, uy = -(mid[:, 1] - c[1]), mid[:, 0] - c[0]
        ex, ey = X[:, l2, 0] - X[:, l1, 0], X[:, l2, 1] - X[:, l1, 1]
        s = np.sign(ey * (mid[:, 0] - cen[:, 0]) - ex * (mid[:, 1] - cen[:, 1]))
        mask |= ((s * (ey * ux - ex * uy) < 0.0) & (mesh.neig[:, f] != 0)).astype(np.int32) << f
    return mask


@pytest.mark.parametrize("name", ["irregular", "synthetic5"])
def test_rotating_field_has_cycles(meshes, name):
    mesh = meshes[name]
    mask = rotating_mask(mesh)
    level, order, nlevels, lagged = pamg.flow_levels(mesh.neig, mask)
    assert lagged > 0
    check_common(mesh.neig, mask, level, order, nlevels, lagged)


def test_bad_arguments():
    neig = np.zeros((2, 3), np.int32)
    neig[0, 0] = 3                               # no element 3
    with pytest.raises(pamg.PamgError):
        pamg.flow_levels(neig, np.ones(2, np.int32))
    with pytest.raises(ValueError):
        pamg.flow_levels(np.zeros((3, 3), np.int32), np.zeros(2, np.int32))
