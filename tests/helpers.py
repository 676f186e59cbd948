"""Shared test helpers: golden meshes -> .msh text, numpy synthetic parents, norms."""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

_meshes = None


def golden_meshes():
    global _meshes
    if _meshes is None:
        _meshes = np.load(os.path.join(GOLDEN, "meshes.npz"))
    return _meshes


def write_msh(name, path):
    """Re-emit a golden mesh as gmsh 2.2 ASCII (same node/element tables as the reference file)."""
    z = golden_meshes()
    nodes, elems = z[name + "__nodes"], z[name + "__elems"]
    with open(path, "w") as f:
        f.write("$MeshFormat\n2.2 0 8\n$EndMeshFormat\n$Nodes\n%d\n" % len(nodes))
        for r in nodes:
            f.write("%d %.17g %.17g %.17g\n" % (int(r[0]), r[1], r[2], r[3]))
        f.write("$EndNodes\n$Elements\n%d\n" % len(elems))
        for e in elems:
            f.write(" ".join(str(int(v)) for v in e if v >= 0) + "\n")
        f.write("$EndElements\n")
    return path


def mesh_triangles(name):
    """(X[U,3,2], region[U]) straight from the golden arrays (no neighbour info)."""
    z = golden_meshes()
    nodes, elems = z[name + "__nodes"], z[name + "__elems"]
    xy = {int(r[0]): (r[1], r[2]) for r in nodes}
    X, reg = [], []
    for e in elems:
        if e[1] in (2, 9, 20, 21, 23, 24, 25):
            nt = e[2]
            ids = e[3 + nt: 6 + nt]
            X.append([xy[int(i)] for i in ids])
            reg.append(e[3])
    return np.array(X, np.float64), np.array(reg, np.int32)


def rel_l2(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    d = np.linalg.norm(b)
    return np.linalg.norm(a - b) / (d if d > 0 else 1.0)


def rng_field(shape, seed=20221):
    return np.random.Generator(np.random.MT19937(seed)).random(shape)


def strip_mesh(nsq=15):
    """[0,1] x [0,1/nsq] cut into nsq squares of two right triangles each: the domain of the reference's thermal
    boundary-layer check (Check_thermal_analytical_validation.py probes y = 0.0333 on x in [0,1]; Mesh_files/untitled8192.msh
    is the same strip) with isotropic parents.  Returns X[U,3,2], all counter-clockwise."""
    H = 1.0 / nsq
    X = []
    for i in range(nsq):
        x0, x1 = i * H, (i + 1) * H
        X.append([(x0, 0.0), (x1, 0.0), (x0, H)])
        X.append([(x1, 0.0), (x1, H), (x0, H)])
    return np.array(X, np.float64)


PERMUTATIONS = ((0, 1, 2), (0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1), (2, 1, 0))


def random_parent_triangulation(seed, m=4, jitter=0.3):
    """(pts, simplices, neighbours) of a jittered (m+1) x (m+1) grid on the unit square: interior points moved by up to
    jitter/m in x and y (MT19937(seed)), Delaunay triangles, the vertices of each triangle in a random one of the 6 orders.
    neighbours[:, i] is the triangle opposite vertex i of the reordered simplex (-1: domain boundary), as in Delaunay."""
    from scipy.spatial import Delaunay
    assert 0.0 <= jitter < 0.5
    rng = np.random.Generator(np.random.MT19937(seed))
    g = np.linspace(0.0, 1.0, m + 1)
    pts = np.stack(np.meshgrid(g, g, indexing="ij"), axis=-1).reshape(-1, 2)
    inner = np.all((pts > 0.0) & (pts < 1.0), axis=1)
    pts[inner] += (jitter / m) * (2.0 * rng.random((int(inner.sum()), 2)) - 1.0)
    tri = Delaunay(pts)
    order = np.array(PERMUTATIONS)[rng.integers(0, len(PERMUTATIONS), len(tri.simplices))]
    return pts, np.take_along_axis(tri.simplices, order, axis=1), np.take_along_axis(tri.neighbors, order, axis=1)


def random_parent_mesh(seed, m=4, jitter=0.3):
    """Parents X[U,3,2] of random_parent_triangulation.  The vertex order decides which gmsh side of a parent a face is and
    its orientation, so such a mesh pairs every parent side with every neighbour side in both reversal senses (see
    face_combinations), which meshes built with one orientation rule, or flipped by one fixed swap, never do.  jitter < 1/2
    keeps the triangles well shaped: the minimum angle is asserted to be at least 15 degrees."""
    pts, simplices, _ = random_parent_triangulation(seed, m, jitter)
    X = np.ascontiguousarray(pts[simplices])
    assert min_angle_deg(X) >= 15.0, (seed, min_angle_deg(X))
    return X


def min_angle_deg(X):
    ang = []
    for i in range(3):
        a = X[:, (i + 1) % 3] - X[:, i]
        b = X[:, (i + 2) % 3] - X[:, i]
        c = np.sum(a * b, axis=1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))
        ang.append(np.degrees(np.arccos(np.clip(c, -1.0, 1.0))))
    return float(np.min(ang))


def face_combinations(neig, fneig, dirv):
    """{(s, ns, dir)} over the interior faces: my gmsh side s (1-3), the neighbour's side ns = fNeig (1-3) and the reversal
    flag Dir (0/1) of the face.  These three pick the branch of the halo tables a face takes; there are 18 of them."""
    u, f = np.nonzero(np.asarray(neig) != 0)
    return {(int(f_ + 1), int(fneig[a, f_]), int(dirv[a, f_])) for a, f_ in zip(u, f)}


ALL_FACE_COMBINATIONS = {(s, ns, d) for s in (1, 2, 3) for ns in (1, 2, 3) for d in (0, 1)}


def write_msh_triangles(X, path, region=1):
    """gmsh 2.2 ASCII file of free-standing triangles X[U,3,2] (coincident vertices are merged)."""
    ids, nodes, tris = {}, [], []
    for t in X:
        row = []
        for p in t:
            key = (float(p[0]), float(p[1]))
            if key not in ids:
                ids[key] = len(nodes) + 1
                nodes.append(key)
            row.append(ids[key])
        tris.append(row)
    with open(path, "w") as f:
        f.write("$MeshFormat\n2.2 0 8\n$EndMeshFormat\n$Nodes\n%d\n" % len(nodes))
        for i, (x, y) in enumerate(nodes):
            f.write("%d %.17g %.17g 0\n" % (i + 1, x, y))
        f.write("$EndNodes\n$Elements\n%d\n" % len(tris))
        for i, t in enumerate(tris):
            f.write("%d 2 2 %d %d %d %d %d\n" % (i + 1, region, region, t[0], t[1], t[2]))
        f.write("$EndElements\n")
    return path


def inlet_open_boundary(X, neig):
    """Boundary data of the boundary-layer case: T = 1 on the inlet x = 0 (kind 1), every other domain-boundary face open
    (kind 2: outflow at x = 1, n.u = 0 on the walls).  Sides in gmsh order: 1 = nodes (1,3), 2 = (1,2), 3 = (2,3)."""
    side_nodes = [(0, 2), (0, 1), (1, 2)]
    U = X.shape[0]
    kind = np.zeros((U, 3), np.int32)
    val = np.zeros((U, 3))
    for f, (a, b) in enumerate(side_nodes):
        xm = 0.5 * (X[:, a, 0] + X[:, b, 0])
        bd = neig[:, f] == 0
        inlet = bd & (np.abs(xm) < 1e-12)
        kind[bd, f] = 2
        kind[inlet, f] = 1
        val[inlet, f] = 1.0
    return kind, val


def probe_p1(xy_children, T, points):
    """Value of the discontinuous P1 field at each point: barycentric interpolation inside the first child triangle that
    contains it (what vtkProbeFilter does in Check_thermal_analytical_validation.py:100-140).
    xy_children [N,3,2], T [N,3], points [M,2]."""
    Xf = np.asarray(xy_children, np.float64).reshape(-1, 3, 2)
    Tf = np.asarray(T, np.float64).reshape(-1, 3)
    v0 = Xf[:, 1] - Xf[:, 0]
    v1 = Xf[:, 2] - Xf[:, 0]
    det = v0[:, 0] * v1[:, 1] - v0[:, 1] * v1[:, 0]
    out = np.empty(len(points))
    for i, pt in enumerate(points):
        d = np.asarray(pt) - Xf[:, 0]
        l1 = (d[:, 0] * v1[:, 1] - d[:, 1] * v1[:, 0]) / det
        l2 = (v0[:, 0] * d[:, 1] - v0[:, 1] * d[:, 0]) / det
        ok = np.where((l1 >= -1e-9) & (l2 >= -1e-9) & (l1 + l2 <= 1 + 1e-9))[0]
        e = ok[0]
        out[i] = (1 - l1[e] - l2[e]) * Tf[e, 0] + l1[e] * Tf[e, 1] + l2[e] * Tf[e, 2]
    return out


def child_coordinates(orc, X, n):
    """x_all_str (U, 4^n, 3, 2) from the oracle's get_splitting (Msh2Tri.F90:69-107)."""
    U, C = X.shape[0], 4 ** n
    out = np.zeros((U, C, 3, 2))
    o = np.zeros(6)
    L = orc.lib()
    for u in range(U):
        xu = np.ascontiguousarray(X[u].reshape(-1))
        for e in range(C):
            L.orc_get_splitting(xu, n, e + 1, o)
            out[u, e] = o.reshape(3, 2)
    return out
