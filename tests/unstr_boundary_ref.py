"""numpy reference of the unstructured front-ends with boundary data (pamg_unstr_set_boundary), on top of velocity_field_ref.

On a face with Nside = 0 (a domain-boundary face) the exterior trace at Gauss point s is g_s = sn(s,1) g1 + sn(s,2) g2, g1 / g2
the data at the face nodes (l1, l2), and the exterior velocity is the element's own trace (u_bc = u_ele,
transport_tri_unstr.F90:93).  The face term of the semi-structured path (INTENDED) then splits into the part HEAD already has
(own trace: outflow flux, own penalty part) and the data's part, which moves to the right-hand side:

    inflow Gauss point (income(s) = 1):   -c_s sn(s, .) g_s,   c_s = sdetwei n.u_s
    penalty (k > 0, face not open):       +(k/dx) sdetwei sum_s sn(s, .) g_s

Kinds as in pamg_set_boundary_data: 0 = sin(x+y) at the face nodes, 1 = given values, 2 = open (no data and no penalty term,
so the own penalty part leaves the matrix too)."""
import numpy as np

from velocity_field_ref import FACES, SN, Geometry, _assemble, advection_rhs, implicit_matrix

OPEN = 2


def face_data(X, neig, fneig, kind, value=None):
    """(g [E,3,2] at the face nodes (l1, l2), has [E,3] faces that take data, open [E,3]) from the ABI's kind / value."""
    X = np.asarray(X, np.float64)
    kind = np.asarray(kind)
    data = (np.asarray(neig) == 0) & (np.asarray(fneig) == 0)
    g = np.zeros(kind.shape + (2,))
    for f, (l1, l2) in enumerate(FACES):
        s0 = np.sin(X[:, l1, 0] + X[:, l1, 1]); s1 = np.sin(X[:, l2, 0] + X[:, l2, 1])
        g[:, f, 0] = np.where(kind[:, f] == 0, s0, 0.0)
        g[:, f, 1] = np.where(kind[:, f] == 0, s1, 0.0)
        if value is not None:
            v = np.asarray(value, np.float64)
            g[:, f, 0] = np.where(kind[:, f] == 1, v[:, f, 0], g[:, f, 0])
            g[:, f, 1] = np.where(kind[:, f] == 1, v[:, f, 1], g[:, f, 1])
    op = data & (kind == OPEN)
    g[op] = 0.0
    g[~data] = 0.0
    return g, data & ~op, op


def _dx_boundary(G, f):
    l1, l2 = FACES[f]
    cen = G.X.mean(axis=1)
    return np.linalg.norm(cen - 0.5 * (G.X[:, l1] + G.X[:, l2]), axis=1)


def boundary_rhs(G, u, g, has, open_, k=0.0):
    """g_bc (E, 3): the data's inflow and penalty terms.  Raises ValueError for an open face with an inflow point of non-zero
    flux (what the library refuses)."""
    out = np.zeros((G.E, 3))
    for f, (l1, l2) in enumerate(FACES):
        n = G.normal[:, f]
        for s in range(2):
            a1, a2 = SN[s]
            us, us2 = G.traces(u, f, s)
            inc = G.income(f, us, np.zeros_like(us))          # the exterior velocity is the own trace: sign of n.us
            c = G.sdet[:, f] * np.einsum("ed,ed->e", n, us)
            bad = open_[:, f] & (inc == 1.0) & (c != 0.0)
            if bad.any():
                e = int(np.nonzero(bad)[0][0])
                raise ValueError(f"open boundary face with inflow: element {e}, face {f + 1}")
            gs = a1 * g[:, f, 0] + a2 * g[:, f, 1]
            w = np.where(has[:, f], inc * c * gs, 0.0)
            out[:, l1] -= a1 * w
            out[:, l2] -= a2 * w
            if k != 0.0:
                p = np.where(has[:, f], (k / _dx_boundary(G, f)) * G.sdet[:, f] * gs, 0.0)
                out[:, l1] += a1 * p
                out[:, l2] += a2 * p
    return out


def open_penalty(G, open_, k, sparse=False):
    """The own penalty blocks of the open faces that implicit_matrix contains and the library leaves out: (3E)^2."""
    P = []
    for f, (l1, l2) in enumerate(FACES):
        sn = np.zeros((2, 3))
        for s in range(2):
            sn[s, l1], sn[s, l2] = SN[s]
        kd = (k / _dx_boundary(G, f)) * G.sdet[:, f] if k != 0.0 else np.zeros(G.E)
        P.append(np.where(open_[:, f, None, None], kd[:, None, None] * sum(np.outer(sn[s], sn[s]) for s in range(2)), 0.0))
    ar = np.arange(G.E)
    return _assemble(ar, ar, P[0] + P[1] + P[2], 3 * G.E, sparse)


def uniform(E, u):
    return np.broadcast_to(np.asarray(u, np.float64), (E, 3, 2)).copy()


def implicit_system(X, neig, fneig, u, dt, k=0.0, use_dir=True, kind=None, value=None, sparse=False):
    """(A, M/dt, g_bc [3E]) of the implicit step with boundary data: A T = (M/dt) told + g_bc.  kind = None: HEAD (g_bc = 0)."""
    A, M = implicit_matrix(X, neig, fneig, u, dt, k, use_dir, sparse=sparse)
    G = Geometry(X, neig, fneig, use_dir)
    if kind is None:
        return A, M, np.zeros(3 * G.E)
    g, has, op = face_data(X, neig, fneig, kind, value)
    A = A - open_penalty(G, op, k, sparse)
    return A, M, boundary_rhs(G, np.asarray(u, np.float64), g, has, op, k).reshape(-1)


def explicit_step(X, neig, fneig, u, T, dt, ntime, nits, njac, exact, use_dir, kind=None, value=None, t_bc=0.0):
    """velocity_field_ref.explicit_step with the data's inflow term added to rhs (faces without data keep t_bc)."""
    G = Geometry(X, neig, fneig, use_dir)
    u = np.asarray(u, np.float64)
    T = np.array(T, np.float64)
    area = G.area
    bc = np.zeros((G.E, 3))
    if kind is not None:
        g, has, op = face_data(X, neig, fneig, kind, value)
        bc = boundary_rhs(G, u, g, has, op, 0.0)
    for _ in range(ntime):
        told = T.copy()
        Mo = (area / 12.0)[:, None] * (told + told.sum(axis=1, keepdims=True))
        for _ in range(nits):
            rj = Mo + dt * (advection_rhs(G, u, T, t_bc) + bc)
            if exact:
                T = (12.0 / area)[:, None] * (rj - 0.25 * rj.sum(axis=1, keepdims=True))
            else:
                ml = (area / 3.0)[:, None]
                x = T.copy()
                for _ in range(njac):
                    x = (ml * x - (area / 12.0)[:, None] * (x + x.sum(axis=1, keepdims=True)) + rj) / ml
                T = x
    return T


def implicit_solve(X, neig, fneig, u, T, dt, ntime, k=0.0, use_dir=True, kind=None, value=None):
    """ntime backward-Euler steps A T = (M/dt) told + g_bc, by one sparse LU."""
    from scipy.sparse.linalg import splu
    A, M, b = implicit_system(X, neig, fneig, u, dt, k, use_dir, kind, value, sparse=True)
    lu = splu(A.tocsc())
    T = np.array(T, np.float64).reshape(-1)
    for _ in range(ntime):
        T = lu.solve(M @ T + b)
    return T.reshape(-1, 3)


def face_values(X, fn):
    """bc_value [E,3,2] of a nodal function fn(x, y) at the face nodes (l1, l2)."""
    X = np.asarray(X, np.float64)
    v = np.zeros((X.shape[0], 3, 2))
    for f, (l1, l2) in enumerate(FACES):
        v[:, f, 0] = fn(X[:, l1, 0], X[:, l1, 1]); v[:, f, 1] = fn(X[:, l2, 0], X[:, l2, 1])
    return v
