"""numpy restatement of the unstructured front-ends with a nodal velocity field u_ele(2,3,E) (transport_tri_unstr.F90:105,
131-134,227,303): the reference's Gauss-point form, vectorised over elements.

    volume   ugi(g) = sum_i n(g,i) u(:,i)  at the three edge midpoints;  rhs_i += sum_g (grad phi_i . ugi(g)) T(g) detwei(g)
    face s   us = sum_q sn(s,q) u(:,q,e),  us2 = sum_q sn2(s,q) u(:,q,npos)  (0 where Nside = 0, us where npos = 0)
             income(s) = 1/2 + 1/2 sign(1, -n.(us + us2)/2)
             flux_i = sum_s sn(s,i) sdet n.((1 - income) us T_s + income us2 T2_s)

u has shape (E, 3, 2) = (element, node, component).  Independent of the library and of the C++ oracle: it is what both are
compared with where the oracle has no field entries."""
import numpy as np

AL, BE = 0.78867513459481288, 0.21132486540518712
SN = ((AL, BE), (BE, AL))                       # sn(s, (l1, l2)) of the two face Gauss points
FACES = ((0, 2), (1, 0), (2, 1))                # gmsh faces (1,3), (2,1), (3,2), 0-based local nodes
GAUSS = ((0, 1), (1, 2), (0, 2))                # nodes with n(g, .) = 1/2 at the volume Gauss points
# get_unstr_sn2: Nside 1 -> neighbour nodes (3,1), 2 -> (1,2), 3 -> (2,3) paired with (l1, l2)


class Geometry:
    """Per-element gradients, areas, face normals and the neighbour node pairing (get_unstr_sn2, or by geometry with use_dir)."""

    def __init__(self, X, neig, fneig, use_dir):
        X = np.asarray(X, np.float64)
        self.X, self.neig, self.fneig = X, np.asarray(neig), np.asarray(fneig)
        E = X.shape[0]
        self.E = E
        x, y = X[:, :, 0], X[:, :, 1]
        det = (x[:, 0] - x[:, 2]) * (y[:, 1] - y[:, 2]) - (y[:, 0] - y[:, 2]) * (x[:, 1] - x[:, 2])
        self.area = 0.5 * np.abs(det)
        # grad phi_i = (y_j - y_k, x_k - x_j) / det over the cyclic (i, j, k)
        self.grad = np.zeros((E, 3, 2))
        for i in range(3):
            j, k = (i + 1) % 3, (i + 2) % 3
            self.grad[:, i, 0] = (y[:, j] - y[:, k]) / det
            self.grad[:, i, 1] = (x[:, k] - x[:, j]) / det
        cen = X.mean(axis=1)
        self.normal = np.zeros((E, 3, 2)); self.sdet = np.zeros((E, 3))
        self.m = np.zeros((E, 3, 2), np.int64)
        for f, (l1, l2) in enumerate(FACES):
            ev = X[:, l2] - X[:, l1]
            L = np.hypot(ev[:, 0], ev[:, 1])
            nrm = np.stack([ev[:, 1], -ev[:, 0]], axis=1) / L[:, None]
            mid = 0.5 * (X[:, l1] + X[:, l2])
            flip = np.einsum("ed,ed->e", nrm, mid - cen) < 0
            nrm[flip] *= -1.0
            self.normal[:, f] = nrm
            self.sdet[:, f] = 0.5 * L
            ns, q = self.fneig[:, f], self.neig[:, f]
            m1 = np.array([0, 2, 0, 1])[ns]; m2 = np.array([0, 0, 1, 2])[ns]
            if use_dir:
                d = X[np.maximum(q - 1, 0), m1] - X[:, l1]
                sw = (q != 0) & (ns >= 1) & (np.hypot(d[:, 0], d[:, 1]) >= 2.220446049250313e-16)
                m1, m2 = np.where(sw, m2, m1), np.where(sw, m1, m2)
            self.m[:, f, 0], self.m[:, f, 1] = m1, m2

    def traces(self, u, f, s, T=None, t_bc=0.0):
        """(us, us2, T_s, T2_s) at Gauss point s of face f of every element; T2_s = sn2 . T2 with T2 = t_bc where npos = 0."""
        l1, l2 = FACES[f]
        a1, a2 = SN[s]
        q, ns = self.neig[:, f], self.fneig[:, f]
        nb = np.maximum(q - 1, 0)
        ar = np.arange(self.E)
        m1, m2 = self.m[:, f, 0], self.m[:, f, 1]
        us = a1 * u[:, l1] + a2 * u[:, l2]
        us2 = a1 * u[nb, m1] + a2 * u[nb, m2]
        us2 = np.where((q == 0)[:, None], us, us2)
        us2 = np.where((ns == 0)[:, None], 0.0, us2)
        if T is None:
            return us, us2
        ts = a1 * T[ar, l1] + a2 * T[ar, l2]
        t2 = np.where(q != 0, a1 * T[nb, m1] + a2 * T[nb, m2], (a1 + a2) * t_bc)
        t2 = np.where(ns == 0, 0.0, t2)
        return us, us2, ts, t2

    def income(self, f, us, us2):
        un = np.einsum("ed,ed->e", self.normal[:, f], 0.5 * (us + us2))
        return 0.5 + 0.5 * np.copysign(1.0, -un)


def advection_rhs(G, u, T, t_bc):
    """rhs of unstr_explicit (:668-746) with the field: volume term minus the upwind face flux, (E, 3)."""
    rhs = np.zeros((G.E, 3))
    for (i0, i1) in GAUSS:
        ug = 0.5 * (u[:, i0] + u[:, i1])
        tg = 0.5 * (T[:, i0] + T[:, i1])
        rhs += np.einsum("eid,ed->ei", G.grad, ug) * (tg * G.area / 3.0)[:, None]
    for f, (l1, l2) in enumerate(FACES):
        for s in range(2):
            us, us2, ts, t2 = G.traces(u, f, s, T, t_bc)
            inc = G.income(f, us, us2)
            n = G.normal[:, f]
            fl = G.sdet[:, f] * ((1.0 - inc) * np.einsum("ed,ed->e", n, us) * ts + inc * np.einsum("ed,ed->e", n, us2) * t2)
            rhs[:, l1] -= SN[s][0] * fl
            rhs[:, l2] -= SN[s][1] * fl
    return rhs


def explicit_step(X, neig, fneig, u, T, dt, ntime, nits, njac, exact, use_dir, t_bc=0.0):
    """Time loop of unstr_explicit (:588-795): told = T ; nits x { T = M^-1 (M told + dt rhs(T)) or njac Jacobi iterations on
    the lumped mass started from T }."""
    G = Geometry(X, neig, fneig, use_dir)
    u = np.asarray(u, np.float64)
    T = np.array(T, np.float64)
    area = G.area
    for _ in range(ntime):
        told = T.copy()
        Mo = (area / 12.0)[:, None] * (told + told.sum(axis=1, keepdims=True))
        for _ in range(nits):
            rj = Mo + dt * advection_rhs(G, u, T, t_bc)
            if exact:                                                       # M^-1 = (12/A)(I - J/4)
                T = (12.0 / area)[:, None] * (rj - 0.25 * rj.sum(axis=1, keepdims=True))
            else:
                ml = (area / 3.0)[:, None]
                x = T.copy()
                for _ in range(njac):
                    x = (ml * x - (area / 12.0)[:, None] * (x + x.sum(axis=1, keepdims=True)) + rj) / ml
                T = x
    return T


def implicit_matrix(X, neig, fneig, u, dt, k=0.0, use_dir=True, literal=False, sparse=False):
    """(3E)^2 lhs + flux (dense, or scipy CSR with sparse=True) of unstr_implicit (:270-364) with the field, and M/dt.  literal=False: every face Gauss point
    puts its sn(s,j) part into the own columns (outflow) or its sn2(s,j) part into the neighbour's (inflow).  literal=True:
    HEAD's rule (:339-342), the whole face block into ONE target chosen by income(1), the neighbour's columns read with the
    own-element and the neighbour's local numbering mixed as the reference does."""
    G = Geometry(X, neig, fneig, use_dir)
    u = np.asarray(u, np.float64)
    E = G.E
    ar = np.arange(E)
    cen = G.X.mean(axis=1)
    Mloc = (np.ones((3, 3)) + np.eye(3)) / 12.0
    m = G.area[:, None, None] * Mloc / dt
    stiff = np.zeros((E, 3, 3))
    for g, (i0, i1) in enumerate(GAUSS):
        ug = 0.5 * (u[:, i0] + u[:, i1])
        ng = np.zeros(3); ng[i0] = ng[i1] = 0.5
        stiff += np.einsum("ei,j->eij", np.einsum("eid,ed->ei", G.grad, ug), ng) * G.area[:, None, None] / 3.0
    diag = m - stiff + (k * G.area[:, None, None] * G.grad) @ G.grad.transpose(0, 2, 1)
    off = np.zeros((3, E, 3, 3))                                     # block (e, neig[e, f] - 1) of face f
    for f, (l1, l2) in enumerate(FACES):
        q, ns = G.neig[:, f], G.fneig[:, f]
        inner = q != 0
        m1, m2 = G.m[:, f, 0], G.m[:, f, 1]
        sn = np.zeros((2, 3)); sn2 = np.zeros((E, 2, 3))
        has = ar[ns >= 1]
        for s in range(2):
            sn[s, l1], sn[s, l2] = SN[s]
            sn2[has, s, m1[has]], sn2[has, s, m2[has]] = SN[s]
        n = G.normal[:, f]
        own = np.zeros((E, 3, 3)); nbr = np.zeros((E, 3, 3))
        for s in range(2):
            us, us2 = G.traces(u, f, s)
            inc = G.income(f, us, us2)
            c = G.sdet[:, f] * np.einsum("ed,ed->e", n, us); c2 = G.sdet[:, f] * np.einsum("ed,ed->e", n, us2)
            own += ((1.0 - inc) * c)[:, None, None] * np.outer(sn[s], sn[s])
            nbr += (inc * c2)[:, None, None] * np.einsum("i,ej->eij", sn[s], sn2[:, s])
            if s == 0:
                to_own = (inc == 0.0) | ~inner                       # literal: the target of the whole face block
        if literal:
            diag[to_own] += (own + nbr)[to_own]
            off[f, ~to_own] += (own + nbr)[~to_own]
        else:
            diag += own
            diag[~inner] += nbr[~inner]
            off[f, inner] += nbr[inner]
        if k != 0.0:
            nb = np.maximum(q - 1, 0)
            dx = np.where(inner, np.linalg.norm(cen - cen[nb], axis=1),
                          np.linalg.norm(cen - 0.5 * (G.X[:, l1] + G.X[:, l2]), axis=1))
            kd = (k / dx) * G.sdet[:, f]
            diag += kd[:, None, None] * sum(np.outer(sn[s], sn[s]) for s in range(2))
            pen = -kd[:, None, None] * sum(np.einsum("i,ej->eij", sn[s], sn2[:, s]) for s in range(2))
            off[f, inner] += pen[inner]
    re = [ar] + [ar[G.neig[:, f] != 0] for f in range(3)]
    ce = [ar] + [G.neig[G.neig[:, f] != 0, f] - 1 for f in range(3)]
    vb = [diag] + [off[f, G.neig[:, f] != 0] for f in range(3)]
    N = 3 * E
    return _assemble(np.concatenate(re), np.concatenate(ce), np.concatenate(vb), N, sparse), _assemble(ar, ar, m, N, sparse)


def _assemble(re, ce, v, N, sparse):
    """(3E)^2 matrix, dense or scipy CSR, of the 3x3 blocks v[i] at block (re[i], ce[i]); repeated blocks add up."""
    r = np.broadcast_to((3 * re)[:, None, None] + np.arange(3)[None, :, None], v.shape).ravel()
    c = np.broadcast_to((3 * ce)[:, None, None] + np.arange(3)[None, None, :], v.shape).ravel()
    if not sparse:
        A = np.zeros((N, N))
        np.add.at(A, (r, c), v.ravel())
        return A
    import scipy.sparse as sp
    return sp.csr_matrix((v.ravel(), (r, c)), shape=(N, N))


def stab(X, u, tnew, told, dt):
    """Petrov-Galerkin diff_coe (E,3) and stab (E,3,3) (:239-267,278) with ugi(g) from the field."""
    X = np.asarray(X, np.float64)
    toler = 1e-11
    x, y = X[:, :, 0], X[:, :, 1]
    A, B, C, D = x[:, 0] - x[:, 2], y[:, 0] - y[:, 2], x[:, 1] - x[:, 2], y[:, 1] - y[:, 2]
    detj = A * D - B * C
    ij = np.stack([np.stack([D / detj, -C / detj], 1), np.stack([-B / detj, A / detj], 1)], 1)   # inv_jac (E,2,2)
    nlx = np.array([[1.0, 0.0, -1.0], [0.0, 1.0, -1.0]])
    grad = np.einsum("ebd,bl->eld", ij, nlx)                      # nx(g, d, l) = sum_b inv_jac(b, d) nlx(b, l): (E, 3, 2)
    tx = np.einsum("eld,el->ed", grad, tnew)
    g2 = (tx ** 2).sum(axis=1)
    dc = np.zeros((X.shape[0], 3))
    for g, (i0, i1) in enumerate(GAUSS):
        ug = 0.5 * (u[:, i0] + u[:, i1])
        tg = 0.5 * (tnew[:, i0] + tnew[:, i1]); tog = 0.5 * (told[:, i0] + told[:, i1])
        rgi = (tg - tog) / dt + (ug * tx).sum(axis=1)
        ac = rgi / np.maximum(toler, g2)
        a_s = ac[:, None] * tx
        ps = np.max(np.abs(np.einsum("eb,ebd->ed", a_s, ij)), axis=1)
        with np.errstate(divide="ignore"):
            ps = np.minimum(1.0 / toler, 0.25 / ps)
        dc[:, g] = 0.25 * rgi * rgi * ps / np.maximum(toler, g2)
    dw = 0.5 * np.abs(detj) / 3.0
    st = dc.sum(axis=1)[:, None, None] * np.einsum("eid,ejd->eij", grad, grad) * dw[:, None, None]
    return dc, st


def implicit_solve(X, neig, fneig, u, T, dt, ntime, nits, use_dir=True, with_stab=False):
    """Time loop of unstr_implicit with the field: told = T ; solve (lhs + flux [+ stab(T, told) on the diagonal blocks]) T =
    (M/dt) told, exactly (dense)."""
    E = np.asarray(X).shape[0]
    sparse = E > 1500
    A, M = implicit_matrix(X, neig, fneig, u, dt, 0.0, use_dir, sparse=sparse)
    if sparse:
        import scipy.sparse as sp
        from scipy.sparse.linalg import spsolve
    T = np.array(T, np.float64).reshape(-1)
    E = A.shape[0] // 3
    for _ in range(ntime):
        told = T.copy()
        rhs = M @ told
        for _ in range(nits):
            As = A
            if with_stab:
                _, st = stab(X, u, T.reshape(E, 3), told.reshape(E, 3), dt)
                if sparse:
                    As = A + sp.block_diag(list(st), format="csr")
                else:
                    As = A.copy()
                    for e in range(E):
                        As[3 * e: 3 * e + 3, 3 * e: 3 * e + 3] += st[e]
            T = spsolve(As.tocsc(), rhs) if sparse else np.linalg.solve(As, rhs)
    return T.reshape(E, 3)


def bsr_to_dense(val, col, sparse=False):
    """(val[E,4,3,3], col[E,4]) of pamg_implicit_get_bsr -> (3E)^2, dense or scipy CSR."""
    E = val.shape[0]
    ok = np.asarray(col) >= 0
    re = np.broadcast_to(np.arange(E)[:, None], ok.shape)[ok]
    return _assemble(re, np.asarray(col)[ok].astype(np.int64), np.asarray(val)[ok], 3 * E, sparse)
