"""Plain NumPy FP64 reference of the operators and functionals, stated from the formulas rather than from the reference's
kernels (oracle/oracle.c restates those in their own order; this second statement catches a misread table or a transposed
layout that a restatement would copy).

Inputs are the library's own host objects: element corners (Mesh2D.vertices / elements), the global map
(H1Space.global_indices, [e, ty, tx]), the face data (FaceSpace.subspace_indices / global_indices), and the 1-D tables of
oracle.setup_np (pinned bit for bit to the reference's tables by tests/test_oracle_golden.py). Element (e, ty, tx) is the
node (x_tx, x_ty) of the Gauss-Lobatto grid under the bilinear map of the element's CCW corners c0..c3; a face runs from the
position of its face DOF 0 to that of its face DOF nb-1, with measure half its length."""
import numpy as np

from oracle import setup_np as S

GL, GLL = 0, 1


def rule(nq, kind=GL):
    return S.gauss_legendre(nq) if kind == GL else S.gauss_lobatto(nq)


def tables(nb, x):
    """P[q, a] = phi_a(x_q), D[q, a] = phi_a'(x_q)"""
    b = S.Basis(nb)
    return b.eval(np.asarray(x, np.float64)), b.deriv(np.asarray(x, np.float64))


def _scatter(n, I, R):
    y = np.zeros(n)
    np.add.at(y, I.reshape(-1), R.reshape(-1))
    return y


def _result(y, c, y0):
    return c * y if y0 is None else np.asarray(y0, np.float64) + c * y


class Space:
    """H1 space of bilinear quadrilaterals (a cb.H1Space)."""

    def __init__(self, fem):
        mesh = fem.mesh()
        self.fem = fem
        self.nb = fem.n_basis
        self.C = mesh.vertices()[mesh.elements()]  # (nel, 4, 2)
        self.I = fem.global_indices()              # (nel, nb, nb): [e, ty, tx]
        self.ndof = fem.size()
        self.xy = fem.physical_coordinates()
        gll = S.Basis(self.nb)
        self.gll_x, self.gll_w = np.asarray(gll.x), np.asarray(gll.w)
        # the local ordering this module assumes: I[e, ty, tx] is the node (x_tx, x_ty) of element e
        X = self.coordinates(self.gll_x)
        scale = max(1.0, float(np.abs(self.xy).max()))
        err = float(np.abs(self.xy[self.I] - X).max()) if self.I.size else 0.0
        assert err <= 1e-14 * scale, ("physical_coordinates()[I] is not the bilinear map at the GLL nodes", err)

    def _b(self, x):
        x = np.asarray(x, np.float64)
        eta, xi = x[:, None], x[None, :]  # [j, i]
        return [0.25 * (1 - xi) * (1 - eta), 0.25 * (1 + xi) * (1 - eta), 0.25 * (1 + xi) * (1 + eta), 0.25 * (1 - xi) * (1 + eta)]

    def coordinates(self, x):
        """(nel, nq, nq, 2) [e, j, i] = bilinear map at (x_i, x_j)"""
        return sum(b[None, :, :, None] * self.C[:, k, None, None, :] for k, b in enumerate(self._b(x)))

    def jacobian(self, x):
        """(dx/dxi, dx/deta), each (nel, nq, nq, 2) [e, j, i, r]"""
        x = np.asarray(x, np.float64)
        eta, xi = x[None, :, None, None], x[None, None, :, None]
        C = self.C[:, :, None, None, :]
        dxi = 0.25 * ((1 - eta) * (C[:, 1] - C[:, 0]) + (1 + eta) * (C[:, 2] - C[:, 3]))
        deta = 0.25 * ((1 - xi) * (C[:, 3] - C[:, 0]) + (1 + xi) * (C[:, 2] - C[:, 1]))
        shape = (len(self.C), len(x), len(x), 2)
        return np.broadcast_to(dxi, shape), np.broadcast_to(deta, shape)

    def measures(self, x):
        a, b = self.jacobian(x)
        return a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]

    def element_metrics(self, x, which):
        """H1Space.element_metrics layout: jacobians (nel, nq, nq, 2, 2) [e, j, i, c, r] = d x_r / d xi_c; measures
        (nel, nq, nq); physical_coordinates (nel, nq, nq, 2)"""
        if which == "jacobians":
            return np.stack(self.jacobian(x), axis=-2)
        if which == "measures":
            return self.measures(x)
        return self.coordinates(x)

    def stiffness(self, u, nq=None, kind=GL, c=1.0, y0=None):
        """y0 + c * S u, S_ab = sum_q w_q grad phi_a . grad phi_b |J| on the nq-point rule of the given kind"""
        nq = self.nb + 1 if nq is None else nq
        x, w = rule(nq, kind)
        P, D = tables(self.nb, x)
        a, b = self.jacobian(x)
        det = a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]
        W = np.outer(w, w)[None] / det
        g00, g01, g11 = W * (b * b).sum(-1), -W * (a * b).sum(-1), W * (a * a).sum(-1)
        U = np.asarray(u, np.float64)[self.I]
        Ux = np.einsum("ia,jb,eba->eji", D, P, U)
        Uy = np.einsum("ia,jb,eba->eji", P, D, U)
        Fx, Fy = g00 * Ux + g01 * Uy, g01 * Ux + g11 * Uy
        R = np.einsum("ia,jb,eji->eba", D, P, Fx) + np.einsum("ia,jb,eji->eba", P, D, Fy)
        return _result(_scatter(self.ndof, self.I, R), c, y0)

    def mass(self, u, nq=None, coef=None, c=1.0, y0=None):
        """y0 + c * M u with the Gauss-Legendre rule; coef: nodal coefficient interpolated to the quadrature points"""
        nq = (self.nb + 1 if coef is None else 1 + 3 * self.nb // 2 + 1) if nq is None else nq
        x, w = rule(nq, GL)
        P, _ = tables(self.nb, x)
        A = np.ones(self.I.shape) if coef is None else np.asarray(coef, np.float64)[self.I]
        aq = np.einsum("ia,jb,eba->eji", P, P, A)
        V = np.outer(w, w)[None] * self.measures(x) * aq * np.einsum("ia,jb,eba->eji", P, P, np.asarray(u, np.float64)[self.I])
        R = np.einsum("ia,jb,eji->eba", P, P, V)
        return _result(_scatter(self.ndof, self.I, R), c, y0)

    def linear_functional(self, f, nq=None, kind=GL, c=1.0, y0=None):
        """y0 + c * (f, phi_i); nq None: the collocated rule on the basis' own Gauss-Lobatto nodes"""
        if nq is None:
            x, w, P = self.gll_x, self.gll_w, np.eye(self.nb)
        else:
            x, w = rule(nq, kind)
            P, _ = tables(self.nb, x)
        X = self.coordinates(x)
        g = np.outer(w, w)[None] * self.measures(x) * f(X[..., 0], X[..., 1])
        R = np.einsum("ia,jb,eji->eba", P, P, g)
        return _result(_scatter(self.ndof, self.I, R), c, y0)


class Faces:
    """FaceSpace over straight edges (a cb.FaceSpace of the H1Space behind `space`)."""

    def __init__(self, space, fs):
        self.space, self.nb = space, space.nb
        self.fI = fs.subspace_indices()  # (nf, nb)
        self.proj = fs.global_indices()
        self.fdof = fs.size()
        pos = space.xy[self.proj[self.fI]] if self.fI.size else np.zeros((0, self.nb, 2))
        self.v0, self.v1 = pos[:, 0], pos[:, -1]
        self.meas = 0.5 * np.linalg.norm(self.v1 - self.v0, axis=1)

    def restrict(self, u):
        return np.asarray(u, np.float64)[self.proj]

    def prolong(self, v, y0):
        y = np.array(y0, np.float64)
        y[self.proj] += v
        return y

    def mass(self, v, nq=None, coef=None, c=1.0, y0=None):
        """y0 + c * H v on FaceSpace vectors, Gauss-Legendre rule; coef: FaceSpace coefficient vector"""
        nq = (self.nb + 1 if coef is None else 1 + 3 * self.nb // 2 + 1) if nq is None else nq
        x, w = rule(nq, GL)
        P, _ = tables(self.nb, x)
        A = np.ones(self.fI.shape) if coef is None else np.asarray(coef, np.float64)[self.fI]
        V = w[None] * self.meas[:, None] * (A @ P.T) * (np.asarray(v, np.float64)[self.fI] @ P.T)  # [f, q]
        return _result(_scatter(self.fdof, self.fI, V @ P), c, y0)

    def points(self, x):
        t = 0.5 * (1.0 + np.asarray(x, np.float64))
        return self.v0[:, None, :] + t[None, :, None] * (self.v1 - self.v0)[:, None, :]  # (nf, nq, 2)

    def linear_functional(self, f, nq=None, kind=GL, c=1.0, y0=None):
        """y0 + c * <f, phi_i> over the faces; nq None: collocated rule on the Gauss-Lobatto nodes"""
        if nq is None:
            x, w, P = self.space.gll_x, self.space.gll_w, np.eye(self.nb)
        else:
            x, w = rule(nq, kind)
            P, _ = tables(self.nb, x)
        X = self.points(x)
        g = w[None] * self.meas[:, None] * f(X[..., 0], X[..., 1])
        return _result(_scatter(self.fdof, self.fI, g @ P), c, y0)


def interior_edges(mesh):
    """every edge of mesh.edges() that is not a boundary edge, ascending"""
    return np.setdiff1d(np.arange(mesh.n_edges()), mesh.boundary_edges()).astype(np.int32)
