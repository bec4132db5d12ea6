"""Host-side mirror of the reference's C++ interface for the solve path (same class / method names, argument
meaning and error behaviour as cuddh.hpp), implemented as thin wrappers over the C ABI in
include/cuddh_b200.h. Device vectors are torch CUDA tensors (torch is only the owner of device memory and
streams here) or raw device addresses (int).

    reference                                  here
    Mesh2D::uniform_rect / from_vertices       Mesh2D.uniform_rect / Mesh2D.from_vertices
    QuadratureRule(n, type)                    QuadratureRule(n, type)
    Basis(n)::eval/deriv                       Basis(n).eval/deriv
    H1Space(mesh, basis)                       H1Space(mesh, basis)
    FaceSpace(fem, nf, faces)                  FaceSpace(fem, faces)
    StiffnessMatrix / MassMatrix / ...         same names; .action(x, y) and .action(c, x, y)
    gmres(n, x, A, b, [P,] m, maxit, tol,..)   gmres(n, x, A, b, m, maxit, tol, P=None, ...)
    DDH(omega, h_a, fem, nx, ny)               DDH(omega, h_a, fem, nx, ny, block=16)
    (new) DDHTransfer(ddh)                     DDHTransfer(ddh, max_bytes=0): the same operator with T assembled
"""
import ctypes as C
import numpy as np

from . import capi
from .capi import check, load

GaussLegendre, GaussLobatto = 0, 1


def _ptr(t):
    """device address of a torch tensor (must be contiguous CUDA) or pass-through of an int / None."""
    if t is None:
        return None
    if isinstance(t, int):
        return t
    if not t.is_cuda:
        raise capi.CuddhError("expected a CUDA tensor (every vector argument is a DEVICE pointer)")
    if not t.is_contiguous():
        raise capi.CuddhError("expected a contiguous tensor")
    return t.data_ptr()


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream if torch.cuda.is_available() else None


def _destroy(fn, obj):
    """release a C handle; safe during interpreter shutdown (module globals may already be gone)"""
    h = getattr(obj, "_h", None)
    lib = getattr(capi, "_lib", None) if capi is not None else None
    if h and lib is not None:
        try:
            getattr(lib, fn)(h)
        except Exception:
            pass
    obj._h = None


def _np(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _vp(a):
    return a.ctypes.data_as(C.c_void_p)


class QuadratureRule:
    """include/QuadratureRule.hpp:13-77."""
    GaussLegendre, GaussLobatto = 0, 1

    def __init__(self, n, type=GaussLobatto):
        self.n, self.type = n, type
        self._x = np.zeros(n)
        self._w = np.zeros(n)
        check(load().cuddh_b200_quadrature(n, type, _vp(self._x), _vp(self._w)))

    def size(self):
        return self.n

    def x(self, i=None):
        return self._x if i is None else self._x[i]

    def w(self, i=None):
        return self._w if i is None else self._w[i]

    def name(self):
        return ("legendre" if self.type == GaussLegendre else "lobatto") + "%05d" % self.n


class Basis:
    """include/Basis.hpp:13-63."""

    def __init__(self, n):
        self.n = n
        self._h = C.c_void_p()
        check(load().cuddh_b200_basis_create(n, C.byref(self._h)))

    def __del__(self):
        _destroy("cuddh_b200_basis_destroy", self)

    def size(self):
        return self.n

    def eval(self, x):
        """P with P[j, i] = phi_i(x_j) (the reference's column-major (m, n) array, returned as numpy (m, n))."""
        x = _np(x, np.float64)
        P = np.zeros((self.n, len(x)))
        check(load().cuddh_b200_basis_eval(self._h, len(x), _vp(x), _vp(P)))
        return P.T.copy()

    def deriv(self, x):
        x = _np(x, np.float64)
        D = np.zeros((self.n, len(x)))
        check(load().cuddh_b200_basis_deriv(self._h, len(x), _vp(x), _vp(D)))
        return D.T.copy()

    def quadrature(self):
        x = np.zeros(self.n)
        w = np.zeros(self.n)
        check(load().cuddh_b200_basis_nodes(self._h, _vp(x), _vp(w)))
        return x, w


class Mesh2D:
    """include/Mesh2D.hpp."""

    def __init__(self, handle):
        self._h = handle
        s = np.zeros(5, np.int64)
        check(load().cuddh_b200_mesh_sizes(self._h, _vp(s)))
        self._sizes = s

    def __del__(self):
        _destroy("cuddh_b200_mesh_destroy", self)

    @staticmethod
    def uniform_rect(nx, ax, bx, ny, ay, by):
        h = C.c_void_p()
        check(load().cuddh_b200_mesh_uniform_rect(nx, ax, bx, ny, ay, by, C.byref(h)))
        return Mesh2D(h)

    @staticmethod
    def from_vertices(xy, elems):
        """xy: (nv, 2) coordinates, elems: (nel, 4) CCW corner indices."""
        xy = _np(xy, np.float64)
        elems = _np(elems, np.int32)
        h = C.c_void_p()
        check(load().cuddh_b200_mesh_from_vertices(len(xy), _vp(xy), len(elems), _vp(elems), C.byref(h)))
        return Mesh2D(h)

    def n_elem(self):
        return int(self._sizes[0])

    def n_nodes(self):
        return int(self._sizes[1])

    def n_edges(self, kind=None):
        return int(self._sizes[2] if kind is None else self._sizes[3] if kind == "boundary" else self._sizes[4])

    def edges(self):
        """(n_edges, 8): nodes0, nodes1, el0, el1, side0, side1, delta, is_boundary."""
        e = np.zeros((self.n_edges(), 8), np.int32)
        check(load().cuddh_b200_mesh_edges(self._h, _vp(e)))
        return e

    def boundary_edges(self):
        b = np.zeros(int(self._sizes[3]), np.int32)
        check(load().cuddh_b200_mesh_boundary_edges(self._h, _vp(b)))
        return b

    def vertices(self):
        """(n_nodes, 2) vertex coordinates"""
        xy = np.zeros((self.n_nodes(), 2))
        check(load().cuddh_b200_mesh_vertices(self._h, _vp(xy)))
        return xy

    def elements(self):
        """(n_elem, 4) CCW corner vertex ids"""
        el = np.zeros((self.n_elem(), 4), np.int32)
        check(load().cuddh_b200_mesh_elements(self._h, _vp(el)))
        return el

    def min_h(self):
        a, b = C.c_double(), C.c_double()
        check(load().cuddh_b200_mesh_h(self._h, C.byref(a), C.byref(b)))
        return a.value

    def max_h(self):
        a, b = C.c_double(), C.c_double()
        check(load().cuddh_b200_mesh_h(self._h, C.byref(a), C.byref(b)))
        return b.value


class H1Space:
    """include/H1Space.hpp:18-65."""

    def __init__(self, mesh, basis):
        self._mesh, self._basis = mesh, basis
        self.n_basis = basis.size()
        self._h = C.c_void_p()
        check(load().cuddh_b200_h1space_create(mesh._h, self.n_basis, C.byref(self._h)))

    def __del__(self):
        _destroy("cuddh_b200_h1space_destroy", self)

    def size(self):
        return int(load().cuddh_b200_h1space_size(self._h))

    def check_plan(self, node_major):
        """host-only self check of the assembly plan (include/cuddh_b200.h): dict of plan sizes and 'mismatches' (0 = ok)."""
        st = (C.c_int64 * 8)()
        check(load().cuddh_b200_h1space_check_plan(self._h, int(node_major), st))
        keys = ("n_patches", "patch_elems", "listed_dofs", "shared_dofs", "max_pdof", "dofs_over_four", "mismatches", "hash")
        return dict(zip(keys, [int(v) for v in st[:8]]))

    def mesh(self):
        return self._mesh

    def basis(self):
        return self._basis

    def global_indices(self):
        """host copy, numpy (n_elem, nb, nb) with [el, j, i] = I(i, j, el)."""
        nb = self.n_basis
        I = np.zeros((self._mesh.n_elem(), nb, nb), np.int32)
        check(load().cuddh_b200_h1space_global_indices(self._h, _vp(I)))
        return I

    def physical_coordinates(self):
        xy = np.zeros((self.size(), 2))
        check(load().cuddh_b200_h1space_physical_coordinates(self._h, _vp(xy)))
        return xy

    def element_metrics(self, xq, which):
        """Mesh2D::ElementMetricCollection (include/Mesh2D.hpp:33-41) on the tensor grid of the 1-D points xq, as a CUDA tensor:
        which = "jacobians" (n_elem, nq, nq, 2, 2) [el, j, i, c, r] = J(r, c, i, j, el); "measures" (n_elem, nq, nq);
        "physical_coordinates" (n_elem, nq, nq, 2)."""
        import torch
        xq = _np(xq, np.float64)
        nq, nel = len(xq), self._mesh.n_elem()
        k = {"jacobians": 0, "measures": 1, "physical_coordinates": 2}[which]
        shape = {0: (nel, nq, nq, 2, 2), 1: (nel, nq, nq), 2: (nel, nq, nq, 2)}[k]
        out = torch.empty(shape, dtype=torch.float64, device="cuda")
        check(load().cuddh_b200_element_metrics(self._h, nq, _vp(xq), k, _ptr(out), _stream()))
        return out


class FaceSpace:
    """include/H1Space.hpp:69-147."""

    def __init__(self, fem, faces):
        self.fem = fem
        faces = _np(faces, np.int32)
        self._faces = faces
        self._nf = len(faces)
        self._h = C.c_void_p()
        check(load().cuddh_b200_facespace_create(fem._h, len(faces), _vp(faces), C.byref(self._h)))

    def __del__(self):
        _destroy("cuddh_b200_facespace_destroy", self)

    def size(self):
        return int(load().cuddh_b200_facespace_size(self._h))

    def n_faces(self):
        return self._nf

    def faces(self):
        return self._faces

    def h1_space(self):
        return self.fem

    def subspace_indices(self):
        I = np.zeros((self._nf, self.fem.n_basis), np.int32)
        check(load().cuddh_b200_facespace_subspace_indices(self._h, _vp(I)))
        return I

    def global_indices(self):
        p = np.zeros(self.size(), np.int32)
        check(load().cuddh_b200_facespace_global_indices(self._h, _vp(p)))
        return p

    def restrict(self, x, y):
        check(load().cuddh_b200_facespace_restrict(self._h, _ptr(x), _ptr(y), _stream()))

    def prolong(self, x, y):
        check(load().cuddh_b200_facespace_prolong(self._h, _ptr(x), _ptr(y), _stream()))

    def orth(self, x):
        check(load().cuddh_b200_facespace_orth(self._h, _ptr(x), _stream()))


class Operator:
    """include/Operator.hpp:6-17: action(c, x, y): y += c*A*x ; action(x, y): y = A*x (device vectors)."""

    _h = None

    def __del__(self):
        _destroy("cuddh_b200_operator_destroy", self)

    def action(self, *args):
        if len(args) == 2:
            x, y = args
            check(load().cuddh_b200_operator_apply(self._h, 1.0, 0, _ptr(x), _ptr(y), _stream()))
        elif len(args) == 3:
            c, x, y = args
            check(load().cuddh_b200_operator_apply(self._h, float(c), 1, _ptr(x), _ptr(y), _stream()))
        else:
            raise TypeError("action(x, y) or action(c, x, y)")

    def algorithmic_bytes(self):
        return int(load().cuddh_b200_operator_bytes(self._h))

    def moved_bytes(self):
        """bytes of the formulation this handle runs (affine meshes: per-element metric constants instead of the stored metric)"""
        return int(load().cuddh_b200_operator_bytes_moved(self._h))

    def is_affine(self):
        return bool(load().cuddh_b200_operator_is_affine(self._h))

    def kernel_kind(self):
        """0 lane-per-row / generic kernel, 1 warp-specialised thread-per-element kernel, 2 fused Helmholtz kernel,
        3 warp-specialised thread-pair-per-element kernel (n_basis 6-9), -1 n/a."""
        return int(load().cuddh_b200_operator_kernel_kind(self._h))

    def is_fused(self):
        return self.kernel_kind() == 2

    def time_phases(self, x, y, reps):
        """(ms of the patch kernel alone, ms of the rest of the action alone), CUDA events on the current stream."""
        a, b = C.c_float(), C.c_float()
        check(load().cuddh_b200_operator_time_phases(self._h, _ptr(x), _ptr(y), reps, C.byref(a), C.byref(b), _stream()))
        return a.value, b.value

    # C callback usable by gmres without a Python trampoline
    def _as_apply(self):
        return C.cast(load().cuddh_b200_operator_as_apply, C.c_void_p), self._h


class StiffnessMatrix(Operator):
    """include/StiffnessMatrix.hpp:11-38."""

    def __init__(self, fem, quad=None):
        self.fem = fem
        self._h = C.c_void_p()
        nq, qt = (0, GaussLegendre) if quad is None else (quad.size(), quad.type)
        check(load().cuddh_b200_stiffness_create(fem._h, nq, qt, C.byref(self._h)))


class MassMatrix(Operator):
    """include/MassMatrix.hpp:14-41: MassMatrix(fem) or MassMatrix(a, fem) with `a` a DEVICE nodal vector."""

    def __init__(self, *args, n_quad=0):
        a, fem = (None, args[0]) if len(args) == 1 else args
        self.fem, self._a = fem, a
        self._h = C.c_void_p()
        check(load().cuddh_b200_mass_create(fem._h, _ptr(a), n_quad, C.byref(self._h)))


class DiagInvMassMatrix(Operator):
    """include/MassMatrix.hpp:44-68."""

    def __init__(self, *args):
        a, fem = (None, args[0]) if len(args) == 1 else args
        self.fem = fem
        self._h = C.c_void_p()
        check(load().cuddh_b200_diag_inv_mass_create(fem._h, _ptr(a), C.byref(self._h)))


class FaceMassMatrix(Operator):
    """include/FaceMassMatrix.hpp: FaceMassMatrix(fs) or FaceMassMatrix(a, fs); vectors are FaceSpace vectors."""

    def __init__(self, *args, n_quad=0):
        a, fs = (None, args[0]) if len(args) == 1 else args
        self.fs = fs
        self._h = C.c_void_p()
        check(load().cuddh_b200_facemass_create(fs._h, _ptr(a), n_quad, C.byref(self._h)))

    def action_h1(self, c, x, y):
        """fused restrict + action + prolong on H1 vectors: y[proj] += c * H * x[proj]."""
        check(load().cuddh_b200_facemass_apply_h1(self._h, float(c), _ptr(x), _ptr(y), _stream()))


class DiagInvFaceMassMatrix(Operator):
    def __init__(self, *args):
        a, fs = (None, args[0]) if len(args) == 1 else args
        self.fs = fs
        self._h = C.c_void_p()
        check(load().cuddh_b200_diag_inv_facemass_create(fs._h, _ptr(a), C.byref(self._h)))


class Helmholtz(Operator):
    """examples/Helmholtz.hpp:10-80: x = [u; v] -> [S u - w^2 M u - w H v ; -(S v - w^2 M v + w H u)]."""

    def __init__(self, omega, a2x, ax, fem, fs):
        self.fem, self.fs, self.omega = fem, fs, omega
        self._h = C.c_void_p()
        check(load().cuddh_b200_helmholtz_create(float(omega), _ptr(a2x), _ptr(ax), fem._h, fs._h, C.byref(self._h)))

    def action(self, *args):
        if len(args) != 2:
            raise capi.CuddhError("Helmholtz::action(c, x, y) not implemented")
        x, y = args
        check(load().cuddh_b200_operator_apply(self._h, 1.0, 0, _ptr(x), _ptr(y), _stream()))


class LinearFunctional:
    """include/LinearFunctional.hpp:11-37: F[i] (+)= c (f, phi_i). LinearFunctional(fem): collocated rule on the basis' own
    Gauss-Lobatto nodes; LinearFunctional(fem, quad): quad.size()-point rule. f is called with CUDA tensors (x, y) of the
    quadrature-point coordinates and returns a tensor of the same shape (the reference takes a __device__ lambda)."""

    def __init__(self, fem, quad=None):
        self.fem = fem
        self.fast = quad is None
        if quad is None:
            self.x, self.w = fem.basis().quadrature()
            self.P = None
        else:
            self.x, self.w = np.array(quad.x(), np.float64), np.array(quad.w(), np.float64)
            self.P = np.ascontiguousarray(fem.basis().eval(self.x).T)  # column-major (nq, nb)

    def action(self, *args):
        import torch
        c, f, F = (1.0,) + tuple(args) if len(args) == 2 else args
        if len(args) == 2:
            F.zero_()
        X = self.fem.element_metrics(self.x, "physical_coordinates")
        detJ = self.fem.element_metrics(self.x, "measures")
        w = torch.as_tensor(self.w, device="cuda")
        g = (w[None, :, None] * w[None, None, :] * detJ * f(X[..., 0], X[..., 1])).contiguous()
        check(load().cuddh_b200_linear_functional_assemble(self.fem._h, len(self.x), None if self.P is None else _vp(self.P), _ptr(g),
                                                           float(c), _ptr(F), _stream()))


class FaceLinearFunctional:
    """include/FaceLinearFunctional.hpp:13-39: F[i] (+)= c <f, phi_i> over the faces of a FaceSpace (FaceSpace vectors). Face
    points: the side of edge->elements[0] the face lies on, in increasing reference coordinate (source/H1Space.cpp:151-157),
    measure = length / 2 (StraightEdge)."""

    def __init__(self, fs, quad=None):
        self.fs = fs
        fem = fs.fem
        if quad is None:
            self.x, self.w = fem.basis().quadrature()
            self.P = None
        else:
            self.x, self.w = np.array(quad.x(), np.float64), np.array(quad.w(), np.float64)
            self.P = np.ascontiguousarray(fem.basis().eval(self.x).T)
        mesh = fem.mesh()
        E = mesh.edges()[fs.faces()]
        V, EL = mesh.vertices(), mesh.elements()
        side_nodes = np.array([[0, 1], [1, 2], [3, 2], [0, 3]])
        el, sd = E[:, 2], E[:, 4]
        v0 = V[EL[el, side_nodes[sd, 0]]]
        v1 = V[EL[el, side_nodes[sd, 1]]]
        t = 0.5 * (1.0 + self.x)
        self.X = v0[:, None, :] + t[None, :, None] * (v1 - v0)[:, None, :]  # (n_faces, nq, 2)
        self.meas = 0.5 * np.linalg.norm(v1 - v0, axis=1)

    def action(self, *args):
        import torch
        c, f, F = (1.0,) + tuple(args) if len(args) == 2 else args
        if len(args) == 2:
            F.zero_()
        X = torch.as_tensor(self.X, device="cuda")
        g = (f(X[..., 0], X[..., 1]) * torch.as_tensor(self.w, device="cuda")[None, :] * torch.as_tensor(self.meas, device="cuda")[:, None]).contiguous()
        check(load().cuddh_b200_face_linear_functional_assemble(self.fs._h, len(self.x), None if self.P is None else _vp(self.P), _ptr(g),
                                                                float(c), _ptr(F), _stream()))


class SolverOut:
    """include/gmres.hpp:14-21 solver_out (+ the orthogonalisation statistics of this library)."""

    def __init__(self, so, res, time, stats=None):
        self.success = bool(so.success)
        self.num_iter = so.num_iter
        self.num_matvec = so.num_matvec
        self.res_norm = list(res[:so.n_res])
        self.time = list(time[:so.n_res])
        self.orth_bytes = stats.orth_bytes if stats is not None else 0.0
        self.orth_ms = stats.orth_ms if stats is not None else 0.0
        self.reorth = stats.reorth if stats is not None else 0
        self.allreduces = stats.allreduces if stats is not None else 0


_callback_error = []


def _callback(A, kind):
    """(function pointer, ctx, keepalive) for an operator: library objects use the in-library trampoline, any
    object with .action(x, y) taking raw device addresses is wrapped in a ctypes callback. The callback runs under the
    stream gmres works on (it is handed over as the 4th argument; for torch-backed operators that is torch's current
    stream, because gmres() below passes exactly that one). An exception in the Python operator aborts the solve."""
    if hasattr(A, "_as_apply"):
        fn, ctx = A._as_apply()
        return fn, ctx, None
    proto = capi.APPLY_D if kind == "d" else capi.APPLY_F

    def tramp(_ctx, x, y, _stream):
        try:
            A.action(int(x), int(y))
            return 0
        except BaseException as e:  # ctypes would swallow it: hand a status back instead and re-raise after the solve
            _callback_error.append(e)
            return -7

    cb = proto(tramp)
    return C.cast(cb, C.c_void_p), None, cb


MGS, CGS2 = 0, 1


def gmres(n, x, A, b, m, maxit, tol=None, P=None, verbose=0, max_seconds=6 * 60 * 60, orth=-1, comm=None, mask=None, time_orth=False,
          flexible=False):
    """include/gmres.hpp:33-36. x, b: device vectors (torch float64 -> FP64 solver, float32 -> FP32 solver).
    A (and P): operators of this module, or any object with .action(x_ptr, y_ptr) on raw device addresses.
    orth: MGS (the reference's arithmetic) / CGS2 / -1 = library default; comm + mask: distributed vectors (Comm, uint8 tensor).
    flexible=True: P is applied on the RIGHT and afresh to every basis vector (FGMRES), so it may be an inner iterative solve."""
    import torch
    single = isinstance(x, torch.Tensor) and x.dtype == torch.float32
    cap = maxit + 2
    res = np.zeros(cap)
    tim = np.zeros(cap)
    so = capi.SolverOut()
    st = capi.GmresStats()
    opts = capi.GmresOptions(int(orth), comm._h if comm is not None else None, _ptr(mask), int(bool(time_orth)), int(bool(flexible)))
    fa, ca, keep_a = _callback(A, "f" if single else "d")
    del _callback_error[:]
    if single:
        if P is not None:
            raise capi.CuddhError("the FP32 gmres overload has no preconditioner argument (include/gmres.hpp:36)")
        tol = 1e-4 if tol is None else tol
        rc = load().cuddh_b200_gmres_f_ex(n, _ptr(x), fa, ca, _ptr(b), m, maxit, tol, verbose, float(max_seconds), C.byref(opts),
                                          C.byref(so), _vp(res), _vp(tim), cap, C.byref(st), _stream())
    else:
        tol = 1e-6 if tol is None else tol
        fp, cp, keep_p = (None, None, None) if P is None else _callback(P, "d")
        rc = load().cuddh_b200_gmres_d_ex(n, _ptr(x), fa, ca, _ptr(b), fp, cp, m, maxit, tol, verbose, float(max_seconds),
                                          C.byref(opts), C.byref(so), _vp(res), _vp(tim), cap, C.byref(st), _stream())
    if _callback_error:
        raise _callback_error.pop()
    check(rc)
    return SolverOut(so, res, tim, st)


def set_option(name, value):
    check(load().cuddh_b200_set_option(name.encode(), int(value)))


def get_option(name):
    return int(load().cuddh_b200_get_option(name.encode()))


class Comm:
    """Library-owned NCCL communicator (include/cuddh_b200.h: cuddh_b200_comm_*), one per process / GPU. The 128-byte unique id
    is made by rank 0 and travels through the caller's bootstrap - here torch.distributed (any backend)."""

    def __init__(self, rank, world, group=None):
        import torch.distributed as dist
        self.rank, self.world = rank, world
        ident = [None]
        if rank == 0:
            buf = (C.c_ubyte * 128)()
            check(load().cuddh_b200_comm_unique_id(buf))
            ident[0] = bytes(buf)
        if world > 1:
            dist.broadcast_object_list(ident, src=0, group=group)
        buf = (C.c_ubyte * 128).from_buffer_copy(ident[0])
        self._h = C.c_void_p()
        check(load().cuddh_b200_comm_create(buf, rank, world, C.byref(self._h)))

    def __del__(self):
        _destroy("cuddh_b200_comm_destroy", self)

    def allreduce(self, t):
        """in-place sum of a float64 CUDA tensor over the ranks (stream-ordered on torch's current stream)"""
        check(load().cuddh_b200_comm_allreduce_d(self._h, _ptr(t), t.numel(), _stream()))


class DDH:
    """include/DDH.hpp:21-84 (SinglePrecisionOperator). h_a: HOST nodal coefficient (numpy, length ndof)."""

    def __init__(self, omega, h_a, fem, nx, ny, block=16):
        self.fem = fem
        h_a = _np(h_a, np.float64)
        if len(h_a) != fem.size():
            raise capi.CuddhError("DDH: coefficient array must have length fem.size()")
        self._h = C.c_void_p()
        check(load().cuddh_b200_ddh_create(float(omega), _vp(h_a), fem._h, nx, ny, block, C.byref(self._h)))

    def __del__(self):
        _destroy("cuddh_b200_ddh_destroy", self)

    def size(self):
        return int(load().cuddh_b200_ddh_size(self._h))

    def rhs(self, f, b):
        check(load().cuddh_b200_ddh_rhs(self._h, _ptr(f), _ptr(b), _stream()))

    def action(self, x, y):
        check(load().cuddh_b200_ddh_action(self._h, _ptr(x), _ptr(y), _stream()))

    def postprocess(self, lam, f, u):
        check(load().cuddh_b200_ddh_postprocess(self._h, _ptr(lam), _ptr(f), _ptr(u), _stream()))

    # subdomain-range variants (multi-GPU sharding, see parallel.ShardedDDH)
    def apply_T_range(self, x, t, dom_begin, dom_end):
        check(load().cuddh_b200_ddh_apply_T_range(self._h, _ptr(x), _ptr(t), dom_begin, dom_end, _stream()))

    def rhs_range(self, f, b, dom_begin, dom_end):
        check(load().cuddh_b200_ddh_rhs_range(self._h, _ptr(f), _ptr(b), dom_begin, dom_end, _stream()))

    def postprocess_range(self, lam, f, u, dom_begin, dom_end):
        check(load().cuddh_b200_ddh_postprocess_range(self._h, _ptr(lam), _ptr(f), _ptr(u), dom_begin, dom_end, _stream()))

    def info(self):
        v = np.zeros(8, np.int64)
        dt = C.c_double()
        check(load().cuddh_b200_ddh_info(self._h, _vp(v), C.byref(dt)))
        keys = ["n_domains", "n_shared", "nt", "mx_dof", "mx_fdof", "mx_elem_per_dom", "n_basis", "block"]
        d = {k: int(x) for k, x in zip(keys, v)}
        d["dt"] = dt.value
        return d

    def array(self, name):
        cnt = C.c_int64()
        check(load().cuddh_b200_ddh_get_array(self._h, name.encode(), None, 0, C.byref(cnt)))
        isf = name in ("m", "gmi", "a", "H", "D", "g", "wh_filter", "cs", "sn")
        out = np.zeros(cnt.value, np.float32 if isf else np.int32)
        check(load().cuddh_b200_ddh_get_array(self._h, name.encode(), _vp(out), out.nbytes, C.byref(cnt)))
        return out

    def flops(self):
        return float(load().cuddh_b200_ddh_flops(self._h))

    def kernel_kind(self):
        """1 = register-tiled thread-per-element kernel (n_basis 4, block 16, uniform metric), 0 = generic kernel"""
        return int(load().cuddh_b200_ddh_kernel_kind(self._h))

    def _as_apply(self):
        return C.cast(load().cuddh_b200_ddh_as_apply, C.c_void_p), self._h

    def transfer_slots(self):
        """Host-only slot maps of the assembled operator (DDHTransfer): (inp, out, orphans). inp[p, k] / out[p, k] is the slot that
        local input / output k of subdomain p reads / writes (-1: face DOF on the physical boundary), shape (n_domains, 2F); k < F is
        the lambda entry, k >= F the mu entry of face position k mod F (boundary ring of the subdomain grid, ascending Y*n1 + X).
        orphans: ascending slots that no subdomain writes."""
        tf = C.c_int()
        check(load().cuddh_b200_ddh_transfer_slots(self._h, None, None, 0, C.byref(tf)))
        nd = self.info()["n_domains"]
        inp = np.zeros((nd, tf.value), np.int32)
        out = np.zeros((nd, tf.value), np.int32)
        check(load().cuddh_b200_ddh_transfer_slots(self._h, _vp(inp), _vp(out), inp.size, C.byref(tf)))
        cnt = C.c_int64()
        check(load().cuddh_b200_ddh_transfer_orphans(self._h, None, 0, C.byref(cnt)))
        orphans = np.zeros(cnt.value, np.int32)
        check(load().cuddh_b200_ddh_transfer_orphans(self._h, _vp(orphans), orphans.size, C.byref(cnt)))
        return inp, out, orphans


class DDHTransfer:
    """The DDH operator with its trace map T assembled: one dense 2F x 2F FP32 block per subdomain, probed once with 2F WaveHoltz
    actions, after which action(x, y) = x - T x is one streaming batched matvec. Same linear map as ddh.action (bitwise on unit
    vectors); rhs / postprocess / array are the DDH's own, so it stands in for the DDH in gmres(...) and DDHPreconditioner.
    max_bytes: device memory it may take (0 = whatever is free); CuddhError naming the bytes needed if the blocks do not fit."""

    def __init__(self, ddh, max_bytes=0):
        self.ddh = ddh  # the DDH handle must outlive this one
        self.fem = ddh.fem
        self._h = C.c_void_p()
        check(load().cuddh_b200_ddh_transfer_create(ddh._h, int(max_bytes), _stream(), C.byref(self._h)))

    def __del__(self):
        _destroy("cuddh_b200_ddh_transfer_destroy", self)

    def size(self):
        return self.ddh.size()

    def action(self, x, y):
        check(load().cuddh_b200_ddh_transfer_action(self._h, _ptr(x), _ptr(y), _stream()))

    def rhs(self, f, b):
        self.ddh.rhs(f, b)

    def postprocess(self, lam, f, u):
        self.ddh.postprocess(lam, f, u)

    def array(self, name):
        return self.ddh.array(name)

    def info(self):
        v = np.zeros(6, np.int64)
        check(load().cuddh_b200_ddh_transfer_info(self._h, _vp(v)))
        keys = ["n_domains", "two_f", "block_bytes", "bytes_per_action", "probe_launches"]
        d = {k: int(x) for k, x in zip(keys, v)}
        d["probe_ms"] = float(v[5]) / 1000.0
        return d

    def block(self, dom):
        """host copy of M_dom, shape (2F, 2F): column k = T's response at the subdomain's outputs to a 1 at its input k"""
        tf = self.info()["two_f"]
        out = np.zeros((tf, tf), np.float32)  # C order of the column-major block -> transpose
        check(load().cuddh_b200_ddh_transfer_get_block(self._h, int(dom), _vp(out)))
        return out.T.copy()

    def _as_apply(self):
        return C.cast(load().cuddh_b200_ddh_transfer_as_apply, C.c_void_p), self._h


class DDHPreconditioner:
    """SURVEY §8(f) rank 4: path B as a preconditioner of path A. P r ~ A^{-1} r for the FP64 Helmholtz composite A of
    examples/Helmholtz.hpp: the residual [r_u; r_v] of A [u; v] = b is the load [F; G] = [r_u; -r_v] of the time-harmonic
    problem DDH solves (the composite negates its second block row, examples/Helmholtz.hpp:55), so
        P r = postprocess( gmres_f32( DDH, rhs( w * [r_u; -r_v] ) ) ),      w_i = 1 / (number of subdomains that hold DOF i)
    - one substructured FP32 DDH-GMRES solve (WaveHoltz local solves, GLL-collocated operators) per application. The weight w is
    needed because DDH::rhs hands the ASSEMBLED load entry to every subdomain that holds the DOF (source/DDH.cpp:208-212), so a
    load on an interface node would otherwise count 2 (4 at cross points) times; on uniform_rect the equal split is also the
    lumped-mass share m * gmi that postprocess uses as partition of unity. P is an inner iterative solve, i.e. not a fixed linear
    map: use it with gmres(..., P=this, flexible=True). The reference has no such composition (its DDH is the system operator of
    the interface problem, SURVEY R1), so there is no parity oracle for this class - its test checks the outer solve against a
    direct FP64 solve of the assembled operator."""

    def __init__(self, ddh, m=20, maxit=100, tol=1e-4, orth=-1):
        import torch
        self.ddh, self.m, self.maxit, self.tol, self.orth = ddh, m, maxit, tol, orth
        self.n = ddh.fem.size()
        nl = ddh.size()
        g = ddh.array("gI")
        mult = np.bincount(g[g >= 0], minlength=self.n).astype(np.float64)
        w = 1.0 / np.maximum(mult, 1.0)
        self.w = torch.as_tensor(np.concatenate([w, -w]), device="cuda")
        self.f = torch.empty(2 * self.n, dtype=torch.float64, device="cuda")
        self.b = torch.empty(nl, dtype=torch.float32, device="cuda")
        self.lam = torch.empty(nl, dtype=torch.float32, device="cuda")
        self.inner_restarts, self.inner_matvecs, self.applications = 0, 0, 0

    def action(self, xp, yp):
        import torch
        from .parallel import _as_tensor
        x = xp if isinstance(xp, torch.Tensor) else _as_tensor(xp, 2 * self.n, torch.float64)
        torch.mul(x, self.w, out=self.f)  # the only torch op of this add-on: split the load, flip the sign of the second block
        self.ddh.rhs(self.f, self.b)
        fill(self.lam.numel(), 0.0, self.lam)
        out = gmres(self.lam.numel(), self.lam, self.ddh, self.b, self.m, self.maxit, self.tol, orth=self.orth)
        self.inner_restarts += out.num_iter
        self.inner_matvecs += out.num_matvec
        self.applications += 1
        self.ddh.postprocess(self.lam, self.f, yp)


class HelmholtzSlab:
    """Path A across GPUs in the library (cuddh_b200_slab_*): the Helmholtz composite on this rank's slab + the interface-row
    exchange with the two neighbours (pack fused into the face-mass launch, one grouped ncclSend/ncclRecv, add)."""

    def __init__(self, op, comm, rank, world, fem, fs_phys, bottom_dofs, top_dofs):
        self.op, self.comm, self.rank, self.world, self.fem = op, comm, rank, world, fem
        b, t = _np(bottom_dofs, np.int32), _np(top_dofs, np.int32)
        self._h = C.c_void_p()
        check(load().cuddh_b200_slab_create(comm._h if comm is not None else None, rank, world, fem._h, fs_phys._h if fs_phys is not None else None,
                                            len(b), _vp(b), len(t), _vp(t), C.byref(self._h)))
        check(load().cuddh_b200_slab_bind(self._h, op._h))
        self.n = 2 * fem.size()

    def __del__(self):
        _destroy("cuddh_b200_slab_destroy", self)

    def bytes_per_apply(self):
        return int(load().cuddh_b200_slab_bytes(self._h))

    def uses_peer_memory(self):
        """True: rows travel as NVLink stores into the neighbours' buffers + epoch flags; False: ncclSend / ncclRecv"""
        return bool(load().cuddh_b200_slab_uses_peer_memory(self._h))

    def apply(self, x, y):
        check(load().cuddh_b200_helmholtz_apply_slab(self.op._h, self._h, _ptr(x), _ptr(y), _stream()))

    def exchange(self, y):
        check(load().cuddh_b200_slab_exchange(self._h, _ptr(y), _stream()))

    def mask(self):
        import torch
        p = load().cuddh_b200_slab_mask(self._h)
        if not p:
            check(-1)
        n = self.n

        class _Raw:
            __cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (int(p), False), "version": 2}
        t = torch.as_tensor(_Raw(), device="cuda")
        t._keepalive = self
        return t

    def _as_apply(self):
        return C.cast(load().cuddh_b200_slab_as_apply, C.c_void_p), self._h

    def solve(self, b, x, m=20, maxit=1000, tol=1e-6, orth=-1):
        """distributed FP64 GMRES(m) in the library on the slab partition: masked inner products + one NCCL allreduce per pass"""
        return gmres(self.n, x, self, b, m, maxit, tol, orth=orth, comm=self.comm, mask=self.mask())


class DDHDist:
    """DDH across GPUs in the library (cuddh_b200_ddh_dist_*): subdomain row slabs, owner = reading subdomain's rank, traces that
    cross a slab boundary packed in the kernel epilogue and moved with ncclSend/ncclRecv. comm=None: partition tables only /
    single rank. Vectors keep the global length ddh.size(); use .mask() as the ownership mask of gmres(..., comm=, mask=)."""

    def __init__(self, ddh, comm, rank, world):
        self.ddh, self.comm, self.rank, self.world = ddh, comm, rank, world
        self._h = C.c_void_p()
        check(load().cuddh_b200_ddh_dist_create(ddh._h, comm._h if comm is not None else None, rank, world, C.byref(self._h)))
        self.n = ddh.size()

    def __del__(self):
        _destroy("cuddh_b200_ddh_dist_destroy", self)

    def size(self):
        return self.n

    def info(self):
        v = np.zeros(8, np.int64)
        check(load().cuddh_b200_ddh_dist_info(self._h, _vp(v)))
        keys = ["dom_begin", "dom_end", "n_owned", "n_send", "n_recv", "n_peers", "bytes_per_action", "size"]
        return {k: int(x) for k, x in zip(keys, v)}

    def array(self, name):
        cnt = C.c_int64()
        check(load().cuddh_b200_ddh_dist_get_array(self._h, name.encode(), None, 0, C.byref(cnt)))
        out = np.zeros(cnt.value, np.int32)
        check(load().cuddh_b200_ddh_dist_get_array(self._h, name.encode(), _vp(out), out.size, C.byref(cnt)))
        return out

    def mask(self):
        """uint8 CUDA tensor view (length size()) of the library's ownership mask"""
        import torch
        p = load().cuddh_b200_ddh_dist_mask(self._h)
        if not p:
            check(-1)

        class _Raw:
            __cuda_array_interface__ = {"shape": (self.n,), "typestr": "|u1", "data": (int(p), False), "version": 2}
        t = torch.as_tensor(_Raw(), device="cuda")
        t._keepalive = self
        return t

    def buffers(self):
        """(send, recv) raw device addresses of the packed (lambda, mu) pair buffers (tests)"""
        a, b = C.c_void_p(), C.c_void_p()
        check(load().cuddh_b200_ddh_dist_buffers(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def rhs(self, f, b):
        check(load().cuddh_b200_ddh_dist_rhs(self._h, _ptr(f), _ptr(b), _stream()))

    def action(self, x, y):
        check(load().cuddh_b200_ddh_dist_action(self._h, _ptr(x), _ptr(y), _stream()))

    def apply_T(self, x, t):
        check(load().cuddh_b200_ddh_dist_apply_T(self._h, _ptr(x), _ptr(t), _stream()))

    def postprocess(self, lam, f, u):
        check(load().cuddh_b200_ddh_dist_postprocess(self._h, _ptr(lam), _ptr(f), _ptr(u), _stream()))

    def _as_apply(self):
        return C.cast(load().cuddh_b200_ddh_dist_as_apply, C.c_void_p), self._h

    def solve(self, b, x, m=20, maxit=100, tol=1e-4, orth=-1, time_orth=False):
        """distributed FP32 GMRES in the library: masked inner products, one NCCL allreduce per pass"""
        return gmres(self.n, x, self, b, m, maxit, tol, orth=orth, comm=self.comm, mask=self.mask(), time_orth=time_orth)


# include/linalg.hpp
def _lin(name, *a):
    check(getattr(load(), name)(*a))


def dot(n, x, y):
    import torch
    if x.dtype == torch.float32:
        r = C.c_float()
        _lin("cuddh_b200_dot_f", n, _ptr(x), _ptr(y), C.byref(r), _stream())
    else:
        r = C.c_double()
        _lin("cuddh_b200_dot_d", n, _ptr(x), _ptr(y), C.byref(r), _stream())
    return r.value


def norm(n, x):
    return float(np.sqrt(dot(n, x, x)))


def dist(n, x, y):
    import torch
    if x.dtype == torch.float32:
        r = C.c_float()
        _lin("cuddh_b200_dist_f", n, _ptr(x), _ptr(y), C.byref(r), _stream())
    else:
        r = C.c_double()
        _lin("cuddh_b200_dist_d", n, _ptr(x), _ptr(y), C.byref(r), _stream())
    return r.value


def _suffix(x):
    import torch
    return {torch.float64: "d", torch.float32: "f", torch.int32: "i"}[x.dtype]


def axpby(n, a, x, b, y):
    _lin("cuddh_b200_axpby_" + _suffix(x), n, a, _ptr(x), b, _ptr(y), _stream())


def copy(n, x, y):
    _lin("cuddh_b200_copy_" + _suffix(x), n, _ptr(x), _ptr(y), _stream())


def scal(n, a, x):
    _lin("cuddh_b200_scal_" + _suffix(x), n, a, _ptr(x), _stream())


def fill(n, a, x):
    _lin("cuddh_b200_fill_" + _suffix(x), n, a, _ptr(x), _stream())


def launch_count():
    return int(load().cuddh_b200_launch_count())
