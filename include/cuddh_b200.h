/* cuddh_b200.h — C ABI of libcuddh_b200.so: the B200 (sm_100a) implementation of CuDDHelmholtz's solve path.
 *
 * This is the drop-in boundary. Every entry point states the reference interface it replaces
 * (file:line relative to the reference tree). Conventions, all taken from the reference:
 *   - every `const double*` / `double*` / `float*` vector argument named x, y, b, u, f, lambda is a DEVICE
 *     pointer (include/gmres.hpp:25-33, include/H1Space.hpp:112-126); arrays named h_* or documented "host"
 *     are HOST pointers;
 *   - arrays are column-major, first index fastest (include/Tensor.hpp:31-47);
 *   - x and y of an action must not alias.
 * Differences by design: explicit stream argument (a cudaStream_t passed as void*; NULL = legacy default
 * stream, which is what the reference always uses), 64-bit sizes, and status codes instead of abort():
 * every function returns 0 on success or a non-zero code, with the text available from
 * cuddh_b200_last_error(). The C++ classes in cuddhelmholtz_b200/cxx map non-zero to cuddh_error().
 *
 * No torch / C++ types cross this boundary.
 */
#ifndef CUDDH_B200_H
#define CUDDH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cuddh_mesh_s * cuddh_mesh_t;
typedef struct cuddh_basis_s * cuddh_basis_t;
typedef struct cuddh_h1space_s * cuddh_h1space_t;
typedef struct cuddh_facespace_s * cuddh_facespace_t;
typedef struct cuddh_operator_s * cuddh_operator_t;   /* any FP64 operator: y (+)= c*A*x */
typedef struct cuddh_ddh_s * cuddh_ddh_t;

#define CUDDH_GAUSS_LEGENDRE 0
#define CUDDH_GAUSS_LOBATTO 1

/* ---- library ------------------------------------------------------------------------------------ */
int cuddh_b200_version(void);
const char * cuddh_b200_last_error(void);
/* number of kernels launched by this library since load (bench.py's gpu_launches) */
int64_t cuddh_b200_launch_count(void);

/* ---- 1-D tables: QuadratureRule(n, type) include/QuadratureRule.hpp:31 ; Basis(n) include/Basis.hpp:16 --- */
int cuddh_b200_quadrature(int n, int type, double * h_x, double * h_w);
int cuddh_b200_basis_create(int n, cuddh_basis_t * out);
int cuddh_b200_basis_destroy(cuddh_basis_t b);
/* Basis::eval / Basis::deriv (include/Basis.hpp:30,37): P, D have shape (m, n) column-major, host */
int cuddh_b200_basis_eval(cuddh_basis_t b, int m, const double * h_x, double * h_P);
int cuddh_b200_basis_deriv(cuddh_basis_t b, int m, const double * h_x, double * h_D);
int cuddh_b200_basis_nodes(cuddh_basis_t b, double * h_x, double * h_w);   /* Basis::quadrature() */

/* ---- Mesh2D: include/Mesh2D.hpp:266-277 --------------------------------------------------------- */
int cuddh_b200_mesh_uniform_rect(int nx, double ax, double bx, int ny, double ay, double by, cuddh_mesh_t * out);
int cuddh_b200_mesh_from_vertices(int64_t nv, const double * h_xy /* (2,nv) */, int64_t nel, const int * h_elems /* (4,nel) */,
                                  cuddh_mesh_t * out);
int cuddh_b200_mesh_destroy(cuddh_mesh_t m);
/* sizes[0..4] = n_elem, n_nodes, n_edges, n_boundary_edges, n_interior_edges (Mesh2D::n_elem/n_nodes/n_edges) */
int cuddh_b200_mesh_sizes(cuddh_mesh_t m, int64_t * sizes);
/* (8, n_edges) records: nodes[0], nodes[1], elements[0], elements[1], sides[0], sides[1], delta, is_boundary
 * (include/Edge.hpp:25-52; elements[1]/sides[1] = -1 on the boundary) */
int cuddh_b200_mesh_edges(cuddh_mesh_t m, int * h_edges);
int cuddh_b200_mesh_boundary_edges(cuddh_mesh_t m, int * h_list);     /* Mesh2D::boundary_edges() */
int cuddh_b200_mesh_h(cuddh_mesh_t m, double * min_h, double * max_h); /* Mesh2D::min_h / max_h */
int cuddh_b200_mesh_vertices(cuddh_mesh_t m, double * h_xy /* (2, n_nodes) */);
int cuddh_b200_mesh_elements(cuddh_mesh_t m, int * h_elems /* (4, n_elem) */);

/* ---- H1Space: include/H1Space.hpp:21-65 --------------------------------------------------------- */
int cuddh_b200_h1space_create(cuddh_mesh_t mesh, int n_basis, cuddh_h1space_t * out);
int cuddh_b200_h1space_destroy(cuddh_h1space_t s);
int64_t cuddh_b200_h1space_size(cuddh_h1space_t s);                       /* H1Space::size() */
/* host-only self check of the deterministic assembly plan behind Operator::action (replaces the atomicAdd scatter of
 * source/StiffnessMatrix.cpp:174-182): plays gather + assembly with integer-valued element contributions and compares with the
 * direct sum over global_indices. node_major: 1 = thread-per-element plan (n_basis <= 5 kernels), 0 = element-major plan.
 * stats[8] = n_patches, elements per patch, listed patch DOFs, shared DOFs, max DOFs per patch, DOFs with more than four
 * contributions, MISMATCHES (0 = ok), FNV-1a hash of all plan arrays. Needs no GPU. */
int cuddh_b200_h1space_check_plan(cuddh_h1space_t s, int node_major, int64_t * stats);
int cuddh_b200_h1space_global_indices(cuddh_h1space_t s, int * h_I);      /* (nb,nb,n_elem) host copy */
int cuddh_b200_h1space_physical_coordinates(cuddh_h1space_t s, double * h_xy); /* (2,ndof) host copy */
const int * cuddh_b200_h1space_device_indices(cuddh_h1space_t s);         /* global_indices(DEVICE) */
const double * cuddh_b200_h1space_device_coordinates(cuddh_h1space_t s);  /* physical_coordinates(DEVICE) */

/* raw views used by the C++ header layer (valid while the handle lives): global_indices(HOST), physical_coordinates(HOST),
 * and the (8, n_elem) corner coordinates on the device */
const int * cuddh_b200_h1space_host_indices(cuddh_h1space_t s);
const double * cuddh_b200_h1space_host_coordinates(cuddh_h1space_t s);
const double * cuddh_b200_h1space_device_corners(cuddh_h1space_t s);
/* Mesh2D::ElementMetricCollection::{jacobians, measures, physical_coordinates}(DEVICE) (include/Mesh2D.hpp:33-41) on the
 * tensor grid of the n_quad points h_xq: which = 0 -> J (2,2,nq,nq,nel), 1 -> detJ (nq,nq,nel), 2 -> x (2,nq,nq,nel) */
int cuddh_b200_element_metrics(cuddh_h1space_t s, int n_quad, const double * h_xq, int which, double * d_out, void * stream);
/* LinearFunctional::action (include/LinearFunctional.hpp:145-181): F += c * sum_e P^T g_e P scattered through the global map in a
 * fixed order; d_g = w_i w_j detJ f(x_ij) on (nq,nq,nel). h_P == NULL: the "fast" collocated rule, d_g is (nb,nb,nel). */
int cuddh_b200_linear_functional_assemble(cuddh_h1space_t s, int n_quad, const double * h_P, const double * d_g, double c, double * d_F,
                                          void * stream);

/* ---- FaceSpace: include/H1Space.hpp:69-147 ------------------------------------------------------ */
int cuddh_b200_facespace_create(cuddh_h1space_t s, int64_t n_faces, const int * h_faces, cuddh_facespace_t * out);
int cuddh_b200_facespace_destroy(cuddh_facespace_t f);
int64_t cuddh_b200_facespace_size(cuddh_facespace_t f);
int cuddh_b200_facespace_subspace_indices(cuddh_facespace_t f, int * h_I);   /* (nb, n_faces) */
int cuddh_b200_facespace_global_indices(cuddh_facespace_t f, int * h_proj);  /* (fdof) */
const int * cuddh_b200_facespace_indices_ptr(cuddh_facespace_t f, int which /* 0 subspace_indices, 1 global_indices, 2 faces */,
                                             int device);
int64_t cuddh_b200_facespace_n_faces(cuddh_facespace_t f);
/* FaceLinearFunctional::action (include/FaceLinearFunctional.hpp:130-164): F += c * sum_f P^T g_f, d_g (nq, n_faces); h_P NULL = collocated */
int cuddh_b200_face_linear_functional_assemble(cuddh_facespace_t f, int n_quad, const double * h_P, const double * d_g, double c,
                                               double * d_F, void * stream);
int cuddh_b200_facespace_restrict(cuddh_facespace_t f, const double * x, double * y, void * stream); /* y[i] = x[proj[i]] */
int cuddh_b200_facespace_prolong(cuddh_facespace_t f, const double * x, double * y, void * stream);  /* y[proj[i]] += x[i] */
int cuddh_b200_facespace_orth(cuddh_facespace_t f, double * x, void * stream);                        /* x[proj[i]] = 0 */

/* ---- operators: Operator::action include/Operator.hpp:12-16 ------------------------------------- */
/* StiffnessMatrix(fem) / StiffnessMatrix(fem, quad): include/StiffnessMatrix.hpp:14-15. n_quad <= 0 -> n_basis + 1 Gauss-Legendre */
int cuddh_b200_stiffness_create(cuddh_h1space_t s, int n_quad, int quad_type, cuddh_operator_t * out);
/* MassMatrix(fem) / MassMatrix(a, fem): include/MassMatrix.hpp:19-24. d_a: DEVICE nodal coefficient or NULL; n_quad <= 0 -> reference default */
int cuddh_b200_mass_create(cuddh_h1space_t s, const double * d_a, int n_quad, cuddh_operator_t * out);
/* DiagInvMassMatrix(fem) / (a, fem): include/MassMatrix.hpp:47-54 */
int cuddh_b200_diag_inv_mass_create(cuddh_h1space_t s, const double * d_a, cuddh_operator_t * out);
/* FaceMassMatrix(fs) / (a, fs): include/FaceMassMatrix.hpp ; vectors are FaceSpace vectors */
int cuddh_b200_facemass_create(cuddh_facespace_t f, const double * d_a, int n_quad, cuddh_operator_t * out);
int cuddh_b200_diag_inv_facemass_create(cuddh_facespace_t f, const double * d_a, cuddh_operator_t * out);
/* the Helmholtz composite of examples/Helmholtz.hpp:10-80 on x = [u; v] (length 2*ndof) */
int cuddh_b200_helmholtz_create(double omega, const double * d_a2, const double * d_a, cuddh_h1space_t s, cuddh_facespace_t f,
                                cuddh_operator_t * out);
/* y <- (accumulate ? y : 0) + c * A * x.  action(c,x,y) == apply(op,c,1,..); action(x,y) == apply(op,1.0,0,..) */
int cuddh_b200_operator_apply(cuddh_operator_t op, double c, int accumulate, const double * x, double * y, void * stream);
/* fused FaceSpace::restrict + FaceMassMatrix::action + FaceSpace::prolong on H1 vectors: y[proj] += c*H*x[proj] */
int cuddh_b200_facemass_apply_h1(cuddh_operator_t op, double c, const double * x, double * y, void * stream);
/* measurement aid (bench.py roofline): MEDIAN CUDA-event time over `reps` (<= 256) repetitions on `stream`, after three warm
 * applies, of the patch kernel alone and of the rest of the action alone (stiffness / mass handles: the shared-DOF assembly pass; Helmholtz
 * handles on the fused path: shared-DOF assembly + face terms; computes y = A x) */
int cuddh_b200_operator_time_phases(cuddh_operator_t op, const double * x, double * y, int reps, float * ms_patch, float * ms_shared,
                                    void * stream);
int cuddh_b200_operator_destroy(cuddh_operator_t op);
/* algorithmic bytes of one apply (SURVEY §8d), 0 if not defined for this operator */
int64_t cuddh_b200_operator_bytes(cuddh_operator_t op);
/* the same count for the formulation the handle actually runs: on meshes whose elements are all parallelograms (every
 * Mesh2D::uniform_rect) the stiffness metric is w_i w_j times three per-element constants, recomputed in registers instead of
 * streamed (24 instead of 24 nq^2 bytes per element; SURVEY §8(f) rank 1). bench.py reports both rooflines.
 * CUDDH_B200_AFFINE=0 in the environment forces the stored-metric kernels. */
int64_t cuddh_b200_operator_bytes_moved(cuddh_operator_t op);
int cuddh_b200_operator_is_affine(cuddh_operator_t op);
/* which kernel family serves this handle: 0 = lane-per-row patch kernel / generic, 1 = warp-specialised thread-per-element
 * kernel (n_basis <= 5), 2 = Helmholtz handle on the fused S - w^2 M path, 3 = warp-specialised thread-pair-per-element kernel
 * (n_basis 6-9); -1 = not a volume operator */
int cuddh_b200_operator_kernel_kind(cuddh_operator_t op);

/* ---- linalg: include/linalg.hpp:16-54 (double and float) ---------------------------------------- */
int cuddh_b200_axpby_d(int64_t n, double a, const double * x, double b, double * y, void * stream);
int cuddh_b200_axpby_f(int64_t n, float a, const float * x, float b, float * y, void * stream);
int cuddh_b200_dot_d(int64_t n, const double * x, const double * y, double * h_result, void * stream);
int cuddh_b200_dot_f(int64_t n, const float * x, const float * y, float * h_result, void * stream);
int cuddh_b200_dist_d(int64_t n, const double * x, const double * y, double * h_result, void * stream);
int cuddh_b200_dist_f(int64_t n, const float * x, const float * y, float * h_result, void * stream);
int cuddh_b200_copy_d(int64_t n, const double * x, double * y, void * stream);
int cuddh_b200_copy_f(int64_t n, const float * x, float * y, void * stream);
int cuddh_b200_copy_i(int64_t n, const int * x, int * y, void * stream);
int cuddh_b200_scal_d(int64_t n, double a, double * x, void * stream);
int cuddh_b200_scal_f(int64_t n, float a, float * x, void * stream);
int cuddh_b200_fill_d(int64_t n, double a, double * x, void * stream);
int cuddh_b200_fill_f(int64_t n, float a, float * x, void * stream);
int cuddh_b200_fill_i(int64_t n, int a, int * x, void * stream);

/* ---- gmres: include/gmres.hpp:14-36 ------------------------------------------------------------- */
/* Operator callback: must enqueue y = A x (device pointers) on `stream` (the stream gmres itself runs its vector kernels on)
 * and return 0; a non-zero return aborts the solve, which then returns that status. */
typedef int (*cuddh_apply_d_fn)(void * ctx, const double * x, double * y, void * stream);
typedef int (*cuddh_apply_f_fn)(void * ctx, const float * x, float * y, void * stream);
typedef struct
{
    int success;      /* solver_out.success */
    int num_iter;     /* solver_out.num_iter */
    int num_matvec;   /* solver_out.num_matvec */
    int n_res;        /* entries written to res_norm / time (<= cap) */
} cuddh_solver_out;
/* P == NULL: gmres(n,x,A,b,m,maxit,tol,verbose,max_seconds); otherwise the left-preconditioned overload.
 * res_norm / time: HOST arrays of capacity `cap` (>= maxit+1 to get everything) or NULL. */
int cuddh_b200_gmres_d(int64_t n, double * x, cuddh_apply_d_fn A, void * A_ctx, const double * b, cuddh_apply_d_fn P, void * P_ctx,
                       int m, int maxit, double tol, int verbose, double max_seconds, cuddh_solver_out * out, double * h_res_norm,
                       double * h_time, int cap, void * stream);
int cuddh_b200_gmres_f(int64_t n, float * x, cuddh_apply_f_fn A, void * A_ctx, const float * b, int m, int maxit, float tol,
                       int verbose, double max_seconds, cuddh_solver_out * out, double * h_res_norm, double * h_time, int cap,
                       void * stream);
/* convenience trampolines so that a cuddh_operator_t / cuddh_ddh_t can be handed to gmres without a host callback */
int cuddh_b200_operator_as_apply(void * op_handle, const double * x, double * y, void * stream);
int cuddh_b200_ddh_as_apply(void * ddh_handle, const float * x, float * y, void * stream);

/* ---- communicator: one process per GPU (new: the reference is single-GPU). NCCL is bound at run time (dlopen). ---- */
typedef struct cuddh_comm_s * cuddh_comm_t;
/* 128-byte ncclUniqueId: call on one rank, hand the bytes to every rank through the host bootstrap (MPI_Bcast, torch.distributed, ...) */
int cuddh_b200_comm_unique_id(unsigned char * id128);
/* ncclCommInitRank on the current device (collective over the `world` ranks) */
int cuddh_b200_comm_create(const unsigned char * id128, int rank, int world, cuddh_comm_t * out);
/* adopt a caller-owned ncclComm_t (not destroyed with the handle) */
int cuddh_b200_comm_wrap(void * nccl_comm, int rank, int world, cuddh_comm_t * out);
int cuddh_b200_comm_destroy(cuddh_comm_t c);
int cuddh_b200_comm_allreduce_d(cuddh_comm_t c, double * d_buf, int64_t count, void * stream); /* in-place sum, stream-ordered */

/* gmres with options: orthogonalisation mode, distributed vectors.
 *   orth   0 = modified Gram-Schmidt: the reference's arithmetic (source/gmres.cpp:167-172), one fused kernel per basis vector;
 *          1 = classical Gram-Schmidt: all inner products in one pass + one update pass, second round on cancellation;
 *         -1 = library default (set_option "gmres_orth", initially 0).
 *   comm / d_mask: vectors are distributed over the ranks of `comm`; inner products count the entries with d_mask[i] != 0
 *          (device array of n bytes: 1 = this rank owns entry i) and are summed with one ncclAllReduce per pass. */
typedef struct
{
    int orth;
    cuddh_comm_t comm;
    const unsigned char * d_mask;
    int time_orth; /* != 0: record the device time of the orthogonalisation kernels (stats.orth_ms) */
    int flexible;  /* gmres_d_ex with P != NULL: 0 = the reference's left preconditioning (solve P A x = P b, source/gmres.cpp:68-89);
                      1 = flexible RIGHT preconditioning (FGMRES): z_k = P v_k stored, true residuals of A x = b, and P may be an
                      inner iterative solve (e.g. the DDH solve as preconditioner of the FP64 Helmholtz system) */
} cuddh_gmres_options;
typedef struct
{
    double orth_bytes; /* vector bytes moved by the orthogonalisation kernels */
    double orth_ms;    /* their device time (time_orth) */
    int reorth;        /* orth 1: second rounds taken */
    int allreduces;
} cuddh_gmres_stats;
int cuddh_b200_gmres_d_ex(int64_t n, double * x, cuddh_apply_d_fn A, void * A_ctx, const double * b, cuddh_apply_d_fn P, void * P_ctx,
                          int m, int maxit, double tol, int verbose, double max_seconds, const cuddh_gmres_options * opts,
                          cuddh_solver_out * out, double * h_res_norm, double * h_time, int cap, cuddh_gmres_stats * stats, void * stream);
int cuddh_b200_gmres_f_ex(int64_t n, float * x, cuddh_apply_f_fn A, void * A_ctx, const float * b, int m, int maxit, float tol,
                          int verbose, double max_seconds, const cuddh_gmres_options * opts, cuddh_solver_out * out, double * h_res_norm,
                          double * h_time, int cap, cuddh_gmres_stats * stats, void * stream);

/* ---- path A across GPUs (new; SURVEY §8e): one slab of element rows per rank ----------------------------------------
 * A rank holds every DOF its elements touch; the node row on a slab interface is mirrored by both neighbours. h_bottom / h_top:
 * slab-local DOF indices of the interface row shared with rank-1 / rank+1, in the same order on both sides (increasing x);
 * n_bottom == 0 on rank 0, n_top == 0 on the last rank. fs_phys: the FaceSpace of the PHYSICAL boundary of this slab (the one
 * the Helmholtz handle was built with) or NULL. apply_slab = local apply + interface rows packed inside the face-mass launch +
 * one grouped ncclSend/ncclRecv + add (4 launches); own + received is the same commutative sum on both sides -> mirrored rows
 * stay bitwise identical. slab_mask: 1 = owned (the lower rank owns a mirrored row) for cuddh_b200_gmres_d_ex. */
typedef struct cuddh_slab_s * cuddh_slab_t;
int cuddh_b200_slab_create(cuddh_comm_t comm, int rank, int world, cuddh_h1space_t s, cuddh_facespace_t fs_phys, int64_t n_bottom,
                           const int * h_bottom, int64_t n_top, const int * h_top, cuddh_slab_t * out);
int cuddh_b200_slab_destroy(cuddh_slab_t h);
int64_t cuddh_b200_slab_bytes(cuddh_slab_t h);                                   /* bytes sent per apply */
/* 1: the interface rows travel as NVLink stores into the neighbours' receive buffers (CUDA IPC mappings made at create time) with an
 * epoch flag (release / acquire at system scope) - no NCCL call on the data path; 0: grouped ncclSend / ncclRecv (CUDDH_B200_PEER=0, or
 * some rank could not map its neighbours). The exchanges of ONE slab handle must be stream-ordered (two receive buffers alternate);
 * requests kept in flight on several streams need one slab handle each. */
int cuddh_b200_slab_uses_peer_memory(cuddh_slab_t h);
int cuddh_b200_slab_exchange(cuddh_slab_t h, double * y, void * stream);         /* y[rows] += neighbours' y[rows], y = [u; v] */
const unsigned char * cuddh_b200_slab_mask(cuddh_slab_t h);                      /* DEVICE, 2*ndof bytes */
int cuddh_b200_helmholtz_apply_slab(cuddh_operator_t op, cuddh_slab_t h, const double * x, double * y, void * stream);
int cuddh_b200_slab_bind(cuddh_slab_t h, cuddh_operator_t helmholtz);            /* operator behind slab_as_apply (not owned) */
int cuddh_b200_slab_as_apply(void * slab_handle, const double * x, double * y, void * stream); /* cuddh_apply_d_fn */

/* ---- tuning / test knobs -------------------------------------------------------------------------
 * "gmres_orth": default orthogonalisation of gmres (0 MGS, 1 CGS2);
 * "max_ctas":   upper bound on the CTAs of the persistent operator kernels (0 = one full wave; tests use a small value to
 *               force many patches per CTA on small meshes);
 * get_option also answers "nccl_available". Unknown names: set returns non-zero, get returns -1. */
int cuddh_b200_set_option(const char * name, int64_t value);
int64_t cuddh_b200_get_option(const char * name);

/* ---- EnsembleSpace: include/EnsembleSpace.hpp:13-140 (host index maps of a labelled decomposition) ------------- */
typedef struct cuddh_ensemble_s * cuddh_ensemble_t;
int cuddh_b200_ensemble_create(cuddh_h1space_t s, int n_spaces, const int * h_labels, cuddh_ensemble_t * out);
int cuddh_b200_ensemble_destroy(cuddh_ensemble_t e);
/* info[0..5] = n_spaces, mx_elems, mx_faces, mx_ndof, mx_fdof, n_shared */
int cuddh_b200_ensemble_info(cuddh_ensemble_t e, int64_t * info);
/* "gI","sizes","elements","n_elems","faces","n_faces","sI","fI","pI","fsizes","cmap": pointer to the host array + element count */
const int * cuddh_b200_ensemble_array(cuddh_ensemble_t e, const char * name, int64_t * count);

/* ---- DDH: include/DDH.hpp:21-84 ----------------------------------------------------------------- */
/* DDH(omega, h_a, fem, nx, ny): h_a HOST nodal coefficient (length ndof). block = 1-D node size of a subdomain
 * (the reference's compile-time DDH_BLOCK_SIZE, source/DDH.cpp:5): 16 or 32. */
int cuddh_b200_ddh_create(double omega, const double * h_a, cuddh_h1space_t s, int nx, int ny, int block, cuddh_ddh_t * out);
int cuddh_b200_ddh_destroy(cuddh_ddh_t d);
int64_t cuddh_b200_ddh_size(cuddh_ddh_t d);                                    /* DDH::size() = 2*n_lambda */
int cuddh_b200_ddh_rhs(cuddh_ddh_t d, const double * f, float * b, void * stream);                 /* DDH::rhs */
int cuddh_b200_ddh_action(cuddh_ddh_t d, const float * x, float * y, void * stream);               /* DDH::action */
int cuddh_b200_ddh_postprocess(cuddh_ddh_t d, const float * lambda, const double * f, double * u, void * stream); /* DDH::postprocess */
/* Multi-GPU sharding of the subdomain loop (new: the reference is single-GPU). Rank r runs subdomains [dom_begin, dom_end):
 * t = T(x) (resp. b, u) restricted to the slots / DOFs those subdomains write, zero elsewhere, so that a sum-allreduce over the
 * ranks reproduces T(x), rhs and postprocess; DDH::action is then x - allreduce(t). */
int cuddh_b200_ddh_apply_T_range(cuddh_ddh_t d, const float * x, float * t, int dom_begin, int dom_end, void * stream);
int cuddh_b200_ddh_rhs_range(cuddh_ddh_t d, const double * f, float * b, int dom_begin, int dom_end, void * stream);
int cuddh_b200_ddh_postprocess_range(cuddh_ddh_t d, const float * lambda, const double * f, double * u, int dom_begin, int dom_end,
                                     void * stream);
/* introspection for parity tests: info[0..7] = n_domains, n_shared, nt, mx_dof, mx_fdof, mx_elem_per_dom, n_basis, block ; dt */
int cuddh_b200_ddh_info(cuddh_ddh_t d, int64_t * info, double * dt);
/* host copies of the index / coefficient arrays in the reference's layouts (names as in source/DDH.cpp):
 * "B" (mx_fdof,2,dom) int, "gI" (mx_dof,dom) int, "sI" (nb,nb,mx_elem,dom) int, "cmap" (4,n_shared) int,
 * "m","gmi","a" (mx_dof,dom) float, "H" (mx_fdof,dom) float, "wh_filter" (nt+1) float. Returns element count in *count. */
int cuddh_b200_ddh_get_array(cuddh_ddh_t d, const char * name, void * h_out, int64_t cap_bytes, int64_t * count);
/* algorithmic FP32 flops of one action (BASELINE.md §3) */
double cuddh_b200_ddh_flops(cuddh_ddh_t d);
/* which kernel serves this handle: 1 = register-tiled thread-per-element kernel (n_basis 4, block 16, uniform metric), 0 = generic */
int cuddh_b200_ddh_kernel_kind(cuddh_ddh_t d);

/* ---- DDH across GPUs (new; SURVEY §8e path B): subdomain row slabs, one per rank --------------------------------
 * Vectors keep the global length DDH::size(); a lambda slot is OWNED by the rank of the subdomain that reads it and is zero
 * on every other rank (use cuddh_b200_ddh_dist_mask as d_mask of cuddh_b200_gmres_f_ex). rhs / action run this rank's
 * subdomains; traces written for a slot another rank owns leave the kernel through a packed send buffer (pack fused into
 * the kernel epilogue) and travel with one grouped ncclSend/ncclRecv per neighbour on `stream`.
 * comm == NULL: partition tables only (host; for tests) or a single rank. */
typedef struct cuddh_ddh_dist_s * cuddh_ddh_dist_t;
int cuddh_b200_ddh_dist_create(cuddh_ddh_t d, cuddh_comm_t comm, int rank, int world, cuddh_ddh_dist_t * out);
int cuddh_b200_ddh_dist_destroy(cuddh_ddh_dist_t h);
/* info[0..7] = dom_begin, dom_end, owned slots, slots sent, slots received, neighbours, bytes sent per action, vector length */
int cuddh_b200_ddh_dist_info(cuddh_ddh_dist_t h, int64_t * info);
/* host tables: "owner" (n_lambda), "send_idx", "recv_idx" (grouped by peer), "segments" (5, neighbours): peer, send_off,
 * send_count, recv_off, recv_count in (lambda, mu) pairs */
int cuddh_b200_ddh_dist_get_array(cuddh_ddh_dist_t h, const char * name, int * h_out, int64_t cap, int64_t * count);
const unsigned char * cuddh_b200_ddh_dist_mask(cuddh_ddh_dist_t h);            /* DEVICE, DDH::size() bytes */
int cuddh_b200_ddh_dist_buffers(cuddh_ddh_dist_t h, void ** d_send, void ** d_recv); /* packed (lambda, mu) float pairs; tests */
int cuddh_b200_ddh_dist_rhs(cuddh_ddh_dist_t h, const double * f, float * b, void * stream);
int cuddh_b200_ddh_dist_action(cuddh_ddh_dist_t h, const float * x, float * y, void * stream);
int cuddh_b200_ddh_dist_apply_T(cuddh_ddh_dist_t h, const float * x, float * t, void * stream);
int cuddh_b200_ddh_dist_postprocess(cuddh_ddh_dist_t h, const float * lambda, const double * f, double * u, void * stream);
int cuddh_b200_ddh_dist_as_apply(void * dist_handle, const float * x, float * y, void * stream); /* cuddh_apply_f_fn */

/* ---- assembled DDH interface operator (new): the same linear map as cuddh_b200_ddh_action, stored -----------------------
 * T is block-sparse: subdomain p reads only its incoming (lambda, mu) slots and writes only its outgoing ones, so T is one dense
 * real block M_p of size 2F x 2F per subdomain (F = face DOFs per subdomain, 48 / 56 / 96 / 112 for n_basis 4 / 8 and block 16 /
 * 32). Face position f numbers the boundary ring of the subdomain's DOF grid in ascending grid index Y*n1 + X (the same order in
 * every subdomain); local input / output k < F is the lambda entry of face position k, k >= F the mu entry of position k - F.
 * Creation probes T with 2F WaveHoltz actions (columns are the DDH kernel's own outputs); an action is then one streaming
 * batched matvec (y = x - T x, deterministic, one launch) instead of 5 x nt time steps per subdomain. Memory: n_domains * 4F^2 * 4
 * bytes. The cuddh_ddh_t handle must outlive the transfer handle. */
typedef struct cuddh_ddh_transfer_s * cuddh_ddh_transfer_t;
/* host only (no GPU needed): slot maps (2F, n_domains) column-major, entry k + 2F p = slot read (h_in) / written (h_out) by
 * local input / output k of subdomain p, -1 on the physical boundary. cap: capacity of each array in ints; with h_in == h_out ==
 * NULL only *two_f is returned. Fails unless every slot has at most one reader and at most one writer. */
int cuddh_b200_ddh_transfer_slots(cuddh_ddh_t d, int * h_in, int * h_out, int64_t cap, int * two_f);
/* host only: ascending slots of [0, DDH::size()) that no subdomain writes (orphans: y = x there); h_out == NULL -> count only */
int cuddh_b200_ddh_transfer_orphans(cuddh_ddh_t d, int * h_out, int64_t cap, int64_t * count);
/* probes the blocks, synchronous on `stream`. max_bytes: device memory the handle may take, 0 = what cudaMemGetInfo reports free;
 * if blocks + maps + probe vectors do not fit, fails with a message naming the bytes needed */
int cuddh_b200_ddh_transfer_create(cuddh_ddh_t d, int64_t max_bytes, void * stream, cuddh_ddh_transfer_t * out);
int cuddh_b200_ddh_transfer_destroy(cuddh_ddh_transfer_t h);
int cuddh_b200_ddh_transfer_action(cuddh_ddh_transfer_t h, const float * x, float * y, void * stream); /* y = x - T x; no overlap */
int cuddh_b200_ddh_transfer_as_apply(void * transfer_handle, const float * x, float * y, void * stream); /* cuddh_apply_f_fn */
/* info[0..5] = n_domains, 2F, block bytes, bytes moved per action, probe launches, probe time in microseconds */
int cuddh_b200_ddh_transfer_info(cuddh_ddh_transfer_t h, int64_t * info);
/* host copy of M_dom: (2F, 2F) column-major floats */
int cuddh_b200_ddh_transfer_get_block(cuddh_ddh_transfer_t h, int dom, float * h_out);

/* ---- many right-hand sides at once (new) -------------------------------------------------------------------------------
 * Batched operator callback: must enqueue y[j] = A x[j] for j < k on `stream` and return 0. x, y: HOST arrays of k DEVICE
 * pointers; a non-zero return aborts the solve, which then returns that status. */
typedef int (*cuddh_apply_batch_f_fn)(void * ctx, int k, const float * const * x, float * const * y, void * stream);
/* y[j] = x[j] - T x[j] for j < k, 1 <= k <= 32. Row j is bitwise cuddh_b200_ddh_transfer_action(x[j]); the blocks are streamed once
 * for up to 16 vectors (ceil(k / 16) launches). Fails if any y[j] overlaps any x[i] or another y[i] (n = DDH::size() floats each). */
int cuddh_b200_ddh_transfer_action_batch(cuddh_ddh_transfer_t h, int k, const float * const * x, float * const * y, void * stream);
int cuddh_b200_ddh_transfer_as_apply_batch(void * transfer_handle, int k, const float * const * x, float * const * y,
                                           void * stream); /* cuddh_apply_batch_f_fn */
/* k (1 <= k <= 32) independent FP32 GMRES(m) solves A x[j] = b[j] in lockstep: each Arnoldi step applies A once to the systems still
 * iterating (A is handed only those), orthogonalises them in the same launches and syncs the host once. Modified Gram-Schmidt
 * only (the "gmres_orth" option is not read); no preconditioner, distributed vectors or verbose output. Each system follows the
 * control flow of cuddh_b200_gmres_f with orth 0 and leaves the batch when it converges: its x, residual norms, num_iter and
 * num_matvec are bitwise those of that solve. max_seconds limits the wall time of the whole batch; h_time is measured from its
 * start. x, b: HOST arrays of k device pointers (the x[j] must not overlap). out: k entries or NULL; h_res_norm / h_time: HOST
 * arrays of k * cap doubles (row j at j * cap) or NULL. */
int cuddh_b200_gmres_f_batch(int64_t n, int k, float * const * x, cuddh_apply_batch_f_fn A, void * A_ctx, const float * const * b, int m,
                             int maxit, float tol, double max_seconds, cuddh_solver_out * out, double * h_res_norm, double * h_time,
                             int cap, void * stream);

#ifdef __cplusplus
}
#endif
#endif
