// extern "C" boundary of libcuddh_b200.so (see include/cuddh_b200.h). Every entry point converts C++
// exceptions into a status code + last-error string; nothing throws across the ABI.
#include "../../include/cuddh_b200.h"
#include "aux.hpp"
#include "common.hpp"
#include "ddh.hpp"
#include "linalg.hpp"
#include "operators.hpp"
#include <algorithm>
#include <atomic>
#include <cstring>

namespace cb200
{
    static thread_local std::string g_last_error;
    void set_last_error(const std::string & msg) { g_last_error = msg; }
    const char * get_last_error() { return g_last_error.c_str(); }
    std::atomic<int64_t> g_launches{0};
    int setup_threads()
    {
        static const int n = [] {
            const char * v = getenv("CUDDH_B200_SETUP_THREADS");
            int k = v ? atoi(v) : (int)std::thread::hardware_concurrency();
            return std::max(1, std::min(k, 64));
        }();
        return n;
    }
} // namespace cb200

using namespace cb200;

#define CB_TRY try {
#define CB_CATCH                                                                        \
    }                                                                                   \
    catch (const cb200::Error & e)                                                      \
    {                                                                                   \
        set_last_error(e.what());                                                       \
        return e.code ? e.code : -1;                                                    \
    }                                                                                   \
    catch (const std::exception & e)                                                    \
    {                                                                                   \
        set_last_error(e.what());                                                       \
        return -2;                                                                      \
    }                                                                                   \
    return 0;

struct cuddh_mesh_s { std::unique_ptr<Mesh> m; };
struct cuddh_basis_s { std::unique_ptr<Basis> b; };
struct cuddh_h1space_s { std::unique_ptr<H1Space> s; };
struct cuddh_facespace_s { std::unique_ptr<FaceSpace> f; };
struct cuddh_operator_s
{
    std::unique_ptr<VolumeOp> vol;
    std::unique_ptr<DiagOp> diag;
    std::unique_ptr<FaceMassOp> face;
    std::unique_ptr<HelmholtzOp> helm;
};
struct cuddh_ddh_s { std::unique_ptr<DDH> d; };
struct cuddh_ensemble_s { std::unique_ptr<Ensemble> e; };
struct cuddh_comm_s { std::unique_ptr<Comm> c; };
struct cuddh_ddh_dist_s { std::unique_ptr<DdhDist> d; };
struct cuddh_slab_s { std::unique_ptr<SlabHalo> h; };
struct cuddh_ddh_transfer_s { std::unique_ptr<DDHTransfer> t; };

static inline cudaStream_t S(void * s) { return (cudaStream_t)s; }

extern "C" {

int cuddh_b200_version(void) { return 100; }
const char * cuddh_b200_last_error(void) { return get_last_error(); }
int64_t cuddh_b200_launch_count(void) { return g_launches.load(); }

// ---- tables ----
int cuddh_b200_quadrature(int n, int type, double * x, double * w)
{
    CB_TRY
    CB_REQUIRE(type == CUDDH_GAUSS_LEGENDRE || type == CUDDH_GAUSS_LOBATTO, "unknown quadrature type");
    quadrature_rule(n, type, x, w);
    CB_CATCH
}
int cuddh_b200_basis_create(int n, cuddh_basis_t * out)
{
    CB_TRY
    *out = new cuddh_basis_s{std::unique_ptr<Basis>(new Basis(n))};
    CB_CATCH
}
int cuddh_b200_basis_destroy(cuddh_basis_t b)
{
    delete b;
    return 0;
}
int cuddh_b200_basis_eval(cuddh_basis_t b, int m, const double * x, double * P)
{
    CB_TRY
    b->b->eval(m, x, P);
    CB_CATCH
}
int cuddh_b200_basis_deriv(cuddh_basis_t b, int m, const double * x, double * D)
{
    CB_TRY
    b->b->deriv(m, x, D);
    CB_CATCH
}
int cuddh_b200_basis_nodes(cuddh_basis_t b, double * x, double * w)
{
    CB_TRY
    std::memcpy(x, b->b->x.data(), sizeof(double) * b->b->n);
    std::memcpy(w, b->b->w.data(), sizeof(double) * b->b->n);
    CB_CATCH
}

// ---- mesh ----
int cuddh_b200_mesh_uniform_rect(int nx, double ax, double bx, int ny, double ay, double by, cuddh_mesh_t * out)
{
    CB_TRY
    *out = new cuddh_mesh_s{Mesh::uniform_rect(nx, ax, bx, ny, ay, by)};
    CB_CATCH
}
int cuddh_b200_mesh_from_vertices(int64_t nv, const double * xy, int64_t nel, const int * elems, cuddh_mesh_t * out)
{
    CB_TRY
    *out = new cuddh_mesh_s{Mesh::from_vertices(nv, xy, nel, elems)};
    CB_CATCH
}
int cuddh_b200_mesh_destroy(cuddh_mesh_t m)
{
    delete m;
    return 0;
}
int cuddh_b200_mesh_sizes(cuddh_mesh_t m, int64_t * sizes)
{
    CB_TRY
    sizes[0] = m->m->n_elem;
    sizes[1] = m->m->n_nodes;
    sizes[2] = m->m->n_edges;
    sizes[3] = (int64_t)m->m->boundary_edges.size();
    sizes[4] = (int64_t)m->m->interior_edges.size();
    CB_CATCH
}
int cuddh_b200_mesh_edges(cuddh_mesh_t m, int * e)
{
    CB_TRY
    std::memcpy(e, m->m->edges.data(), sizeof(int) * m->m->edges.size());
    CB_CATCH
}
int cuddh_b200_mesh_boundary_edges(cuddh_mesh_t m, int * l)
{
    CB_TRY
    std::memcpy(l, m->m->boundary_edges.data(), sizeof(int) * m->m->boundary_edges.size());
    CB_CATCH
}
int cuddh_b200_mesh_h(cuddh_mesh_t m, double * min_h, double * max_h)
{
    CB_TRY
    *min_h = m->m->min_h;
    *max_h = m->m->max_h;
    CB_CATCH
}

// ---- H1 space ----
int cuddh_b200_h1space_create(cuddh_mesh_t mesh, int nb, cuddh_h1space_t * out)
{
    CB_TRY
    *out = new cuddh_h1space_s{std::unique_ptr<H1Space>(new H1Space(mesh->m.get(), nb))};
    CB_CATCH
}
int cuddh_b200_h1space_destroy(cuddh_h1space_t s)
{
    delete s;
    return 0;
}
int64_t cuddh_b200_h1space_size(cuddh_h1space_t s) { return s->s->ndof; }
int cuddh_b200_h1space_check_plan(cuddh_h1space_t s, int node_major, int64_t * stats)
{
    CB_TRY
    plan_self_check(*s->s, node_major != 0, stats);
    CB_CATCH
}
int cuddh_b200_h1space_global_indices(cuddh_h1space_t s, int * I)
{
    CB_TRY
    std::memcpy(I, s->s->I.data(), sizeof(int) * s->s->I.size());
    CB_CATCH
}
int cuddh_b200_h1space_physical_coordinates(cuddh_h1space_t s, double * xy)
{
    CB_TRY
    std::memcpy(xy, s->s->xy.data(), sizeof(double) * s->s->xy.size());
    CB_CATCH
}
const int * cuddh_b200_h1space_device_indices(cuddh_h1space_t s)
{
    try {
        return s->s->device_I();
    }
    catch (const std::exception & e) {
        set_last_error(e.what());
        return nullptr;
    }
}
const double * cuddh_b200_h1space_device_coordinates(cuddh_h1space_t s)
{
    try {
        return s->s->device_xy();
    }
    catch (const std::exception & e) {
        set_last_error(e.what());
        return nullptr;
    }
}

const int * cuddh_b200_h1space_host_indices(cuddh_h1space_t s) { return s->s->I.data(); }
const double * cuddh_b200_h1space_host_coordinates(cuddh_h1space_t s) { return s->s->xy.data(); }
const double * cuddh_b200_h1space_device_corners(cuddh_h1space_t s)
{
    try {
        return s->s->device_corners();
    }
    catch (const std::exception & e) {
        set_last_error(e.what());
        return nullptr;
    }
}
int cuddh_b200_element_metrics(cuddh_h1space_t s, int nq, const double * h_xq, int which, double * d_out, void * stream)
{
    CB_TRY
    CB_REQUIRE(which >= 0 && which <= 2, "element_metrics: which must be 0, 1 or 2");
    element_metrics(s->s.get(), nq, h_xq, which, d_out, S(stream));
    CB_CATCH
}
int cuddh_b200_linear_functional_assemble(cuddh_h1space_t s, int nq, const double * h_P, const double * d_g, double c, double * d_F,
                                          void * stream)
{
    CB_TRY
    linear_functional_assemble(s->s.get(), nq, h_P, d_g, c, d_F, S(stream));
    CB_CATCH
}
int cuddh_b200_mesh_vertices(cuddh_mesh_t m, double * xy)
{
    CB_TRY
    std::memcpy(xy, m->m->xy.data(), sizeof(double) * m->m->xy.size());
    CB_CATCH
}
int cuddh_b200_mesh_elements(cuddh_mesh_t m, int * el)
{
    CB_TRY
    std::memcpy(el, m->m->elems.data(), sizeof(int) * m->m->elems.size());
    CB_CATCH
}

// ---- face space ----
const int * cuddh_b200_facespace_indices_ptr(cuddh_facespace_t f, int which, int device)
{
    try {
        FaceSpace & F = *f->f;
        if (device) {
            F.ensure_device();
            if (which == 2 && !F.d_faces.p)
                F.d_faces.upload(F.faces);
            return which == 0 ? F.d_I.p : which == 1 ? F.d_proj.p : F.d_faces.p;
        }
        return which == 0 ? F.I.data() : which == 1 ? F.proj.data() : F.faces.data();
    }
    catch (const std::exception & e) {
        set_last_error(e.what());
        return nullptr;
    }
}
int64_t cuddh_b200_facespace_n_faces(cuddh_facespace_t f) { return f->f->n_faces; }
int cuddh_b200_face_linear_functional_assemble(cuddh_facespace_t f, int nq, const double * h_P, const double * d_g, double c, double * d_F,
                                               void * stream)
{
    CB_TRY
    face_linear_functional_assemble(f->f.get(), nq, h_P, d_g, c, d_F, S(stream));
    CB_CATCH
}
int cuddh_b200_facespace_create(cuddh_h1space_t s, int64_t nf, const int * faces, cuddh_facespace_t * out)
{
    CB_TRY
    *out = new cuddh_facespace_s{std::unique_ptr<FaceSpace>(new FaceSpace(s->s.get(), nf, faces))};
    CB_CATCH
}
int cuddh_b200_facespace_destroy(cuddh_facespace_t f)
{
    delete f;
    return 0;
}
int64_t cuddh_b200_facespace_size(cuddh_facespace_t f) { return f->f->fdof; }
int cuddh_b200_facespace_subspace_indices(cuddh_facespace_t f, int * I)
{
    CB_TRY
    std::memcpy(I, f->f->I.data(), sizeof(int) * f->f->I.size());
    CB_CATCH
}
int cuddh_b200_facespace_global_indices(cuddh_facespace_t f, int * p)
{
    CB_TRY
    std::memcpy(p, f->f->proj.data(), sizeof(int) * f->f->proj.size());
    CB_CATCH
}
int cuddh_b200_facespace_restrict(cuddh_facespace_t f, const double * x, double * y, void * stream)
{
    CB_TRY
    face_restrict(f->f.get(), x, y, S(stream));
    CB_CATCH
}
int cuddh_b200_facespace_prolong(cuddh_facespace_t f, const double * x, double * y, void * stream)
{
    CB_TRY
    face_prolong(f->f.get(), x, y, S(stream));
    CB_CATCH
}
int cuddh_b200_facespace_orth(cuddh_facespace_t f, double * x, void * stream)
{
    CB_TRY
    face_orth(f->f.get(), x, S(stream));
    CB_CATCH
}

// ---- operators ----
int cuddh_b200_stiffness_create(cuddh_h1space_t s, int nq, int quad_type, cuddh_operator_t * out)
{
    CB_TRY
    auto * op = new cuddh_operator_s;
    std::unique_ptr<cuddh_operator_s> guard(op);
    op->vol = make_stiffness(s->s.get(), nq, quad_type);
    *out = guard.release();
    CB_CATCH
}
int cuddh_b200_mass_create(cuddh_h1space_t s, const double * d_a, int nq, cuddh_operator_t * out)
{
    CB_TRY
    std::unique_ptr<cuddh_operator_s> op(new cuddh_operator_s);
    op->vol = make_mass(s->s.get(), d_a, nq);
    *out = op.release();
    CB_CATCH
}
int cuddh_b200_diag_inv_mass_create(cuddh_h1space_t s, const double * d_a, cuddh_operator_t * out)
{
    CB_TRY
    std::unique_ptr<cuddh_operator_s> op(new cuddh_operator_s);
    op->diag = make_diag_inv_mass(s->s.get(), d_a);
    *out = op.release();
    CB_CATCH
}
int cuddh_b200_facemass_create(cuddh_facespace_t f, const double * d_a, int nq, cuddh_operator_t * out)
{
    CB_TRY
    std::unique_ptr<cuddh_operator_s> op(new cuddh_operator_s);
    op->face = make_facemass(f->f.get(), d_a, nq);
    *out = op.release();
    CB_CATCH
}
int cuddh_b200_diag_inv_facemass_create(cuddh_facespace_t f, const double * d_a, cuddh_operator_t * out)
{
    CB_TRY
    std::unique_ptr<cuddh_operator_s> op(new cuddh_operator_s);
    op->diag = make_diag_inv_facemass(f->f.get(), d_a);
    *out = op.release();
    CB_CATCH
}
int cuddh_b200_helmholtz_create(double omega, const double * d_a2, const double * d_a, cuddh_h1space_t s, cuddh_facespace_t f,
                                cuddh_operator_t * out)
{
    CB_TRY
    std::unique_ptr<cuddh_operator_s> op(new cuddh_operator_s);
    op->helm = make_helmholtz(omega, d_a2, d_a, s->s.get(), f->f.get());
    *out = op.release();
    CB_CATCH
}
int cuddh_b200_operator_apply(cuddh_operator_t op, double c, int accumulate, const double * x, double * y, void * stream)
{
    CB_TRY
    if (op->vol)
        op->vol->apply(c, accumulate, x, y, S(stream));
    else if (op->diag)
        op->diag->apply(c, accumulate, x, y, S(stream));
    else if (op->face)
        op->face->apply(c, accumulate, x, y, S(stream));
    else if (op->helm) {
        // examples/Helmholtz.hpp:62-65: action(c, x, y) is not implemented by the reference composite
        CB_REQUIRE(!accumulate && c == 1.0, "Helmholtz::action(c, x, y) not implemented");
        op->helm->apply(x, y, S(stream));
    }
    else
        throw Error(-1, "operator_apply: empty operator handle");
    CB_CATCH
}
int cuddh_b200_facemass_apply_h1(cuddh_operator_t op, double c, const double * x, double * y, void * stream)
{
    CB_TRY
    CB_REQUIRE(op->face != nullptr, "facemass_apply_h1: not a FaceMassMatrix handle");
    op->face->apply_h1(c, x, y, S(stream));
    CB_CATCH
}
int cuddh_b200_operator_time_phases(cuddh_operator_t op, const double * x, double * y, int reps, float * ms_patch, float * ms_shared,
                                    void * stream)
{
    CB_TRY
    CB_REQUIRE((op->vol != nullptr || op->helm != nullptr) && reps > 0, "operator_time_phases: needs a stiffness / mass / Helmholtz handle and reps > 0");
    auto run = [&](int phases) {
        if (op->vol)
            op->vol->apply(1.0, 0, x, y, S(stream), phases);
        else
            op->helm->apply(x, y, S(stream), phases);
    };
    // three warm launches, then every repetition is timed on its own (patch kernel | rest of the action) and the MEDIAN over the
    // repetitions is reported: a mean over back-to-back launches drifts with the first cold launches and with clock ramps
    const int R = std::min(reps, 256);
    std::vector<cudaEvent_t> ev((size_t)3 * R);
    for (auto & e : ev)
        CB_CUDA(cudaEventCreate(&e));
    for (int i = 0; i < 3; ++i)
        run(3);
    for (int i = 0; i < R; ++i) {
        CB_CUDA(cudaEventRecord(ev[3 * i], S(stream)));
        run(1);
        CB_CUDA(cudaEventRecord(ev[3 * i + 1], S(stream)));
        run(2);
        CB_CUDA(cudaEventRecord(ev[3 * i + 2], S(stream)));
    }
    CB_CUDA(cudaEventSynchronize(ev.back()));
    std::vector<float> ta((size_t)R), tb((size_t)R);
    for (int i = 0; i < R; ++i) {
        CB_CUDA(cudaEventElapsedTime(&ta[i], ev[3 * i], ev[3 * i + 1]));
        CB_CUDA(cudaEventElapsedTime(&tb[i], ev[3 * i + 1], ev[3 * i + 2]));
    }
    for (auto & e : ev)
        cudaEventDestroy(e);
    auto median = [](std::vector<float> & v) {
        std::sort(v.begin(), v.end());
        const size_t n = v.size();
        return n % 2 ? v[n / 2] : 0.5f * (v[n / 2 - 1] + v[n / 2]);
    };
    *ms_patch = median(ta);
    *ms_shared = median(tb);
    CB_CATCH
}
int cuddh_b200_operator_destroy(cuddh_operator_t op)
{
    delete op;
    return 0;
}
int64_t cuddh_b200_operator_bytes(cuddh_operator_t op)
{
    if (op->vol)
        return (int64_t)op->vol->algorithmic_bytes();
    if (op->helm)
        return (int64_t)op->helm->algorithmic_bytes();
    return 0;
}
int64_t cuddh_b200_operator_bytes_moved(cuddh_operator_t op)
{
    if (op->vol)
        return (int64_t)op->vol->moved_bytes();
    if (op->helm)
        return (int64_t)op->helm->moved_bytes();
    return 0;
}
int cuddh_b200_operator_is_affine(cuddh_operator_t op)
{
    if (op->vol)
        return op->vol->affine ? 1 : 0;
    if (op->helm)
        return op->helm->S->affine ? 1 : 0;
    return 0;
}
int cuddh_b200_operator_kernel_kind(cuddh_operator_t op)
{
    auto kind = [](const VolumeOp & v) { return v.kind == VolumeKernel::ThreadPerElement ? 1 : v.kind == VolumeKernel::ThreadPair ? 3 : 0; };
    if (op->vol)
        return kind(*op->vol);
    if (op->helm)
        return op->helm->fused ? 2 : kind(*op->helm->S);
    return -1;
}

// ---- linalg ----
#define CB_LINALG2(NAME, T, SUF)                                                                          \
    int cuddh_b200_axpby_##SUF(int64_t n, T a, const T * x, T b, T * y, void * stream)                    \
    {                                                                                                     \
        CB_TRY axpby<T>(n, a, x, b, y, S(stream));                                                        \
        CB_CATCH                                                                                          \
    }                                                                                                     \
    int cuddh_b200_dot_##SUF(int64_t n, const T * x, const T * y, T * r, void * stream)                   \
    {                                                                                                     \
        CB_TRY * r = dot<T>(n, x, y, S(stream));                                                          \
        CB_CATCH                                                                                          \
    }                                                                                                     \
    int cuddh_b200_dist_##SUF(int64_t n, const T * x, const T * y, T * r, void * stream)                  \
    {                                                                                                     \
        CB_TRY * r = dist<T>(n, x, y, S(stream));                                                         \
        CB_CATCH                                                                                          \
    }                                                                                                     \
    int cuddh_b200_copy_##SUF(int64_t n, const T * x, T * y, void * stream)                               \
    {                                                                                                     \
        CB_TRY copy<T>(n, x, y, S(stream));                                                               \
        CB_CATCH                                                                                          \
    }                                                                                                     \
    int cuddh_b200_scal_##SUF(int64_t n, T a, T * x, void * stream)                                       \
    {                                                                                                     \
        CB_TRY scal<T>(n, a, x, S(stream));                                                               \
        CB_CATCH                                                                                          \
    }                                                                                                     \
    int cuddh_b200_fill_##SUF(int64_t n, T a, T * x, void * stream)                                       \
    {                                                                                                     \
        CB_TRY fill<T>(n, a, x, S(stream));                                                               \
        CB_CATCH                                                                                          \
    }
CB_LINALG2(d, double, d)
CB_LINALG2(f, float, f)
int cuddh_b200_copy_i(int64_t n, const int * x, int * y, void * stream)
{
    CB_TRY copy<int>(n, x, y, S(stream));
    CB_CATCH
}
int cuddh_b200_fill_i(int64_t n, int a, int * x, void * stream)
{
    CB_TRY fill<int>(n, a, x, S(stream));
    CB_CATCH
}

// ---- gmres ----
} // extern "C"
namespace
{
    struct PrecondSystem // source/gmres.cpp:68-89 PreconditionedSystem: y = P (A x)
    {
        cuddh_apply_d_fn A, P;
        void *Actx, *Pctx;
        double * q;
        static int apply(void * self, const double * x, double * y, cudaStream_t st)
        {
            auto * s = (PrecondSystem *)self;
            const int rc = s->A(s->Actx, x, s->q, (void *)st);
            return rc ? rc : s->P(s->Pctx, s->q, y, (void *)st);
        }
    };
    // the C ABI callback type (void* stream) behind the internal one (cudaStream_t)
    template <typename T> struct UserApply
    {
        int (*fn)(void *, const T *, T *, void *);
        void * ctx;
        static int apply(void * self, const T * x, T * y, cudaStream_t st)
        {
            auto * u = (UserApply *)self;
            return u->fn(u->ctx, x, y, (void *)st);
        }
    };

    void fill_out(const GmresResult & r, cuddh_solver_out * out, double * res, double * time, int cap)
    {
        if (out) {
            out->success = r.success ? 1 : 0;
            out->num_iter = r.num_iter;
            out->num_matvec = r.num_matvec;
            out->n_res = (int)std::min<size_t>(r.res_norm.size(), (size_t)std::max(cap, 0));
        }
        const int n = (int)std::min<size_t>(r.res_norm.size(), (size_t)std::max(cap, 0));
        for (int i = 0; i < n; ++i) {
            if (res)
                res[i] = r.res_norm[i];
            if (time)
                time[i] = r.time[i];
        }
    }

    GmresOptions make_options(const cuddh_gmres_options * o)
    {
        GmresOptions g;
        g.orth = default_gmres_orth();
        if (o) {
            if (o->orth >= 0)
                g.orth = o->orth;
            g.comm = o->comm ? o->comm->c.get() : nullptr;
            g.d_mask = o->d_mask;
            g.time_orth = o->time_orth != 0;
        }
        CB_REQUIRE(g.orth == ORTH_MGS || g.orth == ORTH_CGS2, "gmres: unknown orthogonalisation mode");
        return g;
    }
    void fill_stats(const GmresResult & r, cuddh_gmres_stats * st)
    {
        if (!st)
            return;
        st->orth_bytes = r.orth_bytes;
        st->orth_ms = r.orth_ms;
        st->reorth = r.reorth;
        st->allreduces = r.allreduces;
    }
} // namespace
extern "C" {

int cuddh_b200_gmres_d_ex(int64_t n, double * x, cuddh_apply_d_fn A, void * A_ctx, const double * b, cuddh_apply_d_fn P, void * P_ctx,
                          int m, int maxit, double tol, int verbose, double max_seconds, const cuddh_gmres_options * opts,
                          cuddh_solver_out * out, double * res, double * time, int cap, cuddh_gmres_stats * stats, void * stream)
{
    CB_TRY
    CB_REQUIRE(A != nullptr, "gmres: null operator callback");
    const GmresOptions go = make_options(opts);
    GmresResult r;
    if (P && opts && opts->flexible) { // FGMRES: A P y = b, x = P y, P applied afresh to every basis vector
        UserApply<double> ua{A, A_ctx}, up{P, P_ctx};
        GmresOptions gf = go;
        gf.right_precond = (void *)&UserApply<double>::apply;
        gf.right_precond_ctx = &up;
        r = gmres<double>(n, x, &UserApply<double>::apply, &ua, b, m, maxit, tol, verbose, max_seconds, S(stream), gf);
    }
    else if (P) { // gmres.cpp:242-251: solve P A x = P b
        DevBuf<double> q((size_t)n), r0((size_t)n);
        PrecondSystem sys{A, P, A_ctx, P_ctx, q.p};
        const int rc = P(P_ctx, b, r0.p, stream);
        if (rc != 0)
            throw Error(rc, "gmres: the preconditioner callback failed");
        r = gmres<double>(n, x, &PrecondSystem::apply, &sys, r0.p, m, maxit, tol, verbose, max_seconds, S(stream), go);
        CB_CUDA(cudaStreamSynchronize(S(stream)));
    }
    else {
        UserApply<double> ua{A, A_ctx};
        r = gmres<double>(n, x, &UserApply<double>::apply, &ua, b, m, maxit, tol, verbose, max_seconds, S(stream), go);
    }
    fill_out(r, out, res, time, cap);
    fill_stats(r, stats);
    CB_CATCH
}

int cuddh_b200_gmres_f_ex(int64_t n, float * x, cuddh_apply_f_fn A, void * A_ctx, const float * b, int m, int maxit, float tol,
                          int verbose, double max_seconds, const cuddh_gmres_options * opts, cuddh_solver_out * out, double * res,
                          double * time, int cap, cuddh_gmres_stats * stats, void * stream)
{
    CB_TRY
    CB_REQUIRE(A != nullptr, "gmres: null operator callback");
    const GmresOptions go = make_options(opts);
    UserApply<float> ua{A, A_ctx};
    GmresResult r = gmres<float>(n, x, &UserApply<float>::apply, &ua, b, m, maxit, tol, verbose, max_seconds, S(stream), go);
    fill_out(r, out, res, time, cap);
    fill_stats(r, stats);
    CB_CATCH
}

int cuddh_b200_gmres_d(int64_t n, double * x, cuddh_apply_d_fn A, void * A_ctx, const double * b, cuddh_apply_d_fn P, void * P_ctx,
                       int m, int maxit, double tol, int verbose, double max_seconds, cuddh_solver_out * out, double * res,
                       double * time, int cap, void * stream)
{
    return cuddh_b200_gmres_d_ex(n, x, A, A_ctx, b, P, P_ctx, m, maxit, tol, verbose, max_seconds, nullptr, out, res, time, cap, nullptr, stream);
}

int cuddh_b200_gmres_f(int64_t n, float * x, cuddh_apply_f_fn A, void * A_ctx, const float * b, int m, int maxit, float tol,
                       int verbose, double max_seconds, cuddh_solver_out * out, double * res, double * time, int cap, void * stream)
{
    return cuddh_b200_gmres_f_ex(n, x, A, A_ctx, b, m, maxit, tol, verbose, max_seconds, nullptr, out, res, time, cap, nullptr, stream);
}

int cuddh_b200_operator_as_apply(void * h, const double * x, double * y, void * stream)
{
    return cuddh_b200_operator_apply((cuddh_operator_t)h, 1.0, 0, x, y, stream);
}
int cuddh_b200_ddh_as_apply(void * h, const float * x, float * y, void * stream)
{
    return cuddh_b200_ddh_action((cuddh_ddh_t)h, x, y, stream);
}

// ---- options ----
int cuddh_b200_set_option(const char * name, int64_t value)
{
    CB_TRY
    const std::string n(name ? name : "");
    if (n == "gmres_orth")
        set_default_gmres_orth((int)value);
    else if (n == "max_ctas")
        set_max_persistent_ctas((int)value);
    else
        throw Error(-1, "set_option: unknown option " + n);
    CB_CATCH
}
int64_t cuddh_b200_get_option(const char * name)
{
    const std::string n(name ? name : "");
    if (n == "gmres_orth")
        return default_gmres_orth();
    if (n == "max_ctas")
        return max_persistent_ctas();
    if (n == "nccl_available")
        return nccl_available() ? 1 : 0;
    return -1;
}

// ---- communicator (multi-GPU runs: one process per GPU) ----
int cuddh_b200_comm_unique_id(unsigned char * id128)
{
    CB_TRY
    comm_unique_id(id128);
    CB_CATCH
}
int cuddh_b200_comm_create(const unsigned char * id128, int rank, int world, cuddh_comm_t * out)
{
    CB_TRY
    *out = new cuddh_comm_s{comm_create(id128, rank, world)};
    CB_CATCH
}
int cuddh_b200_comm_wrap(void * nccl_comm, int rank, int world, cuddh_comm_t * out)
{
    CB_TRY
    *out = new cuddh_comm_s{comm_wrap(nccl_comm, rank, world)};
    CB_CATCH
}
int cuddh_b200_comm_destroy(cuddh_comm_t c)
{
    delete c;
    return 0;
}
int cuddh_b200_comm_allreduce_d(cuddh_comm_t c, double * d_buf, int64_t count, void * stream)
{
    CB_TRY
    comm_allreduce_sum(c ? c->c.get() : nullptr, d_buf, count, S(stream));
    CB_CATCH
}

// ---- EnsembleSpace ----
int cuddh_b200_ensemble_create(cuddh_h1space_t s, int n_spaces, const int * labels, cuddh_ensemble_t * out)
{
    CB_TRY
    *out = new cuddh_ensemble_s{std::unique_ptr<Ensemble>(new Ensemble(*s->s, n_spaces, labels))};
    CB_CATCH
}
int cuddh_b200_ensemble_destroy(cuddh_ensemble_t e)
{
    delete e;
    return 0;
}
int cuddh_b200_ensemble_info(cuddh_ensemble_t e, int64_t * info)
{
    CB_TRY
    const Ensemble & E = *e->e;
    info[0] = E.n_spaces;
    info[1] = E.mx_elems;
    info[2] = E.mx_faces;
    info[3] = E.mx_ndof;
    info[4] = E.mx_fdof;
    info[5] = E.n_shared;
    CB_CATCH
}
const int * cuddh_b200_ensemble_array(cuddh_ensemble_t e, const char * name, int64_t * count)
{
    const Ensemble & E = *e->e;
    const std::string n(name);
    const std::vector<int> * v = nullptr;
    if (n == "gI") v = &E.gI;
    else if (n == "sizes") v = &E.s_dof;
    else if (n == "elements") v = &E.elems;
    else if (n == "n_elems") v = &E.s_elems;
    else if (n == "faces") v = &E.faces;
    else if (n == "n_faces") v = &E.s_faces;
    else if (n == "sI") v = &E.sI;
    else if (n == "fI") v = &E.fI;
    else if (n == "pI") v = &E.pI;
    else if (n == "fsizes") v = &E.s_fdof;
    else if (n == "cmap") v = &E.cmap;
    if (!v) {
        set_last_error("ensemble_array: unknown array name " + n);
        return nullptr;
    }
    if (count)
        *count = (int64_t)v->size();
    return v->data();
}

// ---- DDH ----
int cuddh_b200_ddh_create(double omega, const double * h_a, cuddh_h1space_t s, int nx, int ny, int block, cuddh_ddh_t * out)
{
    CB_TRY
    *out = new cuddh_ddh_s{std::unique_ptr<DDH>(new DDH(omega, h_a, s->s.get(), nx, ny, block))};
    CB_CATCH
}
int cuddh_b200_ddh_destroy(cuddh_ddh_t d)
{
    delete d;
    return 0;
}
int64_t cuddh_b200_ddh_size(cuddh_ddh_t d) { return 2 * d->d->n_lambda; }
int cuddh_b200_ddh_rhs(cuddh_ddh_t d, const double * f, float * b, void * stream)
{
    CB_TRY
    d->d->rhs(f, b, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_action(cuddh_ddh_t d, const float * x, float * y, void * stream)
{
    CB_TRY
    d->d->action(x, y, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_postprocess(cuddh_ddh_t d, const float * lambda, const double * f, double * u, void * stream)
{
    CB_TRY
    d->d->postprocess(lambda, f, u, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_apply_T_range(cuddh_ddh_t d, const float * x, float * t, int dom_begin, int dom_end, void * stream)
{
    CB_TRY
    d->d->apply_T_range(x, t, dom_begin, dom_end, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_rhs_range(cuddh_ddh_t d, const double * f, float * b, int dom_begin, int dom_end, void * stream)
{
    CB_TRY
    d->d->rhs_range(f, b, dom_begin, dom_end, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_postprocess_range(cuddh_ddh_t d, const float * lambda, const double * f, double * u, int dom_begin, int dom_end,
                                     void * stream)
{
    CB_TRY
    d->d->postprocess_range(lambda, f, u, dom_begin, dom_end, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_info(cuddh_ddh_t d, int64_t * info, double * dt)
{
    CB_TRY
    const DDH & D = *d->d;
    info[0] = D.n_domains;
    info[1] = D.n_shared;
    info[2] = D.nt;
    info[3] = D.mx_dof;
    info[4] = D.mx_fdof;
    info[5] = D.mx_elem;
    info[6] = D.nb;
    info[7] = D.block;
    *dt = D.dt;
    CB_CATCH
}
int cuddh_b200_ddh_get_array(cuddh_ddh_t d, const char * name, void * h_out, int64_t cap_bytes, int64_t * count)
{
    CB_TRY
    d->d->get_array(name, h_out, cap_bytes, count);
    CB_CATCH
}
double cuddh_b200_ddh_flops(cuddh_ddh_t d) { return d->d->flops(); }
int cuddh_b200_ddh_kernel_kind(cuddh_ddh_t d) { return d->d->kernel_kind(); }

// ---- path A across GPUs: slabs of element rows ----
int cuddh_b200_slab_create(cuddh_comm_t comm, int rank, int world, cuddh_h1space_t s, cuddh_facespace_t fs_phys, int64_t n_bottom,
                           const int * h_bottom, int64_t n_top, const int * h_top, cuddh_slab_t * out)
{
    CB_TRY
    *out = new cuddh_slab_s{make_slab_halo(comm ? comm->c.get() : nullptr, rank, world, s->s->ndof, fs_phys ? fs_phys->f.get() : nullptr,
                                            n_bottom, h_bottom, n_top, h_top)};
    CB_CATCH
}
int cuddh_b200_slab_destroy(cuddh_slab_t h)
{
    delete h;
    return 0;
}
int64_t cuddh_b200_slab_bytes(cuddh_slab_t h) { return h->h->bytes_per_apply(); }
int cuddh_b200_slab_uses_peer_memory(cuddh_slab_t h) { return h->h->peer ? 1 : 0; }
int cuddh_b200_slab_exchange(cuddh_slab_t h, double * y, void * stream)
{
    CB_TRY
    h->h->exchange(y, S(stream));
    CB_CATCH
}
const unsigned char * cuddh_b200_slab_mask(cuddh_slab_t h)
{
    try {
        return h->h->mask();
    }
    catch (const std::exception & e) {
        set_last_error(e.what());
        return nullptr;
    }
}
int cuddh_b200_helmholtz_apply_slab(cuddh_operator_t op, cuddh_slab_t h, const double * x, double * y, void * stream)
{
    CB_TRY
    CB_REQUIRE(op->helm != nullptr, "helmholtz_apply_slab: not a Helmholtz handle");
    op->helm->apply_slab(x, y, *h->h, S(stream));
    CB_CATCH
}
int cuddh_b200_slab_bind(cuddh_slab_t h, cuddh_operator_t op)
{
    CB_TRY
    CB_REQUIRE(op->helm != nullptr, "slab_bind: not a Helmholtz handle");
    h->h->op = op->helm.get();
    CB_CATCH
}
int cuddh_b200_slab_as_apply(void * slab, const double * x, double * y, void * stream)
{
    CB_TRY
    SlabHalo & h = *((cuddh_slab_t)slab)->h;
    CB_REQUIRE(h.op != nullptr, "slab_as_apply: no operator bound (cuddh_b200_slab_bind)");
    h.op->apply_slab(x, y, h, S(stream));
    CB_CATCH
}

// ---- DDH across GPUs ----
int cuddh_b200_ddh_dist_create(cuddh_ddh_t d, cuddh_comm_t comm, int rank, int world, cuddh_ddh_dist_t * out)
{
    CB_TRY
    *out = new cuddh_ddh_dist_s{std::unique_ptr<DdhDist>(new DdhDist(d->d.get(), comm ? comm->c.get() : nullptr, rank, world))};
    CB_CATCH
}
int cuddh_b200_ddh_dist_destroy(cuddh_ddh_dist_t h)
{
    delete h;
    return 0;
}
int cuddh_b200_ddh_dist_info(cuddh_ddh_dist_t h, int64_t * info)
{
    CB_TRY
    const DdhDist & D = *h->d;
    info[0] = D.dom_begin;
    info[1] = D.dom_end;
    info[2] = D.n_owned;
    info[3] = (int64_t)D.send_idx.size();
    info[4] = (int64_t)D.recv_idx.size();
    info[5] = (int64_t)D.segs.size();
    info[6] = D.bytes_per_action();
    info[7] = 2 * D.n_lambda;
    CB_CATCH
}
int cuddh_b200_ddh_dist_get_array(cuddh_ddh_dist_t h, const char * name, int * h_out, int64_t cap, int64_t * count)
{
    CB_TRY
    const DdhDist & D = *h->d;
    const std::string n(name ? name : "");
    std::vector<int> tmp;
    const std::vector<int> * v = nullptr;
    if (n == "owner") v = &D.owner;
    else if (n == "send_idx") v = &D.send_idx;
    else if (n == "recv_idx") v = &D.recv_idx;
    else if (n == "segments") { // (5, n_peers): peer, send_off, send_count, recv_off, recv_count
        for (const PeerSeg & g : D.segs) {
            tmp.push_back(g.peer);
            tmp.push_back((int)g.send_off);
            tmp.push_back((int)g.send_count);
            tmp.push_back((int)g.recv_off);
            tmp.push_back((int)g.recv_count);
        }
        v = &tmp;
    }
    else
        throw Error(-1, "ddh_dist_get_array: unknown array name " + n);
    if (count)
        *count = (int64_t)v->size();
    if (h_out) {
        CB_REQUIRE((int64_t)v->size() <= cap, "ddh_dist_get_array: output buffer too small");
        std::memcpy(h_out, v->data(), v->size() * sizeof(int));
    }
    CB_CATCH
}
const unsigned char * cuddh_b200_ddh_dist_mask(cuddh_ddh_dist_t h)
{
    try {
        h->d->ensure_device();
        return h->d->d_mask.p;
    }
    catch (const std::exception & e) {
        set_last_error(e.what());
        return nullptr;
    }
}
int cuddh_b200_ddh_dist_buffers(cuddh_ddh_dist_t h, void ** d_send, void ** d_recv)
{
    CB_TRY
    h->d->ensure_device();
    *d_send = h->d->d_send.p;
    *d_recv = h->d->d_recv.p;
    CB_CATCH
}
int cuddh_b200_ddh_dist_rhs(cuddh_ddh_dist_t h, const double * f, float * b, void * stream)
{
    CB_TRY
    h->d->rhs(f, b, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_dist_action(cuddh_ddh_dist_t h, const float * x, float * y, void * stream)
{
    CB_TRY
    h->d->action(x, y, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_dist_apply_T(cuddh_ddh_dist_t h, const float * x, float * t, void * stream)
{
    CB_TRY
    h->d->apply_T(x, t, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_dist_postprocess(cuddh_ddh_dist_t h, const float * lambda, const double * f, double * u, void * stream)
{
    CB_TRY
    h->d->postprocess(lambda, f, u, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_dist_as_apply(void * h, const float * x, float * y, void * stream)
{
    return cuddh_b200_ddh_dist_action((cuddh_ddh_dist_t)h, x, y, stream);
}

// ---- assembled DDH interface operator ----
int cuddh_b200_ddh_transfer_slots(cuddh_ddh_t d, int * h_in, int * h_out, int64_t cap, int * two_f)
{
    CB_TRY
    TransferSlots S;
    transfer_slots(*d->d, S);
    if (two_f)
        *two_f = S.two_f;
    if (h_in || h_out)
        CB_REQUIRE((int64_t)S.in.size() <= cap, "ddh_transfer_slots: output buffer too small");
    if (h_in)
        std::memcpy(h_in, S.in.data(), S.in.size() * sizeof(int));
    if (h_out)
        std::memcpy(h_out, S.out.data(), S.out.size() * sizeof(int));
    CB_CATCH
}
int cuddh_b200_ddh_transfer_orphans(cuddh_ddh_t d, int * h_out, int64_t cap, int64_t * count)
{
    CB_TRY
    TransferSlots S;
    transfer_slots(*d->d, S);
    if (count)
        *count = (int64_t)S.orphans.size();
    if (h_out) {
        CB_REQUIRE((int64_t)S.orphans.size() <= cap, "ddh_transfer_orphans: output buffer too small");
        std::memcpy(h_out, S.orphans.data(), S.orphans.size() * sizeof(int));
    }
    CB_CATCH
}
int cuddh_b200_ddh_transfer_create(cuddh_ddh_t d, int64_t max_bytes, void * stream, cuddh_ddh_transfer_t * out)
{
    CB_TRY
    *out = new cuddh_ddh_transfer_s{std::unique_ptr<DDHTransfer>(new DDHTransfer(d->d.get(), max_bytes, S(stream)))};
    CB_CATCH
}
int cuddh_b200_ddh_transfer_destroy(cuddh_ddh_transfer_t h)
{
    delete h;
    return 0;
}
int cuddh_b200_ddh_transfer_action(cuddh_ddh_transfer_t h, const float * x, float * y, void * stream)
{
    CB_TRY
    h->t->action(x, y, S(stream));
    CB_CATCH
}
int cuddh_b200_ddh_transfer_as_apply(void * h, const float * x, float * y, void * stream)
{
    return cuddh_b200_ddh_transfer_action((cuddh_ddh_transfer_t)h, x, y, stream);
}
int cuddh_b200_ddh_transfer_info(cuddh_ddh_transfer_t h, int64_t * info)
{
    CB_TRY
    const DDHTransfer & T = *h->t;
    info[0] = T.slots.n_domains;
    info[1] = T.slots.two_f;
    info[2] = T.block_bytes();
    info[3] = T.bytes_per_action();
    info[4] = T.probe_launches;
    info[5] = (int64_t)(T.probe_ms * 1000.0 + 0.5);
    CB_CATCH
}
int cuddh_b200_ddh_transfer_get_block(cuddh_ddh_transfer_t h, int dom, float * h_out)
{
    CB_TRY
    h->t->get_block(dom, h_out);
    CB_CATCH
}

} // extern "C"
