// BLAS-1 + GMRES declarations (see linalg.cu).
#pragma once
#include "common.hpp"
#include "dist.hpp"
#include <vector>

namespace cb200
{
    template <typename T> void axpby(int64_t n, T a, const T * x, T b, T * y, cudaStream_t s);
    template <typename T> void scal(int64_t n, T a, T * x, cudaStream_t s);
    template <typename T> void fill(int64_t n, T a, T * x, cudaStream_t s);
    template <typename T> void copy(int64_t n, const T * x, T * y, cudaStream_t s);
    template <typename T> T dot(int64_t n, const T * x, const T * y, cudaStream_t s);   // blocks the host (returns the scalar)
    template <typename T> T dist(int64_t n, const T * x, const T * y, cudaStream_t s);

    // y = A x enqueued on stream s; non-zero return aborts the solve with that status
    template <typename T> using ApplyFn = int (*)(void * ctx, const T * x, T * y, cudaStream_t s);

    struct GmresResult
    {
        bool success;
        int num_iter, num_matvec;
        std::vector<double> res_norm, time;
        // vector traffic of the orthogonalisation (bytes moved by the Gram-Schmidt kernels) and its device time, for bench.py
        double orth_bytes = 0, orth_ms = 0;
        int reorth = 0;     // CGS: second passes taken (cancellation)
        int allreduces = 0; // distributed runs
    };

    enum GmresOrth
    {
        ORTH_MGS = 0, // modified Gram-Schmidt, the reference's arithmetic (source/gmres.cpp:167-172): k+2 fused passes per step
        ORTH_CGS2 = 1 // classical Gram-Schmidt, all inner products in one pass + one update pass; second round on cancellation
    };

    struct GmresOptions
    {
        int orth = ORTH_MGS;
        const Comm * comm = nullptr;             // distributed vectors: inner products are summed over the ranks
        const unsigned char * d_mask = nullptr;  // 1 = this rank owns the entry (counted in inner products), 0 = mirror copy / foreign slot
        bool time_orth = false;                  // record CUDA-event time of the orthogonalisation kernels (adds two event records per step)
        // flexible right preconditioning (FGMRES): z_k = P(v_k) is stored, w = A z_k, x += sum eta_k z_k; P may change from
        // step to step (e.g. an inner iterative solve). ApplyFn<T> cast to void*; null = none.
        void * right_precond = nullptr;
        void * right_precond_ctx = nullptr;
    };

    // Restarted GMRES(m) with the reference's control flow (source/gmres.cpp:91-235). A is a callback that
    // must enqueue y = A x on the stream it is handed.
    template <typename T>
    GmresResult gmres(int64_t n, T * x, ApplyFn<T> A, void * ctx, const T * b, int m, int maxit, T tol, int verbose,
                      double max_seconds, cudaStream_t s, const GmresOptions & opt = GmresOptions());

    // y_j = A x_j for the k systems listed, enqueued on stream s (x, y: HOST arrays of k device pointers); non-zero aborts the solve
    template <typename T> using ApplyBatchFn = int (*)(void * ctx, int k, const T * const * x, T * const * y, cudaStream_t s);
    constexpr int GMRES_BATCH_KMAX = 32;

    // k (<= GMRES_BATCH_KMAX) independent GMRES(m) solves A x_j = b_j in lockstep: every Arnoldi step applies A once to all systems
    // still in their Arnoldi loop (A is handed only those), runs their MGS sweeps in the same launches and syncs the host once.
    // Each system keeps the control flow of gmres(..., ORTH_MGS): its own initial-residual exit, inner break (|eta| < tol ||b||
    // or w = 0; it then waits for the restart boundary), true residual per restart, and it leaves the batch when it converges.
    // Results (x, res_norm, num_iter, num_matvec) are bitwise those of k sequential gmres(..., ORTH_MGS) calls; time[] is measured
    // from the start of the batch, and max_seconds limits the wall time of the whole batch. MGS only (GmresOptions::orth is not
    // read); no CGS2, distributed vectors, preconditioning or verbose output. Only float is instantiated.
    template <typename T>
    std::vector<GmresResult> gmres_batch(int64_t n, int k, T * const * x, ApplyBatchFn<T> A, void * ctx, const T * const * b, int m, int maxit,
                                         T tol, double max_seconds, cudaStream_t s);

    // process-wide default of GmresOptions::orth for the entry points without an options argument (set_option "gmres_orth")
    int default_gmres_orth();
    void set_default_gmres_orth(int v);
} // namespace cb200
