// DDH: the FP32 substructured (domain-decomposition, WaveHoltz local solves) Helmholtz operator
// (reference include/DDH.hpp:21-84). One batched sm_100a kernel per action (csrc/ddh.cu).
#ifndef CUDDH_DDH_HPP
#define CUDDH_DDH_HPP

#include <algorithm>
#include <assert.h>
#include <functional>
#include <memory>
#include <unordered_set>
#include <vector>

#include <cuda_runtime.h>

#include "EnsembleSpace.hpp"
#include "HostDeviceArray.hpp"
#include "MassMatrix.hpp"
#include "Operator.hpp"
#include "forall.hpp"
#include "gmres.hpp"
#include "linalg.hpp"

#ifndef DDH_BLOCK_SIZE
#define DDH_BLOCK_SIZE 16 // 1-D node size of a subdomain block (the reference's compile-time constant); 16 or 32
#endif

namespace cuddh
{
    class DDH : public SinglePrecisionOperator
    {
    public:
        /// h_a: HOST array, the variable coefficient a at the H1 nodes; fem's mesh must come from Mesh2D::uniform_rect(nx, .., ny, ..)
        DDH(double omega, const double * h_a, const H1Space & fem, int nx, int ny)
        {
            cuddh_ddh_t raw = nullptr;
            cuddh_check(cuddh_b200_ddh_create(omega, h_a, fem.handle(), nx, ny, DDH_BLOCK_SIZE, &raw));
            h.reset(raw, [](cuddh_ddh_t p) { cuddh_b200_ddh_destroy(p); });
        }
        ~DDH() = default;

        /// number of degrees of freedom of the substructured problem
        int size() const { return (int)cuddh_b200_ddh_size(h.get()); }

        /// b <- right-hand side of the substructured problem from the Helmholtz forcing f
        void rhs(const double * f, float * b) const { cuddh_check(cuddh_b200_ddh_rhs(h.get(), f, b, nullptr)); }
        /// u <- finite element solution from lambda and f
        void postprocess(const float * lambda, const double * f, double * u) const { cuddh_check(cuddh_b200_ddh_postprocess(h.get(), lambda, f, u, nullptr)); }
        /// y <- (I - T) x
        void action(const float * x, float * y) const override { cuddh_check(cuddh_b200_ddh_action(h.get(), x, y, nullptr)); }

        /// the library handle (include/cuddh_b200.h)
        cuddh_ddh_t handle() const { return h.get(); }

    private:
        std::shared_ptr<cuddh_ddh_s> h;
    };

    /// The same operator as DDH with its interface map T assembled: one dense 2F x 2F block per subdomain, probed once with 2F
    /// WaveHoltz actions; action() is then one streaming batched matvec, y <- (I - T) x. The DDH must outlive this object.
    class DDHTransfer : public SinglePrecisionOperator
    {
    public:
        /// max_bytes: device memory the blocks may take, 0 = whatever is free (throws with the bytes needed if they do not fit)
        explicit DDHTransfer(const DDH & ddh, int64_t max_bytes = 0) : ddh(ddh)
        {
            cuddh_ddh_transfer_t raw = nullptr;
            cuddh_check(cuddh_b200_ddh_transfer_create(ddh.handle(), max_bytes, nullptr, &raw));
            h.reset(raw, [](cuddh_ddh_transfer_t p) { cuddh_b200_ddh_transfer_destroy(p); });
        }

        int size() const { return ddh.size(); }
        void rhs(const double * f, float * b) const { ddh.rhs(f, b); }
        void postprocess(const float * lambda, const double * f, double * u) const { ddh.postprocess(lambda, f, u); }
        /// y <- (I - T) x  (x and y must not overlap)
        void action(const float * x, float * y) const override { cuddh_check(cuddh_b200_ddh_transfer_action(h.get(), x, y, nullptr)); }
        /// y[j] <- (I - T) x[j] for j < k, 1 <= k <= 32; x, y: host arrays of k device pointers, no y[j] overlapping any x[i] or
        /// another y[i]. Row j is bitwise action(x[j], y[j]); the blocks are streamed once for up to 16 vectors.
        void action(int k, const float * const * x, float * const * y) const
        {
            cuddh_check(cuddh_b200_ddh_transfer_action_batch(h.get(), k, x, y, nullptr));
        }

        /// the library handle (include/cuddh_b200.h)
        cuddh_ddh_transfer_t handle() const { return h.get(); }

    private:
        const DDH & ddh;
        std::shared_ptr<cuddh_ddh_transfer_s> h;
    };

    /// k independent single-precision GMRES(m) solves A x[j] = b[j] in lockstep, 1 <= k <= 32: every Arnoldi step applies A once to
    /// all systems still iterating and syncs the host once. x, b: host arrays of k device pointers. Each result is bitwise that of
    /// gmres(n, x[j], &A, b[j], m, maxit, tol) with modified Gram-Schmidt (the library default); a system leaves the batch when it
    /// converges. max_seconds limits the whole batch, and time[] is measured from its start.
    inline std::vector<solver_out> gmres(int n, int k, float * const * x, const DDHTransfer & A, const float * const * b, int m, int maxit,
                                         float tol = 1e-4, double max_seconds = 6 * 60 * 60)
    {
        const int cap = maxit + 2;
        const size_t rows = (size_t)std::max(k, 1);
        std::vector<cuddh_solver_out> so(rows);
        std::vector<double> res(rows * cap), tim(rows * cap);
        cuddh_check(cuddh_b200_gmres_f_batch(n, k, x, &cuddh_b200_ddh_transfer_as_apply_batch, A.handle(), b, m, maxit, tol, max_seconds,
                                             so.data(), res.data(), tim.data(), cap, nullptr));
        std::vector<solver_out> out;
        for (int j = 0; j < k; ++j)
            out.push_back(detail::unpack(so[j], std::vector<double>(res.begin() + (size_t)j * cap, res.begin() + (size_t)(j + 1) * cap),
                                         std::vector<double>(tim.begin() + (size_t)j * cap, tim.begin() + (size_t)(j + 1) * cap)));
        return out;
    }
} // namespace cuddh

#endif
