// DDH: the FP32 substructured (domain-decomposition, WaveHoltz local solves) Helmholtz operator
// (reference include/DDH.hpp:21-84). One batched sm_100a kernel per action (csrc/ddh.cu).
#ifndef CUDDH_DDH_HPP
#define CUDDH_DDH_HPP

#include <assert.h>
#include <functional>
#include <memory>
#include <unordered_set>

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

    private:
        const DDH & ddh;
        std::shared_ptr<cuddh_ddh_transfer_s> h;
    };
} // namespace cuddh

#endif
