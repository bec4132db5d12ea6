// BLAS-1 kernels and restarted GMRES (reference include/linalg.hpp, source/linalg.cpp, source/gmres.cpp).
//
// Reference behaviour being replaced: 32-thread reduction CTAs with one same-address atomicAdd per 256
// elements, a cudaMalloc + memset + blocking D2H + cudaFree per dot, and k+1 (dot, axpy) launch pairs with
// k+1 host syncs per Arnoldi step. Here:
//   * reductions are two-stage and deterministic: per-CTA partials in fixed slots, summed in slot order (by the last
//     CTA to finish, or by a one-block-per-value finishing kernel); grid = a multiple of the SM count;
//   * Krylov vectors live in a basis with a 16-byte-aligned leading dimension, so every orthogonalisation kernel
//     moves them with 128-bit loads / stores;
//   * two orthogonalisation modes (GmresOptions::orth):
//       MGS  - the reference's arithmetic (h_j = <w, v_j> AFTER w has been updated with h_{j-1}), every step ONE fused
//              kernel (w -= h_{j-1} v_{j-1} and the partial dot with v_j in the same pass, h_{j-1} read from device
//              memory), one host sync per Arnoldi step instead of k+1. This is what the parity tests pin.
//       CGS2 - all k+1 inner products and <w,w> in ONE pass over the basis (multi_dot), then ONE update pass
//              w <- (w - V h) / ||w - V h|| with the norm from Pythagoras; a second round (h2 = V^T w, w -= V h2,
//              h += h2) only when the first one cancelled more than half of ||w||^2 (the DGKS criterion). Traffic per
//              step ~ (2k+5) vectors instead of ~4(k+2), two launches + one sync instead of k+3;
//   * distributed vectors (GmresOptions::comm / d_mask): inner products count the entries this rank owns and are
//     summed with NCCL on the same stream - one allreduce of k+2 doubles per Arnoldi step in CGS2 mode;
//   * x += sum_k eta_k v_k is one pass (same left-to-right order as the reference's axpby chain).
// No process-wide mutable state: reduction workspaces are per (device, stream) for the BLAS-1 entry points and per call
// for gmres().
#include "linalg.hpp"
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <iostream>
#include <iomanip>
#include <map>
#include <mutex>

namespace cb200
{
    namespace
    {
        constexpr int RED_THREADS = 256;
        constexpr int MAX_RED_BLOCKS = 1184; // 8 CTAs x 148 SMs
        constexpr int JT = 8;                // basis vectors per multi_dot CTA row

        int sm_count()
        {
            int dev = 0, n = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
            return n > 0 ? n : 148;
        }

        int red_blocks(int64_t n, int per_sm = 8)
        {
            const int64_t want = (n + RED_THREADS * 4 - 1) / (RED_THREADS * 4);
            return (int)std::max<int64_t>(1, std::min<int64_t>(want, std::min(MAX_RED_BLOCKS, per_sm * sm_count())));
        }

        template <typename T>
        __device__ __forceinline__ T warp_sum(T v)
        {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1)
                v += __shfl_down_sync(0xffffffffu, v, o);
            return v;
        }

        // 16-byte packets of T
        template <typename T> struct Pack;
        template <> struct Pack<double>
        {
            static constexpr int N = 2;
            using V = double2;
            using M = uchar2;
            static __device__ __forceinline__ void get(const V & v, double (&a)[2]) { a[0] = v.x; a[1] = v.y; }
            static __device__ __forceinline__ V put(const double (&a)[2]) { return make_double2(a[0], a[1]); }
            static __device__ __forceinline__ void getm(const M & m, unsigned char (&a)[2]) { a[0] = m.x; a[1] = m.y; }
        };
        template <> struct Pack<float>
        {
            static constexpr int N = 4;
            using V = float4;
            using M = uchar4;
            static __device__ __forceinline__ void get(const V & v, float (&a)[4]) { a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w; }
            static __device__ __forceinline__ V put(const float (&a)[4]) { return make_float4(a[0], a[1], a[2], a[3]); }
            static __device__ __forceinline__ void getm(const M & m, unsigned char (&a)[4]) { a[0] = m.x; a[1] = m.y; a[2] = m.z; a[3] = m.w; }
        };

        // block partial -> slot; last block sums slots in order and writes result[0] (optionally sqrt)
        template <typename T>
        __device__ __forceinline__ void block_finish(T acc, T * __restrict__ partials, unsigned * __restrict__ ticket,
                                                     T * __restrict__ result, const bool take_sqrt)
        {
            __shared__ T wsum[RED_THREADS / 32];
            __shared__ bool last;
            acc = warp_sum(acc);
            if ((threadIdx.x & 31) == 0)
                wsum[threadIdx.x >> 5] = acc;
            __syncthreads();
            if (threadIdx.x == 0) {
                T b = 0;
#pragma unroll
                for (int w = 0; w < RED_THREADS / 32; ++w)
                    b += wsum[w];
                partials[blockIdx.x] = b;
                __threadfence();
                const unsigned t = atomicAdd(ticket, 1u);
                last = (t == gridDim.x - 1);
            }
            __syncthreads();
            if (last) {
                __threadfence();
                T s = 0;
                for (int i = threadIdx.x; i < (int)gridDim.x; i += RED_THREADS)
                    s += ((volatile T *)partials)[i];
                // fixed-shape tree over the 256 per-thread sums
                s = warp_sum(s);
                __syncthreads();
                if ((threadIdx.x & 31) == 0)
                    wsum[threadIdx.x >> 5] = s;
                __syncthreads();
                if (threadIdx.x == 0) {
                    T tot = 0;
#pragma unroll
                    for (int w = 0; w < RED_THREADS / 32; ++w)
                        tot += wsum[w];
                    result[0] = take_sqrt ? sqrt(tot) : tot;
                    *ticket = 0;
                }
            }
        }

        // body of reduce_kernel, shared with the batched solve (one system per grid row: same partition, same tree)
        template <typename T, int MODE> // MODE 0: x.y   1: (x-y)^2
        __device__ __forceinline__ void reduce_block(const int64_t n, const T * __restrict__ x, const T * __restrict__ y, T * __restrict__ partials,
                                                     unsigned * __restrict__ ticket, T * __restrict__ result, const int take_sqrt)
        {
            T acc = 0;
            const int64_t stride = (int64_t)gridDim.x * RED_THREADS;
            for (int64_t i = blockIdx.x * (int64_t)RED_THREADS + threadIdx.x; i < n; i += stride) {
                if (MODE == 0)
                    acc = fma(x[i], y[i], acc);
                else {
                    const T e = x[i] - y[i];
                    acc = fma(e, e, acc);
                }
            }
            block_finish(acc, partials, ticket, result, take_sqrt != 0);
        }

        template <typename T, int MODE>
        __global__ void __launch_bounds__(RED_THREADS)
        reduce_kernel(const int64_t n, const T * __restrict__ x, const T * __restrict__ y, T * __restrict__ partials,
                      unsigned * __restrict__ ticket, T * __restrict__ result, const int take_sqrt)
        {
            reduce_block<T, MODE>(n, x, y, partials, ticket, result, take_sqrt);
        }

        // fused MGS step on 16-byte-aligned basis columns: w -= h[prev] * vprev (if vprev), then <w, vnext> -> hout
        // (vnext == null: <w, w>, square root on the device unless the result still has to be summed over ranks).
        // Inner products count the entries with mask != 0 (mask == null: all).
        // (body of mgs_step_kernel, shared with the batched solve)
        template <typename T>
        __device__ __forceinline__ void mgs_step_block(const int64_t n, T * __restrict__ w, const T * __restrict__ vprev, const T * __restrict__ vnext,
                                                       const T * __restrict__ hprev, const unsigned char * __restrict__ mask, T * __restrict__ partials,
                                                       unsigned * __restrict__ ticket, T * __restrict__ hout, const int take_sqrt)
        {
            using P = Pack<T>;
            constexpr int N = P::N;
            const T hp = vprev ? hprev[0] : T(0);
            T acc = 0;
            const int64_t nv = n / N;
            const int64_t stride = (int64_t)gridDim.x * RED_THREADS;
            typename P::V * wv = reinterpret_cast<typename P::V *>(w);
            const typename P::V * pv = reinterpret_cast<const typename P::V *>(vprev);
            const typename P::V * qv = reinterpret_cast<const typename P::V *>(vnext);
            const typename P::M * mv = reinterpret_cast<const typename P::M *>(mask);
            for (int64_t i = blockIdx.x * (int64_t)RED_THREADS + threadIdx.x; i < nv; i += stride) {
                T a[N], b[N], c[N];
                unsigned char mk[N];
                P::get(wv[i], a);
                if (vprev) {
                    P::get(pv[i], b);
#pragma unroll
                    for (int t = 0; t < N; ++t)
                        a[t] = fma(-hp, b[t], a[t]);
                    wv[i] = P::put(a);
                }
                if (vnext)
                    P::get(qv[i], c);
                if (mask)
                    P::getm(mv[i], mk);
#pragma unroll
                for (int t = 0; t < N; ++t) {
                    const T term = vnext ? c[t] : a[t];
                    if (!mask || mk[t])
                        acc = fma(a[t], term, acc);
                }
            }
            // tail (n not a multiple of the packet width)
            if (blockIdx.x == 0 && threadIdx.x < n - nv * N) {
                const int64_t i = nv * N + threadIdx.x;
                T wi = w[i];
                if (vprev) {
                    wi = fma(-hp, vprev[i], wi);
                    w[i] = wi;
                }
                if (!mask || mask[i])
                    acc = fma(wi, vnext ? vnext[i] : wi, acc);
            }
            block_finish(acc, partials, ticket, hout, take_sqrt != 0);
        }

        template <typename T>
        __global__ void __launch_bounds__(RED_THREADS)
        mgs_step_kernel(const int64_t n, T * __restrict__ w, const T * __restrict__ vprev, const T * __restrict__ vnext,
                        const T * __restrict__ hprev, const unsigned char * __restrict__ mask, T * __restrict__ partials,
                        unsigned * __restrict__ ticket, T * __restrict__ hout, const int take_sqrt)
        {
            mgs_step_block(n, w, vprev, vnext, hprev, mask, partials, ticket, hout, take_sqrt);
        }

        // CGS pass 1: partial sums of <w, v_j> for the JT basis columns of CTA row blockIdx.y (and of <w, w> in row 0), FP64
        // accumulators whatever T is. partials[(value) * gridDim.x + blockIdx.x], values 0..k1-1 = columns, k1 = <w, w>.
        template <typename T>
        __global__ void __launch_bounds__(RED_THREADS)
        multi_dot_kernel(const int64_t n, const int64_t ldv, const int k1, const T * __restrict__ V, const T * __restrict__ w,
                         const unsigned char * __restrict__ mask, double * __restrict__ partials)
        {
            using P = Pack<T>;
            constexpr int N = P::N;
            const int j0 = blockIdx.y * JT;
            const int nj = min(JT, k1 - j0);
            const bool with_ww = blockIdx.y == 0;
            double acc[JT + 1];
#pragma unroll
            for (int j = 0; j <= JT; ++j)
                acc[j] = 0.0;
            const int64_t nv = n / N;
            const int64_t stride = (int64_t)gridDim.x * RED_THREADS;
            const typename P::V * wv = reinterpret_cast<const typename P::V *>(w);
            const typename P::M * mv = reinterpret_cast<const typename P::M *>(mask);
            for (int64_t i = blockIdx.x * (int64_t)RED_THREADS + threadIdx.x; i < nv; i += stride) {
                T a[N];
                unsigned char mk[N];
                P::get(wv[i], a);
                if (mask) {
                    P::getm(mv[i], mk);
#pragma unroll
                    for (int t = 0; t < N; ++t)
                        a[t] = mk[t] ? a[t] : T(0);
                }
                if (with_ww) {
#pragma unroll
                    for (int t = 0; t < N; ++t)
                        acc[JT] = fma((double)a[t], (double)a[t], acc[JT]);
                }
#pragma unroll
                for (int j = 0; j < JT; ++j)
                    if (j < nj) {
                        T b[N];
                        P::get(reinterpret_cast<const typename P::V *>(V + (size_t)(j0 + j) * ldv)[i], b);
#pragma unroll
                        for (int t = 0; t < N; ++t)
                            acc[j] = fma((double)a[t], (double)b[t], acc[j]);
                    }
            }
            if (blockIdx.x == 0 && threadIdx.x < n - nv * N) {
                const int64_t i = nv * N + threadIdx.x;
                const T wi = (!mask || mask[i]) ? w[i] : T(0);
                if (with_ww)
                    acc[JT] = fma((double)wi, (double)wi, acc[JT]);
                for (int j = 0; j < nj; ++j)
                    acc[j] = fma((double)wi, (double)V[(size_t)(j0 + j) * ldv + i], acc[j]);
            }
            __shared__ double wsum[JT + 1][RED_THREADS / 32];
#pragma unroll
            for (int j = 0; j <= JT; ++j) {
                const double v = warp_sum(acc[j]);
                if ((threadIdx.x & 31) == 0)
                    wsum[j][threadIdx.x >> 5] = v;
            }
            __syncthreads();
            if (threadIdx.x <= JT) {
                const int j = threadIdx.x;
                double b = 0.0;
#pragma unroll
                for (int q = 0; q < RED_THREADS / 32; ++q)
                    b += wsum[j][q];
                if (j < nj)
                    partials[(size_t)(j0 + j) * gridDim.x + blockIdx.x] = b;
                else if (j == JT && with_ww)
                    partials[(size_t)k1 * gridDim.x + blockIdx.x] = b;
            }
        }

        // out[v] = sum of the nb partials of value v, fixed order (one CTA per value)
        __global__ void __launch_bounds__(RED_THREADS) finish_sums_kernel(const int nb, const double * __restrict__ partials, double * __restrict__ out)
        {
            __shared__ double wsum[RED_THREADS / 32];
            const double * p = partials + (size_t)blockIdx.x * nb;
            double s = 0.0;
            for (int i = threadIdx.x; i < nb; i += RED_THREADS)
                s += p[i];
            s = warp_sum(s);
            if ((threadIdx.x & 31) == 0)
                wsum[threadIdx.x >> 5] = s;
            __syncthreads();
            if (threadIdx.x == 0) {
                double tot = 0.0;
#pragma unroll
                for (int q = 0; q < RED_THREADS / 32; ++q)
                    tot += wsum[q];
                out[blockIdx.x] = tot;
            }
        }

        // CGS pass 2: w <- (w - sum_j h[j] v_j) * scale, columns left to right, FP64 arithmetic on the way
        template <typename T>
        __global__ void __launch_bounds__(RED_THREADS)
        multi_update_kernel(const int64_t n, const int64_t ldv, const int k1, const T * __restrict__ V, const double * __restrict__ h,
                            const double scale, T * __restrict__ w)
        {
            using P = Pack<T>;
            constexpr int N = P::N;
            extern __shared__ double hs[];
            for (int j = threadIdx.x; j < k1; j += RED_THREADS)
                hs[j] = h[j];
            __syncthreads();
            const int64_t nv = n / N;
            const int64_t stride = (int64_t)gridDim.x * RED_THREADS;
            typename P::V * wv = reinterpret_cast<typename P::V *>(w);
            for (int64_t i = blockIdx.x * (int64_t)RED_THREADS + threadIdx.x; i < nv; i += stride) {
                T a[N];
                P::get(wv[i], a);
                double acc[N];
#pragma unroll
                for (int t = 0; t < N; ++t)
                    acc[t] = (double)a[t];
#pragma unroll 4
                for (int j = 0; j < k1; ++j) {
                    T b[N];
                    P::get(reinterpret_cast<const typename P::V *>(V + (size_t)j * ldv)[i], b);
                    const double hj = hs[j];
#pragma unroll
                    for (int t = 0; t < N; ++t)
                        acc[t] = fma(-hj, (double)b[t], acc[t]);
                }
#pragma unroll
                for (int t = 0; t < N; ++t)
                    a[t] = (T)(acc[t] * scale);
                wv[i] = P::put(a);
            }
            if (blockIdx.x == 0 && threadIdx.x < n - nv * N) {
                const int64_t i = nv * N + threadIdx.x;
                double acc = (double)w[i];
                for (int j = 0; j < k1; ++j)
                    acc = fma(-hs[j], (double)V[(size_t)j * ldv + i], acc);
                w[i] = (T)(acc * scale);
            }
        }

        // element bodies shared by the single and the batched kernels (same expression, same contraction)
        template <typename T>
        __device__ __forceinline__ void axpby_at(const int64_t i, const T a, const T * __restrict__ x, const T b, T * __restrict__ y)
        {
            y[i] = a * x[i] + b * y[i];
        }
        template <typename T>
        __device__ __forceinline__ T inv_norm(const T * __restrict__ s, const int take_sqrt)
        {
            return T(1) / (take_sqrt ? sqrt(s[0]) : s[0]);
        }
        template <typename T>
        __device__ __forceinline__ void multi_axpy_at(const int64_t i, const int64_t ldv, const int k1, const T * __restrict__ eta,
                                                      const T * __restrict__ V, T * __restrict__ x)
        {
            T acc = x[i];
            for (int k = 0; k < k1; ++k)
                acc = eta[k] * V[i + (size_t)k * ldv] + acc;
            x[i] = acc;
        }

        template <typename T>
        __global__ void axpby_kernel(const int64_t n, const T a, const T * __restrict__ x, const T b, T * __restrict__ y)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (i < n)
                axpby_at(i, a, x, b, y);
        }
        template <typename T>
        __global__ void scal_kernel(const int64_t n, const T a, T * __restrict__ x)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (i < n)
                x[i] *= a;
        }
        // x <- x / s[0] (or / sqrt(s[0])) with s on the device (no host round trip)
        template <typename T>
        __global__ void scal_inv_dev_kernel(const int64_t n, const T * __restrict__ s, const int take_sqrt, T * __restrict__ x)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            const T a = inv_norm(s, take_sqrt);
            if (i < n)
                x[i] *= a;
        }
        template <typename T>
        __global__ void fill_kernel(const int64_t n, const T a, T * __restrict__ x)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (i < n)
                x[i] = a;
        }
        template <typename T>
        __global__ void copy_kernel(const int64_t n, const T * __restrict__ x, T * __restrict__ y)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (i < n)
                y[i] = x[i];
        }
        // x <- x + sum_k eta[k] V[:,k], left to right (gmres.cpp:190-191)
        template <typename T>
        __global__ void multi_axpy_kernel(const int64_t n, const int64_t ldv, const int k1, const T * __restrict__ eta, const T * __restrict__ V,
                                          T * __restrict__ x)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (i < n)
                multi_axpy_at(i, ldv, k1, eta, V, x);
        }
        // masked sum of squares / products in T (the residual norms of the distributed solve)
        template <typename T>
        __global__ void __launch_bounds__(RED_THREADS)
        masked_dot_kernel(const int64_t n, const T * __restrict__ x, const T * __restrict__ y, const unsigned char * __restrict__ mask,
                          double * __restrict__ partials)
        {
            double acc = 0.0;
            const int64_t stride = (int64_t)gridDim.x * RED_THREADS;
            for (int64_t i = blockIdx.x * (int64_t)RED_THREADS + threadIdx.x; i < n; i += stride)
                if (!mask || mask[i])
                    acc = fma((double)x[i], (double)y[i], acc);
            __shared__ double wsum[RED_THREADS / 32];
            acc = warp_sum(acc);
            if ((threadIdx.x & 31) == 0)
                wsum[threadIdx.x >> 5] = acc;
            __syncthreads();
            if (threadIdx.x == 0) {
                double b = 0.0;
#pragma unroll
                for (int q = 0; q < RED_THREADS / 32; ++q)
                    b += wsum[q];
                partials[blockIdx.x] = b;
            }
        }

        inline unsigned nblk(int64_t n, int bs = 256) { return (unsigned)((n + bs - 1) / bs); }

        // ---- batched solve (gmres_batch): grid row blockIdx.y = one active system, kernel arguments passed by value ----
        template <typename T>
        struct BatchArgs
        {
            const T * x[GMRES_BATCH_KMAX];
            T * y[GMRES_BATCH_KMAX];
            T a[GMRES_BATCH_KMAX], b[GMRES_BATCH_KMAX];
            int k1[GMRES_BATCH_KMAX];  // multi_axpy: basis columns of each system
            int sys[GMRES_BATCH_KMAX]; // system index: its slice of the basis, Hessenberg column, partials and ticket
        };

        template <typename T>
        __global__ void axpby_batch_kernel(const int64_t n, const BatchArgs<T> p)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            const int j = blockIdx.y;
            if (i < n)
                axpby_at(i, p.a[j], p.x[j], p.b[j], p.y[j]);
        }

        // x_j += sum_k eta_j[k] V_j[:, k], eta_j at eta + sys * m1
        template <typename T>
        __global__ void multi_axpy_batch_kernel(const int64_t n, const int64_t ldv, const T * __restrict__ eta, const int m1, const BatchArgs<T> p)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            const int j = blockIdx.y;
            if (i < n)
                multi_axpy_at(i, ldv, p.k1[j], eta + (size_t)p.sys[j] * m1, p.x[j], p.y[j]);
        }

        // <x_j, x_j> -> result[j], each system with its own partials and ticket
        template <typename T>
        __global__ void __launch_bounds__(RED_THREADS)
        norm2_batch_kernel(const int64_t n, T * __restrict__ partials, unsigned * __restrict__ tickets, T * __restrict__ result, const BatchArgs<T> p)
        {
            const int j = blockIdx.y, s = p.sys[j];
            reduce_block<T, 0>(n, p.x[j], p.x[j], partials + (size_t)s * gridDim.x, tickets + s, result + j, 0);
        }

        // step j of the fused MGS sweep at Arnoldi index k1 - 1 for every listed system (basis of system s at V + s * vstride,
        // Hessenberg column at H + s * hstride)
        template <typename T>
        __global__ void __launch_bounds__(RED_THREADS)
        mgs_step_batch_kernel(const int64_t n, T * __restrict__ V, const int64_t ldv, const int64_t vstride, T * __restrict__ H, const int hstride,
                              const int k1, const int jstep, T * __restrict__ partials, unsigned * __restrict__ tickets, const BatchArgs<T> p)
        {
            const int s = p.sys[blockIdx.y];
            T * Vs = V + (size_t)s * vstride;
            T * hs = H + (size_t)s * hstride;
            mgs_step_block<T>(n, Vs + (size_t)k1 * ldv, jstep > 0 ? Vs + (size_t)(jstep - 1) * ldv : nullptr, jstep < k1 ? Vs + (size_t)jstep * ldv : nullptr,
                              hs + (jstep > 0 ? jstep - 1 : 0), nullptr, partials + (size_t)s * gridDim.x, tickets + s, hs + jstep, jstep == k1 ? 1 : 0);
        }

        // w_s /= ||w_s|| (w_s = column k1 of system s, the norm at H[s * hstride + k1])
        template <typename T>
        __global__ void scal_inv_batch_kernel(const int64_t n, T * __restrict__ V, const int64_t ldv, const int64_t vstride, const T * __restrict__ H,
                                              const int hstride, const int k1, const BatchArgs<T> p)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            const int s = p.sys[blockIdx.y];
            const T a = inv_norm(H + (size_t)s * hstride + k1, 0);
            if (i < n)
                V[(size_t)s * vstride + (size_t)k1 * ldv + i] *= a;
        }

        // reduction workspace of one thread of execution
        struct RedWork
        {
            DevBuf<double> part_d, res_d;
            DevBuf<float> part_f, res_f;
            DevBuf<unsigned> ticket;
            void init()
            {
                part_d.alloc(MAX_RED_BLOCKS);
                part_f.alloc(MAX_RED_BLOCKS);
                res_d.alloc(64);
                res_f.alloc(64);
                ticket.alloc(1);
                CB_CUDA(cudaMemset(ticket.p, 0, sizeof(unsigned)));
            }
            template <typename T> T * part();
            template <typename T> T * res();
        };
        template <> double * RedWork::part<double>() { return part_d.p; }
        template <> float * RedWork::part<float>() { return part_f.p; }
        template <> double * RedWork::res<double>() { return res_d.p; }
        template <> float * RedWork::res<float>() { return res_f.p; }

        // BLAS-1 entry points (dot, dist): one workspace per (device, stream), so two streams / two devices of a process
        // never share a ticket or a partial buffer (the reference allocates a scalar per call, source/linalg.cpp:69)
        RedWork & work(cudaStream_t s)
        {
            static std::mutex mu;
            static std::map<std::pair<int, cudaStream_t>, std::unique_ptr<RedWork>> table;
            int dev = 0;
            cudaGetDevice(&dev);
            std::lock_guard<std::mutex> lock(mu);
            auto & slot = table[std::make_pair(dev, s)];
            if (!slot) {
                slot.reset(new RedWork);
                slot->init();
            }
            return *slot;
        }

        std::atomic<int> g_default_orth{ORTH_MGS};
    } // namespace

    int default_gmres_orth() { return g_default_orth.load(); }
    void set_default_gmres_orth(int v) { g_default_orth.store(v == ORTH_CGS2 ? ORTH_CGS2 : ORTH_MGS); }

    template <typename T> void axpby(int64_t n, T a, const T * x, T b, T * y, cudaStream_t s)
    {
        if (n <= 0) return;
        axpby_kernel<T><<<nblk(n), 256, 0, s>>>(n, a, x, b, y);
        CB_LAUNCHED();
    }
    template <typename T> void scal(int64_t n, T a, T * x, cudaStream_t s)
    {
        if (n <= 0) return;
        scal_kernel<T><<<nblk(n), 256, 0, s>>>(n, a, x);
        CB_LAUNCHED();
    }
    template <typename T> void fill(int64_t n, T a, T * x, cudaStream_t s)
    {
        if (n <= 0) return;
        fill_kernel<T><<<nblk(n), 256, 0, s>>>(n, a, x);
        CB_LAUNCHED();
    }
    template <typename T> void copy(int64_t n, const T * x, T * y, cudaStream_t s)
    {
        if (n <= 0) return;
        copy_kernel<T><<<nblk(n), 256, 0, s>>>(n, x, y);
        CB_LAUNCHED();
    }

    namespace
    {
        template <typename T, int MODE> T reduce_with(RedWork & w, int64_t n, const T * x, const T * y, cudaStream_t s)
        {
            reduce_kernel<T, MODE><<<red_blocks(n), RED_THREADS, 0, s>>>(n, x, y, w.part<T>(), w.ticket.p, w.res<T>(), 0);
            CB_LAUNCHED();
            T h;
            CB_CUDA(cudaMemcpyAsync(&h, w.res<T>(), sizeof(T), cudaMemcpyDeviceToHost, s));
            CB_CUDA(cudaStreamSynchronize(s));
            return h;
        }
    } // namespace

    template <typename T> T dot(int64_t n, const T * x, const T * y, cudaStream_t s)
    {
        if (n <= 0) return T(0);
        return reduce_with<T, 0>(work(s), n, x, y, s);
    }
    template <typename T> T dist(int64_t n, const T * x, const T * y, cudaStream_t s)
    {
        if (n <= 0) return T(0);
        return std::sqrt(reduce_with<T, 1>(work(s), n, x, y, s));
    }

#define CB_INST(T)                                                                         \
    template void axpby<T>(int64_t, T, const T *, T, T *, cudaStream_t);                   \
    template void scal<T>(int64_t, T, T *, cudaStream_t);                                  \
    template void fill<T>(int64_t, T, T *, cudaStream_t);                                  \
    template void copy<T>(int64_t, const T *, T *, cudaStream_t);                          \
    template T dot<T>(int64_t, const T *, const T *, cudaStream_t);                        \
    template T dist<T>(int64_t, const T *, const T *, cudaStream_t);
    CB_INST(double)
    CB_INST(float)
    template void fill<int>(int64_t, int, int *, cudaStream_t);
    template void copy<int>(int64_t, const int *, int *, cudaStream_t);
#undef CB_INST

    // ---------------------------------------------------------------------------------------------
    // GMRES(m): reference source/gmres.cpp:91-235 (t_gmres). Same control flow and stopping rules:
    //   it starts at 1 and runs while it < maxit; inner break on |eta_{k+1}| < tol*||b|| or H(k+1,k) == 0;
    //   true residual recomputed every restart; num_iter = it.
    // ---------------------------------------------------------------------------------------------
    namespace
    {
        template <typename T>
        void givens(T * h, T * cs, T * sn, int k) // gmres.cpp:7-23
        {
            for (int i = 0; i < k; ++i) {
                const T h1 = h[i], h2 = h[i + 1];
                h[i] = cs[i] * h1 + sn[i] * h2;
                h[i + 1] = -sn[i] * h1 + cs[i] * h2;
            }
            const T t = std::hypot(h[k], h[k + 1]);
            cs[k] = h[k] / t;
            sn[k] = h[k + 1] / t;
            h[k] = cs[k] * h[k] + sn[k] * h[k + 1];
            h[k + 1] = 0.0;
        }

        // upper-triangular solve R x = b in place (what dtrsv_/strsv_("U","N","N") compute; gmres.cpp:26-44)
        template <typename T>
        void trsv_upper(int n, const T * R, int ldr, T * b)
        {
            for (int j = n - 1; j >= 0; --j) {
                if (b[j] != T(0)) {
                    b[j] /= R[j + (size_t)ldr * j];
                    const T t = b[j];
                    for (int i = j - 1; i >= 0; --i)
                        b[i] -= t * R[i + (size_t)ldr * j];
                }
            }
        }

        struct Progress // gmres.cpp:46-66
        {
            int it = 0, nt;
            std::string bar;
            explicit Progress(int nt_) : nt(nt_), bar(30, ' ') {}
            void step()
            {
                it = std::min(it + 1, nt - 1);
                bar.at(30 * (it - 1) / nt) = '#';
            }
        };

        struct EventPair
        {
            cudaEvent_t a = nullptr, b = nullptr;
            bool on;
            explicit EventPair(bool on_) : on(on_)
            {
                if (on) {
                    CB_CUDA(cudaEventCreate(&a));
                    CB_CUDA(cudaEventCreate(&b));
                }
            }
            ~EventPair()
            {
                if (a) cudaEventDestroy(a);
                if (b) cudaEventDestroy(b);
            }
        };
    } // namespace

    template <typename T>
    GmresResult gmres(int64_t n, T * x, ApplyFn<T> A, void * ctx, const T * b, int m, int maxit, T tol, int verbose,
                      double max_seconds, cudaStream_t s, const GmresOptions & opt)
    {
        NvtxRange nvtx_solve(sizeof(T) == 8 ? "cuddh::gmres<double>" : "cuddh::gmres<float>");
        GmresResult out;
        out.success = false;
        out.num_iter = 0;
        out.num_matvec = 0;
        CB_REQUIRE(m >= 1, "gmres: m must be >= 1");
        CB_REQUIRE(n >= 0, "gmres: negative size");
        const T one = 1, zero = 0;
        const int m1 = m + 1;
        const Comm * comm = (opt.comm && opt.comm->world > 1) ? opt.comm : nullptr;
        const unsigned char * mask = opt.d_mask;
        const bool cgs = opt.orth == ORTH_CGS2;
        // basis columns on 16-byte boundaries (vector loads in every orthogonalisation kernel)
        const int64_t ldv = (n + 3) & ~int64_t(3);

        RedWork wk; // per call: concurrent solves never share a ticket
        wk.init();
        const int gx = red_blocks(n, 4);
        DevBuf<double> partials((size_t)(m1 + 1) * gx), sums((size_t)m1 + 2);
        std::vector<double> hsum((size_t)m1 + 2);

        auto apply = [&](const T * in, T * o) {
            const int rc = A(ctx, in, o, s);
            if (rc != 0)
                throw Error(rc, std::string("gmres: the operator callback failed (status ") + std::to_string(rc) + "): " + get_last_error());
            out.num_matvec++;
        };
        // <x, y> over the owned entries, summed over the ranks
        auto gdot = [&](const T * xx, const T * yy) -> double {
            if (!comm && !mask)
                return (double)reduce_with<T, 0>(wk, n, xx, yy, s);
            masked_dot_kernel<T><<<gx, RED_THREADS, 0, s>>>(n, xx, yy, mask, partials.p);
            CB_LAUNCHED();
            finish_sums_kernel<<<1, RED_THREADS, 0, s>>>(gx, partials.p, sums.p);
            CB_LAUNCHED();
            if (comm) {
                comm_allreduce_sum(comm, sums.p, 1, s);
                out.allreduces++;
            }
            double h;
            CB_CUDA(cudaMemcpyAsync(&h, sums.p, sizeof(double), cudaMemcpyDeviceToHost, s));
            CB_CUDA(cudaStreamSynchronize(s));
            return h;
        };

        const T bnrm = (T)std::sqrt(gdot(b, b));

        DevBuf<T> r_((size_t)n), V_((size_t)ldv * m1), hdev((size_t)m1 + 2), etadev((size_t)m1);
        T * r = r_.p;
        T * V = V_.p;
        CB_CUDA(cudaMemsetAsync(V, 0, sizeof(T) * (size_t)ldv * m1, s));
        // flexible right preconditioning: the preconditioned directions z_k = P v_k are kept (they, not the v_k, update x)
        ApplyFn<T> Pr = reinterpret_cast<ApplyFn<T>>(opt.right_precond);
        DevBuf<T> Z_;
        if (Pr)
            Z_.alloc((size_t)ldv * m);
        T * Z = Z_.p;

        std::vector<T> H((size_t)m1 * m, T(0)), sn(m, T(0)), cs(m, T(0)), eta(m1, T(0)), hcol((size_t)m1 + 2);

        apply(x, r);
        axpby<T>(n, one, b, -one, r, s);
        T r_nrm = (T)std::sqrt(gdot(r, r));
        out.res_norm.push_back((double)r_nrm);
        out.time.push_back(0.0);
        const auto t0 = std::chrono::high_resolution_clock::now();

        if (r_nrm < tol * bnrm) {
            out.success = true;
            if (verbose) {
                std::cout << "After 0 iterations, GMRES achieved rel. residual of " << out.res_norm.back() / bnrm << std::endl;
                std::cout << "GMRES successfully converged within desired tolerance." << std::endl;
            }
            return out;
        }

        Progress bar(maxit);
        if (verbose)
            std::cout << std::setprecision(5) << std::scientific;

        EventPair ev(opt.time_orth);
        const int rb = red_blocks(n);
        const double vb = (double)n * sizeof(T);

        // one CGS round on w against the k1 columns of V: sums[0..k1) = V^T w, sums[k1] = <w, w> (host copy in hsum)
        auto cgs_dots = [&](const T * w, int k1) {
            multi_dot_kernel<T><<<dim3((unsigned)gx, (unsigned)((k1 + JT - 1) / JT)), RED_THREADS, 0, s>>>(n, ldv, k1, V, w, mask, partials.p);
            CB_LAUNCHED();
            finish_sums_kernel<<<(unsigned)(k1 + 1), RED_THREADS, 0, s>>>(gx, partials.p, sums.p);
            CB_LAUNCHED();
            if (comm) {
                comm_allreduce_sum(comm, sums.p, k1 + 1, s);
                out.allreduces++;
            }
            CB_CUDA(cudaMemcpyAsync(hsum.data(), sums.p, sizeof(double) * (size_t)(k1 + 1), cudaMemcpyDeviceToHost, s));
            CB_CUDA(cudaStreamSynchronize(s));
            out.orth_bytes += vb * (k1 + 1 + (k1 + JT - 1) / JT - 1);
        };
        auto cgs_update = [&](T * w, int k1, double scale) {
            multi_update_kernel<T><<<(unsigned)gx * 2, RED_THREADS, sizeof(double) * (size_t)k1, s>>>(n, ldv, k1, V, sums.p, scale, w);
            CB_LAUNCHED();
            out.orth_bytes += vb * (k1 + 2);
        };

        int it = 1;
        for (; it < maxit; ++it) {
            NvtxRange nvtx_cycle("gmres restart cycle");
            axpby<T>(n, one / r_nrm, r, zero, V, s); // v0 = r / ||r||
            std::fill(eta.begin(), eta.end(), T(0));
            eta[0] = r_nrm;

            int k1 = 0;
            for (int k = 0; k < m; ++k) {
                k1 = k + 1;
                T * vk = V + (size_t)k * ldv;
                T * w = vk + ldv;
                if (Pr) {
                    T * zk = Z + (size_t)k * ldv;
                    const int rc = Pr(opt.right_precond_ctx, vk, zk, s);
                    if (rc != 0)
                        throw Error(rc, std::string("gmres: the preconditioner callback failed (status ") + std::to_string(rc) + "): " + get_last_error());
                    apply(zk, w);
                }
                else
                    apply(vk, w);
                T * Hk = &H[(size_t)m1 * k];

                if (ev.on)
                    CB_CUDA(cudaEventRecord(ev.a, s));
                NvtxRange nvtx_orth(cgs ? "gmres orthogonalise (CGS2)" : "gmres orthogonalise (MGS)");
                bool zero_w = false;
                if (cgs) {
                    cgs_dots(w, k1);
                    double ww = hsum[k1], hh = 0.0;
                    for (int j = 0; j < k1; ++j) {
                        Hk[j] = (T)hsum[j];
                        hh += hsum[j] * hsum[j];
                    }
                    double nn = ww - hh;
                    if (ww == 0.0)
                        zero_w = true;
                    else if (nn >= 0.5 * ww) // no cancellation: ||w - V h||^2 = <w,w> - h.h to full accuracy
                        cgs_update(w, k1, 1.0 / std::sqrt(nn));
                    else { // re-orthogonalise once ("twice is enough"): h2 = V^T w', w' -= V h2, h += h2
                        cgs_update(w, k1, 1.0);
                        cgs_dots(w, k1);
                        out.reorth++;
                        double h2 = 0.0;
                        for (int j = 0; j < k1; ++j) {
                            Hk[j] = (T)((double)Hk[j] + hsum[j]);
                            h2 += hsum[j] * hsum[j];
                        }
                        nn = std::max(hsum[k1] - h2, 0.0);
                        if (nn == 0.0)
                            zero_w = true;
                        else
                            cgs_update(w, k1, 1.0 / std::sqrt(nn));
                    }
                    Hk[k1] = zero_w ? T(0) : (T)std::sqrt(nn);
                }
                else {
                    // fused MGS sweep: step j computes h_j = <w, v_j> after applying h_{j-1}; the last step applies
                    // h_k and produces ||w|| (sqrt on the device, after the sum over ranks in a distributed run)
                    for (int j = 0; j <= k1; ++j) {
                        const T * vprev = (j > 0) ? V + (size_t)(j - 1) * ldv : nullptr;
                        const T * vnext = (j < k1) ? V + (size_t)j * ldv : nullptr;
                        mgs_step_kernel<T><<<rb, RED_THREADS, 0, s>>>(n, w, vprev, vnext, hdev.p + (j > 0 ? j - 1 : 0), mask, wk.part<T>(),
                                                                      wk.ticket.p, hdev.p + j, (j == k1 && !comm) ? 1 : 0);
                        CB_LAUNCHED();
                        if (comm) {
                            comm_allreduce_sum(comm, hdev.p + j, 1, s);
                            out.allreduces++;
                        }
                    }
                    scal_inv_dev_kernel<T><<<nblk(n), 256, 0, s>>>(n, hdev.p + k1, comm ? 1 : 0, w); // w /= ||w|| (inf/nan if 0: caught below)
                    CB_LAUNCHED();
                    CB_CUDA(cudaMemcpyAsync(hcol.data(), hdev.p, sizeof(T) * (size_t)(k1 + 1), cudaMemcpyDeviceToHost, s));
                    CB_CUDA(cudaStreamSynchronize(s));
                    for (int j = 0; j <= k1; ++j)
                        Hk[j] = hcol[j];
                    if (comm)
                        Hk[k1] = std::sqrt(Hk[k1]);
                    zero_w = Hk[k1] == T(0);
                    out.orth_bytes += vb * (2 + 4.0 * (k1 - 1) + 3 + 2);
                }
                if (ev.on) {
                    CB_CUDA(cudaEventRecord(ev.b, s));
                    CB_CUDA(cudaEventSynchronize(ev.b));
                    float ms = 0;
                    CB_CUDA(cudaEventElapsedTime(&ms, ev.a, ev.b));
                    out.orth_ms += ms;
                }

                if (zero_w) // gmres.cpp:176 (w was all zeros: undo the 0/0 scaling)
                {
                    CB_CUDA(cudaMemsetAsync(w, 0, sizeof(T) * (size_t)n, s));
                    break;
                }

                givens(Hk, cs.data(), sn.data(), k);
                eta[k1] = -sn[k] * eta[k];
                eta[k] = cs[k] * eta[k];

                if (std::abs(eta[k1]) < tol * bnrm)
                    break;
            }

            trsv_upper<T>(k1, H.data(), m1, eta.data());
            CB_CUDA(cudaMemcpyAsync(etadev.p, eta.data(), sizeof(T) * (size_t)k1, cudaMemcpyHostToDevice, s));
            multi_axpy_kernel<T><<<nblk(n), 256, 0, s>>>(n, ldv, k1, etadev.p, Pr ? Z : V, x);
            CB_LAUNCHED();

            apply(x, r);
            axpby<T>(n, one, b, -one, r, s);
            r_nrm = (T)std::sqrt(gdot(r, r));
            out.res_norm.push_back((double)r_nrm);
            const auto t1 = std::chrono::high_resolution_clock::now();
            const double dur = 1e-9 * std::chrono::duration_cast<std::chrono::nanoseconds>(t1 - t0).count();
            out.time.push_back(dur);
            if (dur > max_seconds)
                break;

            if (verbose == 1) {
                bar.step();
                std::cout << "[" << bar.bar << "] || iteration " << std::setw(10) << it + 1 << " / " << maxit
                          << " || rel. res. = " << std::setw(10) << r_nrm / bnrm << "\r" << std::flush;
            }
            else if (verbose >= 2)
                std::cout << "iteration " << std::setw(10) << it + 1 << " / " << maxit << " || rel. res. = " << std::setw(10)
                          << r_nrm / bnrm << std::endl;

            if (r_nrm < tol * bnrm) {
                out.success = true;
                break;
            }
        }

        if (verbose == 1)
            std::cout << std::endl;
        if (verbose) {
            std::cout << "After " << it << " iterations, GMRES achieved rel. residual of " << out.res_norm.back() / bnrm << std::endl;
            if (out.success)
                std::cout << "GMRES successfully converged within desired tolerance." << std::endl;
            else
                std::cout << "GMRES failed to converge within desired tolerance." << std::endl;
        }
        out.num_iter = it;
        return out;
    }

    // ---------------------------------------------------------------------------------------------
    // Lockstep batched GMRES(m), MGS arithmetic: k independent gmres(..., ORTH_MGS) solves that share their launches. All active
    // systems sit at the same Arnoldi index; every reduction of a system runs the single solve's kernel body on its own grid row
    // with red_blocks(n) blocks, its own partials and ticket, so each system's results are bitwise those of its own solve.
    // ---------------------------------------------------------------------------------------------
    template <typename T>
    std::vector<GmresResult> gmres_batch(int64_t n, int k, T * const * x, ApplyBatchFn<T> A, void * ctx, const T * const * b, int m, int maxit,
                                         T tol, double max_seconds, cudaStream_t s)
    {
        NvtxRange nvtx_solve("cuddh::gmres_batch<float>");
        CB_REQUIRE(k >= 1 && k <= GMRES_BATCH_KMAX, "gmres_batch: k must be in [1, " + std::to_string(GMRES_BATCH_KMAX) + "]");
        CB_REQUIRE(x != nullptr && b != nullptr, "gmres_batch: null pointer array");
        CB_REQUIRE(A != nullptr, "gmres_batch: null operator callback");
        CB_REQUIRE(m >= 1, "gmres_batch: m must be >= 1");
        CB_REQUIRE(n >= 0, "gmres_batch: negative size");
        for (int j = 0; j < k; ++j) {
            CB_REQUIRE(x[j] != nullptr && b[j] != nullptr, "gmres_batch: null vector pointer");
            for (int i = 0; i < j; ++i)
                CB_REQUIRE(x[j] + n <= x[i] || x[i] + n <= x[j], "gmres_batch: solution vectors " + std::to_string(i) + " and " + std::to_string(j) + " overlap");
        }

        std::vector<GmresResult> out((size_t)k);
        for (auto & o : out) {
            o.success = false;
            o.num_iter = 0;
            o.num_matvec = 0;
        }
        const T one = 1, zero = 0;
        const int m1 = m + 1, hstride = m1 + 2;
        const int64_t ldv = (n + 3) & ~int64_t(3), vstride = ldv * m1;
        const int rb = red_blocks(n);

        DevBuf<T> R_((size_t)ldv * k), V_((size_t)vstride * k), H_((size_t)hstride * k), part_((size_t)rb * k), res_((size_t)2 * k),
            eta_((size_t)m1 * k);
        DevBuf<unsigned> tick_((size_t)k);
        CB_CUDA(cudaMemsetAsync(tick_.p, 0, sizeof(unsigned) * (size_t)k, s));
        CB_CUDA(cudaMemsetAsync(V_.p, 0, sizeof(T) * (size_t)vstride * k, s));
        auto Rv = [&](int j) { return R_.p + (size_t)j * ldv; };
        auto Vv = [&](int j, int col) { return V_.p + (size_t)j * vstride + (size_t)col * ldv; };

        // per-system host state of the single solve
        std::vector<T> H((size_t)k * m1 * m, T(0)), sn((size_t)k * m, T(0)), cs((size_t)k * m, T(0)), eta((size_t)k * m1, T(0)),
            hcol((size_t)k * hstride), hres((size_t)2 * k), bnrm(k), r_nrm(k);
        std::vector<int> k1s(k, 0);

        std::vector<const T *> ain;
        std::vector<T *> aout;
        // A on the listed systems, in[j] -> out[j]
        auto apply = [&](const std::vector<int> & sys, auto in_of, auto out_of) {
            ain.clear();
            aout.clear();
            for (int j : sys) {
                ain.push_back(in_of(j));
                aout.push_back(out_of(j));
            }
            const int rc = A(ctx, (int)sys.size(), ain.data(), aout.data(), s);
            if (rc != 0)
                throw Error(rc, std::string("gmres_batch: the operator callback failed (status ") + std::to_string(rc) + "): " + get_last_error());
            for (int j : sys)
                out[j].num_matvec++;
        };
        auto args_of = [&](const std::vector<int> & sys) {
            BatchArgs<T> a{};
            for (size_t i = 0; i < sys.size(); ++i)
                a.sys[i] = sys[i];
            return a;
        };
        // r_j = b_j - r_j
        auto residual = [&](const std::vector<int> & sys) {
            BatchArgs<T> a = args_of(sys);
            for (size_t i = 0; i < sys.size(); ++i) {
                a.x[i] = b[sys[i]];
                a.y[i] = Rv(sys[i]);
                a.a[i] = one;
                a.b[i] = -one;
            }
            axpby_batch_kernel<T><<<dim3(nblk(n), (unsigned)sys.size()), 256, 0, s>>>(n, a);
            CB_LAUNCHED();
        };
        // <v_j, v_j> of the listed systems -> res_[off + i]
        auto norms2 = [&](const std::vector<int> & sys, auto vec_of, int off) {
            BatchArgs<T> a = args_of(sys);
            for (size_t i = 0; i < sys.size(); ++i)
                a.x[i] = vec_of(sys[i]);
            norm2_batch_kernel<T><<<dim3((unsigned)rb, (unsigned)sys.size()), RED_THREADS, 0, s>>>(n, part_.p, tick_.p, res_.p + off, a);
            CB_LAUNCHED();
        };
        auto fetch = [&](T * dst, const T * src, size_t count) {
            CB_CUDA(cudaMemcpyAsync(dst, src, sizeof(T) * count, cudaMemcpyDeviceToHost, s));
            CB_CUDA(cudaStreamSynchronize(s));
        };

        std::vector<int> active(k);
        for (int j = 0; j < k; ++j)
            active[j] = j;
        apply(active, [&](int j) { return (const T *)x[j]; }, Rv);
        residual(active);
        norms2(active, [&](int j) { return b[j]; }, 0);
        norms2(active, [&](int j) { return (const T *)Rv(j); }, k);
        fetch(hres.data(), res_.p, (size_t)2 * k);
        {
            std::vector<int> still;
            for (int j = 0; j < k; ++j) {
                bnrm[j] = (T)std::sqrt((double)hres[j]);
                r_nrm[j] = (T)std::sqrt((double)hres[k + j]);
                out[j].res_norm.push_back((double)r_nrm[j]);
                out[j].time.push_back(0.0);
                if (r_nrm[j] < tol * bnrm[j])
                    out[j].success = true; // converged at the initial guess: 0 iterations
                else
                    still.push_back(j);
            }
            active.swap(still);
        }
        const auto t0 = std::chrono::high_resolution_clock::now();

        int it = 1;
        for (; it < maxit && !active.empty(); ++it) {
            NvtxRange nvtx_cycle("gmres_batch restart cycle");
            {
                BatchArgs<T> a = args_of(active); // v0 = r / ||r||
                for (size_t i = 0; i < active.size(); ++i) {
                    const int j = active[i];
                    a.x[i] = Rv(j);
                    a.y[i] = Vv(j, 0);
                    a.a[i] = one / r_nrm[j];
                    a.b[i] = zero;
                    std::fill(eta.begin() + (size_t)j * m1, eta.begin() + (size_t)(j + 1) * m1, T(0));
                    eta[(size_t)j * m1] = r_nrm[j];
                    k1s[j] = 0;
                }
                axpby_batch_kernel<T><<<dim3(nblk(n), (unsigned)active.size()), 256, 0, s>>>(n, a);
                CB_LAUNCHED();
            }

            std::vector<int> inner = active; // systems still in this cycle's Arnoldi loop
            for (int kk = 0; kk < m && !inner.empty(); ++kk) {
                const int k1 = kk + 1;
                for (int j : inner)
                    k1s[j] = k1;
                apply(inner, [&](int j) { return (const T *)Vv(j, kk); }, [&](int j) { return Vv(j, k1); });
                const BatchArgs<T> a = args_of(inner);
                const dim3 grid_red((unsigned)rb, (unsigned)inner.size()), grid_el(nblk(n), (unsigned)inner.size());
                {
                    NvtxRange nvtx_orth("gmres_batch orthogonalise (MGS)");
                    for (int js = 0; js <= k1; ++js) {
                        mgs_step_batch_kernel<T><<<grid_red, RED_THREADS, 0, s>>>(n, V_.p, ldv, vstride, H_.p, hstride, k1, js, part_.p, tick_.p, a);
                        CB_LAUNCHED();
                    }
                    scal_inv_batch_kernel<T><<<grid_el, 256, 0, s>>>(n, V_.p, ldv, vstride, H_.p, hstride, k1, a);
                    CB_LAUNCHED();
                    fetch(hcol.data(), H_.p, (size_t)k * hstride);
                }
                std::vector<int> next;
                for (int j : inner) {
                    T * Hk = &H[(size_t)j * m1 * m + (size_t)m1 * kk];
                    for (int i = 0; i <= k1; ++i)
                        Hk[i] = hcol[(size_t)j * hstride + i];
                    if (Hk[k1] == T(0)) { // w was all zeros: undo the 0/0 scaling and wait for the restart
                        CB_CUDA(cudaMemsetAsync(Vv(j, k1), 0, sizeof(T) * (size_t)n, s));
                        continue;
                    }
                    T * e = &eta[(size_t)j * m1];
                    T * c = &cs[(size_t)j * m];
                    T * sg = &sn[(size_t)j * m];
                    givens(Hk, c, sg, kk);
                    e[k1] = -sg[kk] * e[kk];
                    e[kk] = c[kk] * e[kk];
                    if (std::abs(e[k1]) < tol * bnrm[j])
                        continue;
                    next.push_back(j);
                }
                inner.swap(next);
            }

            // restart tail: x += V eta, true residual
            for (int j : active)
                trsv_upper<T>(k1s[j], &H[(size_t)j * m1 * m], m1, &eta[(size_t)j * m1]);
            CB_CUDA(cudaMemcpyAsync(eta_.p, eta.data(), sizeof(T) * eta.size(), cudaMemcpyHostToDevice, s));
            {
                BatchArgs<T> a = args_of(active);
                for (size_t i = 0; i < active.size(); ++i) {
                    const int j = active[i];
                    a.x[i] = Vv(j, 0);
                    a.y[i] = x[j];
                    a.k1[i] = k1s[j];
                }
                multi_axpy_batch_kernel<T><<<dim3(nblk(n), (unsigned)active.size()), 256, 0, s>>>(n, ldv, eta_.p, m1, a);
                CB_LAUNCHED();
            }
            apply(active, [&](int j) { return (const T *)x[j]; }, Rv);
            residual(active);
            norms2(active, [&](int j) { return (const T *)Rv(j); }, 0);
            fetch(hres.data(), res_.p, active.size());
            const auto t1 = std::chrono::high_resolution_clock::now();
            const double dur = 1e-9 * std::chrono::duration_cast<std::chrono::nanoseconds>(t1 - t0).count();
            std::vector<int> still;
            for (size_t i = 0; i < active.size(); ++i) {
                const int j = active[i];
                r_nrm[j] = (T)std::sqrt((double)hres[i]);
                out[j].res_norm.push_back((double)r_nrm[j]);
                out[j].time.push_back(dur);
                if (dur > max_seconds)
                    out[j].num_iter = it;
                else if (r_nrm[j] < tol * bnrm[j]) {
                    out[j].success = true;
                    out[j].num_iter = it;
                }
                else
                    still.push_back(j);
            }
            active.swap(still);
        }
        for (int j : active)
            out[j].num_iter = it;
        return out;
    }

    template std::vector<GmresResult> gmres_batch<float>(int64_t, int, float * const *, ApplyBatchFn<float>, void *, const float * const *, int, int,
                                                         float, double, cudaStream_t);

    template GmresResult gmres<double>(int64_t, double *, ApplyFn<double>, void *, const double *, int, int, double, int, double, cudaStream_t,
                                       const GmresOptions &);
    template GmresResult gmres<float>(int64_t, float *, ApplyFn<float>, void *, const float *, int, int, float, int, double, cudaStream_t,
                                      const GmresOptions &);
} // namespace cb200
