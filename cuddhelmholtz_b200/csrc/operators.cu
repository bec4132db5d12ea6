// FP64 matrix-free operator actions for sm_100a (path A): stiffness, mass, face mass.
//
// What the reference does (source/StiffnessMatrix.cpp:83-184, source/MassMatrix.cpp:137-211): one CTA of
// nq*nq threads per element, 1-D tables re-read from global memory by every CTA, 4 barriers, FP64
// atomicAdd scatter preceded by a cudaMemset. What this file does instead:
//
//   * one CTA per PATCH of elements (assembly plan, h1space.cpp). The patch's unique DOFs are gathered once,
//     coalesced, into shared memory; element results are accumulated into a patch-local vector colour by
//     colour (fixed order, no atomics) and written back with plain coalesced stores. Only DOFs on patch
//     boundaries (~12%) take a detour through a partial buffer that a second tiny kernel sums in patch
//     order. The result is bitwise reproducible and needs no memset.
//   * inside a patch, a warp processes EPW = 32/NQ elements at a time with NQ lanes per element. Each
//     lane owns a whole tensor row/column in registers, so the sum-factorised contractions are pure
//     register DFMA chains whose table operands (P, D) come from the kernel-parameter constant bank
//     (__grid_constant__): no shared-memory reads for the tables at all. The two transposes an element
//     needs go through a small per-warp scratch with __syncwarp only.
//   * the metric data (G for stiffness, a*w*w*detJ for mass) is stored in "lane-major" plan order so that
//     every load instruction of a warp reads one contiguous run; it is prefetched into registers before
//     the first contraction, streamed with an evict-first hint.
//
// Contraction order. Let U = u[I] (nb x nb), F = metric applied at quadrature points. The reference forms
//   Su[a][b] = sum_j P(j,b) (sum_i D(i,a) F0[i][j]) + D(j,b) (sum_i P(i,a) F1[i][j]);
// here the j-sum (local to a lane) is done first and the i-sum second: same flops, one transpose fewer.
// The difference is floating-point re-association only (tests bound it at 1e-12 relative).
#include "operators.hpp"
#include <algorithm>
#include <cmath>
#include <type_traits>

namespace cb200
{
    namespace
    {
        constexpr int MAXQ = 32;
        constexpr int MAX_DEVICES = 64;
        std::atomic<int> g_max_ctas{0};

        struct PlanDev
        {
            const PatchHdr * hdr;
            const int * gid;
            const int * slot;
            const uint16_t * L;
            const uint16_t * cptr;
            const uint16_t * cent;
            int PE;
            const int * Ig; // node-major plans: global DOF of (patch, node / 4, slot, node % 4)
            const uint2 * cent4; // node-major plans: first four CSR entries of every patch-local DOF (Plan::cent4)
            const int * target;  // node-major plans: global DOF / partial slot of every patch-local DOF
        };

        // 1-D tables as a kernel parameter (constant bank). Both orientations are stored so that every inner loop
        // reads one contiguous, even-padded row: Prow[q][k] = P(q,k) (contractions over the basis index),
        // Pcol[t][i] = P(i,t) (contractions over the quadrature index).
        template <int NB, int NQ, bool STIFF>
        struct Tables
        {
            static constexpr int NBP = (NB + 1) & ~1;
            static constexpr int NQP = (NQ + 1) & ~1;
            double Prow[NQ][NBP];
            double Pcol[NB][NQP];
            double Drow[STIFF ? NQ : 1][NBP];
            double Dcol[STIFF ? NB : 1][NQP];
            // rows scaled by the quadrature weight, PWrow[q][k] = w_q P(q,k): back-contractions of the affine stiffness phase
            double PWrow[STIFF ? NQ : 1][NBP];
            double DWrow[STIFF ? NQ : 1][NBP];
            // mass: msc * P(q,k), the phase scale (1, or -omega^2 inside the Helmholtz composite) folded into the last back-contraction
            double PSrow[STIFF ? 1 : NQ][NBP];
        };

        // Padded layout of the per-element transpose scratch: element stride S, row stride RS, offset HALF of the second
        // (derivative) plane, all in doubles. Chosen by exhaustive search (profiles/r01_notes.md) so that the four access
        // patterns of the two transposes (column writes, row reads, row writes, column reads of NQ-lane groups, 64-bit
        // accesses resolved per half-warp) hit distinct bank pairs: e.g. n_basis 5 / n_quad 6 stiffness goes from 176 to
        // 88 shared-memory wavefronts per warp pass, the minimum for 44 64-bit instructions.
        struct ScrLayout
        {
            int S, RS, HALF;
        };
        template <int NB, int NQ, bool STIFF>
        __host__ __device__ constexpr ScrLayout scr_layout()
        {
            if (STIFF == true && NB == 2 && NQ == 3) return {25, 3, 9};
            if (STIFF == true && NB == 3 && NQ == 4) return {28, 3, 12};
            if (STIFF == true && NB == 4 && NQ == 5) return {74, 7, 35};
            if (STIFF == true && NB == 5 && NQ == 6) return {70, 5, 30}; // 128 wavefronts; {118, 9, 54} reaches 88 but costs a CTA per SM
            if (STIFF == true && NB == 6 && NQ == 7) return {87, 6, 42};
            if (STIFF == true && NB == 7 && NQ == 8) return {120, 7, 56};
            if (STIFF == true && NB == 8 && NQ == 9) return {201, 11, 99};
            if (STIFF == true && NB == 9 && NQ == 10) return {186, 9, 90};
            if (STIFF == true && NB == 3 && NQ == 5) return {83, 7, 35};
            if (STIFF == true && NB == 4 && NQ == 6) return {90, 7, 42};
            if (STIFF == true && NB == 5 && NQ == 7) return {71, 5, 35};
            if (STIFF == true && NB == 6 && NQ == 8) return {103, 6, 48};
            if (STIFF == true && NB == 7 && NQ == 9) return {201, 11, 99};
            if (STIFF == true && NB == 8 && NQ == 10) return {186, 9, 90};
            if (STIFF == false && NB == 2 && NQ == 3) return {9, 3, 0};
            if (STIFF == false && NB == 3 && NQ == 4) return {12, 3, 0};
            if (STIFF == false && NB == 4 && NQ == 5) return {42, 7, 0};
            if (STIFF == false && NB == 5 && NQ == 6) return {54, 9, 0};
            if (STIFF == false && NB == 6 && NQ == 7) return {54, 7, 0};
            if (STIFF == false && NB == 7 && NQ == 8) return {56, 7, 0};
            if (STIFF == false && NB == 8 && NQ == 9) return {105, 11, 0};
            if (STIFF == false && NB == 9 && NQ == 10) return {90, 9, 0};
            if (STIFF == false && NB == 3 && NQ == 5) return {35, 7, 0};
            if (STIFF == false && NB == 4 && NQ == 6) return {42, 7, 0};
            if (STIFF == false && NB == 5 && NQ == 7) return {39, 5, 0};
            if (STIFF == false && NB == 6 && NQ == 8) return {55, 6, 0};
            if (STIFF == false && NB == 7 && NQ == 9) return {105, 11, 0};
            if (STIFF == false && NB == 8 && NQ == 10) return {90, 9, 0};
            if (STIFF == false && NB == 2 && NQ == 5) return {25, 5, 0};
            if (STIFF == false && NB == 3 && NQ == 6) return {42, 7, 0};
            if (STIFF == false && NB == 4 && NQ == 8) return {40, 5, 0};
            if (STIFF == false && NB == 5 && NQ == 9) return {54, 5, 0};
            if (STIFF == false && NB == 6 && NQ == 11) return {71, 6, 0};
            if (STIFF == false && NB == 7 && NQ == 12) return {108, 9, 0};
            if (STIFF == false && NB == 8 && NQ == 14) return {126, 9, 0};
            if (STIFF == false && NB == 9 && NQ == 15) return {137, 9, 0};
            return {(STIFF ? 2 : 1) * NQ * NB, NB, STIFF ? NQ * NB : 0};
        }

        __device__ __forceinline__ double ld_stream(const double * p)
        {
            return __ldcs(p);
        }

        // cp.async.bulk.prefetch.L2 (TMA bulk prefetch): size a multiple of 16 bytes, 16-byte aligned address
        __device__ __forceinline__ void bulk_prefetch_l2(const void * p, size_t bytes)
        {
            // align the window inwards/down to 16 bytes: a prefetch is a hint, losing a few bytes at the edges is fine
            const size_t a = reinterpret_cast<size_t>(p);
            const size_t a0 = a & ~size_t(15);
            const unsigned n = (unsigned)((bytes + (a - a0)) & ~size_t(15));
            if (n)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a0), "r"(n) : "memory");
        }

        // ------------------------------------------------------------------------------------------
        // main action kernel
        // ------------------------------------------------------------------------------------------
        // ------------------------------------------------------------------------------------------
        // Phase B of the action kernels: the sum-factorised contractions of one patch. A warp processes EPW = 32/NQ
        // elements per pass with NQ lanes per element; results go to su[(slot, node)].
        // ------------------------------------------------------------------------------------------
        template <int NB, int NQ, bool STIFF>
        __device__ __forceinline__ void contract_patch(const Tables<NB, NQ, STIFF> & tab, const double * __restrict__ G, const int patch,
                                                       const int n_pass_patch, const int n_elem, const int lane, const int warp,
                                                       const int nwarps, const double * xloc, const uint16_t * Ls, double * scratch,
                                                       double * su)
        {
            constexpr int EPW = 32 / NQ;
            constexpr int LW = EPW * NQ;
            constexpr int NB2 = NB * NB;
            constexpr int NK = STIFF ? 3 * NQ : NQ;
            constexpr int NKI = STIFF ? 3 : 1;
            constexpr int PD = STIFF ? 2 : 4;
            constexpr ScrLayout LY = scr_layout<NB, NQ, STIFF>();
            constexpr int SCR = LY.S, RS = LY.RS, HALF = LY.HALF;
            const int el_local = lane / NQ;
            const int r = lane - el_local * NQ; // row / column owned by this lane
            double * sc = scratch + (warp * EPW + el_local) * SCR;
            const int n_pass = (n_elem + EPW - 1) / EPW;

            for (int pass = warp; pass < n_pass; pass += nwarps) {
                const int e = pass * EPW + el_local;
                const bool live = (lane < LW) && (e < n_elem);
                // this lane's metric values: row r of the element, NKI values per quadrature column, kept PD columns
                // ahead of the contraction in a register ring (the loads hit L2: the whole patch was bulk-prefetched)
                const double * gp = G + ((size_t)patch * n_pass_patch + pass) * (size_t)(NK * LW) + lane;
                double gring[PD][NKI];
                if (lane < LW) {
#pragma unroll
                    for (int i = 0; i < PD; ++i)
#pragma unroll
                        for (int a = 0; a < NKI; ++a)
                            gring[i][a] = (i < NQ) ? ld_stream(gp + (NKI * i + a) * LW) : 0.0;
                }

                // stage 1: lane j = r < NB holds column j of U; contracts the first index with P (and D)
                if (live && r < NB) {
                    double u[NB];
                    const uint16_t * Le = Ls + e * NB2 + NB * r;
#pragma unroll
                    for (int k = 0; k < NB; ++k)
                        u[k] = xloc[Le[k]];
#pragma unroll 1
                    for (int q = 0; q < NQ; ++q) {
                        double pu = 0.0, du = 0.0;
#pragma unroll
                        for (int k = 0; k < NB; ++k) {
                            pu = fma(tab.Prow[q][k], u[k], pu);
                            if (STIFF)
                                du = fma(tab.Drow[q][k], u[k], du);
                        }
                        sc[q * RS + r] = pu;
                        if (STIFF)
                            sc[HALF + q * RS + r] = du;
                    }
                }
                __syncwarp();

                // stage 2: lane q = r holds row q; second-index contraction, metric, and the transposed
                // second-index contraction back to the basis
                double a0[NB], a1[STIFF ? NB : 1];
                if (lane < LW) {
                    double pu[NB], du[STIFF ? NB : 1];
#pragma unroll
                    for (int l = 0; l < NB; ++l) {
                        pu[l] = live ? sc[r * RS + l] : 0.0;
                        if (STIFF)
                            du[l] = live ? sc[HALF + r * RS + l] : 0.0;
                    }
#pragma unroll
                    for (int t = 0; t < NB; ++t) {
                        a0[t] = 0.0;
                        if (STIFF)
                            a1[t] = 0.0;
                    }
#pragma unroll 1
                    for (int ty0 = 0; ty0 < NQ; ty0 += PD) {
#pragma unroll
                        for (int i = 0; i < PD; ++i) {
                            const int ty = ty0 + i;
                            if (ty < NQ) {
                                double gcur[NKI];
#pragma unroll
                                for (int a = 0; a < NKI; ++a)
                                    gcur[a] = gring[i][a];
                                if (ty + PD < NQ) {
#pragma unroll
                                    for (int a = 0; a < NKI; ++a)
                                        gring[i][a] = ld_stream(gp + (NKI * (ty + PD) + a) * LW);
                                }
                                if (STIFF) {
                                    double Dx = 0.0, Dy = 0.0;
#pragma unroll
                                    for (int l = 0; l < NB; ++l) {
                                        Dx = fma(tab.Prow[ty][l], du[l], Dx);
                                        Dy = fma(tab.Drow[ty][l], pu[l], Dy);
                                    }
                                    const double A = gcur[0], B = gcur[NKI > 1 ? 1 : 0], C = gcur[NKI > 2 ? 2 : 0];
                                    const double F0 = A * Dx + B * Dy;
                                    const double F1 = B * Dx + C * Dy;
#pragma unroll
                                    for (int t = 0; t < NB; ++t) {
                                        a0[t] = fma(tab.Prow[ty][t], F0, a0[t]);
                                        a1[t] = fma(tab.Drow[ty][t], F1, a1[t]);
                                    }
                                }
                                else {
                                    double ppu = 0.0;
#pragma unroll
                                    for (int l = 0; l < NB; ++l)
                                        ppu = fma(tab.Prow[ty][l], pu[l], ppu);
                                    const double val = gcur[0] * ppu;
#pragma unroll
                                    for (int t = 0; t < NB; ++t)
                                        a0[t] = fma(tab.Prow[ty][t], val, a0[t]);
                                }
                            }
                        }
                    }
                }
                __syncwarp();
                if (live) {
#pragma unroll
                    for (int t = 0; t < NB; ++t) {
                        sc[r * RS + t] = a0[t];
                        if (STIFF)
                            sc[HALF + r * RS + t] = a1[t];
                    }
                }
                __syncwarp();

                // stage 3: lane b = r < NB contracts the first index back to the basis
                if (live && r < NB) {
                    double A0[NQ], A1[STIFF ? NQ : 1];
#pragma unroll
                    for (int i = 0; i < NQ; ++i) {
                        A0[i] = sc[i * RS + r];
                        if (STIFF)
                            A1[i] = sc[HALF + i * RS + r];
                    }
                    double * so = su + e * NB2 + NB * r;
#pragma unroll 1
                    for (int t = 0; t < NB; ++t) {
                        double s0 = 0.0, s1 = 0.0;
#pragma unroll
                        for (int i = 0; i < NQ; ++i) {
                            if (STIFF) {
                                s0 = fma(tab.Dcol[t][i], A0[i], s0);
                                s1 = fma(tab.Pcol[t][i], A1[i], s1);
                            }
                            else
                                s0 = fma(tab.Pcol[t][i], A0[i], s0);
                        }
                        so[t] = STIFF ? (s0 + s1) : s0;
                    }
                }
                __syncwarp();
            }
        }

        // Outer loops of the three contraction stages are deliberately NOT unrolled (#pragma unroll 1): with rolled
        // loops ptxas streams each table row through uniform registers (one LDCU per DFMA pair) and the kernel needs
        // ~70 registers; fully unrolled it runs out of the 63 uniform registers, parks the tables in ~120 regular
        // registers and shuffles them back with R2UR (190 registers, 1 CTA / SM, issue-bound: profiles/r01_*).
        template <int NB, int NQ, bool STIFF>
        __global__ void __launch_bounds__(256, (NB <= 6 ? 3 : 2))
        volume_action_kernel(const __grid_constant__ Tables<NB, NQ, STIFF> tab, const PlanDev plan,
                             const double * __restrict__ G, const double * __restrict__ x, double * __restrict__ y,
                             double * __restrict__ partial, const double c, const int accumulate, const int max_pdof,
                             const int n_patches, const int pf_dist)
        {
            constexpr int EPW = 32 / NQ;          // elements per warp pass
            constexpr int LW = EPW * NQ;          // active lanes
            constexpr int NB2 = NB * NB;
            constexpr int NK = STIFF ? 3 * NQ : NQ; // metric values per lane
            constexpr int SCR = scr_layout<NB, NQ, STIFF>().S; // scratch doubles per element (padded; layout: contract_patch)

            extern __shared__ __align__(16) unsigned char smem_raw[];
            const int PE = plan.PE;
            const int n_pass_patch = (PE + EPW - 1) / EPW;
            const int nwarps = blockDim.x >> 5;
            double * xloc = reinterpret_cast<double *>(smem_raw);
            double * su = xloc + max_pdof;
            double * scratch = su + PE * NB2;
            int * gids = reinterpret_cast<int *>(scratch + nwarps * EPW * SCR);
            uint16_t * Ls = reinterpret_cast<uint16_t *>(gids + max_pdof);
            uint16_t * cents = Ls + PE * NB2;          // PE*NB2 is even: stays 4-byte aligned
            uint16_t * cptrs = cents + PE * NB2;       // max_pdof + 1 (+1 pad) entries

            const int tid = threadIdx.x;
            const int lane = tid & 31;
            const int warp = tid >> 5;
            const PatchHdr hdr = plan.hdr[blockIdx.x];

            // The patch's metric data is one contiguous block (plan order): pull it into L2 with a single bulk
            // prefetch while the gather below is in flight, so that the per-column loads of stage 2 are L2 hits.
            // The same is done one scheduling wave ahead (patch blockIdx.x + pf_dist) for that patch's metric block,
            // local map and assembly lists, so that its staging phase runs at L2 instead of DRAM latency.
            const int pnext = (pf_dist > 0 && (int)blockIdx.x + pf_dist < n_patches) ? (int)blockIdx.x + pf_dist : -1;
            const size_t g_patch = (size_t)n_pass_patch * NK * LW;
            if (tid == 0) {
                bulk_prefetch_l2(G + (size_t)blockIdx.x * g_patch, g_patch * sizeof(double));
                if (pnext >= 0) {
                    bulk_prefetch_l2(G + (size_t)pnext * g_patch, g_patch * sizeof(double));
                    bulk_prefetch_l2(plan.L + (size_t)pnext * PE * NB2, (size_t)PE * NB2 * sizeof(uint16_t));
                    bulk_prefetch_l2(plan.cent + (size_t)pnext * PE * NB2, (size_t)PE * NB2 * sizeof(uint16_t));
                }
            }
            PatchHdr hnext;
            if (tid == 32 && pnext >= 0)
                hnext = plan.hdr[pnext];

            // ---- A. stage the patch: gather x, zero the accumulator, copy the local map ----
            // (index loads, then value loads, then stores: AU independent gathers in flight per thread)
            {
                constexpr int AU = 6;
                const int * gidp = plan.gid + hdr.pdof_begin;
                for (int base = tid; base < hdr.n_pdof; base += AU * blockDim.x) {
                    int gi[AU];
                    double xv[AU];
#pragma unroll
                    for (int a = 0; a < AU; ++a) {
                        const int d = base + a * blockDim.x;
                        gi[a] = (d < hdr.n_pdof) ? __ldg(gidp + d) : -1;
                    }
#pragma unroll
                    for (int a = 0; a < AU; ++a)
                        xv[a] = (gi[a] >= 0) ? __ldg(x + gi[a]) : 0.0;
#pragma unroll
                    for (int a = 0; a < AU; ++a) {
                        const int d = base + a * blockDim.x;
                        if (d < hdr.n_pdof) {
                            xloc[d] = xv[a];
                            gids[d] = gi[a];
                        }
                    }
                }
                // local map: PE*NB2 is even for every patch shape, so copy two 16-bit entries at a time
                const uint32_t * Lg = reinterpret_cast<const uint32_t *>(plan.L + (size_t)hdr.elem_begin * NB2);
                uint32_t * Ls32 = reinterpret_cast<uint32_t *>(Ls);
                const int n32 = (hdr.n_elem * NB2 + 1) >> 1;
                const uint32_t * Cg = reinterpret_cast<const uint32_t *>(plan.cent + (size_t)hdr.elem_begin * NB2);
                uint32_t * Cs32 = reinterpret_cast<uint32_t *>(cents);
                for (int k = tid; k < n32; k += blockDim.x) {
                    Ls32[k] = __ldg(Lg + k);
                    Cs32[k] = __ldg(Cg + k);
                }
                const uint16_t * cpg = plan.cptr + hdr.cptr_begin;
                for (int k = tid; k <= hdr.n_pdof; k += blockDim.x)
                    cptrs[k] = __ldg(cpg + k);
            }
            if (tid == 32 && pnext >= 0) { // 16-byte aligned windows around the next patch's index lists
                const int * g0 = plan.gid + (hnext.pdof_begin & ~3);
                bulk_prefetch_l2(g0, ((size_t)hnext.n_pdof + 4) * sizeof(int));
                const uint16_t * c0 = plan.cptr + (hnext.cptr_begin & ~7);
                bulk_prefetch_l2(c0, ((size_t)hnext.n_pdof + 9) * sizeof(uint16_t));
            }
            __syncthreads();

            // ---- B. element contractions ----
            contract_patch<NB, NQ, STIFF>(tab, G, (int)blockIdx.x, n_pass_patch, hdr.n_elem, lane, warp, nwarps, xloc, Ls, scratch, su);
            __syncthreads();

            // ---- C. deterministic assembly + write-back. One thread per patch-local DOF adds the DOF's element
            //      contributions in the fixed order of the plan's CSR (no atomics, no colouring, no accumulator
            //      array); patch-private DOFs go straight to y, shared ones to their slot of the partial buffer. ----
            {
                const int * slotp = plan.slot + hdr.slot_begin - hdr.n_int;
                for (int d = tid; d < hdr.n_pdof; d += blockDim.x) {
                    const int b = cptrs[d], e = cptrs[d + 1];
                    double sum = 0.0;
                    for (int k = b; k < e; ++k)
                        sum += su[cents[k]];
                    if (d < hdr.n_int) {
                        const int gi = gids[d];
                        const double v = c * sum;
                        y[gi] = accumulate ? (y[gi] + v) : v;
                    }
                    else
                        partial[__ldg(slotp + d)] = sum;
                }
            }
        }

#include "volume_ws.cuh" // the warp-specialised thread-per-element kernel and its metric ring (device code only)
#include "volume_pair.cuh" // the thread-pair-per-element kernel of the high orders (device code only)

        // generic fallback for (nb, nq) pairs without a template instance: same algorithm and data layout
        // with EPW = 1 (one element per warp pass), runtime loops, tables in global memory.
        __global__ void __launch_bounds__(256)
        volume_action_generic(const int NB, const int NQ, const int STIFF, const double * __restrict__ Pt,
                              const double * __restrict__ Dt, const PlanDev plan, const double * __restrict__ G,
                              const double * __restrict__ x, double * __restrict__ y, double * __restrict__ partial,
                              const double c, const int accumulate, const int max_pdof)
        {
            extern __shared__ __align__(16) unsigned char smem_raw[];
            const int NB2 = NB * NB;
            const int NK = STIFF ? 3 * NQ : NQ;
            const int SCR = (STIFF ? 2 : 1) * NQ * NB;
            const int PE = plan.PE;
            const int nwarps = blockDim.x >> 5;
            double * xloc = reinterpret_cast<double *>(smem_raw);
            double * su = xloc + max_pdof;
            double * scratch = su + PE * NB2;
            uint16_t * Ls = reinterpret_cast<uint16_t *>(scratch + nwarps * SCR);
            const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
            const PatchHdr hdr = plan.hdr[blockIdx.x];

            for (int d = tid; d < hdr.n_pdof; d += blockDim.x)
                xloc[d] = __ldg(x + __ldg(plan.gid + hdr.pdof_begin + d));
            const uint16_t * Lg = plan.L + (size_t)hdr.elem_begin * NB2;
            for (int k = tid; k < hdr.n_elem * NB2; k += blockDim.x)
                Ls[k] = __ldg(Lg + k);
            __syncthreads();

            double * sc = scratch + warp * SCR;
            const int r = lane;
            for (int e = warp; e < hdr.n_elem; e += nwarps) {
                const double * gp = G + ((size_t)blockIdx.x * PE + e) * (size_t)(NK * NQ) + lane;
                if (r < NB) {
                    const uint16_t * Le = Ls + e * NB2 + NB * r;
                    for (int q = 0; q < NQ; ++q) {
                        double pu = 0.0, du = 0.0;
                        for (int k = 0; k < NB; ++k) {
                            const double uk = xloc[Le[k]];
                            pu = fma(Pt[q + NQ * k], uk, pu);
                            if (STIFF)
                                du = fma(Dt[q + NQ * k], uk, du);
                        }
                        sc[q * NB + r] = pu;
                        if (STIFF)
                            sc[NQ * NB + q * NB + r] = du;
                    }
                }
                __syncwarp();
                double a0[MAXQ], a1[MAXQ];
                if (r < NQ) {
                    for (int t = 0; t < NB; ++t)
                        a0[t] = a1[t] = 0.0;
                    for (int ty = 0; ty < NQ; ++ty) {
                        if (STIFF) {
                            double Dx = 0.0, Dy = 0.0;
                            for (int l = 0; l < NB; ++l) {
                                Dx = fma(Pt[ty + NQ * l], sc[NQ * NB + r * NB + l], Dx);
                                Dy = fma(Dt[ty + NQ * l], sc[r * NB + l], Dy);
                            }
                            const double A = gp[(3 * ty) * NQ], B = gp[(3 * ty + 1) * NQ], C = gp[(3 * ty + 2) * NQ];
                            const double F0 = A * Dx + B * Dy, F1 = B * Dx + C * Dy;
                            for (int t = 0; t < NB; ++t) {
                                a0[t] = fma(Pt[ty + NQ * t], F0, a0[t]);
                                a1[t] = fma(Dt[ty + NQ * t], F1, a1[t]);
                            }
                        }
                        else {
                            double ppu = 0.0;
                            for (int l = 0; l < NB; ++l)
                                ppu = fma(Pt[ty + NQ * l], sc[r * NB + l], ppu);
                            const double val = gp[ty * NQ] * ppu;
                            for (int t = 0; t < NB; ++t)
                                a0[t] = fma(Pt[ty + NQ * t], val, a0[t]);
                        }
                    }
                }
                __syncwarp();
                if (r < NQ)
                    for (int t = 0; t < NB; ++t) {
                        sc[r * NB + t] = a0[t];
                        if (STIFF)
                            sc[NQ * NB + r * NB + t] = a1[t];
                    }
                __syncwarp();
                if (r < NB) {
                    double * so = su + e * NB2 + NB * r;
                    for (int t = 0; t < NB; ++t) {
                        double s = 0.0;
                        for (int i = 0; i < NQ; ++i) {
                            if (STIFF) {
                                s = fma(Dt[i + NQ * t], sc[i * NB + r], s);
                                s = fma(Pt[i + NQ * t], sc[NQ * NB + i * NB + r], s);
                            }
                            else
                                s = fma(Pt[i + NQ * t], sc[i * NB + r], s);
                        }
                        so[t] = s;
                    }
                }
                __syncwarp();
            }
            __syncthreads();
            const uint16_t * cp = plan.cptr + hdr.cptr_begin;
            const uint16_t * ce = plan.cent + (size_t)hdr.elem_begin * NB2;
            for (int d = tid; d < hdr.n_pdof; d += blockDim.x) {
                const int b = cp[d], e = cp[d + 1];
                double sum = 0.0;
                for (int k = b; k < e; ++k)
                    sum += su[ce[k]];
                if (d < hdr.n_int) {
                    const int gi = __ldg(plan.gid + hdr.pdof_begin + d);
                    const double v = c * sum;
                    y[gi] = accumulate ? (y[gi] + v) : v;
                }
                else
                    partial[__ldg(plan.slot + hdr.slot_begin + d - hdr.n_int)] = sum;
            }
        }

        // second pass: DOFs shared between patches, partial slots summed in patch order
        __global__ void assemble_shared_kernel(const int64_t n_shared, const int * __restrict__ sh_gid,
                                               const int * __restrict__ sh_ptr, const double * __restrict__ partial,
                                               double * __restrict__ y, const double c, const int accumulate)
        {
            const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (s >= n_shared)
                return;
            const int b = sh_ptr[s], e = sh_ptr[s + 1];
            double sum = 0.0;
            for (int k = b; k < e; ++k)
                sum += partial[k];
            const int gi = sh_gid[s];
            const double v = c * sum;
            y[gi] = accumulate ? (y[gi] + v) : v;
        }

        // both block rows of the fused Helmholtz apply in one launch: blockIdx.y = field
        __global__ void assemble_shared_fields_kernel(const int64_t n_shared, const int * __restrict__ sh_gid,
                                                      const int * __restrict__ sh_ptr, const double * __restrict__ partial,
                                                      const int64_t partial_stride, double * __restrict__ y, const int64_t y_stride,
                                                      const double c0, const double c1)
        {
            const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (s >= n_shared)
                return;
            const int f = blockIdx.y;
            const double * pf = partial + f * partial_stride;
            const int b = sh_ptr[s], e = sh_ptr[s + 1];
            double sum = 0.0;
            for (int k = b; k < e; ++k)
                sum += pf[k];
            y[f * y_stride + sh_gid[s]] = (f == 0 ? c0 : c1) * sum;
        }

        // ------------------------------------------------------------------------------------------
        // setup kernels: metric data in plan ("lane-major") order.
        //   index(slot e of patch p, q = first quad index, k) =
        //       ((p * n_pass + e / EPW) * NK + k) * LW + (e % EPW) * NQ + q
        // Jacobian of the bilinear map: source/Element.cpp:21-27; G: source/StiffnessMatrix.cpp:5-38;
        // mass weights: source/MassMatrix.cpp:5-67.
        // ------------------------------------------------------------------------------------------
        __device__ __forceinline__ void bilinear_jacobian(const double * c, double xi0, double xi1, double * J)
        {
            J[0] = 0.25 * ((1.0 - xi1) * (c[2] - c[0]) + (1.0 + xi1) * (c[4] - c[6]));
            J[1] = 0.25 * ((1.0 - xi1) * (c[3] - c[1]) + (1.0 + xi1) * (c[5] - c[7]));
            J[2] = 0.25 * ((1.0 - xi0) * (c[6] - c[0]) + (1.0 + xi0) * (c[4] - c[2]));
            J[3] = 0.25 * ((1.0 - xi0) * (c[7] - c[1]) + (1.0 + xi0) * (c[5] - c[3]));
        }

        // position of metric value (tx, ty, component a of NKI) of element slot e of patch p. EPW > 0: lane-major layout of
        // volume_action_kernel; EPW == 0: thread-per-element layout [pair of values][element] of volume_action_ws.
        __device__ __forceinline__ size_t metric_index(const int64_t p, const int e, const int PE, const int NQ, const int EPW,
                                                       const int n_pass, const int NKI, const int tx, const int ty, const int a)
        {
            if (EPW == 0) {
                const int KR = (NKI * NQ + 1) & ~1;
                const int NK2 = NQ * KR / 2;
                const int k = tx * KR + ty * NKI + a;
                return (((size_t)p * NK2 + (k >> 1)) * PE + e) * 2 + (k & 1);
            }
            const int LW = EPW * NQ, NK = NKI * NQ;
            return ((size_t)(p * n_pass + e / EPW) * NK + (NKI * ty + a)) * LW + (size_t)(e % EPW) * NQ + tx;
        }

        // thread-pair layout of volume_action_pair (EPW == -1): [patch][row tx][pair of values][thread slot 0..127]; thread slot
        // s = (e / 16) * 32 + h * 16 + e % 16 of half h holds, for its local quadrature column tt (ty = tt in the natural frame
        // h = 0, ty = nq-1-tt in the mirrored frame h = 1), the NKI values at k = tt * NKI + a. The middle column of an odd nq
        // belongs to h = 0 (the h = 1 copy stays zero); *sign is -1 for the off-diagonal stiffness term in the mirrored frame.
        __device__ __forceinline__ size_t metric_index_pair(const int64_t p, const int e, const int NQ, const int NKI, const int tx,
                                                            const int ty, const int a, double * sign)
        {
            const int TA = (NQ + 1) / 2;
            const int h = ty < TA ? 0 : 1;
            const int tt = h ? NQ - 1 - ty : ty;
            const int KR = (NKI * TA + 1) & ~1, NPR = KR / 2;
            const int k = tt * NKI + a;
            const int s = (e >> 4) * 32 + h * 16 + (e & 15);
            *sign = (h && NKI == 3 && a == 1) ? -1.0 : 1.0;
            return ((((size_t)p * NQ + tx) * NPR + (k >> 1)) * 128 + s) * 2 + (k & 1);
        }

        __global__ void setup_stiffness_kernel(const int64_t n_slots, const int PE, const int NQ, const int EPW,
                                               const int n_pass, const int * __restrict__ slot_elem,
                                               const double * __restrict__ corners, const double * __restrict__ xq,
                                               const double * __restrict__ wq, double * __restrict__ G)
        {
            const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            const int nq2 = NQ * NQ;
            if (t >= n_slots * nq2)
                return;
            const int64_t slot = t / nq2;
            const int rem = (int)(t - slot * nq2);
            const int i = rem % NQ, j = rem / NQ;
            const int64_t p = slot / PE;
            const int e = (int)(slot - p * PE);
            const int el = slot_elem[slot];
            double g0 = 0.0, g1 = 0.0, g2 = 0.0;
            if (el >= 0) {
                double J[4];
                bilinear_jacobian(corners + 8 * (size_t)el, xq[i], xq[j], J);
                const double W = wq[i] * wq[j];
                const double X_xi = J[0], Y_xi = J[1], X_eta = J[2], Y_eta = J[3];
                const double det = X_xi * Y_eta - X_eta * Y_xi;
                g0 = W * (Y_eta * Y_eta + X_eta * X_eta) / det;
                g1 = -W * (Y_xi * Y_eta + X_xi * X_eta) / det;
                g2 = W * (Y_xi * Y_xi + X_xi * X_xi) / det;
            }
            if (EPW < 0) {
                double sg;
                G[metric_index_pair(p, e, NQ, 3, i, j, 0, &sg)] = g0;
                const size_t i1 = metric_index_pair(p, e, NQ, 3, i, j, 1, &sg);
                G[i1] = sg * g1;
                G[metric_index_pair(p, e, NQ, 3, i, j, 2, &sg)] = g2;
                return;
            }
            G[metric_index(p, e, PE, NQ, EPW, n_pass, 3, i, j, 0)] = g0;
            G[metric_index(p, e, PE, NQ, EPW, n_pass, 3, i, j, 1)] = g1;
            G[metric_index(p, e, PE, NQ, EPW, n_pass, 3, i, j, 2)] = g2;
        }

        // affine stiffness: gA, gB, gC of the element in slot (p, e), layout ((p * 3 + c) * PE + e); Jacobian of a parallelogram
        // (source/Element.cpp:21-27 with x1 - x0 == x2 - x3), the W = w_i w_j factor lives in the kernel's weighted tables
        __global__ void setup_stiffness_affine_kernel(const int64_t n_slots, const int PE, const int * __restrict__ slot_elem,
                                                      const double * __restrict__ corners, double * __restrict__ Gc)
        {
            const int64_t slot = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (slot >= n_slots)
                return;
            const int64_t p = slot / PE;
            const int e = (int)(slot - p * PE);
            const int el = slot_elem[slot];
            double gA = 0.0, gB = 0.0, gC = 0.0;
            if (el >= 0) {
                double J[4];
                bilinear_jacobian(corners + 8 * (size_t)el, 0.0, 0.0, J);
                const double X_xi = J[0], Y_xi = J[1], X_eta = J[2], Y_eta = J[3];
                const double det = X_xi * Y_eta - X_eta * Y_xi;
                gA = (Y_eta * Y_eta + X_eta * X_eta) / det;
                gB = -(Y_xi * Y_eta + X_xi * X_eta) / det;
                gC = (Y_xi * Y_xi + X_xi * X_xi) / det;
            }
            Gc[((size_t)p * 3 + 0) * PE + e] = gA;
            Gc[((size_t)p * 3 + 1) * PE + e] = gB;
            Gc[((size_t)p * 3 + 2) * PE + e] = gC;
        }

        __global__ void setup_mass_kernel(const int64_t n_slots, const int PE, const int NB, const int NQ, const int EPW,
                                          const int n_pass, const int * __restrict__ slot_elem,
                                          const double * __restrict__ corners, const int * __restrict__ I,
                                          const double * __restrict__ coef, const double * __restrict__ P,
                                          const double * __restrict__ xq, const double * __restrict__ wq,
                                          double * __restrict__ A)
        {
            const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            const int nq2 = NQ * NQ;
            if (t >= n_slots * nq2)
                return;
            const int64_t slot = t / nq2;
            const int rem = (int)(t - slot * nq2);
            const int tx = rem % NQ, ty = rem / NQ;
            const int64_t p = slot / PE;
            const int e = (int)(slot - p * PE);
            const int el = slot_elem[slot];
            double sg_;
            const size_t idx = EPW < 0 ? metric_index_pair(p, e, NQ, 1, tx, ty, 0, &sg_) : metric_index(p, e, PE, NQ, EPW, n_pass, 1, tx, ty, 0);
            double val = 0.0;
            if (el >= 0) {
                double ppx = 0.0;
                const int * Ie = I + (size_t)NB * NB * el;
                for (int l = 0; l < NB; ++l) {
                    double z = 0.0; // z[tx][l] = sum_k P(tx,k) Q[k][l]
                    for (int k = 0; k < NB; ++k)
                        z += P[tx + NQ * k] * (coef ? coef[Ie[k + NB * l]] : 1.0);
                    ppx += P[ty + NQ * l] * z;
                }
                double J[4];
                bilinear_jacobian(corners + 8 * (size_t)el, xq[tx], xq[ty], J);
                const double det = J[0] * J[3] - J[1] * J[2];
                ppx *= wq[tx] * wq[ty] * det;
                val = ppx;
            }
            A[idx] = val;
        }

        // lumped (GLL-collocated) mass diagonal, DOF-centric and deterministic: one thread per element node
        // writes its contribution into an element-local array, a second kernel sums per DOF through the plan?
        // Setup-only and tiny: use a simple two-step (element-local products, then ordered gather by a
        // transposed map built on the host).
        __global__ void diag_mass_contrib_kernel(const int64_t nel, const int NB, const int * __restrict__ I,
                                                 const double * __restrict__ corners, const double * __restrict__ coef,
                                                 const double * __restrict__ xg, const double * __restrict__ wg,
                                                 double * __restrict__ contrib)
        {
            const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            const int nb2 = NB * NB;
            if (t >= nel * nb2)
                return;
            const int64_t el = t / nb2;
            const int rem = (int)(t - el * nb2);
            const int i = rem % NB, j = rem / NB;
            double J[4];
            bilinear_jacobian(corners + 8 * (size_t)el, xg[i], xg[j], J);
            double m = wg[i] * wg[j] * (J[0] * J[3] - J[1] * J[2]);
            if (coef)
                m *= coef[I[t]];
            contrib[t] = m;
        }

        __global__ void gather_sum_recip_kernel(const int64_t n, const int * __restrict__ ptr, const int * __restrict__ src,
                                                const double * __restrict__ contrib, double * __restrict__ out)
        {
            const int64_t d = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (d >= n)
                return;
            double s = 0.0;
            for (int k = ptr[d]; k < ptr[d + 1]; ++k)
                s += contrib[src[k]];
            out[d] = 1.0 / s;
        }

        __global__ void diag_apply_kernel(const int64_t n, const double * __restrict__ p, const double c, const int accumulate,
                                          const double * __restrict__ x, double * __restrict__ y)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (i >= n)
                return;
            // reference source/MassMatrix.cpp:316-334: y += c*p*x  /  y = p*x
            y[i] = accumulate ? (y[i] + c * p[i] * x[i]) : (c * p[i] * x[i]);
        }

        // ------------------------------------------------------------------------------------------
        // face mass: reference source/FaceMassMatrix.cpp:141-193. One thread per face-space DOF walks its
        // incident (face, k) pairs in fixed order (deterministic; replaces atomicAdd). `gather`/`scatter`
        // fuse FaceSpace::restrict / prolong (source/H1Space.cpp:189-211) when operating on H1 vectors.
        // ------------------------------------------------------------------------------------------
        __global__ void facemass_action_kernel(const int64_t fdof, const int NB, const int NQ, const double * __restrict__ P,
                                               const double * __restrict__ a, const int * __restrict__ If,
                                               const int * __restrict__ inc_ptr, const int * __restrict__ inc,
                                               const int * __restrict__ proj /* null: face-space vectors */,
                                               const double c, const int accumulate, const double * __restrict__ x,
                                               double * __restrict__ y)
        {
            const int64_t d = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (d >= fdof)
                return;
            double sum = 0.0;
            for (int t = inc_ptr[d]; t < inc_ptr[d + 1]; ++t) {
                const int fk = inc[t];
                const int f = fk / NB, k = fk - f * NB;
                const int * Ifa = If + (size_t)NB * f;
                double Mu = 0.0;
                for (int i = 0; i < NQ; ++i) {
                    double pu = 0.0;
                    for (int l = 0; l < NB; ++l) {
                        const int xi = proj ? proj[Ifa[l]] : Ifa[l];
                        pu += P[i + NQ * l] * x[xi];
                    }
                    pu *= a[i + (size_t)NQ * f];
                    Mu += P[i + NQ * k] * pu;
                }
                sum += c * Mu;
            }
            const int64_t yi = proj ? proj[d] : d;
            y[yi] = accumulate ? (y[yi] + sum) : sum;
        }

        // interface rows of a slab (SlabHalo): position of (field f, row entry e) in the send / recv buffers
        struct HaloDev
        {
            const int * row_dof;    // (n_bottom + n_top)
            const int * face_entry; // per face DOF: row entry or -1
            const int * plain;      // row entries packed by plain copy
            double * send;
            int64_t n_bottom, n_top, n_plain;
            // peer path (NVLink stores into the neighbours' receive buffers instead of a send buffer + ncclSend/ncclRecv):
            double * peer_dst[2];               // where the bottom / top segment of THIS apply goes in the lower / upper neighbour's memory
            unsigned long long * peer_flag[2];  // the neighbours' arrival flags for this rank
            unsigned * ticket;                  // last-block detection of the packing launch
            unsigned long long epoch;           // value to publish (monotone: one per exchange)
            int peer;
        };
        __device__ __forceinline__ int64_t halo_pos(const HaloDev & h, const int f, const int e)
        {
            return e < h.n_bottom ? f * h.n_bottom + e : 2 * h.n_bottom + f * h.n_top + (e - h.n_bottom);
        }
        __device__ __forceinline__ void halo_put(const HaloDev & h, const int f, const int e, const double v)
        {
            const int64_t pos = halo_pos(h, f, e);
            if (!h.peer)
                h.send[pos] = v;
            else if (pos < 2 * h.n_bottom)
                h.peer_dst[0][pos] = v;
            else
                h.peer_dst[1][pos - 2 * h.n_bottom] = v;
        }
        // peer path: after the last block of the packing launch has made its stores visible system-wide, publish the epoch in the
        // neighbours' flags (release at system scope). Every thread of the launch must call this exactly once, at its end.
        __device__ __forceinline__ void halo_publish(const HaloDev & h)
        {
            if (!h.peer)
                return;
            __threadfence_system();
            __syncthreads();
            if (threadIdx.x == 0) {
                const unsigned total = gridDim.x * gridDim.y;
                if (atomicAdd(h.ticket, 1u) == total - 1) {
                    *h.ticket = 0;
                    __threadfence_system();
                    for (int side = 0; side < 2; ++side)
                        if (h.peer_flag[side])
                            asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(h.peer_flag[side]), "l"(h.epoch) : "memory");
                }
            }
        }

        // the two boundary terms of the Helmholtz composite in one launch: blockIdx.y = 0: y[0:n] += c H x[n:2n]; 1: y[n:2n] += c H x[0:n].
        // With a halo (slab of a partitioned mesh) the same launch packs the two interface rows of the finished result: the
        // thread that adds the face term of a corner node writes that node's final value, blocks beyond the face DOFs copy the rest.
        __global__ void facemass_pair_kernel(const int64_t fdof, const int NB, const int NQ, const double * __restrict__ P,
                                             const double * __restrict__ a, const int * __restrict__ If,
                                             const int * __restrict__ inc_ptr, const int * __restrict__ inc,
                                             const int * __restrict__ proj, const double c, const int64_t n,
                                             const double * __restrict__ x, double * __restrict__ y, const HaloDev halo, const int face_blocks)
        {
            const int fld = blockIdx.y;
            double * yd = fld == 0 ? y : y + n;
            if ((int)blockIdx.x >= face_blocks) { // pack-only part
                const int64_t k = (int64_t)(blockIdx.x - face_blocks) * blockDim.x + threadIdx.x;
                if (k < halo.n_plain) {
                    const int e = halo.plain[k];
                    halo_put(halo, fld, e, yd[halo.row_dof[e]]);
                }
            }
            else {
                const int64_t d = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
                if (d < fdof) {
                    const double * xs = fld == 0 ? x + n : x;
                    double sum = 0.0;
                    for (int t = inc_ptr[d]; t < inc_ptr[d + 1]; ++t) {
                        const int fk = inc[t];
                        const int f = fk / NB, k = fk - f * NB;
                        const int * Ifa = If + (size_t)NB * f;
                        double Mu = 0.0;
                        for (int i = 0; i < NQ; ++i) {
                            double pu = 0.0;
                            for (int l = 0; l < NB; ++l)
                                pu += P[i + NQ * l] * xs[proj[Ifa[l]]];
                            pu *= a[i + (size_t)NQ * f];
                            Mu += P[i + NQ * k] * pu;
                        }
                        sum += c * Mu;
                    }
                    const double v = yd[proj[d]] + sum;
                    yd[proj[d]] = v;
                    if (halo.face_entry) {
                        const int e = halo.face_entry[d];
                        if (e >= 0)
                            halo_put(halo, fld, e, v);
                    }
                }
            }
            halo_publish(halo);
        }

        // stand-alone pack of every row entry (SlabHalo::exchange) and the add of the received rows
        __global__ void halo_pack_kernel(const HaloDev halo, const int64_t n, const double * __restrict__ y)
        {
            const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (e < halo.n_bottom + halo.n_top)
                halo_put(halo, blockIdx.y, (int)e, y[blockIdx.y * n + halo.row_dof[e]]);
            halo_publish(halo);
        }
        // recv: this rank's receive buffer of the current parity. Peer path: wait (acquire at system scope) until both neighbours
        // have published `epoch` in this rank's flags; their stores bypass this SM's L1, so the data is read with ld.cg.
        __global__ void halo_add_kernel(const HaloDev halo, const double * __restrict__ recv, const int64_t n, double * __restrict__ y,
                                        const unsigned long long * __restrict__ own_flags, const int wait_bottom, const int wait_top)
        {
            if (halo.peer) {
                if (threadIdx.x == 0) {
                    unsigned long long t0 = 0;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
                    for (int side = 0; side < 2; ++side) {
                        if (!(side == 0 ? wait_bottom : wait_top))
                            continue;
                        unsigned long long seen = 0;
                        for (;;) {
                            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(own_flags + side) : "memory");
                            if (seen >= halo.epoch)
                                break;
                            unsigned long long t1;
                            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                            if (t1 - t0 > 120000000000ull) // two minutes without the neighbour's rows: fail loudly instead of hanging the GPU
                                __trap();
                            __nanosleep(200);
                        }
                    }
                }
                __syncthreads();
            }
            const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (e < halo.n_bottom + halo.n_top) {
                const double r = halo.peer ? __ldcg(recv + halo_pos(halo, blockIdx.y, (int)e)) : recv[halo_pos(halo, blockIdx.y, (int)e)];
                y[blockIdx.y * n + halo.row_dof[e]] += r; // own + received: same sum on both sides
            }
        }

        __global__ void setup_facemass_kernel(const int64_t nf, const int NB, const int NQ, const double * __restrict__ wq,
                                              const double * __restrict__ P, const double * __restrict__ meas,
                                              const double * __restrict__ coef, const int * __restrict__ If,
                                              double * __restrict__ op)
        {
            const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (t >= nf * NQ)
                return;
            const int64_t f = t / NQ;
            const int k = (int)(t - f * NQ);
            double pa = 0.0;
            for (int l = 0; l < NB; ++l)
                pa += P[k + NQ * l] * (coef ? coef[If[l + (size_t)NB * f]] : 1.0);
            pa *= wq[k] * meas[f];
            op[t] = pa;
        }

        __global__ void diag_facemass_kernel(const int64_t fdof, const int NB, const double * __restrict__ wg,
                                             const double * __restrict__ meas, const double * __restrict__ coef,
                                             const int * __restrict__ inc_ptr, const int * __restrict__ inc,
                                             double * __restrict__ out)
        {
            const int64_t d = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (d >= fdof)
                return;
            double s = 0.0;
            for (int t = inc_ptr[d]; t < inc_ptr[d + 1]; ++t) {
                const int fk = inc[t];
                const int f = fk / NB, i = fk - f * NB;
                double m = wg[i] * meas[f];
                if (coef)
                    m *= coef[d];
                s += m;
            }
            out[d] = 1.0 / s;
        }

        __global__ void restrict_kernel(const int64_t n, const int * __restrict__ proj, const double * __restrict__ x, double * __restrict__ y)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (i < n)
                y[i] = x[proj[i]];
        }
        __global__ void prolong_kernel(const int64_t n, const int * __restrict__ proj, const double * __restrict__ x, double * __restrict__ y)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (i < n)
                y[proj[i]] += x[i]; // proj is injective: no atomics needed
        }
        __global__ void orth_kernel(const int64_t n, const int * __restrict__ proj, double * __restrict__ x)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (i < n)
                x[proj[i]] = 0.0;
        }
        __global__ void negate_kernel(const int64_t n, double * __restrict__ x)
        {
            const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (i < n)
                x[i] = -x[i];
        }

        inline unsigned blocks_for(int64_t n, int bs) { return (unsigned)((n + bs - 1) / bs); }

        // ------------------------------------------------------------------------------------------
        // launch plumbing
        // ------------------------------------------------------------------------------------------
        int pick_warps(int n_pass)
        {
            int best = std::min(8, n_pass);
            for (int w = 8; w >= 4; --w)
                if (n_pass % w == 0) {
                    best = w;
                    break;
                }
            return std::max(best, 1);
        }

        int env_int(const char * name, int dflt)
        {
            const char * v = getenv(name);
            return v ? atoi(v) : dflt;
        }

        PlanDev plan_dev(const Plan & plan)
        {
            return PlanDev{plan.d_hdr.p, plan.d_gid.p, plan.d_slot.p, plan.d_L.p, plan.d_cptr.p, plan.d_cent.p, plan.PE, plan.d_Ig.p,
                           reinterpret_cast<const uint2 *>(plan.d_cent4.p), plan.d_target.p};
        }

        // launch configuration of `grid` CTAs of 256 threads in clusters of `cluster` along x (attr must outlive it)
        cudaLaunchConfig_t cluster_config(int grid, size_t smem, int cluster, cudaLaunchAttribute & attr, cudaStream_t s = 0)
        {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)grid);
            cfg.blockDim = dim3(256);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = s;
            attr.id = cudaLaunchAttributeClusterDimension;
            attr.val.clusterDim.x = (unsigned)cluster;
            attr.val.clusterDim.y = 1;
            attr.val.clusterDim.z = 1;
            cfg.attrs = &attr;
            cfg.numAttrs = 1;
            return cfg;
        }

        // what one kernel instance has been set up for on one device (function attributes are per device)
        struct DeviceSetup
        {
            size_t smem = 0; // dynamic shared-memory limit set so far
            int wave = 0;    // one wave of resident CTAs: resident CTAs per SM x SM count
        };

        // Raises the instance's dynamic shared-memory limit whenever a launch needs more than before and asks for the largest
        // carve-out (several CTAs per SM are needed to overlap the staging / assembly phases of one patch with the contractions
        // of another). Sizes the wave at the first launch on the device; cluster > 1: the kernel runs as clusters of that many
        // CTAs, and the wave is clamped to the co-resident clusters.
        template <class Kern>
        const DeviceSetup & setup_kernel(DeviceSetup (&per_device)[MAX_DEVICES], Kern kern, int threads, size_t smem, int cluster = 1)
        {
            int dev = 0;
            cudaGetDevice(&dev);
            CB_REQUIRE(dev >= 0 && dev < MAX_DEVICES, "device ordinal out of range");
            DeviceSetup & st = per_device[dev];
            if (smem > st.smem) {
                CB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max(smem, (size_t)49152)));
                CB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
                st.smem = std::max(smem, (size_t)49152);
            }
            if (!st.wave) {
                int sms = 148, occ = 1;
                cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
                CB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
                st.wave = std::max(1, occ) * sms;
                if (cluster > 1) {
                    cudaLaunchAttribute at;
                    const cudaLaunchConfig_t cfg = cluster_config(st.wave, smem, cluster, at);
                    int ncl = 0;
                    if (cudaOccupancyMaxActiveClusters(&ncl, kern, &cfg) == cudaSuccess && ncl > 0)
                        st.wave = std::min(st.wave, cluster * ncl);
                    else
                        cudaGetLastError();
                }
            }
            return st;
        }

        template <int NB, int NQ, bool STIFF>
        void fill_tables(Tables<NB, NQ, STIFF> & tab, const VolumeOp & op, const double msc = 1.0)
        {
            std::memset(&tab, 0, sizeof(tab));
            for (int q = 0; q < NQ; ++q)
                for (int k = 0; k < NB; ++k) {
                    if (!STIFF)
                        tab.PSrow[q][k] = msc * op.P[q + NQ * k];
                    tab.Prow[q][k] = op.P[q + NQ * k];
                    tab.Pcol[k][q] = op.P[q + NQ * k];
                    if (STIFF) {
                        tab.Drow[q][k] = op.D[q + NQ * k];
                        tab.Dcol[k][q] = op.D[q + NQ * k];
                        if (!op.wq.empty()) {
                            tab.PWrow[q][k] = op.wq[q] * op.P[q + NQ * k];
                            tab.DWrow[q][k] = op.wq[q] * op.D[q + NQ * k];
                        }
                    }
                }
        }

        using LaunchFn = decltype(VolumeOp::launch);
        using FusedFn = decltype(HelmholtzOp::fused);

        template <int NB, int NQ, bool STIFF>
        void launch_volume(const VolumeOp & op, double c, int accumulate, const double * x, double * y, cudaStream_t s)
        {
            constexpr int EPW = 32 / NQ;
            constexpr int SCR = scr_layout<NB, NQ, STIFF>().S;
            const Plan & plan = *op.plan;
            const int n_pass = (plan.PE + EPW - 1) / EPW;
            static const int warps_override = env_int("CUDDH_B200_WARPS", 0);
            const int nwarps = warps_override > 0 ? std::min(warps_override, 16) : pick_warps(n_pass);
            size_t smem = sizeof(double) * ((size_t)plan.max_pdof + (size_t)plan.PE * NB * NB + (size_t)nwarps * EPW * SCR) +
                          sizeof(int) * (size_t)plan.max_pdof + sizeof(uint16_t) * ((size_t)2 * plan.PE * NB * NB + plan.max_pdof + 2);
            smem = (smem + 15) & ~size_t(15);
            Tables<NB, NQ, STIFF> tab;
            fill_tables(tab, op); // the weighted / scaled rows are not read by this kernel
            auto kern = volume_action_kernel<NB, NQ, STIFF>;
            static DeviceSetup per_device[MAX_DEVICES];
            const DeviceSetup & st = setup_kernel(per_device, kern, nwarps * 32, smem);
            // L2 prefetch distance in patches: one scheduling wave unless CUDDH_B200_PFDIST is set
            static const bool pf_set = getenv("CUDDH_B200_PFDIST") != nullptr;
            static const int pf_env = env_int("CUDDH_B200_PFDIST", 0);
            const int pf_dist = pf_set ? pf_env : st.wave;
            kern<<<(unsigned)plan.n_patches, nwarps * 32, smem, s>>>(tab, plan_dev(plan), op.d_G.p, x, y, op.d_partial.p, c, accumulate,
                                                                       plan.max_pdof, (int)plan.n_patches, pf_dist);
            CB_LAUNCHED();
        }

        template <int NB, int NQ, bool STIFF, int NQ2, int RING = 0, bool AFFINE = false>
        void launch_ws(const VolumeOp & op, const VolumeOp * op2, WsArgs args, cudaStream_t s)
        {
            const Plan & plan = *op.plan;
            CB_REQUIRE(plan.PE == 128, "warp-specialised kernel: patches must hold 128 elements");
            constexpr int NI = (NB > 2 ? NB - 2 : 0) * (NB > 2 ? NB - 2 : 0);
            constexpr int NPRa = TpeCfg<NB, NQ, STIFF>::KR / 2, NPRb = NQ2 > 0 ? TpeCfg<NB, (NQ2 > 0 ? NQ2 : 1), false>::KR / 2 : 0;
            constexpr int CHUNK_PAIRS = ring_cp(NPRa) > (NQ2 > 0 ? ring_cp(NPRb) : 0) ? ring_cp(NPRa) : ring_cp(NPRb);
            constexpr int NBUF = (RING > 2 || RING < 0) ? 2 : 3; // as in the kernel
            constexpr int RSLOTS = RING < 0 ? -RING : RING;
            constexpr int SLOT_PAIRS = (RING < 0 && AFFINE && NQ2 > 0) ? NPRb : CHUNK_PAIRS; // per-thread ring of mass rows: one slot = one row
            const size_t smem = sizeof(double) * NBUF * (size_t)NB * NB * 128 + sizeof(int) * NBUF * (size_t)NI * 128 +
                                (size_t)RSLOTS * SLOT_PAIRS * 128 * sizeof(double2) + (size_t)RSLOTS * 8 + 16;
            Tables<NB, NQ, STIFF> tab;
            fill_tables(tab, op);
            typename Phase2<NB, NQ2>::type tab2;
            std::memset(&tab2, 0, sizeof(tab2));
            if constexpr (NQ2 > 0)
                fill_tables(tab2, *op2, args.msc);
            auto kern = volume_action_ws<NB, NQ, STIFF, NQ2, RING, AFFINE>;
            static DeviceSetup per_device[MAX_DEVICES];
            const int grid = setup_kernel(per_device, kern, 256, smem, NQ2 > 0 ? 2 : 1).wave;
            const int nf = std::max(args.n_fields, 1);
            const int cap = max_persistent_ctas(); // test / tuning knob: fewer CTAs = more patches per persistent CTA
            const int wave = cap > 0 ? std::max(nf, std::min(grid, cap)) : grid;
            const int g = (int)std::min<int64_t>(wave / nf, plan.n_patches) * nf;
            const PlanDev pd = plan_dev(plan);
            args.n_patches = (int)plan.n_patches;
            if (nf > 1) { // one cluster = the CTAs that walk the same patches, one field each
                cudaLaunchAttribute at;
                const cudaLaunchConfig_t cfg = cluster_config(g, smem, nf, at, s);
                CB_CUDA(cudaLaunchKernelEx(&cfg, kern, tab, tab2, pd, args));
            }
            else
                kern<<<g, 256, smem, s>>>(tab, tab2, pd, args);
            CB_LAUNCHED();
        }

        template <int NB, int NQ, bool STIFF, int RING = 0, bool AFFINE = false>
        void launch_volume_ws(const VolumeOp & op, double c, int accumulate, const double * x, double * y, cudaStream_t s)
        {
            WsArgs a{};
            a.G1 = reinterpret_cast<const double2 *>(op.d_G.p);
            a.G2 = nullptr;
            a.Gc = op.d_Gc.p;
            a.x = x;
            a.y = y;
            a.partial = op.d_partial.p;
            a.c[0] = a.c[1] = c;
            a.msc = 1.0;
            a.accumulate = accumulate;
            a.n_fields = 1;
            launch_ws<NB, NQ, STIFF, 0, RING, AFFINE>(op, nullptr, a, s);
        }

        // thread-pair-per-element kernel (volume_pair.cuh): n_basis 6-9
        // depth of the per-thread metric ring of a thread-pair instance: the (short-row) mass operator where two CTAs per SM still
        // fit with 3 rows of ring; 0 = registers, one row ahead
        template <int NB, int NQ, bool STIFF, bool AFFINE>
        constexpr int pair_ring_depth()
        {
            if (STIFF || AFFINE)
                return 0;
            constexpr int NI = 2, TA = (NQ + 1) / 2, NPR = ((TA + 1) & ~1) / 2; // NI: ids handed over per element (see volume_action_pair)
            constexpr size_t base = sizeof(double) * 2 * (size_t)NB * NB * 64 + sizeof(int) * 2 * (size_t)NI * 64 + 16;
            return (base + 3 * (size_t)NPR * 128 * 16 + 1024) * 2 <= 233472 ? 3 : 0;
        }

        template <int NB, int NQ, bool STIFF>
        void fill_pair_tables(PairTables<NB, NQ, STIFF> & tab, const VolumeOp & op, const double msc = 1.0)
        {
            std::memset(&tab, 0, sizeof(tab));
            for (int q = 0; q < NQ; ++q)
                for (int k = 0; k < NB; ++k) {
                    tab.Prow[q][k] = op.P[q + NQ * k];
                    if (!STIFF)
                        tab.PSrow[q][k] = msc * op.P[q + NQ * k];
                    if (STIFF) {
                        tab.Drow[q][k] = op.D[q + NQ * k];
                        if (!op.wq.empty()) {
                            tab.PWrow[q][k] = op.wq[q] * op.P[q + NQ * k];
                            tab.DWrow[q][k] = op.wq[q] * op.D[q + NQ * k];
                        }
                    }
                }
        }

        // one launch of the thread-pair kernel: a single operator (NQ2 == 0, op2 == nullptr) or the fused S + msc * M of one field
        template <int NB, int NQ, bool STIFF, bool AFFINE, int NQ2>
        void launch_pair(const VolumeOp & op, const VolumeOp * op2, PairArgs a, cudaStream_t s)
        {
            const Plan & plan = *op.plan;
            CB_REQUIRE(plan.PE == 64 && plan.interior_affine, "thread-pair kernel: needs 64-element patches and affine element-interior ids");
            constexpr int NI = 2;
            constexpr int RD = pair_ring_depth<NB, NQ, STIFF, AFFINE>();
            constexpr int RD2 = NQ2 > 0 ? pair_ring_depth<NB, (NQ2 > 0 ? NQ2 : 1), false, false>() : 0;
            static_assert(NQ2 == 0 || RD2 > 0, "fused thread-pair instances need the metric ring for their mass phase");
            constexpr int NPRR = RD > 0 ? PairCfg<NB, NQ, STIFF>::NPR : PairCfg<NB, (NQ2 > 0 ? NQ2 : 1), false>::NPR;
            constexpr int RDR = RD > 0 ? RD : RD2;
            const size_t smem = sizeof(double) * 2 * (size_t)NB * NB * 64 + sizeof(int) * 2 * (size_t)NI * 64 + (size_t)RDR * NPRR * 128 * 16 + 16;
            PairTables<NB, NQ, STIFF> tab;
            fill_pair_tables(tab, op);
            PairTables<NB, (NQ2 > 0 ? NQ2 : 1), false> tab2;
            std::memset(&tab2, 0, sizeof(tab2));
            if constexpr (NQ2 > 0)
                fill_pair_tables(tab2, *op2, a.msc);
            auto kern = volume_action_pair<NB, NQ, STIFF, AFFINE, RD, NQ2, RD2>;
            static DeviceSetup per_device[MAX_DEVICES];
            const int grid = setup_kernel(per_device, kern, 256, smem).wave;
            a.n_patches = (int)plan.n_patches;
            a.zero = 0;
            const int cap = max_persistent_ctas();
            const int wave = cap > 0 ? std::min(grid, cap) : grid;
            const int g = (int)std::min<int64_t>(wave, plan.n_patches);
            kern<<<g, 256, smem, s>>>(tab, tab2, plan_dev(plan), a);
            CB_LAUNCHED();
        }

        template <int NB, int NQ, bool STIFF, bool AFFINE = false>
        void launch_volume_pair(const VolumeOp & op, double c, int accumulate, const double * x, double * y, cudaStream_t s)
        {
            PairArgs a{};
            a.G = reinterpret_cast<const double2 *>(op.d_G.p);
            a.G2 = nullptr;
            a.Gc = op.d_Gc.p;
            a.x = x;
            a.y = y;
            a.partial = op.d_partial.p;
            a.c = c;
            a.msc = 1.0;
            a.accumulate = accumulate;
            launch_pair<NB, NQ, STIFF, AFFINE, 0>(op, nullptr, a, s);
        }

        // stride of the two fields in HelmholtzOp::d_partial2
        int64_t partial_stride(const HelmholtzOp & h) { return std::max<int64_t>(h.S->plan->n_slots_total, 1); }

        // the volume phase of the fused Helmholtz apply, both fields in one launch (the two CTAs of a cluster); the sign of the
        // second block row is applied on write
        template <int NB, int NQS, int NQM, int RING, bool AFFINE>
        void launch_fused_ws(const HelmholtzOp & h, const double * x, double * y, cudaStream_t s)
        {
            WsArgs a{};
            a.G1 = reinterpret_cast<const double2 *>(h.S->d_G.p);
            a.G2 = reinterpret_cast<const double2 *>(h.M->d_G.p);
            a.Gc = h.S->d_Gc.p;
            a.x = x;
            a.y = y;
            a.partial = h.d_partial2.p;
            a.x_stride = a.y_stride = h.fem->ndof;
            a.partial_stride = partial_stride(h);
            a.c[0] = 1.0;
            a.c[1] = -1.0;
            a.msc = -h.omega * h.omega;
            a.accumulate = 0;
            a.n_fields = 2;
            launch_ws<NB, NQS, true, NQM, RING, AFFINE>(*h.S, h.M.get(), a, s);
        }

        // the shared-DOF pass of the fused apply, both fields in one launch
        void assemble_shared_fields(const HelmholtzOp & h, double * y, cudaStream_t s)
        {
            const Plan & plan = *h.S->plan;
            if (plan.n_shared > 0) {
                assemble_shared_fields_kernel<<<dim3(blocks_for(plan.n_shared, 256), 2), 256, 0, s>>>(
                    plan.n_shared, plan.d_sh_gid.p, plan.d_sh_ptr.p, h.d_partial2.p, partial_stride(h), y, h.fem->ndof, 1.0, -1.0);
                CB_LAUNCHED();
            }
        }

        // n_basis 6-9: the thread-pair kernel runs S - omega^2 M of one field per launch
        template <int NB, int NQS, int NQM>
        void launch_fused_pair(const HelmholtzOp & h, const double * x, double * y, cudaStream_t s)
        {
            const int64_t n = h.fem->ndof;
            for (int f = 0; f < 2; ++f) {
                PairArgs a{};
                a.G = reinterpret_cast<const double2 *>(h.S->d_G.p);
                a.G2 = reinterpret_cast<const double2 *>(h.M->d_G.p);
                a.Gc = h.S->d_Gc.p;
                a.x = x + f * n;
                a.y = y + f * n;
                a.partial = h.d_partial2.p + f * partial_stride(h);
                a.c = f == 0 ? 1.0 : -1.0;
                a.msc = -h.omega * h.omega;
                a.accumulate = 0;
                launch_pair<NB, NQS, true, true, NQM>(*h.S, h.M.get(), a, s);
            }
        }

        // ------------------------------------------------------------------------------------------
        // kernel selection
        // ------------------------------------------------------------------------------------------
        // The metric-ring variants of one instance family: ring knob value -> instance. A value that is not listed gets the
        // first entry.
        template <class Fn>
        struct RingVariant
        {
            int ring;
            Fn fn;
        };
        template <class Fn, size_t N>
        Fn ring_variant(const RingVariant<Fn> (&family)[N], int ring)
        {
            for (const RingVariant<Fn> & v : family)
                if (v.ring == ring)
                    return v.fn;
            return family[0].fn;
        }

        // stand-alone thread-per-element operators and stored-metric fused ones: 0 = metric rows through registers, 2 / 5 =
        // shared-memory TMA ring of that many chunks (contract_phase_ring), -5 = per-thread cp.async ring (no row barrier)
        template <int NB, int NQ, bool STIFF>
        const RingVariant<LaunchFn> tpe_rings[4] = {{0, &launch_volume_ws<NB, NQ, STIFF, 0>},
                                                    {-5, &launch_volume_ws<NB, NQ, STIFF, -5>},
                                                    {2, &launch_volume_ws<NB, NQ, STIFF, 2>},
                                                    {5, &launch_volume_ws<NB, NQ, STIFF, 5>}};
        template <int NB, int NQS, int NQM>
        const RingVariant<FusedFn> fused_stored_rings[4] = {{0, &launch_fused_ws<NB, NQS, NQM, 0, false>},
                                                            {-5, &launch_fused_ws<NB, NQS, NQM, -5, false>},
                                                            {2, &launch_fused_ws<NB, NQS, NQM, 2, false>},
                                                            {5, &launch_fused_ws<NB, NQS, NQM, 5, false>}};
        // fused affine operators (the ring carries the mass rows): 0 = straight from global memory into registers, 5 = the TMA
        // ring; any other value: the per-thread cp.async ring of -TR rows
        template <int NB, int NQS, int NQM, int TR>
        const RingVariant<FusedFn> fused_affine_rings[3] = {{TR, &launch_fused_ws<NB, NQS, NQM, TR, true>},
                                                            {0, &launch_fused_ws<NB, NQS, NQM, 0, true>},
                                                            {5, &launch_fused_ws<NB, NQS, NQM, 5, true>}};

        template <bool STIFF>
        LaunchFn find_pair_instance(int nb, int nq, bool affine = false)
        {
#define CB_CASE(NB_, NQ_)                                                                                              \
    if (nb == NB_ && nq == NQ_) {                                                                                      \
        if constexpr (STIFF) {                                                                                         \
            if (affine)                                                                                                \
                return &launch_volume_pair<NB_, NQ_, true, true>;                                                      \
        }                                                                                                              \
        return &launch_volume_pair<NB_, NQ_, STIFF, false>;                                                            \
    }
            // the stored-metric stiffness at n_basis 9 spills its result tile in this kernel (2.73 ms at 1024^2 against 2.11 ms of the
            // lane-per-row kernel): only the affine instance is offered there
            if (STIFF && nb == 9 && !affine)
                return nullptr;
            // default rules nq = nb + 1 (reference StiffnessMatrix.cpp:45, MassMatrix.cpp:74)
            CB_CASE(6, 7) CB_CASE(7, 8) CB_CASE(8, 9) CB_CASE(9, 10)
            if constexpr (!STIFF) { // weighted mass: nq = 1 + 3nb/2 + 1 (MassMatrix.cpp:108)
                CB_CASE(6, 11) CB_CASE(7, 12) CB_CASE(8, 14) CB_CASE(9, 15)
            }
#undef CB_CASE
            return nullptr;
        }

        // thread-per-element instances: n_basis <= 5 (U and the result fit in registers next to the row temporaries)
        // stiffness on all-affine meshes (VolumeOp::affine): per-element metric constants, no metric stream
        LaunchFn find_affine_instance(int nb, int nq)
        {
            if (nb == 5 && nq == 6)
                return &launch_volume_ws<5, 6, true, 0, true>;
            if (nb == 4 && nq == 5)
                return &launch_volume_ws<4, 5, true, 0, true>;
            return nullptr;
        }

        // ring5 / ring4: metric ring of the n_basis 5 / 4 instances of the default rules (stiffness nq = nb + 1, weighted mass)
        template <bool STIFF>
        LaunchFn find_tpe_instance(int nb, int nq, int ring5, int ring4)
        {
#define CB_CASE(NB_, NQ_)                                                                                              \
    if (nb == NB_ && nq == NQ_)                                                                                        \
        return &launch_volume_ws<NB_, NQ_, STIFF>;
            constexpr int NQ5 = STIFF ? 6 : 9, NQ4 = STIFF ? 5 : 8;
            if (nb == 5 && nq == NQ5)
                return ring_variant(tpe_rings<5, NQ5, STIFF>, ring5);
            if (nb == 4 && nq == NQ4)
                return ring_variant(tpe_rings<4, NQ4, STIFF>, ring4);
            CB_CASE(2, 3) CB_CASE(3, 4) CB_CASE(4, 5) CB_CASE(5, 6)
            CB_CASE(3, 5) CB_CASE(4, 6) CB_CASE(5, 7)
            if constexpr (!STIFF) {
                CB_CASE(2, 5) CB_CASE(3, 6)
            }
#undef CB_CASE
            return nullptr;
        }

        template <bool STIFF>
        LaunchFn find_instance(int nb, int nq)
        {
#define CB_CASE(NB_, NQ_)                                                                                              \
    if (nb == NB_ && nq == NQ_)                                                                                        \
        return &launch_volume<NB_, NQ_, STIFF>;
            // default rules: nq = nb + 1 (reference StiffnessMatrix.cpp:45, MassMatrix.cpp:74)
            CB_CASE(2, 3) CB_CASE(3, 4) CB_CASE(4, 5) CB_CASE(5, 6) CB_CASE(6, 7) CB_CASE(7, 8) CB_CASE(8, 9) CB_CASE(9, 10)
            // the reference tests' nb + 2 rules (tests/stiffness.cpp:84, tests/mass.cpp:94)
            CB_CASE(3, 5) CB_CASE(4, 6) CB_CASE(5, 7) CB_CASE(6, 8) CB_CASE(7, 9) CB_CASE(8, 10)
            if constexpr (!STIFF) { // weighted mass: nq = 1 + 3nb/2 + 1 (MassMatrix.cpp:108)
                CB_CASE(2, 5) CB_CASE(3, 6) CB_CASE(4, 8) CB_CASE(5, 9) CB_CASE(6, 11) CB_CASE(7, 12) CB_CASE(8, 14) CB_CASE(9, 15)
            }
#undef CB_CASE
            return nullptr;
        }

        struct VolumeChoice
        {
            VolumeKernel kind;
            bool affine;     // stiffness from per-element metric constants (every element a parallelogram)
            LaunchFn launch; // null for Generic
            Plan * plan;
        };

        // Which kernel runs a stiffness / mass operator. The only reader of the knobs that select one: CUDDH_B200_FORCE_GENERIC,
        // CUDDH_B200_TPE, CUDDH_B200_PAIR, CUDDH_B200_AFFINE (0 = stored metric), CUDDH_B200_RING1 / RING4 (metric ring of the
        // n_basis 5 / 4 thread-per-element operators).
        VolumeChoice select_volume_kernel(H1Space * fem, int nb, int nq, bool stiff, bool want_affine)
        {
            const LaunchFn lane = stiff ? find_instance<true>(nb, nq) : find_instance<false>(nb, nq);
            if (getenv("CUDDH_B200_FORCE_GENERIC") != nullptr || !lane)
                return {VolumeKernel::Generic, false, nullptr, &fem->get_plan()};
            auto affine_ok = [&] { return want_affine && stiff && env_int("CUDDH_B200_AFFINE", 1) != 0 && fem->all_affine(); };
            if (env_int("CUDDH_B200_TPE", 1) != 0) {
                const int ring5 = env_int("CUDDH_B200_RING1", 5), ring4 = env_int("CUDDH_B200_RING4", 5);
                const LaunchFn tpe = stiff ? find_tpe_instance<true>(nb, nq, ring5, ring4) : find_tpe_instance<false>(nb, nq, ring5, ring4);
                if (tpe) {
                    const LaunchFn aff = stiff ? find_affine_instance(nb, nq) : nullptr;
                    const bool affine = aff && affine_ok();
                    return {VolumeKernel::ThreadPerElement, affine, affine ? aff : tpe, &fem->get_plan_tpe()};
                }
            }
            if (env_int("CUDDH_B200_PAIR", 1) != 0) {
                const bool affine = nb >= 6 && affine_ok();
                const LaunchFn pair = stiff ? find_pair_instance<true>(nb, nq, affine) : find_pair_instance<false>(nb, nq);
                // never with H1Space's own numbering and the default patch shape (the CUDDH_B200_TPE_PX / PY experiment knobs can
                // change the latter): the lane-per-row kernel serves such a plan
                if (pair) {
                    Plan & plan = fem->get_plan_tpe();
                    if (plan.PE == 64 && plan.interior_affine)
                        return {VolumeKernel::ThreadPair, affine, pair, &plan};
                }
            }
            return {VolumeKernel::LanePerRow, false, lane, &fem->get_plan()};
        }

        // The fused volume phase of the Helmholtz composite, or null when S and M run one by one. The only reader of the knobs
        // of the fused kernels: CUDDH_B200_FUSED, CUDDH_B200_AFFINE_RING, CUDDH_B200_RING (n_basis 5) / RING4F (n_basis 4).
        FusedFn select_fused_kernel(const VolumeOp & S, const VolumeOp & M)
        {
            if (S.kind != M.kind || S.plan != M.plan || env_int("CUDDH_B200_FUSED", 1) == 0)
                return nullptr;
            // default stiffness rule nq = nb + 1 with the weighted-mass rule nq = 1 + 3nb/2 + 1 (examples/Helmholtz.hpp)
            auto rule = [&](int nb, int nqs, int nqm) { return S.nb == nb && S.nq == nqs && M.nq == nqm; };
            if (S.kind == VolumeKernel::ThreadPerElement && S.affine) {
                const int ring = env_int("CUDDH_B200_AFFINE_RING", -5);
                if (rule(5, 6, 9)) return ring_variant(fused_affine_rings<5, 6, 9, -5>, ring);
                if (rule(4, 5, 8)) return ring_variant(fused_affine_rings<4, 5, 8, -4>, ring);
            }
            else if (S.kind == VolumeKernel::ThreadPerElement) {
                // stored metric: per-thread chunk ring (n_basis 5: 0.704 ms against 0.719 ms of the TMA ring, n_basis 4: 0.388 / 0.437)
                if (rule(5, 6, 9)) return ring_variant(fused_stored_rings<5, 6, 9>, env_int("CUDDH_B200_RING", -5));
                if (rule(4, 5, 8)) return ring_variant(fused_stored_rings<4, 5, 8>, env_int("CUDDH_B200_RING4F", -5));
                if (rule(2, 3, 5)) return &launch_fused_ws<2, 3, 5, 0, false>;
                if (rule(3, 4, 6)) return &launch_fused_ws<3, 4, 6, 0, false>;
            }
            else if (S.kind == VolumeKernel::ThreadPair && S.affine) { // stored-metric meshes keep the per-operator launches (see volume_action_pair)
                if (rule(6, 7, 11)) return &launch_fused_pair<6, 7, 11>;
                if (rule(7, 8, 12)) return &launch_fused_pair<7, 8, 12>;
                if (rule(8, 9, 14)) return &launch_fused_pair<8, 9, 14>;
                if (rule(9, 10, 15)) return &launch_fused_pair<9, 10, 15>;
            }
            return nullptr;
        }
    } // namespace

    int max_persistent_ctas() { return g_max_ctas.load(); }
    void set_max_persistent_ctas(int n) { g_max_ctas.store(n > 0 ? n : 0); }

    void VolumeOp::apply(double c, int accumulate, const double * x, double * y, cudaStream_t s, int phases)
    {
        NvtxRange nvtx_(stiff ? "cuddh::StiffnessMatrix::action" : "cuddh::MassMatrix::action");
        const Plan & plan = *this->plan;
        if ((phases & 1) && launch)
            launch(*this, c, accumulate, x, y, s);
        else if (phases & 1) {
            const int nwarps = std::min(8, plan.PE);
            const int SCR = (stiff ? 2 : 1) * nq * nb;
            size_t smem = sizeof(double) * ((size_t)plan.max_pdof + (size_t)plan.PE * nb * nb + (size_t)nwarps * SCR) +
                          sizeof(uint16_t) * (size_t)plan.PE * nb * nb;
            smem = (smem + 15) & ~size_t(15);
            CB_REQUIRE(smem <= 227 * 1024, "operator action: patch does not fit in shared memory for this (n_basis, n_quad)");
            CB_CUDA(cudaFuncSetAttribute(volume_action_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max(smem, (size_t)49152)));
            volume_action_generic<<<(unsigned)plan.n_patches, nwarps * 32, smem, s>>>(nb, nq, stiff ? 1 : 0, d_P.p, d_D.p, plan_dev(plan), d_G.p, x,
                                                                                      y, d_partial.p, c, accumulate, plan.max_pdof);
            CB_LAUNCHED();
        }
        if (plan.n_shared > 0 && (phases & 2)) {
            assemble_shared_kernel<<<blocks_for(plan.n_shared, 256), 256, 0, s>>>(plan.n_shared, plan.d_sh_gid.p, plan.d_sh_ptr.p,
                                                                                  d_partial.p, y, c, accumulate);
            CB_LAUNCHED();
        }
    }

    size_t VolumeOp::algorithmic_bytes() const
    {
        // SURVEY §8(d): stiffness 24nq^2 + 4nb^2 + 16(nb-1)^2 ; mass 8nq^2 + 4nb^2 + 16(nb-1)^2 bytes per element
        const size_t per = (size_t)(stiff ? 24 : 8) * nq * nq + 4 * (size_t)nb * nb + 16 * (size_t)(nb - 1) * (nb - 1);
        return per * (size_t)fem->n_elem;
    }

    size_t VolumeOp::moved_bytes() const
    {
        if (!affine)
            return algorithmic_bytes();
        const size_t per = 24 + 4 * (size_t)nb * nb + 16 * (size_t)(nb - 1) * (nb - 1);
        return per * (size_t)fem->n_elem;
    }

    namespace
    {
        // layout of the metric data for the setup kernels (metric_index / metric_index_pair): EPW -1 thread-pair, 0 thread-per-element,
        // otherwise the elements per warp pass of the lane-per-row (32 / nq) or generic (1) kernel, n_pass passes per patch
        struct MetricLayout
        {
            int epw, n_pass;
        };

        // chooses the kernel, allocates the metric data and returns its layout
        MetricLayout init_volume_common(VolumeOp & op, H1Space * fem, int nq, bool stiff, bool want_affine = false)
        {
            op.fem = fem;
            op.nb = fem->nb;
            op.nq = nq;
            op.stiff = stiff;
            CB_REQUIRE(nq >= 1 && nq <= MAXQ, stiff ? "StiffnessMatrix::action does not support quadrature rules with more than 24 points."
                                                    : "MassMatrix error: quadrature rules with more than 32 points not yet supported.");
            const VolumeChoice k = select_volume_kernel(fem, op.nb, nq, stiff, want_affine);
            op.kind = k.kind;
            op.affine = k.affine;
            op.launch = k.launch;
            op.plan = k.plan;
            const Plan & plan = *op.plan;
            const int nki = stiff ? 3 : 1; // metric values per quadrature point
            MetricLayout ml{0, 0};
            size_t n_metric;
            if (op.kind == VolumeKernel::ThreadPair) { // [row][pair of metric values][thread slot], see metric_index_pair
                const int TA = (nq + 1) / 2, KR = (nki * TA + 1) & ~1;
                ml.epw = -1;
                n_metric = (size_t)plan.n_patches * (size_t)nq * KR * 128;
            }
            else if (op.kind == VolumeKernel::ThreadPerElement) // [pair of metric values][element], see volume_action_ws
                n_metric = (size_t)plan.n_patches * (size_t)(nq * ((nki * nq + 1) & ~1)) * plan.PE;
            else { // lane-major per warp pass, see metric_index
                ml.epw = op.kind == VolumeKernel::Generic ? 1 : 32 / nq;
                ml.n_pass = (plan.PE + ml.epw - 1) / ml.epw;
                n_metric = (size_t)plan.n_patches * ml.n_pass * (nki * nq) * (ml.epw * nq);
            }
            if (op.affine)
                op.d_Gc.alloc((size_t)plan.n_patches * 3 * plan.PE);
            else
                op.d_G.alloc(n_metric);
            op.d_partial.alloc((size_t)std::max<int64_t>(plan.n_slots_total, 1));
            if (op.d_G.n)
                CB_CUDA(cudaMemset(op.d_G.p, 0, op.d_G.n * sizeof(double)));
            return ml;
        }
    } // namespace

    std::unique_ptr<VolumeOp> make_stiffness(H1Space * fem, int nq, int quad_type)
    {
        std::unique_ptr<VolumeOp> op(new VolumeOp);
        if (nq <= 0)
            nq = fem->nb + 1; // mesh.max_element_order() (=1) + n_basis, StiffnessMatrix.cpp:45
        CB_REQUIRE(nq <= 24, "StiffnessMatrix::action does not support quadrature rules with more than 24 points.");
        const MetricLayout ml = init_volume_common(*op, fem, nq, true, quad_type == GAUSS_LEGENDRE);
        std::vector<double> xq(nq), wq(nq);
        quadrature_rule(nq, quad_type, xq.data(), wq.data());
        op->wq = wq;
        op->P.resize((size_t)nq * fem->nb);
        op->D.resize((size_t)nq * fem->nb);
        fem->basis->eval(nq, xq.data(), op->P.data());
        fem->basis->deriv(nq, xq.data(), op->D.data());
        op->d_P.upload(op->P);
        op->d_D.upload(op->D);
        DevBuf<double> d_x, d_w;
        d_x.upload(xq);
        d_w.upload(wq);
        Plan & plan = *op->plan;
        const int64_t n_slots = plan.n_patches * plan.PE;
        if (op->affine)
            setup_stiffness_affine_kernel<<<blocks_for(n_slots, 256), 256>>>(n_slots, plan.PE, plan.d_slot_elem.p, fem->device_corners(), op->d_Gc.p);
        else
            setup_stiffness_kernel<<<blocks_for(n_slots * nq * nq, 256), 256>>>(n_slots, plan.PE, nq, ml.epw, ml.n_pass, plan.d_slot_elem.p,
                                                                                fem->device_corners(), d_x.p, d_w.p, op->d_G.p);
        CB_LAUNCHED();
        CB_CUDA(cudaDeviceSynchronize());
        return op;
    }

    std::unique_ptr<VolumeOp> make_mass(H1Space * fem, const double * d_coef, int nq)
    {
        std::unique_ptr<VolumeOp> op(new VolumeOp);
        if (nq <= 0) // MassMatrix.cpp:74 (unweighted) / :108 (weighted)
            nq = d_coef ? (1 + 3 * fem->nb / 2 + 1) : (fem->nb + 1);
        const MetricLayout ml = init_volume_common(*op, fem, nq, false);
        std::vector<double> xq(nq), wq(nq);
        quadrature_rule(nq, GAUSS_LEGENDRE, xq.data(), wq.data());
        op->P.resize((size_t)nq * fem->nb);
        fem->basis->eval(nq, xq.data(), op->P.data());
        op->d_P.upload(op->P);
        DevBuf<double> d_x, d_w;
        d_x.upload(xq);
        d_w.upload(wq);
        Plan & plan = *op->plan;
        const int64_t n_slots = plan.n_patches * plan.PE;
        setup_mass_kernel<<<blocks_for(n_slots * nq * nq, 256), 256>>>(n_slots, plan.PE, fem->nb, nq, ml.epw, ml.n_pass, plan.d_slot_elem.p,
                                                                       fem->device_corners(), fem->device_I(), d_coef, op->d_P.p, d_x.p,
                                                                       d_w.p, op->d_G.p);
        CB_LAUNCHED();
        CB_CUDA(cudaDeviceSynchronize());
        return op;
    }

    void DiagOp::apply(double c, int accumulate, const double * x, double * y, cudaStream_t s)
    {
        if (n == 0)
            return;
        diag_apply_kernel<<<blocks_for(n, 256), 256, 0, s>>>(n, d_p.p, c, accumulate, x, y);
        CB_LAUNCHED();
    }

    std::unique_ptr<DiagOp> make_diag_inv_mass(H1Space * fem, const double * d_coef)
    {
        // reference source/MassMatrix.cpp:241-314: p = 1 / sum_e w_i w_j detJ(x_i,x_j) [a], GLL collocation
        std::unique_ptr<DiagOp> op(new DiagOp);
        op->n = fem->ndof;
        op->d_p.alloc((size_t)fem->ndof);
        const int nb = fem->nb;
        const int64_t N = (int64_t)nb * nb * fem->n_elem;
        // transposed map (DOF -> element-local entries, ascending) for an ordered, atomic-free sum
        std::vector<int> ptr((size_t)fem->ndof + 1, 0), src((size_t)N);
        for (int64_t t = 0; t < N; ++t)
            ptr[fem->I[t] + 1]++;
        for (int64_t d = 0; d < fem->ndof; ++d)
            ptr[d + 1] += ptr[d];
        {
            std::vector<int> cur(ptr.begin(), ptr.end() - 1);
            for (int64_t t = 0; t < N; ++t)
                src[cur[fem->I[t]]++] = (int)t;
        }
        DevBuf<int> d_ptr, d_src;
        d_ptr.upload(ptr);
        d_src.upload(src);
        DevBuf<double> contrib((size_t)N), d_x, d_w;
        d_x.upload(fem->basis->x);
        d_w.upload(fem->basis->w);
        diag_mass_contrib_kernel<<<blocks_for(N, 256), 256>>>(fem->n_elem, nb, fem->device_I(), fem->device_corners(), d_coef, d_x.p, d_w.p,
                                                              contrib.p);
        CB_LAUNCHED();
        gather_sum_recip_kernel<<<blocks_for(fem->ndof, 256), 256>>>(fem->ndof, d_ptr.p, d_src.p, contrib.p, op->d_p.p);
        CB_LAUNCHED();
        CB_CUDA(cudaDeviceSynchronize());
        return op;
    }

    std::unique_ptr<FaceMassOp> make_facemass(FaceSpace * fs, const double * d_coef, int nq)
    {
        std::unique_ptr<FaceMassOp> op(new FaceMassOp);
        fs->ensure_device();
        op->fs = fs;
        op->nb = fs->nb;
        if (nq <= 0) // FaceMassMatrix.cpp:56 / :103
            nq = d_coef ? (1 + 3 * fs->nb / 2 + 1) : (fs->nb + 1);
        CB_REQUIRE(nq <= 64, "FaceMassMatrix does not support quadrature rules with more than 64 points.");
        op->nq = nq;
        std::vector<double> xq(nq), wq(nq), P((size_t)nq * fs->nb);
        quadrature_rule(nq, GAUSS_LEGENDRE, xq.data(), wq.data());
        fs->fem->basis->eval(nq, xq.data(), P.data());
        op->d_P.upload(P);
        DevBuf<double> d_w;
        d_w.upload(wq);
        op->d_a.alloc((size_t)nq * fs->n_faces);
        if (fs->n_faces > 0) {
            setup_facemass_kernel<<<blocks_for(fs->n_faces * nq, 128), 128>>>(fs->n_faces, fs->nb, nq, d_w.p, op->d_P.p, fs->d_meas.p, d_coef,
                                                                              fs->d_I.p, op->d_a.p);
            CB_LAUNCHED();
            CB_CUDA(cudaDeviceSynchronize());
        }
        return op;
    }

    void FaceMassOp::apply(double c, int accumulate, const double * x, double * y, cudaStream_t s)
    {
        NvtxRange nvtx_("cuddh::FaceMassMatrix::action");
        if (fs->fdof == 0)
            return;
        facemass_action_kernel<<<blocks_for(fs->fdof, 128), 128, 0, s>>>(fs->fdof, nb, nq, d_P.p, d_a.p, fs->d_I.p, fs->d_inc_ptr.p,
                                                                         fs->d_inc.p, nullptr, c, accumulate, x, y);
        CB_LAUNCHED();
    }

    void FaceMassOp::apply_h1(double c, const double * x, double * y, cudaStream_t s)
    {
        if (fs->fdof == 0)
            return;
        facemass_action_kernel<<<blocks_for(fs->fdof, 128), 128, 0, s>>>(fs->fdof, nb, nq, d_P.p, d_a.p, fs->d_I.p, fs->d_inc_ptr.p,
                                                                         fs->d_inc.p, fs->d_proj.p, c, 1, x, y);
        CB_LAUNCHED();
    }

    namespace
    {
        // device view for ONE exchange; begin_exchange() has advanced the epoch
        HaloDev halo_dev(SlabHalo & h)
        {
            HaloDev d{};
            d.row_dof = h.d_row_dof.p;
            d.face_entry = h.d_face_entry.p;
            d.plain = h.d_plain.p;
            d.send = h.d_send.p;
            d.n_bottom = h.n_bottom;
            d.n_top = h.n_top;
            d.n_plain = h.n_plain;
            d.peer = h.peer ? 1 : 0;
            if (h.peer) {
                const int par = (int)(h.epoch & 1);
                for (int side = 0; side < 2; ++side) {
                    d.peer_dst[side] = h.peer_recv[side] ? h.peer_recv[side] + par * h.peer_tot[side] + h.peer_off[side] : nullptr;
                    d.peer_flag[side] = h.peer_flag[side];
                }
                d.ticket = h.d_ticket.p;
                d.epoch = h.epoch;
            }
            return d;
        }
    } // namespace

    void FaceMassOp::apply_h1_pair(double c, const double * x, double * y, int64_t n, cudaStream_t s, SlabHalo * halo)
    {
        const unsigned fb = fs->fdof > 0 ? blocks_for(fs->fdof, 128) : 0;
        const unsigned pb = halo ? blocks_for(halo->n_plain, 128) : 0;
        if (fb + pb == 0)
            return;
        HaloDev hd{};
        if (halo)
            hd = halo_dev(*halo);
        facemass_pair_kernel<<<dim3(fb + pb, 2), 128, 0, s>>>(fs->fdof, nb, nq, d_P.p, d_a.p, fs->d_I.p, fs->d_inc_ptr.p, fs->d_inc.p,
                                                              fs->d_proj.p, c, n, x, y, hd, (int)fb);
        CB_LAUNCHED();
    }

    // ---- peer path of the halo exchange: CUDA IPC mappings of the neighbours' receive buffers ----
    namespace
    {
        struct PeerHello // what neighbours tell each other at setup (through NCCL, 128 bytes)
        {
            cudaIpcMemHandle_t handle;
            int64_t n_bottom, tot;
            char pad[128 - sizeof(cudaIpcMemHandle_t) - 16];
        };
        static_assert(sizeof(PeerHello) == 128, "hello size");
    } // namespace

    SlabHalo::~SlabHalo()
    {
        for (int side = 0; side < 2; ++side)
            if (peer_base[side])
                cudaIpcCloseMemHandle(peer_base[side]);
    }

    void SlabHalo::setup_peer()
    {
        peer = false;
        if (!comm || world == 1 || env_int("CUDDH_B200_PEER", 1) == 0)
            return;
        const int64_t tot = (int64_t)n_fields * (n_bottom + n_top);
        // own block: two parity buffers + two arrival flags (64-byte aligned tail)
        const size_t flag_off = (((size_t)2 * tot * sizeof(double)) + 63) & ~size_t(63);
        d_peer_block.alloc(flag_off + 64);
        CB_CUDA(cudaMemset(d_peer_block.p, 0, d_peer_block.n));
        d_ticket.alloc(1);
        CB_CUDA(cudaMemset(d_ticket.p, 0, sizeof(unsigned)));
        own_recv = reinterpret_cast<double *>(d_peer_block.p);
        own_flags = reinterpret_cast<unsigned long long *>(d_peer_block.p + flag_off);
        own_tot = tot;
        PeerHello mine{};
        int ok = cudaIpcGetMemHandle(&mine.handle, d_peer_block.p) == cudaSuccess ? 1 : 0;
        if (!ok)
            cudaGetLastError();
        mine.n_bottom = n_bottom;
        mine.tot = tot;
        // hello exchange with the two neighbours (device staging: slot 0 <-> lower neighbour, slot 1 <-> upper neighbour)
        DevBuf<unsigned char> d_hs(256), d_hr(256);
        PeerHello both[2] = {mine, mine};
        CB_CUDA(cudaMemcpy(d_hs.p, both, 256, cudaMemcpyHostToDevice));
        std::vector<PeerSeg> hs;
        if (n_bottom > 0)
            hs.push_back(PeerSeg{rank - 1, 0, 128, 0, 128});
        if (n_top > 0)
            hs.push_back(PeerSeg{rank + 1, 128, 128, 128, 128});
        comm_exchange(comm, hs, d_hs.p, d_hr.p, 1, 0);
        CB_CUDA(cudaDeviceSynchronize());
        PeerHello theirs[2];
        CB_CUDA(cudaMemcpy(theirs, d_hr.p, 256, cudaMemcpyDeviceToHost));
        for (int side = 0; side < 2 && ok; ++side) {
            if ((side == 0 ? n_bottom : n_top) == 0)
                continue;
            void * base = nullptr;
            if (cudaIpcOpenMemHandle(&base, theirs[side].handle, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                ok = 0;
                break;
            }
            peer_base[side] = base;
            const int64_t ptot = theirs[side].tot;
            const size_t pflag = (((size_t)2 * ptot * sizeof(double)) + 63) & ~size_t(63);
            peer_recv[side] = reinterpret_cast<double *>(base);
            peer_tot[side] = ptot;
            // my bottom segment is the lower neighbour's TOP segment (after its own bottom segment); my top segment is the upper
            // neighbour's bottom segment (offset 0). Flags: I am the lower neighbour's upper side (flag 1) and vice versa.
            peer_off[side] = side == 0 ? 2 * theirs[side].n_bottom : 0;
            peer_flag[side] = reinterpret_cast<unsigned long long *>(reinterpret_cast<unsigned char *>(base) + pflag) + (side == 0 ? 1 : 0);
        }
        // all ranks or none: a rank that cannot map its neighbours sends everybody back to ncclSend / ncclRecv
        DevBuf<double> d_ok(1);
        const double bad = ok ? 0.0 : 1.0;
        CB_CUDA(cudaMemcpy(d_ok.p, &bad, sizeof(double), cudaMemcpyHostToDevice));
        comm_allreduce_sum(comm, d_ok.p, 1, 0);
        double nbad = 0.0;
        CB_CUDA(cudaMemcpy(&nbad, d_ok.p, sizeof(double), cudaMemcpyDeviceToHost));
        peer = nbad == 0.0;
        if (!peer)
            for (int side = 0; side < 2; ++side) {
                if (peer_base[side])
                    cudaIpcCloseMemHandle(peer_base[side]);
                peer_base[side] = nullptr;
                peer_recv[side] = nullptr;
                peer_flag[side] = nullptr;
            }
    }

    std::unique_ptr<SlabHalo> make_slab_halo(const Comm * comm, int rank, int world, int64_t ndof, FaceSpace * fs_phys, int64_t n_bottom,
                                             const int * h_bottom, int64_t n_top, const int * h_top)
    {
        CB_REQUIRE(world >= 1 && rank >= 0 && rank < world, "slab halo: rank out of range");
        CB_REQUIRE((rank > 0) == (n_bottom > 0) || world == 1, "slab halo: rank > 0 needs a bottom interface row, rank 0 must not have one");
        CB_REQUIRE((rank < world - 1) == (n_top > 0) || world == 1, "slab halo: every rank but the last needs a top interface row");
        std::unique_ptr<SlabHalo> h(new SlabHalo);
        h->comm = comm;
        h->rank = rank;
        h->world = world;
        h->ndof = ndof;
        h->n_bottom = n_bottom;
        h->n_top = n_top;
        std::vector<int> row((size_t)(n_bottom + n_top));
        std::copy(h_bottom, h_bottom + n_bottom, row.begin());
        std::copy(h_top, h_top + n_top, row.begin() + n_bottom);
        for (int v : row)
            CB_REQUIRE(v >= 0 && v < ndof, "slab halo: interface DOF out of range");
        // entries that are also face DOFs of the physical boundary are packed by the face-mass thread that finishes them
        std::vector<int> entry_of_dof;
        std::vector<int> face_entry;
        std::vector<char> covered(row.size(), 0);
        if (fs_phys) {
            fs_phys->ensure_device();
            entry_of_dof.assign((size_t)ndof, -1);
            for (size_t e = 0; e < row.size(); ++e)
                entry_of_dof[row[e]] = (int)e;
            face_entry.assign((size_t)fs_phys->fdof, -1);
            for (int64_t d = 0; d < fs_phys->fdof; ++d) {
                const int e = entry_of_dof[fs_phys->proj[d]];
                face_entry[d] = e;
                if (e >= 0)
                    covered[e] = 1;
            }
        }
        std::vector<int> plain;
        for (size_t e = 0; e < row.size(); ++e)
            if (!covered[e])
                plain.push_back((int)e);
        h->n_plain = (int64_t)plain.size();
        h->d_row_dof.upload(row);
        if (!face_entry.empty())
            h->d_face_entry.upload(face_entry);
        if (!plain.empty())
            h->d_plain.upload(plain);
        const size_t tot = (size_t)h->n_fields * (size_t)(n_bottom + n_top);
        h->d_send.alloc(std::max<size_t>(tot, 1));
        h->d_recv.alloc(std::max<size_t>(tot, 1));
        if (n_bottom > 0)
            h->segs.push_back(PeerSeg{rank - 1, 0, 2 * n_bottom, 0, 2 * n_bottom});
        if (n_top > 0)
            h->segs.push_back(PeerSeg{rank + 1, 2 * n_bottom, 2 * n_top, 2 * n_bottom, 2 * n_top});
        h->setup_peer();
        return h;
    }

    const unsigned char * SlabHalo::mask()
    {
        if (!d_mask.p) {
            std::vector<unsigned char> m((size_t)n_fields * (size_t)ndof, 1);
            if (n_bottom > 0) { // rank > 0 mirrors its bottom row: the rank below owns it (SURVEY §8e: owner = lower rank)
                const std::vector<int> row = d_row_dof.download();
                for (int f = 0; f < n_fields; ++f)
                    for (int64_t e = 0; e < n_bottom; ++e)
                        m[(size_t)f * ndof + row[e]] = 0;
            }
            d_mask.upload(m);
        }
        return d_mask.p;
    }

    void SlabHalo::unpack_add(double * y, cudaStream_t s)
    {
        const int64_t ne = n_bottom + n_top;
        if (ne == 0)
            return;
        const double * recv = peer ? own_recv + (epoch & 1) * own_tot : d_recv.p;
        halo_add_kernel<<<dim3(blocks_for(ne, 256), (unsigned)n_fields), 256, 0, s>>>(halo_dev(*this), recv, ndof, y, own_flags, n_bottom > 0 ? 1 : 0,
                                                                                      n_top > 0 ? 1 : 0);
        CB_LAUNCHED();
    }

    void SlabHalo::exchange(double * y, cudaStream_t s)
    {
        NvtxRange nvtx_("cuddh::SlabHalo::exchange");
        const int64_t ne = n_bottom + n_top;
        if (ne == 0 || world == 1)
            return;
        ++epoch;
        halo_pack_kernel<<<dim3(blocks_for(ne, 256), (unsigned)n_fields), 256, 0, s>>>(halo_dev(*this), ndof, y);
        CB_LAUNCHED();
        if (!peer)
            comm_exchange(comm, segs, d_send.p, d_recv.p, sizeof(double), s);
        unpack_add(y, s);
    }

    std::unique_ptr<DiagOp> make_diag_inv_facemass(FaceSpace * fs, const double * d_coef)
    {
        // reference source/FaceMassMatrix.cpp:226-270
        std::unique_ptr<DiagOp> op(new DiagOp);
        fs->ensure_device();
        op->n = fs->fdof;
        op->d_p.alloc((size_t)std::max<int64_t>(fs->fdof, 1));
        DevBuf<double> d_w;
        d_w.upload(fs->fem->basis->w);
        if (fs->fdof > 0) {
            diag_facemass_kernel<<<blocks_for(fs->fdof, 128), 128>>>(fs->fdof, fs->nb, d_w.p, fs->d_meas.p, d_coef, fs->d_inc_ptr.p,
                                                                     fs->d_inc.p, op->d_p.p);
            CB_LAUNCHED();
            CB_CUDA(cudaDeviceSynchronize());
        }
        return op;
    }

    void face_restrict(FaceSpace * fs, const double * x, double * y, cudaStream_t s)
    {
        if (fs->fdof == 0)
            return;
        fs->ensure_device();
        restrict_kernel<<<blocks_for(fs->fdof, 256), 256, 0, s>>>(fs->fdof, fs->d_proj.p, x, y);
        CB_LAUNCHED();
    }
    void face_prolong(FaceSpace * fs, const double * x, double * y, cudaStream_t s)
    {
        if (fs->fdof == 0)
            return;
        fs->ensure_device();
        prolong_kernel<<<blocks_for(fs->fdof, 256), 256, 0, s>>>(fs->fdof, fs->d_proj.p, x, y);
        CB_LAUNCHED();
    }
    void face_orth(FaceSpace * fs, double * x, cudaStream_t s)
    {
        if (fs->fdof == 0)
            return;
        fs->ensure_device();
        orth_kernel<<<blocks_for(fs->fdof, 256), 256, 0, s>>>(fs->fdof, fs->d_proj.p, x);
        CB_LAUNCHED();
    }

    std::unique_ptr<HelmholtzOp> make_helmholtz(double omega, const double * d_a2, const double * d_a, H1Space * fem, FaceSpace * fs)
    {
        std::unique_ptr<HelmholtzOp> op(new HelmholtzOp);
        op->omega = omega;
        op->fem = fem;
        op->fs = fs;
        op->S = make_stiffness(fem, 0, GAUSS_LEGENDRE);
        op->M = make_mass(fem, d_a2, 0);
        op->H = make_facemass(fs, d_a, 0);
        op->fused = select_fused_kernel(*op->S, *op->M);
        if (op->fused)
            op->d_partial2.alloc(2 * (size_t)partial_stride(*op));
        return op;
    }

    void HelmholtzOp::apply(const double * x, double * y, cudaStream_t s, int phases)
    {
        NvtxRange nvtx_("cuddh::Helmholtz::action");
        // examples/Helmholtz.hpp:28-56:  Au = S u - w^2 M u - w H v ;  Av = -(S v - w^2 M v + w H u)
        const int64_t n = fem->ndof;
        const double * u = x;
        const double * v = x + n;
        double * Au = y;
        double * Av = y + n;
        if (fused) {
            // one volume kernel walks (patch, field) units: S and M share the gather, the index lists and the assembly, the
            // sign of the second block row is applied on write: 3 launches instead of 11 + 4 memsets
            if (phases & 1)
                fused(*this, x, y, s);
            if (phases & 2) {
                assemble_shared_fields(*this, y, s);
                H->apply_h1_pair(-omega, x, y, n, s); // Au -= w H v ; Av -= w H u in one launch
            }
            return;
        }
        // 7 launches + 4 tiny assembly passes instead of the reference's 11 kernels + 4 memsets.
        S->apply(1.0, 0, u, Au, s);
        S->apply(1.0, 0, v, Av, s);
        M->apply(-omega * omega, 1, u, Au, s);
        M->apply(-omega * omega, 1, v, Av, s);
        H->apply_h1(-omega, v, Au, s);
        H->apply_h1(omega, u, Av, s);
        negate_kernel<<<blocks_for(n, 256), 256, 0, s>>>(n, Av);
        CB_LAUNCHED();
    }

    void HelmholtzOp::apply_slab(const double * x, double * y, SlabHalo & halo, cudaStream_t s)
    {
        NvtxRange nvtx_("cuddh::Helmholtz::action (slab + halo exchange)");
        CB_REQUIRE(halo.ndof == fem->ndof && halo.n_fields == 2, "apply_slab: halo was built for another space");
        if (halo.world == 1) {
            apply(x, y, s);
            return;
        }
        if (fused) {
            // volume kernel + shared-DOF pass, then ONE launch for both face terms and the pack of the interface rows
            apply(x, y, s, 1);
            assemble_shared_fields(*this, y, s);
            ++halo.epoch;
            H->apply_h1_pair(-omega, x, y, fem->ndof, s, &halo);
            if (!halo.peer)
                comm_exchange(halo.comm, halo.segs, halo.d_send.p, halo.d_recv.p, sizeof(double), s);
            halo.unpack_add(y, s);
        }
        else {
            apply(x, y, s);
            halo.exchange(y, s);
        }
    }

    size_t HelmholtzOp::moved_bytes() const
    {
        const size_t nb = S->nb, nqs = S->nq, nqm = M->nq;
        const size_t metric_s = S->affine ? 24 : 24 * nqs * nqs;
        return (metric_s + 8 * nqm * nqm + 4 * nb * nb + 32 * (nb - 1) * (nb - 1)) * (size_t)fem->n_elem;
    }

    size_t HelmholtzOp::algorithmic_bytes() const
    {
        // SURVEY §8(d), fused complex apply: metric data and index map read once for u and v
        const size_t nb = S->nb, nqs = S->nq, nqm = M->nq;
        return (24 * nqs * nqs + 8 * nqm * nqm + 4 * nb * nb + 32 * (nb - 1) * (nb - 1)) * (size_t)fem->n_elem;
    }
} // namespace cb200
