// Assembled DDH interface operator for sm_100a: T probed once per subdomain, then applied as a batched matvec.
//
// T (DDH::action = x - T x) is linear and block-sparse: subdomain p reads only its incoming slots (lambda, mu) at B(j,0,p) and writes
// only its outgoing slots B(i,1,p). Every slot has at most one reader and at most one writer (cross-point overwrites of B included;
// transfer_slots() checks it), so T is one dense 2F x 2F block M_p per subdomain between a gather and a scatter.
//
// Probing: probe k sets local input k of EVERY subdomain to 1 (one slot each, no slot shared) and runs the WaveHoltz kernel that
// serves the DDH handle (reg4 / reg8 / generic): column k of every M_p is that kernel's output, gathered at the subdomain's
// outgoing slots. 2F actions fill all blocks.
//
// Action: one launch. A CTA takes SPB subdomains; it gathers their 2F inputs into shared memory (0 for face DOFs on the physical
// boundary), then each thread owns four consecutive rows of one block and walks the columns in ascending k with 128-bit
// streaming loads (no L1 allocation, L2 evict-first: the blocks stream through while the Krylov vectors stay in L2), so the sum
// order is fixed and the result deterministic. y[out(i,p)] = x[out(i,p)] - r_i; extra CTAs copy the orphan slots (y = x).
// For a unit vector the matvec adds exact zeros to the probed entry, so it reproduces DDH::action bit for bit.
#include "ddh.hpp"

namespace cb200
{
    void transfer_slots(const DDH & D, TransferSlots & S)
    {
        const int n1 = D.n1, nd = n1 * n1;
        std::vector<char> ring(nd, 0);
        S.face_at.clear();
        for (int at = 0; at < nd; ++at) {
            const int X = at % n1, Y = at / n1;
            if (X == 0 || Y == 0 || X == n1 - 1 || Y == n1 - 1) {
                ring[at] = 1;
                S.face_at.push_back(at);
            }
        }
        const int F = (int)S.face_at.size();
        CB_REQUIRE(F == D.mx_fdof, "DDH transfer: the face DOFs of a subdomain are not the boundary ring of its grid");
        S.two_f = 2 * F;
        S.n_domains = D.n_domains;
        S.n_lambda = D.n_lambda;
        const int64_t n = 2 * D.n_lambda, TF = S.two_f;
        S.in.assign((size_t)TF * D.n_domains, -1);
        S.out.assign((size_t)TF * D.n_domains, -1);
        std::vector<char> read((size_t)n, 0), written((size_t)n, 0);
        auto claim = [&](std::vector<char> & seen, int64_t slot, const char * what) {
            if (seen[(size_t)slot])
                throw Error(-1, "DDH transfer: slot " + std::to_string(slot) + " has more than one " + what);
            seen[(size_t)slot] = 1;
        };
        for (int p = 0; p < D.n_domains; ++p) {
            const size_t g0 = (size_t)nd * p;
            for (int at = 0; at < nd; ++at)
                if (!ring[at])
                    CB_REQUIRE(D.hg_bin[g0 + at] < 0 && D.hg_bout[g0 + at] < 0, "DDH transfer: a subdomain-interior DOF carries an interface slot");
            for (int f = 0; f < F; ++f) {
                const int bi = D.hg_bin[g0 + S.face_at[f]], bo = D.hg_bout[g0 + S.face_at[f]];
                CB_REQUIRE(bi < D.n_lambda && bo < D.n_lambda, "DDH transfer: slot index out of range");
                const size_t c = (size_t)TF * p;
                if (bi >= 0) {
                    claim(read, bi, "reader");
                    claim(read, D.n_lambda + bi, "reader");
                    S.in[c + f] = bi;
                    S.in[c + F + f] = (int)(D.n_lambda + bi);
                }
                if (bo >= 0) {
                    claim(written, bo, "writer");
                    claim(written, D.n_lambda + bo, "writer");
                    S.out[c + f] = bo;
                    S.out[c + F + f] = (int)(D.n_lambda + bo);
                }
            }
        }
        S.orphans.clear();
        for (int64_t s = 0; s < n; ++s)
            if (!written[(size_t)s])
                S.orphans.push_back((int)s);
    }

    namespace
    {
        constexpr int TR_THREADS = 256;

        // L2 policy that marks lines evict-first (the blocks are read once per action)
        __device__ __forceinline__ uint64_t evict_first_policy()
        {
            uint64_t pol;
            asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
            return pol;
        }

        // 128-bit load that does not allocate in L1, with the L2 policy above
        __device__ __forceinline__ float4 ld_stream(const float4 * p, const uint64_t pol)
        {
            float4 v;
            asm("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
                : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                : "l"(p), "l"(pol));
            return v;
        }

        // TF = 2F rows / columns per block; Q = TF / 4 threads per subdomain, SPB subdomains per CTA
        template <int TF>
        struct TransferShape
        {
            static constexpr int Q = TF / 4;
            static constexpr int SPB = TR_THREADS / Q;
            static constexpr int NT = Q * SPB;
            static constexpr int XS = TF + 1; // shared-memory row stride of the gathered inputs (TF is a multiple of 16: pad off bank 0)
        };

        template <int TF>
        __global__ void __launch_bounds__(TR_THREADS)
        ddh_transfer_action_kernel(const float * __restrict__ M, const int * __restrict__ in, const int * __restrict__ out,
                                   const int * __restrict__ orphans, const int n_orphans, const float * __restrict__ x, float * __restrict__ y,
                                   const int n_domains, const int n_dom_ctas)
        {
            using SH = TransferShape<TF>;
            constexpr int Q = SH::Q, SPB = SH::SPB, NT = SH::NT, XS = SH::XS;
            __shared__ float s_x[SPB * XS];

            if ((int)blockIdx.x >= n_dom_ctas) { // slots no subdomain writes: y = x
                const int i = ((int)blockIdx.x - n_dom_ctas) * NT + (int)threadIdx.x;
                if (i < n_orphans) {
                    const int o = __ldg(orphans + i);
                    y[o] = __ldg(x + o);
                }
                return;
            }
            const int dom0 = blockIdx.x * SPB;
            const int nloc = min(SPB, n_domains - dom0);
            const int * inb = in + (size_t)dom0 * TF;
            for (int t = threadIdx.x; t < nloc * TF; t += NT) {
                const int s = __ldg(inb + t);
                s_x[(t / TF) * XS + t % TF] = s >= 0 ? __ldg(x + s) : 0.0f;
            }
            __syncthreads();
            const int sub = threadIdx.x / Q, q = threadIdx.x % Q;
            if (sub >= nloc)
                return;
            const int dom = dom0 + sub;
            const float4 * Mp = reinterpret_cast<const float4 *>(M + (size_t)dom * TF * TF) + q;
            const float * xs = s_x + sub * XS;
            const uint64_t pol = evict_first_policy();
            float r0 = 0.0f, r1 = 0.0f, r2 = 0.0f, r3 = 0.0f;
#pragma unroll 16
            for (int k = 0; k < TF; ++k) {
                const float4 m = ld_stream(Mp + (size_t)k * Q, pol);
                const float xk = xs[k];
                r0 = fmaf(m.x, xk, r0);
                r1 = fmaf(m.y, xk, r1);
                r2 = fmaf(m.z, xk, r2);
                r3 = fmaf(m.w, xk, r3);
            }
            const int4 o = __ldg(reinterpret_cast<const int4 *>(out + (size_t)dom * TF) + q);
            if (o.x >= 0) y[o.x] = __ldg(x + o.x) - r0;
            if (o.y >= 0) y[o.y] = __ldg(x + o.y) - r1;
            if (o.z >= 0) y[o.z] = __ldg(x + o.z) - r2;
            if (o.w >= 0) y[o.w] = __ldg(x + o.w) - r3;
        }

        // probe k: local input k of every subdomain to 1, input k - 1 of the previous probe back to 0 (no slot has two readers,
        // so the two writes never meet)
        __global__ void ddh_transfer_probe_scatter(const int * __restrict__ in, const int TF, const int k, const int n_domains,
                                                   float * __restrict__ xk)
        {
            const int p = blockIdx.x * blockDim.x + threadIdx.x;
            if (p >= n_domains)
                return;
            const size_t c = (size_t)TF * p;
            if (k > 0) {
                const int s = in[c + k - 1];
                if (s >= 0)
                    xk[s] = 0.0f;
            }
            const int s = in[c + k];
            if (s >= 0)
                xk[s] = 1.0f;
        }

        // column k of every block: t at the subdomain's outgoing slots (0 where it has no input k or no outgoing slot)
        __global__ void ddh_transfer_probe_gather(const int * __restrict__ in, const int * __restrict__ out, const float * __restrict__ t,
                                                  const int TF, const int k, const int n_domains, float * __restrict__ M)
        {
            const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
            if (g >= (int64_t)TF * n_domains)
                return;
            const int64_t p = g / TF, i = g % TF;
            const int o = out[g];
            const bool has = in[TF * p + k] >= 0;
            M[(size_t)p * TF * TF + (size_t)k * TF + i] = (has && o >= 0) ? t[o] : 0.0f;
        }

        template <int TF>
        void launch_action(const DDHTransfer & T, const float * x, float * y, cudaStream_t s)
        {
            using SH = TransferShape<TF>;
            const int nd = T.slots.n_domains, no = (int)T.slots.orphans.size();
            const int dom_ctas = (nd + SH::SPB - 1) / SH::SPB;
            const int orph_ctas = (no + SH::NT - 1) / SH::NT;
            ddh_transfer_action_kernel<TF><<<dom_ctas + orph_ctas, SH::NT, 0, s>>>(T.d_M.p, T.d_in.p, T.d_out.p, T.d_orphans.p, no, x, y, nd,
                                                                                 dom_ctas);
            CB_LAUNCHED();
        }
    } // namespace

    DDHTransfer::DDHTransfer(DDH * ddh_, int64_t max_bytes, cudaStream_t s) : ddh(ddh_)
    {
        NvtxRange nvtx_("cuddh::DDHTransfer probe");
        transfer_slots(*ddh, slots);
        const int TF = slots.two_f, nd = slots.n_domains;
        CB_REQUIRE(TF == 96 || TF == 112 || TF == 192 || TF == 224, "DDH transfer: no action kernel for this n_basis / block");
        CB_REQUIRE(max_bytes >= 0, "DDH transfer: max_bytes must be >= 0");
        const int64_t n = 2 * slots.n_lambda;
        const int64_t maps = (int64_t)(slots.in.size() + slots.out.size() + slots.orphans.size()) * (int64_t)sizeof(int);
        const int64_t needed = block_bytes() + maps + 2 * n * (int64_t)sizeof(float); // + the two probe vectors
        if (max_bytes == 0) {
            size_t fr = 0, tot = 0;
            CB_CUDA(cudaMemGetInfo(&fr, &tot));
            max_bytes = (int64_t)fr;
        }
        if (needed > max_bytes)
            throw Error(-1, "DDH transfer: needs " + std::to_string(needed) + " bytes of device memory (" + std::to_string(block_bytes()) +
                                " for the blocks), only " + std::to_string(max_bytes) + " available");

        ddh->ensure_device();
        d_in.upload(slots.in);
        d_out.upload(slots.out);
        d_orphans.upload(slots.orphans);
        d_M.alloc((size_t)TF * TF * nd);
        DevBuf<float> xk((size_t)n), t((size_t)n);
        xk.zero(s);

        cudaEvent_t e0, e1;
        CB_CUDA(cudaEventCreate(&e0));
        CB_CUDA(cudaEventCreate(&e1));
        const int64_t launches0 = g_launches.load();
        try {
            CB_CUDA(cudaEventRecord(e0, s));
            const unsigned sc_blocks = (unsigned)((nd + 255) / 256);
            const unsigned ga_blocks = (unsigned)(((int64_t)TF * nd + 255) / 256);
            for (int k = 0; k < TF; ++k) {
                ddh_transfer_probe_scatter<<<sc_blocks, 256, 0, s>>>(d_in.p, TF, k, nd, xk.p);
                CB_LAUNCHED();
                ddh->run(nullptr, nullptr, xk.p, t.p, s);
                ddh_transfer_probe_gather<<<ga_blocks, 256, 0, s>>>(d_in.p, d_out.p, t.p, TF, k, nd, d_M.p);
                CB_LAUNCHED();
            }
            CB_CUDA(cudaEventRecord(e1, s));
            CB_CUDA(cudaEventSynchronize(e1));
            float ms = 0.0f;
            CB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
            probe_ms = ms;
        }
        catch (...) {
            cudaStreamSynchronize(s);
            cudaEventDestroy(e0);
            cudaEventDestroy(e1);
            throw;
        }
        probe_launches = g_launches.load() - launches0;
        CB_CUDA(cudaEventDestroy(e0));
        CB_CUDA(cudaEventDestroy(e1));
    }

    int64_t DDHTransfer::bytes_per_action() const
    {
        const int64_t v = (int64_t)slots.two_f * slots.n_domains;
        // blocks, in / out maps, gathered x, x and y at the written slots, orphan index + x + y
        return block_bytes() + 2 * v * 4 + v * 4 + 2 * v * 4 + 3 * (int64_t)slots.orphans.size() * 4;
    }

    void DDHTransfer::action(const float * x, float * y, cudaStream_t s)
    {
        NvtxRange nvtx_("cuddh::DDHTransfer::action");
        const int64_t n = 2 * slots.n_lambda;
        CB_REQUIRE(x + n <= y || y + n <= x, "DDH transfer action: x and y must not overlap");
        switch (slots.two_f) {
        case 96: launch_action<96>(*this, x, y, s); break;
        case 112: launch_action<112>(*this, x, y, s); break;
        case 192: launch_action<192>(*this, x, y, s); break;
        case 224: launch_action<224>(*this, x, y, s); break;
        default: throw Error(-1, "DDH transfer: no action kernel for this n_basis / block");
        }
    }

    void DDHTransfer::get_block(int dom, float * h_out) const
    {
        CB_REQUIRE(dom >= 0 && dom < slots.n_domains, "DDH transfer: subdomain out of range");
        const size_t bb = (size_t)slots.two_f * slots.two_f;
        CB_CUDA(cudaMemcpy(h_out, d_M.p + bb * dom, bb * sizeof(float), cudaMemcpyDeviceToHost));
    }
} // namespace cb200
