// DDH: the FP32 substructured Helmholtz operator (path B of SURVEY §8a) — reference include/DDH.hpp,
// source/DDH.cpp, source/EnsembleSpace.cpp.
#pragma once
#include "common.hpp"
#include "dist.hpp"

namespace cb200
{
    // Subdomain index maps with the reference's numbering (source/EnsembleSpace.cpp:11-287); host only.
    struct Ensemble
    {
        int n_spaces = 0, nb = 0;
        int mx_elems = 0, mx_faces = 0, mx_ndof = 0, mx_fdof = 0;
        int64_t n_shared = 0;
        std::vector<int> s_elems, s_faces, s_dof, s_fdof;
        std::vector<int> elems;      // (mx_elems, p)
        std::vector<int> faces;      // (mx_faces, p) global edge ids
        std::vector<int> face_side;  // (mx_faces, p)
        std::vector<int> sI;         // (nb, nb, mx_elems, p)
        std::vector<int> gI;         // (mx_ndof, p)
        std::vector<int> fI;         // (nb, mx_faces, p)
        std::vector<int> pI;         // (mx_fdof, p)
        std::vector<int> cmap;       // (4, n_shared)
        Ensemble(const H1Space & fem, int n_spaces, const int * labels);
    };

    struct DDH
    {
        H1Space * fem;
        int nb, block, nel1;         // nel1 = block / nb elements per subdomain side
        int n1;                      // unique DOFs per subdomain side = nel1*(nb-1)+1
        int64_t g_ndof, n_shared, n_lambda;
        int n_domains, nt, mx_dof, mx_fdof, mx_elem;
        double omega, dt;
        std::unique_ptr<Ensemble> en;

        // reference-layout host arrays (kept for parity tests / introspection)
        std::vector<int> B, gI, sI;
        std::vector<float> m, gmi, a, H, D, wh_filter, cs, sn;
        std::vector<float> g_first;       // (3, nb, nb) geometric factors of one element (all elements alike on uniform_rect)
        mutable std::vector<float> g;     // (3, nb, nb, mx_elem, dom), built on demand by full_metric()
        bool uniform_metric = false;
        const std::vector<float> & full_metric() const;

        // device arrays in the kernel's grid layout: per subdomain, per unique DOF (Y*n1 + X)
        DevBuf<int> d_gid, d_bin, d_bout;
        DevBuf<float> d_a, d_m, d_pou, d_H, d_g, d_D, d_whf, d_cs, d_sn;
        // deterministic partition-of-unity assembly of postprocess(): per-DOF contribution slots
        DevBuf<int> d_asm_ptr, d_asm_src;
        DevBuf<double> d_contrib;
        // host copies of the grid-layout tables (uploaded lazily so that the index data can be built and
        // inspected without a GPU)
        std::vector<int> hg_gid, hg_bin, hg_bout, h_asm_ptr, h_asm_src;
        std::vector<float> hg_a, hg_m, hg_pou, hg_H;
        bool on_device = false;
        void ensure_device();
        // metric diagonal and identical in every element (uniform_rect): enables the register-tiled kernel
        bool reg_tiled_ok = false;

        DDH(double omega, const double * h_a, H1Space * fem, int nx, int ny, int block);
        void rhs(const double * f, float * b, cudaStream_t s);
        void action(const float * x, float * y, cudaStream_t s);
        void postprocess(const float * lambda, const double * f, double * u, cudaStream_t s);
        void apply_T_range(const float * x, float * t, int dom_begin, int dom_end, cudaStream_t s);
        void rhs_range(const double * f, float * b, int dom_begin, int dom_end, cudaStream_t s);
        void postprocess_range(const float * lambda, const double * f, double * u, int dom_begin, int dom_end, cudaStream_t s);
        void get_array(const char * name, void * out, int64_t cap_bytes, int64_t * count) const;
        double flops() const;

        int kernel_kind() const { return (((nb == 4 && block == 16) || nb == 8) && reg_tiled_ok) ? 1 : 0; } // 1 = register-tiled kernel (ddh_kernel_reg4 / reg8)

        // outgoing-trace redirection of a distributed run (DdhDist): slots owned by another rank go to a packed send buffer
        struct Redirect
        {
            const int * bout = nullptr; // remapped table of the local subdomain range; entry <= -2: pair -2 - entry of `send`
            int64_t bout_off = 0;       // index of the first local entry in the full (n1*n1, n_domains) table
            float2 * send = nullptr;
        };
        void run(const double * x, double * y, const float * lambda, float * update, cudaStream_t s, int dom_begin = 0, int dom_end = -1,
                 const Redirect * redirect = nullptr);
    };

    // Slot maps of the assembled interface operator (DDHTransfer). T = DDH's trace map is block-sparse: subdomain p reads the
    // (lambda, mu) pairs of its own incoming slots and writes its own outgoing slots, so T is one dense 2F x 2F block per subdomain
    // (F = mx_fdof face DOFs) between a gather and a scatter. Face position f = 0..F-1 numbers the boundary ring of the n1 x n1
    // subdomain grid in ascending grid index Y*n1 + X, the same for every subdomain. Local input / output k < F is the lambda
    // entry of face position k, k >= F the mu entry of face position k - F. Host only.
    struct TransferSlots
    {
        int two_f = 0, n_domains = 0;
        int64_t n_lambda = 0;
        std::vector<int> face_at;    // (F) grid index of face position f
        std::vector<int> in, out;    // (2F, n_domains): slot of the vector that local input / output k of subdomain p reads / writes,
                                     // -1 = face DOF on the physical boundary (no slot)
        std::vector<int> orphans;    // ascending slots of [0, 2 n_lambda) that no subdomain writes
    };
    // builds the maps from hg_bin / hg_bout; throws unless every slot has at most one reader and at most one writer
    void transfer_slots(const DDH & D, TransferSlots & S);

    // Assembled DDH operator: y = x - T x with T stored as the probed per-subdomain blocks M_p (2F x 2F, FP32, column-major,
    // subdomain-contiguous). Creation probes T with 2F actions of the WaveHoltz kernel (input k set to 1 in every subdomain at
    // once), so every column is that kernel's own output; an action is one streaming batched matvec. `ddh` must outlive this.
    struct DDHTransfer
    {
        DDH * ddh;
        TransferSlots slots;
        DevBuf<float> d_M;
        DevBuf<int> d_in, d_out, d_orphans;
        int64_t probe_launches = 0;
        double probe_ms = 0.0;

        // max_bytes: device memory the handle may take (0 = what cudaMemGetInfo reports free); creation is synchronous on s
        DDHTransfer(DDH * ddh, int64_t max_bytes, cudaStream_t s);
        int64_t block_bytes() const { return (int64_t)slots.two_f * slots.two_f * slots.n_domains * (int64_t)sizeof(float); }
        int64_t bytes_per_action() const;   // blocks + maps + gathered inputs + written outputs + orphan copies
        void action(const float * x, float * y, cudaStream_t s); // y = x - T x; x and y must not overlap
        void get_block(int dom, float * h_out) const;            // host copy of M_dom (2F x 2F, column-major)
    };

    // contiguous block of subdomains of `rank` (subdomain ids are row-major over the subdomain grid -> row slabs)
    void subdomain_range(int n_domains, int rank, int world, int & begin, int & end);

    // Path B across GPUs (SURVEY §8e, north_star): subdomains are dealt to the ranks in contiguous row slabs; a lambda slot
    // lives on ONE rank - the rank of the subdomain that reads it (slots nobody reads: the writer's rank; untouched slots:
    // rank 0) - and Krylov vectors are distributed accordingly (global length, zero outside the owned slots). The action
    // kernel writes the traces that cross a slab boundary straight into a packed send buffer (fused pack in the kernel
    // epilogue); one grouped ncclSend/ncclRecv pair per neighbour moves them; a small unpack kernel drops them into the
    // owner's vector. Reader / writer of every slot come from the B table (source/DDH.cpp:425-440, cross-point overwrites
    // included).
    struct DdhDist
    {
        DDH * ddh;
        const Comm * comm; // may be null (tables only / single rank)
        int rank, world, dom_begin, dom_end;
        int64_t n_lambda;
        std::vector<int> owner;               // (n_lambda) owning rank of slot k (the lambda and mu entries share it)
        std::vector<int> send_idx, recv_idx;  // slots grouped by peer (ascending peer, ascending slot)
        std::vector<PeerSeg> segs;            // offsets / counts in (lambda, mu) pairs
        std::vector<unsigned char> mask;      // (2 n_lambda) 1 = owned
        int64_t n_owned = 0;
        // device
        DevBuf<int> d_bout, d_recv_idx;
        DevBuf<float2> d_send, d_recv;
        DevBuf<unsigned char> d_mask;
        bool on_device = false;

        DdhDist(DDH * ddh, const Comm * comm, int rank, int world);
        void ensure_device();
        int64_t bytes_per_action() const { return (int64_t)send_idx.size() * 8; }
        // t = T(x) on the owned slots (0 elsewhere); x holds valid values on the owned slots
        void apply_T(const float * x, float * t, cudaStream_t s);
        void action(const float * x, float * y, cudaStream_t s);      // y = x - T(x) on the owned slots, 0 elsewhere
        void rhs(const double * f, float * b, cudaStream_t s);        // b = T_f(0) on the owned slots
        void postprocess(const float * lambda, const double * f, double * u, cudaStream_t s); // u complete on every rank
    private:
        void exchange_and_finish(const float * x, float * t, int mode, cudaStream_t s);
    };
} // namespace cb200
