// Operator objects behind the C ABI (FP64 path A of SURVEY §8a): stiffness, mass, face mass, their
// diagonal inverses, face restrict/prolong/orth and the fused Helmholtz composite.
#pragma once
#include "common.hpp"
#include "dist.hpp"

namespace cb200
{
    struct SlabHalo;
    struct HelmholtzOp;

    // kernel family of a volume operator, chosen once at construction (select_volume_kernel in operators.cu)
    enum class VolumeKernel { Generic, LanePerRow, ThreadPerElement, ThreadPair };

    // y = (accumulate ? y : 0) + c * A x  for a patch-planned volume operator
    struct VolumeOp
    {
        H1Space * fem = nullptr;
        int nb = 0, nq = 0;
        bool stiff = false;
        std::vector<double> P, D;     // (nq, nb) column-major tables
        DevBuf<double> d_P, d_D;      // device copies (generic kernel)
        std::vector<double> wq;       // quadrature weights (stiffness; folded into the tables of the affine path)
        DevBuf<double> d_G;           // plan-ordered metric data: stiffness 3 comps, mass 1 comp
        DevBuf<double> d_Gc;          // affine stiffness: per patch (3, PE) element constants gA, gB, gC instead of d_G
        bool affine = false;          // stiffness on a mesh whose elements are all parallelograms: metric = w_i w_j * per-element constants
        DevBuf<double> d_partial;     // partial sums of patch-boundary DOFs
        VolumeKernel kind = VolumeKernel::Generic; // and the template instance that runs it (null: Generic)
        void (*launch)(const VolumeOp &, double c, int accumulate, const double * x, double * y, cudaStream_t s) = nullptr;
        Plan * plan = nullptr;        // the assembly plan this operator was laid out for (owned by fem)

        // phases: bit 0 = patch kernel, bit 1 = shared-DOF assembly pass (3 = the full action)
        void apply(double c, int accumulate, const double * x, double * y, cudaStream_t s, int phases = 3);
        size_t algorithmic_bytes() const; // SURVEY §8(d) per-element bytes * n_elem (the reference's stored-metric formulation)
        size_t moved_bytes() const;       // the same count for the formulation this handle actually runs (affine: 24 B of metric per element)
    };

    std::unique_ptr<VolumeOp> make_stiffness(H1Space * fem, int nq, int quad_type);
    std::unique_ptr<VolumeOp> make_mass(H1Space * fem, const double * d_coef /* device nodal coefficient or null */, int nq /* <=0: reference default */);

    struct DiagOp // y (+)= c * p .* x
    {
        int64_t n = 0;
        DevBuf<double> d_p;
        void apply(double c, int accumulate, const double * x, double * y, cudaStream_t s);
    };
    std::unique_ptr<DiagOp> make_diag_inv_mass(H1Space * fem, const double * d_coef);

    struct FaceMassOp
    {
        FaceSpace * fs = nullptr;
        int nb = 0, nq = 0;
        DevBuf<double> d_P, d_a; // P (nq,nb); a (nq, n_faces) = coef * w * measure
        // face-space vectors
        void apply(double c, int accumulate, const double * x, double * y, cudaStream_t s);
        // fused restrict + action + prolong on H1 vectors: y[proj] += c * H * x[proj]
        void apply_h1(double c, const double * x, double * y, cudaStream_t s);
        // both boundary terms of the Helmholtz composite on [u; v] (n DOFs each): y_u += c H x_v ; y_v += c H x_u
        void apply_h1_pair(double c, const double * x, double * y, int64_t n, cudaStream_t s, SlabHalo * halo = nullptr);
    };
    std::unique_ptr<FaceMassOp> make_facemass(FaceSpace * fs, const double * d_coef /* device face-space coefficient or null */, int nq);
    std::unique_ptr<DiagOp> make_diag_inv_facemass(FaceSpace * fs, const double * d_coef);

    void face_restrict(FaceSpace * fs, const double * x, double * y, cudaStream_t s);
    void face_prolong(FaceSpace * fs, const double * x, double * y, cudaStream_t s);
    void face_orth(FaceSpace * fs, double * x, cudaStream_t s);

    // upper bound on the CTAs of the persistent kernels (0 = one full wave of resident CTAs); test / tuning knob
    int max_persistent_ctas();
    void set_max_persistent_ctas(int n);

    // Path A across GPUs (SURVEY §8e): the mesh is cut into slabs of element rows, one per rank; a rank holds every DOF its
    // elements touch, so the node row on a slab interface is held by both neighbours and gets partial sums from both. After
    // the local apply the two interface rows of [u; v] are packed (fused into the face-mass launch), exchanged with the two
    // neighbours (one grouped ncclSend/ncclRecv) and added: own + received is the same commutative two-term sum on both
    // sides, so the mirrored rows stay bitwise identical and the result does not depend on the rank count.
    struct SlabHalo
    {
        const Comm * comm = nullptr;
        int rank = 0, world = 1, n_fields = 2;
        int64_t n_bottom = 0, n_top = 0, ndof = 0; // entries of the bottom / top interface row (one field); DOFs of one field
        std::vector<PeerSeg> segs;                 // offsets / counts in doubles
        DevBuf<int> d_row_dof;                     // (n_bottom + n_top) slab-local DOF of every row entry
        DevBuf<int> d_face_entry;                  // per face-space DOF of the physical boundary: its row entry or -1
        DevBuf<int> d_plain;                       // row entries that are not physical-boundary face DOFs (packed by copy)
        DevBuf<double> d_send, d_recv;             // [bottom: field 0 entries, field 1 entries | top: field 0, field 1]
        int64_t n_plain = 0;
        // peer path (default when every rank can map its neighbours' buffers with CUDA IPC; CUDDH_B200_PEER=0 or a failed mapping
        // anywhere -> ncclSend / ncclRecv): the packing launch stores the rows straight into the neighbours' receive buffers over
        // NVLink and publishes an epoch in their flags, the add kernel acquires its own flags. Two parity buffers: a neighbour can be
        // at most one exchange ahead (its next pack needs this rank's rows of the current exchange).
        bool peer = false;
        unsigned long long epoch = 0;
        DevBuf<unsigned char> d_peer_block;       // own: [2 parities][n_fields * (n_bottom + n_top)] doubles, then 2 arrival flags
        DevBuf<unsigned> d_ticket;
        double * own_recv = nullptr;
        unsigned long long * own_flags = nullptr; // [0]: from the lower neighbour, [1]: from the upper neighbour
        int64_t own_tot = 0;
        void * peer_base[2] = {nullptr, nullptr};
        double * peer_recv[2] = {nullptr, nullptr};
        unsigned long long * peer_flag[2] = {nullptr, nullptr};
        int64_t peer_tot[2] = {0, 0}, peer_off[2] = {0, 0};
        void setup_peer();
        ~SlabHalo();
        HelmholtzOp * op = nullptr;         // bound operator (gmres callback), not owned
        DevBuf<unsigned char> d_mask;              // (n_fields * ndof) 1 = owned: the lower rank owns a mirrored row (built lazily)
        const unsigned char * mask();
        int64_t bytes_per_apply() const { return (int64_t)sizeof(double) * n_fields * (n_bottom + n_top); }
        // y <- y + neighbours' copies on the interface rows (stand-alone: makes a vector consistent / sums partial results)
        void exchange(double * y, cudaStream_t s);
        void unpack_add(double * y, cudaStream_t s);
    };
    struct FaceSpace;
    std::unique_ptr<SlabHalo> make_slab_halo(const Comm * comm, int rank, int world, int64_t ndof, FaceSpace * fs_phys, int64_t n_bottom,
                                             const int * h_bottom, int64_t n_top, const int * h_top);

    // examples/Helmholtz.hpp:28-56 composite on [u;v]
    struct HelmholtzOp
    {
        double omega = 0;
        H1Space * fem = nullptr;
        FaceSpace * fs = nullptr;
        std::unique_ptr<VolumeOp> S, M;
        std::unique_ptr<FaceMassOp> H;
        DevBuf<double> d_partial2;    // fused path: partial sums of patch-boundary DOFs for both fields
        // fused path: S - omega^2 M on u and v, one launch for both fields (n_basis <= 5) or one per field (6-9); null: one by one
        void (*fused)(const HelmholtzOp &, const double * x, double * y, cudaStream_t s) = nullptr;
        // phases (fused path only): bit 0 = the fused volume kernel, bit 1 = shared-DOF assembly + face terms
        void apply(const double * x, double * y, cudaStream_t s, int phases = 3);
        // the apply of one slab of a partitioned mesh: local apply, interface rows packed inside the face-mass launch,
        // neighbour exchange, add. 4 launches + one grouped send/recv (fused path).
        void apply_slab(const double * x, double * y, SlabHalo & halo, cudaStream_t s);
        size_t algorithmic_bytes() const;
        size_t moved_bytes() const;
    };
    std::unique_ptr<HelmholtzOp> make_helmholtz(double omega, const double * d_a2, const double * d_a, H1Space * fem, FaceSpace * fs);
} // namespace cb200
