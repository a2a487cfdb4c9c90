// internal.h -- shared declarations of the b200ldu library (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <memory>
#include <string>
#include <vector>

#include "../../include/b200ldu.h"

// ---------------------------------------------------------------------------
// error handling: nothing throws across the ABI
// ---------------------------------------------------------------------------
void b200_set_error(const char *fmt, ...);

#define CUDA_TRY(expr)                                                                   \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            b200_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                 \
                           cudaGetErrorString(_e));                                      \
            return B200LDU_ECUDA;                                                        \
        }                                                                                \
    } while (0)

#define TRY(expr)                          \
    do {                                   \
        int _rc = (expr);                  \
        if (_rc != B200LDU_OK) return _rc; \
    } while (0)

#define KERNEL_CHECK() CUDA_TRY(cudaGetLastError())

// ---------------------------------------------------------------------------
// owning buffers: every device (and pinned host) allocation of the library is one of these
// ---------------------------------------------------------------------------
// Move-only; the destructor frees.  An empty buffer makes no CUDA call (the host-only layout path needs no
// GPU).  Never give one static storage duration: it would be freed after the CUDA runtime has shut down.
template <class T, bool Pinned = false>
class DevBuf {
  public:
    DevBuf() = default;
    DevBuf(DevBuf &&o) noexcept { std::swap(p_, o.p_), std::swap(n_, o.n_); }
    DevBuf &operator=(DevBuf &&o) noexcept
    {
        if (this != &o) {
            reset();
            std::swap(p_, o.p_), std::swap(n_, o.n_);
        }
        return *this;
    }
    ~DevBuf() { reset(); }
    T *get() const { return p_; }
    size_t size() const { return n_; }
    void reset()
    {
        if (p_) Pinned ? cudaFreeHost(p_) : cudaFree(p_);
        p_ = nullptr, n_ = 0;
    }
    // n elements, replacing what was held (contents undefined)
    int alloc(size_t n)
    {
        reset();
        const size_t bytes = sizeof(T) * n;
        cudaError_t e = Pinned ? cudaMallocHost((void **)&p_, bytes) : cudaMalloc((void **)&p_, bytes);
        if (e != cudaSuccess) {
            p_ = nullptr;
            b200_set_error("%s of %zu bytes -> %s", Pinned ? "cudaMallocHost" : "cudaMalloc", bytes, cudaGetErrorString(e));
            return B200LDU_ECUDA;
        }
        n_ = n;
        return B200LDU_OK;
    }
    // a copy of h; one element when h is empty
    int upload(const std::vector<T> &h)
    {
        TRY(alloc(h.size() ? h.size() : 1));
        if (h.size()) CUDA_TRY(cudaMemcpy(p_, h.data(), sizeof(T) * h.size(), cudaMemcpyHostToDevice));
        return B200LDU_OK;
    }
    // at least n elements: never shrinks, does not keep the contents when it reallocates
    int grow(size_t n) { return p_ && n_ >= n ? B200LDU_OK : alloc(n); }

  private:
    T *p_ = nullptr;
    size_t n_ = 0;
};
template <class T>
using PinnedBuf = DevBuf<T, true>;

// an owning handle that is released through its C ABI destroy function (device set, stream synchronised)
template <class H, int (*Destroy)(H *)>
struct AbiDestroy {
    void operator()(H *h) const { Destroy(h); }
};
template <class H, int (*Destroy)(H *)>
using AbiHandle = std::unique_ptr<H, AbiDestroy<H, Destroy>>;

// ---------------------------------------------------------------------------
// banded layout constants
// ---------------------------------------------------------------------------
// A "band" is BAND_ROWS consecutive rows of the renumbered matrix, processed by one
// CTA with the band's psi values staged in shared memory.  A "slice" is SLICE_ROWS
// consecutive rows handled by one warp, each lane owning two adjacent rows so that the
// coefficient stream is read with 128-bit loads (double2) and the 16-bit local column
// indices with 32-bit loads (ushort2).
constexpr int SLICE_ROWS = 64;
constexpr int ENGINE_THREADS = 256;

// workspace slots (fixed indices: a slot is allocated at its first use and kept)
enum PoolSlot { POOL_X, POOL_Y, POOL_B, POOL_SLOTS }; // b200ldu_addr::pool, the caller-order matrix operations
enum WorkSlot {                                        // b200ldu_matrix::work
    WORK_SOLVER_SLOTS = 8,                             // [0, 8): the vectors of the running solver (Solve::vec)
    WORK_HOST_PSI = 12, WORK_HOST_SRC,                 // b200ldu_solve_host: caller-order device copies
    WORK_PSI_B, WORK_SRC_B,                            // b200ldu_solve: banded psi and source
    WORK_SLOTS
};
enum FvmSlot {       // b200ldu_addr::fvmScratch, grown to the largest request
    FVM_DIAG,        // fvm_solve: boundary-folded diagonal; fvm_residual: boundary-folded source
    FVM_SOURCE,      // fvm_solve: boundary-folded source, all components
    FVM_CMPT_SOURCE, // fvm_solve: source of one component
    FVM_CMPT_PSI,    // fvm_solve: psi of one component; fv_patch_neighbour_field: the send buffer
    FVM_SLOTS
};

struct SolverScalars; // ops.cuh

struct b200ldu_ctx {
    int device = 0;
    cudaStream_t stream = 0;
    cudaStream_t ownStream = 0; // created by ctx_create, destroyed with the context
    int smCount = 148;
    long long launches = 0;
    // NCCL (comm.cu)
    void *nccl = nullptr; // ncclComm_t
    int rank = 0, nRanks = 1;
    // pinned staging for *_host entry points and scalar read-back
    PinnedBuf<char> pinned;
    // peer-memory (CUDA IPC over NVLink) collectives, see comm.cu
    bool p2p = false;
    DevBuf<char> region;             // this rank's shared region
    char *peerRegion[8] = {nullptr}; // every rank's region mapped here (own included)
    DevBuf<unsigned long long> d_seq; // local device counters: [0] reduction seq, [1] halo seq, [2..] scratch
};

// layout of the IPC-shared region of every rank
constexpr int P2P_MAXR = 8;
constexpr size_t P2P_MAIL_OFF = 0;        // double mail[2][P2P_MAXR][8]
constexpr size_t P2P_MAILFLAG_OFF = 2048; // u64 mailFlag[2][P2P_MAXR]
constexpr size_t P2P_HALOFLAG_OFF = 4096; // u64 haloFlag[P2P_MAXR]   (indexed by source rank)
constexpr int PACK_CHUNK = 4096; // faces per packing CTA of the fused halo send (comm.cu); layout.cu reserves their CTA slots
constexpr int P2P_GMAX = 256;             // doubles per rank in the coarsest-level gather
constexpr size_t P2P_GATHER_OFF = 8192;   // double gather[2][P2P_MAXR][P2P_GMAX]
constexpr size_t P2P_GFLAG_OFF = 8192 + 2 * P2P_MAXR * P2P_GMAX * sizeof(double); // u64 gflag[2][P2P_MAXR]
constexpr size_t P2P_RECV_OFF = 49152;    // double recv[2][P2P_RECV_CAP]
constexpr size_t P2P_RECV_CAP = 1u << 20; // doubles per parity
constexpr size_t P2P_REGION_BYTES = P2P_RECV_OFF + 2 * P2P_RECV_CAP * sizeof(double);
static_assert(P2P_GFLAG_OFF + 2 * P2P_MAXR * sizeof(unsigned long long) <= P2P_RECV_OFF, "gather area overlaps the receive buffers");

struct P2PRed { // passed by value to scalar_kernel
    int rank = 0, nRanks = 1;
    double *mail[P2P_MAXR] = {nullptr};
    unsigned long long *flag[P2P_MAXR] = {nullptr};
    unsigned long long *seq = nullptr;
};

// peer-memory halo send descriptors (comm.cu builds them, engine.cuh executes them)
struct PackPatch {
    double *dst[2];            // neighbour's receive buffer (parity 0/1) + this patch's offset there
    unsigned long long *flag;  // neighbour's arrival flag for this rank
    int start, n, nChunks;
};
struct PackChunk {
    int patch, begin, end;
};

// device view of the banded addressing, passed by value to kernels
struct LayoutDev {
    int nCells;         // real rows
    int nPad;           // rows incl. padding (multiple of bandRows)
    int nBands;
    int bandRows;       // rows per band (multiple of SLICE_ROWS)
    int slicesPerBand;
    int nRecv;          // halo tail length (values received from coupled patches)
    int maxHalo;        // max halo columns of any band (smem sizing)
    const long long *sliceStart; // [nSlices+1] entry offset of each slice (multiple of 64)
    const uint16_t *sliceW;      // slots per row in the slice, all entries
    const uint16_t *sliceWL;     // slots holding owner/neighbour entries only (no interfaces)
    const uint16_t *col;         // [nEntries] band-local column: < bandRows own band, else halo slot
    const int *haloStart;        // [nBands+1]
    const int *haloIdx;          // banded extended index: < nPad local row, else nPad + recv slot
    const int *perm;             // [nCells] caller cell -> banded row
    const int *iperm;            // [nPad]  banded row -> caller cell, -1 padding
    // peer-memory halo (null/0 when the exchange goes through NCCL into the vector's own tail)
    const unsigned long long *haloFlags; // this rank's arrival flags, indexed by source rank
    const unsigned long long *haloSeq;   // device counter of completed exchanges
    const double *tail0, *tail1;         // receive buffers by exchange parity
    int nNbr;
    int nbr[8];
    const PackChunk *packChunks;   // fused halo send: first nPackChunks CTAs of a consuming kernel
    const PackPatch *packPatches;
    const int *sendRows;           // banded row of every coupled-patch face cell
    unsigned long long *seqs;      // device counters: [1] halo sequence, [6] CTAs done, [8+p] chunks done
    int nPackChunks;
};

struct b200ldu_addr {
    b200ldu_ctx *ctx = nullptr;
    int nCells = 0, nFaces = 0;
    std::vector<int> l, u; // host copies (GAMG agglomeration, FV CSR build)
    int nPatches = 0;
    std::vector<int> patchStart, faceCells, neighbRank;
    // layout (host mirrors kept only where later setup steps need them)
    LayoutDev L{};
    long long nEntries = 0;
    long long nHaloTotal = 0;
    std::vector<int> perm_h, iperm_h;
    std::vector<double> centres_h; // optional cell centres (kept for GAMG coarse-level banding)
    // device arrays owned
    DevBuf<long long> d_sliceStart;
    DevBuf<uint16_t> d_sliceW, d_sliceWL, d_col;
    DevBuf<int> d_code; // [nEntries] value source: 2f+side | -1 pad | -2-pf interface
    DevBuf<int> d_haloStart, d_haloIdx, d_perm, d_iperm;
    DevBuf<int> d_sendRows; // [nRecv] banded row of faceCells (pack kernel)
    bool p2pHalo = false;   // peer-store halo usable for this addressing
    DevBuf<PackPatch> d_packPatches; // peer-memory halo send descriptors (comm.cu)
    DevBuf<PackChunk> d_packChunks;
    int nPackChunks = 0;
    double nCellsGlobal = 0;
    // caller-order CSR views for the FV face-sum kernels and faceH
    DevBuf<int> d_cyclicSrc; // per coupled-patch face: banded row supplying it (cyclic partner) | -1
    DevBuf<int> d_l, d_u, d_ownerStart, d_losort, d_losortStart;
    int nBFaces = 0;
    DevBuf<int> d_bFaceCells;              // boundary faces (all patches, patch order)
    DevBuf<int> d_bCellStart, d_bCellFaces; // per boundary cell lists
    // fvMatrix glue (fvmatrix.cu): per-cell lists over the coupled patch faces, built at first use, and
    // grow-only scratch vectors
    int nCFaces = 0;
    DevBuf<int> d_cCellStart, d_cCellFaces, d_cFaceCells;
    DevBuf<double> mulesScratch; // MULES limiter: six cell fields + the received limiters (mules.cu)
    DevBuf<double> fvmScratch[FVM_SLOTS];
    // host-only structural self-check (b200ldu_layout_debug_*): no GPU, no compute
    bool hostOnly = false;
    std::vector<long long> dbg_sliceStart;
    std::vector<uint16_t> dbg_sliceW, dbg_sliceWL, dbg_col;
    std::vector<int> dbg_code, dbg_haloStart, dbg_haloIdx;
    // workspace pool for caller-order entry points (banded vectors)
    DevBuf<double> pool[POOL_SLOTS];
    long long vecLen = 0; // nPad + nRecv (padded to even)
};

struct b200ldu_matrix {
    b200ldu_addr *a = nullptr;
    bool symmetric = true;
    bool haveT = false;
    DevBuf<double> d_val;  // banded coefficients for Amul   [nEntries]
    DevBuf<double> d_valT; // banded coefficients for Tmul   (only when haveT: A != A^T)
    DevBuf<double> d_diag; // banded diagonal [nPad] (padding rows = 1)
    DevBuf<double> d_rD;   // 1/diag, filled by matrix_set
    const double *valT() const { return haveT ? d_valT.get() : d_val.get(); }
    // caller-order coefficients OWNED by the matrix (copied by matrix_set): diag, upper, lower, interfaceBouCoeffs,
    // interfaceIntCoeffs -- read by faceH, the fvMatrix glue and the GAMG coarse-level assembly
    DevBuf<double> own[5];
    // current views of them (diag_ext is re-pointed at the boundary-folded diagonal for the duration of fvm_solve;
    // lower_ext aliases upper_ext when symmetric, int_ext aliases bou_ext when the caller passed one array for both)
    const double *upper_ext = nullptr, *lower_ext = nullptr, *diag_ext = nullptr, *bou_ext = nullptr,
                 *int_ext = nullptr;
    // solver workspace (allocated once, reused across solves -- PCGCache.H:9-58)
    DevBuf<double> work[WORK_SLOTS];
    DevBuf<double> d_partials;       // reduction partials
    DevBuf<SolverScalars> d_scal;
    DevBuf<double> d_hist;           // device residual history
    DevBuf<double> d_sendBuf;        // packed psi at coupled-patch face cells
};

// ---------------------------------------------------------------------------
// cross-file helpers
// ---------------------------------------------------------------------------
int layout_build(b200ldu_addr *a, const double *centres);
int addr_alloc_vec(b200ldu_addr *a, DevBuf<double> &v); // banded vector of vecLen doubles, zeroed
double *addr_reuse_vec(b200ldu_addr *a, DevBuf<double> &v); // the same, allocated at first use; null on failure
