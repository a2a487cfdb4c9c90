// ldu.cu -- contexts, lduAddressing / lduMatrix handles and the caller-order matrix
// operations of the C ABI (include/b200ldu.h).
#include <stdarg.h>

#include <cstdlib>

#include "comm.h"
#include "ldu.h"
#include "ops.cuh"

// ---------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------
static thread_local char g_err[1024] = "";

void b200_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *b200ldu_last_error(void) { return g_err; }

extern "C" void b200ldu_controls_default(b200ldu_controls *c)
{
    memset(c, 0, sizeof(*c));
    c->tolerance = 1e-6; // LDU/lduMatrix/lduMatrixSolver.C:167-173
    c->relTol = 0;
    c->maxIter = 1000;
    c->minIter = 0;
    c->nSweeps = 1;  // smoothSolver.C:80
    c->omega = 0.9;  // JacobiSmoother.C:34
    c->nCellsInCoarsestLevel = 10; // GAMGSolver.C:67-77
    c->mergeLevels = 1;
    c->nPreSweeps = 0;
    c->preSweepsLevelMultiplier = 1;
    c->maxPreSweeps = 4;
    c->nPostSweeps = 2;
    c->postSweepsLevelMultiplier = 1;
    c->maxPostSweeps = 4;
    c->nFinestSweeps = 2;
    c->interpolateCorrection = 0;
    c->scaleCorrection = -1;
    c->directSolveCoarsest = 1;
    c->checkEvery = 0;
}

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
extern "C" int b200ldu_ctx_create(int device, b200ldu_ctx **out)
{
    if (!out) return B200LDU_EINVAL;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        b200_set_error("no CUDA device available (%s); this library has no CPU fallback",
                       e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        return B200LDU_ECUDA;
    }
    if (device < 0 || device >= n) {
        b200_set_error("ctx_create: device %d out of range [0,%d)", device, n);
        return B200LDU_EINVAL;
    }
    CUDA_TRY(cudaSetDevice(device));
    AbiHandle<b200ldu_ctx, b200ldu_ctx_destroy> c(new b200ldu_ctx());
    c->device = device;
    cudaDeviceProp p;
    CUDA_TRY(cudaGetDeviceProperties(&p, device));
    c->smCount = p.multiProcessorCount;
    CUDA_TRY(cudaStreamCreateWithFlags(&c->ownStream, cudaStreamNonBlocking));
    c->stream = c->ownStream;
    TRY(c->pinned.alloc(1 << 16));
    *out = c.release();
    return B200LDU_OK;
}

extern "C" int b200ldu_ctx_destroy(b200ldu_ctx *c)
{
    if (!c) return B200LDU_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    comm_destroy(c);
    if (c->ownStream) cudaStreamDestroy(c->ownStream);
    delete c;
    return B200LDU_OK;
}

extern "C" int b200ldu_ctx_set_stream(b200ldu_ctx *c, void *s)
{
    if (!c) return B200LDU_EINVAL;
    c->stream = (cudaStream_t)s;
    return B200LDU_OK;
}

extern "C" int b200ldu_ctx_sync(b200ldu_ctx *c)
{
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return B200LDU_OK;
}

extern "C" long long b200ldu_launch_count(const b200ldu_ctx *c) { return c ? c->launches : 0; }

// ---------------------------------------------------------------------------
// addressing
// ---------------------------------------------------------------------------
extern "C" int b200ldu_addr_create(b200ldu_ctx *ctx, int nCells, int nFaces, const int *lower_h,
                                   const int *upper_h, int nPatches, const int *patchStart_h,
                                   const int *faceCells_h, const int *neighbRank_h,
                                   const double *cellCentres_h, b200ldu_addr **out)
{
    if (!ctx || !out || nCells <= 0 || nFaces < 0 || (nFaces && (!lower_h || !upper_h)) ||
        nPatches < 0 || (nPatches && (!patchStart_h || !faceCells_h || !neighbRank_h))) {
        b200_set_error("addr_create: bad arguments");
        return B200LDU_EINVAL;
    }
    CUDA_TRY(cudaSetDevice(ctx->device));
    AbiHandle<b200ldu_addr, b200ldu_addr_destroy> a(new b200ldu_addr());
    a->ctx = ctx;
    a->nCells = nCells;
    a->nFaces = nFaces;
    a->l.assign(lower_h, lower_h + nFaces);
    a->u.assign(upper_h, upper_h + nFaces);
    a->nPatches = nPatches;
    if (nPatches) {
        a->patchStart.assign(patchStart_h, patchStart_h + nPatches + 1);
        a->faceCells.assign(faceCells_h, faceCells_h + a->patchStart[nPatches]);
        a->neighbRank.assign(neighbRank_h, neighbRank_h + nPatches);
        for (int i = 0; i < a->patchStart[nPatches]; i++)
            if (a->faceCells[i] < 0 || a->faceCells[i] >= nCells) {
                b200_set_error("addr_create: patch faceCells out of range");
                return B200LDU_EINVAL;
            }
    }
    if (cellCentres_h) a->centres_h.assign(cellCentres_h, cellCentres_h + 3 * (size_t)nCells);
    TRY(layout_build(a.get(), cellCentres_h));
    TRY(comm_addr_setup(a.get()));
    // cyclic patches: neighbRank[p] = -(q+1) pairs patch p with patch q of this addressing, face i
    // with face i (cyclicLduInterface: neighbPatchID).  Their "received" values are psi at the
    // partner's face cells, copied on the device (comm_halo_exchange).
    {
        bool any = false;
        for (int p = 0; p < nPatches; p++) any = any || a->neighbRank[p] < 0;
        if (any) {
            std::vector<int> src((size_t)a->patchStart[nPatches], -1);
            for (int p = 0; p < nPatches; p++) {
                if (a->neighbRank[p] >= 0) continue;
                const int q = -a->neighbRank[p] - 1;
                const int n = a->patchStart[p + 1] - a->patchStart[p];
                if (q < 0 || q >= nPatches || q == p || a->neighbRank[q] != -(p + 1) ||
                    a->patchStart[q + 1] - a->patchStart[q] != n) {
                    b200_set_error("addr_create: cyclic patch %d has no matching partner patch", p);
                    return B200LDU_EINVAL;
                }
                for (int i = 0; i < n; i++)
                    src[(size_t)a->patchStart[p] + i] = a->perm_h[a->faceCells[(size_t)a->patchStart[q] + i]];
            }
            TRY(a->d_cyclicSrc.upload(src));
        }
    }
    *out = a.release();
    return B200LDU_OK;
}

extern "C" int b200ldu_addr_destroy(b200ldu_addr *a)
{
    if (!a) return B200LDU_OK;
    cudaSetDevice(a->ctx->device);
    cudaStreamSynchronize(a->ctx->stream);
    delete a;
    return B200LDU_OK;
}

extern "C" int b200ldu_addr_info(const b200ldu_addr *a, long long *nPadRows, long long *nEntries,
                                 long long *nHalo, int *bandRows, int *nBands)
{
    if (!a) return B200LDU_EINVAL;
    if (nPadRows) *nPadRows = a->L.nPad;
    if (nEntries) *nEntries = a->nEntries;
    if (nHalo) *nHalo = a->nHaloTotal;
    if (bandRows) *bandRows = a->L.bandRows;
    if (nBands) *nBands = a->L.nBands;
    return B200LDU_OK;
}

extern "C" int b200ldu_addr_perm(const b200ldu_addr *a, int *perm_h)
{
    if (!a || !perm_h) return B200LDU_EINVAL;
    memcpy(perm_h, a->perm_h.data(), sizeof(int) * (size_t)a->nCells);
    return B200LDU_OK;
}

extern "C" long long b200ldu_vec_len(const b200ldu_addr *a) { return a ? a->vecLen : 0; }

int addr_alloc_vec(b200ldu_addr *a, DevBuf<double> &v)
{
    TRY(v.alloc((size_t)a->vecLen));
    CUDA_TRY(cudaMemsetAsync(v.get(), 0, sizeof(double) * (size_t)a->vecLen, a->ctx->stream));
    return B200LDU_OK;
}

double *addr_reuse_vec(b200ldu_addr *a, DevBuf<double> &v)
{
    if (!v.get() && addr_alloc_vec(a, v) != B200LDU_OK) return nullptr;
    return v.get();
}

static double *addr_pool_vec(b200ldu_addr *a, PoolSlot slot) { return addr_reuse_vec(a, a->pool[slot]); }

// ---- caller order <-> banded order ----
__global__ void to_banded_kernel(int nPad, const int *__restrict__ iperm, const double *__restrict__ x,
                                 double *__restrict__ xb)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < nPad) {
        int c = iperm[r];
        xb[r] = c >= 0 ? x[c] : 0.0;
    }
}

__global__ void from_banded_kernel(int nCells, const int *__restrict__ iperm,
                                   const double *__restrict__ xb, double *__restrict__ x)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < nCells) x[iperm[r]] = xb[r];
}

int to_banded(b200ldu_addr *a, const double *x, double *xb)
{
    to_banded_kernel<<<(a->L.nPad + 255) / 256, 256, 0, a->ctx->stream>>>(a->L.nPad, a->d_iperm.get(), x, xb);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

int from_banded(b200ldu_addr *a, const double *xb, double *x)
{
    // rows [0, nCells) are the real rows (padding sits at the end)
    from_banded_kernel<<<(a->nCells + 255) / 256, 256, 0, a->ctx->stream>>>(a->nCells, a->d_iperm.get(), xb, x);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_to_banded(b200ldu_addr *a, const double *x_d, double *xb_d)
{
    if (!a || !x_d || !xb_d) return B200LDU_EINVAL;
    return to_banded(a, x_d, xb_d);
}

extern "C" int b200ldu_from_banded(b200ldu_addr *a, const double *xb_d, double *x_d)
{
    if (!a || !x_d || !xb_d) return B200LDU_EINVAL;
    return from_banded(a, xb_d, x_d);
}

// ---------------------------------------------------------------------------
// matrix
// ---------------------------------------------------------------------------
extern "C" int b200ldu_matrix_create(b200ldu_addr *a, b200ldu_matrix **out)
{
    if (!a || !out) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    AbiHandle<b200ldu_matrix, b200ldu_matrix_destroy> m(new b200ldu_matrix());
    m->a = a;
    // coefficient streams are allocated by matrix_set (which layout is used depends on symmetry)
    TRY(m->d_diag.alloc((size_t)a->vecLen));
    TRY(m->d_rD.alloc((size_t)a->vecLen));
    int np = a->L.nBands > a->ctx->smCount * 8 ? a->L.nBands : a->ctx->smCount * 8;
    TRY(m->d_partials.alloc(4 * (size_t)np));
    TRY(m->d_scal.alloc(1));
    CUDA_TRY(cudaMemset(m->d_scal.get(), 0, sizeof(SolverScalars)));
    TRY(m->d_sendBuf.alloc((size_t)(a->L.nRecv > 0 ? a->L.nRecv : 1)));
    *out = m.release();
    return B200LDU_OK;
}

extern "C" int b200ldu_matrix_destroy(b200ldu_matrix *m)
{
    if (!m) return B200LDU_OK;
    cudaSetDevice(m->a->ctx->device);
    cudaStreamSynchronize(m->a->ctx->stream);
    delete m;
    return B200LDU_OK;
}

// code: 2f+side (side 0: owner-side entry, row = owner; side 1: neighbour-side entry),
// -1 padding, -2-pf coupled-patch face.  A uses upper on the owner side and lower on the
// neighbour side (lduMatrixATmul.C:90-136); the transpose swaps them (:298-329) and
// takes interfaceIntCoeffs instead of interfaceBouCoeffs (PBiCG.C:96).  Interface
// entries carry -coeff: result[cell] -= coeff*psiNbr (lduAddressingFunctors.H:252-261).
__global__ void fill_val_kernel(long long n, const int *__restrict__ code,
                                const double *__restrict__ upper, const double *__restrict__ lower,
                                const double *__restrict__ ifc, double *__restrict__ val, int transpose)
{
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    int c = code[e];
    double v;
    if (c >= 0) {
        int side = (c & 1) ^ transpose;
        v = side ? lower[c >> 1] : upper[c >> 1];
    } else if (c == -1) {
        v = 0.0;
    } else {
        v = -ifc[-2 - c];
    }
    val[e] = v;
}

__global__ void fill_diag_kernel(long long n, int nPad, const int *__restrict__ iperm,
                                 const double *__restrict__ diag, double *__restrict__ out,
                                 double *__restrict__ rD)
{
    long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double d = 1.0;
    if (r < nPad) {
        int c = iperm[r];
        if (c >= 0) d = diag[c];
    }
    out[r] = d;
    rD[r] = __ddiv_rn(1.0, d); // AINVPreconditioner.C:34-41, diagonalPreconditioner.C:60-66
}

// caller-order copy kept by the matrix (slot k of m->own), grown on demand
static int own_copy(b200ldu_matrix *m, int k, const double *src, size_t n, const double **out)
{
    *out = nullptr;
    if (!src || n == 0) return B200LDU_OK;
    TRY(m->own[k].grow(n));
    if (src != m->own[k].get())
        CUDA_TRY(cudaMemcpyAsync(m->own[k].get(), src, sizeof(double) * n, cudaMemcpyDeviceToDevice, m->a->ctx->stream));
    *out = m->own[k].get();
    return B200LDU_OK;
}

// banded diagonal + reciprocal from a caller-order diagonal (also used by fvm_solve, which folds the
// boundary coefficients into the diagonal for the duration of a solve: fvScalarMatrix.C:161-185)
int matrix_set_diag(b200ldu_matrix *m, const double *diag_d)
{
    b200ldu_addr *a = m->a;
    fill_diag_kernel<<<(unsigned)((a->vecLen + 255) / 256), 256, 0, a->ctx->stream>>>(a->vecLen, a->L.nPad, a->d_iperm.get(),
                                                                                      diag_d, m->d_diag.get(), m->d_rD.get());
    a->ctx->launches++;
    KERNEL_CHECK();
    m->diag_ext = diag_d;
    return B200LDU_OK;
}

extern "C" int b200ldu_matrix_set(b200ldu_matrix *m, const double *diag_d, const double *upper_d,
                                  const double *lower_d, const double *bou_d, const double *int_d)
{
    if (!m || !diag_d || (m->a->nFaces && !upper_d)) {
        b200_set_error("matrix_set: diag/upper required");
        return B200LDU_EINVAL;
    }
    b200ldu_addr *a = m->a;
    if (a->L.nRecv && (!bou_d || !int_d)) {
        b200_set_error("matrix_set: interface coefficients required for coupled patches");
        return B200LDU_EINVAL;
    }
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    cudaStream_t st = a->ctx->stream;
    m->symmetric = (lower_d == nullptr);
    const bool sameIfc = (bou_d == int_d);
    // The matrix keeps its own caller-order copies (the reference's lduMatrix owns diag/upper/lower,
    // lduMatrix.C:202-218): faceH, the fvMatrix glue and the GAMG coarse-level assembly read them
    // later, so the caller may free or overwrite its arrays as soon as this call returns.
    const double *dg, *up, *lw, *bo, *in;
    TRY(own_copy(m, 0, diag_d, (size_t)a->nCells, &dg));
    TRY(own_copy(m, 1, upper_d, (size_t)a->nFaces, &up));
    TRY(own_copy(m, 2, lower_d, (size_t)a->nFaces, &lw));
    TRY(own_copy(m, 3, bou_d, (size_t)a->L.nRecv, &bo));
    if (sameIfc)
        in = bo;
    else
        TRY(own_copy(m, 4, int_d, (size_t)a->L.nRecv, &in));
    const double *lo = lw ? lw : up;
    long long ne = a->nEntries;
    // Tmul needs its own coefficient stream when A != A^T (asymmetric coefficients or
    // interfaceIntCoeffs != interfaceBouCoeffs)
    bool needT = !m->symmetric || (a->L.nRecv && !sameIfc);
    size_t nb = (size_t)(ne > 0 ? ne : 1);
    if (!m->d_val.get()) TRY(m->d_val.alloc(nb));
    if (!needT)
        m->d_valT.reset(); // A^T == A
    else if (!m->d_valT.get())
        TRY(m->d_valT.alloc(nb));
    m->haveT = needT;
    if (ne > 0) {
        unsigned g = (unsigned)((ne + 255) / 256);
        fill_val_kernel<<<g, 256, 0, st>>>(ne, a->d_code.get(), up, lo, bo, m->d_val.get(), 0);
        a->ctx->launches++;
        if (needT) {
            fill_val_kernel<<<g, 256, 0, st>>>(ne, a->d_code.get(), up, lo, in, m->d_valT.get(), 1);
            a->ctx->launches++;
        }
    }
    KERNEL_CHECK();
    m->upper_ext = up;
    m->bou_ext = bo;
    m->int_ext = in;
    m->lower_ext = lo;
    return matrix_set_diag(m, dg);
}

// ---------------------------------------------------------------------------
// banded-order operations used by the solvers
// ---------------------------------------------------------------------------
int mat_halo(b200ldu_matrix *m, double *x, const int *stop, int *usedP2P)
{
    return comm_halo_exchange(m->a, x, m->d_sendBuf.get(), stop, usedP2P);
}

int mat_amul(b200ldu_matrix *m, bool transpose, double *x, double *out, int mode, const double *aux,
             double *partials, const int *stop)
{
    int wait = 0;
    TRY(mat_halo(m, x, stop, &wait));
#define LAUNCH_AMUL(MODE)                  \
    {                                      \
        AmulOp<MODE> op;                   \
        op.stop = stop;                    \
        op.waitHalo = wait;                \
        op.partials = partials;            \
        op.x = x;                          \
        op.diag = m->d_diag.get();         \
        op.aux = aux;                      \
        op.out = out;                      \
        return engine_launch_m(m, transpose, op); \
    }
    switch (mode) {
    case 0: LAUNCH_AMUL(0)
    case 1: LAUNCH_AMUL(1)
    case 2: LAUNCH_AMUL(2)
    case 3: LAUNCH_AMUL(3)
    case 4: LAUNCH_AMUL(4)
    }
#undef LAUNCH_AMUL
    return B200LDU_EINVAL;
}

int mat_ainv(b200ldu_matrix *m, bool transpose, const double *r, double *w, bool fuseDot,
             const double *dotv, double *partials, const int *stop)
{
    if (fuseDot) {
        AinvOp<1> op;
        op.stop = stop;
        op.partials = partials;
        op.r = r;
        op.rD = m->d_rD.get();
        op.dotv = dotv;
        op.out = w;
        return engine_launch_m(m, transpose, op);
    }
    AinvOp<0> op;
    op.stop = stop;
    op.partials = partials;
    op.r = r;
    op.rD = m->d_rD.get();
    op.dotv = nullptr;
    op.out = w;
    return engine_launch_m(m, transpose, op);
}

int mat_jacobi(b200ldu_matrix *m, double omega, double *x, const double *b, double *out, const int *stop)
{
    int wait = 0;
    TRY(mat_halo(m, x, stop, &wait));
    JacobiOp op;
    op.stop = stop;
    op.waitHalo = wait;
    op.x = x;
    op.diag = m->d_diag.get();
    op.b = b;
    op.out = out;
    op.omega = omega;
    op.nCells = m->a->nCells;
    return engine_launch_m(m, false, op);
}

int mat_residual(b200ldu_matrix *m, double *x, const double *b, double *out, bool fuseSumMag,
                 double *partials, const int *stop)
{
    int wait = 0;
    TRY(mat_halo(m, x, stop, &wait));
    if (fuseSumMag) {
        ResidualOp<1> op;
        op.stop = stop;
        op.waitHalo = wait;
        op.partials = partials;
        op.x = x;
        op.diag = m->d_diag.get();
        op.b = b;
        op.out = out;
        return engine_launch_m(m, false, op);
    }
    ResidualOp<0> op;
    op.stop = stop;
    op.waitHalo = wait;
    op.x = x;
    op.diag = m->d_diag.get();
    op.b = b;
    op.out = out;
    return engine_launch_m(m, false, op);
}

int mat_sumA(b200ldu_matrix *m, double *out, const int *stop)
{
    CoeffSumOp<false, false> op;
    op.stop = stop;
    op.diag = m->d_diag.get();
    op.out = out;
    return engine_launch_m(m, false, op);
}

int mat_H1(b200ldu_matrix *m, double *out)
{
    CoeffSumOp<true, true> op;
    op.diag = nullptr;
    op.out = out;
    return engine_launch_m(m, false, op);
}

int mat_H(b200ldu_matrix *m, const double *x, double *out)
{
    OffDiagOp<true, false> op;
    op.x = x;
    op.diag = m->d_diag.get();
    op.out = out;
    return engine_launch_m(m, false, op);
}

int mat_interpolate(b200ldu_matrix *m, double *x, double *out, const int *stop)
{
    int wait = 0;
    TRY(mat_halo(m, x, stop, &wait));
    OffDiagOp<false, true> op;
    op.stop = stop;
    op.waitHalo = wait;
    op.x = x;
    op.diag = m->d_diag.get();
    op.out = out;
    return engine_launch_m(m, false, op);
}

// ---------------------------------------------------------------------------
// caller-order entry points
// ---------------------------------------------------------------------------
#define CHECK_M(m)                               \
    if (!(m)) {                                  \
        b200_set_error("null matrix handle");    \
        return B200LDU_EINVAL;                   \
    }                                            \
    CUDA_TRY(cudaSetDevice((m)->a->ctx->device));

static int amul_ext(b200ldu_matrix *m, bool T, const double *psi, double *out)
{
    CHECK_M(m);
    if (!psi || !out) return B200LDU_EINVAL;
    b200ldu_addr *a = m->a;
    double *xb = addr_pool_vec(a, POOL_X), *yb = addr_pool_vec(a, POOL_Y);
    if (!xb || !yb) return B200LDU_ECUDA;
    TRY(to_banded(a, psi, xb));
    TRY(mat_amul(m, T, xb, yb, 0, nullptr, nullptr, nullptr));
    return from_banded(a, yb, out);
}

extern "C" int b200ldu_amul(b200ldu_matrix *m, const double *psi_d, double *Apsi_d)
{
    return amul_ext(m, false, psi_d, Apsi_d);
}

extern "C" int b200ldu_tmul(b200ldu_matrix *m, const double *psi_d, double *Tpsi_d)
{
    return amul_ext(m, true, psi_d, Tpsi_d);
}

extern "C" int b200ldu_amul_banded(b200ldu_matrix *m, const double *psib_d, double *Apsib_d)
{
    CHECK_M(m);
    return mat_amul(m, false, const_cast<double *>(psib_d), Apsib_d, 0, nullptr, nullptr, nullptr);
}

extern "C" int b200ldu_sumA(b200ldu_matrix *m, double *sumA_d)
{
    CHECK_M(m);
    double *yb = addr_pool_vec(m->a, POOL_Y);
    if (!yb) return B200LDU_ECUDA;
    TRY(mat_sumA(m, yb, nullptr));
    return from_banded(m->a, yb, sumA_d);
}

extern "C" int b200ldu_residual(b200ldu_matrix *m, const double *psi_d, const double *source_d,
                                double *rA_d)
{
    CHECK_M(m);
    b200ldu_addr *a = m->a;
    double *xb = addr_pool_vec(a, POOL_X), *yb = addr_pool_vec(a, POOL_Y), *bb = addr_pool_vec(a, POOL_B);
    if (!xb || !yb || !bb) return B200LDU_ECUDA;
    TRY(to_banded(a, psi_d, xb));
    TRY(to_banded(a, source_d, bb));
    TRY(mat_residual(m, xb, bb, yb, false, nullptr, nullptr));
    return from_banded(a, yb, rA_d);
}

extern "C" int b200ldu_H(b200ldu_matrix *m, const double *psi_d, double *Hpsi_d)
{
    CHECK_M(m);
    b200ldu_addr *a = m->a;
    double *xb = addr_pool_vec(a, POOL_X), *yb = addr_pool_vec(a, POOL_Y);
    if (!xb || !yb) return B200LDU_ECUDA;
    TRY(to_banded(a, psi_d, xb));
    TRY(mat_H(m, xb, yb));
    return from_banded(a, yb, Hpsi_d);
}

extern "C" int b200ldu_H1(b200ldu_matrix *m, double *H1_d)
{
    CHECK_M(m);
    double *yb = addr_pool_vec(m->a, POOL_Y);
    if (!yb) return B200LDU_ECUDA;
    TRY(mat_H1(m, yb));
    return from_banded(m->a, yb, H1_d);
}

// faceH: per internal face upper*psi[u] - lower*psi[l], caller order, face-parallel
// (lduMatrixTemplates.C:40-49,108-149)
__global__ void faceH_kernel(int nFaces, const int *__restrict__ l, const int *__restrict__ u,
                             const double *__restrict__ upper, const double *__restrict__ lower,
                             const double *__restrict__ psi, double *__restrict__ out)
{
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < nFaces) out[f] = __dsub_rn(__dmul_rn(upper[f], psi[u[f]]), __dmul_rn(lower[f], psi[l[f]]));
}

extern "C" int b200ldu_faceH(b200ldu_matrix *m, const double *psi_d, double *faceHpsi_d)
{
    CHECK_M(m);
    b200ldu_addr *a = m->a;
    if (!m->upper_ext) {
        b200_set_error("faceH: the matrix does not have any off-diagonal coefficients");
        return B200LDU_EINVAL;
    }
    if (a->nFaces == 0) return B200LDU_OK;
    faceH_kernel<<<(a->nFaces + 255) / 256, 256, 0, a->ctx->stream>>>(a->nFaces, a->d_l.get(), a->d_u.get(), m->upper_ext,
                                                                        m->lower_ext, psi_d, faceHpsi_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

int precond_kind(const char *name, char *printed)
{
    // lduMatrixPreconditioner.C:40-65: word or sub-dict; DIC/DILU silently become AINV (:58-61)
    if (!name || !*name || !strcmp(name, "none")) {
        strcpy(printed, "none");
        return 0;
    }
    if (!strcmp(name, "diagonal")) {
        strcpy(printed, "diagonal");
        return 1;
    }
    if (!strcmp(name, "AINV") || !strcmp(name, "DIC") || !strcmp(name, "DILU")) {
        strcpy(printed, "AINV");
        return 2;
    }
    b200_set_error("Unknown lduMatrix preconditioner %s; valid: (AINV DIC DILU diagonal none)", name);
    return -1;
}

int mat_precondition(b200ldu_matrix *m, int kind, bool transpose, const double *r, double *w, bool fuseDot,
                     const double *dotv, double *partials, int *nPartials, const int *stop)
{
    b200ldu_addr *a = m->a;
    if (kind == 2) {
        if (nPartials) *nPartials = a->L.nBands;
        return mat_ainv(m, transpose, r, w, fuseDot, dotv, partials, stop);
    }
    const double *rD = m->d_rD.get();
    const double *dv = dotv ? dotv : r;
    int n2 = a->L.nPad / 2;
    if (kind == 1) { // diagonalPreconditioner.C:76-89
        if (fuseDot)
            return ew_launch<1>(a->ctx, n2, stop, partials, nPartials, [=] __device__(int i, double *red) {
                double2 rr = reinterpret_cast<const double2 *>(r)[i];
                double2 dd = reinterpret_cast<const double2 *>(rD)[i];
                double2 d2 = reinterpret_cast<const double2 *>(dv)[i];
                double2 ww = make_double2(__dmul_rn(dd.x, rr.x), __dmul_rn(dd.y, rr.y));
                reinterpret_cast<double2 *>(w)[i] = ww;
                red[0] += ww.x * d2.x + ww.y * d2.y;
            });
        return ew_launch<0>(a->ctx, n2, stop, nullptr, nullptr, [=] __device__(int i, double *) {
            double2 rr = reinterpret_cast<const double2 *>(r)[i];
            double2 dd = reinterpret_cast<const double2 *>(rD)[i];
            reinterpret_cast<double2 *>(w)[i] = make_double2(__dmul_rn(dd.x, rr.x), __dmul_rn(dd.y, rr.y));
        });
    }
    // noPreconditioner.C:58-72
    if (fuseDot)
        return ew_launch<1>(a->ctx, n2, stop, partials, nPartials, [=] __device__(int i, double *red) {
            double2 rr = reinterpret_cast<const double2 *>(r)[i];
            double2 d2 = reinterpret_cast<const double2 *>(dv)[i];
            reinterpret_cast<double2 *>(w)[i] = rr;
            red[0] += rr.x * d2.x + rr.y * d2.y;
        });
    return ew_launch<0>(a->ctx, n2, stop, nullptr, nullptr, [=] __device__(int i, double *) {
        reinterpret_cast<double2 *>(w)[i] = reinterpret_cast<const double2 *>(r)[i];
    });
}

extern "C" int b200ldu_precondition(b200ldu_matrix *m, const char *name, int transpose, const double *rA_d,
                                    double *wA_d)
{
    CHECK_M(m);
    char printed[32];
    int k = precond_kind(name, printed);
    if (k < 0) return B200LDU_ENOPRECOND;
    b200ldu_addr *a = m->a;
    double *xb = addr_pool_vec(a, POOL_X), *yb = addr_pool_vec(a, POOL_Y);
    if (!xb || !yb) return B200LDU_ECUDA;
    TRY(to_banded(a, rA_d, xb));
    TRY(mat_precondition(m, k, transpose != 0, xb, yb, false, nullptr, nullptr, nullptr, nullptr));
    return from_banded(a, yb, wA_d);
}

int smoother_ok(const char *name)
{
    // GaussSeidel is an alias of the Jacobi smoother (GaussSeidelSmoother.C:43-69)
    if (!name || !*name || !strcmp(name, "Jacobi") || !strcmp(name, "GaussSeidel")) return 1;
    b200_set_error("Unknown lduMatrix smoother %s; valid: (GaussSeidel Jacobi)", name);
    return 0;
}

extern "C" int b200ldu_smooth(b200ldu_matrix *m, const char *name, double omega, double *psi_d,
                              const double *source_d, int nSweeps)
{
    CHECK_M(m);
    if (!smoother_ok(name)) return B200LDU_ENOPRECOND;
    b200ldu_addr *a = m->a;
    double *xb = addr_pool_vec(a, POOL_X), *yb = addr_pool_vec(a, POOL_Y), *bb = addr_pool_vec(a, POOL_B);
    if (!xb || !yb || !bb) return B200LDU_ECUDA;
    TRY(to_banded(a, psi_d, xb));
    TRY(to_banded(a, source_d, bb));
    double *cur = xb, *nxt = yb;
    for (int s = 0; s < nSweeps; s++) { // ping-pong instead of psi = Apsi copies (JacobiSmoother.C:146)
        TRY(mat_jacobi(m, omega, cur, bb, nxt, nullptr));
        double *t = cur;
        cur = nxt;
        nxt = t;
    }
    return from_banded(a, cur, psi_d);
}

// banded-order single-kernel entry for the kernel table of bench.py (--kernels): vectors are
// b200ldu_vec_len() doubles in banded order, exactly as the solvers hold them
extern "C" int b200ldu_bench_op(b200ldu_matrix *m, const char *op, double *xb, double *yb, const double *bb)
{
    CHECK_M(m);
    if (!op || !xb || !yb) return B200LDU_EINVAL;
    if (!strcmp(op, "amul")) return mat_amul(m, false, xb, yb, 0, nullptr, nullptr, nullptr);
    if (!strcmp(op, "tmul")) return mat_amul(m, true, xb, yb, 0, nullptr, nullptr, nullptr);
    if (!strcmp(op, "amul_dot")) return mat_amul(m, false, xb, yb, 1, nullptr, m->d_partials.get(), nullptr);
    if (!strcmp(op, "ainv")) return mat_ainv(m, false, xb, yb, false, nullptr, nullptr, nullptr);
    if (!strcmp(op, "ainv_dot")) return mat_ainv(m, false, xb, yb, true, nullptr, m->d_partials.get(), nullptr);
    if (!strcmp(op, "jacobi")) return bb ? mat_jacobi(m, 0.9, xb, bb, yb, nullptr) : B200LDU_EINVAL;
    if (!strcmp(op, "residual")) return bb ? mat_residual(m, xb, bb, yb, true, m->d_partials.get(), nullptr) : B200LDU_EINVAL;
    if (!strcmp(op, "sumA")) return mat_sumA(m, yb, nullptr);
    if (!strcmp(op, "H")) return mat_H(m, xb, yb);
    b200_set_error("bench_op: unknown op %s", op);
    return B200LDU_EINVAL;
}
