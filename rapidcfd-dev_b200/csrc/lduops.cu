// lduops.cu -- lduMatrix algebra on caller-order coefficient arrays: the row sums sumDiag / negSumDiag /
// sumMagOffDiag (LDU/lduMatrix/lduMatrixOperations.C:36-104) and operator+= / -= / *= (:235-465), which
// fvMatrix uses to combine the matrices of an equation's terms (fvm::ddt + fvm::div - fvm::laplacian,
// fvMatrix.C:1750-1815).  A matrix is (diag[nCells], upper[nFaces], lower[nFaces]) with a presence flag per
// array, as the reference's lduMatrix holds optional arrays: symmetric = diag and upper only, asymmetric = all
// three, diagonal = diag only (lduMatrix.H:626-639).
#include "internal.h"

namespace {

__global__ void row_sum_kernel(int nCells, int mode, const int *__restrict__ ownerStart, const int *__restrict__ losortStart,
                               const int *__restrict__ losort, const double *__restrict__ upper,
                               const double *__restrict__ lower, double *__restrict__ io)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nCells) return;
    double acc = io[c];
    // a row receives lower[f] from the faces it owns and upper[f] from the faces where it is neighbour
    // (sumMagOffDiag: |upper| / |lower| the other way round, lduMatrixOperations.C:83-104); owner faces first
    for (int f = ownerStart[c]; f < ownerStart[c + 1]; f++) {
        const double v = mode == 2 ? fabs(upper[f]) : lower[f];
        acc = mode == 1 ? __dsub_rn(acc, v) : __dadd_rn(acc, v);
    }
    for (int k = losortStart[c]; k < losortStart[c + 1]; k++) {
        const int f = losort[k];
        const double v = mode == 2 ? fabs(lower[f]) : upper[f];
        acc = mode == 1 ? __dsub_rn(acc, v) : __dadd_rn(acc, v);
    }
    io[c] = acc;
}

// y = y (+|-) x ; or y = (+|-) x when assign
__global__ void axpy_kernel(long long n, int sub, int assign, const double *__restrict__ x, double *__restrict__ y)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = x[i];
    if (assign)
        y[i] = sub ? -v : v;
    else
        y[i] = sub ? __dsub_rn(y[i], v) : __dadd_rn(y[i], v);
}

// y[i] *= s[idx ? idx[i] : i]   (idx: face -> cell), or y[i] *= scalar
__global__ void scale_kernel(long long n, const int *__restrict__ idx, const double *__restrict__ s, double scalar,
                             double *__restrict__ y)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    y[i] = __dmul_rn(y[i], s ? s[idx ? idx[i] : i] : scalar);
}

int axpy(b200ldu_ctx *ctx, long long n, int sub, int assign, const double *x, double *y)
{
    if (n <= 0) return B200LDU_OK;
    axpy_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, sub, assign, x, y);
    ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

} // namespace

// mode 0: sumDiag (diag += ...), 1: negSumDiag (diag -= ...), 2: sumMagOffDiag (sumOff += |...|); lower_d NULL = symmetric
extern "C" int b200ldu_ldu_row_sum(b200ldu_addr *a, int mode, const double *upper_d, const double *lower_d, double *inout_d)
{
    if (!a || !inout_d || mode < 0 || mode > 2 || (a->nFaces && !upper_d)) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    row_sum_kernel<<<(a->nCells + 127) / 128, 128, 0, a->ctx->stream>>>(a->nCells, mode, a->d_ownerStart.get(), a->d_losortStart.get(),
                                                                        a->d_losort.get(), upper_d, lower_d ? lower_d : upper_d, inout_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

// A (+|-)= B with the reference's rules for the kinds of the two matrices (lduMatrixOperations.C:235-397).
// hasA[3] / hasB[3]: which of {diag, upper, lower} each matrix holds; hasA is updated (a symmetric A becomes
// asymmetric when B is: its lower starts as a copy of its upper, lduMatrix.C:238-254).  The three A pointers
// must be valid storage whenever the result can hold that array.
extern "C" int b200ldu_ldu_add_assign(b200ldu_addr *a, int subtract, double *diagA_d, double *upperA_d, double *lowerA_d, int *hasA,
                                      const double *diagB_d, const double *upperB_d, const double *lowerB_d, const int *hasB)
{
    if (!a || !hasA || !hasB) return B200LDU_EINVAL;
    b200ldu_ctx *ctx = a->ctx;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const long long n = a->nCells, nF = a->nFaces;
    const size_t fb = sizeof(double) * (size_t)nF;
    if (hasB[0]) { // diag() (+|-)= A.diag(): the non-const accessor allocates a zero diagonal (lduMatrix.C:272-283)
        if (!diagA_d || !diagB_d) return B200LDU_EINVAL;
        if (!hasA[0]) CUDA_TRY(cudaMemsetAsync(diagA_d, 0, sizeof(double) * (size_t)n, ctx->stream));
        hasA[0] = 1;
        TRY(axpy(ctx, n, subtract, 0, diagB_d, diagA_d));
    }
    const bool symA = hasA[0] && hasA[1] && !hasA[2], asymA = hasA[0] && hasA[1] && hasA[2], diagonalA = hasA[0] && !hasA[1] && !hasA[2];
    const bool symB = hasB[0] && hasB[1] && !hasB[2], asymB = hasB[0] && hasB[1] && hasB[2];
    if ((hasA[1] && !upperA_d) || (hasA[2] && !lowerA_d) || (hasB[1] && !upperB_d) || (hasB[2] && !lowerB_d)) return B200LDU_EINVAL;
    if (symA && symB) {
        TRY(axpy(ctx, nF, subtract, 0, upperB_d, upperA_d));
    } else if (symA && asymB) {
        if (!lowerA_d) return B200LDU_EINVAL;
        CUDA_TRY(cudaMemcpyAsync(lowerA_d, upperA_d, fb, cudaMemcpyDeviceToDevice, ctx->stream)); // lower(): copy of upper
        hasA[2] = 1;
        TRY(axpy(ctx, nF, subtract, 0, upperB_d, upperA_d));
        TRY(axpy(ctx, nF, subtract, 0, lowerB_d, lowerA_d));
    } else if (asymA && symB) {
        TRY(axpy(ctx, nF, subtract, 0, upperB_d, lowerA_d));
        TRY(axpy(ctx, nF, subtract, 0, upperB_d, upperA_d));
    } else if (asymA && asymB) {
        TRY(axpy(ctx, nF, subtract, 0, lowerB_d, lowerA_d));
        TRY(axpy(ctx, nF, subtract, 0, upperB_d, upperA_d));
    } else if (diagonalA) { // takes B's triangles (negated for -=)
        if (hasB[1]) {
            if (!upperA_d) return B200LDU_EINVAL;
            TRY(axpy(ctx, nF, subtract, 1, upperB_d, upperA_d));
            hasA[1] = 1;
        }
        if (hasB[2]) {
            if (!lowerA_d) return B200LDU_EINVAL;
            TRY(axpy(ctx, nF, subtract, 1, lowerB_d, lowerA_d));
            hasA[2] = 1;
        }
    } // B diagonal, or an unknown combination: nothing more (the reference warns at debug > 1)
    return B200LDU_OK;
}

// A *= sf (a cell field: diag by the cell, upper by the owner's value, lower by the neighbour's, :400-441) or A *= s (:444-462)
extern "C" int b200ldu_ldu_scale(b200ldu_addr *a, const double *sf_d, double s, double *diagA_d, double *upperA_d, double *lowerA_d,
                                 const int *hasA)
{
    if (!a || !hasA) return B200LDU_EINVAL;
    b200ldu_ctx *ctx = a->ctx;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const long long n = a->nCells, nF = a->nFaces;
    if (hasA[0] && diagA_d && n) scale_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, nullptr, sf_d, s, diagA_d);
    if (hasA[1] && upperA_d && nF) scale_kernel<<<(unsigned)((nF + 255) / 256), 256, 0, ctx->stream>>>(nF, a->d_l.get(), sf_d, s, upperA_d);
    if (hasA[2] && lowerA_d && nF) scale_kernel<<<(unsigned)((nF + 255) / 256), 256, 0, ctx->stream>>>(nF, a->d_u.get(), sf_d, s, lowerA_d);
    ctx->launches += 3;
    KERNEL_CHECK();
    return B200LDU_OK;
}
