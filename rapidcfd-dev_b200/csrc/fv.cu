// fv.cu -- finite-volume face-sum loops that assemble the fvMatrix (caller-order fields).
//
// Reference (FV/ = src/finiteVolume/): fvc::surfaceIntegrate / surfaceSum
// FV/finiteVolume/fvc/fvcSurfaceIntegrate.C:41-97,138-203,264-360; gaussGrad::gradf
// FV/finiteVolume/gradSchemes/gaussGrad/gaussGrad.C:34-139,143-242; Laplacian fill
// gaussLaplacianScheme.C:63-64; convection fill gaussConvectionScheme.C:95-97; linear
// interpolation surfaceInterpolationScheme.C:272-351; addBoundaryDiag/Source
// FV/fvMatrices/fvMatrix/fvMatrix.C:209-226,290-312.
//
// One thread per cell walks the cell's owner faces (contiguous) and neighbour faces
// (losort); the boundary-face contributions and the division by the cell volume are
// fused into the same kernel through a per-cell boundary-face list, so each output is
// written once (the reference runs one kernel per patch plus a separate divide).
// Summation order = owner faces, neighbour faces, boundary faces (ascending), then /V,
// products rounded separately -- bit-comparable with oracle/ldu_oracle_fv.c.
#include <algorithm>

#include "internal.h"

#include "fv_kernels.cuh"

using namespace fvk;

extern "C" int b200ldu_fv_boundary_set(b200ldu_addr *a, int nBFaces, const int *bFaceCells_h)
{
    if (!a || nBFaces < 0 || (nBFaces && !bFaceCells_h)) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    for (int i = 0; i < nBFaces; i++)
        if (bFaceCells_h[i] < 0 || bFaceCells_h[i] >= a->nCells) {
            b200_set_error("fv_boundary_set: face cell out of range");
            return B200LDU_EINVAL;
        }
    // per cell CSR over boundary faces, ascending boundary-face index inside a cell
    std::vector<int> start((size_t)a->nCells + 1, 0), faces(std::max(nBFaces, 1));
    for (int i = 0; i < nBFaces; i++) start[bFaceCells_h[i] + 1]++;
    for (int c = 0; c < a->nCells; c++) start[c + 1] += start[c];
    {
        std::vector<int> cur(start.begin(), start.end() - 1);
        for (int i = 0; i < nBFaces; i++) faces[cur[bFaceCells_h[i]]++] = i;
    }
    std::vector<int> fc(bFaceCells_h, bFaceCells_h + nBFaces);
    TRY(a->d_bFaceCells.upload(fc));
    TRY(a->d_bCellStart.upload(start));
    TRY(a->d_bCellFaces.upload(faces));
    a->nBFaces = nBFaces;
    return B200LDU_OK;
}

extern "C" int b200ldu_fv_surface_integrate(b200ldu_addr *a, int nComp, const double *ssf_d,
                                            const double *bssf_d, const double *V_d, double *out_d,
                                            int divideByV, int neiSign)
{
    if (!a || !ssf_d || !out_d || (divideByV && !V_d) || (nComp != 1 && nComp != 3)) return B200LDU_EINVAL;
    if (a->nBFaces && !bssf_d) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    const int *bs = a->nBFaces ? a->d_bCellStart.get() : nullptr;
    dim3 g((a->nCells + 127) / 128), b(128);
    if (nComp == 1)
        surface_integrate_kernel<1><<<g, b, 0, a->ctx->stream>>>(a->nCells, a->d_ownerStart.get(), a->d_losortStart.get(),
                                                                  a->d_losort.get(), bs, a->d_bCellFaces.get(), ssf_d, bssf_d,
                                                                  V_d, out_d, divideByV, neiSign);
    else
        surface_integrate_kernel<3><<<g, b, 0, a->ctx->stream>>>(a->nCells, a->d_ownerStart.get(), a->d_losortStart.get(),
                                                                  a->d_losort.get(), bs, a->d_bCellFaces.get(), ssf_d, bssf_d,
                                                                  V_d, out_d, divideByV, neiSign);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_fv_gauss_grad(b200ldu_addr *a, int nComp, const double *Sf_d, const double *ssf_d,
                                     const double *bSf_d, const double *bssf_d, const double *V_d,
                                     double *out_d)
{
    if (!a || !Sf_d || !ssf_d || !V_d || !out_d || (nComp != 1 && nComp != 3)) return B200LDU_EINVAL;
    if (a->nBFaces && (!bSf_d || !bssf_d)) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    const int *bs = a->nBFaces ? a->d_bCellStart.get() : nullptr;
    dim3 g((a->nCells + 127) / 128), b(128);
    if (nComp == 1)
        gauss_grad_kernel<1><<<g, b, 0, a->ctx->stream>>>(a->nCells, a->d_ownerStart.get(), a->d_losortStart.get(),
                                                           a->d_losort.get(), bs, a->d_bCellFaces.get(), Sf_d, ssf_d, bSf_d,
                                                           bssf_d, V_d, out_d);
    else
        gauss_grad_kernel<3><<<g, b, 0, a->ctx->stream>>>(a->nCells, a->d_ownerStart.get(), a->d_losortStart.get(),
                                                           a->d_losort.get(), bs, a->d_bCellFaces.get(), Sf_d, ssf_d, bSf_d,
                                                           bssf_d, V_d, out_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

// fused coefficient fills: one pass over the cells writes the diagonal as the negated
// sum of the just-computed face coefficients (negSumDiag, lduMatrixOperations.C:59-80)
// while one pass over the faces writes upper/lower.
__global__ void laplacian_upper_kernel(int nFaces, const double *__restrict__ dc, const double *__restrict__ g,
                                       double *__restrict__ upper)
{
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < nFaces) upper[f] = __dmul_rn(dc[f], g[f]);
}

__global__ void convection_faces_kernel(int nFaces, const double *__restrict__ w, const double *__restrict__ phi,
                                        double *__restrict__ lower, double *__restrict__ upper)
{
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < nFaces) {
        double lo = __dmul_rn(-w[f], phi[f]);
        lower[f] = lo;
        upper[f] = __dadd_rn(lo, phi[f]);
    }
}

extern "C" int b200ldu_fv_laplacian_fill(b200ldu_addr *a, const double *deltaCoeffs_d,
                                         const double *gammaMagSf_d, double *upper_d, double *diag_d)
{
    if (!a || !deltaCoeffs_d || !gammaMagSf_d || !upper_d || !diag_d) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    cudaStream_t st = a->ctx->stream;
    if (a->nFaces) laplacian_upper_kernel<<<(a->nFaces + 255) / 256, 256, 0, st>>>(a->nFaces, deltaCoeffs_d, gammaMagSf_d, upper_d);
    neg_sum_diag_kernel<<<(a->nCells + 127) / 128, 128, 0, st>>>(a->nCells, a->d_ownerStart.get(), a->d_losortStart.get(),
                                                                  a->d_losort.get(), upper_d, upper_d, diag_d);
    a->ctx->launches += 2;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_fv_convection_fill(b200ldu_addr *a, const double *weights_d, const double *phi_d,
                                          double *lower_d, double *upper_d, double *diag_d)
{
    if (!a || !weights_d || !phi_d || !lower_d || !upper_d || !diag_d) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    cudaStream_t st = a->ctx->stream;
    if (a->nFaces) convection_faces_kernel<<<(a->nFaces + 255) / 256, 256, 0, st>>>(a->nFaces, weights_d, phi_d, lower_d, upper_d);
    neg_sum_diag_kernel<<<(a->nCells + 127) / 128, 128, 0, st>>>(a->nCells, a->d_ownerStart.get(), a->d_losortStart.get(),
                                                                  a->d_losort.get(), upper_d, lower_d, diag_d);
    a->ctx->launches += 2;
    KERNEL_CHECK();
    return B200LDU_OK;
}

template <int NC>
__global__ void interpolate_linear_kernel(int nFaces, const int *__restrict__ l, const int *__restrict__ u,
                                          const double *__restrict__ w, const double *__restrict__ vf,
                                          double *__restrict__ sf)
{
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nFaces) return;
    double ww = w[f];
    int o = l[f], n = u[f];
#pragma unroll
    for (int k = 0; k < NC; k++)
        sf[(size_t)f * NC + k] = lin_face(ww, vf[(size_t)o * NC + k], vf[(size_t)n * NC + k]);
}

extern "C" int b200ldu_fv_interpolate_linear(b200ldu_addr *a, int nComp, const double *w_d,
                                             const double *vf_d, double *sf_d)
{
    if (!a || !w_d || !vf_d || !sf_d || (nComp != 1 && nComp != 3)) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    if (a->nFaces == 0) return B200LDU_OK;
    dim3 g((a->nFaces + 255) / 256), b(256);
    if (nComp == 1)
        interpolate_linear_kernel<1><<<g, b, 0, a->ctx->stream>>>(a->nFaces, a->d_l.get(), a->d_u.get(), w_d, vf_d, sf_d);
    else
        interpolate_linear_kernel<3><<<g, b, 0, a->ctx->stream>>>(a->nFaces, a->d_l.get(), a->d_u.get(), w_d, vf_d, sf_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

// x[cell] += sum of coeffs over the cell's boundary faces (ascending boundary face)
__global__ void add_boundary_kernel(int nCells, const int *__restrict__ bStart, const int *__restrict__ bFaces,
                                    const double *__restrict__ coeffs, double *__restrict__ x)
{
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nCells) return;
    int s = bStart[c], e = bStart[c + 1];
    if (s == e) return;
    double acc = x[c];
    for (int j = s; j < e; j++) acc = __dadd_rn(acc, coeffs[bFaces[j]]);
    x[c] = acc;
}

static int add_boundary(b200ldu_addr *a, const double *coeffs, double *x)
{
    if (!a || !coeffs || !x) return B200LDU_EINVAL;
    if (!a->nBFaces) return B200LDU_OK;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    add_boundary_kernel<<<(a->nCells + 255) / 256, 256, 0, a->ctx->stream>>>(a->nCells, a->d_bCellStart.get(),
                                                                             a->d_bCellFaces.get(), coeffs, x);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_fv_add_boundary_diag(b200ldu_addr *a, const double *internalCoeffs_d, double *diag_d)
{
    return add_boundary(a, internalCoeffs_d, diag_d);
}

extern "C" int b200ldu_fv_add_boundary_source(b200ldu_addr *a, const double *boundaryCoeffs_d, double *source_d)
{
    return add_boundary(a, boundaryCoeffs_d, source_d);
}


// ---------------------------------------------------------------------------
// SURVEY.md section 8(f) rank 1: surface interpolation fused into the face sums (grad_linear_kernel, fv_kernels.cuh), so the
// F-sized interpolated face field (401 MB - 1.2 GB at 256^3) is never written or re-read.
// ---------------------------------------------------------------------------
extern "C" int b200ldu_fv_grad_linear(b200ldu_addr *a, int nComp, const double *Sf_d, const double *w_d,
                                      const double *vf_d, const double *bSf_d, const double *bvf_d,
                                      const double *V_d, double *out_d)
{
    if (!a || !Sf_d || !w_d || !vf_d || !V_d || !out_d || (nComp != 1 && nComp != 3)) return B200LDU_EINVAL;
    if (a->nBFaces && (!bSf_d || !bvf_d)) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    const int *bs = a->nBFaces ? a->d_bCellStart.get() : nullptr;
    dim3 g((a->nCells + 127) / 128), b(128);
    if (nComp == 1)
        grad_linear_kernel<1><<<g, b, 0, a->ctx->stream>>>(a->nCells, a->d_ownerStart.get(), a->d_u.get(), a->d_losortStart.get(),
                                                            a->d_losort.get(), a->d_l.get(), bs, a->d_bCellFaces.get(), Sf_d, w_d, vf_d,
                                                            bSf_d, bvf_d, V_d, out_d);
    else
        grad_linear_kernel<3><<<g, b, 0, a->ctx->stream>>>(a->nCells, a->d_ownerStart.get(), a->d_u.get(), a->d_losortStart.get(),
                                                            a->d_losort.get(), a->d_l.get(), bs, a->d_bCellFaces.get(), Sf_d, w_d, vf_d,
                                                            bSf_d, bvf_d, V_d, out_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

// phi = interpolate(U) & Sf per internal face (icoFoam.C:73-78 phiHbyA; face-parallel):
// component-wise linear interpolation, then Sf.x*Ux + Sf.y*Uy + Sf.z*Uz added left to right
__global__ void flux_linear_kernel(int nFaces, const int *__restrict__ l, const int *__restrict__ u,
                                   const double *__restrict__ Sf, const double *__restrict__ w,
                                   const double *__restrict__ U, double *__restrict__ phi)
{
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nFaces) return;
    const double ww = w[f];
    const int o = l[f], n = u[f];
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const double fv = lin_face(ww, U[(size_t)o * 3 + k], U[(size_t)n * 3 + k]);
        const double p = __dmul_rn(Sf[(size_t)f * 3 + k], fv);
        acc = k == 0 ? p : __dadd_rn(acc, p);
    }
    phi[f] = acc;
}

extern "C" int b200ldu_fv_flux_linear(b200ldu_addr *a, const double *Sf_d, const double *w_d, const double *U_d,
                                      double *phi_d)
{
    if (!a || !Sf_d || !w_d || !U_d || !phi_d) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    if (a->nFaces == 0) return B200LDU_OK;
    flux_linear_kernel<<<(a->nFaces + 255) / 256, 256, 0, a->ctx->stream>>>(a->nFaces, a->d_l.get(), a->d_u.get(), Sf_d, w_d, U_d,
                                                                             phi_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}
