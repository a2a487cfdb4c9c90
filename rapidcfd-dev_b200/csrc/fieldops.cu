// fieldops.cu -- the element-wise field operators an application composes between the hot kernels (SURVEY.md
// section 8(f) rank 2: the icoFoam step).  The reference evaluates every `a*b`, `a + b`, `1.0/a`, `min(a, s)` of a
// field expression as one thrust::transform with one rounding per element
// (src/OpenFOAM/fields/Fields/gpuField/gpuFieldFunctionsM.C:283-330 BINARY_OPERATOR, :200-280 UNARY_FUNCTION /
// BINARY_TYPE_OPERATOR; the functors in gpuFieldFunctions.C); these entry points are that operator set over plain
// device pointers, so that a caller composing them in the reference's order gets the reference's roundings.  A
// scalar field (1 component per element) may be combined with a 3-component one (scalargpuField * vectorgpuField:
// every component times the scalar, VectorSpaceI.H:604-630).  Pure streaming; fusing whole expressions into the
// producing kernels is what csrc/fv.cu and csrc/fvmatrix.cu do for the heavy ones.
#include "internal.h"

#include "fieldops_kernels.cuh"

using namespace fieldk;


extern "C" int b200ldu_field_binary(b200ldu_ctx *ctx, int op, long long n, int ncA, const double *a_d, int ncB,
                                    const double *b_d, double *out_d)
{
    if (!ctx || !a_d || !b_d || !out_d || n < 0 || op < OP_ADD || op > OP_MAX) return B200LDU_EINVAL;
    if ((ncA != 1 && ncA != 3) || (ncB != 1 && ncB != 3)) return B200LDU_EINVAL;
    if (n == 0) return B200LDU_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int nc = ncA > ncB ? ncA : ncB;
    const long long tot = n * nc;
    binary_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, ctx->stream>>>(n, nc, ncA, ncB, op, a_d, b_d, out_d);
    ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_field_unary(b200ldu_ctx *ctx, int op, long long n, double s, const double *a_d, double *out_d)
{
    if (!ctx || !a_d || !out_d || n < 0 || op < UN_NEG || op > UN_POS) return B200LDU_EINVAL;
    if (n == 0) return B200LDU_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    unary_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, op, s, a_d, out_d);
    ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_field_dot3(b200ldu_ctx *ctx, long long n, const double *a_d, const double *b_d, double *out_d)
{
    if (!ctx || !a_d || !b_d || !out_d || n < 0) return B200LDU_EINVAL;
    if (n == 0) return B200LDU_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    dot3_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, a_d, b_d, out_d);
    ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_field_symm_magsqr(b200ldu_ctx *ctx, long long n, const double *tensor_d, double *out_d)
{
    if (!ctx || !tensor_d || !out_d || n < 0) return B200LDU_EINVAL;
    if (n == 0) return B200LDU_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    symm_magsqr_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, tensor_d, out_d);
    ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_field_gather(b200ldu_ctx *ctx, int n, int nComp, const int *cells_d, const double *field_d,
                                    double *out_d)
{
    if (!ctx || !cells_d || !field_d || !out_d || n < 0 || (nComp != 1 && nComp != 3)) return B200LDU_EINVAL;
    if (n == 0) return B200LDU_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    gather_kernel<<<(unsigned)(((long long)n * nComp + 255) / 256), 256, 0, ctx->stream>>>(n, nComp, cells_d, field_d, out_d);
    ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

// snGradScheme::snGrad of a cell field on the internal faces (the boundary values come from the boundary conditions)
extern "C" int b200ldu_fv_sngrad(b200ldu_addr *a, int nComp, const double *deltaCoeffs_d, const double *vf_d, double *out_d)
{
    if (!a || !deltaCoeffs_d || !vf_d || !out_d || (nComp != 1 && nComp != 3)) return B200LDU_EINVAL;
    if (a->nFaces == 0) return B200LDU_OK;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    const long long tot = (long long)a->nFaces * nComp;
    sngrad_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, a->ctx->stream>>>(a->nFaces, nComp, a->d_l.get(), a->d_u.get(), deltaCoeffs_d, vf_d,
                                                                             out_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

// ---- limited / upwind interpolation weights (SURVEY.md section 8(f) rank 1) ----
// limiter field of a limited scheme on the internal faces (LimitedScheme.C:60-140); gradc = fvc::grad(vf) (b200ldu_fv_grad_linear),
// C = cell centres.  scheme: "upwind" | "linear" | "limitedLinear" (coefficient k) | "vanLeer" | "Minmod"
extern "C" int b200ldu_fv_limiter(b200ldu_addr *a, const char *scheme, double k, const double *faceFlux_d, const double *vf_d,
                                  const double *gradc_d, const double *C_d, double *limiter_d)
{
    if (!a || !scheme || !limiter_d) return B200LDU_EINVAL;
    int sch;
    if (!strcmp(scheme, "upwind"))
        sch = LIM_UPWIND;
    else if (!strcmp(scheme, "linear"))
        sch = LIM_LINEAR;
    else if (!strcmp(scheme, "limitedLinear"))
        sch = LIM_LIMITED_LINEAR;
    else if (!strcmp(scheme, "vanLeer"))
        sch = LIM_VANLEER;
    else if (!strcmp(scheme, "Minmod"))
        sch = LIM_MINMOD;
    else {
        b200_set_error("Unknown discretisation scheme %s; valid schemes are: (Minmod limitedLinear linear upwind vanLeer)", scheme);
        return B200LDU_EINVAL;
    }
    if (sch >= LIM_LIMITED_LINEAR && (!faceFlux_d || !vf_d || !gradc_d || !C_d)) return B200LDU_EINVAL;
    if (sch == LIM_LIMITED_LINEAR && (k < 0 || k > 1)) {
        b200_set_error("limitedLinear: coefficient = %g should be >= 0 and <= 1 (limitedLinear.H:66-72)", k);
        return B200LDU_EINVAL;
    }
    if (a->nFaces == 0) return B200LDU_OK;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    const double kk = k > 1e-15 ? k : 1e-15;   // twoByk_ = 2.0/max(k_, SMALL), SMALL = 1e-15 (doubleScalar.H)
    limiter_kernel<<<(a->nFaces + 255) / 256, 256, 0, a->ctx->stream>>>(a->nFaces, sch, 2.0 / kk, a->d_l.get(), a->d_u.get(), faceFlux_d, vf_d,
                                                                       gradc_d, C_d, limiter_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

// weights of a limited scheme from its limiter field (limitedSurfaceInterpolationScheme.C:155-212); limiter_d NULL: upwind
// (upwind.H:120-123).  n faces: internal faces, or the faces of a coupled patch.
extern "C" int b200ldu_fv_limited_weights(b200ldu_ctx *ctx, long long n, const double *limiter_d, const double *cdWeights_d,
                                          const double *faceFlux_d, double *weights_d)
{
    if (!ctx || !faceFlux_d || !weights_d || n < 0 || (limiter_d && !cdWeights_d)) return B200LDU_EINVAL;
    if (n == 0) return B200LDU_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    limited_weights_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, limiter_d, cdWeights_d, faceFlux_d, weights_d);
    ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}
