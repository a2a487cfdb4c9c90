// mules.cu -- MULES: multidimensional universal limiter for explicit solution (SURVEY.md section 8(f) rank 4).
// b200ldu_mules_limiter = MULES::limiter (FV/fvMatrices/solvers/MULES/MULESTemplates.C:381-745): the face limiters
// lambda of the anti-diffusive flux phiCorr = phiPsi - phiBD such that psi stays within [psiMin, psiMax] and within
// the extrema of its face neighbours.  MULES::limit (:748-813) and MULES::explicitSolve (:36-78) are compositions of
// this entry with the upwind flux, the field operators and fvc::surfaceIntegrate (rapidcfd-dev_b200/mules.py).
// Static mesh; boundary faces = the faces given to b200ldu_fv_boundary_set, the coupled patch faces last (nCoupledFaces of them, in
// the patch order of b200ldu_addr_create): psiB holds their patchNeighbourField(), and after every sweep their limiters take the
// minimum with the other side's (syncTools::syncFaceList, :743) through the patch exchange of comm.cu.
#include "internal.h"
#include "comm.h"

#include "mules_kernels.cuh"

using namespace mulesk;

static int mules_limiter_impl(int corr, double extrema, b200ldu_addr *a, int nLimiterIter, double rDeltaT, const double *rho_d, const double *rho0_d,
                                     const double *psi_d, const double *psi0_d, const double *psiB_d, const double *phiBD_d,
                                     const double *phiBDB_d, const double *phiCorr_d, const double *phiCorrB_d,
                                     const double *Sp_d, const double *Su_d, const double *V_d, double psiMax, double psiMin,
                                     double *lambda_d, double *lambdaB_d, int nCoupledFaces)
{
    if (!a || !psi_d || !psi0_d || (!corr && !phiBD_d) || !phiCorr_d || !V_d || !lambda_d || nLimiterIter < 0) return B200LDU_EINVAL;
    if (a->nBFaces && (!psiB_d || !phiBDB_d || !phiCorrB_d || !lambdaB_d)) return B200LDU_EINVAL;
    const int nPF = a->nPatches ? a->patchStart[a->nPatches] : 0;
    if (nCoupledFaces < 0 || nCoupledFaces > a->nBFaces || (nCoupledFaces && nCoupledFaces != nPF)) {
        b200_set_error("b200ldu_mules_limiter: nCoupledFaces must be 0 or the number of coupled patch faces of the addressing, "
                       "listed last in b200ldu_fv_boundary_set");
        return B200LDU_EINVAL;
    }
    b200ldu_ctx *ctx = a->ctx;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int n = a->nCells, nF = a->nFaces, nB = a->nBFaces;
    // scratch: psiMaxn, psiMinn, sumPhip, mSumPhim, lambdam, lambdap (six cell fields, kept across calls) + the received limiters
    const size_t need = (size_t)6 * n + (size_t)nCoupledFaces;
    TRY(a->mulesScratch.grow(need));
    double *psiMaxn = a->mulesScratch.get(), *psiMinn = psiMaxn + n, *sumPhip = psiMinn + n, *mSumPhim = sumPhip + n,
           *lambdam = mSumPhim + n, *lambdap = lambdam + n, *theirs = lambdap + n;
    const int *bs = nB ? a->d_bCellStart.get() : nullptr;
    // lambda_d / lambdaB_d come in holding the starting limiter (MULES::limit: allLambda(mesh.nFaces(), 1.0))
    mules_bounds_kernel<<<(n + 127) / 128, 128, 0, st>>>(n, a->d_ownerStart.get(), a->d_u.get(), a->d_losortStart.get(), a->d_losort.get(), a->d_l.get(), bs,
                                                         a->d_bCellFaces.get(), psi_d, psiB_d, phiBD_d, phiBDB_d, phiCorr_d, phiCorrB_d,
                                                         psi0_d, rho_d, rho0_d, Sp_d, Su_d, V_d, rDeltaT, psiMax, psiMin, psiMaxn,
                                                         psiMinn, sumPhip, mSumPhim, corr, extrema);
    ctx->launches++;
    for (int j = 0; j < nLimiterIter; j++) {
        mules_cell_lambda_kernel<<<(n + 127) / 128, 128, 0, st>>>(n, a->d_ownerStart.get(), a->d_losortStart.get(), a->d_losort.get(), bs,
                                                                  a->d_bCellFaces.get(), lambda_d, lambdaB_d, phiCorr_d, phiCorrB_d,
                                                                  psiMaxn, psiMinn, sumPhip, mSumPhim, lambdam, lambdap);
        mules_face_lambda_kernel<<<(nF + nB + 255) / 256, 256, 0, st>>>(nF, nB, nCoupledFaces, corr, a->d_l.get(), a->d_u.get(), a->d_bFaceCells.get(), phiCorr_d,
                                                                        phiCorrB_d, phiBDB_d, lambdam, lambdap, lambda_d,
                                                                        lambdaB_d);
        ctx->launches += 2;
        if (nCoupledFaces) {
            double *mine = lambdaB_d + (nB - nCoupledFaces);
            TRY(comm_exchange_patch_field(a, 1, mine, theirs));
            mules_sync_min_kernel<<<(nCoupledFaces + 255) / 256, 256, 0, st>>>(nCoupledFaces, mine, theirs);
            ctx->launches++;
        }
    }
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_mules_limiter(b200ldu_addr *a, int nLimiterIter, double rDeltaT, const double *rho_d, const double *rho0_d,
                                     const double *psi_d, const double *psi0_d, const double *psiB_d, const double *phiBD_d,
                                     const double *phiBDB_d, const double *phiCorr_d, const double *phiCorrB_d,
                                     const double *Sp_d, const double *Su_d, const double *V_d, double psiMax, double psiMin,
                                     double *lambda_d, double *lambdaB_d, int nCoupledFaces)
{
    return mules_limiter_impl(0, 0.0, a, nLimiterIter, rDeltaT, rho_d, rho0_d, psi_d, psi0_d, psiB_d, phiBD_d, phiBDB_d, phiCorr_d,
                              phiCorrB_d, Sp_d, Su_d, V_d, psiMax, psiMin, lambda_d, lambdaB_d, nCoupledFaces);
}

// MULES::limiterCorr (CMULESTemplates.C:375-704): the limiter of a flux CORRECTION applied to an already bounded psi -- the same
// sweeps around budgets without a bounded-flux sum, the extrema widened by extremaCoeff*(psiMax - psiMin) (the reference reads
// extremaCoeff from the field's solver dictionary, default 0), the current psi and rho, and the outflow test of the non-coupled
// boundary faces on the total flux phiB_d.
extern "C" int b200ldu_mules_limiter_corr(b200ldu_addr *a, int nLimiterIter, double rDeltaT, const double *rho_d, const double *psi_d,
                                          const double *psiB_d, const double *phiB_d, const double *phiCorr_d,
                                          const double *phiCorrB_d, const double *Sp_d, const double *Su_d, const double *V_d,
                                          double psiMax, double psiMin, double extremaCoeff, double *lambda_d, double *lambdaB_d,
                                          int nCoupledFaces)
{
    if (a && a->nBFaces && !phiB_d) return B200LDU_EINVAL;
    return mules_limiter_impl(1, extremaCoeff * (psiMax - psiMin), a, nLimiterIter, rDeltaT, rho_d, nullptr, psi_d, psi_d, psiB_d, nullptr,
                              phiB_d, phiCorr_d, phiCorrB_d, Sp_d, Su_d, V_d, psiMax, psiMin, lambda_d, lambdaB_d, nCoupledFaces);
}
