// fvmatrix.cu -- the fvMatrix glue around the linear solvers (SURVEY.md section 8, row a17), caller-order
// fields.  Reference (FV/ = src/finiteVolume/): addBoundaryDiag / addCmptAvBoundaryDiag / addBoundarySource
// FV/fvMatrices/fvMatrix/fvMatrix.C:209-348; setReference :965-983; relax :1088-1345; D / A :1375-1455;
// H :1458-1508 (scalar: fvScalarMatrix.C:252-283); flux :1591-1660; residual fvScalarMatrix.C:195-240;
// solveSegregated fvScalarMatrix.C:142-192 (scalar), fvMatrixSolve.C:104-226 (component loop).
//
// Boundary model (same as oracle/fvm_oracle.py): the non-coupled boundary faces of all patches are the flat list
// given to b200ldu_fv_boundary_set (patch order), with internalCoeffs / boundaryCoeffs [nBFaces*nComp]; the coupled
// patches are those of the addressing and their coefficients the interfaceIntCoeffs / interfaceBouCoeffs of the
// last b200ldu_matrix_set (one scalar per face, used for every component).  Where the reference asks a coupled
// patch for patchNeighbourField() the caller passes it (pnf [nCoupledFaces*nComp]).
//
// The reference runs one small kernel per patch and operation; here a cell walks its boundary faces (ascending,
// non-coupled list first, then the coupled patches -- mesh order) inside ONE kernel per operation, and the
// element-wise field algebra around it (the /V, the +source, the max / divide / subtract of relax) is fused
// into the same pass.  Products are rounded separately and summed in the reference's order, so the results
// are bit-comparable with the oracle.
#include "comm.h"
#include "fieldops_kernels.cuh"
#include "fvmatrix_kernels.cuh"
#include "internal.h"
#include "ldu.h"

using namespace fvmk;

namespace
{
int coupled_lists(b200ldu_addr *a)
{
    if (a->d_cCellStart.get() || a->nPatches == 0) return B200LDU_OK;
    const int tot = a->patchStart.empty() ? 0 : a->patchStart[a->nPatches];
    if (tot == 0) return B200LDU_OK;
    std::vector<int> start((size_t)a->nCells + 1, 0), faces((size_t)tot);
    for (int i = 0; i < tot; i++) start[a->faceCells[i] + 1]++;
    for (int c = 0; c < a->nCells; c++) start[c + 1] += start[c];
    std::vector<int> cur(start.begin(), start.end() - 1);
    for (int i = 0; i < tot; i++) faces[cur[a->faceCells[i]]++] = i;
    TRY(a->d_cCellStart.upload(start));
    TRY(a->d_cCellFaces.upload(faces));
    TRY(a->d_cFaceCells.upload(a->faceCells));
    a->nCFaces = tot;
    return B200LDU_OK;
}

int lists(b200ldu_addr *a, BoundaryLists *L)
{
    TRY(coupled_lists(a));
    L->bStart = a->nBFaces ? a->d_bCellStart.get() : nullptr;
    L->bFaces = a->d_bCellFaces.get();
    L->cStart = a->nCFaces ? a->d_cCellStart.get() : nullptr;
    L->cFaces = a->d_cCellFaces.get();
    return B200LDU_OK;
}

inline dim3 grid(int n, int b) { return dim3((unsigned)((n + b - 1) / b)); }

bool bad_nc(int nc) { return nc != 1 && nc != 3; }

int need_boundary(const b200ldu_addr *a, const void *ic, const char *what)
{
    if (a->nBFaces && !ic) {
        b200_set_error("%s: boundary coefficients required (b200ldu_fv_boundary_set holds %d faces)", what, a->nBFaces);
        return B200LDU_EINVAL;
    }
    return B200LDU_OK;
}
} // namespace

// patchNeighbourField of every coupled patch face (what the fvm_* calls take as pnf_d): the patchInternalField is
// gathered, processor patches exchange it with their neighbour rank, cyclic patches read their partner patch
extern "C" int b200ldu_fv_patch_neighbour_field(b200ldu_addr *a, int nComp, const double *field_d, double *pnf_d)
{
    if (!a || !field_d || bad_nc(nComp)) return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    TRY(coupled_lists(a));
    if (a->nCFaces == 0) return B200LDU_OK;
    if (!pnf_d) return B200LDU_EINVAL;
    DevBuf<double> &send = a->fvmScratch[FVM_CMPT_PSI];
    TRY(send.grow((size_t)a->nCFaces * nComp));
    fieldk::gather_kernel<<<grid(a->nCFaces * nComp, 256), 256, 0, a->ctx->stream>>>(a->nCFaces, nComp, a->d_cFaceCells.get(),
                                                                                      field_d, send.get());
    a->ctx->launches++;
    KERNEL_CHECK();
    return comm_exchange_patch_field(a, nComp, send.get(), pnf_d);
}

extern "C" int b200ldu_fvm_add_boundary_diag(b200ldu_matrix *m, int nComp, int cmpt, const double *internalCoeffs_d,
                                             const double *diagIn_d, double *diagOut_d)
{
    if (!m || !diagOut_d || bad_nc(nComp) || cmpt >= nComp) return B200LDU_EINVAL;
    b200ldu_addr *a = m->a;
    TRY(need_boundary(a, internalCoeffs_d, "fvm_add_boundary_diag"));
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    BoundaryLists L;
    TRY(lists(a, &L));
    boundary_diag_kernel<<<grid(a->nCells, 256), 256, 0, a->ctx->stream>>>(a->nCells, L, internalCoeffs_d, nComp, cmpt,
                                                                           m->int_ext, diagIn_d, diagOut_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_fvm_add_boundary_source(b200ldu_matrix *m, int nComp, const double *boundaryCoeffs_d,
                                               const double *pnf_d, const double *sourceIn_d, double *sourceOut_d)
{
    if (!m || !sourceIn_d || !sourceOut_d || bad_nc(nComp)) return B200LDU_EINVAL;
    b200ldu_addr *a = m->a;
    TRY(need_boundary(a, boundaryCoeffs_d, "fvm_add_boundary_source"));
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    BoundaryLists L;
    TRY(lists(a, &L));
    if (nComp == 1)
        boundary_source_kernel<1><<<grid(a->nCells, 256), 256, 0, a->ctx->stream>>>(a->nCells, L, boundaryCoeffs_d,
                                                                                    m->bou_ext, pnf_d, sourceIn_d, sourceOut_d);
    else
        boundary_source_kernel<3><<<grid(a->nCells, 256), 256, 0, a->ctx->stream>>>(a->nCells, L, boundaryCoeffs_d,
                                                                                    m->bou_ext, pnf_d, sourceIn_d, sourceOut_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_fvm_A(b200ldu_matrix *m, int nComp, const double *internalCoeffs_d, const double *V_d,
                             double *A_d)
{
    if (!m || !V_d || !A_d || bad_nc(nComp) || !m->diag_ext) return B200LDU_EINVAL;
    b200ldu_addr *a = m->a;
    TRY(need_boundary(a, internalCoeffs_d, "fvm_A"));
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    BoundaryLists L;
    TRY(lists(a, &L));
    A_kernel<<<grid(a->nCells, 256), 256, 0, a->ctx->stream>>>(a->nCells, L, internalCoeffs_d, nComp, m->int_ext,
                                                               m->diag_ext, V_d, A_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_fvm_H(b200ldu_matrix *m, int nComp, const double *psi_d, const double *source_d,
                             const double *boundaryCoeffs_d, const double *pnf_d, const double *V_d, double *H_d)
{
    if (!m || !psi_d || !source_d || !V_d || !H_d || bad_nc(nComp) || !m->diag_ext) return B200LDU_EINVAL;
    b200ldu_addr *a = m->a;
    TRY(need_boundary(a, boundaryCoeffs_d, "fvm_H"));
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    BoundaryLists L;
    TRY(lists(a, &L));
    if (L.cStart && !pnf_d) {
        b200_set_error("fvm_H: the coupled patches need their patchNeighbourField (fvMatrix.C:318-346)");
        return B200LDU_EINVAL;
    }
    if (nComp == 1)
        H_kernel<1><<<grid(a->nCells, 128), 128, 0, a->ctx->stream>>>(
            a->nCells, a->d_ownerStart.get(), a->d_u.get(), a->d_losortStart.get(), a->d_losort.get(), a->d_l.get(),
            m->upper_ext, m->lower_ext, L, boundaryCoeffs_d, m->bou_ext, pnf_d, psi_d, source_d, V_d, H_d);
    else
        H_kernel<3><<<grid(a->nCells, 128), 128, 0, a->ctx->stream>>>(
            a->nCells, a->d_ownerStart.get(), a->d_u.get(), a->d_losortStart.get(), a->d_losort.get(), a->d_l.get(),
            m->upper_ext, m->lower_ext, L, boundaryCoeffs_d, m->bou_ext, pnf_d, psi_d, source_d, V_d, H_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_fvm_flux(b200ldu_matrix *m, int nComp, const double *psi_d, const double *internalCoeffs_d,
                                const double *boundaryCoeffs_d, const double *pnf_d, double *flux_d,
                                double *boundaryFlux_d, double *coupledFlux_d)
{
    if (!m || !psi_d || bad_nc(nComp) || !m->diag_ext) return B200LDU_EINVAL;
    b200ldu_addr *a = m->a;
    if ((a->nFaces && !flux_d) || (a->nBFaces && (!boundaryFlux_d || !internalCoeffs_d || !boundaryCoeffs_d)))
        return B200LDU_EINVAL;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    BoundaryLists L;
    TRY(lists(a, &L));
    if (a->nCFaces && (!coupledFlux_d || !pnf_d)) {
        b200_set_error("fvm_flux: the coupled patches need their patchNeighbourField and an output (fvMatrix.C:1636-1648)");
        return B200LDU_EINVAL;
    }
    cudaStream_t st = a->ctx->stream;
    if (a->nFaces) {
        if (nComp == 1)
            flux_internal_kernel<1><<<grid(a->nFaces, 256), 256, 0, st>>>(a->nFaces, a->d_l.get(), a->d_u.get(), m->upper_ext,
                                                                          m->lower_ext, psi_d, flux_d);
        else
            flux_internal_kernel<3><<<grid(a->nFaces, 256), 256, 0, st>>>(a->nFaces, a->d_l.get(), a->d_u.get(), m->upper_ext,
                                                                          m->lower_ext, psi_d, flux_d);
        a->ctx->launches++;
    }
    if (a->nBFaces) {
        if (nComp == 1)
            flux_boundary_kernel<1><<<grid(a->nBFaces, 256), 256, 0, st>>>(a->nBFaces, a->d_bFaceCells.get(), internalCoeffs_d,
                                                                           1, boundaryCoeffs_d, 1, nullptr, psi_d,
                                                                           boundaryFlux_d);
        else
            flux_boundary_kernel<3><<<grid(a->nBFaces, 256), 256, 0, st>>>(a->nBFaces, a->d_bFaceCells.get(), internalCoeffs_d,
                                                                           3, boundaryCoeffs_d, 3, nullptr, psi_d,
                                                                           boundaryFlux_d);
        a->ctx->launches++;
    }
    if (a->nCFaces) {
        if (nComp == 1)
            flux_boundary_kernel<1><<<grid(a->nCFaces, 256), 256, 0, st>>>(a->nCFaces, a->d_cFaceCells.get(), m->int_ext, 1,
                                                                           m->bou_ext, 1, pnf_d, psi_d, coupledFlux_d);
        else
            flux_boundary_kernel<3><<<grid(a->nCFaces, 256), 256, 0, st>>>(a->nCFaces, a->d_cFaceCells.get(), m->int_ext, 1,
                                                                           m->bou_ext, 1, pnf_d, psi_d, coupledFlux_d);
        a->ctx->launches++;
    }
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_fvm_residual(b200ldu_matrix *m, const double *psi_d, const double *source_d,
                                    const double *internalCoeffs_d, const double *boundaryCoeffs_d,
                                    const double *pnf_d, double *residual_d)
{
    if (!m || !psi_d || !source_d || !residual_d || !m->diag_ext) return B200LDU_EINVAL;
    b200ldu_addr *a = m->a;
    TRY(need_boundary(a, internalCoeffs_d, "fvm_residual"));
    TRY(need_boundary(a, boundaryCoeffs_d, "fvm_residual"));
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    BoundaryLists L;
    TRY(lists(a, &L));
    if (L.cStart && !pnf_d) {
        b200_set_error("fvm_residual: the coupled patches need their patchNeighbourField (addBoundarySource)");
        return B200LDU_EINVAL;
    }
    DevBuf<double> &tmp = a->fvmScratch[FVM_DIAG];
    TRY(tmp.grow((size_t)a->nCells));
    residual_source_kernel<<<grid(a->nCells, 256), 256, 0, a->ctx->stream>>>(a->nCells, L, internalCoeffs_d, m->int_ext,
                                                                             psi_d, source_d, tmp.get());
    a->ctx->launches++;
    KERNEL_CHECK();
    TRY(b200ldu_residual(m, psi_d, tmp.get(), residual_d)); // lduMatrix::residual incl. the interface update
    return b200ldu_fvm_add_boundary_source(m, 1, boundaryCoeffs_d, pnf_d, residual_d, residual_d);
}

extern "C" int b200ldu_fvm_relax(b200ldu_matrix *m, int nComp, double alpha, const double *psi_d,
                                 const double *internalCoeffs_d, double *diag_d, double *source_d)
{
    if (!m || !psi_d || !diag_d || !source_d || bad_nc(nComp) || !m->diag_ext) return B200LDU_EINVAL;
    if (alpha <= 0) return B200LDU_OK; // fvMatrix.C:1090-1093
    b200ldu_addr *a = m->a;
    TRY(need_boundary(a, internalCoeffs_d, "fvm_relax"));
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    BoundaryLists L;
    TRY(lists(a, &L));
    if (nComp == 1)
        relax_kernel<1><<<grid(a->nCells, 128), 128, 0, a->ctx->stream>>>(
            a->nCells, a->d_ownerStart.get(), a->d_losortStart.get(), a->d_losort.get(), m->upper_ext, m->lower_ext, L,
            internalCoeffs_d, m->int_ext, m->bou_ext, alpha, psi_d, diag_d, source_d);
    else
        relax_kernel<3><<<grid(a->nCells, 128), 128, 0, a->ctx->stream>>>(
            a->nCells, a->d_ownerStart.get(), a->d_losortStart.get(), a->d_losort.get(), m->upper_ext, m->lower_ext, L,
            internalCoeffs_d, m->int_ext, m->bou_ext, alpha, psi_d, diag_d, source_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

extern "C" int b200ldu_fvm_set_reference(b200ldu_matrix *m, int celli, int nComp, const double *value_h,
                                         double *diag_d, double *source_d)
{
    if (!m || !value_h || !diag_d || !source_d || bad_nc(nComp) || celli >= m->a->nCells) return B200LDU_EINVAL;
    if (celli < 0) return B200LDU_OK; // the reference cell lives on another rank (fvMatrix.C:972)
    b200ldu_addr *a = m->a;
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    set_reference_kernel<<<1, 1, 0, a->ctx->stream>>>(celli, nComp, value_h[0], nComp > 1 ? value_h[1] : 0.0,
                                                      nComp > 2 ? value_h[2] : 0.0, diag_d, source_d);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

// solveSegregated: fold the boundary into diagonal and source, solve, put the diagonal back.
// Scalar: fvScalarMatrix.C:142-192.  Vector: fvMatrixSolve.C:104-226 -- the coupled boundary source goes in once
// for all components and is taken out again per component through the interface update on the source.
extern "C" int b200ldu_fvm_solve(b200ldu_matrix *m, int nComp, const char *solver, const char *precondOrSmoother,
                                 const b200ldu_controls *controls, b200ldu_gamg *gamg, double *psi_d,
                                 const double *source_d, const double *internalCoeffs_d,
                                 const double *boundaryCoeffs_d, const double *pnf_d, b200ldu_perf *perf)
{
    if (!m || !solver || !psi_d || !source_d || !perf || bad_nc(nComp) || !m->diag_ext) return B200LDU_EINVAL;
    b200ldu_addr *a = m->a;
    TRY(need_boundary(a, internalCoeffs_d, "fvm_solve"));
    TRY(need_boundary(a, boundaryCoeffs_d, "fvm_solve"));
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    BoundaryLists L;
    TRY(lists(a, &L));
    if (nComp > 1 && L.cStart && !pnf_d) {
        b200_set_error("fvm_solve: the component loop needs the patchNeighbourField of the coupled patches");
        return B200LDU_EINVAL;
    }
    const int n = a->nCells;
    cudaStream_t st = a->ctx->stream;
    // the caller's coefficient arrays: the matrix is re-pointed at the folded diagonal for the solve
    const double *diag0 = m->diag_ext;
    const double *bou = m->bou_ext, *intc = m->int_ext;
    DevBuf<double> *scr = a->fvmScratch;
    TRY(scr[FVM_DIAG].grow((size_t)n));
    TRY(scr[FVM_SOURCE].grow((size_t)n * nComp));
    double *dK = scr[FVM_DIAG].get(), *total = scr[FVM_SOURCE].get();
    int rc = B200LDU_OK;
    if (nComp == 1) {
        boundary_diag_kernel<<<grid(n, 256), 256, 0, st>>>(n, L, internalCoeffs_d, 1, 0, intc, diag0, dK);
        boundary_source_kernel<1><<<grid(n, 256), 256, 0, st>>>(n, L, boundaryCoeffs_d, bou, nullptr, source_d, total);
        a->ctx->launches += 2;
        KERNEL_CHECK();
        rc = matrix_set_diag(m, dK); // the off-diagonal streams are unchanged
        if (rc == B200LDU_OK) rc = b200ldu_solve(m, solver, precondOrSmoother, controls, gamg, psi_d, total, &perf[0], nullptr, 0);
    } else {
        TRY(scr[FVM_CMPT_SOURCE].grow((size_t)n));
        TRY(scr[FVM_CMPT_PSI].grow((size_t)n));
        double *sK = scr[FVM_CMPT_SOURCE].get(), *pK = scr[FVM_CMPT_PSI].get();
        boundary_source_kernel<3><<<grid(n, 256), 256, 0, st>>>(n, L, boundaryCoeffs_d, bou, pnf_d, source_d, total);
        a->ctx->launches++;
        KERNEL_CHECK();
        BoundaryLists none = L;
        none.cStart = nullptr;
        for (int k = 0; k < nComp && rc == B200LDU_OK; k++) {
            boundary_diag_kernel<<<grid(n, 256), 256, 0, st>>>(n, L, internalCoeffs_d, nComp, k, intc, diag0, dK);
            component_kernel<<<grid(n, 256), 256, 0, st>>>(n, nComp, k, L, bou, pnf_d, total, sK);
            component_kernel<<<grid(n, 256), 256, 0, st>>>(n, nComp, k, none, nullptr, nullptr, psi_d, pK);
            a->ctx->launches += 3;
            KERNEL_CHECK();
            rc = matrix_set_diag(m, dK);
            if (rc == B200LDU_OK) rc = b200ldu_solve(m, solver, precondOrSmoother, controls, gamg, pK, sK, &perf[k], nullptr, 0);
            if (rc == B200LDU_OK) {
                set_component_kernel<<<grid(n, 256), 256, 0, st>>>(n, nComp, k, pK, psi_d);
                a->ctx->launches++;
                KERNEL_CHECK();
            }
        }
    }
    const int rc2 = matrix_set_diag(m, diag0); // diag() = saveDiag
    return rc != B200LDU_OK ? rc : rc2;
}
