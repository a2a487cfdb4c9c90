// gamg.cu -- GAMG: cached pair agglomeration (host, like the reference) + device-resident
// V-cycle on the banded kernels.
//
// Reference (GAMG/ = LDU/solvers/GAMG/): pair agglomeration
// GAMG/GAMGAgglomerations/pairGAMGAgglomeration/pairGAMGAgglomerate.C:31-313; coarse
// addressing GAMG/GAMGAgglomerations/GAMGAgglomeration/GAMGAgglomerateLduAddressing.C:245-461;
// restrict/prolong GAMGAgglomerationTemplates.C:35-308; coarse matrices
// GAMG/GAMGSolverAgglomerateMatrix.C:37-322 (+ F.H:9-160); solve / Vcycle
// GAMG/GAMGSolverSolve.C:59-619; scale GAMGSolverScale.C:59-171; interpolate
// GAMGSolverInterpolate.C:45-110; defaults GAMGSolver.C:67-77.
//
// What is different from the reference's execution (not its numerics):
//  * restriction, prolongation and the Galerkin-by-summation coarse matrices are
//    deterministic segmented sums (ascending fine index, the order of the reference's
//    sorted non-atomic path) -- no atomics;
//  * the whole cycle is enqueued without host synchronisation: scaling factors and the
//    convergence decision stay on the device; the coarsest level is solved on the device
//    with the inverse of the (tiny) coarsest matrix computed once per solve on the host,
//    instead of a D2H/host-LU/H2D round trip in every cycle (GAMGSolverSolve.C:564-569).
// Multi-rank: processor interfaces are agglomerated level by level like
// processorGAMGInterface.C:60-140 (the neighbour side's restrict map is exchanged over NCCL at
// set-up), interface coefficients are restricted by deterministic segmented sums, every coarse
// level gets its own peer-memory halo descriptors, and the coarsest level is solved against
// the inverse of the matrix assembled from ALL ranks (LUscalarMatrix.C:60-160 gathers it on the
// master; here every rank holds its own rows of the inverse and the right-hand sides are
// all-gathered through peer memory inside the solve kernel).
#include <algorithm>
#include <cmath>

#include "comm.h"
#include "ldu.h"
#include "solver_steps.cuh"

constexpr int MAX_LEVELS = 50; // GAMGAgglomeration.C:94

struct GamgLevel {
    int nFine = 0, nFineFaces = 0, nCoarse = 0, nCoarseFaces = 0;
    std::vector<int> restrictAddr;      // fine cell -> coarse cell (caller orders)
    std::vector<int> faceRestrict;      // fine face -> coarse face | -(cell+1)
    std::vector<unsigned char> faceFlip;
    // coarse level addressing (banded layout built) and matrix (values refreshed every solve): the matrix is
    // declared after the addressing so that it is destroyed first
    AbiHandle<b200ldu_addr, b200ldu_addr_destroy> addr;
    AbiHandle<b200ldu_matrix, b200ldu_matrix_destroy> mat;
    // device maps, banded vector space
    DevBuf<int> d_childStart, d_child; // coarse banded row -> fine banded rows (asc. fine cell)
    DevBuf<int> d_pmap;                // fine banded row -> coarse banded row (-1 padding)
    // device maps, caller order (coefficients)
    DevBuf<int> d_cellChildStart, d_cellChild; // coarse cell -> fine cells ascending
    DevBuf<int> d_faceChildStart, d_faceChild; // coarse face -> (fine face << 1 | flip) ascending
    DevBuf<int> d_diagFaceStart, d_diagFace;   // coarse cell -> collapsed fine faces ascending
    DevBuf<double> d_diag, d_upper, d_lower;   // caller-order coarse coefficients
    // coupled patches of the coarse level
    int nFinePF = 0, nCoarsePF = 0;
    std::vector<int> cPatchStart, cFaceCells;
    DevBuf<int> d_pfChildStart, d_pfChild; // coarse patch face -> fine patch faces ascending
    DevBuf<double> d_bou, d_int;
    // level vectors (banded, vecLen of the coarse level)
    DevBuf<double> corr, src, tmp, acf, pre;
};

struct b200ldu_gamg {
    b200ldu_addr *finest = nullptr;
    int nLevels = 0;
    std::vector<GamgLevel> lev;
    DevBuf<double> d_inv; // this rank's rows of the inverse of the (global) coarsest matrix
    int invN = 0;         // global size of the coarsest system
    // multi-rank coarsest solve
    std::vector<int> coarsestCounts, coarsestOffs, coarsestNbrCell;
    int nMaxCoarsest = 0;
    DevBuf<double> d_gatherAll; // NCCL fallback of the peer-memory gather
    bool metaUploaded = false;
};

// ---------------------------------------------------------------------------
// host agglomeration
// ---------------------------------------------------------------------------
// pairGAMGAgglomeration::agglomerate(nCoarseCells, addr, faceWeights): pairGAMGAgglomerate.C:135-313
static void pair_agglomerate(int n, const std::vector<int> &lo, const std::vector<int> &up,
                             const std::vector<double> &w, bool &forward, std::vector<int> &map, int &nCoarse)
{
    const int nf = (int)lo.size();
    std::vector<int> off((size_t)n + 1, 0), cnt((size_t)n, 0), cf((size_t)2 * nf + 1);
    for (int f = 0; f < nf; f++) off[up[f] + 1]++;
    for (int f = 0; f < nf; f++) off[lo[f] + 1]++;
    for (int c = 0; c < n; c++) off[c + 1] += off[c];
    // neighbour-side faces first, then owned faces (:172-192)
    for (int f = 0; f < nf; f++) cf[off[up[f]] + cnt[up[f]]++] = f;
    for (int f = 0; f < nf; f++) cf[off[lo[f]] + cnt[lo[f]]++] = f;
    map.assign(n, -1);
    nCoarse = 0;
    const double GREAT = 1e20;
    for (int ci = 0; ci < n; ci++) {
        int c = forward ? ci : n - ci - 1;
        if (map[c] >= 0) continue;
        int match = -1;
        double best = -GREAT;
        for (int k = off[c]; k < off[c + 1]; k++) {
            int f = cf[k];
            if (map[up[f]] < 0 && map[lo[f]] < 0 && w[f] > best) {
                match = f;
                best = w[f];
            }
        }
        if (match >= 0) {
            map[up[match]] = nCoarse;
            map[lo[match]] = nCoarse;
            nCoarse++;
        } else {
            int cm = -1;
            double cbest = -GREAT;
            for (int k = off[c]; k < off[c + 1]; k++) {
                int f = cf[k];
                if (w[f] > cbest) {
                    cm = f;
                    cbest = w[f];
                }
            }
            if (cm >= 0) map[c] = std::max(map[up[cm]], map[lo[cm]]);
        }
    }
    for (int ci = 0; ci < n; ci++) {
        int c = forward ? ci : n - ci - 1;
        if (map[c] < 0) map[c] = nCoarse++;
    }
    if (!forward) {
        nCoarse--;
        for (int c = 0; c < n; c++) map[c] = nCoarse - map[c];
        nCoarse++;
    }
    forward = !forward;
}

// GAMGAgglomeration::agglomerateLduAddressing: GAMGAgglomerateLduAddressing.C:245-461
static void coarse_addressing(const std::vector<int> &lo, const std::vector<int> &up, const std::vector<int> &rmap,
                              int nCoarse, std::vector<int> &cOwner, std::vector<int> &cNeigh,
                              std::vector<int> &fr, std::vector<unsigned char> &flip)
{
    const int nff = (int)lo.size();
    // per coarse owner: its coarse faces in order of discovery, as singly linked lists in flat arrays (a vector per
    // coarse cell cost seconds of allocator time on the first levels of a 16 M cell mesh)
    std::vector<int> head(nCoarse, -1), tail(nCoarse, -1), nxt, initNei;
    nxt.reserve(nff / 2 + 16);
    initNei.reserve(nff / 2 + 16);
    fr.assign(nff, 0);
    for (int f = 0; f < nff; f++) {
        int ru = rmap[up[f]], rl = rmap[lo[f]];
        if (ru == rl) {
            fr[f] = -(ru + 1);
            continue;
        }
        int cOwn = std::min(ru, rl), cNei = std::max(ru, rl);
        int found = -1;
        for (int cfi = head[cOwn]; cfi >= 0; cfi = nxt[cfi])
            if (initNei[cfi] == cNei) {
                found = cfi;
                break;
            }
        if (found < 0) {
            found = (int)initNei.size();
            initNei.push_back(cNei);
            nxt.push_back(-1);
            if (tail[cOwn] >= 0)
                nxt[tail[cOwn]] = found;
            else
                head[cOwn] = found;
            tail[cOwn] = found;
        }
        fr[f] = found;
    }
    const int nCF = (int)initNei.size();
    cOwner.resize(nCF);
    cNeigh.resize(nCF);
    std::vector<int> cMap(nCF);
    int k = 0;
    for (int cc = 0; cc < nCoarse; cc++)
        for (int cfi = head[cc]; cfi >= 0; cfi = nxt[cfi]) {
            cOwner[k] = cc;
            cNeigh[k] = initNei[cfi];
            cMap[cfi] = k++;
        }
    flip.assign(nff, 0);
    for (int f = 0; f < nff; f++)
        if (fr[f] >= 0) {
            fr[f] = cMap[fr[f]];
            int ru = rmap[up[f]], rl = rmap[lo[f]];
            if (cOwner[fr[f]] == ru && cNeigh[fr[f]] == rl) flip[f] = 1;
        }
}

static void csr_from_map(const std::vector<int> &map, int nTargets, std::vector<int> &start, std::vector<int> &items)
{
    start.assign((size_t)nTargets + 1, 0);
    for (int v : map)
        if (v >= 0) start[v + 1]++;
    for (int t = 0; t < nTargets; t++) start[t + 1] += start[t];
    items.resize(std::max(start[nTargets], 1));
    std::vector<int> cur(start.begin(), start.end() - 1);
    for (int i = 0; i < (int)map.size(); i++)
        if (map[i] >= 0) items[cur[map[i]]++] = i;
}

extern "C" int b200ldu_gamg_destroy(b200ldu_gamg *g)
{
    if (!g) return B200LDU_OK;
    cudaSetDevice(g->finest->ctx->device);
    cudaStreamSynchronize(g->finest->ctx->stream);
    delete g;
    return B200LDU_OK;
}

extern "C" int b200ldu_gamg_create(b200ldu_addr *a, const double *faceWeights_h, int nCellsInCoarsestLevel,
                                   int mergeLevels, int *forwardInOut, b200ldu_gamg **out)
{
    if (!a || !faceWeights_h || !out) return B200LDU_EINVAL;
    if (mergeLevels < 1) {
        b200_set_error("GAMG: mergeLevels must be >= 1");
        return B200LDU_EINVAL;
    }
    for (int p = 0; p < a->nPatches; p++)
        if (a->neighbRank[p] == a->ctx->rank && a->ctx->nRanks > 1) {
            b200_set_error("GAMG: patch %d names this rank as its neighbour; cyclic patches are declared with neighbRank = -(partnerPatch + 1)", p);
            return B200LDU_EINVAL;
        }
    CUDA_TRY(cudaSetDevice(a->ctx->device));
    AbiHandle<b200ldu_gamg, b200ldu_gamg_destroy> g(new b200ldu_gamg());
    g->finest = a;
    bool forward = forwardInOut ? (*forwardInOut != 0) : true; // pairGAMGAgglomeration.C:33
    std::vector<int> lo = a->l, up = a->u;
    std::vector<int> fPatchStart = a->patchStart, fFaceCells = a->faceCells; // coupled patches of the fine level
    const int nPatches = a->nPatches;
    std::vector<double> w(faceWeights_h, faceWeights_h + a->nFaces);
    std::vector<double> centres = a->centres_h;
    int nFine = a->nCells;
    int rc = B200LDU_OK;

    // One pairing step on the host (pairGAMGAgglomerate.C:46-107): maps from the current fine
    // level to the next coarser one.  With mergeLevels > 1 consecutive steps are composed
    // (combineLevels) before the device structures of the level are built.
    struct HostStep {
        int nFine = 0, nFineFaces = 0, nCoarse = 0, nCoarseFaces = 0, nFinePF = 0, nCoarsePF = 0;
        std::vector<int> map, faceRestrict, cOwner, cNeigh, pfRestrict, cPatchStart, cFaceCells;
        std::vector<unsigned char> faceFlip;
        std::vector<double> cc;
    };

    // build the device side of a finished level
    auto finalize = [&](HostStep &H) -> int {
        g->lev.emplace_back();
        GamgLevel &L = g->lev.back();
        b200ldu_addr *fineAddr = g->lev.size() >= 2 ? g->lev[g->lev.size() - 2].addr.get() : a;
        const std::vector<int> &finePerm = fineAddr->perm_h, &fiperm = fineAddr->iperm_h;
        L.nFine = H.nFine;
        L.nFineFaces = H.nFineFaces;
        L.nCoarse = H.nCoarse;
        L.nCoarseFaces = H.nCoarseFaces;
        L.nFinePF = H.nFinePF;
        L.nCoarsePF = H.nCoarsePF;
        L.restrictAddr.swap(H.map);
        L.faceRestrict.swap(H.faceRestrict);
        L.faceFlip.swap(H.faceFlip);
        L.cPatchStart.swap(H.cPatchStart);
        L.cFaceCells.swap(H.cFaceCells);
        const std::vector<int> &map = L.restrictAddr;
        const int nCoarse = L.nCoarse, nFineL = L.nFine;
        b200ldu_addr *ca = nullptr;
        TRY(b200ldu_addr_create(a->ctx, nCoarse, L.nCoarseFaces, H.cOwner.data(), H.cNeigh.data(), nPatches,
                                nPatches ? L.cPatchStart.data() : nullptr, nPatches ? L.cFaceCells.data() : nullptr,
                                nPatches ? a->neighbRank.data() : nullptr, H.cc.empty() ? nullptr : H.cc.data(), &ca));
        L.addr.reset(ca);
        if (nPatches) {
            std::vector<int> ps, pi;
            csr_from_map(H.pfRestrict, L.nCoarsePF, ps, pi);
            TRY(L.d_pfChildStart.upload(ps));
            TRY(L.d_pfChild.upload(pi));
            TRY(L.d_bou.alloc((size_t)std::max(L.nCoarsePF, 1)));
            TRY(L.d_int.alloc((size_t)std::max(L.nCoarsePF, 1)));
        }
        b200ldu_matrix *cm = nullptr;
        TRY(b200ldu_matrix_create(L.addr.get(), &cm));
        L.mat.reset(cm);
        // ---- device maps ----
        {
            std::vector<int> cs, ci;
            csr_from_map(map, nCoarse, cs, ci); // coarse cell -> fine cells ascending
            TRY(L.d_cellChildStart.upload(cs));
            TRY(L.d_cellChild.upload(ci));
            // banded versions
            const std::vector<int> &cperm = L.addr->perm_h, &ciperm = L.addr->iperm_h;
            const int nPadC = L.addr->L.nPad, nPadF = fineAddr->L.nPad;
            std::vector<int> bs((size_t)nPadC + 1, 0), bi(std::max(nFineL, 1));
            for (int R = 0; R < nPadC; R++) {
                int C = ciperm[R];
                int cntC = C >= 0 ? cs[C + 1] - cs[C] : 0;
                bs[R + 1] = bs[R] + cntC;
                for (int k = 0; k < cntC; k++) bi[bs[R] + k] = finePerm[ci[cs[C] + k]];
            }
            std::vector<int> pm(nPadF, -1);
            for (int q = 0; q < nPadF; q++)
                if (fiperm[q] >= 0) pm[q] = cperm[map[fiperm[q]]];
            TRY(L.d_childStart.upload(bs));
            TRY(L.d_child.upload(bi));
            TRY(L.d_pmap.upload(pm));
            // face maps (caller order)
            std::vector<int> fmap(L.nFineFaces), dmap(L.nFineFaces);
            for (int f = 0; f < L.nFineFaces; f++) {
                fmap[f] = L.faceRestrict[f] >= 0 ? L.faceRestrict[f] : -1;
                dmap[f] = L.faceRestrict[f] < 0 ? -1 - L.faceRestrict[f] : -1;
            }
            std::vector<int> fs, fi, ds, di;
            csr_from_map(fmap, L.nCoarseFaces, fs, fi);
            csr_from_map(dmap, nCoarse, ds, di);
            for (int k = 0; k < fs[L.nCoarseFaces]; k++) fi[k] = (fi[k] << 1) | (L.faceFlip[fi[k]] ? 1 : 0);
            TRY(L.d_faceChildStart.upload(fs));
            TRY(L.d_faceChild.upload(fi));
            TRY(L.d_diagFaceStart.upload(ds));
            TRY(L.d_diagFace.upload(di));
        }
        size_t nf = (size_t)std::max(L.nCoarseFaces, 1);
        TRY(L.d_diag.alloc((size_t)nCoarse));
        TRY(L.d_upper.alloc(nf));
        TRY(L.d_lower.alloc(nf));
        for (DevBuf<double> *v : {&L.corr, &L.src, &L.tmp, &L.acf, &L.pre}) TRY(addr_alloc_vec(L.addr.get(), *v));
        return B200LDU_OK;
    };

    // combineLevels (GAMGAgglomerateLduAddressing.C:606-765): fold step N (built on the coarse side
    // of P) into P.  The flip of a composed face is the flip of the second step alone, as in the
    // reference (:631); a face that collapses into a cell carries no flip.
    auto combine = [&](HostStep &P, HostStep &N) {
        for (int f = 0; f < P.nFineFaces; f++) {
            if (P.faceRestrict[f] >= 0) {
                const int mid = P.faceRestrict[f];
                P.faceRestrict[f] = N.faceRestrict[mid];
                P.faceFlip[f] = N.faceFlip[mid];
            } else {
                P.faceRestrict[f] = -N.map[-P.faceRestrict[f] - 1] - 1;
                P.faceFlip[f] = 0;
            }
        }
        for (int c = 0; c < P.nFine; c++) P.map[c] = N.map[P.map[c]];
        for (int i = 0; i < P.nFinePF; i++) P.pfRestrict[i] = N.pfRestrict[P.pfRestrict[i]];
        P.nCoarse = N.nCoarse;
        P.nCoarseFaces = N.nCoarseFaces;
        P.nCoarsePF = N.nCoarsePF;
        P.cOwner.swap(N.cOwner);
        P.cNeigh.swap(N.cNeigh);
        P.cPatchStart.swap(N.cPatchStart);
        P.cFaceCells.swap(N.cFaceCells);
        P.cc.swap(N.cc);
    };

    HostStep pend;
    bool havePend = false;
    int nPairLevels = 0;
    while ((int)g->lev.size() + (havePend ? 1 : 0) < MAX_LEVELS - 1) {
        HostStep H;
        int nCoarse = -1;
        pair_agglomerate(nFine, lo, up, w, forward, H.map, nCoarse);
        // continueAgglomerating (GAMGAgglomeration.C:72-84): and-reduced over the ranks
        {
            double votes = (nCoarse >= nCellsInCoarsestLevel) ? 0.0 : 1.0;
            std::vector<double> all((size_t)a->ctx->nRanks, 0.0);
            rc = comm_allgather_host(a->ctx, &votes, 1, all.data());
            if (rc != B200LDU_OK) break;
            double stopVotes = 0;
            for (double v : all) stopVotes += v;
            if (stopVotes > 0) break;
        }
        H.nFine = nFine;
        H.nFineFaces = (int)lo.size();
        H.nCoarse = nCoarse;
        coarse_addressing(lo, up, H.map, nCoarse, H.cOwner, H.cNeigh, H.faceRestrict, H.faceFlip);
        H.nCoarseFaces = (int)H.cOwner.size();
        // coarse centres = mean of the children (only used to pick the band renumbering)
        if (!centres.empty()) {
            H.cc.assign((size_t)3 * nCoarse, 0.0);
            std::vector<int> cn(nCoarse, 0);
            for (int c = 0; c < nFine; c++) {
                for (int k = 0; k < 3; k++) H.cc[3 * (size_t)H.map[c] + k] += centres[3 * (size_t)c + k];
                cn[H.map[c]]++;
            }
            for (int C = 0; C < nCoarse; C++)
                for (int k = 0; k < 3; k++) H.cc[3 * (size_t)C + k] /= cn[C];
        }
        // processor / cyclic interfaces of the coarse level (processorGAMGInterface.C:60-140,
        // cyclicGAMGInterface.C:70-150): unique
        // (master cell, slave cell) pairs in order of first appearance along every fine patch
        H.nFinePF = nPatches ? fPatchStart[nPatches] : 0;
        H.pfRestrict.assign(std::max(H.nFinePF, 1), 0);
        H.cPatchStart.assign((size_t)nPatches + 1, 0);
        if (nPatches) {
            std::vector<int> sendMap(H.nFinePF), nbrMap(H.nFinePF);
            for (int i = 0; i < H.nFinePF; i++) sendMap[i] = H.map[fFaceCells[i]];
            rc = comm_exchange_patch_ints(a->ctx, nPatches, fPatchStart.data(), a->neighbRank.data(), sendMap.data(),
                                          nbrMap.data());
            if (rc != B200LDU_OK) break;
            int nC = 0;
            for (int p = 0; p < nPatches; p++) {
                const int nb = a->neighbRank[p], me = a->ctx->rank;
                // master side first so that both sides enumerate the same pairs: the lower rank of a processor
                // patch, the owner (= lower patch index) of a cyclic pair (cyclicGAMGInterface.C:104-127)
                const bool master = nb >= 0 ? (me < nb) : (p < -nb - 1);
                H.cPatchStart[p] = nC;
                std::vector<std::pair<int, int>> pairs;
                for (int i = fPatchStart[p]; i < fPatchStart[p + 1]; i++) {
                    std::pair<int, int> pr = master ? std::make_pair(sendMap[i], nbrMap[i])
                                                    : std::make_pair(nbrMap[i], sendMap[i]);
                    int found = -1;
                    for (int k = (int)pairs.size() - 1; k >= 0; k--)
                        if (pairs[k] == pr) {
                            found = k;
                            break;
                        }
                    if (found < 0) {
                        found = (int)pairs.size();
                        pairs.push_back(pr);
                        H.cFaceCells.push_back(sendMap[i]);
                    }
                    H.pfRestrict[i] = nC + found;
                }
                nC += (int)pairs.size();
            }
            H.cPatchStart[nPatches] = nC;
            H.nCoarsePF = nC;
        }
        // restrictFaceField of the weights for the next step (pairGAMGAgglomerate.C:86-107)
        std::vector<double> cw(H.nCoarseFaces, 0.0);
        for (int f = 0; f < H.nFineFaces; f++)
            if (H.faceRestrict[f] >= 0) cw[H.faceRestrict[f]] += w[f];
        w.swap(cw);
        lo = H.cOwner;
        up = H.cNeigh;
        fPatchStart = H.cPatchStart;
        fFaceCells = H.cFaceCells;
        centres = H.cc;
        nFine = nCoarse;
        if (nPairLevels % mergeLevels) { // pairGAMGAgglomerate.C:110-117
            combine(pend, H);
        } else {
            if (havePend) {
                rc = finalize(pend);
                if (rc != B200LDU_OK) break;
            }
            pend = std::move(H);
            havePend = true;
        }
        nPairLevels++;
    }
    if (rc == B200LDU_OK && havePend) rc = finalize(pend);
    if (forwardInOut) *forwardInOut = forward ? 1 : 0;
    if (rc != B200LDU_OK) return rc;
    g->nLevels = (int)g->lev.size();
    // coarsest level across the ranks: sizes, offsets and the neighbour-side cell of every
    // coarsest processor-patch face (columns of the global matrix, LUscalarMatrix.C:201-270)
    if (g->nLevels > 0 && (a->ctx->nRanks > 1 || nPatches)) {
        GamgLevel &LC = g->lev[g->nLevels - 1];
        const int R = a->ctx->nRanks;
        double mine = LC.nCoarse;
        std::vector<double> all(R);
        rc = comm_allgather_host(a->ctx, &mine, 1, all.data());
        if (rc == B200LDU_OK) {
            g->coarsestCounts.resize(R);
            g->coarsestOffs.assign(R + 1, 0);
            g->nMaxCoarsest = 0;
            for (int r = 0; r < R; r++) {
                g->coarsestCounts[r] = (int)all[r];
                g->coarsestOffs[r + 1] = g->coarsestOffs[r] + g->coarsestCounts[r];
                g->nMaxCoarsest = std::max(g->nMaxCoarsest, g->coarsestCounts[r]);
            }
            if (R > 1 && g->nMaxCoarsest > P2P_GMAX) {
                b200_set_error("GAMG: coarsest level has %d cells on one rank; the multi-rank direct solve "
                               "supports up to %d (lower nCellsInCoarsestLevel)", g->nMaxCoarsest, P2P_GMAX);
                rc = B200LDU_EINVAL;
            }
        }
        if (rc == B200LDU_OK && nPatches) {
            g->coarsestNbrCell.resize(std::max(LC.nCoarsePF, 1));
            rc = comm_exchange_patch_ints(a->ctx, nPatches, LC.cPatchStart.data(), a->neighbRank.data(),
                                          LC.cFaceCells.data(), g->coarsestNbrCell.data());
        }
        if (rc != B200LDU_OK) return rc;
    }
    *out = g.release();
    return B200LDU_OK;
}

extern "C" int b200ldu_gamg_nlevels(const b200ldu_gamg *g) { return g ? g->nLevels : 0; }

extern "C" int b200ldu_gamg_level_size(const b200ldu_gamg *g, int lev, int *nCells, int *nFaces)
{
    if (!g || lev < 0 || lev >= g->nLevels) return B200LDU_EINVAL;
    if (nCells) *nCells = g->lev[lev].nCoarse;
    if (nFaces) *nFaces = g->lev[lev].nCoarseFaces;
    return B200LDU_OK;
}

extern "C" int b200ldu_gamg_restrict_addr(const b200ldu_gamg *g, int lev, int *out_h)
{
    if (!g || lev < 0 || lev >= g->nLevels || !out_h) return B200LDU_EINVAL;
    memcpy(out_h, g->lev[lev].restrictAddr.data(), sizeof(int) * g->lev[lev].restrictAddr.size());
    return B200LDU_OK;
}

// ---------------------------------------------------------------------------
// device kernels
// ---------------------------------------------------------------------------
// restrictField (GAMGAgglomerationF.H:10-40): coarse = sum of fine values in ascending
// fine index, starting from zero
__global__ void restrict_kernel(int nRows, const int *__restrict__ start, const int *__restrict__ child,
                                const double *__restrict__ ff, double *__restrict__ cf, const int *stop)
{
    if (stop && *stop) return;
    int R = blockIdx.x * blockDim.x + threadIdx.x;
    if (R >= nRows) return;
    double s = 0.0;
    for (int k = start[R]; k < start[R + 1]; k++) s = __dadd_rn(s, ff[child[k]]);
    cf[R] = s;
}

// prolongField (GAMGAgglomerationTemplates.C:273-308): ff[c] = cf[map[c]]
__global__ void prolong_kernel(int nRows, const int *__restrict__ pmap, const double *__restrict__ cf,
                               double *__restrict__ ff, const int *stop)
{
    if (stop && *stop) return;
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nRows) return;
    int R = pmap[r];
    ff[r] = R >= 0 ? cf[R] : 0.0;
}

// coarse diagonal: restrict(fine diag) then the collapsed faces, ascending
// (GAMGSolverAgglomerateMatrix.C:59-71, F.H diagSym/diagAsymAgglomerate)
__global__ void agg_diag_kernel(int nCoarse, const int *__restrict__ cStart, const int *__restrict__ cChild,
                                const int *__restrict__ dStart, const int *__restrict__ dFace,
                                const double *__restrict__ fDiag, const double *__restrict__ fUpper,
                                const double *__restrict__ fLower, double *__restrict__ cDiag)
{
    int C = blockIdx.x * blockDim.x + threadIdx.x;
    if (C >= nCoarse) return;
    double s = 0.0;
    for (int k = cStart[C]; k < cStart[C + 1]; k++) s = __dadd_rn(s, fDiag[cChild[k]]);
    for (int k = dStart[C]; k < dStart[C + 1]; k++) {
        int f = dFace[k];
        double add = fLower ? __dadd_rn(fUpper[f], fLower[f]) : __dmul_rn(2.0, fUpper[f]);
        s = __dadd_rn(s, add);
    }
    cDiag[C] = s;
}

// coarse upper/lower: sums of the mapped fine faces, ascending, flipped faces swapped
// (F.H sym/asymAgglomerate)
__global__ void agg_faces_kernel(int nCF, const int *__restrict__ fStart, const int *__restrict__ fChild,
                                 const double *__restrict__ fUpper, const double *__restrict__ fLower,
                                 double *__restrict__ cUpper, double *__restrict__ cLower)
{
    int F = blockIdx.x * blockDim.x + threadIdx.x;
    if (F >= nCF) return;
    double u = 0.0, l = 0.0;
    for (int k = fStart[F]; k < fStart[F + 1]; k++) {
        int f = fChild[k] >> 1, flip = fChild[k] & 1;
        if (!fLower) {
            u = __dadd_rn(u, fUpper[f]);
        } else if (!flip) {
            u = __dadd_rn(u, fUpper[f]);
            l = __dadd_rn(l, fLower[f]);
        } else {
            u = __dadd_rn(u, fLower[f]);
            l = __dadd_rn(l, fUpper[f]);
        }
    }
    cUpper[F] = u;
    if (fLower) cLower[F] = l;
}

// coarse interface coefficients: sums over the patch face map, ascending fine patch face
// (agglomerateInterfaceCoefficients, GAMGSolverAgglomerateMatrix.C:325-447)
__global__ void agg_patch_kernel(int nCPF, const int *__restrict__ start, const int *__restrict__ child,
                                 const double *__restrict__ fBou, const double *__restrict__ fInt,
                                 double *__restrict__ cBou, double *__restrict__ cInt)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nCPF) return;
    double b = 0.0, c = 0.0;
    for (int k = start[i]; k < start[i + 1]; k++) {
        b = __dadd_rn(b, fBou[child[k]]);
        c = __dadd_rn(c, fInt[child[k]]);
    }
    cBou[i] = b;
    cInt[i] = c;
}

// multi-rank coarsest solve: all-gather the (tiny) coarsest right-hand sides through peer
// memory -- every rank stores its part + a sequence flag into every rank's gather area -- then
// apply this rank's rows of the global inverse.  One CTA.  seqs[2] = gather sequence.
struct P2PGather {
    int rank = 0, nRanks = 1;
    double *area[P2P_MAXR] = {nullptr};
    unsigned long long *flag[P2P_MAXR] = {nullptr};
    unsigned long long *seq = nullptr;
    int counts[P2P_MAXR] = {0}, offs[P2P_MAXR + 1] = {0};
};

__global__ void dense_apply_p2p_kernel(int nLocal, int nGlobal, const double *__restrict__ invRows,
                                       const double *__restrict__ b, double *__restrict__ x, P2PGather G,
                                       const int *stop)
{
    if (stop && *stop) return;
    __shared__ double bg[P2P_MAXR * P2P_GMAX];
    const unsigned long long seq = *G.seq + 1;
    const int par = (int)(seq & 1);
    for (int i = threadIdx.x; i < nLocal * G.nRanks; i += blockDim.x) {
        int r = i / nLocal, k = i % nLocal;
        G.area[r][(size_t)(par * P2P_MAXR + G.rank) * P2P_GMAX + k] = b[k];
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < G.nRanks) {
        unsigned long long *f = G.flag[threadIdx.x] + (par * P2P_MAXR + G.rank);
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(f), "l"(seq) : "memory");
        spin_until(G.flag[G.rank] + (par * P2P_MAXR + threadIdx.x), seq, G.seq + 5); // seqs[2] + 5 = the error word seqs[7]
    }
    __syncthreads();
    for (int r = 0; r < G.nRanks; r++)
        for (int k = threadIdx.x; k < G.counts[r]; k += blockDim.x)
            bg[G.offs[r] + k] = __ldcg(G.area[G.rank] + (size_t)(par * P2P_MAXR + r) * P2P_GMAX + k);
    __syncthreads();
    for (int i = threadIdx.x; i < nLocal; i += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < nGlobal; j++) s += invRows[(size_t)i * nGlobal + j] * bg[j];
        x[i] = s;
    }
    if (threadIdx.x == 0) *G.seq = seq;
}

// NCCL fallback: gathered right-hand sides arrive padded to P2P_GMAX per rank
__global__ void dense_apply_gathered_kernel(int nLocal, int nGlobal, int nRanks, const double *__restrict__ invRows,
                                            const double *__restrict__ gathered, const int *__restrict__ offs,
                                            const int *__restrict__ counts, double *__restrict__ x, const int *stop)
{
    if (stop && *stop) return;
    __shared__ double bg[P2P_MAXR * P2P_GMAX];
    for (int r = 0; r < nRanks; r++)
        for (int k = threadIdx.x; k < counts[r]; k += blockDim.x) bg[offs[r] + k] = gathered[(size_t)r * P2P_GMAX + k];
    __syncthreads();
    for (int i = threadIdx.x; i < nLocal; i += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < nGlobal; j++) s += invRows[(size_t)i * nGlobal + j] * bg[j];
        x[i] = s;
    }
}

// x = Ainv * b for the coarsest level (one CTA; row-major inverse, fixed order)
__global__ void dense_apply_kernel(int n, const double *__restrict__ inv, const double *__restrict__ b,
                                   double *__restrict__ x, const int *stop)
{
    if (stop && *stop) return;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < n; j++) s += inv[(size_t)i * n + j] * b[j];
        x[i] = s;
    }
}

#define LAUNCH1D(kernel, n, st, ...)                                      \
    do {                                                                  \
        if ((n) > 0) {                                                    \
            kernel<<<((n) + 255) / 256, 256, 0, st>>>(__VA_ARGS__);       \
            S.ctx->launches++;                                            \
        }                                                                 \
    } while (0)

// ---------------------------------------------------------------------------
// solve
// ---------------------------------------------------------------------------
namespace {

struct LevelView { // uniform access to the finest matrix (-1) and coarse level k
    b200ldu_matrix *m;
};

int smooth_in_place(Solve &S, b200ldu_matrix *m, double omega, DevBuf<double> &x, DevBuf<double> &spare,
                    const double *b, int nSweeps, const int *stop)
{
    for (int s = 0; s < nSweeps; s++) {
        TRY(mat_jacobi(m, omega, x.get(), b, spare.get(), stop));
        std::swap(x, spare);
    }
    return B200LDU_OK;
}

// GAMGSolver::scale (GAMGSolverScale.C:59-171); field updated in place
int gamg_scale(Solve &S, b200ldu_matrix *m, double *field, double *Acf, const double *source, const int *stop)
{
    SolverScalars *sc = S.sc;
    TRY(mat_amul(m, false, field, Acf, 2, source, m->d_partials.get(), stop));
    TRY(scalar_step_on<2>(S, m->d_partials.get(), m->a->L.nBands, [=] __device__(SolverScalars *s) {
        double den = s->sum[1];
        double sden = den >= 0 ? den + VSMALL_ : den - VSMALL_; // stabilise(y, VSMALL)
        s->alpha = s->sum[0] / sden;
    }));
    const double *D = m->d_diag.get();
    return ew_launch<0>(S.ctx, m->a->L.nPad / 2, stop, nullptr, nullptr, [=] __device__(int i, double *) {
        double sf = sc->alpha;
        double2 f = CV2(field)[i], a = CV2(Acf)[i], b = CV2(source)[i], d = CV2(D)[i];
        f.x = __dadd_rn(__dmul_rn(sf, f.x), __ddiv_rn(__dsub_rn(b.x, __dmul_rn(sf, a.x)), d.x));
        f.y = __dadd_rn(__dmul_rn(sf, f.y), __ddiv_rn(__dsub_rn(b.y, __dmul_rn(sf, a.y)), d.y));
        V2(field)[i] = f;
    });
}

} // namespace

// rebuilds every coarse matrix from the current finest coefficients (GAMGSolver.C:85-96:
// done at every solver construction, i.e. every solve; only the agglomeration is cached)
static int gamg_build_matrices(Solve &S, b200ldu_gamg *g)
{
    b200ldu_matrix *fm = S.m;
    cudaStream_t st = S.ctx->stream;
    const double *fd = fm->diag_ext, *fu = fm->upper_ext, *fl = fm->symmetric ? nullptr : fm->lower_ext;
    const double *fb = fm->bou_ext, *fi = fm->int_ext;
    if (!fd || !fu) {
        b200_set_error("GAMG: matrix coefficients not set");
        return B200LDU_EINVAL;
    }
    for (int k = 0; k < g->nLevels; k++) {
        GamgLevel &L = g->lev[k];
        LAUNCH1D(agg_diag_kernel, L.nCoarse, st, L.nCoarse, L.d_cellChildStart.get(), L.d_cellChild.get(),
                 L.d_diagFaceStart.get(), L.d_diagFace.get(), fd, fu, fl, L.d_diag.get());
        LAUNCH1D(agg_faces_kernel, L.nCoarseFaces, st, L.nCoarseFaces, L.d_faceChildStart.get(), L.d_faceChild.get(),
                 fu, fl, L.d_upper.get(), L.d_lower.get());
        if (L.nCoarsePF > 0) {
            LAUNCH1D(agg_patch_kernel, L.nCoarsePF, st, L.nCoarsePF, L.d_pfChildStart.get(), L.d_pfChild.get(), fb, fi,
                     L.d_bou.get(), L.d_int.get());
        }
        KERNEL_CHECK();
        // identical boundary/internal interface coefficients on the finest level stay identical
        const double *cInt = (fm->bou_ext == fm->int_ext) ? L.d_bou.get() : L.d_int.get();
        TRY(b200ldu_matrix_set(L.mat.get(), L.d_diag.get(), L.d_upper.get(), fl ? L.d_lower.get() : nullptr,
                               L.nCoarsePF > 0 ? L.d_bou.get() : nullptr, L.nCoarsePF > 0 ? cInt : nullptr));
        fb = L.d_bou.get();
        fi = L.d_int.get();
        fd = L.d_diag.get();
        fu = L.d_upper.get();
        fl = fl ? L.d_lower.get() : nullptr;
    }
    return B200LDU_OK;
}

// Inverse of the coarsest matrix on the host (partial-pivot Gauss-Jordan), standing in for
// LUscalarMatrix (GAMGSolver.C:144-172).  Single rank: the local matrix in banded order.
// Multi rank: every rank contributes its rows of the global matrix (local coefficients +
// processor-interface coefficients at the neighbour's global column, LUscalarMatrix.C:201-270),
// all rows are all-gathered, every rank inverts the same matrix and keeps its own rows.
static int gamg_coarsest_inverse(Solve &S, b200ldu_gamg *g)
{
    GamgLevel &L = g->lev[g->nLevels - 1];
    b200ldu_ctx *ctx = S.ctx;
    const int R = ctx->nRanks;
    int n = L.nCoarse, nf = L.nCoarseFaces, npf = L.nCoarsePF;
    bool asym = !S.m->symmetric;
    std::vector<double> d(std::max(n, 1)), u(std::max(nf, 1)), l(std::max(nf, 1)), bou(std::max(npf, 1));
    cudaStream_t st = ctx->stream;
    CUDA_TRY(cudaMemcpyAsync(d.data(), L.d_diag.get(), sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    if (nf) CUDA_TRY(cudaMemcpyAsync(u.data(), L.d_upper.get(), sizeof(double) * nf, cudaMemcpyDeviceToHost, st));
    if (nf && asym) CUDA_TRY(cudaMemcpyAsync(l.data(), L.d_lower.get(), sizeof(double) * nf, cudaMemcpyDeviceToHost, st));
    if (npf) CUDA_TRY(cudaMemcpyAsync(bou.data(), L.d_bou.get(), sizeof(double) * npf, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (!asym) l = u;
    const std::vector<int> &perm = L.addr->perm_h;
    // global numbering: rank offset + banded row (the solve kernel works on banded vectors)
    const int me = ctx->rank;
    const int N = R > 1 ? g->coarsestOffs[R] : n;
    const int off = R > 1 ? g->coarsestOffs[me] : 0;
    const int nMax = R > 1 ? g->nMaxCoarsest : n;
    std::vector<double> rows((size_t)std::max(nMax, 1) * N, 0.0);
    for (int c = 0; c < n; c++) rows[(size_t)perm[c] * N + off + perm[c]] = d[c];
    for (int f = 0; f < nf; f++) {
        int o = perm[L.addr->l[f]], nb = perm[L.addr->u[f]];
        rows[(size_t)o * N + off + nb] += u[f];
        rows[(size_t)nb * N + off + o] += l[f];
    }
    std::vector<double> A;
    if (L.addr->nPatches) {
        // coupled patches: the coefficient sits at the neighbour cell's column -- another rank's block for a
        // processor patch (LUscalarMatrix.C:201-270), this rank's own for a cyclic pair.  The neighbour's banded
        // numbering is not known here: the neighbour-side cell index was exchanged in caller order, so all ranks
        // also gather their perm to translate columns
        std::vector<double> permD((size_t)std::max(nMax, 1), -1.0), permAll((size_t)std::max(nMax, 1) * R);
        for (int c = 0; c < n; c++) permD[c] = perm[c];
        TRY(comm_allgather_host(ctx, permD.data(), std::max(nMax, 1), permAll.data()));
        for (int p = 0; p < L.addr->nPatches; p++) {
            const int nbr = L.addr->neighbRank[p] >= 0 ? L.addr->neighbRank[p] : me;
            const int nbrOff = R > 1 ? g->coarsestOffs[nbr] : 0;
            for (int i = L.cPatchStart[p]; i < L.cPatchStart[p + 1]; i++) {
                int row = perm[L.cFaceCells[i]];
                int col = nbrOff + (int)permAll[(size_t)nbr * std::max(nMax, 1) + g->coarsestNbrCell[i]];
                rows[(size_t)row * N + col] -= bou[i];
            }
        }
    }
    if (R > 1) {
        std::vector<double> all((size_t)R * nMax * N);
        TRY(comm_allgather_host(ctx, rows.data(), nMax * N, all.data()));
        A.assign((size_t)N * N, 0.0);
        for (int r = 0; r < R; r++)
            for (int i = 0; i < g->coarsestCounts[r]; i++)
                memcpy(&A[(size_t)(g->coarsestOffs[r] + i) * N], &all[((size_t)r * nMax + i) * N], sizeof(double) * N);
    } else
        A = rows;
    std::vector<double> I((size_t)N * N, 0.0);
    for (int c = 0; c < N; c++) I[(size_t)c * N + c] = 1.0;
    for (int k = 0; k < N; k++) {
        int p = k;
        double mx = fabs(A[(size_t)k * N + k]);
        for (int i = k + 1; i < N; i++)
            if (fabs(A[(size_t)i * N + k]) > mx) {
                mx = fabs(A[(size_t)i * N + k]);
                p = i;
            }
        if (mx == 0.0) {
            b200_set_error("GAMG: coarsest-level matrix is singular");
            return B200LDU_EINVAL;
        }
        if (p != k)
            for (int j = 0; j < N; j++) {
                std::swap(A[(size_t)k * N + j], A[(size_t)p * N + j]);
                std::swap(I[(size_t)k * N + j], I[(size_t)p * N + j]);
            }
        double piv = 1.0 / A[(size_t)k * N + k];
        for (int j = 0; j < N; j++) {
            A[(size_t)k * N + j] *= piv;
            I[(size_t)k * N + j] *= piv;
        }
        for (int i = 0; i < N; i++) {
            if (i == k) continue;
            double fct = A[(size_t)i * N + k];
            if (fct == 0.0) continue;
            for (int j = 0; j < N; j++) {
                A[(size_t)i * N + j] -= fct * A[(size_t)k * N + j];
                I[(size_t)i * N + j] -= fct * I[(size_t)k * N + j];
            }
        }
    }
    TRY(g->d_inv.grow((size_t)std::max(n, 1) * N));
    g->invN = N;
    CUDA_TRY(cudaMemcpyAsync(g->d_inv.get(), &I[(size_t)off * N], sizeof(double) * (size_t)n * N, cudaMemcpyHostToDevice, st));
    if (R > 1 && !ctx->p2p) // R + 1 gather rows, then 64 ints of offsets and counts
        TRY(g->d_gatherAll.grow((size_t)(R + 1) * P2P_GMAX + sizeof(int) * 64 / sizeof(double)));
    CUDA_TRY(cudaStreamSynchronize(st)); // I goes out of scope
    return B200LDU_OK;
}

template <class Body>
int run_iterations(Solve &S, long long maxBodies, Body body); // solvers.cu
int init_residual(Solve &S, const double *psi, const double *b, const double *wA, double *rA, double *tmp,
                  const double *wT, double *rT); // solvers.cu
int gamg_run_cycles(Solve &S, long long maxBodies, int (*body)(void *), void *arg); // solvers.cu

struct CycleArgs {
    Solve *S;
    b200ldu_gamg *g;
    int scaleCorrection;
    double *psiBuf[2];
    long long finestSweeps;
    double *Apsi, *finestCorr, *finestRes;
};

static int gamg_cycle(void *vp)
{
    CycleArgs &A = *(CycleArgs *)vp;
    Solve &S = *A.S;
    b200ldu_gamg *g = A.g;
    const b200ldu_controls &c = S.c;
    SolverScalars *sc = S.sc;
    double *hist = S.hist;
    const int *stop = &sc->stop;
    cudaStream_t st = S.ctx->stream;
    b200ldu_matrix *fm = S.m;
    const int nL = g->nLevels, coarsest = nL - 1;
    const double omega = c.omega;
    auto imin = [](int a, int b) { return a < b ? a : b; };

    // ---- Vcycle (GAMGSolverSolve.C:181-474) ----
    {
        GamgLevel &L0 = g->lev[0];
        LAUNCH1D(restrict_kernel, L0.nCoarse, st, L0.nCoarse, L0.d_childStart.get(), L0.d_child.get(), A.finestRes, L0.src.get(), stop);
    }
    for (int k = 0; k < coarsest; k++) {
        GamgLevel &L = g->lev[k], &Ln = g->lev[k + 1];
        if (c.nPreSweeps) {
            CUDA_TRY(cudaMemsetAsync(L.corr.get(), 0, sizeof(double) * (size_t)L.addr->vecLen, st));
            TRY(smooth_in_place(S, L.mat.get(), omega, L.corr, L.tmp, L.src.get(),
                                imin(c.nPreSweeps + c.preSweepsLevelMultiplier * k, c.maxPreSweeps), stop));
            if (A.scaleCorrection && k < coarsest - 1) TRY(gamg_scale(S, L.mat.get(), L.corr.get(), L.acf.get(), L.src.get(), stop));
            TRY(mat_amul(L.mat.get(), false, L.corr.get(), L.acf.get(), 0, nullptr, nullptr, stop));
            double *src = L.src.get(), *acf = L.acf.get();
            TRY(ew_launch<0>(S.ctx, L.addr->L.nPad / 2, stop, nullptr, nullptr, [=] __device__(int i, double *) {
                double2 s2 = CV2(src)[i], a2 = CV2(acf)[i];
                V2(src)[i] = make_double2(__dsub_rn(s2.x, a2.x), __dsub_rn(s2.y, a2.y));
            }));
        }
        LAUNCH1D(restrict_kernel, Ln.nCoarse, st, Ln.nCoarse, Ln.d_childStart.get(), Ln.d_child.get(), L.src.get(), Ln.src.get(), stop);
    }
    { // solveCoarsestLevel :552-619
        GamgLevel &L = g->lev[coarsest];
        if (c.directSolveCoarsest) {
            if (S.ctx->nRanks == 1) {
                dense_apply_kernel<<<1, 256, 0, st>>>(L.nCoarse, g->d_inv.get(), L.src.get(), L.corr.get(), stop);
            } else if (S.ctx->p2p) {
                P2PGather G;
                G.rank = S.ctx->rank;
                G.nRanks = S.ctx->nRanks;
                for (int r = 0; r < G.nRanks; r++) {
                    G.area[r] = (double *)(S.ctx->peerRegion[r] + P2P_GATHER_OFF);
                    G.flag[r] = (unsigned long long *)(S.ctx->peerRegion[r] + P2P_GFLAG_OFF);
                    G.counts[r] = g->coarsestCounts[r];
                    G.offs[r] = g->coarsestOffs[r];
                }
                G.offs[G.nRanks] = g->coarsestOffs[G.nRanks];
                G.seq = S.ctx->d_seq.get() + 2;
                dense_apply_p2p_kernel<<<1, 256, 0, st>>>(L.nCoarse, g->invN, g->d_inv.get(), L.src.get(), L.corr.get(), G, stop);
            } else {
                // NCCL fallback: pad to P2P_GMAX per rank, all-gather, apply
                double *mine = g->d_gatherAll.get() + (size_t)S.ctx->nRanks * P2P_GMAX;
                CUDA_TRY(cudaMemsetAsync(mine, 0, sizeof(double) * P2P_GMAX, st));
                CUDA_TRY(cudaMemcpyAsync(mine, L.src.get(), sizeof(double) * L.nCoarse, cudaMemcpyDeviceToDevice, st));
                TRY(comm_allgather_dev(S.ctx, mine, P2P_GMAX, g->d_gatherAll.get()));
                int *meta = (int *)(g->d_gatherAll.get() + (size_t)(S.ctx->nRanks + 1) * P2P_GMAX);
                if (!g->metaUploaded) {
                    std::vector<int> h(64, 0);
                    for (int r = 0; r <= S.ctx->nRanks; r++) h[r] = g->coarsestOffs[r];
                    for (int r = 0; r < S.ctx->nRanks; r++) h[32 + r] = g->coarsestCounts[r];
                    CUDA_TRY(cudaMemcpyAsync(meta, h.data(), sizeof(int) * 64, cudaMemcpyHostToDevice, st));
                    CUDA_TRY(cudaStreamSynchronize(st));
                    g->metaUploaded = true;
                }
                dense_apply_gathered_kernel<<<1, 256, 0, st>>>(L.nCoarse, g->invN, S.ctx->nRanks, g->d_inv.get(),
                                                                g->d_gatherAll.get(), meta, meta + 32, L.corr.get(), stop);
            }
            S.ctx->launches++;
        } else {
            // ICCG / BICCG to the GAMG tolerances, from a zero correction (:568-606).  The nested
            // solve decides its own iteration count, so this mode runs cycle by cycle (no graph;
            // gamg_solve sets checkEvery = 1): skip the work once the outer solve has stopped.
            int stopped = 0;
            CUDA_TRY(cudaMemcpyAsync(&stopped, stop, sizeof(int), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            if (!stopped) {
                CUDA_TRY(cudaMemsetAsync(L.corr.get(), 0, sizeof(double) * (size_t)L.addr->vecLen, st));
                b200ldu_controls cc;
                b200ldu_controls_default(&cc);
                cc.tolerance = c.tolerance;
                cc.relTol = c.relTol;
                b200ldu_perf cp;
                double *res = nullptr;
                TRY(solve_banded(L.mat.get(), L.mat->symmetric ? "ICCG" : "BICCG", nullptr, &cc, nullptr, L.corr.get(),
                                 L.src.get(), &cp, nullptr, 0, &res));
                if (res != L.corr.get())
                    CUDA_TRY(cudaMemcpyAsync(L.corr.get(), res, sizeof(double) * (size_t)L.addr->vecLen,
                                             cudaMemcpyDeviceToDevice, st));
            }
        }
    }
    for (int k = coarsest - 1; k >= 0; k--) {
        GamgLevel &L = g->lev[k], &Ln = g->lev[k + 1];
        int nPadL = L.addr->L.nPad;
        if (c.nPreSweeps)
            CUDA_TRY(cudaMemcpyAsync(L.pre.get(), L.corr.get(), sizeof(double) * (size_t)L.addr->vecLen, cudaMemcpyDeviceToDevice, st));
        LAUNCH1D(prolong_kernel, nPadL, st, nPadL, Ln.d_pmap.get(), Ln.corr.get(), L.corr.get(), stop);
        if (c.interpolateCorrection) {
            TRY(mat_interpolate(L.mat.get(), L.corr.get(), L.tmp.get(), stop));
            std::swap(L.corr, L.tmp);
        }
        if (A.scaleCorrection && (c.interpolateCorrection || k < coarsest - 1))
            TRY(gamg_scale(S, L.mat.get(), L.corr.get(), L.acf.get(), L.src.get(), stop));
        if (c.nPreSweeps) {
            double *corr = L.corr.get(), *pre = L.pre.get();
            TRY(ew_launch<0>(S.ctx, nPadL / 2, stop, nullptr, nullptr, [=] __device__(int i, double *) {
                double2 a2 = CV2(corr)[i], p2 = CV2(pre)[i];
                V2(corr)[i] = make_double2(__dadd_rn(a2.x, p2.x), __dadd_rn(a2.y, p2.y));
            }));
        }
        TRY(smooth_in_place(S, L.mat.get(), omega, L.corr, L.tmp, L.src.get(),
                            imin(c.nPostSweeps + c.postSweepsLevelMultiplier * k, c.maxPostSweeps), stop));
    }
    {
        GamgLevel &L0 = g->lev[0];
        int nPadF = fm->a->L.nPad;
        LAUNCH1D(prolong_kernel, nPadF, st, nPadF, L0.d_pmap.get(), L0.corr.get(), A.finestCorr, stop);
        KERNEL_CHECK();
    }
    double *psi = A.psiBuf[A.finestSweeps & 1], *spare = A.psiBuf[(A.finestSweeps + 1) & 1];
    if (c.interpolateCorrection) {
        TRY(mat_interpolate(fm, A.finestCorr, A.Apsi, stop));
        std::swap(A.finestCorr, A.Apsi);
    }
    if (A.scaleCorrection) TRY(gamg_scale(S, fm, A.finestCorr, A.Apsi, A.finestRes, stop));
    {
        double *fc = A.finestCorr;
        TRY(ew_launch<0>(S.ctx, fm->a->L.nPad / 2, stop, nullptr, nullptr, [=] __device__(int i, double *) {
            double2 p2 = CV2(psi)[i], c2 = CV2(fc)[i];
            V2(psi)[i] = make_double2(__dadd_rn(p2.x, c2.x), __dadd_rn(p2.y, c2.y));
        }));
    }
    for (int s = 0; s < c.nFinestSweeps; s++) {
        TRY(mat_jacobi(fm, omega, psi, S.src, spare, stop));
        std::swap(psi, spare);
        A.finestSweeps++;
    }
    // ---- finest residual + convergence (:146-175) ----
    TRY(mat_amul(fm, false, psi, A.Apsi, 0, nullptr, nullptr, stop));
    int np = 0;
    {
        const double *b = S.src, *Ap = A.Apsi;
        double *fr = A.finestRes;
        TRY(ew_launch<1>(S.ctx, fm->a->L.nPad / 2, stop, S.partials, &np, [=] __device__(int i, double *red) {
            double2 b2 = CV2(b)[i], a2 = CV2(Ap)[i];
            double2 r = make_double2(__dsub_rn(b2.x, a2.x), __dsub_rn(b2.y, a2.y));
            V2(fr)[i] = r;
            red[0] += fabs(r.x) + fabs(r.y);
        }));
    }
    TRY(scalar_step<1>(S, np, [=] __device__(SolverScalars *s) {
        s->finalResidual = s->sum[0] / s->normFactor;
        hist_put(s, hist, s->nIterations + 1, s->finalResidual);
        bool conv = check_convergence(s);
        s->nIterations++; // (++nIterations < maxIter && !conv) || nIterations < minIter  (:166-175)
        bool cont = (s->nIterations < s->maxIter && !conv) || s->nIterations < s->minIter;
        if (!cont) s->stop = 1;
    }));
    return B200LDU_OK;
}

int gamg_solve(Solve &S, b200ldu_gamg *g, const char *smoother)
{
    (void)smoother; // validated by the caller; Jacobi is the only smoother (GaussSeidel aliases to it)
    if (!g || g->nLevels == 0) {
        b200_set_error("GAMG: No coarse levels created, either matrix too small for GAMG or "
                       "nCellsInCoarsestLevel too large (GAMGSolver.C:174-192)");
        return B200LDU_ENOLEVELS;
    }
    if (g->finest != S.m->a) {
        b200_set_error("GAMG: agglomeration was built for a different addressing");
        return B200LDU_EINVAL;
    }
    b200ldu_matrix *fm = S.m;
    CycleArgs A;
    A.S = &S;
    A.g = g;
    A.scaleCorrection = S.c.scaleCorrection < 0 ? (fm->symmetric ? 1 : 0) : S.c.scaleCorrection;
    A.psiBuf[0] = S.psi;
    A.psiBuf[1] = S.vec(0);
    A.Apsi = S.vec(1);
    A.finestCorr = S.vec(2);
    A.finestRes = S.vec(3);
    A.finestSweeps = 0;
    if (!A.psiBuf[1] || !A.Apsi || !A.finestCorr || !A.finestRes) return B200LDU_ECUDA;

    TRY(gamg_build_matrices(S, g));
    if (S.c.directSolveCoarsest) {
        TRY(gamg_coarsest_inverse(S, g));
    } else {
        S.useGraph = false; // the coarsest-level Krylov solve synchronises with the host
        S.c.checkEvery = 1;
    }
    TRY(mat_amul(fm, false, S.psi, A.Apsi, 0, nullptr, nullptr, nullptr));
    TRY(init_residual(S, S.psi, S.src, A.Apsi, A.finestRes, A.finestCorr, nullptr, nullptr));
    long long maxBodies = S.c.maxIter > S.c.minIter ? S.c.maxIter : S.c.minIter;
    if (maxBodies < 1) maxBodies = 1;
    TRY(gamg_run_cycles(S, maxBodies, gamg_cycle, &A));
    S.sweepParityUnknown = S.c.nFinestSweeps > 0;
    S.smoothBuf[0] = A.psiBuf[0];
    S.smoothBuf[1] = A.psiBuf[1];
    S.gamgFinestSweeps = S.c.nFinestSweeps;
    return B200LDU_OK;
}
