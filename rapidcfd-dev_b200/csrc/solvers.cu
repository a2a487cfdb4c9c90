// solvers.cu -- lduMatrix::solver run-time selection and the Krylov / smooth solvers,
// running entirely on the device: alpha, beta and the convergence decision live in a
// device-resident SolverScalars block, every kernel of an iteration early-exits once
// the device has decided to stop, and the host only polls that flag every few
// iterations (pipelined, so polling never drains the GPU).  The iteration count and
// residual history are therefore exactly those of the reference's host-driven loop.
//
// Reference: LDU/lduMatrix/lduMatrixSolver.C:43-236 (selection, controls, normFactor),
// LDU/solvers/PCG/PCG.C:69-208, PBiCG/PBiCG.C:68-246, PBiCGStab/PBiCGStab.C:66-300,
// smoothSolver/smoothSolver.C:77-193, diagonalSolver/diagonalSolver.C:62-81,
// LduMatrix/LduMatrix/SolverPerformance.C:32-92.
#include "ldu.h"

#include <cstdlib>

#include <algorithm>

#include "solver_steps.cuh"

// initial residual, normFactor and the first convergence test, common to all solvers
// (PCG.C:92-128; lduMatrixSolver.C:205-236).  wA must hold A.psi; tmp receives sumA.
int init_residual(Solve &S, const double *psi, const double *b, const double *wA, double *rA, double *tmp,
                  const double *wT = nullptr, double *rT = nullptr)
{
    b200ldu_addr *a = S.m->a;
    SolverScalars *sc = S.sc;
    double *hist = S.hist;
    const int n2 = a->L.nPad / 2;
    int np = 0;
    TRY(ew_launch<2>(S.ctx, n2, nullptr, S.partials, &np, [=] __device__(int i, double *red) {
        double2 bb = CV2(b)[i], ww = CV2(wA)[i], pp = CV2(psi)[i];
        double2 r = make_double2(__dsub_rn(bb.x, ww.x), __dsub_rn(bb.y, ww.y));
        V2(rA)[i] = r;
        if (rT) {
            double2 wt = CV2(wT)[i];
            V2(rT)[i] = make_double2(__dsub_rn(bb.x, wt.x), __dsub_rn(bb.y, wt.y));
        }
        red[0] += fabs(r.x) + fabs(r.y);
        red[1] += pp.x + pp.y;
    }));
    TRY(scalar_step<2>(S, np, [=] __device__(SolverScalars *s) {
        s->sumMag0 = s->sum[0];
        s->average = s->sum[1] / s->nCellsGlobal; // gAverage: gpuFieldCommonFunctions.C:611-635
    }));
    TRY(mat_sumA(S.m, tmp, nullptr));
    const int nCells = a->nCells;
    TRY(ew_launch<1>(S.ctx, n2, nullptr, S.partials, &np, [=] __device__(int i, double *red) {
        double avg = sc->average;
        double2 bb = CV2(b)[i], ww = CV2(wA)[i], tt = CV2(tmp)[i];
        double t0 = __dmul_rn(avg, tt.x), t1 = __dmul_rn(avg, tt.y);
        if (2 * i < nCells) red[0] += fabs(ww.x - t0) + fabs(bb.x - t0);
        if (2 * i + 1 < nCells) red[0] += fabs(ww.y - t1) + fabs(bb.y - t1);
    }));
    TRY(scalar_step<1>(S, np, [=] __device__(SolverScalars *s) {
        s->normFactor = s->sum[0] + SMALL_;
        s->initialResidual = s->sumMag0 / s->normFactor;
        s->finalResidual = s->initialResidual;
        hist_put(s, hist, 0, s->finalResidual);
        bool conv = check_convergence(s);
        if (!(s->minIter > 0 || !conv)) s->stop = 1;
    }));
    return B200LDU_OK;
}

// ---------------------------------------------------------------------------
// host driver: enqueue iteration bodies, poll the device stop flag (pipelined)
// ---------------------------------------------------------------------------
template <class Body>
int run_iterations(Solve &S, long long maxBodies, Body body)
{
    b200ldu_ctx *ctx = S.ctx;
    int every = S.c.checkEvery > 0 ? S.c.checkEvery : 8;
    volatile int *flags = (volatile int *)S.pinnedFlags; // two slots
    cudaEvent_t ev[2] = {S.ev[0], S.ev[1]};
    long long enq = 0;
    int chunk = 0;
    bool pending[2] = {false, false};
    cudaGraphExec_t graphExec = nullptr;
    long long launchesPerGraph = 0;
    struct GraphGuard {
        cudaGraphExec_t &g;
        ~GraphGuard()
        {
            if (g) cudaGraphExecDestroy(g);
        }
    } guard{graphExec};
    for (;;) {
        int slot = chunk & 1;
        // before reusing a slot, consume its previous result
        if (pending[slot]) {
            CUDA_TRY(cudaEventSynchronize(ev[slot]));
            pending[slot] = false;
            if (flags[slot]) break;
        }
        if (enq >= maxBodies) {
            // nothing more to enqueue: drain the other slot and leave
            int o = slot ^ 1;
            if (pending[o]) {
                CUDA_TRY(cudaEventSynchronize(ev[o]));
                pending[o] = false;
            }
            break;
        }
        // CUDA graph: after one chunk launched kernel by kernel (attribute set-up, warm caches) a full
        // chunk of `every` bodies (even, so every ping-pong returns to its starting buffers) is captured
        // once and replayed -- the device-side stop flag makes replayed bodies after convergence no-ops.
        const bool fullChunk = (enq + every <= maxBodies) && (every % 2 == 0) && (enq % 2 == 0);
        if (S.useGraph && fullChunk && chunk >= 1) {
            if (!graphExec) {
                long long l0 = ctx->launches;
                cudaGraph_t g = nullptr;
                CUDA_TRY(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed));
                int rcb = B200LDU_OK;
                for (int k = 0; k < every && rcb == B200LDU_OK; k++) rcb = body(enq + k);
                cudaError_t ce = cudaStreamEndCapture(ctx->stream, &g);
                if (rcb != B200LDU_OK) return rcb;
                if (ce != cudaSuccess || !g) {
                    b200_set_error("CUDA graph capture failed: %s", cudaGetErrorString(ce));
                    return B200LDU_ECUDA;
                }
                launchesPerGraph = ctx->launches - l0;
                ctx->launches = l0;
                CUDA_TRY(cudaGraphInstantiate(&graphExec, g, 0));
                cudaGraphDestroy(g);
            }
            CUDA_TRY(cudaGraphLaunch(graphExec, ctx->stream));
            ctx->launches += launchesPerGraph;
            enq += every;
        } else {
            for (int k = 0; k < every && enq < maxBodies; k++, enq++) TRY(body(enq));
        }
        CUDA_TRY(cudaMemcpyAsync((void *)&flags[slot], &S.sc->stop, sizeof(int), cudaMemcpyDeviceToHost,
                                 ctx->stream));
        CUDA_TRY(cudaEventRecord(ev[slot], ctx->stream));
        pending[slot] = true;
        chunk++;
    }
    return B200LDU_OK;
}

// ---------------------------------------------------------------------------
// PCG (PCG.C:69-208)
// ---------------------------------------------------------------------------
int solve_pcg(Solve &S, int pk)
{
    b200ldu_matrix *m = S.m;
    b200ldu_addr *a = m->a;
    SolverScalars *sc = S.sc;
    double *hist = S.hist;
    const int *stop = &sc->stop;
    const int n2 = a->L.nPad / 2;
    double *psi = S.psi, *b = S.src;
    double *pA = S.vec(0), *wA = S.vec(1), *rA = S.vec(2);
    if (!pA || !wA || !rA) return B200LDU_ECUDA;

    TRY(mat_amul(m, false, psi, wA, 0, nullptr, nullptr, nullptr));
    TRY(init_residual(S, psi, b, wA, rA, pA));

    auto body = [&](long long) -> int {
        int np = 0;
        // wA = M^-1 rA ; wArA = <wA, rA>
        TRY(mat_precondition(m, pk, false, rA, wA, true, nullptr, S.partials, &np, stop));
        TRY(scalar_step<1>(S, np, [=] __device__(SolverScalars *s) {
            s->wArAold = s->wArA;
            s->wArA = s->sum[0];
            s->beta = s->wArA / s->wArAold;
        }));
        // pA = wA (first) | wA + beta*pA
        TRY(ew_launch<0>(S.ctx, n2, stop, nullptr, nullptr, [=] __device__(int i, double *) {
            double2 w = CV2(wA)[i];
            if (sc->nIterations == 0) {
                V2(pA)[i] = w;
            } else {
                double beta = sc->beta;
                double2 p = CV2(pA)[i];
                V2(pA)[i] = make_double2(fma(beta, p.x, w.x), fma(beta, p.y, w.y));
            }
        }));
        // wA = A pA ; wApA = <wA, pA>
        TRY(mat_amul(m, false, pA, wA, 1, nullptr, S.partials, stop));
        TRY(scalar_step<1>(S, a->L.nBands, [=] __device__(SolverScalars *s) {
            s->wApA = s->sum[0];
            if (!(fabs(s->wApA) / s->normFactor > VSMALL_)) { // checkSingularity PCG.C:170
                s->singular = 1;
                s->stop = 1;
                return;
            }
            s->alpha = s->wArA / s->wApA;
        }));
        // psi += alpha pA ; rA -= alpha wA ; sum|rA|
        TRY(ew_launch<1>(S.ctx, n2, stop, S.partials, &np, [=] __device__(int i, double *red) {
            double alpha = sc->alpha;
            double2 x = CV2(psi)[i], p = CV2(pA)[i], r = CV2(rA)[i], w = CV2(wA)[i];
            x.x = fma(alpha, p.x, x.x);
            x.y = fma(alpha, p.y, x.y);
            r.x = fma(-alpha, w.x, r.x);
            r.y = fma(-alpha, w.y, r.y);
            V2(psi)[i] = x;
            V2(rA)[i] = r;
            red[0] += fabs(r.x) + fabs(r.y);
        }));
        TRY(scalar_step<1>(S, np, [=] __device__(SolverScalars *s) { end_of_body(s, hist, s->sum[0]); }));
        return B200LDU_OK;
    };
    return run_iterations(S, (long long)S.c.maxIter + 1 > S.c.minIter ? (long long)S.c.maxIter + 1 : S.c.minIter,
                          body);
}

// ---------------------------------------------------------------------------
// PCG, fused form: TWO launches per iteration (the reference: 8 Thrust launches + 3 host synchronisations,
// PCG.C:131-205).  Sweep A (PcgAinvOp) applies the psi/r update of the previous body while staging r,
// preconditions and reduces <z,r>, sum|r|; sweep B (PcgAmulOp) forms p = z + beta p while staging, multiplies
// and reduces <Ap,p>.  The scalar step that closes each sweep (sum of the per-band partials in fixed order,
// cross-rank all-reduce over the peer mailboxes, alpha / beta / convergence test) runs in the prologue of the
// NEXT sweep's kernel (ops.cuh DeferredStep) -- round 1 spent two one-CTA launches per iteration on it.
// Same recurrences and per-row arithmetic as solve_pcg; the convergence decision of body k is taken at the
// start of sweep B of body k+1 (the preconditioner sweep that has then already run only overwrote scratch).
// ---------------------------------------------------------------------------
// scalar step A of the fused PCG: closes body k-1 (residual, convergence: PCG.C:190-205), then beta of body k
struct PcgStepA {
    double *hist;
    __device__ void operator()(SolverScalars *s) const
    {
        if (s->bodies > 0) {
            end_of_body(s, hist, s->sum[1]);
            if (s->stop) return;
        }
        s->wArAold = s->wArA;
        s->wArA = s->sum[0];
        s->beta = s->wArA / s->wArAold;
    }
};
// scalar step B: alpha of body k (PCG.C:166-175)
struct PcgStepB {
    __device__ void operator()(SolverScalars *s) const
    {
        s->wApA = s->sum[0];
        if (!(fabs(s->wApA) / s->normFactor > VSMALL_)) { // checkSingularity PCG.C:170
            s->singular = 1;
            s->stop = 1;
            return;
        }
        s->alpha = s->wArA / s->wApA;
        s->bodies++;
    }
};

int solve_pcg_fused(Solve &S, int pk)
{
    b200ldu_matrix *m = S.m;
    b200ldu_addr *a = m->a;
    SolverScalars *sc = S.sc;
    double *hist = S.hist;
    const int *stop = &sc->stop;
    const int n2 = a->L.nPad / 2;
    double *psi = S.psi, *b = S.src;
    double *pb[2] = {S.vec(0), S.vec(4)}, *w = S.vec(1), *rb[2] = {S.vec(2), S.vec(3)}, *z = S.vec(5);
    if (!pb[0] || !pb[1] || !w || !rb[0] || !rb[1] || !z) return B200LDU_ECUDA;
    const double *rD = m->d_rD.get();
    const P2PRed pr = (S.ctx->nRanks > 1 && S.ctx->p2p) ? comm_p2p_red(S.ctx) : P2PRed();
    // the two sweeps leave their partials in separate buffers: a deferred step reads one while the sweep that
    // runs it writes the other
    double *partA = S.partials, *partB = S.partials + 2 * (size_t)(a->L.nBands > S.ctx->smCount * 8 ? a->L.nBands : S.ctx->smCount * 8);

    TRY(mat_amul(m, false, psi, w, 0, nullptr, nullptr, nullptr));
    TRY(init_residual(S, psi, b, w, rb[0], pb[0]));

    const PcgStepA gA{hist};
    const PcgStepB gB{};
    typedef DeferredStep<1, PcgStepB> PreA; // sweep A starts by closing sweep B of the previous body
    typedef DeferredStep<2, PcgStepA> PreB; // sweep B starts by closing sweep A of this body
    const int every = S.c.checkEvery > 0 ? S.c.checkEvery : 8;
    const unsigned mod = 2u * (unsigned)every;

    auto body = [&](long long k) -> int {
        const double *rOld = rb[k & 1], *pPrev = pb[k & 1];
        double *rNew = rb[(k + 1) & 1], *pNew = pb[(k + 1) & 1];
        int npA = a->L.nBands;
        const PreA preA{partB, a->L.nBands, sc, gB, pr, (unsigned)(2 * (k % every)), mod, k > 0 ? 1 : 0};
        if (pk == 2) {
            PcgAinvOp<PreA> op;
            op.stop = stop;
            op.partials = partA;
            op.rOld = rOld, op.rNew = rNew, op.w = w, op.p = pPrev, op.psi = psi, op.z = z, op.rD = m->d_rD.get();
            op.sc = sc;
            op.pre = preA;
            TRY(engine_launch_m(m, false, op));
        } else {
            // diagonal / no preconditioner: sweep A is element-wise; its deferred step runs as CTA 0's prologue too
            TRY(ew_launch<2>(S.ctx, n2, stop, partA, &npA, [=] __device__(int i, double *red) {
                double2 r = CV2(rOld)[i];
                if (sc->bodies > 0) {
                    const double alpha = sc->alpha;
                    double2 ww = CV2(w)[i], pp = CV2(pPrev)[i], x = CV2(psi)[i];
                    r.x = fma(-alpha, ww.x, r.x);
                    r.y = fma(-alpha, ww.y, r.y);
                    V2(psi)[i] = make_double2(fma(alpha, pp.x, x.x), fma(alpha, pp.y, x.y));
                }
                V2(rNew)[i] = r;
                double2 zz = r;
                if (pk == 1) {
                    double2 d = CV2(rD)[i];
                    zz = make_double2(__dmul_rn(d.x, r.x), __dmul_rn(d.y, r.y));
                }
                V2(z)[i] = zz;
                red[0] += zz.x * r.x + zz.y * r.y;
                red[1] += fabs(r.x) + fabs(r.y);
            }, preA));
        }
        int wait = 0;
        TRY(mat_halo(m, pNew, stop, &wait)); // peer-memory path: nothing is launched, the send is fused
        const PreB preB{partA, npA, sc, gA, pr, (unsigned)(2 * (k % every) + 1), mod, 1};
        PcgAmulOp<PreB> op;
        op.stop = stop;
        op.partials = partB;
        op.waitHalo = wait;
        op.z = z, op.pOld = pPrev, op.pNew = pNew, op.out = w, op.diag = m->d_diag.get();
        op.sc = sc;
        op.pre = preB;
        TRY(engine_launch_m(m, false, op));
        return B200LDU_OK;
    };
    long long mb = (long long)S.c.maxIter + 1 > S.c.minIter ? (long long)S.c.maxIter + 1 : S.c.minIter;
    TRY(run_iterations(S, mb + 1, body)); // +1: the last body's update is applied (and judged) by the next sweeps
    // the loop ends on a decision taken in a prologue (or when the bodies run out): one last scalar step closes
    // whatever sweep ran last without one -- a no-op once the stop flag is set
    return B200LDU_OK;
}

// ---------------------------------------------------------------------------
// PBiCG (PBiCG.C:68-246)
// ---------------------------------------------------------------------------
int solve_pbicg(Solve &S, int pk)
{
    b200ldu_matrix *m = S.m;
    b200ldu_addr *a = m->a;
    SolverScalars *sc = S.sc;
    double *hist = S.hist;
    const int *stop = &sc->stop;
    const int n2 = a->L.nPad / 2;
    double *psi = S.psi, *b = S.src;
    double *pA = S.vec(0), *wA = S.vec(1), *rA = S.vec(2), *pT = S.vec(3), *wT = S.vec(4), *rT = S.vec(5);
    if (!pA || !wA || !rA || !pT || !wT || !rT) return B200LDU_ECUDA;
    CUDA_TRY(cudaMemsetAsync(pT, 0, sizeof(double) * (size_t)a->vecLen, S.ctx->stream)); // pT = 0 :86

    TRY(mat_amul(m, false, psi, wA, 0, nullptr, nullptr, nullptr));
    TRY(mat_amul(m, true, psi, wT, 0, nullptr, nullptr, nullptr));
    TRY(init_residual(S, psi, b, wA, rA, pA, wT, rT));

    auto body = [&](long long) -> int {
        int np = 0;
        TRY(mat_precondition(m, pk, true, rT, wT, false, nullptr, nullptr, nullptr, stop));
        TRY(mat_precondition(m, pk, false, rA, wA, true, rT, S.partials, &np, stop)); // wArT = <wA, rT>
        TRY(scalar_step<1>(S, np, [=] __device__(SolverScalars *s) {
            s->wArAold = s->wArA;
            s->wArA = s->sum[0];
            s->beta = s->wArA / s->wArAold;
        }));
        TRY(ew_launch<0>(S.ctx, n2, stop, nullptr, nullptr, [=] __device__(int i, double *) {
            double2 w = CV2(wA)[i], wt = CV2(wT)[i];
            if (sc->nIterations == 0) {
                V2(pA)[i] = w;
                V2(pT)[i] = wt;
            } else {
                double beta = sc->beta;
                double2 p = CV2(pA)[i], pt = CV2(pT)[i];
                V2(pA)[i] = make_double2(fma(beta, p.x, w.x), fma(beta, p.y, w.y));
                V2(pT)[i] = make_double2(fma(beta, pt.x, wt.x), fma(beta, pt.y, wt.y));
            }
        }));
        TRY(mat_amul(m, true, pT, wT, 0, nullptr, nullptr, stop));
        TRY(mat_amul(m, false, pA, wA, 3, pT, S.partials, stop)); // wApT = <wA, pT>
        TRY(scalar_step<1>(S, a->L.nBands, [=] __device__(SolverScalars *s) {
            s->wApA = s->sum[0];
            if (!(fabs(s->wApA) / s->normFactor > VSMALL_)) {
                s->singular = 1;
                s->stop = 1;
                return;
            }
            s->alpha = s->wArA / s->wApA;
        }));
        TRY(ew_launch<1>(S.ctx, n2, stop, S.partials, &np, [=] __device__(int i, double *red) {
            double alpha = sc->alpha;
            double2 x = CV2(psi)[i], p = CV2(pA)[i], r = CV2(rA)[i], w = CV2(wA)[i];
            double2 rt = CV2(rT)[i], wt = CV2(wT)[i];
            x.x = fma(alpha, p.x, x.x);
            x.y = fma(alpha, p.y, x.y);
            r.x = fma(-alpha, w.x, r.x);
            r.y = fma(-alpha, w.y, r.y);
            rt.x = fma(-alpha, wt.x, rt.x);
            rt.y = fma(-alpha, wt.y, rt.y);
            V2(psi)[i] = x;
            V2(rA)[i] = r;
            V2(rT)[i] = rt;
            red[0] += fabs(r.x) + fabs(r.y);
        }));
        TRY(scalar_step<1>(S, np, [=] __device__(SolverScalars *s) { end_of_body(s, hist, s->sum[0]); }));
        return B200LDU_OK;
    };
    return run_iterations(S, (long long)S.c.maxIter + 1 > S.c.minIter ? (long long)S.c.maxIter + 1 : S.c.minIter,
                          body);
}

// ---------------------------------------------------------------------------
// PBiCGStab (PBiCGStab.C:66-300)
// ---------------------------------------------------------------------------
int solve_pbicgstab(Solve &S, int pk)
{
    b200ldu_matrix *m = S.m;
    b200ldu_addr *a = m->a;
    SolverScalars *sc = S.sc;
    double *hist = S.hist;
    const int *stop = &sc->stop;
    const int n2 = a->L.nPad / 2;
    const int quirk = S.c.bicgstabRefQuirk;
    double *psi = S.psi, *b = S.src;
    double *pA = S.vec(0), *yA = S.vec(1), *rA = S.vec(2), *AyA = S.vec(3), *sA = S.vec(4), *zA = S.vec(5),
           *tA = S.vec(6), *rA0 = S.vec(7);
    if (!pA || !yA || !rA || !AyA || !sA || !zA || !tA || !rA0) return B200LDU_ECUDA;

    TRY(mat_amul(m, false, psi, yA, 0, nullptr, nullptr, nullptr));
    TRY(init_residual(S, psi, b, yA, rA, pA));
    CUDA_TRY(cudaMemcpyAsync(rA0, rA, sizeof(double) * (size_t)a->vecLen, cudaMemcpyDeviceToDevice,
                             S.ctx->stream)); // rA0 = rA :127

    auto body = [&](long long) -> int {
        int np = 0;
        // rA0rA = <rA0, rA>
        TRY(ew_launch<1>(S.ctx, n2, stop, S.partials, &np, [=] __device__(int i, double *red) {
            double2 x = CV2(rA0)[i], y = CV2(rA)[i];
            red[0] += x.x * y.x + x.y * y.y;
        }));
        TRY(scalar_step<1>(S, np, [=] __device__(SolverScalars *s) {
            s->rA0rAold = s->rA0rA;
            s->rA0rA = s->sum[0];
            if (!(fabs(s->rA0rA) > VSMALL_)) { // :141-144
                s->singular = 1;
                s->stop = 1;
                return;
            }
            if (s->nIterations > 0) {
                if (!(fabs(s->omega) > VSMALL_)) { // :153-156
                    s->singular = 1;
                    s->stop = 1;
                    return;
                }
                s->beta = (s->rA0rA / s->rA0rAold) * (s->alpha / s->omega);
            }
        }));
        // pA = rA (first) | rA + beta*(pA - omega*AyA)
        TRY(ew_launch<0>(S.ctx, n2, stop, nullptr, nullptr, [=] __device__(int i, double *) {
            double2 r = CV2(rA)[i];
            if (sc->nIterations == 0) {
                V2(pA)[i] = r;
            } else {
                double beta = sc->beta, omega = sc->omega;
                double2 p = CV2(pA)[i], ay = CV2(AyA)[i];
                double r1x = fma(-omega, ay.x, p.x), r1y = fma(-omega, ay.y, p.y);
                V2(pA)[i] = make_double2(fma(beta, r1x, r.x), fma(beta, r1y, r.y));
            }
        }));
        TRY(mat_precondition(m, pk, false, pA, yA, false, nullptr, nullptr, nullptr, stop));
        TRY(mat_amul(m, false, yA, AyA, 3, rA0, S.partials, stop)); // rA0AyA
        TRY(scalar_step<1>(S, a->L.nBands, [=] __device__(SolverScalars *s) { s->alpha = s->rA0rA / s->sum[0]; }));
        // sA = rA - alpha*AyA ; psi += alpha*yA (both exits of the body need it) ; sum|sA|
        TRY(ew_launch<1>(S.ctx, n2, stop, S.partials, &np, [=] __device__(int i, double *red) {
            double alpha = sc->alpha;
            double2 r = CV2(rA)[i], ay = CV2(AyA)[i], x = CV2(psi)[i], y = CV2(yA)[i];
            double2 s2 = make_double2(fma(-alpha, ay.x, r.x), fma(-alpha, ay.y, r.y));
            V2(sA)[i] = s2;
            V2(psi)[i] = make_double2(fma(alpha, y.x, x.x), fma(alpha, y.y, x.y));
            red[0] += fabs(s2.x) + fabs(s2.y);
        }));
        TRY(scalar_step<1>(S, np, [=] __device__(SolverScalars *s) {
            s->finalResidual = s->sum[0] / s->normFactor;
            if (check_convergence(s)) { // early return :198-213
                s->nIterations++;
                hist_put(s, hist, s->nIterations, s->finalResidual);
                s->stop = 1;
            }
        }));
        TRY(mat_precondition(m, pk, false, sA, zA, false, nullptr, nullptr, nullptr, stop));
        TRY(mat_amul(m, false, zA, tA, 4, sA, S.partials, stop)); // tAtA, tAsA
        TRY(scalar_step<2>(S, a->L.nBands, [=] __device__(SolverScalars *s) { s->omega = s->sum[1] / s->sum[0]; }));
        TRY(ew_launch<1>(S.ctx, n2, stop, S.partials, &np, [=] __device__(int i, double *red) {
            double omega = sc->omega;
            const double *second = quirk ? yA : zA; // PBiCGStab.C:263-270 passes yA
            double2 x = CV2(psi)[i], z = CV2(second)[i], s2 = CV2(sA)[i], t = CV2(tA)[i];
            V2(psi)[i] = make_double2(fma(omega, z.x, x.x), fma(omega, z.y, x.y));
            double2 r = make_double2(fma(-omega, t.x, s2.x), fma(-omega, t.y, s2.y));
            V2(rA)[i] = r;
            red[0] += fabs(r.x) + fabs(r.y);
        }));
        TRY(scalar_step<1>(S, np, [=] __device__(SolverScalars *s) { end_of_body(s, hist, s->sum[0]); }));
        return B200LDU_OK;
    };
    return run_iterations(S, (long long)S.c.maxIter + 1 > S.c.minIter ? (long long)S.c.maxIter + 1 : S.c.minIter,
                          body);
}

// ---------------------------------------------------------------------------
// smoothSolver (smoothSolver.C:77-193) with the Jacobi smoother
// ---------------------------------------------------------------------------
int solve_smooth(Solve &S)
{
    b200ldu_matrix *m = S.m;
    b200ldu_addr *a = m->a;
    SolverScalars *sc = S.sc;
    double *hist = S.hist;
    const int *stop = &sc->stop;
    double *b = S.src;
    double *buf[2] = {S.psi, S.vec(0)};
    double *tmp = S.vec(1), *Apsi = S.vec(2);
    if (!buf[1] || !tmp || !Apsi) return B200LDU_ECUDA;
    const double omega = S.c.omega;
    long long sweepsDone = 0;

    if (S.c.nSweeps < 0) { // fixed number of sweeps, no residual evaluation (:88-110)
        int ns = -S.c.nSweeps;
        for (int s = 0; s < ns; s++, sweepsDone++)
            TRY(mat_jacobi(m, omega, buf[sweepsDone & 1], b, buf[(sweepsDone + 1) & 1], nullptr));
        S.resultBuf = buf[sweepsDone & 1];
        S.fixedSweeps = ns;
        return B200LDU_OK;
    }
    TRY(mat_amul(m, false, S.psi, Apsi, 0, nullptr, nullptr, nullptr));
    TRY(init_residual(S, S.psi, b, Apsi, tmp, buf[1]));
    const int nSweeps = S.c.nSweeps;
    auto body = [&](long long) -> int {
        for (int s = 0; s < nSweeps; s++, sweepsDone++)
            TRY(mat_jacobi(m, omega, buf[sweepsDone & 1], b, buf[(sweepsDone + 1) & 1], stop));
        TRY(mat_residual(m, buf[sweepsDone & 1], b, tmp, true, S.partials, stop));
        TRY(scalar_step<1>(S, a->L.nBands, [=] __device__(SolverScalars *s) {
            s->finalResidual = s->sum[0] / s->normFactor;
            int k = s->nIterations / (nSweeps > 0 ? nSweeps : 1) + 1;
            hist_put(s, hist, k, s->finalResidual);
            bool conv = check_convergence(s);
            s->nIterations += nSweeps; // ((nIterations += nSweeps) < maxIter && !conv) || nIterations < minIter
            bool cont = (s->nIterations < s->maxIter && !conv) || s->nIterations < s->minIter;
            if (!cont) s->stop = 1;
        }));
        return B200LDU_OK;
    };
    int per = nSweeps > 0 ? nSweeps : 1;
    long long maxBodies = ((long long)(S.c.maxIter > S.c.minIter ? S.c.maxIter : S.c.minIter) + per - 1) / per + 1;
    TRY(run_iterations(S, maxBodies, body));
    S.sweepParityUnknown = true; // resolved from nIterations after the read-back
    S.smoothBuf[0] = buf[0];
    S.smoothBuf[1] = buf[1];
    return B200LDU_OK;
}

// diagonalSolver.C:62-81
int solve_diagonal(Solve &S)
{
    const double *d = S.m->d_diag.get();
    double *psi = S.psi;
    const double *b = S.src;
    return ew_launch<0>(S.ctx, S.m->a->L.nPad / 2, nullptr, nullptr, nullptr, [=] __device__(int i, double *) {
        double2 bb = CV2(b)[i], dd = CV2(d)[i];
        V2(psi)[i] = make_double2(__ddiv_rn(bb.x, dd.x), __ddiv_rn(bb.y, dd.y));
    });
}

int gamg_run_cycles(Solve &S, long long maxBodies, int (*body)(void *), void *arg)
{
    return run_iterations(S, maxBodies, [&](long long) -> int { return body(arg); });
}

double *Solve::vec(int k) { return addr_reuse_vec(m->a, m->work[k]); }

int gamg_solve(Solve &S, b200ldu_gamg *g, const char *smoother); // gamg.cu

// run-time selection: lduMatrixSolver.C:43-140.  psi_b / src_b are banded vectors.
int solve_banded(b200ldu_matrix *m, const char *solver, const char *pre, const b200ldu_controls *controls,
                 b200ldu_gamg *gamg, double *psi_b, double *src_b, b200ldu_perf *perf, double *hist_h,
                 int histCap, double **resultBuf)
{
    b200ldu_addr *a = m->a;
    b200ldu_ctx *ctx = a->ctx;
    Solve S;
    S.m = m;
    S.ctx = ctx;
    S.sc = m->d_scal.get();
    S.partials = m->d_partials.get();
    S.psi = psi_b;
    S.src = src_b;
    if (controls)
        S.c = *controls;
    else
        b200ldu_controls_default(&S.c);
    memset(perf, 0, sizeof(*perf));
    *resultBuf = psi_b;

    // residual history buffer on the device
    if (histCap > 0 && hist_h) {
        TRY(m->d_hist.grow((size_t)histCap));
        S.hist = m->d_hist.get();
    }
    // pinned flags + events
    TRY(ctx->pinned.grow(4096));
    char *pin = ctx->pinned.get();
    // a solve nested in another one (GAMG coarsest level) polls its own pair of flags
    static thread_local int depth = 0;
    struct Depth {
        int &d;
        Depth(int &x) : d(x) { d++; }
        ~Depth() { d--; }
    } depthGuard(depth);
    if (depth > 8) {
        b200_set_error("solve: nesting too deep");
        return B200LDU_EINVAL;
    }
    S.pinnedFlags = (int *)pin + 2 * (depth - 1);
    S.pinnedFlags[0] = S.pinnedFlags[1] = 0;
    struct Events { // destroyed on every way out
        cudaEvent_t *ev;
        ~Events()
        {
            for (int i = 0; i < 2; i++)
                if (ev[i]) cudaEventDestroy(ev[i]);
        }
    } events{S.ev};
    CUDA_TRY(cudaEventCreateWithFlags(&S.ev[0], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&S.ev[1], cudaEventDisableTiming));

    // CUDA graphs need a capturable stream: if the context runs on the legacy default stream the
    // solve moves to the context's own stream, ordered against the caller's stream by events
    {
        const char *ev = getenv("B200LDU_GRAPH");
        S.useGraph = !(ev && atoi(ev) == 0) && (ctx->nRanks == 1 || ctx->p2p);
    }
    cudaStream_t userStream = ctx->stream;
    const bool swapStream = S.useGraph && ctx->ownStream && userStream != ctx->ownStream;
    if (swapStream) {
        CUDA_TRY(cudaEventRecord(S.ev[0], userStream));
        CUDA_TRY(cudaStreamWaitEvent(ctx->ownStream, S.ev[0], 0));
        ctx->stream = ctx->ownStream;
    }
    struct StreamRestore {
        b200ldu_ctx *c;
        cudaStream_t user;
        bool on;
        ~StreamRestore()
        {
            if (!on) return;
            cudaEvent_t e;
            if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess) {
                cudaEventRecord(e, c->ownStream);
                cudaStreamWaitEvent(user, e, 0);
                cudaEventDestroy(e);
            }
            c->stream = user;
        }
    } restore{ctx, userStream, swapStream};

    SolverScalars h;
    memset(&h, 0, sizeof(h));
    h.wArA = GREAT_; // PCG.C:88
    h.wArAold = GREAT_;
    h.tolerance = S.c.tolerance;
    h.relTol = S.c.relTol;
    h.maxIter = S.c.maxIter;
    h.minIter = S.c.minIter;
    h.histCap = S.hist ? histCap : 0;
    h.nSweeps = S.c.nSweeps;
    h.nCellsGlobal = a->nCellsGlobal > 0 ? a->nCellsGlobal : (double)a->nCells; // all-reduced at addr_create
    CUDA_TRY(cudaMemcpyAsync(S.sc, &h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));

    int rc = B200LDU_OK;
    bool diagonalOnly = (a->nFaces == 0 && a->L.nRecv == 0);
    const char *sv = solver ? solver : "";
    char pname[32] = "";
    if (diagonalOnly || !strcmp(sv, "diagonal")) {
        strcpy(perf->solverName, "diagonal");
        rc = solve_diagonal(S);
        perf->converged = 1;
        S.noScalars = true;
    } else {
        // ICCG / BICCG wrappers (ICCG.C:40-51)
        if (!strcmp(sv, "ICCG")) {
            sv = "PCG";
            pre = "DIC";
        } else if (!strcmp(sv, "BICCG")) {
            sv = "PBiCG";
            pre = "DILU";
        }
        if (!strcmp(sv, "PCG") || !strcmp(sv, "PBiCG") || !strcmp(sv, "PBiCGStab")) {
            // solver::New looks the name up in the table of the matrix kind first (lduMatrixSolver.C:70-133); the
            // preconditioner is selected inside solve() from the tables of the same kind: DIC symmetric, DILU
            // asymmetric, AINV / diagonal / none both (DICPreconditioner.C:35, DILUPreconditioner.C:35, ...)
            const bool wantSym = !strcmp(sv, "PCG");
            int pk = -1;
            if (wantSym != (bool)m->symmetric) {
                b200_set_error("%s is registered for %s matrices only (PCG.C:36, PBiCG.C:36, PBiCGStab.C:36)", sv,
                               wantSym ? "symmetric" : "asymmetric");
                rc = B200LDU_EMATRIX;
            } else if ((pk = precond_kind(pre, pname)) < 0) {
                rc = B200LDU_ENOPRECOND;
            } else if (pre && ((!strcmp(pre, "DILU") && m->symmetric) || (!strcmp(pre, "DIC") && !m->symmetric))) {
                b200_set_error("Unknown %s matrix preconditioner %s; valid %s matrix preconditioners: (AINV %s diagonal none)",
                               m->symmetric ? "symmetric" : "asymmetric", pre, m->symmetric ? "symmetric" : "asymmetric",
                               m->symmetric ? "DIC" : "DILU");
                rc = B200LDU_ENOPRECOND;
            } else {
                snprintf(perf->solverName, sizeof(perf->solverName), "%s%s", pname, sv);
                if (!strcmp(sv, "PCG")) {
                    // the fused form needs every exchange inside the kernels: the peer-memory halo (or no halo)
                    // and the peer-memory all-reduce (or one rank); otherwise -- cyclic patches, NCCL fall-back --
                    // and with B200LDU_PCG_FUSED=0 the reference's op list runs kernel by kernel
                    const char *ev = getenv("B200LDU_PCG_FUSED");
                    bool fused = !(ev && atoi(ev) == 0) && (a->L.nRecv == 0 || a->p2pHalo) && (ctx->nRanks == 1 || ctx->p2p);
                    rc = fused ? solve_pcg_fused(S, pk) : solve_pcg(S, pk);
                } else if (!strcmp(sv, "PBiCG")) {
                    rc = solve_pbicg(S, pk);
                } else {
                    rc = solve_pbicgstab(S, pk);
                }
            }
        } else if (!strcmp(sv, "smoothSolver")) {
            if (!smoother_ok(pre))
                rc = B200LDU_ENOPRECOND;
            else {
                strcpy(perf->solverName, "smoothSolver");
                rc = solve_smooth(S);
            }
        } else if (!strcmp(sv, "GAMG")) {
            if (!smoother_ok(pre))
                rc = B200LDU_ENOPRECOND;
            else if (!gamg) {
                b200_set_error("GAMG needs an agglomeration handle (b200ldu_gamg_create)");
                rc = B200LDU_EINVAL;
            } else {
                strcpy(perf->solverName, "GAMG");
                rc = gamg_solve(S, gamg, pre);
            }
        } else {
            b200_set_error("Unknown %s solver %s; valid solvers: (BICCG GAMG ICCG PBiCG PBiCGStab PCG "
                           "diagonal smoothSolver)",
                           m->symmetric ? "symmetric" : "asymmetric", sv);
            rc = B200LDU_ENOSOLVER;
        }
    }
    if (rc == B200LDU_OK) {
        // read back the scalars (one synchronisation per solve)
        SolverScalars *hp = (SolverScalars *)(pin + 1024);
        CUDA_TRY(cudaMemcpyAsync(hp, S.sc, sizeof(SolverScalars), cudaMemcpyDeviceToHost, ctx->stream));
        unsigned long long *peerErr = (unsigned long long *)(pin + 2048);
        *peerErr = 0;
        if (ctx->d_seq.get()) // a bounded wait on a peer's flag gave up (engine.cuh spin_until)
            CUDA_TRY(cudaMemcpyAsync(peerErr, ctx->d_seq.get() + 7, sizeof(*peerErr), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        if (*peerErr) {
            b200_set_error("solve: timed out waiting for a peer GPU's halo / all-reduce flag (a rank died or did not "
                           "enter the matching solve)");
            rc = B200LDU_ENCCL;
        }
        if (!S.noScalars) {
            perf->initialResidual = hp->initialResidual;
            perf->finalResidual = hp->finalResidual;
            perf->normFactor = hp->normFactor;
            perf->nIterations = hp->nIterations;
            perf->converged = hp->converged;
            perf->singular = hp->singular;
        }
        if (S.fixedSweeps) perf->nIterations = S.fixedSweeps;
        if (S.sweepParityUnknown) {
            long long sweeps = perf->nIterations; // smoothSolver: nIterations counts sweeps
            if (S.gamgFinestSweeps) sweeps = (long long)perf->nIterations * S.gamgFinestSweeps;
            S.resultBuf = S.smoothBuf[sweeps & 1];
        }
        if (S.resultBuf) *resultBuf = S.resultBuf;
        if (S.hist && hist_h) {
            int k = perf->nIterations + 1;
            if (!strcmp(perf->solverName, "smoothSolver") && S.c.nSweeps > 0) k = perf->nIterations / S.c.nSweeps + 1;
            if (k > histCap) k = histCap;
            if (S.noScalars || S.fixedSweeps) k = 0;
            if (k > 0) CUDA_TRY(cudaMemcpy(hist_h, m->d_hist.get(), sizeof(double) * (size_t)k, cudaMemcpyDeviceToHost));
            for (int i = k; i < histCap; i++) hist_h[i] = NAN;
        }
    } else {
        cudaStreamSynchronize(ctx->stream);
    }
    return rc;
}

extern "C" int b200ldu_solve(b200ldu_matrix *m, const char *solver, const char *pre,
                             const b200ldu_controls *controls, b200ldu_gamg *gamg, double *psi_d,
                             const double *source_d, b200ldu_perf *perf, double *hist_h, int histCap)
{
    if (!m || !psi_d || !source_d || !perf) {
        b200_set_error("solve: null argument");
        return B200LDU_EINVAL;
    }
    CUDA_TRY(cudaSetDevice(m->a->ctx->device));
    b200ldu_addr *a = m->a;
    // banded copies of psi and source live with the matrix workspace
    double *psi_b = addr_reuse_vec(a, m->work[WORK_PSI_B]), *src_b = addr_reuse_vec(a, m->work[WORK_SRC_B]);
    if (!psi_b || !src_b) return B200LDU_ECUDA;
    TRY(to_banded(a, psi_d, psi_b));
    TRY(to_banded(a, source_d, src_b));
    double *res = nullptr;
    TRY(solve_banded(m, solver, pre, controls, gamg, psi_b, src_b, perf, hist_h, histCap, &res));
    TRY(from_banded(a, res, psi_d));
    CUDA_TRY(cudaStreamSynchronize(a->ctx->stream));
    return B200LDU_OK;
}

extern "C" int b200ldu_solve_host(b200ldu_matrix *m, const char *solver, const char *pre,
                                  const b200ldu_controls *controls, b200ldu_gamg *gamg, double *psi_h,
                                  const double *source_h, b200ldu_perf *perf, double *hist_h, int histCap)
{
    if (!m || !psi_h || !source_h || !perf) {
        b200_set_error("solve_host: null argument");
        return B200LDU_EINVAL;
    }
    b200ldu_addr *a = m->a;
    b200ldu_ctx *ctx = a->ctx;
    CUDA_TRY(cudaSetDevice(ctx->device));
    size_t bytes = sizeof(double) * (size_t)a->nCells;
    double *psi_d = addr_reuse_vec(a, m->work[WORK_HOST_PSI]), *src_d = addr_reuse_vec(a, m->work[WORK_HOST_SRC]);
    if (!psi_d || !src_d) return B200LDU_ECUDA;
    // host buffers may be pageable: cudaMemcpyAsync then stages through the driver's pinned pool
    CUDA_TRY(cudaMemcpyAsync(psi_d, psi_h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(src_d, source_h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    TRY(b200ldu_solve(m, solver, pre, controls, gamg, psi_d, src_d, perf, hist_h, histCap));
    CUDA_TRY(cudaMemcpyAsync(psi_h, psi_d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return B200LDU_OK;
}
