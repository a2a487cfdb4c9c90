// comm.cu -- multi-GPU plumbing: one process per GPU, one NCCL communicator per context,
// plus hand-written peer-memory collectives over NVLink / NVSwitch for the two latency-
// bound exchanges of the hot path.
//
// Replaces the reference's Pstream-over-MPI layer: processor-patch halo exchange
// (src/Pstream/mpi/UOPwrite.C:73-122, UIPread.C:260-316,
// LDU/lduAddressing/lduInterface/processorLduInterfaceTemplates.C:128-298, host-staged
// unless gpuDirectTransfer) and the scalar all-reduces behind gSumProd/gSumMag/gAverage
// (src/Pstream/mpi/allReduceTemplates.C:197).
//
// Peer-memory path (default when CUDA IPC works; B200LDU_P2P=0 forces NCCL):
//  * every rank allocates one small device region and publishes its IPC handle (all-gathered
//    with NCCL at b200ldu_comm_init); every rank maps every other region;
//  * halo: the pack kernel gathers psi at the patch face cells and stores it STRAIGHT INTO
//    THE NEIGHBOUR'S receive buffer over NVLink (coalesced peer stores), then releases a
//    sequence flag there; the SpMV kernel of the neighbour lets its interior bands run and
//    makes only the bands that reference received values wait on the flag (engine.cuh) --
//    pack, transfer and interior compute overlap with no NCCL call and no extra kernel;
//  * all-reduce of the 1..4 solver scalars: fused into the scalar-step kernel (ops.cuh):
//    peer stores of the partial sums + flag into every rank's mailbox, rank-ordered sum.
// Receive buffers and mailboxes are double-buffered by sequence parity; the sequence
// counters live on the device and only advance when a kernel really executed, so the
// early-exit of a converged solve cannot desynchronise the ranks.
// NCCL remains the bootstrap (handle exchange) and the fallback data path.
#include <nccl.h>

#include <cstdlib>

#include "comm.h"

#define NCCL_TRY(expr)                                                                      \
    do {                                                                                    \
        ncclResult_t _r = (expr);                                                           \
        if (_r != ncclSuccess) {                                                            \
            b200_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, ncclGetErrorString(_r)); \
            return B200LDU_ENCCL;                                                           \
        }                                                                                   \
    } while (0)

// PACK_CHUNK (faces per packing CTA of the fused halo send): internal.h

extern "C" int b200ldu_comm_unique_id(void *out128)
{
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    NCCL_TRY(ncclGetUniqueId(&id));
    memcpy(out128, &id, 128);
    return B200LDU_OK;
}

static int p2p_setup(b200ldu_ctx *ctx)
{
    const char *e = getenv("B200LDU_P2P");
    if (e && atoi(e) == 0) return B200LDU_OK;
    if (ctx->nRanks > P2P_MAXR) return B200LDU_OK;
    cudaStream_t st = ctx->stream;
    ncclComm_t comm = (ncclComm_t)ctx->nccl;
    TRY(ctx->region.alloc(P2P_REGION_BYTES));
    CUDA_TRY(cudaMemsetAsync(ctx->region.get(), 0, P2P_REGION_BYTES, st));
    TRY(ctx->d_seq.alloc(64));
    CUDA_TRY(cudaMemsetAsync(ctx->d_seq.get(), 0, 64 * sizeof(unsigned long long), st));
    cudaIpcMemHandle_t mine;
    cudaError_t ce = cudaIpcGetMemHandle(&mine, ctx->region.get());
    int ok = (ce == cudaSuccess) ? 1 : 0;
    if (!ok) cudaGetLastError();
    // all-gather {ok, handle} through NCCL (device buffers)
    const int rec = 128;
    std::vector<char> sendH(rec, 0), allH((size_t)rec * ctx->nRanks, 0);
    memcpy(sendH.data(), &ok, sizeof(int));
    memcpy(sendH.data() + 64, &mine, sizeof(mine));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
    {
        DevBuf<char> d_send, d_all;
        TRY(d_send.alloc(rec));
        TRY(d_all.alloc((size_t)rec * ctx->nRanks));
        CUDA_TRY(cudaMemcpyAsync(d_send.get(), sendH.data(), rec, cudaMemcpyHostToDevice, st));
        NCCL_TRY(ncclAllGather(d_send.get(), d_all.get(), rec, ncclChar, comm, st));
        CUDA_TRY(cudaMemcpyAsync(allH.data(), d_all.get(), (size_t)rec * ctx->nRanks, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    bool all = true;
    for (int r = 0; r < ctx->nRanks; r++) {
        int okr;
        memcpy(&okr, allH.data() + (size_t)rec * r, sizeof(int));
        all = all && okr;
    }
    int opened = all ? 1 : 0;
    if (all) {
        for (int r = 0; r < ctx->nRanks && opened; r++) {
            if (r == ctx->rank) {
                ctx->peerRegion[r] = ctx->region.get();
                continue;
            }
            cudaIpcMemHandle_t h;
            memcpy(&h, allH.data() + (size_t)rec * r + 64, sizeof(h));
            void *p = nullptr;
            ce = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
            if (ce != cudaSuccess) {
                cudaGetLastError();
                opened = 0;
            } else
                ctx->peerRegion[r] = (char *)p;
        }
    }
    // every rank must agree (a rank that failed to map falls everybody back to NCCL)
    DevBuf<int> d_flag;
    TRY(d_flag.alloc(1));
    CUDA_TRY(cudaMemcpyAsync(d_flag.get(), &opened, sizeof(int), cudaMemcpyHostToDevice, st));
    NCCL_TRY(ncclAllReduce(d_flag.get(), d_flag.get(), 1, ncclInt, ncclMin, comm, st));
    CUDA_TRY(cudaMemcpyAsync(&opened, d_flag.get(), sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    ctx->p2p = opened != 0;
    return B200LDU_OK;
}

extern "C" int b200ldu_comm_init(b200ldu_ctx *ctx, const void *id128, int rank, int nRanks)
{
    if (!ctx || nRanks < 1 || rank < 0 || rank >= nRanks) {
        b200_set_error("comm_init: bad arguments");
        return B200LDU_EINVAL;
    }
    ctx->rank = rank;
    ctx->nRanks = nRanks;
    if (nRanks == 1) return B200LDU_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclComm_t comm;
    NCCL_TRY(ncclCommInitRank(&comm, nRanks, id, rank));
    ctx->nccl = (void *)comm;
    return p2p_setup(ctx);
}

// which data path the two exchanges of the hot path take (reported by bench.py): 1 = hand-written peer-memory
// kernels over NVLink, 0 = NCCL (ncclSend/ncclRecv halo, ncclAllReduce of the solver scalars), -1 = not applicable
extern "C" int b200ldu_comm_info(const b200ldu_ctx *ctx, const b200ldu_addr *a, int *allreduceP2P, int *haloP2P)
{
    if (!ctx) return B200LDU_EINVAL;
    if (allreduceP2P) *allreduceP2P = ctx->nRanks > 1 ? (ctx->p2p ? 1 : 0) : -1;
    if (haloP2P) *haloP2P = (a && a->L.nRecv > 0) ? (a->p2pHalo ? 1 : 0) : -1;
    return B200LDU_OK;
}

int comm_destroy(b200ldu_ctx *ctx)
{
    // the peers' regions are unmapped before this rank's own is released
    if (ctx->region.get())
        for (int r = 0; r < ctx->nRanks; r++)
            if (r != ctx->rank && ctx->peerRegion[r]) cudaIpcCloseMemHandle(ctx->peerRegion[r]);
    ctx->region.reset();
    ctx->d_seq.reset();
    if (ctx->nccl) {
        ncclCommDestroy((ncclComm_t)ctx->nccl);
        ctx->nccl = nullptr;
    }
    return B200LDU_OK;
}

int comm_allreduce_sum(b200ldu_ctx *ctx, double *d_buf, int n)
{
    if (ctx->nRanks == 1) return B200LDU_OK;
    NCCL_TRY(ncclAllReduce(d_buf, d_buf, n, ncclDouble, ncclSum, (ncclComm_t)ctx->nccl, ctx->stream));
    return B200LDU_OK;
}

P2PRed comm_p2p_red(b200ldu_ctx *ctx)
{
    P2PRed p;
    p.rank = ctx->rank;
    p.nRanks = ctx->nRanks;
    for (int r = 0; r < ctx->nRanks; r++) {
        p.mail[r] = (double *)(ctx->peerRegion[r] + P2P_MAIL_OFF);
        p.flag[r] = (unsigned long long *)(ctx->peerRegion[r] + P2P_MAILFLAG_OFF);
    }
    p.seq = ctx->d_seq.get(); // [0]
    return p;
}

// Per-addressing setup (collective over the communicator when the addressing has processor
// patches): global cell count for gAverage, and -- for the peer-memory halo -- where each of
// this rank's patches lands in its neighbour's receive buffer.
int comm_addr_setup(b200ldu_addr *a)
{
    b200ldu_ctx *ctx = a->ctx;
    a->nCellsGlobal = (double)a->nCells;
    a->L.haloFlags = nullptr;
    a->L.haloSeq = nullptr;
    a->L.tail0 = a->L.tail1 = nullptr;
    a->L.nNbr = 0;
    // COLLECTIVE over the communicator: every rank takes part in the gather below, also one whose addressing
    // has no processor patch (it contributes an empty row and still learns the global cell count)
    if (ctx->nRanks == 1 || !ctx->nccl) return B200LDU_OK;
    cudaStream_t st = ctx->stream;
    ncclComm_t comm = (ncclComm_t)ctx->nccl;
    const int R = ctx->nRanks;
    // table row of this rank: [0..R) offset of my patch facing rank r (-1 none, -2 not representable),
    // [R..2R) its size, [2R] my cell count
    std::vector<int> row(2 * R + 1, -1), all((size_t)(2 * R + 1) * R, 0);
    bool simple = (a->L.nRecv <= (int)P2P_RECV_CAP);
    for (int p = 0; p < a->nPatches; p++) {
        int nb = a->neighbRank[p];
        if (nb == ctx->rank || nb < 0 || nb >= R || row[nb] != -1) {
            simple = false; // cyclic, or several patches towards one rank: NCCL path
            continue;
        }
        row[nb] = a->patchStart[p];
        row[R + nb] = a->patchStart[p + 1] - a->patchStart[p];
    }
    if (a->L.nRecv == 0) simple = true; // nothing to exchange: does not block the peers' peer-memory halo
    if (!simple)
        for (int r = 0; r < R; r++) row[r] = -2;
    row[2 * R] = a->nCells;
    {
        DevBuf<int> d_row, d_all;
        TRY(d_row.alloc(row.size()));
        TRY(d_all.alloc(all.size()));
        CUDA_TRY(cudaMemcpyAsync(d_row.get(), row.data(), sizeof(int) * row.size(), cudaMemcpyHostToDevice, st));
        NCCL_TRY(ncclAllGather(d_row.get(), d_all.get(), row.size(), ncclInt, comm, st));
        CUDA_TRY(cudaMemcpyAsync(all.data(), d_all.get(), sizeof(int) * all.size(), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    double ncg = 0;
    bool everySimple = true;
    for (int r = 0; r < R; r++) {
        ncg += all[(size_t)(2 * R + 1) * r + 2 * R];
        for (int q = 0; q < R; q++)
            if (all[(size_t)(2 * R + 1) * r + q] == -2) everySimple = false;
    }
    a->nCellsGlobal = ncg;
    if (!ctx->p2p || !everySimple || a->nPatches == 0) return B200LDU_OK;
    std::vector<PackPatch> pp(a->nPatches);
    std::vector<PackChunk> pc;
    for (int p = 0; p < a->nPatches; p++) {
        int nb = a->neighbRank[p];
        int remoteOff = all[(size_t)(2 * R + 1) * nb + ctx->rank];
        int remoteN = all[(size_t)(2 * R + 1) * nb + R + ctx->rank];
        int n = a->patchStart[p + 1] - a->patchStart[p];
        if (remoteOff < 0 || remoteN != n) {
            b200_set_error("processor patch %d towards rank %d has no matching patch of %d faces there", p, nb, n);
            return B200LDU_EINVAL;
        }
        double *base = (double *)(ctx->peerRegion[nb] + P2P_RECV_OFF);
        pp[p].dst[0] = base + remoteOff;
        pp[p].dst[1] = base + P2P_RECV_CAP + remoteOff;
        pp[p].flag = (unsigned long long *)(ctx->peerRegion[nb] + P2P_HALOFLAG_OFF) + ctx->rank;
        pp[p].start = a->patchStart[p];
        pp[p].n = n;
        pp[p].nChunks = (n + PACK_CHUNK - 1) / PACK_CHUNK;
        for (int c = 0; c < pp[p].nChunks; c++)
            pc.push_back({p, a->patchStart[p] + c * PACK_CHUNK, std::min(a->patchStart[p] + (c + 1) * PACK_CHUNK, a->patchStart[p + 1])});
        a->L.nbr[a->L.nNbr++] = nb;
    }
    TRY(a->d_packPatches.alloc(pp.size()));
    TRY(a->d_packChunks.alloc(pc.size()));
    CUDA_TRY(cudaMemcpy(a->d_packPatches.get(), pp.data(), sizeof(PackPatch) * pp.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(a->d_packChunks.get(), pc.data(), sizeof(PackChunk) * pc.size(), cudaMemcpyHostToDevice));
    a->nPackChunks = (int)pc.size();
    a->L.haloFlags = (const unsigned long long *)(ctx->region.get() + P2P_HALOFLAG_OFF);
    a->L.haloSeq = ctx->d_seq.get() + 1;
    a->L.tail0 = (const double *)(ctx->region.get() + P2P_RECV_OFF);
    a->L.tail1 = a->L.tail0 + P2P_RECV_CAP;
    a->L.packChunks = a->d_packChunks.get();
    a->L.packPatches = a->d_packPatches.get();
    a->L.sendRows = a->d_sendRows.get();
    a->L.seqs = ctx->d_seq.get();
    a->L.nPackChunks = (int)pc.size();
    a->p2pHalo = true;
    return B200LDU_OK;
}

__global__ void pack_kernel(int n, const int *__restrict__ rows, const double *__restrict__ x,
                            double *__restrict__ send, const int *stop)
{
    if (stop && *stop) return;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) send[i] = x[rows[i]];
}

__global__ void cyclic_fill_kernel(int n, const int *__restrict__ src, const double *__restrict__ x,
                                   double *__restrict__ tail, const int *stop)
{
    if (stop && *stop) return;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && src[i] >= 0) tail[i] = x[src[i]];
}

// x is a banded vector of vecLen doubles.  NCCL path: received neighbour values land in its
// tail [nPad, nPad + nRecv) where the band halo lists point.  Peer-memory path: they land
// in this rank's shared receive buffer (the engine reads it for columns >= nPad).
// *usedP2P tells the caller to make the consuming kernel wait on the arrival flags.
int comm_halo_exchange(b200ldu_addr *a, double *x, double *sendBuf, const int *stop, int *usedP2P)
{
    if (usedP2P) *usedP2P = 0;
    const int nRecv = a->L.nRecv;
    if (nRecv == 0) return B200LDU_OK;
    b200ldu_ctx *ctx = a->ctx;
    if (a->p2pHalo) { // the send is fused into the consuming kernel (engine.cuh)
        if (usedP2P) *usedP2P = 1;
        return B200LDU_OK;
    }
    bool remote = false;
    for (int p = 0; p < a->nPatches; p++)
        if (a->neighbRank[p] >= 0) remote = true;
    if (a->d_cyclicSrc.get()) { // cyclic partners: x[nPad + face] = x[partner's face cell]
        cyclic_fill_kernel<<<(nRecv + 255) / 256, 256, 0, ctx->stream>>>(nRecv, a->d_cyclicSrc.get(), x, x + a->L.nPad, stop);
        ctx->launches++;
        KERNEL_CHECK();
    }
    if (!remote) return B200LDU_OK;
    pack_kernel<<<(nRecv + 255) / 256, 256, 0, ctx->stream>>>(nRecv, a->d_sendRows.get(), x, sendBuf, stop);
    ctx->launches++;
    KERNEL_CHECK();
    if (remote && !ctx->nccl) {
        b200_set_error("halo exchange: processor patches present but no communicator (b200ldu_comm_init)");
        return B200LDU_ENCCL;
    }
    if (remote) NCCL_TRY(ncclGroupStart());
    for (int p = 0; p < a->nPatches; p++) {
        int s = a->patchStart[p], n = a->patchStart[p + 1] - s;
        int nb = a->neighbRank[p];
        if (nb < 0) continue; // cyclic: filled above
        if (nb == ctx->rank) {
            b200_set_error("halo exchange: patch %d names this rank as its neighbour; cyclic patches are "
                           "declared with neighbRank = -(partnerPatch + 1)", p);
            return B200LDU_EINVAL;
        }
        NCCL_TRY(ncclSend(sendBuf + s, n, ncclDouble, nb, (ncclComm_t)ctx->nccl, ctx->stream));
        NCCL_TRY(ncclRecv(x + a->L.nPad + s, n, ncclDouble, nb, (ncclComm_t)ctx->nccl, ctx->stream));
    }
    if (remote) NCCL_TRY(ncclGroupEnd());
    return B200LDU_OK;
}

// ---------------------------------------------------------------------------
// setup-time helpers for the multi-rank GAMG agglomeration (host data, collective calls)
// ---------------------------------------------------------------------------
// exchange one int per coupled-patch face with the neighbour rank of each patch
// (the reference's internalFieldTransfer of the restrict map,
// GAMGAgglomerateLduAddressing.C:487-500)
int comm_exchange_patch_ints(b200ldu_ctx *ctx, int nPatches, const int *patchStart, const int *neighbRank,
                             const int *send, int *recv)
{
    int tot = nPatches ? patchStart[nPatches] : 0;
    if (tot == 0) return B200LDU_OK;
    // cyclic pairs (neighbRank = -(q+1)): the neighbour values are this rank's own, at the partner patch
    // (cyclicGAMGInterface::internalFieldTransfer, cyclicGAMGInterface.C:163-180)
    bool remote = false;
    for (int p = 0; p < nPatches; p++) {
        if (neighbRank[p] >= 0) {
            remote = true;
            continue;
        }
        const int q = -neighbRank[p] - 1, n = patchStart[p + 1] - patchStart[p];
        for (int i = 0; i < n; i++) recv[patchStart[p] + i] = send[patchStart[q] + i];
    }
    if (!remote) return B200LDU_OK;
    if (!ctx->nccl) {
        b200_set_error("processor patches present but no communicator (b200ldu_comm_init)");
        return B200LDU_ENCCL;
    }
    DevBuf<int> d_s, d_r;
    TRY(d_s.alloc((size_t)tot));
    TRY(d_r.alloc((size_t)tot));
    cudaStream_t st = ctx->stream;
    CUDA_TRY(cudaMemcpyAsync(d_s.get(), send, sizeof(int) * (size_t)tot, cudaMemcpyHostToDevice, st));
    NCCL_TRY(ncclGroupStart());
    for (int p = 0; p < nPatches; p++) {
        int s = patchStart[p], n = patchStart[p + 1] - s;
        if (neighbRank[p] < 0) continue;
        NCCL_TRY(ncclSend(d_s.get() + s, n, ncclInt, neighbRank[p], (ncclComm_t)ctx->nccl, st));
        NCCL_TRY(ncclRecv(d_r.get() + s, n, ncclInt, neighbRank[p], (ncclComm_t)ctx->nccl, st));
    }
    NCCL_TRY(ncclGroupEnd());
    std::vector<int> got((size_t)tot);
    CUDA_TRY(cudaMemcpyAsync(got.data(), d_r.get(), sizeof(int) * (size_t)tot, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    for (int p = 0; p < nPatches; p++)
        if (neighbRank[p] >= 0)
            for (int i = patchStart[p]; i < patchStart[p + 1]; i++) recv[i] = got[i];
    return B200LDU_OK;
}

// all-gather of n doubles per rank (host in, host out: all[r*n + i])
int comm_allgather_host(b200ldu_ctx *ctx, const double *mine, int n, double *all)
{
    if (ctx->nRanks == 1) {
        memcpy(all, mine, sizeof(double) * (size_t)n);
        return B200LDU_OK;
    }
    DevBuf<double> d_s, d_a;
    cudaStream_t st = ctx->stream;
    TRY(d_s.alloc((size_t)n));
    TRY(d_a.alloc((size_t)n * ctx->nRanks));
    CUDA_TRY(cudaMemcpyAsync(d_s.get(), mine, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    NCCL_TRY(ncclAllGather(d_s.get(), d_a.get(), n, ncclDouble, (ncclComm_t)ctx->nccl, st));
    CUDA_TRY(cudaMemcpyAsync(all, d_a.get(), sizeof(double) * (size_t)n * ctx->nRanks, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return B200LDU_OK;
}

// in-stream all-gather of GMAX doubles per rank (device buffers), NCCL fallback of the
// peer-memory gather used by the coarsest-level solve
int comm_allgather_dev(b200ldu_ctx *ctx, const double *d_mine, int n, double *d_all)
{
    if (ctx->nRanks == 1) return B200LDU_OK;
    NCCL_TRY(ncclAllGather(d_mine, d_all, n, ncclDouble, (ncclComm_t)ctx->nccl, ctx->stream));
    return B200LDU_OK;
}

// coupled-patch exchange of a caller-order field (processorFvPatchField::initEvaluate / evaluate,
// processorFvPatchField.C:196-262; cyclic: cyclicFvPatchField::patchNeighbourField, :133-160): send_d holds the
// patchInternalField of every coupled face (nComp values each, patches concatenated), recv_d receives the
// neighbour's.  In stream; processor patches through one NCCL group, cyclic pairs by a device copy.
int comm_exchange_patch_field(b200ldu_addr *a, int nComp, const double *send_d, double *recv_d)
{
    b200ldu_ctx *ctx = a->ctx;
    bool remote = false;
    for (int p = 0; p < a->nPatches; p++) {
        const int s = a->patchStart[p], n = a->patchStart[p + 1] - s, nb = a->neighbRank[p];
        if (nb >= 0) {
            remote = true;
            continue;
        }
        const int q = -nb - 1; // validated at addr_create
        CUDA_TRY(cudaMemcpyAsync(recv_d + (size_t)s * nComp, send_d + (size_t)a->patchStart[q] * nComp,
                                 sizeof(double) * (size_t)n * nComp, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    if (!remote) return B200LDU_OK;
    if (!ctx->nccl) {
        b200_set_error("patch field exchange: processor patches present but no communicator (b200ldu_comm_init)");
        return B200LDU_ENCCL;
    }
    NCCL_TRY(ncclGroupStart());
    for (int p = 0; p < a->nPatches; p++) {
        const int s = a->patchStart[p], n = a->patchStart[p + 1] - s, nb = a->neighbRank[p];
        if (nb < 0) continue;
        NCCL_TRY(ncclSend(send_d + (size_t)s * nComp, (size_t)n * nComp, ncclDouble, nb, (ncclComm_t)ctx->nccl, ctx->stream));
        NCCL_TRY(ncclRecv(recv_d + (size_t)s * nComp, (size_t)n * nComp, ncclDouble, nb, (ncclComm_t)ctx->nccl, ctx->stream));
    }
    NCCL_TRY(ncclGroupEnd());
    return B200LDU_OK;
}
