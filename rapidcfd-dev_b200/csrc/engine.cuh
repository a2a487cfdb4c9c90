// engine.cuh -- the banded row-gather kernel engine (sm_100a).
//
// One CTA per band.  Phase 1 stages the band's input vector(s) into shared memory:
// the band's own rows with coalesced 128-bit loads, then the band's halo columns
// (rows of neighbouring bands or values received from coupled patches) with a sorted
// gather.  Phase 2: each warp walks its slices of 64 rows; lane k owns rows 2k, 2k+1 and
// reads slot j of both rows with one 128-bit coefficient load (double2) and one 32-bit
// column load (ushort2); the gathers hit shared memory only.  Row sums follow the
// reference's order exactly (diag, owner faces, neighbour faces, interface faces; products
// rounded separately: __dmul_rn/__dadd_rn) so results are bit-comparable with the oracle.
// Fused reductions (dot products needed by the Krylov solvers) are reduced with warp
// shuffles, then across the CTA through shared memory, and written as one partial per
// band -- summed in fixed order by the scalar-step kernel (deterministic, no atomics).
//
// Replaces the reference's Thrust functors: matrixMultiplyFunctor
// (LDU/lduMatrix/lduMatrixATmul.C:42-138), lduAddressingFunctor family
// (LDU/lduAddressing/lduAddressingFunctors.H:10-185), AINVPreconditionerFunctor
// (LDU/preconditioners/AINVPreconditioner/AINVPreconditionerF.H:5-100),
// JacobiSmootherFunctor (LDU/smoothers/Jacobi/JacobiSmootherF.H:8-110).
#pragma once
#include "internal.h"

__device__ __forceinline__ double2 ldg_stream2(const double *p)
{
    // coefficients and columns are read exactly once per kernel: keep them out of L1
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];"
                 : "=d"(r.x), "=d"(r.y)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ uint32_t ldg_stream_u32(const void *p)
{
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}

__device__ __forceinline__ void cp_async16(void *smemDst, const void *gsrc)
{
    unsigned d = (unsigned)__cvta_generic_to_shared(smemDst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}

__device__ __forceinline__ bool spin_until(const unsigned long long *f, unsigned long long seq, unsigned long long *err)
{
    // bounded wait on a flag written by a peer GPU (ld.acquire.sys): a peer that died or never entered the
    // matching kernel must not hang this GPU for ever -- after ~20 s the error word is set and the wait ends
    unsigned long long v, t0 = 0;
    unsigned spins = 0;
    for (;;) {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
        if (v >= seq) return true;
        if ((++spins & 0x3ffu) == 0) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (!t0) t0 = now;
            if (now - t0 > 20000000000ull) {
                if (err) atomicExch(err, 1ull);
                return false;
            }
        }
    }
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sums of NRED per-thread values -> out[blockIdx.x * NRED + k].
// Fixed combination order: lanes by xor-butterfly, warps in index order.
template <int NRED, int THREADS>
__device__ __forceinline__ void block_reduce_store(double (&red)[NRED], double *partials,
                                                   int slot)
{
    __shared__ double wsum[NRED][THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NRED; k++) {
        double v = warp_sum(red[k]);
        if (lane == 0) wsum[k][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < NRED) {
        double s = 0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; w++) s += wsum[threadIdx.x][w];
        partials[(size_t)slot * NRED + threadIdx.x] = s;
    }
}

// ---------------------------------------------------------------------------
// Op concept
//   static constexpr int  NVEC   1 or 2 vectors staged in shared memory
//   static constexpr int  NRED   number of fused reductions (0..3)
//   static constexpr bool LOCAL  true: owner/neighbour entries only (no interfaces)
//   const int *stop              device flag; kernel exits at once when *stop != 0
//   bool prologue(L)             runs first in every CTA (default: nothing); false => the CTA exits
//   double *partials             [nBands*NRED]
//   void   stage(int g, double &a, double &b)        value(s) of extended index g
//   void   stage_own(int r, double2 &a, double2 &b)  rows r, r+1 of the own band (may
//                                                    also write a fused vector update)
//   double init(int r, double a, double b)           start of the row sum
//   double term(double acc, double v, double a, double b)   acc (+) v*...
//   void   finish(int r, double acc0, double acc1, a0,b0,a1,b1, double *red)
//                                                    writes rows r, r+1; adds reductions
// ---------------------------------------------------------------------------
template <class Op>
__global__ void __launch_bounds__(ENGINE_THREADS, 6) engine_kernel(const LayoutDev L, const double *__restrict__ val, Op op)
{
    extern __shared__ double smem[];
    if (!op.prologue(L)) return; // stop flag (OpBase) or the deferred scalar step of the fused PCG (ops.cuh)
    // Fused halo send (peer-memory path): the first nPackChunks CTAs of the grid gather psi
    // at the processor-patch face cells, store it straight into the neighbours' receive
    // buffers over NVLink and release their arrival flags; all other CTAs are SpMV bands
    // (those that reference received values wait for the neighbours' flags below).
    const bool fusedPack = op.waitHalo && L.nPackChunks > 0;
    unsigned long long haloSeqNow = 0;
    if (fusedPack) {
        haloSeqNow = L.seqs[1] + 1; // seqs[1] only advances when the whole grid has finished
        if ((int)blockIdx.x < L.nPackChunks) {
            const PackChunk c = L.packChunks[blockIdx.x];
            const PackPatch P = L.packPatches[c.patch];
            double *dst = P.dst[haloSeqNow & 1];
            for (int i = c.begin + threadIdx.x; i < c.end; i += ENGINE_THREADS)
                dst[i - P.start] = op.pack_val(__ldg(L.sendRows + i));
            __threadfence_system();
            __syncthreads();
            if (threadIdx.x == 0) {
                unsigned long long done = atomicAdd(&L.seqs[8 + c.patch], 1ull) + 1;
                if (done == (unsigned long long)P.nChunks) {
                    L.seqs[8 + c.patch] = 0;
                    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(P.flag), "l"(haloSeqNow) : "memory");
                }
                if (atomicAdd(&L.seqs[6], 1ull) + 1 == (unsigned long long)gridDim.x) {
                    L.seqs[6] = 0;
                    __threadfence();
                    L.seqs[1] = haloSeqNow;
                }
            }
            return;
        }
    }
    const int band = blockIdx.x - (fusedPack ? L.nPackChunks : 0);
    const int rowBase = band * L.bandRows;
    const int stride = (L.bandRows + L.maxHalo + 1) & ~1; // keep the second tile 16-byte aligned
    double *xs = smem;
    double *ys = smem + ((Op::NVEC > 1) ? stride : 0);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = ENGINE_THREADS / 32;

    // ---- phase 1: stage the band's vector tile + halo ----
    if (Op::NVEC > 0) {
    for (int i = tid; i < (L.bandRows >> 1); i += ENGINE_THREADS) {
        double2 a, b = make_double2(0, 0);
        op.stage_own(rowBase + 2 * i, a, b);
        reinterpret_cast<double2 *>(xs)[i] = a;
        if (Op::NVEC > 1) reinterpret_cast<double2 *>(ys)[i] = b;
    }
    {
        const int hs = L.haloStart[band], hn = L.haloStart[band + 1] - hs;
        // peer-memory halo: bands that reference received values wait for the neighbours'
        // arrival flags here, so interior bands overlap with the exchange
        const double *remoteTail = nullptr;
        if (op.waitHalo && L.haloFlags) {
            const unsigned long long seq = fusedPack ? haloSeqNow : *L.haloSeq;
            remoteTail = (seq & 1) ? L.tail1 : L.tail0;
            if (hn > 0 && __ldg(L.haloIdx + hs + hn - 1) >= L.nPad) {
                if (tid < L.nNbr) spin_until(L.haloFlags + L.nbr[tid], seq, L.seqs ? L.seqs + 7 : nullptr);
                __syncthreads();
            }
        }
        for (int i = tid; i < hn; i += ENGINE_THREADS) {
            int g = __ldg(L.haloIdx + hs + i);
            double a, b = 0;
            if (remoteTail && g >= L.nPad)
                a = __ldcg(remoteTail + (g - L.nPad));
            else
                op.stage(g, a, b);
            xs[L.bandRows + i] = a;
            if (Op::NVEC > 1) ys[L.bandRows + i] = b;
        }
    }
    __syncthreads();
    }

    // ---- phase 2: row sums ----
    double red[Op::NRED > 0 ? Op::NRED : 1];
#pragma unroll
    for (int k = 0; k < (Op::NRED > 0 ? Op::NRED : 1); k++) red[k] = 0;

    for (int sl = warp; sl < L.slicesPerBand; sl += NW) {
        const int s = band * L.slicesPerBand + sl;
        const long long base = L.sliceStart[s];
        const int W = Op::LOCAL ? L.sliceWL[s] : L.sliceW[s];
        const int lr = sl * SLICE_ROWS + 2 * lane; // local row of this lane's first row
        const double a0 = (Op::NVEC > 0) ? xs[lr] : 0, a1 = (Op::NVEC > 0) ? xs[lr + 1] : 0;
        const double b0 = (Op::NVEC > 1) ? ys[lr] : 0, b1 = (Op::NVEC > 1) ? ys[lr + 1] : 0;
        double acc0 = op.init(rowBase + lr, a0, b0);
        double acc1 = op.init(rowBase + lr + 1, a1, b1);
        const double *vp = val + base + 2 * lane;
        const uint16_t *cp = L.col + base + 2 * lane;
        int j = 0;
        // slots in groups of 4: all loads of a group are issued before any use
        for (; j + 4 <= W; j += 4) {
            double2 v[4];
            uint32_t c[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                v[k] = ldg_stream2(vp + (size_t)(j + k) * SLICE_ROWS);
                c[k] = ldg_stream_u32(cp + (size_t)(j + k) * SLICE_ROWS);
            }
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int c0 = c[k] & 0xffffu, c1 = c[k] >> 16;
                acc0 = op.term(acc0, v[k].x, (Op::NVEC > 0) ? xs[c0] : 0, (Op::NVEC > 1) ? ys[c0] : 0);
                acc1 = op.term(acc1, v[k].y, (Op::NVEC > 0) ? xs[c1] : 0, (Op::NVEC > 1) ? ys[c1] : 0);
            }
        }
        for (; j < W; j++) {
            double2 v = ldg_stream2(vp + (size_t)j * SLICE_ROWS);
            uint32_t c = ldg_stream_u32(cp + (size_t)j * SLICE_ROWS);
            const int c0 = c & 0xffffu, c1 = c >> 16;
            acc0 = op.term(acc0, v.x, (Op::NVEC > 0) ? xs[c0] : 0, (Op::NVEC > 1) ? ys[c0] : 0);
            acc1 = op.term(acc1, v.y, (Op::NVEC > 0) ? xs[c1] : 0, (Op::NVEC > 1) ? ys[c1] : 0);
        }
        op.finish(rowBase + lr, acc0, acc1, a0, b0, a1, b1, red);
    }
    if (Op::NRED > 0) block_reduce_store<(Op::NRED > 0 ? Op::NRED : 1), ENGINE_THREADS>(red, op.partials, band);
    if (fusedPack && threadIdx.x == 0) {
        if (atomicAdd(&L.seqs[6], 1ull) + 1 == (unsigned long long)gridDim.x) {
            L.seqs[6] = 0;
            __threadfence();
            L.seqs[1] = haloSeqNow;
        }
    }
}

template <class Op>
int engine_launch(b200ldu_addr *a, const double *val, const Op &op)
{
    const LayoutDev &L = a->L;
    size_t smem = sizeof(double) * (size_t)((L.bandRows + L.maxHalo + 1) & ~1) * (size_t)Op::NVEC;
    // the kernel also owns a little static shared memory (reduction scratch): opt in to large dynamic shared
    // memory well before the 48 KB default limit.  The attribute is per device and instantiation.
    static size_t configured[64] = {0};
    const int dev = a->ctx->device & 63;
    if (smem > 40 * 1024 && smem > configured[dev]) {
        CUDA_TRY(cudaFuncSetAttribute(engine_kernel<Op>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[dev] = smem;
    }
    int grid = L.nBands + ((op.waitHalo && L.nPackChunks > 0) ? L.nPackChunks : 0);
    engine_kernel<Op><<<grid, ENGINE_THREADS, smem, a->ctx->stream>>>(L, val, op);
    a->ctx->launches++;
    KERNEL_CHECK();
    return B200LDU_OK;
}

// matrix sweep with A's coefficients, or A^T's
template <class Op>
int engine_launch_m(b200ldu_matrix *m, bool transpose, const Op &op)
{
    return engine_launch(m->a, transpose ? m->valT() : m->d_val.get(), op);
}
