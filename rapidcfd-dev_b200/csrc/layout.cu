// layout.cu -- host-side construction of the banded block layout ("warp-contiguous
// bands") from OpenFOAM lduAddressing.  Replaces the reference's derived addressing
// (LDU/lduAddressing/lduAddressing.C:169-400: losort, ownerStart, losortStart,
// ownerSortAddr, patchSort*) and lduMatrix::calcSortCoeffs (LDU/lduMatrix/lduMatrix.C:380-471).
//
// Design (DESIGN.md section 3):
//  * cells are renumbered so that BAND_ROWS consecutive rows form a spatially compact
//    brick (Morton order over power-of-two tiles of the cell-centre bounding box, caller
//    order inside a tile; without centres a graph-distance embedding stands in);
//  * every row keeps its entries in the reference's summation order (owner faces by
//    face index, neighbour faces in losort order, coupled-patch faces in patch order);
//  * entries of 64 consecutive rows are stored slot-major ("slice"): slot j of row q
//    sits at sliceStart + 64*j + q, so a warp reads one slot of its 64 rows with a
//    single 128-bit load per lane;
//  * columns are 16-bit indices into the band's shared-memory psi tile: the band's own
//    rows first, then the band's halo list (rows of other bands / received interface
//    values) which is gathered once per band.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <numeric>
#include <queue>

#include "internal.h"

namespace {

struct Csr {
    std::vector<int> start, item;
};

// cell -> faces it owns is contiguous (faces sorted by owner); cell -> faces where it
// is neighbour needs the stable counting sort the reference calls losort.
void build_losort(int nCells, const std::vector<int> &u, std::vector<int> &losortStart,
                  std::vector<int> &losort)
{
    int nF = (int)u.size();
    losortStart.assign((size_t)nCells + 1, 0);
    for (int f = 0; f < nF; f++) losortStart[u[f] + 1]++;
    for (int c = 0; c < nCells; c++) losortStart[c + 1] += losortStart[c];
    losort.resize(nF);
    std::vector<int> cur(losortStart.begin(), losortStart.end() - 1);
    for (int f = 0; f < nF; f++) losort[cur[u[f]]++] = f;
}

void build_owner_start(int nCells, const std::vector<int> &l, std::vector<int> &ownerStart)
{
    ownerStart.assign((size_t)nCells + 1, 0);
    for (size_t f = 0; f < l.size(); f++) ownerStart[l[f] + 1]++;
    for (int c = 0; c < nCells; c++) ownerStart[c + 1] += ownerStart[c];
}

// breadth-first graph distance from `seed` (used when no cell centres are given);
// further components, if any, restart from their lowest cell
void bfs_dist(int nCells, const std::vector<int> &l, const std::vector<int> &u,
              const std::vector<int> &ownerStart, const std::vector<int> &losortStart,
              const std::vector<int> &losort, int seed, std::vector<int> &dist)
{
    dist.assign(nCells, -1);
    std::vector<int> q;
    q.reserve(nCells);
    auto grow = [&](int s) {
        size_t head = q.size();
        dist[s] = 0;
        q.push_back(s);
        while (head < q.size()) {
            int c = q[head++];
            for (int f = ownerStart[c]; f < ownerStart[c + 1]; f++)
                if (dist[u[f]] < 0) {
                    dist[u[f]] = dist[c] + 1;
                    q.push_back(u[f]);
                }
            for (int k = losortStart[c]; k < losortStart[c + 1]; k++) {
                int nb = l[losort[k]];
                if (dist[nb] < 0) {
                    dist[nb] = dist[c] + 1;
                    q.push_back(nb);
                }
            }
        }
    };
    grow(seed);
    for (int c = 0; c < nCells; c++)
        if (dist[c] < 0) grow(c);
}

int argmax(const std::vector<int> &v)
{
    return (int)(std::max_element(v.begin(), v.end()) - v.begin());
}

uint64_t interleave(const uint32_t idx[3], const int bits[3])
{
    // axis 0 provides the lowest bit of each round so that consecutive tiles are
    // x-neighbours first
    uint64_t code = 0;
    int pos = 0;
    int maxb = std::max(bits[0], std::max(bits[1], bits[2]));
    for (int b = 0; b < maxb; b++)
        for (int ax = 0; ax < 3; ax++)
            if (b < bits[ax]) code |= (uint64_t)((idx[ax] >> b) & 1u) << pos++;
    return code;
}

// set while layout_build retries with narrower bands (tile did not fit in shared memory)
thread_local int g_bandRowsRetry = 0;

// a band's tile is (bandRows + halo) doubles per staged vector, two vectors at most (engine.cuh);
// B200 gives a CTA 227 KB, the kernel keeps a little static scratch
constexpr size_t TILE_BYTES_MAX = 200 * 1024;

int pick_band_rows(int nCells, int smCount, int packCtas)
{
    if (g_bandRowsRetry) return g_bandRowsRetry;
    if (const char *e = getenv("B200LDU_BAND_ROWS")) {
        int v = atoi(e);
        if (v >= SLICE_ROWS && v % SLICE_ROWS == 0 && v <= 16384) return v;
    }
    // A sweep is one CTA per band, 6 resident per SM (888 slots on B200).  Measured on B200, fused PCG, Mcell-iters/s
    // (profiles/r02_band_rows.txt):
    //   128^3 (2.1 M cells):  512 rows (4.6 waves) 18.8 k | 1024 rows (2.3 waves) 19.2 k | 2368 rows (ONE wave, 886 CTAs) 19.9-20.3 k
    //   161^3 (4.2 M):       1024 rows (4.6 waves) 20.7 k | 2048 rows (2.3 waves) 19.8 k | 2368 rows (two whole waves) 17.7 k
    //   256^3 (16.8 M):      2048 rows (9.2 waves) 23.6 k | 2368 rows (eight whole waves) 23.1 k
    // A mesh that fits one wave is best served by exactly one (every CTA resident at once, 886 partial sums instead of 4096 for
    // the scalar step).  Beyond that, whole waves are the WORST choice -- the CTAs of a wave stage and stream in lock-step, so the
    // SM alternates between a latency-bound and a bandwidth-bound phase -- and 4+ waves of smaller bands, which drift out of
    // phase, are best; the bands grow to 2048 rows as the mesh allows.
    // the packing CTAs of the fused halo send share the grid with the bands: keep bands + packers within the one wave
    const long long slots = (long long)(smCount > 0 ? smCount : 148) * 6 - packCtas;
    const long long maxRows = 2432; // the tile of a band + its halo must leave room for 6 CTAs per SM
    if (nCells <= slots * maxRows) {
        const long long perBand = (nCells + slots - 1) / slots;
        long long rows = ((perBand + SLICE_ROWS - 1) / SLICE_ROWS) * SLICE_ROWS;
        return (int)std::max<long long>(rows, SLICE_ROWS);
    }
    const long long target = nCells / (slots * 4);
    int b = SLICE_ROWS;
    while (b * 2 <= target && b < 2048) b *= 2;
    return b;
}

} // namespace

int layout_build(b200ldu_addr *a, const double *centres)
{
    const int nCells = a->nCells, nFaces = a->nFaces;
    const std::vector<int> &l = a->l, &u = a->u;
    if (nCells <= 0) {
        b200_set_error("layout_build: nCells must be positive");
        return B200LDU_EINVAL;
    }
    for (int f = 0; f < nFaces; f++) {
        if (l[f] < 0 || u[f] >= nCells || l[f] >= u[f] || (f && l[f] < l[f - 1])) {
            b200_set_error("layout_build: face %d violates upper-triangular owner-sorted order", f);
            return B200LDU_EINVAL;
        }
    }
    std::vector<int> ownerStart, losortStart, losort;
    build_owner_start(nCells, l, ownerStart);
    build_losort(nCells, u, losortStart, losort);

    int packCtas = 0;
    for (int p = 0; p < a->nPatches; p++)
        if (p < (int)a->neighbRank.size() && a->neighbRank[p] >= 0) packCtas += (a->patchStart[p + 1] - a->patchStart[p] + PACK_CHUNK - 1) / PACK_CHUNK;
    const int bandRows = pick_band_rows(nCells, a->ctx ? a->ctx->smCount : 148, packCtas);
    const int nBands = (nCells + bandRows - 1) / bandRows;
    const int nPad = nBands * bandRows;
    const int slicesPerBand = bandRows / SLICE_ROWS;
    const int nSlices = nPad / SLICE_ROWS;
    const int nRecv = a->nPatches ? a->patchStart[a->nPatches] : 0;

    // ---- 1. cell renumbering ------------------------------------------------
    std::vector<double> emb; // 3 coordinates per cell
    const double *xyz = centres;
    if (!xyz) {
        std::vector<int> d0, d1, d2, d3;
        bfs_dist(nCells, l, u, ownerStart, losortStart, losort, 0, d0);
        int s1 = argmax(d0);
        bfs_dist(nCells, l, u, ownerStart, losortStart, losort, s1, d1);
        int s2 = argmax(d1);
        bfs_dist(nCells, l, u, ownerStart, losortStart, losort, s2, d2);
        std::vector<int> sum(nCells);
        for (int c = 0; c < nCells; c++) sum[c] = d1[c] + d2[c];
        int s3 = argmax(sum);
        bfs_dist(nCells, l, u, ownerStart, losortStart, losort, s3, d3);
        emb.resize((size_t)3 * nCells);
        for (int c = 0; c < nCells; c++) {
            emb[3 * (size_t)c + 0] = d1[c];
            emb[3 * (size_t)c + 1] = d2[c];
            emb[3 * (size_t)c + 2] = d3[c];
        }
        xyz = emb.data();
    }
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (int c = 0; c < nCells; c++)
        for (int k = 0; k < 3; k++) {
            double v = xyz[3 * (size_t)c + k];
            lo[k] = std::min(lo[k], v);
            hi[k] = std::max(hi[k], v);
        }
    double ext[3];
    for (int k = 0; k < 3; k++) ext[k] = std::max(hi[k] - lo[k], 1e-300);
    int bits[3] = {0, 0, 0};
    {
        long long tiles = 1;
        // tiles of ~one slice (64 rows): slices become small cubes (most of a row's faces stay inside its slice) and Morton order keeps
        // every run of bandRows/64 consecutive tiles a compact brick
        while ((double)nCells / (double)tiles > (double)SLICE_ROWS && bits[0] + bits[1] + bits[2] < 45) {
            int best = 2; // ties go to the last axis so x keeps the longest runs
            double bestExt = -1;
            for (int k = 2; k >= 0; k--) {
                double e = ext[k] / (double)(1 << bits[k]);
                if (e > bestExt * (1 + 1e-9)) {
                    bestExt = e;
                    best = k;
                }
            }
            bits[best]++;
            tiles *= 2;
        }
    }
    std::vector<uint64_t> key(nCells);
#pragma omp parallel for schedule(static)
    for (int c = 0; c < nCells; c++) {
        uint32_t idx[3];
        for (int k = 0; k < 3; k++) {
            double t = (xyz[3 * (size_t)c + k] - lo[k]) / ext[k];
            long long q = (long long)(t * (double)(1 << bits[k]));
            long long mx = (1ll << bits[k]) - 1;
            idx[k] = (uint32_t)std::min(std::max(q, 0ll), mx);
        }
        key[c] = interleave(idx, bits);
    }
    std::vector<int> order(nCells); // banded row -> caller cell
    {
        int kb = bits[0] + bits[1] + bits[2];
        if (kb <= 26) { // counting sort (stable => caller order inside a tile)
            size_t nT = (size_t)1 << kb;
            std::vector<int> cnt(nT + 1, 0);
            for (int c = 0; c < nCells; c++) cnt[key[c] + 1]++;
            for (size_t t = 0; t < nT; t++) cnt[t + 1] += cnt[t];
            for (int c = 0; c < nCells; c++) order[cnt[key[c]]++] = c;
        } else {
            std::iota(order.begin(), order.end(), 0);
            std::stable_sort(order.begin(), order.end(),
                             [&](int x, int y) { return key[x] < key[y]; });
        }
    }
    key.clear();
    key.shrink_to_fit();
    a->perm_h.assign(nCells, 0);
    a->iperm_h.assign(nPad, -1);
    for (int r = 0; r < nCells; r++) {
        a->perm_h[order[r]] = r;
        a->iperm_h[r] = order[r];
    }
    const std::vector<int> &perm = a->perm_h, &iperm = a->iperm_h;

    // cell -> coupled-patch faces, in (patch, patch face) order
    std::vector<int> pfStart((size_t)nCells + 1, 0), pfItem(nRecv);
    for (int i = 0; i < nRecv; i++) pfStart[a->faceCells[i] + 1]++;
    for (int c = 0; c < nCells; c++) pfStart[c + 1] += pfStart[c];
    {
        std::vector<int> cur(pfStart.begin(), pfStart.end() - 1);
        for (int i = 0; i < nRecv; i++) pfItem[cur[a->faceCells[i]]++] = i;
    }

    // ---- 2. slice widths ----------------------------------------------------
    std::vector<uint16_t> sliceW(nSlices, 0), sliceWL(nSlices, 0);
    int bad = 0;
#pragma omp parallel for schedule(static) reduction(+ : bad)
    for (int s = 0; s < nSlices; s++) {
        int wl = 0, wi = 0;
        for (int q = 0; q < SLICE_ROWS; q++) {
            int c = iperm[(size_t)s * SLICE_ROWS + q];
            if (c < 0) continue;
            int nl = (ownerStart[c + 1] - ownerStart[c]) + (losortStart[c + 1] - losortStart[c]);
            int ni = pfStart[c + 1] - pfStart[c];
            wl = std::max(wl, nl);
            wi = std::max(wi, ni);
        }
        if (wl + wi > 65535) bad++;
        sliceWL[s] = (uint16_t)wl;
        sliceW[s] = (uint16_t)(wl + wi);
    }
    if (bad) {
        b200_set_error("layout_build: a row has more than 65535 entries");
        return B200LDU_ELAYOUT;
    }
    std::vector<long long> sliceStart((size_t)nSlices + 1, 0);
    for (int s = 0; s < nSlices; s++)
        sliceStart[s + 1] = sliceStart[s] + (long long)sliceW[s] * SLICE_ROWS;
    const long long nEntries = sliceStart[nSlices];

    // ---- 3. per-band halo lists and entries ---------------------------------
    std::vector<uint16_t> col((size_t)std::max<long long>(nEntries, 1));
    std::vector<int> code((size_t)std::max<long long>(nEntries, 1));
    std::vector<std::vector<int>> halo(nBands);
    int tooWide = 0;
#pragma omp parallel for schedule(dynamic, 4) reduction(+ : tooWide)
    for (int b = 0; b < nBands; b++) {
        const int r0 = b * bandRows, r1 = r0 + bandRows;
        std::vector<int> &h = halo[b];
        for (int r = r0; r < r1; r++) {
            int c = iperm[r];
            if (c < 0) continue;
            for (int f = ownerStart[c]; f < ownerStart[c + 1]; f++) {
                int t = perm[u[f]];
                if (t < r0 || t >= r1) h.push_back(t);
            }
            for (int k = losortStart[c]; k < losortStart[c + 1]; k++) {
                int t = perm[l[losort[k]]];
                if (t < r0 || t >= r1) h.push_back(t);
            }
            for (int k = pfStart[c]; k < pfStart[c + 1]; k++) h.push_back(nPad + pfItem[k]);
        }
        std::sort(h.begin(), h.end());
        h.erase(std::unique(h.begin(), h.end()), h.end());
        if ((long long)bandRows + (long long)h.size() > 65536) {
            tooWide++;
            continue;
        }
        auto colOf = [&](int t) -> uint16_t {
            if (t >= r0 && t < r1) return (uint16_t)(t - r0);
            int pos = (int)(std::lower_bound(h.begin(), h.end(), t) - h.begin());
            return (uint16_t)(bandRows + pos);
        };
        for (int sl = 0; sl < slicesPerBand; sl++) {
            int s = b * slicesPerBand + sl;
            long long base = sliceStart[s];
            int W = sliceW[s], WL = sliceWL[s];
            for (int q = 0; q < SLICE_ROWS; q++) {
                int r = s * SLICE_ROWS + q;
                int c = iperm[r];
                uint16_t self = (uint16_t)(r - r0);
                int j = 0;
                if (c >= 0) {
                    for (int f = ownerStart[c]; f < ownerStart[c + 1]; f++, j++) {
                        col[base + (long long)j * SLICE_ROWS + q] = colOf(perm[u[f]]);
                        code[base + (long long)j * SLICE_ROWS + q] = 2 * f;
                    }
                    for (int k = losortStart[c]; k < losortStart[c + 1]; k++, j++) {
                        int f = losort[k];
                        col[base + (long long)j * SLICE_ROWS + q] = colOf(perm[l[f]]);
                        code[base + (long long)j * SLICE_ROWS + q] = 2 * f + 1;
                    }
                }
                for (; j < WL; j++) { // padding: zero coefficient, own column
                    col[base + (long long)j * SLICE_ROWS + q] = self;
                    code[base + (long long)j * SLICE_ROWS + q] = -1;
                }
                if (c >= 0) {
                    for (int k = pfStart[c]; k < pfStart[c + 1]; k++, j++) {
                        col[base + (long long)j * SLICE_ROWS + q] = colOf(nPad + pfItem[k]);
                        code[base + (long long)j * SLICE_ROWS + q] = -2 - pfItem[k];
                    }
                }
                for (; j < W; j++) {
                    col[base + (long long)j * SLICE_ROWS + q] = self;
                    code[base + (long long)j * SLICE_ROWS + q] = -1;
                }
            }
        }
    }
    if (tooWide) {
        if (bandRows > SLICE_ROWS) { // retry with narrower bands (see the tile check below)
            const int saved = g_bandRowsRetry;
            g_bandRowsRetry = bandRows / 2;
            int rc = layout_build(a, centres);
            g_bandRowsRetry = saved;
            return rc;
        }
        b200_set_error("layout_build: %d band(s) of %d rows reference more than 65535 distinct columns",
                       tooWide, bandRows);
        return B200LDU_ELAYOUT;
    }
    std::vector<int> haloStart((size_t)nBands + 1, 0);
    int maxHalo = 0;
    for (int b = 0; b < nBands; b++) {
        haloStart[b + 1] = haloStart[b] + (int)halo[b].size();
        maxHalo = std::max(maxHalo, (int)halo[b].size());
    }
    if ((size_t)(bandRows + maxHalo + 2) * 2 * sizeof(double) > TILE_BYTES_MAX) {
        // poorly clustered numbering (no cell centres, high-degree graph): the halo of a band does not fit
        // next to its rows in shared memory.  Narrower bands shrink both terms; the ordering is unchanged.
        if (bandRows > SLICE_ROWS) {
            const int saved = g_bandRowsRetry;
            g_bandRowsRetry = bandRows / 2;
            int rc = layout_build(a, centres);
            g_bandRowsRetry = saved;
            return rc;
        }
        b200_set_error("layout_build: a band of %d rows references %d outside columns: the tile does not fit in "
                       "shared memory; pass cell centres (or renumber the mesh) so that neighbours are close",
                       bandRows, maxHalo);
        return B200LDU_ELAYOUT;
    }
    std::vector<int> haloIdx((size_t)std::max(haloStart[nBands], 1));
#pragma omp parallel for schedule(static)
    for (int b = 0; b < nBands; b++)
        std::copy(halo[b].begin(), halo[b].end(), haloIdx.begin() + haloStart[b]);

    std::vector<int> sendRows(std::max(nRecv, 1));
    for (int i = 0; i < nRecv; i++) sendRows[i] = perm[a->faceCells[i]];

    a->nEntries = nEntries;
    a->nHaloTotal = haloStart[nBands];
    a->vecLen = ((long long)nPad + nRecv + 1) & ~1ll;
    a->L.nCells = nCells;
    a->L.nPad = nPad;
    a->L.nBands = nBands;
    a->L.bandRows = bandRows;
    a->L.slicesPerBand = slicesPerBand;
    a->L.nRecv = nRecv;
    a->L.maxHalo = maxHalo;
    if (a->hostOnly) { // structural self-check path (tests): keep the host arrays, no GPU
        a->dbg_sliceStart.swap(sliceStart);
        a->dbg_sliceW.swap(sliceW);
        a->dbg_sliceWL.swap(sliceWL);
        a->dbg_col.swap(col);
        a->dbg_code.swap(code);
        a->dbg_haloStart.swap(haloStart);
        a->dbg_haloIdx.swap(haloIdx);
        return B200LDU_OK;
    }

    // ---- 4. upload ----------------------------------------------------------
    TRY(a->d_sliceStart.upload(sliceStart));
    TRY(a->d_sliceW.upload(sliceW));
    TRY(a->d_sliceWL.upload(sliceWL));
    TRY(a->d_col.upload(col));
    TRY(a->d_code.upload(code));
    TRY(a->d_haloStart.upload(haloStart));
    TRY(a->d_haloIdx.upload(haloIdx));
    TRY(a->d_perm.upload(a->perm_h));
    TRY(a->d_iperm.upload(a->iperm_h));
    TRY(a->d_sendRows.upload(sendRows));
    TRY(a->d_l.upload(a->l));
    TRY(a->d_u.upload(a->u));
    TRY(a->d_ownerStart.upload(ownerStart));
    TRY(a->d_losort.upload(losort));
    TRY(a->d_losortStart.upload(losortStart));

    LayoutDev &L = a->L;
    L.nCells = nCells;
    L.nPad = nPad;
    L.nBands = nBands;
    L.bandRows = bandRows;
    L.slicesPerBand = slicesPerBand;
    L.nRecv = nRecv;
    L.maxHalo = maxHalo;
    L.sliceStart = a->d_sliceStart.get();
    L.sliceW = a->d_sliceW.get();
    L.sliceWL = a->d_sliceWL.get();
    L.col = a->d_col.get();
    L.haloStart = a->d_haloStart.get();
    L.haloIdx = a->d_haloIdx.get();
    L.perm = a->d_perm.get();
    L.iperm = a->d_iperm.get();
    a->nEntries = nEntries;
    a->nHaloTotal = haloStart[nBands];
    a->vecLen = ((long long)nPad + nRecv + 1) & ~1ll;
    return B200LDU_OK;
}

// ---------------------------------------------------------------------------
// structural self-check entry points (host only; used by the CPU test-suite to verify
// the renumbering and the banded entries without a GPU -- no arithmetic happens here)
// ---------------------------------------------------------------------------
extern "C" int b200ldu_layout_debug_create(int nCells, int nFaces, const int *lower_h, const int *upper_h,
                                           int nPatches, const int *patchStart_h, const int *faceCells_h,
                                           const double *cellCentres_h, b200ldu_addr **out)
{
    if (!out || nCells <= 0) return B200LDU_EINVAL;
    std::unique_ptr<b200ldu_addr> a(new b200ldu_addr()); // plain delete: no CUDA call on this path
    a->hostOnly = true;
    a->nCells = nCells;
    a->nFaces = nFaces;
    a->l.assign(lower_h, lower_h + nFaces);
    a->u.assign(upper_h, upper_h + nFaces);
    a->nPatches = nPatches;
    if (nPatches) {
        a->patchStart.assign(patchStart_h, patchStart_h + nPatches + 1);
        a->faceCells.assign(faceCells_h, faceCells_h + a->patchStart[nPatches]);
    }
    TRY(layout_build(a.get(), cellCentres_h));
    *out = a.release();
    return B200LDU_OK;
}

// what: 0 perm(int32) 1 iperm(int32) 2 sliceStart(int64) 3 sliceW(u16) 4 sliceWL(u16) 5 col(u16)
//       6 code(int32) 7 haloStart(int32) 8 haloIdx(int32) 9 dims {nPad,nBands,bandRows,nRecv,maxHalo}(int32)
// returns the element count (copies min(count, cap) elements when out != NULL)
extern "C" long long b200ldu_layout_debug_get(const b200ldu_addr *a, int what, void *out, long long cap)
{
    if (!a || !a->hostOnly) return -1;
    auto give = [&](const void *src, size_t elem, long long n) -> long long {
        if (out) memcpy(out, src, elem * (size_t)std::min(n, cap));
        return n;
    };
    int dims[5] = {a->L.nPad, a->L.nBands, a->L.bandRows, a->L.nRecv, a->L.maxHalo};
    switch (what) {
    case 0: return give(a->perm_h.data(), 4, (long long)a->perm_h.size());
    case 1: return give(a->iperm_h.data(), 4, (long long)a->iperm_h.size());
    case 2: return give(a->dbg_sliceStart.data(), 8, (long long)a->dbg_sliceStart.size());
    case 3: return give(a->dbg_sliceW.data(), 2, (long long)a->dbg_sliceW.size());
    case 4: return give(a->dbg_sliceWL.data(), 2, (long long)a->dbg_sliceWL.size());
    case 5: return give(a->dbg_col.data(), 2, a->nEntries);
    case 6: return give(a->dbg_code.data(), 4, a->nEntries);
    case 7: return give(a->dbg_haloStart.data(), 4, (long long)a->dbg_haloStart.size());
    case 8: return give(a->dbg_haloIdx.data(), 4, a->nHaloTotal);
    case 9: return give(dims, 4, 5);
    }
    return -1;
}

extern "C" int b200ldu_layout_debug_destroy(b200ldu_addr *a)
{
    if (a && a->hostOnly) delete a;
    return B200LDU_OK;
}
