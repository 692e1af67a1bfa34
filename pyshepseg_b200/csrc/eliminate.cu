// eliminate.cu -- K4..K8: single-pixel elimination, per-segment spectra, pixel lists and the
// small-segment merge passes, plus the order-preserving relabel.
// Replaces shepseg.eliminateSinglePixels / mergeSinglePixels / findNearestNeighbourPixel
// (shepseg.py:572-736), relabelSegments (739-777), buildSegmentSpectra (780-813),
// makeSegmentLocations (880-915), eliminateSmallSegments / findMergeSegment / doMerge
// (918-1123).
//
// The reference is a chain of sequential loops; what makes it data parallel is that every
// decision phase reads a frozen state (shepseg.py:649-660 and 983-986) and every apply phase
// only depends on order within one target segment (ascending source id, shepseg.py:989-994).
// The kernels keep exactly those two orders and nothing else:
//   * single pixels: per round a decide kernel over the candidates, then an apply kernel;
//   * spectra: exact integer band sums by warp-aggregated 64-bit atomics; a float32 running
//     sum of non-negative integers is exact in any order while the total stays below 2^24,
//     so only segments above that take the ordered float32 chain (raster order, one thread
//     per (segment, band));
//   * pixel lists: every small segment's pixels in raster order, in a region of minSegSize-1
//     entries of its own, or, where the regions would take too much memory, in a slice of a
//     packed array (merge.cuh describes both);
//   * passes: the targetSize loop itself runs in merge.cu, a few persistent launches in all,
//     so that ~100 passes do not cost ~500 launches and host round trips.
#include "common.cuh"
#include "merge.cuh"

#include <stdlib.h>
#include <type_traits>
#include <cub/device/device_scan.cuh>

// ====================================================================================
// single pixels
// ====================================================================================
// findNearestNeighbourPixel (shepseg.py:677-736): rows outer, columns inner, first strict
// minimum of the int64 squared distance, only neighbours whose segment has more than one pixel.
// The loads go out level by level (labels, sizes, then one band of all neighbours at a time) so
// that their latencies overlap.
// The label raster itself is not touched while single pixels move (scattered 4-byte stores into a
// raster of tens of megabytes are what this GPU does worst: each is a read-modify-write of a DRAM
// sector): a moved pixel's OLD id has size 0 and moveTo[old id] names the segment it joined, and
// whoever looks at such a pixel follows that link (stored + 1; 0 = not moved).  The raster catches up in the relabel that
// ends the stage (shepseg.py:615), which rewrites every label anyway.
template <typename T, bool FOUR>
__device__ bool nearest_neighbour(const T *__restrict__ img, int nB, int64_t nRows, int64_t nCols,
                                  const unsigned *__restrict__ seg,
                                  const unsigned *__restrict__ segSize,
                                  const unsigned *__restrict__ moveTo, int64_t p,
                                  unsigned *newSeg)
{
    const int64_t N = nRows * nCols;
    const int64_t i = p / nCols, j = p % nCols;
    unsigned sn[8], sz[8];
    int64_t qi[8];
    bool ok[8];
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const int w = q < 4 ? q : q + 1;            // window cell, centre skipped
        const int dy = w / 3 - 1, dx = w % 3 - 1;
        const int64_t ii = i + dy, jj = j + dx;
        ok[q] = ii >= 0 && ii < nRows && jj >= 0 && jj < nCols && !(FOUR && dy != 0 && dx != 0);
        qi[q] = ok[q] ? ii * nCols + jj : p;
        sn[q] = ok[q] ? seg[qi[q]] : 0u;
    }
#pragma unroll
    for (int q = 0; q < 8; q++) sz[q] = ok[q] ? segSize[sn[q]] : 0u;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        if (ok[q] && sz[q] == 0) {          // a single pixel that moved in an earlier round
            sn[q] = moveTo[sn[q]] - 1u;       // (stored + 1: segment 0, the null segment, is a possible target)
            sz[q] = segSize[sn[q]];
        }
    }
    bool any = false;
#pragma unroll
    for (int q = 0; q < 8; q++) { ok[q] = ok[q] && sz[q] > 1; any |= ok[q]; }
    *newSeg = 0;
    if (!any) return false;
    unsigned long long d[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // wraps like the reference's int64
    for (int b = 0; b < nB; b++) {
        const T *plane = img + (size_t)b * N;
        if constexpr (sizeof(T) == 4) {
            // the difference is exact in int64; its square (up to 2^64) and the sum wrap
            const long long own = (long long)plane[p];
#pragma unroll
            for (int q = 0; q < 8; q++) {
                if (!ok[q]) continue;
                const unsigned long long df = (unsigned long long)(own - (long long)plane[qi[q]]);
                d[q] += df * df;
            }
        } else {
            const int own = (int)plane[p];
#pragma unroll
            for (int q = 0; q < 8; q++) {
                if (!ok[q]) continue;
                const int df = own - (int)plane[qi[q]];
                d[q] += (unsigned long long)((long long)df * (long long)df);
            }
        }
    }
    long long minD = -1;
    unsigned best = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        if (!ok[q]) continue;
        const long long dq = (long long)d[q];
        if (minD < 0 || dq < minD) { minD = dq; best = sn[q]; }
    }
    *newSeg = best;
    return true;
}

// decide phase of mergeSinglePixels (shepseg.py:649-660).  candIn == nullptr: scan every
// pixel (first round); otherwise scan the pixels left over from the previous round.
template <typename T, bool FOUR>
__global__ void __launch_bounds__(256)
k_single_decide(const T *__restrict__ img, int nB, int64_t nRows, int64_t nCols,
                const unsigned *__restrict__ seg, const unsigned *__restrict__ segSize,
                const unsigned *__restrict__ moveTo,
                const unsigned *__restrict__ candIn, int64_t nIn, unsigned *moveOld,
                unsigned *moveSeg, unsigned *candOut, unsigned long long *counters)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool cand = false;
    int64_t p = 0;
    unsigned own = 0;
    if (t < nIn) {
        p = candIn ? (int64_t)candIn[t] : t;
        own = seg[p];
        cand = segSize[own] == 1;      // (a pixel that has moved has size 0 under its old id)
    }
    unsigned newSeg = 0;
    bool found = false;
    if (cand) found = nearest_neighbour<T, FOUR>(img, nB, nRows, nCols, seg, segSize, moveTo, p, &newSeg);
    unsigned long long s0 = warp_claim(&counters[C_NUM_MOVES], cand && found);
    if (cand && found) { moveOld[s0] = own; moveSeg[s0] = newSeg; }
    unsigned long long s1 = warp_claim(&counters[C_NUM_LEFT], cand && !found);
    if (cand && !found) candOut[s1] = (unsigned)p;
}

// apply phase (shepseg.py:664-672), on the per-segment tables only
__global__ void __launch_bounds__(256)
k_single_apply(const unsigned *__restrict__ moveOld, const unsigned *__restrict__ moveSeg,
               int64_t n, unsigned *moveTo, unsigned *segSize)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const unsigned old = moveOld[t], ns = moveSeg[t];
    moveTo[old] = ns + 1u;
    segSize[old] = 0;
    atomicAdd(&segSize[ns], 1u);
}

__global__ void __launch_bounds__(256)
k_count_size_eq(const unsigned *__restrict__ segSize, int64_t lo, int64_t len, unsigned value,
                unsigned long long *counter)
{
    const int64_t s = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool hit = s < len && segSize[s] == value;
    block_add(counter, hit ? 1u : 0u);
}

template <typename T>
static int eliminate_single_t(ssg_ctx *ctx, const T *img, int nB, int64_t nRows, int64_t nCols,
                              const unsigned *seg, unsigned *segSize, int64_t len, int four,
                              int64_t *numMoved, unsigned *numRounds, const unsigned *cand0,
                              int64_t nCand0, const unsigned **moveToOut)
{
    const int64_t N = nRows * nCols;
    unsigned long long *counters = bufp<unsigned long long>(ctx->counters);
    *numMoved = 0;
    *numRounds = 0;
    *moveToOut = nullptr;
    if (N == 0) return SSG_OK;
    // how many single-pixel segments are there (the lone null pixel counts, shepseg.py:652)
    int64_t nSingles = nCand0;
    if (cand0 == nullptr || nCand0 < 0) {
        cand0 = nullptr;
        SSG_CUDA(ctx, cudaMemsetAsync(counters + C_NUM_SINGLES, 0, sizeof(unsigned long long), ctx->stream));
        SSG_PROF_BEGIN(ctx, "k_count_size_eq");
        k_count_size_eq<<<gridFor(len, 256), 256, 0, ctx->stream>>>(segSize, 0, len, 1u, counters + C_NUM_SINGLES);
        SSG_LAUNCHED(ctx);
        SSG_TRY(ssg_fetch_counters(ctx));
        nSingles = (int64_t)ctx->hostCounters[C_NUM_SINGLES];
    }
    if (nSingles == 0) return SSG_OK;
    const size_t cap = (size_t)nSingles * sizeof(unsigned);
    SSG_TRY(ssg_reserve(ctx, ctx->aux0, cap));
    SSG_TRY(ssg_reserve(ctx, ctx->aux1, cap));
    SSG_TRY(ssg_reserve(ctx, ctx->aux2, 2 * cap));
    SSG_TRY(ssg_reserve(ctx, ctx->mergeTo, (size_t)len * sizeof(unsigned)));
    unsigned *moveOld = bufp<unsigned>(ctx->aux0), *moveSeg = bufp<unsigned>(ctx->aux1);
    unsigned *candA = bufp<unsigned>(ctx->aux2), *candB = candA + nSingles;
    unsigned *moveTo = bufp<unsigned>(ctx->mergeTo);
    SSG_CUDA(ctx, cudaMemsetAsync(moveTo, 0, (size_t)len * sizeof(unsigned), ctx->stream));

    const unsigned *candIn = cand0;
    int64_t nIn = cand0 ? nSingles : N;
    unsigned *candOut = candA;
    while (true) {
        SSG_CUDA(ctx, cudaMemsetAsync(counters + C_NUM_MOVES, 0, 2 * sizeof(unsigned long long), ctx->stream));
        SSG_PROF_BEGIN(ctx, "k_single_decide");
        if (four)
            k_single_decide<T, true><<<gridFor(nIn, 256), 256, 0, ctx->stream>>>(img, nB, nRows, nCols, seg, segSize, moveTo,
                                                                                 candIn, nIn, moveOld, moveSeg, candOut, counters);
        else
            k_single_decide<T, false><<<gridFor(nIn, 256), 256, 0, ctx->stream>>>(img, nB, nRows, nCols, seg, segSize, moveTo,
                                                                                  candIn, nIn, moveOld, moveSeg, candOut, counters);
        SSG_LAUNCHED(ctx);
        SSG_TRY(ssg_fetch_counters(ctx));
        const int64_t nMoves = (int64_t)ctx->hostCounters[C_NUM_MOVES];
        const int64_t nLeft = (int64_t)ctx->hostCounters[C_NUM_LEFT];
        (*numRounds)++;
        if (nMoves == 0) break;   // the reference's last, empty round (shepseg.py:610)
        SSG_PROF_BEGIN(ctx, "k_single_apply");
        k_single_apply<<<gridFor(nMoves, 256), 256, 0, ctx->stream>>>(moveOld, moveSeg, nMoves, moveTo, segSize);
        SSG_LAUNCHED(ctx);
        *numMoved += nMoves;
        if (nLeft == 0) { (*numRounds)++; break; }   // nothing left to examine: the empty round is implied
        candIn = candOut;
        nIn = nLeft;
        candOut = (candOut == candA) ? candB : candA;
    }
    if (*numMoved > 0) *moveToOut = moveTo;
    return SSG_OK;
}

// seg is NOT modified: *moveToOut (len entries, scratch of this call; nullptr if nothing moved) maps
// the old id of every moved pixel to the segment it joined and must be handed to ssgk_relabel
int ssgk_eliminate_single(ssg_ctx *ctx, const void *imgDev, int dtype, int nBands, int64_t nRows,
                          int64_t nCols, const uint32_t *segDev, uint32_t *sizeDev, int64_t len,
                          int four, int64_t *numMoved, uint32_t *numRounds, const uint32_t **moveToOut,
                          const unsigned *cand0, int64_t nCand0)
{
    switch (dtype) {
    case SSG_U8: return eliminate_single_t<uint8_t>(ctx, (const uint8_t *)imgDev, nBands, nRows, nCols, segDev, sizeDev, len, four, numMoved, numRounds, cand0, nCand0, moveToOut);
    case SSG_U16: return eliminate_single_t<uint16_t>(ctx, (const uint16_t *)imgDev, nBands, nRows, nCols, segDev, sizeDev, len, four, numMoved, numRounds, cand0, nCand0, moveToOut);
    case SSG_I16: return eliminate_single_t<int16_t>(ctx, (const int16_t *)imgDev, nBands, nRows, nCols, segDev, sizeDev, len, four, numMoved, numRounds, cand0, nCand0, moveToOut);
    case SSG_U32: return eliminate_single_t<uint32_t>(ctx, (const uint32_t *)imgDev, nBands, nRows, nCols, segDev, sizeDev, len, four, numMoved, numRounds, cand0, nCand0, moveToOut);
    case SSG_I32: return eliminate_single_t<int32_t>(ctx, (const int32_t *)imgDev, nBands, nRows, nCols, segDev, sizeDev, len, four, numMoved, numRounds, cand0, nCand0, moveToOut);
    default: SSG_FAIL(ctx, SSG_ERR_ARG, "unsupported dtype code %d", dtype);
    }
}

// ====================================================================================
// relabelSegments (shepseg.py:739-777): new = old - #{j in [minSegId, old-1] : size[j]==0}
// ====================================================================================
__global__ void __launch_bounds__(256)
k_zero_flags(const unsigned *__restrict__ segSize, int64_t len, unsigned minSegId, unsigned *flag)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < len) flag[s] = (s >= minSegId && segSize[s] == 0) ? 1u : 0u;
}

// lut[s] = s - (zeros before s); also the number of ids >= minSegId that own pixels
__global__ void __launch_bounds__(256)
k_make_lut(const unsigned *__restrict__ zerosBefore, const unsigned *__restrict__ segSize,
           int64_t len, unsigned minSegId, unsigned *lut, unsigned long long *counters)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool alive = false;
    if (s < len) {
        lut[s] = (unsigned)s - zerosBefore[s];
        alive = s >= minSegId && segSize[s] != 0;
    }
    block_add(&counters[C_NUM_ALIVE], alive ? 1u : 0u);
}

__global__ void __launch_bounds__(256)
k_apply_lut(unsigned *seg, int64_t N, const unsigned *__restrict__ lut)
{
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t p0 = g * 4;
    if (p0 + 4 <= N && ((uintptr_t)seg % 16 == 0)) {
        uint4 v = *reinterpret_cast<uint4 *>(seg + p0);
        v.x = __ldg(lut + v.x); v.y = __ldg(lut + v.y); v.z = __ldg(lut + v.z); v.w = __ldg(lut + v.w);
        *reinterpret_cast<uint4 *>(seg + p0) = v;
    } else {
        for (int64_t p = p0; p < p0 + 4 && p < N; p++) seg[p] = __ldg(lut + seg[p]);
    }
}

// sizes of the surviving ids at their new positions (segSize of the compacted numbering)
__global__ void __launch_bounds__(256)
k_compact_sizes(const unsigned *__restrict__ segSize, const unsigned *__restrict__ lut, int64_t len,
                unsigned minSegId, unsigned *sizeOut)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= len) return;
    const unsigned z = segSize[s];
    if (s < minSegId) sizeOut[s] = z;          // ids below minSegId keep their place (a null id whose one pixel moved: 0)
    else if (z != 0) sizeOut[lut[s]] = z;
}

// ids whose pixels have moved elsewhere take the new id of the segment they joined
__global__ void __launch_bounds__(256)
k_redirect_lut(const unsigned *__restrict__ segSize, const unsigned *__restrict__ moveTo, int64_t len, unsigned *lut)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= len) return;
    const unsigned to = moveTo[s];
    if (to != 0 && segSize[s] == 0) lut[s] = lut[to - 1u];     // (the target is alive: its entry is final)
}

int ssgk_relabel(ssg_ctx *ctx, uint32_t *segDev, int64_t N, const uint32_t *sizeDev, int64_t len,
                 uint32_t minSegId, uint32_t *numAlive, uint32_t *sizeOutDev, const uint32_t **lutOut,
                 const uint32_t *moveTo)
{
    if (lutOut) *lutOut = nullptr;
    unsigned long long *counters = bufp<unsigned long long>(ctx->counters);
    *numAlive = 0;
    if (len <= 0) return SSG_OK;
    SSG_TRY(ssg_reserve(ctx, ctx->lut, (size_t)len * 2 * sizeof(unsigned)));
    unsigned *flag = bufp<unsigned>(ctx->lut), *lut = flag + len;
    SSG_PROF_BEGIN(ctx, "k_zero_flags");
    k_zero_flags<<<gridFor(len, 256), 256, 0, ctx->stream>>>(sizeDev, len, minSegId, flag);
    SSG_LAUNCHED(ctx);
    size_t tmpBytes = 0;
    SSG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes, flag, flag, (int)len, ctx->stream));
    SSG_TRY(ssg_reserve(ctx, ctx->cubTemp, tmpBytes));
    SSG_PROF_BEGIN(ctx, "cub_DeviceScan_ExclusiveSum");
    SSG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->cubTemp.p, tmpBytes, flag, flag, (int)len, ctx->stream));
    SSG_LAUNCHED(ctx);
    SSG_CUDA(ctx, cudaMemsetAsync(counters + C_NUM_ALIVE, 0, sizeof(unsigned long long), ctx->stream));
    SSG_PROF_BEGIN(ctx, "k_make_lut");
    k_make_lut<<<gridFor(len, 256), 256, 0, ctx->stream>>>(flag, sizeDev, len, minSegId, lut, counters);
    SSG_LAUNCHED(ctx);
    if (moveTo) {
        SSG_PROF_BEGIN(ctx, "k_redirect_lut");
        k_redirect_lut<<<gridFor(len, 256), 256, 0, ctx->stream>>>(sizeDev, moveTo, len, lut);
        SSG_LAUNCHED(ctx);
    }
    if (lutOut) *lutOut = lut;        // the caller applies it (in a pass it makes over the labels anyway)
    else if (N > 0) {
        SSG_PROF_BEGIN(ctx, "k_apply_lut");
        k_apply_lut<<<gridFor((N + 3) / 4, 256), 256, 0, ctx->stream>>>(segDev, N, lut);
        SSG_LAUNCHED(ctx);
    }
    if (sizeOutDev) {
        SSG_PROF_BEGIN(ctx, "k_compact_sizes");
        k_compact_sizes<<<gridFor(len, 256), 256, 0, ctx->stream>>>(sizeDev, lut, len, minSegId, sizeOutDev);
        SSG_LAUNCHED(ctx);
    }
    SSG_TRY(ssg_fetch_counters(ctx));
    *numAlive = (uint32_t)ctx->hostCounters[C_NUM_ALIVE];
    return SSG_OK;
}

// ====================================================================================
// per-segment spectra (buildSegmentSpectra, shepseg.py:780-813)
// ====================================================================================
// ordered float32 chain for one (segment, band): s = RN32(s + x) in raster order.  One warp
// per chain: the lanes fetch 32 values at a time (the next batch is in flight while the
// current one is added), the adds themselves run in order through shuffles.  The values travel
// as float for 8/16-bit images (exact there) and as double for 32-bit ones.
template <typename T>
__global__ void __launch_bounds__(128)
k_ordered_sums(const T *__restrict__ img, int nB, int64_t N, const unsigned *__restrict__ pixSorted,
               const unsigned *__restrict__ keysSorted, const unsigned *__restrict__ runStart,
               unsigned numRuns, int64_t M, float *fsum)
{
    using X = typename std::conditional<sizeof(T) == 4, double, float>::type;
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned lane = lane_id();
    const int64_t run = w / nB;
    const int b = (int)(w % nB);
    if (run >= numRuns) return;
    const int64_t lo = runStart[run];
    const int64_t hi = (run + 1 < numRuns) ? (int64_t)runStart[run + 1] : M;
    const unsigned s = keysSorted[lo];
    const T *plane = img + (size_t)b * N;
    float acc = 0.0f;
    X next = (lo + lane < hi) ? (X)plane[pixSorted[lo + lane]] : (X)0;
    for (int64_t i0 = lo; i0 < hi; i0 += 32) {
        const X cur = next;
        const int64_t i1 = i0 + 32 + lane;
        next = (i1 < hi) ? (X)plane[pixSorted[i1]] : (X)0;
        const int n = (int)((hi - i0) < 32 ? (hi - i0) : 32);
        for (int k = 0; k < n; k++)
            acc = __double2float_rn((double)acc + (double)__shfl_sync(0xffffffffu, cur, k));
    }
    if (lane == 0) fsum[(size_t)s * nB + b] = acc;
}

// ====================================================================================
// One pass over the pixels for everything the merge stage needs from them
// ====================================================================================
// Per pixel: the pending order-preserving relabel (relabelSegments after the single-pixel stage,
// shepseg.py:615 -- applied here instead of in a pass of its own), the band sums of
// buildSegmentSpectra (shepseg.py:780-813) as exact integers, and the pixel lists of the small
// segments (makeSegmentLocations, shepseg.py:880-915).  A thread takes V consecutive pixels
// with one wide load per plane, aggregates its own runs of equal labels in registers and issues
// one atomic per run and band PAIR: two unsigned bands share a 64-bit word (32 bits each; a
// half can only overflow in a segment of more than 2^32 / maxValue pixels, and such a segment
// takes the ordered path below anyway, which recomputes every band).  32-bit values get one
// 64-bit sum per band, with 64-bit run partials.
//   lutF[old] = new id | (1u << 31 if the segment is small, i.e. its pixels are listed)
template <typename T>
__device__ __forceinline__ void load4(const T *p, unsigned (&x)[4])
{
    if constexpr (sizeof(T) == 2) {
        const uint2 r = __ldg(reinterpret_cast<const uint2 *>(p));
        const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
        for (int i = 0; i < 4; i++) x[i] = (unsigned)(int)e[i];      // sign-extended for int16
    } else {
        const unsigned r = __ldg(reinterpret_cast<const unsigned *>(p));
        const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
        for (int i = 0; i < 4; i++) x[i] = (unsigned)(int)e[i];
    }
}

template <typename T, bool PACKED>
__device__ __forceinline__ void add_band_pair(unsigned long long *isum, int NP, int nB, int j, unsigned id,
                                              unsigned a, unsigned b)
{
    if (PACKED) atomicAdd(&isum[(size_t)id * NP + j], (unsigned long long)a | ((unsigned long long)b << 32));
    else {      // signed values: one 64-bit sum per band (a, b are sign-extended 32-bit partial sums)
        atomicAdd(&isum[(size_t)id * NP + 2 * j], (unsigned long long)(long long)(int)a);
        if (2 * j + 1 < nB) atomicAdd(&isum[(size_t)id * NP + 2 * j + 1], (unsigned long long)(long long)(int)b);
    }
}

template <typename T, bool PACKED>
__global__ void __launch_bounds__(256)
k_pixel_pass(const T *__restrict__ img, int nB, int64_t N, unsigned *seg, const unsigned *__restrict__ lutF,
             int writeSeg, int vec, unsigned long long *isum, const unsigned *__restrict__ sliceOff, unsigned *fill,
             unsigned *pix)
{
    const int NP = PACKED ? (nB + 1) / 2 : nB;      // words per segment in isum
    const int nPairs = (nB + 1) / 2;
    const int64_t nGroups = (N + 3) / 4;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < nGroups; g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p0 = g * 4;
        if (vec && p0 + 4 <= N) {
            const uint4 o = *reinterpret_cast<const uint4 *>(seg + p0);
            unsigned s[4];
            s[0] = __ldg(lutF + o.x); s[1] = __ldg(lutF + o.y); s[2] = __ldg(lutF + o.z); s[3] = __ldg(lutF + o.w);
            if (writeSeg)
                *reinterpret_cast<uint4 *>(seg + p0) = make_uint4(s[0] & 0x7fffffffu, s[1] & 0x7fffffffu,
                                                                  s[2] & 0x7fffffffu, s[3] & 0x7fffffffu);
            // runs of equal labels among my four pixels
            bool last[4];
            last[0] = s[1] != s[0]; last[1] = s[2] != s[1]; last[2] = s[3] != s[2]; last[3] = true;
            // pixel lists of the small segments: one slot claim per run (any order: sorted afterwards)
            if ((s[0] | s[1] | s[2] | s[3]) >> 31) {
                unsigned base = 0, pos = 0;
#pragma unroll
                for (int v = 0; v < 4; v++) {
                    const bool head = v == 0 || last[v > 0 ? v - 1 : 0];
                    const unsigned id = s[v] & 0x7fffffffu;
                    if (head) {
                        pos = 0;
                        if (s[v] >> 31) {
                            unsigned n = 1;
#pragma unroll
                            for (int w = v; w < 3; w++) {
                                bool cont = true;
#pragma unroll
                                for (int z = v; z <= w; z++) cont = cont && !last[z];
                                n += cont ? 1u : 0u;
                            }
                            base = atomicAdd(&fill[id], n) + __ldg(sliceOff + id);
                        }
                    }
                    if (s[v] >> 31) pix[base + pos] = (unsigned)(p0 + v);
                    pos++;
                }
            }
            if constexpr (sizeof(T) == 4) {
                // band sums: one atomic per run and band
                for (int b = 0; b < nB; b++) {
                    const uint4 r = __ldg(reinterpret_cast<const uint4 *>(img + (size_t)b * N + p0));
                    const T *e = reinterpret_cast<const T *>(&r);
                    long long a = 0;
#pragma unroll
                    for (int v = 0; v < 4; v++) {
                        a += (long long)e[v];       // zero-extended for uint32, sign-extended for int32
                        if (last[v]) {
                            const unsigned id = s[v] & 0x7fffffffu;
                            if (id != 0) atomicAdd(&isum[(size_t)id * nB + b], (unsigned long long)a);
                            a = 0;
                        }
                    }
                }
            } else {
                // band sums: one atomic per run and band pair
                for (int j = 0; j < nPairs; j++) {
                    unsigned xa[4], xb[4];
                    load4<T>(img + (size_t)(2 * j) * N + p0, xa);
                    if (2 * j + 1 < nB) load4<T>(img + (size_t)(2 * j + 1) * N + p0, xb);
                    else { xb[0] = xb[1] = xb[2] = xb[3] = 0; }
                    unsigned a = 0, b = 0;
#pragma unroll
                    for (int v = 0; v < 4; v++) {
                        a += xa[v]; b += xb[v];
                        if (last[v]) {
                            const unsigned id = s[v] & 0x7fffffffu;
                            if (id != 0) add_band_pair<T, PACKED>(isum, NP, nB, j, id, a, b);
                            a = 0; b = 0;
                        }
                    }
                }
            }
        } else {
            for (int v = 0; v < 4 && p0 + v < N; v++) {
                const int64_t p = p0 + v;
                const unsigned sv = __ldg(lutF + seg[p]);
                const unsigned id = sv & 0x7fffffffu;
                if (writeSeg) seg[p] = id;
                if (id == 0) continue;
                if (sv >> 31) pix[__ldg(sliceOff + id) + atomicAdd(&fill[id], 1u)] = (unsigned)p;
                if constexpr (sizeof(T) == 4) {
                    for (int b = 0; b < nB; b++)
                        atomicAdd(&isum[(size_t)id * nB + b], (unsigned long long)(long long)img[(size_t)b * N + p]);
                } else {
                    for (int j = 0; j < nPairs; j++) {
                        const unsigned a = (unsigned)(int)img[(size_t)(2 * j) * N + p];
                        const unsigned b = 2 * j + 1 < nB ? (unsigned)(int)img[(size_t)(2 * j + 1) * N + p] : 0u;
                        add_band_pair<T, PACKED>(isum, NP, nB, j, id, a, b);
                    }
                }
            }
        }
    }
}

// integer sums -> float32 sums where that is exact; flag the segments where it is not
template <bool PACKED, bool SIGNED>
__global__ void __launch_bounds__(256)
k_finalize_sums2(const unsigned long long *__restrict__ isum, const unsigned *__restrict__ segSize,
                 int nB, int64_t len, unsigned maxAbs, float *fsum, unsigned char *bigFlag,
                 unsigned long long *counters)
{
    const int NP = PACKED ? (nB + 1) / 2 : nB;
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool big = false;
    if (s < len) {
        for (int b = 0; b < nB; b++) {
            long long v;
            if (PACKED) {
                const unsigned long long w = isum[(size_t)s * NP + b / 2];
                v = (long long)((b & 1) ? (w >> 32) : (w & 0xffffffffull));
            } else {
                v = (long long)isum[(size_t)s * NP + b];
            }
            fsum[(size_t)s * nB + b] = (float)v;
            if (PACKED) big |= (v >= (1ll << 24));
            else if (!SIGNED) big |= ((unsigned long long)v >= (1ull << 24));
        }
        // packed halves are exact while size * maxValue < 2^32; signed sums may cancel, so there the
        // bound on the running sum decides
        if (PACKED) big |= (unsigned long long)segSize[s] * maxAbs >= (1ull << 32);
        else if (SIGNED) big = (unsigned long long)segSize[s] * maxAbs >= (1ull << 24);
        if (s == 0) big = false;
        bigFlag[s] = big ? 1 : 0;
    }
    block_add(&counters[C_NUM_BIGSUM], big ? 1u : 0u);
}

// lutF[i] = (lut ? lut[i] : i) | small flag of the new id
__global__ void __launch_bounds__(256)
k_flag_lut(const unsigned *__restrict__ lut, int64_t n, const unsigned *__restrict__ sliceLen, int64_t len,
           unsigned *lutF)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned v = lut ? lut[i] : (unsigned)i;
    unsigned f = 0;
    if (v != 0 && (int64_t)v < len && sliceLen[v] != 0) f = 0x80000000u;
    lutF[i] = v | f;
}

// ====================================================================================
// pixel lists and size buckets of the small segments (makeSegmentLocations, shepseg.py:880-915)
// ====================================================================================
#define SMALL_MAX_MINSEG 8192   // size-histogram bins kept in shared memory

// per segment: listed pixel count (its size if 0 < size < minSegSize) for the chunk-offset
// scan, the histogram of those sizes, and the totals
__global__ void __launch_bounds__(256)
k_small_census(const unsigned *__restrict__ segSize, int64_t len, unsigned minSegSize,
               unsigned *cnt /* len + 1 */, unsigned *isSmall /* len + 1 */,
               unsigned *sizeHist /* minSegSize + 1 */, unsigned long long *counters)
{
    extern __shared__ unsigned hist[];
    for (unsigned i = threadIdx.x; i < minSegSize; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned c = 0;
    if (s >= 1 && s < len) {
        const unsigned z = segSize[s];
        if (z > 0 && z < minSegSize) c = z;
    }
    if (s <= len) { cnt[s] = c; isSmall[s] = c ? 1u : 0u; }
    if (c) atomicAdd(&hist[c], 1u);
    block_add(&counters[C_NUM_SMALLSEG], c != 0 ? 1u : 0u);
    block_add(&counters[C_NUM_SMALLPIX], c);
    __syncthreads();
    for (unsigned i = threadIdx.x; i < minSegSize; i += blockDim.x)
        if (hist[i]) atomicAdd(&sizeHist[i], hist[i]);
}

// the small segments grouped by size: bucketList[bucketStart[z] ..) holds the ids of size z
__global__ void __launch_bounds__(256)
k_bucket_fill(const unsigned *__restrict__ segSize, int64_t len, unsigned minSegSize,
              const unsigned *__restrict__ bucketStart, unsigned *bucketFill, unsigned *bucketList)
{
    extern __shared__ unsigned sh[];
    unsigned *hist = sh, *base = sh + minSegSize;
    for (unsigned i = threadIdx.x; i < minSegSize; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned z = 0, myRank = 0;
    if (s >= 1 && s < len) {
        z = segSize[s];
        if (z >= minSegSize) z = 0;
    }
    if (z) myRank = atomicAdd(&hist[z], 1u);
    __syncthreads();
    for (unsigned i = threadIdx.x; i < minSegSize; i += blockDim.x)
        if (hist[i]) base[i] = bucketStart[i] + atomicAdd(&bucketFill[i], hist[i]);
    __syncthreads();
    if (z) bucketList[base[z] + myRank] = (unsigned)s;
}

// per-segment state of the passes.  A small segment's pixel list lives either in a region of its
// own of minSegSize-1 entries (regionCap != 0: the list only ever grows by appending, and cannot
// outgrow the region while the segment is still small) or, when that would take too much memory,
// in a slice of a packed array (merged lists are then copied into an arena or chained, merge.cu).
__global__ void __launch_bounds__(256)
k_list_init(const unsigned *__restrict__ off, const unsigned *__restrict__ smallRank,
            const unsigned *__restrict__ segSize, int64_t len, unsigned minSegSize, unsigned regionCap,
            unsigned *sliceOff, unsigned *sliceLen, unsigned *nextChunk, unsigned *tailChunk,
            unsigned *mergeTo, unsigned *fill)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= len) return;
    const unsigned n = off[s + 1] - off[s];
    sliceOff[s] = regionCap ? smallRank[s] * regionCap : off[s];
    sliceLen[s] = n;
    nextChunk[s] = SSG_NIL;
    tailChunk[s] = (unsigned)s;
    mergeTo[s] = 0;
    fill[s] = 0;
}

// slots were claimed in arbitrary order: put every list back into raster order
__global__ void __launch_bounds__(128)
k_list_sort(const unsigned *__restrict__ sliceOff, const unsigned *__restrict__ sliceLen, int64_t len,
            unsigned *pix)
{
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= len) return;
    const unsigned o = sliceOff[s], n = sliceLen[s];
    for (unsigned i = 1; i < n; i++) {
        unsigned v = pix[o + i];
        unsigned j = i;
        while (j > 0 && pix[o + j - 1] > v) { pix[o + j] = pix[o + j - 1]; j--; }
        pix[o + j] = v;
    }
}

// lut may be null: nothing to relabel
int ssgk_apply_lut(ssg_ctx *ctx, unsigned *seg, int64_t N, const unsigned *lut)
{
    if (!lut || N == 0) return SSG_OK;
    SSG_PROF_BEGIN(ctx, "k_apply_lut");
    k_apply_lut<<<gridFor((N + 3) / 4, 256), 256, 0, ctx->stream>>>(seg, N, lut);
    SSG_LAUNCHED(ctx);
    return SSG_OK;
}

// pendingLut (optional, lutLen entries): an order-preserving relabel of `seg` that has been worked
// out but not applied yet (segSize, maxSegId and everything else refer to the NEW ids); it is
// applied by the pixel pass of this stage, which reads and writes every label anyway.
template <typename T>
static int eliminate_small_t(ssg_ctx *ctx, const T *img, int nB, int64_t nRows, int64_t nCols,
                             unsigned *seg, unsigned *segSize, uint32_t maxSegId, int minSegSize,
                             double thr, int four, int64_t *numElim, uint32_t *numPasses,
                             const unsigned *pendingLut, int64_t lutLen)
{
    const int64_t N = nRows * nCols;
    const int64_t len = (int64_t)maxSegId + 1;
    *numElim = 0;
    *numPasses = 0;
    if (N == 0 || minSegSize <= 1)      // the targetSize loop never runs (shepseg.py:970)
        return ssgk_apply_lut(ctx, seg, N, pendingLut);     // the pending relabel on its own
    if (minSegSize > SMALL_MAX_MINSEG)
        SSG_FAIL(ctx, SSG_ERR_ARG, "minSegmentSize=%d is above the supported maximum of %d", minSegSize, SMALL_MAX_MINSEG);
    unsigned long long *counters = bufp<unsigned long long>(ctx->counters);

    // census of the small segments: listed sizes (-> slice offsets), 0/1 flags (-> rank among the
    // small segments) and the size histogram (-> buckets); the three scans share one scratch
    // array: [off: len+1][rank: len+1][hist: m+1][start: m+1][fill: m+1]
    const size_t m1 = (size_t)minSegSize + 1;
    SSG_TRY(ssg_reserve(ctx, ctx->listOff, (2 * (size_t)(len + 1) + 3 * m1) * sizeof(unsigned)));
    unsigned *off = bufp<unsigned>(ctx->listOff);
    unsigned *smallRank = off + (len + 1);
    unsigned *sizeHist = smallRank + (len + 1), *bucketStart = sizeHist + m1, *bucketFill = bucketStart + m1;
    SSG_CUDA(ctx, cudaMemsetAsync(sizeHist, 0, 3 * m1 * sizeof(unsigned), ctx->stream));
    SSG_CUDA(ctx, cudaMemsetAsync(counters + C_NUM_SMALLSEG, 0, 2 * sizeof(unsigned long long), ctx->stream));
    SSG_PROF_BEGIN(ctx, "k_small_census");
    k_small_census<<<gridFor(len + 1, 256), 256, (size_t)minSegSize * sizeof(unsigned), ctx->stream>>>(
        segSize, len, (unsigned)minSegSize, off, smallRank, sizeHist, counters);
    SSG_LAUNCHED(ctx);
    size_t tmpBytes = 0, tmpBytes2 = 0;
    SSG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes, off, off, (int)(len + 1), ctx->stream));
    SSG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes2, sizeHist, bucketStart, (int)m1, ctx->stream));
    SSG_TRY(ssg_reserve(ctx, ctx->cubTemp, tmpBytes > tmpBytes2 ? tmpBytes : tmpBytes2));
    SSG_PROF_BEGIN(ctx, "cub_DeviceScan_ExclusiveSum");
    SSG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->cubTemp.p, tmpBytes, off, off, (int)(len + 1), ctx->stream));
    SSG_LAUNCHED(ctx);
    SSG_PROF_BEGIN(ctx, "cub_DeviceScan_ExclusiveSum");
    SSG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->cubTemp.p, tmpBytes, smallRank, smallRank, (int)(len + 1), ctx->stream));
    SSG_LAUNCHED(ctx);
    SSG_PROF_BEGIN(ctx, "cub_DeviceScan_ExclusiveSum");
    SSG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->cubTemp.p, tmpBytes2, sizeHist, bucketStart, (int)m1, ctx->stream));
    SSG_LAUNCHED(ctx);
    SSG_TRY(ssg_fetch_counters(ctx));
    const size_t numSmall = (size_t)ctx->hostCounters[C_NUM_SMALLSEG];
    const size_t numSmallPix = (size_t)ctx->hostCounters[C_NUM_SMALLPIX];
    if (numSmall == 0)      // nothing can be a candidate, now or later
        return ssgk_apply_lut(ctx, seg, N, pendingLut);

    // Pixel lists.  By default every small segment gets a region of minSegSize-1 entries of its
    // own: a list only ever grows by appending the lists of merged sources, and it cannot outgrow
    // the region while its segment is still below minSegSize -- so merging never moves the
    // target's pixels, needs no allocation and lists never fragment.  That takes
    // (minSegSize-1) * 4 bytes per small segment (170 MB for a 7908^2 tile at minSegSize=50); if
    // it would exceed the limit (a very large minSegSize) the lists are packed instead and merged
    // lists are copied into an arena of twice their size, chained when that runs out.
    size_t regionLimit = (size_t)8 << 30;
    if (const char *e = getenv("SSG_SMALL_REGION_MB")) regionLimit = (size_t)atoll(e) << 20;
    const size_t regionEntries = numSmall * (size_t)(minSegSize - 1);
    const bool regions = regionEntries * sizeof(unsigned) <= regionLimit && regionEntries < 0xFFFFFFF0ull;
    size_t arenaCap = 0;
    if (!regions) {
        arenaCap = 2 * numSmallPix;
        if (const char *e = getenv("SSG_SMALL_ARENA_PCT")) arenaCap = numSmallPix * (size_t)atoi(e) / 100;
        if (numSmallPix + arenaCap > 0xFFFFFFF0ull) arenaCap = 0xFFFFFFF0ull - numSmallPix;
    }
    const size_t pixEntries = regions ? regionEntries : numSmallPix + arenaCap;
    const size_t tbl = (size_t)len * sizeof(unsigned);
    SSG_TRY(ssg_reserve(ctx, ctx->aux0, pixEntries * sizeof(unsigned)));                 // pixel store
    SSG_TRY(ssg_reserve(ctx, ctx->aux1, 2 * tbl));                                       // slices
    SSG_TRY(ssg_reserve(ctx, ctx->nextChunk, tbl));
    SSG_TRY(ssg_reserve(ctx, ctx->tailChunk, tbl));
    SSG_TRY(ssg_reserve(ctx, ctx->mergeTo, tbl));
    SSG_TRY(ssg_reserve(ctx, ctx->pendNext, tbl));
    SSG_TRY(ssg_reserve(ctx, ctx->candList, numSmall * sizeof(unsigned)));              // buckets
    unsigned *pix = bufp<unsigned>(ctx->aux0);
    unsigned *sliceOff = bufp<unsigned>(ctx->aux1), *sliceLen = sliceOff + len;
    unsigned *fill = bufp<unsigned>(ctx->pendNext);   // free until the passes start
    unsigned *bucketList = bufp<unsigned>(ctx->candList);

    SSG_PROF_BEGIN(ctx, "k_bucket_fill");
    k_bucket_fill<<<gridFor(len, 256), 256, 2 * (size_t)minSegSize * sizeof(unsigned), ctx->stream>>>(
        segSize, len, (unsigned)minSegSize, bucketStart, bucketFill, bucketList);
    SSG_LAUNCHED(ctx);
    SSG_PROF_BEGIN(ctx, "k_list_init");
    k_list_init<<<gridFor(len, 256), 256, 0, ctx->stream>>>(off, smallRank, segSize, len, (unsigned)minSegSize,
        regions ? (unsigned)(minSegSize - 1) : 0u, sliceOff, sliceLen, bufp<unsigned>(ctx->nextChunk),
        bufp<unsigned>(ctx->tailChunk), bufp<unsigned>(ctx->mergeTo), fill);
    SSG_LAUNCHED(ctx);
    // the one pass over the pixels: pending relabel + integer band sums + pixel lists
    {
        constexpr bool isSigned = std::is_signed<T>::value;
        constexpr bool packed = sizeof(T) < 4 && !isSigned;
        const int NP = packed ? (nB + 1) / 2 : nB;
        const size_t nSum = (size_t)len * NP;
        SSG_TRY(ssg_reserve(ctx, ctx->isum, nSum * sizeof(unsigned long long)));
        SSG_TRY(ssg_reserve(ctx, ctx->fsum, (size_t)len * nB * sizeof(float)));
        SSG_TRY(ssg_reserve(ctx, ctx->flags, (size_t)len));
        const int64_t nLut = pendingLut ? lutLen : len;
        SSG_TRY(ssg_reserve(ctx, ctx->sortVals0, (size_t)nLut * sizeof(unsigned)));
        unsigned *lutF = bufp<unsigned>(ctx->sortVals0);
        unsigned long long *isum = bufp<unsigned long long>(ctx->isum);
        float *fsum = bufp<float>(ctx->fsum);
        unsigned char *bigFlag = bufp<unsigned char>(ctx->flags);
        SSG_CUDA(ctx, cudaMemsetAsync(isum, 0, nSum * sizeof(unsigned long long), ctx->stream));
        SSG_CUDA(ctx, cudaMemsetAsync(counters + C_NUM_BIGSUM, 0, sizeof(unsigned long long), ctx->stream));
        SSG_PROF_BEGIN(ctx, "k_flag_lut");
        k_flag_lut<<<gridFor(nLut, 256), 256, 0, ctx->stream>>>(pendingLut, nLut, sliceLen, len, lutF);
        SSG_LAUNCHED(ctx);
        // wide loads need every band plane and the label raster 16 / 8 / 4-byte aligned
        const int vec = (N % 4 == 0) && ((uintptr_t)seg % 16 == 0) && ((uintptr_t)img % (sizeof(T) == 4 ? 16 : 8) == 0);
        int64_t blocks = ((N + 3) / 4 + 255) / 256;
        if (blocks > (int64_t)ctx->numSMs * 16) blocks = (int64_t)ctx->numSMs * 16;
        SSG_PROF_BEGIN(ctx, "k_pixel_pass");
        k_pixel_pass<T, packed><<<(unsigned)blocks, 256, 0, ctx->stream>>>(img, nB, N, seg, lutF, pendingLut != nullptr, vec,
                                                                         isum, sliceOff, fill, pix);
        SSG_LAUNCHED(ctx);
        const unsigned maxAbs = sizeof(T) == 1 ? 255u : sizeof(T) == 2 ? (packed ? 65535u : 32768u)
                                                                       : (isSigned ? 2147483648u : 4294967295u);
        SSG_PROF_BEGIN(ctx, "k_finalize_sums");
        k_finalize_sums2<packed, isSigned><<<gridFor(len, 256), 256, 0, ctx->stream>>>(isum, segSize, nB, len, maxAbs, fsum, bigFlag, counters);
        SSG_LAUNCHED(ctx);
    }
    SSG_PROF_BEGIN(ctx, "k_list_sort");
    k_list_sort<<<gridFor(len, 128), 128, 0, ctx->stream>>>(sliceOff, sliceLen, len, pix);
    SSG_LAUNCHED(ctx);

    SSG_TRY(ssg_fetch_counters(ctx));
    if (ctx->hostCounters[C_NUM_BIGSUM] > 0) {
        // float32 sums that are not exact integers: re-accumulated in raster order (shepseg.py:805-811)
        const unsigned *pixSorted = nullptr, *keysSorted = nullptr, *runStart = nullptr;
        int64_t M = 0;
        unsigned numRuns = 0;
        SSG_TRY(ssgk_group_pixels(ctx, seg, N, bufp<unsigned char>(ctx->flags), &pixSorted, &keysSorted, &runStart, &M, &numRuns));
        if (M > 0) {
            SSG_PROF_BEGIN(ctx, "k_ordered_sums");
            k_ordered_sums<T><<<gridFor((int64_t)numRuns * nB * 32, 128), 128, 0, ctx->stream>>>(
                img, nB, N, pixSorted, keysSorted, runStart, numRuns, M, bufp<float>(ctx->fsum));
            SSG_LAUNCHED(ctx);
        }
    }

    // the passes (merge.cu: 32-byte segment records, per-size candidate lists, grid kernels for
    // the first sizes + one cluster for the tail)
    const size_t m1g = (size_t)minSegSize + 1;
    ctx->grownStartStage.assign(m1g, 0ull);
    unsigned long long total = 0;
    for (size_t z = 0; z < m1g; z++) {
        ctx->grownStartStage[z] = total;
        // a merge at size t makes at least 2t+1 >= 3 pixels; the segments that ever have exactly
        // z pixels are disjoint sets of listed pixels
        if (z >= 3) total += numSmallPix / z;
    }
    SSG_TRY(ssg_reserve(ctx, ctx->lut, ssgk_merge_rec_bytes(nB, len)));
    SSG_TRY(ssg_reserve(ctx, ctx->targetList, (size_t)(total + 1) * sizeof(unsigned)));
    SSG_TRY(ssg_reserve(ctx, ctx->sortKeys0, m1g * sizeof(unsigned long long) + m1g * sizeof(unsigned) +
                                             (size_t)(len + 1) * sizeof(unsigned long long) + ssgk_merge_ctr_bytes() + 64));
    unsigned long long *grownStart = bufp<unsigned long long>(ctx->sortKeys0);
    unsigned long long *pendHead64 = grownStart + m1g;
    unsigned long long *arenaUsed = pendHead64 + len;
    unsigned long long *mctr = arenaUsed + 1;
    unsigned *grownCount = reinterpret_cast<unsigned *>(
        reinterpret_cast<char *>(mctr) + ssgk_merge_ctr_bytes());
    SSG_CUDA(ctx, cudaMemcpyAsync(grownStart, ctx->grownStartStage.data(), m1g * sizeof(unsigned long long),
                                  cudaMemcpyHostToDevice, ctx->stream));
    SSG_CUDA(ctx, cudaMemsetAsync(pendHead64, 0, (size_t)(len + 1) * sizeof(unsigned long long), ctx->stream));
    SSG_CUDA(ctx, cudaMemsetAsync(grownCount, 0, m1g * sizeof(unsigned), ctx->stream));
    MergeState ms;
    ms.seg = seg; ms.segSize = segSize; ms.rec = bufp<unsigned>(ctx->lut); ms.pix = pix;
    ms.mergeTo = bufp<unsigned>(ctx->mergeTo); ms.pendHead = pendHead64; ms.pendNext = bufp<unsigned>(ctx->pendNext);
    ms.bucketStart = bucketStart; ms.bucketList = bucketList;
    ms.grownList = bufp<unsigned>(ctx->targetList); ms.grownStart = grownStart; ms.grownCount = grownCount;
    ms.ctr = mctr;
    ms.bar = nullptr;       // (set by the merge stage, which knows the layout of its counters)
    ms.stage = 0; ms.exitSlots = 0;
    ms.nB = nB; ms.nRows = (unsigned)nRows; ms.nCols = (unsigned)nCols; ms.four = four;
    ms.minSegSize = minSegSize; ms.thr = thr;
    ms.sliceLen = sliceLen; ms.nextChunk = bufp<unsigned>(ctx->nextChunk); ms.tailChunk = bufp<unsigned>(ctx->tailChunk);
    ms.arenaUsed = arenaUsed; ms.arenaBase = (unsigned)numSmallPix; ms.arenaCap = (unsigned)arenaCap;
    ms.means = nullptr; ms.nBP = 0;      // (set by the merge stage for 17 to 64 bands)
    MergePlan plan;
    plan.fsum = bufp<float>(ctx->fsum); plan.sliceOff = sliceOff; plan.len = len; plan.packed = !regions;
    return ssgk_merge(ctx, ms, plan, numPasses, numElim);
}

int ssgk_eliminate_small(ssg_ctx *ctx, const void *imgDev, int dtype, int nBands, int64_t nRows,
                         int64_t nCols, uint32_t *segDev, uint32_t *sizeDev, uint32_t maxSegId,
                         int minSegSize, double thr, int four, int64_t *numElim, uint32_t *numPasses,
                         const uint32_t *pendingLut, int64_t lutLen)
{
    switch (dtype) {
    case SSG_U8: return eliminate_small_t<uint8_t>(ctx, (const uint8_t *)imgDev, nBands, nRows, nCols, segDev, sizeDev, maxSegId, minSegSize, thr, four, numElim, numPasses, pendingLut, lutLen);
    case SSG_U16: return eliminate_small_t<uint16_t>(ctx, (const uint16_t *)imgDev, nBands, nRows, nCols, segDev, sizeDev, maxSegId, minSegSize, thr, four, numElim, numPasses, pendingLut, lutLen);
    case SSG_I16: return eliminate_small_t<int16_t>(ctx, (const int16_t *)imgDev, nBands, nRows, nCols, segDev, sizeDev, maxSegId, minSegSize, thr, four, numElim, numPasses, pendingLut, lutLen);
    case SSG_U32: return eliminate_small_t<uint32_t>(ctx, (const uint32_t *)imgDev, nBands, nRows, nCols, segDev, sizeDev, maxSegId, minSegSize, thr, four, numElim, numPasses, pendingLut, lutLen);
    case SSG_I32: return eliminate_small_t<int32_t>(ctx, (const int32_t *)imgDev, nBands, nRows, nCols, segDev, sizeDev, maxSegId, minSegSize, thr, four, numElim, numPasses, pendingLut, lutLen);
    default: SSG_FAIL(ctx, SSG_ERR_ARG, "unsupported dtype code %d", dtype);
    }
}
