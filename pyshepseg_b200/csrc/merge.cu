// merge.cu -- K8: the targetSize loop of eliminateSmallSegments (shepseg.py:970-997) with
// findMergeSegment (1003-1063) and doMerge (1066-1123).
//
// What the reference fixes and what is kept here exactly:
//   * sizes are visited in ascending order; within a size up to ten passes, each pass first
//     DECIDES for every segment of exactly that size with the state frozen (shepseg.py:983-986),
//     then MERGES in ascending id of the merged segment (989-994);
//   * a decision scans the segment's pixels in list order and the 3x3 window rows outer, columns
//     inner; float32 means, float32 squared differences summed in band order; the first strict
//     minimum wins (1046-1057); it is dropped if it exceeds maxSpectralDiff**2 (1060);
//   * a merge appends the source's pixel list to the target's, adds the float32 sums and the
//     sizes (1099-1123): with several sources for one target in a pass the order is ascending
//     source id.
//
// How it runs here.  A pass is two phases separated by a barrier, nothing else:
//   find   a group of G lanes per candidate (G = the candidate's size rounded up to a power of two,
//          at most 32): ONE 32-byte record {band MEANS, size, list offset} per segment means one
//          gather tells everything about the candidate and one gather per neighbouring segment
//          tells whether it is larger and how far away it is spectrally.  The winner is recorded as
//          mergeTo[s] and s is pushed on the target's pending stack (one atomic exchange; the
//          stack head carries the pass number, so it never has to be cleared).
//   merge  again a group per candidate that found a target: it relabels its own pixels, and the
//          group of the SMALLEST source id of a target also does the target's bookkeeping: sums
//          and sizes in ascending source id, the sources' pixel lists appended to the target's
//          list in that order.  A target that is still small afterwards is entered in the
//          candidate list of its new size (a merge at size t makes segments of at least 2t+1
//          pixels, so that list is complete before its size comes up; its capacity is bounded by
//          listedPixels / size because the segments that ever have exactly `size` pixels are
//          pairwise disjoint sets of listed pixels).
// The candidates of a size are its bucket of initially small segments followed by that list; a
// later pass of the same size rescans them and skips what has merged (size 0) or grown.
//
// Where the pixel lists live is the one thing the two instantiations of the kernels differ in:
//   regions  (PACKED = false, the default) every small segment has a region of minSegSize-1
//            entries of its own; a merge appends the sources' lists in place at off + size.
//   packed   (PACKED = true, when the regions would take too much memory) the lists start as
//            consecutive slices of one array; a list is a chain of slices (sliceLen, nextChunk).
//            A merge copies the target's chain and then the sources' into a fresh slice of an
//            arena behind the initial lists, and when the arena has run out it links the
//            sources' chains to the target's instead.  A list position is counted across slices.
//
// Two kernels share the code: a cooperative grid for the sizes with many candidates (the first
// few: hundreds of thousands of gathers per phase) and ONE thread-block cluster of 16 CTAs for the
// tail, where a phase is a handful of dependent gathers and the barrier itself is what a pass pays
// for: a hardware cluster barrier costs 0.35 us against 1.2 us for a grid barrier, and the skew
// between 16 CTAs is far below that between 148 (measured: tools/bench_barrier.cu, profiles/).
#include "common.cuh"
#include "merge.cuh"

#include <cooperative_groups.h>
namespace cg = cooperative_groups;

#define MERGE_THREADS 512
#define MERGE_SORT_MAX 64
#define MERGE_CLUSTER 16

enum MergeCtr {
    MF_MERGED = 0,    // candidates that found a target (per parity set)
    MF_LEFT,          // candidates that did not
    MF_COUNT = 2,
    MC_ELIM = 4,      // merges done
    MC_PASSES,
    MC_RESUME_T,      // the size the tail kernel starts at
    MC_STAMP,         // pass number at hand-over
    MC_COUNT = 8      // one block of MC_COUNT per launch of the chain (parity sets; the MC_* of the first count)
};

__device__ __forceinline__ float rec_mean(float sum, unsigned n)
{
    // float32 mean as the reference gets it (float64 division rounded to float32, shepseg.py:1042,
    // 1053); for n < 2^24 a float32 division gives the same bits
    if (n < (1u << 24)) return __fdiv_rn(sum, (float)n);
    return __double2float_rn(__ddiv_rn((double)sum, (double)n));
}

__device__ __forceinline__ unsigned width_for(unsigned t)
{
    unsigned g = 1;
    while (g < t && g < 32u) g <<= 1;
    return g;
}

template <int NBMAX>
struct Rec {
    float f[NBMAX];
    unsigned size, off;
};
template <>
struct Rec<64> {         // 17 to 64 bands: the means are read from MergeState::means where needed
    unsigned size, off;
};

// one segment record: everything in it sits in one (NBMAX <= 4) or two / four 32-byte sectors
template <int NBMAX>
__device__ __forceinline__ Rec<NBMAX> load_rec(const unsigned *rec, unsigned s)
{
    constexpr int W = MergeRecWords<NBMAX>::value;
    if constexpr (NBMAX > 16) {
        const uint2 t = __ldcg(reinterpret_cast<const uint2 *>(rec + (size_t)s * W));
        Rec<NBMAX> r;
        r.size = t.x; r.off = t.y;
        return r;
    } else {
        const uint4 *p = reinterpret_cast<const uint4 *>(rec + (size_t)s * W);
        Rec<NBMAX> r;
#pragma unroll
        for (int i = 0; i < NBMAX / 4; i++) {
            const uint4 v = __ldcg(p + i);
            r.f[4 * i] = __uint_as_float(v.x); r.f[4 * i + 1] = __uint_as_float(v.y);
            r.f[4 * i + 2] = __uint_as_float(v.z); r.f[4 * i + 3] = __uint_as_float(v.w);
        }
        const uint2 t = __ldcg(reinterpret_cast<const uint2 *>(rec + (size_t)s * W + NBMAX));
        r.size = t.x; r.off = t.y;
        return r;
    }
}

// 17 to 64 bands: the float32 distance of the means of segments a and b, streamed from the means
// array, in band order (the zero padding of both rows adds exact zeros)
__device__ __forceinline__ float means_dist(const MergeState &st, unsigned a, unsigned b)
{
    const float4 *pa = reinterpret_cast<const float4 *>(st.means + (size_t)a * st.nBP);
    const float4 *pb = reinterpret_cast<const float4 *>(st.means + (size_t)b * st.nBP);
    float d = 0.0f;
    for (int q = 0; q < st.nBP / 4; q++) {
        const float4 x = __ldcg(pa + q), y = __ldcg(pb + q);
        float df = __fsub_rn(x.x, y.x);
        d = __fadd_rn(d, __fmul_rn(df, df));
        df = __fsub_rn(x.y, y.y);
        d = __fadd_rn(d, __fmul_rn(df, df));
        df = __fsub_rn(x.z, y.z);
        d = __fadd_rn(d, __fmul_rn(df, df));
        df = __fsub_rn(x.w, y.w);
        d = __fadd_rn(d, __fmul_rn(df, df));
    }
    return d;
}

// packed lists: f(offset, length, list position) for every slice of the chain that starts with the
// slice of segment ch at pix[o ..)
template <int NBMAX, typename F>
__device__ __forceinline__ void for_slices(const MergeState &st, unsigned ch, unsigned o, F f)
{
    constexpr int W = MergeRecWords<NBMAX>::value;
    for (unsigned pos = 0;;) {
        const unsigned n = __ldcg(st.sliceLen + ch);
        f(o, n, pos);
        pos += n;
        ch = __ldcg(st.nextChunk + ch);
        if (ch == SSG_NIL) return;
        o = __ldcg(st.rec + (size_t)ch * W + MergeRecSizeAt<NBMAX>::value + 1);
    }
}

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Barrier over the whole launch: the grid (cooperative launch: every block is resident) or the one
// cluster.  On the way out every block picks up the find counters of parity `set`.
// tallySh: what the warps of this block counted in the phase that ends here (candidates merged /
// left, merges done): one global atomic per block and counter instead of one per warp -- a
// thousand atomics on one address take microseconds, and the barrier waits for them
template <bool CLUSTER>
__device__ __forceinline__ void merge_barrier(const MergeState &st, unsigned long long *ctr, unsigned &phase, int set,
                                              unsigned long long *curSh, unsigned *tallySh)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        if (tallySh[0]) atomicAdd(&ctr[set * MF_COUNT + MF_MERGED], (unsigned long long)tallySh[0]);
        if (tallySh[1]) atomicAdd(&ctr[set * MF_COUNT + MF_LEFT], (unsigned long long)tallySh[1]);
        if (tallySh[2]) atomicAdd(&st.ctr[MC_ELIM], (unsigned long long)tallySh[2]);
        tallySh[0] = tallySh[1] = tallySh[2] = 0;
    }
    if (CLUSTER) {
        if (threadIdx.x == 0) __threadfence();
        cg::this_cluster().sync();
    } else if (threadIdx.x == 0) {
        const unsigned target = (phase + 1) * gridDim.x;
        __threadfence();
        atomicAdd(&st.bar[st.stage].arrive, 1u);
        while (ld_acquire_gpu(&st.bar[st.stage].arrive) < target) { }
    }
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < MF_COUNT; i++) curSh[i] = __ldcg(&ctr[set * MF_COUNT + i]);
    }
    phase++;
    __syncthreads();
}

// ---- find ---------------------------------------------------------------------------------------
template <int NBMAX, bool FOUR, bool PACKED>
__device__ __forceinline__ void merge_find(const MergeState &st, unsigned *tallySh, unsigned t,
                                           const unsigned *listA, unsigned nA, const unsigned *listB, unsigned nCand,
                                           unsigned stamp, unsigned gtid, unsigned gsize)
{
    const unsigned G = width_for(t);
    const unsigned lane = lane_id();
    const unsigned sub = lane % G;
    const unsigned perWarp = 32u / G;
    const unsigned warpId = gtid >> 5, nWarps = gsize >> 5;
    const int nB = st.nB;
    const unsigned nCols = st.nCols, nRows = st.nRows;
    unsigned tallyMerged = 0, tallyLeft = 0;

    for (unsigned c0 = warpId * perWarp; c0 < nCand; c0 += nWarps * perWarp) {
        const unsigned c = c0 + lane / G;
        bool active = c < nCand;
        unsigned s = 0;
        if (active) s = c < nA ? __ldg(listA + c) : __ldcg(listB + (c - nA));
        Rec<NBMAX> me;
        me.size = 0; me.off = 0;
        if (active) me = load_rec<NBMAX>(st.rec, s);
        active = active && me.size == t;          // merged (size 0) or grown since it was listed
        unsigned long long bestKey = ~0ull;
        unsigned bestU = 0;
        if (active) {
            float ms[NBMAX <= 16 ? NBMAX : 1];       // (the records hold the float32 MEANS: see k_rec_init)
            if constexpr (NBMAX <= 16) {
#pragma unroll
                for (int b = 0; b < NBMAX; b++) ms[b] = me.f[b];
            }
            // pixel p at list position pos
            auto visit = [&](unsigned p, unsigned pos) {
                // row = p / nCols by multiplication (colMagic = floor(2^40 / nCols) + 1 overshoots by at
                // most one for p < 2^32)
                unsigned y = (unsigned)(((unsigned long long)p * st.colMagic) >> 40);
                if (y * nCols > p) y--;
                const unsigned x = p - y * nCols;
                constexpr int NQ = FOUR ? 4 : 8;
                unsigned nu[NQ];
                bool ok[NQ];
#pragma unroll
                for (int q = 0; q < NQ; q++) {
                    // window cells in the reference's scan order, rows outer, columns inner
                    // (shepseg.py:1046-1047); four-connected: N, W, E, S
                    const int cell = FOUR ? (q == 0 ? 1 : (q == 1 ? 3 : (q == 2 ? 5 : 7))) : (q < 4 ? q : q + 1);
                    const int dy = cell / 3 - 1, dx = cell % 3 - 1;
                    const unsigned yy = y + (unsigned)dy, xx = x + (unsigned)dx;   // wraps below zero
                    ok[q] = yy < nRows && xx < nCols;
                    nu[q] = ok[q] ? st.seg[(size_t)yy * nCols + xx] : 0u;
                }
#pragma unroll
                for (int q = 0; q < NQ; q++) {
                    ok[q] = ok[q] && nu[q] != s && nu[q] != 0;
#pragma unroll
                    for (int r = 0; r < q; r++)          // a repeat can never win: same distance, later
                        if (nu[r] == nu[q]) ok[q] = false;
                }
                constexpr int BATCH = (NBMAX <= 4 || NBMAX > 16) ? 4 : 2;
#pragma unroll
                for (int q0 = 0; q0 < NQ; q0 += BATCH) {
                    Rec<NBMAX> nr[BATCH];
#pragma unroll
                    for (int e = 0; e < BATCH; e++) {
                        nr[e].size = 0;
                        if (ok[q0 + e]) nr[e] = load_rec<NBMAX>(st.rec, nu[q0 + e]);
                    }
#pragma unroll
                    for (int e = 0; e < BATCH; e++) {
                        if (!ok[q0 + e] || !(nr[e].size > t)) continue;     // strictly larger, shepseg.py:1052
                        float d = 0.0f;
                        if constexpr (NBMAX > 16) {
                            d = means_dist(st, s, nu[q0 + e]);
                        } else {
#pragma unroll
                            for (int b = 0; b < NBMAX; b++) {
                                if (b < nB) {
                                    const float df = __fsub_rn(ms[b], nr[e].f[b]);
                                    d = __fadd_rn(d, __fmul_rn(df, df));
                                }
                            }
                        }
                        const int q = q0 + e;
                        const unsigned cell = FOUR ? (q == 0 ? 1u : (q == 1 ? 3u : (q == 2 ? 5u : 7u)))
                                                   : (unsigned)(q < 4 ? q : q + 1);
                        const unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) |
                                                       (unsigned long long)(pos * 16u + cell);
                        if (key < bestKey) { bestKey = key; bestU = nu[q]; }
                    }
                }
            };
            if constexpr (PACKED) {
                for_slices<NBMAX>(st, s, me.off, [&](unsigned o, unsigned n, unsigned pos0) {
                    for (unsigned i = sub; i < n; i += G) visit(__ldcg(st.pix + o + i), pos0 + i);
                });
            } else {
                for (unsigned i = sub; i < t; i += G) visit(__ldcg(st.pix + me.off + i), i);
            }
        }
        // the minimum over the group (keys embed the list position: distinct across lanes)
        for (unsigned o = G >> 1; o > 0; o >>= 1) {
            const unsigned long long k2 = __shfl_xor_sync(0xffffffffu, bestKey, o);
            const unsigned u2 = __shfl_xor_sync(0xffffffffu, bestU, o);
            if (k2 < bestKey) { bestKey = k2; bestU = u2; }
        }
        if (active && sub == 0) {
            bool merged = false;
            if (bestKey != ~0ull) {
                const float d = __uint_as_float((unsigned)(bestKey >> 32));
                merged = !((double)d > st.thr);       // shepseg.py:1060
            }
            if (merged) {
                st.mergeTo[s] = bestU;
                const unsigned long long old =
                    atomicExch(&st.pendHead[bestU], ((unsigned long long)stamp << 32) | (unsigned long long)s);
                st.pendNext[s] = (unsigned)(old >> 32) == stamp ? (unsigned)old : 0u;
                tallyMerged++;
            } else {
                tallyLeft++;
            }
        }
    }
    tallyMerged = __reduce_add_sync(0xffffffffu, tallyMerged);
    tallyLeft = __reduce_add_sync(0xffffffffu, tallyLeft);
    if (lane == 0) {
        if (tallyMerged) atomicAdd(&tallySh[0], tallyMerged);
        if (tallyLeft) atomicAdd(&tallySh[1], tallyLeft);
    }
}

// ---- merge --------------------------------------------------------------------------------------
template <int NBMAX, bool PACKED>
__device__ __forceinline__ void merge_apply(const MergeState &st, unsigned *tallySh, unsigned t,
                                            const unsigned *listA, unsigned nA, const unsigned *listB, unsigned nCand,
                                            unsigned stamp, unsigned gtid, unsigned gsize)
{
    constexpr int W = MergeRecWords<NBMAX>::value;
    constexpr int SZ = MergeRecSizeAt<NBMAX>::value;
    const unsigned G = width_for(t);
    const unsigned lane = lane_id();
    const unsigned sub = lane % G;
    const unsigned perWarp = 32u / G;
    const unsigned warpId = gtid >> 5, nWarps = gsize >> 5;
    const int nB = st.nB;
    unsigned elim = 0;

    for (unsigned c0 = warpId * perWarp; c0 < nCand; c0 += nWarps * perWarp) {
        // The lanes of a group work on one candidate but are not in lock step on their own (a lane
        // that is done with a sweep goes on to the next one), and what a group writes (its
        // candidate's size word, its target's record) is what its lanes read to decide what to
        // do: all reads of a sweep come first, then a warp barrier, then the writes.
        __syncwarp();
        const unsigned c = c0 + lane / G;
        bool active = c < nCand;
        unsigned s = 0, u = 0;
        unsigned sSize = 0, sOff = 0;
        if (active) {
            s = c < nA ? __ldg(listA + c) : __ldcg(listB + (c - nA));
            u = __ldcg(st.mergeTo + s);
            const uint2 so = __ldcg(reinterpret_cast<const uint2 *>(st.rec + (size_t)s * W + SZ));
            sSize = so.x; sOff = so.y;
        }
        // merged in THIS pass: it has a target and still its size (an earlier pass zeroed it)
        active = active && u != 0 && sSize == t;
        unsigned long long head = 0;
        Rec<NBMAX> tg;
        tg.size = 0; tg.off = 0;
        unsigned ids[MERGE_SORT_MAX];
        unsigned k = 0, below = 0;
        if (active) {
            head = __ldcg(st.pendHead + u);
            tg = load_rec<NBMAX>(st.rec, u);        // only the target's own group uses it
            // the other sources of my target (pushed this pass: the head carries the stamp)
            for (unsigned q = (unsigned)(head >> 32) == stamp ? (unsigned)head : 0u; q != 0; q = __ldcg(st.pendNext + q)) {
                if (k < MERGE_SORT_MAX) {
                    unsigned j = k;
                    while (j > 0 && ids[j - 1] > q) { ids[j] = ids[j - 1]; j--; }
                    ids[j] = q;
                }
                below += q < s;
                k++;
            }
        }
        __syncwarp();
        if (active) {
            // my own pixels now belong to the target (first half of doMerge, shepseg.py:1107-1110)
            if constexpr (PACKED) {
                // The target's group may link chains while this runs (see below), and the one
                // thing it changes under my feet is the last link of my chain: following that link
                // only relabels the next source of the SAME target, which is harmless.
                for_slices<NBMAX>(st, s, sOff, [&](unsigned o, unsigned n, unsigned) {
                    for (unsigned i = sub; i < n; i += G) st.seg[__ldcg(st.pix + o + i)] = u;
                });
            } else {
                for (unsigned i = sub; i < t; i += G) st.seg[__ldcg(st.pix + sOff + i)] = u;
            }
            if (sub == 0) {
                st.rec[(size_t)s * W + SZ] = 0u;     // size 0: dead
                st.segSize[s] = 0u;
            }
        }
        if (active && below == 0) {      // the group of the target's smallest source goes on
            const unsigned newSize = tg.size + k * t;              // every source has exactly t pixels
            const bool keepList = newSize < (unsigned)st.minSegSize;   // then the target was small all along
            // float32 band sums of the target (spectSum, shepseg.py:1117-1120); from 17 bands on they
            // are updated in memory, each lane of the group taking every G-th band
            float fu[NBMAX <= 16 ? NBMAX : 1];
            if constexpr (NBMAX <= 16) {
#pragma unroll
                for (int b = 0; b < NBMAX; b++) fu[b] = b < nB ? __ldcg(st.fsum + (size_t)u * nB + b) : 0.0f;
            }
            // Packed lists: the merged list is copied into a fresh slice of the arena while the
            // arena lasts; after that the sources' chains are linked to the target's.
            const unsigned gmask = G == 32 ? 0xffffffffu : ((1u << G) - 1u) << (lane & ~(G - 1u));
            unsigned arenaOff = SSG_NIL, w = 0;
            auto copy = [&](unsigned o, unsigned n, unsigned) {
                for (unsigned i = sub; i < n; i += G) st.pix[arenaOff + w + i] = __ldcg(st.pix + o + i);
                w += n;
            };
            if (PACKED && keepList) {
                unsigned long long a = 0;
                if (sub == 0) a = atomicAdd(st.arenaUsed, (unsigned long long)newSize);
                a = __shfl_sync(gmask, a, lane & ~(G - 1u));
                if (a + newSize <= st.arenaCap) {
                    arenaOff = st.arenaBase + (unsigned)a;
                    for_slices<NBMAX>(st, u, tg.off, copy);
                }
            }
            unsigned last = 0;   // ids are >= 1
            for (unsigned m = 0; m < k; m++) {
                unsigned sm;
                if (k <= MERGE_SORT_MAX) sm = ids[m];
                else {               // long stacks: the smallest pending source above `last`
                    sm = SSG_NIL;
                    for (unsigned q = (unsigned)head; q != 0; q = __ldcg(st.pendNext + q))
                        if (q > last && q < sm) sm = q;
                }
                if constexpr (NBMAX > 16) {
                    for (int b = sub; b < nB; b += G)
                        st.fsum[(size_t)u * nB + b] = __fadd_rn(__ldcg(st.fsum + (size_t)u * nB + b),
                                                                __ldcg(st.fsum + (size_t)sm * nB + b));
                } else {
#pragma unroll
                    for (int b = 0; b < NBMAX; b++)
                        if (b < nB) fu[b] = __fadd_rn(fu[b], __ldcg(st.fsum + (size_t)sm * nB + b));
                }
                if (keepList) {
                    const unsigned srcOff = __ldcg(st.rec + (size_t)sm * W + SZ + 1);
                    if constexpr (PACKED) {
                        if (arenaOff != SSG_NIL) {
                            for_slices<NBMAX>(st, sm, srcOff, copy);
                        } else if (sub == 0) {
                            st.nextChunk[__ldcg(st.tailChunk + u)] = sm;
                            st.tailChunk[u] = __ldcg(st.tailChunk + sm);
                        }
                    } else {
                        const unsigned dst = tg.off + tg.size + m * t;
                        for (unsigned i = sub; i < t; i += G) st.pix[dst + i] = __ldcg(st.pix + srcOff + i);
                    }
                }
                last = sm;
            }
            if (PACKED && keepList) __syncwarp(gmask);     // the group has read the target's chain
            if constexpr (NBMAX > 16) {
                for (int b = sub; b < nB; b += G)
                    st.means[(size_t)u * st.nBP + b] = rec_mean(__ldcg(st.fsum + (size_t)u * nB + b), newSize);
            }
            if (sub == 0) {
                unsigned *r = st.rec + (size_t)u * W;
                if constexpr (NBMAX <= 16) {
#pragma unroll
                    for (int b = 0; b < NBMAX; b++) {
                        if (b < nB) {
                            st.fsum[(size_t)u * nB + b] = fu[b];
                            r[b] = __float_as_uint(rec_mean(fu[b], newSize));
                        }
                    }
                }
                r[SZ] = newSize;
                st.segSize[u] = newSize;
                if (PACKED && arenaOff != SSG_NIL) {      // one slice again
                    r[SZ + 1] = arenaOff;
                    st.sliceLen[u] = newSize;
                    st.nextChunk[u] = SSG_NIL;
                    st.tailChunk[u] = u;
                }
                elim += k;
                if (keepList) {      // a candidate itself when its new size comes up
                    const unsigned slot = atomicAdd(&st.grownCount[newSize], 1u);
                    st.grownList[st.grownStart[newSize] + slot] = u;
                }
            }
        }
    }
    elim = __reduce_add_sync(0xffffffffu, elim);
    if (lane == 0 && elim) atomicAdd(&tallySh[2], elim);
}

// ---- the loop over sizes --------------------------------------------------------------------------
template <int NBMAX, bool FOUR, bool CLUSTER, int MINB, bool PACKED>
__global__ void __launch_bounds__(MERGE_THREADS, MINB)
k_merge(MergeState st)
{
    __shared__ unsigned long long cur[MF_COUNT];
    __shared__ unsigned tally[4];
    if (threadIdx.x < 4) tally[threadIdx.x] = 0;
    __syncthreads();
    const unsigned gtid = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned gsize = gridDim.x * blockDim.x;
    unsigned long long *ctrG = st.ctr;                                // MC_* live in the first block
    unsigned long long *ctr = st.ctr + st.stage * MC_COUNT;           // parity sets of this launch
    unsigned phase = 0;
    unsigned long long base[2][MF_COUNT] = {{0, 0}, {0, 0}};
    unsigned long long passes = 0;
    unsigned stamp = 0;
    unsigned tBegin = 1;
    if (st.stage > 0) {
        tBegin = (unsigned)__ldcg(&ctrG[MC_RESUME_T]);
        stamp = (unsigned)__ldcg(&ctrG[MC_STAMP]);
        if (tBegin == 0 || tBegin >= (unsigned)st.minSegSize) return;    // an earlier launch did it all
    }
    constexpr unsigned switchMinT = 2;      // size 1 always runs in the first launch
    for (unsigned t = tBegin; t < (unsigned)st.minSegSize; t++) {
        const unsigned a0 = st.bucketStart[t];
        const unsigned nA = st.bucketStart[t + 1] - a0;
        const unsigned nCand = nA + __ldcg(&st.grownCount[t]);
        if (st.exitSlots != 0 && t >= switchMinT && (unsigned long long)nCand * width_for(t) <= st.exitSlots) {
            // few enough candidates for the next launch of the chain (fewer, leaner blocks; in the
            // end one cluster).  Every block takes this branch: the counts are the same for all.
            if (gtid == 0) {
                ctrG[MC_RESUME_T] = t;
                ctrG[MC_STAMP] = stamp;
                ctrG[MC_PASSES] = __ldcg(&ctrG[MC_PASSES]) + passes;
            }
            return;
        }
        if (nCand == 0) continue;
        const unsigned *listA = st.bucketList + a0;
        const unsigned *listB = st.grownList + st.grownStart[t];
        for (int pass = 0; pass < 10; pass++) {              // shepseg.py:979-980
            const int set = (int)(phase & 1u);
            stamp++;
            merge_find<NBMAX, FOUR, PACKED>(st, tally, t, listA, nA, listB, nCand, stamp, gtid, gsize);
            merge_barrier<CLUSTER>(st, ctr, phase, set, cur, tally);
            const unsigned long long merged = cur[MF_MERGED] - base[set][MF_MERGED];
            const unsigned long long left = cur[MF_LEFT] - base[set][MF_LEFT];
#pragma unroll
            for (int i = 0; i < MF_COUNT; i++) base[set][i] = cur[i];
            passes++;
            if (merged == 0) break;      // the count of this size did not change (shepseg.py:980,996)
            merge_apply<NBMAX, PACKED>(st, tally, t, listA, nA, listB, nCand, stamp, gtid, gsize);
            merge_barrier<CLUSTER>(st, ctr, phase, set, cur, tally);    // (the find counters did not move)
            if (left == 0) break;        // nobody left of this size: the next pass would merge nothing
        }
    }
    if (gtid == 0) {
        ctrG[MC_PASSES] = __ldcg(&ctrG[MC_PASSES]) + passes;
        ctrG[MC_RESUME_T] = 0;
    }
}

// ---- records -------------------------------------------------------------------------------------
template <int NBMAX>
__global__ void __launch_bounds__(256)
k_rec_init(const float *__restrict__ fsum, const unsigned *__restrict__ segSize, const unsigned *__restrict__ sliceOff,
           int nB, int64_t len, unsigned *rec)
{
    constexpr int W = MergeRecWords<NBMAX>::value;
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= len) return;
    unsigned r[W];
    const unsigned size = segSize[s];
#pragma unroll
    for (int b = 0; b < NBMAX; b++)
        r[b] = (b < nB && size != 0) ? __float_as_uint(rec_mean(fsum[(size_t)s * nB + b], size)) : 0u;
    r[NBMAX] = size;
    r[NBMAX + 1] = sliceOff[s];
#pragma unroll
    for (int b = NBMAX + 2; b < W; b++) r[b] = 0u;
    uint4 *o = reinterpret_cast<uint4 *>(rec + (size_t)s * W);      // whole sectors, not words
#pragma unroll
    for (int i = 0; i < W / 4; i++) o[i] = make_uint4(r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
}

// 17 to 64 bands: the records {size, list offset} and the means array, one thread per (segment,
// padded band)
__global__ void __launch_bounds__(256)
k_rec_init_many(const float *__restrict__ fsum, const unsigned *__restrict__ segSize, const unsigned *__restrict__ sliceOff,
                int nB, int nBP, int64_t len, unsigned *rec, float *means)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len * nBP) return;
    const int64_t s = i / nBP;
    const int b = (int)(i % nBP);
    const unsigned size = segSize[s];
    means[i] = (b < nB && size != 0) ? rec_mean(fsum[(size_t)s * nB + b], size) : 0.0f;
    if (b == 0) reinterpret_cast<uint2 *>(rec)[s] = make_uint2(size, sliceOff[s]);
}

// the means array of the 17-64-band class starts behind the records, 16-byte aligned
static size_t means_offset_words(int64_t len) { return ((size_t)len * MergeRecWords<64>::value + 3) & ~(size_t)3; }

#define MERGE_STAGES 3

template <int NBMAX, bool FOUR, bool PACKED>
static int run_merge_t(ssg_ctx *ctx, MergeState &st, const MergePlan &plan, uint32_t *numPasses, int64_t *numElim)
{
    const size_t ctrBytes = MERGE_STAGES * MC_COUNT * sizeof(unsigned long long) + MERGE_STAGES * sizeof(SmallBarrier);
    st.bar = reinterpret_cast<SmallBarrier *>(st.ctr + MERGE_STAGES * MC_COUNT);
    SSG_CUDA(ctx, cudaMemsetAsync(st.ctr, 0, ctrBytes, ctx->stream));
    if constexpr (NBMAX > 16) {
        st.nBP = (st.nB + 3) & ~3;
        st.means = reinterpret_cast<float *>(st.rec + means_offset_words(plan.len));
        SSG_PROF_BEGIN(ctx, "k_rec_init_many");
        k_rec_init_many<<<gridFor(plan.len * st.nBP, 256), 256, 0, ctx->stream>>>(plan.fsum, st.segSize, plan.sliceOff,
                                                                                   st.nB, st.nBP, plan.len, st.rec, st.means);
        SSG_LAUNCHED(ctx);
    } else {
        SSG_PROF_BEGIN(ctx, "k_rec_init");
        k_rec_init<NBMAX><<<gridFor(plan.len, 256), 256, 0, ctx->stream>>>(plan.fsum, st.segSize, plan.sliceOff, st.nB, plan.len, st.rec);
        SSG_LAUNCHED(ctx);
    }
    st.fsum = const_cast<float *>(plan.fsum);
    st.colMagic = ((1ull << 40) / st.nCols) + 1ull;

    // A chain of three launches, each picking up where the previous one stopped:
    //   wide    two blocks per SM (64 registers): the first sizes, whose phases are hundreds of
    //           thousands of gathers and want every warp the GPU can hold;
    //   lean    one block per SM with all the registers it wants (no spills): the long run of sizes
    //           whose phases are one dependent chain per candidate;
    //   cluster one cluster of 16 blocks: the end, when a hardware cluster barrier beats a grid barrier.
    // Where the cluster cannot be launched the lean grid runs to the end.
    bool tail = true;
    auto kTail = k_merge<NBMAX, FOUR, true, 1, PACKED>;
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    if (cudaFuncSetAttribute(kTail, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
        cudaGetLastError();
        tail = false;
    }
    if (tail) {
        cfg.gridDim = dim3(MERGE_CLUSTER);
        cfg.blockDim = dim3(MERGE_THREADS);
        cfg.stream = ctx->stream;
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = MERGE_CLUSTER; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int nClusters = 0;
        if (cudaOccupancyMaxActiveClusters(&nClusters, kTail, &cfg) != cudaSuccess || nClusters < 1) {
            cudaGetLastError();
            tail = false;
        }
    }
    const unsigned tailCands = 320;      // measured (profiles/): below this a 16-CTA cluster finishes a pass sooner than the grid

    void *kWide = (void *)k_merge<NBMAX, FOUR, false, 2, PACKED>;
    void *kLean = (void *)k_merge<NBMAX, FOUR, false, 1, PACKED>;
    int perSM = 0;
    SSG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, kWide, MERGE_THREADS, 0));
    if (perSM < 1) SSG_FAIL(ctx, SSG_ERR_CUDA, "merge kernel does not fit on an SM");
    if (perSM > 2) perSM = 2;
    dim3 block(MERGE_THREADS);
    {
        MergeState s0 = st;
        s0.stage = 0;
        // the wide launch hands over when one sweep of the lean grid covers the candidates
        s0.exitSlots = (unsigned long long)ctx->numSMs * MERGE_THREADS;
        void *args[] = {&s0};
        SSG_PROF_BEGIN(ctx, "k_merge_wide");
        SSG_CUDA(ctx, cudaLaunchCooperativeKernel(kWide, dim3((unsigned)(ctx->numSMs * perSM)), block, args, 0, ctx->stream));
        SSG_LAUNCHED(ctx);
    }
    {
        MergeState s1 = st;
        s1.stage = 1;
        s1.exitSlots = tail ? (unsigned long long)tailCands * 32ull : 0ull;
        void *args[] = {&s1};
        SSG_PROF_BEGIN(ctx, "k_merge_lean");
        SSG_CUDA(ctx, cudaLaunchCooperativeKernel(kLean, dim3((unsigned)ctx->numSMs), block, args, 0, ctx->stream));
        SSG_LAUNCHED(ctx);
    }
    if (tail) {
        MergeState s2 = st;
        s2.stage = 2;
        s2.exitSlots = 0;
        SSG_PROF_BEGIN(ctx, "k_merge_tail");
        SSG_CUDA(ctx, cudaLaunchKernelEx(&cfg, kTail, s2));
        SSG_LAUNCHED(ctx);
    }
    uint64_t *host = ctx->hostCounters;   // the pinned mirror doubles as the landing zone
    SSG_CUDA(ctx, cudaMemcpyAsync(host, st.ctr, MC_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *numPasses = (uint32_t)host[MC_PASSES];
    *numElim = (int64_t)host[MC_ELIM];
    return SSG_OK;
}

size_t ssgk_merge_rec_bytes(int nB, int64_t len)
{
    if (nB > 16) return (means_offset_words(len) + (size_t)len * ((nB + 3) & ~3)) * sizeof(unsigned);
    const int w = nB <= 4 ? MergeRecWords<4>::value : (nB <= 8 ? MergeRecWords<8>::value : MergeRecWords<16>::value);
    return (size_t)len * w * sizeof(unsigned);
}

size_t ssgk_merge_ctr_bytes(void) { return MERGE_STAGES * MC_COUNT * sizeof(unsigned long long) + MERGE_STAGES * sizeof(SmallBarrier) + 64; }

int ssgk_merge(ssg_ctx *ctx, MergeState &st, const MergePlan &plan, uint32_t *numPasses, int64_t *numElim)
{
    const int nB = st.nB;
#define RUN_P(NBMAX, FOUR) (plan.packed ? run_merge_t<NBMAX, FOUR, true>(ctx, st, plan, numPasses, numElim) \
                                        : run_merge_t<NBMAX, FOUR, false>(ctx, st, plan, numPasses, numElim))
#define RUN(NBMAX) (st.four ? RUN_P(NBMAX, true) : RUN_P(NBMAX, false))
    if (nB <= 4) return RUN(4);
    if (nB <= 8) return RUN(8);
    if (nB <= 16) return RUN(16);
    return RUN(64);
#undef RUN
#undef RUN_P
}
