// common.cuh -- context, scratch-memory and error plumbing shared by the kernels of
// libshepseg_b200.so.  Device code here is sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <math.h>
#include <string>
#include <vector>

#include "../../include/shepseg_b200.h"

#define SSG_NIL 0xFFFFFFFFu          // "no pixel / no root / no chunk"
#define SSG_MAX_CLUMP_SIZE 10000u    // shepseg.py:481

// geometry of the pruning grid of the assignment kernel (assign.cu)
struct GridGeom {
    int nB;
    int base[4], shift[4], q[4];     // cell of value x in band b: clamp((x - base) >> shift, 0, q - 1)
    int tmin, tmax;                  // limits of the data type
};

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool scratch = false;   // carved out of the context's slab, valid for one entry-point call
};

// One context per worker thread: a stream, named scratch buffers that only ever grow,
// a few pinned words for device->host scalars, per-stage events.
struct ssg_ctx {
    int device = 0;
    int numSMs = 148;
    cudaStream_t stream = nullptr;
    std::string err;
    uint64_t launches = 0;

    // N-sized arrays (N = pixels of the current tile)
    DevBuf img;       // staged image when the caller gave host memory
    DevBuf cluster;   // int32 cluster ids (assign -> clump); later scratch
    DevBuf label;     // uint32 root pixel per pixel (clump); later scratch
    DevBuf seg;       // uint32 segment ids
    DevBuf aux0, aux1, aux2;   // N-sized scratch (lists, moves)
    DevBuf singles;   // pixels of the single-pixel clumps, listed while the clumps are numbered
    // per-segment tables
    DevBuf segSize, isum, fsum, listOff, nextChunk, tailChunk, mergeTo, pendNext,
           candList, targetList, lut, flags;
    DevBuf blockCnt;  // per-block counts for the numbering scan
    DevBuf cubTemp;   // temp storage for the CUB scans / sorts
    DevBuf sortKeys0, sortKeys1, sortVals0, sortVals1;   // slow paths (oversized, ordered sums)
    DevBuf emuStack;
    DevBuf centres;   // double k*nBands
    DevBuf assignGrid;                  // candidate-centre masks of the pruning grid (kept between calls)
    std::vector<double> gridCentres;    // the centres it was built for
    int gridDtype = -1, gridK = 0;
    GridGeom gridGeom = {};
    std::vector<double> centresStage;
    std::vector<unsigned long long> grownStartStage;   // host copy of the merge kernel's list offsets
    DevBuf counters;  // small device counter block (see enum Counter)
    DevBuf stitch0, stitch1, stitch2, stitch3, stitch4, stitch5;

    // Scratch of one call comes out of one slab by bumping a pointer (cudaMalloc / cudaFree
    // synchronise the whole device, and the worker contexts of a tiled run would otherwise each
    // grow three dozen buffers the first time they meet the largest tile).  A call that needs
    // more than the slab holds gets plain allocations for the excess; the slab is regrown to the
    // observed need at the start of the next call.
    char *slab = nullptr;
    size_t slabCap = 0, slabUsed = 0, slabNeed = 0, spillBytes = 0;
    std::vector<void *> spills;
    std::vector<DevBuf *> scratchBufs;

    uint64_t *hostCounters = nullptr;   // pinned mirror of `counters`
    cudaEvent_t ev[8] = {};

    // optional per-kernel timing (ssg_profile_enable): every launch bracketed by two events
    bool profiling = false;
    std::vector<std::string> profNames;
    std::vector<int> profRecName;
    std::vector<cudaEvent_t> profEvents;   // 2 per record
    size_t profUsed = 0;                   // records in use
    bool profOpen = false;

    // stitch tables of the last ssg_tile_tables_device call
    int64_t stitchLen = 0;
    uint32_t stitchPairs = 0;
    std::vector<uint32_t> lutStage;

    // resident tile
    int64_t resRows = 0, resCols = 0;
    bool haveResident = false;
};

enum Counter {
    C_NUM_ROOTS = 0,
    C_NUM_OVERSIZED,
    C_NUM_SINGLES,
    C_NUM_SINGLEPIX,   // single-pixel clumps listed by the numbering pass
    C_NULL_SINGLE,     // exactly one null pixel (it counts as a single-pixel segment)
    C_NUM_MOVES,
    C_NUM_LEFT,
    C_NUM_ALIVE,
    C_NUM_SMALLSEG,
    C_NUM_SMALLPIX,
    C_NUM_BIGSUM,
    C_NUM_ELIM,
    C_MAXLABEL,
    C_SCRATCH0,
    C_SCRATCH1,
    C_SCRATCH2,
    C_SCRATCH3,
    C_MAXRANKTRIM,     // stitch: highest rank of a self-numbered segment inside the trimmed window
    C_COUNT = 32
};

#define SSG_FAIL(ctx, code, ...)                                        \
    do {                                                                \
        char _b[512];                                                   \
        snprintf(_b, sizeof(_b), __VA_ARGS__);                          \
        (ctx)->err = _b;                                                \
        return (code);                                                  \
    } while (0)

#define SSG_CUDA(ctx, call)                                             \
    do {                                                                \
        cudaError_t _e = (call);                                        \
        if (_e != cudaSuccess) {                                        \
            char _b[512];                                               \
            snprintf(_b, sizeof(_b), "%s:%d: %s: %s", __FILE__, __LINE__, #call, \
                     cudaGetErrorString(_e));                           \
            (ctx)->err = _b;                                            \
            return _e == cudaErrorMemoryAllocation ? SSG_ERR_NOMEM : SSG_ERR_CUDA; \
        }                                                               \
    } while (0)

#define SSG_TRY(call)                                                   \
    do {                                                                \
        int _rc = (call);                                               \
        if (_rc != SSG_OK) return _rc;                                  \
    } while (0)

// per-kernel timing: SSG_PROF_BEGIN before a launch, SSG_LAUNCHED after it
static inline void ssg_prof_begin(ssg_ctx *ctx, const char *name)
{
    if (!ctx->profiling) return;
    int id = -1;
    for (size_t i = 0; i < ctx->profNames.size(); i++)
        if (ctx->profNames[i] == name) { id = (int)i; break; }
    if (id < 0) { ctx->profNames.push_back(name); id = (int)ctx->profNames.size() - 1; }
    if (ctx->profEvents.size() < 2 * (ctx->profUsed + 1)) {
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        ctx->profEvents.push_back(a);
        ctx->profEvents.push_back(b);
    }
    if (ctx->profRecName.size() <= ctx->profUsed) ctx->profRecName.push_back(id);
    else ctx->profRecName[ctx->profUsed] = id;
    cudaEventRecord(ctx->profEvents[2 * ctx->profUsed], ctx->stream);
    ctx->profOpen = true;
}
static inline void ssg_prof_end(ssg_ctx *ctx)
{
    if (!ctx->profOpen) return;
    cudaEventRecord(ctx->profEvents[2 * ctx->profUsed + 1], ctx->stream);
    ctx->profUsed++;
    ctx->profOpen = false;
}
#define SSG_PROF_BEGIN(ctx, name) ssg_prof_begin(ctx, name)

// check the launch that has just been issued
#define SSG_LAUNCHED(ctx)                                               \
    do {                                                                \
        (ctx)->launches++;                                              \
        ssg_prof_end(ctx);                                              \
        SSG_CUDA(ctx, cudaGetLastError());                              \
    } while (0)

// device buffer of at least `bytes`: scratch buffers come out of the slab (contents are lost
// when they grow), the few persistent ones are grow-only allocations of their own
static inline int ssg_reserve(ssg_ctx *ctx, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return SSG_OK;
    if (b.scratch) {
        const size_t want = (bytes + 255) & ~(size_t)255;
        if (ctx->slabUsed + want <= ctx->slabCap) {
            b.p = ctx->slab + ctx->slabUsed;
            ctx->slabUsed += want;
        } else {
            void *q = nullptr;
            cudaError_t e = cudaMalloc(&q, want);
            if (e != cudaSuccess) {
                cudaGetLastError();
                SSG_FAIL(ctx, SSG_ERR_NOMEM, "cudaMalloc of %zu scratch bytes failed: %s", want, cudaGetErrorString(e));
            }
            ctx->spills.push_back(q);
            ctx->spillBytes += want;
            if (getenv("SSG_DEBUG_ALLOC")) fprintf(stderr, "[ssg %p] scratch spill %zu bytes (slab %zu used of %zu)\n", (void *)ctx, want, ctx->slabUsed, ctx->slabCap);
            b.p = q;
        }
        b.cap = want;
        if (ctx->slabUsed + ctx->spillBytes > ctx->slabNeed) ctx->slabNeed = ctx->slabUsed + ctx->spillBytes;
        return SSG_OK;
    }
    if (b.p) {
        SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        SSG_CUDA(ctx, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = bytes + bytes / 8 + 256;   // a little headroom: tiles of one run vary in size
    if (getenv("SSG_DEBUG_ALLOC")) fprintf(stderr, "[ssg %p] persistent buffer grows to %zu bytes\n", (void *)ctx, want);
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        e = cudaMalloc(&b.p, bytes);
        want = bytes;
    }
    if (e != cudaSuccess) {
        b.p = nullptr;
        cudaGetLastError();
        SSG_FAIL(ctx, SSG_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", bytes,
                 cudaGetErrorString(e));
    }
    b.cap = want;
    return SSG_OK;
}

// start of an entry-point call: every scratch buffer is forgotten, spilled allocations of the
// previous call are returned and the slab is regrown if that call needed more than it holds
static inline int ssg_scratch_reset(ssg_ctx *ctx, size_t atLeast = 0)
{
    for (DevBuf *b : ctx->scratchBufs) { b->p = nullptr; b->cap = 0; }
    ctx->slabUsed = 0;
    size_t need = ctx->slabNeed > atLeast ? ctx->slabNeed : atLeast;
    if (!ctx->spills.empty() || need > ctx->slabCap) {
        SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (void *q : ctx->spills) cudaFree(q);
        ctx->spills.clear();
        ctx->spillBytes = 0;
    }
    if (need > ctx->slabCap) {
        if (ctx->slab) cudaFree(ctx->slab);
        ctx->slab = nullptr;
        ctx->slabCap = 0;
        size_t want = need + need / 8 + (1u << 20);
        if (getenv("SSG_DEBUG_ALLOC")) fprintf(stderr, "[ssg %p] slab regrown to %zu bytes\n", (void *)ctx, want);
        void *q = nullptr;
        if (cudaMalloc(&q, want) != cudaSuccess) {
            cudaGetLastError();
            want = need;
            if (cudaMalloc(&q, want) != cudaSuccess) { cudaGetLastError(); q = nullptr; want = 0; }
        }
        ctx->slab = (char *)q;      // without a slab every reservation spills: slow, still correct
        ctx->slabCap = want;
    }
    return SSG_OK;
}

template <typename T>
static inline T *bufp(DevBuf &b) { return reinterpret_cast<T *>(b.p); }

static inline unsigned gridFor(int64_t n, int block)
{
    int64_t g = (n + block - 1) / block;
    if (g < 1) g = 1;
    return (unsigned)g;
}

// copy the counter block to the pinned mirror and wait for it
static inline int ssg_fetch_counters(ssg_ctx *ctx)
{
    SSG_CUDA(ctx, cudaMemcpyAsync(ctx->hostCounters, ctx->counters.p, C_COUNT * sizeof(uint64_t),
                                  cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSG_OK;
}

static inline size_t dtypeSize(int dt) { return dt == SSG_U8 ? 1 : (dt == SSG_U32 || dt == SSG_I32) ? 4 : 2; }

// ---- device helpers ----------------------------------------------------------------
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }

// one atomicAdd per warp for a per-thread 0/1 vote; returns this thread's slot (valid only
// where pred is true).  All 32 lanes of the warp must call it.
__device__ __forceinline__ unsigned long long warp_claim(unsigned long long *counter, bool pred)
{
    unsigned m = __ballot_sync(0xffffffffu, pred);
    unsigned long long base = 0;
    if (m == 0) return 0;
    int leader = __ffs(m) - 1;
    if ((int)lane_id() == leader) base = atomicAdd(counter, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + __popc(m & ((1u << lane_id()) - 1u));
}

// A per-thread count added to a global counter with ONE atomic per block (every thread of the
// block must call it): a counter that every warp of a large grid hits directly serialises
// thousands of atomics on one address, which costs more than the kernels that do the counting.
__device__ __forceinline__ void block_add(unsigned long long *counter, unsigned v)
{
    __shared__ unsigned long long blockAddSh;
    if (threadIdx.x == 0) blockAddSh = 0ull;
    __syncthreads();
    v = __reduce_add_sync(0xffffffffu, v);
    if (lane_id() == 0 && v) atomicAdd(&blockAddSh, (unsigned long long)v);
    __syncthreads();
    if (threadIdx.x == 0 && blockAddSh) atomicAdd(counter, blockAddSh);
    __syncthreads();
}

// Runs of equal keys over the lanes of a warp (consecutive pixels of a label raster are mostly
// runs of a few segments).  A run never spans an invalid lane or a lane flagged `breakBefore`.
// Cheaper than __match_any_sync + masked reductions: fixed cost, no divergence; a segment that
// shows up in two separate runs of the warp simply contributes twice.
struct WarpRuns {
    bool head;       // first lane of its run (does the atomics)
    unsigned end;    // last lane of my run
    unsigned len;    // run length (valid at the head)
};
__device__ __forceinline__ WarpRuns warp_runs(unsigned key, bool valid, bool breakBefore = false)
{
    const unsigned lane = lane_id();
    const unsigned prev = __shfl_up_sync(0xffffffffu, key, 1);
    const bool prevValid = __shfl_up_sync(0xffffffffu, (int)valid, 1) != 0;
    WarpRuns r;
    r.head = valid && (lane == 0 || !prevValid || prev != key || breakBefore);
    const unsigned bounds = __ballot_sync(0xffffffffu, r.head || !valid);
    const unsigned above = lane == 31 ? 0u : (bounds & ~((2u << lane) - 1u));
    r.end = above ? (unsigned)(__ffs(above) - 2) : 31u;
    r.len = r.end - lane + 1u;
    return r;
}
// sum of v over the lanes [lane, end] of the run; the head lane gets the run total
__device__ __forceinline__ unsigned run_suffix_add(unsigned v, const WarpRuns &r)
{
    const unsigned lane = lane_id();
#pragma unroll
    for (unsigned d = 1; d < 32; d <<= 1) {
        const unsigned t = __shfl_down_sync(0xffffffffu, v, d);
        if (lane + d <= r.end) v += t;
    }
    return v;
}

// Pixels whose segment is flagged (segFlag[seg[p]] != 0), grouped by segment with raster
// order kept inside each segment.  Outputs live in ctx scratch until the next call:
// pixSorted[M], keysSorted[M] (segment id of each entry, may be requested as nullptr),
// runStart[numRuns] (index of the first entry of every segment).
int ssgk_group_pixels(ssg_ctx *ctx, const unsigned *segDev, int64_t N, const unsigned char *segFlag,
                      const unsigned **pixSorted, const unsigned **keysSorted,
                      const unsigned **runStart, int64_t *M, unsigned *numRuns);

// stage entry points implemented in the other translation units ------------------------
int ssgk_apply_lut_extents(ssg_ctx *ctx, unsigned *seg, int64_t ysize, int64_t xsize, const unsigned *lut,
                           uint32_t numIds, const ssg_tile_params *prm, uint32_t *stride, bool *done);
int ssgk_apply_lut(ssg_ctx *ctx, unsigned *seg, int64_t N, const unsigned *lut);
int ssgk_assign(ssg_ctx *ctx, const void *imgDev, int dtype, int nBands, int64_t N,
                const double *centresHost, int k, int hasNull, double nullVal, int32_t *outDev);
// singlesOut (optional): receives the number of single-pixel clumps whose pixels were listed in
// ctx->singles, or -1 if the list cannot stand in for a scan (a lone null pixel exists)
int ssgk_clump(ssg_ctx *ctx, const int32_t *clusterDev, int64_t nRows, int64_t nCols,
               int32_t ignoreVal, int four, uint32_t clumpId, uint32_t *segDev,
               uint32_t *numClumps, uint32_t *numOversized, int64_t *singlesOut = nullptr);
int ssgk_seg_size(ssg_ctx *ctx, const uint32_t *segDev, int64_t N, uint32_t *sizeDev, int64_t len);
// cand0 / nCand0: the pixels of all single-pixel segments if the caller has them (device list),
// else nullptr / -1 and the first round scans the raster.  The label raster is not modified:
// *moveToOut (nullptr if nothing moved) goes to ssgk_relabel, which ends the stage.
int ssgk_eliminate_single(ssg_ctx *ctx, const void *imgDev, int dtype, int nBands, int64_t nRows,
                          int64_t nCols, const uint32_t *segDev, uint32_t *sizeDev, int64_t len,
                          int four, int64_t *numMoved, uint32_t *numRounds, const uint32_t **moveToOut,
                          const unsigned *cand0 = nullptr, int64_t nCand0 = -1);
int ssgk_eliminate_small(ssg_ctx *ctx, const void *imgDev, int dtype, int nBands, int64_t nRows,
                         int64_t nCols, uint32_t *segDev, uint32_t *sizeDev, uint32_t maxSegId,
                         int minSegSize, double thr, int four, int64_t *numElim,
                         uint32_t *numPasses, const uint32_t *pendingLut = nullptr, int64_t lutLen = 0);
// sizeOutDev (optional, len entries, must not alias sizeDev): the sizes under the new numbering.
// lutOut (optional): the relabel is only worked out, *lutOut (len entries, scratch of this call)
// maps old to new ids and the caller applies it.  moveTo (optional): see ssgk_eliminate_single.
int ssgk_relabel(ssg_ctx *ctx, uint32_t *segDev, int64_t N, const uint32_t *sizeDev, int64_t len,
                 uint32_t minSegId, uint32_t *numAlive, uint32_t *sizeOutDev = nullptr,
                 const uint32_t **lutOut = nullptr, const uint32_t *moveTo = nullptr);
