// api.cu -- the extern "C" boundary of libshepseg_b200.so (see include/shepseg_b200.h).
// Context lifetime, host<->device staging for the stage-level entry points, and the fused
// tile pipeline assign -> clump -> single pixels -> small segments -> relabel
// (shepseg.doShepherdSegmentation, shepseg.py:130-249).
#include "common.cuh"

static thread_local std::string g_noCtxError;

extern "C" {

int ssg_abi_version(void) { return SSG_ABI_VERSION; }

int ssg_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

static int ctx_create(int device, int highPriority, ssg_ctx **out);

int ssg_ctx_create(int device, ssg_ctx **out) { return ctx_create(device, 0, out); }
int ssg_ctx_create_priority(int device, ssg_ctx **out) { return ctx_create(device, 1, out); }

static int ctx_create(int device, int highPriority, ssg_ctx **out)
{
    if (!out) return SSG_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return SSG_ERR_CUDA; }
    if (device < 0 || device >= n) return SSG_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return SSG_ERR_CUDA; }
    ssg_ctx *ctx = new ssg_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->numSMs = prop.multiProcessorCount;
    int prLow = 0, prHigh = 0;
    cudaDeviceGetStreamPriorityRange(&prLow, &prHigh);     // (numerically lower = more urgent)
    if (cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, highPriority ? prHigh : prLow) != cudaSuccess) { delete ctx; return SSG_ERR_CUDA; }
    if (cudaMalloc(&ctx->counters.p, C_COUNT * sizeof(uint64_t)) != cudaSuccess) { cudaStreamDestroy(ctx->stream); delete ctx; return SSG_ERR_NOMEM; }
    ctx->counters.cap = C_COUNT * sizeof(uint64_t);
    cudaMemsetAsync(ctx->counters.p, 0, ctx->counters.cap, ctx->stream);
    if (cudaMallocHost(&ctx->hostCounters, C_COUNT * sizeof(uint64_t)) != cudaSuccess) {
        cudaFree(ctx->counters.p); cudaStreamDestroy(ctx->stream); delete ctx; return SSG_ERR_NOMEM;
    }
    for (auto &e : ctx->ev) cudaEventCreate(&e);
    // everything that lives for one call only comes out of the slab; what outlives a call (the
    // staged image, the resident labels, the stitch tables read by ssg_tile_tables_fetch, the
    // centres, the counters) keeps an allocation of its own
    DevBuf *scratch[] = {&ctx->cluster, &ctx->label, &ctx->aux0, &ctx->aux1, &ctx->aux2, &ctx->singles,
                         &ctx->segSize, &ctx->isum, &ctx->fsum, &ctx->listOff, &ctx->nextChunk, &ctx->tailChunk,
                         &ctx->mergeTo, &ctx->pendNext, &ctx->candList, &ctx->targetList, &ctx->lut,
                         &ctx->flags, &ctx->blockCnt, &ctx->cubTemp, &ctx->sortKeys0, &ctx->sortKeys1, &ctx->sortVals0,
                         &ctx->sortVals1, &ctx->emuStack, &ctx->stitch0, &ctx->stitch2, &ctx->stitch3};
    for (DevBuf *b : scratch) { b->scratch = true; ctx->scratchBufs.push_back(b); }
    cudaStreamSynchronize(ctx->stream);
    *out = ctx;
    return SSG_OK;
}

void ssg_ctx_destroy(ssg_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    DevBuf *bufs[] = {&ctx->img, &ctx->cluster, &ctx->label, &ctx->seg, &ctx->aux0, &ctx->aux1, &ctx->aux2, &ctx->singles,
                      &ctx->segSize, &ctx->isum, &ctx->fsum, &ctx->listOff, &ctx->nextChunk, &ctx->tailChunk,
                      &ctx->mergeTo, &ctx->pendNext, &ctx->candList, &ctx->targetList, &ctx->lut,
                      &ctx->flags, &ctx->blockCnt, &ctx->cubTemp, &ctx->sortKeys0, &ctx->sortKeys1, &ctx->sortVals0,
                      &ctx->sortVals1, &ctx->emuStack, &ctx->centres, &ctx->assignGrid, &ctx->counters, &ctx->stitch0, &ctx->stitch1,
                      &ctx->stitch2, &ctx->stitch3, &ctx->stitch4, &ctx->stitch5};
    for (DevBuf *b : bufs) if (b->p && !b->scratch) cudaFree(b->p);
    for (void *q : ctx->spills) cudaFree(q);
    if (ctx->slab) cudaFree(ctx->slab);
    if (ctx->hostCounters) cudaFreeHost(ctx->hostCounters);
    for (auto &e : ctx->ev) if (e) cudaEventDestroy(e);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *ssg_last_error(const ssg_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context"; }
void *ssg_ctx_stream(ssg_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
uint64_t ssg_launch_count(const ssg_ctx *ctx) { return ctx ? ctx->launches : 0; }

#define CTX_ENTER(ctx)                                                  \
    if (!(ctx)) return SSG_ERR_ARG;                                     \
    (ctx)->err.clear();                                                 \
    SSG_CUDA(ctx, cudaSetDevice((ctx)->device))

int ssg_profile_enable(ssg_ctx *ctx, int on)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->profiling = on != 0;
    ctx->profUsed = 0;
    ctx->profOpen = false;
    return SSG_OK;
}

// "name count total_ms\n" per kernel, since the last fetch / enable
int ssg_profile_fetch(ssg_ctx *ctx, char *buf, size_t cap)
{
    CTX_ENTER(ctx);
    if (!buf || cap == 0) SSG_FAIL(ctx, SSG_ERR_ARG, "null buffer");
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    std::vector<double> total(ctx->profNames.size(), 0.0);
    std::vector<long long> count(ctx->profNames.size(), 0);
    for (size_t r = 0; r < ctx->profUsed; r++) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->profEvents[2 * r], ctx->profEvents[2 * r + 1]) == cudaSuccess) {
            total[ctx->profRecName[r]] += ms;
            count[ctx->profRecName[r]]++;
        } else {
            cudaGetLastError();
        }
    }
    std::string out;
    char line[256];
    for (size_t i = 0; i < ctx->profNames.size(); i++) {
        if (!count[i]) continue;
        snprintf(line, sizeof(line), "%s %lld %.6f\n", ctx->profNames[i].c_str(), count[i], total[i]);
        out += line;
    }
    ctx->profUsed = 0;
    if (out.size() + 1 > cap) SSG_FAIL(ctx, SSG_ERR_ARG, "profile buffer too small (%zu needed)", out.size() + 1);
    memcpy(buf, out.c_str(), out.size() + 1);
    return SSG_OK;
}

int ssg_ctx_synchronize(ssg_ctx *ctx)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSG_OK;
}

int ssg_host_alloc(size_t bytes, void **out)
{
    if (!out) return SSG_ERR_ARG;
    if (cudaMallocHost(out, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); *out = nullptr; return SSG_ERR_NOMEM; }
    return SSG_OK;
}

int ssg_host_free(void *p)
{
    if (p && cudaFreeHost(p) != cudaSuccess) { cudaGetLastError(); return SSG_ERR_CUDA; }
    return SSG_OK;
}

int ssg_ctx_reserve(ssg_ctx *ctx, int64_t maxPixels, int nBands, int dtype, int64_t scratchBytes)
{
    CTX_ENTER(ctx);
    if (maxPixels < 0 || nBands < 0 || nBands > SSG_MAX_BANDS || scratchBytes < 0) SSG_FAIL(ctx, SSG_ERR_ARG, "bad argument");
    // measured on noisy 4-band imagery: about 40 bytes of scratch per pixel (cluster, root and
    // single-pixel rasters, pixel lists, per-segment tables); a tile that needs more spills once
    // and the slab follows
    const size_t slab = scratchBytes > 0 ? (size_t)scratchBytes
                                         : (size_t)maxPixels * (size_t)(40 + 2 * nBands) + ((size_t)64 << 20);
    SSG_TRY(ssg_scratch_reset(ctx, slab));
    if (nBands > 0 && maxPixels > 0) {
        SSG_TRY(ssg_reserve(ctx, ctx->img, (size_t)maxPixels * nBands * dtypeSize(dtype)));
        SSG_TRY(ssg_reserve(ctx, ctx->seg, (size_t)maxPixels * sizeof(uint32_t)));
    }
    return SSG_OK;
}

// ---- plain memory helpers --------------------------------------------------------------------
int ssg_dev_alloc(ssg_ctx *ctx, size_t bytes, void **out)
{
    CTX_ENTER(ctx);
    if (!out) SSG_FAIL(ctx, SSG_ERR_ARG, "null out pointer");
    SSG_CUDA(ctx, cudaMalloc(out, bytes ? bytes : 1));
    return SSG_OK;
}
int ssg_dev_free(ssg_ctx *ctx, void *p)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (p) SSG_CUDA(ctx, cudaFree(p));
    return SSG_OK;
}
int ssg_memcpy_h2d(ssg_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return SSG_OK;
}
int ssg_memcpy_d2h(ssg_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSG_OK;
}
int ssg_memcpy_d2d(ssg_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return SSG_OK;
}
int ssg_memcpy2d_d2d(ssg_ctx *ctx, void *dst, size_t dpitch, const void *src, size_t spitch, size_t widthBytes, size_t rows)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaMemcpy2DAsync(dst, dpitch, src, spitch, widthBytes, rows, cudaMemcpyDeviceToDevice, ctx->stream));
    return SSG_OK;
}
int ssg_memcpy2d_d2h(ssg_ctx *ctx, void *dst, size_t dpitch, const void *src, size_t spitch, size_t widthBytes, size_t rows)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaMemcpy2DAsync(dst, dpitch, src, spitch, widthBytes, rows, cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSG_OK;
}
int ssg_memcpy2d_h2d(ssg_ctx *ctx, void *dst, size_t dpitch, const void *src, size_t spitch, size_t widthBytes, size_t rows)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaMemcpy2DAsync(dst, dpitch, src, spitch, widthBytes, rows, cudaMemcpyHostToDevice, ctx->stream));
    return SSG_OK;
}
int ssg_memcpy_d2h_async(ssg_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return SSG_OK;
}
int ssg_memcpy2d_d2h_async(ssg_ctx *ctx, void *dst, size_t dpitch, const void *src, size_t spitch, size_t widthBytes, size_t rows)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaMemcpy2DAsync(dst, dpitch, src, spitch, widthBytes, rows, cudaMemcpyDeviceToHost, ctx->stream));
    return SSG_OK;
}
int ssg_mark(ssg_ctx *ctx, int slot)
{
    CTX_ENTER(ctx);
    if (slot < 0 || slot > 2) SSG_FAIL(ctx, SSG_ERR_ARG, "mark slot %d not in 0..2", slot);
    SSG_CUDA(ctx, cudaEventRecord(ctx->ev[5 + slot], ctx->stream));
    return SSG_OK;
}
int ssg_wait_mark(ssg_ctx *ctx, int slot)
{
    CTX_ENTER(ctx);
    if (slot < 0 || slot > 2) SSG_FAIL(ctx, SSG_ERR_ARG, "mark slot %d not in 0..2", slot);
    SSG_CUDA(ctx, cudaEventSynchronize(ctx->ev[5 + slot]));
    return SSG_OK;
}
int ssg_memset_d(ssg_ctx *ctx, void *dst, int value, size_t bytes)
{
    CTX_ENTER(ctx);
    SSG_CUDA(ctx, cudaMemsetAsync(dst, value, bytes, ctx->stream));
    return SSG_OK;
}

// ---- argument checks -------------------------------------------------------------------------
static int check_image_args(ssg_ctx *ctx, const void *img, int dtype, int nBands, int64_t nRows, int64_t nCols)
{
    if (!img && nRows * nCols > 0) SSG_FAIL(ctx, SSG_ERR_ARG, "null image pointer");
    if (dtype < SSG_U8 || dtype > SSG_I32) SSG_FAIL(ctx, SSG_ERR_ARG, "unsupported dtype code %d (uint8, uint16, int16, uint32 and int32 images are supported)", dtype);
    if (nBands < 1 || nBands > SSG_MAX_BANDS) SSG_FAIL(ctx, SSG_ERR_ARG, "nBands=%d not in 1..%d", nBands, SSG_MAX_BANDS);
    if (nRows < 0 || nCols < 0) SSG_FAIL(ctx, SSG_ERR_ARG, "negative image size");
    if (nRows * nCols >= 0x7FFFFFF0ll) SSG_FAIL(ctx, SSG_ERR_ARG, "tile of %lld pixels is too large (use the tiled entry point)", (long long)(nRows * nCols));
    return SSG_OK;
}

static int upload_image(ssg_ctx *ctx, const void *imgHost, int dtype, int nBands, int64_t N)
{
    const size_t bytes = (size_t)N * nBands * dtypeSize(dtype);
    SSG_TRY(ssg_reserve(ctx, ctx->img, bytes ? bytes : 16));
    if (bytes) SSG_CUDA(ctx, cudaMemcpyAsync(ctx->img.p, imgHost, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return SSG_OK;
}

// ---- stage-level entry points (host buffers) ---------------------------------------------------
int ssg_assign(ssg_ctx *ctx, const void *img, int dtype, int nBands, int64_t nRows, int64_t nCols,
               const double *centres, int k, int hasNull, double nullVal, int32_t *out)
{
    CTX_ENTER(ctx);
    SSG_TRY(ssg_scratch_reset(ctx));
    SSG_TRY(check_image_args(ctx, img, dtype, nBands, nRows, nCols));
    if (!centres || (!out && nRows * nCols > 0)) SSG_FAIL(ctx, SSG_ERR_ARG, "null pointer argument");
    const int64_t N = nRows * nCols;
    if (N == 0) return SSG_OK;
    SSG_TRY(upload_image(ctx, img, dtype, nBands, N));
    SSG_TRY(ssg_reserve(ctx, ctx->cluster, (size_t)N * sizeof(int32_t)));
    SSG_TRY(ssgk_assign(ctx, ctx->img.p, dtype, nBands, N, centres, k, hasNull, nullVal, bufp<int32_t>(ctx->cluster)));
    SSG_CUDA(ctx, cudaMemcpyAsync(out, ctx->cluster.p, (size_t)N * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSG_OK;
}

int ssg_clump(ssg_ctx *ctx, const int32_t *img, int64_t nRows, int64_t nCols, int32_t ignoreVal,
              int fourConnected, uint32_t clumpId, uint32_t *out, uint32_t *nextId)
{
    CTX_ENTER(ctx);
    SSG_TRY(ssg_scratch_reset(ctx));
    if (nRows < 0 || nCols < 0 || nRows * nCols >= 0x7FFFFFF0ll) SSG_FAIL(ctx, SSG_ERR_ARG, "bad raster size");
    const int64_t N = nRows * nCols;
    if (nextId) *nextId = clumpId;
    if (N == 0) return SSG_OK;
    if (!img || !out) SSG_FAIL(ctx, SSG_ERR_ARG, "null pointer argument");
    SSG_TRY(ssg_reserve(ctx, ctx->cluster, (size_t)N * sizeof(int32_t)));
    SSG_TRY(ssg_reserve(ctx, ctx->seg, (size_t)N * sizeof(uint32_t)));
    SSG_CUDA(ctx, cudaMemcpyAsync(ctx->cluster.p, img, (size_t)N * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    uint32_t numClumps = 0, numOver = 0;
    SSG_TRY(ssgk_clump(ctx, bufp<int32_t>(ctx->cluster), nRows, nCols, ignoreVal, fourConnected, clumpId,
                       bufp<uint32_t>(ctx->seg), &numClumps, &numOver));
    SSG_CUDA(ctx, cudaMemcpyAsync(out, ctx->seg.p, (size_t)N * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (nextId) *nextId = clumpId + numClumps;
    return SSG_OK;
}

int ssg_make_seg_size(ssg_ctx *ctx, const uint32_t *seg, int64_t nPixels, uint32_t *segSize, int64_t len)
{
    CTX_ENTER(ctx);
    SSG_TRY(ssg_scratch_reset(ctx));
    if (nPixels < 0 || len < 0 || (!seg && nPixels > 0) || (!segSize && len > 0)) SSG_FAIL(ctx, SSG_ERR_ARG, "bad argument");
    if (len == 0) return SSG_OK;
    SSG_TRY(ssg_reserve(ctx, ctx->seg, (size_t)(nPixels ? nPixels : 1) * sizeof(uint32_t)));
    SSG_TRY(ssg_reserve(ctx, ctx->segSize, (size_t)len * sizeof(uint32_t)));
    if (nPixels) SSG_CUDA(ctx, cudaMemcpyAsync(ctx->seg.p, seg, (size_t)nPixels * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    SSG_TRY(ssgk_seg_size(ctx, bufp<uint32_t>(ctx->seg), nPixels, bufp<uint32_t>(ctx->segSize), len));
    SSG_CUDA(ctx, cudaMemcpyAsync(segSize, ctx->segSize.p, (size_t)len * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSG_OK;
}

int ssg_eliminate_single_pixels(ssg_ctx *ctx, const void *img, int dtype, int nBands, int64_t nRows,
                                int64_t nCols, uint32_t *seg, uint32_t *segSize, int64_t len,
                                uint32_t minSegId, int fourConnected, int64_t *numMoved)
{
    CTX_ENTER(ctx);
    SSG_TRY(ssg_scratch_reset(ctx));
    SSG_TRY(check_image_args(ctx, img, dtype, nBands, nRows, nCols));
    const int64_t N = nRows * nCols;
    if (numMoved) *numMoved = 0;
    if (N == 0) return SSG_OK;
    if (!seg || !segSize || len < 1) SSG_FAIL(ctx, SSG_ERR_ARG, "null pointer argument");
    SSG_TRY(upload_image(ctx, img, dtype, nBands, N));
    SSG_TRY(ssg_reserve(ctx, ctx->seg, (size_t)N * sizeof(uint32_t)));
    SSG_TRY(ssg_reserve(ctx, ctx->segSize, (size_t)len * sizeof(uint32_t)));
    SSG_CUDA(ctx, cudaMemcpyAsync(ctx->seg.p, seg, (size_t)N * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    SSG_CUDA(ctx, cudaMemcpyAsync(ctx->segSize.p, segSize, (size_t)len * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    int64_t moved = 0;
    uint32_t rounds = 0, alive = 0;
    const uint32_t *moveTo = nullptr;
    SSG_TRY(ssgk_eliminate_single(ctx, ctx->img.p, dtype, nBands, nRows, nCols, bufp<uint32_t>(ctx->seg),
                                  bufp<uint32_t>(ctx->segSize), len, fourConnected, &moved, &rounds, &moveTo));
    // the reference leaves segSize as mergeSinglePixels updated it and relabels seg (shepseg.py:615)
    SSG_CUDA(ctx, cudaMemcpyAsync(segSize, ctx->segSize.p, (size_t)len * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_TRY(ssgk_relabel(ctx, bufp<uint32_t>(ctx->seg), N, bufp<uint32_t>(ctx->segSize), len, minSegId, &alive,
                         nullptr, nullptr, moveTo));
    SSG_CUDA(ctx, cudaMemcpyAsync(seg, ctx->seg.p, (size_t)N * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (numMoved) *numMoved = moved;
    return SSG_OK;
}

int ssg_relabel_segments(ssg_ctx *ctx, uint32_t *seg, int64_t nPixels, const uint32_t *segSize, int64_t len,
                         uint32_t minSegId)
{
    CTX_ENTER(ctx);
    SSG_TRY(ssg_scratch_reset(ctx));
    if (nPixels < 0 || len < 0 || (!seg && nPixels > 0) || (!segSize && len > 0)) SSG_FAIL(ctx, SSG_ERR_ARG, "bad argument");
    if (nPixels == 0 || len == 0) return SSG_OK;
    SSG_TRY(ssg_reserve(ctx, ctx->seg, (size_t)nPixels * sizeof(uint32_t)));
    SSG_TRY(ssg_reserve(ctx, ctx->segSize, (size_t)len * sizeof(uint32_t)));
    SSG_CUDA(ctx, cudaMemcpyAsync(ctx->seg.p, seg, (size_t)nPixels * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    SSG_CUDA(ctx, cudaMemcpyAsync(ctx->segSize.p, segSize, (size_t)len * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    uint32_t alive = 0;
    SSG_TRY(ssgk_relabel(ctx, bufp<uint32_t>(ctx->seg), nPixels, bufp<uint32_t>(ctx->segSize), len, minSegId, &alive));
    SSG_CUDA(ctx, cudaMemcpyAsync(seg, ctx->seg.p, (size_t)nPixels * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSG_OK;
}

int ssg_eliminate_small_segments(ssg_ctx *ctx, uint32_t *seg, const void *img, int dtype, int nBands,
                                 int64_t nRows, int64_t nCols, uint32_t maxSegId, int minSegSize,
                                 double spectralThreshold, int fourConnected, uint32_t minSegId,
                                 int64_t *numEliminated)
{
    CTX_ENTER(ctx);
    SSG_TRY(ssg_scratch_reset(ctx));
    SSG_TRY(check_image_args(ctx, img, dtype, nBands, nRows, nCols));
    const int64_t N = nRows * nCols;
    if (numEliminated) *numEliminated = 0;
    if (N == 0) return SSG_OK;
    if (!seg) SSG_FAIL(ctx, SSG_ERR_ARG, "null pointer argument");
    if (minSegId != 1) SSG_FAIL(ctx, SSG_ERR_ARG, "minSegId must be 1 (shepseg.MINSEGID)");
    const int64_t len = (int64_t)maxSegId + 1;
    SSG_TRY(upload_image(ctx, img, dtype, nBands, N));
    SSG_TRY(ssg_reserve(ctx, ctx->seg, (size_t)N * sizeof(uint32_t)));
    SSG_TRY(ssg_reserve(ctx, ctx->segSize, (size_t)len * sizeof(uint32_t)));
    SSG_CUDA(ctx, cudaMemcpyAsync(ctx->seg.p, seg, (size_t)N * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    SSG_TRY(ssgk_seg_size(ctx, bufp<uint32_t>(ctx->seg), N, bufp<uint32_t>(ctx->segSize), len));
    int64_t numElim = 0;
    uint32_t passes = 0, alive = 0;
    SSG_TRY(ssgk_eliminate_small(ctx, ctx->img.p, dtype, nBands, nRows, nCols, bufp<uint32_t>(ctx->seg),
                                 bufp<uint32_t>(ctx->segSize), maxSegId, minSegSize, spectralThreshold,
                                 fourConnected, &numElim, &passes));
    SSG_TRY(ssgk_relabel(ctx, bufp<uint32_t>(ctx->seg), N, bufp<uint32_t>(ctx->segSize), len, minSegId, &alive));
    SSG_CUDA(ctx, cudaMemcpyAsync(seg, ctx->seg.p, (size_t)N * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (numEliminated) *numEliminated = numElim;
    return SSG_OK;
}

// ---- the fused tile pipeline -------------------------------------------------------------------
static int segment_tile_impl(ssg_ctx *ctx, const void *imgDev, const ssg_tile_params *prm,
                             uint32_t *segDev, ssg_tile_result *res)
{
    const int64_t N = prm->nRows * prm->nCols;
    memset(res, 0, sizeof(*res));
    if (N == 0) return SSG_OK;
    unsigned long long *counters = bufp<unsigned long long>(ctx->counters);
    SSG_TRY(ssg_reserve(ctx, ctx->cluster, (size_t)N * sizeof(int32_t)));

    SSG_CUDA(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
    SSG_TRY(ssgk_assign(ctx, imgDev, prm->dtype, prm->nBands, N, prm->centres, prm->k, prm->hasNull,
                        prm->nullVal, bufp<int32_t>(ctx->cluster)));
    SSG_CUDA(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));

    uint32_t numClumps = 0, numOver = 0;
    int64_t numSingles = -1;
    SSG_TRY(ssgk_clump(ctx, bufp<int32_t>(ctx->cluster), prm->nRows, prm->nCols, 0, prm->fourConnected, 1,
                       segDev, &numClumps, &numOver, &numSingles));
    SSG_CUDA(ctx, cudaEventRecord(ctx->ev[2], ctx->stream));
    const int64_t len = (int64_t)numClumps + 1;
    unsigned *segSize = bufp<unsigned>(ctx->segSize);

    int64_t moved = 0;
    uint32_t rounds = 0;
    const uint32_t *moveTo = nullptr;
    SSG_TRY(ssgk_eliminate_single(ctx, imgDev, prm->dtype, prm->nBands, prm->nRows, prm->nCols, segDev,
                                  segSize, len, prm->fourConnected, &moved, &rounds, &moveTo,
                                  numSingles >= 0 ? bufp<unsigned>(ctx->singles) : nullptr, numSingles));
    // the reference relabels here (eliminateSinglePixels ends with relabelSegments,
    // shepseg.py:615), and so do we: three quarters of the clump ids are gone, and every table
    // of the next stage is that much smaller (they then sit in L2 instead of HBM).
    // singlePixelsEliminated = oldMaxSegId - seg.max() (shepseg.py:226-227)
    uint32_t afterSingles = numClumps;
    const uint32_t *pendingLut = nullptr;
    if (numClumps > 0) {
        SSG_TRY(ssg_reserve(ctx, ctx->aux2, (size_t)len * sizeof(unsigned)));
        unsigned *compact = bufp<unsigned>(ctx->aux2);
        // (worked out here, applied by the pixel pass of the next stage)
        SSG_TRY(ssgk_relabel(ctx, segDev, N, segSize, len, 1, &afterSingles, compact, &pendingLut, moveTo));
        segSize = compact;
    }
    const int64_t len1 = (int64_t)afterSingles + 1;
    SSG_CUDA(ctx, cudaEventRecord(ctx->ev[3], ctx->stream));

    int64_t numElim = 0;
    uint32_t passes = 0, alive = 0;
    SSG_TRY(ssgk_eliminate_small(ctx, imgDev, prm->dtype, prm->nBands, prm->nRows, prm->nCols, segDev, segSize,
                                 afterSingles, prm->minSegSize, prm->spectralThreshold, prm->fourConnected,
                                 &numElim, &passes, pendingLut, len));
    // the final relabel; for a tile that will be stitched the same pass fills the existence tables
    const uint32_t *finalLut = nullptr;
    SSG_TRY(ssgk_relabel(ctx, segDev, N, segSize, len1, 1, &alive, nullptr, &finalLut));
    bool extDone = false;
    uint32_t extStride = 0;
    SSG_TRY(ssgk_apply_lut_extents(ctx, segDev, prm->nRows, prm->nCols, finalLut, alive, prm, &extStride, &extDone));
    if (!extDone) SSG_TRY(ssgk_apply_lut(ctx, segDev, N, finalLut));
    SSG_CUDA(ctx, cudaEventRecord(ctx->ev[4], ctx->stream));
    SSG_TRY(ssg_fetch_counters(ctx));

    res->numClumps = numClumps;
    res->numOversized = numOver;
    res->numSegments = alive;
    res->singlePixelsEliminated = numClumps - afterSingles;
    res->smallSegmentsEliminated = numElim;
    res->numSinglePixelRounds = rounds;
    res->numSmallPasses = passes;
    res->extentsDone = extDone ? 1u : 0u;
    res->extentsStride = extStride;
    cudaEventElapsedTime(&res->msAssign, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&res->msClump, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&res->msSingle, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&res->msSmall, ctx->ev[3], ctx->ev[4]);
    cudaEventElapsedTime(&res->msTotal, ctx->ev[0], ctx->ev[4]);
    return SSG_OK;
}

static int check_tile_params(ssg_ctx *ctx, const void *img, const ssg_tile_params *prm, ssg_tile_result *res)
{
    if (!prm || !res) SSG_FAIL(ctx, SSG_ERR_ARG, "null params/result");
    SSG_TRY(check_image_args(ctx, img, prm->dtype, prm->nBands, prm->nRows, prm->nCols));
    if (!prm->centres) SSG_FAIL(ctx, SSG_ERR_ARG, "null centres");
    if (prm->k < 1 || prm->k > SSG_MAX_CLUSTERS) SSG_FAIL(ctx, SSG_ERR_ARG, "k=%d not in 1..%d", prm->k, SSG_MAX_CLUSTERS);
    return SSG_OK;
}

int ssg_segment_tile_device(ssg_ctx *ctx, const void *imgDev, const ssg_tile_params *prm,
                            uint32_t *segOutDev, ssg_tile_result *res)
{
    CTX_ENTER(ctx);
    SSG_TRY(ssg_scratch_reset(ctx));
    SSG_TRY(check_tile_params(ctx, imgDev, prm, res));
    const int64_t N = prm->nRows * prm->nCols;
    uint32_t *segDev = segOutDev;
    if (!segDev) {
        SSG_TRY(ssg_reserve(ctx, ctx->seg, (size_t)(N ? N : 1) * sizeof(uint32_t)));
        segDev = bufp<uint32_t>(ctx->seg);
    }
    SSG_TRY(segment_tile_impl(ctx, imgDev, prm, segDev, res));
    ctx->resRows = prm->nRows;
    ctx->resCols = prm->nCols;
    ctx->haveResident = (segOutDev == nullptr);
    return SSG_OK;
}

int ssg_segment_tile(ssg_ctx *ctx, const void *imgHost, const ssg_tile_params *prm,
                     uint32_t *segOutHost, ssg_tile_result *res)
{
    CTX_ENTER(ctx);
    SSG_TRY(ssg_scratch_reset(ctx));
    SSG_TRY(check_tile_params(ctx, imgHost, prm, res));
    const int64_t N = prm->nRows * prm->nCols;
    SSG_TRY(upload_image(ctx, imgHost, prm->dtype, prm->nBands, N));
    SSG_TRY(ssg_reserve(ctx, ctx->seg, (size_t)(N ? N : 1) * sizeof(uint32_t)));
    SSG_TRY(segment_tile_impl(ctx, ctx->img.p, prm, bufp<uint32_t>(ctx->seg), res));
    ctx->resRows = prm->nRows;
    ctx->resCols = prm->nCols;
    ctx->haveResident = true;
    if (segOutHost && N > 0) {
        SSG_CUDA(ctx, cudaMemcpyAsync(segOutHost, ctx->seg.p, (size_t)N * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return SSG_OK;
}

int ssg_upload_image(ssg_ctx *ctx, const void *imgHost, int dtype, int nBands, int64_t nRows, int64_t nCols)
{
    CTX_ENTER(ctx);
    SSG_TRY(check_image_args(ctx, imgHost, dtype, nBands, nRows, nCols));
    return upload_image(ctx, imgHost, dtype, nBands, nRows * nCols);
}

void *ssg_staged_image(ssg_ctx *ctx) { return ctx ? ctx->img.p : nullptr; }

int ssg_download_labels(ssg_ctx *ctx, uint32_t *segOutHost)
{
    CTX_ENTER(ctx);
    if (!ctx->haveResident) SSG_FAIL(ctx, SSG_ERR_STATE, "no resident tile labels");
    const int64_t N = ctx->resRows * ctx->resCols;
    if (N > 0) {
        SSG_CUDA(ctx, cudaMemcpyAsync(segOutHost, ctx->seg.p, (size_t)N * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return SSG_OK;
}

uint32_t *ssg_resident_labels(ssg_ctx *ctx)
{
    if (!ctx || !ctx->haveResident) return nullptr;
    return bufp<uint32_t>(ctx->seg);
}

}  // extern "C"
