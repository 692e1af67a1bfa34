/*
 * shepseg_b200.h -- C ABI of libshepseg_b200.so, the B200 (sm_100a) implementation of
 * pyshepseg's Shepherd-segmentation hot path.
 *
 * The reference (ubarsc/pyshepseg 2.0.3) is pure Python + numba and has no FFI of its
 * own: the path is reached through the Python functions of pyshepseg/shepseg.py and
 * pyshepseg/tiling.py.  Each entry point below therefore cites the reference FUNCTION it
 * replaces; pyshepseg_b200/shepseg.py and pyshepseg_b200/tiling.py bind them with ctypes
 * behind the reference's own signatures (see INTEGRATION.md for the stub a maintainer
 * would add to the reference).
 *
 * Conventions
 *  - plain pointers and sizes only; no C++ or torch types cross this boundary;
 *  - every function returns 0 on success or an SSG_ERR_* code; the message is kept per
 *    context and read with ssg_last_error(); nothing throws across the boundary;
 *  - "host" pointers are caller-owned C-contiguous memory (pageable or pinned; pinned
 *    memory obtained from ssg_host_alloc makes the copies asynchronous and full speed);
 *    "device" pointers are CUDA device memory on the context's device;
 *  - images are band-sequential (nBands, nRows, nCols) like the reference's `img`
 *    (shepseg.py:140); label rasters are uint32 (nRows, nCols), 0 = null (shepseg.py:97-101);
 *  - a context owns one CUDA stream and its scratch memory, is bound to one device and
 *    must be used by one host thread at a time (use one context per worker thread, as the
 *    reference uses one worker per tile, tiling.py:1548-1613);
 *  - there is no CPU fallback: a context cannot be created without a CUDA device.
 */
#ifndef SHEPSEG_B200_H
#define SHEPSEG_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSG_ABI_VERSION 2

/* image element types (numpy dtypes the reference is used with) */
#define SSG_U8 0
#define SSG_U16 1
#define SSG_I16 2
#define SSG_U32 3      /* 32-bit values: the float32 band sums of most segments are not exact, */
#define SSG_I32 4      /* so they are accumulated in raster order (slower than 8/16-bit images) */

#define SSG_OK 0
#define SSG_ERR_ARG 1       /* bad argument (shape, dtype, null pointer, more than SSG_MAX_BANDS bands) */
#define SSG_ERR_CUDA 2      /* CUDA runtime error; ssg_last_error() has the string */
#define SSG_ERR_NOMEM 3     /* device or pinned allocation failed */
#define SSG_ERR_STATE 4     /* call sequence error (e.g. no resident tile) */

#define SSG_MAX_BANDS 64
#define SSG_MAX_CLUSTERS 1024

typedef struct ssg_ctx ssg_ctx;

/* ---- library / context -------------------------------------------------------------- */
int ssg_abi_version(void);
int ssg_device_count(void);
int ssg_ctx_create(int device, ssg_ctx **out);
/* the same with the context's stream at the device's highest priority: for the short
 * latency-critical work of a pipeline (the stitch kernels of the tiled driver, which would
 * otherwise queue behind the segmentation kernels of the worker contexts) */
int ssg_ctx_create_priority(int device, ssg_ctx **out);
void ssg_ctx_destroy(ssg_ctx *ctx);
const char *ssg_last_error(const ssg_ctx *ctx);
/* the context's cudaStream_t, so a caller can order its own work / events against it */
void *ssg_ctx_stream(ssg_ctx *ctx);
int ssg_ctx_synchronize(ssg_ctx *ctx);
/* size the context's device memory before the first tile arrives: the image staging and label
 * buffers for tiles of up to maxPixels pixels of nBands bands of `dtype` (skipped when either is
 * 0) and the per-call scratch slab (scratchBytes, or an estimate from maxPixels when 0).
 * Optional: everything grows on demand, but growing means cudaMalloc / cudaFree mid-run. */
int ssg_ctx_reserve(ssg_ctx *ctx, int64_t maxPixels, int nBands, int dtype, int64_t scratchBytes);
/* pinned host memory for full-speed asynchronous copies */
int ssg_host_alloc(size_t bytes, void **out);
int ssg_host_free(void *p);

/* ---- stage-level entry points: host buffers in, host buffers out --------------------- */

/* shepseg.applySpectralClusters (shepseg.py:317-361): out[p] = 1 + index of the nearest
 * centre (float64 ||c||^2 - 2 x.c, first minimum), 0 where any band equals nullVal. */
int ssg_assign(ssg_ctx *ctx, const void *img, int dtype, int nBands, int64_t nRows,
               int64_t nCols, const double *centres, int k, int hasNull, double nullVal,
               int32_t *out);

/* shepseg.clump (shepseg.py:452-541) including its MAX_CLUMP_SIZE=10000 splitting rule
 * and raster-scan numbering from clumpId; *nextId = highest id used + 1. */
int ssg_clump(ssg_ctx *ctx, const int32_t *img, int64_t nRows, int64_t nCols,
              int32_t ignoreVal, int fourConnected, uint32_t clumpId, uint32_t *out,
              uint32_t *nextId);

/* shepseg.makeSegSize (shepseg.py:544-569): segSize must hold max(seg)+1 entries. */
int ssg_make_seg_size(ssg_ctx *ctx, const uint32_t *seg, int64_t nPixels, uint32_t *segSize,
                      int64_t len);

/* shepseg.eliminateSinglePixels (shepseg.py:572-615): seg and segSize are updated in
 * place exactly as the reference leaves them (segSize stale after the final relabel). */
int ssg_eliminate_single_pixels(ssg_ctx *ctx, const void *img, int dtype, int nBands,
                                int64_t nRows, int64_t nCols, uint32_t *seg,
                                uint32_t *segSize, int64_t len, uint32_t minSegId,
                                int fourConnected, int64_t *numMoved);

/* shepseg.relabelSegments (shepseg.py:739-777): ids >= minSegId that own no pixel
 * (segSize == 0) are squeezed out, order preserved; seg is recoded in place, segSize (len
 * entries) is left as it is, like the reference leaves it.  Every id in seg must be below len. */
int ssg_relabel_segments(ssg_ctx *ctx, uint32_t *seg, int64_t nPixels, const uint32_t *segSize,
                         int64_t len, uint32_t minSegId);

/* shepseg.eliminateSmallSegments (shepseg.py:918-1000).  spectralThreshold is
 * maxSpectralDiff**2 evaluated in maxSpectralDiff's own type (float32 product for a
 * numpy.float32, shepseg.py:1060) and widened to double by the caller. */
int ssg_eliminate_small_segments(ssg_ctx *ctx, uint32_t *seg, const void *img, int dtype,
                                 int nBands, int64_t nRows, int64_t nCols, uint32_t maxSegId,
                                 int minSegSize, double spectralThreshold, int fourConnected,
                                 uint32_t minSegId, int64_t *numEliminated);

/* ---- the whole tile: shepseg.doShepherdSegmentation with kmeansObj given -------------- */
typedef struct ssg_tile_params {
    int dtype;             /* SSG_U8 / SSG_U16 / SSG_I16 / SSG_U32 / SSG_I32 */
    int nBands;
    int64_t nRows, nCols;
    const double *centres; /* host, k x nBands row-major (kmeansObj.cluster_centers_) */
    int k;
    int hasNull;           /* imgNullVal is not None */
    double nullVal;
    int fourConnected;
    int minSegSize;
    double spectralThreshold;
    /* Optional, for tiles that will be stitched (all zero / NULL otherwise): the final relabel of
     * the segmentation touches every pixel anyway, so it also fills the per-segment existence
     * tables that ssg_tile_tables_device needs (crossesMidline, tiling.py:1271-1306, and the
     * bounding-box corner test of relabelSegments, tiling.py:1255-1265) and the stitch does not
     * have to read the labels again.  [trimTop,trimBottom) x [trimLeft,trimRight) is the trimmed
     * window (tiling.py:997-1022), stripRows / stripCols the overlap with the upper / left
     * neighbour (0 without one).  extentsDev: device memory for SSG_EXTENT_TABLES byte tables of
     * extentsCap entries each; used only if the tile ends up with fewer than extentsCap ids. */
    int64_t trimTop, trimBottom, trimLeft, trimRight;
    int64_t stripRows, stripCols;
    uint8_t *extentsDev;
    int64_t extentsCap;
} ssg_tile_params;

#define SSG_EXTENT_TABLES 10

typedef struct ssg_tile_result {
    uint32_t numClumps;             /* ids after clump (shepseg.py:214) */
    uint32_t numSegments;           /* seg.max() of the final raster */
    uint32_t singlePixelsEliminated;/* shepseg.py:226-227 */
    int64_t smallSegmentsEliminated;/* shepseg.py:235 */
    uint32_t numOversized;          /* connected components that hit MAX_CLUMP_SIZE */
    uint32_t numSinglePixelRounds;
    uint32_t numSmallPasses;
    float msAssign, msClump, msSingle, msSmall, msTotal; /* device time of each stage */
    uint32_t extentsDone;           /* 1: the tables at ssg_tile_params.extentsDev are filled ... */
    uint32_t extentsStride;         /* ... table i starts at extentsDev + i * extentsStride */
} ssg_tile_result;

/* host image in, host labels out (segOut may be NULL: labels stay resident on the device
 * for ssg_stitch_* / ssg_download_labels).  Copies are inside the call. */
int ssg_segment_tile(ssg_ctx *ctx, const void *imgHost, const ssg_tile_params *prm,
                     uint32_t *segOutHost, ssg_tile_result *res);
/* device image in (already in HBM), labels stay on the device (segOutDev may be NULL to
 * keep them in the context; otherwise a device pointer to nRows*nCols uint32). */
int ssg_segment_tile_device(ssg_ctx *ctx, const void *imgDev, const ssg_tile_params *prm,
                            uint32_t *segOutDev, ssg_tile_result *res);
/* stage a host image in the context's device image buffer (asynchronous on the context's
 * stream when imgHost is pinned); ssg_staged_image returns that device pointer, to be passed
 * to ssg_segment_tile_device together with a per-tile device label buffer */
int ssg_upload_image(ssg_ctx *ctx, const void *imgHost, int dtype, int nBands, int64_t nRows,
                     int64_t nCols);
void *ssg_staged_image(ssg_ctx *ctx);
/* copy the resident labels of the last tile to host memory */
int ssg_download_labels(ssg_ctx *ctx, uint32_t *segOutHost);
/* device pointer of the resident labels of the last tile (owned by the context) */
uint32_t *ssg_resident_labels(ssg_ctx *ctx);

/* ---- spectral-cluster fit: the KMeans.fit call of shepseg.fitSpectralClusters
 *      (shepseg.py:252-314; tiling.fitSpectralClustersWholeFile, tiling.py:154-226) --------
 * The two steps of a Lloyd iteration as scikit-learn runs them ("lloyd" algorithm, float64), on
 * the device; the loop around them (stop when no label changes, when the summed squared centre
 * shift is <= tol, or after max_iter iterations) and the relocation of empty clusters are the
 * host's (pyshepseg_b200.shepseg._fitOnDevice).  X is the host sample matrix (n x nBands,
 * row-major), centres the initial centres (k x nBands).  Not bit identical to scikit-learn (order
 * of the sums, ties): centres agree to a tolerance stated in the tests.  One fit at a time per
 * host thread. */
int ssg_kmeans_begin(ssg_ctx *ctx, const double *X, int64_t n, int nBands, const double *centres, int k);
/* the assignment step with the current centres: samples per cluster, inertia, labels changed */
int ssg_kmeans_step(ssg_ctx *ctx, uint64_t *countsOut, double *inertia, uint64_t *changed);
/* labels of the last step (host, n) -- only needed when a cluster came out empty */
int ssg_kmeans_labels(ssg_ctx *ctx, int32_t *labelsOut);
/* sample farIdx[i] becomes the only member of empty cluster emptyIds[i] (scikit-learn's
 * _relocate_empty_clusters_dense; which samples is decided on the host with numpy, as there) */
int ssg_kmeans_relocate(ssg_ctx *ctx, int m, const int64_t *farIdx, const int32_t *emptyIds);
/* centres = mean of the samples assigned by the last step; summed squared shift; new centres (optional) */
int ssg_kmeans_update(ssg_ctx *ctx, double *shift, double *centresOut);
int ssg_kmeans_centres(ssg_ctx *ctx, double *centresOut);

/* ---- per-segment statistics: tilingstats.calcPerSegmentStatsTiled (tilingstats.py:85-215),
 *      accumulateSegDict (467-517), SegmentStats (923-1008) ---------------------------------
 * Statistics of one image band over the segments of a label raster of the same shape.  seg and
 * img are device pointers when onDevice (labels that are still resident), host pointers
 * otherwise.  Pixels of segment 0 and pixels equal to nullVal (when hasNull) do not count.
 * statIds: 0 min, 1 max, 2 mean, 3 stddev, 4 median, 5 mode, 6 percentile (params[i] = the
 * percentile), 7 pixcount -- the reference's STATID_* (tilingstats.py:770-777).  mean and
 * stddev go to float32 columns, the others to int64 columns (RatPage, tilingstats.py:1972-1996),
 * numbered in the order given: intOut is (number of int statistics, maxSegId + 1) row-major,
 * floatOut likewise.  A segment without valid pixels gets `missing` everywhere except in a
 * pixcount column (0, SegmentStats.getStat, 1006-1007); row 0 is zero.  totalOut (maxSegId + 1,
 * may be NULL) receives every segment's pixel count with the null-valued pixels included -- what
 * the reference compares with the Histogram column to decide a segment is complete
 * (checkSegComplete, 519-554).  A label above maxSegId is an error. */
int ssg_segment_stats(ssg_ctx *ctx, const uint32_t *seg, const void *img, int dtype, int64_t nPixels,
                      int onDevice, int hasNull, int64_t nullVal, uint32_t maxSegId, int nStats,
                      const int32_t *statIds, const int32_t *params, int64_t missing,
                      int64_t *intOut, float *floatOut, uint32_t *totalOut);

/* ---- tile stitching: tiling.stitchTiles / recodeTile / recodeSharedSegments /
 *      relabelSegments / crossesMidline (tiling.py:950-1306) --------------------------
 *
 * The reference stitches tile after tile in row-major order, carrying a running maxSegId
 * and the recoded overlap strips of the finished neighbours.  Here the per-pixel work is
 * done on the device in two parallel phases around a tiny sequential resolve on the host
 * (pyshepseg_b200/tiling.py), which is what lets tiles live on different GPUs:
 *
 *   ssg_tile_tables_device  per tile, independent of all other tiles' FINAL ids: bounding-box
 *                           corner of every segment (relabelSegments, tiling.py:1255-1265),
 *                           which segments cross the overlap midlines (crossesMidline,
 *                           tiling.py:1271-1306), the rank of every segment the tile numbers
 *                           itself (ascending id, tiling.py:1250-1267), and for the crossing
 *                           segments the histogram of the neighbour tile's LOCAL labels under
 *                           their strip pixels (the input of scipy.stats.mode, tiling.py:1194);
 *   (host)                  lut = offset + rank; neighbour labels mapped through the
 *                           neighbour's lut, counts of equal final ids added, mode taken
 *                           (smallest id on ties), left overlap overriding top
 *                           (tiling.py:1107-1121); offset = max(offset, max lut inside the
 *                           trimmed window) (tiling.py:1042-1043);
 *   ssg_apply_lut_device    out = lut[tile] over the trimmed window, straight into the mosaic
 *                           (or a staging buffer) + histogram (tiling.py:1032-1035).
 */
typedef struct ssg_tile_tables {
    uint32_t maxId;     /* largest label in the tile */
    uint32_t countNew;  /* segments numbered by this tile (flag SSG_SEG_NUMBERED) */
    uint32_t numPairs;  /* distinct (strip, segment, neighbour label) triples */
    uint32_t maxRankInTrim; /* highest rank among the numbered segments with a pixel in the trimmed window */
} ssg_tile_tables;

#define SSG_SEG_PRESENT 1u   /* id owns at least one pixel of the tile */
#define SSG_SEG_NUMBERED 2u  /* numbered by this tile: lut = offset + rank */
#define SSG_SEG_KEYTOP 4u    /* crosses the midline of the top overlap */
#define SSG_SEG_KEYLEFT 8u   /* crosses the midline of the left overlap */
#define SSG_SEG_INTRIM 16u   /* has a pixel inside the trimmed window */
#define SSG_PAIR_LEFT (1ull << 63) /* pair key = strip bit | segment << 32 | neighbour label */

/* tileDev: device labels (ysize, xsize) with contiguous ids 1..max.  topBDev / leftBDev:
 * the labels of the upper / left neighbour under this tile's top `overlap` rows / left
 * `overlap` columns (row strides in elements, so they may point into the neighbour's
 * resident label raster), or NULL on the first tile row / column.  [top,bottom) x
 * [left,right) is the trimmed window (tiling.py:997-1022).  maxIdHint is the largest label of
 * the tile when the caller knows it (ssg_tile_result.numSegments), 0 to have it searched.
 * extentsDev / extentsStride: the existence tables the segmentation of this tile filled
 * (ssg_tile_result.extentsDone, for the same window and overlaps), or NULL / 0 to have them
 * computed here from the labels.
 * Results stay in the context until the next call; sizes come back in *out. */
int ssg_tile_tables_device(ssg_ctx *ctx, const uint32_t *tileDev, int64_t ysize, int64_t xsize,
                           int64_t overlap, const uint32_t *topBDev, int64_t topBStride,
                           const uint32_t *leftBDev, int64_t leftBStride, int64_t top,
                           int64_t bottom, int64_t left, int64_t right, uint32_t maxIdHint,
                           const uint8_t *extentsDev, int64_t extentsStride,
                           ssg_tile_tables *out);
/* rank[maxId+1] (1-based among the numbered segments, 0 otherwise), flags[maxId+1]
 * (SSG_SEG_*), pairKeys[numPairs] ascending, pairCounts[numPairs]; host buffers. */
int ssg_tile_tables_fetch(ssg_ctx *ctx, uint32_t *rank, uint8_t *flags, uint64_t *pairKeys,
                          uint32_t *pairCounts);
/* out[(r-top)*outStride + (c-left)] = lut[tile[r,c]] for the trimmed window; lutHost has
 * maxId+1 entries.  outDev is device memory (a mosaic window or a staging buffer).  If
 * histDev is not NULL, histDev[v] += 1 for every written value v < histLen. */
int ssg_apply_lut_device(ssg_ctx *ctx, const uint32_t *tileDev, int64_t ysize, int64_t xsize,
                         const uint32_t *lutHost, uint32_t maxId, int64_t top, int64_t bottom,
                         int64_t left, int64_t right, uint32_t *outDev, int64_t outStride,
                         uint64_t *histDev, int64_t histLen);
/* The same with the lut put together on the device: lut[i] = offset + rankHost[i] where
 * flagsHost[i] has SSG_SEG_NUMBERED (a segment the tile numbered itself, tiling.py:1264-1267;
 * both as ssg_tile_tables_fetch returned them; rankHost NULL: every label numbers itself, the
 * simple recode of tiling.py:1067-1092), 0 elsewhere, then
 * lut[crossLabelsHost[j]] = crossIdsHost[j] for the nCross segments that take a neighbour's id.
 * Used when the offset is the last thing to become known (tiles sharded over several GPUs). */
int ssg_apply_rel_lut_device(ssg_ctx *ctx, const uint32_t *tileDev, int64_t ysize, int64_t xsize,
                             const uint32_t *rankHost, const uint8_t *flagsHost, uint32_t maxId,
                             uint32_t offset, int64_t nCross,
                             const uint32_t *crossLabelsHost, const uint32_t *crossIdsHost,
                             int64_t top, int64_t bottom, int64_t left, int64_t right,
                             uint32_t *outDev, int64_t outStride, uint64_t *histDev, int64_t histLen);
/* Overviews of a window that is in device memory (TilingSegmenter.writeOverviews,
 * tiling.py:1360-1383): for every level L the sub-sampled window arr[L/2::L, L/2::L], all levels
 * packed one after the other (each row-major) into outHost; startsOut (nLevels + 1) receives the
 * element offset of every level and the total.  Level l has len(range(L/2, wRows, L)) rows and
 * len(range(L/2, wCols, L)) columns.  Synchronous. */
int ssg_window_overviews(ssg_ctx *ctx, const uint32_t *winDev, int64_t wRows, int64_t wCols,
                         int64_t winStride, int nLevels, const int32_t *levels, uint32_t *outHost,
                         int64_t outCapacity, int64_t *startsOut);

/* ---- plain device memory helpers (so the Python side needs nothing but ctypes) -------- */
int ssg_dev_alloc(ssg_ctx *ctx, size_t bytes, void **out);
int ssg_dev_free(ssg_ctx *ctx, void *p);
int ssg_memcpy_h2d(ssg_ctx *ctx, void *dst, const void *src, size_t bytes);
int ssg_memcpy_d2h(ssg_ctx *ctx, void *dst, const void *src, size_t bytes);
int ssg_memcpy_d2d(ssg_ctx *ctx, void *dst, const void *src, size_t bytes);
/* strided 2-D copies on the context's stream (rows of `widthBytes`, pitches in bytes) */
int ssg_memcpy2d_d2d(ssg_ctx *ctx, void *dst, size_t dpitch, const void *src, size_t spitch,
                     size_t widthBytes, size_t rows);
int ssg_memcpy2d_d2h(ssg_ctx *ctx, void *dst, size_t dpitch, const void *src, size_t spitch,
                     size_t widthBytes, size_t rows);
int ssg_memcpy2d_h2d(ssg_ctx *ctx, void *dst, size_t dpitch, const void *src, size_t spitch,
                     size_t widthBytes, size_t rows);
int ssg_memset_d(ssg_ctx *ctx, void *dst, int value, size_t bytes);
/* the same device-to-host copies without waiting for them, and marks to wait on later: the tiled
 * driver lets the last (largest) window travel while the host already works on the histogram
 * (HistogramAccumulator / utils.estimateStatsFromHisto, tiling.py:1915-1963, utils.py:47-95).
 * The host buffer should be pinned (ssg_host_alloc) or the copy is not asynchronous. */
int ssg_memcpy_d2h_async(ssg_ctx *ctx, void *dst, const void *src, size_t bytes);
int ssg_memcpy2d_d2h_async(ssg_ctx *ctx, void *dst, size_t dpitch, const void *src, size_t spitch,
                           size_t widthBytes, size_t rows);
/* record mark `slot` (0..2) on the context's stream / block the host until it has been reached */
int ssg_mark(ssg_ctx *ctx, int slot);
int ssg_wait_mark(ssg_ctx *ctx, int slot);


/* per-kernel device timing: while enabled every kernel launch is bracketed by two CUDA
 * events on the context's stream; ssg_profile_fetch writes "name count total_ms" lines for
 * the launches since the last fetch into buf (NUL terminated) and resets the records */
int ssg_profile_enable(ssg_ctx *ctx, int on);
int ssg_profile_fetch(ssg_ctx *ctx, char *buf, size_t cap);

/* number of kernels this library has launched on the context since creation */
uint64_t ssg_launch_count(const ssg_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* SHEPSEG_B200_H */
