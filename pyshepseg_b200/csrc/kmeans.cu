// kmeans.cu -- Lloyd iterations of the spectral-cluster fit on the device.
// Replaces the scikit-learn KMeans.fit call of shepseg.fitSpectralClusters (shepseg.py:252-314,
// tiling.py:154-226) when the caller asks for it: the same algorithm as scikit-learn's "lloyd"
// (assign every sample to its nearest centre, move every centre to the mean of its samples,
// stop when the labels do not change any more or the summed squared centre shift falls below
// tol = 1e-4 * mean feature variance, at most max_iter iterations), in float64.  It is NOT bit
// identical to scikit-learn (the sums are accumulated in another order, ties may break
// differently): the centres agree to a stated tolerance, which tests/ holds it to.
// An empty cluster keeps its centre (scikit-learn moves it to the sample farthest from its centre).
#include "common.cuh"

#define KM_THREADS 256

// one Lloyd step: labels, per-cluster sums and counts, inertia, number of labels that changed.
// NBMAX (16 or 64) bounds nB: a sample is held in registers
template <int NBMAX>
__global__ void __launch_bounds__(KM_THREADS)
k_lloyd_step(const double *__restrict__ X, int64_t n, int nB, const double *__restrict__ centres, int k,
             int *labels, double *sums, unsigned long long *counts, double *scalars /* [0] inertia */,
             unsigned long long *changed, int useShared)
{
    extern __shared__ double sh[];
    double *cs = sh;                       // k*nB centres
    double *cn = cs + (size_t)k * nB;      // k squared norms
    double *bs = cn + k;                   // k*nB block sums   (useShared)
    unsigned long long *bc = reinterpret_cast<unsigned long long *>(bs + (size_t)k * nB);   // k block counts
    for (int i = threadIdx.x; i < k * nB; i += blockDim.x) cs[i] = centres[i];
    __syncthreads();
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        double s = 0.0;
        for (int b = 0; b < nB; b++) s += cs[j * nB + b] * cs[j * nB + b];
        cn[j] = s;
    }
    if (useShared) {
        for (int i = threadIdx.x; i < k * nB; i += blockDim.x) bs[i] = 0.0;
        for (int j = threadIdx.x; j < k; j += blockDim.x) bc[j] = 0ull;
    }
    __syncthreads();
    double inertia = 0.0;
    unsigned nChanged = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double x[NBMAX];
        double xx = 0.0;
        for (int b = 0; b < nB; b++) { x[b] = X[i * nB + b]; xx += x[b] * x[b]; }
        int best = 0;
        double bestD = 0.0;
        for (int j = 0; j < k; j++) {
            double dot = 0.0;
            for (int b = 0; b < nB; b++) dot += x[b] * cs[j * nB + b];
            const double d = cn[j] - 2.0 * dot;
            if (j == 0 || d < bestD) { bestD = d; best = j; }
        }
        inertia += bestD + xx;
        if (labels[i] != best) { nChanged++; labels[i] = best; }
        if (useShared) {
            for (int b = 0; b < nB; b++) atomicAdd(&bs[best * nB + b], x[b]);
            atomicAdd(&bc[best], 1ull);
        } else {
            for (int b = 0; b < nB; b++) atomicAdd(&sums[(size_t)best * nB + b], x[b]);
            atomicAdd(&counts[best], 1ull);
        }
    }
    __syncthreads();
    if (useShared) {
        for (int i = threadIdx.x; i < k * nB; i += blockDim.x)
            if (bs[i] != 0.0) atomicAdd(&sums[i], bs[i]);
        for (int j = threadIdx.x; j < k; j += blockDim.x)
            if (bc[j]) atomicAdd(&counts[j], bc[j]);
    }
    // block totals of inertia and changes
    __shared__ double redI[KM_THREADS / 32];
    __shared__ unsigned redC[KM_THREADS / 32];
    for (int o = 16; o > 0; o >>= 1) {
        inertia += __shfl_xor_sync(0xffffffffu, inertia, o);
        nChanged += __shfl_xor_sync(0xffffffffu, nChanged, o);
    }
    if (lane_id() == 0) { redI[threadIdx.x >> 5] = inertia; redC[threadIdx.x >> 5] = nChanged; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ti = 0.0;
        unsigned tc = 0;
        for (int w = 0; w < KM_THREADS / 32; w++) { ti += redI[w]; tc += redC[w]; }
        atomicAdd(&scalars[0], ti);
        if (tc) atomicAdd(changed, (unsigned long long)tc);
    }
}

// centres = sums / counts; scalars[1] = summed squared shift; the accumulators are cleared
__global__ void __launch_bounds__(256)
k_lloyd_update(double *centres, int k, int nB, double *sums, unsigned long long *counts, double *scalars)
{
    __shared__ double red[256];
    double shift = 0.0;
    for (int i = threadIdx.x; i < k * nB; i += blockDim.x) {
        const int j = i / nB;
        const unsigned long long c = counts[j];
        const double old = centres[i];
        const double neu = c ? sums[i] / (double)c : old;      // an empty cluster keeps its centre
        centres[i] = neu;
        shift += (neu - old) * (neu - old);
        sums[i] = 0.0;
    }
    red[threadIdx.x] = shift;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    for (int j = threadIdx.x; j < k; j += blockDim.x) counts[j] = 0ull;
    if (threadIdx.x == 0) scalars[1] = red[0];
}

// sums[old cluster of sample far] -= x, sums[empty] = x, counts likewise: scikit-learn's
// _relocate_empty_clusters_dense, applied to the accumulators of the step that has just run
__global__ void k_lloyd_relocate(const double *__restrict__ X, int nB, const int *__restrict__ labels, int m,
                                 const long long *__restrict__ farIdx, const int *__restrict__ emptyIds, double *sums,
                                 unsigned long long *counts)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    for (int i = 0; i < m; i++) {
        const long long f = farIdx[i];
        const int oldC = labels[f], newC = emptyIds[i];
        for (int b = 0; b < nB; b++) {
            sums[(size_t)oldC * nB + b] -= X[f * nB + b];
            sums[(size_t)newC * nB + b] = X[f * nB + b];
        }
        counts[newC] = 1ull;
        counts[oldC] -= 1ull;
    }
}

struct KmState {
    double *X, *C, *sums, *scalars;
    int *labels;
    unsigned long long *counts, *changed;
    int64_t n;
    int nB, k, useShared;
    void (*step)(const double *, int64_t, int, const double *, int, int *, double *, unsigned long long *, double *,
                 unsigned long long *, int);
    size_t smem;
    int64_t blocks;
};
static thread_local KmState g_km;      // the fit in progress on this thread's context

extern "C" int ssg_kmeans_begin(ssg_ctx *ctx, const double *X, int64_t n, int nB, const double *centres, int k)
{
    if (!ctx) return SSG_ERR_ARG;
    ctx->err.clear();
    SSG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!X || !centres || n < 1 || nB < 1 || nB > SSG_MAX_BANDS || k < 1 || k > SSG_MAX_CLUSTERS)
        SSG_FAIL(ctx, SSG_ERR_ARG, "bad argument");
    SSG_TRY(ssg_scratch_reset(ctx));
    const size_t xBytes = (size_t)n * nB * sizeof(double), cBytes = (size_t)k * nB * sizeof(double);
    SSG_TRY(ssg_reserve(ctx, ctx->aux0, xBytes));
    SSG_TRY(ssg_reserve(ctx, ctx->aux1, (size_t)n * sizeof(int)));
    SSG_TRY(ssg_reserve(ctx, ctx->aux2, 2 * cBytes + (size_t)k * sizeof(unsigned long long) + 64 +
                                        (size_t)k * (sizeof(long long) + sizeof(int))));
    KmState &km = g_km;
    km.X = bufp<double>(ctx->aux0);
    km.labels = bufp<int>(ctx->aux1);
    km.C = bufp<double>(ctx->aux2);
    km.sums = km.C + (size_t)k * nB;
    km.counts = reinterpret_cast<unsigned long long *>(km.sums + (size_t)k * nB);
    km.scalars = reinterpret_cast<double *>(km.counts + k);      // [0] inertia, [1] shift, [2] changed (u64)
    km.changed = reinterpret_cast<unsigned long long *>(km.scalars + 2);
    km.n = n; km.nB = nB; km.k = k;
    SSG_CUDA(ctx, cudaMemcpyAsync(km.X, X, xBytes, cudaMemcpyHostToDevice, ctx->stream));
    SSG_CUDA(ctx, cudaMemcpyAsync(km.C, centres, cBytes, cudaMemcpyHostToDevice, ctx->stream));
    SSG_CUDA(ctx, cudaMemsetAsync(km.labels, 0xff, (size_t)n * sizeof(int), ctx->stream));
    SSG_CUDA(ctx, cudaMemsetAsync(km.sums, 0, cBytes + (size_t)k * sizeof(unsigned long long) + 32, ctx->stream));
    km.smem = ((size_t)k * nB + k) * sizeof(double);
    const size_t smemSums = km.smem + (size_t)k * nB * sizeof(double) + (size_t)k * sizeof(unsigned long long);
    km.useShared = smemSums <= 96 * 1024;
    if (km.useShared) km.smem = smemSums;
    if (km.smem > 200 * 1024)
        SSG_FAIL(ctx, SSG_ERR_ARG, "the device k-means fit holds the centres in 200 KB of shared memory: "
                 "%d clusters x %d bands need %zu bytes; use fewer clusters or the scikit-learn fit",
                 k, nB, (size_t)(k * nB + k) * sizeof(double));
    km.step = nB <= 16 ? k_lloyd_step<16> : k_lloyd_step<64>;
    if (km.smem > 48 * 1024)
        SSG_CUDA(ctx, cudaFuncSetAttribute(km.step, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)km.smem));
    km.blocks = (n + KM_THREADS - 1) / KM_THREADS;
    if (km.blocks > (int64_t)ctx->numSMs * 4) km.blocks = (int64_t)ctx->numSMs * 4;
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));      // (X may be reused by the caller)
    return SSG_OK;
}

// the assignment step with the current centres: counts per cluster (k), inertia, labels changed
extern "C" int ssg_kmeans_step(ssg_ctx *ctx, uint64_t *countsOut, double *inertia, uint64_t *changed)
{
    if (!ctx) return SSG_ERR_ARG;
    ctx->err.clear();
    SSG_CUDA(ctx, cudaSetDevice(ctx->device));
    KmState &km = g_km;
    if (!km.X) SSG_FAIL(ctx, SSG_ERR_STATE, "ssg_kmeans_begin has not been called");
    const size_t cBytes = (size_t)km.k * km.nB * sizeof(double);
    SSG_CUDA(ctx, cudaMemsetAsync(km.sums, 0, cBytes + (size_t)km.k * sizeof(unsigned long long) + 32, ctx->stream));
    SSG_PROF_BEGIN(ctx, "k_lloyd_step");
    km.step<<<(unsigned)km.blocks, KM_THREADS, km.smem, ctx->stream>>>(km.X, km.n, km.nB, km.C, km.k, km.labels, km.sums,
                                                                       km.counts, km.scalars, km.changed, km.useShared);
    SSG_LAUNCHED(ctx);
    struct { double inertia, shift; unsigned long long changed; } h;
    if (countsOut) SSG_CUDA(ctx, cudaMemcpyAsync(countsOut, km.counts, (size_t)km.k * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaMemcpyAsync(&h, km.scalars, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (inertia) *inertia = h.inertia;
    if (changed) *changed = h.changed;
    return SSG_OK;
}

extern "C" int ssg_kmeans_labels(ssg_ctx *ctx, int32_t *labelsOut)
{
    if (!ctx) return SSG_ERR_ARG;
    ctx->err.clear();
    SSG_CUDA(ctx, cudaSetDevice(ctx->device));
    KmState &km = g_km;
    if (!km.X || !labelsOut) SSG_FAIL(ctx, SSG_ERR_STATE, "no fit in progress");
    SSG_CUDA(ctx, cudaMemcpyAsync(labelsOut, km.labels, (size_t)km.n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSG_OK;
}

extern "C" int ssg_kmeans_relocate(ssg_ctx *ctx, int m, const int64_t *farIdx, const int32_t *emptyIds)
{
    if (!ctx) return SSG_ERR_ARG;
    ctx->err.clear();
    SSG_CUDA(ctx, cudaSetDevice(ctx->device));
    KmState &km = g_km;
    if (!km.X) SSG_FAIL(ctx, SSG_ERR_STATE, "no fit in progress");
    if (m < 1) return SSG_OK;
    if (m > km.k || !farIdx || !emptyIds) SSG_FAIL(ctx, SSG_ERR_ARG, "bad argument");
    long long *dFar = reinterpret_cast<long long *>(km.changed + 2);
    int *dEmpty = reinterpret_cast<int *>(dFar + km.k);
    SSG_CUDA(ctx, cudaMemcpyAsync(dFar, farIdx, (size_t)m * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
    SSG_CUDA(ctx, cudaMemcpyAsync(dEmpty, emptyIds, (size_t)m * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    SSG_PROF_BEGIN(ctx, "k_lloyd_relocate");
    k_lloyd_relocate<<<1, 32, 0, ctx->stream>>>(km.X, km.nB, km.labels, m, dFar, dEmpty, km.sums, km.counts);
    SSG_LAUNCHED(ctx);
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSG_OK;
}

// centres = sums / counts of the last step; returns the summed squared shift; centresOut optional
extern "C" int ssg_kmeans_update(ssg_ctx *ctx, double *shift, double *centresOut)
{
    if (!ctx) return SSG_ERR_ARG;
    ctx->err.clear();
    SSG_CUDA(ctx, cudaSetDevice(ctx->device));
    KmState &km = g_km;
    if (!km.X) SSG_FAIL(ctx, SSG_ERR_STATE, "no fit in progress");
    SSG_PROF_BEGIN(ctx, "k_lloyd_update");
    k_lloyd_update<<<1, 256, 0, ctx->stream>>>(km.C, km.k, km.nB, km.sums, km.counts, km.scalars);
    SSG_LAUNCHED(ctx);
    double h[2];
    SSG_CUDA(ctx, cudaMemcpyAsync(h, km.scalars, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    if (centresOut) SSG_CUDA(ctx, cudaMemcpyAsync(centresOut, km.C, (size_t)km.k * km.nB * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (shift) *shift = h[1];
    return SSG_OK;
}

extern "C" int ssg_kmeans_centres(ssg_ctx *ctx, double *centresOut)
{
    if (!ctx) return SSG_ERR_ARG;
    ctx->err.clear();
    SSG_CUDA(ctx, cudaSetDevice(ctx->device));
    KmState &km = g_km;
    if (!km.X || !centresOut) SSG_FAIL(ctx, SSG_ERR_STATE, "no fit in progress");
    SSG_CUDA(ctx, cudaMemcpyAsync(centresOut, km.C, (size_t)km.k * km.nB * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SSG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SSG_OK;
}
