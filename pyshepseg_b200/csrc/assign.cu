// assign.cu -- K1: per-pixel nearest-centre assignment.
// Replaces shepseg.applySpectralClusters (shepseg.py:317-361), i.e. scikit-learn's
// KMeans.predict on the band-interleaved pixel matrix plus the +1 / null masking.
//
// Result contract (what the reference computes): argmin_j of the float64 value
// ||c_j||^2 - 2 x.c_j, first minimum on ties, +1; 0 if any band equals imgNullVal.
//
// How it is done here: each thread takes V consecutive pixels of every band plane with one
// wide load per band (coalesced, 16 B per lane for uint16 at V=8), the centres sit in
// shared memory (float32 copies of -2c and ||c||^2 for the fast pass, float64 copies for the
// exact pass) and are read as warp-wide broadcasts.  The fast pass evaluates
// ||c_j||^2 - 2 x.c_j as nB chained FFMAs per centre (half the FP32 work of sum (x-c)^2) and
// tracks the best and second-best value.  With u = 2^-24 every such value is within
// E = (nB+1) * 1.01 * u * (max||c||^2 + 2 max|c| sum_b |x_b|) of the real one, so whenever
// second - best > 2E (+ the float64 margin) the float32 argmin IS the float64 argmin; otherwise
// the pixel is re-evaluated in float64 with exactly the operation sequence of the oracle
// (separate multiply and add, no FMA), so the label equals the float64 first-minimum argmin
// in every case, ties included.
#include "common.cuh"

template <typename T, int V>
__device__ __forceinline__ void load_vec(const T *p, float (&x)[V])
{
    constexpr int BYTES = V * (int)sizeof(T);
    if constexpr (BYTES == 16) {
        uint4 r = __ldg(reinterpret_cast<const uint4 *>(p));
        const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
        for (int i = 0; i < V; i++) x[i] = (float)e[i];
    } else if constexpr (BYTES == 8) {
        uint2 r = __ldg(reinterpret_cast<const uint2 *>(p));
        const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
        for (int i = 0; i < V; i++) x[i] = (float)e[i];
    } else if constexpr (BYTES == 4) {
        unsigned r = __ldg(reinterpret_cast<const unsigned *>(p));
        const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
        for (int i = 0; i < V; i++) x[i] = (float)e[i];
    } else if constexpr (BYTES == 2 && V == 2) {
        unsigned short r = __ldg(reinterpret_cast<const unsigned short *>(p));
        const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
        for (int i = 0; i < V; i++) x[i] = (float)e[i];
    } else {
#pragma unroll
        for (int i = 0; i < V; i++) x[i] = (float)__ldg(p + i);
    }
}

struct AssignBounds {
    float perAbsX, constant;   // tolerance on second - best = perAbsX * sum_b |x_b| + constant
};

// exact pass for one pixel: same float64 sequence as the oracle / scikit-learn form.  X is float
// for 8/16-bit images (every such value is exact in float32) and double for 32-bit ones.
template <int NB, typename X>
__device__ __noinline__ int assign_exact(const X (&x)[NB], const double *cd, const double *cn,
                                         int k)
{
    int best = 0;
    double bestD = 0.0;
    for (int j = 0; j < k; j++) {
        double dot = 0.0;
#pragma unroll
        for (int b = 0; b < NB; b++)
            dot = __dadd_rn(dot, __dmul_rn((double)x[b], cd[j * NB + b]));
        double d = __dadd_rn(cn[j], __dmul_rn(-2.0, dot));
        if (j == 0 || d < bestD) { bestD = d; best = j; }
    }
    return best;
}

template <typename T, int NB, int V>
__global__ void __launch_bounds__(256)
k_assign(const T *__restrict__ img, int64_t N, const double *__restrict__ centres, int k,
         int hasNull, double nullVal, AssignBounds bnd, int32_t *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smemRaw[];
    double *cd = reinterpret_cast<double *>(smemRaw);          // k*NB
    double *cn = cd + (size_t)k * NB;                          // k
    float *cf = reinterpret_cast<float *>(cn + k);             // k*(NB+1): ||c||^2, then -2c

    for (int i = threadIdx.x; i < k * NB; i += blockDim.x) {
        double c = centres[i];
        cd[i] = c;
        cf[(i / NB) * (NB + 1) + 1 + (i % NB)] = (float)(-2.0 * c);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        double s = 0.0;
#pragma unroll
        for (int b = 0; b < NB; b++) s = __dadd_rn(s, __dmul_rn(cd[j * NB + b], cd[j * NB + b]));
        cn[j] = s;
        cf[j * (NB + 1)] = (float)s;
    }
    __syncthreads();

    const int64_t nGroups = (N + V - 1) / V;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < nGroups;
         g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p0 = g * V;
        float x[V][NB];
        const bool full = (p0 + V <= N);
        if (full) {
#pragma unroll
            for (int b = 0; b < NB; b++) {
                float t[V];
                load_vec<T, V>(img + (size_t)b * N + p0, t);
#pragma unroll
                for (int v = 0; v < V; v++) x[v][b] = t[v];
            }
        } else {
#pragma unroll
            for (int b = 0; b < NB; b++)
#pragma unroll
                for (int v = 0; v < V; v++)
                    x[v][b] = (p0 + v < N) ? (float)__ldg(img + (size_t)b * N + p0 + v) : 0.0f;
        }

        float best[V], second[V];
        int idx[V];
#pragma unroll
        for (int v = 0; v < V; v++) { best[v] = 3.0e38f; second[v] = 3.0e38f; idx[v] = 0; }

        for (int j = 0; j < k; j++) {
            float c[NB + 1];
#pragma unroll
            for (int b = 0; b <= NB; b++) c[b] = cf[j * (NB + 1) + b];
#pragma unroll
            for (int v = 0; v < V; v++) {
                float acc = c[0];
#pragma unroll
                for (int b = 0; b < NB; b++) acc = fmaf(x[v][b], c[b + 1], acc);
                second[v] = fminf(second[v], fmaxf(acc, best[v]));
                bool lt = acc < best[v];
                best[v] = fminf(acc, best[v]);
                idx[v] = lt ? j : idx[v];
            }
        }

        int32_t res[V];
#pragma unroll
        for (int v = 0; v < V; v++) {
            if constexpr (sizeof(T) == 4) {
                // (the pixel is read again below: a padding slot of the last group has none)
                if (p0 + v >= N) { res[v] = 0; continue; }
            }
            float gap = second[v] - best[v];
            float absSum = 0.0f;
#pragma unroll
            for (int b = 0; b < NB; b++) absSum += fabsf(x[v][b]);
            float tol = fmaf(bnd.perAbsX, absSum, bnd.constant);
            int lab = idx[v];
            if (k > 1 && !(gap > tol)) {
                if constexpr (sizeof(T) == 4) {
                    // x[][] holds 32-bit values rounded to float32: the exact pass reads the integers
                    double xv[NB];
#pragma unroll
                    for (int b = 0; b < NB; b++) xv[b] = (double)__ldg(img + (size_t)b * N + p0 + v);
                    lab = assign_exact<NB>(xv, cd, cn, k);
                } else {
                    float xv[NB];   // copy: keeps x[][] itself in registers
#pragma unroll
                    for (int b = 0; b < NB; b++) xv[b] = x[v][b];
                    lab = assign_exact<NB>(xv, cd, cn, k);
                }
            }
            bool isNull = false;
            if (hasNull) {
                if constexpr (sizeof(T) == 4) {
                    // rounding to float32 is monotonic, so x == nullVal implies (float)x == (float)nullVal;
                    // the integer itself decides (4294967295 and 4294967200 round to the same float)
#pragma unroll
                    for (int b = 0; b < NB; b++) isNull |= (x[v][b] == (float)nullVal);
                    if (isNull) {
                        isNull = false;
#pragma unroll
                        for (int b = 0; b < NB; b++)
                            isNull |= ((double)__ldg(img + (size_t)b * N + p0 + v) == nullVal);
                    }
                } else {
#pragma unroll
                    for (int b = 0; b < NB; b++) isNull |= ((double)x[v][b] == nullVal);
                }
            }
            res[v] = isNull ? 0 : lab + 1;
        }
        bool stored = false;
        if constexpr (V == 8) {
            if (full) {
                int4 *o = reinterpret_cast<int4 *>(out + p0);
                o[0] = make_int4(res[0], res[1], res[2], res[3]);
                o[1] = make_int4(res[4], res[5], res[6], res[7]);
                stored = true;
            }
        } else if constexpr (V == 4) {
            if (full) {
                *reinterpret_cast<int4 *>(out + p0) = make_int4(res[0], res[1], res[2], res[3]);
                stored = true;
            }
        } else if constexpr (V == 2) {
            if (full) {
                *reinterpret_cast<int2 *>(out + p0) = make_int2(res[0], res[1]);
                stored = true;
            }
        }
        if (!stored) {
#pragma unroll
            for (int v = 0; v < V; v++)
                if (p0 + v < N) out[p0 + v] = res[v];
        }
    }
}

// ---- 17 to 64 bands ------------------------------------------------------------------------------
// The same fast pass and exact recheck with the band count known at run time, up to NBMAX (32 or
// 64).  All k centres no longer fit in shared memory as float32 rows next to their float64 copies
// (k (12 nB + 12) bytes: 780 KB at 64 bands and k = 1024), so the float32 rows {-2c} come in tiles
// of ASSIGN_TILE centres and every pixel carries its best and second-best value from tile to tile.
// Rows are padded with zeros to a multiple of four bands (x is padded with zeros too: the padding
// adds exact zeros to the chain).  The exact pass reads the float64 centres from global memory
// (L2) and the pixel's integers from the image, so it needs no per-band array of its own.
constexpr int ASSIGN_TILE = 128;

// exact pass with nB known at run time: the operation sequence of assign_exact
template <typename T>
__device__ __noinline__ int assign_exact_rt(const T *__restrict__ img, int64_t N, int64_t p, int nB,
                                            const double *__restrict__ cd, const double *cn, int k)
{
    int best = 0;
    double bestD = 0.0;
    for (int j = 0; j < k; j++) {
        double dot = 0.0;
        for (int b = 0; b < nB; b++)
            dot = __dadd_rn(dot, __dmul_rn((double)__ldg(img + (size_t)b * N + p), __ldg(cd + (size_t)j * nB + b)));
        double d = __dadd_rn(cn[j], __dmul_rn(-2.0, dot));
        if (j == 0 || d < bestD) { bestD = d; best = j; }
    }
    return best;
}

template <typename T, int NBMAX, int V>
__global__ void __launch_bounds__(256)
k_assign_many(const T *__restrict__ img, int64_t N, int nB, const double *__restrict__ centres, int k,
              int hasNull, double nullVal, AssignBounds bnd, int32_t *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smemRaw[];
    const int nBP = (nB + 3) & ~3;                               // padded row length
    // (each array starts on 16 bytes: the rows of cf are read as float4)
    double *cn = reinterpret_cast<double *>(smemRaw);            // k float64 ||c||^2
    float *cnf = reinterpret_cast<float *>(cn + ((k + 1) & ~1)); // k float32 ||c||^2
    float *cf = cnf + ((k + 3) & ~3);                            // ASSIGN_TILE x nBP float32 -2c

    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        double s = 0.0;
        for (int b = 0; b < nB; b++) {
            const double c = centres[(size_t)j * nB + b];
            s = __dadd_rn(s, __dmul_rn(c, c));
        }
        cn[j] = s;
        cnf[j] = (float)s;
    }
    const int nTiles = (k + ASSIGN_TILE - 1) / ASSIGN_TILE;
    auto loadTile = [&](int t) {
        const int j0 = t * ASSIGN_TILE;
        const int kt = min(ASSIGN_TILE, k - j0);
        for (int i = threadIdx.x; i < kt * nBP; i += blockDim.x) {
            const int j = i / nBP, b = i % nBP;
            cf[i] = b < nB ? (float)(-2.0 * centres[(size_t)(j0 + j) * nB + b]) : 0.0f;
        }
    };
    if (nTiles == 1) loadTile(0);          // (then the tile stays for every pixel of the block)
    __syncthreads();

    // the pixel loop runs the same number of times in every thread of the block: the tiles are
    // loaded between barriers
    const int64_t perIter = (int64_t)blockDim.x * V;
    for (int64_t base = (int64_t)blockIdx.x * perIter; base < N; base += (int64_t)gridDim.x * perIter) {
        const int64_t p0 = base + (int64_t)threadIdx.x * V;
        float x[V][NBMAX];
#pragma unroll
        for (int b = 0; b < NBMAX; b++) {
#pragma unroll
            for (int v = 0; v < V; v++)
                x[v][b] = (b < nB && p0 + v < N) ? (float)__ldg(img + (size_t)b * N + p0 + v) : 0.0f;
        }
        float best[V], second[V];
        int idx[V];
#pragma unroll
        for (int v = 0; v < V; v++) { best[v] = 3.0e38f; second[v] = 3.0e38f; idx[v] = 0; }

        for (int t = 0; t < nTiles; t++) {
            const int j0 = t * ASSIGN_TILE;
            const int kt = min(ASSIGN_TILE, k - j0);
            if (nTiles > 1) {
                __syncthreads();
                loadTile(t);
                __syncthreads();
            }
            for (int jj = 0; jj < kt; jj++) {
                const float4 *row = reinterpret_cast<const float4 *>(cf + jj * nBP);
                float acc[V];
#pragma unroll
                for (int v = 0; v < V; v++) acc[v] = cnf[j0 + jj];
#pragma unroll
                for (int q = 0; q < NBMAX / 4; q++) {
                    if (4 * q >= nBP) break;       // (uniform: nB is the same for every thread)
                    const float4 c = row[q];
#pragma unroll
                    for (int v = 0; v < V; v++) {
                        acc[v] = fmaf(x[v][4 * q], c.x, acc[v]);
                        acc[v] = fmaf(x[v][4 * q + 1], c.y, acc[v]);
                        acc[v] = fmaf(x[v][4 * q + 2], c.z, acc[v]);
                        acc[v] = fmaf(x[v][4 * q + 3], c.w, acc[v]);
                    }
                }
#pragma unroll
                for (int v = 0; v < V; v++) {
                    second[v] = fminf(second[v], fmaxf(acc[v], best[v]));
                    const bool lt = acc[v] < best[v];
                    best[v] = fminf(acc[v], best[v]);
                    idx[v] = lt ? j0 + jj : idx[v];
                }
            }
        }

#pragma unroll
        for (int v = 0; v < V; v++) {
            const int64_t p = p0 + v;
            if (p >= N) continue;
            const float gap = second[v] - best[v];
            float absSum = 0.0f;
#pragma unroll
            for (int b = 0; b < NBMAX; b++) absSum += fabsf(x[v][b]);
            const float tol = fmaf(bnd.perAbsX, absSum, bnd.constant);
            int lab = idx[v];
            if (k > 1 && !(gap > tol)) lab = assign_exact_rt<T>(img, N, p, nB, centres, cn, k);
            bool isNull = false;
            if (hasNull) {
                // rounding to float32 is monotonic, so x == nullVal implies (float)x == (float)nullVal;
                // the integer itself decides
#pragma unroll
                for (int b = 0; b < NBMAX; b++) isNull |= (b < nB && x[v][b] == (float)nullVal);
                if (isNull) {
                    isNull = false;
                    for (int b = 0; b < nB; b++) isNull |= ((double)__ldg(img + (size_t)b * N + p) == nullVal);
                }
            }
            out[p] = isNull ? 0 : lab + 1;
        }
    }
}

template <typename T, int NBMAX>
static int launch_assign_many(ssg_ctx *ctx, const void *img, int nB, int64_t N, const double *centresDev, int k,
                              int hasNull, double nullVal, AssignBounds bnd, int32_t *out)
{
    constexpr int V = NBMAX <= 32 ? 4 : 2;       // x[][] is V * NBMAX registers
    const int nBP = (nB + 3) & ~3;
    const int kt = k < ASSIGN_TILE ? k : ASSIGN_TILE;
    const size_t smem = (size_t)((k + 1) & ~1) * sizeof(double) + (size_t)((k + 3) & ~3) * sizeof(float) +
                        (size_t)kt * nBP * sizeof(float);
    auto kern = k_assign_many<T, NBMAX, V>;
    if (smem > 48 * 1024)
        SSG_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t blocks = (N + 256 * V - 1) / (256 * V);
    const int64_t cap = (int64_t)ctx->numSMs * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    SSG_PROF_BEGIN(ctx, "k_assign_many");
    kern<<<(unsigned)blocks, 256, smem, ctx->stream>>>(reinterpret_cast<const T *>(img), N, nB, centresDev, k,
                                                       hasNull, nullVal, bnd, out);
    SSG_LAUNCHED(ctx);
    return SSG_OK;
}

// ---- pruned assignment for few bands ---------------------------------------------------------
// With up to four bands the band space is cut into a grid of boxes (power-of-two widths over the
// range the centres span, one outer box on either side out to the limits of the data type) and
// every box knows which centres can be nearest to ANY integer point inside it:
//     U = min_j maxdist^2(box, c_j)   is an upper bound of the best distance of every such point,
//     centre j stays  <=>  mindist^2(box, c_j) <= U (+ a float64 rounding margin),
// since a centre farther than U from the whole box is strictly farther than the best one from
// every point of it (ties are within the margin and stay).  A pixel then evaluates only the
// centres of its box -- a few instead of all k -- in ascending j with the same float32 fast pass
// and guarded float64 recheck as the full scan, so the label is still the float64 first-minimum
// argmin over all k centres.  The table is a 64-bit mask per box (k <= 64), built on the device
// when the centres change and kept in the context.

__global__ void __launch_bounds__(256)
k_grid_build(const double *__restrict__ centres, int k, GridGeom g, unsigned long long *__restrict__ grid, int64_t nCells)
{
    extern __shared__ double sc[];      // k * nB
    for (int i = threadIdx.x; i < k * g.nB; i += blockDim.x) sc[i] = centres[i];
    __syncthreads();
    const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= nCells) return;
    double lo[4], hi[4];
    int64_t rest = cell;
    bool empty = false;
    for (int b = g.nB - 1; b >= 0; b--) {
        const int qb = (int)(rest % g.q[b]);
        rest /= g.q[b];
        const long long w = 1ll << g.shift[b];
        long long a = qb == 0 ? (long long)g.tmin : (long long)g.base[b] + qb * w;
        long long z = qb == g.q[b] - 1 ? (long long)g.tmax : (long long)g.base[b] + (qb + 1) * w - 1;
        if (a < g.tmin) a = g.tmin;
        if (z > g.tmax) z = g.tmax;
        empty |= a > z;
        lo[b] = (double)a;
        hi[b] = (double)z;
    }
    if (empty) { grid[cell] = 0ull; return; }
    double U = 1e300;
    for (int j = 0; j < k; j++) {
        double far2 = 0.0;
        for (int b = 0; b < g.nB; b++) {
            const double c = sc[j * g.nB + b];
            const double d0 = c - lo[b], d1 = hi[b] - c;
            const double d = fmax(fabs(d0), fabs(d1));
            far2 += d * d;
        }
        U = fmin(U, far2);
    }
    const double limit = U * (1.0 + 1e-9) + 1e-6;
    unsigned long long mask = 0ull;
    for (int j = 0; j < k; j++) {
        double near2 = 0.0;
        for (int b = 0; b < g.nB; b++) {
            const double c = sc[j * g.nB + b];
            const double d = c < lo[b] ? lo[b] - c : (c > hi[b] ? c - hi[b] : 0.0);
            near2 += d * d;
        }
        if (near2 <= limit) mask |= 1ull << j;
    }
    grid[cell] = mask;
}

template <typename T, int V>
__device__ __forceinline__ void load_raw(const T *p, int (&x)[V])
{
    constexpr int BYTES = V * (int)sizeof(T);
    if constexpr (BYTES == 8) {
        const uint2 r = __ldg(reinterpret_cast<const uint2 *>(p));
        const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
        for (int i = 0; i < V; i++) x[i] = (int)e[i];
    } else {
        const unsigned r = __ldg(reinterpret_cast<const unsigned *>(p));
        const T *e = reinterpret_cast<const T *>(&r);
#pragma unroll
        for (int i = 0; i < V; i++) x[i] = (int)e[i];
    }
}

// pixels per thread of k_assign_grid: 4 leaves room for twice the warps of 8 (the loop waits on
// shared memory)
constexpr int GRID_V = 4;

template <typename T, int NB>
__global__ void __launch_bounds__(256)
k_assign_grid(const T *__restrict__ img, int64_t N, const double *__restrict__ centres, int k,
              int hasNull, double nullVal, AssignBounds bnd, GridGeom g,
              const unsigned long long *__restrict__ grid, int32_t *__restrict__ out)
{
    // rows of NB+1 floats {||c||^2, -2c}: an odd stride, so lanes that look at different centres
    // hit different banks (lanes that look at the same one are a broadcast)
    constexpr int CS = NB + 1 + ((NB + 1) % 2 == 0 ? 1 : 0);
    constexpr int V = GRID_V;
    extern __shared__ __align__(16) unsigned char smemRaw[];
    double *cd = reinterpret_cast<double *>(smemRaw);          // k*NB
    double *cn = cd + (size_t)k * NB;                          // k
    float *cf = reinterpret_cast<float *>(cn + k);             // k x CS
    for (int i = threadIdx.x; i < k * NB; i += blockDim.x) cd[i] = centres[i];
    __syncthreads();
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        double s = 0.0;
#pragma unroll
        for (int b = 0; b < NB; b++) {
            s = __dadd_rn(s, __dmul_rn(cd[j * NB + b], cd[j * NB + b]));
            cf[j * CS + 1 + b] = (float)(-2.0 * cd[j * NB + b]);
        }
        cn[j] = s;
        cf[j * CS] = (float)s;
    }
    __syncthreads();

    const int64_t nGroups = N / V;        // (the launcher takes this path only when N is a multiple of V)
    for (int64_t gi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; gi < nGroups; gi += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p0 = gi * V;
        float x[V][NB];
        int cellOf[V];
#pragma unroll
        for (int v = 0; v < V; v++) cellOf[v] = 0;
#pragma unroll
        for (int b = 0; b < NB; b++) {
            int t[V];
            load_raw<T, V>(img + (size_t)b * N + p0, t);
#pragma unroll
            for (int v = 0; v < V; v++) {
                x[v][b] = (float)t[v];
                int qb = (t[v] - g.base[b]) >> g.shift[b];
                qb = min(max(qb, 0), g.q[b] - 1);
                cellOf[v] = cellOf[v] * g.q[b] + qb;
            }
        }
        // the centres that can be nearest to any of my V (adjacent, hence similar) pixels: evaluating
        // a centre for a pixel whose box does not list it costs a little and changes nothing
        unsigned long long M = 0ull;
#pragma unroll
        for (int v = 0; v < V; v++) M |= __ldg(grid + cellOf[v]);

        float best[V], second[V];
        int idx[V];
#pragma unroll
        for (int v = 0; v < V; v++) { best[v] = 3.0e38f; second[v] = 3.0e38f; idx[v] = 0; }
#pragma unroll
        for (int half = 0; half < 2; half++) {
            unsigned m = half == 0 ? (unsigned)M : (unsigned)(M >> 32);
            while (m) {
                const int j = (__ffs(m) - 1) + 32 * half;
                m &= m - 1;
                float c[NB + 1];
#pragma unroll
                for (int b = 0; b <= NB; b++) c[b] = cf[j * CS + b];
#pragma unroll
                for (int v = 0; v < V; v++) {
                    float acc = c[0];
#pragma unroll
                    for (int b = 0; b < NB; b++) acc = fmaf(x[v][b], c[b + 1], acc);
                    second[v] = fminf(second[v], fmaxf(acc, best[v]));
                    const bool lt = acc < best[v];
                    best[v] = fminf(acc, best[v]);
                    idx[v] = lt ? j : idx[v];
                }
            }
        }
        int32_t res[V];
#pragma unroll
        for (int v = 0; v < V; v++) {
            const float gap = second[v] - best[v];
            float absSum = 0.0f;
#pragma unroll
            for (int b = 0; b < NB; b++) absSum += fabsf(x[v][b]);
            const float tol = fmaf(bnd.perAbsX, absSum, bnd.constant);
            int lab = idx[v];
            if (!(gap > tol)) {
                float xv[NB];
#pragma unroll
                for (int b = 0; b < NB; b++) xv[b] = x[v][b];
                lab = assign_exact<NB>(xv, cd, cn, k);
            }
            bool isNull = false;
            if (hasNull) {
#pragma unroll
                for (int b = 0; b < NB; b++) isNull |= ((double)x[v][b] == nullVal);
            }
            res[v] = isNull ? 0 : lab + 1;
        }
        *reinterpret_cast<int4 *>(out + p0) = make_int4(res[0], res[1], res[2], res[3]);
    }
}

template <typename T, int NB, int V>
static int launch_assign(ssg_ctx *ctx, const void *img, int64_t N, const double *centresDev, int k,
                         int hasNull, double nullVal, AssignBounds bnd, int32_t *out)
{
    size_t smem = (size_t)k * NB * sizeof(double) + (size_t)k * sizeof(double) + (size_t)k * (NB + 1) * sizeof(float);
    auto kern = k_assign<T, NB, V>;
    if (smem > 48 * 1024)
        SSG_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t nGroups = (N + V - 1) / V;
    int64_t blocks = (nGroups + 255) / 256;
    // a few resident waves, grid-stride beyond: every block first builds the centre tables in
    // shared memory (float64 norms, two barriers), which with one block per 2048 pixels was a
    // tenth of the kernel (ncu: barrier stalls)
    int64_t cap = (int64_t)ctx->numSMs * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    SSG_PROF_BEGIN(ctx, "k_assign");
    kern<<<(unsigned)blocks, 256, smem, ctx->stream>>>(reinterpret_cast<const T *>(img), N, centresDev,
                                                      k, hasNull, nullVal, bnd, out);
    SSG_LAUNCHED(ctx);
    return SSG_OK;
}

template <typename T, int NB>
static int dispatch_v(ssg_ctx *ctx, const void *img, int64_t N, const double *centresDev, int k,
                      int hasNull, double nullVal, AssignBounds bnd, int32_t *out)
{
    // widest load the alignment of every band plane allows (at most 16 bytes per band)
    constexpr int VMAX = sizeof(T) == 4 ? (NB <= 8 ? 4 : 2) : (NB <= 4 ? 8 : (NB <= 8 ? 4 : 2));
    const size_t planeBytes = (size_t)N * sizeof(T);
    const bool aligned = ((uintptr_t)img % 16 == 0) && ((uintptr_t)out % 16 == 0) &&
                         (planeBytes % (VMAX * sizeof(T)) == 0);
    if (aligned) return launch_assign<T, NB, VMAX>(ctx, img, N, centresDev, k, hasNull, nullVal, bnd, out);
    return launch_assign<T, NB, 1>(ctx, img, N, centresDev, k, hasNull, nullVal, bnd, out);
}

template <typename T>
static int dispatch_nb(ssg_ctx *ctx, const void *img, int nBands, int64_t N, const double *c, int k,
                       int hasNull, double nullVal, AssignBounds bnd, int32_t *out)
{
    switch (nBands) {
#define CASE(NB) case NB: return dispatch_v<T, NB>(ctx, img, N, c, k, hasNull, nullVal, bnd, out);
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
        CASE(9) CASE(10) CASE(11) CASE(12) CASE(13) CASE(14) CASE(15) CASE(16)
#undef CASE
    default:
        if (nBands >= 17 && nBands <= 32) return launch_assign_many<T, 32>(ctx, img, nBands, N, c, k, hasNull, nullVal, bnd, out);
        if (nBands >= 33 && nBands <= SSG_MAX_BANDS) return launch_assign_many<T, 64>(ctx, img, nBands, N, c, k, hasNull, nullVal, bnd, out);
        SSG_FAIL(ctx, SSG_ERR_ARG, "nBands=%d not in 1..%d", nBands, SSG_MAX_BANDS);
    }
}

int ssgk_assign(ssg_ctx *ctx, const void *imgDev, int dtype, int nBands, int64_t N,
                const double *centresHost, int k, int hasNull, double nullVal, int32_t *outDev)
{
    if (N == 0) return SSG_OK;
    if (k < 1 || k > SSG_MAX_CLUSTERS) SSG_FAIL(ctx, SSG_ERR_ARG, "k=%d not in 1..%d", k, SSG_MAX_CLUSTERS);
    const size_t nc = (size_t)k * nBands;
    SSG_TRY(ssg_reserve(ctx, ctx->centres, nc * sizeof(double)));
    // the caller's centre array may be reused as soon as we return: stage through a copy
    // that lives until the stream has consumed it
    ctx->centresStage.assign(centresHost, centresHost + nc);
    SSG_CUDA(ctx, cudaMemcpyAsync(ctx->centres.p, ctx->centresStage.data(), nc * sizeof(double),
                                  cudaMemcpyHostToDevice, ctx->stream));
    const double *centresDev = bufp<double>(ctx->centres);
    double cmax = 0.0, cnmax = 0.0;
    for (int j = 0; j < k; j++) {
        double n2 = 0.0;
        for (int b = 0; b < nBands; b++) {
            const double a = fabs(centresHost[(size_t)j * nBands + b]);
            if (a > cmax) cmax = a;
            n2 += a * a;
        }
        if (n2 > cnmax) cnmax = n2;
    }
    const double xmax = dtype == SSG_U8 ? 255.0 : dtype == SSG_U16 ? 65535.0 : dtype == SSG_I16 ? 32768.0 :
                        dtype == SSG_U32 ? 4294967295.0 : 2147483648.0;
    const size_t itemSize = dtypeSize(dtype);
    const double u = ldexp(1.0, -24);
    // 2E of the fast pass (see the header) + what float64 itself can be off by in the reference
    const double e32 = 2.0 * (nBands + 1) * 1.01 * u;
    const double margin64 = ldexp(1.0, -50) * (nBands + 2) * (cnmax + 2.0 * nBands * xmax * cmax) + 1e-30;
    // 32-bit values are rounded to float32 on load (|x_f - x| <= u |x|), which moves the difference of
    // two values by up to 2 u |x|.|c_i - c_j| <= 4 u max|c| sum_b |x_b| more
    const double xRound = itemSize == 4 ? 4.0 * u * cmax * 1.01 : 0.0;
    AssignBounds bnd;
    bnd.perAbsX = (float)((e32 * 2.0 * cmax + xRound) * 1.001);
    bnd.constant = (float)((e32 * cnmax + margin64) * 1.001);
    // few bands, at most 64 centres, wide loads possible, 8/16-bit values: the pruned kernel
    const bool gridOff = getenv("SSG_ASSIGN_GRID") && atoi(getenv("SSG_ASSIGN_GRID")) == 0;
    if (!gridOff && itemSize <= 2 && nBands <= 4 && k >= 2 && k <= 64 && N % 8 == 0 && ((uintptr_t)imgDev % 16 == 0) &&
        ((uintptr_t)outDev % 16 == 0) && ((size_t)N * itemSize) % 16 == 0) {
        const int tmin = dtype == SSG_I16 ? -32768 : 0;
        const int tmax = dtype == SSG_U8 ? 255 : (dtype == SSG_U16 ? 65535 : 32767);
        const bool same = ctx->gridDtype == dtype && ctx->gridK == k && ctx->gridGeom.nB == nBands &&
                          ctx->gridCentres.size() == nc && memcmp(ctx->gridCentres.data(), centresHost, nc * sizeof(double)) == 0;
        static const int cellsPerBand[5] = {0, 4096, 512, 64, 32};
        if (!same) {
            GridGeom g = {};
            g.nB = nBands;
            g.tmin = tmin; g.tmax = tmax;
            int64_t nCells = 1;
            for (int b = 0; b < nBands; b++) {
                double lo = centresHost[b], hi = centresHost[b];
                for (int j = 1; j < k; j++) {
                    const double c = centresHost[(size_t)j * nBands + b];
                    if (c < lo) lo = c;
                    if (c > hi) hi = c;
                }
                // The fine boxes should cover the DATA, which reaches beyond the outermost centres by
                // about a cluster radius: the range of the centres widened by 40 % on either side
                // (pixels beyond that land in the two outer boxes, which reach to the limits of the
                // data type and list many centres: correct, just slower).  Centres outside the data
                // type's range cannot make the grid wider than the data.
                const double widen = 0.4 * (hi - lo);
                lo -= widen;
                hi += widen;
                long long cmin = (long long)floor(lo < tmin ? (double)tmin : (lo > tmax ? (double)tmax : lo));
                long long cmax = (long long)ceil(hi > tmax ? (double)tmax : (hi < tmin ? (double)tmin : hi));
                const int q = cellsPerBand[nBands];
                int shift = 0;
                while (((long long)(q - 2) << shift) < cmax - cmin + 1) shift++;
                g.q[b] = q;
                g.shift[b] = shift;
                g.base[b] = (int)(cmin - (1ll << shift));
                nCells *= q;
            }
            SSG_TRY(ssg_reserve(ctx, ctx->assignGrid, (size_t)nCells * sizeof(unsigned long long)));
            SSG_PROF_BEGIN(ctx, "k_grid_build");
            k_grid_build<<<gridFor(nCells, 256), 256, nc * sizeof(double), ctx->stream>>>(centresDev, k, g,
                bufp<unsigned long long>(ctx->assignGrid), nCells);
            SSG_LAUNCHED(ctx);
            ctx->gridGeom = g;
            ctx->gridDtype = dtype;
            ctx->gridK = k;
            ctx->gridCentres.assign(centresHost, centresHost + nc);
        }
        const GridGeom g = ctx->gridGeom;
        const size_t smem = nc * sizeof(double) + (size_t)k * sizeof(double) + (size_t)k * 6 * sizeof(float);
        int64_t blocks = (N / GRID_V + 255) / 256;
        if (blocks > (int64_t)ctx->numSMs * 16) blocks = (int64_t)ctx->numSMs * 16;
        const unsigned long long *grid = bufp<unsigned long long>(ctx->assignGrid);
        SSG_PROF_BEGIN(ctx, "k_assign_grid");
#define GRID_CASE(T, NB)                                                                                   \
        k_assign_grid<T, NB><<<(unsigned)blocks, 256, smem, ctx->stream>>>(reinterpret_cast<const T *>(imgDev), N, \
            centresDev, k, hasNull, nullVal, bnd, g, grid, outDev)
#define GRID_NB(T)                                                           \
        switch (nBands) {                                                    \
        case 1: GRID_CASE(T, 1); break;                                      \
        case 2: GRID_CASE(T, 2); break;                                      \
        case 3: GRID_CASE(T, 3); break;                                      \
        default: GRID_CASE(T, 4); break;                                     \
        }
        if (dtype == SSG_U8) { GRID_NB(uint8_t) }
        else if (dtype == SSG_U16) { GRID_NB(uint16_t) }
        else { GRID_NB(int16_t) }
#undef GRID_NB
#undef GRID_CASE
        SSG_LAUNCHED(ctx);
        return SSG_OK;
    }
    switch (dtype) {
    case SSG_U8: return dispatch_nb<uint8_t>(ctx, imgDev, nBands, N, centresDev, k, hasNull, nullVal, bnd, outDev);
    case SSG_U16: return dispatch_nb<uint16_t>(ctx, imgDev, nBands, N, centresDev, k, hasNull, nullVal, bnd, outDev);
    case SSG_I16: return dispatch_nb<int16_t>(ctx, imgDev, nBands, N, centresDev, k, hasNull, nullVal, bnd, outDev);
    case SSG_U32: return dispatch_nb<uint32_t>(ctx, imgDev, nBands, N, centresDev, k, hasNull, nullVal, bnd, outDev);
    case SSG_I32: return dispatch_nb<int32_t>(ctx, imgDev, nBands, N, centresDev, k, hasNull, nullVal, bnd, outDev);
    default: SSG_FAIL(ctx, SSG_ERR_ARG, "unsupported dtype code %d", dtype);
    }
}
