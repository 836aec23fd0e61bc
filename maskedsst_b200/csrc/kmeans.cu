// k-means clustering of embeddings (msst_kmeans_*, include/msst.h): Lloyd's algorithm with k-means++ seeding on fp32 rows, all
// restarts of a fit in the same launches.  FP32 FFMA distances in the direct difference form, fp64 sums in a fixed order.
//
//   kmeans_assign_kernel     CTA = (4096-row slice, restart), 256 threads.  The restart's K centroids are staged once into shared
//                            memory [K][dim + 4]; the slice is walked in 32-row tiles, each row loaded (and normalised) by one warp
//                            into shared memory [32][dim + 4].  Distances: thread = 1 row x 4 clusters (cl + 8j) per chunk of 32
//                            clusters, float4 reads along dim, sum_d (y_d - c_d)^2 in ascending d; the (distance, index) minimum
//                            is taken lexicographically within the thread, over the 8 lanes of the row and over the chunks, so the
//                            lowest index wins a tie.  With a workspace: thread = feature adds the tile's rows in ascending order
//                            into the per-cluster fp64 sums in shared memory [K][dim]; thread 0 counts, sums the minima (fp64) and
//                            counts changed labels.  The slice's partials go to the workspace (sums rounded to fp32 once).
//   kmeans_update_kernel     CTA = (restart, cluster), thread = feature: the slices' sums and counts added in ascending slice order
//                            (fp64), centroid = sum / count, an empty cluster keeps its centroid.  The CTA of cluster 0 also writes
//                            the restart's inertia, changed count and number of empty clusters.
//   kmeans_seed_pick_kernel  CTA = restart: one k-means++ choice from the fp64 slice sums of mindist (one thread scans the slices,
//                            then the rows of the chosen slice, in ascending order), the chosen row copied into the centroids.
//   kmeans_seed_dist_kernel  CTA = (slice, restart), warp = row: mindist = min(mindist, d(y, c_j)) and the slice's fp64 sum of it.
//
// No float atomics: a restart's results depend only on x, its own u row or centroids and the dims, never on the other restarts, the
// grid or the SM count, and a row's label / distance does not depend on the rows it was launched with.
#include "common.cuh"

namespace msst {

constexpr int KM_SLICE = 4096;               // rows of a slice (fixed: the partials and their order never depend on the launch)
constexpr int KM_TR = 32;                    // rows of a tile
constexpr int KM_CH = 32;                    // clusters per register pass (8 lanes x 4)
constexpr int KM_THREADS = 256;
constexpr int KM_MAX_DIM = 256, KM_MAX_K = 256;
constexpr int KM_SMEM_MAX = 227 * 1024;
static_assert(KM_THREADS >= KM_MAX_DIM, "thread = feature in the sums");

// [fp64 sums K*dim (with a workspace)] [centroids K][dim + 4] [rows 32][dim + 4] [counts K] [label, min distance, changed of 32 rows]
// dim + 4 keeps the row stride at 16 bytes mod 128: conflict-free float4 reads.  At the K*dim cap (K = 64, dim = 256) 226 KB.
static size_t km_assign_smem(int dim, int k, bool with_sums) {
    return (with_sums ? (size_t)k * dim * 8 : 0) + (size_t)(k + KM_TR) * (dim + 4) * 4 + (size_t)k * 4 + (size_t)KM_TR * 4 * 3;
}

struct KmSmem {
    double* sums;
    float *cent, *xs, *dmin;
    int *cnt, *lab, *chg;
    int ld;
    __device__ KmSmem(unsigned char* p, int k, int dim, bool with_sums) {
        ld = dim + 4;
        sums = reinterpret_cast<double*>(p);
        cent = reinterpret_cast<float*>(p + (with_sums ? (size_t)k * dim * 8 : 0));
        xs = cent + k * ld;
        cnt = reinterpret_cast<int*>(xs + KM_TR * ld);
        lab = cnt + k; dmin = reinterpret_cast<float*>(lab + KM_TR); chg = reinterpret_cast<int*>(dmin + KM_TR);
    }
};

// The workspace: per (restart, slice) the fp64 inertia (seeding: the slice sum of mindist), the per-cluster fp32 sums [K][dim] and
// int32 counts [K], and the int32 changed count.  S = number of slices.
struct KmWs {
    double* inertia;   // [R][S]
    float* sums;       // [R][S][K][dim]
    int* counts;       // [R][S][K]
    int* changed;      // [R][S]
};

static KmWs km_ws(void* base, int R, int64_t S, int k, int dim) {
    KmWs w;
    w.inertia = static_cast<double*>(base);
    w.sums = reinterpret_cast<float*>(w.inertia + R * S);
    w.counts = reinterpret_cast<int*>(w.sums + R * S * k * dim);
    w.changed = w.counts + R * S * k;
    return w;
}

static int64_t km_slices(int64_t n) { return ceil_div(n, KM_SLICE); }

// row xr (nullptr: zeros) into v (element lane + 32i), as F.normalize(x, dim=1, eps=1e-12) when normalize: x / max(||x||, 1e-12).
// The one row staging of every kernel here, so assignment, seeding and the copied centroids see the same bits.
__device__ __forceinline__ void km_row(const float* __restrict__ xr, int dim, int lane, int normalize, float (&v)[KM_MAX_DIM / 32]) {
#pragma unroll
    for (int i = 0; i < KM_MAX_DIM / 32; ++i) {
        const int c = lane + 32 * i;
        v[i] = (xr != nullptr && c < dim) ? xr[c] : 0.f;
    }
    if (normalize) {
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < KM_MAX_DIM / 32; ++i) sq = fmaf(v[i], v[i], sq);
        const float den = fmaxf(sqrtf(warp_sum(sq)), 1e-12f);
#pragma unroll
        for (int i = 0; i < KM_MAX_DIM / 32; ++i) v[i] = __fdiv_rn(v[i], den);
    }
}

// (d2, i2) before (d1, i1): smaller distance, then lower index
__device__ __forceinline__ bool km_before(float d2, int i2, float d1, int i1) { return d2 < d1 || (d2 == d1 && i2 < i1); }

__global__ void __launch_bounds__(KM_THREADS) kmeans_assign_kernel(const msst_kmeans_dims d, int64_t slices, const float* __restrict__ x,
                                                                   const float* __restrict__ centroids, int64_t* __restrict__ labels,
                                                                   float* __restrict__ dist, const KmWs ws, bool with_ws) {
    extern __shared__ float4 km_smem_raw[];
    const int R = d.restarts, K = d.k, dim = d.dim, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r = (int)(blockIdx.x % R);                 // restarts of a slice are neighbours in the grid: they share its rows in L2
    const int64_t slice = blockIdx.x / R;
    const KmSmem s(reinterpret_cast<unsigned char*>(km_smem_raw), K, dim, with_ws);
    const float* C = centroids + (int64_t)r * K * dim;
    for (int i = tid; i < K * dim; i += KM_THREADS) {
        const int k = i / dim;
        s.cent[k * s.ld + i - k * dim] = C[i];
    }
    if (with_ws) {
        for (int i = tid; i < K * dim; i += KM_THREADS) s.sums[i] = 0.0;
        for (int i = tid; i < K; i += KM_THREADS) s.cnt[i] = 0;
    }
    const int64_t first = slice * KM_SLICE;
    const int rows = (int)min((int64_t)KM_SLICE, d.n - first);
    int64_t* lab_r = labels + (int64_t)r * d.n;
    float* dist_r = dist ? dist + (int64_t)r * d.n : nullptr;
    double inertia = 0.0;                                  // thread 0
    int changed = 0;
    const int cl = tid & 7, rw = tid >> 3;
    for (int t0 = 0; t0 < rows; t0 += KM_TR) {
        const int cnt = min(KM_TR, rows - t0);
        __syncthreads();                                   // centroids staged / the previous tile's rows consumed
#pragma unroll
        for (int q = 0; q < KM_TR / 8; ++q) {
            const int rr = warp + 8 * q;
            float v[KM_MAX_DIM / 32];
            km_row(rr < cnt ? x + (first + t0 + rr) * dim : nullptr, dim, lane, d.normalize, v);
#pragma unroll
            for (int i = 0; i < KM_MAX_DIM / 32; ++i)
                if (lane + 32 * i < dim) s.xs[rr * s.ld + lane + 32 * i] = v[i];
        }
        __syncthreads();
        float bd = INFINITY;
        int bi = 0x7fffffff;
        const float* z = s.xs + rw * s.ld;
        for (int c0 = 0; c0 < K; c0 += KM_CH) {
            const float* w[4];
            bool ok[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int k = c0 + cl + 8 * j;
                ok[j] = k < K;
                w[j] = s.cent + (ok[j] ? k : 0) * s.ld;
            }
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int c = 0; c < dim; c += 4) {
                const float4 zz = *reinterpret_cast<const float4*>(z + c);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 ww = *reinterpret_cast<const float4*>(w[j] + c);
                    float e;
                    e = __fsub_rn(zz.x, ww.x); acc[j] = fmaf(e, e, acc[j]);
                    e = __fsub_rn(zz.y, ww.y); acc[j] = fmaf(e, e, acc[j]);
                    e = __fsub_rn(zz.z, ww.z); acc[j] = fmaf(e, e, acc[j]);
                    e = __fsub_rn(zz.w, ww.w); acc[j] = fmaf(e, e, acc[j]);
                }
            }
            float cd = INFINITY;
            int ci = 0x7fffffff;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (ok[j] && km_before(acc[j], c0 + cl + 8 * j, cd, ci)) { cd = acc[j]; ci = c0 + cl + 8 * j; }
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {               // the row's 8 lanes
                const float od = __shfl_xor_sync(0xffffffffu, cd, o);
                const int oi = __shfl_xor_sync(0xffffffffu, ci, o);
                if (km_before(od, oi, cd, ci)) { cd = od; ci = oi; }
            }
            if (km_before(cd, ci, bd, bi)) { bd = cd; bi = ci; }
        }
        if (bi == 0x7fffffff) bi = 0;                       // every distance NaN
        if (cl == 0 && rw < cnt) {
            const int64_t i = first + t0 + rw;
            int ch = 0;
            if (with_ws) ch = lab_r[i] != bi;
            lab_r[i] = bi;
            if (dist_r) dist_r[i] = bd;
            s.lab[rw] = bi; s.dmin[rw] = bd; s.chg[rw] = ch;
        }
        __syncthreads();
        if (with_ws) {
            if (tid < dim)                                  // thread = feature, rows in ascending order
                for (int rr = 0; rr < cnt; ++rr) {
                    double* a = s.sums + s.lab[rr] * dim + tid;
                    *a = __dadd_rn(*a, (double)s.xs[rr * s.ld + tid]);
                }
            if (tid == 0)
                for (int rr = 0; rr < cnt; ++rr) {
                    ++s.cnt[s.lab[rr]];
                    inertia = __dadd_rn(inertia, (double)s.dmin[rr]);
                    changed += s.chg[rr];
                }
        }
    }
    if (!with_ws) return;
    __syncthreads();
    const int64_t p = (int64_t)r * slices + slice;
    float* so = ws.sums + p * K * dim;
    for (int i = tid; i < K * dim; i += KM_THREADS) so[i] = __double2float_rn(s.sums[i]);
    for (int i = tid; i < K; i += KM_THREADS) ws.counts[p * K + i] = s.cnt[i];
    if (tid == 0) { ws.inertia[p] = inertia; ws.changed[p] = changed; }
}

__device__ __forceinline__ int km_warp_isum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// blockDim.x = dim
__global__ void kmeans_update_kernel(const msst_kmeans_dims d, int64_t slices, const KmWs ws, float* __restrict__ centroids,
                                     double* __restrict__ inertia, int* __restrict__ changed, int* __restrict__ empty) {
    __shared__ int total, n_empty;
    const int K = d.k, dim = d.dim, tid = threadIdx.x;
    const int r = blockIdx.x / K, k = blockIdx.x % K;
    if (tid < 32) {                                         // integer count: any order gives the same value
        int c = 0;
        for (int64_t s = tid; s < slices; s += 32) c += ws.counts[((int64_t)r * slices + s) * K + k];
        c = km_warp_isum(c);
        if (tid == 0) { total = c; n_empty = 0; }
    }
    __syncthreads();
    double acc = 0.0;
    const float* src = ws.sums + ((int64_t)r * slices * K + k) * dim + tid;
    for (int64_t s = 0; s < slices; ++s) acc = __dadd_rn(acc, (double)src[s * K * dim]);
    if (total > 0) centroids[((int64_t)r * K + k) * dim + tid] = __double2float_rn(__ddiv_rn(acc, (double)total));
    if (k != 0) return;
    const int64_t p = (int64_t)r * slices;
    if (tid == 0) {
        double in = 0.0;
        int ch = 0;
        for (int64_t s = 0; s < slices; ++s) { in = __dadd_rn(in, ws.inertia[p + s]); ch += ws.changed[p + s]; }
        inertia[r] = in;
        changed[r] = ch;
    }
    for (int kk = tid; kk < K; kk += blockDim.x) {
        int c = 0;
        for (int64_t s = 0; s < slices; ++s) c += ws.counts[(p + s) * K + kk];
        if (c == 0) atomicAdd(&n_empty, 1);                 // an integer count: the total does not depend on the order
    }
    __syncthreads();
    if (tid == 0) empty[r] = n_empty;
}

__global__ void __launch_bounds__(KM_THREADS) kmeans_seed_pick_kernel(const msst_kmeans_dims d, int64_t slices, int j,
                                                                      const float* __restrict__ x, const double* __restrict__ u,
                                                                      float* __restrict__ centroids, int64_t* __restrict__ index,
                                                                      const float* __restrict__ mindist,
                                                                      const double* __restrict__ slice_sums) {
    __shared__ float m[KM_SLICE];
    __shared__ int64_t s_found, pick;
    __shared__ double base, thr;
    const int K = d.k, tid = threadIdx.x, r = blockIdx.x;
    const int64_t n = d.n;
    const double ur = u[r * K + j];
    const double f = floor(__dmul_rn(ur, (double)n));
    const int64_t fallback = f >= 0.0 ? (int64_t)fmin(f, (double)(n - 1)) : 0;   // NaN -> 0
    if (tid == 0) {
        int64_t sf = -1;
        double P = 0.0, t = 0.0;
        if (j > 0) {
            const double* S = slice_sums + (int64_t)r * slices;
            double T = 0.0;
            for (int64_t s = 0; s < slices; ++s) T = __dadd_rn(T, S[s]);
            if (T > 0.0) {
                t = __dmul_rn(ur, T);
                for (int64_t s = 0; s < slices; ++s) {
                    const double Pn = __dadd_rn(P, S[s]);
                    if (Pn > t) { sf = s; break; }
                    P = Pn;
                }
            }
        }
        s_found = sf; base = P; thr = t; pick = fallback;
    }
    __syncthreads();
    if (s_found >= 0) {
        const int64_t first = s_found * KM_SLICE;
        const int rows = (int)min((int64_t)KM_SLICE, n - first);
        for (int i = tid; i < rows; i += KM_THREADS) m[i] = mindist[(int64_t)r * n + first + i];
        __syncthreads();
        if (tid == 0) {
            double L = 0.0;
            for (int i = 0; i < rows; ++i) {
                L = __dadd_rn(L, (double)m[i]);
                if (__dadd_rn(base, L) > thr) { pick = first + i; break; }
            }
        }
        __syncthreads();
    }
    const int64_t p = pick;
    if (tid == 0) index[r * K + j] = p;
    if (tid < 32) {
        float v[KM_MAX_DIM / 32];
        km_row(x + p * d.dim, d.dim, tid, d.normalize, v);
        float* c = centroids + ((int64_t)r * K + j) * d.dim;
#pragma unroll
        for (int i = 0; i < KM_MAX_DIM / 32; ++i)
            if (tid + 32 * i < d.dim) c[tid + 32 * i] = v[i];
    }
}

__global__ void __launch_bounds__(KM_THREADS) kmeans_seed_dist_kernel(const msst_kmeans_dims d, int64_t slices, int j,
                                                                      const float* __restrict__ x, const float* __restrict__ centroids,
                                                                      float* __restrict__ mindist, double* __restrict__ slice_sums) {
    __shared__ float m[KM_SLICE];
    const int R = d.restarts, dim = d.dim, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r = (int)(blockIdx.x % R);
    const int64_t slice = blockIdx.x / R, first = slice * KM_SLICE;
    const int rows = (int)min((int64_t)KM_SLICE, d.n - first);
    float c[KM_MAX_DIM / 32];
    const float* cj = centroids + ((int64_t)r * d.k + j) * dim;
#pragma unroll
    for (int i = 0; i < KM_MAX_DIM / 32; ++i) c[i] = lane + 32 * i < dim ? cj[lane + 32 * i] : 0.f;
    float* md = mindist + (int64_t)r * d.n + first;
    for (int rr = warp; rr < rows; rr += KM_THREADS / 32) {
        float v[KM_MAX_DIM / 32];
        km_row(x + (first + rr) * dim, dim, lane, d.normalize, v);
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < KM_MAX_DIM / 32; ++i) { const float e = __fsub_rn(v[i], c[i]); sq = fmaf(e, e, sq); }
        const float dd = warp_sum(sq);
        if (lane == 0) {
            const float out = j == 0 ? dd : fminf(md[rr], dd);
            md[rr] = out;
            m[rr] = out;
        }
    }
    __syncthreads();
    if (tid == 0) {                                         // ascending row order: the order the pick kernel scans
        double s = 0.0;
        for (int i = 0; i < rows; ++i) s = __dadd_rn(s, (double)m[i]);
        slice_sums[(int64_t)r * slices + slice] = s;
    }
}

static bool km_dim_ok(int dim) { return dim >= 32 && dim <= KM_MAX_DIM && dim % 32 == 0; }

// fitting: seeding and assignment with a workspace need K <= n; prediction needs one row
static int km_check(const msst_kmeans_dims* d, const char* who, bool fitting) {
    MSST_REQUIRE(d, "%s: dims must be set", who);
    MSST_REQUIRE(km_dim_ok(d->dim), "%s: dim=%d must be a multiple of 32 in [32, %d]", who, d->dim, KM_MAX_DIM);
    MSST_REQUIRE(d->k >= 1 && d->k <= KM_MAX_K, "%s: k=%d outside [1, %d]", who, d->k, KM_MAX_K);
    MSST_REQUIRE((int64_t)d->k * d->dim <= MSST_KMEANS_MAX_KD, "%s: k*dim=%lld exceeds %d", who, (long long)d->k * d->dim,
                 MSST_KMEANS_MAX_KD);
    MSST_REQUIRE(d->restarts >= 1 && d->restarts <= MSST_KMEANS_MAX_RESTARTS, "%s: restarts=%d outside [1, %d]", who, d->restarts,
                 MSST_KMEANS_MAX_RESTARTS);
    MSST_REQUIRE(d->normalize == 0 || d->normalize == 1, "%s: normalize=%d must be 0 or 1", who, d->normalize);
    const int64_t lo = fitting ? d->k : 1;
    MSST_REQUIRE(d->n >= lo && d->n < 2147483648LL, "%s: n=%lld rows outside [%lld, 2^31)", who, (long long)d->n, (long long)lo);
    return MSST_OK;
}

}  // namespace msst
using namespace msst;

extern "C" int64_t msst_kmeans_workspace(const msst_kmeans_dims* d) {
    if (km_check(d, "kmeans_workspace", true) != MSST_OK) return -1;
    const int64_t rs = (int64_t)d->restarts * km_slices(d->n);
    return rs * (8 + 4 * (int64_t)d->k * d->dim + 4 * (int64_t)d->k + 4);
}

extern "C" int msst_kmeans_seed(const msst_kmeans_dims* d, int round, const float* x, const double* u, float* centroids, int64_t* index,
                                float* mindist, void* workspace, msst_stream_t stream) {
    if (int rc = km_check(d, "kmeans_seed", true)) return rc;
    MSST_REQUIRE(round >= 0 && round < d->k, "kmeans_seed: round=%d outside [0, k=%d)", round, d->k);
    MSST_REQUIRE(x && u && centroids && index && mindist && workspace, "kmeans_seed: x / u / centroids / index / mindist / workspace must be set");
    const int64_t S = km_slices(d->n);
    const KmWs ws = km_ws(workspace, d->restarts, S, d->k, d->dim);
    const cudaStream_t st = (cudaStream_t)stream;
    kmeans_seed_pick_kernel<<<(unsigned)d->restarts, KM_THREADS, 0, st>>>(*d, S, round, x, u, centroids, index, mindist, ws.inertia);
    MSST_LAUNCH_CHECK();
    if (round + 1 < d->k) {
        kmeans_seed_dist_kernel<<<(unsigned)(S * d->restarts), KM_THREADS, 0, st>>>(*d, S, round, x, centroids, mindist, ws.inertia);
        MSST_LAUNCH_CHECK();
    }
    return MSST_OK;
}

extern "C" int msst_kmeans_assign(const msst_kmeans_dims* d, const float* x, const float* centroids, int64_t* labels, float* dist,
                                  void* workspace, msst_stream_t stream) {
    const bool with_ws = workspace != nullptr;
    if (int rc = km_check(d, "kmeans_assign", with_ws)) return rc;
    MSST_REQUIRE(x && centroids && labels, "kmeans_assign: x / centroids / labels must be set");
    static PerDeviceOnce once;
    if (once.first()) MSST_CUDA(cudaFuncSetAttribute((const void*)kmeans_assign_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, KM_SMEM_MAX));
    const int64_t S = km_slices(d->n);
    const KmWs ws = with_ws ? km_ws(workspace, d->restarts, S, d->k, d->dim) : KmWs{nullptr, nullptr, nullptr, nullptr};
    kmeans_assign_kernel<<<(unsigned)(S * d->restarts), KM_THREADS, km_assign_smem(d->dim, d->k, with_ws), (cudaStream_t)stream>>>(
        *d, S, x, centroids, labels, dist, ws, with_ws);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

extern "C" int msst_kmeans_update(const msst_kmeans_dims* d, const void* workspace, float* centroids, double* inertia, int32_t* changed,
                                  int32_t* empty, msst_stream_t stream) {
    if (int rc = km_check(d, "kmeans_update", true)) return rc;
    MSST_REQUIRE(workspace && centroids && inertia && changed && empty, "kmeans_update: workspace / centroids / inertia / changed / empty must be set");
    const int64_t S = km_slices(d->n);
    const KmWs ws = km_ws(const_cast<void*>(workspace), d->restarts, S, d->k, d->dim);
    kmeans_update_kernel<<<(unsigned)(d->restarts * d->k), (unsigned)d->dim, 0, (cudaStream_t)stream>>>(*d, S, ws, centroids, inertia,
                                                                                                        changed, empty);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}
