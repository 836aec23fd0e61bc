// Mean, covariance and projection of fp32 rows (msst_moments_*, include/msst.h): the device half of PCA and of the global RX anomaly
// detector.  All arithmetic is FP64 on the CUDA cores: rows are centred as c = (double)x - mean, and every sum runs in a fixed order.
//
//   moments_mean_kernel      CTA = one 16384-row slice, thread = column: the slice's fp64 column sums, rows added in ascending order
//                            (32-row tiles staged in shared memory so that all 256 threads load).
//   moments_mean_reduce      thread = column: the slices added in ascending order, / n.
//   moments_cov_kernel       CTA = (slice, 64 x 64 tile of the upper triangle), 256 threads, each a 4 x 4 block of fp64 accumulators
//                            (rows tr + 16a, columns tc + 16b).  Centred 32-row tiles of both column blocks are staged in shared
//                            memory as fp64; every entry is an fp64 FMA chain over the slice's rows in ascending order.
//   moments_cov_reduce       thread = (i <= j): the slices added in ascending order, / (n - 1), written to (i, j) and (j, i).
//   moments_project_kernel   CTA = 4 TR rows, thread = 4 rows x 4 components; the components run in chunks of 4 * (256 / TR) in
//                            ascending order and dim in 32-wide stages: y_ij = sum_d c_id W_jd as one fp64 FMA chain in ascending d.
//                            One thread per row then adds the chunk's y_ij^2 (unrounded fp64) to the row's score in ascending j.
//                            TR = 64 (16 components per chunk) for k <= 16, else TR = 16 (64 components).
//
// No atomics: a slice partial depends only on the slice's rows, the sums over slices run in ascending order, and a projected row depends
// only on that row, so every result is bitwise independent of the grid, the SM count and (for the projection) the rows it ran with.
// The two-pass covariance is deliberate: the one-pass E[xx^T] - mu mu^T cancels catastrophically for rows far from the origin.
#include "common.cuh"

namespace msst {

constexpr int MO_SLICE = 16384;              // rows of a slice (fixed: the partials and their order never depend on the launch)
constexpr int MO_THREADS = 256;
constexpr int MO_MAX_DIM = 256;
constexpr int MO_TILE = 64;                  // covariance tile side
constexpr int MO_KR = 32;                    // rows (covariance) or features (projection) per shared-memory stage
static_assert(MO_THREADS >= MO_MAX_DIM, "thread = column in the mean");

static int64_t mo_slices(int64_t n) { return ceil_div(n, MO_SLICE); }
static int mo_tiles(int dim) { const int t = (int)ceil_div(dim, MO_TILE); return t * (t + 1) / 2; }

__global__ void __launch_bounds__(MO_THREADS) moments_mean_kernel(int64_t n, int dim, const float* __restrict__ x,
                                                                  double* __restrict__ part) {
    __shared__ float xs[MO_KR * MO_MAX_DIM];
    const int tid = threadIdx.x;
    const int64_t first = (int64_t)blockIdx.x * MO_SLICE;
    const int rows = (int)min((int64_t)MO_SLICE, n - first);
    const float* xb = x + first * dim;
    double acc = 0.0;
    for (int r0 = 0; r0 < rows; r0 += MO_KR) {
        const int cnt = min(MO_KR, rows - r0);
        __syncthreads();
        for (int i = tid; i < cnt * dim; i += MO_THREADS) xs[i] = xb[(int64_t)r0 * dim + i];
        __syncthreads();
        if (tid < dim)
            for (int r = 0; r < cnt; ++r) acc = __dadd_rn(acc, (double)xs[r * dim + tid]);
    }
    if (tid < dim) part[(int64_t)blockIdx.x * dim + tid] = acc;
}

__global__ void moments_mean_reduce(int64_t n, int dim, int64_t slices, const double* __restrict__ part, double* __restrict__ mean) {
    const int c = threadIdx.x;
    if (c >= dim) return;
    double acc = 0.0;
    for (int64_t s = 0; s < slices; ++s) acc = __dadd_rn(acc, part[s * dim + c]);
    mean[c] = __ddiv_rn(acc, (double)n);
}

// blockIdx.y = upper-triangle tile (I, J), I <= J, row-major
__global__ void __launch_bounds__(MO_THREADS) moments_cov_kernel(int64_t n, int dim, const float* __restrict__ x,
                                                                 const double* __restrict__ mean, double* __restrict__ part) {
    __shared__ double as[MO_KR][MO_TILE], bs[MO_KR][MO_TILE];
    __shared__ double ma[MO_TILE], mb[MO_TILE];
    const int tid = threadIdx.x, tr = tid / 16, tc = tid % 16;
    int I = 0, t = blockIdx.y;
    const int T = (int)ceil_div(dim, MO_TILE);
    while (t >= T - I) { t -= T - I; ++I; }
    const int J = I + t, ca = I * MO_TILE, cb = J * MO_TILE;
    if (tid < MO_TILE) {
        ma[tid] = ca + tid < dim ? mean[ca + tid] : 0.0;
        mb[tid] = cb + tid < dim ? mean[cb + tid] : 0.0;
    }
    const int64_t first = (int64_t)blockIdx.x * MO_SLICE;
    const int rows = (int)min((int64_t)MO_SLICE, n - first);
    double acc[4][4] = {};
    for (int r0 = 0; r0 < rows; r0 += MO_KR) {
        const int cnt = min(MO_KR, rows - r0);
        __syncthreads();                                   // means staged / the previous tile consumed
        for (int i = tid; i < MO_KR * MO_TILE; i += MO_THREADS) {
            const int r = i / MO_TILE, cc = i % MO_TILE;
            const float* xr = x + (first + r0 + r) * dim;
            as[r][cc] = r < cnt && ca + cc < dim ? __dsub_rn((double)xr[ca + cc], ma[cc]) : 0.0;
            bs[r][cc] = r < cnt && cb + cc < dim ? __dsub_rn((double)xr[cb + cc], mb[cc]) : 0.0;
        }
        __syncthreads();
        for (int r = 0; r < cnt; ++r) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = as[r][tr + 16 * i]; b[i] = bs[r][tc + 16 * i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = __fma_rn(a[i], b[j], acc[i][j]);
        }
    }
    double* out = part + (int64_t)blockIdx.x * dim * dim;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ri = ca + tr + 16 * i, cj = cb + tc + 16 * j;
            if (ri < dim && cj < dim) out[ri * dim + cj] = acc[i][j];
        }
}

__global__ void moments_cov_reduce(int64_t n, int dim, int64_t slices, const double* __restrict__ part, double* __restrict__ cov) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= dim * dim) return;
    const int i = e / dim, j = e % dim;
    if (i > j) return;
    double acc = 0.0;
    for (int64_t s = 0; s < slices; ++s) acc = __dadd_rn(acc, part[s * dim * dim + e]);
    const double v = __ddiv_rn(acc, (double)(n - 1));
    cov[(int64_t)i * dim + j] = v;
    cov[(int64_t)j * dim + i] = v;
}

template <int TR>
struct ProjShape {
    static constexpr int TC = MO_THREADS / TR, ROWS = 4 * TR, COMPS = 4 * TC;
    // [MO_KR][ROWS + 1] centred rows and [MO_KR][COMPS + 1] components (transposed: feature-major), later reused as y [ROWS][COMPS + 1]
    static constexpr size_t STAGE = (size_t)MO_KR * (ROWS + 1 + COMPS + 1), YS = (size_t)ROWS * (COMPS + 1);
    static constexpr size_t SMEM = 8 * (STAGE > YS ? STAGE : YS);
};

template <int TR>
__global__ void __launch_bounds__(MO_THREADS) moments_project_kernel(int64_t n, int dim, int k, const float* __restrict__ x,
                                                                     const double* __restrict__ mean, const double* __restrict__ W,
                                                                     float* __restrict__ y, float* __restrict__ score) {
    using S = ProjShape<TR>;
    extern __shared__ double mo_smem[];
    double* cs = mo_smem;                                  // [MO_KR][ROWS + 1]
    double* ws = mo_smem + MO_KR * (S::ROWS + 1);          // [MO_KR][COMPS + 1]
    double* ys = mo_smem;                                  // [ROWS][COMPS + 1]
    const int tid = threadIdx.x, tr = tid / S::TC, tc = tid % S::TC;
    const int64_t row0 = (int64_t)blockIdx.x * S::ROWS;
    const int rows = (int)min((int64_t)S::ROWS, n - row0);
    double sc = 0.0;                                       // thread tid < rows: the score of row row0 + tid
    for (int j0 = 0; j0 < k; j0 += S::COMPS) {
        const int nc = min(S::COMPS, k - j0);
        double acc[4][4] = {};
        for (int d0 = 0; d0 < dim; d0 += MO_KR) {
            const int nd = min(MO_KR, dim - d0);
            __syncthreads();                               // the previous stage / y of the previous chunk consumed
            for (int i = tid; i < S::ROWS * MO_KR; i += MO_THREADS) {
                const int r = i / MO_KR, dd = i % MO_KR;
                cs[dd * (S::ROWS + 1) + r] =
                    r < rows && dd < nd ? __dsub_rn((double)x[(row0 + r) * dim + d0 + dd], mean[d0 + dd]) : 0.0;
            }
            for (int i = tid; i < S::COMPS * MO_KR; i += MO_THREADS) {
                const int c = i / MO_KR, dd = i % MO_KR;
                ws[dd * (S::COMPS + 1) + c] = c < nc && dd < nd ? W[(int64_t)(j0 + c) * dim + d0 + dd] : 0.0;
            }
            __syncthreads();
            for (int dd = 0; dd < nd; ++dd) {
                double a[4], b[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) { a[i] = cs[dd * (S::ROWS + 1) + tr + TR * i]; b[i] = ws[dd * (S::COMPS + 1) + tc + S::TC * i]; }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = __fma_rn(a[i], b[j], acc[i][j]);
            }
        }
        __syncthreads();                                   // the last stage consumed: ys overwrites it
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) ys[(tr + TR * i) * (S::COMPS + 1) + tc + S::TC * j] = acc[i][j];
        __syncthreads();
        if (y)
            for (int i = tid; i < rows * nc; i += MO_THREADS) {
                const int r = i / nc, c = i % nc;
                y[(row0 + r) * k + j0 + c] = __double2float_rn(ys[r * (S::COMPS + 1) + c]);
            }
        if (score && tid < rows)
            for (int c = 0; c < nc; ++c) {
                const double v = ys[tid * (S::COMPS + 1) + c];
                sc = __fma_rn(v, v, sc);
            }
    }
    if (score && tid < rows) score[row0 + tid] = __double2float_rn(sc);
}

template <int TR>
static int mo_project_launch(int64_t n, int dim, int k, const float* x, const double* mean, const double* W, float* y, float* score,
                             cudaStream_t st) {
    using S = ProjShape<TR>;
    static PerDeviceOnce once;
    if (once.first())
        MSST_CUDA(cudaFuncSetAttribute((const void*)moments_project_kernel<TR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::SMEM));
    moments_project_kernel<TR><<<(unsigned)ceil_div(n, S::ROWS), MO_THREADS, S::SMEM, st>>>(n, dim, k, x, mean, W, y, score);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

static int mo_check(int64_t n, int dim, int64_t lo, const char* who) {
    MSST_REQUIRE(dim >= 1 && dim <= MO_MAX_DIM, "%s: dim=%d outside [1, %d]", who, dim, MO_MAX_DIM);
    MSST_REQUIRE(n >= lo && n < 2147483648LL, "%s: n=%lld rows outside [%lld, 2^31)", who, (long long)n, (long long)lo);
    return MSST_OK;
}

}  // namespace msst
using namespace msst;

extern "C" int64_t msst_moments_workspace(int64_t n, int dim) {
    if (mo_check(n, dim, 2, "moments_workspace") != MSST_OK) return -1;
    return 8 * mo_slices(n) * dim * (int64_t)(dim + 1);
}

extern "C" int msst_moments_mean(int64_t n, int dim, const float* x, void* workspace, double* mean, msst_stream_t stream) {
    if (int rc = mo_check(n, dim, 2, "moments_mean")) return rc;
    MSST_REQUIRE(x && workspace && mean, "moments_mean: x / workspace / mean must be set");
    const int64_t S = mo_slices(n);
    double* part = static_cast<double*>(workspace);
    const cudaStream_t st = (cudaStream_t)stream;
    moments_mean_kernel<<<(unsigned)S, MO_THREADS, 0, st>>>(n, dim, x, part);
    MSST_LAUNCH_CHECK();
    moments_mean_reduce<<<1, MO_MAX_DIM, 0, st>>>(n, dim, S, part, mean);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

extern "C" int msst_moments_cov(int64_t n, int dim, const float* x, const double* mean, void* workspace, double* cov, msst_stream_t stream) {
    if (int rc = mo_check(n, dim, 2, "moments_cov")) return rc;
    MSST_REQUIRE(x && mean && workspace && cov, "moments_cov: x / mean / workspace / cov must be set");
    const int64_t S = mo_slices(n);
    double* part = static_cast<double*>(workspace) + S * dim;     // after the mean partials
    const cudaStream_t st = (cudaStream_t)stream;
    moments_cov_kernel<<<dim3((unsigned)S, (unsigned)mo_tiles(dim)), MO_THREADS, 0, st>>>(n, dim, x, mean, part);
    MSST_LAUNCH_CHECK();
    moments_cov_reduce<<<(unsigned)ceil_div((int64_t)dim * dim, MO_THREADS), MO_THREADS, 0, st>>>(n, dim, S, part, cov);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

extern "C" int msst_moments_project(int64_t n, int dim, int k, const float* x, const double* mean, const double* W, float* y, float* score,
                                    msst_stream_t stream) {
    if (int rc = mo_check(n, dim, 1, "moments_project")) return rc;
    MSST_REQUIRE(k >= 1 && k <= dim, "moments_project: k=%d outside [1, dim=%d]", k, dim);
    MSST_REQUIRE(x && mean && W, "moments_project: x / mean / W must be set");
    MSST_REQUIRE(y || score, "moments_project: y and score are both NULL");
    const cudaStream_t st = (cudaStream_t)stream;
    return k <= 16 ? mo_project_launch<64>(n, dim, k, x, mean, W, y, score, st) : mo_project_launch<16>(n, dim, k, x, mean, W, y, score, st);
}
