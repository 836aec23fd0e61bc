// Linear probing of embeddings (msst_linprobe_*, include/msst.h): softmax regression on LayerNorm'ed fp32 feature rows, all heads of a
// fit trained in the same two launches per minibatch, and prediction.  FP32 FFMA throughout (the probe's accuracy contract rules out
// bf16 / TF32 operands).
//
//   linprobe_grad_kernel     CTA = (128-row slice of the minibatch, head).  Gathers the slice's rows through the index and normalises
//                            each once (lp_ln_row, one warp per row, four rows in flight) into shared memory z [128][dim].  Pass 1, per chunk of 32
//                            classes: W_h chunk -> shared memory, logits [128][32] (thread tile 4 rows x 4 classes, float4 along
//                            dim), online row max / sum of exp in ascending class order, the label's logit.  Pass 2, per chunk:
//                            G = softmax - onehot, dW chunk = G^T z (thread tile 4 classes x 4 features, rows in ascending order),
//                            db chunk = column sums of G.  With nc <= 32 the one chunk's logits stay in shared memory; otherwise pass
//                            2 recomputes them with the same code, so both passes see the same bits.  The slice's dW, db and CE sum
//                            go to the workspace.
//   linprobe_update_kernel   thread = parameter of one head: the slices' partials summed in ascending slice order, / batch, AdamW
//                            (adam_one, adam.cuh) with the head's lr / wd.  One thread per head writes the step's CE sum.
//   linprobe_predict_kernel  CTA = 128 query rows: the same normalisation and logits code, softmax, argmax (lowest class on ties).
//
// Nothing a head computes depends on the number of heads or CTAs, and no atomics are used: results are bitwise reproducible, a head
// fitted with others equals the head fitted alone, and a query's prediction does not depend on the chunk it ran in.
#include "adam.cuh"

namespace msst {

constexpr int LP_ROWS = 128;                 // rows of a slice / a prediction tile
constexpr int LP_CH = 32;                    // classes per chunk
constexpr int LP_THREADS = 256;
constexpr int LP_LDL = LP_CH + 1;            // row stride of the logits tile
constexpr int LP_MAX_DIM = 256, LP_MAX_CLASSES = 256;
constexpr int LP_SMEM_MAX = 227 * 1024;

// z [128][dim + 4] (float4 rows; +4 keeps the row stride at 16 bytes mod 128 for conflict-free float4 reads), W chunk [32][dim + 4],
// logits / G [128][33], per-row max, sum of exp, label logit and label
static size_t lp_smem(int dim) {
    return (size_t)(LP_ROWS + LP_CH) * (dim + 4) * 4 + (size_t)LP_ROWS * LP_LDL * 4 + (size_t)LP_ROWS * 4 * 4;
}

struct LpTile {
    float *z, *w, *L, *m, *s, *ly;
    int* lab;
    int ldz;
    __device__ LpTile(float* sm, int dim) {
        ldz = dim + 4;
        z = sm; w = z + LP_ROWS * ldz; L = w + LP_CH * ldz;
        m = L + LP_ROWS * LP_LDL; s = m + LP_ROWS; ly = s + LP_ROWS; lab = reinterpret_cast<int*>(ly + LP_ROWS);
    }
};

constexpr int LP_LOAD_ROWS = 4;             // rows a warp loads before it normalises them (the gather is latency-bound)

__device__ __forceinline__ void lp_read_row(const float* __restrict__ xr, int dim, int lane, float (&v)[LP_MAX_DIM / 32]) {
#pragma unroll
    for (int i = 0; i < LP_MAX_DIM / 32; ++i) {
        const int c = lane + 32 * i;
        v[i] = (xr != nullptr && c < dim) ? xr[c] : 0.f;
    }
}

// out = (x - mean) / sqrt(var + 1e-5), mean and biased variance over dim (F.layer_norm(x, (dim,))), x = the row lp_read_row read.
// The one normalisation of training and prediction.
__device__ __forceinline__ void lp_ln_row(float (&v)[LP_MAX_DIM / 32], int dim, int lane, float* __restrict__ out) {
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < LP_MAX_DIM / 32; ++i) sum += v[i];
    const float mean = __fdiv_rn(warp_sum(sum), (float)dim);
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < LP_MAX_DIM / 32; ++i)
        if (lane + 32 * i < dim) { v[i] = __fsub_rn(v[i], mean); sq = fmaf(v[i], v[i], sq); }
    const float rstd = __fdiv_rn(1.f, sqrtf(__fadd_rn(__fdiv_rn(warp_sum(sq), (float)dim), 1e-5f)));
#pragma unroll
    for (int i = 0; i < LP_MAX_DIM / 32; ++i)
        if (lane + 32 * i < dim) out[lane + 32 * i] = __fmul_rn(v[i], rstd);
}

// rows r < count of the tile: x[index[first + r]] (index == nullptr: x[first + r]), normalised; the other rows (and rows whose index is
// outside [0, n)) are zero.  Warp w owns rows w + 8k and reads LP_LOAD_ROWS of them before normalising them.
__device__ void lp_load_rows(const LpTile& t, const float* __restrict__ x, const int64_t* __restrict__ index, int64_t first, int count,
                             int64_t n, int dim) {
    constexpr int NW = LP_THREADS / 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int k0 = 0; k0 < LP_ROWS / NW; k0 += LP_LOAD_ROWS) {
        float v[LP_LOAD_ROWS][LP_MAX_DIM / 32];
#pragma unroll
        for (int q = 0; q < LP_LOAD_ROWS; ++q) {
            const int r = warp + NW * (k0 + q);
            const float* xr = nullptr;
            if (r < count) {
                const int64_t i = index ? index[first + r] : first + r;
                if (i >= 0 && i < n) xr = x + i * dim;
            }
            lp_read_row(xr, dim, lane, v[q]);
        }
#pragma unroll
        for (int q = 0; q < LP_LOAD_ROWS; ++q) lp_ln_row(v[q], dim, lane, t.z + (warp + NW * (k0 + q)) * t.ldz);
    }
}

// L[r][j] = b[c0 + j] + sum_d z[r][d] W[c0 + j][d] for the tile's 128 rows and classes c0 + j < nc (-inf beyond); W [nc][dim], b [nc].
// Thread tile: rows rw + 32i x classes cl + 8j, the sum over d in ascending order.  Starts and ends with a barrier.
__device__ void lp_logits(const LpTile& t, const float* __restrict__ W, const float* __restrict__ b, int c0, int nc, int dim) {
    const int tid = threadIdx.x, ncc = min(LP_CH, nc - c0);
    __syncthreads();
    for (int i = tid; i < LP_CH * dim; i += LP_THREADS) {
        const int c = i / dim, d = i - c * dim;
        t.w[c * t.ldz + d] = c < ncc ? W[(int64_t)(c0 + c) * dim + d] : 0.f;
    }
    __syncthreads();
    const int cl = tid & 7, rw = tid >> 3;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int d = 0; d < dim; d += 4) {
        float4 z[4], w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) z[i] = *reinterpret_cast<const float4*>(t.z + (rw + 32 * i) * t.ldz + d);
#pragma unroll
        for (int j = 0; j < 4; ++j) w[j] = *reinterpret_cast<const float4*>(t.w + (cl + 8 * j) * t.ldz + d);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                acc[i][j] = fmaf(z[i].x, w[j].x, acc[i][j]); acc[i][j] = fmaf(z[i].y, w[j].y, acc[i][j]);
                acc[i][j] = fmaf(z[i].z, w[j].z, acc[i][j]); acc[i][j] = fmaf(z[i].w, w[j].w, acc[i][j]);
            }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = cl + 8 * j;
            t.L[(rw + 32 * i) * LP_LDL + c] = c < ncc ? __fadd_rn(acc[i][j], b[c0 + c]) : -INFINITY;
        }
    __syncthreads();
}

// pass 1 over all chunks: per row (threads 0..127) the running max m and sum of exp(l - m) in ascending class order, and the label's
// logit.  Leaves the last chunk's logits in L.
__device__ void lp_row_stats(const LpTile& t, const float* __restrict__ W, const float* __restrict__ b, int nc, int dim) {
    const int tid = threadIdx.x;
    float m = -INFINITY, s = 0.f, ly = 0.f;
    const int lab = tid < LP_ROWS ? t.lab[tid] : -1;
    for (int c0 = 0; c0 < nc; c0 += LP_CH) {
        lp_logits(t, W, b, c0, nc, dim);
        if (tid < LP_ROWS) {
            const int ncc = min(LP_CH, nc - c0);
            for (int j = 0; j < ncc; ++j) {
                const float l = t.L[tid * LP_LDL + j];
                if (l > m) { s = __fadd_rn(__fmul_rn(s, expf(__fsub_rn(m, l))), 1.f); m = l; }
                else s = __fadd_rn(s, expf(__fsub_rn(l, m)));
            }
            if (lab >= c0 && lab < c0 + ncc) ly = t.L[tid * LP_LDL + lab - c0];
        }
    }
    if (tid < LP_ROWS) { t.m[tid] = m; t.s[tid] = s; t.ly[tid] = ly; }
    __syncthreads();
}

__device__ __forceinline__ float lp_prob(const LpTile& t, int r, float l) { return __fdiv_rn(expf(__fsub_rn(l, t.m[r])), t.s[r]); }

__global__ void __launch_bounds__(LP_THREADS) linprobe_grad_kernel(const msst_linprobe_dims d, const float* __restrict__ x,
                                                                   const int64_t* __restrict__ labels, const int64_t* __restrict__ index,
                                                                   const float* __restrict__ params, float* __restrict__ ws) {
    extern __shared__ float4 lp_smem_raw[];
    const LpTile t(reinterpret_cast<float*>(lp_smem_raw), d.dim);
    const int slice = blockIdx.x, h = blockIdx.y, tid = threadIdx.x, dim = d.dim, nc = d.nc;
    const int64_t first = (int64_t)slice * LP_ROWS;
    const int count = (int)min((int64_t)LP_ROWS, (int64_t)d.batch - first);
    const int64_t P = (int64_t)nc * dim + nc;
    const float* W = params + h * P;
    const float* b = W + (int64_t)nc * dim;
    float* out = ws + ((int64_t)slice * d.heads + h) * (P + 1);

    if (tid < LP_ROWS) {   // label of the row, -1 when the row contributes nothing
        int lab = -1;
        if (tid < count) {
            const int64_t i = index[first + tid];
            if (i >= 0 && i < d.n) { const int64_t y = labels[i]; if (y >= 0 && y < nc) lab = (int)y; }
        }
        t.lab[tid] = lab;
    }
    lp_load_rows(t, x, index, first, count, d.n, dim);
    lp_row_stats(t, W, b, nc, dim);
    if (tid == 0) {   // the slice's CE sum, rows in ascending order
        float ce = 0.f;
        for (int r = 0; r < LP_ROWS; ++r)
            if (t.lab[r] >= 0) ce = __fadd_rn(ce, __fsub_rn(__fadd_rn(t.m[r], logf(t.s[r])), t.ly[r]));
        out[P] = ce;
    }
    const bool one_chunk = nc <= LP_CH;
    for (int c0 = 0; c0 < nc; c0 += LP_CH) {
        const int ncc = min(LP_CH, nc - c0);
        if (!one_chunk) lp_logits(t, W, b, c0, nc, dim);
        for (int i = tid; i < LP_ROWS * LP_CH; i += LP_THREADS) {   // G = softmax - onehot in place
            const int r = i / LP_CH, j = i - r * LP_CH;
            float g = 0.f;
            const int lab = t.lab[r];
            if (lab >= 0 && j < ncc) g = __fsub_rn(lp_prob(t, r, t.L[r * LP_LDL + j]), c0 + j == lab ? 1.f : 0.f);
            t.L[r * LP_LDL + j] = g;
        }
        __syncthreads();
        for (int tile = tid; tile < 8 * (dim / 4); tile += LP_THREADS) {   // dW chunk: classes cl + 8j x features 4*d4 .. 4*d4 + 3
            const int cl = tile & 7, d4 = tile >> 3;
            float acc[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int k = 0; k < 4; ++k) acc[j][k] = 0.f;
            for (int r = 0; r < LP_ROWS; ++r) {
                const float4 z = *reinterpret_cast<const float4*>(t.z + r * t.ldz + 4 * d4);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float g = t.L[r * LP_LDL + cl + 8 * j];
                    acc[j][0] = fmaf(g, z.x, acc[j][0]); acc[j][1] = fmaf(g, z.y, acc[j][1]);
                    acc[j][2] = fmaf(g, z.z, acc[j][2]); acc[j][3] = fmaf(g, z.w, acc[j][3]);
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = cl + 8 * j;
                if (c < ncc) {
                    float* o = out + (int64_t)(c0 + c) * dim + 4 * d4;
                    o[0] = acc[j][0]; o[1] = acc[j][1]; o[2] = acc[j][2]; o[3] = acc[j][3];
                }
            }
        }
        if (tid < ncc) {   // db chunk
            float a = 0.f;
            for (int r = 0; r < LP_ROWS; ++r) a = __fadd_rn(a, t.L[r * LP_LDL + tid]);
            out[(int64_t)nc * dim + c0 + tid] = a;
        }
        __syncthreads();   // G is read above before the next chunk overwrites L
    }
}

struct LpUpdate {
    AdamK a;
    float lr[MSST_LINPROBE_MAX_HEADS], wd[MSST_LINPROBE_MAX_HEADS];
    int heads, slices, batch;
    int64_t P;
};

__global__ void __launch_bounds__(256) linprobe_update_kernel(const LpUpdate u, const float* __restrict__ ws, float* __restrict__ params,
                                                              float* __restrict__ m, float* __restrict__ v, float* __restrict__ loss_sum) {
    const int64_t total = (int64_t)u.heads * u.P, stride = u.P + 1;
    const float nb = (float)u.batch;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int h = (int)(i / u.P);
        const int64_t e = i - h * u.P;
        const float* w = ws + (int64_t)h * stride + e;
        float g = 0.f;
        for (int s = 0; s < u.slices; ++s) g = __fadd_rn(g, w[(int64_t)s * u.heads * stride]);
        AdamK a = u.a;
        a.lr = u.lr[h]; a.wd = u.wd[h];
        float p = params[i], mi = m[i], vi = v[i];
        adam_one(a, p, __fdiv_rn(g, nb), mi, vi);
        params[i] = p; m[i] = mi; v[i] = vi;
    }
    if (blockIdx.x == 0 && threadIdx.x < u.heads) {
        const int h = threadIdx.x;
        float ce = 0.f;
        for (int s = 0; s < u.slices; ++s) ce = __fadd_rn(ce, ws[((int64_t)s * u.heads + h) * stride + u.P]);
        loss_sum[h] = ce;
    }
}

__global__ void __launch_bounds__(LP_THREADS) linprobe_predict_kernel(int64_t nq, int dim, int nc, const float* __restrict__ x,
                                                                      const float* __restrict__ params, float* __restrict__ probs,
                                                                      int64_t* __restrict__ pred) {
    extern __shared__ float4 lp_smem_raw[];
    const LpTile t(reinterpret_cast<float*>(lp_smem_raw), dim);
    const int tid = threadIdx.x;
    const int64_t first = (int64_t)blockIdx.x * LP_ROWS;
    const int count = (int)min((int64_t)LP_ROWS, nq - first);
    const float* W = params;
    const float* b = params + (int64_t)nc * dim;
    if (tid < LP_ROWS) t.lab[tid] = -1;
    lp_load_rows(t, x, nullptr, first, count, nq, dim);
    lp_row_stats(t, W, b, nc, dim);
    float best = -1.f;
    int best_c = 0;
    for (int c0 = 0; c0 < nc; c0 += LP_CH) {
        const int ncc = min(LP_CH, nc - c0);
        if (nc > LP_CH) lp_logits(t, W, b, c0, nc, dim);
        for (int i = tid; i < LP_ROWS * LP_CH; i += LP_THREADS) {
            const int r = i / LP_CH, j = i - r * LP_CH;
            if (r < count && j < ncc) {
                const float p = lp_prob(t, r, t.L[r * LP_LDL + j]);
                t.L[r * LP_LDL + j] = p;
                probs[(first + r) * nc + c0 + j] = p;
            }
        }
        __syncthreads();
        if (tid < count)   // argmax in ascending class order, lowest class on ties
            for (int j = 0; j < ncc; ++j) {
                const float p = t.L[tid * LP_LDL + j];
                if (p > best) { best = p; best_c = c0 + j; }
            }
        __syncthreads();
    }
    if (tid < count) pred[first + tid] = best_c;
}

static bool lp_dim_ok(int dim) { return dim >= 32 && dim <= LP_MAX_DIM && dim % 32 == 0; }

static bool lp_finite_nonneg(float f) { return f >= 0.f && f <= 3.402823466e38f; }   // NaN and +inf fail

static int lp_check(const msst_linprobe_dims* d, const char* who) {
    MSST_REQUIRE(d, "%s: dims must be set", who);
    MSST_REQUIRE(lp_dim_ok(d->dim), "%s: dim=%d must be a multiple of 32 in [32, %d]", who, d->dim, LP_MAX_DIM);
    MSST_REQUIRE(d->nc >= 1 && d->nc <= LP_MAX_CLASSES, "%s: nc=%d outside [1, %d]", who, d->nc, LP_MAX_CLASSES);
    MSST_REQUIRE(d->heads >= 1 && d->heads <= MSST_LINPROBE_MAX_HEADS, "%s: heads=%d outside [1, %d]", who, d->heads, MSST_LINPROBE_MAX_HEADS);
    MSST_REQUIRE(d->n >= 1 && d->n < 2147483648LL, "%s: n=%lld rows outside [1, 2^31)", who, (long long)d->n);
    MSST_REQUIRE(d->batch >= 1, "%s: batch=%d < 1", who, d->batch);
    return MSST_OK;
}

static int lp_smem_setup(const void* kernel, PerDeviceOnce& once) {
    if (once.first()) MSST_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LP_SMEM_MAX));
    return MSST_OK;
}

}  // namespace msst
using namespace msst;

extern "C" int64_t msst_linprobe_workspace(const msst_linprobe_dims* d) {
    if (lp_check(d, "linprobe_workspace") != MSST_OK) return -1;
    return ceil_div(d->batch, LP_ROWS) * d->heads * ((int64_t)d->nc * d->dim + d->nc + 1) * 4;
}

extern "C" int msst_linprobe_grad(const msst_linprobe_dims* d, const float* x, const int64_t* labels, const int64_t* index,
                                  const float* params, float* workspace, msst_stream_t stream) {
    if (int rc = lp_check(d, "linprobe_grad")) return rc;
    MSST_REQUIRE(x && labels && index && params && workspace, "linprobe_grad: x / labels / index / params / workspace must be set");
    static PerDeviceOnce once;
    if (int rc = lp_smem_setup((const void*)linprobe_grad_kernel, once)) return rc;
    const dim3 grid((unsigned)ceil_div(d->batch, LP_ROWS), (unsigned)d->heads);
    linprobe_grad_kernel<<<grid, LP_THREADS, lp_smem(d->dim), (cudaStream_t)stream>>>(*d, x, labels, index, params, workspace);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

extern "C" int msst_linprobe_update(const msst_linprobe_dims* d, const float* workspace, float* params, float* m, float* v,
                                    float* loss_sum, msst_stream_t stream) {
    if (int rc = lp_check(d, "linprobe_update")) return rc;
    MSST_REQUIRE(d->step >= 1, "linprobe_update: step=%d must be >= 1", d->step);
    for (int h = 0; h < d->heads; ++h)
        MSST_REQUIRE(lp_finite_nonneg(d->lr[h]) && lp_finite_nonneg(d->wd[h]), "linprobe_update: lr[%d] / wd[%d] must be finite and >= 0", h, h);
    MSST_REQUIRE(workspace && params && m && v && loss_sum, "linprobe_update: workspace / params / m / v / loss_sum must be set");
    LpUpdate u{};
    u.a.b1 = 0.9f; u.a.b2 = 0.999f; u.a.omb1 = (float)(1.0 - 0.9); u.a.omb2 = (float)(1.0 - 0.999); u.a.eps = 1e-8f; u.a.clamp = 0.f; u.a.gscale = 1.f; u.a.decoupled = 1; u.a.step_dev = nullptr;
    u.a.inv_bc1 = (float)(1.0 / (1.0 - pow(0.9, (double)d->step)));          // bias corrections as msst_adam_step forms them
    u.a.inv_sqrt_bc2 = (float)(1.0 / sqrt(1.0 - pow(0.999, (double)d->step)));
    for (int h = 0; h < d->heads; ++h) { u.lr[h] = d->lr[h]; u.wd[h] = d->wd[h]; }
    u.heads = d->heads; u.slices = (int)ceil_div(d->batch, LP_ROWS); u.batch = d->batch;
    u.P = (int64_t)d->nc * d->dim + d->nc;
    int64_t blocks = ceil_div(u.heads * u.P, 256);
    if (blocks > 8 * kNumSMs) blocks = 8 * kNumSMs;
    linprobe_update_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(u, workspace, params, m, v, loss_sum);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

extern "C" int msst_linprobe_predict(int64_t n_query, int dim, int nc, const float* x, const float* params, float* probs, int64_t* pred,
                                     msst_stream_t stream) {
    MSST_REQUIRE(lp_dim_ok(dim), "linprobe_predict: dim=%d must be a multiple of 32 in [32, %d]", dim, LP_MAX_DIM);
    MSST_REQUIRE(nc >= 1 && nc <= LP_MAX_CLASSES, "linprobe_predict: nc=%d outside [1, %d]", nc, LP_MAX_CLASSES);
    MSST_REQUIRE(n_query >= 1 && n_query < 2147483648LL, "linprobe_predict: n_query=%lld outside [1, 2^31)", (long long)n_query);
    MSST_REQUIRE(x && params && probs && pred, "linprobe_predict: x / params / probs / pred must be set");
    static PerDeviceOnce once;
    if (int rc = lp_smem_setup((const void*)linprobe_predict_kernel, once)) return rc;
    linprobe_predict_kernel<<<(unsigned)ceil_div(n_query, LP_ROWS), LP_THREADS, lp_smem(dim), (cudaStream_t)stream>>>(n_query, dim, nc, x,
                                                                                                                  params, probs, pred);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}
