// k-nearest-neighbour probing of embeddings (msst_knn_prepare / msst_knn_topk / msst_knn_vote, include/msst.h): cosine similarity
// between fp32 feature rows, the k best references of every query kept on chip, a weighted class vote.
//
//   knn_prepare_kernel  y = x / max(||x||, 1e-12) in fp32 (F.normalize), split y = hi + mid + lo into three bf16 parts, written as one
//                       bf16 row [hi | mid | lo] of 3*D elements: the operand format of the search kernel
//   knn_topk_kernel     persistent warp-specialised CTA (warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM allocator, warps 4-7 =
//                       selection).  A CTA owns 128 queries at a time and streams the references past them in tiles of 128 rows: per
//                       32-element k-block one ring stage holds the three parts of both sides (SWIZZLE_64B boxes, 6 x 8 KB).  The six
//                       products a_i . b_j with i + j <= 2 give fp32 accuracy (bound: DESIGN.md §3): hi . hi accumulates in one TMEM
//                       accumulator, the five small products in a second one, so the truncating tensor-core accumulation rounds the
//                       many small updates at their own magnitude (~2^-8 of the score), not at the score's; the selection adds the two.
//                       Two such pairs, so the MMAs of reference tile j + 1 overlap the selection on tile j.  The
//                       selection thread of query row r reads its row with tcgen05.ld and compares every score with the row's k-th best
//                       (a register); the rare winners are inserted into the row's sorted list in shared memory.
//   knn_vote_kernel     one warp per query: w_j = exp((s_j - s_0) / T), probs = per-class sums of w / sum of w, pred = argmax
//
// Order: (score descending, reference index ascending).  References arrive in ascending index, so a candidate that only ties the k-th
// best is rejected (strict >) and an inserted one goes behind every equal score already in the list.  A query's result depends only on
// its own row and the reference set: the reference tiling is fixed, every score is one accumulator element summed in a fixed order, and
// no atomics are used -- so it is bitwise independent of the query chunking and of the CTA that ran it.
#include "common.cuh"
#include "ptx.cuh"
#include <cuda.h>

namespace msst {
using namespace ptx;

int make_tmap_nd(CUtensorMap* m, const void* base, int elem_bytes, int rank, const int64_t* dims, const int64_t* strides, const int* box,
                 int swizzle_bytes);   // gemm_bf16.cu

constexpr int KN_M = 128;                         // queries per tile: UMMA M, TMEM lane = query row
constexpr int KN_N = 128;                         // references per tile: UMMA N
constexpr int KN_KB = 32;                         // elements per k-block: one 64-byte SWIZZLE_64B row
constexpr uint32_t KN_PART = 128 * KN_KB * 2;     // one part's [128 rows][32] box: 8 KB
constexpr uint32_t KN_STAGE = 6 * KN_PART;        // query hi / mid / lo + reference hi / mid / lo: 48 KB
constexpr int KN_MAX_STAGES = 4;
constexpr int KN_THREADS = 256;                   // TMA, MMA, TMEM-alloc, spare + 4 selection warps
constexpr uint32_t KN_TMEM_COLS = 4 * KN_N;       // two buffers x (hi . hi accumulator, small-product accumulator), fp32
constexpr int KN_MAX_K = 64, KN_MAX_DIM = 256, KN_MAX_CLASSES = 256;
constexpr int KN_SMEM_MAX = 227 * 1024;

struct alignas(8) KnnBars {
    uint64_t full[KN_MAX_STAGES], empty[KN_MAX_STAGES], tmem_full[2], tmem_empty[2];
    uint32_t tmem_base;
};
constexpr uint32_t KN_BARS_BYTES = 128;
static_assert(sizeof(KnnBars) <= KN_BARS_BYTES, "barrier block");

struct KnnParams {
    int64_t nq; int n_ref, dim, k, stages, q_tiles, r_tiles;
    float* scores; int64_t* index;
};

__global__ void __launch_bounds__(256) knn_prepare_kernel(const float* __restrict__ x, int64_t n, int dim, __nv_bfloat16* __restrict__ out) {
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const float* xr = x + row * dim;
    float v[KN_MAX_DIM / 32];
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < KN_MAX_DIM / 32; ++i) {
        const int c = lane + 32 * i;
        v[i] = c < dim ? xr[c] : 0.f;
        ss = fmaf(v[i], v[i], ss);
    }
    const float nrm = fmaxf(sqrtf(warp_sum(ss)), 1e-12f);
    __nv_bfloat16* o = out + row * 3 * dim;
#pragma unroll
    for (int i = 0; i < KN_MAX_DIM / 32; ++i) {
        const int c = lane + 32 * i;
        if (c >= dim) break;
        const float y = __fdiv_rn(v[i], nrm);
        const __nv_bfloat16 h = __float2bfloat16_rn(y);
        const float r = __fsub_rn(y, __bfloat162float(h));          // exact: y and h agree in their leading bits
        const __nv_bfloat16 m = __float2bfloat16_rn(r);
        const __nv_bfloat16 l = __float2bfloat16_rn(__fsub_rn(r, __bfloat162float(m)));
        o[c] = h; o[dim + c] = m; o[2 * dim + c] = l;
    }
}

// inserts (s, idx) into the row's list (column `row` of [k][KN_M]) behind every entry with score >= s; returns the new k-th best score
__device__ __forceinline__ float knn_insert(float* ls, int* li, int k, float s, int idx) {
    int pos = k - 1;
    while (pos > 0) {
        const float prev = ls[(pos - 1) * KN_M];
        if (prev >= s) break;
        ls[pos * KN_M] = prev;
        li[pos * KN_M] = li[(pos - 1) * KN_M];
        --pos;
    }
    ls[pos * KN_M] = s;
    li[pos * KN_M] = idx;
    return ls[(k - 1) * KN_M];
}

__global__ void __launch_bounds__(KN_THREADS, 1)
knn_topk_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_r, const KnnParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    KnnBars* bars = reinterpret_cast<KnnBars*>(smem + (size_t)p.stages * KN_STAGE);
    float* lsc = reinterpret_cast<float*>(smem + (size_t)p.stages * KN_STAGE + KN_BARS_BYTES);   // [k][KN_M] scores
    int* lix = reinterpret_cast<int*>(lsc + (size_t)p.k * KN_M);                                // [k][KN_M] reference indices
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nkb = p.dim / KN_KB;

    if (warp == 0 && elect_one()) { prefetch_tmap(&tma_q); prefetch_tmap(&tma_r); }
    if (warp == 1 && elect_one()) {
        for (int s = 0; s < KN_MAX_STAGES; ++s) { mbar_init(&bars->full[s], 1); mbar_init(&bars->empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&bars->tmem_full[s], 1); mbar_init(&bars->tmem_empty[s], 4); }
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc(&bars->tmem_base, KN_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp == 0) {
        // ===== TMA producer: per (query tile, reference tile, k-block) one stage with the three parts of both sides =====
        if (elect_one()) {
            int stage = 0; uint32_t phase = 0;
            for (int qt = blockIdx.x; qt < p.q_tiles; qt += gridDim.x)
                for (int rt = 0; rt < p.r_tiles; ++rt)
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait(&bars->empty[stage], phase ^ 1);
                        uint8_t* s = smem + (size_t)stage * KN_STAGE;
                        mbar_arrive_expect_tx(&bars->full[stage], KN_STAGE);
#pragma unroll
                        for (int part = 0; part < 3; ++part) {
                            const int col = part * p.dim + kb * KN_KB;
                            tma_load_2d(s + part * KN_PART, &tma_q, &bars->full[stage], col, qt * KN_M);
                            tma_load_2d(s + (3 + part) * KN_PART, &tma_r, &bars->full[stage], col, rt * KN_N);
                        }
                        if (++stage == p.stages) { stage = 0; phase ^= 1; }
                    }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (single elected thread): scores[128 queries][128 references] = sum of the six part products =====
        if (elect_one()) {
            const uint32_t idesc = make_idesc_bf16(KN_M, KN_N, 0, 0);
            // the six products, small terms last: (hi, hi), (hi, mid), (mid, hi), (mid, mid), (hi, lo), (lo, hi)
            constexpr int kPartA[6] = {0, 0, 1, 1, 0, 2}, kPartB[6] = {0, 1, 0, 1, 2, 0};
            int stage = 0; uint32_t phase = 0; int it = 0;
            for (int qt = blockIdx.x; qt < p.q_tiles; qt += gridDim.x)
                for (int rt = 0; rt < p.r_tiles; ++rt, ++it) {
                    const int acc = it & 1;
                    mbar_wait(&bars->tmem_empty[acc], ((uint32_t)(it >> 1) & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t d_hi = tmem_base + (uint32_t)(acc * 2 * KN_N), d_lo = d_hi + KN_N;
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait(&bars->full[stage], phase);
                        tc_fence_after();
                        const uint32_t s = smem_u32(smem + (size_t)stage * KN_STAGE);
#pragma unroll
                        for (int t = 0; t < 6; ++t) {
                            const uint64_t da = make_smem_desc_sw64(s + kPartA[t] * KN_PART), db = make_smem_desc_sw64(s + (3 + kPartB[t]) * KN_PART);
#pragma unroll
                            for (int ks = 0; ks < 2; ++ks)   // +32 B per UMMA_K = 16 step inside the 64-byte swizzle row
                                umma_bf16(t == 0 ? d_hi : d_lo, da + (uint64_t)(ks * 2), db + (uint64_t)(ks * 2), idesc,
                                          !(kb == 0 && ks == 0 && t <= 1));
                        }
                        umma_commit(&bars->empty[stage]);
                        if (++stage == p.stages) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(&bars->tmem_full[acc]);
                }
        }
    } else if (warp >= 4) {
        // ===== selection: thread = query row (TMEM lane quarter q = warp - 4) =====
        const int q = warp - 4, row = q * 32 + lane;
        float* ls = lsc + row;
        int* li = lix + row;
        int it = 0;
        for (int qt = blockIdx.x; qt < p.q_tiles; qt += gridDim.x) {
            for (int i = 0; i < p.k; ++i) { ls[i * KN_M] = -INFINITY; li[i * KN_M] = -1; }
            float thr = -INFINITY;   // the row's k-th best score so far
            for (int rt = 0; rt < p.r_tiles; ++rt, ++it) {
                const int acc = it & 1;
                mbar_wait(&bars->tmem_full[acc], (uint32_t)(it >> 1) & 1);
                tc_fence_after();
                const int base = rt * KN_N;
                const int lim = min(KN_N, p.n_ref - base);   // rows past the end of the references were zero-filled by TMA
                const uint32_t t_hi = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * 2 * KN_N);
                for (int c = 0; c < KN_N / 32; ++c) {
                    uint32_t vh[32], vl[32];
                    tmem_ld_32x32(t_hi + (uint32_t)(c * 32), vh);
                    tmem_ld_32x32(t_hi + (uint32_t)(KN_N + c * 32), vl);
                    tmem_ld_wait();
#pragma unroll
                    for (int t = 0; t < 32; ++t) {
                        const float s = __fadd_rn(__uint_as_float(vh[t]), __uint_as_float(vl[t]));
                        if (s > thr && c * 32 + t < lim) thr = knn_insert(ls, li, p.k, s, base + c * 32 + t);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->tmem_empty[acc]);
            }
            const int64_t qrow = (int64_t)qt * KN_M + row;
            if (qrow < p.nq) {
                for (int i = 0; i < p.k; ++i) {
                    p.scores[qrow * p.k + i] = ls[i * KN_M];
                    p.index[qrow * p.k + i] = (int64_t)li[i * KN_M];
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, KN_TMEM_COLS); }
}

// one warp per query; labels outside [0, nc) and indices outside [0, n_ref) carry no vote (their weight still counts in the sum)
constexpr int KV_WARPS = 8;
__global__ void __launch_bounds__(KV_WARPS * 32) knn_vote_kernel(int64_t nq, int k, int64_t n_ref, const float* __restrict__ scores,
                                                                 const int64_t* __restrict__ index, const int64_t* __restrict__ labels,
                                                                 int nc, float temperature, float* __restrict__ probs, int64_t* __restrict__ pred) {
    __shared__ float s_acc[KV_WARPS][KN_MAX_CLASSES];
    __shared__ float s_w[KV_WARPS][KN_MAX_K];
    __shared__ int s_c[KV_WARPS][KN_MAX_K];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t qi = (int64_t)blockIdx.x * KV_WARPS + warp;
    if (qi >= nq) return;   // warp-uniform; the kernel synchronises warps only
    float* a = s_acc[warp];
    for (int c = lane; c < nc; c += 32) a[c] = 0.f;
    const float* sr = scores + qi * k;
    const float s0 = sr[0];
    for (int j = lane; j < k; j += 32) {
        s_w[warp][j] = expf(__fdiv_rn(__fsub_rn(sr[j], s0), temperature));   // <= 1: the top score is subtracted first
        const int64_t r = index[qi * k + j];
        const int64_t lab = (r >= 0 && r < n_ref) ? labels[r] : -1;
        s_c[warp][j] = (lab >= 0 && lab < nc) ? (int)lab : -1;
    }
    __syncwarp();
    float z = 0.f;
    if (lane == 0) {   // ascending neighbour order: fixed summation order
        for (int j = 0; j < k; ++j) {
            const float w = s_w[warp][j];
            z = __fadd_rn(z, w);
            if (s_c[warp][j] >= 0) a[s_c[warp][j]] = __fadd_rn(a[s_c[warp][j]], w);
        }
    }
    __syncwarp();
    z = __shfl_sync(0xffffffffu, z, 0);
    float best = -1.f;
    int best_c = nc;
    for (int c = lane; c < nc; c += 32) {
        const float pc = __fdiv_rn(a[c], z);
        probs[qi * nc + c] = pc;
        if (pc > best) { best = pc; best_c = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {   // argmax, lowest class on ties
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oc = __shfl_xor_sync(0xffffffffu, best_c, o);
        if (ob > best || (ob == best && oc < best_c)) { best = ob; best_c = oc; }
    }
    if (lane == 0) pred[qi] = best_c;
}

static bool knn_dim_ok(int dim) { return dim >= 32 && dim <= KN_MAX_DIM && dim % 32 == 0; }

static size_t knn_topk_smem(int k, int stages) { return 1024 + (size_t)stages * KN_STAGE + KN_BARS_BYTES + (size_t)k * KN_M * 8; }

}  // namespace msst
using namespace msst;

extern "C" int msst_knn_prepare(const float* x, int64_t n, int dim, void* out, msst_stream_t stream) {
    MSST_REQUIRE(knn_dim_ok(dim), "knn_prepare: dim=%d must be a multiple of 32 in [32, %d]", dim, KN_MAX_DIM);
    MSST_REQUIRE(n >= 1 && n < 2147483647LL, "knn_prepare: n=%lld rows outside [1, 2^31)", (long long)n);
    MSST_REQUIRE(x && out, "knn_prepare: x / out must be set");
    knn_prepare_kernel<<<(unsigned)ceil_div(n, 8), 256, 0, (cudaStream_t)stream>>>(x, n, dim, reinterpret_cast<__nv_bfloat16*>(out));
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

extern "C" int msst_knn_topk(const msst_knn_dims* d, const void* ref, const void* query, float* scores, int64_t* index, msst_stream_t stream) {
    MSST_REQUIRE(d, "knn_topk: dims must be set");
    MSST_REQUIRE(knn_dim_ok(d->dim), "knn_topk: dim=%d must be a multiple of 32 in [32, %d]", d->dim, KN_MAX_DIM);
    MSST_REQUIRE(d->k >= 1 && d->k <= KN_MAX_K, "knn_topk: k=%d outside [1, %d]", d->k, KN_MAX_K);
    MSST_REQUIRE(d->n_ref >= d->k && d->n_ref < 2147483647LL, "knn_topk: n_ref=%lld must satisfy k=%d <= n_ref < 2^31", (long long)d->n_ref, d->k);
    MSST_REQUIRE(d->n_query >= 1 && d->n_query < 2147483647LL - KN_M, "knn_topk: n_query=%lld outside [1, 2^31 - 128)", (long long)d->n_query);
    MSST_REQUIRE(ref && query && scores && index, "knn_topk: ref / query / scores / index must be set");
    int stages = KN_MAX_STAGES;
    while (stages > 2 && knn_topk_smem(d->k, stages) > (size_t)KN_SMEM_MAX) --stages;
    const size_t smem = knn_topk_smem(d->k, stages);
    MSST_REQUIRE(smem <= (size_t)KN_SMEM_MAX, "knn_topk: %zu bytes of shared memory exceed %d", smem, KN_SMEM_MAX);
    CUtensorMap tq, tr;
    auto map = [](CUtensorMap* m, const void* base, int64_t rows, int dim) {
        const int64_t dims[2] = {3 * (int64_t)dim, rows}, strides[1] = {3 * (int64_t)dim};
        const int box[2] = {KN_KB, 128};
        return make_tmap_nd(m, base, 2, 2, dims, strides, box, 64);
    };
    if (int rc = map(&tq, query, d->n_query, d->dim)) return rc;
    if (int rc = map(&tr, ref, d->n_ref, d->dim)) return rc;
    KnnParams p{};
    p.nq = d->n_query; p.n_ref = (int)d->n_ref; p.dim = d->dim; p.k = d->k; p.stages = stages;
    p.q_tiles = (int)ceil_div(d->n_query, KN_M); p.r_tiles = (int)ceil_div(d->n_ref, KN_N);
    p.scores = scores; p.index = index;
    static PerDeviceOnce once;
    if (once.first()) MSST_CUDA(cudaFuncSetAttribute(knn_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, KN_SMEM_MAX));
    const int grid = p.q_tiles < kNumSMs ? p.q_tiles : kNumSMs;
    knn_topk_kernel<<<grid, KN_THREADS, smem, (cudaStream_t)stream>>>(tq, tr, p);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

extern "C" int msst_knn_vote(int64_t n_query, int k, int64_t n_ref, const float* scores, const int64_t* index, const int64_t* ref_labels,
                             int nc, float temperature, float* probs, int64_t* pred, msst_stream_t stream) {
    MSST_REQUIRE(k >= 1 && k <= KN_MAX_K, "knn_vote: k=%d outside [1, %d]", k, KN_MAX_K);
    MSST_REQUIRE(n_ref >= k && n_ref < 2147483647LL, "knn_vote: n_ref=%lld must satisfy k=%d <= n_ref < 2^31", (long long)n_ref, k);
    MSST_REQUIRE(n_query >= 1, "knn_vote: n_query=%lld < 1", (long long)n_query);
    MSST_REQUIRE(nc >= 1 && nc <= KN_MAX_CLASSES, "knn_vote: nc=%d outside [1, %d]", nc, KN_MAX_CLASSES);
    MSST_REQUIRE(temperature > 0.f, "knn_vote: temperature must be > 0 (+inf: uniform vote)");   // NaN fails too
    MSST_REQUIRE(scores && index && ref_labels && probs && pred, "knn_vote: scores / index / ref_labels / probs / pred must be set");
    knn_vote_kernel<<<(unsigned)ceil_div(n_query, KV_WARPS), KV_WARPS * 32, 0, (cudaStream_t)stream>>>(n_query, k, n_ref, scores, index,
                                                                                                     ref_labels, nc, temperature, probs, pred);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}
