// dfx_build.cu -- building a shard on device: k-means (coarse centroids, PQ codebooks),
// assign + encode, and folding staged rows into contiguous inverted lists.
//
// Replaces `faiss_index.train(x)` (reference distributed_faiss/index.py:217) and
// `faiss_index.add(x)` (index.py:425).  Not on the timed search path (SURVEY.md 8f next-1),
// but required to produce a searchable shard without any CPU fallback.
// faiss semantics restated: Clustering = Lloyd iterations from a random subset, at most
// 256 points per centroid, empty clusters re-seeded from a large one; ProductQuantizer
// trained on residuals of <= 256*ksub training vectors; add = nearest centroid under the
// quantizer's metric, ids sequential, ids ascending inside every list.
#include "dfx_internal.h"
#include "dfx_ptx.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <numeric>
#include <random>

// ------------------------------------------------------------------ small kernels
__global__ void gather_rows_kernel(const float* __restrict__ src, const int32_t* __restrict__ rows,
                                   int64_t n, int d, int col0, int dsrc, float* __restrict__ dst) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * d) return;
    int64_t i = t / d;
    int c = (int)(t - i * d);
    int64_t r = rows ? rows[i] : i;
    dst[t] = src[r * dsrc + col0 + c];
}

__global__ void residual_kernel(const float* __restrict__ x, const float* __restrict__ cent,
                                const int32_t* __restrict__ assign, int64_t n, int d,
                                float* __restrict__ out) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * d) return;
    int64_t i = t / d;
    int c = (int)(t - i * d);
    out[t] = x[t] - cent[(size_t)assign[i] * d + c];
}

__global__ void count_kernel(const int32_t* __restrict__ keys, int64_t n, int32_t* __restrict__ cnt) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicAdd(&cnt[keys[i]], 1);
}

__global__ void iota_kernel(int32_t* p, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = (int32_t)i;
}

// one CTA per centroid: mean of its rows, rows visited in ascending row index (deterministic)
__global__ void centroid_update_kernel(const float* __restrict__ x, int d,
                                       const int32_t* __restrict__ order,
                                       const int32_t* __restrict__ seg_off,
                                       float* __restrict__ cent) {
    const int c = blockIdx.x;
    const int beg = seg_off[c], end = seg_off[c + 1];
    if (end <= beg) return;  // empty: keep the old centroid, handled by the host
    const float inv = 1.0f / (float)(end - beg);
    for (int k = threadIdx.x; k < d; k += blockDim.x) {
        float s = 0.f;
        for (int r = beg; r < end; r++) s += x[(size_t)order[r] * d + k];
        cent[(size_t)c * d + k] = s * inv;
    }
}

__global__ void split_cluster_kernel(float* cent, int d, int empty, int big) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= d) return;
    const float eps = 1.f / 1024.f;
    float v = cent[(size_t)big * d + k];
    if ((k & 1) == 0) {
        cent[(size_t)empty * d + k] = v * (1 + eps);
        cent[(size_t)big * d + k] = v * (1 - eps);
    } else {
        cent[(size_t)empty * d + k] = v * (1 - eps);
        cent[(size_t)big * d + k] = v * (1 + eps);
    }
}

// PQ encode: grid (ceil(n/256), row bytes); code_m = argmin_j l2_seq(r_m, P[m][j]), ties -> smaller
// j.  A thread writes one whole byte of a row: one code at 8 bits, the two codes that share the
// byte at 4 bits (so no two threads write the same byte).  The residual sub-vector lives in
// registers (DS = dsub when it is one of the common sizes).
template <int DS>
__device__ __forceinline__ int pq_encode_one(const float* __restrict__ xi, const float* __restrict__ c,
                                             const float* __restrict__ s_cb, int ksub, int dsub) {
    float best = FLT_MAX;
    int bj = 0;
    if (DS > 0) {
        float r[DS > 0 ? DS : 1];
#pragma unroll
        for (int t = 0; t < DS; t++) r[t] = xi[t] - c[t];
        for (int j = 0; j < ksub; j++) {
            float acc = 0.f;
#pragma unroll
            for (int t = 0; t < DS; t++) {
                float df = r[t] - s_cb[j * DS + t];
                acc = __fmaf_rn(df, df, acc);
            }
            if (acc < best) {
                best = acc;
                bj = j;
            }
        }
    } else {
        for (int j = 0; j < ksub; j++) {
            float acc = 0.f;
            for (int t = 0; t < dsub; t++) {
                float df = (xi[t] - c[t]) - s_cb[j * dsub + t];
                acc = __fmaf_rn(df, df, acc);
            }
            if (acc < best) {
                best = acc;
                bj = j;
            }
        }
    }
    return bj;
}

template <int DS>
__global__ void __launch_bounds__(256)
pq_encode_kernel(const float* __restrict__ x, const float* __restrict__ cent,
                 const int32_t* __restrict__ assign, int64_t n, int d, int M, int ksub, int dsub, int nbits,
                 const float* __restrict__ codebooks, uint8_t* __restrict__ codes) {
    DFX_DYN_SMEM0(float, s_cb);  // [per][ksub][dsub]: the codebooks of the byte's sub-quantizers
    const int per = 8 / nbits;   // codes per byte
    const int b = blockIdx.y, m0 = b * per;
    for (int i = threadIdx.x; i < per * ksub * dsub; i += blockDim.x)
        s_cb[i] = codebooks[(size_t)m0 * ksub * dsub + i];
    __syncthreads();
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* xi = x + i * d + m0 * dsub;
    const float* c = cent + (size_t)assign[i] * d + m0 * dsub;
    const int c0 = pq_encode_one<DS>(xi, c, s_cb, ksub, dsub);
    const int64_t rb = (int64_t)M * nbits / 8;
    if (nbits == 8) {
        codes[i * rb + b] = (uint8_t)c0;
    } else {
        const int c1 = pq_encode_one<DS>(xi + dsub, c + dsub, s_cb + ksub * dsub, ksub, dsub);
        codes[i * rb + b] = dfx_pq4_byte(c0, c1);
    }
}

// tvals[i] = sum_m ( |p_m|^2 + 2 <c_m, p_m> ), sequential in m (oracle orc_pq_tvals)
__global__ void pq_tvals_kernel(const uint8_t* __restrict__ codes, const int32_t* __restrict__ list_of,
                                const int64_t* __restrict__ list_off, int64_t nlist, int64_t n, int d,
                                int M, int ksub, int dsub, int nbits, const float* __restrict__ codebooks,
                                const float* __restrict__ cent, float* __restrict__ tvals) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t l;
    if (list_of) {
        l = list_of[i];
    } else {  // list-sorted storage: binary search the list owning row i
        int64_t lo = 0, hi = nlist;
        while (hi - lo > 1) {
            int64_t mid = (lo + hi) >> 1;
            if (list_off[mid] <= i) lo = mid; else hi = mid;
        }
        l = lo;
    }
    const float* c = cent + (size_t)l * d;
    const uint8_t* row = codes + i * ((int64_t)M * nbits / 8);
    float t = 0.f;
    for (int m = 0; m < M; m++) {
        const float* p = codebooks + ((size_t)m * ksub + dfx_pq_code(row, m, nbits)) * dsub;
        float ipcp = 0.f, ippp = 0.f;
        for (int tt = 0; tt < dsub; tt++) ipcp = __fmaf_rn(c[m * dsub + tt], p[tt], ipcp);
        for (int tt = 0; tt < dsub; tt++) ippp = __fmaf_rn(p[tt], p[tt], ippp);
        float tm = __fmaf_rn(2.f, ipcp, ippp);
        t = t + tm;
    }
    tvals[i] = t;
}

__global__ void sq_encode_kernel(const float* __restrict__ x, const float* __restrict__ cent,
                                 const int32_t* __restrict__ assign, int64_t n, int d,
                                 __half* __restrict__ codes) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * d) return;
    int64_t i = t / d;
    int c = (int)(t - i * d);
    codes[t] = __float2half_rn(x[t] - cent[(size_t)assign[i] * d + c]);
}

// list id of every row of the list-sorted storage
__global__ void expand_lists_kernel(const int64_t* __restrict__ list_off, int64_t nlist, int64_t n,
                                    int32_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t lo = 0, hi = nlist;
    while (hi - lo > 1) {
        int64_t mid = (lo + hi) >> 1;
        if (list_off[mid] <= i) lo = mid; else hi = mid;
    }
    out[i] = (int32_t)lo;
}

// new[i] = (src < n_sorted ? old_sorted[src] : pending[src - n_sorted]) in 4-byte words
__global__ void gather_words_kernel(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b,
                                    int64_t n_a, const int32_t* __restrict__ order, int64_t n,
                                    int words, uint32_t* __restrict__ out) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * words) return;
    int64_t i = t / words;
    int w = (int)(t - i * words);
    int64_t src = order[i];
    out[t] = (src < n_a) ? a[src * words + w] : b[(src - n_a) * words + w];
}
__global__ void gather_ids_kernel(const int32_t* __restrict__ old_ids, int64_t n_a,
                                  const int32_t* __restrict__ order, int64_t n,
                                  int32_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t src = order[i];
    out[i] = (src < n_a) ? old_ids[src] : (int32_t)src;  // pending row j gets id n_a + j == src
}
__global__ void widen_kernel(const int32_t* __restrict__ in, int64_t n, int64_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}

static inline unsigned blocks_for(int64_t n, int t) { return (unsigned)dfx_ceil_div(n, t); }

// ------------------------------------------------------------------ assign
void dfx_assign_impl(dfx_index* idx, const float* d_cent, const float* d_cnorm, int64_t nlist,
                     int metric, int d, int64_t n, const float* d_x, int32_t* d_assign,
                     cudaStream_t st) {
    if (n <= 0) return;
    if (idx->tc_enabled && dfx_tc_supported(d) && nlist >= 1024) {
        dfx_tc_assign(idx, d, d_cent, d_cnorm, nlist, metric, n, d_x, d_assign, st);
        return;
    }
    idx->w_best.reserve((size_t)n * 8);
    dfx_launch_assign_fused(d_x, n, d_cent, d_cnorm, nlist, d, metric,
                            idx->w_best.as<unsigned long long>(), d_assign, st);
}

// ------------------------------------------------------------------ k-means on device
static void kmeans_device(dfx_index* idx, int d, int64_t n, const float* d_x, int64_t k, int niter,
                          uint64_t seed, float* d_cent, cudaStream_t st) {
    DFX_REQUIRE(n >= k, "k-means: need at least as many training points as centroids (" +
                            std::to_string(n) + " < " + std::to_string(k) + ")");
    DFX_REQUIRE(n < (1ll << 31), "k-means: too many training points");
    // init = random subset without replacement
    std::vector<int32_t> perm((size_t)n);
    std::iota(perm.begin(), perm.end(), 0);
    std::mt19937_64 rng(seed);
    for (int64_t i = 0; i < k; i++) {
        int64_t j = i + (int64_t)(rng() % (uint64_t)(n - i));
        std::swap(perm[(size_t)i], perm[(size_t)j]);
    }
    DevBuf d_sel, d_assign, d_order_in, d_order, d_keys_out, d_cnt, d_off, d_cnorm, d_tmp;
    d_sel.reserve((size_t)k * 4);
    DFX_CUDA(cudaMemcpyAsync(d_sel.p, perm.data(), (size_t)k * 4, cudaMemcpyHostToDevice, st));
    DFX_LAUNCH(gather_rows_kernel, blocks_for(k * d, 256), 256, 0, st, d_x, d_sel.as<int32_t>(), k, d,
               0, d, d_cent);
    DFX_CUDA(cudaStreamSynchronize(st));

    d_assign.reserve((size_t)n * 4);
    d_order_in.reserve((size_t)n * 4);
    d_order.reserve((size_t)n * 4);
    d_keys_out.reserve((size_t)n * 4);
    d_cnt.reserve((size_t)(k + 1) * 4);
    d_off.reserve((size_t)(k + 1) * 4);
    d_cnorm.reserve((size_t)k * 4);
    DFX_LAUNCH(iota_kernel, blocks_for(n, 256), 256, 0, st, d_order_in.as<int32_t>(), n);
    int bits = 1;
    while ((1ll << bits) < k) bits++;
    size_t tmp_sort = 0, tmp_scan = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, d_assign.as<int32_t>(), d_keys_out.as<int32_t>(),
                                    d_order_in.as<int32_t>(), d_order.as<int32_t>(), (int)n, 0, bits, st);
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_scan, d_cnt.as<int32_t>(), d_off.as<int32_t>(),
                                  (int)(k + 1), st);
    d_tmp.reserve(std::max(tmp_sort, tmp_scan));
    std::vector<int32_t> h_cnt((size_t)k + 1);

    for (int it = 0; it < niter; it++) {
        dfx_launch_row_norms(d_cent, k, d, d_cnorm.as<float>(), st);
        dfx_assign_impl(idx, d_cent, d_cnorm.as<float>(), k, DFX_METRIC_L2, d, n, d_x,
                        d_assign.as<int32_t>(), st);
        DFX_CUDA(cudaMemsetAsync(d_cnt.p, 0, (size_t)(k + 1) * 4, st));
        DFX_LAUNCH(count_kernel, blocks_for(n, 256), 256, 0, st, d_assign.as<int32_t>(), n,
                   d_cnt.as<int32_t>());
        size_t tb = d_tmp.cap;
        DFX_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp.p, tb, d_cnt.as<int32_t>(), d_off.as<int32_t>(),
                                               (int)(k + 1), st));
        tb = d_tmp.cap;
        DFX_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp.p, tb, d_assign.as<int32_t>(),
                                                 d_keys_out.as<int32_t>(), d_order_in.as<int32_t>(),
                                                 d_order.as<int32_t>(), (int)n, 0, bits, st));
        g_dfx_launches.fetch_add(2, std::memory_order_relaxed);
        int threads = d >= 128 ? 128 : (d >= 64 ? 64 : 32);
        DFX_LAUNCH(centroid_update_kernel, (unsigned)k, threads, 0, st, d_x, d, d_order.as<int32_t>(),
                   d_off.as<int32_t>(), d_cent);
        // empty clusters: split the currently largest (host decides, like the oracle)
        DFX_CUDA(cudaMemcpyAsync(h_cnt.data(), d_cnt.p, (size_t)k * 4, cudaMemcpyDeviceToHost, st));
        DFX_CUDA(cudaStreamSynchronize(st));
        for (int64_t c = 0; c < k; c++) {
            if (h_cnt[(size_t)c] != 0) continue;
            int64_t big = std::max_element(h_cnt.begin(), h_cnt.begin() + k) - h_cnt.begin();
            if (h_cnt[(size_t)big] < 2) break;
            DFX_LAUNCH(split_cluster_kernel, blocks_for(d, 128), 128, 0, st, d_cent, d, (int)c, (int)big);
            h_cnt[(size_t)c] = h_cnt[(size_t)big] / 2;
            h_cnt[(size_t)big] -= h_cnt[(size_t)c];
        }
    }
    DFX_CUDA(cudaStreamSynchronize(st));
}

// ------------------------------------------------------------------ train
void dfx_train_impl(dfx_index* idx, int64_t n, const float* d_x, cudaStream_t st) {
    const int kind = idx->cfg.kind;
    if (kind == DFX_FLAT) {
        idx->trained = true;
        return;
    }
    const int d = idx->cfg.d;
    const int64_t nlist = idx->cfg.nlist;
    DFX_REQUIRE(n >= nlist, "train: need at least nlist=" + std::to_string(nlist) +
                                " training vectors, got " + std::to_string(n));
    const int niter = idx->kmeans_niter > 0 ? idx->kmeans_niter : 25;
    const uint64_t seed = idx->train_seed;

    // faiss Clustering: at most 256 points per centroid (random subset)
    const float* xt = d_x;
    int64_t nt = n;
    DevBuf sub;
    const int64_t maxpts = (int64_t)idx->max_points_per_centroid * nlist;
    if (n > maxpts) {
        std::vector<int32_t> perm((size_t)n);
        std::iota(perm.begin(), perm.end(), 0);
        std::mt19937_64 rng(seed ^ 0x5bd1e995u);
        for (int64_t i = 0; i < maxpts; i++) {
            int64_t j = i + (int64_t)(rng() % (uint64_t)(n - i));
            std::swap(perm[(size_t)i], perm[(size_t)j]);
        }
        DevBuf d_sel;
        d_sel.reserve((size_t)maxpts * 4);
        DFX_CUDA(cudaMemcpyAsync(d_sel.p, perm.data(), (size_t)maxpts * 4, cudaMemcpyHostToDevice, st));
        sub.reserve((size_t)maxpts * d * 4);
        DFX_LAUNCH(gather_rows_kernel, blocks_for(maxpts * d, 256), 256, 0, st, d_x,
                   d_sel.as<int32_t>(), maxpts, d, 0, d, sub.as<float>());
        DFX_CUDA(cudaStreamSynchronize(st));
        xt = sub.as<float>();
        nt = maxpts;
    }
    idx->centroids.reserve((size_t)nlist * d * 4);
    idx->cnorm.reserve((size_t)nlist * 4);
    kmeans_device(idx, d, nt, xt, nlist, niter, seed, idx->centroids.as<float>(), st);
    dfx_launch_row_norms(idx->centroids.as<float>(), nlist, d, idx->cnorm.as<float>(), st);
    dfx_tc_prepare_centroids(idx, st);

    if (kind == DFX_IVF_PQ) {
        const int M = idx->M, ksub = idx->ksub, dsub = idx->dsub;
        int64_t ns = std::min<int64_t>(nt, 256ll * ksub);
        DFX_REQUIRE(ns >= ksub, "train: need at least " + std::to_string(ksub) + " vectors for PQ");
        DevBuf d_assign, d_res, d_subv, d_cb;
        d_assign.reserve((size_t)ns * 4);
        d_res.reserve((size_t)ns * d * 4);
        d_subv.reserve((size_t)ns * dsub * 4);
        dfx_assign_impl(idx, idx->centroids.as<float>(), idx->cnorm.as<float>(), nlist, idx->cfg.metric,
                        d, ns, xt, d_assign.as<int32_t>(), st);
        DFX_LAUNCH(residual_kernel, blocks_for(ns * d, 256), 256, 0, st, xt, idx->centroids.as<float>(),
                   d_assign.as<int32_t>(), ns, d, d_res.as<float>());
        idx->codebooks.reserve((size_t)M * ksub * dsub * 4);
        idx->cbT_valid = false;
        for (int m = 0; m < M; m++) {
            DFX_LAUNCH(gather_rows_kernel, blocks_for(ns * dsub, 256), 256, 0, st, d_res.as<float>(),
                       (const int32_t*)nullptr, ns, dsub, m * dsub, d, d_subv.as<float>());
            kmeans_device(idx, dsub, ns, d_subv.as<float>(), ksub, niter, seed + 1 + m,
                          idx->codebooks.as<float>() + (size_t)m * ksub * dsub, st);
        }
    }
    // an empty, trained index
    idx->h_list_off.assign((size_t)nlist + 1, 0);
    idx->list_off.reserve((size_t)(nlist + 1) * 8);
    DFX_CUDA(cudaMemsetAsync(idx->list_off.p, 0, (size_t)(nlist + 1) * 8, st));
    DFX_CUDA(cudaStreamSynchronize(st));
    idx->n_sorted = 0;
    idx->n_pending = 0;
    idx->trained = true;
}

// ------------------------------------------------------------------ add
static void ensure_pending(dfx_index* idx, int64_t need, cudaStream_t st) {
    if (need <= idx->p_cap) return;
    int64_t cap = std::max<int64_t>(need, idx->p_cap * 2);
    if (idx->reserve_hint > idx->n_sorted)
        cap = std::max<int64_t>(cap, std::min<int64_t>(idx->reserve_hint - idx->n_sorted, need * 64));
    const size_t rb = idx->row_bytes();
    idx->p_list.reserve((size_t)cap * 4, (size_t)idx->n_pending * 4, st);
    idx->p_payload.reserve((size_t)cap * rb, (size_t)idx->n_pending * rb, st);
    if (idx->cfg.kind == DFX_IVF_PQ)
        idx->p_tvals.reserve((size_t)cap * 4, (size_t)idx->n_pending * 4, st);
    idx->p_cap = cap;
}

void dfx_add_impl(dfx_index* idx, int64_t n, const float* d_x, cudaStream_t st) {
    if (n <= 0) return;
    const int kind = idx->cfg.kind;
    const int d = idx->cfg.d;
    DFX_REQUIRE(idx->ntotal() + n < (1ll << 31), "a shard holds at most 2^31-1 vectors");
    if (kind == DFX_FLAT) {
        const int64_t N = idx->n_sorted;
        if ((size_t)(N + n) * d * 4 > idx->payload.cap) {
            int64_t cap = std::max<int64_t>({N + n, 2 * N, idx->reserve_hint});
            idx->payload.reserve((size_t)cap * d * 4, (size_t)N * d * 4, st);
            if (idx->cfg.metric == DFX_METRIC_L2) idx->xnorm.reserve((size_t)cap * 4, (size_t)N * 4, st);
        }
        DFX_CUDA(cudaMemcpyAsync(idx->payload.as<float>() + N * d, d_x, (size_t)n * d * 4,
                                 cudaMemcpyDeviceToDevice, st));
        if (idx->cfg.metric == DFX_METRIC_L2)
            dfx_launch_row_norms(d_x, n, d, idx->xnorm.as<float>() + N, st);
        idx->n_sorted += n;
        return;
    }
    DFX_REQUIRE(idx->trained, "add: index is not trained");
    const int64_t nlist = idx->cfg.nlist;
    ensure_pending(idx, idx->n_pending + n, st);
    int32_t* plist = idx->p_list.as<int32_t>() + idx->n_pending;
    dfx_assign_impl(idx, idx->centroids.as<float>(), idx->cnorm.as<float>(), nlist, idx->cfg.metric, d, n,
                    d_x, plist, st);
    const size_t rb = idx->row_bytes();
    unsigned char* prow = idx->p_payload.as<unsigned char>() + (size_t)idx->n_pending * rb;
    if (kind == DFX_IVF_FLAT) {
        DFX_CUDA(cudaMemcpyAsync(prow, d_x, (size_t)n * rb, cudaMemcpyDeviceToDevice, st));
    } else if (kind == DFX_IVF_PQ) {
        const int M = idx->M, ksub = idx->ksub, dsub = idx->dsub, nbits = idx->nbits;
        dim3 grid(blocks_for(n, 256), (unsigned)rb);  // one thread per (vector, row byte)
        const size_t cb_smem = (size_t)(8 / nbits) * ksub * dsub * 4;
#define DFX_PQ_ENCODE(DS)                                                                       \
    do {                                                                                        \
        auto kern = pq_encode_kernel<DS>;                                                       \
        DFX_LAUNCH(kern, grid, 256, cb_smem, st, d_x, idx->centroids.as<float>(),               \
                   plist, n, d, M, ksub, dsub, nbits, idx->codebooks.as<float>(), (uint8_t*)prow); \
    } while (0)
        if (dsub == 2) DFX_PQ_ENCODE(2);
        else if (dsub == 4) DFX_PQ_ENCODE(4);
        else if (dsub == 8) DFX_PQ_ENCODE(8);
        else if (dsub == 16) DFX_PQ_ENCODE(16);
        else DFX_PQ_ENCODE(0);
#undef DFX_PQ_ENCODE
        DFX_LAUNCH(pq_tvals_kernel, blocks_for(n, 128), 128, 0, st, (const uint8_t*)prow, plist,
                   (const int64_t*)nullptr, nlist, n, d, M, ksub, dsub, nbits, idx->codebooks.as<float>(),
                   idx->centroids.as<float>(), idx->p_tvals.as<float>() + idx->n_pending);
    } else {  // IVF_SQ16
        DFX_LAUNCH(sq_encode_kernel, blocks_for(n * d, 256), 256, 0, st, d_x, idx->centroids.as<float>(),
                   plist, n, d, (__half*)prow);
    }
    idx->n_pending += n;
}

void dfx_compute_tvals_sorted(dfx_index* idx, cudaStream_t st) {
    const int64_t n = idx->n_sorted;
    idx->tvals.reserve((size_t)std::max<int64_t>(n, 1) * 4);
    if (n == 0) return;
    DFX_LAUNCH(pq_tvals_kernel, blocks_for(n, 128), 128, 0, st, idx->payload.as<uint8_t>(),
               (const int32_t*)nullptr, idx->list_off.as<int64_t>(), idx->cfg.nlist, n, idx->cfg.d,
               idx->M, idx->ksub, idx->dsub, idx->nbits, idx->codebooks.as<float>(), idx->centroids.as<float>(),
               idx->tvals.as<float>());
}

// ------------------------------------------------------------------ finalize: stage -> lists
void dfx_finalize_impl(dfx_index* idx, cudaStream_t st) {
    if (!idx->is_ivf() || idx->n_pending == 0) return;
    if (idx->il) dfx_pq_il_to_rm(idx, st);  // merge happens on the row-major form
    const int64_t na = idx->n_sorted, nb = idx->n_pending, n = na + nb;
    const int64_t nlist = idx->cfg.nlist;
    const size_t rb = idx->row_bytes();
    DFX_REQUIRE(rb % 4 == 0, "row size must be a multiple of 4 bytes");
    DevBuf keys_in, keys_out, order_in, order, cnt, off32, tmp;
    keys_in.reserve((size_t)n * 4);
    keys_out.reserve((size_t)n * 4);
    order_in.reserve((size_t)n * 4);
    order.reserve((size_t)n * 4);
    cnt.reserve((size_t)(nlist + 1) * 4);
    off32.reserve((size_t)(nlist + 1) * 4);
    if (na > 0)
        DFX_LAUNCH(expand_lists_kernel, blocks_for(na, 256), 256, 0, st, idx->list_off.as<int64_t>(),
                   nlist, na, keys_in.as<int32_t>());
    DFX_CUDA(cudaMemcpyAsync(keys_in.as<int32_t>() + na, idx->p_list.p, (size_t)nb * 4,
                             cudaMemcpyDeviceToDevice, st));
    DFX_LAUNCH(iota_kernel, blocks_for(n, 256), 256, 0, st, order_in.as<int32_t>(), n);
    int bits = 1;
    while ((1ll << bits) < nlist) bits++;
    size_t tmp_sort = 0, tmp_scan = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, keys_in.as<int32_t>(), keys_out.as<int32_t>(),
                                    order_in.as<int32_t>(), order.as<int32_t>(), (int)n, 0, bits, st);
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_scan, cnt.as<int32_t>(), off32.as<int32_t>(),
                                  (int)(nlist + 1), st);
    tmp.reserve(std::max(tmp_sort, tmp_scan));
    size_t tb = tmp.cap;
    DFX_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tb, keys_in.as<int32_t>(), keys_out.as<int32_t>(),
                                             order_in.as<int32_t>(), order.as<int32_t>(), (int)n, 0,
                                             bits, st));
    DFX_CUDA(cudaMemsetAsync(cnt.p, 0, (size_t)(nlist + 1) * 4, st));
    DFX_LAUNCH(count_kernel, blocks_for(n, 256), 256, 0, st, keys_in.as<int32_t>(), n, cnt.as<int32_t>());
    tb = tmp.cap;
    DFX_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb, cnt.as<int32_t>(), off32.as<int32_t>(),
                                           (int)(nlist + 1), st));
    g_dfx_launches.fetch_add(2, std::memory_order_relaxed);
    keys_in.release();
    keys_out.release();
    order_in.release();

    // gather into fresh list-sorted storage
    DevBuf new_payload, new_ids, new_tvals;
    new_payload.reserve((size_t)n * rb);
    new_ids.reserve((size_t)n * 4);
    const int words = (int)(rb / 4);
    DFX_LAUNCH(gather_words_kernel, blocks_for(n * words, 256), 256, 0, st, idx->payload.as<uint32_t>(),
               idx->p_payload.as<uint32_t>(), na, order.as<int32_t>(), n, words,
               new_payload.as<uint32_t>());
    DFX_LAUNCH(gather_ids_kernel, blocks_for(n, 256), 256, 0, st, idx->ids.as<int32_t>(), na,
               order.as<int32_t>(), n, new_ids.as<int32_t>());
    if (idx->cfg.kind == DFX_IVF_PQ) {
        new_tvals.reserve((size_t)n * 4);
        DFX_LAUNCH(gather_words_kernel, blocks_for(n, 256), 256, 0, st, idx->tvals.as<uint32_t>(),
                   idx->p_tvals.as<uint32_t>(), na, order.as<int32_t>(), n, 1, new_tvals.as<uint32_t>());
    }
    idx->list_off.reserve((size_t)(nlist + 1) * 8);
    DFX_LAUNCH(widen_kernel, blocks_for(nlist + 1, 256), 256, 0, st, off32.as<int32_t>(), nlist + 1,
               idx->list_off.as<int64_t>());
    idx->h_list_off.resize((size_t)nlist + 1);
    DFX_CUDA(cudaMemcpyAsync(idx->h_list_off.data(), idx->list_off.p, (size_t)(nlist + 1) * 8,
                             cudaMemcpyDeviceToHost, st));
    DFX_CUDA(cudaStreamSynchronize(st));
    std::swap(idx->payload, new_payload);
    std::swap(idx->ids, new_ids);
    if (idx->cfg.kind == DFX_IVF_PQ) std::swap(idx->tvals, new_tvals);
    idx->p_list.release();
    idx->p_payload.release();
    idx->p_tvals.release();
    idx->p_cap = 0;
    idx->n_sorted = n;
    idx->n_pending = 0;
    idx->inv_valid = false;
    dfx_pq_rm_to_il(idx, st);  // IVF-PQ 32 x 8 / 64 x 4 bit: interleaved blocks for the scan (no-op otherwise)
}

// ------------------------------------------------------------------ reconstruct
__global__ void invert_ids_kernel(const int32_t* __restrict__ ids, int64_t n, int32_t* __restrict__ inv) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && ids[i] >= 0) inv[ids[i]] = (int32_t)i;
}

// il != 0 (IVF-PQ interleaved, il = block layout 1 or 2): `inv` holds padded block positions and
// codes are read from the interleaved blocks (dfx_il_byte_of(il, pos%32, m & 31) of block pos/32;
// at 4 bits that byte is the pair of columns m & 31, dfx_il2_pair_code)
__global__ void reconstruct_kernel(int kind, int d, int M, int ksub, int dsub, int nbits, int64_t ntotal,
                                   int64_t nlist, const int64_t* __restrict__ want,
                                   const int32_t* __restrict__ inv, const void* __restrict__ rows,
                                   const int64_t* __restrict__ list_off, const float* __restrict__ cent,
                                   const float* __restrict__ codebooks, int il,
                                   const int64_t* __restrict__ blk_off, float* __restrict__ out,
                                   int64_t tag) {
    const int64_t r = blockIdx.x;
    int64_t id = want[r];
    if (tag >= 0) {
        // exchange ids ((shard tag << 40) | local id, see encode_ids_kernel): decode only the rows
        // this shard owns and leave every other row of `out` untouched
        if (id < 0 || ((id >> 40) & 0xfffff) != tag) return;
        id &= (1ll << 40) - 1;
    }
    if (id < 0 || id >= ntotal) {
        for (int k = threadIdx.x; k < d; k += blockDim.x) out[r * d + k] = __int_as_float(0x7fc00000);
        return;
    }
    const int64_t pos = (kind == DFX_FLAT) ? id : inv[id];
    int64_t l = 0;
    if (kind == DFX_IVF_PQ || kind == DFX_IVF_SQ16) {
        const int64_t* off = il ? blk_off : list_off;
        const int64_t key = il ? (pos >> 5) : pos;
        int64_t lo = 0, hi = nlist;
        while (hi - lo > 1) {
            int64_t mid = (lo + hi) >> 1;
            if (off[mid] <= key) lo = mid; else hi = mid;
        }
        l = lo;
    }
    for (int k = threadIdx.x; k < d; k += blockDim.x) {
        float v;
        if (kind == DFX_FLAT || kind == DFX_IVF_FLAT) {
            v = reinterpret_cast<const float*>(rows)[pos * d + k];
        } else if (kind == DFX_IVF_SQ16) {
            v = cent[(size_t)l * d + k] + __half2float(reinterpret_cast<const __half*>(rows)[pos * d + k]);
        } else {
            int m = k / dsub;
            int code;
            if (il) {
                const uint8_t b = reinterpret_cast<const uint8_t*>(rows)[(pos >> 5) * 1024 + dfx_il_byte_of(il, (int)(pos & 31), m & 31)];
                code = (nbits == 8) ? (int)b : dfx_il2_pair_code(b, m);
            } else {
                code = dfx_pq_code(reinterpret_cast<const uint8_t*>(rows) + pos * ((int64_t)M * nbits / 8), m, nbits);
            }
            v = cent[(size_t)l * d + k] + codebooks[((size_t)m * ksub + code) * dsub + (k - m * dsub)];
        }
        out[r * d + k] = v;
    }
}

void dfx_reconstruct_impl(dfx_index* idx, int64_t n, const int64_t* d_ids, float* d_out,
                          cudaStream_t st, int64_t tag) {
    if (n <= 0) return;
    if (idx->n_pending > 0) dfx_finalize_impl(idx, st);
    const int64_t nt = idx->n_sorted;
    const int il = idx->il ? 2 : 0;  // 0 = row-major, else the block layout
    if (idx->is_ivf() && !idx->inv_valid) {
        idx->inv.reserve((size_t)std::max<int64_t>(nt, 1) * 4);
        const int64_t npos = il ? idx->nblk * 32 : nt;
        if (npos > 0)
            DFX_LAUNCH(invert_ids_kernel, blocks_for(npos, 256), 256, 0, st,
                       il ? idx->il_ids.as<int32_t>() : idx->ids.as<int32_t>(), npos, idx->inv.as<int32_t>());
        idx->inv_valid = true;
    }
    DFX_LAUNCH(reconstruct_kernel, (unsigned)n, 128, 0, st, idx->cfg.kind, idx->cfg.d, idx->M, idx->ksub,
               idx->dsub, idx->nbits, nt, idx->cfg.nlist, d_ids, idx->inv.as<int32_t>(),
               il ? (const void*)idx->il_codes.p : (const void*)idx->payload.p, idx->list_off.as<int64_t>(),
               idx->centroids.as<float>(), idx->codebooks.as<float>(), il, idx->blk_off.as<int64_t>(), d_out, tag);
}
