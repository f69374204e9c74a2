// dfx_search.cu -- the search hot path of one shard on one B200 (sm_100a).
//
// Replaces `self.faiss_index.search(query_batch, top_k)` (reference
// distributed_faiss/index.py:257) for the four builders of index.py:93-100 and
// `IndexClient._aggregate_results` (client.py:265-310):
//   K1a  gemm_values      coarse quantizer / flat contraction, fp32 FFMA, seq-k canonical order
//   K_sel select_rows     exact k-selection (dfx_select.cuh)
//   K3   pq_prep          per-query PQ table  -2<q_m,P[m][j]>  + exact ||q-c||^2 of probed lists
//   K4   scan_pq          inverted-list scan of PQ codes, per-warp k-selection
//   K2/5 scan_rows        inverted-list scan of fp32 rows / fp16 residual codes
//   K6   merge            cross-shard merge (float_maxheap_array_t semantics)
// Arithmetic orders are the canonical ones of oracle/dfx_oracle.c (bit-exact parity).
#include "dfx_internal.h"
#include "dfx_select.cuh"
#include "dfx_topk.cuh"
#include "dfx_ptx.cuh"

// =====================================================================================
// K1a: values GEMM (fp32 FFMA).  acc = fmaf(q[k], x[k], acc), k ascending.
// =====================================================================================
template <int BM, int BN, int BK, int TM, int TN>
__global__ void __launch_bounds__((BM / TM) * (BN / TN))
gemm_values_kernel(const float* __restrict__ Q, int64_t nq, const float* __restrict__ X,
                   const float* __restrict__ xnorm, int64_t ncols, int d, int metric,
                   float* __restrict__ out, int64_t ld_out) {
    constexpr int THREADS = (BM / TM) * (BN / TN);
    __shared__ float sQ[BK][BM + 4];
    __shared__ float sX[BK][BN + 4];
    const int tid = threadIdx.x;
    const int tx = tid % (BN / TN), ty = tid / (BN / TN);
    const int64_t m0 = (int64_t)blockIdx.y * BM;
    const int64_t n0 = (int64_t)blockIdx.x * BN;

    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; i++)
#pragma unroll
        for (int j = 0; j < TN; j++) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < d; k0 += BK) {
        for (int e = tid; e < BM * BK; e += THREADS) {
            int m = e / BK, kk = e % BK;
            int64_t gm = m0 + m;
            int gk = k0 + kk;
            sQ[kk][m] = (gm < nq && gk < d) ? Q[gm * d + gk] : 0.f;
        }
        for (int e = tid; e < BN * BK; e += THREADS) {
            int n = e / BK, kk = e % BK;
            int64_t gn = n0 + n;
            int gk = k0 + kk;
            sX[kk][n] = (gn < ncols && gk < d) ? X[gn * d + gk] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; kk++) {
            float a[TM], b[TN];
#pragma unroll
            for (int i = 0; i < TM; i++) a[i] = sQ[kk][ty * TM + i];
#pragma unroll
            for (int j = 0; j < TN; j++) b[j] = sX[kk][tx * TN + j];
#pragma unroll
            for (int i = 0; i < TM; i++)
#pragma unroll
                for (int j = 0; j < TN; j++) acc[i][j] = __fmaf_rn(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
    // NOTE: zero padding of the k tail adds fmaf(0,0,acc) == acc exactly (acc is never -0 here
    // in a way that matters: acc + (+0) keeps acc), so the canonical order is preserved.
#pragma unroll
    for (int i = 0; i < TM; i++) {
        int64_t gm = m0 + ty * TM + i;
        if (gm >= nq) continue;
#pragma unroll
        for (int j = 0; j < TN; j++) {
            int64_t gn = n0 + tx * TN + j;
            if (gn >= ncols) continue;
            float ip = acc[i][j];
            float v = (metric == DFX_METRIC_IP) ? -ip : __fmaf_rn(-2.f, ip, xnorm[gn]);
            out[gm * ld_out + gn] = v;
        }
    }
}

void dfx_launch_gemm_values(const float* Q, int64_t nq, const float* X, const float* xnorm,
                            int64_t ncols, int d, int metric, float* out, int64_t ld_out,
                            cudaStream_t st) {
    if (nq <= 0 || ncols <= 0) return;
    if (nq <= 16) {
        constexpr int BM = 16, BN = 128, BK = 16, TM = 2, TN = 4;
        dim3 grid((unsigned)dfx_ceil_div(ncols, BN), (unsigned)dfx_ceil_div(nq, BM));
        auto kern = gemm_values_kernel<BM, BN, BK, TM, TN>;
        DFX_LAUNCH(kern, grid, (BM / TM) * (BN / TN), 0, st, Q, nq, X, xnorm, ncols, d, metric, out,
                   ld_out);
    } else {
        constexpr int BM = 128, BN = 128, BK = 8, TM = 8, TN = 8;
        dim3 grid((unsigned)dfx_ceil_div(ncols, BN), (unsigned)dfx_ceil_div(nq, BM));
        auto kern = gemm_values_kernel<BM, BN, BK, TM, TN>;
        DFX_LAUNCH(kern, grid, (BM / TM) * (BN / TN), 0, st, Q, nq, X, xnorm, ncols, d, metric, out,
                   ld_out);
    }
}

// |x|^2 in seq-k order
__global__ void row_norms_kernel(const float* __restrict__ X, int64_t n, int d,
                                 float* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* x = X + i * d;
    float acc = 0.f;
    for (int k = 0; k < d; k++) acc = __fmaf_rn(x[k], x[k], acc);
    out[i] = acc;
}
void dfx_launch_row_norms(const float* X, int64_t n, int d, float* out, cudaStream_t st) {
    if (n <= 0) return;
    DFX_LAUNCH(row_norms_kernel, (unsigned)dfx_ceil_div(n, 128), 128, 0, st, X, n, d, out);
}

// =====================================================================================
// loaders / writers for the selection kernel
// =====================================================================================
struct ColsLoader {  // a row of a values matrix; sec = col_base + column
    const float* vals;
    int64_t ld;
    uint32_t col_base;
    __device__ __forceinline__ uint64_t operator()(int64_t row, int e) const {
        return dfx_comp(vals[row * ld + e], col_base + (uint32_t)e);
    }
};
struct KeysWriter {  // -> int32 keys (+ optional values, + optional composite copy)
    int32_t* keys;
    float* kvals;
    uint64_t* comp;
    int64_t comp_ld;
    int k;
    __device__ __forceinline__ void operator()(int64_t row, int j, uint64_t c) const {
        if (keys) keys[row * k + j] = (c == DFX_COMP_NONE) ? -1 : (int32_t)(uint32_t)c;
        if (kvals) kvals[row * k + j] = (c == DFX_COMP_NONE) ? FLT_MAX : dfx_key2f((uint32_t)(c >> 32));
        if (comp) comp[row * comp_ld + j] = c;
    }
};
struct CompLoader {  // a row of composites
    const uint64_t* comp;
    int64_t ld;
    __device__ __forceinline__ uint64_t operator()(int64_t row, int e) const {
        return comp[row * ld + e];
    }
};
struct ResultWriter {  // composites -> faiss-style (D, I)
    float* D;
    int64_t* I;
    int k;
    int metric;
    float qnorm_add;             // unused (0)
    const float* qnorm;          // FLAT L2: add |q|^2 back and clamp at 0
    __device__ __forceinline__ void operator()(int64_t row, int j, uint64_t c) const {
        if (c == DFX_COMP_NONE) {
            D[row * k + j] = (metric == DFX_METRIC_IP) ? -FLT_MAX : FLT_MAX;
            I[row * k + j] = -1;
        } else {
            float v = dfx_key2f((uint32_t)(c >> 32));
            if (metric == DFX_METRIC_IP) {
                v = -v;
            } else if (qnorm) {
                v = v + qnorm[row];
                v = v < 0.f ? 0.f : v;
            }
            D[row * k + j] = v;
            I[row * k + j] = (int64_t)(uint32_t)c;
        }
    }
};

void dfx_launch_select_cols(const float* vals, int64_t nrows, int n, int64_t ld, int k,
                            uint32_t col_base, int32_t* keys, float* kvals, uint64_t* comp_out,
                            int64_t comp_ld, cudaStream_t st) {
    ColsLoader ldr{vals, ld, col_base};
    KeysWriter wr{keys, kvals, comp_out, comp_ld, k};
    dfx_launch_select<256>(ldr, wr, nrows, n, k, st);
}

void dfx_launch_select_comp(const uint64_t* comp, int64_t nrows, int n, int64_t ld, int k, int32_t* keys,
                            cudaStream_t st) {
    CompLoader ldr{comp, ld};
    KeysWriter wr{keys, nullptr, nullptr, 0, k};
    dfx_launch_select<256>(ldr, wr, nrows, n, k, st);
}

#include "dfx_pq_prep_dev.cuh"

// =====================================================================================
// K4: scan_pq.  one CTA = (query, group of G consecutive probes).  lane-per-vector:
//   v = dis0 + (t + S),  S = halving-tree sum of lut[m][code_m] (oracle pq_sum)
// =====================================================================================
template <int MT>
__global__ void __launch_bounds__(128)
scan_pq_kernel(const float* __restrict__ lut, const float* __restrict__ dis0,
               const int32_t* __restrict__ keys, int nprobe, int G, int ngroups,
               const int64_t* __restrict__ list_off, const uint8_t* __restrict__ codes,
               const float* __restrict__ tvals, const int32_t* __restrict__ ids, int Mrt, int ksub,
               int nbits, int k, int cap, uint64_t* __restrict__ part) {
    DFX_DYN_SMEM(unsigned char, smem_raw, 16);
    const int M = (MT > 0) ? MT : Mrt;
    float* s_lut = reinterpret_cast<float*>(smem_raw);
    uint64_t* s_buf = reinterpret_cast<uint64_t*>(smem_raw + (size_t)M * ksub * 4);
    const int64_t q = blockIdx.x / ngroups;
    const int g = blockIdx.x % ngroups;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    {
        const float4* src = reinterpret_cast<const float4*>(lut + q * (int64_t)M * ksub);
        float4* dst = reinterpret_cast<float4*>(s_lut);
        for (int i = tid; i < (M * ksub) / 4; i += 128) dst[i] = src[i];
    }
    WarpTopK wt;
    wt.init(s_buf + (size_t)warp * cap, cap, k);
    __syncthreads();

    const int p_end = min(nprobe, (g + 1) * G);
    for (int p = g * G; p < p_end; p++) {
        const int l = keys[q * nprobe + p];
        if (l < 0) continue;
        const float d0 = dis0[q * nprobe + p];
        const int64_t beg = list_off[l], end = list_off[l + 1];
        for (int64_t base = beg + warp * 32; base < end; base += 128) {
            const int64_t i = base + lane;
            const bool valid = i < end;
            float v = 0.f;
            uint32_t my_id = DFX_SEC_NONE;  // loaded with the code: never a dependent load on admission
            if (valid) {
                my_id = (uint32_t)__ldg(ids + i);
                // table values of this vector, then the canonical halving tree (oracle pq_sum)
                constexpr int P = (MT > 0) ? MT : 64;  // MT is a power of two when > 0
                float val[P];
                if (nbits == 4) {  // ksub = 16, rows of M / 2 bytes (M % 8 == 0): 8 codes per word
                    const uint32_t* cp = reinterpret_cast<const uint32_t*>(codes + i * (int64_t)(M / 2));
#pragma unroll
                    for (int w = 0; w < (P + 7) / 8; w++) {
                        const int m = w * 8;
                        if (m < M) {
                            const uint32_t c = __ldg(cp + w);
#pragma unroll
                            for (int u = 0; u < 8; u++) val[m + u] = s_lut[(m + u) * 16 + dfx_pq4_word_code(c, u)];
                        } else {
#pragma unroll
                            for (int u = 0; u < 8; u++) val[m + u] = 0.f;
                        }
                    }
                } else if (MT > 0 && (MT % 16) == 0) {
                    const uint4* cp = reinterpret_cast<const uint4*>(codes + i * (int64_t)M);
#pragma unroll
                    for (int w4 = 0; w4 < MT / 16; w4++) {
                        uint4 c = __ldg(cp + w4);
                        uint32_t wv[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
                        for (int w = 0; w < 4; w++) {
                            const int m = w4 * 16 + w * 4;
                            val[m + 0] = s_lut[(m + 0) * ksub + (wv[w] & 255u)];
                            val[m + 1] = s_lut[(m + 1) * ksub + ((wv[w] >> 8) & 255u)];
                            val[m + 2] = s_lut[(m + 2) * ksub + ((wv[w] >> 16) & 255u)];
                            val[m + 3] = s_lut[(m + 3) * ksub + (wv[w] >> 24)];
                        }
                    }
                } else {
                    const uint32_t* cp = reinterpret_cast<const uint32_t*>(codes + i * (int64_t)M);
#pragma unroll
                    for (int w = 0; w < P / 4; w++) {
                        const int m = w * 4;
                        if (m < M) {
                            uint32_t c = __ldg(cp + w);
                            val[m + 0] = s_lut[(m + 0) * ksub + (c & 255u)];
                            val[m + 1] = s_lut[(m + 1) * ksub + ((c >> 8) & 255u)];
                            val[m + 2] = s_lut[(m + 2) * ksub + ((c >> 16) & 255u)];
                            val[m + 3] = s_lut[(m + 3) * ksub + (c >> 24)];
                        } else {
                            val[m + 0] = val[m + 1] = val[m + 2] = val[m + 3] = 0.f;
                        }
                    }
                }
#pragma unroll
                for (int off = P / 2; off >= 1; off >>= 1)
#pragma unroll
                    for (int r = 0; r < off; r++) val[r] = val[r] + val[r + off];
                v = d0 + (__ldg(tvals + i) + val[0]);
            }
            uint32_t sec = 0;
            const bool want = valid && wt.admits(v, [&] { return my_id; }, sec);
            wt.push_lanes(want, v, sec);
        }
    }
    cta_merge_and_write<128>(wt, s_buf, cap, k, part + ((int64_t)q * ngroups + g) * k);
}

// =====================================================================================
// K2 / K5: scan_rows.  warp-per-vector, warp-dot canonical order.
//   MODE 0: fp32 rows, value = -<q,x>      (IVF-Flat, IP)
//   MODE 1: fp32 rows, value = ||q-x||^2   (IVF-Flat, L2)
//   MODE 2: fp16 residual codes, value = ||(q-c) - half2float(code)||^2   (IVF-SQ fp16)
// =====================================================================================
// U = vectors in flight per warp: 4 (default), 8 = EXPERIMENTAL (dfx_set_param "rows_inflight"):
// the kernel is bound by memory-level parallelism, not by instructions -- C2 (512 B per vector)
// reaches 0.46 of the HBM peak and C4 (1536 B per vector) 0.68 with the same code.
template <int MODE, int U = 4>
__global__ void __launch_bounds__(128)
scan_rows_kernel(const float* __restrict__ Q, int d, const float* __restrict__ cent,
                 const int32_t* __restrict__ keys, int nprobe, int G, int ngroups,
                 const int64_t* __restrict__ list_off, const void* __restrict__ rows,
                 const int32_t* __restrict__ ids, int k, int cap, uint64_t* __restrict__ part) {
    DFX_DYN_SMEM(unsigned char, smem_raw, 16);
    float* s_q = reinterpret_cast<float*>(smem_raw);   // query (MODE 2: residual q - c)
    float* s_q0 = s_q + d;                              // MODE 2: the raw query
    const int dpad = (MODE == 2) ? 2 * d : d;
    uint64_t* s_buf = reinterpret_cast<uint64_t*>(smem_raw + (((size_t)dpad * 4 + 15) / 16) * 16);
    const int64_t q = blockIdx.x / ngroups;
    const int g = blockIdx.x % ngroups;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    for (int i = tid; i < d; i += 128) {
        float qv = Q[q * d + i];
        s_q[i] = qv;
        if (MODE == 2) s_q0[i] = qv;
    }
    WarpTopK wt;
    wt.init(s_buf + (size_t)warp * cap, cap, k);
    __syncthreads();

    const int p_end = min(nprobe, (g + 1) * G);
    for (int p = g * G; p < p_end; p++) {
        const int l = keys[q * nprobe + p];
        if (l < 0) continue;
        if (MODE == 2) {
            __syncthreads();
            for (int i = tid; i < d; i += 128) s_q[i] = s_q0[i] - cent[(size_t)l * d + i];
            __syncthreads();
        }
        const int64_t beg = list_off[l], end = list_off[l + 1];
        for (int64_t base = beg + warp * U; base < end; base += 4 * U) {
            float acc[U];
            uint32_t vid[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                acc[u] = 0.f;
                vid[u] = (base + u < end) ? (uint32_t)__ldg(ids + base + u) : DFX_SEC_NONE;
            }
            for (int kb = 4 * lane; kb < d; kb += 128) {
                const float4 qv = *reinterpret_cast<const float4*>(s_q + kb);
                float4 xv[U];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int64_t i = base + u;
                    if (i < end) {
                        if (MODE == 2) {
                            const uint2 h = __ldg(reinterpret_cast<const uint2*>(
                                reinterpret_cast<const __half*>(rows) + i * (int64_t)d + kb));
                            const __half2 h01 = *reinterpret_cast<const __half2*>(&h.x);
                            const __half2 h23 = *reinterpret_cast<const __half2*>(&h.y);
                            const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                            xv[u] = make_float4(f01.x, f01.y, f23.x, f23.y);
                        } else {
                            xv[u] = __ldg(reinterpret_cast<const float4*>(
                                reinterpret_cast<const float*>(rows) + i * (int64_t)d + kb));
                        }
                    } else {
                        xv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    if (MODE == 0) {
                        acc[u] = __fmaf_rn(qv.x, xv[u].x, acc[u]);
                        acc[u] = __fmaf_rn(qv.y, xv[u].y, acc[u]);
                        acc[u] = __fmaf_rn(qv.z, xv[u].z, acc[u]);
                        acc[u] = __fmaf_rn(qv.w, xv[u].w, acc[u]);
                    } else {
                        float df;
                        df = qv.x - xv[u].x; acc[u] = __fmaf_rn(df, df, acc[u]);
                        df = qv.y - xv[u].y; acc[u] = __fmaf_rn(df, df, acc[u]);
                        df = qv.z - xv[u].z; acc[u] = __fmaf_rn(df, df, acc[u]);
                        df = qv.w - xv[u].w; acc[u] = __fmaf_rn(df, df, acc[u]);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                const int64_t i = base + u;
                float v = dfx_warp_butterfly(acc[u]);
                if (MODE == 0) v = -v;
                uint32_t sec = 0;
                if (i < end && wt.admits(v, [&] { return vid[u]; }, sec))
                    wt.push_uniform(v, sec);
            }
        }
    }
    cta_merge_and_write<128>(wt, s_buf, cap, k, part + ((int64_t)q * ngroups + g) * k);
}

// =====================================================================================
// K6: cross-shard merge (client.py:265-310 / float_maxheap_array_t)
// =====================================================================================
struct MergeLoader {
    const float* D;
    int64_t nq;
    int k;
    int negate;
    __device__ __forceinline__ uint64_t operator()(int64_t row, int e) const {
        int s = e / k, j = e - s * k;
        float v = D[((int64_t)s * nq + row) * k + j];
        if (negate) v = -v;
        if (!(v < FLT_MAX)) return DFX_COMP_NONE;  // heapify(): admitted only if FLT_MAX > v
        return dfx_comp(v, (uint32_t)e);
    }
};
struct MergeWriter {
    const int64_t* I;
    int64_t nq;
    int k;
    float* outD;
    int64_t* outI;
    __device__ __forceinline__ void operator()(int64_t row, int j, uint64_t c) const {
        if (c == DFX_COMP_NONE) {
            outD[row * k + j] = FLT_MAX;
            outI[row * k + j] = -1;
        } else {
            uint32_t e = (uint32_t)c;
            int s = e / k, jj = e - s * k;
            outD[row * k + j] = dfx_key2f((uint32_t)(c >> 32));
            outI[row * k + j] = I[((int64_t)s * nq + row) * k + jj];
        }
    }
};

void dfx_merge_impl(int64_t S, int64_t nq, int64_t k, const float* d_D, const int64_t* d_I,
                    int negate, float* d_outD, int64_t* d_outI, cudaStream_t st) {
    DFX_REQUIRE(S >= 1 && k >= 1 && S * k < (1ll << 31), "merge: bad S/k");
    if (nq <= 0) return;
    MergeLoader ldr{d_D, nq, (int)k, negate};
    MergeWriter wr{d_I, nq, (int)k, d_outD, d_outI};
    dfx_launch_select<128>(ldr, wr, nq, (int)(S * k), (int)k, st);
}

__global__ void map_ids_kernel(int64_t n, const int64_t* __restrict__ ids,
                               const int64_t* __restrict__ table, int64_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        int64_t v = ids[i];
        out[i] = v < 0 ? -1 : table[v];
    }
}
void dfx_map_ids_impl(int64_t n, const int64_t* d_ids, const int64_t* d_table, int64_t* d_out,
                      cudaStream_t st) {
    if (n <= 0) return;
    DFX_LAUNCH(map_ids_kernel, (unsigned)dfx_ceil_div(n, 256), 256, 0, st, n, d_ids, d_table, d_out);
}

// ---- packed exchange form: what ONE all-gather over the ranks delivers.  Rank r's block starts at
// base + r * rank_stride and holds D f32[S_loc][nq][k] at offset 0 and I i64[S_loc][nq][k] at
// off_I.  Shard s = r * S_loc + j (rank-major), same total order as dfx_merge_impl.
struct MergePackedLoader {
    const unsigned char* base;
    int64_t rank_stride, nq;
    int k, s_loc, negate;
    __device__ __forceinline__ uint64_t operator()(int64_t row, int e) const {
        int s = e / k, j = e - s * k;
        int r = s / s_loc, sl = s - r * s_loc;
        const float* D = reinterpret_cast<const float*>(base + (int64_t)r * rank_stride);
        float v = D[((int64_t)sl * nq + row) * k + j];
        if (negate) v = -v;
        if (!(v < FLT_MAX)) return DFX_COMP_NONE;
        return dfx_comp(v, (uint32_t)e);
    }
};
struct MergePackedWriter {
    const unsigned char* base;
    int64_t rank_stride, off_I, nq;
    int k, s_loc;
    float* outD;
    int64_t* outI;
    __device__ __forceinline__ void operator()(int64_t row, int j, uint64_t c) const {
        if (c == DFX_COMP_NONE) {
            outD[row * k + j] = FLT_MAX;
            outI[row * k + j] = -1;
        } else {
            uint32_t e = (uint32_t)c;
            int s = e / k, jj = e - s * k;
            int r = s / s_loc, sl = s - r * s_loc;
            const int64_t* I = reinterpret_cast<const int64_t*>(base + (int64_t)r * rank_stride + off_I);
            outD[row * k + j] = dfx_key2f((uint32_t)(c >> 32));
            outI[row * k + j] = I[((int64_t)sl * nq + row) * k + jj];
        }
    }
};
void dfx_merge_packed_impl(int64_t R, int64_t S_loc, int64_t nq, int64_t k, const void* d_packed,
                           int64_t rank_stride, int64_t off_I, int negate, float* d_outD,
                           int64_t* d_outI, cudaStream_t st) {
    DFX_REQUIRE(R >= 1 && S_loc >= 1 && k >= 1 && R * S_loc * k < (1ll << 31), "merge: bad R/S/k");
    DFX_REQUIRE(rank_stride % 8 == 0 && off_I % 8 == 0 && off_I >= S_loc * nq * k * 4,
                "merge: the packed blocks must be 8-byte aligned and I must follow D");
    if (nq <= 0) return;
    const unsigned char* b = reinterpret_cast<const unsigned char*>(d_packed);
    MergePackedLoader ldr{b, rank_stride, nq, (int)k, (int)S_loc, negate};
    MergePackedWriter wr{b, rank_stride, off_I, nq, (int)k, (int)S_loc, d_outD, d_outI};
    dfx_launch_select<128>(ldr, wr, nq, (int)(R * S_loc * k), (int)k, st);
}

// shard-local ids -> exchange ids: (shard tag << 40) | local id, -1 stays -1.  With a metadata
// column (int32 code per local id; -2 = the entry has no such metadata position) the entries the
// reference's post-filter would drop (client.py:235-243: meta[filter_pos] == filter_value, or no
// metadata / too short) get bit 62 set; the flag rides through all-gather + merge untouched.
__global__ void encode_ids_kernel(int64_t n, const int64_t* __restrict__ ids, int64_t tag,
                                  const int32_t* __restrict__ col, int32_t drop_code,
                                  int64_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t v = ids[i];
    if (v < 0) {
        out[i] = -1;
        return;
    }
    int64_t e = (tag << 40) | v;
    if (col) {
        int32_t c = col[v];
        if (c == drop_code || c == -2) e |= (1ll << 62);
    }
    out[i] = e;
}
void dfx_encode_ids_impl(int64_t n, const int64_t* d_ids, int64_t tag, const int32_t* d_col,
                         int32_t drop_code, int64_t* d_out, cudaStream_t st) {
    DFX_REQUIRE(tag >= 0 && tag < (1ll << 20), "encode_ids: shard tag out of range");
    if (n <= 0) return;
    DFX_LAUNCH(encode_ids_kernel, (unsigned)dfx_ceil_div(n, 256), 256, 0, st, n, d_ids, tag, d_col, drop_code, d_out);
}

// post-filter of search_with_filter on device (client.py:229-250): per query walk the kin merged
// slots in rank order, keep the entries that exist (I >= 0) and do not carry the drop flag, stop
// at kout.  One warp per query; ballot + prefix popcount keeps the order.
__global__ void filter_compact_kernel(int64_t nq, int kin, int kout, const float* __restrict__ D,
                                      const int64_t* __restrict__ I, float* __restrict__ outD,
                                      int64_t* __restrict__ outI, int32_t* __restrict__ outCount) {
    const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (q >= nq) return;
    int kept = 0;
    for (int j0 = 0; j0 < kin && kept < kout; j0 += 32) {
        int j = j0 + lane;
        int64_t id = (j < kin) ? I[q * kin + j] : -1;
        bool keep = id >= 0 && !(id & (1ll << 62));
        unsigned m = __ballot_sync(0xffffffffu, keep);
        int pos = kept + __popc(m & ((1u << lane) - 1u));
        if (keep && pos < kout) {
            outD[q * kout + pos] = D[q * kin + j];
            outI[q * kout + pos] = id;
        }
        kept += __popc(m);
    }
    if (kept > kout) kept = kout;
    for (int j = kept + lane; j < kout; j += 32) {
        outD[q * kout + j] = FLT_MAX;
        outI[q * kout + j] = -1;
    }
    if (lane == 0) outCount[q] = kept;
}
void dfx_filter_compact_impl(int64_t nq, int64_t kin, int64_t kout, const float* d_D, const int64_t* d_I,
                             float* d_outD, int64_t* d_outI, int32_t* d_count, cudaStream_t st) {
    DFX_REQUIRE(kin >= 1 && kout >= 1 && kin < (1 << 20), "filter: bad k");
    if (nq <= 0) return;
    DFX_LAUNCH(filter_compact_kernel, (unsigned)dfx_ceil_div(nq, 4), 128, 0, st, nq, (int)kin, (int)kout, d_D, d_I,
               d_outD, d_outI, d_count);
}

// ndis of the last search = sum over (q,p) of len(list keys[q][p])
__global__ void ndis_kernel(const int32_t* __restrict__ keys, int64_t n,
                            const int64_t* __restrict__ list_off, unsigned long long* out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long v = 0;
    if (i < n) {
        int l = keys[i];
        if (l >= 0) v = (unsigned long long)(list_off[l + 1] - list_off[l]);
    }
    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(out, v);
}
void dfx_stats_impl(dfx_index* idx, int64_t* ndis, cudaStream_t st) {
    *ndis = 0;
    if (!idx->is_ivf() || !idx->last_keys_valid) return;
    int64_t n = idx->last_nq * idx->last_nprobe;
    if (n <= 0) return;
    idx->w_misc.reserve(8);
    DFX_CUDA(cudaMemsetAsync(idx->w_misc.p, 0, 8, st));
    DFX_LAUNCH(ndis_kernel, (unsigned)dfx_ceil_div(n, 256), 256, 0, st, idx->w_keys.as<int32_t>(), n,
               idx->list_off.as<int64_t>(), idx->w_misc.as<unsigned long long>());
    unsigned long long h = 0;
    DFX_CUDA(cudaMemcpyAsync(&h, idx->w_misc.p, 8, cudaMemcpyDeviceToHost, st));
    DFX_CUDA(cudaStreamSynchronize(st));
    *ndis = (int64_t)h;
}

// =====================================================================================
// the per-shard search driver
// =====================================================================================
static int choose_group(int64_t nq, int nprobe) {
    // keep >= ~8 CTAs per SM in flight; at large batch let one CTA walk several lists so the
    // query's table is staged into shared memory once.
    const int64_t target = 148 * 8;
    int64_t G = (nq * (int64_t)nprobe) / target;
    if (G < 1) G = 1;
    if (G > nprobe) G = nprobe;
    if (G > 16) G = 16;
    return (int)G;
}

void dfx_search_impl(dfx_index* idx, int64_t nq, const float* d_x, int64_t k64, float* d_D,
                     int64_t* d_I, cudaStream_t st) {
    DFX_REQUIRE(idx->trained || idx->cfg.kind == DFX_FLAT, "index is not trained");
    DFX_REQUIRE(k64 >= 1, "k must be >= 1");
    if (nq <= 0) return;
    if (idx->n_pending > 0) dfx_finalize_impl(idx, st);
    const int d = idx->cfg.d;
    const int k = (int)k64;
    const int kind = idx->cfg.kind;
    idx->last_keys_valid = false;

    if (kind == DFX_FLAT) {
        DFX_REQUIRE(k64 <= 4096, "flat search supports k <= 4096");
        const int64_t N = idx->n_sorted;
        const int metric = idx->cfg.metric;
        if (N == 0) {
            ResultWriter wr{d_D, d_I, k, metric, 0.f, nullptr};
            CompLoader ldr{nullptr, 0};
            dfx_launch_select<128>(ldr, wr, nq, 0, k, st);
            return;
        }
        float* qnorm_tc = nullptr;
        if (idx->flat_tc && idx->tc_enabled) {  // screening on tensor cores + exact re-rank
            const int64_t ng = dfx_ceil_div(N, 128) * 4;
            const int64_t QT = std::max<int64_t>(128, ((64ll << 20) / (ng * 4)) / 128 * 128);
            bool handled = true;
            for (int64_t q0 = 0; q0 < nq && handled; q0 += QT) {
                const int64_t qc = std::min(QT, nq - q0);
                const int ncand = dfx_tc_flat_candidates(idx, d_x + q0 * d, qc, k, st);
                if (ncand == 0) {
                    handled = false;  // shape not covered (only possible on the first chunk)
                    break;
                }
                if (metric == DFX_METRIC_L2 && !qnorm_tc) {
                    idx->w_dis0.reserve((size_t)nq * 4);
                    qnorm_tc = idx->w_dis0.as<float>();
                    dfx_launch_row_norms(d_x, nq, d, qnorm_tc, st);
                }
                CompLoader ldr{idx->tc_cand.as<uint64_t>(), ncand};
                ResultWriter wr{d_D + q0 * k, d_I + q0 * k, k, metric, 0.f, qnorm_tc ? qnorm_tc + q0 : nullptr};
                dfx_launch_select<128>(ldr, wr, qc, ncand, k, st);
            }
            if (handled) return;
        }
        const int64_t NT = 32768;
        const int64_t ntiles = dfx_ceil_div(N, NT);
        int64_t QC = (32ll << 20) / NT;  // 1024 queries per chunk (128 MB of values)
        if (QC > nq) QC = nq;
        idx->w_vals.reserve((size_t)QC * NT * 4);
        idx->w_part.reserve((size_t)QC * ntiles * k * 8);
        float* qnorm = nullptr;
        if (metric == DFX_METRIC_L2) {
            idx->w_dis0.reserve((size_t)nq * 4);
            qnorm = idx->w_dis0.as<float>();
            dfx_launch_row_norms(d_x, nq, d, qnorm, st);
        }
        for (int64_t q0 = 0; q0 < nq; q0 += QC) {
            const int64_t qc = (nq - q0 < QC) ? (nq - q0) : QC;
            for (int64_t t = 0; t < ntiles; t++) {
                const int64_t c0 = t * NT;
                const int64_t nc = (N - c0 < NT) ? (N - c0) : NT;
                dfx_launch_gemm_values(d_x + q0 * d, qc, idx->payload.as<float>() + c0 * d,
                                       idx->xnorm.as<float>() ? idx->xnorm.as<float>() + c0 : nullptr,
                                       nc, d, metric, idx->w_vals.as<float>(), NT, st);
                dfx_launch_select_cols(idx->w_vals.as<float>(), qc, (int)nc, NT, k, (uint32_t)c0,
                                       nullptr, nullptr, idx->w_part.as<uint64_t>() + t * k,
                                       ntiles * k, st);
            }
            CompLoader ldr{idx->w_part.as<uint64_t>(), ntiles * k};
            ResultWriter wr{d_D + q0 * k, d_I + q0 * k, k, metric, 0.f, qnorm ? qnorm + q0 : nullptr};
            dfx_launch_select<128>(ldr, wr, qc, (int)(ntiles * k), k, st);
        }
        return;
    }

    // ---------------- IVF kinds
    DFX_REQUIRE(k64 <= 1024, "IVF search supports k <= 1024");
    const int64_t nlist = idx->cfg.nlist;
    int nprobe = (int)std::min<int64_t>(std::max<int64_t>(idx->nprobe, 1), nlist);
    DFX_REQUIRE(nprobe <= 4096, "nprobe <= 4096");
    const int cmetric = idx->cfg.metric;  // coarse quantizer metric
    const int smetric = (kind == DFX_IVF_FLAT) ? idx->cfg.metric : DFX_METRIC_L2;

    // query chunk: bounds the workspace (values matrix on the FFMA coarse path, tables and
    // partial results otherwise)
    const bool use_tc = idx->tc_enabled && idx->tc_ready && nlist >= 1024 && nprobe <= 512;
    int64_t QC = use_tc ? 8192 : (32ll << 20) / nlist;
    if (QC < 1) QC = 1;
    if (QC > 8192) QC = 8192;
    if (QC > nq) QC = nq;
    const int KP = dfx_next_pow2(k < 32 ? 32 : k);
    const int cap = 2 * KP;

    idx->w_keys.reserve((size_t)nq * nprobe * 4);
    int32_t* keys_all = idx->w_keys.as<int32_t>();

    for (int64_t q0 = 0; q0 < nq; q0 += QC) {
        const int64_t qc = (nq - q0 < QC) ? (nq - q0) : QC;
        const float* xq = d_x + q0 * d;
        int32_t* keys = keys_all + q0 * nprobe;
        // K1: coarse quantizer -- tensor cores (screen) + canonical fp32 (decide), or plain FFMA
        if (use_tc) {
            dfx_tc_coarse_search(idx, xq, qc, nprobe, keys, st);
        } else {
            idx->w_vals.reserve((size_t)QC * nlist * 4);
            dfx_launch_gemm_values(xq, qc, idx->centroids.as<float>(), idx->cnorm.as<float>(), nlist, d,
                                   cmetric, idx->w_vals.as<float>(), nlist, st);
            dfx_launch_select_cols(idx->w_vals.as<float>(), qc, (int)nlist, nlist, nprobe, 0, keys,
                                   nullptr, nullptr, 0, st);
        }
        const int G = choose_group(qc, nprobe);
        const int ngroups = (nprobe + G - 1) / G;
        idx->w_part.reserve((size_t)qc * ngroups * k * 8);
        uint64_t* part = idx->w_part.as<uint64_t>();
        std::pair<cudaEvent_t, cudaEvent_t>* pev = nullptr;
        if (idx->prof_on) {
            if (idx->prof_used == idx->prof_events.size()) {
                cudaEvent_t a, b;
                DFX_CUDA(cudaEventCreate(&a));
                DFX_CUDA(cudaEventCreate(&b));
                idx->prof_events.emplace_back(a, b);
            }
            pev = &idx->prof_events[idx->prof_used++];
            DFX_CUDA(cudaEventRecord(pev->first, st));
        }

        bool final_written = false;
        if (kind == DFX_IVF_PQ && idx->il) {
            // M == 32 x 8 / 64 x 4 bit: table build + exact |q-c|^2 + block scan in ONE kernel; with a single probe
            // group per query it also writes the final rows (dfx_scan_il2.cu)
            final_written = dfx_launch_scan_pq_il2(idx, xq, qc, keys, nprobe, G, ngroups, k, cap, part, d_D + q0 * k,
                                                   d_I + q0 * k, st);
        } else if (kind == DFX_IVF_PQ) {
            const int M = idx->M, ksub = idx->ksub;
            idx->w_lut.reserve((size_t)qc * M * ksub * 4);
            idx->w_dis0.reserve((size_t)qc * nprobe * 4);
            const size_t prep_smem = (size_t)((d + 3) / 4) * 16;
            DFX_LAUNCH(pq_prep_kernel, (unsigned)qc, 256, prep_smem, st, xq, d, M, ksub, idx->dsub,
                       idx->codebooks.as<float>(), idx->centroids.as<float>(), keys, nprobe,
                       idx->w_lut.as<float>(), idx->w_dis0.as<float>());
            {
            const size_t smem = (size_t)M * ksub * 4 + (size_t)4 * cap * 8;
#define DFX_SCAN_PQ(MT)                                                                          \
    do {                                                                                         \
        auto kern = scan_pq_kernel<MT>;                                                          \
        DFX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,         \
                                      (int)smem));                                               \
        DFX_LAUNCH(kern, (unsigned)(qc * ngroups), 128, smem, st, idx->w_lut.as<float>(),        \
                   idx->w_dis0.as<float>(), keys, nprobe, G, ngroups, idx->list_off.as<int64_t>(), \
                   idx->payload.as<uint8_t>(), idx->tvals.as<float>(), idx->ids.as<int32_t>(), M, \
                   ksub, idx->nbits, k, cap, part);                                              \
    } while (0)
            if (M == 32) DFX_SCAN_PQ(32);
            else if (M == 64) DFX_SCAN_PQ(64);
            else if (M == 16) DFX_SCAN_PQ(16);
            else if (M == 8) DFX_SCAN_PQ(8);
            else DFX_SCAN_PQ(0);  // any other M <= 64: values padded to 64 with +0
#undef DFX_SCAN_PQ
            }
        } else {
            const int dq = (kind == DFX_IVF_SQ16) ? 2 * d : d;
            const size_t smem = (((size_t)dq * 4 + 15) / 16) * 16 + (size_t)4 * cap * 8;
            // vectors in flight per warp: rows of up to 1 KB need 8 to cover the DRAM latency
            // (B200, C2 512 B rows: 3.0 -> 4.6 TB/s), longer rows are faster with 4 (C4 1536 B rows:
            // 4.5 vs 3.2 TB/s); profiles/r02_other_configs.json
            const int inflight = idx->rows_inflight ? idx->rows_inflight : (idx->row_bytes() <= 1024 ? 8 : 4);
#define DFX_SCAN_ROWS(MODE)                                                                      \
    do {                                                                                         \
        auto kern = (inflight == 8) ? scan_rows_kernel<MODE, 8> : scan_rows_kernel<MODE, 4>; \
        DFX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,         \
                                      (int)smem));                                               \
        DFX_LAUNCH(kern, (unsigned)(qc * ngroups), 128, smem, st, xq, d, idx->centroids.as<float>(), \
                   keys, nprobe, G, ngroups, idx->list_off.as<int64_t>(), idx->payload.p,        \
                   idx->ids.as<int32_t>(), k, cap, part);                                        \
    } while (0)
            if (kind == DFX_IVF_SQ16) DFX_SCAN_ROWS(2);
            else if (smetric == DFX_METRIC_IP) DFX_SCAN_ROWS(0);
            else DFX_SCAN_ROWS(1);
#undef DFX_SCAN_ROWS
        }
        if (pev) DFX_CUDA(cudaEventRecord(pev->second, st));
        if (!final_written) {
            CompLoader ldr{part, (int64_t)ngroups * k};
            ResultWriter wr{d_D + q0 * k, d_I + q0 * k, k, smetric, 0.f, nullptr};
            dfx_launch_select<128>(ldr, wr, qc, ngroups * k, k, st);
        }
    }
    idx->last_nq = nq;
    idx->last_nprobe = nprobe;
    idx->last_keys_valid = true;
}

// =====================================================================================
// K7a: fused nearest-centroid assignment (build path).  Same FFMA tile as K1a, but the
// epilogue reduces each row's tile to one composite (value, column) and folds it into
// best[row] with a 64-bit atomicMin -- the values matrix is never written.  The minimum of
// composites is exactly the oracle's argmin with ties -> smaller index.
// =====================================================================================
template <int BM, int BN, int BK, int TM, int TN>
__global__ void __launch_bounds__((BM / TM) * (BN / TN))
gemm_argmin_kernel(const float* __restrict__ Q, int64_t nq, const float* __restrict__ X,
                   const float* __restrict__ xnorm, int64_t ncols, int d, int metric,
                   unsigned long long* __restrict__ best) {
    constexpr int THREADS = (BM / TM) * (BN / TN);
    __shared__ float sQ[BK][BM + 4];
    __shared__ float sX[BK][BN + 4];
    const int tid = threadIdx.x;
    const int tx = tid % (BN / TN), ty = tid / (BN / TN);
    const int64_t m0 = (int64_t)blockIdx.y * BM;
    const int64_t n0 = (int64_t)blockIdx.x * BN;
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; i++)
#pragma unroll
        for (int j = 0; j < TN; j++) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < d; k0 += BK) {
        for (int e = tid; e < BM * BK; e += THREADS) {
            int m = e / BK, kk = e % BK;
            int64_t gm = m0 + m;
            int gk = k0 + kk;
            sQ[kk][m] = (gm < nq && gk < d) ? Q[gm * d + gk] : 0.f;
        }
        for (int e = tid; e < BN * BK; e += THREADS) {
            int n = e / BK, kk = e % BK;
            int64_t gn = n0 + n;
            int gk = k0 + kk;
            sX[kk][n] = (gn < ncols && gk < d) ? X[gn * d + gk] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; kk++) {
            float a[TM], b[TN];
#pragma unroll
            for (int i = 0; i < TM; i++) a[i] = sQ[kk][ty * TM + i];
#pragma unroll
            for (int j = 0; j < TN; j++) b[j] = sX[kk][tx * TN + j];
#pragma unroll
            for (int i = 0; i < TM; i++)
#pragma unroll
                for (int j = 0; j < TN; j++) acc[i][j] = __fmaf_rn(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
    constexpr int TXN = BN / TN;  // threads sharing a row (consecutive lanes)
#pragma unroll
    for (int i = 0; i < TM; i++) {
        unsigned long long c = DFX_COMP_NONE;
#pragma unroll
        for (int j = 0; j < TN; j++) {
            int64_t gn = n0 + tx * TN + j;
            if (gn < ncols) {
                float ip = acc[i][j];
                float v = (metric == DFX_METRIC_IP) ? -ip : __fmaf_rn(-2.f, ip, xnorm[gn]);
                unsigned long long cc = dfx_comp(v, (uint32_t)gn);
                c = cc < c ? cc : c;
            }
        }
#pragma unroll
        for (int off = TXN / 2; off >= 1; off >>= 1) {
            unsigned long long o = __shfl_xor_sync(0xffffffffu, c, off);
            c = o < c ? o : c;
        }
        int64_t gm = m0 + ty * TM + i;
        if (tx == 0 && gm < nq && c != DFX_COMP_NONE) atomicMin(&best[gm], c);
    }
}

__global__ void unpack_best_kernel(const unsigned long long* __restrict__ best, int64_t n,
                                   int32_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int32_t)(uint32_t)best[i];
}

void dfx_launch_assign_fused(const float* X, int64_t n, const float* cent, const float* cnorm,
                             int64_t nlist, int d, int metric, unsigned long long* best,
                             int32_t* out, cudaStream_t st) {
    if (n <= 0) return;
    DFX_CUDA(cudaMemsetAsync(best, 0xff, (size_t)n * 8, st));
    constexpr int BM = 128, BN = 128, BK = 8, TM = 8, TN = 8;
    static_assert(BN / TN == 16, "row group must be 16 consecutive lanes");
    const int64_t max_y = 65535;
    for (int64_t r0 = 0; r0 < n; r0 += max_y * BM) {
        int64_t rc = std::min<int64_t>(n - r0, max_y * BM);
        dim3 grid((unsigned)dfx_ceil_div(nlist, BN), (unsigned)dfx_ceil_div(rc, BM));
        auto kern = gemm_argmin_kernel<BM, BN, BK, TM, TN>;
        DFX_LAUNCH(kern, grid, (BM / TM) * (BN / TN), 0, st, X + r0 * d, rc, cent, cnorm, nlist, d, metric,
                   best + r0);
    }
    DFX_LAUNCH(unpack_best_kernel, (unsigned)dfx_ceil_div(n, 256), 256, 0, st, best, n, out);
}
