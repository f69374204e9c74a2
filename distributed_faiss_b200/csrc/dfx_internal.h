// dfx_internal.h -- index object + launcher declarations shared by the .cu files.
#pragma once
#include "dfx_common.cuh"
#include <vector>
#include <atomic>
#include <mutex>
#include <memory>
#include <algorithm>

struct dfx_index {
    dfx_cfg cfg{};
    int M = 0, ksub = 0, dsub = 0;
    int nbits = 8;  // IVF-PQ bits per sub-quantizer code (4 or 8); ksub = 1 << nbits
    int64_t nprobe = 1;  // faiss default (index.py:47 copies it back into cfg for knnlm)
    bool trained = false;

    // list-sorted storage ("sorted") and arrival-order staging ("pending")
    int64_t n_sorted = 0, n_pending = 0;
    DevBuf centroids, cnorm, codebooks;
    DevBuf list_off;                    // int64[nlist+1]
    std::vector<int64_t> h_list_off;    // host mirror
    DevBuf ids;                         // int32[n_sorted] shard-local ids, list-sorted
    DevBuf payload;                     // kind-specific rows, list-sorted (FLAT: arrival order)
    DevBuf tvals;                       // IVF_PQ: f32[n_sorted]
    DevBuf xnorm;                       // FLAT + L2: f32[n]
    DevBuf p_list, p_payload, p_tvals;  // pending: int32 list per row, payload rows, tvals
    int64_t p_cap = 0;
    int64_t reserve_hint = 0;

    // search workspace (grow-only)
    DevBuf w_vals, w_keys, w_dis0, w_lut, w_part, w_q, w_D, w_I, w_misc, w_best;
    // reconstruct support: inverse of ids (shard-local id -> storage position)
    DevBuf inv;
    bool inv_valid = false;
    // training knobs (dfx_set_param)
    int kmeans_niter = 25;            // faiss Clustering default niter
    int max_points_per_centroid = 256;  // faiss Clustering default
    uint64_t train_seed = 1234;       // faiss Clustering default seed

    // IVF-PQ, M == 32 x 8 bit or M == 64 x 4 bit: block-interleaved storage for the lane-per-vector
    // scan (dfx_scan_il2.cu, layout dfx_il2_byte / dfx_il2_pair).  While `il` is set the row-major
    // payload/tvals/ids are released.
    bool il = false, il_enabled = true;
    DevBuf il_codes, il_tvals, il_ids, blk_off;
    int64_t nblk = 0;
    DevBuf codebooksT;  // [ksub][M][dsub]: the order the fused table build reads (dfx_scan_il2.cu)
    bool cbT_valid = false;

    // tensor-core coarse quantizer (dfx_tc.cu): fp16 copies (1 or 2 planes) and screening workspace
    DevBuf tc_cent, tc_cent_tmp, tc_q, tc_qmult, tc_gmin, tc_tmin, tc_gmin2, tc_gargc, tc_groups, tc_cand, tc_qn, tc_amb, tc_ovf;
    float tc_cmax2 = 0.f;
    float tc_cscale = 1.f;      // power-of-two scale of the fp16 copy tc_cent
    // screening precision (dfx_tc.cu): tc_mode 0 = AUTO, 1 = FAST (one fp16 MMA per k-step),
    // 2 = PRECISE (hi/lo split, three MMAs).  AUTO starts PRECISE and moves to FAST once a launch
    // shows that FAST's wider tolerance would not overflow the kept groups (and back if it does).
    int tc_mode = 0;
    bool tc_fast = false;       // the precision the next screening launch uses (AUTO state)
    int tc_cent_npl = 0;        // planes currently held by tc_cent (0: none)
    int32_t* tc_stat_h = nullptr;      // pinned [2]: {overflow rows, rows that FAST would overflow} of a past launch
    cudaEvent_t tc_stat_ev = nullptr;
    bool tc_stat_pending = false, tc_stat_fast = false;
    int64_t tc_stat_rows = 0;
    int64_t tc_last_rows = 0, tc_last_overflow = 0, tc_last_fast_would = 0;  // of the last launch polled
    int64_t tc_auto_window = 16384;            // AUTO: rows observed before PRECISE may become FAST
    int64_t tc_acc_rows = 0, tc_acc_bad = 0;   // AUTO: rows / rows that (would) overflow since the last decision
    bool tc_ready = false;
    bool tc_enabled = true;
    int rows_inflight = 0;      // vectors in flight per warp of scan_rows_kernel: 0 = by row size, else 4 / 8
    int il2_threads = 0;        // scan_pq_il2 CTA shape: 0 = default (env DFX_IL2_THREADS or 256), 256, 512
    int il2_prefetch = -1;      // L2 prefetch distance in blocks: -1 = default (env DFX_IL2_PREFETCH or 4)
    bool flat_tc = true;        // FLAT: search through the tensor-core screening (dfx_tc_flat_candidates)
    int64_t tc_flat_rows = -1;  // rows covered by the fp16 copy of a FLAT index (-1: none)

    // scan-kernel profiling (dfx_profile_enable)
    bool prof_on = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    size_t prof_used = 0;

    // last-search bookkeeping
    int64_t last_nq = 0, last_nprobe = 0;
    bool last_keys_valid = false;

    // bumped by every call that can change what a search launches (train / add / finalize /
    // import / set_param / set_nprobe): CUDA-graph replays of a search are keyed on it
    std::atomic<long long> generation{0};

    cudaStream_t stream = nullptr;  // used by the host-pointer entry points
    // stream of the most recent *_dev call; host-pointer entry points (which run on `stream`,
    // a non-blocking stream) wait for it first so that the two never race
    cudaStream_t last_dev_stream = nullptr;
    bool dev_work_pending = false;
    // An EVENT after the call's own work, not the stream: the caller may queue unrelated work
    // behind it on the same stream -- the search plane queues the wait for the NEXT header
    // broadcast, which only completes when the client rank sends one, and a socket search served
    // meanwhile by another thread of the same process must not wait for that (it deadlocked the
    // 2-GPU bench: rank 0 waited for the socket reply, rank 1's reply for rank 0's next header).
    cudaEvent_t dev_done = nullptr;
    bool dev_done_recorded = false;
    void note_dev(cudaStream_t st) {
        last_dev_stream = st;
        dev_work_pending = true;
        dev_done_recorded = false;
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) cudaGetLastError();
        if (cs != cudaStreamCaptureStatusNone) return;  // inside a graph capture: the capturing caller orders its replays
        if (!dev_done && cudaEventCreateWithFlags(&dev_done, cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            dev_done = nullptr;
        }
        if (dev_done && cudaEventRecord(dev_done, st) == cudaSuccess) dev_done_recorded = true;
        else cudaGetLastError();
    }
    // a *_dev call on a different stream than the previous one: order them
    void join_dev_if_other(cudaStream_t st) {
        if (dev_work_pending && st != last_dev_stream) join_dev();
    }
    void join_dev() {
        if (dev_work_pending) {
            if (dev_done_recorded) cudaEventSynchronize(dev_done);
            else cudaStreamSynchronize(last_dev_stream);
            dev_work_pending = false;
        }
    }
    std::mutex mu;

    size_t row_bytes() const {
        switch (cfg.kind) {
            case DFX_FLAT:
            case DFX_IVF_FLAT: return (size_t)cfg.d * 4;
            case DFX_IVF_PQ: return (size_t)M * nbits / 8;
            case DFX_IVF_SQ16: return (size_t)cfg.d * 2;
        }
        return 0;
    }
    int64_t ntotal() const { return n_sorted + n_pending; }
    bool is_ivf() const { return cfg.kind != DFX_FLAT; }
};

// ---- dfx_search.cu
// values[q][j] = ranking value of row (col0+j) of X for query q (IP: -q.x ; L2: |x|^2 - 2 q.x)
void dfx_launch_gemm_values(const float* Q, int64_t nq, const float* X, const float* xnorm,
                            int64_t ncols, int d, int metric, float* out, int64_t ld_out,
                            cudaStream_t st);
void dfx_launch_row_norms(const float* X, int64_t n, int d, float* out, cudaStream_t st);
// top-k columns per row of a values matrix -> keys int32[nrows,k] (and optional values)
void dfx_launch_select_cols(const float* vals, int64_t nrows, int n, int64_t ld, int k,
                            uint32_t col_base, int32_t* keys, float* kvals, uint64_t* comp_out,
                            int64_t comp_ld, cudaStream_t st);
void dfx_search_impl(dfx_index* idx, int64_t nq, const float* d_x, int64_t k, float* d_D,
                     int64_t* d_I, cudaStream_t st);
void dfx_merge_impl(int64_t S, int64_t nq, int64_t k, const float* d_D, const int64_t* d_I,
                    int negate, float* d_outD, int64_t* d_outI, cudaStream_t st);
void dfx_merge_packed_impl(int64_t R, int64_t S_loc, int64_t nq, int64_t k, const void* d_packed,
                           int64_t rank_stride, int64_t off_I, int negate, float* d_outD,
                           int64_t* d_outI, cudaStream_t st);
void dfx_encode_ids_impl(int64_t n, const int64_t* d_ids, int64_t tag, const int32_t* d_col,
                         int32_t drop_code, int64_t* d_out, cudaStream_t st);
void dfx_filter_compact_impl(int64_t nq, int64_t kin, int64_t kout, const float* d_D, const int64_t* d_I,
                             float* d_outD, int64_t* d_outI, int32_t* d_count, cudaStream_t st);
void dfx_map_ids_impl(int64_t n, const int64_t* d_ids, const int64_t* d_table, int64_t* d_out,
                      cudaStream_t st);
void dfx_stats_impl(dfx_index* idx, int64_t* ndis, cudaStream_t st);

void dfx_launch_select_comp(const uint64_t* comp, int64_t nrows, int n, int64_t ld, int k, int32_t* keys,
                            cudaStream_t st);

// Interleaved IVF-PQ block (M == 32 x 8 bit; M == 64 x 4 bit stores code pairs, dfx_il2_pair below):
// 32 vectors x 32 bytes = 1 KB, one lane per vector.
// Lane v of the scanning warp owns vector v of
// the block and walks its 32 subquantizers in the rotated order m = (t + v) & 31, t = 0..31, so
// that at every step the 32 lanes read 32 different table columns (bank == column).  Byte t of
// the lane's 32 code bytes therefore holds the code of subquantizer (t + v) & 31; the two 16-byte
// halves of all lanes are stored contiguously (bytes 0..511: t = 0..15 of lanes 0..31, bytes
// 512..1023: t = 16..31) so that each of the two 128-bit loads of a warp is one 512-byte run.
__host__ __device__ __forceinline__ int dfx_il2_byte(int v, int m) {
    const int t = (m - v) & 31;
    return (t >> 4) * 512 + v * 16 + (t & 15);
}
// (the `layout` argument of the C-ABI probe dfx_debug_il_byte is kept for compatibility; there is
// one block layout)
__host__ __device__ __forceinline__ int dfx_il_byte_of(int /*layout*/, int v, int m) { return dfx_il2_byte(v, m); }

// ---- PQ code format.  Every reader and writer of PQ codes goes through the helpers below.
// Row-major (exchange) form, faiss bit order (PQEncoderGeneric, LSB first): a row is M * nbits / 8
// bytes; at nbits = 8 byte m is code m, at nbits = 4 byte m >> 1 holds code m in its low nibble
// when m is even and in its high nibble when m is odd.
__host__ __device__ __forceinline__ int dfx_pq_code(const uint8_t* row, int m, int nbits) {
    return nbits == 8 ? (int)row[m] : (int)((row[m >> 1] >> ((m & 1) * 4)) & 15u);
}
// byte b of a 4-bit row from its two codes (sub-quantizers 2b and 2b + 1)
__host__ __device__ __forceinline__ uint8_t dfx_pq4_byte(int c_even, int c_odd) {
    return (uint8_t)(c_even | (c_odd << 4));
}
// code u (0..7) of 4-byte word w of a 4-bit row (sub-quantizer 8w + u; the row is little endian)
__host__ __device__ __forceinline__ int dfx_pq4_word_code(uint32_t word, int u) {
    return (int)((word >> (4 * u)) & 15u);
}
// Blocks of the fused M = 64 x 4-bit scan: byte dfx_il2_byte(v, p), p < 32, holds the PAIR
// c_p | c_{p+32} << 4 of vector v -- one byte per column of the pair table (dfx_scan_il2_dev.cuh),
// so the block bytes, offsets and addressing are those of the M = 32 x 8-bit blocks.
__host__ __device__ __forceinline__ uint8_t dfx_il2_pair(int c_p, int c_p32) { return (uint8_t)(c_p | (c_p32 << 4)); }
// code of sub-quantizer m < 64 in the pair byte of column m & 31
__host__ __device__ __forceinline__ int dfx_il2_pair_code(uint8_t pair, int m) { return (int)((pair >> ((m >> 5) * 4)) & 15u); }

// ---- dfx_scan_il.cu
bool dfx_il_wanted(const dfx_index* idx);
void dfx_pq_rm_to_il(dfx_index* idx, cudaStream_t st);
void dfx_pq_il_to_rm(dfx_index* idx, cudaStream_t st);
// ---- dfx_scan_il2.cu: K3 + K4 fused; returns true when it wrote the final (D, I) rows itself
bool dfx_launch_scan_pq_il2(dfx_index* idx, const float* xq, int64_t qc, const int32_t* keys, int nprobe, int G,
                            int ngroups, int k, int cap, uint64_t* part, float* outD, int64_t* outI,
                            cudaStream_t st);

// ---- dfx_tc.cu
bool dfx_tc_supported(int d);
void dfx_tc_stats_sync(dfx_index* idx);  // wait for and fold in the statistics of the last screening launch
void dfx_tc_prepare_centroids(dfx_index* idx, cudaStream_t st);
void dfx_tc_coarse_search(dfx_index* idx, const float* d_x, int64_t nq, int nprobe, int32_t* keys,
                          cudaStream_t st);
int dfx_tc_flat_candidates(dfx_index* idx, const float* d_x, int64_t nq, int k, cudaStream_t st);
void dfx_tc_assign(dfx_index* idx, int d, const float* d_cent, const float* d_cnorm, int64_t nlist, int metric,
                   int64_t n, const float* d_x, int32_t* d_assign, cudaStream_t st);

// ---- dfx_build.cu
void dfx_train_impl(dfx_index* idx, int64_t n, const float* d_x, cudaStream_t st);
void dfx_add_impl(dfx_index* idx, int64_t n, const float* d_x, cudaStream_t st);
void dfx_finalize_impl(dfx_index* idx, cudaStream_t st);
// tag < 0: d_ids are shard-local ids (unknown / -1 rows become NaN); tag >= 0: d_ids are exchange
// ids and only the rows owned by shard `tag` are written
void dfx_reconstruct_impl(dfx_index* idx, int64_t n, const int64_t* d_ids, float* d_out,
                          cudaStream_t st, int64_t tag = -1);
// fused nearest-centroid (GEMM + argmin epilogue), no values matrix
void dfx_launch_assign_fused(const float* X, int64_t n, const float* cent, const float* cnorm,
                             int64_t nlist, int d, int metric, unsigned long long* best,
                             int32_t* out, cudaStream_t st);
void dfx_assign_impl(dfx_index* idx, const float* d_cent, const float* d_cnorm, int64_t nlist,
                     int metric, int d, int64_t n, const float* d_x, int32_t* d_assign,
                     cudaStream_t st);
void dfx_compute_tvals_sorted(dfx_index* idx, cudaStream_t st);
