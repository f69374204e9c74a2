// dfx_api.cu -- extern "C" surface of libdfx.so (include/dfx.h) + synthetic data generator.
#include "dfx_internal.h"
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <vector>

static thread_local std::string g_last_error;
std::atomic<long long> g_dfx_launches{0};

void dfx_set_error(const std::string& msg) { g_last_error = msg; }

#define DFX_API_BEGIN try {
#define DFX_API_END                                   \
    }                                                 \
    catch (const DfxError& e) {                       \
        g_last_error = e.msg;                         \
        return 1;                                     \
    }                                                 \
    catch (const std::exception& e) {                 \
        g_last_error = std::string("dfx: ") + e.what(); \
        return 2;                                     \
    }                                                 \
    return 0;

static void require_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        throw DfxError{std::string("libdfx needs a CUDA device (no CPU fallback): ") +
                       (e != cudaSuccess ? cudaGetErrorString(e) : "no device found")};
    DFX_REQUIRE(device >= 0 && device < n, "bad device ordinal " + std::to_string(device));
    cudaDeviceProp p;
    DFX_CUDA(cudaGetDeviceProperties(&p, device));
    DFX_REQUIRE(p.major == 10, std::string("libdfx is built for sm_100a only; device is sm_") +
                                   std::to_string(p.major) + std::to_string(p.minor));
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

extern "C" {

const char* dfx_last_error(void) { return g_last_error.c_str(); }
#ifndef DFX_SRC_HASH
#define DFX_SRC_HASH "unknown"
#endif
// ends with the hash of the sources the library was compiled from (build.py: source_hash)
const char* dfx_version(void) { return "dfx 0.2 (sm_100a) dfx-src-sha256=" DFX_SRC_HASH; }
int64_t dfx_launch_count(void) { return (int64_t)g_dfx_launches.load(); }
int dfx_debug_il_byte(int layout, int v, int m) { return dfx_il_byte_of(layout, v & 31, m & 31); }

int dfx_create(const dfx_cfg* cfg, dfx_index** out) {
    DFX_API_BEGIN
    DFX_REQUIRE(cfg && out, "null argument");
    DFX_REQUIRE(cfg->kind >= DFX_FLAT && cfg->kind <= DFX_IVF_SQ16, "unknown index kind");
    DFX_REQUIRE(cfg->metric == DFX_METRIC_IP || cfg->metric == DFX_METRIC_L2,
                "Only dot and l2 metrics are supported.");
    DFX_REQUIRE(cfg->d > 0 && cfg->d <= 4096, "dimension must be in [1, 4096]");
    require_device(cfg->device);
    std::unique_ptr<dfx_index> idx(new dfx_index());
    idx->cfg = *cfg;
    if (cfg->kind != DFX_FLAT) {
        DFX_REQUIRE(cfg->nlist >= 1 && cfg->nlist < (1ll << 24), "nlist must be in [1, 2^24)");
        DFX_REQUIRE(cfg->d % 4 == 0, "IVF indexes need a dimension that is a multiple of 4");
    }
    if (cfg->kind == DFX_IVF_PQ) {
        DFX_REQUIRE(cfg->pq_nbits == 8 || cfg->pq_nbits == 4,
                    "IVF-PQ: bits per sub-quantizer must be 4 or 8, got " + std::to_string(cfg->pq_nbits));
        DFX_REQUIRE(cfg->pq_m >= 4 && cfg->pq_m % 4 == 0 && cfg->d % cfg->pq_m == 0,
                    "IVF-PQ: the number of sub-quantizers must be a multiple of 4 that divides d");
        DFX_REQUIRE(cfg->pq_m <= 64, "IVF-PQ: at most 64 sub-quantizers are supported");
        // 4-bit rows are M / 2 bytes; M % 8 == 0 keeps them whole 4-byte words (finalize, scan loads)
        DFX_REQUIRE(cfg->pq_nbits == 8 || cfg->pq_m % 8 == 0,
                    "IVF-PQ with 4-bit codes: the number of sub-quantizers must be a multiple of 8, got " +
                        std::to_string(cfg->pq_m));
        idx->M = cfg->pq_m;
        idx->nbits = cfg->pq_nbits;
        idx->ksub = 1 << cfg->pq_nbits;
        idx->dsub = cfg->d / cfg->pq_m;
    }
    DeviceGuard g(cfg->device);
    DFX_CUDA(cudaStreamCreateWithFlags(&idx->stream, cudaStreamNonBlocking));
    *out = idx.release();
    DFX_API_END
}

void dfx_destroy(dfx_index* idx) {
    if (!idx) return;
    {
        DeviceGuard g(idx->cfg.device);
        if (idx->stream) {
            cudaStreamSynchronize(idx->stream);
            cudaStreamDestroy(idx->stream);
        }
        for (auto& e : idx->prof_events) {
            cudaEventDestroy(e.first);
            cudaEventDestroy(e.second);
        }
        if (idx->tc_stat_ev) cudaEventDestroy(idx->tc_stat_ev);
        if (idx->dev_done) cudaEventDestroy(idx->dev_done);
        if (idx->tc_stat_h) cudaFreeHost(idx->tc_stat_h);
        delete idx;
    }
}

int dfx_set_param(dfx_index* idx, const char* name, double value) {
    DFX_API_BEGIN
    idx->generation++;
    std::string n(name);
    if (n == "kmeans_niter") idx->kmeans_niter = (int)value;
    else if (n == "max_points_per_centroid") idx->max_points_per_centroid = (int)value;
    else if (n == "train_seed") idx->train_seed = (uint64_t)value;
    else if (n == "tensor_cores") idx->tc_enabled = value != 0;
    else if (n == "interleaved") {
        std::lock_guard<std::mutex> lk(idx->mu);
        DeviceGuard g(idx->cfg.device);
        idx->join_dev();
        idx->il_enabled = value != 0;
        if (!idx->il_enabled) dfx_pq_il_to_rm(idx, idx->stream);
        else if (idx->trained && idx->n_pending == 0 && idx->n_sorted > 0) dfx_pq_rm_to_il(idx, idx->stream);
    }
    else if (n == "flat_tensor_cores") idx->flat_tc = value != 0;
    else if (n == "rows_inflight") {
        DFX_REQUIRE(value == 0 || value == 4 || value == 8, "rows_inflight must be 0 (by row size), 4 or 8");
        idx->rows_inflight = (int)value;
    }
    else if (n == "tc_screen_mode") {  // 0 = AUTO, 1 = FAST (one fp16 MMA), 2 = PRECISE (hi/lo split, three MMAs)
        DFX_REQUIRE(value == 0 || value == 1 || value == 2, "tc_screen_mode must be 0 (auto), 1 (fast) or 2 (precise)");
        idx->tc_mode = (int)value;
        idx->tc_fast = value == 1;
        idx->tc_stat_pending = false;
        idx->tc_acc_rows = idx->tc_acc_bad = 0;
    }
    else if (n == "tc_auto_window") {
        DFX_REQUIRE(value >= 1 && value <= (double)(1 << 30), "tc_auto_window must be 1 .. 2^30 rows");
        idx->tc_auto_window = (int64_t)value;
        idx->tc_acc_rows = idx->tc_acc_bad = 0;
    }
    else if (n == "il2_threads") {
        DFX_REQUIRE(value == 0 || value == 256 || value == 512, "il2_threads must be 0 (default), 256 or 512");
        idx->il2_threads = (int)value;
    }
    else if (n == "il2_prefetch") {
        DFX_REQUIRE(value >= -1 && value <= 32, "il2_prefetch must be -1 (default) or 0..32 blocks");
        idx->il2_prefetch = (int)value;
    }
    else throw DfxError{"unknown parameter " + n};
    DFX_API_END
}

int dfx_get_param(dfx_index* idx, const char* name, double* value) {
    DFX_API_BEGIN
    DFX_REQUIRE(idx && name && value, "null argument");
    std::string n(name);
    if (n.rfind("tc_stat_", 0) == 0 || n == "tc_fast") {
        DeviceGuard g(idx->cfg.device);
        dfx_tc_stats_sync(idx);  // fold the outstanding launch statistics in (AUTO precision)
    }
    if (n == "kmeans_niter") *value = idx->kmeans_niter;
    else if (n == "max_points_per_centroid") *value = idx->max_points_per_centroid;
    else if (n == "train_seed") *value = (double)idx->train_seed;
    else if (n == "tensor_cores") *value = idx->tc_enabled;
    else if (n == "tc_screen_mode") *value = idx->tc_mode;
    else if (n == "tc_fast") *value = idx->tc_fast;
    else if (n == "tc_auto_window") *value = (double)idx->tc_auto_window;
    else if (n == "tc_cmax2") *value = idx->tc_cmax2;
    else if (n == "tc_stat_rows") *value = (double)idx->tc_last_rows;
    else if (n == "tc_stat_overflow") *value = (double)idx->tc_last_overflow;
    else if (n == "tc_stat_fast_would") *value = (double)idx->tc_last_fast_would;
    else if (n == "flat_tensor_cores") *value = idx->flat_tc;
    else if (n == "interleaved") *value = idx->il_enabled;
    else if (n == "il2_threads") *value = idx->il2_threads;
    else if (n == "il2_prefetch") *value = idx->il2_prefetch;
    else if (n == "rows_inflight") *value = idx->rows_inflight;
    else throw DfxError{"unknown parameter " + n};
    DFX_API_END
}

int dfx_train_dev(dfx_index* idx, int64_t n, const float* d_x, void* stream) {
    DFX_API_BEGIN
    idx->generation++;
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev_if_other((cudaStream_t)stream);
    dfx_train_impl(idx, n, d_x, (cudaStream_t)stream);
    idx->note_dev((cudaStream_t)stream);
    DFX_API_END
}
int dfx_add_dev(dfx_index* idx, int64_t n, const float* d_x, void* stream) {
    DFX_API_BEGIN
    idx->generation++;
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev_if_other((cudaStream_t)stream);
    dfx_add_impl(idx, n, d_x, (cudaStream_t)stream);
    idx->note_dev((cudaStream_t)stream);
    DFX_API_END
}
int dfx_train(dfx_index* idx, int64_t n, const float* x) {
    DFX_API_BEGIN
    idx->generation++;
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    DevBuf buf;
    buf.reserve((size_t)std::max<int64_t>(n, 1) * idx->cfg.d * 4);
    DFX_CUDA(cudaMemcpyAsync(buf.p, x, (size_t)n * idx->cfg.d * 4, cudaMemcpyHostToDevice, idx->stream));
    dfx_train_impl(idx, n, buf.as<float>(), idx->stream);
    DFX_CUDA(cudaStreamSynchronize(idx->stream));
    DFX_API_END
}
int dfx_add(dfx_index* idx, int64_t n, const float* x) {
    DFX_API_BEGIN
    idx->generation++;
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    const int64_t chunk = 1 << 20;
    DevBuf buf;
    buf.reserve((size_t)std::min<int64_t>(std::max<int64_t>(n, 1), chunk) * idx->cfg.d * 4);
    for (int64_t i0 = 0; i0 < n; i0 += chunk) {
        int64_t c = std::min(chunk, n - i0);
        DFX_CUDA(cudaMemcpyAsync(buf.p, x + i0 * idx->cfg.d, (size_t)c * idx->cfg.d * 4,
                                 cudaMemcpyHostToDevice, idx->stream));
        dfx_add_impl(idx, c, buf.as<float>(), idx->stream);
        DFX_CUDA(cudaStreamSynchronize(idx->stream));
    }
    DFX_API_END
}
int dfx_reserve(dfx_index* idx, int64_t n_total) {
    DFX_API_BEGIN
    idx->reserve_hint = n_total;
    DFX_API_END
}
int dfx_finalize(dfx_index* idx, void* stream) {
    DFX_API_BEGIN
    idx->generation++;
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    cudaStream_t st = stream ? (cudaStream_t)stream : idx->stream;
    dfx_finalize_impl(idx, st);
    DFX_CUDA(cudaStreamSynchronize(st));
    DFX_API_END
}

int dfx_search_dev(dfx_index* idx, int64_t nq, const float* d_x, int64_t k, float* d_D, int64_t* d_I,
                   void* stream) {
    DFX_API_BEGIN
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev_if_other((cudaStream_t)stream);
    dfx_search_impl(idx, nq, d_x, k, d_D, d_I, (cudaStream_t)stream);
    idx->note_dev((cudaStream_t)stream);
    DFX_API_END
}
int dfx_search(dfx_index* idx, int64_t nq, const float* x, int64_t k, float* D, int64_t* I) {
    DFX_API_BEGIN
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    if (nq <= 0) return 0;
    DFX_REQUIRE(k >= 1, "k must be >= 1");
    const int d = idx->cfg.d;
    idx->w_q.reserve((size_t)nq * d * 4);
    idx->w_D.reserve((size_t)nq * k * 4);
    idx->w_I.reserve((size_t)nq * k * 8);
    DFX_CUDA(cudaMemcpyAsync(idx->w_q.p, x, (size_t)nq * d * 4, cudaMemcpyHostToDevice, idx->stream));
    dfx_search_impl(idx, nq, idx->w_q.as<float>(), k, idx->w_D.as<float>(), idx->w_I.as<int64_t>(),
                    idx->stream);
    DFX_CUDA(cudaMemcpyAsync(D, idx->w_D.p, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, idx->stream));
    DFX_CUDA(cudaMemcpyAsync(I, idx->w_I.p, (size_t)nq * k * 8, cudaMemcpyDeviceToHost, idx->stream));
    DFX_CUDA(cudaStreamSynchronize(idx->stream));
    DFX_API_END
}

int dfx_reconstruct(dfx_index* idx, int64_t n, const int64_t* ids, float* out) {
    DFX_API_BEGIN
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    if (n <= 0) return 0;
    DevBuf d_ids, d_out;
    d_ids.reserve((size_t)n * 8);
    d_out.reserve((size_t)n * idx->cfg.d * 4);
    DFX_CUDA(cudaMemcpyAsync(d_ids.p, ids, (size_t)n * 8, cudaMemcpyHostToDevice, idx->stream));
    dfx_reconstruct_impl(idx, n, d_ids.as<int64_t>(), d_out.as<float>(), idx->stream);
    DFX_CUDA(cudaMemcpyAsync(out, d_out.p, (size_t)n * idx->cfg.d * 4, cudaMemcpyDeviceToHost, idx->stream));
    DFX_CUDA(cudaStreamSynchronize(idx->stream));
    DFX_API_END
}

int dfx_reconstruct_dev(dfx_index* idx, int64_t n, const int64_t* d_ids, int64_t shard_tag, float* d_out,
                        void* stream) {
    DFX_API_BEGIN
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev_if_other((cudaStream_t)stream);
    dfx_reconstruct_impl(idx, n, d_ids, d_out, (cudaStream_t)stream, shard_tag);
    idx->note_dev((cudaStream_t)stream);
    DFX_API_END
}

int dfx_set_nprobe(dfx_index* idx, int64_t nprobe) {
    DFX_API_BEGIN
    idx->generation++;
    DFX_REQUIRE(nprobe >= 1, "nprobe must be >= 1");
    idx->nprobe = nprobe;
    DFX_API_END
}
int64_t dfx_get_nprobe(const dfx_index* idx) { return idx->nprobe; }
int64_t dfx_generation(const dfx_index* idx) { return (int64_t)idx->generation.load(); }
int64_t dfx_ntotal(const dfx_index* idx) { return idx->ntotal(); }
int64_t dfx_nlist(const dfx_index* idx) { return idx->cfg.kind == DFX_FLAT ? 0 : idx->cfg.nlist; }
int dfx_is_trained(const dfx_index* idx) { return (idx->trained || idx->cfg.kind == DFX_FLAT) ? 1 : 0; }

int dfx_get_centroids(dfx_index* idx, float* out) {
    DFX_API_BEGIN
    DFX_REQUIRE(idx->is_ivf() && idx->trained, "index has no trained coarse quantizer");
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    DFX_CUDA(cudaMemcpy(out, idx->centroids.p, (size_t)idx->cfg.nlist * idx->cfg.d * 4, cudaMemcpyDeviceToHost));
    DFX_API_END
}

int dfx_merge_dev(int64_t S, int64_t nq, int64_t k, const float* d_D, const int64_t* d_I, int negate,
                  float* d_outD, int64_t* d_outI, void* stream) {
    DFX_API_BEGIN
    dfx_merge_impl(S, nq, k, d_D, d_I, negate, d_outD, d_outI, (cudaStream_t)stream);
    DFX_API_END
}
int dfx_merge(int64_t S, int64_t nq, int64_t k, const float* D, const int64_t* I, int negate, float* outD,
              int64_t* outI) {
    DFX_API_BEGIN
    int dev = 0;
    DFX_CUDA(cudaGetDevice(&dev));
    require_device(dev);
    if (nq <= 0) return 0;
    DevBuf dD, dI, oD, oI;
    size_t n = (size_t)S * nq * k;
    dD.reserve(n * 4);
    dI.reserve(n * 8);
    oD.reserve((size_t)nq * k * 4);
    oI.reserve((size_t)nq * k * 8);
    DFX_CUDA(cudaMemcpy(dD.p, D, n * 4, cudaMemcpyHostToDevice));
    DFX_CUDA(cudaMemcpy(dI.p, I, n * 8, cudaMemcpyHostToDevice));
    dfx_merge_impl(S, nq, k, dD.as<float>(), dI.as<int64_t>(), negate, oD.as<float>(), oI.as<int64_t>(), 0);
    DFX_CUDA(cudaMemcpy(outD, oD.p, (size_t)nq * k * 4, cudaMemcpyDeviceToHost));
    DFX_CUDA(cudaMemcpy(outI, oI.p, (size_t)nq * k * 8, cudaMemcpyDeviceToHost));
    DFX_API_END
}
int dfx_merge_packed_dev(int64_t R, int64_t S_loc, int64_t nq, int64_t k, const void* d_packed,
                         int64_t rank_stride_bytes, int64_t off_I_bytes, int negate, float* d_outD,
                         int64_t* d_outI, void* stream) {
    DFX_API_BEGIN
    dfx_merge_packed_impl(R, S_loc, nq, k, d_packed, rank_stride_bytes, off_I_bytes, negate, d_outD, d_outI,
                          (cudaStream_t)stream);
    DFX_API_END
}
int dfx_encode_ids_dev(int64_t n, const int64_t* d_ids, int64_t shard_tag, const int32_t* d_col,
                       int32_t drop_code, int64_t* d_out, void* stream) {
    DFX_API_BEGIN
    dfx_encode_ids_impl(n, d_ids, shard_tag, d_col, drop_code, d_out, (cudaStream_t)stream);
    DFX_API_END
}
int dfx_filter_compact_dev(int64_t nq, int64_t k_in, int64_t k_out, const float* d_D, const int64_t* d_I,
                           float* d_outD, int64_t* d_outI, int32_t* d_count, void* stream) {
    DFX_API_BEGIN
    dfx_filter_compact_impl(nq, k_in, k_out, d_D, d_I, d_outD, d_outI, d_count, (cudaStream_t)stream);
    DFX_API_END
}
int dfx_map_ids_dev(int64_t n, const int64_t* d_ids, const int64_t* d_table, int64_t* d_out, void* stream) {
    DFX_API_BEGIN
    dfx_map_ids_impl(n, d_ids, d_table, d_out, (cudaStream_t)stream);
    DFX_API_END
}

int dfx_last_stats(dfx_index* idx, int64_t* ndis, int64_t* nq, int64_t* nprobe) {
    DFX_API_BEGIN
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    int64_t nd = 0;
    dfx_stats_impl(idx, &nd, idx->stream);
    if (ndis) *ndis = nd;
    if (nq) *nq = idx->last_nq;
    if (nprobe) *nprobe = idx->last_nprobe;
    DFX_API_END
}

int dfx_profile_enable(dfx_index* idx, int on) {
    DFX_API_BEGIN
    std::lock_guard<std::mutex> lk(idx->mu);
    idx->prof_on = on != 0;
    DFX_API_END
}
int dfx_profile_read(dfx_index* idx, double* scan_ms, int64_t* scan_launches, int reset) {
    DFX_API_BEGIN
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    double ms = 0;
    for (size_t i = 0; i < idx->prof_used; i++) {
        DFX_CUDA(cudaEventSynchronize(idx->prof_events[i].second));
        float t = 0;
        DFX_CUDA(cudaEventElapsedTime(&t, idx->prof_events[i].first, idx->prof_events[i].second));
        ms += t;
    }
    if (scan_ms) *scan_ms = ms;
    if (scan_launches) *scan_launches = (int64_t)idx->prof_used;
    if (reset) idx->prof_used = 0;
    DFX_API_END
}

// ------------------------------------------------------------------ state exchange
static const char* payload_name(int kind) {
    switch (kind) {
        case DFX_FLAT: return "xb";
        case DFX_IVF_FLAT: return "vecs";
        case DFX_IVF_PQ: return "codes";
        case DFX_IVF_SQ16: return "codes16";
    }
    return "";
}

int dfx_get_array(dfx_index* idx, const char* name, void* out, int64_t max_bytes, int64_t* nbytes) {
    DFX_API_BEGIN
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    if (idx->n_pending > 0) dfx_finalize_impl(idx, idx->stream);
    std::string n(name);
    struct Restore {  // the exchange format is row-major; put the interleaved form back afterwards
        dfx_index* i;
        bool on;
        ~Restore() {
            if (on) {
                try {
                    dfx_pq_rm_to_il(i, i->stream);
                } catch (...) {
                }
            }
        }
    } restore{idx, false};
    if (idx->il && (n == "codes" || n == "tvals" || n == "ids")) {
        dfx_pq_il_to_rm(idx, idx->stream);
        restore.on = true;
    }
    const int64_t nt = idx->n_sorted, nlist = idx->cfg.nlist, d = idx->cfg.d;
    const void* src = nullptr;
    int64_t bytes = 0;
    bool widen_ids = false;
    if (n == "centroids" && idx->is_ivf() && idx->trained) { src = idx->centroids.p; bytes = nlist * d * 4; }
    else if (n == "codebooks" && idx->cfg.kind == DFX_IVF_PQ && idx->trained) { src = idx->codebooks.p; bytes = (int64_t)idx->M * idx->ksub * idx->dsub * 4; }
    else if (n == "list_off" && idx->is_ivf() && idx->trained) { src = idx->list_off.p; bytes = (nlist + 1) * 8; }
    else if (n == "ids" && idx->is_ivf()) { widen_ids = true; bytes = nt * 8; }
    else if (n == "tvals" && idx->cfg.kind == DFX_IVF_PQ) { src = idx->tvals.p; bytes = nt * 4; }
    else if (n == payload_name(idx->cfg.kind)) { src = idx->payload.p; bytes = nt * (int64_t)idx->row_bytes(); }
    else throw DfxError{"no array named '" + n + "' in this index"};
    if (nbytes) *nbytes = bytes;
    if (!out) return 0;
    DFX_REQUIRE(max_bytes >= bytes, "output buffer too small for '" + n + "'");
    if (bytes == 0) return 0;
    if (widen_ids) {
        std::vector<int32_t> tmp((size_t)nt);
        DFX_CUDA(cudaMemcpy(tmp.data(), idx->ids.p, (size_t)nt * 4, cudaMemcpyDeviceToHost));
        int64_t* o = (int64_t*)out;
        for (int64_t i = 0; i < nt; i++) o[i] = tmp[(size_t)i];
    } else {
        DFX_CUDA(cudaMemcpy(out, src, (size_t)bytes, cudaMemcpyDeviceToHost));
    }
    DFX_API_END
}

int dfx_set_array(dfx_index* idx, const char* name, const void* in, int64_t nbytes) {
    DFX_API_BEGIN
    idx->generation++;
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    std::string n(name);
    if (idx->il) dfx_pq_il_to_rm(idx, idx->stream);  // imports arrive row-major
    const int64_t nlist = idx->cfg.nlist, d = idx->cfg.d;
    auto upload = [&](DevBuf& b, int64_t bytes) {
        b.reserve((size_t)std::max<int64_t>(bytes, 4));
        if (bytes) DFX_CUDA(cudaMemcpy(b.p, in, (size_t)bytes, cudaMemcpyHostToDevice));
    };
    if (n == "centroids" && idx->is_ivf()) {
        DFX_REQUIRE(nbytes == nlist * d * 4, "centroids: wrong size");
        upload(idx->centroids, nbytes);
        idx->cnorm.reserve((size_t)nlist * 4);
        dfx_launch_row_norms(idx->centroids.as<float>(), nlist, (int)d, idx->cnorm.as<float>(), idx->stream);
        DFX_CUDA(cudaStreamSynchronize(idx->stream));
    } else if (n == "codebooks" && idx->cfg.kind == DFX_IVF_PQ) {
        DFX_REQUIRE(nbytes == (int64_t)idx->M * idx->ksub * idx->dsub * 4, "codebooks: wrong size");
        upload(idx->codebooks, nbytes);
        idx->cbT_valid = false;
    } else if (n == "list_off" && idx->is_ivf()) {
        DFX_REQUIRE(nbytes == (nlist + 1) * 8, "list_off: wrong size");
        upload(idx->list_off, nbytes);
        idx->h_list_off.assign((const int64_t*)in, (const int64_t*)in + nlist + 1);
        DFX_REQUIRE(idx->h_list_off[0] == 0, "list_off[0] must be 0");
        idx->n_sorted = idx->h_list_off[(size_t)nlist];
        idx->n_pending = 0;
    } else if (n == "ids" && idx->is_ivf()) {
        DFX_REQUIRE(nbytes == idx->n_sorted * 8, "ids: wrong size (set list_off first)");
        std::vector<int32_t> tmp((size_t)idx->n_sorted);
        const int64_t* s = (const int64_t*)in;
        for (int64_t i = 0; i < idx->n_sorted; i++) {
            DFX_REQUIRE(s[i] >= 0 && s[i] < (1ll << 31), "ids must be in [0, 2^31)");
            tmp[(size_t)i] = (int32_t)s[i];
        }
        idx->ids.reserve((size_t)std::max<int64_t>(idx->n_sorted, 1) * 4);
        if (idx->n_sorted)
            DFX_CUDA(cudaMemcpy(idx->ids.p, tmp.data(), (size_t)idx->n_sorted * 4, cudaMemcpyHostToDevice));
    } else if (n == payload_name(idx->cfg.kind)) {
        if (idx->cfg.kind == DFX_FLAT) {
            DFX_REQUIRE(nbytes % (d * 4) == 0, "xb: wrong size");
            idx->n_sorted = nbytes / (d * 4);
            idx->tc_flat_rows = -1;  // imported rows: any bf16 planes are stale
            upload(idx->payload, nbytes);
            if (idx->cfg.metric == DFX_METRIC_L2) {
                idx->xnorm.reserve((size_t)std::max<int64_t>(idx->n_sorted, 1) * 4);
                dfx_launch_row_norms(idx->payload.as<float>(), idx->n_sorted, (int)d, idx->xnorm.as<float>(), idx->stream);
                DFX_CUDA(cudaStreamSynchronize(idx->stream));
            }
        } else {
            DFX_REQUIRE(nbytes == idx->n_sorted * (int64_t)idx->row_bytes(), "payload: wrong size (set list_off first)");
            upload(idx->payload, nbytes);
        }
    } else {
        throw DfxError{"cannot import array '" + n + "'"};
    }
    idx->inv_valid = false;
    DFX_API_END
}

int dfx_import_done(dfx_index* idx) {
    DFX_API_BEGIN
    idx->generation++;
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->cfg.device);
    idx->join_dev();
    if (idx->is_ivf()) {
        DFX_REQUIRE(idx->centroids.p && idx->list_off.p, "import: centroids and list_off are required");
        if (idx->cfg.kind == DFX_IVF_PQ) {
            DFX_REQUIRE(idx->codebooks.p, "import: codebooks are required");
            dfx_compute_tvals_sorted(idx, idx->stream);  // K7 recomputes the per-vector term
            dfx_pq_rm_to_il(idx, idx->stream);
        }
        dfx_tc_prepare_centroids(idx, idx->stream);
        DFX_CUDA(cudaStreamSynchronize(idx->stream));
    }
    idx->trained = true;
    DFX_API_END
}

int dfx_free(void* p) {
    DFX_API_BEGIN
    if (p) DFX_CUDA(cudaFree(p));
    DFX_API_END
}

}  // extern "C"

// =====================================================================================
// synthetic data (bench harness).  Stateless: every value is a hash of (seed, stream, row, j).
// =====================================================================================
__host__ __device__ static inline uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
__host__ __device__ static inline uint64_t hash4(uint64_t seed, uint64_t stream, uint64_t a, uint64_t b) {
    uint64_t h = mix64(seed + 0x9e3779b97f4a7c15ull);
    h = mix64(h ^ (stream * 0xd1342543de82ef95ull + 0x632be59bd9b4e019ull));
    h = mix64(h ^ (a * 0x9e3779b97f4a7c15ull));
    h = mix64(h ^ (b * 0xc2b2ae3d27d4eb4full + 0x165667b19e3779f9ull));
    return h;
}
// standard normal from one 64-bit hash (Box-Muller on two 32-bit halves)
__device__ static inline float hash_normal(uint64_t h) {
    float u1 = ((float)(uint32_t)(h >> 32) + 0.5f) * (1.0f / 4294967296.0f);
    float u2 = ((float)(uint32_t)h + 0.5f) * (1.0f / 4294967296.0f);
    return sqrtf(-2.0f * __logf(u1)) * __cosf(6.28318530718f * u2);
}

// one CTA (128 threads) per row, d <= 4096, r <= 64
__global__ void synth_rows_kernel(dfx_synth p, const float* __restrict__ A, int64_t row0,
                                  const int64_t* __restrict__ rows, int64_t n, uint64_t noise_stream,
                                  float* __restrict__ out) {
    __shared__ float s_z[64];
    const int64_t r = blockIdx.x;
    if (r >= n) return;
    const int64_t row = rows ? rows[r] : row0 + r;
    const uint64_t cluster = (uint64_t)(row % p.nclusters);
    const uint64_t zkey = p.ngroups > 0 ? (uint64_t)(row % p.ngroups) : (uint64_t)row;
    if (threadIdx.x < p.r) {
        float z = hash_normal(hash4(p.seed, 2, zkey, threadIdx.x));
        z = p.sigma * fminf(4.f, fmaxf(-4.f, z));
        if (p.delta > 0.f) z += p.delta * hash_normal(hash4(p.seed, 5, (uint64_t)row, threadIdx.x));
        s_z[threadIdx.x] = z;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < p.d; k += blockDim.x) {
        float mu = hash_normal(hash4(p.seed, 1, cluster, k));
        float az = 0.f;
        for (int j = 0; j < p.r; j++) az += A[k * p.r + j] * s_z[j];
        float v = mu + az;
        if (p.eps > 0.f) v += p.eps * hash_normal(hash4(p.seed, 4, (uint64_t)row, k));
        if (p.sigma_q > 0.f && noise_stream)
            v += p.sigma_q * hash_normal(hash4(p.seed, noise_stream, (uint64_t)row, k));
        out[r * p.d + k] = v;
    }
}

extern "C" {

// A: d x r with orthonormal columns (Gram-Schmidt of a hashed Gaussian matrix, on the host)
int dfx_synth_init(const dfx_synth* p, float** d_A_out, void* stream) {
    DFX_API_BEGIN
    DFX_REQUIRE(p && d_A_out, "null argument");
    DFX_REQUIRE(p->r >= 1 && p->r <= 64 && p->r <= p->d && p->d <= 4096, "synth: need 1 <= r <= min(64, d)");
    const int d = p->d, r = p->r;
    std::vector<double> A((size_t)d * r);
    for (int k = 0; k < d; k++)
        for (int j = 0; j < r; j++) {
            uint64_t h = hash4(p->seed, 3, (uint64_t)k, (uint64_t)j);
            double u1 = ((double)(uint32_t)(h >> 32) + 0.5) / 4294967296.0;
            double u2 = ((double)(uint32_t)h + 0.5) / 4294967296.0;
            A[(size_t)k * r + j] = std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586 * u2);
        }
    for (int j = 0; j < r; j++) {
        for (int j2 = 0; j2 < j; j2++) {
            double dot = 0;
            for (int k = 0; k < d; k++) dot += A[(size_t)k * r + j] * A[(size_t)k * r + j2];
            for (int k = 0; k < d; k++) A[(size_t)k * r + j] -= dot * A[(size_t)k * r + j2];
        }
        double nrm = 0;
        for (int k = 0; k < d; k++) nrm += A[(size_t)k * r + j] * A[(size_t)k * r + j];
        nrm = std::sqrt(nrm);
        for (int k = 0; k < d; k++) A[(size_t)k * r + j] /= nrm;
    }
    std::vector<float> Af(A.begin(), A.end());
    float* dA = nullptr;
    DFX_CUDA(cudaMalloc(&dA, Af.size() * 4));
    DFX_CUDA(cudaMemcpyAsync(dA, Af.data(), Af.size() * 4, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    DFX_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    *d_A_out = dA;
    DFX_API_END
}

int dfx_synth_rows_dev(const dfx_synth* p, const float* d_A, int64_t row0, const int64_t* d_rows, int64_t n,
                       uint64_t noise_stream, float* d_out, void* stream) {
    DFX_API_BEGIN
    if (n <= 0) return 0;
    DFX_REQUIRE(p->nclusters >= 1, "synth: nclusters >= 1");
    DFX_REQUIRE(p->ngroups == 0 || p->ngroups % p->nclusters == 0, "synth: ngroups must be a multiple of nclusters");
    DFX_LAUNCH(synth_rows_kernel, (unsigned)n, 128, 0, (cudaStream_t)stream, *p, d_A, row0, d_rows, n,
               noise_stream, d_out);
    DFX_API_END
}

}  // extern "C"
