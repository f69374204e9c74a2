// dfx_scan_il2.cu -- launcher of the IVF-PQ (M == 32 x 8 bit, M == 64 x 4 bit) table build +
// inverted-list scan, K3 + K4.
// Kernel: dfx_scan_il2_dev.cuh.
#include "dfx_scan_il2_dev.cuh"
#include <cstdlib>

template <bool REG, int THREADS, int MINB, bool PQ4>
static void launch_il2_t(dfx_index* idx, const float* xq, int64_t qc, const int32_t* keys, int nprobe, int G,
                       int ngroups, int k, int cap, uint64_t* part, float* outD, int64_t* outI, cudaStream_t st) {
    constexpr int NW = THREADS / 32;
    const size_t smem = (size_t)IL2_LUT_BYTES + (REG ? (size_t)NW * IL2_QCAP * 8 : (size_t)NW * cap * 8);
    auto kern = scan_pq_il2_kernel<REG, THREADS, MINB, PQ4>;
    DFX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DFX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    // blocks the L2 prefetch cursor runs ahead of the register loads (0 = off; DFX_IL2_PREFETCH)
    static const int pf_default = [] {
        const char* e = getenv("DFX_IL2_PREFETCH");
        const int v = e ? atoi(e) : 4;
        return v < 0 ? 0 : (v > 32 ? 32 : v);
    }();
    const int pf_ahead = idx->il2_prefetch >= 0 ? idx->il2_prefetch : pf_default;
    DFX_LAUNCH(kern, (unsigned)(qc * ngroups), THREADS, smem, st, xq, idx->codebooksT.as<float>(),
               idx->centroids.as<float>(), idx->cfg.d, idx->dsub, keys, nprobe, G, ngroups, idx->blk_off.as<int64_t>(),
               idx->il_codes.as<uint4>(), idx->il_tvals.as<float>(), idx->il_ids.as<int32_t>(), k, cap, part, outD, outI,
               pf_ahead);
}

// CTA shape: 256 threads x 3 CTAs per SM (default) or, DFX_IL2_THREADS=512, 512 threads x 2 CTAs
// (16 warps share one query's table: 32 instead of 24 warps per SM, half the table builds per SM)
template <bool REG, bool PQ4>
static void launch_il2(dfx_index* idx, const float* xq, int64_t qc, const int32_t* keys, int nprobe, int G,
                       int ngroups, int k, int cap, uint64_t* part, float* outD, int64_t* outI, cudaStream_t st) {
    static const int threads_default = [] {
        const char* e = getenv("DFX_IL2_THREADS");
        return e ? atoi(e) : IL2_THREADS;
    }();
    const int threads = idx->il2_threads ? idx->il2_threads : threads_default;
    if (threads == 512) launch_il2_t<REG, 512, 2, PQ4>(idx, xq, qc, keys, nprobe, G, ngroups, k, cap, part, outD, outI, st);
    else launch_il2_t<REG, 256, 3, PQ4>(idx, xq, qc, keys, nprobe, G, ngroups, k, cap, part, outD, outI, st);
}

// outD / outI: when ngroups == 1 and k <= 32 the kernel writes the final rows there and the
// function returns true (the caller skips the per-query reduction of `part`).
bool dfx_launch_scan_pq_il2(dfx_index* idx, const float* xq, int64_t qc, const int32_t* keys, int nprobe, int G,
                            int ngroups, int k, int cap, uint64_t* part, float* outD, int64_t* outI,
                            cudaStream_t st) {
    DFX_REQUIRE(G <= IL2_MAXG, "scan_pq_il2: more than 16 probes per CTA");
    const bool pq4 = idx->nbits == 4;
    DFX_REQUIRE(((idx->M == 32 && idx->nbits == 8) || (idx->M == 64 && pq4)) && idx->cfg.d == idx->M * idx->dsub,
                "scan_pq_il2: M == 32 x 8 bit or M == 64 x 4 bit only");
    if (!idx->cbT_valid) {  // transposed codebook PT[j][m][dsub], once per trained / imported codebook
        const int tot = idx->M * idx->ksub * idx->dsub;
        idx->codebooksT.reserve((size_t)tot * 4);
        DFX_LAUNCH(cb_transpose_kernel, (unsigned)((tot + 255) / 256), 256, 0, st, idx->codebooks.as<float>(), idx->M,
                   idx->ksub, idx->dsub, idx->codebooksT.as<float>());
        idx->cbT_valid = true;
    }
    const bool reg = k <= 32;
    const bool direct = reg && ngroups == 1 && outD != nullptr;
    float* dD = direct ? outD : nullptr;
    int64_t* dI = direct ? outI : nullptr;
    if (reg && pq4) launch_il2<true, true>(idx, xq, qc, keys, nprobe, G, ngroups, k, cap, part, dD, dI, st);
    else if (reg) launch_il2<true, false>(idx, xq, qc, keys, nprobe, G, ngroups, k, cap, part, dD, dI, st);
    else if (pq4) launch_il2<false, true>(idx, xq, qc, keys, nprobe, G, ngroups, k, cap, part, nullptr, nullptr, st);
    else launch_il2<false, false>(idx, xq, qc, keys, nprobe, G, ngroups, k, cap, part, nullptr, nullptr, st);
    return direct;
}
