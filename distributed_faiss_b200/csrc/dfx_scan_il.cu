// dfx_scan_il.cu -- layout conversion drivers of the block-interleaved IVF-PQ storage (M == 32 x 8 bit
// and M == 64 x 4 bit).
// Kernels: dfx_scan_il_dev.cuh; the scan itself: dfx_scan_il2.cu.
#include "dfx_scan_il_dev.cuh"

bool dfx_il_wanted(const dfx_index* idx) {
    return idx->cfg.kind == DFX_IVF_PQ && idx->il_enabled &&
           ((idx->M == 32 && idx->nbits == 8) || (idx->M == 64 && idx->nbits == 4));
}

// payload/tvals/ids (row-major, list-sorted) -> il_* ; frees the row-major arrays
void dfx_pq_rm_to_il(dfx_index* idx, cudaStream_t st) {
    if (!dfx_il_wanted(idx)) return;
    if (idx->il) return;
    const int64_t nlist = idx->cfg.nlist;
    std::vector<int64_t> h_blk((size_t)nlist + 1);
    h_blk[0] = 0;
    for (int64_t l = 0; l < nlist; l++)
        h_blk[(size_t)l + 1] = h_blk[(size_t)l] + dfx_ceil_div(idx->h_list_off[(size_t)l + 1] - idx->h_list_off[(size_t)l], 32);
    const int64_t nblk = h_blk[(size_t)nlist];
    idx->blk_off.reserve((size_t)(nlist + 1) * 8);
    DFX_CUDA(cudaMemcpyAsync(idx->blk_off.p, h_blk.data(), (size_t)(nlist + 1) * 8, cudaMemcpyHostToDevice, st));
    idx->il_codes.reserve((size_t)std::max<int64_t>(nblk, 1) * 1024);
    idx->il_tvals.reserve((size_t)std::max<int64_t>(nblk, 1) * 32 * 4);
    idx->il_ids.reserve((size_t)std::max<int64_t>(nblk, 1) * 32 * 4);
    if (nblk > 0)
        DFX_LAUNCH(pq_rm_to_il_kernel, (unsigned)nblk, 256, 0, st, idx->list_off.as<int64_t>(),
                   idx->blk_off.as<int64_t>(), nlist, idx->nbits, idx->payload.as<uint8_t>(), idx->tvals.as<float>(),
                   idx->ids.as<int32_t>(), idx->il_codes.as<uint8_t>(), idx->il_tvals.as<float>(),
                   idx->il_ids.as<int32_t>());
    DFX_CUDA(cudaStreamSynchronize(st));  // h_blk is on the stack of this call
    idx->payload.release();
    idx->tvals.release();
    idx->ids.release();
    idx->nblk = nblk;
    idx->il = true;
    idx->inv_valid = false;
}

// il_* -> payload/tvals/ids (row-major); frees the interleaved arrays
void dfx_pq_il_to_rm(dfx_index* idx, cudaStream_t st) {
    if (!idx->il) return;
    const int64_t n = idx->n_sorted;
    idx->payload.reserve((size_t)std::max<int64_t>(n, 1) * idx->row_bytes());
    idx->tvals.reserve((size_t)std::max<int64_t>(n, 1) * 4);
    idx->ids.reserve((size_t)std::max<int64_t>(n, 1) * 4);
    if (idx->nblk > 0)
        DFX_LAUNCH(pq_il_to_rm_kernel, (unsigned)idx->nblk, 256, 0, st, idx->list_off.as<int64_t>(),
                   idx->blk_off.as<int64_t>(), idx->cfg.nlist, idx->nbits, idx->il_codes.as<uint8_t>(),
                   idx->il_tvals.as<float>(), idx->il_ids.as<int32_t>(), idx->payload.as<uint8_t>(),
                   idx->tvals.as<float>(), idx->ids.as<int32_t>());
    DFX_CUDA(cudaStreamSynchronize(st));
    idx->il_codes.release();
    idx->il_tvals.release();
    idx->il_ids.release();
    idx->nblk = 0;
    idx->il = false;
    idx->inv_valid = false;
}

