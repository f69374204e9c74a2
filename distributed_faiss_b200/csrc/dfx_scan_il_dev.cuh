// dfx_scan_il_dev.cuh -- device code of dfx_scan_il.cu (also compiled by the CPU emulator, tests/emu/).
// Conversion between the row-major exchange form of an IVF-PQ shard (M == 32 x 8 bit or
// M == 64 x 4 bit: 32 bytes per vector either way) and the 1 KB
// blocks of 32 vectors the scan reads (block layout: dfx_il2_byte, dfx_internal.h; scan kernel:
// dfx_scan_il2_dev.cuh).  Lists are padded to whole blocks; padding carries t = +inf so it can
// never enter a result.
#pragma once
#include "dfx_internal.h"
#include "dfx_topk.cuh"
#include "dfx_ptx.cuh"

// ------------------------------------------------------------------ layout conversion
__device__ __forceinline__ int64_t il_list_of_block(const int64_t* __restrict__ blk_off, int64_t nlist, int64_t blk) {
    int64_t lo = 0, hi = nlist;
    while (hi - lo > 1) {
        int64_t mid = (lo + hi) >> 1;
        if (blk_off[mid] <= blk) lo = mid; else hi = mid;
    }
    return lo;
}

// row-major (list-sorted) -> interleaved blocks.  one CTA per block.  nbits = 8: M = 32, block byte
// of column p is code p; nbits = 4: M = 64, it is the pair (c_p, c_{p+32}) (dfx_il2_pair).
__global__ void __launch_bounds__(256)
pq_rm_to_il_kernel(const int64_t* __restrict__ list_off, const int64_t* __restrict__ blk_off, int64_t nlist,
                   int nbits, const uint8_t* __restrict__ codes, const float* __restrict__ tvals,
                   const int32_t* __restrict__ ids, uint8_t* __restrict__ il_codes, float* __restrict__ il_tvals,
                   int32_t* __restrict__ il_ids) {
    const int64_t blk = blockIdx.x;
    const int64_t l = il_list_of_block(blk_off, nlist, blk);
    const int64_t base = list_off[l] + (blk - blk_off[l]) * 32, end = list_off[l + 1];
    for (int e = threadIdx.x; e < 1024; e += 256) {
        const int v = e >> 5, p = e & 31;
        const int64_t i = base + v;
        uint8_t b = 0;
        if (i < end) {
            const uint8_t* row = codes + i * 32;  // 32 bytes per row in both configurations
            b = (nbits == 8) ? (uint8_t)dfx_pq_code(row, p, 8)
                             : dfx_il2_pair(dfx_pq_code(row, p, 4), dfx_pq_code(row, p + 32, 4));
        }
        il_codes[blk * 1024 + dfx_il2_byte(v, p)] = b;
    }
    if (threadIdx.x < 32) {
        const int64_t i = base + threadIdx.x;
        il_tvals[blk * 32 + threadIdx.x] = (i < end) ? tvals[i] : __int_as_float(0x7f800000);
        il_ids[blk * 32 + threadIdx.x] = (i < end) ? ids[i] : -1;
    }
}

__global__ void __launch_bounds__(256)
pq_il_to_rm_kernel(const int64_t* __restrict__ list_off, const int64_t* __restrict__ blk_off, int64_t nlist,
                   int nbits, const uint8_t* __restrict__ il_codes, const float* __restrict__ il_tvals,
                   const int32_t* __restrict__ il_ids, uint8_t* __restrict__ codes, float* __restrict__ tvals,
                   int32_t* __restrict__ ids) {
    const int64_t blk = blockIdx.x;
    const int64_t l = il_list_of_block(blk_off, nlist, blk);
    const int64_t base = list_off[l] + (blk - blk_off[l]) * 32, end = list_off[l + 1];
    const uint8_t* bk = il_codes + blk * 1024;
    for (int e = threadIdx.x; e < 1024; e += 256) {
        const int v = e >> 5, j = e & 31;  // byte j of row v
        const int64_t i = base + v;
        if (i >= end) continue;
        if (nbits == 8) {
            codes[i * 32 + j] = bk[dfx_il2_byte(v, j)];
        } else {  // sub-quantizers 2j and 2j + 1, each from the pair byte of its column
            const int m0 = 2 * j, m1 = 2 * j + 1;
            codes[i * 32 + j] = dfx_pq4_byte(dfx_il2_pair_code(bk[dfx_il2_byte(v, m0 & 31)], m0),
                                             dfx_il2_pair_code(bk[dfx_il2_byte(v, m1 & 31)], m1));
        }
    }
    if (threadIdx.x < 32) {
        const int64_t i = base + threadIdx.x;
        if (i < end) {
            tvals[i] = il_tvals[blk * 32 + threadIdx.x];
            ids[i] = il_ids[blk * 32 + threadIdx.x];
        }
    }
}

