// dfx_pq_prep_dev.cuh -- K3 device code (included by dfx_search.cu; also compiled by the CPU
// emulator, tests/emu/).
#pragma once
#include "dfx_common.cuh"
#include "dfx_ptx.cuh"

// =====================================================================================
// K3 (row-major scan: any other (M, nbits), or interleaving switched off): lut[q][m][j] =
// -2 * ip_seq(q_m, P[m][j]), j < ksub (256 or 16); dis0[q][p] = warp-dot ||q - c||^2.  (The block
// scan of M == 32 x 8 / M == 64 x 4 bit builds its table in its own prologue, dfx_scan_il2_dev.cuh.)
// =====================================================================================
__global__ void __launch_bounds__(256)
pq_prep_kernel(const float* __restrict__ Q, int d, int M, int ksub, int dsub,
               const float* __restrict__ codebooks, const float* __restrict__ cent,
               const int32_t* __restrict__ keys, int nprobe, float* __restrict__ lut,
               float* __restrict__ dis0) {
    DFX_DYN_SMEM0(float, s_q);
    const int64_t q = blockIdx.x;
    for (int i = threadIdx.x; i < d; i += blockDim.x) s_q[i] = Q[q * d + i];
    __syncthreads();
    if (lut) {
        const int tot = M * ksub;
#pragma unroll 4
        for (int idx = threadIdx.x; idx < tot; idx += blockDim.x) {
            const int m = (ksub == 256) ? (idx >> 8) : (idx / ksub);
            const float* p = codebooks + (size_t)idx * dsub;
            const float* qm = s_q + m * dsub;
            float acc = 0.f;
            if (dsub == 4) {  // same seq-k order, one 16-byte load
                const float4 pv = __ldg(reinterpret_cast<const float4*>(p));
                acc = __fmaf_rn(qm[0], pv.x, acc);
                acc = __fmaf_rn(qm[1], pv.y, acc);
                acc = __fmaf_rn(qm[2], pv.z, acc);
                acc = __fmaf_rn(qm[3], pv.w, acc);
            } else {
                for (int t = 0; t < dsub; t++) acc = __fmaf_rn(qm[t], p[t], acc);
            }
            lut[q * tot + idx] = -2.f * acc;
        }
    }
    if (dis0) {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
        for (int p = warp; p < nprobe; p += nw) {
            int l = keys[q * nprobe + p];
            float acc = 0.f;
            if (l >= 0) {
                const float* c = cent + (size_t)l * d;
                for (int base = 4 * lane; base < d; base += 128) {
                    float4 cv = *reinterpret_cast<const float4*>(c + base);
                    float4 qv = *reinterpret_cast<const float4*>(s_q + base);
                    float df;
                    df = qv.x - cv.x; acc = __fmaf_rn(df, df, acc);
                    df = qv.y - cv.y; acc = __fmaf_rn(df, df, acc);
                    df = qv.z - cv.z; acc = __fmaf_rn(df, df, acc);
                    df = qv.w - cv.w; acc = __fmaf_rn(df, df, acc);
                }
            }
            acc = dfx_warp_butterfly(acc);
            if (lane == 0) dis0[q * nprobe + p] = acc;
        }
    }
}
