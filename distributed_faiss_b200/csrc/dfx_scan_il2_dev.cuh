// dfx_scan_il2_dev.cuh -- device code of dfx_scan_il2.cu (also compiled by the CPU emulator, tests/emu/).
// K3 + K4: per-query PQ table build fused into the inverted-list scan of PQ codes (M == 32), one
// lane per vector, wide table.  The default IVF-PQ scan since round 2 (validated on B200:
// profiles/r02_*; the 8-lanes-per-vector kernel of round 1 and the other candidates are gone).
//
// Replaces the inner loop of faiss IndexIVFPQ::search (reached from reference
// distributed_faiss/index.py:257) -- `dis = dis0 + sum_m table[m][code[m]]` over every code of
// every probed list; same canonical arithmetic as the other scan kernels (oracle pq_sum).
//
// Design (each point answers a line of the ncu profile of the round-1 kernel):
//   * Block layout 2 (dfx_il2_byte): lane v owns vector v; the two 16-byte halves of all lanes are
//     contiguous, so each 128-bit load of the warp is one 512-byte run (4 wavefronts).
//   * One lane per vector needs no shuffles: lane v walks m = (t + v) & 31, t = 0..31.  The table
//     rows are 64 floats wide (column c holds m = c & 31), so the lane reads column v + t with no
//     wrap-around and the 32 lanes hit 32 different banks at every step.  The halving tree of
//     oracle pq_sum joins, at each level, the residue classes of m modulo a power of two; a
//     rotation of m maps classes to classes, so the tree over t joins the same sets (operands of
//     a node possibly swapped: fp32 addition is commutative) -> bit-identical sums.
//   * The shared-memory address of a lookup is ONE instruction: PRMT drops the code byte into
//     byte 1 of (4 * lane), giving code * 256 + 4 * lane; the table base (uniform register) and
//     4 * t (immediate) ride in the LDS address.  The tree is 15 packed FADD2 + 1 FADD.
//   * k <= 32: the k best of a warp live in REGISTERS (lane i = i-th best, 64-bit composite);
//     admitted candidates go to a 64-slot queue; whenever 32 are queued they are merged with a
//     bitonic network over shuffles, the remainder stays queued.
//     Ids are not streamed: the queue holds positions, ids are gathered when the queue is
//     merged (one latency per merge) or on an exact tie with the k-th best.
//   * A warp scans a CONTIGUOUS eighth of the CTA's blocks (the probed lists laid end to end),
//     two blocks in flight in registers and an L2 prefetch pf_ahead blocks further in the same
//     segment; the stream crosses list boundaries, the head of the next segment is prefetched when
//     a segment is entered.
//   * K3 fused (round 2): the CTA builds its query's table in the prologue -- lut[m][j] =
//     -2 * ip_seq(q_m, P[m][j]) from the transposed codebook PT[j][m][dsub] (L2-resident, 128 KB),
//     warp w produces rows j = w, w+8, ... with lane = m, so codebook reads are 512-byte runs and
//     the shared-memory stores are conflict-free -- and the exact |q - c|^2 of its probed lists
//     (warp-dot).  The 64 KB per (query, shard) table no longer makes a round trip through global
//     memory (268 MB written + 268 MB read per 4096-query launch) and the K3 launch is gone.
//   * A CTA that owns ALL probes of its query (ngroups == 1, the large-batch regime) writes the
//     final (D, I) rows itself; the per-query reduction launch is skipped.
//   * M = 64 x 4 bit (PQ4) runs the same main loop: block byte p of a vector is the pair
//     c_p | c_{p+32} << 4 and the prologue builds the pair table T[b][p] = lut[p][b & 15] +
//     lut[p+32][b >> 4] in place of the 8-bit table.  That sum is the first level (s[p] + s[p+32])
//     of the oracle's M = 64 tree; its other five levels are the M = 32 tree the loop already
//     reproduces, so the sums are bit-identical with 32 lookups per vector (DESIGN.md 4.2).
#pragma once
#include "dfx_internal.h"
#include "dfx_topk.cuh"
#include "dfx_ptx.cuh"

constexpr int IL2_THREADS = 256;             // default: 8 warps; 3 CTAs per SM (64 KB table each)
constexpr int IL2_LUT_BYTES = 256 * 64 * 4;  // wide table of one query
constexpr int IL2_QCAP = 64;                 // queue slots per warp (register top-k path)
constexpr int IL2_MAXG = 16;                 // probes per CTA (choose_group caps G at 16)

// codebook in the order the fused table build of the block scan reads it: PT[j][m][dsub]
__global__ void cb_transpose_kernel(const float* __restrict__ cb, int M, int ksub, int dsub,
                                    float* __restrict__ cbT) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // over M * ksub * dsub
    if (i >= M * ksub * dsub) return;
    const int t = i % dsub, e = i / dsub, j = e % ksub, m = e / ksub;
    cbT[((size_t)j * M + m) * dsub + t] = cb[i];
}

// Merge the first min(cnt, 32) entries of a warp's queue (key << 32 | position) into its
// register-resident set and move the rest to the front of the queue; the ids of the merged
// positions are gathered here.  Returns the new set, the new count and, once k candidates are held,
// the k-th best (value, id), which is also folded into the CTA-wide bound.  Everything travels by
// value so that the caller's state stays in registers.
struct Il2Flushed {
    uint64_t kept;
    float thr;
    uint32_t thr_sec;
    int cnt;
};
__device__ __noinline__ Il2Flushed il2_flush(uint64_t kept, uint64_t* queue, int cnt, int k,
                                             const int32_t* __restrict__ il_ids, unsigned int* cta_key, float thr,
                                             uint32_t thr_sec, int lane) {
    const int n = cnt < 32 ? cnt : 32;
    uint64_t x = DFX_COMP_NONE;
    if (lane < n) {
        const uint64_t c = queue[lane];
        x = (c & 0xffffffff00000000ull) | (uint64_t)dfx_ld_nc_u(il_ids + (uint32_t)c);
    }
    const int rest = cnt - n;  // < 32: the pusher flushes as soon as 32 entries are queued
    const uint64_t moved = (lane < rest) ? queue[32 + lane] : 0;
    __syncwarp();  // queue fully read before it is rewritten
    if (lane < rest) queue[lane] = moved;
    __syncwarp();
    kept = dfx_warp_merge_sorted32(kept, dfx_warp_sort32_asc(x, lane), lane);
    const uint64_t kth = __shfl_sync(0xffffffffu, kept, k - 1);
    if (kth != DFX_COMP_NONE) {
        thr = dfx_key2f((uint32_t)(kth >> 32));
        thr_sec = (uint32_t)kth;
        if (lane == 0) atomicMin(cta_key, (unsigned int)(kth >> 32));
    }
    Il2Flushed r;
    r.kept = kept;
    r.thr = thr;
    r.thr_sec = thr_sec;
    r.cnt = rest;
    return r;
}

// Prologue of the M = 64 x 4-bit block scan (out of line: it keeps the main loop's register
// allocation that of the 8-bit kernel).  (a) lut[m][j] = -2 * ip_seq(q_m, P[m][j]), m < 64,
// j < 16, into s_l16 (the queue area, free until the scan starts; >= 4 KB for every k), stored
// [j][m] so that (b) reads it conflict-free.  (b) the pair table T[b][p] = lut[p][b & 15] +
// lut[p + 32][b >> 4] -- the first level of the oracle's M = 64 halving tree (s[p] + s[p + 32]);
// b = pair byte of column p (dfx_il2_pair).  Row b is 64 floats wide with columns p and p + 32
// equal, as in the 8-bit table.
template <int THREADS>
__device__ __noinline__ void il2_pair_table(float* s_lut, float* s_l16, const float* __restrict__ qrow,
                                            const float* __restrict__ cbT, int dsub, int tid) {
#pragma unroll 1
    for (int e = tid; e < 16 * 64; e += THREADS) {  // e = j * 64 + m: cbT row e is P[m][j]
        const int m = e & 63;
        const float* pv = cbT + (size_t)e * dsub;
        const float* qm = qrow + m * dsub;
        float acc = 0.f;
        for (int t = 0; t < dsub; t++) acc = __fmaf_rn(__ldg(qm + t), __ldg(pv + t), acc);
        s_l16[e] = -2.f * acc;
    }
    __syncthreads();
#pragma unroll 1
    for (int e = tid; e < 256 * 32; e += THREADS) {
        const int b = e >> 5, p = e & 31;
        const float val = s_l16[(b & 15) * 64 + p] + s_l16[(b >> 4) * 64 + 32 + p];
        s_lut[b * 64 + p] = val;
        s_lut[b * 64 + 32 + p] = val;
    }
}

// REG: k <= 32, register-resident top-k;  !REG: WarpTopK buffers in shared memory (any k)
// PQ4: M = 64 x 4 bit (pair table, blocks of pair bytes); else M = 32 x 8 bit.
// Q [nq][d] queries; cbT: transposed codebook PT[j][m][dsub]; cent [nlist][d]; d = M * dsub.
// outD / outI != nullptr (requires ngroups == 1): final faiss-style rows are written directly.
template <bool REG, int THREADS, int MINB, bool PQ4>
__global__ void __launch_bounds__(THREADS, MINB)
scan_pq_il2_kernel(const float* __restrict__ Q, const float* __restrict__ cbT, const float* __restrict__ cent, int d,
                   int dsub, const int32_t* __restrict__ keys, int nprobe, int G, int ngroups,
                   const int64_t* __restrict__ blk_off, const uint4* __restrict__ il_codes,
                   const float* __restrict__ il_tvals, const int32_t* __restrict__ il_ids, int k, int cap,
                   uint64_t* __restrict__ part, float* __restrict__ outD, int64_t* __restrict__ outI, int pf_ahead) {
    DFX_DYN_SMEM(unsigned char, smem_raw, 128);
    float* s_lut = reinterpret_cast<float*>(smem_raw);                      // [256][64]
    uint64_t* s_buf = reinterpret_cast<uint64_t*>(smem_raw + IL2_LUT_BYTES);  // queues / WarpTopK buffers
    __shared__ unsigned int s_cta_key;  // CTA-wide admission bound (order-preserving key)
    __shared__ int s_lb[IL2_MAXG], s_le[IL2_MAXG];  // first / end block of each probed list
    __shared__ float s_ld0[IL2_MAXG];               // |q - c|^2 of each probed list
    __shared__ int s_lkey[IL2_MAXG];
    __shared__ int s_cum[IL2_MAXG + 1];             // blocks of the probed lists before list p

    constexpr int IL2_NW = THREADS / 32;
    const int64_t q = blockIdx.x / ngroups;
    const int g = blockIdx.x % ngroups;
    const int tid = threadIdx.x, lane = tid & 31;
    // through a shuffle so that the compiler knows `warp` (and with it the block cursor and the
    // loop branches) is warp-uniform: the table base then stays in a uniform register and the
    // lookups become LDS [R + UR + imm]
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int np = min(nprobe, (g + 1) * G) - g * G;  // probes of this CTA (<= IL2_MAXG)
    const float* qrow = Q + q * d;

    if (tid == 0) s_cta_key = 0xff800000u;  // key of +inf: no bound yet
    if (tid < np) {
        const int l = keys[q * nprobe + g * G + tid];
        s_lkey[tid] = l;
        s_lb[tid] = (l < 0) ? 0 : (int)blk_off[l];
        s_le[tid] = (l < 0) ? 0 : (int)blk_off[l + 1];
    }
    // ---- K3, part 1: the query's table, rows j = warp, warp + 8, ...; lane = subquantizer m.
    // seq-k order (oracle): acc = fma(q0, p0, 0), fma(q1, p1, acc), ...; entry = -2 * acc.
    if (PQ4) {
        il2_pair_table<THREADS>(s_lut, reinterpret_cast<float*>(s_buf), qrow, cbT, dsub, tid);
    } else if (dsub == 4) {
        const float4 qm = __ldg(reinterpret_cast<const float4*>(qrow) + lane);
        const float4* pt4 = reinterpret_cast<const float4*>(cbT);
#pragma unroll 8
        for (int j = warp; j < 256; j += IL2_NW) {
            const float4 pv = __ldg(pt4 + j * 32 + lane);
            float acc = __fmaf_rn(qm.x, pv.x, 0.f);
            acc = __fmaf_rn(qm.y, pv.y, acc);
            acc = __fmaf_rn(qm.z, pv.z, acc);
            acc = __fmaf_rn(qm.w, pv.w, acc);
            const float val = -2.f * acc;
            s_lut[j * 64 + lane] = val;
            s_lut[j * 64 + 32 + lane] = val;
        }
    } else {
        const float* qm = qrow + lane * dsub;
        for (int j = warp; j < 256; j += IL2_NW) {
            const float* pv = cbT + ((size_t)j * 32 + lane) * dsub;
            float acc = 0.f;
            for (int t = 0; t < dsub; t++) acc = __fmaf_rn(__ldg(qm + t), __ldg(pv + t), acc);
            const float val = -2.f * acc;
            s_lut[j * 64 + lane] = val;
            s_lut[j * 64 + 32 + lane] = val;
        }
    }
    __syncthreads();  // s_lkey visible (and the table complete)
    if (tid == THREADS - 1) {  // the CTA's block stream: the probed lists end to end
        int c = 0;
        for (int p = 0; p < np; p++) {
            s_cum[p] = c;
            c += s_le[p] - s_lb[p];
        }
        s_cum[np] = c;
    }
    // ---- K3, part 2: exact |q - c|^2 of the probed lists, canonical warp-dot order
    for (int p = warp; p < np; p += IL2_NW) {
        const int l = s_lkey[p];
        float acc = 0.f;
        if (l >= 0) {
            const float* c = cent + (size_t)l * d;
            for (int base = 4 * lane; base < d; base += 128) {
                const float4 cv = __ldg(reinterpret_cast<const float4*>(c + base));
                const float4 qv = __ldg(reinterpret_cast<const float4*>(qrow + base));
                float df;
                df = qv.x - cv.x; acc = __fmaf_rn(df, df, acc);
                df = qv.y - cv.y; acc = __fmaf_rn(df, df, acc);
                df = qv.z - cv.z; acc = __fmaf_rn(df, df, acc);
                df = qv.w - cv.w; acc = __fmaf_rn(df, df, acc);
            }
        }
        acc = dfx_warp_butterfly(acc);
        if (lane == 0) s_ld0[p] = acc;
    }
    __syncthreads();

    // ---- candidate set
    WarpTopK wt;                                     // !REG
    uint64_t kept = DFX_COMP_NONE;                   // REG: lane i = i-th best of this warp
    uint64_t* queue = s_buf + (size_t)warp * IL2_QCAP;  // REG: (key << 32 | position)
    int cnt = 0;
    float thr = __int_as_float(0x7f800000);  // value of this warp's k-th best
    uint32_t thr_sec = DFX_SEC_NONE;         // and its id
    float bnd = __int_as_float(0x7f800000);  // register copy of the CTA bound (may lag: only looser)
    if (!REG) wt.init(s_buf + (size_t)warp * cap, cap, k, &s_cta_key);

    // merge 32 queued candidates into `kept` (out of line: rare, and called from three places)
    auto flush = [&]() {
        const Il2Flushed f = il2_flush(kept, queue, cnt, k, il_ids, &s_cta_key, thr, thr_sec, lane);
        kept = f.kept;
        thr = f.thr;
        thr_sec = f.thr_sec;
        cnt = f.cnt;
    };

    const uint32_t lut_base = dfx_smem_addr(s_lut);
    const uint32_t cu = (uint32_t)lane * 4u;  // byte offset of column `lane`; byte 1 receives the code

    // one 32-vector block: lane = vector.  32 lookups (column lane + t of row code_t), the
    // halving tree, then the admission test.
    auto process = [&](const uint4& ca, const uint4& cb, float tv, float d0, int pos) {
        const uint32_t w[8] = {ca.x, ca.y, ca.z, ca.w, cb.x, cb.y, cb.z, cb.w};
        float y[32];
#pragma unroll
        for (int t = 0; t < 32; t++) {
            // byte t&3 of word t>>2 -> byte 1 of (4 * lane): code * 256 + 4 * lane (one PRMT);
            // table base + 4 * t fold into the LDS address (uniform register + immediate)
            const uint32_t r = __byte_perm(w[t >> 2], cu, 0x6504u | ((uint32_t)(t & 3) << 4));
            y[t] = dfx_lds_f32(r + lut_base + 4u * (uint32_t)t);
        }
        // tree levels 16, 8, 4, 2 on pairs (y[2i], y[2i+1]); level 1 joins the two halves
        dfx_f32x2 p2[16];
#pragma unroll
        for (int i = 0; i < 16; i++) p2[i] = dfx_pack2(y[2 * i], y[2 * i + 1]);
#pragma unroll
        for (int off = 8; off >= 1; off >>= 1) {
#pragma unroll
            for (int i = 0; i < off; i++) p2[i] = dfx_add2(p2[i], p2[i + off]);
        }
        float s0, s1;
        dfx_unpack2(p2[0], s0, s1);
        const float v = d0 + (tv + (s0 + s1));  // padding has tv = +inf

        if (REG) {
            bool pass = v <= bnd;
            if (__any_sync(0xffffffffu, pass)) {
                bnd = dfx_key2f(*reinterpret_cast<volatile unsigned int*>(&s_cta_key));
                pass = v <= bnd;  // equal to the bound: still admitted (rank decided by the id)
                bool want = false;
                if (pass) {
                    if (v < thr) want = true;
                    else if (v == thr) want = dfx_ld_nc_u(il_ids + (int64_t)pos * 32 + lane) < thr_sec;
                }
                const unsigned mask = __ballot_sync(0xffffffffu, want);
                if (mask) {
                    if (want)
                        queue[cnt + __popc(mask & ((1u << lane) - 1u))] =
                            ((uint64_t)dfx_f2key(v) << 32) | (uint64_t)((uint32_t)pos * 32u + (uint32_t)lane);
                    cnt += __popc(mask);
                    __syncwarp();
                    if (cnt >= 32) flush();  // keeps cnt <= 31 between pushes (a push adds <= 32)
                }
            }
        } else {
            uint32_t sec = 0;
            const bool want = (v + 0.0f <= wt.cta_bound()) &&
                              wt.admits(v, [&] { return dfx_ld_nc_u(il_ids + (int64_t)pos * 32 + lane); }, sec);
            wt.push_lanes(want, v, sec);
        }
    };

    // ---- the warp's block stream: a CONTIGUOUS eighth of the CTA's blocks (the probed lists laid
    // end to end, s_cum), so that the cursor is one increment and one compare per block, the L2
    // prefetch is "the same segment, pf_ahead blocks further" and the warps finish together.
    // (The profile of the strided walk -- blocks lb + warp, + 8, ... of every list, with a second
    // cursor for the prefetch -- showed ~68 bookkeeping instructions per block next to the 82 of
    // the lookups and the tree.)  A warp's range spans one or two lists; entering a segment is the
    // rare path and prefetches the head of the segment after it.
    const int nblk_cta = s_cum[np];
    const int r0 = (int)(((int64_t)nblk_cta * warp) / IL2_NW);
    int rem = (int)(((int64_t)nblk_cta * (warp + 1)) / IL2_NW) - r0;  // blocks not yet assigned to a segment
    int cur_p = 0, cur_b = 0, cur_e = 0;
    float cur_d0 = 0.f;
    const bool pf_lane = pf_ahead > 0 && lane < 9;  // lanes 0..7: the 8 code lines of a block, lane 8: its t-values
    const unsigned char* pf_base = (lane < 8) ? reinterpret_cast<const unsigned char*>(il_codes) + lane * 128
                                              : reinterpret_cast<const unsigned char*>(il_tvals);
    const int pf_stride = (lane < 8) ? 1024 : 128;
    auto prefetch_head = [&](int b, int n) {  // first min(n, pf_ahead) blocks of a segment
        n = n < pf_ahead ? n : pf_ahead;
        if (pf_lane)
            for (int i = 0; i < n; i++) dfx_prefetch_l2(pf_base + (int64_t)(b + i) * pf_stride);
    };
    auto peek_next_segment = [&]() {  // prefetch the head of the segment that follows the current one
        if (rem <= 0 || pf_ahead == 0) return;
        int p2 = cur_p + 1;
        while (s_le[p2] == s_lb[p2]) p2++;  // rem > 0: a non-empty list lies ahead
        const int len = s_le[p2] - s_lb[p2];
        prefetch_head(s_lb[p2], len < rem ? len : rem);
    };
    if (rem > 0) {
        while (s_cum[cur_p + 1] <= r0) cur_p++;  // the list holding block r0 of the CTA's stream
        cur_b = s_lb[cur_p] + (r0 - s_cum[cur_p]);
        const int len = min(s_le[cur_p] - cur_b, rem);
        cur_e = cur_b + len;
        rem -= len;
        cur_d0 = s_ld0[cur_p];
        prefetch_head(cur_b, len);
        peek_next_segment();
    }
    // next block of the range, or -1
    auto next_block = [&]() -> int {
        if (cur_b == cur_e) {  // segment exhausted (once or twice per warp)
            if (rem <= 0) return -1;
            do cur_p++; while (s_le[cur_p] == s_lb[cur_p]);
            cur_b = s_lb[cur_p];
            const int len = min(s_le[cur_p] - cur_b, rem);
            cur_e = cur_b + len;
            rem -= len;
            cur_d0 = s_ld0[cur_p];
            peek_next_segment();
        }
        return cur_b++;
    };
    const uint4* pc_lane = il_codes + lane;
    const float* pt_lane = il_tvals + lane;
#define IL2_FETCH(A, B, T, D0, POS)                                          \
    do {                                                                     \
        POS = next_block();                                                  \
        if (POS >= 0) {                                                      \
            const uint4* pc_ = pc_lane + (int64_t)POS * 64;                  \
            A = dfx_ld_stream(pc_);                                          \
            B = dfx_ld_stream(pc_ + 32);                                     \
            T = dfx_ld_stream_f(pt_lane + (int64_t)POS * 32);                \
            D0 = cur_d0;                                                     \
            if (pf_lane && POS + pf_ahead < cur_e)                           \
                dfx_prefetch_l2(pf_base + (int64_t)(POS + pf_ahead) * pf_stride); \
        }                                                                    \
    } while (0)

    {
    uint4 a0 = {}, b0 = {}, a1 = {}, b1 = {}, a2 = {}, b2 = {};
    float t0 = 0.f, t1 = 0.f, t2 = 0.f, e0 = 0.f, e1 = 0.f, e2 = 0.f;
    int p0, p1, p2;
    IL2_FETCH(a0, b0, t0, e0, p0);
    IL2_FETCH(a1, b1, t1, e1, p1);
    for (;;) {  // two blocks in flight while one is processed
        IL2_FETCH(a2, b2, t2, e2, p2);
        if (p0 < 0) break;
        process(a0, b0, t0, e0, p0);
        IL2_FETCH(a0, b0, t0, e0, p0);
        if (p1 < 0) break;
        process(a1, b1, t1, e1, p1);
        IL2_FETCH(a1, b1, t1, e1, p1);
        if (p2 < 0) break;
        process(a2, b2, t2, e2, p2);
    }
    }
#undef IL2_FETCH

    uint64_t* out = part + ((int64_t)q * ngroups + g) * k;
    if (REG) {
        if (cnt > 0) flush();
        __syncthreads();  // every warp is done with its queue: the area is reused for the merge
        s_buf[warp * 32 + lane] = kept;
        __syncthreads();
        if (warp == 0) {
#pragma unroll 1
            for (int w2 = 1; w2 < IL2_NW; w2++) kept = dfx_warp_merge_sorted32(kept, s_buf[w2 * 32 + lane], lane);
            if (lane < k) {
                if (outD) {  // this CTA saw every probe of the query: final faiss-style row
                    const bool none = kept == DFX_COMP_NONE;
                    outD[q * k + lane] = none ? FLT_MAX : dfx_key2f((uint32_t)(kept >> 32));
                    outI[q * k + lane] = none ? -1 : (int64_t)(uint32_t)kept;
                } else {
                    out[lane] = kept;
                }
            }
        }
    } else {
        cta_merge_and_write<THREADS>(wt, s_buf, cap, k, out);
    }
}
