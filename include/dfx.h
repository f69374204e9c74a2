/*
 * dfx.h -- C-ABI of the B200-native shard engine (libdfx.so).
 *
 * This is the drop-in boundary for the SEARCH PATH of
 * facebookresearch/distributed-faiss.  The reference is pure Python and
 * reaches its numeric kernels through the SWIG-wrapped `faiss` object that
 * `distributed_faiss/index.py` keeps in `Index.faiss_index`; each entry point
 * below names the reference call site (file:line under /root/reference) whose
 * faiss call it replaces.  Plain pointers and sizes only -- no torch types.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; the message is
 *     available from dfx_last_error() (thread-local).  The Python binding
 *     turns it into RuntimeError, which IndexServer forwards to the client as
 *     rpc.ServerException exactly like a faiss exception (server.py:229-236).
 *   - "_dev" variants take DEVICE pointers and a cudaStream_t (passed as
 *     void*), enqueue work and return without synchronising; the others take
 *     HOST pointers, copy in/out and synchronise (the reference-facing path).
 *   - float32 row-major C-contiguous inputs, like faiss (index.py:151 casts,
 *     index.py:257 does not).
 *   - results follow faiss: L2 ascending / IP descending, missing entries
 *     id -1 and distance +FLT_MAX (L2) or -FLT_MAX (IP).  Ties are broken by
 *     the total order (value asc, id asc) -- see DESIGN.md.
 *   - there is no CPU fallback: every entry point that computes requires a
 *     CUDA device of compute capability 10.x and fails otherwise.
 */
#ifndef DFX_H
#define DFX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dfx_index dfx_index;

/* which faiss object the reference builder would have made (index.py:93-100) */
enum {
    DFX_FLAT = 0,     /* faiss.IndexFlatIP / IndexFlatL2         index.py:94, 25-33 */
    DFX_IVF_FLAT = 1, /* faiss.IndexIVFFlat                       index.py:36-40     */
    DFX_IVF_PQ = 2,   /* faiss.IndexIVFPQ (L2, by_residual)       index.py:43-48     */
    DFX_IVF_SQ16 = 3  /* faiss.IndexIVFScalarQuantizer(QT_fp16)   index.py:63-68     */
};

/* faiss.METRIC_INNER_PRODUCT / faiss.METRIC_L2 (index_cfg.py:44-52) */
enum { DFX_METRIC_IP = 0, DFX_METRIC_L2 = 1 };

typedef struct dfx_cfg {
    int32_t kind;     /* DFX_FLAT ... */
    int32_t metric;   /* FLAT / IVF_FLAT: search metric.  IVF_PQ / IVF_SQ16: metric of the
                         coarse quantizer only -- the reference never forwards it to the
                         index, which is therefore always L2 (index.py:44-46, 64-66). */
    int32_t d;        /* vector dimension (cfg.dim) */
    int32_t pq_m;     /* IVF_PQ: sub-quantizers  (cfg.extra["code_size"], index.py:44) */
    int32_t pq_nbits; /* IVF_PQ: bits per code, 8 or 4 (cfg.extra["bits_per_vector"], index.py:45);
                         4 needs pq_m % 8 == 0 */
    int32_t device;   /* CUDA device ordinal this shard lives on */
    int64_t nlist;    /* IVF_*: number of inverted lists (cfg.centroids) */
} dfx_cfg;

/* ---- lifetime: replaces the faiss constructors at index.py:25-48,63-68,94 ---- */
int dfx_create(const dfx_cfg *cfg, dfx_index **out);
void dfx_destroy(dfx_index *idx);

/* ---- build: faiss_index.train(x) index.py:217 ; faiss_index.add(x) index.py:425 ---- */
int dfx_train(dfx_index *idx, int64_t n, const float *x);
int dfx_add(dfx_index *idx, int64_t n, const float *x);
int dfx_train_dev(dfx_index *idx, int64_t n, const float *d_x, void *stream);
int dfx_add_dev(dfx_index *idx, int64_t n, const float *d_x, void *stream);
/* knobs (every setting returns the same results; they only move the cost):
 * training: "kmeans_niter" (default 25), "max_points_per_centroid" (256), "train_seed" (1234) --
 *   the faiss Clustering defaults;
 * "tensor_cores" (1): 0 forces the plain fp32 FFMA coarse quantizer instead of the tcgen05
 *   screening path;
 * "tc_screen_mode" (0): precision of the tcgen05 screening: 0 = AUTO (starts PRECISE, moves to
 *   FAST once enough rows have shown that FAST's wider tolerance would not overflow the kept
 *   groups, and back as soon as it does),
 *   1 = FAST (fp16 operands, one MMA per k-step), 2 = PRECISE (fp16 hi/lo split, three MMAs);
 *   "tc_auto_window" (16384): rows AUTO observes before PRECISE may become FAST;
 * "flat_tensor_cores" (1): 0 runs FLAT searches through the FFMA GEMM instead of the tensor-core
 *   screening + exact re-rank;
 * "interleaved" (1): 0 keeps IVF-PQ (M = 32 x 8 bit, M = 64 x 4 bit) codes row-major (one vector
 *   per lane, table from pq_prep_kernel) instead of the block-interleaved layout of the fused
 *   table-build + scan;
 * "il2_threads" (0 = 256) / "il2_prefetch" (-1 = 4 blocks): CTA shape and L2 prefetch distance of
 *   that scan (tuning);
 * "rows_inflight" (0 = by row size): 4 or 8 vectors per warp in flight in the IVF-Flat / IVF-SQ
 *   list scan */
int dfx_set_param(dfx_index *idx, const char *name, double value);
/* read back a knob or a counter: the names of dfx_set_param, plus "tc_fast" (the precision the
 * next screening launch will use: 1 = FAST), "tc_stat_rows" / "tc_stat_overflow" /
 * "tc_stat_fast_would" (rows, rows re-done exactly, and rows FAST would have re-done, of the last
 * launch whose statistics came back; synchronises with that launch) */
int dfx_get_param(dfx_index *idx, const char *name, double *value);
/* pre-size the shard for n_total vectors (optional; avoids regrowth while bulk loading) */
int dfx_reserve(dfx_index *idx, int64_t n_total);
/* fold pending adds into the inverted lists now (otherwise done by the next search) */
int dfx_finalize(dfx_index *idx, void *stream);

/* ---- THE HOT PATH: faiss_index.search(query_batch, top_k) index.py:257 ----
 * D float32[nq,k], I int64[nq,k]. */
int dfx_search(dfx_index *idx, int64_t nq, const float *x, int64_t k, float *D, int64_t *I);
int dfx_search_dev(dfx_index *idx, int64_t nq, const float *d_x, int64_t k, float *d_D,
                   int64_t *d_I, void *stream);

/* faiss_index.search_and_reconstruct: decode rows by id (index.py:255); id -1 -> NaN row */
int dfx_reconstruct(dfx_index *idx, int64_t n, const int64_t *ids, float *out);

/* device form, for winners that travelled through the all-gather + merge (client.py:287-289,
 * 299-307 carry per-shard embeddings to the client; here only the WINNERS are decoded, by the
 * shard that owns them).  shard_tag < 0: d_ids are shard-local ids, as dfx_reconstruct.
 * shard_tag >= 0: d_ids are exchange ids (dfx_encode_ids_dev); rows owned by another shard (or
 * empty, -1) are left untouched, so every rank decodes into a zeroed [n, d] buffer and the
 * buffers are summed. */
int dfx_reconstruct_dev(dfx_index *idx, int64_t n, const int64_t *d_ids, int64_t shard_tag,
                        float *d_out, void *stream);

/* ---- attributes the wrapper touches: .nprobe (index.py:356,495) .ntotal (index.py:184)
 *      .nlist / .quantizer.reconstruct_n(0, nlist) (index.py:350) ---- */
int dfx_set_nprobe(dfx_index *idx, int64_t nprobe);
int64_t dfx_get_nprobe(const dfx_index *idx);
int64_t dfx_ntotal(const dfx_index *idx);
/* changes whenever a call may have changed what a search launches (train / add / finalize /
 * import / set_param / set_nprobe); callers that replay captured CUDA graphs key them on it */
int64_t dfx_generation(const dfx_index *idx);
int64_t dfx_nlist(const dfx_index *idx);
int dfx_is_trained(const dfx_index *idx);
int dfx_get_centroids(dfx_index *idx, float *out /* [nlist, d] host */);

/* ---- cross-shard merge: faiss.float_maxheap_array_t as driven by ResultHeap /
 *      IndexClient._aggregate_results (client.py:29-54, 265-310).
 * D, I: [S][nq][k].  negate != 0 reproduces client.py:291-292 (search for -D when
 * metric == "dot"; the returned scores stay negated).  Keeps the k smallest, ascending;
 * an entry is admitted only if FLT_MAX > value (heapify() semantics); pads (FLT_MAX,-1).
 * outI[q][j] = I of the winner. */
int dfx_merge(int64_t S, int64_t nq, int64_t k, const float *D, const int64_t *I, int negate,
              float *outD, int64_t *outI);
int dfx_merge_dev(int64_t S, int64_t nq, int64_t k, const float *d_D, const int64_t *d_I,
                  int negate, float *d_outD, int64_t *d_outI, void *stream);

/* the same merge over what ONE all-gather of the ranks' result blocks delivers: rank r's block
 * starts at d_packed + r * rank_stride_bytes and holds D f32[S_loc][nq][k] at offset 0 and
 * I i64[S_loc][nq][k] at off_I_bytes (both multiples of 8).  Shard s = r * S_loc + j. */
int dfx_merge_packed_dev(int64_t R, int64_t S_loc, int64_t nq, int64_t k, const void *d_packed,
                         int64_t rank_stride_bytes, int64_t off_I_bytes, int negate,
                         float *d_outD, int64_t *d_outI, void *stream);

/* shard-local ids -> exchange ids: out = ids < 0 ? -1 : (shard_tag << 40) | ids, so that the
 * client can tell which (shard, local id) won after the merge (the reference's synthetic
 * positions, client.py:288).  d_col (optional): one int32 code per local id for ONE metadata
 * position (-2 = no metadata / tuple too short); entries whose code == drop_code or -2 are what
 * search_with_filter's post-filter drops (client.py:235-243) and get bit 62 set. */
int dfx_encode_ids_dev(int64_t n, const int64_t *d_ids, int64_t shard_tag, const int32_t *d_col,
                       int32_t drop_code, int64_t *d_out, void *stream);
/* search_with_filter's post-filter on device (client.py:229-250): per query, walk the k_in merged
 * slots in rank order, keep existing entries without the drop flag, stop at k_out; pads
 * (FLT_MAX, -1); d_count[q] = number kept. */
int dfx_filter_compact_dev(int64_t nq, int64_t k_in, int64_t k_out, const float *d_D,
                           const int64_t *d_I, float *d_outD, int64_t *d_outI, int32_t *d_count,
                           void *stream);

/* map shard-local ids to caller ids on device: out[i] = ids[i] < 0 ? -1 : table[ids[i]]
 * (the device form of Index.search's id -> metadata loop, index.py:260-268, for the
 * integer-metadata convention of scripts/load_data.py:120-124). */
int dfx_map_ids_dev(int64_t n, const int64_t *d_ids, const int64_t *d_table, int64_t *d_out,
                    void *stream);

/* ---- state exchange (tests, persistence; not on the timed path) ----
 * named arrays, host memory, list-sorted storage order:
 *   "centroids" f32[nlist,d]   "codebooks" f32[M,ksub,dsub]   "list_off" i64[nlist+1]
 *   "ids" i64[ntotal]   "codes" u8[ntotal,M*nbits/8]   "tvals" f32[ntotal]
 *   ("codes" in faiss bit order: at nbits = 4 code m is the low nibble of byte m/2 when m is
 *   even, the high nibble when m is odd; ksub = 1 << nbits)
 *   "vecs" f32[ntotal,d] (IVF_FLAT)   "codes16" u16[ntotal,d]   "xb" f32[ntotal,d] (FLAT)
 * dfx_get_array with out == NULL only reports the size.  Import order: centroids,
 * codebooks, then list_off, ids and the payload, then dfx_import_done(). */
int dfx_get_array(dfx_index *idx, const char *name, void *out, int64_t max_bytes,
                  int64_t *nbytes);
int dfx_set_array(dfx_index *idx, const char *name, const void *in, int64_t nbytes);
int dfx_import_done(dfx_index *idx);

/* statistics of the most recent search (device work, synchronises):
 * ndis = sum over (query, probed list) of the list length -- faiss's `ndis`. */
int dfx_last_stats(dfx_index *idx, int64_t *ndis, int64_t *nq, int64_t *nprobe);
/* per-kernel timing of the dominant kernel (the inverted-list scan): when enabled, every scan
 * launch is bracketed by CUDA events on the launching stream; dfx_profile_read synchronises
 * those events and returns the summed device time and the number of launches. */
int dfx_profile_enable(dfx_index *idx, int on);
int dfx_profile_read(dfx_index *idx, double *scan_ms, int64_t *scan_launches, int reset);
/* number of kernel launches issued by this library since process start */
int64_t dfx_launch_count(void);

/* ---- synthetic data on device (bench harness; SURVEY.md 8d generator, see DESIGN.md) ----
 * x_i = mu_{c(i)} + A (sigma * z_{g(i)} + delta * w_i) + eps * n_i
 *   C cluster centres mu_c ~ N(0, I_d);  c(i) = i mod C
 *   G groups ("near-duplicate" micro-clusters), g(i) = i mod G (G multiple of C; G = 0: one
 *   group per row); latent z_g ~ N(0, I_r) clipped to |z| <= 4;  A: d x r, orthonormal columns
 *   w_i ~ N(0, I_r), n_i ~ N(0, I_d) per row.
 * Counter-based: any row is regenerable anywhere from (seed, row).  rows: optional explicit row
 * ids (else row0 .. row0+n-1).  noise_stream != 0 adds sigma_q * N(0, I_d) (queries). */
typedef struct dfx_synth {
    uint64_t seed;
    int32_t d;
    int32_t r;        /* intrinsic dimension of the cluster-level structure */
    int64_t nclusters;
    int64_t ngroups;
    float sigma;
    float eps;
    float sigma_q;
    float delta;
} dfx_synth;
int dfx_synth_init(const dfx_synth *p, float **d_A_out /* device [d,r], caller frees with dfx_free */,
                   void *stream);
int dfx_synth_rows_dev(const dfx_synth *p, const float *d_A, int64_t row0, const int64_t *d_rows,
                       int64_t n, uint64_t noise_stream, float *d_out, void *stream);
int dfx_free(void *d_ptr);

const char *dfx_last_error(void);
const char *dfx_version(void);
/* byte offset, inside a 1 KB block of 32 IVF-PQ vectors, of subquantizer m of vector v for block
 * layout 1 or 2 (host function; lets the layout be checked without a GPU) */
int dfx_debug_il_byte(int layout, int v, int m);

#ifdef __cplusplus
}
#endif
#endif /* DFX_H */
