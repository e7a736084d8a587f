/*
 * semtools_b200.h -- C ABI of the B200-native `search` hot path of semtools.
 *
 * The reference (run-llama/semtools v3.0.0, paths relative to /root/reference)
 * has no FFI layer of its own: the seam is a set of Rust calls into two
 * third-party crates (model2vec-rs, simsimd) plus its own scan/sort loop.  Each
 * entry point below names the reference interface it replaces; INTEGRATION.md
 * shows the `extern "C"` block a semtools maintainer would add.
 *
 * Conventions
 *   - every function returns 0 (STB_OK) or a negative stb_status;
 *     stb_last_error() returns the message of the calling thread's last failure
 *   - nothing throws or aborts across this boundary
 *   - the caller owns every buffer it passes; the library owns everything
 *     behind the opaque handles; outputs go to caller-allocated arrays with
 *     explicit capacities
 *   - one host thread per context at a time (the reference runs the whole
 *     search path on one blocking thread, src/bin/semtools.rs:134-135)
 *   - pointers named *_dev are CUDA device pointers on the context's device,
 *     everything else is host memory
 *   - there is NO CPU fallback: without a usable sm_100 device every call fails
 *     with STB_ERR_CUDA
 *
 * Vector width is fixed at 256 f32 (LINE_EMBEDDING_SIZE,
 * src/workspace/store.rs:37); other widths fail with STB_ERR_ARG.
 *
 * Environment switches (read per call; results are identical whatever their
 * value -- they select how candidates are found, never how the returned
 * distances are computed): STB_SCAN_TIER=f32|h16|q8 (narrowest candidate copy K1
 * may read, default q8), STB_DIRECT_OUT=0, STB_BATCH_V1=1, STB_IVFPQ_V1=1
 * (INTEGRATION.md, 5b).
 */
#ifndef SEMTOOLS_B200_H
#define SEMTOOLS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STB_DIM 256u

typedef enum stb_status {
  STB_OK = 0,
  STB_ERR_ARG = -1,      /* bad argument (null handle, wrong width, ...)          */
  STB_ERR_CUDA = -2,     /* CUDA runtime failure / no sm_100 device                */
  STB_ERR_NOMEM = -3,    /* host or device allocation failed                       */
  STB_ERR_RANGE = -4,    /* token id / row range outside the table or corpus       */
  STB_ERR_CAPACITY = -5, /* result does not fit `cap`; *out_n holds the full count */
  STB_ERR_STATE = -6     /* call not valid in the handle's current state           */
} stb_status;

typedef struct stb_ctx stb_ctx;       /* one CUDA device + stream + scratch        */
typedef struct stb_table stb_table;   /* model2vec embedding table resident in HBM */
typedef struct stb_corpus stb_corpus; /* row-major N x 256 f32 line-vector matrix  */

/* One search hit: (distance, global row) -- 16 bytes, the unit of the
 * cross-GPU top-k exchange.  `row` is the line's position in (document order,
 * line order), i.e. the reference's iteration order (src/search/mod.rs:84-85),
 * so ordering by (distance, row) reproduces its stable sort (:107-111). */
typedef struct stb_hit {
  double distance;
  uint64_t row;
} stb_hit;

int stb_version(void);
const char *stb_last_error(void);

/* Device count visible to the library (0 if no driver / no GPU). */
int stb_device_count(void);

/* ---- context ----------------------------------------------------------------
 * `cuda_stream` may be NULL (the library creates its own non-blocking stream) or
 * an existing cudaStream_t that every kernel/copy of this context is issued on
 * (lets a host framework time the work with its own events).  NULL never means
 * "the default stream": pass cudaStreamLegacy / cudaStreamPerThread for those.
 * Tables and corpora may be destroyed after their context (any order is safe). */
int stb_ctx_create(int device, void *cuda_stream, stb_ctx **out);
int stb_ctx_destroy(stb_ctx *ctx);
int stb_ctx_sync(stb_ctx *ctx);
/* cudaStream_t the context launches on. */
void *stb_ctx_stream(stb_ctx *ctx);

/* ---- embedding table ---------------------------------------------------------
 * Replaces the tensors held by StaticModel after
 * StaticModel::from_pretrained(MODEL_NAME, None, None, None)
 * (src/cmds/search.rs:123-128, src/search/mod.rs:16): table E[V][256] f32,
 * optional per-token weights[n_weights], optional token->row mapping[n_mapping],
 * and the `normalize` flag from config.json.  Uploaded once, read-only after. */
int stb_table_load(stb_ctx *ctx, const float *E, uint64_t V, uint32_t D,
                   const float *weights, uint64_t n_weights,
                   const uint32_t *mapping, uint64_t n_mapping, int normalize,
                   stb_table **out);
int stb_table_destroy(stb_table *table);

/* ---- corpus -------------------------------------------------------------------
 * Replaces Document.embeddings: Vec<Vec<f32>> (src/search/mod.rs:18-22) and the
 * line_embeddings shard's vectors (src/workspace/store.rs:140-160) with ONE
 * contiguous matrix in HBM.  `row_base` is the global row id of local row 0
 * (non-zero when this context holds one row-shard of a larger corpus). */
int stb_corpus_create(stb_ctx *ctx, uint32_t D, uint64_t capacity_rows,
                      uint64_t row_base, stb_corpus **out);
int stb_corpus_destroy(stb_corpus *corpus);
int stb_corpus_append(stb_corpus *corpus, const float *rows, uint64_t n);
int stb_corpus_append_dev(stb_corpus *corpus, const float *rows_dev, uint64_t n);
int stb_corpus_clear(stb_corpus *corpus);
int stb_corpus_rows(const stb_corpus *corpus, uint64_t *n);
/* device pointer of local row 0 (for zero-copy producers). */
int stb_corpus_data_dev(const stb_corpus *corpus, float **rows_dev);
/* copy rows [first, first+n) back to the host (tests, store write-back). */
int stb_corpus_read(const stb_corpus *corpus, uint64_t first, uint64_t n,
                    float *rows);

/* ---- K3: gather + mean-pool + L2-normalise -------------------------------------
 * Replaces model.encode_with_args(&lines, Some(2048), 16384)
 * (src/search/mod.rs:69, src/cmds/search.rs:154) and model.encode_single(q)
 * (src/search/mod.rs:138,153; src/cmds/search.rs:136) MINUS tokenisation, which
 * stays on the host: the caller passes the token ids of each line as a CSR batch
 * (offsets[n_lines+1], ids[offsets[n_lines]]), already unk-dropped and truncated
 * (2048 ids per corpus line, 512 for the query).  Output row i is bit-identical
 * to pool_ids(ids of line i) of model2vec-rs 0.1.3.
 * `out` (host, n_lines x 256) and `append_to` may each be NULL; with `append_to`
 * the rows are written straight into the corpus in HBM and never visit the host.
 * A token whose table row is out of range fails the call with STB_ERR_RANGE
 * (upstream panics) and appends nothing. */
int stb_embed(stb_ctx *ctx, const stb_table *table, const uint64_t *offsets,
              const uint32_t *ids, uint64_t n_lines, float *out,
              stb_corpus *append_to);

/* Asynchronous device-resident form of stb_embed: CSR and output already in HBM
 * (out_dev: n_lines x 256 f32, e.g. a slice of stb_corpus_data_dev), nothing
 * synchronises.  A token outside the table sets a sticky flag instead of failing;
 * stb_embed_status() synchronises the stream, returns STB_ERR_RANGE if the flag was
 * set since the last call, and clears it. */
int stb_embed_dev(stb_ctx *ctx, const stb_table *table, const uint64_t *offsets_dev,
                  const uint32_t *ids_dev, uint64_t n_lines, float *out_dev);
int stb_embed_status(stb_ctx *ctx);

/* ---- K1 + K4: cosine scan, top-k / threshold, exact re-rank ---------------------
 * Replaces search_documents' scan/filter/sort/take (src/search/mod.rs:84-119,
 * one f32::cosine per line at :86) and, with `row_ranges`, the filtered query of
 * Store::search_line_embeddings (src/workspace/store.rs:481-546).
 *
 *   q            256 f32 query vector (host)
 *   top_k        config.top_k (:118)
 *   has_max /    config.max_distance (:88): a hit needs distance < max_distance
 *   max_distance (strict; 100.0 when absent).
 *   mode         STB_MODE_SEARCH_DOCUMENTS: has_max lifts the top_k cap (:115-119)
 *                STB_MODE_STORE_QUERY:      top_k always caps (store.rs:517,543)
 *   row_ranges   NULL, or n_ranges half-open [begin,end) pairs of GLOBAL rows,
 *                ascending and disjoint: only these rows are scanned
 *   out_hits     cap entries; on return the first min(*out_n, cap) are filled,
 *                ordered by (distance asc, row asc); distances are the canonical
 *                f64 cosine distance (oracle/semtools_oracle.c: orc_cosine_f32)
 *   out_n        full result count; if it exceeds cap the call returns
 *                STB_ERR_CAPACITY after filling cap entries
 * On a sharded corpus (row_base != 0 or several contexts) the result is the
 * shard-local answer; merge shards with stb_hits_merge*. */
#define STB_MODE_SEARCH_DOCUMENTS 0
#define STB_MODE_STORE_QUERY 1
int stb_search(stb_ctx *ctx, const stb_corpus *corpus, const float *q,
               uint32_t top_k, int has_max, double max_distance, int mode,
               const uint64_t *row_ranges, uint32_t n_ranges, stb_hit *out_hits,
               uint64_t cap, uint64_t *out_n);

/* Candidate tiers.  The scan is HBM-bound, so the way to go faster than the f32 roofline is
 * to read fewer bytes: stb_search can draw its candidates from a reduced-width copy of the
 * corpus -- "q8": int8 codes + one f32 scale per row, 260 B/row, top_k <= 16; "h16": the
 * 16-bit L2-normalised shadow K2 multiplies, 512 B/row -- and re-ranks them in the canonical
 * f64 arithmetic on the f32 rows exactly as before.  Each tier proves its own result (rounding
 * bound of the copy vs. the gap to the best row it dropped); an unproven query is retried on
 * the next wider tier, so the hits are identical to the f32 path's.  stb_search builds the
 * copies lazily (second query on an unchanged corpus of >= 32768 rows);
 * stb_corpus_prepare builds them now.  Costs +25 % / +50 % HBM.  No reference analogue
 * (the reference keeps Vec<Vec<f32>>, src/search/mod.rs:18-22). */
#define STB_PREPARE_Q8 1
#define STB_PREPARE_H16 2
int stb_corpus_prepare(stb_corpus *corpus, int what);
/* Per-tier bookkeeping of stb_search on this corpus since its last change, index = tier
 * (0 f32, 1 h16, 2 q8): fast-path scans tried / proven, and the rows each copy covers
 * (0 = not built or refused).  Any pointer may be NULL. */
int stb_corpus_tier_stats(const stb_corpus *corpus, uint32_t tries[3], uint32_t proven[3],
                          uint64_t built_rows[3]);

/* Asynchronous device-resident form of the top-k search (no threshold, no
 * ranges): query and results stay in HBM, nothing synchronises.  out_hits_dev
 * receives top_k entries (unused tail: distance = +inf, row = UINT64_MAX) and
 * out_status_dev[0] the hit count, out_status_dev[1] a completeness flag
 * (1 = provably the exact top-k; 0 = the candidate margin check failed and the
 * caller must fall back to stb_search, which handles it internally),
 * out_status_dev[3] = K' | tier << 16 (tier: 0 f32, 1 h16, 2 q8).  Reads the
 * narrowest copy that is already built (never builds one). */
int stb_search_topk_dev(stb_ctx *ctx, const stb_corpus *corpus,
                        const float *q_dev, uint32_t top_k, stb_hit *out_hits_dev,
                        uint32_t *out_status_dev);

/* ---- K2: batched queries on the tensor cores ------------------------------------------
 * Q independent top-k searches (the semantics of Q calls of search_documents,
 * src/search/mod.rs:77-120, without max_distance) in one pass over the corpus: an
 * L2-normalised bf16 copy of the corpus (built lazily, 512 B/row, rebuilt after the
 * corpus changes; stb_corpus_prepare_batch builds it ahead of time) is multiplied with
 * the query tile on tcgen05 tensor cores, the 32 most promising 32-row sub-tiles per
 * query are re-scored exactly (canonical f64 distance on the f32 rows) and the result is
 * accepted only if the bf16 error bound proves no other row can enter the top-k;
 * unproven queries are answered by the single-query path (stb_search).  Results are
 * therefore identical to stb_search.
 *   q         nq x 256 f32 (host);  out_hits nq x top_k (unused tail: +inf / UINT64_MAX)
 *   out_n     nq counts */
int stb_corpus_prepare_batch(stb_corpus *corpus);
int stb_search_batch(stb_ctx *ctx, const stb_corpus *corpus, const float *q, uint32_t nq,
                     uint32_t top_k, stb_hit *out_hits, uint32_t *out_n);
/* Asynchronous device-resident form: out_status_dev[2*i] = hits of query i,
 * [2*i+1] = 1 iff proven exact (0: re-run query i through stb_search). */
int stb_search_batch_dev(stb_ctx *ctx, const stb_corpus *corpus, const float *q_dev,
                         uint32_t nq, uint32_t top_k, stb_hit *out_hits_dev,
                         uint32_t *out_status_dev);

/* ---- fused multi-GPU search: K1 -> exchange over NVLink peer memory -> K4 -------------
 * One process (or thread) per GPU, one stb_xchg per rank.  Each rank allocates an
 * exchange buffer; the ranks trade its 64-byte CUDA IPC handle through whatever channel
 * the host has (MPI, torch.distributed, a pipe ...) and connect.  After that
 * stb_search_topk_xchg is ONE kernel per query per rank: the scan's final CTA stores its
 * k hits directly into every peer's buffer, release-stores a sequence flag, waits for
 * the peers' flags and merges by (distance,row) -- no NCCL call, no second launch.
 * All ranks must issue the same sequence of stb_search_topk_xchg calls (same top_k).
 * Within one process (several contexts), use stb_xchg_connect_local instead of IPC.
 *   out_status_dev[0] = hits, [1] = 1 iff every rank proved its shard result exact
 *   (0 -> run the per-shard stb_search + stb_hits_merge path), [2] = 0xfffffffe if a
 *   peer never arrived.  The wait is bounded (~15 s of SM cycles): ranks may enter a call seconds
 *   apart, not more.  After a timeout the ranks no longer agree on what was exchanged: stop using
 *   the exchange (destroy it on every rank); do NOT re-run queries on it, a surplus call waits a
 *   full bound for peers that will not come.  The synchronous entry points (stb_search_xchg,
 *   stb_search_many) mark the exchange dead when they see the timeout: every later call on it
 *   returns STB_ERR_STATE at once. */
typedef struct stb_xchg stb_xchg;
#define STB_IPC_HANDLE_BYTES 64
#define STB_XCHG_MAX_RANKS 8
int stb_xchg_create(stb_ctx *ctx, uint32_t world, uint32_t rank, uint32_t max_k,
                    stb_xchg **out);
int stb_xchg_destroy(stb_xchg *x);
int stb_xchg_local_handle(stb_xchg *x, uint8_t handle[STB_IPC_HANDLE_BYTES]);
/* handles: world x 64 bytes, entry r = rank r's handle (own entry ignored). */
int stb_xchg_connect(stb_xchg *x, const uint8_t *handles);
/* same-process variant: peers[r] = the stb_xchg of rank r (peers[rank] == x). */
int stb_xchg_connect_local(stb_xchg *x, stb_xchg *const *peers);
int stb_search_topk_xchg(stb_ctx *ctx, const stb_corpus *corpus, const float *q_dev,
                         uint32_t top_k, stb_xchg *x, stb_hit *out_hits_dev,
                         uint32_t *out_status_dev);
/* Sharded K2 over the same peer-memory exchange.  stb_xchg_create_batch allocates, behind the single-query
 * area, two batch slots of world x max_nq x max_k hits (+ flags and per-query proof bits); everything else
 * (handles, connect, destroy, stb_search_topk_xchg) works as with stb_xchg_create.
 * stb_search_batch_xchg_dev = stb_search_batch_dev on the local shard, then a push kernel (this rank's
 * nq x k hits into every peer's slot over NVLink, release-stored sequence flag) and a merge kernel (waits
 * for every peer's flag, merges each query's world x k hits by (distance,row)): two launches, no NCCL.
 *   out_status_dev[2q] = hits of query q, [2q+1] = 1 iff every rank proved its part (0: re-run query q
 *   through stb_search_xchg / stb_search_many on every rank; 2: a peer never arrived -- see above:
 *   treat the exchange as dead, the flags of this batch are not the same on every rank).
 * All ranks must issue the same sequence of calls. */
int stb_xchg_create_batch(stb_ctx *ctx, uint32_t world, uint32_t rank, uint32_t max_k, uint32_t max_nq,
                          stb_xchg **out);
int stb_search_batch_xchg_dev(stb_ctx *ctx, const stb_corpus *corpus, const float *q_dev, uint32_t nq,
                              uint32_t top_k, stb_xchg *x, stb_hit *out_hits_dev, uint32_t *out_status_dev);

/* ---- K5: IVF-PQ index (approximate) ------------------------------------------------------
 * NOT a replacement of any reference code: this snapshot of semtools has no IVF_PQ (the
 * store is qdrant-edge with a plain index, src/workspace/store.rs:129-130,156-157; the
 * string survives only in README.md:125).  Self-specified for BASELINE config 5 and
 * measured by recall against stb_search: coarse spherical k-means (nlist lists), 32 x 8-bit
 * product quantiser on the residual, ADC lookup-table scan of the nprobe best lists,
 * exact re-rank of the `rerank` best candidates.  Returned distances are exact canonical
 * distances; only the candidate set is approximate.  The index refers to the corpus it
 * was built on (rows [0, n) at build time) and must be destroyed before it. */
typedef struct stb_ivfpq stb_ivfpq;
int stb_ivfpq_build(stb_ctx *ctx, const stb_corpus *corpus, uint32_t nlist, uint32_t train_rows,
                    uint32_t iters, stb_ivfpq **out);
int stb_ivfpq_destroy(stb_ivfpq *index);
int stb_ivfpq_stats(const stb_ivfpq *index, uint64_t *rows, uint32_t *nlist, uint32_t *max_list,
                    uint64_t *index_bytes);
int stb_ivfpq_search(stb_ivfpq *index, const float *q, uint32_t nprobe, uint32_t top_k,
                     uint32_t rerank, stb_hit *out_hits, uint32_t *out_n, uint64_t *out_scanned);
/* Asynchronous device-resident form (query, hits and status stay in HBM, nothing synchronises): the
 * sharded index is one of these per rank, an all-gather of the k hits and stb_hits_merge_dev.
 * out_hits_dev: top_k entries (unused tail +inf / UINT64_MAX); out_status_dev[0] = hits, [1] = codes
 * scanned.  rerank is capped at 1024. */
int stb_ivfpq_search_dev(stb_ivfpq *index, const float *q_dev, uint32_t nprobe, uint32_t top_k,
                         uint32_t rerank, stb_hit *out_hits_dev, uint32_t *out_status_dev);

/* Host-buffer form of the fused multi-GPU search (the call a sharded host makes per query):
 * pinned H2D of the query, ONE kernel (scan + NVLink exchange + merge), D2H of the merged
 * hits, stream sync.  *out_complete = 0 means some rank could not prove its shard result
 * (all ranks see the same flag): run stb_search per shard + stb_hits_merge instead. */
int stb_search_xchg(stb_ctx *ctx, const stb_corpus *corpus, const float *q, uint32_t top_k,
                    stb_xchg *x, stb_hit *out_hits, uint32_t *out_n, int *out_complete);

/* Many independent single queries, one synchronisation (a host that has several queries in hand:
 * an agent's tool calls, a batch of CLI invocations).  q: nq x 256 f32 (host); out_hits: nq x top_k
 * (entry i*top_k.. of query i), out_n: nq counts.  Each query is its own scan (use stb_search_batch
 * when nq is in the hundreds: one pass over the corpus for all of them); the kernels are enqueued
 * back to back, so every tail overlaps the next scan, and hits are written straight to pinned host
 * memory.  x == NULL: results are exactly stb_search's (an unproven query is re-run through it).
 * x != NULL: the sharded form of stb_search_xchg -- out_complete[i] = 0 marks a query some rank could
 * not prove (every rank sees the same flags).  out_complete may be NULL when x is NULL.
 * Validation state: the x == NULL form is covered by the GPU suite; the x != NULL form is the same kernel
 * stb_search_xchg launches, enqueued nq times, but has not yet run on a multi-GPU box. */
int stb_search_many(stb_ctx *ctx, const stb_corpus *corpus, const float *q, uint32_t nq, uint32_t top_k,
                    stb_xchg *x, stb_hit *out_hits, uint32_t *out_n, uint8_t *out_complete);

/* ---- K4: merge per-shard hit lists -----------------------------------------------
 * The final sort_by + take of src/search/mod.rs:107-119 applied across row
 * shards: `lists_dev` holds n_lists x per_list hits (e.g. the all-gathered
 * per-GPU top-k; padding entries have distance = +inf); writes the top_k best by
 * (distance, row) to out_dev.  Asynchronous on the context's stream. */
int stb_hits_merge_dev(stb_ctx *ctx, const stb_hit *lists_dev, uint32_t n_lists,
                       uint32_t per_list, uint32_t top_k, stb_hit *out_dev);
/* Batched form for sharded K2: lists_dev[n_lists][nq][per_list] (e.g. the all-gathered
 * per-rank results of stb_search_batch_dev) -> out_dev[nq][top_k]; n_lists*per_list <= 2048. */
int stb_hits_merge_batch_dev(stb_ctx *ctx, const stb_hit *lists_dev, uint32_t n_lists,
                             uint32_t nq, uint32_t per_list, uint32_t top_k, stb_hit *out_dev);
/* Host-buffer convenience wrapper (copies in, merges on the GPU, copies out). */
int stb_hits_merge(stb_ctx *ctx, const stb_hit *lists, uint32_t n_lists,
                   uint32_t per_list, uint32_t top_k, stb_hit *out,
                   uint32_t *out_n);

/* ---- ids -------------------------------------------------------------------------
 * fnv1a_hash (src/workspace/store.rs:651-661); DocMeta::id (:75-80) is
 * stb_fnv1a64(path); LineEmbedding::id (:82-89) is stb_line_id. Pure host code. */
uint64_t stb_fnv1a64(const uint8_t *bytes, uint64_t len);
uint64_t stb_line_id(const uint8_t *path, uint64_t path_len, int32_t line_number);
/* stb_line_id for n_rows (path index, line_number) int32 pairs at once (rebuilding a store's
 * id map): paths = one byte blob + n_paths+1 offsets.  STB_ERR_RANGE on a bad path index. */
int stb_line_ids(const uint8_t *path_bytes, const uint64_t *path_offsets, uint32_t n_paths,
                 const int32_t *rows, uint64_t n_rows, uint64_t *out_ids);

/* ---- introspection (bench / tests) -------------------------------------------------
 * Counters since context creation: kernels launched by this library on the
 * context, and how many searches needed the fallback pass. */
int stb_ctx_counters(const stb_ctx *ctx, uint64_t *kernel_launches,
                     uint64_t *fallback_searches);
/* Consistency check of K1's dynamic tile schedule (synchronises): the device-side ticket counter
 * must equal the value the host booked over all launches so far; STB_ERR_STATE otherwise. */
int stb_debug_ticket_check(stb_ctx *ctx, uint64_t *device_value, uint64_t *host_value);
/* Tuning aid: K1's scan front, the virtual row at which the next ticketed top-k launch starts its
 * wrapped scan (any value is correct; consecutive scans share HBM traffic by starting where the
 * running one is).  set != 0 stores *value, else reads it into *value.  Synchronises. */
int stb_debug_scan_front(stb_ctx *ctx, int set, uint64_t *value);
/* Tuning aid: phase timestamps (ns, %globaltimer) of the last K1 launch; only filled by
 * libraries built with -DSTB_TAIL_TIMING.  reset=1 arms, reset=0 reads 8 values:
 * [0] first CTA start, [1] last scan end, [2] last CTA merge end, [3] final ticket,
 * [4] select done, [5] re-rank done. */
int stb_debug_timestamps(stb_ctx *ctx, int reset, uint64_t out[8]);
/* Test hook for K2: shadow build + tcgen05 GEMM on host inputs; out_full receives the
 * approximate cosine matrix [ceil(nq/128)*128][ceil(n/256)*256] (f32), out_submax (may be
 * NULL) the per-32-row maxima [ceil(nq/128)][ceil(n/256)*8][128]. */
int stb_debug_batch_gemm(stb_ctx *ctx, const float *q, uint32_t nq, const float *rows,
                         uint64_t n, float *out_full, float *out_submax);
/* Build parameters of K2 (host-only): element type of the shadow the tensor-core pass runs on
 * (0 = bf16, 1 = fp16) and the bound |approximate - exact cosine| <= eps its selection uses. */
int stb_debug_batch_params(int *shadow_is_f16, double *eps);

#ifdef __cplusplus
}
#endif
#endif /* SEMTOOLS_B200_H */
