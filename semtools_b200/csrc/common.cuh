// Internal declarations shared by the translation units of libsemtools_b200.so.
// Everything here is sm_100a-only product code; nothing in this directory may
// include, link or call anything under oracle/.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/semtools_b200.h"

#define STB_D 256           // floats per row
#define STB_ROW_F4 64       // float4 per row
#ifndef STB_SCAN_THREADS
#define STB_SCAN_THREADS 256
#endif
#ifndef STB_SCAN_MINB
#define STB_SCAN_MINB 2     // CTAs per SM the scan kernels are register-budgeted for
#endif
#define STB_SCAN_WARPS (STB_SCAN_THREADS / 32)
#define STB_SORT_CAP 1024   // keys one CTA sorts in shared memory
// Rigorous bound (with ~4x slack) on |approx cosine - exact cosine| for the fp32
// scan arithmetic on rows whose squared norm is a normal fp32 number; derivation
// in DESIGN.md "Candidate completeness".  Rows outside that range are forced
// into the candidate set instead of being scored.
#define STB_SCORE_EPS 1.0e-5
// Element type of the 16-bit L2-normalised corpus shadow (K2 operand; K1's opt-in half-width
// scan): fp16 by default (same tcgen05 kind::f16 rate as bf16, 8x smaller rounding bound for unit
// rows; validated on hardware in round 2), bf16 with -DSTB_SHADOW_F16=0.
#ifndef STB_SHADOW_F16
#define STB_SHADOW_F16 1
#endif
// |q^ . shadow(x) - exact cosine| when only the ROW is rounded (K1 shadow scan: the query stays
// f32): <= u * ||q^|| * ||x^|| = u (unit roundoff: 2^-8 bf16, 2^-11 fp16; fp16 components below 2^-14 add
// <= 16 * 2^-25 * ||q^||_1 <= 8e-6), plus f32 accumulation and rsqrt (< 2e-5).
#if STB_SHADOW_F16
#define STB_SHADOW_SCAN_EPS 0.00052
#else
#define STB_SHADOW_SCAN_EPS 0.0040
#endif
// K1 candidate tiers (which copy of the corpus the streaming pass reads; the exact f64 re-rank
// and the completeness proof are common to all): f32 rows (1 KiB/row), 16-bit normalised shadow
// (512 B/row, also K2's operand), int8 codes + per-row scale (260 B/row).
#define STB_TIER_F32 0
#define STB_TIER_H16 1
#define STB_TIER_Q8 2
// Not a tier of its own: a 4-bit coarse pass (136 B/row) whose candidates each CTA re-scores with the
// q8 copy; built and invalidated with q8, counted and reported as q8 (scan_topk.cu: stb_scan_q4).
#define STB_TIER_Q4Q8 3
// q8 scores are upper bounds of the exact cosine up to the fp32 evaluation of the bound itself
// and of the two normalisations (< 4e-6, scan_topk.cu: stb_scan_q8); proof slack:
#define STB_Q8_SCAN_EPS 2.0e-5
// the q8 tier always keeps K' = 128 candidates; beyond this top_k the gap between the k-th and
// the 128th best is too small for its ~0.01 per-row error term to prove anything
#define STB_Q8_MAX_K 16

void stb_set_error(const char *fmt, ...);

#define STB_CUDA(call)                                                             \
  do {                                                                             \
    cudaError_t _e = (call);                                                       \
    if (_e != cudaSuccess) {                                                       \
      stb_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,                  \
                    cudaGetErrorString(_e));                                       \
      return STB_ERR_CUDA;                                                         \
    }                                                                              \
  } while (0)

struct stb_ctx {
  int device;
  int sm_count;
  cudaStream_t stream;
  bool own_stream;
  // --- scan scratch (device) ---
  uint64_t *block_keys;     // candidate keys of every tree level
  size_t block_keys_cap;    // in keys
  unsigned int *counters;   // tree arrival counters (zeroed; kernels re-zero)
  size_t counters_cap;
  // K1 tile-ticket counters (monotonic; scan_topk.cu: stb_for_each_tile).  A ring of STB_TICKET_SLOTS
  // counters, one per launch in turn: two consecutive scans may run concurrently and must not draw
  // from the same counter.
  unsigned long long *tickets;         // [STB_TICKET_SLOTS] counters, then the words below
  unsigned long long *scan_start;      // [STB_TICKET_SLOTS] per slot: (launch seq << 32) | start tile
  unsigned long long *scan_front;      // [1] a virtual row a running scan reached (synchronized scans)
  unsigned long long ticket_next[8];   // per slot: its value when the next launch using it starts
  unsigned long long topk_launches;    // picks the slot
  float *q_dev;             // 256 f32 staging for host queries
  stb_hit *hits_dev;        // result hits (top-k path)
  size_t hits_cap;
  uint32_t *status_dev;     // [0]=n hits, [1]=complete flag, [2..] debug
  uint32_t *collect_rows;   // threshold/fallback compaction: local row ids
  size_t collect_cap;
  unsigned long long *collect_count;
  stb_hit *collect_hits;    // exact hits of collected rows (sorted in place)
  size_t collect_hits_cap;
  uint64_t *ranges_dev;     // [3 * n] : begin(local), end(local), vstart
  size_t ranges_cap;
  int *err_flag;            // device int for K3 range errors
  unsigned int *hist_dev;       // 4096-bin score histogram (large-k path)
  unsigned long long *dbg_dev;  // 8 u64 phase timestamps (STB_TAIL_TIMING builds; else unused)
  // cudaFuncSetAttribute is per DEVICE: remembered per context, never in function statics
  // (one process may hold contexts on several GPUs)
  uint32_t func_attr_mask;
  size_t finish2_smem_set;
  // --- K2 scratch ---
  uint8_t *bq_tiles; size_t bq_tiles_cap;     // query shadow tiles
  float *b_submax; size_t b_submax_cap;       // [n_sub][q_pad]
  float *b_tilemax; size_t b_tilemax_cap;     // [n_tiles][q_pad]
  uint64_t *b_cand; size_t b_cand_cap;        // [q_pad][slices][32]
  float *b_thr; size_t b_thr_cap;             // v2: [q_pad] emission thresholds
  uint32_t *b_cnt; size_t b_cnt_cap;          // v2: [q_pad] emitted-candidate counters
  uint64_t *b_keys; size_t b_keys_cap;        // v2: [q_pad][cand_cap] emitted keys
  float *bq_dev; size_t bq_dev_cap;           // host-call staging: queries
  stb_hit *bh_dev; size_t bh_dev_cap;         // host-call staging: hits
  uint32_t *bs_dev; size_t bs_dev_cap;        // host-call staging: status
  uint64_t *embed_off_dev;  // K3 staging: CSR offsets
  size_t embed_off_cap;
  uint32_t *embed_ids_dev;  // K3 staging: token ids
  size_t embed_ids_cap;
  float *embed_out_dev;     // K3 output when not appending to a corpus
  size_t embed_out_cap;
  // --- pinned host staging ---
  float *q_pin;
  stb_hit *hits_pin;
  size_t hits_pin_cap;
  uint32_t *status_pin;
  float *many_q_pin;          // stb_search_many: queries / per-query status (kernels write the latter directly)
  uint32_t *many_status_pin;
  size_t many_q_pin_cap;      // in floats
  // --- counters ---
  uint64_t kernel_launches;
  uint64_t fallback_searches;
};

#define STB_TICKET_SLOTS 8
// Spin-wait bound of the peer-memory exchanges (SM cycles, ~15 s): long enough that ranks entering a sharded
// search a few seconds apart (first-call allocations, a busy host) still meet; a peer that is really gone
// costs one bound, the call reports it (status 0xfffffffe / 2) and the caller must stop using the exchange:
// ranks that disagree on whether an exchange happened no longer issue the same sequence of calls.
#define STB_XCHG_TIMEOUT_CYCLES 30000000000ll
#define STB_XCHG_SLOTS 4
#define STB_XCHG_MAX_WORLD 8
struct StbXchgArgs {
  unsigned char *base[STB_XCHG_MAX_WORLD];   // exchange buffer of every rank (peer-mapped)
  uint32_t world, rank, max_k, slot;
  unsigned long long seq;
};

struct stb_xchg {
  stb_ctx *ctx;
  uint32_t world, rank, max_k;
  unsigned char *local;                      // this rank's buffer (cudaMalloc)
  size_t bytes;
  unsigned char *peers[STB_XCHG_MAX_WORLD];  // peers[rank] == local
  bool ipc_opened[STB_XCHG_MAX_WORLD];
  bool connected;
  unsigned long long seq;
  // batch area (stb_xchg_create_batch; sharded K2): 2 slots x { flags[world] u64 | status[world][max_nq] u32 |
  // hits[world][max_nq][max_k] } behind the single-query area
  uint32_t max_nq;
  size_t batch_off, batch_slot_bytes;
  unsigned long long batch_seq;
  unsigned int *batch_ticket;                // device: arrival counter of the push kernel
  bool dead;                                 // a synchronous call saw a peer time-out: every later call is refused
};

struct stb_table {
  stb_ctx *ctx;
  float *E;            // V x 256
  uint64_t V;
  float *weights;      // or nullptr
  uint64_t n_weights;
  uint32_t *mapping;   // or nullptr
  uint64_t n_mapping;
  int normalize;
};

struct stb_corpus {
  stb_ctx *ctx;
  float *rows;         // capacity x 256
  uint64_t n;
  uint64_t capacity;
  uint64_t row_base;
  // K2: L2-normalised bf16 copy in tcgen05 tile layout (built lazily, rebuilt when n changes)
  uint8_t *shadow;
  uint64_t shadow_rows;      // rows covered by `shadow` (== n when valid)
  uint64_t shadow_cap_tiles;
  int shadow_bad;            // 1: some row cannot be normalised in fp32 -> tensor path refused
  // K1 tier q8: int8 codes [capacity][256] + per-row scale, built lazily / by stb_corpus_prepare
  uint8_t *q8;
  float *q8_scale;
  uint64_t q8_rows;          // rows covered (== n when valid)
  uint64_t q8_cap_rows;
  int q8_bad;
  // coarse copy in front of q8 (same rows, capacity and bad flag): 4-bit codes [capacity][128] + (s4, r)
  uint8_t *q4;
  float2 *q4_sr;
  // per-tier bookkeeping: a reduced-width tier is skipped once it proves fewer than half of its
  // results on this corpus (index = STB_TIER_*)
  uint32_t tier_tries[3], tier_proven[3];
  uint32_t coarse_tries, coarse_proven;   // the same rule for the coarse stage in front of q8
  uint32_t searches_since_change;   // lazy builds wait for the second query on an unchanged corpus
};

// ---- scan_topk.cu -------------------------------------------------------------
// Fast path: one kernel = scan + per-warp running top-K' + CTA/tree merge +
// exact f64 re-rank + completeness check.  q_dev: 256 f32 on device.
// n_ranges > 0: ranges_dev holds local [begin,end,vstart] triples.
// tier: STB_TIER_* or STB_TIER_Q4Q8 -- which copy of `c` the streaming pass reads (must exist and be current).
// overlapped: the launch is one of a pipelined series (asynchronous entry points): the grid is sized
// for ONE CTA per SM and releases its dependent at its START, so the next query's scan co-runs with
// this one instead of waiting for it to drain (scan_topk.cu: "overlapped launches").
int stb_launch_scan_topk(stb_ctx *ctx, const stb_corpus *c, int tier, const float *q_dev, uint32_t top_k,
                         const uint64_t *ranges_dev, uint32_t n_ranges,
                         uint64_t n_virtual, stb_hit *out_hits_dev,
                         uint32_t *out_status_dev, const StbXchgArgs *xchg = nullptr, bool overlapped = false);
// int8 codes + scales of rows [first_row, n_rows) (q8 tier)
int stb_launch_q8_build(stb_ctx *ctx, const float *rows_dev, uint64_t first_row, uint64_t n_rows, uint8_t *out,
                        float *scale, int *bad_flag_dev);
// 4-bit codes + (s4, r) of rows [first_row, n_rows) (coarse stage in front of q8)
int stb_launch_q4_build(stb_ctx *ctx, const float *rows_dev, uint64_t first_row, uint64_t n_rows, uint8_t *out,
                        float2 *sr, int *bad_flag_dev);
// Largest top_k the fast path serves.
uint32_t stb_scan_topk_max_k(void);
// Collect path: every row whose approximate cosine >= cos_floor (or that cannot be
// scored safely) is appended to ctx->collect_rows; total count -> collect_count.
// tier: STB_TIER_F32 (approximate cosine of the f32 rows) or STB_TIER_Q8 (upper bounds from the int8 copy)
int stb_launch_scan_collect(stb_ctx *ctx, const stb_corpus *c, int tier,
                            const float *q_dev, float cos_floor,
                            const uint64_t *ranges_dev, uint32_t n_ranges,
                            uint64_t n_virtual);
// Large-k support: 4096-bin histogram of the approximate cosine over the scanned rows
// (bin b: cos in (1-(b+1)/2048, 1-b/2048]).  hist_dev: 4096 u32 on device.
int stb_launch_scan_hist(stb_ctx *ctx, const stb_corpus *c, int tier, const float *q_dev, const uint64_t *ranges_dev,
                         uint32_t n_ranges, uint64_t n_virtual, unsigned int *hist_dev);
// Exact canonical distances of m collected rows -> hits (invalid/failing rows get
// distance=+inf,row=UINT64_MAX); counts passing rows into pass_count.
int stb_launch_exact(stb_ctx *ctx, const float *rows, uint64_t row_base,
                     const float *q_dev, const uint32_t *row_ids, uint64_t m,
                     double limit, stb_hit *hits, uint64_t m_padded,
                     unsigned long long *pass_count);
// In-place ascending sort by (distance,row) of m_padded (power of two) hits.
int stb_launch_sort_hits(stb_ctx *ctx, stb_hit *hits, uint64_t m_padded);

// ---- hits_merge.cu --------------------------------------------------------------
int stb_launch_hits_merge(stb_ctx *ctx, const stb_hit *lists_dev, uint32_t n_lists,
                          uint32_t per_list, uint32_t top_k, stb_hit *out_dev);

int stb_launch_hits_merge_batch(stb_ctx *ctx, const stb_hit *lists_dev, uint32_t n_lists, uint32_t nq,
                                uint32_t per_list, uint32_t top_k, stb_hit *out_dev);
// sharded K2 exchange over peer memory: push this rank's nq x k hits + per-query status into every
// peer's batch slot, then (second launch) wait for all peers and merge per query
struct StbBatchXchgArgs {
  unsigned char *slot[STB_XCHG_MAX_WORLD];   // batch slot of every rank (peer-mapped), this batch's parity
  uint32_t world, rank, max_nq, max_k, nq, top_k;
  unsigned long long seq;
  unsigned int *ticket;
};
int stb_launch_batch_xchg(stb_ctx *ctx, const StbBatchXchgArgs &a, const stb_hit *local_hits, const uint32_t *local_status,
                          stb_hit *out_hits, uint32_t *out_status);

// opt-in to > 48 KiB dynamic shared memory (or another function attribute) once per context
enum { STB_ATTR_GEMM0 = 0, STB_ATTR_GEMM1, STB_ATTR_MERGE, STB_ATTR_IVF_PROBE, STB_ATTR_IVF_V2, STB_ATTR_FINISH2 };
#define STB_ATTR_ONCE(ctx, bit, call)                         \
  do {                                                        \
    if (!((ctx)->func_attr_mask & (1u << (bit)))) {           \
      STB_CUDA(call);                                         \
      (ctx)->func_attr_mask |= 1u << (bit);                   \
    }                                                         \
  } while (0)

// ---- embed_pool.cu --------------------------------------------------------------
int stb_launch_embed(stb_ctx *ctx, const stb_table *t, const uint64_t *offsets_dev,
                     const uint32_t *ids_dev, uint64_t n_lines, float *out_dev,
                     int *err_flag_dev);

// ---- batch_scan.cu (K2) ------------------------------------------------------------------
int stb_launch_shadow_build(stb_ctx *ctx, const float *rows_dev, uint64_t n_rows, int tile,
                            uint8_t *out, int *bad_flag_dev, uint64_t first_row = 0);
int stb_launch_batch_gemm(stb_ctx *ctx, const uint8_t *a_tiles, uint32_t m_tiles,
                          const uint8_t *b_tiles, uint32_t n_tiles, float *submax,
                          float *tilemax, float *full_out);
int stb_launch_batch_gemm_strided(stb_ctx *ctx, const uint8_t *a_tiles, uint32_t m_tiles,
                                  const uint8_t *b_tiles, uint32_t n_tiles, uint32_t tile_stride,
                                  float *submax, float *tilemax, float *full_out);
int stb_launch_batch_gemm_emit(stb_ctx *ctx, const uint8_t *a_tiles, uint32_t m_tiles,
                               const uint8_t *b_tiles, uint32_t n_tiles, uint64_t n_rows,
                               const float *thr, uint32_t *cand_cnt, uint64_t *cand_keys,
                               uint32_t cand_cap);
int stb_launch_batch_thresh(stb_ctx *ctx, const float *tilemax, uint32_t n_sample, uint32_t nq,
                            uint32_t q_pad, uint32_t top_k, float *thr);
// candidates live in per-(query, CTA) segments: keys [q_pad][n_seg][seg_cap], counts [q_pad][n_seg];
// n_seg = stb_batch_emit_grid() = the grid the emitting GEMM runs with
uint32_t stb_batch_emit_grid(const stb_ctx *ctx, uint32_t n_tiles);
int stb_launch_batch_finish2(stb_ctx *ctx, const uint64_t *cand_keys, const uint32_t *cand_cnt, uint32_t n_seg,
                             uint32_t seg_cap, uint32_t nq, uint32_t top_k, const float *rows,
                             uint64_t n_rows, uint64_t row_base, const float *queries_dev,
                             stb_hit *out_hits, uint32_t *out_status);
void stb_batch_build_params(int *shadow_is_f16, double *eps);
int stb_launch_batch_select(stb_ctx *ctx, const float *submax, uint32_t n_sub, uint32_t q_pad,
                            uint32_t n_slices, uint64_t *cand);
int stb_launch_batch_finish(stb_ctx *ctx, const uint64_t *cand, uint32_t n_slices, uint32_t n_sub,
                            uint32_t nq, uint32_t top_k, const float *rows, uint64_t n_rows,
                            uint64_t row_base, const float *queries_dev, stb_hit *out_hits,
                            uint32_t *out_status, const float *submax, uint32_t q_pad);

// ---- device helpers ---------------------------------------------------------------
#ifdef __CUDACC__
// Monotone map float -> uint32 (larger float -> larger uint), total order with
// -inf lowest; NaN never reaches it.
__device__ __forceinline__ uint32_t stb_f2ord(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float stb_ord2f(uint32_t o) {
  uint32_t b = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
  return __uint_as_float(b);
}
// Candidate key: ascending key order == (score descending, row ascending).
__device__ __forceinline__ uint64_t stb_make_key(float score, uint32_t row) {
  return ((uint64_t)(~stb_f2ord(score)) << 32) | (uint64_t)row;
}
#define STB_KEY_INVALID 0xffffffffffffffffull
__device__ __forceinline__ float stb_key_score(uint64_t k) {
  return stb_ord2f(~(uint32_t)(k >> 32));
}
__device__ __forceinline__ uint32_t stb_key_row(uint64_t k) { return (uint32_t)k; }

__device__ __forceinline__ bool stb_hit_less(double da, uint64_t ra, double db,
                                             uint64_t rb) {
  return (da < db) || (da == db && ra < rb);
}

// Ascending bitonic sort of n keys (power of two, <= R*256) held in shared memory,
// done in registers: element i = r*256 + tid lives in register k[r] of thread tid, so a
// compare-exchange at distance j is a register swap (j >= 256), a shuffle (j < 32) or a
// shared-memory exchange (32 <= j < 256; the only steps that need __syncthreads).
// Requires blockDim.x == 256.
template <int R>
__device__ __forceinline__ void stb_cta_sort_keys_t(uint64_t *keys, int n) {
  const int tid = threadIdx.x;
  uint64_t k[R];
#pragma unroll
  for (int r = 0; r < R; ++r) k[r] = (r * 256 + tid < n) ? keys[r * 256 + tid] : STB_KEY_INVALID;
  __syncthreads();
  for (int kk = 2; kk <= n; kk <<= 1) {
    for (int j = kk >> 1; j > 0; j >>= 1) {
      if (j >= 256) {
        // in-thread exchange; dr spelled out so k[] stays in registers
#pragma unroll
        for (int dr = 1; dr < R; dr <<= 1) {
          if (j == dr * 256) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
              if ((r & dr) == 0) {
                const bool up = (((r * 256 + tid) & kk) == 0);
                uint64_t x = k[r], y = k[r | dr];
                if ((x > y) == up) { k[r] = y; k[r | dr] = x; }
              }
            }
          }
        }
      } else if (j >= 32) {
#pragma unroll
        for (int r = 0; r < R; ++r) keys[r * 256 + tid] = k[r];
        __syncthreads();
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const int i = r * 256 + tid;
          const uint64_t other = keys[i ^ j];
          const bool keep_min = (((i & j) == 0) == ((i & kk) == 0));
          k[r] = keep_min ? (k[r] < other ? k[r] : other) : (k[r] > other ? k[r] : other);
        }
        __syncthreads();
      } else {
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const int i = r * 256 + tid;
          const uint64_t other = __shfl_xor_sync(0xffffffffu, k[r], j);
          const bool keep_min = (((i & j) == 0) == ((i & kk) == 0));
          k[r] = keep_min ? (k[r] < other ? k[r] : other) : (k[r] > other ? k[r] : other);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) keys[r * 256 + tid] = k[r];
  __syncthreads();
}

#endif
