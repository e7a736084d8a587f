// C ABI of libsemtools_b200.so (include/semtools_b200.h).  Host-side orchestration
// only: argument checking, HBM residency, staging copies, and the exact
// fallback ladder around the scan kernel.  No CPU implementation of any kernel
// exists in this library: without an sm_100 device every entry point fails.
#include <stdarg.h>
#include <stdlib.h>

#include <chrono>

#include <algorithm>
#include <mutex>
#include <new>
#include <unordered_set>
#include <vector>

#include "common.cuh"

static thread_local char g_err[512] = "";

void stb_set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ------------------------------------------------------------------- context ---
// Live-context registry: tables/corpora may outlive their context (garbage-collected
// host languages destroy in any order); their destructors must not touch a dead one.
static std::mutex g_ctx_mu;
static std::unordered_set<const stb_ctx *> g_ctx_live;
static bool ctx_alive(const stb_ctx *ctx) {
  std::lock_guard<std::mutex> lk(g_ctx_mu);
  return g_ctx_live.count(ctx) != 0;
}

static int ctx_use(const stb_ctx *ctx) {
  if (!ctx) { stb_set_error("null context"); return STB_ERR_ARG; }
  if (!ctx_alive(ctx)) { stb_set_error("context was destroyed"); return STB_ERR_STATE; }
  STB_CUDA(cudaSetDevice(ctx->device));
  return STB_OK;
}

template <class T>
static int dev_reserve(T **p, size_t *cap, size_t need, size_t floor_cap = 0) {
  if (need <= *cap && *p) return STB_OK;
  size_t ncap = std::max(std::max(need, floor_cap), *cap + *cap / 2);
  T *np = nullptr;
  cudaError_t e = cudaMalloc((void **)&np, ncap * sizeof(T));
  if (e != cudaSuccess) {
    cudaGetLastError();
    stb_set_error("cudaMalloc(%zu bytes) failed: %s", ncap * sizeof(T), cudaGetErrorString(e));
    return STB_ERR_NOMEM;
  }
  if (*p) cudaFree(*p);
  *p = np;
  *cap = ncap;
  return STB_OK;
}

extern "C" {

int stb_version(void) { return 100; }
const char *stb_last_error(void) { return g_err; }

int stb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int stb_ctx_create(int device, void *cuda_stream, stb_ctx **out) {
  if (!out) { stb_set_error("out is null"); return STB_ERR_ARG; }
  *out = nullptr;
  int n = stb_device_count();
  if (n <= 0) { stb_set_error("no CUDA device visible (this library has no CPU path)"); return STB_ERR_CUDA; }
  if (device < 0 || device >= n) { stb_set_error("device %d out of range (0..%d)", device, n - 1); return STB_ERR_ARG; }
  STB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  STB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    stb_set_error("device %d is sm_%d%d; libsemtools_b200 ships sm_100a code only", device, prop.major, prop.minor);
    return STB_ERR_CUDA;
  }
  stb_ctx *c = new (std::nothrow) stb_ctx();
  if (!c) { stb_set_error("out of host memory"); return STB_ERR_NOMEM; }
  memset(c, 0, sizeof(*c));
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if (cuda_stream) { c->stream = (cudaStream_t)cuda_stream; c->own_stream = false; }
  else {
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { stb_set_error("cudaStreamCreate: %s", cudaGetErrorString(e)); delete c; return STB_ERR_CUDA; }
    c->own_stream = true;
  }
  int rc = STB_OK;
  const size_t max_grid = (size_t)c->sm_count * 8;
  if ((rc = dev_reserve(&c->block_keys, &c->block_keys_cap, 2 * max_grid * 129 + STB_SORT_CAP)) != STB_OK) goto fail;
  if ((rc = dev_reserve(&c->counters, &c->counters_cap, max_grid + 64)) != STB_OK) goto fail;
  {
    size_t one = 0;
    if ((rc = dev_reserve(&c->q_dev, &one, STB_D)) != STB_OK) goto fail;
    one = 0;
    if ((rc = dev_reserve(&c->status_dev, &one, 8)) != STB_OK) goto fail;
    one = 0;
    if ((rc = dev_reserve(&c->collect_count, &one, 2)) != STB_OK) goto fail;
    one = 0;
    if ((rc = dev_reserve(&c->err_flag, &one, 1)) != STB_OK) goto fail;
    one = 0;
    if ((rc = dev_reserve(&c->dbg_dev, &one, 8)) != STB_OK) goto fail;
    one = 0;
    if ((rc = dev_reserve(&c->hist_dev, &one, 4096)) != STB_OK) goto fail;
    one = 0;
    if ((rc = dev_reserve(&c->tickets, &one, 2 * STB_TICKET_SLOTS + 1)) != STB_OK) goto fail;
    c->scan_start = c->tickets + STB_TICKET_SLOTS;
    c->scan_front = c->scan_start + STB_TICKET_SLOTS;
  }
  if ((rc = dev_reserve(&c->hits_dev, &c->hits_cap, 1024)) != STB_OK) goto fail;
  if (cudaMemset(c->counters, 0, c->counters_cap * sizeof(unsigned int)) != cudaSuccess ||
      cudaMemset(c->tickets, 0, (2 * STB_TICKET_SLOTS + 1) * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMemset(c->err_flag, 0, sizeof(int)) != cudaSuccess ||
      cudaMallocHost((void **)&c->q_pin, STB_D * sizeof(float)) != cudaSuccess ||
      cudaMallocHost((void **)&c->status_pin, 8 * sizeof(uint32_t)) != cudaSuccess ||
      cudaMallocHost((void **)&c->hits_pin, 1024 * sizeof(stb_hit)) != cudaSuccess) {
    stb_set_error("context staging allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    rc = STB_ERR_NOMEM;
    goto fail;
  }
  c->hits_pin_cap = 1024;
  { std::lock_guard<std::mutex> lk(g_ctx_mu); g_ctx_live.insert(c); }
  *out = c;
  return STB_OK;
fail:
  stb_ctx_destroy(c);
  return rc;
}

int stb_ctx_destroy(stb_ctx *c) {
  if (!c) return STB_OK;
  { std::lock_guard<std::mutex> lk(g_ctx_mu); g_ctx_live.erase(c); }
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  cudaFree(c->block_keys); cudaFree(c->counters); cudaFree(c->q_dev); cudaFree(c->hits_dev);
  cudaFree(c->status_dev); cudaFree(c->collect_rows); cudaFree(c->collect_count);
  cudaFree(c->collect_hits); cudaFree(c->ranges_dev); cudaFree(c->err_flag);
  cudaFree(c->tickets);
  cudaFree(c->dbg_dev); cudaFree(c->hist_dev); cudaFree(c->bq_tiles); cudaFree(c->b_submax); cudaFree(c->b_tilemax); cudaFree(c->b_cand);
  cudaFree(c->b_thr); cudaFree(c->b_cnt); cudaFree(c->b_keys);
  cudaFree(c->bq_dev); cudaFree(c->bh_dev); cudaFree(c->bs_dev); cudaFree(c->embed_off_dev); cudaFree(c->embed_ids_dev); cudaFree(c->embed_out_dev);
  if (c->q_pin) cudaFreeHost(c->q_pin);
  if (c->hits_pin) cudaFreeHost(c->hits_pin);
  if (c->status_pin) cudaFreeHost(c->status_pin);
  if (c->many_q_pin) cudaFreeHost(c->many_q_pin);
  if (c->many_status_pin) cudaFreeHost(c->many_status_pin);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  cudaGetLastError();
  delete c;
  return STB_OK;
}

int stb_ctx_sync(stb_ctx *ctx) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  return STB_OK;
}

void *stb_ctx_stream(stb_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

// Tuning aid (STB_TAIL_TIMING builds): reset=1 arms the timestamps, reset=0 reads them.
int stb_debug_timestamps(stb_ctx *ctx, int reset, uint64_t out[8]) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (reset) {
    unsigned long long init[8] = {~0ull, 0, 0, 0, 0, 0, 0, 0};
    STB_CUDA(cudaMemcpyAsync(ctx->dbg_dev, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
    STB_CUDA(cudaStreamSynchronize(ctx->stream));
  } else {
    STB_CUDA(cudaMemcpyAsync(out, ctx->dbg_dev, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    STB_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return STB_OK;
}

// K1's tile tickets: every top-k launch must advance the device counter by exactly what the host
// booked for it (n_tickets + total_warps); a mismatch would make later launches skip or repeat
// tiles.  Synchronises; returns STB_ERR_STATE on a mismatch.
int stb_debug_ticket_check(stb_ctx *ctx, uint64_t *device_value, uint64_t *host_value) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  unsigned long long v[STB_TICKET_SLOTS];
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  STB_CUDA(cudaMemcpy(v, ctx->tickets, sizeof(v), cudaMemcpyDeviceToHost));
  unsigned long long dsum = 0, hsum = 0;
  int bad = -1;
  for (int i = 0; i < STB_TICKET_SLOTS; ++i) { dsum += v[i]; hsum += ctx->ticket_next[i]; if (v[i] != ctx->ticket_next[i] && bad < 0) bad = i; }
  if (device_value) *device_value = dsum;          // sums over the counter ring
  if (host_value) *host_value = hsum;
  if (bad >= 0) { stb_set_error("ticket counter %d is %llu, host expects %llu", bad, v[bad], ctx->ticket_next[bad]); return STB_ERR_STATE; }
  return STB_OK;
}

int stb_debug_scan_front(stb_ctx *ctx, int set, uint64_t *value) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!value) { stb_set_error("scan_front: null value"); return STB_ERR_ARG; }
  unsigned long long v = *value;
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  if (set) STB_CUDA(cudaMemcpy(ctx->scan_front, &v, sizeof(v), cudaMemcpyHostToDevice));
  else STB_CUDA(cudaMemcpy(&v, ctx->scan_front, sizeof(v), cudaMemcpyDeviceToHost));
  *value = v;
  return STB_OK;
}

int stb_ctx_counters(const stb_ctx *ctx, uint64_t *kernel_launches, uint64_t *fallback_searches) {
  if (!ctx) { stb_set_error("null context"); return STB_ERR_ARG; }
  if (kernel_launches) *kernel_launches = ctx->kernel_launches;
  if (fallback_searches) *fallback_searches = ctx->fallback_searches;
  return STB_OK;
}

// --------------------------------------------------------------------- table ---
int stb_table_load(stb_ctx *ctx, const float *E, uint64_t V, uint32_t D, const float *weights,
                   uint64_t n_weights, const uint32_t *mapping, uint64_t n_mapping, int normalize,
                   stb_table **out) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!out || !E || V == 0) { stb_set_error("table_load: null/empty table"); return STB_ERR_ARG; }
  if (D != STB_D) { stb_set_error("table_load: D=%u, only %u supported", D, STB_D); return STB_ERR_ARG; }
  if (V > 0xffffffffull) { stb_set_error("table_load: V exceeds 2^32 rows"); return STB_ERR_ARG; }
  stb_table *t = new (std::nothrow) stb_table();
  if (!t) { stb_set_error("out of host memory"); return STB_ERR_NOMEM; }
  memset(t, 0, sizeof(*t));
  t->ctx = ctx; t->V = V; t->normalize = normalize ? 1 : 0;
  t->n_weights = weights ? n_weights : 0;
  t->n_mapping = mapping ? n_mapping : 0;
  cudaError_t e = cudaMalloc((void **)&t->E, V * STB_D * sizeof(float));
  if (e == cudaSuccess && t->n_weights) e = cudaMalloc((void **)&t->weights, t->n_weights * sizeof(float));
  if (e == cudaSuccess && t->n_mapping) e = cudaMalloc((void **)&t->mapping, t->n_mapping * sizeof(uint32_t));
  if (e != cudaSuccess) {
    cudaGetLastError();
    stb_set_error("table_load: device allocation failed: %s", cudaGetErrorString(e));
    stb_table_destroy(t);
    return STB_ERR_NOMEM;
  }
  e = cudaMemcpyAsync(t->E, E, V * STB_D * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess && t->n_weights)
    e = cudaMemcpyAsync(t->weights, weights, t->n_weights * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess && t->n_mapping)
    e = cudaMemcpyAsync(t->mapping, mapping, t->n_mapping * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    stb_set_error("table_load: upload failed: %s", cudaGetErrorString(e));
    stb_table_destroy(t);
    return STB_ERR_CUDA;
  }
  *out = t;
  return STB_OK;
}

int stb_table_destroy(stb_table *t) {
  if (!t) return STB_OK;
  if (t->ctx && ctx_alive(t->ctx)) { cudaSetDevice(t->ctx->device); cudaStreamSynchronize(t->ctx->stream); }
  else cudaDeviceSynchronize();
  cudaFree(t->E); cudaFree(t->weights); cudaFree(t->mapping);
  cudaGetLastError();
  delete t;
  return STB_OK;
}

// -------------------------------------------------------------------- corpus ---
static int corpus_reserve(stb_corpus *c, uint64_t need) {
  if (need <= c->capacity && c->rows) return STB_OK;
  if (need > 0xfffffffeull) { stb_set_error("corpus shard exceeds 2^32-2 rows; shard it"); return STB_ERR_ARG; }
  uint64_t ncap = std::max<uint64_t>(std::max<uint64_t>(need, 1024), c->capacity + c->capacity / 2);
  float *np = nullptr;
  cudaError_t e = cudaMalloc((void **)&np, ncap * STB_D * sizeof(float));
  if (e != cudaSuccess) {
    cudaGetLastError();
    stb_set_error("corpus: cudaMalloc(%llu rows) failed: %s", (unsigned long long)ncap, cudaGetErrorString(e));
    return STB_ERR_NOMEM;
  }
  if (c->rows && c->n) {
    e = cudaMemcpyAsync(np, c->rows, c->n * STB_D * sizeof(float), cudaMemcpyDeviceToDevice, c->ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->ctx->stream);
    if (e != cudaSuccess) { cudaFree(np); stb_set_error("corpus grow copy: %s", cudaGetErrorString(e)); return STB_ERR_CUDA; }
  }
  if (c->rows) cudaFree(c->rows);
  c->rows = np;
  c->capacity = ncap;
  return STB_OK;
}

int stb_corpus_create(stb_ctx *ctx, uint32_t D, uint64_t capacity_rows, uint64_t row_base, stb_corpus **out) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!out) { stb_set_error("out is null"); return STB_ERR_ARG; }
  if (D != STB_D) { stb_set_error("corpus_create: D=%u, only %u supported", D, STB_D); return STB_ERR_ARG; }
  stb_corpus *c = new (std::nothrow) stb_corpus();
  if (!c) { stb_set_error("out of host memory"); return STB_ERR_NOMEM; }
  memset(c, 0, sizeof(*c));
  c->ctx = ctx; c->row_base = row_base;
  rc = corpus_reserve(c, std::max<uint64_t>(capacity_rows, 1));
  if (rc) { delete c; return rc; }
  *out = c;
  return STB_OK;
}

int stb_corpus_destroy(stb_corpus *c) {
  if (!c) return STB_OK;
  if (c->ctx && ctx_alive(c->ctx)) { cudaSetDevice(c->ctx->device); cudaStreamSynchronize(c->ctx->stream); }
  else cudaDeviceSynchronize();
  cudaFree(c->shadow);
  cudaFree(c->q8);
  cudaFree(c->q8_scale);
  cudaFree(c->q4);
  cudaFree(c->q4_sr);
  cudaFree(c->rows);
  cudaGetLastError();
  delete c;
  return STB_OK;
}

// The reduced-width copies (K2 shadow, K1 tiers) cover a PREFIX of the rows: an append leaves the
// prefix valid and the next query / prepare only converts the new rows (q8_rows / shadow_rows < n);
// anything else (clear) drops them.
static void corpus_changed(stb_corpus *c, bool appended_only = false) {
  if (!appended_only) { c->shadow_rows = 0; c->q8_rows = 0; }
  c->searches_since_change = 0;
  memset(c->tier_tries, 0, sizeof(c->tier_tries));
  memset(c->tier_proven, 0, sizeof(c->tier_proven));
  c->coarse_tries = c->coarse_proven = 0;
}

static int corpus_append_impl(stb_corpus *c, const float *rows, uint64_t n, cudaMemcpyKind kind) {
  if (!c) { stb_set_error("null corpus"); return STB_ERR_ARG; }
  int rc = ctx_use(c->ctx);
  if (rc) return rc;
  if (n == 0) return STB_OK;
  if (!rows) { stb_set_error("corpus_append: rows is null"); return STB_ERR_ARG; }
  if ((rc = corpus_reserve(c, c->n + n)) != STB_OK) return rc;
  STB_CUDA(cudaMemcpyAsync(c->rows + c->n * STB_D, rows, n * STB_D * sizeof(float), kind, c->ctx->stream));
  STB_CUDA(cudaStreamSynchronize(c->ctx->stream));
  c->n += n;
  corpus_changed(c, true);
  return STB_OK;
}

int stb_corpus_append(stb_corpus *c, const float *rows, uint64_t n) {
  return corpus_append_impl(c, rows, n, cudaMemcpyHostToDevice);
}
int stb_corpus_append_dev(stb_corpus *c, const float *rows_dev, uint64_t n) {
  return corpus_append_impl(c, rows_dev, n, cudaMemcpyDeviceToDevice);
}
int stb_corpus_clear(stb_corpus *c) {
  if (!c) { stb_set_error("null corpus"); return STB_ERR_ARG; }
  if (!ctx_alive(c->ctx)) { stb_set_error("context was destroyed"); return STB_ERR_STATE; }
  c->n = 0;
  corpus_changed(c);
  return STB_OK;
}
int stb_corpus_rows(const stb_corpus *c, uint64_t *n) {
  if (!c || !n) { stb_set_error("null argument"); return STB_ERR_ARG; }
  *n = c->n;
  return STB_OK;
}
int stb_corpus_data_dev(const stb_corpus *c, float **rows_dev) {
  if (!c || !rows_dev) { stb_set_error("null argument"); return STB_ERR_ARG; }
  *rows_dev = c->rows;
  return STB_OK;
}
int stb_corpus_read(const stb_corpus *c, uint64_t first, uint64_t n, float *rows) {
  if (!c || (!rows && n)) { stb_set_error("null argument"); return STB_ERR_ARG; }
  int rc = ctx_use(c->ctx);
  if (rc) return rc;
  if (first > c->n || n > c->n - first) { stb_set_error("corpus_read: rows [%llu,+%llu) outside corpus of %llu",
      (unsigned long long)first, (unsigned long long)n, (unsigned long long)c->n); return STB_ERR_RANGE; }
  if (n == 0) return STB_OK;
  STB_CUDA(cudaMemcpyAsync(rows, c->rows + first * STB_D, n * STB_D * sizeof(float), cudaMemcpyDeviceToHost, c->ctx->stream));
  STB_CUDA(cudaStreamSynchronize(c->ctx->stream));
  return STB_OK;
}

// ---------------------------------------------------------------------- embed ---
int stb_embed(stb_ctx *ctx, const stb_table *table, const uint64_t *offsets, const uint32_t *ids,
              uint64_t n_lines, float *out, stb_corpus *append_to) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!table) { stb_set_error("embed: null table"); return STB_ERR_ARG; }
  if (table->ctx != ctx || (append_to && append_to->ctx != ctx)) { stb_set_error("embed: handles belong to another context"); return STB_ERR_ARG; }
  if (n_lines == 0) return STB_OK;
  if (!offsets) { stb_set_error("embed: offsets is null"); return STB_ERR_ARG; }
  if (offsets[0] != 0) { stb_set_error("embed: offsets[0] must be 0"); return STB_ERR_ARG; }
  const uint64_t total = offsets[n_lines];
  for (uint64_t i = 0; i < n_lines; ++i)
    if (offsets[i + 1] < offsets[i]) { stb_set_error("embed: offsets not monotone at line %llu", (unsigned long long)i); return STB_ERR_ARG; }
  if (total && !ids) { stb_set_error("embed: ids is null"); return STB_ERR_ARG; }
  if ((rc = dev_reserve(&ctx->embed_off_dev, &ctx->embed_off_cap, n_lines + 1, 4096)) != STB_OK) return rc;
  if ((rc = dev_reserve(&ctx->embed_ids_dev, &ctx->embed_ids_cap, std::max<uint64_t>(total, 1), 65536)) != STB_OK) return rc;
  float *dst = nullptr;
  if (append_to) {
    if ((rc = corpus_reserve(append_to, append_to->n + n_lines)) != STB_OK) return rc;
    dst = append_to->rows + append_to->n * STB_D;
  } else {
    if ((rc = dev_reserve(&ctx->embed_out_dev, &ctx->embed_out_cap, n_lines * STB_D, 4096 * STB_D)) != STB_OK) return rc;
    dst = ctx->embed_out_dev;
  }
  STB_CUDA(cudaMemcpyAsync(ctx->embed_off_dev, offsets, (n_lines + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
  if (total) STB_CUDA(cudaMemcpyAsync(ctx->embed_ids_dev, ids, total * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  STB_CUDA(cudaMemsetAsync(ctx->err_flag, 0, sizeof(int), ctx->stream));
  if ((rc = stb_launch_embed(ctx, table, ctx->embed_off_dev, ctx->embed_ids_dev, n_lines, dst, ctx->err_flag)) != STB_OK) return rc;
  int flag = 0;
  STB_CUDA(cudaMemcpyAsync(&flag, ctx->err_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  if (out) STB_CUDA(cudaMemcpyAsync(out, dst, n_lines * STB_D * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  if (flag) { stb_set_error("embed: a token id maps outside the %llu-row table", (unsigned long long)table->V); return STB_ERR_RANGE; }
  if (append_to) { append_to->n += n_lines; corpus_changed(append_to, true); }
  return STB_OK;
}

int stb_embed_dev(stb_ctx *ctx, const stb_table *table, const uint64_t *offsets_dev,
                  const uint32_t *ids_dev, uint64_t n_lines, float *out_dev) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!table || table->ctx != ctx) { stb_set_error("embed_dev: bad table"); return STB_ERR_ARG; }
  if (n_lines == 0) return STB_OK;
  if (!offsets_dev || !ids_dev || !out_dev) { stb_set_error("embed_dev: null device pointer"); return STB_ERR_ARG; }
  return stb_launch_embed(ctx, table, offsets_dev, ids_dev, n_lines, out_dev, ctx->err_flag);
}

int stb_embed_status(stb_ctx *ctx) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  int flag = 0;
  STB_CUDA(cudaMemcpyAsync(&flag, ctx->err_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  STB_CUDA(cudaMemsetAsync(ctx->err_flag, 0, sizeof(int), ctx->stream));
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  if (flag) { stb_set_error("embed: a token id maps outside the table"); return STB_ERR_RANGE; }
  return STB_OK;
}

// --------------------------------------------------------------------- search ---
static int corpus_ensure_shadow(stb_ctx *ctx, stb_corpus *c);   // defined with the K2 entry points
static int corpus_ensure_q8(stb_ctx *ctx, stb_corpus *c);

// STB_SCAN_TIER = f32 | h16 | q8: the narrowest candidate tier K1 may use (default q8).  Read per
// call so one process can compare tiers; results are identical whatever the value.
static int stb_env_max_tier() {
  const char *e = getenv("STB_SCAN_TIER");
  if (!e || !e[0]) return STB_TIER_Q8;
  if (e[0] == 'f') return STB_TIER_F32;
  if (e[0] == 'h') return STB_TIER_H16;
  return STB_TIER_Q8;
}
// STB_Q8_COARSE=0: no 4-bit coarse stage in front of the q8 scan.  Read per call like STB_SCAN_TIER, so
// one process can compare the two; results are identical either way.
static bool stb_env_coarse() {
  const char *e = getenv("STB_Q8_COARSE");
  return !(e && e[0] == '0');
}
// a reduced-width stage that proves fewer than half of its results on this corpus is skipped
static bool stage_keeps_failing(uint32_t tries, uint32_t proven) { return tries >= 8 && 2 * proven < tries; }
static bool coarse_usable(const stb_corpus *c) {
  return stb_env_coarse() && c->q4 && !stage_keeps_failing(c->coarse_tries, c->coarse_proven);
}
static bool stb_env_direct_out() {
  const char *e = getenv("STB_DIRECT_OUT");
  return !(e && e[0] == '0');
}
static int best_built_tier(const stb_corpus *c, uint32_t top_k) {
  const int max_tier = stb_env_max_tier();
  if (max_tier >= STB_TIER_Q8 && top_k <= STB_Q8_MAX_K && c->q8 && c->q8_rows == c->n && !c->q8_bad)
    return coarse_usable(c) ? STB_TIER_Q4Q8 : STB_TIER_Q8;
  if (max_tier >= STB_TIER_H16 && c->shadow && c->shadow_rows == c->n && !c->shadow_bad) return STB_TIER_H16;
  return STB_TIER_F32;
}

static int ensure_hits_pin(stb_ctx *ctx, size_t need) {
  if (need <= ctx->hits_pin_cap) return STB_OK;
  stb_hit *np = nullptr;
  size_t ncap = std::max(need, ctx->hits_pin_cap * 2);
  if (cudaMallocHost((void **)&np, ncap * sizeof(stb_hit)) != cudaSuccess) {
    cudaGetLastError();
    stb_set_error("pinned staging allocation failed");
    return STB_ERR_NOMEM;
  }
  cudaFreeHost(ctx->hits_pin);
  ctx->hits_pin = np;
  ctx->hits_pin_cap = ncap;
  return STB_OK;
}

// Exact path for any input: collect rows whose approximate cosine >= cos_floor,
// score them canonically, keep distance < limit, sort by (distance,row).
// On return ctx->collect_hits holds the sorted hits and *n_pass their count.
static int collect_exact_sorted(stb_ctx *ctx, const stb_corpus *c, float cos_floor, double limit,
                                const uint64_t *ranges_dev, uint32_t n_ranges, uint64_t n_virtual,
                                uint64_t *n_pass, int tier = STB_TIER_F32) {
  int rc;
  unsigned long long count = 0;
  if ((rc = dev_reserve(&ctx->collect_rows, &ctx->collect_cap, 1, 1u << 20)) != STB_OK) return rc;
  for (int attempt = 0; attempt < 3; ++attempt) {
    if ((rc = stb_launch_scan_collect(ctx, c, tier, ctx->q_dev, cos_floor, ranges_dev, n_ranges, n_virtual)) != STB_OK) return rc;
    STB_CUDA(cudaMemcpyAsync(&count, ctx->collect_count, sizeof(count), cudaMemcpyDeviceToHost, ctx->stream));
    STB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (count <= ctx->collect_cap) break;
    if ((rc = dev_reserve(&ctx->collect_rows, &ctx->collect_cap, (size_t)count)) != STB_OK) return rc;
  }
  if (count > ctx->collect_cap) { stb_set_error("collect buffer could not be sized"); return STB_ERR_STATE; }
  uint64_t m = count, m_padded = 1024;
  while (m_padded < m) m_padded <<= 1;
  if ((rc = dev_reserve(&ctx->collect_hits, &ctx->collect_hits_cap, (size_t)m_padded)) != STB_OK) return rc;
  if ((rc = stb_launch_exact(ctx, c->rows, c->row_base, ctx->q_dev, ctx->collect_rows, m, limit,
                             ctx->collect_hits, m_padded, ctx->collect_count + 1)) != STB_OK) return rc;
  if ((rc = stb_launch_sort_hits(ctx, ctx->collect_hits, m_padded)) != STB_OK) return rc;
  unsigned long long pass = 0;
  STB_CUDA(cudaMemcpyAsync(&pass, ctx->collect_count + 1, sizeof(pass), cudaMemcpyDeviceToHost, ctx->stream));
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  *n_pass = pass;
  return STB_OK;
}

int stb_search(stb_ctx *ctx, const stb_corpus *corpus, const float *q, uint32_t top_k, int has_max,
               double max_distance, int mode, const uint64_t *row_ranges, uint32_t n_ranges,
               stb_hit *out_hits, uint64_t cap, uint64_t *out_n) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!corpus || !q || !out_n) { stb_set_error("search: null argument"); return STB_ERR_ARG; }
  if (corpus->ctx != ctx) { stb_set_error("search: corpus belongs to another context"); return STB_ERR_ARG; }
  if (mode != STB_MODE_SEARCH_DOCUMENTS && mode != STB_MODE_STORE_QUERY) { stb_set_error("search: bad mode %d", mode); return STB_ERR_ARG; }
  if (n_ranges && !row_ranges) { stb_set_error("search: row_ranges is null"); return STB_ERR_ARG; }
  if (cap && !out_hits) { stb_set_error("search: out_hits is null"); return STB_ERR_ARG; }
  *out_n = 0;
  const bool threshold_all = (mode == STB_MODE_SEARCH_DOCUMENTS) && has_max;   // src/search/mod.rs:115-116
  if (!threshold_all && top_k == 0) return STB_OK;                             // take(0) / store.rs:489-491
  if (mode == STB_MODE_STORE_QUERY && row_ranges && n_ranges == 0) return STB_OK;  // empty subset, store.rs:489
  if (corpus->n == 0) return STB_OK;

  // ---- row ranges: global -> local, clipped to this shard ----------------------
  const uint64_t *ranges_dev = nullptr;
  uint32_t n_loc = 0;
  uint64_t n_virtual = corpus->n;
  if (row_ranges) {
    std::vector<uint64_t> vstart, rbegin;
    vstart.reserve(n_ranges + 1); rbegin.reserve(n_ranges);
    uint64_t acc = 0, prev_end = 0;
    const uint64_t lo = corpus->row_base, hi = corpus->row_base + corpus->n;
    for (uint32_t i = 0; i < n_ranges; ++i) {
      uint64_t b = row_ranges[2 * i], e = row_ranges[2 * i + 1];
      if (e < b || (i > 0 && b < prev_end)) { stb_set_error("search: row_ranges must be ascending, disjoint, half-open"); return STB_ERR_RANGE; }
      prev_end = e;
      b = std::max(b, lo); e = std::min(e, hi);
      if (b >= e) continue;
      vstart.push_back(acc); rbegin.push_back(b - lo);
      acc += e - b;
    }
    if (acc == 0) return STB_OK;
    vstart.push_back(acc);
    n_loc = (uint32_t)rbegin.size();
    n_virtual = acc;
    std::vector<uint64_t> packed(vstart);
    packed.insert(packed.end(), rbegin.begin(), rbegin.end());
    if ((rc = dev_reserve(&ctx->ranges_dev, &ctx->ranges_cap, packed.size(), 4096)) != STB_OK) return rc;
    STB_CUDA(cudaMemcpyAsync(ctx->ranges_dev, packed.data(), packed.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    STB_CUDA(cudaStreamSynchronize(ctx->stream));   // `packed` dies at scope end
    ranges_dev = ctx->ranges_dev;
  }

  memcpy(ctx->q_pin, q, STB_D * sizeof(float));
  STB_CUDA(cudaMemcpyAsync(ctx->q_dev, ctx->q_pin, STB_D * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));

  uint64_t total = 0;
  const stb_hit *src_dev = nullptr;   // sorted device hits to copy out (collect path)
  if (!threshold_all && top_k <= stb_scan_topk_max_k()) {
    // ---- fast path: one kernel, k*16+16 bytes back -----------------------------
    // The kernel's last CTA stores the k hits + status straight into the pinned host buffers
    // (UVA: cudaMallocHost memory is device-accessible), which takes the two D2H copies off the
    // stream; kernel completion makes the stores visible to the host.  STB_DIRECT_OUT=0 restores
    // the device buffers + two cudaMemcpyAsync.
    const bool direct = stb_env_direct_out();
    auto run_fast = [&](int tier) -> int {
      int r;
      if (direct) {
        if ((r = stb_launch_scan_topk(ctx, corpus, tier, ctx->q_dev, top_k, ranges_dev, n_loc, n_virtual, ctx->hits_pin,
                                      ctx->status_pin)) != STB_OK) return r;
      } else {
        if ((r = stb_launch_scan_topk(ctx, corpus, tier, ctx->q_dev, top_k, ranges_dev, n_loc, n_virtual, ctx->hits_dev,
                                      ctx->status_dev)) != STB_OK) return r;
        STB_CUDA(cudaMemcpyAsync(ctx->status_pin, ctx->status_dev, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        STB_CUDA(cudaMemcpyAsync(ctx->hits_pin, ctx->hits_dev, top_k * sizeof(stb_hit), cudaMemcpyDeviceToHost, ctx->stream));
      }
      STB_CUDA(cudaStreamSynchronize(ctx->stream));
      return STB_OK;
    };
    // Tier ladder: coarse + q8 (136 B/row + a few q8 rows) -> q8 (260 B/row) -> h16 (512 B/row) -> f32 (1 KiB/row).  Every tier ends in the
    // same exact f64 re-rank and proves its own result; one that cannot is retried one tier up, so
    // the answer is the oracle's whichever tier produced it.  Reduced-width copies are used when
    // they exist (stb_corpus_prepare) and built lazily from the second query on an unchanged
    // corpus of >= 32768 rows (a one-shot CLI query must not pay a full extra pass to save half
    // of one); a tier that keeps failing its proofs on this corpus is dropped.
    stb_corpus *cm = const_cast<stb_corpus *>(corpus);
    const int max_tier = stb_env_max_tier();
    const bool lazy_ok = cm->searches_since_change >= 1 && cm->n >= 32768;
    cm->searches_since_change++;
    bool proven = false;
    for (int tier = STB_TIER_Q8; tier >= STB_TIER_H16 && !proven; --tier) {
      if (tier > max_tier) continue;
      if (tier == STB_TIER_Q8 && top_k > STB_Q8_MAX_K) continue;
      if (stage_keeps_failing(cm->tier_tries[tier], cm->tier_proven[tier])) continue;
      const bool built = (tier == STB_TIER_Q8) ? (cm->q8 && cm->q8_rows == cm->n) : (cm->shadow && cm->shadow_rows == cm->n);
      // a copy that covers a prefix (rows were appended since) is extended right away: converting the
      // new rows costs far less than scanning everything at 1 KiB/row
      const bool extendable = (tier == STB_TIER_Q8) ? (cm->q8 && cm->q8_rows > 0 && !cm->q8_bad) : (cm->shadow && cm->shadow_rows > 0 && !cm->shadow_bad);
      if (!built && !lazy_ok && !extendable) continue;
      const int src = (tier == STB_TIER_Q8) ? corpus_ensure_q8(ctx, cm) : corpus_ensure_shadow(ctx, cm);
      if (src == STB_ERR_STATE) continue;                  // rows that cannot be normalised in fp32
      if (src != STB_OK) return src;
      if (tier == STB_TIER_Q8 && coarse_usable(cm)) {
        // the coarse stage is part of the q8 tier: a proven result counts there, an unproven one is
        // retried by the single-stage q8 scan and counts only against the coarse stage
        if ((rc = run_fast(STB_TIER_Q4Q8)) != STB_OK) return rc;
        proven = ctx->status_pin[1] != 0;
        cm->coarse_tries++;
        if (proven) { cm->coarse_proven++; cm->tier_tries[tier]++; cm->tier_proven[tier]++; continue; }
      }
      if ((rc = run_fast(tier)) != STB_OK) return rc;
      proven = ctx->status_pin[1] != 0;
      cm->tier_tries[tier]++;
      if (proven) cm->tier_proven[tier]++;
    }
    if (!proven) {
      if ((rc = run_fast(STB_TIER_F32)) != STB_OK) return rc;
      cm->tier_tries[STB_TIER_F32]++;
      if (ctx->status_pin[1]) cm->tier_proven[STB_TIER_F32]++;
    }
    const uint32_t n_hits = ctx->status_pin[0];
    if (ctx->status_pin[1]) {
      uint64_t n = 0;
      for (uint32_t i = 0; i < n_hits; ++i) {
        if (has_max && !(ctx->hits_pin[i].distance < max_distance)) break;   // strict, sorted ascending
        if (n < cap) out_hits[n] = ctx->hits_pin[i];
        ++n;
      }
      *out_n = n;
      if (n > cap) { stb_set_error("search: %llu hits, capacity %llu", (unsigned long long)n, (unsigned long long)cap); return STB_ERR_CAPACITY; }
      return STB_OK;
    }
    // ---- candidate margin not provable: exact collect pass --------------------
    ctx->fallback_searches++;
    float floor_cos = -INFINITY;
    if (n_hits == top_k) floor_cos = (float)(1.0 - ctx->hits_pin[top_k - 1].distance - 2.0 * STB_SCORE_EPS);
    uint64_t n_pass = 0;
    if ((rc = collect_exact_sorted(ctx, corpus, floor_cos, has_max ? std::min(max_distance, 100.0) : 100.0,
                                   ranges_dev, n_loc, n_virtual, &n_pass)) != STB_OK) return rc;
    total = std::min<uint64_t>(n_pass, top_k);
    src_dev = ctx->collect_hits;
  } else {
    // ---- threshold mode / top_k beyond the register lists: collect -> exact -> sort --------------
    // When the int8 copy exists (or may be built: same lazy rule as the top-k tiers) the streaming
    // passes read it instead of the f32 rows: its scores are upper bounds u >= c - 2e-5 of the exact
    // cosine, so "u >= floor" collects a superset of "c >= floor" at a quarter of the bytes.
    stb_corpus *cm = const_cast<stb_corpus *>(corpus);
    const bool lazy_ok = cm->searches_since_change >= 1 && cm->n >= 32768;
    cm->searches_since_change++;
    bool use_q8 = stb_env_max_tier() >= STB_TIER_Q8;
    if (use_q8) {
      const bool built = cm->q8 && cm->q8_rows == cm->n;
      const bool extendable = cm->q8 && cm->q8_rows > 0 && !cm->q8_bad;
      if (!built && !lazy_ok && !extendable) use_q8 = false;
      else {
        const int src = corpus_ensure_q8(ctx, cm);
        if (src == STB_ERR_STATE) use_q8 = false;
        else if (src != STB_OK) return src;
      }
    }
    float floor_cos = -INFINITY;
    double limit = 100.0;
    uint64_t n_pass = 0;
    bool done = false;
    if (threshold_all) {
      limit = max_distance;
      floor_cos = (float)(1.0 - max_distance - (use_q8 ? 2.0 * STB_Q8_SCAN_EPS : STB_SCORE_EPS));
      if (!(max_distance == max_distance)) floor_cos = INFINITY;   // NaN threshold: nothing passes
      if ((rc = collect_exact_sorted(ctx, corpus, floor_cos, limit, ranges_dev, n_loc, n_virtual, &n_pass,
                                     use_q8 ? STB_TIER_Q8 : STB_TIER_F32)) != STB_OK) return rc;
      done = true;
    } else {
      if (has_max) {
        limit = std::min(max_distance, 100.0);
        if (!(max_distance == max_distance)) limit = -1.0;
      }
      // top_k beyond the register lists: histogram pass to find the score bin of the k-th
      // best, then collect only rows at or above that bin (instead of the whole shard)
      std::vector<unsigned int> hist(4096);
      auto kth_bin = [&](int tier, int *bin) -> int {
        int r;
        if ((r = stb_launch_scan_hist(ctx, corpus, tier, ctx->q_dev, ranges_dev, n_loc, n_virtual, ctx->hist_dev)) != STB_OK) return r;
        STB_CUDA(cudaMemcpyAsync(hist.data(), ctx->hist_dev, 4096 * sizeof(unsigned int), cudaMemcpyDeviceToHost, ctx->stream));
        STB_CUDA(cudaStreamSynchronize(ctx->stream));
        uint64_t cum = 0;
        int b = 0;
        for (; b < 4096; ++b) { cum += hist[b]; if (cum >= top_k) break; }
        *bin = b;
        return STB_OK;
      };
      if (use_q8) {
        // q8: the histogram is over UPPER BOUNDS, which sit up to ~0.02-0.04 above the exact cosines, so the
        // floor is put 0.04 below the k-th best bound and the result is PROVEN afterwards: every row that
        // was not collected has c < floor + 2e-5; if the k-th exact distance found is below
        // 1 - floor - 2e-5 nothing outside can enter or tie.  Otherwise the f32 passes below answer.
        int b = 0;
        if ((rc = kth_bin(STB_TIER_Q8, &b)) != STB_OK) return rc;
        floor_cos = (b < 4095) ? (float)(1.0 - (double)(b + 1) / 2048.0 - 0.04) : -INFINITY;
        if ((rc = collect_exact_sorted(ctx, corpus, floor_cos, limit, ranges_dev, n_loc, n_virtual, &n_pass, STB_TIER_Q8)) != STB_OK) return rc;
        if (floor_cos == -INFINITY) done = true;             // everything was collected
        else if (n_pass >= top_k) {
          stb_hit kth;
          STB_CUDA(cudaMemcpyAsync(&kth, ctx->collect_hits + (top_k - 1), sizeof(kth), cudaMemcpyDeviceToHost, ctx->stream));
          STB_CUDA(cudaStreamSynchronize(ctx->stream));
          done = kth.distance < 1.0 - (double)floor_cos - 2.0 * STB_Q8_SCAN_EPS;
        }
        if (!done) ctx->fallback_searches++;
      }
      if (!done) {
        int b = 0;
        if ((rc = kth_bin(STB_TIER_F32, &b)) != STB_OK) return rc;
        floor_cos = (b < 4095) ? (float)(1.0 - (double)(b + 1) / 2048.0 - 2.0 * STB_SCORE_EPS) : -INFINITY;   // else: fewer than k rows, take all
        if ((rc = collect_exact_sorted(ctx, corpus, floor_cos, limit, ranges_dev, n_loc, n_virtual, &n_pass)) != STB_OK) return rc;
      }
    }
    total = threshold_all ? n_pass : std::min<uint64_t>(n_pass, top_k);
    src_dev = ctx->collect_hits;
  }
  *out_n = total;
  uint64_t ncopy = std::min(total, cap);
  if (ncopy) {
    STB_CUDA(cudaMemcpyAsync(out_hits, src_dev, ncopy * sizeof(stb_hit), cudaMemcpyDeviceToHost, ctx->stream));
    STB_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  if (total > cap) { stb_set_error("search: %llu hits, capacity %llu", (unsigned long long)total, (unsigned long long)cap); return STB_ERR_CAPACITY; }
  return STB_OK;
}

int stb_search_topk_dev(stb_ctx *ctx, const stb_corpus *corpus, const float *q_dev, uint32_t top_k,
                        stb_hit *out_hits_dev, uint32_t *out_status_dev) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!corpus || !q_dev || !out_hits_dev || !out_status_dev) { stb_set_error("search_topk_dev: null argument"); return STB_ERR_ARG; }
  if (corpus->ctx != ctx) { stb_set_error("search_topk_dev: corpus belongs to another context"); return STB_ERR_ARG; }
  if (top_k == 0 || top_k > stb_scan_topk_max_k()) { stb_set_error("search_topk_dev: top_k must be 1..%u", stb_scan_topk_max_k()); return STB_ERR_ARG; }
  if (corpus->n == 0) { stb_set_error("search_topk_dev: empty corpus"); return STB_ERR_STATE; }
  // candidates from the narrowest copy that already exists (this asynchronous entry point never
  // builds one: stb_corpus_prepare does); status[1] says whether the result is proven, the
  // caller's fallback is unchanged
  return stb_launch_scan_topk(ctx, corpus, best_built_tier(corpus, top_k), q_dev, top_k, nullptr, 0, corpus->n,
                              out_hits_dev, out_status_dev, nullptr, /*overlapped=*/true);
}

// ------------------------------------------------------------ peer-memory exchange ---
static size_t xchg_bytes(uint32_t world, uint32_t max_k) {
  return (size_t)STB_XCHG_SLOTS * world * 16 + (size_t)STB_XCHG_SLOTS * world * max_k * sizeof(stb_hit);
}

static size_t xchg_batch_slot_bytes(uint32_t world, uint32_t max_nq, uint32_t max_k) {
  const size_t head = ((size_t)world * 8 + (size_t)world * max_nq * 4 + 15) & ~(size_t)15;   // flags | status, 16-byte aligned
  return ((head + (size_t)world * max_nq * max_k * sizeof(stb_hit)) + 255) & ~(size_t)255;
}

static int xchg_create_impl(stb_ctx *ctx, uint32_t world, uint32_t rank, uint32_t max_k, uint32_t max_nq, stb_xchg **out) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!out) { stb_set_error("xchg_create: out is null"); return STB_ERR_ARG; }
  if (world < 1 || world > STB_XCHG_MAX_WORLD || rank >= world) { stb_set_error("xchg_create: world must be 1..%d and rank < world", STB_XCHG_MAX_WORLD); return STB_ERR_ARG; }
  if (max_k < 1 || max_k > stb_scan_topk_max_k()) { stb_set_error("xchg_create: max_k must be 1..%u", stb_scan_topk_max_k()); return STB_ERR_ARG; }
  if (max_nq > 65536 || (uint64_t)world * max_k > 2048) { stb_set_error("xchg_create: batch area too large (max_nq <= 65536, world * max_k <= 2048)"); return STB_ERR_ARG; }
  stb_xchg *x = new (std::nothrow) stb_xchg();
  if (!x) { stb_set_error("out of host memory"); return STB_ERR_NOMEM; }
  memset(x, 0, sizeof(*x));
  x->ctx = ctx; x->world = world; x->rank = rank; x->max_k = max_k; x->max_nq = max_nq;
  x->batch_off = (xchg_bytes(world, max_k) + 255) & ~(size_t)255;
  x->batch_slot_bytes = max_nq ? xchg_batch_slot_bytes(world, max_nq, max_k) : 0;
  x->bytes = x->batch_off + 2 * x->batch_slot_bytes;
  // plain cudaMalloc memory: required for cudaIpcGetMemHandle
  cudaError_t e = cudaMalloc((void **)&x->local, x->bytes);
  if (e == cudaSuccess) e = cudaMemset(x->local, 0, x->bytes);
  if (e == cudaSuccess) e = cudaMalloc((void **)&x->batch_ticket, sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaMemset(x->batch_ticket, 0, sizeof(unsigned int));
  // cudaMemset on device memory may return before it ran (legacy default stream, which a non-blocking
  // stream does not order against): the zeroed flags must be in place before any peer can store to them
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { cudaGetLastError(); cudaFree(x->local); stb_set_error("xchg_create: %s", cudaGetErrorString(e)); delete x; return STB_ERR_NOMEM; }
  x->peers[rank] = x->local;
  x->connected = (world == 1);
  *out = x;
  return STB_OK;
}

int stb_xchg_create(stb_ctx *ctx, uint32_t world, uint32_t rank, uint32_t max_k, stb_xchg **out) {
  return xchg_create_impl(ctx, world, rank, max_k, 0, out);
}
int stb_xchg_create_batch(stb_ctx *ctx, uint32_t world, uint32_t rank, uint32_t max_k, uint32_t max_nq, stb_xchg **out) {
  if (max_nq == 0) { stb_set_error("xchg_create_batch: max_nq must be > 0"); return STB_ERR_ARG; }
  return xchg_create_impl(ctx, world, rank, max_k, max_nq, out);
}

int stb_xchg_destroy(stb_xchg *x) {
  if (!x) return STB_OK;
  if (x->ctx && ctx_alive(x->ctx)) { cudaSetDevice(x->ctx->device); cudaStreamSynchronize(x->ctx->stream); }
  else cudaDeviceSynchronize();
  for (uint32_t r = 0; r < x->world; ++r)
    if (x->ipc_opened[r] && x->peers[r]) cudaIpcCloseMemHandle(x->peers[r]);
  cudaFree(x->batch_ticket);
  cudaFree(x->local);
  cudaGetLastError();
  delete x;
  return STB_OK;
}

int stb_xchg_local_handle(stb_xchg *x, uint8_t handle[STB_IPC_HANDLE_BYTES]) {
  if (!x || !handle) { stb_set_error("xchg_local_handle: null argument"); return STB_ERR_ARG; }
  int rc = ctx_use(x->ctx);
  if (rc) return rc;
  static_assert(sizeof(cudaIpcMemHandle_t) == STB_IPC_HANDLE_BYTES, "IPC handle size");
  cudaIpcMemHandle_t h;
  STB_CUDA(cudaIpcGetMemHandle(&h, x->local));
  memcpy(handle, &h, sizeof(h));
  return STB_OK;
}

int stb_xchg_connect(stb_xchg *x, const uint8_t *handles) {
  if (!x || !handles) { stb_set_error("xchg_connect: null argument"); return STB_ERR_ARG; }
  int rc = ctx_use(x->ctx);
  if (rc) return rc;
  for (uint32_t r = 0; r < x->world; ++r) {
    if (r == x->rank || x->peers[r]) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * STB_IPC_HANDLE_BYTES, sizeof(h));
    void *p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      stb_set_error("xchg_connect: cannot map rank %u's buffer (%s); use the NCCL path", r, cudaGetErrorString(e));
      return STB_ERR_CUDA;
    }
    x->peers[r] = (unsigned char *)p;
    x->ipc_opened[r] = true;
  }
  x->connected = true;
  return STB_OK;
}

int stb_xchg_connect_local(stb_xchg *x, stb_xchg *const *peers) {
  if (!x || !peers) { stb_set_error("xchg_connect_local: null argument"); return STB_ERR_ARG; }
  int rc = ctx_use(x->ctx);
  if (rc) return rc;
  for (uint32_t r = 0; r < x->world; ++r) {
    if (r == x->rank) continue;
    if (!peers[r] || peers[r]->world != x->world || peers[r]->rank != r || peers[r]->max_k != x->max_k || peers[r]->max_nq != x->max_nq) { stb_set_error("xchg_connect_local: peer %u mismatched", r); return STB_ERR_ARG; }
    const int pd = peers[r]->ctx->device;
    if (pd != x->ctx->device) {
      int can = 0;
      STB_CUDA(cudaDeviceCanAccessPeer(&can, x->ctx->device, pd));
      if (!can) { stb_set_error("xchg_connect_local: device %d cannot access device %d", x->ctx->device, pd); return STB_ERR_CUDA; }
      cudaError_t e = cudaDeviceEnablePeerAccess(pd, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { stb_set_error("cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e)); return STB_ERR_CUDA; }
      cudaGetLastError();
    }
    x->peers[r] = peers[r]->local;
  }
  x->connected = true;
  return STB_OK;
}

static int search_topk_xchg_impl(stb_ctx *ctx, const stb_corpus *corpus, const float *q_dev, uint32_t top_k,
                                 stb_xchg *x, stb_hit *out_hits_dev, uint32_t *out_status_dev, bool overlapped) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!corpus || !q_dev || !x || !out_hits_dev || !out_status_dev) { stb_set_error("search_topk_xchg: null argument"); return STB_ERR_ARG; }
  if (corpus->ctx != ctx || x->ctx != ctx) { stb_set_error("search_topk_xchg: handles belong to another context"); return STB_ERR_ARG; }
  if (!x->connected) { stb_set_error("search_topk_xchg: exchange not connected"); return STB_ERR_STATE; }
  if (x->dead) { stb_set_error("search_topk_xchg: this exchange saw a peer time-out; destroy it on every rank"); return STB_ERR_STATE; }
  if (top_k == 0 || top_k > x->max_k) { stb_set_error("search_topk_xchg: top_k must be 1..%u", x->max_k); return STB_ERR_ARG; }
  StbXchgArgs a;
  memset(&a, 0, sizeof(a));
  for (uint32_t r = 0; r < x->world; ++r) a.base[r] = x->peers[r];
  a.world = x->world; a.rank = x->rank; a.max_k = x->max_k;
  a.seq = ++x->seq;
  a.slot = (uint32_t)(a.seq % STB_XCHG_SLOTS);
  return stb_launch_scan_topk(ctx, corpus, best_built_tier(corpus, top_k), q_dev, top_k, nullptr, 0, corpus->n,
                              out_hits_dev, out_status_dev, &a, overlapped);
}

int stb_search_topk_xchg(stb_ctx *ctx, const stb_corpus *corpus, const float *q_dev, uint32_t top_k,
                         stb_xchg *x, stb_hit *out_hits_dev, uint32_t *out_status_dev) {
  return search_topk_xchg_impl(ctx, corpus, q_dev, top_k, x, out_hits_dev, out_status_dev, /*overlapped=*/false);
}

// ----------------------------------------------------------------- K2 batched search ---
static int corpus_ensure_shadow(stb_ctx *ctx, stb_corpus *c) {
  if (c->shadow && c->shadow_rows == c->n) {
    if (c->shadow_bad) { stb_set_error("search_batch: corpus holds rows whose norm is not a normal fp32 number; use stb_search"); return STB_ERR_STATE; }
    return STB_OK;
  }
  const uint64_t tiles = (c->n + 255) / 256;
  uint64_t first = (c->shadow && c->shadow_rows < c->n && !c->shadow_bad) ? (c->shadow_rows / 256) * 256 : 0;   // valid prefix, whole tiles
  if (tiles > c->shadow_cap_tiles || !c->shadow) {
    uint8_t *np = nullptr;
    const uint64_t cap_tiles = std::max<uint64_t>(tiles, (c->capacity + 255) / 256);
    cudaError_t e = cudaMalloc((void **)&np, cap_tiles * 131072ull);
    if (e != cudaSuccess) { cudaGetLastError(); stb_set_error("search_batch: cannot allocate the %llu MiB 16-bit shadow", (unsigned long long)(cap_tiles >> 3)); return STB_ERR_NOMEM; }
    if (c->shadow && first) STB_CUDA(cudaMemcpyAsync(np, c->shadow, (first / 256) * 131072ull, cudaMemcpyDeviceToDevice, ctx->stream));
    else first = 0;
    STB_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaFree(c->shadow);
    c->shadow = np;
    c->shadow_cap_tiles = cap_tiles;
  }
  int rc;
  STB_CUDA(cudaMemsetAsync(ctx->err_flag, 0, sizeof(int), ctx->stream));
  if ((rc = stb_launch_shadow_build(ctx, c->rows, c->n, 256, c->shadow, ctx->err_flag, first)) != STB_OK) return rc;
  int flag = 0;
  STB_CUDA(cudaMemcpyAsync(&flag, ctx->err_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  STB_CUDA(cudaMemsetAsync(ctx->err_flag, 0, sizeof(int), ctx->stream));
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  c->shadow_rows = c->n;
  c->shadow_bad = (first ? c->shadow_bad : 0) | flag;
  if (c->shadow_bad) { stb_set_error("search_batch: corpus holds rows whose norm is not a normal fp32 number; use stb_search"); return STB_ERR_STATE; }
  return STB_OK;
}

static int corpus_ensure_q8(stb_ctx *ctx, stb_corpus *c) {
  if (c->q8 && c->q8_rows == c->n) {
    if (c->q8_bad) { stb_set_error("q8 tier: corpus holds rows whose norm is not a normal fp32 number"); return STB_ERR_STATE; }
    return STB_OK;
  }
  uint64_t first = (c->q8 && c->q8_rows < c->n && !c->q8_bad) ? c->q8_rows : 0;      // valid prefix: convert only the new rows
  if (c->n > c->q8_cap_rows || !c->q8) {
    // the int8 copy (260 B/row) and the coarse copy in front of it (136 B/row) live and grow together
    uint8_t *np = nullptr, *n4 = nullptr;
    float *ns = nullptr;
    float2 *n4s = nullptr;
    const uint64_t cap = std::max<uint64_t>(c->n, c->capacity);
    cudaError_t e = cudaMalloc((void **)&np, cap * 256ull);
    if (e == cudaSuccess) e = cudaMalloc((void **)&ns, cap * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc((void **)&n4, cap * 128ull);
    if (e == cudaSuccess) e = cudaMalloc((void **)&n4s, cap * sizeof(float2));
    if (e != cudaSuccess) {
      cudaGetLastError(); cudaFree(np); cudaFree(ns); cudaFree(n4);
      stb_set_error("q8 tier: cannot allocate %llu MiB", (unsigned long long)(cap * 396 >> 20));
      return STB_ERR_NOMEM;
    }
    if (c->q8 && first) {
      STB_CUDA(cudaMemcpyAsync(np, c->q8, first * 256ull, cudaMemcpyDeviceToDevice, ctx->stream));
      STB_CUDA(cudaMemcpyAsync(ns, c->q8_scale, first * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
      STB_CUDA(cudaMemcpyAsync(n4, c->q4, first * 128ull, cudaMemcpyDeviceToDevice, ctx->stream));
      STB_CUDA(cudaMemcpyAsync(n4s, c->q4_sr, first * sizeof(float2), cudaMemcpyDeviceToDevice, ctx->stream));
      STB_CUDA(cudaStreamSynchronize(ctx->stream));
    } else first = 0;
    cudaFree(c->q8); cudaFree(c->q8_scale); cudaFree(c->q4); cudaFree(c->q4_sr);
    c->q8 = np; c->q8_scale = ns; c->q4 = n4; c->q4_sr = n4s; c->q8_cap_rows = cap;
  }
  int rc;
  STB_CUDA(cudaMemsetAsync(ctx->err_flag, 0, sizeof(int), ctx->stream));
  if ((rc = stb_launch_q8_build(ctx, c->rows, first, c->n, c->q8, c->q8_scale, ctx->err_flag)) != STB_OK) return rc;
  if ((rc = stb_launch_q4_build(ctx, c->rows, first, c->n, c->q4, c->q4_sr, ctx->err_flag)) != STB_OK) return rc;
  int flag = 0;
  STB_CUDA(cudaMemcpyAsync(&flag, ctx->err_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  STB_CUDA(cudaMemsetAsync(ctx->err_flag, 0, sizeof(int), ctx->stream));
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  c->q8_rows = c->n;
  c->q8_bad = (first ? c->q8_bad : 0) | flag;
  if (c->q8_bad) { stb_set_error("q8 tier: corpus holds rows whose norm is not a normal fp32 number"); return STB_ERR_STATE; }
  return STB_OK;
}

int stb_corpus_prepare(stb_corpus *corpus, int what) {
  if (!corpus) { stb_set_error("null corpus"); return STB_ERR_ARG; }
  if (what & ~(STB_PREPARE_Q8 | STB_PREPARE_H16)) { stb_set_error("corpus_prepare: unknown flag"); return STB_ERR_ARG; }
  int rc = ctx_use(corpus->ctx);
  if (rc) return rc;
  if (corpus->n == 0) return STB_OK;
  // rows that cannot be normalised in fp32 make a copy unusable (STB_ERR_STATE): not an error of
  // this call -- searches simply stay on the f32 rows
  if (what & STB_PREPARE_Q8) { rc = corpus_ensure_q8(corpus->ctx, corpus); if (rc != STB_OK && rc != STB_ERR_STATE) return rc; }
  if (what & STB_PREPARE_H16) { rc = corpus_ensure_shadow(corpus->ctx, corpus); if (rc != STB_OK && rc != STB_ERR_STATE) return rc; }
  return STB_OK;
}

int stb_corpus_tier_stats(const stb_corpus *corpus, uint32_t tries[3], uint32_t proven[3], uint64_t built_rows[3]) {
  if (!corpus) { stb_set_error("null corpus"); return STB_ERR_ARG; }
  for (int t = 0; t < 3; ++t) {
    if (tries) tries[t] = corpus->tier_tries[t];
    if (proven) proven[t] = corpus->tier_proven[t];
  }
  if (built_rows) {
    built_rows[STB_TIER_F32] = corpus->n;
    built_rows[STB_TIER_H16] = (corpus->shadow && !corpus->shadow_bad) ? corpus->shadow_rows : 0;   // < n after an append: a valid prefix
    built_rows[STB_TIER_Q8] = (corpus->q8 && !corpus->q8_bad) ? corpus->q8_rows : 0;
  }
  return STB_OK;
}

int stb_corpus_prepare_batch(stb_corpus *corpus) {
  if (!corpus) { stb_set_error("null corpus"); return STB_ERR_ARG; }
  int rc = ctx_use(corpus->ctx);
  if (rc) return rc;
  if (corpus->n == 0) return STB_OK;
  return corpus_ensure_shadow(corpus->ctx, corpus);
}

int stb_search_batch_dev(stb_ctx *ctx, const stb_corpus *corpus_c, const float *q_dev, uint32_t nq,
                         uint32_t top_k, stb_hit *out_hits_dev, uint32_t *out_status_dev) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  stb_corpus *corpus = const_cast<stb_corpus *>(corpus_c);
  if (!corpus || !q_dev || !out_hits_dev || !out_status_dev) { stb_set_error("search_batch_dev: null argument"); return STB_ERR_ARG; }
  if (corpus->ctx != ctx) { stb_set_error("search_batch_dev: corpus belongs to another context"); return STB_ERR_ARG; }
  if (nq == 0) return STB_OK;
  if (top_k == 0 || top_k > 1024) { stb_set_error("search_batch_dev: top_k must be 1..1024"); return STB_ERR_ARG; }
  if (corpus->n == 0) { stb_set_error("search_batch_dev: empty corpus"); return STB_ERR_STATE; }
  if ((rc = corpus_ensure_shadow(ctx, corpus)) != STB_OK) return rc;
  const uint32_t m_tiles = (nq + 127) / 128, q_pad = m_tiles * 128;
  const uint32_t n_tiles = (uint32_t)((corpus->n + 255) / 256), n_sub = n_tiles * 8;
  // Pipeline v2 (default): sampled threshold -> candidate-emitting tcgen05 epilogue -> exact finish
  // (batch_scan.cu).  Proves every query for any top_k <= 64 unless a capacity overflows.
  // STB_BATCH_V1=1 forces the round-1 maxima/select/finish pipeline (also used when v2 does not fit).
  const char *v1_env = getenv("STB_BATCH_V1");            // read per call so one process can compare both
  const bool force_v1 = v1_env != nullptr && v1_env[0] == '1';
  // v2 sampling: ~4 COMPLETE tiles per SM, strided over the shard (a padding row must never stand
  // in for a real one).  Expected candidates per query ~ top_k * n_full / n_sample * e^(2 EPS x / sigma^2)
  // (x = top score, sigma = 1/16 for the benchmark's rows: factor ~1.2 with the fp16 shadow's
  // EPS = 0.0012, ~3.8 with bf16's 0.0080).  Shards so large that this exceeds half of the finish
  // kernel's 4096-key capacity sample 1/64 of the tiles instead (threshold kernel: CTA-per-query
  // variant, <= 8192 tiles); beyond that, v1.
  const uint32_t n_full = (uint32_t)(corpus->n / 256);
  uint32_t n_sample = std::min<uint32_t>(n_full, std::min<uint32_t>(4u * (uint32_t)ctx->sm_count, 608u));
  const uint32_t margin_factor = STB_SHADOW_F16 ? 2u : 4u;
  auto expected_emitted = [&](uint32_t ns) { return ns ? (uint64_t)top_k * margin_factor * ((n_full + ns - 1) / ns) : 0; };
  if (expected_emitted(n_sample) > 2048) {
    const uint32_t sm = (uint32_t)ctx->sm_count;
    n_sample = std::min<uint32_t>(std::min<uint32_t>(n_full, 8192u), (n_full / 64 + sm - 1) / sm * sm);
  }
  const bool v2_fits = n_sample >= top_k && expected_emitted(n_sample) <= 2048;
  if (!force_v1 && top_k <= 64 && v2_fits) {
    constexpr uint32_t kSegCap = 64;                      // per (query, CTA): ~5 expected at 10M rows / 148 CTAs
    const uint32_t n_seg = stb_batch_emit_grid(ctx, n_tiles);
    const uint32_t stride = n_full / n_sample;
    if ((rc = dev_reserve(&ctx->bq_tiles, &ctx->bq_tiles_cap, (size_t)q_pad * 512)) != STB_OK) return rc;
    if ((rc = dev_reserve(&ctx->b_tilemax, &ctx->b_tilemax_cap, (size_t)n_sample * q_pad)) != STB_OK) return rc;
    if ((rc = dev_reserve(&ctx->b_thr, &ctx->b_thr_cap, (size_t)q_pad)) != STB_OK) return rc;
    if ((rc = dev_reserve(&ctx->b_cnt, &ctx->b_cnt_cap, (size_t)q_pad * n_seg)) != STB_OK) return rc;
    if ((rc = dev_reserve(&ctx->b_keys, &ctx->b_keys_cap, (size_t)q_pad * n_seg * kSegCap)) != STB_OK) return rc;
    STB_CUDA(cudaMemsetAsync(ctx->err_flag, 0, sizeof(int), ctx->stream));
    STB_CUDA(cudaMemsetAsync(ctx->b_cnt, 0, (size_t)q_pad * n_seg * sizeof(uint32_t), ctx->stream));
    if ((rc = stb_launch_shadow_build(ctx, q_dev, nq, 128, ctx->bq_tiles, ctx->err_flag)) != STB_OK) return rc;
    if ((rc = stb_launch_batch_gemm_strided(ctx, ctx->bq_tiles, m_tiles, corpus->shadow, n_sample, stride, nullptr,
                                            ctx->b_tilemax, nullptr)) != STB_OK) return rc;
    if ((rc = stb_launch_batch_thresh(ctx, ctx->b_tilemax, n_sample, nq, q_pad, top_k, ctx->b_thr)) != STB_OK) return rc;
    if ((rc = stb_launch_batch_gemm_emit(ctx, ctx->bq_tiles, m_tiles, corpus->shadow, n_tiles, corpus->n, ctx->b_thr,
                                         ctx->b_cnt, ctx->b_keys, kSegCap)) != STB_OK) return rc;
    return stb_launch_batch_finish2(ctx, ctx->b_keys, ctx->b_cnt, n_seg, kSegCap, nq, top_k, corpus->rows, corpus->n,
                                    corpus->row_base, q_dev, out_hits_dev, out_status_dev);
  }
  // selection slices: enough CTAs (m_tiles x n_slices) to hide the latency of the streaming
  // read; the finish kernel merges n_slices x 32 <= 4096 candidate tiles per query
  uint32_t n_slices = std::max<uint32_t>(1, std::min<uint32_t>(128, 1536 / m_tiles));
  n_slices = std::min<uint32_t>(n_slices, std::max<uint32_t>(1, n_tiles / 48));
  if ((rc = dev_reserve(&ctx->bq_tiles, &ctx->bq_tiles_cap, (size_t)q_pad * 512)) != STB_OK) return rc;
  if ((rc = dev_reserve(&ctx->b_submax, &ctx->b_submax_cap, (size_t)n_sub * q_pad)) != STB_OK) return rc;
  if ((rc = dev_reserve(&ctx->b_tilemax, &ctx->b_tilemax_cap, (size_t)n_tiles * q_pad)) != STB_OK) return rc;
  if ((rc = dev_reserve(&ctx->b_cand, &ctx->b_cand_cap, (size_t)q_pad * n_slices * 32)) != STB_OK) return rc;
  // query tiles: padding queries beyond nq are written as zeros by the shadow builder
  STB_CUDA(cudaMemsetAsync(ctx->err_flag, 0, sizeof(int), ctx->stream));
  if ((rc = stb_launch_shadow_build(ctx, q_dev, nq, 128, ctx->bq_tiles, ctx->err_flag)) != STB_OK) return rc;
  if ((rc = stb_launch_batch_gemm(ctx, ctx->bq_tiles, m_tiles, corpus->shadow, n_tiles, ctx->b_submax, ctx->b_tilemax, nullptr)) != STB_OK) return rc;
  // two-level selection: the best tiles by tile maximum (1/8 of the data), refined to
  // sub-tiles inside the finish kernel
  if ((rc = stb_launch_batch_select(ctx, ctx->b_tilemax, n_tiles, q_pad, n_slices, ctx->b_cand)) != STB_OK) return rc;
  return stb_launch_batch_finish(ctx, ctx->b_cand, n_slices, n_sub, nq, top_k, corpus->rows, corpus->n,
                                 corpus->row_base, q_dev, out_hits_dev, out_status_dev, ctx->b_submax, q_pad);
}

int stb_search_batch(stb_ctx *ctx, const stb_corpus *corpus, const float *q, uint32_t nq, uint32_t top_k,
                     stb_hit *out_hits, uint32_t *out_n) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!corpus || !q || !out_hits || !out_n) { stb_set_error("search_batch: null argument"); return STB_ERR_ARG; }
  if (nq == 0) return STB_OK;
  for (uint32_t i = 0; i < nq; ++i) out_n[i] = 0;
  if (top_k == 0 || corpus->n == 0) return STB_OK;
  bool tensor_ok = top_k <= 1024;
  std::vector<uint32_t> status((size_t)nq * 2, 0);
  if (tensor_ok) {
    if ((rc = dev_reserve(&ctx->bq_dev, &ctx->bq_dev_cap, (size_t)nq * STB_D)) != STB_OK) return rc;
    if ((rc = dev_reserve(&ctx->bh_dev, &ctx->bh_dev_cap, (size_t)nq * top_k)) != STB_OK) return rc;
    if ((rc = dev_reserve(&ctx->bs_dev, &ctx->bs_dev_cap, (size_t)nq * 2)) != STB_OK) return rc;
    STB_CUDA(cudaMemcpyAsync(ctx->bq_dev, q, (size_t)nq * STB_D * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    rc = stb_search_batch_dev(ctx, corpus, ctx->bq_dev, nq, top_k, ctx->bh_dev, ctx->bs_dev);
    if (rc == STB_ERR_STATE) { tensor_ok = false; }        // un-normalisable rows: K1 handles them
    else if (rc != STB_OK) return rc;
    else {
      int qbad = 0;
      STB_CUDA(cudaMemcpyAsync(&qbad, ctx->err_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
      STB_CUDA(cudaMemsetAsync(ctx->err_flag, 0, sizeof(int), ctx->stream));
      STB_CUDA(cudaMemcpyAsync(out_hits, ctx->bh_dev, (size_t)nq * top_k * sizeof(stb_hit), cudaMemcpyDeviceToHost, ctx->stream));
      STB_CUDA(cudaMemcpyAsync(status.data(), ctx->bs_dev, (size_t)nq * 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
      STB_CUDA(cudaStreamSynchronize(ctx->stream));
      if (qbad) std::fill(status.begin(), status.end(), 0u);   // a query could not be normalised: trust none
    }
  }
  // queries the tensor path could not prove (or could not run): exact single-query path
  for (uint32_t i = 0; i < nq; ++i) {
    if (tensor_ok && status[2 * i + 1]) { out_n[i] = status[2 * i]; continue; }
    ctx->fallback_searches++;
    uint64_t n = 0;
    rc = stb_search(ctx, corpus, q + (size_t)i * STB_D, top_k, 0, 0.0, STB_MODE_SEARCH_DOCUMENTS, nullptr, 0,
                    out_hits + (size_t)i * top_k, top_k, &n);
    if (rc != STB_OK) return rc;
    out_n[i] = (uint32_t)n;
    for (uint64_t j = n; j < top_k; ++j) { out_hits[(size_t)i * top_k + j].distance = INFINITY; out_hits[(size_t)i * top_k + j].row = 0xffffffffffffffffull; }
  }
  return STB_OK;
}

// Sharded K2: every rank answers the nq queries on its shard (stb_search_batch_dev), then ONE exchange over
// NVLink peer memory -- each rank stores its nq x k hits + per-query proof flags into every peer's batch slot
// (push kernel), waits for all peers' sequence flags and merges per query (merge kernel).  Two launches, no
// NCCL call.  out_status_dev[2q] = hits of query q, [2q+1] = 1 iff EVERY rank proved its part, 2 = a peer
// never arrived.  Unproven queries: re-run them with stb_search_xchg / stb_search_many(x) (collective: every
// rank sees the same flags).
int stb_search_batch_xchg_dev(stb_ctx *ctx, const stb_corpus *corpus, const float *q_dev, uint32_t nq, uint32_t top_k,
                              stb_xchg *x, stb_hit *out_hits_dev, uint32_t *out_status_dev) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!corpus || !q_dev || !x || !out_hits_dev || !out_status_dev) { stb_set_error("search_batch_xchg_dev: null argument"); return STB_ERR_ARG; }
  if (corpus->ctx != ctx || x->ctx != ctx) { stb_set_error("search_batch_xchg_dev: handles belong to another context"); return STB_ERR_ARG; }
  if (!x->connected) { stb_set_error("search_batch_xchg_dev: exchange not connected"); return STB_ERR_STATE; }
  if (x->dead) { stb_set_error("search_batch_xchg_dev: this exchange saw a peer time-out; destroy it on every rank"); return STB_ERR_STATE; }
  if (nq == 0) return STB_OK;
  if (x->max_nq == 0 || nq > x->max_nq || top_k == 0 || top_k > x->max_k) { stb_set_error("search_batch_xchg_dev: needs stb_xchg_create_batch with max_nq >= %u, max_k >= %u", nq, top_k); return STB_ERR_ARG; }
  if ((rc = dev_reserve(&ctx->bh_dev, &ctx->bh_dev_cap, (size_t)nq * top_k)) != STB_OK) return rc;
  if ((rc = dev_reserve(&ctx->bs_dev, &ctx->bs_dev_cap, (size_t)nq * 2)) != STB_OK) return rc;
  if ((rc = stb_search_batch_dev(ctx, corpus, q_dev, nq, top_k, ctx->bh_dev, ctx->bs_dev)) != STB_OK) return rc;
  StbBatchXchgArgs a;
  memset(&a, 0, sizeof(a));
  a.world = x->world; a.rank = x->rank; a.max_nq = x->max_nq; a.max_k = x->max_k; a.nq = nq; a.top_k = top_k;
  a.seq = ++x->batch_seq;
  a.ticket = x->batch_ticket;
  for (uint32_t r = 0; r < x->world; ++r) a.slot[r] = x->peers[r] + x->batch_off + (size_t)(a.seq & 1) * x->batch_slot_bytes;
  return stb_launch_batch_xchg(ctx, a, ctx->bh_dev, ctx->bs_dev, out_hits_dev, out_status_dev);
}

int stb_debug_batch_params(int *shadow_is_f16, double *eps) {
  stb_batch_build_params(shadow_is_f16, eps);
  return STB_OK;
}

// ------------------------------------------------------------------- K2 debug hook ---
// Runs shadow build + tcgen05 GEMM on host inputs and returns the FULL approximate score
// matrix (tests only: validates descriptors / TMEM / epilogue against a reference matmul).
int stb_debug_batch_gemm(stb_ctx *ctx, const float *q, uint32_t nq, const float *rows, uint64_t n,
                         float *out_full, float *out_submax) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!q || !rows || !out_full || nq == 0 || n == 0) { stb_set_error("debug_batch_gemm: bad argument"); return STB_ERR_ARG; }
  const uint32_t m_tiles = (nq + 127) / 128;
  const uint32_t n_tiles = (uint32_t)((n + 255) / 256);
  const size_t q_pad = (size_t)m_tiles * 128, n_pad = (size_t)n_tiles * 256;
  float *dq = nullptr, *dr = nullptr, *dfull = nullptr, *dsub = nullptr, *dtile = nullptr;
  uint8_t *da = nullptr, *db = nullptr;
  int *dbad = nullptr;
  cudaError_t e = cudaMalloc(&dq, (size_t)nq * 1024);
  if (e == cudaSuccess) e = cudaMalloc(&dr, n * 1024);
  if (e == cudaSuccess) e = cudaMalloc(&da, q_pad * 512);
  if (e == cudaSuccess) e = cudaMalloc(&db, n_pad * 512);
  if (e == cudaSuccess) e = cudaMalloc(&dfull, q_pad * n_pad * 4);
  if (e == cudaSuccess) e = cudaMalloc(&dsub, (size_t)n_tiles * 8 * q_pad * 4);
  if (e == cudaSuccess) e = cudaMalloc(&dtile, (size_t)n_tiles * q_pad * 4);
  if (e == cudaSuccess) e = cudaMalloc(&dbad, 4);
  if (e == cudaSuccess) e = cudaMemsetAsync(dbad, 0, 4, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(dq, q, (size_t)nq * 1024, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(dr, rows, n * 1024, cudaMemcpyHostToDevice, ctx->stream);
  rc = STB_OK;
  if (e == cudaSuccess) rc = stb_launch_shadow_build(ctx, dq, nq, 128, da, dbad);
  if (e == cudaSuccess && rc == STB_OK) rc = stb_launch_shadow_build(ctx, dr, n, 256, db, dbad);
  if (e == cudaSuccess && rc == STB_OK) rc = stb_launch_batch_gemm(ctx, da, m_tiles, db, n_tiles, dsub, dtile, dfull);
  if (e == cudaSuccess && rc == STB_OK) e = cudaMemcpyAsync(out_full, dfull, q_pad * n_pad * 4, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess && rc == STB_OK && out_submax) e = cudaMemcpyAsync(out_submax, dsub, (size_t)n_tiles * 8 * q_pad * 4, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess && rc == STB_OK) e = cudaStreamSynchronize(ctx->stream);
  cudaFree(dq); cudaFree(dr); cudaFree(da); cudaFree(db); cudaFree(dfull); cudaFree(dsub); cudaFree(dtile); cudaFree(dbad);
  if (e != cudaSuccess) { stb_set_error("debug_batch_gemm: %s", cudaGetErrorString(e)); cudaGetLastError(); return STB_ERR_CUDA; }
  return rc;
}

int stb_search_xchg(stb_ctx *ctx, const stb_corpus *corpus, const float *q, uint32_t top_k, stb_xchg *x,
                    stb_hit *out_hits, uint32_t *out_n, int *out_complete) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!q || !out_hits || !out_n || !out_complete) { stb_set_error("search_xchg: null argument"); return STB_ERR_ARG; }
  static const bool prof = getenv("STB_XCHG_PROFILE") != nullptr;
  static double t_enq = 0, t_sync = 0; static long n_calls = 0;
  auto t0 = std::chrono::steady_clock::now();
  memcpy(ctx->q_pin, q, STB_D * sizeof(float));
  STB_CUDA(cudaMemcpyAsync(ctx->q_dev, ctx->q_pin, STB_D * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  if (stb_env_direct_out()) {        // the merge CTA stores the hits + status straight into pinned host memory
    if ((rc = search_topk_xchg_impl(ctx, corpus, ctx->q_dev, top_k, x, ctx->hits_pin, ctx->status_pin, false)) != STB_OK) return rc;
  } else {
    if ((rc = search_topk_xchg_impl(ctx, corpus, ctx->q_dev, top_k, x, ctx->hits_dev, ctx->status_dev, false)) != STB_OK) return rc;
    STB_CUDA(cudaMemcpyAsync(ctx->status_pin, ctx->status_dev, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    STB_CUDA(cudaMemcpyAsync(ctx->hits_pin, ctx->hits_dev, top_k * sizeof(stb_hit), cudaMemcpyDeviceToHost, ctx->stream));
  }
  auto t1 = std::chrono::steady_clock::now();
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  if (prof) {
    auto t2 = std::chrono::steady_clock::now();
    t_enq += std::chrono::duration<double, std::micro>(t1 - t0).count();
    t_sync += std::chrono::duration<double, std::micro>(t2 - t1).count();
    if (++n_calls % 50 == 0) fprintf(stderr, "[stb_search_xchg rank %u] calls %ld  enqueue %.1f us  sync %.1f us (avg)\n", x->rank, n_calls, t_enq / n_calls, t_sync / n_calls);
  }
  const uint32_t n = std::min<uint32_t>(ctx->status_pin[0], top_k);
  memcpy(out_hits, ctx->hits_pin, n * sizeof(stb_hit));
  *out_n = n;
  *out_complete = ctx->status_pin[1] ? 1 : 0;
  if (ctx->status_pin[2] == 0xfffffffeu) { x->dead = true; stb_set_error("search_xchg: a peer rank never arrived (timeout)"); return STB_ERR_STATE; }
  return STB_OK;
}

// Many independent single queries with ONE synchronisation: queries are staged through pinned
// memory in one H2D copy, the nq scan kernels are enqueued back to back (PDL overlaps each tail
// with the next scan) and every kernel's final CTA stores its hits + status straight into pinned
// host memory.  Unproven queries are re-run through stb_search (x == NULL) or reported
// (x != NULL: all ranks see the same flag and fall back together).
int stb_search_many(stb_ctx *ctx, const stb_corpus *corpus, const float *q, uint32_t nq, uint32_t top_k, stb_xchg *x,
                    stb_hit *out_hits, uint32_t *out_n, uint8_t *out_complete) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!corpus || !q || !out_hits || !out_n) { stb_set_error("search_many: null argument"); return STB_ERR_ARG; }
  if (corpus->ctx != ctx || (x && x->ctx != ctx)) { stb_set_error("search_many: handles belong to another context"); return STB_ERR_ARG; }
  if (nq == 0) return STB_OK;
  for (uint32_t i = 0; i < nq; ++i) { out_n[i] = 0; if (out_complete) out_complete[i] = 1; }
  if (top_k == 0 || corpus->n == 0) {
    if (x && corpus->n == 0) { stb_set_error("search_many: empty shard in a sharded search"); return STB_ERR_STATE; }
    return STB_OK;
  }
  if (top_k > (x ? x->max_k : stb_scan_topk_max_k())) {
    if (x) { stb_set_error("search_many: top_k must be 1..%u", x->max_k); return STB_ERR_ARG; }
    for (uint32_t i = 0; i < nq; ++i) {                    // beyond the register lists: the general path, query by query
      uint64_t n = 0;
      rc = stb_search(ctx, corpus, q + (size_t)i * STB_D, top_k, 0, 0.0, STB_MODE_SEARCH_DOCUMENTS, nullptr, 0,
                      out_hits + (size_t)i * top_k, top_k, &n);
      if (rc != STB_OK) return rc;
      out_n[i] = (uint32_t)n;
    }
    return STB_OK;
  }
  // many queries amortise the reduced-width copy: build it now (same size rule as the lazy build)
  stb_corpus *cm = const_cast<stb_corpus *>(corpus);
  if (nq >= 2 && cm->n >= 32768 && stb_env_max_tier() >= STB_TIER_Q8 && top_k <= STB_Q8_MAX_K && !(cm->q8 && cm->q8_rows == cm->n)) {
    rc = corpus_ensure_q8(ctx, cm);
    if (rc != STB_OK && rc != STB_ERR_STATE) return rc;
  }
  if ((rc = dev_reserve(&ctx->bq_dev, &ctx->bq_dev_cap, (size_t)nq * STB_D)) != STB_OK) return rc;
  if ((rc = ensure_hits_pin(ctx, (size_t)nq * top_k)) != STB_OK) return rc;
  if ((size_t)nq * STB_D > ctx->many_q_pin_cap) {
    float *np = nullptr; uint32_t *ns = nullptr;
    const size_t cap = std::max<size_t>((size_t)nq, 64);
    if (cudaMallocHost((void **)&np, cap * STB_D * sizeof(float)) != cudaSuccess ||
        cudaMallocHost((void **)&ns, cap * 4 * sizeof(uint32_t)) != cudaSuccess) {
      cudaGetLastError(); if (np) cudaFreeHost(np);
      stb_set_error("search_many: pinned staging allocation failed"); return STB_ERR_NOMEM;
    }
    if (ctx->many_q_pin) cudaFreeHost(ctx->many_q_pin);
    if (ctx->many_status_pin) cudaFreeHost(ctx->many_status_pin);
    ctx->many_q_pin = np; ctx->many_status_pin = ns; ctx->many_q_pin_cap = cap * STB_D;
  }
  memcpy(ctx->many_q_pin, q, (size_t)nq * STB_D * sizeof(float));
  STB_CUDA(cudaMemcpyAsync(ctx->bq_dev, ctx->many_q_pin, (size_t)nq * STB_D * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  const int tier = best_built_tier(corpus, top_k);
  for (uint32_t i = 0; i < nq; ++i) {
    stb_hit *oh = ctx->hits_pin + (size_t)i * top_k;
    uint32_t *os = ctx->many_status_pin + 4 * (size_t)i;
    if (x) rc = search_topk_xchg_impl(ctx, corpus, ctx->bq_dev + (size_t)i * STB_D, top_k, x, oh, os, /*overlapped=*/false);
    else rc = stb_launch_scan_topk(ctx, corpus, tier, ctx->bq_dev + (size_t)i * STB_D, top_k, nullptr, 0, corpus->n, oh, os, nullptr,
                                   /*overlapped=*/nq > 1);
    if (rc != STB_OK) { cudaStreamSynchronize(ctx->stream); return rc; }
  }
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  for (uint32_t i = 0; i < nq; ++i) {
    const uint32_t *st = ctx->many_status_pin + 4 * (size_t)i;
    if (x && st[2] == 0xfffffffeu) { x->dead = true; stb_set_error("search_many: a peer rank never arrived (timeout)"); return STB_ERR_STATE; }
    if (st[1]) {
      const uint32_t n = std::min<uint32_t>(st[0], top_k);
      memcpy(out_hits + (size_t)i * top_k, ctx->hits_pin + (size_t)i * top_k, n * sizeof(stb_hit));
      out_n[i] = n;
    } else if (x) {
      if (out_complete) out_complete[i] = 0;               // every rank sees the same flag: fall back together
    } else {
      uint64_t n = 0;                                      // tier ladder / collect path
      rc = stb_search(ctx, corpus, q + (size_t)i * STB_D, top_k, 0, 0.0, STB_MODE_SEARCH_DOCUMENTS, nullptr, 0,
                      out_hits + (size_t)i * top_k, top_k, &n);
      if (rc != STB_OK) return rc;
      out_n[i] = (uint32_t)n;
    }
  }
  return STB_OK;
}

// ---------------------------------------------------------------------- merge ---
int stb_hits_merge_dev(stb_ctx *ctx, const stb_hit *lists_dev, uint32_t n_lists, uint32_t per_list,
                       uint32_t top_k, stb_hit *out_dev) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!lists_dev || !out_dev || n_lists == 0 || per_list == 0 || top_k == 0) { stb_set_error("hits_merge: bad argument"); return STB_ERR_ARG; }
  return stb_launch_hits_merge(ctx, lists_dev, n_lists, per_list, top_k, out_dev);
}

int stb_hits_merge_batch_dev(stb_ctx *ctx, const stb_hit *lists_dev, uint32_t n_lists, uint32_t nq,
                             uint32_t per_list, uint32_t top_k, stb_hit *out_dev) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!lists_dev || !out_dev || n_lists == 0 || per_list == 0 || top_k == 0) { stb_set_error("hits_merge_batch: bad argument"); return STB_ERR_ARG; }
  if (nq == 0) return STB_OK;
  return stb_launch_hits_merge_batch(ctx, lists_dev, n_lists, nq, per_list, top_k, out_dev);
}

int stb_hits_merge(stb_ctx *ctx, const stb_hit *lists, uint32_t n_lists, uint32_t per_list,
                   uint32_t top_k, stb_hit *out, uint32_t *out_n) {
  int rc = ctx_use(ctx);
  if (rc) return rc;
  if (!lists || !out || !out_n || n_lists == 0 || per_list == 0) { stb_set_error("hits_merge: bad argument"); return STB_ERR_ARG; }
  *out_n = 0;
  if (top_k == 0) return STB_OK;
  const size_t total = (size_t)n_lists * per_list;
  if ((rc = dev_reserve(&ctx->hits_dev, &ctx->hits_cap, total + top_k)) != STB_OK) return rc;
  if ((rc = ensure_hits_pin(ctx, std::max<size_t>(total, top_k))) != STB_OK) return rc;
  memcpy(ctx->hits_pin, lists, total * sizeof(stb_hit));
  STB_CUDA(cudaMemcpyAsync(ctx->hits_dev, ctx->hits_pin, total * sizeof(stb_hit), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = stb_launch_hits_merge(ctx, ctx->hits_dev, n_lists, per_list, top_k, ctx->hits_dev + total)) != STB_OK) return rc;
  STB_CUDA(cudaMemcpyAsync(ctx->hits_pin, ctx->hits_dev + total, top_k * sizeof(stb_hit), cudaMemcpyDeviceToHost, ctx->stream));
  STB_CUDA(cudaStreamSynchronize(ctx->stream));
  uint32_t n = 0;
  for (uint32_t i = 0; i < top_k; ++i) {
    if (ctx->hits_pin[i].row == 0xffffffffffffffffull) break;
    out[n++] = ctx->hits_pin[i];
  }
  *out_n = n;
  return STB_OK;
}

// ------------------------------------------------------------------------ ids ---
uint64_t stb_fnv1a64(const uint8_t *bytes, uint64_t len) {
  uint64_t h = 0xcbf29ce484222325ull;
  for (uint64_t i = 0; i < len; ++i) { h ^= bytes[i]; h *= 0x100000001b3ull; }
  return h;
}

uint64_t stb_line_id(const uint8_t *path, uint64_t path_len, int32_t line_number) {
  uint64_t h = 0xcbf29ce484222325ull;
  for (uint64_t i = 0; i < path_len; ++i) { h ^= path[i]; h *= 0x100000001b3ull; }
  const uint32_t u = (uint32_t)line_number;
  for (int b = 0; b < 4; ++b) { h ^= (u >> (8 * b)) & 0xffu; h *= 0x100000001b3ull; }
  return h;
}

// LineEmbedding::id for many rows at once: rows = n_rows x (path index, line_number) int32, paths
// given as one byte blob + n_paths+1 offsets.  The FNV state after each path is computed once.
int stb_line_ids(const uint8_t *path_bytes, const uint64_t *path_offsets, uint32_t n_paths, const int32_t *rows,
                 uint64_t n_rows, uint64_t *out_ids) {
  if ((n_paths && (!path_bytes || !path_offsets)) || (n_rows && (!rows || !out_ids))) { stb_set_error("line_ids: null argument"); return STB_ERR_ARG; }
  std::vector<uint64_t> prefix(n_paths);
  for (uint32_t p = 0; p < n_paths; ++p) {
    uint64_t h = 0xcbf29ce484222325ull;
    for (uint64_t i = path_offsets[p]; i < path_offsets[p + 1]; ++i) { h ^= path_bytes[i]; h *= 0x100000001b3ull; }
    prefix[p] = h;
  }
  for (uint64_t r = 0; r < n_rows; ++r) {
    const int32_t pi = rows[2 * r];
    if (pi < 0 || (uint32_t)pi >= n_paths) { stb_set_error("line_ids: row %llu refers to path %d of %u", (unsigned long long)r, pi, n_paths); return STB_ERR_RANGE; }
    uint64_t h = prefix[pi];
    const uint32_t u = (uint32_t)rows[2 * r + 1];
    for (int b = 0; b < 4; ++b) { h ^= (u >> (8 * b)) & 0xffu; h *= 0x100000001b3ull; }
    out_ids[r] = h;
  }
  return STB_OK;
}

}  // extern "C"
