// K1 (+ in-kernel K4): cosine scan with running top-K', tree merge, exact re-rank.
//
// Replaces the loop/sort/take of search_documents (reference
// src/search/mod.rs:84-119; one simsimd f32::cosine per line at :86) and the
// filtered nearest query of Store::search_line_embeddings
// (src/workspace/store.rs:495-543).
//
// HBM-bound: the only large traffic is the corpus matrix, 1 KiB per row, read
// exactly once with 128-bit coalesced loads (8 lanes cover one 128-byte line of a
// row; a warp instruction touches 4 full lines).  Everything else (query, K'
// candidates per CTA, k results) is bytes.
//
// Exactness: the streaming pass ranks rows by an fp32 approximate cosine and keeps
// the best K' = 32*E per warp; the surviving K' of the whole grid are re-scored by
// one thread each in the oracle's canonical arithmetic (f64 accumulation in index
// order) and sorted by (distance,row).  The result is accepted only if the worst
// kept approximate score proves that no dropped row can reach the k-th exact
// distance (STB_SCORE_EPS); otherwise status[1]=0 and the host runs the collect
// path below, which is exact for any input.
#include <math_constants.h>

#include <cuda_fp16.h>

#include <algorithm>

#include "common.cuh"

#ifndef STB_SCAN_U
#define STB_SCAN_U 2   // rows per 8-lane group per iteration (loads in flight = 8*U float4)
#endif
#ifndef STB_SCAN_LD
#define STB_SCAN_LD 0  // 0: ld.global.nc.L1::no_allocate  1: __ldcs  2: __ldg
#endif

__device__ __forceinline__ float4 stb_ld_stream(const float4 *p) {
#if STB_SCAN_LD == 0
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
#elif STB_SCAN_LD == 1
  return __ldcs(p);
#else
  return __ldg(p);
#endif
}

struct ScanArgs {
  const float4 *rows;        // local row 0
  uint64_t n_virtual;        // rows to scan (== n_rows when no ranges)
  const float *q;            // 256 f32 (device)
  const uint64_t *vstart;    // [n_ranges+1] virtual prefix (ranges mode)
  const uint64_t *rbegin;    // [n_ranges]   local first row of each range
  uint32_t n_ranges;
  // dynamic tile schedule (top-k kernel; null = static warp-strided schedule):
  unsigned long long *tickets;   // this launch's counter of the context's ring (monotonic)
  unsigned long long t_base;     // its value when this launch starts (host-tracked)
  uint64_t t_bulk;               // tickets [0, t_bulk) cover STB_TICKET_TILES tiles each, later ones one tile
  unsigned long long *start;     // this launch's ring word: (seq << 32) | first tile, once published
  unsigned long long *front;     // the context's scan front: a virtual row some running scan reached
  uint32_t seq;                  // launch number (never 0): tells this launch's start from a stale one
};
#define STB_TICKET_TILES 4
#define STB_FRONT_EVERY 64       // tickets per store to the scan front

// ---- tile schedule + row map shared by the three scans -----------------------------------
// RANGES == 0: whole shard, tiles are warp-strided (the grid streams one contiguous window).
// RANGES == 1: row ranges (workspace path filter).  Blocks of WB consecutive tiles are
// warp-strided and a warp walks each block in order, so the virtual->local row map costs one
// binary search per block per lane and a forward step per row afterwards (the per-row
// 15-step search of round 1 held this mode at 0.52 of the HBM peak).
// Dynamic schedule (args.tickets != null): warps draw tickets from one atomic counter; a ticket is
// STB_TICKET_TILES consecutive tiles, except that the last ~2 tiles per warp are handed out one
// by one so the grid drains evenly.  Tickets are issued in row order, so the grid still streams
// one contiguous window.  Why: the grid fills every CTA slot, and with a static partition a CTA
// that starts late finishes late -- under PDL the next query's last CTA cannot start before this
// query's final (merge) CTA exits, which exposed the whole tail (10 us at K'=32, 77 us at
// K'=128) on every pipelined query.  With tickets a late CTA simply finds less work.
// Every warp makes exactly one failing draw, so a launch advances the counter by
// n_tickets + total_warps -- the host tracks the base of the next launch with that.
// Synchronized scans: a launch does not start at tile 0 but at the tile s where some running scan of the
// context currently is, and wraps around: ticket t covers tiles (s + first_tile(t) + i) mod n_tiles.  Two
// co-resident grids (overlapped launches) then stream the same lines at the same time, so each line comes
// from HBM once for both; a launch that follows a finished one starts on the lines still in L2.  Warps
// store the first virtual row of every STB_FRONT_EVERY-th ticket to args.front; any value is correct,
// only the sharing depends on it.  body(tile, restart): restart is set at a ticket's first tile and at
// the wrap to tile 0 (the row-ranges map walks forward only).
__device__ __forceinline__ void stb_st_release_gpu(unsigned long long *p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long stb_ld_acquire_gpu(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void stb_st_relaxed_gpu(unsigned long long *p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long stb_ld_relaxed_gpu(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

template <int RANGES, int WB, class Body>
__device__ __forceinline__ void stb_for_each_tile(const ScanArgs &args, uint64_t n_tiles, uint64_t tile_rows, Body &&body) {
  if (args.tickets) {
    // The next ticket is drawn BEFORE the current one is processed, so the atomic's L2 round trip
    // (~1 us under load) overlaps a ticket's worth of loads instead of stalling the warp 4-6 times per
    // query (at 1.25M rows per GPU that was ~10 % of the scan).  A warp stops drawing at its first
    // failing draw, so the "exactly one failing draw per warp" bookkeeping holds.
    const int lane = threadIdx.x & 31;
    auto draw = [&]() -> unsigned long long {
      unsigned long long t = 0;
      if (lane == 0) t = atomicAdd(args.tickets, 1ull);
      return __shfl_sync(0xffffffffu, t, 0) - args.t_base;
    };
    auto first_tile = [&](unsigned long long t) -> uint64_t {
      return t < args.t_bulk ? t * STB_TICKET_TILES : args.t_bulk * STB_TICKET_TILES + (t - args.t_bulk);
    };
    unsigned long long cur = draw();
    if (first_tile(cur) >= n_tiles) return;
    // The start tile s: the warp that drew ticket 0 reads the front and publishes s for this launch; the
    // others wait for it.  No deadlock: a waiter depends only on a warp of its own grid, and that warp is
    // resident (it has drawn ticket 0) and publishes before it waits on anything.  The word is tagged with
    // the launch number, so nothing is reset between launches.
    uint64_t s = 0;
    if (lane == 0) {
      if (cur == 0) {
        s = (stb_ld_relaxed_gpu(args.front) % args.n_virtual) / tile_rows;
        stb_st_release_gpu(args.start, ((unsigned long long)args.seq << 32) | s);
      } else {
        unsigned long long w;
        while (((w = stb_ld_acquire_gpu(args.start)) >> 32) != args.seq) __nanosleep(100);
        s = w & 0xffffffffull;
      }
    }
    s = __shfl_sync(0xffffffffu, s, 0);
    do {
      const unsigned long long nxt = draw();
      const uint64_t t0 = first_tile(cur);
      const uint64_t t1 = cur < args.t_bulk ? t0 + STB_TICKET_TILES : t0 + 1;
      uint64_t tile = s + t0;
      if (tile >= n_tiles) tile -= n_tiles;
      if (lane == 0 && cur % STB_FRONT_EVERY == 0) stb_st_relaxed_gpu(args.front, tile * tile_rows);
      for (uint64_t i = t0; i < t1; ++i) {
        body(tile, i == t0 || tile == 0);
        if (++tile == n_tiles) tile = 0;
      }
      cur = nxt;
    } while (first_tile(cur) < n_tiles);
    return;
  }
  const uint64_t warps_total = (uint64_t)gridDim.x * (blockDim.x >> 5);
  const uint64_t warp_id = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if constexpr (RANGES == 0) {
    for (uint64_t tile = warp_id; tile < n_tiles; tile += warps_total) body(tile, false);
  } else {
    const uint64_t n_blocks = (n_tiles + WB - 1) / WB;
    for (uint64_t blk = warp_id; blk < n_blocks; blk += warps_total) {
      const uint64_t t0 = blk * WB;
      const uint64_t t1 = t0 + WB < n_tiles ? t0 + WB : n_tiles;
      for (uint64_t tile = t0; tile < t1; ++tile) body(tile, tile == t0);
    }
  }
}

template <int RANGES>
struct StbRowMap {
  uint32_t rlo;
  bool fresh;
  __device__ __forceinline__ void restart() { fresh = true; }
  // virtual row -> local row: largest idx with vstart[idx] <= v.  A lane's virtual rows only
  // grow inside a block: search once, then step to the next range(s).
  __device__ __forceinline__ uint32_t map(const ScanArgs &a, uint64_t v) {
    if constexpr (RANGES == 0) return (uint32_t)v;
    else {
      if (fresh) {
        uint32_t lo = 0, hi = a.n_ranges;
        while (hi - lo > 1) {
          const uint32_t mid = (lo + hi) >> 1;
          if (__ldg(a.vstart + mid) <= v) lo = mid; else hi = mid;
        }
        rlo = lo;
        fresh = false;
      } else {
        while (rlo + 1 < a.n_ranges && __ldg(a.vstart + rlo + 1) <= v) ++rlo;
      }
      return (uint32_t)(__ldg(a.rbegin + rlo) + (v - __ldg(a.vstart + rlo)));
    }
  }
};

// fixed-order ||q||^2 of a lane's 8 float4 + 8-lane group reduction; classifies the query
struct StbQueryNorm { float rq; bool q_zero, q_bad; };
__device__ __forceinline__ StbQueryNorm stb_query_norm(const float4 (&q)[8]) {
  float qx = 0.f, qy = 0.f, qz = 0.f, qw = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    qx = fmaf(q[i].x, q[i].x, qx); qy = fmaf(q[i].y, q[i].y, qy);
    qz = fmaf(q[i].z, q[i].z, qz); qw = fmaf(q[i].w, q[i].w, qw);
  }
  float b2 = (qx + qy) + (qz + qw);
  b2 += __shfl_xor_sync(0xffffffffu, b2, 4);
  b2 += __shfl_xor_sync(0xffffffffu, b2, 2);
  b2 += __shfl_xor_sync(0xffffffffu, b2, 1);
  // b2 == 0 in fp32 is either a true zero vector or an underflowed tiny one
  bool q_any = false;
#pragma unroll
  for (int i = 0; i < 8; ++i)
    q_any |= (q[i].x != 0.f) | (q[i].y != 0.f) | (q[i].z != 0.f) | (q[i].w != 0.f);
  q_any = __any_sync(0xffffffffu, q_any);   // all four groups hold the same query
  StbQueryNorm r;
  r.q_zero = (b2 == 0.f) && !q_any;
  r.q_bad = !r.q_zero && !(b2 >= 1e-30f && b2 <= 1e30f);  // NaN/inf/denormal/underflow
  r.rq = r.q_zero ? 0.f : rsqrtf(b2);
  return r;
}

// Approximate-cosine scan over the f32 rows.  Calls sink(score, local_row) once per 4*U-row
// tile with a warp-uniform control flow; lanes that do not represent a row pass -inf.
template <int U, int RANGES, class Sink>
__device__ __forceinline__ void stb_scan_rows(const ScanArgs &args, Sink &sink) {
  const int lane = threadIdx.x & 31;
  const int g = lane >> 3;   // row group inside the warp
  const int j = lane & 7;    // 16-byte column slot inside the group
  // query slice of this lane: float4 index j + 8*i
  float4 q[8];
  const float4 *q4 = reinterpret_cast<const float4 *>(args.q);
#pragma unroll
  for (int i = 0; i < 8; ++i) q[i] = __ldg(q4 + j + 8 * i);
  const StbQueryNorm qn = stb_query_norm(q);
  const bool q_zero = qn.q_zero, q_bad = qn.q_bad;
  const float rq = qn.rq;

  constexpr uint64_t tile_rows = 4 * U;
  const uint64_t n_tiles = (args.n_virtual + tile_rows - 1) / tile_rows;
  StbRowMap<RANGES> rmap;
  rmap.restart();
  stb_for_each_tile<RANGES, 64 / (4 * U)>(args, n_tiles, tile_rows, [&](uint64_t tile, bool first) {
    if (first) rmap.restart();
    float4 a[U][8];
    uint32_t row[U];
    bool valid[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      uint64_t v = tile * tile_rows + (uint64_t)(u * 4 + g);
      valid[u] = v < args.n_virtual;
      uint64_t vc = valid[u] ? v : (args.n_virtual - 1);
      row[u] = rmap.map(args, vc);
      const float4 *p = args.rows + (size_t)row[u] * STB_ROW_F4 + j;
#pragma unroll
      for (int i = 0; i < 8; ++i) a[u][i] = stb_ld_stream(p + 8 * i);
    }
    float sc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float dx = 0.f, dy = 0.f, dz = 0.f, dw = 0.f;
      float nx = 0.f, ny = 0.f, nz = 0.f, nw = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        dx = fmaf(a[u][i].x, q[i].x, dx); dy = fmaf(a[u][i].y, q[i].y, dy);
        dz = fmaf(a[u][i].z, q[i].z, dz); dw = fmaf(a[u][i].w, q[i].w, dw);
        nx = fmaf(a[u][i].x, a[u][i].x, nx); ny = fmaf(a[u][i].y, a[u][i].y, ny);
        nz = fmaf(a[u][i].z, a[u][i].z, nz); nw = fmaf(a[u][i].w, a[u][i].w, nw);
      }
      float ab = (dx + dy) + (dz + dw);
      float a2 = (nx + ny) + (nz + nw);
      ab += __shfl_xor_sync(0xffffffffu, ab, 4);
      a2 += __shfl_xor_sync(0xffffffffu, a2, 4);
      ab += __shfl_xor_sync(0xffffffffu, ab, 2);
      a2 += __shfl_xor_sync(0xffffffffu, a2, 2);
      ab += __shfl_xor_sync(0xffffffffu, ab, 1);
      a2 += __shfl_xor_sync(0xffffffffu, a2, 1);
      float s;
      if (a2 == 0.f) {
        // rare: a true zero row (simsimd rules: d = 0 vs a zero query, else d = 1) or a
        // row so small that its fp32 squared norm underflowed -> forced candidate.
        // All 8 lanes of the group hold the same a2, so the group votes together.
        bool nz = false;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          nz |= (a[u][i].x != 0.f) | (a[u][i].y != 0.f) | (a[u][i].z != 0.f) | (a[u][i].w != 0.f);
        nz = __any_sync(0xffu << (8 * g), nz);
        s = nz ? CUDART_INF_F : (q_zero ? 1.f : 0.f);
      } else if (q_bad || !(a2 >= 1e-30f && a2 <= 1e30f)) s = CUDART_INF_F;  // forced candidate
      else s = ab * rsqrtf(a2) * rq;
      sc[u] = valid[u] ? s : -CUDART_INF_F;
    }
    float s = -CUDART_INF_F;
    uint32_t r = 0;
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (j == u) { s = sc[u]; r = row[u]; }
    sink.template consume<4 * U>(s, r);
  });
}

// Half-width scan (tier "h16"): the same running top-K' selection, but the scores come from the
// 16-bit L2-normalised shadow that K2 uses (512 B per row instead of 1 KiB), so the HBM-bound
// pass moves half the bytes.  The exact f64 re-rank and the completeness proof are unchanged
// except for the margin (STB_SHADOW_SCAN_EPS: only the row is rounded, the query stays f32).
// Shadow layout (batch_scan.cu): tile t = row / 256 -> 4 K-slabs x [256 rows x 128 B],
// 16-byte chunk index XOR (row % 8).  Lane j of a row's 8-lane group reads PHYSICAL chunk
// j ^ (row % 8) of every slab, i.e. LOGICAL chunk j = elements s*64 + 8j .. +8 (s = 0..3), so
// each lane pairs a fixed 32-element slice of the query with every row; the group still
// covers each 128-byte line completely.
__device__ __forceinline__ float2 stb_shadow_pair(uint32_t w) {
#if STB_SHADOW_F16
  return __half22float2(*reinterpret_cast<const __half2 *>(&w));
#else
  return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
#endif
}

template <int U, int RANGES, class Sink>
__device__ __forceinline__ void stb_scan_shadow(const ScanArgs &args, const uint8_t *shadow, Sink &sink) {
  const int lane = threadIdx.x & 31;
  const int g = lane >> 3;   // row group inside the warp
  const int j = lane & 7;    // logical 16-byte chunk of every K-slab
  // query slice: elements s*64 + 8j + e  (s < 4, e < 8) = float4 index s*16 + 2j + {0,1}
  float4 q[8];
  const float4 *q4 = reinterpret_cast<const float4 *>(args.q);
#pragma unroll
  for (int sl = 0; sl < 4; ++sl) { q[2 * sl] = __ldg(q4 + sl * 16 + 2 * j); q[2 * sl + 1] = __ldg(q4 + sl * 16 + 2 * j + 1); }
  const StbQueryNorm qn = stb_query_norm(q);
  const bool q_bad = qn.q_bad;
  const float rq = qn.rq;

  constexpr uint64_t tile_rows = 4 * U;
  const uint64_t n_tiles = (args.n_virtual + tile_rows - 1) / tile_rows;
  StbRowMap<RANGES> rmap;
  rmap.restart();
  stb_for_each_tile<RANGES, 64 / (4 * U)>(args, n_tiles, tile_rows, [&](uint64_t tile, bool first) {
    if (first) rmap.restart();
    uint4 a[U][4];
    uint32_t row[U];
    bool valid[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint64_t v = tile * tile_rows + (uint64_t)(u * 4 + g);
      valid[u] = v < args.n_virtual;
      const uint64_t vc = valid[u] ? v : (args.n_virtual - 1);
      row[u] = rmap.map(args, vc);
      const uint32_t rr = row[u] & 255u;
      const uint8_t *p = shadow + (size_t)(row[u] >> 8) * (size_t)(256 * 512) + (size_t)(rr >> 3) * 1024 + (size_t)(rr & 7u) * 128 +
                         (size_t)((j ^ (int)(rr & 7u)) * 16);
#pragma unroll
      for (int sl = 0; sl < 4; ++sl) {
        const float4 t = stb_ld_stream(reinterpret_cast<const float4 *>(p + (size_t)sl * (256 * 128)));
        a[u][sl] = make_uint4(__float_as_uint(t.x), __float_as_uint(t.y), __float_as_uint(t.z), __float_as_uint(t.w));
      }
    }
    float sc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float dx = 0.f, dy = 0.f, dz = 0.f, dw = 0.f;
#pragma unroll
      for (int sl = 0; sl < 4; ++sl) {
        const float2 e0 = stb_shadow_pair(a[u][sl].x), e1 = stb_shadow_pair(a[u][sl].y);
        const float2 e2 = stb_shadow_pair(a[u][sl].z), e3 = stb_shadow_pair(a[u][sl].w);
        dx = fmaf(e0.x, q[2 * sl].x, dx); dy = fmaf(e0.y, q[2 * sl].y, dy);
        dz = fmaf(e1.x, q[2 * sl].z, dz); dw = fmaf(e1.y, q[2 * sl].w, dw);
        dx = fmaf(e2.x, q[2 * sl + 1].x, dx); dy = fmaf(e2.y, q[2 * sl + 1].y, dy);
        dz = fmaf(e3.x, q[2 * sl + 1].z, dz); dw = fmaf(e3.y, q[2 * sl + 1].w, dw);
      }
      float ab = (dx + dy) + (dz + dw);
      ab += __shfl_xor_sync(0xffffffffu, ab, 4);
      ab += __shfl_xor_sync(0xffffffffu, ab, 2);
      ab += __shfl_xor_sync(0xffffffffu, ab, 1);
      // the shadow row is already unit-norm (zero rows stay zero: score 0 = distance 1)
      const float s = q_bad ? CUDART_INF_F : ab * rq;
      sc[u] = valid[u] ? s : -CUDART_INF_F;
    }
    float s = -CUDART_INF_F;
    uint32_t r = 0;
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (j == u) { s = sc[u]; r = row[u]; }
    sink.template consume<4 * U>(s, r);
  });
}

// Quarter-width scan (tier "q8"): candidates come from an 8-bit copy of the corpus -- row x is
// L2-normalised in fp32 (x^), scaled by its own s = max|x^_i| / 127 and rounded to int8
// (stb_q8_build_kernel): 256 B + one f32 scale per row = 260 B instead of 1 KiB.  The query is
// normalised and quantised to 16 bits per component (q16 = rint(q^ * S), S = 32639 / max|q^_i|),
// split into two signed bytes (q16 = 256 * hi + lo) so the dot product is two dp4a chains,
// exact in int32 (|dot| <= 127 * 32639 * 256 < 2^31).  What the list ranks by is not the
// approximate cosine a = s * dot / S but an UPPER BOUND of the exact one:
//     |c - a| <= sum_i |q~_i| |x^_i - s x8_i|  +  sum_i |q^_i - q~_i| |x^_i|
//             <= s * (0.5 + 3e-5) * ||q16||_1 / S   +   (0.6 / S) * ||x^||_1 ,  ||x^||_1 <= 16.001
//     u = s * (dot / S + 0.50025 * ||q16||_1 / S) + 9.7 / S          >=  c - 1e-5
// (||q16||_1 is an exact integer sum).  Every row dropped from the lists has u <= u_min, hence
// exact cosine <= u_min + 1e-5: the completeness proof is the f32 one with the per-row error
// term folded into the score, so rows with a large scale are promoted instead of widening a
// global margin.  A zero or unscorable query makes every score +inf: the proof fails and the
// caller falls through to the f32 tiers.
// max |q^_i| of the lane's 8 float4 (the 8 lanes of a group hold the whole query)
__device__ __forceinline__ float stb_query_amax(const float4 (&q)[8], float rq) {
  float amax = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    amax = fmaxf(amax, fmaxf(fmaxf(fabsf(q[i].x), fabsf(q[i].y)), fmaxf(fabsf(q[i].z), fabsf(q[i].w))));
  }
  amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 4));
  amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
  amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
  return amax * rq;
}

// The q8 tier's query side for lane j of a row group: q16 split into two signed bytes for the row
// bytes [16j, 16j+16) and [128+16j, 128+16j+16), plus the terms of the upper bound.  Called by the
// full warp (group reductions).
struct StbQ8Query {
  uint32_t hi[8], lo[8];
  float inv_S, h_l1, e_q;
  bool unusable;
  __device__ __forceinline__ void load(const float *qp, int j) {
    float4 q[8];
    const float4 *q4 = reinterpret_cast<const float4 *>(qp);
#pragma unroll
    for (int i = 0; i < 4; ++i) { q[i] = __ldg(q4 + 4 * j + i); q[4 + i] = __ldg(q4 + 32 + 4 * j + i); }
    const StbQueryNorm qn = stb_query_norm(q);
    const float amax = stb_query_amax(q, qn.rq);            // max |q^_i|
    unusable = qn.q_zero || qn.q_bad || !(amax > 0.f && amax <= 1.0001f);
    const float S = unusable ? 1.f : 32639.0f / amax;
    const float qs = qn.rq * S;
    int l1 = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float f[4] = {q[i].x, q[i].y, q[i].z, q[i].w};
      uint32_t hw = 0, lw = 0;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        int v = unusable ? 0 : __float2int_rn(f[e] * qs);
        v = max(-32639, min(32639, v));
        l1 += abs(v);
        const int l = ((v + 128) & 255) - 128;              // signed low byte
        const int h = (v - l) >> 8;                         // exact: v - l is a multiple of 256
        hw |= (uint32_t)(h & 255) << (8 * e);
        lw |= (uint32_t)(l & 255) << (8 * e);
      }
      hi[i] = hw; lo[i] = lw;
    }
    l1 += __shfl_xor_sync(0xffffffffu, l1, 4);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    inv_S = 1.0f / S;
    h_l1 = 0.50025f * (float)l1 * inv_S;                    // (0.5 + 3e-5 + fp slack) * ||q~||_1
    e_q = 9.7f * inv_S;
  }
  // upper bound of the exact cosine of the row whose 32 code bytes this lane holds (full warp: group reduction)
  __device__ __forceinline__ float bound(const uint4 &a0, const uint4 &a1, float scale) const {
    int dh = 0, dl = 0;
    const uint32_t w[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      dh = __dp4a((int)w[i], (int)hi[i], dh);
      dl = __dp4a((int)w[i], (int)lo[i], dl);
    }
    int dot = dh * 256 + dl;
    dot += __shfl_xor_sync(0xffffffffu, dot, 4);
    dot += __shfl_xor_sync(0xffffffffu, dot, 2);
    dot += __shfl_xor_sync(0xffffffffu, dot, 1);
    return unusable ? CUDART_INF_F : fmaf(scale, fmaf((float)dot, inv_S, h_l1), e_q);
  }
};

template <int U, int RANGES, class Sink>
__device__ __forceinline__ void stb_scan_q8(const ScanArgs &args, const uint8_t *q8, const float *q8_scale, Sink &sink) {
  const int lane = threadIdx.x & 31;
  const int g = lane >> 3;   // row group inside the warp
  const int j = lane & 7;    // this lane reads row bytes [16j, 16j+16) and [128+16j, 128+16j+16)
  StbQ8Query qq;
  qq.load(args.q, j);

  constexpr uint64_t tile_rows = 4 * U;
  const uint64_t n_tiles = (args.n_virtual + tile_rows - 1) / tile_rows;
  StbRowMap<RANGES> rmap;
  rmap.restart();
  stb_for_each_tile<RANGES, 2>(args, n_tiles, tile_rows, [&](uint64_t tile, bool first) {
    if (first) rmap.restart();
    uint4 a[U][2];
    float sc_row[U];
    uint32_t row[U];
    bool valid[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint64_t v = tile * tile_rows + (uint64_t)(u * 4 + g);
      valid[u] = v < args.n_virtual;
      const uint64_t vc = valid[u] ? v : (args.n_virtual - 1);
      row[u] = rmap.map(args, vc);
      const uint8_t *p = q8 + (size_t)row[u] * 256 + (size_t)j * 16;
      const float4 t0 = stb_ld_stream(reinterpret_cast<const float4 *>(p));
      const float4 t1 = stb_ld_stream(reinterpret_cast<const float4 *>(p + 128));
      a[u][0] = make_uint4(__float_as_uint(t0.x), __float_as_uint(t0.y), __float_as_uint(t0.z), __float_as_uint(t0.w));
      a[u][1] = make_uint4(__float_as_uint(t1.x), __float_as_uint(t1.y), __float_as_uint(t1.z), __float_as_uint(t1.w));
      sc_row[u] = __ldg(q8_scale + row[u]);                 // 8 lanes, one address
    }
    float sc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const float s = qq.bound(a[u][0], a[u][1], sc_row[u]);
      sc[u] = valid[u] ? s : -CUDART_INF_F;
    }
    float s = -CUDART_INF_F;
    uint32_t r = 0;
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (j == u) { s = sc[u]; r = row[u]; }
    sink.template consume<4 * U>(s, r);
  });
}

// dp4a with unsigned bytes in a and signed bytes in b (PTX dp4a.u32.s32)
__device__ __forceinline__ int stb_dp4a_us(uint32_t a, uint32_t b, int c) {
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// Coarse pass in front of the q8 tier ("q4"): a 4-bit copy, 128 B of codes + (s4, r) per row = 136 B.
// Row model (stb_q4_build_kernel): x~_i = s4 * (c_i - 7.5), c_i in [0, 15] (16 mid-rise levels) on the
// fp32-normalised row x^, with s4 picked per row to minimise r = ||x^ - x~||_2, stored rounded up.
// Byte b of the row's 32-bit word l holds c[8l+b] in its low nibble and c[8l+4+b] in its high one, so
// lane j of a row group reads one 16-byte chunk = elements 32j .. 32j+31, and the query, quantised per
// call to int8 (q8_i = rint(q^_i * S8), S8 = 127 / max|q^_i|), lines up byte for byte with the two
// nibble planes: two masks and two dp4a per word, exact in int32.  With q~ = q8 / S8 and
// f = q^ - q~, Cauchy-Schwarz gives for the exact cosine c = q^ . x^:
//     c = q~ . x~ + q~ . (x^ - x~) + f . x^  <=  q~ . x~ + r (1 + ||f||) + ||f||
//     q~ . x~ = s4 * (2 dot - 15 sum(q8)) / (2 S8)          (integer part exact)
//     u4 = s4 * (2 dot - 15 sum(q8)) / (2 S8) + r (1 + ||f||) + ||f|| + 4e-6   >=  c - 1e-5
// (||f|| is evaluated in fp32 and inflated; the fp32 normalisations of row and query stay inside the
// 1e-5, as for q8).  u4 is ~0.1 wide against q8's ~0.01, so it only ranks: the warps keep their best
// 64 by u4, the CTA re-scores the few that can matter with the q8 codes (stb_scan_topk_kernel, SRC 3)
// and the tree above sees q8 bounds only.
template <int U, int RANGES, class Sink>
__device__ __forceinline__ void stb_scan_q4(const ScanArgs &args, const uint8_t *q4, const float2 *q4_sr, Sink &sink) {
  static_assert(U % 8 == 0, "a lane carries rows u = j + 8h to the sink");
  const int lane = threadIdx.x & 31;
  const int g = lane >> 3;   // row group inside the warp
  const int j = lane & 7;    // this lane reads row bytes [16j, 16j+16) = elements 32j .. 32j+31
  float4 q[8];
  const float4 *qf4 = reinterpret_cast<const float4 *>(args.q);
#pragma unroll
  for (int i = 0; i < 8; ++i) q[i] = __ldg(qf4 + 8 * j + i);
  const StbQueryNorm qn = stb_query_norm(q);
  const float amax = stb_query_amax(q, qn.rq);
  const bool q_unusable = qn.q_zero || qn.q_bad || !(amax > 0.f && amax <= 1.0001f);
  const float S = q_unusable ? 1.f : 127.0f / amax;
  const float qs = qn.rq * S, inv_S = 1.0f / S;
  // qw[2i] pairs with the low nibbles of word i (elements 32j+8i .. +3), qw[2i+1] with the high ones
  uint32_t qw[8];
  int qsum = 0;
  float f2 = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float f[4] = {q[i].x, q[i].y, q[i].z, q[i].w};
    uint32_t w = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      int v = q_unusable ? 0 : __float2int_rn(f[e] * qs);
      v = max(-127, min(127, v));
      qsum += v;
      const float d = fmaf(-(float)v, inv_S, f[e] * qn.rq);   // f_i = q^_i - q~_i
      f2 = fmaf(d, d, f2);
      w |= (uint32_t)(v & 255) << (8 * e);
    }
    qw[i] = w;
  }
  qsum += __shfl_xor_sync(0xffffffffu, qsum, 4);
  qsum += __shfl_xor_sync(0xffffffffu, qsum, 2);
  qsum += __shfl_xor_sync(0xffffffffu, qsum, 1);
  f2 += __shfl_xor_sync(0xffffffffu, f2, 4);
  f2 += __shfl_xor_sync(0xffffffffu, f2, 2);
  f2 += __shfl_xor_sync(0xffffffffu, f2, 1);
  const float nf = sqrtf(f2) * 1.001f + 2e-6f;              // ||f||, rounded up (each f_i is within 1 ulp)
  const float coef = 0.5f * inv_S;
  const int qsum15 = 15 * qsum;
  const float r_mul = 1.0f + nf, slack = nf + 4e-6f;

  constexpr uint64_t tile_rows = 4 * U;
  const uint64_t n_tiles = (args.n_virtual + tile_rows - 1) / tile_rows;
  StbRowMap<RANGES> rmap;
  rmap.restart();
  stb_for_each_tile<RANGES, 1>(args, n_tiles, tile_rows, [&](uint64_t tile, bool first) {
    if (first) rmap.restart();
    uint4 a[U];
    uint32_t own_row[U / 8];   // the rows this lane hands to the sink: u = j + 8h
    const uint64_t v0 = tile * tile_rows;
    const bool full = RANGES == 0 && v0 + tile_rows <= args.n_virtual;   // warp-uniform
    if (full) {
      // every row exists and is its own local row: one base address, the rows at immediate offsets
      const float4 *p = reinterpret_cast<const float4 *>(q4 + (size_t)(v0 + g) * 128 + (size_t)j * 16);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float4 t = stb_ld_stream(p + u * 32);   // + 4 rows of 128 B
        a[u] = make_uint4(__float_as_uint(t.x), __float_as_uint(t.y), __float_as_uint(t.z), __float_as_uint(t.w));
      }
#pragma unroll
      for (int h = 0; h < U / 8; ++h) own_row[h] = (uint32_t)(v0 + (uint64_t)((8 * h + j) * 4 + g));
    } else {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const uint64_t v = v0 + (uint64_t)(u * 4 + g);
        const uint64_t vc = v < args.n_virtual ? v : (args.n_virtual - 1);
        const uint32_t row = rmap.map(args, vc);
        const float4 t = stb_ld_stream(reinterpret_cast<const float4 *>(q4 + (size_t)row * 128 + (size_t)j * 16));
        a[u] = make_uint4(__float_as_uint(t.x), __float_as_uint(t.y), __float_as_uint(t.z), __float_as_uint(t.w));
        if ((u & 7) == j) own_row[u >> 3] = row;
      }
    }
#pragma unroll
    for (int h = 0; h < U / 8; ++h) {
      const float2 sr = __ldg(q4_sr + own_row[h]);
      // x[uu] = 16 * this lane's part of the dot of row u = 8h + uu: the high nibbles are dotted in place
      // (w & 0xF0F0F0F0 = 16 * code, unsigned bytes against the signed query bytes), so no shift per word
      int x[8];
#pragma unroll
      for (int uu = 0; uu < 8; ++uu) {
        const uint4 &w = a[8 * h + uu];
        const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
        int dl = 0, dh = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          dl = __dp4a((int)(ww[i] & 0x0f0f0f0fu), (int)qw[2 * i], dl);
          dh = stb_dp4a_us(ww[i] & 0xf0f0f0f0u, qw[2 * i + 1], dh);
        }
        x[uu] = dh + 16 * dl;
      }
      // transpose-reduce over the 8 lanes of the group by recursive halving: at each step a lane keeps the
      // half of its rows whose index agrees with j on that bit and adds its partner's copy of the same rows,
      // so lane j ends with the full sum of row uu = j (7 shuffles for 8 rows instead of 24)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool hi = j & 4;
        const int keep = hi ? x[i + 4] : x[i], send = hi ? x[i] : x[i + 4];
        x[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
      }
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const bool hi = j & 2;
        const int keep = hi ? x[i + 2] : x[i], send = hi ? x[i] : x[i + 2];
        x[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
      }
      {
        const bool hi = j & 1;
        const int keep = hi ? x[1] : x[0], send = hi ? x[0] : x[1];
        x[0] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
      }
      const int own_dot = x[0] >> 4;                      // exact: x[0] = 16 * dot
      float s = q_unusable ? CUDART_INF_F : fmaf(sr.x * coef, (float)(2 * own_dot - qsum15), fmaf(sr.y, r_mul, slack));
      if (!full && v0 + (uint64_t)((8 * h + j) * 4 + g) >= args.n_virtual) s = -CUDART_INF_F;
      sink.template consume<32>(s, own_row[h]);
    }
  });
}

// q4 builder: one warp per row, lane l owns elements 8l .. 8l+7 and writes word l of the row's codes.
// Normalisation and the bad-row flag are stb_q8_build_kernel's.  s4 = t * max|x^| / 7.5 with t from a
// fixed set: the one with the smallest ||x^ - x~||_2 (fp32, first on ties).  r is that norm for the
// stored s4 and codes, evaluated in f64 and rounded up to f32 (a proof input).  Zero rows: s4 = r = 0.
#define STB_Q4_T_STEPS 8
__global__ void __launch_bounds__(256)
stb_q4_build_kernel(const float4 *__restrict__ rows, uint64_t first_row, uint64_t n_rows, uint8_t *__restrict__ out,
                    float2 *__restrict__ sr, int *bad_flag) {
  const int lane = threadIdx.x & 31;
  const uint64_t row = first_row + (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const float4 v0 = __ldg(rows + row * STB_ROW_F4 + 2 * lane);
  const float4 v1 = __ldg(rows + row * STB_ROW_F4 + 2 * lane + 1);
  float ss = v0.x * v0.x + v0.y * v0.y + v0.z * v0.z + v0.w * v0.w + v1.x * v1.x + v1.y * v1.y + v1.z * v1.z + v1.w * v1.w;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
  float inv = 0.f;
  if (ss != 0.f) {
    if (!(ss >= 1e-30f && ss <= 1e30f)) { if (lane == 0) atomicExch(bad_flag, 1); }   // NaN/inf/extreme
    else inv = rsqrtf(ss);
  } else {
    const bool nz = (v0.x != 0.f) | (v0.y != 0.f) | (v0.z != 0.f) | (v0.w != 0.f) | (v1.x != 0.f) | (v1.y != 0.f) |
                    (v1.z != 0.f) | (v1.w != 0.f);
    if (__any_sync(0xffffffffu, nz) && lane == 0) atomicExch(bad_flag, 1);             // underflowed tiny row
  }
  const float x[8] = {v0.x * inv, v0.y * inv, v0.z * inv, v0.w * inv, v1.x * inv, v1.y * inv, v1.z * inv, v1.w * inv};
  float am = 0.f;
#pragma unroll
  for (int e = 0; e < 8; ++e) am = fmaxf(am, fabsf(x[e]));
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) am = fmaxf(am, __shfl_xor_sync(0xffffffffu, am, off));
  auto code = [](float xe, float inv_s) { return max(0, min(15, __float2int_rn(fmaf(xe, inv_s, 7.5f)))); };
  float s = 0.f, best = CUDART_INF_F;
  if (am > 0.f) {
    for (int k = 0; k < STB_Q4_T_STEPS; ++k) {
      const float sk = (0.65f + 0.05f * (float)k) * am * (1.0f / 7.5f);
      const float inv_s = 1.0f / sk;
      float err = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float d = x[e] - sk * ((float)code(x[e], inv_s) - 7.5f);
        err = fmaf(d, d, err);
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) err += __shfl_xor_sync(0xffffffffu, err, off);
      if (err < best) { best = err; s = sk; }
    }
  }
  const float inv_s = s > 0.f ? 1.0f / s : 0.f;
  uint32_t w = 0;
  double e2 = 0.0;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = s > 0.f ? code(x[e], inv_s) : 8;
    w |= (uint32_t)c << (e < 4 ? 8 * e + 0 : 8 * (e - 4) + 4);
    const double d = (double)x[e] - (double)s * ((double)c - 7.5);   // s * (c - 7.5) is exact in f64
    e2 = fma(d, d, e2);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) e2 += __shfl_xor_sync(0xffffffffu, e2, off);
  reinterpret_cast<uint32_t *>(out + row * 128)[lane] = w;
  // f64 sum and sqrt are within a few 1e-16 relative: the 1e-9 margin and upward rounding keep r >= the true norm
  if (lane == 0) sr[row] = make_float2(s, s > 0.f ? __double2float_ru(sqrt(e2) * (1.0 + 1e-9)) : 0.f);
}

int stb_launch_q4_build(stb_ctx *ctx, const float *rows_dev, uint64_t first_row, uint64_t n_rows, uint8_t *out,
                        float2 *sr, int *bad_flag_dev) {
  if (first_row >= n_rows) return STB_OK;
  const unsigned blocks = (unsigned)((n_rows - first_row + 7) / 8);
  stb_q4_build_kernel<<<blocks, 256, 0, ctx->stream>>>(reinterpret_cast<const float4 *>(rows_dev), first_row, n_rows, out, sr,
                                                       bad_flag_dev);
  STB_CUDA(cudaGetLastError());
  ctx->kernel_launches++;
  return STB_OK;
}

// q8 builder: one warp per row; lane l owns elements 8l .. 8l+7.  Rows whose fp32 squared norm
// is not a normal number set *bad_flag (the tier is then refused for this corpus, like the
// 16-bit shadow); true zero rows get scale 0 and all-zero codes (score = the query's slack).
__global__ void __launch_bounds__(256)
stb_q8_build_kernel(const float4 *__restrict__ rows, uint64_t first_row, uint64_t n_rows, uint8_t *__restrict__ out,
                    float *__restrict__ scale, int *bad_flag) {
  const int lane = threadIdx.x & 31;
  const uint64_t row = first_row + (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const float4 v0 = __ldg(rows + row * STB_ROW_F4 + 2 * lane);
  const float4 v1 = __ldg(rows + row * STB_ROW_F4 + 2 * lane + 1);
  float ss = v0.x * v0.x + v0.y * v0.y + v0.z * v0.z + v0.w * v0.w + v1.x * v1.x + v1.y * v1.y + v1.z * v1.z + v1.w * v1.w;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
  float inv = 0.f;
  if (ss != 0.f) {
    if (!(ss >= 1e-30f && ss <= 1e30f)) { if (lane == 0) atomicExch(bad_flag, 1); }   // NaN/inf/extreme
    else inv = rsqrtf(ss);
  } else {
    const bool nz = (v0.x != 0.f) | (v0.y != 0.f) | (v0.z != 0.f) | (v0.w != 0.f) | (v1.x != 0.f) | (v1.y != 0.f) |
                    (v1.z != 0.f) | (v1.w != 0.f);
    if (__any_sync(0xffffffffu, nz) && lane == 0) atomicExch(bad_flag, 1);             // underflowed tiny row
  }
  const float x[8] = {v0.x * inv, v0.y * inv, v0.z * inv, v0.w * inv, v1.x * inv, v1.y * inv, v1.z * inv, v1.w * inv};
  float am = 0.f;
#pragma unroll
  for (int e = 0; e < 8; ++e) am = fmaxf(am, fabsf(x[e]));
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) am = fmaxf(am, __shfl_xor_sync(0xffffffffu, am, off));
  const float s = am * (1.0f / 127.0f);
  const float inv_s = am > 0.f ? 127.0f / am : 0.f;
  uint32_t w0 = 0, w1 = 0;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int c0 = max(-127, min(127, __float2int_rn(x[e] * inv_s)));
    const int c1 = max(-127, min(127, __float2int_rn(x[4 + e] * inv_s)));
    w0 |= (uint32_t)(c0 & 255) << (8 * e);
    w1 |= (uint32_t)(c1 & 255) << (8 * e);
  }
  *reinterpret_cast<uint2 *>(out + row * 256 + (size_t)lane * 8) = make_uint2(w0, w1);
  if (lane == 0) scale[row] = s;
}

int stb_launch_q8_build(stb_ctx *ctx, const float *rows_dev, uint64_t first_row, uint64_t n_rows, uint8_t *out,
                        float *scale, int *bad_flag_dev) {
  if (first_row >= n_rows) return STB_OK;
  const unsigned blocks = (unsigned)((n_rows - first_row + 7) / 8);
  stb_q8_build_kernel<<<blocks, 256, 0, ctx->stream>>>(reinterpret_cast<const float4 *>(rows_dev), first_row, n_rows, out, scale,
                                                       bad_flag_dev);
  STB_CUDA(cudaGetLastError());
  ctx->kernel_launches++;
  return STB_OK;
}

// ---------------------------------------------------------------- top-K' sink ---
template <int E>
struct TopSink {
  float ls[E];
  uint32_t lr[E];
  float thr;   // min score in the list (warp-uniform); -inf while not full
  int lane;
  int fill;    // slots bulk-filled so far (warp-uniform); 32*E once the fill phase is over
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int e = 0; e < E; ++e) { ls[e] = -CUDART_INF_F; lr[e] = 0xffffffffu; }
    thr = -CUDART_INF_F;
    lane = threadIdx.x & 31;
    fill = 0;
  }
  __device__ __forceinline__ float warp_min(float m) const {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, off));
    return m;
  }
  __device__ __forceinline__ void insert(float cs, uint32_t cr) {
    float m = ls[0];
    int mi = 0;
#pragma unroll
    for (int e = 1; e < E; ++e)
      if (ls[e] < m) { m = ls[e]; mi = e; }
    unsigned owners = __ballot_sync(0xffffffffu, m == thr);
    int owner = __ffs(owners) - 1;
    if (lane == owner) {
#pragma unroll
      for (int e = 0; e < E; ++e)
        if (e == mi) { ls[e] = cs; lr[e] = cr; }
    }
    m = ls[0];
#pragma unroll
    for (int e = 1; e < E; ++e) m = fminf(m, ls[e]);
    thr = warp_min(m);
  }
  // Bulk fill: while the list has room and tiles are complete, the tile's rows are
  // gathered straight into the free slots (slot -> lane slot%32, entry slot/32) with two
  // shuffles, instead of one min-reduction per row.  ROWS = rows a full tile carries,
  // sitting in lanes g*8+u (g < 4, u < ROWS/4).
  template <int ROWS>
  __device__ __forceinline__ bool try_fill(float s, uint32_t r, unsigned vmask) {
    constexpr int KP = 32 * E;
    constexpr int UU = ROWS / 4;
    unsigned full = 0u;
#pragma unroll
    for (int g = 0; g < 4; ++g)
#pragma unroll
      for (int u = 0; u < UU; ++u) full |= 1u << (g * 8 + u);
    if (fill >= KP) return false;
    if (vmask != full || fill + ROWS > KP) {      // ragged tile: leave the fill phase for good
      fill = KP;
      return false;
    }
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int d = e * 32 + lane - fill;          // which row of the tile this slot takes
      const bool want = (d >= 0 && d < ROWS);
      const int src = want ? ((d / UU) * 8 + (d % UU)) : 0;
      const float cs = __shfl_sync(0xffffffffu, s, src);
      const uint32_t cr = __shfl_sync(0xffffffffu, r, src);
      if (want) { ls[e] = cs; lr[e] = cr; }
    }
    fill += ROWS;
    if (fill >= KP) {
      float m = ls[0];
#pragma unroll
      for (int e = 1; e < E; ++e) m = fminf(m, ls[e]);
      thr = warp_min(m);
    }
    return true;
  }
  template <int ROWS>
  __device__ __forceinline__ void consume(float s, uint32_t r) {
    if (fill < 32 * E) {
      const unsigned vmask = __ballot_sync(0xffffffffu, s > -CUDART_INF_F);
      if (try_fill<ROWS>(s, r, vmask)) return;
    }
    (*this)(s, r);
  }
  __device__ __forceinline__ void operator()(float s, uint32_t r) {
    unsigned mask = __ballot_sync(0xffffffffu, s > thr);
    while (mask) {
      int src = __ffs(mask) - 1;
      mask &= mask - 1;
      float cs = __shfl_sync(0xffffffffu, s, src);
      uint32_t cr = __shfl_sync(0xffffffffu, r, src);
      if (cs > thr) insert(cs, cr);
    }
  }
};

__device__ __forceinline__ void stb_cta_sort_keys(uint64_t *keys, int n) {
  static_assert(STB_SCAN_THREADS == 256, "register sort assumes 256 threads");
  if (n <= 256) stb_cta_sort_keys_t<1>(keys, n);
  else stb_cta_sort_keys_t<4>(keys, n);
}

struct TopkArgs {
  ScanArgs scan;
  uint64_t row_base;
  uint64_t *keys;            // sorted best-KP lists of every tree level
  unsigned int *counters;    // one arrival ticket per tree group, all levels
  stb_hit *out_hits;
  uint32_t *out_status;
  uint32_t top_k;
  StbXchgArgs xchg;          // world == 0: no cross-GPU exchange
  unsigned long long *dbg;   // STB_TAIL_TIMING builds only: phase timestamps (ns)
  const uint8_t *shadow;     // SRC == 1: 16-bit normalised corpus shadow (UMMA tile layout)
  uint32_t early_trigger;    // overlapped launch: release the dependent launch at kernel start
  const uint8_t *q8;         // SRC == 2, 3: int8 codes [n][256] ...
  const float *q8_scale;     //              ... and per-row scales [n]
  const uint8_t *q4;         // SRC == 3: 4-bit codes [n][128] ...
  const float2 *q4_sr;       //           ... and per-row (s4, r) [n]
};

// SRC 3, after the scan: the CTA's coarse candidates sit in keys[0, c) as (u4, row).  Each is re-scored
// with the q8 codes (StbQ8Query::bound) and its key replaced by min(u4, u8) -- both are upper bounds of
// the exact cosine.  32 row groups of 8 lanes, 4 rows per group per pass (<= 512 candidates).
__device__ __forceinline__ void stb_q8_refine(const TopkArgs &args, uint64_t *keys, int c) {
  constexpr int R = 4;
  const int grp = threadIdx.x >> 3, j = threadIdx.x & 7;
  StbQ8Query qq;
  qq.load(args.scan.q, j);
  for (int base = 0; base < c; base += 32 * R) {           // c is CTA-uniform
    uint4 a[R][2];
    float sc[R];
#pragma unroll
    for (int u = 0; u < R; ++u) {
      const int idx = base + grp + 32 * u;
      a[u][0] = a[u][1] = make_uint4(0u, 0u, 0u, 0u);
      sc[u] = 0.f;
      if (idx < c) {
        const uint32_t row = stb_key_row(keys[idx]);
        const uint4 *p = reinterpret_cast<const uint4 *>(args.q8 + (size_t)row * 256 + (size_t)j * 16);
        a[u][0] = __ldg(p);
        a[u][1] = __ldg(p + 8);
        sc[u] = __ldg(args.q8_scale + row);
      }
    }
#pragma unroll
    for (int u = 0; u < R; ++u) {
      const int idx = base + grp + 32 * u;
      const float u8 = qq.bound(a[u][0], a[u][1], sc[u]);
      if (idx < c && j == 0) {
        const uint64_t key = keys[idx];
        keys[idx] = stb_make_key(fminf(stb_key_score(key), u8), stb_key_row(key));
      }
    }
  }
}

__device__ __forceinline__ unsigned long long stb_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#ifdef STB_TAIL_TIMING
#define STB_T_MIN(i) do { if (threadIdx.x == 0 && args.dbg) atomicMin(args.dbg + (i), stb_globaltimer()); } while (0)
#define STB_T_MAX(i) do { if (threadIdx.x == 0 && args.dbg) atomicMax(args.dbg + (i), stb_globaltimer()); } while (0)
#else
#define STB_T_MIN(i) do { } while (0)
#define STB_T_MAX(i) do { } while (0)
#endif

// ---- peer-memory exchange (fused K1 -> all-gather -> K4) ------------------------------
// Every rank owns one exchange buffer (cudaMalloc, mapped into all peers through CUDA
// IPC or peer access):  flags[S][world] u64 | status[S][world] u32 | hits[S][world][max_k].
// The final CTA of rank r stores its k hits into slot (seq % S), lane r of EVERY peer's
// buffer over NVLink, fences, release-stores seq into the peers' flags, then
// acquire-spins on its own flags until all `world` lanes carry seq, and merges.
__device__ __forceinline__ void stb_st_release_sys(unsigned long long *p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long stb_ld_acquire_sys(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long *stb_x_flags(const StbXchgArgs &x, int peer) {
  return reinterpret_cast<unsigned long long *>(x.base[peer]);
}
__device__ __forceinline__ uint32_t *stb_x_status(const StbXchgArgs &x, int peer) {
  return reinterpret_cast<uint32_t *>(x.base[peer] + (size_t)STB_XCHG_SLOTS * x.world * 8);
}
__device__ __forceinline__ stb_hit *stb_x_hits(const StbXchgArgs &x, int peer) {
  return reinterpret_cast<stb_hit *>(x.base[peer] + (size_t)STB_XCHG_SLOTS * x.world * 16);
}

// Sort the first `c` keys of skeys (padded with INVALID to a power of two >= KP).
__device__ __forceinline__ int stb_pad_and_sort(uint64_t *skeys, int c, int min_n) {
  int n = min_n;
  while (n < c) n <<= 1;
  const int span = n <= 256 ? 256 : STB_SORT_CAP;   // the register sort writes back its whole span
  for (int i = c + threadIdx.x; i < span; i += blockDim.x) skeys[i] = STB_KEY_INVALID;
  __syncthreads();
  stb_cta_sort_keys(skeys, n);
  return n;
}

#define STB_RR_STRIDE 260   // floats per staged row (1 KiB + 16 B pad: conflict-free LDS.128)

// E: 32*E candidates per warp / CTA / inner tree list.  EF: the ROOT of the merge tree (the CTA
// itself when the grid is one CTA) keeps 32*EF >= 32*E candidates for the exact re-rank.
// EF > E lets a tier with a wide error term (q8) re-rank 128 rows while every level below the
// root moves 32-key lists -- the tail costs what the f32 tier's does.  Completeness is tracked
// explicitly: every node that drops keys publishes the best score it dropped (<= its last kept
// key), the bounds are max-reduced up the tree, and the proof compares the k-th exact distance
// with that bound instead of "the K'-th key of one uniform list".
template <int E, int U, int RANGES, int SRC = 0, int EF = E>
__global__ void __launch_bounds__(STB_SCAN_THREADS, STB_SCAN_MINB)
stb_scan_topk_kernel(const TopkArgs args) {
  // SRC 0: scores from the f32 rows; SRC 1: from the 16-bit shadow (wider proof margin);
  // SRC 2: upper bounds of the exact cosine from the int8 copy (margin folded into the score);
  // SRC 3: 4-bit coarse bounds in the warps, re-scored with the int8 copy in the CTA (stb_scan_q4)
  constexpr double kScoreEps = SRC == 1 ? STB_SHADOW_SCAN_EPS : (SRC >= 2 ? STB_Q8_SCAN_EPS : STB_SCORE_EPS);
  constexpr uint32_t kTierReported = SRC == 3 ? STB_TIER_Q8 : SRC;   // the status word knows tiers 0..2
  // SRC 3: the warps rank by the ~0.1-wide 4-bit bound, so their lists are 64 long (room for the rows that
  // can reach c_k, DESIGN.md section 5); the CTA re-scores them with q8 and publishes KP keys like every tier
  constexpr int ES = SRC == 3 ? 2 : E;
  constexpr int KP = 32 * E;          // list length below the root
  constexpr int KF = 32 * EF;         // candidates the root keeps
  constexpr int KPS = KP + 1;         // published list stride: KP keys + the node's drop bound
  static_assert(EF >= E && 8 * 32 * ES <= STB_SORT_CAP && KF <= STB_SORT_CAP / 2, "list sizes");
  __shared__ uint64_t skeys[STB_SORT_CAP];
  __shared__ unsigned int s_T, s_cnt, s_ticket, s_bound, s_nin;
  __shared__ unsigned long long s_T64;
  __shared__ double sqd[STB_D];                  // query in f64 (exact conversion)
  __shared__ __align__(16) float srows[32 * STB_RR_STRIDE];
  __shared__ double s_d[KF], s_r2[KF], s_q2;
  __shared__ uint64_t s_r[KF];
  __shared__ int s_nv[2];

  STB_T_MIN(0);                      // first CTA starts
  // Overlapped launches (asynchronous entry points): the grid is sized for one CTA per SM and lets the
  // NEXT query's grid in right away, so two scans share the SMs and the ~10 us in which a draining
  // grid leaves HBM idle (CTA merge before exit, launch, ramp-up) are covered by the other scan.
  // Tails stay ordered: everything after the scan sits behind griddepcontrol.wait.
  if (args.early_trigger) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  TopSink<ES> sink;
  sink.init();
  if constexpr (SRC == 3) stb_scan_q4<U, RANGES>(args.scan, args.q4, args.q4_sr, sink);
  else if constexpr (SRC == 2) stb_scan_q8<U, RANGES>(args.scan, args.q8, args.q8_scale, sink);
  else if constexpr (SRC == 1) stb_scan_shadow<U, RANGES>(args.scan, args.shadow, sink);
  else stb_scan_rows<U, RANGES>(args.scan, sink);
  STB_T_MAX(1);                      // last CTA leaves the scan loop
  // Programmatic dependent launch: the scan above reads only the corpus and the query,
  // so the NEXT query's kernel may start streaming as soon as every CTA of this one has
  // left its scan loop; this kernel's merge / re-rank tail then overlaps with it.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  // ---- CTA merge ------------------------------------------------------------------
  // T = max over warps of the warp list minimum is a lower bound of the CTA's KP-th
  // best score (that warp alone holds KP keys >= its minimum), so only keys >= T can
  // matter: compact those (typically ~KP..2KP of the 8*KP) and sort the small set.
  // Drop bounds are ordered scores (stb_f2ord); 0 = "nothing dropped so far".
  const int lane = threadIdx.x & 31;
  const unsigned kOrdNegInf = 0x007fffffu;       // stb_f2ord(-inf): a list that never filled
  if (threadIdx.x == 0) { s_T = 0u; s_cnt = 0u; }
  __syncthreads();
  if (lane == 0) atomicMax(&s_T, stb_f2ord(sink.thr));
  __syncthreads();
  {
    const unsigned T = s_T;
#pragma unroll
    for (int e = 0; e < ES; ++e) {
      const bool take = sink.lr[e] != 0xffffffffu && stb_f2ord(sink.ls[e]) >= T;
      const unsigned m = __ballot_sync(0xffffffffu, take);
      unsigned base = 0u;
      if (lane == 0 && m) base = atomicAdd(&s_cnt, (unsigned)__popc(m));   // <= 8*32*ES <= STB_SORT_CAP
      base = __shfl_sync(0xffffffffu, base, 0);
      if (take) skeys[base + __popc(m & ((1u << lane) - 1u))] = stb_make_key(sink.ls[e], sink.lr[e]);
    }
  }
  __syncthreads();
  if constexpr (SRC == 3) {
    // the keys are u4 bounds so far: T (= T4) covers every row they dropped, the q8 re-score decides the rest
    stb_q8_refine(args, skeys, (int)s_cnt);
    __syncthreads();
  }
  unsigned bound;                                // uniform per CTA from here on
  {
    const int c = (int)s_cnt;
    stb_pad_and_sort(skeys, c, KP);
    const int keep = (gridDim.x == 1) ? KF : KP;
    // warps dropped keys below their own minimum (<= T); the compaction dropped keys < T
    bound = (s_T > kOrdNegInf) ? s_T : 0u;
    if (c > keep) bound = max(bound, stb_f2ord(stb_key_score(skeys[keep - 1])));
  }
  STB_T_MAX(2);                      // last CTA-level merge done

  // Everything below writes scratch shared with the PREVIOUS launch on this stream
  // (keys, tickets, exchange slots): wait until that grid has completed and flushed.
  asm volatile("griddepcontrol.wait;" ::: "memory");

  // ---- tree merge across CTAs ------------------------------------------------------------
  // Lists of KP sorted keys (+ their drop bound) are merged F = 1024/KP at a time by the last
  // CTA to arrive in each group (atomic ticket + fences), level by level: 296 -> 10 -> 1 lists
  // at E = 1.  Each merge is one register/shuffle bitonic sort of <= 1024 keys; the groups of a
  // level run in parallel on different SMs.  Level l's lists live at key offset
  // lvl_key_off*KPS, its tickets at counters[lvl_cnt_off + group].
  {
    constexpr int F = STB_SORT_CAP / KP;
    uint32_t lists = gridDim.x, my_id = blockIdx.x, lvl_key_off = 0, lvl_cnt_off = 0;
    while (lists > 1) {
      uint64_t *lvl = args.keys + (size_t)lvl_key_off * KPS;
      for (int i = threadIdx.x; i < KP; i += blockDim.x) lvl[(size_t)my_id * KPS + i] = skeys[i];
      if (threadIdx.x == 0) lvl[(size_t)my_id * KPS + KP] = (uint64_t)bound;
      __threadfence();
      __syncthreads();
      const uint32_t group = my_id / F, first = group * F;
      const uint32_t n_in = min((uint32_t)F, lists - first);
      if (threadIdx.x == 0) s_ticket = atomicAdd(args.counters + lvl_cnt_off + group, 1u);
      __syncthreads();
      if (s_ticket != n_in - 1) return;            // not the last of my group: done
      __threadfence();
      if (threadIdx.x == 0) args.counters[lvl_cnt_off + group] = 0u;   // re-arm for the next launch
      const uint32_t groups = (lists + F - 1) / F;
      const int keep = (groups == 1) ? KF : KP;     // the root keeps the re-rank set
      {
        // Pre-filter before sorting: every list is sorted best-first, so with
        // r = ceil(keep / n_in) - 1 the worst of the lists' r-th keys is a lower bound of the
        // group's keep-th best (n_in * (r+1) >= keep keys are at least that good).  Only keys at
        // or above it can survive the merge -- typically ~100 of the 1024 -- and the sort
        // shrinks from the 1024-key to the 256-key network.  r >= KP (fewer than `keep` keys
        // in total): nothing can be filtered.
        constexpr int PER = STB_SORT_CAP / STB_SCAN_THREADS;
        uint64_t v[PER];
        const uint32_t r = (keep + n_in - 1) / n_in - 1;
        if (threadIdx.x == 0) { s_T64 = (r >= (uint32_t)KP) ? STB_KEY_INVALID : 0ull; s_cnt = 0u; s_bound = 0u; s_nin = 0u; }
        __syncthreads();
        unsigned my_valid = 0;
#pragma unroll
        for (int u = 0; u < PER; ++u) {
          const int i = threadIdx.x + u * STB_SCAN_THREADS;
          const uint32_t li = i / KP;
          v[u] = (li < n_in) ? __ldcg(lvl + (size_t)(first + li) * KPS + (i % KP)) : STB_KEY_INVALID;
          my_valid += (v[u] != STB_KEY_INVALID) ? 1u : 0u;
          if (li < n_in && (uint32_t)(i % KP) == r) atomicMax(&s_T64, v[u]);   // INVALID (all ones) disables the filter
        }
        if (threadIdx.x < n_in) atomicMax(&s_bound, (unsigned)__ldcg(lvl + (size_t)(first + threadIdx.x) * KPS + KP));
        my_valid = __reduce_add_sync(0xffffffffu, my_valid);
        if (lane == 0 && my_valid) atomicAdd(&s_nin, my_valid);
        __syncthreads();
        const uint64_t T = s_T64;
#pragma unroll
        for (int u = 0; u < PER; ++u) {
          const bool take = v[u] != STB_KEY_INVALID && v[u] <= T;
          const unsigned m = __ballot_sync(0xffffffffu, take);
          unsigned base = 0u;
          if (lane == 0 && m) base = atomicAdd(&s_cnt, (unsigned)__popc(m));
          base = __shfl_sync(0xffffffffu, base, 0);
          if (take) skeys[base + __popc(m & ((1u << lane) - 1u))] = v[u];
        }
      }
      __syncthreads();
      stb_pad_and_sort(skeys, (int)s_cnt, KP);
      bound = s_bound;
      if ((int)s_nin > keep) bound = max(bound, stb_f2ord(stb_key_score(skeys[keep - 1])));
      lvl_key_off += lists;
      lvl_cnt_off += groups;
      lists = groups;
      my_id = group;
    }
  }
  STB_T_MAX(3);                      // survivor holds the global best KF
  STB_T_MAX(4);

  // ---- exact re-rank of the best KF in canonical arithmetic --------------------------
  // Rows are staged through shared memory (coalesced, one DRAM latency), then one
  // thread per candidate accumulates (ab, q2, r2) with f64 FMAs in index order:
  // f32 x f32 products are exact in f64, so this equals orc_cosine_f32 bit for bit.
  for (int i = threadIdx.x; i < STB_D; i += blockDim.x) sqd[i] = (double)__ldg(args.scan.q + i);
  if (threadIdx.x < 2) s_nv[threadIdx.x] = 0;
  if (threadIdx.x < KF) { s_d[threadIdx.x] = CUDART_INF; s_r[threadIdx.x] = 0xffffffffffffffffull; }
  __syncthreads();
  if (threadIdx.x == 5 * 32) {                       // an otherwise idle warp: ||q||^2 once
    double q2 = 0.0;
#pragma unroll 8
    for (int i = 0; i < STB_D; ++i) q2 = fma(sqd[i], sqd[i], q2);
    s_q2 = q2;
  }
  // Candidates are sorted by approximate score (or upper bound) best-first and re-scored 32 at a
  // time.  After the first 32 the k-th best EXACT cosine c_k among them is known; a later
  // candidate whose score + eps is below c_k cannot enter the top-k, and neither can anything
  // after it -- with K' = 128 (q8) this usually ends the re-rank after one pass instead of four.
  __shared__ double s_cthr;
  __shared__ int s_done;
  if (threadIdx.x == 0) { s_cthr = -CUDART_INF; s_done = 0; }
  for (int chunk = 0; chunk < EF; ++chunk) {
    if (chunk > 0) {
      const uint64_t nk = skeys[chunk * 32];                            // uniform
      if (nk == STB_KEY_INVALID || (double)stb_key_score(nk) + kScoreEps < s_cthr) break;
    }
    {
      constexpr int PER = 32 * STB_ROW_F4 / STB_SCAN_THREADS;   // float4 per thread
      float4 v[PER];
#pragma unroll
      for (int u = 0; u < PER; ++u) {
        const int t = threadIdx.x + u * STB_SCAN_THREADS;
        const uint64_t key = skeys[chunk * 32 + (t >> 6)];
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (key != STB_KEY_INVALID)
          v[u] = __ldg(args.scan.rows + (size_t)stb_key_row(key) * STB_ROW_F4 + (t & 63));
      }
#pragma unroll
      for (int u = 0; u < PER; ++u) {
        const int t = threadIdx.x + u * STB_SCAN_THREADS;
        *reinterpret_cast<float4 *>(srows + (t >> 6) * STB_RR_STRIDE + (t & 63) * 4) = v[u];
      }
    }
    __syncthreads();
    // 8 candidates per warp on 4 warps (one per SM sub-partition): the f64 chains are
    // latency-bound, so spreading them quarters the issue time
    if (threadIdx.x < 128 && lane < 8) {
      const int cl = (threadIdx.x >> 5) * 8 + lane;          // candidate inside the chunk
      const int ci = chunk * 32 + cl;
      if (skeys[ci] != STB_KEY_INVALID) {
        const float4 *rp = reinterpret_cast<const float4 *>(srows + cl * STB_RR_STRIDE);
        double ab = 0.0, r2 = 0.0;
#pragma unroll 8
        for (int i = 0; i < STB_ROW_F4; ++i) {
          const float4 v = rp[i];
          const double vx = (double)v.x, vy = (double)v.y, vz = (double)v.z, vw = (double)v.w;
          // oracle order (orc_cosine_f32(q,row)): index order, one rounding per step
          ab = fma(sqd[4 * i + 0], vx, ab); r2 = fma(vx, vx, r2);
          ab = fma(sqd[4 * i + 1], vy, ab); r2 = fma(vy, vy, r2);
          ab = fma(sqd[4 * i + 2], vz, ab); r2 = fma(vz, vz, r2);
          ab = fma(sqd[4 * i + 3], vw, ab); r2 = fma(vw, vw, r2);
        }
        s_d[ci] = ab;          // finalised below once ||q||^2 is known
        s_r2[ci] = r2;
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) s_done = chunk + 1;
    if (chunk == 0 && EF > 1 && args.top_k <= 32) {
      if (threadIdx.x < 32) {
        const uint64_t key = skeys[lane];
        double dist = CUDART_INF;
        if (key != STB_KEY_INVALID) {
          const double ab = s_d[lane], r2 = s_r2[lane], q2 = s_q2;
          if (q2 == 0.0 && r2 == 0.0) dist = 0.0;
          else if (ab == 0.0) dist = 1.0;
          else { const double t = 1.0 - ab / (sqrt(q2) * sqrt(r2)); dist = t > 0.0 ? t : 0.0; }
          if (!(dist < 100.0)) dist = CUDART_INF;
        }
        int rank = 0;
#pragma unroll
        for (int jj = 0; jj < 32; ++jj) {
          const double dj = __shfl_sync(0xffffffffu, dist, jj);
          rank += (dj < dist || (dj == dist && jj < lane)) ? 1 : 0;
        }
        const unsigned passing = __ballot_sync(0xffffffffu, dist < CUDART_INF);
        if ((uint32_t)__popc(passing) >= args.top_k && rank == (int)args.top_k - 1) s_cthr = 1.0 - dist;
      }
      __syncthreads();
    }
  }
  __syncthreads();
  if (threadIdx.x < KF) {
    const uint64_t key = skeys[threadIdx.x];
    double d = CUDART_INF;
    uint64_t grow = 0xffffffffffffffffull;
    if (key != STB_KEY_INVALID) atomicAdd(&s_nv[0], 1);     // valid candidates (re-scored or provably outside the top-k)
    if (key != STB_KEY_INVALID && (int)threadIdx.x < 32 * s_done) {
      const double ab = s_d[threadIdx.x], r2 = s_r2[threadIdx.x], q2 = s_q2;
      double dist;
      if (q2 == 0.0 && r2 == 0.0) dist = 0.0;
      else if (ab == 0.0) dist = 1.0;
      else {
        double t = 1.0 - ab / (sqrt(q2) * sqrt(r2));
        dist = t > 0.0 ? t : 0.0;
      }
      if (dist < 100.0) {                         // max_distance.unwrap_or(100.0), strict
        d = dist;
        grow = args.row_base + (uint64_t)stb_key_row(key);
        atomicAdd(&s_nv[1], 1);                   // passing
      }
    }
    s_d[threadIdx.x] = d;
    s_r[threadIdx.x] = grow;
  }
  __syncthreads();
  // bitonic sort of the KF (distance,row) pairs
  for (int k = 2; k <= KF; k <<= 1) {
    for (int jj = k >> 1; jj > 0; jj >>= 1) {
      int i = threadIdx.x;
      if (i < KF) {
        int ixj = i ^ jj;
        if (ixj > i) {
          double da = s_d[i], db = s_d[ixj];
          uint64_t ra = s_r[i], rb = s_r[ixj];
          bool up = ((i & k) == 0);
          bool gt = stb_hit_less(db, rb, da, ra);
          if (gt == up) { s_d[i] = db; s_r[i] = rb; s_d[ixj] = da; s_r[ixj] = ra; }
        }
      }
      __syncthreads();
    }
  }
  STB_T_MAX(5);                      // exact re-rank + hit sort done
  const int n_valid = s_nv[0], n_pass = s_nv[1];
  const uint32_t k = args.top_k;
  const uint32_t n_out = min((uint32_t)n_pass, k);
  bool complete;
  if (bound == 0u) complete = true;    // no node dropped a key: every scorable row is a candidate
  else {
    // every row that is not a candidate scored <= the best dropped score
    const float s_drop = stb_ord2f(bound);
    complete = (n_out == k) && ((1.0 - (double)s_drop - kScoreEps) > s_d[k - 1]);
  }
  if (args.xchg.world <= 1) {
    for (uint32_t i = threadIdx.x; i < k; i += blockDim.x) {
      stb_hit h;
      h.distance = (i < n_out) ? s_d[i] : CUDART_INF;
      h.row = (i < n_out) ? s_r[i] : 0xffffffffffffffffull;
      args.out_hits[i] = h;
    }
    if (threadIdx.x == 0) {
      args.out_status[0] = n_out;
      args.out_status[1] = complete ? 1u : 0u;
      args.out_status[2] = (uint32_t)n_valid;
      args.out_status[3] = (uint32_t)KF | (kTierReported << 16);
    }
    return;
  }

  // ---- fused exchange over NVLink peer memory + global merge ---------------------------
  const StbXchgArgs &X = args.xchg;
  const int world = (int)X.world, me = (int)X.rank;
  const size_t lane_off = (size_t)X.slot * world + me;
  for (int idx = threadIdx.x; idx < world * (int)k; idx += blockDim.x) {
    const int p = idx / (int)k, i = idx % (int)k;
    stb_hit h;
    h.distance = ((uint32_t)i < n_out) ? s_d[i] : CUDART_INF;
    h.row = ((uint32_t)i < n_out) ? s_r[i] : 0xffffffffffffffffull;
    stb_x_hits(X, p)[lane_off * X.max_k + i] = h;
  }
  if (threadIdx.x < world) stb_x_status(X, threadIdx.x)[lane_off] = (complete ? 1u : 0u) | (n_out << 8);
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < world) stb_st_release_sys(stb_x_flags(X, threadIdx.x) + lane_off, X.seq);
  __shared__ unsigned int s_timeout;
  if (threadIdx.x == 0) s_timeout = 0u;
  __syncthreads();
  if (threadIdx.x < world) {
    const unsigned long long *f = stb_x_flags(X, me) + (size_t)X.slot * world + threadIdx.x;
    const long long t0 = clock64();
    while (stb_ld_acquire_sys(f) != X.seq) {
      if (clock64() - t0 > STB_XCHG_TIMEOUT_CYCLES) { s_timeout = 1u; break; }   // a peer is gone
    }
  }
  __syncthreads();
  // merge world x k hits by (distance,row); buffers alias the re-rank staging area
  double *md = reinterpret_cast<double *>(srows);
  uint64_t *mr = reinterpret_cast<uint64_t *>(srows) + 1024;
  const int n_in = world * (int)k;
  int n_sort = 2;
  while (n_sort < n_in) n_sort <<= 1;
  const stb_hit *lh = stb_x_hits(X, me) + (size_t)X.slot * world * X.max_k;
  for (int i = threadIdx.x; i < n_sort; i += blockDim.x) {
    double d = CUDART_INF;
    uint64_t r = 0xffffffffffffffffull;
    if (i < n_in) {
      const stb_hit *src = lh + (size_t)(i / (int)k) * X.max_k + (i % (int)k);
      d = __ldcv(&src->distance);
      r = __ldcv(&src->row);
    }
    md[i] = d; mr[i] = r;
  }
  __syncthreads();
  for (int kk = 2; kk <= n_sort; kk <<= 1) {
    for (int jj = kk >> 1; jj > 0; jj >>= 1) {
      for (int i = threadIdx.x; i < n_sort; i += blockDim.x) {
        int ixj = i ^ jj;
        if (ixj > i) {
          bool up = ((i & kk) == 0);
          bool gt = stb_hit_less(md[ixj], mr[ixj], md[i], mr[i]);
          if (gt == up) {
            double td = md[i]; uint64_t tr = mr[i];
            md[i] = md[ixj]; mr[i] = mr[ixj]; md[ixj] = td; mr[ixj] = tr;
          }
        }
      }
      __syncthreads();
    }
  }
  for (uint32_t i = threadIdx.x; i < k; i += blockDim.x) {
    stb_hit h;
    h.distance = md[i];
    h.row = mr[i];
    args.out_hits[i] = h;
  }
  if (threadIdx.x == 0) {
    uint32_t all_complete = s_timeout ? 0u : 1u, total = 0u;
    const uint32_t *st = stb_x_status(X, me) + (size_t)X.slot * world;
    for (int p = 0; p < world; ++p) {
      uint32_t v = __ldcv(st + p);
      all_complete &= (v & 1u);
      total += v >> 8;
    }
    args.out_status[0] = min(total, k);
    args.out_status[1] = all_complete;
    args.out_status[2] = s_timeout ? 0xfffffffeu : (uint32_t)n_valid;
    args.out_status[3] = (uint32_t)KF | (kTierReported << 16);
  }
}

uint32_t stb_scan_topk_max_k(void) { return 96; }

static int stb_pick_e(uint32_t top_k) {
  if (top_k <= 16) return 1;   // K' = 32
  if (top_k <= 40) return 2;   // K' = 64
  return 4;                    // K' = 128
}

#define STB_SHADOW_SCAN_U 4     // 4 rows x 4 LDG.128 per lane in flight = the f32 path's 2 x 8
#define STB_Q8_SCAN_U 8         // 8 rows x 2 LDG.128
#define STB_Q4_SCAN_U 16        // 16 rows x 1 LDG.128: 128 KiB in flight per SM at 2 CTAs, as q8

// STB_SCAN_CTAS_PER_SM (tuning aid): resident CTAs per SM the top-k grid is sized for
// (default: what the occupancy calculator allows, 2 with the 128-register budget).
// STB_SCAN_TICKETS=0 (tuning aid): static warp-strided tile partition instead of tickets.
static bool stb_scan_tickets_enabled() {
  static const bool v = [] { const char *e = getenv("STB_SCAN_TICKETS"); return !(e && e[0] == '0'); }();
  return v;
}
static int stb_scan_ctas_per_sm_override() {
  static const int v = [] { const char *e = getenv("STB_SCAN_CTAS_PER_SM"); return e ? atoi(e) : 0; }();
  return v;
}

template <int E, int RANGES, int SRC = 0, int EF = E>
static int stb_launch_topk_t(stb_ctx *ctx, const TopkArgs &a_in, bool overlapped) {
  constexpr int kU = SRC == 3 ? STB_Q4_SCAN_U : SRC == 2 ? STB_Q8_SCAN_U : (SRC == 1 ? STB_SHADOW_SCAN_U : STB_SCAN_U);
  auto kern = stb_scan_topk_kernel<E, kU, RANGES, SRC, EF>;
  int occ = 0;
  STB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, STB_SCAN_THREADS, 0));
  if (occ < 1) occ = 1;
  const int ovr = stb_scan_ctas_per_sm_override();
  if (ovr >= 1 && ovr < occ) occ = ovr;
  TopkArgs a = a_in;
  const bool use_tickets = stb_scan_tickets_enabled();
  overlapped = overlapped && use_tickets && occ >= 2;
  if (overlapped) occ = 1;                 // two consecutive grids co-reside, one CTA per SM each
  a.early_trigger = overlapped ? 1u : 0u;
  const uint64_t tiles = (a.scan.n_virtual + 4 * kU - 1) / (4 * kU);
  uint64_t want = (tiles + STB_SCAN_WARPS - 1) / STB_SCAN_WARPS;
  uint64_t grid = (uint64_t)ctx->sm_count * occ;
  if (want < grid) grid = want < 1 ? 1 : want;
  // scratch: lists (KP keys + bound) for all tree levels (< 2 * grid lists), counters (< grid groups)
  size_t need_keys = (size_t)2 * grid * (32 * E + 1) + STB_SORT_CAP;
  if (need_keys > ctx->block_keys_cap || grid + 8 > ctx->counters_cap) {
    stb_set_error("scan scratch too small (grid=%llu)", (unsigned long long)grid);
    return STB_ERR_STATE;
  }
  // tile tickets (stb_for_each_tile): bulk tickets of STB_TICKET_TILES tiles, then the last ~2 tiles
  // per warp one by one.  The launch advances the counter by n_tickets + total_warps exactly.
  const uint64_t warps_total = grid * STB_SCAN_WARPS;
  if (use_tickets) {
    const uint64_t single = std::min<uint64_t>(tiles, 2 * warps_total);
    a.scan.t_bulk = (tiles - single) / STB_TICKET_TILES;
    const uint64_t n_tickets = a.scan.t_bulk + (tiles - a.scan.t_bulk * STB_TICKET_TILES);
    // consecutive launches draw from different counters of the ring: two overlapped scans co-run, and a
    // straggler warp of a finished scan must not take a ticket of the next one (at most ~3 grids are ever
    // in flight, far fewer than STB_TICKET_SLOTS)
    const int slot = (int)(ctx->topk_launches++ % STB_TICKET_SLOTS);
    a.scan.tickets = ctx->tickets + slot;
    a.scan.t_base = ctx->ticket_next[slot];
    ctx->ticket_next[slot] += n_tickets + warps_total;
    a.scan.start = ctx->scan_start + slot;
    a.scan.front = ctx->scan_front;
    a.scan.seq = (uint32_t)ctx->topk_launches;   // the slot's previous launch had seq - STB_TICKET_SLOTS; never 0 mod 2^32 twice in a row
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(STB_SCAN_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = ctx->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // PDL, see the kernel
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  STB_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
  STB_CUDA(cudaGetLastError());
  ctx->kernel_launches++;
  return STB_OK;
}

template <int RANGES>
static int stb_launch_topk_r(stb_ctx *ctx, const TopkArgs &a, int tier, uint32_t top_k, bool ov) {
  const int e = stb_pick_e(top_k);
  // q8: 32-key lists below the root, 128 candidates re-ranked at the root (see stb_scan_q8)
  if (tier == STB_TIER_Q8) return stb_launch_topk_t<1, RANGES, 2, 4>(ctx, a, ov);
  // coarse + q8: 64-key warp lists by the 4-bit bound, re-scored with q8 in the CTA; 32-key lists above
  if (tier == STB_TIER_Q4Q8) return stb_launch_topk_t<1, RANGES, 3, 4>(ctx, a, ov);
  if (tier == STB_TIER_H16) {
    switch (e) {
      case 1: return stb_launch_topk_t<1, RANGES, 1>(ctx, a, ov);
      case 2: return stb_launch_topk_t<2, RANGES, 1>(ctx, a, ov);
      default: return stb_launch_topk_t<4, RANGES, 1>(ctx, a, ov);
    }
  }
  switch (e) {
    case 1: return stb_launch_topk_t<1, RANGES, 0>(ctx, a, ov);
    case 2: return stb_launch_topk_t<2, RANGES, 0>(ctx, a, ov);
    default: return stb_launch_topk_t<4, RANGES, 0>(ctx, a, ov);
  }
}

int stb_launch_scan_topk(stb_ctx *ctx, const stb_corpus *c, int tier, const float *q_dev, uint32_t top_k,
                         const uint64_t *ranges_dev, uint32_t n_ranges,
                         uint64_t n_virtual, stb_hit *out_hits_dev,
                         uint32_t *out_status_dev, const StbXchgArgs *xchg, bool overlapped) {
  TopkArgs a;
  a.scan.rows = reinterpret_cast<const float4 *>(c->rows);
  a.scan.n_virtual = n_virtual;
  a.scan.q = q_dev;
  a.scan.vstart = ranges_dev;
  a.scan.rbegin = ranges_dev ? ranges_dev + (n_ranges + 1) : nullptr;
  a.scan.n_ranges = n_ranges;
  a.scan.tickets = nullptr; a.scan.t_base = 0; a.scan.t_bulk = 0; a.scan.start = a.scan.front = nullptr; a.scan.seq = 0;
  a.row_base = c->row_base;
  a.keys = ctx->block_keys;
  a.counters = ctx->counters;
  a.out_hits = out_hits_dev;
  a.out_status = out_status_dev;
  a.top_k = top_k;
  if (xchg) a.xchg = *xchg; else memset(&a.xchg, 0, sizeof(a.xchg));
  a.dbg = ctx->dbg_dev;
  a.early_trigger = 0;
  a.shadow = c->shadow;
  a.q8 = c->q8;
  a.q8_scale = c->q8_scale;
  a.q4 = c->q4;
  a.q4_sr = c->q4_sr;
  if (tier == STB_TIER_Q8 && (top_k > STB_Q8_MAX_K || !c->q8)) { stb_set_error("scan_topk: q8 tier unavailable"); return STB_ERR_STATE; }
  if (tier == STB_TIER_Q4Q8 && (top_k > STB_Q8_MAX_K || !c->q8 || !c->q4)) { stb_set_error("scan_topk: coarse q8 stage unavailable"); return STB_ERR_STATE; }
  if (tier == STB_TIER_H16 && !c->shadow) { stb_set_error("scan_topk: h16 tier unavailable"); return STB_ERR_STATE; }
  return n_ranges > 0 ? stb_launch_topk_r<1>(ctx, a, tier, top_k, overlapped) : stb_launch_topk_r<0>(ctx, a, tier, top_k, overlapped);
}

// ------------------------------------------------------------------ collect path ---
struct CollectSink {
  float floor_;
  uint32_t *out;
  unsigned long long *count;
  uint64_t cap;
  template <int ROWS>
  __device__ __forceinline__ void consume(float s, uint32_t r) { (*this)(s, r); }
  __device__ __forceinline__ void operator()(float s, uint32_t r) {
    bool hit = (s >= floor_) && (s > -CUDART_INF_F);   // -inf marks lanes that carry no row
    unsigned mask = __ballot_sync(0xffffffffu, hit);
    if (mask == 0) return;
    int lane = threadIdx.x & 31;
    int leader = __ffs(mask) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(count, (unsigned long long)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (hit) {
      unsigned long long idx = base + __popc(mask & ((1u << lane) - 1));
      if (idx < cap) out[idx] = r;
    }
  }
};

struct CollectArgs {
  ScanArgs scan;
  float cos_floor;
  uint32_t *out;
  unsigned long long *count;
  uint64_t cap;
  const uint8_t *q8;         // SRC == 2: scores are the q8 tier's upper bounds of the exact cosine
  const float *q8_scale;
};

template <int U, bool RANGES, int SRC = 0>
__global__ void __launch_bounds__(STB_SCAN_THREADS, STB_SCAN_MINB)
stb_scan_collect_kernel(const CollectArgs args) {
  CollectSink sink{args.cos_floor, args.out, args.count, args.cap};
  if constexpr (SRC == 2) stb_scan_q8<U, RANGES>(args.scan, args.q8, args.q8_scale, sink);
  else stb_scan_rows<U, RANGES>(args.scan, sink);
}

int stb_launch_scan_collect(stb_ctx *ctx, const stb_corpus *c, int tier,
                            const float *q_dev, float cos_floor,
                            const uint64_t *ranges_dev, uint32_t n_ranges,
                            uint64_t n_virtual) {
  CollectArgs a;
  a.scan.rows = reinterpret_cast<const float4 *>(c->rows);
  a.q8 = c->q8; a.q8_scale = c->q8_scale;
  a.scan.n_virtual = n_virtual;
  a.scan.q = q_dev;
  a.scan.vstart = ranges_dev;
  a.scan.rbegin = ranges_dev ? ranges_dev + (n_ranges + 1) : nullptr;
  a.scan.n_ranges = n_ranges;
  a.scan.tickets = nullptr; a.scan.t_base = 0; a.scan.t_bulk = 0; a.scan.start = a.scan.front = nullptr; a.scan.seq = 0;
  a.cos_floor = cos_floor;
  a.out = ctx->collect_rows;
  a.count = ctx->collect_count;
  a.cap = ctx->collect_cap;
  STB_CUDA(cudaMemsetAsync(ctx->collect_count, 0, sizeof(unsigned long long), ctx->stream));
  const int u = tier == STB_TIER_Q8 ? STB_Q8_SCAN_U : STB_SCAN_U;
  uint64_t tiles = (n_virtual + 4 * u - 1) / (4 * u);
  uint64_t want = (tiles + STB_SCAN_WARPS - 1) / STB_SCAN_WARPS;
  uint64_t grid = (uint64_t)ctx->sm_count * STB_SCAN_MINB;
  if (want < grid) grid = want < 1 ? 1 : want;
  if (tier == STB_TIER_Q8) {
    if (!c->q8) { stb_set_error("scan_collect: q8 tier unavailable"); return STB_ERR_STATE; }
    if (n_ranges > 0) stb_scan_collect_kernel<STB_Q8_SCAN_U, true, 2><<<(unsigned)grid, STB_SCAN_THREADS, 0, ctx->stream>>>(a);
    else stb_scan_collect_kernel<STB_Q8_SCAN_U, false, 2><<<(unsigned)grid, STB_SCAN_THREADS, 0, ctx->stream>>>(a);
  } else if (n_ranges > 0)
    stb_scan_collect_kernel<STB_SCAN_U, true><<<(unsigned)grid, STB_SCAN_THREADS, 0, ctx->stream>>>(a);
  else
    stb_scan_collect_kernel<STB_SCAN_U, false><<<(unsigned)grid, STB_SCAN_THREADS, 0, ctx->stream>>>(a);
  STB_CUDA(cudaGetLastError());
  ctx->kernel_launches++;
  return STB_OK;
}

// ------------------------------------------------------------ histogram pass (large k) ---
// For top_k beyond the register lists: one scan builds a 4096-bin histogram of the
// approximate cosine (bin b covers cos in (1-(b+1)/2048, 1-b/2048]; forced candidates fall
// in bin 0), the host picks the bin that contains the k-th best, and the collect pass
// gathers everything at or above that bin's lower edge (minus the score error bound).
#define STB_HIST_BINS 4096
struct HistSink {
  unsigned int *hist;   // shared-memory histogram of this CTA
  template <int ROWS>
  __device__ __forceinline__ void consume(float s, uint32_t) {
    if (s > -CUDART_INF_F) {
      float b = floorf((1.0f - s) * (STB_HIST_BINS / 2.0f));
      int bin = b < 0.f ? 0 : (b > (float)(STB_HIST_BINS - 1) ? STB_HIST_BINS - 1 : (int)b);   // +inf -> 0, NaN cannot occur
      atomicAdd(hist + bin, 1u);
    }
  }
};

template <int U, bool RANGES, int SRC = 0>
__global__ void __launch_bounds__(STB_SCAN_THREADS, STB_SCAN_MINB)
stb_scan_hist_kernel(const ScanArgs scan, unsigned int *global_hist, const uint8_t *q8, const float *q8_scale) {
  __shared__ unsigned int s_hist[STB_HIST_BINS];
  for (int i = threadIdx.x; i < STB_HIST_BINS; i += blockDim.x) s_hist[i] = 0u;
  __syncthreads();
  HistSink sink{s_hist};
  if constexpr (SRC == 2) stb_scan_q8<U, RANGES>(scan, q8, q8_scale, sink);
  else stb_scan_rows<U, RANGES>(scan, sink);
  __syncthreads();
  for (int i = threadIdx.x; i < STB_HIST_BINS; i += blockDim.x)
    if (s_hist[i]) atomicAdd(global_hist + i, s_hist[i]);
}

int stb_launch_scan_hist(stb_ctx *ctx, const stb_corpus *c, int tier, const float *q_dev, const uint64_t *ranges_dev,
                         uint32_t n_ranges, uint64_t n_virtual, unsigned int *hist_dev) {
  ScanArgs a;
  a.rows = reinterpret_cast<const float4 *>(c->rows);
  a.n_virtual = n_virtual;
  a.q = q_dev;
  a.vstart = ranges_dev;
  a.rbegin = ranges_dev ? ranges_dev + (n_ranges + 1) : nullptr;
  a.n_ranges = n_ranges;
  a.tickets = nullptr; a.t_base = 0; a.t_bulk = 0; a.start = a.front = nullptr; a.seq = 0;
  STB_CUDA(cudaMemsetAsync(hist_dev, 0, STB_HIST_BINS * sizeof(unsigned int), ctx->stream));
  const int u = tier == STB_TIER_Q8 ? STB_Q8_SCAN_U : STB_SCAN_U;
  uint64_t tiles = (n_virtual + 4 * u - 1) / (4 * u);
  uint64_t want = (tiles + STB_SCAN_WARPS - 1) / STB_SCAN_WARPS;
  uint64_t grid = (uint64_t)ctx->sm_count * STB_SCAN_MINB;
  if (want < grid) grid = want < 1 ? 1 : want;
  if (tier == STB_TIER_Q8) {
    if (!c->q8) { stb_set_error("scan_hist: q8 tier unavailable"); return STB_ERR_STATE; }
    if (n_ranges > 0) stb_scan_hist_kernel<STB_Q8_SCAN_U, true, 2><<<(unsigned)grid, STB_SCAN_THREADS, 0, ctx->stream>>>(a, hist_dev, c->q8, c->q8_scale);
    else stb_scan_hist_kernel<STB_Q8_SCAN_U, false, 2><<<(unsigned)grid, STB_SCAN_THREADS, 0, ctx->stream>>>(a, hist_dev, c->q8, c->q8_scale);
  } else if (n_ranges > 0)
    stb_scan_hist_kernel<STB_SCAN_U, true><<<(unsigned)grid, STB_SCAN_THREADS, 0, ctx->stream>>>(a, hist_dev, nullptr, nullptr);
  else
    stb_scan_hist_kernel<STB_SCAN_U, false><<<(unsigned)grid, STB_SCAN_THREADS, 0, ctx->stream>>>(a, hist_dev, nullptr, nullptr);
  STB_CUDA(cudaGetLastError());
  ctx->kernel_launches++;
  return STB_OK;
}

// Exact canonical distance of each collected row; one thread per row.
__global__ void stb_exact_kernel(const float4 *rows, uint64_t row_base, const float *q,
                                 const uint32_t *row_ids, uint64_t m, double limit,
                                 stb_hit *hits, uint64_t m_padded,
                                 unsigned long long *pass_count) {
  __shared__ __align__(16) float sq[STB_D];
  for (int i = threadIdx.x; i < STB_D; i += blockDim.x) sq[i] = __ldg(q + i);
  __syncthreads();
  uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= m_padded) return;
  stb_hit h;
  h.distance = CUDART_INF;
  h.row = 0xffffffffffffffffull;
  if (idx < m) {
    uint32_t row = row_ids[idx];
    const float4 *rp = rows + (size_t)row * STB_ROW_F4;
    const float4 *qp = reinterpret_cast<const float4 *>(sq);
    double ab = 0.0, q2 = 0.0, r2 = 0.0;
#pragma unroll 4
    for (int i = 0; i < STB_ROW_F4; ++i) {
      float4 v = __ldg(rp + i);
      float4 w = qp[i];
      ab = fma((double)w.x, (double)v.x, ab); q2 = fma((double)w.x, (double)w.x, q2); r2 = fma((double)v.x, (double)v.x, r2);
      ab = fma((double)w.y, (double)v.y, ab); q2 = fma((double)w.y, (double)w.y, q2); r2 = fma((double)v.y, (double)v.y, r2);
      ab = fma((double)w.z, (double)v.z, ab); q2 = fma((double)w.z, (double)w.z, q2); r2 = fma((double)v.z, (double)v.z, r2);
      ab = fma((double)w.w, (double)v.w, ab); q2 = fma((double)w.w, (double)w.w, q2); r2 = fma((double)v.w, (double)v.w, r2);
    }
    double dist;
    if (q2 == 0.0 && r2 == 0.0) dist = 0.0;
    else if (ab == 0.0) dist = 1.0;
    else {
      double t = 1.0 - ab / (sqrt(q2) * sqrt(r2));
      dist = t > 0.0 ? t : 0.0;
    }
    if (dist < limit) {
      h.distance = dist;
      h.row = row_base + (uint64_t)row;
      atomicAdd(pass_count, 1ull);
    }
  }
  hits[idx] = h;
}

int stb_launch_exact(stb_ctx *ctx, const float *rows, uint64_t row_base,
                     const float *q_dev, const uint32_t *row_ids, uint64_t m,
                     double limit, stb_hit *hits, uint64_t m_padded,
                     unsigned long long *pass_count) {
  STB_CUDA(cudaMemsetAsync(pass_count, 0, sizeof(unsigned long long), ctx->stream));
  if (m_padded == 0) return STB_OK;
  unsigned blocks = (unsigned)((m_padded + 127) / 128);
  stb_exact_kernel<<<blocks, 128, 0, ctx->stream>>>(reinterpret_cast<const float4 *>(rows),
                                                     row_base, q_dev, row_ids, m, limit, hits,
                                                     m_padded, pass_count);
  STB_CUDA(cudaGetLastError());
  ctx->kernel_launches++;
  return STB_OK;
}

// Global bitonic sort of hits by (distance,row): one launch per (k,j) step above
// the shared-memory span, fused steps inside a 1024-element span.
__global__ void stb_bitonic_global_step(stb_hit *h, uint64_t n, uint64_t k, uint64_t j) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t ixj = i ^ j;
  if (ixj > i) {
    stb_hit a = h[i], b = h[ixj];
    bool up = ((i & k) == 0);
    bool gt = stb_hit_less(b.distance, b.row, a.distance, a.row);
    if (gt == up) { h[i] = b; h[ixj] = a; }
  }
}

// Sorts all steps with j < 1024 of stage k inside shared memory (span 1024).
__global__ void stb_bitonic_local(stb_hit *h, uint64_t n, uint64_t k_first, uint64_t k_last) {
  __shared__ double sd[1024];
  __shared__ uint64_t sr[1024];
  const uint64_t base = (uint64_t)blockIdx.x * 1024;
  for (int t = threadIdx.x; t < 1024; t += blockDim.x) {
    stb_hit x = h[base + t];
    sd[t] = x.distance; sr[t] = x.row;
  }
  __syncthreads();
  for (uint64_t k = k_first; k <= k_last; k <<= 1) {
    uint64_t jstart = (k >> 1) < 512 ? (k >> 1) : 512;
    for (uint64_t j = jstart; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < 1024; t += blockDim.x) {
        uint64_t i = base + t, ixj = i ^ j;
        if (ixj > i) {
          int u = (int)(ixj - base);
          bool up = ((i & k) == 0);
          bool gt = stb_hit_less(sd[u], sr[u], sd[t], sr[t]);
          if (gt == up) {
            double td = sd[t]; uint64_t tr = sr[t];
            sd[t] = sd[u]; sr[t] = sr[u]; sd[u] = td; sr[u] = tr;
          }
        }
      }
      __syncthreads();
    }
  }
  for (int t = threadIdx.x; t < 1024; t += blockDim.x) {
    stb_hit x; x.distance = sd[t]; x.row = sr[t];
    h[base + t] = x;
  }
}

int stb_launch_sort_hits(stb_ctx *ctx, stb_hit *hits, uint64_t n) {
  if (n < 2) return STB_OK;
  if (n < 1024 || (n & (n - 1))) { stb_set_error("sort size must be a power of two >= 1024"); return STB_ERR_ARG; }
  unsigned lblocks = (unsigned)(n / 1024);
  // stages k = 2..1024 entirely local
  stb_bitonic_local<<<lblocks, 256, 0, ctx->stream>>>(hits, n, 2, 1024);
  ctx->kernel_launches++;
  for (uint64_t k = 2048; k <= n; k <<= 1) {
    for (uint64_t j = k >> 1; j >= 1024; j >>= 1) {
      unsigned gblocks = (unsigned)((n + 255) / 256);
      stb_bitonic_global_step<<<gblocks, 256, 0, ctx->stream>>>(hits, n, k, j);
      ctx->kernel_launches++;
    }
    stb_bitonic_local<<<lblocks, 256, 0, ctx->stream>>>(hits, n, k, k);
    ctx->kernel_launches++;
  }
  STB_CUDA(cudaGetLastError());
  return STB_OK;
}
