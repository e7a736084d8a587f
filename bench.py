#!/usr/bin/env python
"""bench.py -- queries/sec of the semtools `search` scan on B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 200 --warmup 10
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference            # the reference's CPU scan on the host cores

A "step" is one query: one pass of the hot path (K1 cosine scan + running top-k + exact f64
re-rank [+ fused NVLink exchange + merge when sharded]) over the whole corpus.
Workload: the 10M-line x 256 f32 corpus BASELINE.json's metric is quoted on, top-k 10, single
query.  The scan reads the narrowest copy of the corpus the library has built (tier q8: int8
codes + per-row scale, 2.6 GB for 10M rows >> 126 MB L2, so every step streams from HBM and no L2
flush is needed); the re-rank reads the f32 rows; results are bit-identical to the f32 scan's.
N > 1 shards the SAME corpus row-wise across ranks ("strong" scaling), one process per GPU.

stdout: one compact JSON line per side section ({"side": name, ...}; with --side-json PATH also written
together, with the untrimmed headline, to PATH), then the headline line LAST.  bench.py writes nothing
into the source tree.

--dump-outputs DIR writes the hits of the last timed step (what a caller of the timed path receives:
distances and global row numbers, ordered by (distance,row)) as DIR/hits_distance.npy and
DIR/hits_row.npy, both float64.  The inputs depend on the arguments only (seeded generators), so two
builds run with the same arguments can be compared output for output.

PyTorch is used here for plumbing only: device allocation of the synthetic corpus, CUDA events on
the launching stream, torch.distributed (NCCL) to trade IPC handles and for barriers.  All compute
is libsemtools_b200.so via its C ABI.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import tempfile
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CHUNK = 1_000_000
SEED = 0x5E117003
METRIC = "queries/sec over 10M-line corpus, top-k=10"
TIER_BYTES = {"f32": 1024, "h16": 512, "q8": 260}
TIER_NAMES = ("f32", "h16", "q8")


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--rows", type=int, default=10_000_000)
    p.add_argument("--topk", type=int, default=10)
    p.add_argument("--ref-rows", type=int, default=0, help="--impl reference: rows per step (default: --rows, the full workload)")
    p.add_argument("--no-side", action="store_true", help="headline only (no side sections, no cpu_baseline)")
    p.add_argument("--no-cpu-baseline", action="store_true", help="alias of --no-side (round-1 name)")
    p.add_argument("--config4-rows", type=int, default=100_000_000, help="BASELINE configs[3]: rows of the sharded 100M-line section (0 = skip)")
    p.add_argument("--config2-rows", type=int, default=1_000_000, help="BASELINE configs[1]: rows of the 1M-line section")
    p.add_argument("--embed-lines", type=int, default=1_000_000, help="K3 side section: lines of the synthetic ingestion batch")
    p.add_argument("--embed-vocab", type=int, default=500_000, help="K3 side section: rows of the embedding table")
    p.add_argument("--batch-queries", type=int, default=1024, help="K2 side section: queries per batch (BASELINE configs[2]: 1024)")
    p.add_argument("--clock-load-queries", type=int, default=1200,
                   help="untimed queries (x N) run right after the timed region so the 100 ms clock samples are taken under load")
    p.add_argument("--ivfpq-rows", type=int, default=4_000_000, help="N=1 IVF-PQ side section rows")
    p.add_argument("--ivfpq-rows-per-gpu", type=int, default=12_500_000, help="N>1: clustered rows per GPU of the IVF-PQ section (x8 = configs[4])")
    p.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                   help="N>1: p2p = fused in-kernel exchange over NVLink peer memory; nccl = all-gather + merge kernel")
    p.add_argument("--side-json", metavar="PATH", help="also write the untrimmed headline and every side section to PATH")
    p.add_argument("--dump-outputs", metavar="DIR", help="write the hits of the last timed step to DIR/hits_{distance,row}.npy")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    a.no_side = a.no_side or a.no_cpu_baseline
    return a


def dump_outputs(dir_, hits):
    """hits["distance"], hits["row"]: one step's result, already trimmed to its hit count."""
    os.makedirs(dir_, exist_ok=True)
    np.save(os.path.join(dir_, "hits_distance.npy"), np.asarray(hits["distance"], dtype=np.float64))
    np.save(os.path.join(dir_, "hits_row.npy"), np.asarray(hits["row"], dtype=np.float64))   # rows < 2**53: exact


def workload_name(rows, topk):
    return f"{rows} lines x 256 f32 (unit rows, 0.1% dup, 0.01% zero), 1 query, top-k={topk}, brute-force cosine scan"


# ------------------------------------------------------------------ synthetic data ---
def gen_chunk_torch(torch, dev, chunk_id, rows):
    """Chunk `chunk_id` of the global corpus: identical whatever the rank count."""
    g = torch.Generator(device=dev)
    g.manual_seed(SEED + chunk_id)
    x = torch.randn((rows, 256), generator=g, device=dev, dtype=torch.float32)
    x /= x.norm(dim=1, keepdim=True)
    n_dup, n_zero = max(rows // 1000, 1), max(rows // 10000, 1)
    idx = torch.randint(0, rows, (2 * n_dup + n_zero,), generator=g, device=dev)
    x[idx[:n_dup]] = x[idx[n_dup:2 * n_dup]]
    x[idx[2 * n_dup:]] = 0.0
    return x


def gen_chunk_numpy(chunk_id, rows):
    rng = np.random.default_rng(SEED + chunk_id)
    x = rng.standard_normal((rows, 256), dtype=np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    n_dup, n_zero = max(rows // 1000, 1), max(rows // 10000, 1)
    idx = rng.integers(0, rows, 2 * n_dup + n_zero)
    x[idx[:n_dup]] = x[idx[n_dup:2 * n_dup]]
    x[idx[2 * n_dup:]] = 0.0
    return np.ascontiguousarray(x, dtype=np.float32)


def gen_queries(n):
    rng = np.random.default_rng(SEED - 1)
    q = rng.standard_normal((n, 256)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    return np.ascontiguousarray(q, dtype=np.float32)


def fill_shard(torch, dev, capi, ctx, rows_total, world, rank, seed_shift=0):
    """Rank's contiguous row block of the chunk-seeded global corpus -> a capi.Corpus in HBM."""
    per = (rows_total + world - 1) // world
    lo, hi = min(rank * per, rows_total), min((rank + 1) * per, rows_total)
    corpus = capi.Corpus(ctx, max(hi - lo, 1), row_base=lo)
    for c in range(lo // CHUNK, (max(hi, lo + 1) - 1) // CHUNK + 1):
        c_lo, c_hi = c * CHUNK, min((c + 1) * CHUNK, rows_total)
        a, b = max(lo, c_lo), min(hi, c_hi)
        if a >= b:
            continue
        x = gen_chunk_torch(torch, dev, c + seed_shift, c_hi - c_lo)
        torch.cuda.synchronize(dev)
        sl = x[a - c_lo:b - c_lo]
        corpus.append_dev(sl.data_ptr(), b - a)
        del x, sl
    assert len(corpus) == hi - lo
    return corpus, lo, hi


# ------------------------------------------------------------------ clock sampling ---
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            f = [s.strip() for s in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(smax) if smax else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------ reference arm ----
def run_reference(args):
    """--impl reference: the reference's own CPU path on the host cores, SAME workload (all
    --rows rows, same step count).  The Rust reference cannot be built here (no cargo/rustc;
    model2vec-rs / simsimd not vendored), so this is the oracle port of search_documents
    (oracle/cpu_baseline.c): one SIMD cosine per row (AVX-512 when the host has it, as simsimd
    dispatches), the full result vector, a stable sort, take(top_k) -- single-threaded like the
    reference's loop (src/search/mod.rs:84-104)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    n = args.ref_rows or args.rows
    rows = np.empty((n, 256), dtype=np.float32)
    for c in range((n + CHUNK - 1) // CHUNK):
        a, b = c * CHUNK, min((c + 1) * CHUNK, n)
        rows[a:b] = gen_chunk_numpy(c, min(CHUNK, args.rows - a))[: b - a]
    queries = gen_queries(64)
    steps, warm = max(1, args.steps), min(args.warmup, 2)
    for i in range(warm):
        oracle.baseline_search(rows, queries[i], args.topk, threads=1)
    t0 = time.perf_counter()
    for i in range(steps):
        last = oracle.baseline_search(rows, queries[(warm + i) % 64], args.topk, threads=1)
    dt = (time.perf_counter() - t0) / steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"row": last[0], "distance": last[1]})
    scale = args.rows / n
    qps = 1.0 / (dt * scale)
    nt = oracle.baseline_threads()
    t1 = time.perf_counter()
    oracle.baseline_search(rows, queries[0], args.topk, threads=nt)
    dt_omp = time.perf_counter() - t1
    line = {
        "impl": "reference", "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": 0,
        "steps": steps, "warmup": warm, "ms_per_step": dt * scale * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(args.rows, args.topk), "rows": args.rows, "top_k": args.topk},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": 1, "kind": "port", "isa": oracle.baseline_isa(),
                         "sample": (f"all {n} rows per step" if n == args.rows else f"{n} of {args.rows} rows per step, time scaled x{scale:g}")
                                   + f", {steps} steps, {warm} warm-up (each ~{dt:.1f} s)",
                         "host_cores": os.cpu_count(),
                         "all_cores_not_reference_behaviour": {"threads": nt, "value": 1.0 / (dt_omp * scale)}},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------ helpers -----------
class Env:
    """Everything a section needs."""
    def __init__(self, **kw):
        self.__dict__.update(kw)


class Dist:
    """torch.distributed with one switch: STB_BENCH_ONE_GPU=1 puts every rank on cuda:0 (NCCL refuses two
    ranks on one device) and runs the few collectives bench.py needs on gloo through CPU copies.  That
    mode validates the N>1 code path on a single-GPU box -- its timings mean nothing and the line says so."""
    def __init__(self, dist, torch, dev, one_gpu):
        self.d, self.torch, self.dev, self.one_gpu = dist, torch, dev, one_gpu
        self.ReduceOp = dist.ReduceOp

    def __getattr__(self, name):                                  # barrier, all_gather_object, get_rank, ...
        return getattr(self.d, name)

    def _cpu(self, t):
        return t.detach().cpu() if self.one_gpu else t

    def all_reduce(self, t, op=None):
        c = self._cpu(t)
        self.d.all_reduce(c, op=op)
        if self.one_gpu:
            t.copy_(c)

    def broadcast(self, t, src=0):
        c = self._cpu(t)
        self.d.broadcast(c, src=src)
        if self.one_gpu:
            t.copy_(c)

    def all_gather_into_tensor(self, out, t):
        if not self.one_gpu:
            return self.d.all_gather_into_tensor(out, t)
        self.torch.cuda.synchronize(self.dev)
        parts = [self.torch.empty_like(t, device="cpu") for _ in range(self.d.get_world_size())]
        self.d.all_gather(parts, t.detach().cpu())
        out.copy_(self.torch.stack(parts).reshape(out.shape))


# The stdout line must stay below 1.5 kB, so that a consumer keeping a bounded tail of stdout still gets all of
# it.  The full line goes to --side-json; on stdout the least important keys are dropped, in this order, until it fits.
LINE_LIMIT = 1480
DROPPABLE = (("tier_stats",), ("roofline", "algorithmic_bytes"), ("cpu_baseline", "all_cores_threads"), ("cpu_baseline", "host_cores"),
             ("e2e", "steps"), ("roofline", "peak_source"), ("config", "rows"), ("e2e", "ms_per_step"), ("cpu_baseline", "gpu_rows_equal_cpu_rows"),
             ("per_rank_ms_per_step",), ("clocks", "samples"), ("clocks", "window"), ("roofline", "bytes_read"), ("cpu_baseline", "all_cores_value"),
             ("cpu_baseline", "isa"), ("side",))


def shrink_line(full):
    line = json.loads(json.dumps(full))
    for k in [k for k, v in line.items() if v is None and k not in ("vs_baseline",)]:
        del line[k]                                                   # ranks_agree at N=1, parity_spot_check at N>1, ...
    for path in DROPPABLE:
        if len(json.dumps(line)) <= LINE_LIMIT:
            break
        d = line
        for key in path[:-1]:
            d = d.get(key, {}) if isinstance(d, dict) else {}
        if isinstance(d, dict):
            d.pop(path[-1], None)
    return line


class Watchdog:
    """Deadlines for the multi-rank run.  The fused exchanges are spin-waits on peer memory and the few
    NCCL calls block until every rank arrives: a rank that fails (or a peer that stalls) would otherwise
    leave the job waiting for NCCL's own 10-minute watchdog with nothing printed.  Every rank runs this
    thread; the main thread arms a deadline per phase.  When one passes, rank 0 prints the headline built
    from what has been measured so far (marked "truncated") and every rank leaves with os._exit(0) --
    hung kernels go down with the process.  No collective, no store traffic: the ranks' clocks are aligned
    by the barrier that precedes every arm()."""

    def __init__(self, rank, emit, total_s=720.0):
        self.rank, self.emit = rank, emit
        self.deadline, self.label, self.budget = None, None, 0.0
        self.total_s, self.t_end = float(total_s), time.monotonic() + float(total_s)   # the whole run, whatever the phases do
        # one node: a file every rank can see tells the others that one rank is leaving (same parent = the
        # torchrun agent, so the name is unique to this job); no collective, no store traffic
        self.flag = os.path.join(tempfile.gettempdir(), f"stb_bench_leave_{os.getppid()}_{os.environ.get('MASTER_PORT', '0')}")
        if rank == 0:
            try:
                os.unlink(self.flag)
            except OSError:
                pass
        self.lock = threading.Lock()
        self.done = False
        t = threading.Thread(target=self._run, daemon=True)
        t.start()

    def arm(self, label, seconds):
        seconds = float(seconds) * float(os.environ.get("STB_BENCH_DEADLINE_SCALE", "1"))   # tests shrink the deadlines
        with self.lock:
            self.label, self.budget, self.deadline = label, float(seconds), time.monotonic() + float(seconds)

    def disarm(self):
        with self.lock:
            self.deadline = None

    def fire(self, reason):
        """Print what exists (rank 0) and leave.  Also called by a rank whose section raised."""
        with self.lock:
            if self.done:
                return
            self.done = True
        print(f"[rank {self.rank}] leaving: {reason}", file=sys.stderr, flush=True)
        try:
            open(self.flag, "w").write(f"rank {self.rank}: {reason}\n")
        except OSError:
            pass
        if self.emit is None:                                  # nothing measured yet: an error, not a result
            if self.rank == 0:
                print(json.dumps({"error": reason}), flush=True)
            os._exit(1)
        if self.rank == 0:
            try:
                self.emit(reason)
            finally:
                sys.stdout.flush()
        os._exit(0)

    def park(self, reason):
        """A non-zero rank whose section raised: the peers are inside a collective or a spin-wait and will
        run into their own deadline; stay alive until ours (torchrun kills the job if a rank dies)."""
        print(f"[rank {self.rank}] {reason}; leaving shortly", file=sys.stderr, flush=True)
        try:
            open(self.flag, "w").write(f"rank {self.rank}: {reason}\n")       # rank 0 prints the line when it sees this
        except OSError:
            pass
        with self.lock:                                        # 10 s for rank 0 to print, then this rank goes too
            self.deadline = min(self.deadline or float("inf"), time.monotonic() + 10.0)
        while True:
            time.sleep(1.0)

    def _run(self):
        while True:
            time.sleep(0.25)
            with self.lock:
                d, label, budget = self.deadline, self.label, self.budget
            if d is not None and time.monotonic() > d:
                self.fire(f"phase '{label}' exceeded its {budget:.0f} s deadline")
            if time.monotonic() > self.t_end:
                self.fire(f"the run exceeded {self.total_s:.0f} s (phase '{label}')")
            if os.path.exists(self.flag):
                try:
                    why = open(self.flag).read().strip()
                except OSError:
                    why = "another rank left"
                self.fire(f"phase '{label}': {why}")


def timed_queries(E, corpus, q_dev, k, steps, warm, xchg=None):
    """Pipelined device-timed top-k queries (stb_search_topk_dev / stb_search_topk_xchg).
    Returns (ms per query [max over ranks], status array of the timed steps, hits tensor)."""
    torch, dev, stream = E.torch, E.dev, E.stream
    n_q = q_dev.shape[0]
    hits = torch.zeros((steps + warm, k, 2), dtype=torch.float64, device=dev)
    st = torch.zeros((steps + warm, 4), dtype=torch.int32, device=dev)

    def step(i):
        if xchg is not None:
            xchg.search_topk(corpus, q_dev[i % n_q].data_ptr(), k, hits[i].data_ptr(), st[i].data_ptr())
        else:
            corpus.search_topk_dev(q_dev[i % n_q].data_ptr(), k, hits[i].data_ptr(), st[i].data_ptr())

    for i in range(warm):
        step(i)
    E.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(warm, warm + steps):
        step(i)
    e1.record(stream)
    E.barrier()
    mine = e0.elapsed_time(e1) / steps
    E.last_per_rank_ms = E.gather_over_ranks(mine)
    ms = max(E.last_per_rank_ms)
    return ms, st[warm:].cpu().numpy(), hits[warm:]


def clock_load(E, corpus, q_dev, k, n, xchg=None):
    """nvidia-smi reports a clock sample every 100 ms; the timed region is a few milliseconds.  Right after it,
    the SAME queries keep running (untimed, n of them, ~0.4 s) so that the samples bench.py reports are taken
    under this load and not on an idle GPU."""
    torch, dev = E.torch, E.dev
    hits = torch.zeros((64, k, 2), dtype=torch.float64, device=dev)
    st = torch.zeros((64, 4), dtype=torch.int32, device=dev)
    n_q = q_dev.shape[0]
    for i in range(n):
        if xchg is not None:
            xchg.search_topk(corpus, q_dev[i % n_q].data_ptr(), k, hits[i % 64].data_ptr(), st[i % 64].data_ptr())
        else:
            corpus.search_topk_dev(q_dev[i % n_q].data_ptr(), k, hits[i % 64].data_ptr(), st[i % 64].data_ptr())
    torch.cuda.synchronize(dev)


def e2e_queries(E, corpus, queries_h, k, steps, xchg=None):
    """Synchronous host calls: host query in, host hits out (stb_search / stb_search_xchg)."""
    n_q = len(queries_h)

    def one(i):
        if xchg is not None:
            return xchg.search(corpus, queries_h[i % n_q], k)[0]
        return corpus.search(queries_h[i % n_q], top_k=k)

    for i in range(3):
        one(i)
    E.barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        one(i)
    E.torch.cuda.synchronize(E.dev)
    return E.max_over_ranks(time.perf_counter() - t0) / steps * 1e3


def e2e_queries_many(E, corpus, queries_h, k, steps, xchg=None, group=16):
    """Host queries in, host hits out through stb_search_many: `group` independent queries per call (ONE
    H2D copy of the group's queries from pinned memory, one kernel per query enqueued back to back, hits
    written to pinned host memory, ONE synchronisation per call).  Every query's input and result cross the
    PCIe bus inside the timed region.  Returns ms per query."""
    n_q = len(queries_h)
    calls = max(1, steps // group)

    def one(c):
        idx = [(c * group + j) % n_q for j in range(group)]
        return corpus.search_many(queries_h[idx], top_k=k, xchg=xchg)

    one(0)
    E.barrier()
    t0 = time.perf_counter()
    for c in range(calls):
        one(c)
    E.torch.cuda.synchronize(E.dev)
    return E.max_over_ranks(time.perf_counter() - t0) / (calls * group) * 1e3


# ------------------------------------------------------------------ side sections -----
def side_k1_tiers(E, corpus, q_dev, queries_h, k, rows):
    """The three candidate tiers on the headline corpus, same loop as `value` (N=1)."""
    out = {}
    ref = None
    corpus.prepare()                                     # q8 + h16
    for tier in TIER_NAMES:
        os.environ["STB_SCAN_TIER"] = tier
        try:
            ms, st, hits = timed_queries(E, corpus, q_dev, k, 32, 4)
            e2e_ms = e2e_queries(E, corpus, queries_h, k, 16)
        finally:
            os.environ.pop("STB_SCAN_TIER", None)
        if ref is None:
            ref = hits.clone()
        out[tier] = {"us_per_query": ms * 1e3, "GBps_read": rows * TIER_BYTES[tier] / ms / 1e6, "e2e_ms": e2e_ms,
                     "proven": int((st[:, 1] == 1).sum()), "of": len(st),
                     "bit_identical_to_f32": bool(E.torch.equal(hits.view(E.torch.int64), ref.view(E.torch.int64)))}
    return out


def side_config2(E, k, n=1_000_000):
    """BASELINE configs[1]: 1M-line corpus, single query, top-k=10, 1xB200."""
    capi, torch, dev = E.capi, E.torch, E.dev
    x = gen_chunk_torch(torch, dev, 2002, n)
    c = capi.Corpus(E.ctx, n)
    torch.cuda.synchronize(dev); c.append_dev(x.data_ptr(), n); del x
    c.prepare()
    qh = gen_queries(96)[64:]
    q_dev = torch.from_numpy(qh).to(dev)
    out = {"workload": "%d-line corpus, single query, top-k=%d (BASELINE configs[1])" % (n, k)}
    for tier in ("q8", "f32"):
        os.environ["STB_SCAN_TIER"] = tier
        try:
            ms, st, _ = timed_queries(E, c, q_dev, k, 100, 10)
            e2e_ms = e2e_queries(E, c, qh, k, 50)
        finally:
            os.environ.pop("STB_SCAN_TIER", None)
        out[tier] = {"us_per_query": ms * 1e3, "qps": 1e3 / ms, "e2e_us": e2e_ms * 1e3, "proven": int((st[:, 1] == 1).sum()), "of": len(st),
                     "frac_of_hbm_peak_algorithmic": n * 1024 / ms / 1e6 / E.peak_gbs,
                     "frac_of_hbm_peak_bytes_read": n * TIER_BYTES[tier] / ms / 1e6 / E.peak_gbs}
    c.close()
    return out


def side_batch(E, corpus, rows, k, nq=1024, iters=5, make_xchg=None):
    """BASELINE configs[2]: 10M-line corpus, batch of 1024 queries, top-k=10 through the tcgen05
    path.  Sharded (N>1): K2 per shard, then ONE exchange of the nq x k hits over NVLink peer memory
    inside two small kernels (stb_search_batch_xchg_dev: push + wait/merge; NCCL all-gather + merge
    kernel with --exchange nccl).  Unproven queries are re-run INSIDE the timed region (round 1 left
    them out): N=1 through the single-query path, N>1 through the fused single-query exchange on
    every rank (all ranks see the same proof flags)."""
    torch, dev, stream, dist, world, capi = E.torch, E.dev, E.stream, E.dist, E.world, E.capi
    qh = gen_queries(nq + 64)[64:]
    q_dev = torch.from_numpy(qh).to(dev)
    hits = torch.zeros((nq, k, 2), dtype=torch.float64, device=dev)
    st = torch.zeros((nq, 2), dtype=torch.int32, device=dev)
    st1 = torch.zeros((4,), dtype=torch.int32, device=dev)
    merged = torch.zeros((nq, k, 2), dtype=torch.float64, device=dev)
    gathered = st_all = None
    xb = None
    if world > 1 and make_xchg is not None:
        xb = make_xchg(max_nq=nq)
    elif world > 1:
        gathered = torch.zeros((world, nq, k, 2), dtype=torch.float64, device=dev)
        st_all = torch.zeros((world, nq, 2), dtype=torch.int32, device=dev)
    corpus.prepare()
    if world > 1:
        # first-call costs (shadow build, kernel attributes, workspaces) stay local; the ranks then enter the
        # exchange together: its wait is bounded (STB_XCHG_TIMEOUT_CYCLES), a rank arriving later than that is "gone"
        corpus.search_batch_dev(q_dev.data_ptr(), nq, k, hits.data_ptr(), st.data_ptr())
        E.barrier()
    fused_note = None
    if xb is not None:
        # probe: one fused exchange; if ANY rank saw a peer time out, every rank switches to the NCCL exchange
        # (a timed-out exchange object is dead -- include/semtools_b200.h -- and the ranks must keep issuing
        # the same calls)
        xb.search_batch_dev(corpus, q_dev.data_ptr(), nq, k, merged.data_ptr(), st.data_ptr())
        flag = torch.tensor([int(bool((st[:, 1] == 2).any()))], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if int(flag.item()):
            xb.close()
            xb = None
            fused_note = "the fused peer-memory exchange timed out on at least one rank in its probe batch; measured with the NCCL exchange"
            gathered = torch.zeros((world, nq, k, 2), dtype=torch.float64, device=dev)
            st_all = torch.zeros((world, nq, 2), dtype=torch.int32, device=dev)
    fallbacks = []

    def one():
        if world == 1:
            corpus.search_batch_dev(q_dev.data_ptr(), nq, k, hits.data_ptr(), st.data_ptr())
            bad = (st[:, 1] != 1).nonzero().flatten().tolist()          # synchronises: the product path does too
            for i in bad:                                                # exact single-query path for the unproven
                corpus.search_topk_dev(q_dev[i].data_ptr(), k, hits[i].data_ptr(), st1.data_ptr())
        elif xb is not None:
            xb.search_batch_dev(corpus, q_dev.data_ptr(), nq, k, merged.data_ptr(), st.data_ptr())
            if bool((st[:, 1] == 2).any()):                              # a peer never arrived: the ranks no longer agree on
                raise RuntimeError("fused batch exchange: a peer rank timed out")   # what to re-run -- stop here
            bad = (st[:, 1] != 1).nonzero().flatten().tolist()          # identical on every rank
            for i in bad:
                xb.search_topk(corpus, q_dev[i].data_ptr(), k, merged[i].data_ptr(), st1.data_ptr())
        else:
            corpus.search_batch_dev(q_dev.data_ptr(), nq, k, hits.data_ptr(), st.data_ptr())
            dist.all_gather_into_tensor(gathered, hits)
            dist.all_gather_into_tensor(st_all, st)
            E.ctx.hits_merge_batch_dev(gathered.data_ptr(), world, nq, k, k, merged.data_ptr())
            bad = (st_all[:, :, 1].min(dim=0).values != 1).nonzero().flatten().tolist()
            for i in bad:                                                # every rank re-runs its shard, then one more exchange
                corpus.search_topk_dev(q_dev[i].data_ptr(), k, hits[i].data_ptr(), st1.data_ptr())
            if bad:
                dist.all_gather_into_tensor(gathered, hits)
                E.ctx.hits_merge_batch_dev(gathered.data_ptr(), world, nq, k, k, merged.data_ptr())
        fallbacks.append(len(bad))

    for _ in range(2):
        one()
    E.barrier()
    fallbacks.clear()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(iters):
        one()
    e1.record(stream)
    E.barrier()
    ms = E.max_over_ranks(e0.elapsed_time(e1)) / iters
    out = {"workload": f"{rows}-line corpus{'' if world == 1 else f' row-sharded x{world}'}, batch of {nq} queries, top-k={k} (BASELINE configs[2])",
           "value": nq / ms * 1e3, "unit": "queries/s", "ms_per_batch": ms, "dtype": "fp16 candidates (tcgen05 kind::f16, f32 TMEM) + f64 exact re-rank",
           "TFLOPs_pipeline": 2.0 * nq * rows * 256 / ms / 1e9, "fallback_queries_per_batch": float(np.mean(fallbacks)),
           "fallbacks_timed": True}
    out["frac_of_bf16_peak_pipeline"] = out["TFLOPs_pipeline"] / (E.peak_tf * world)
    if world == 1:
        t0 = time.perf_counter()
        res = corpus.search_batch(qh, top_k=k)                       # host queries in, host hits out
        e2e_s = time.perf_counter() - t0
        out["e2e"] = {"value": nq / e2e_s, "unit": "queries/s", "ms_per_batch": e2e_s * 1e3, "h2d_bytes_per_step": nq * 1024,
                      "d2h_bytes_per_step": nq * (16 * k + 8)}
        out["agrees_with_single_query_path"] = all(np.array_equal(res[i], corpus.search(qh[i], top_k=k)) for i in range(4))
    else:
        ref = merged.clone()
        dist.broadcast(ref, src=0)
        agree = torch.tensor([int(torch.equal(ref.view(torch.int64), merged.view(torch.int64)))], device=dev)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
        out["ranks_agree"] = bool(agree.item())
        out["exchange"] = ("fused: push + wait/merge kernels over NVLink peer memory (stb_search_batch_xchg_dev)" if xb is not None
                           else "nccl all_gather of nq x k hits + stb_hits_merge_batch_dev")
        if fused_note:
            out["note"] = fused_note
        # spot-check against the single-query fused path (exact by its own proof)
        chk = torch.zeros((k, 2), dtype=torch.float64, device=dev)
        same = True
        if xb is not None:
            for i in (0, nq // 2, nq - 1):
                xb.search_topk(corpus, q_dev[i].data_ptr(), k, chk.data_ptr(), st1.data_ptr())
                torch.cuda.synchronize(dev)
                same = same and bool(torch.equal(chk.view(torch.int64), merged[i].view(torch.int64)))
            out["agrees_with_single_query_path"] = same
            xb.close()
    return out


def side_config4(E, args, k, xchg_factory):
    """BASELINE configs[3]: 100M-line corpus row-sharded over the ranks (N=1: the whole corpus on
    one GPU, 102.4 GB f32 + 26 GB q8 -- the comparator the >=6x claim needs), single query."""
    capi, torch, dev = E.capi, E.torch, E.dev
    rows = args.config4_rows
    if E.world > 1 and xchg_factory is None:
        return {"skipped": "the sharded 100M-line section runs on the fused peer-memory exchange (--exchange p2p)"}
    torch.cuda.empty_cache()
    corpus, lo, hi = fill_shard(torch, dev, capi, E.ctx, rows, E.world, E.rank, seed_shift=4000)
    corpus.prepare(1)                                                 # q8 only: K2's shadow is not needed here
    qh = gen_queries(128)[96:]
    q_dev = torch.from_numpy(qh).to(dev)
    xchg = xchg_factory() if E.world > 1 else None
    steps = 40 if E.world > 1 else 20
    ms, st, hits = timed_queries(E, corpus, q_dev, k, steps, 4, xchg=xchg)
    e2e_ms = e2e_queries(E, corpus, qh, k, 10, xchg=xchg)
    tier = TIER_NAMES[int(st[0, 3]) >> 16]
    rpg = hi - lo
    out = {"workload": f"{rows}-line corpus row-sharded x{E.world} ({rpg} rows/GPU), single query, top-k={k} (BASELINE configs[3])",
           "value": 1e3 / ms, "unit": "queries/s", "ms_per_query": ms, "e2e_ms_per_query": e2e_ms, "tier": tier,
           "proven": int((st[:, 1] == 1).sum()), "of": len(st),
           "per_gpu_GBps_algorithmic": rpg * 1024 / ms / 1e6, "per_gpu_GBps_read": rpg * TIER_BYTES[tier] / ms / 1e6,
           "frac_of_hbm_peak_bytes_read": rpg * TIER_BYTES[tier] / ms / 1e6 / E.peak_gbs}
    if xchg is not None:
        xchg.close()
    corpus.close()
    torch.cuda.empty_cache()
    return out


def clustered_shard(E, rows_total, lo, hi, n_centers, spread=0.6):
    """Clustered synthetic rows (random unit vectors have no neighbourhood structure for an IVF to
    exploit): row = normalise(center + noise); chunk-seeded, identical for any world size."""
    capi, torch, dev = E.capi, E.torch, E.dev
    g = torch.Generator(device=dev); g.manual_seed(SEED + 5)
    centers = torch.randn((n_centers, 256), generator=g, device=dev); centers /= centers.norm(dim=1, keepdim=True)
    c = capi.Corpus(E.ctx, max(hi - lo, 1), row_base=lo)
    for chunk_id in range(lo // CHUNK, (hi + CHUNK - 1) // CHUNK):
        gc = torch.Generator(device=dev); gc.manual_seed(SEED + 1000 + chunk_id)
        idx = torch.randint(0, n_centers, (CHUNK,), generator=gc, device=dev)
        x = centers[idx] + spread / 16.0 * torch.randn((CHUNK, 256), generator=gc, device=dev)
        x /= x.norm(dim=1, keepdim=True)
        a, b = max(lo, chunk_id * CHUNK), min(hi, (chunk_id + 1) * CHUNK)
        part = x[a - chunk_id * CHUNK: b - chunk_id * CHUNK].contiguous()
        torch.cuda.synchronize(dev); c.append_dev(part.data_ptr(), b - a)
        del x, part
    gq = torch.Generator(device=dev); gq.manual_seed(SEED + 6)
    idx = torch.randint(0, n_centers, (64,), generator=gq, device=dev)
    q = centers[idx] + spread / 16.0 * torch.randn((64, 256), generator=gq, device=dev); q /= q.norm(dim=1, keepdim=True)
    return c, q.cpu().numpy()


def side_ivfpq(E, args, nlist=4096, nprobe=64, make_xchg=None):
    """BASELINE configs[4] (IVF-PQ; self-specified: the reference has no IVF_PQ, so no parity --
    recall@10 against the exact scan of the same rows is the quality metric).  N=1: --ivfpq-rows
    clustered rows on one GPU.  N>1: --ivfpq-rows-per-gpu rows per GPU, sharded by ROW (one index
    per rank over its block, per-rank top-k, all-gather of k hits, K4 merge); at N=8 that is the
    named 100M-line / nlist 4096 / nprobe 64 configuration."""
    from semtools_b200.sharded import ShardedCorpus, shard_bounds
    capi, torch, dev, dist = E.capi, E.torch, E.dev, E.dist
    rows = args.ivfpq_rows if E.world == 1 else args.ivfpq_rows_per_gpu * E.world
    lo, hi = shard_bounds(rows, E.world, E.rank)
    # exact re-scores per query per shard: the PQ ranking gets noisier as the lists grow (12.5M-row shards scan
    # ~195k codes per query), so the large configuration re-ranks the kernel's maximum
    rerank = 512 if (hi - lo) <= 5_000_000 else 1024
    torch.cuda.empty_cache()
    c, qh = clustered_shard(E, rows, lo, hi, max(rows // 100, 1000))
    t0 = time.perf_counter()
    index = capi.IvfPq(c, nlist=nlist, train_rows=262144, iters=8)
    E.torch.cuda.synchronize(dev)
    build_s = E.max_over_ranks(time.perf_counter() - t0)
    xq = None
    if E.world == 1:
        search_exact = lambda i: c.search(qh[i], top_k=10)
        search_ivf = lambda i: index.search(qh[i], nprobe=nprobe, top_k=10, rerank=rerank)
    else:
        # exact comparator: the fused single-query exchange (stb_search_xchg) over the same shards;
        # IVF-PQ: stb_ivfpq_search_dev per rank -> all-gather of the k hits -> stb_hits_merge_dev -> one D2H
        c.prepare(1)
        xq = make_xchg() if make_xchg is not None else None
        exact_sc = ShardedCorpus.on_gpu(E.ctx, c, dist, dev)
        search_exact = (lambda i: xq.search(c, qh[i], 10)[0]) if xq is not None else (lambda i: exact_sc.search(qh[i], 10))
        q_pin = torch.from_numpy(qh).pin_memory()
        q_d = torch.empty(256, dtype=torch.float32, device=dev)
        loc = torch.zeros((10, 2), dtype=torch.float64, device=dev)
        st2 = torch.zeros(2, dtype=torch.int32, device=dev)
        gat = torch.zeros((E.world, 10, 2), dtype=torch.float64, device=dev)
        mer = torch.zeros((10, 2), dtype=torch.float64, device=dev)
        out_pin = torch.zeros((10, 2), dtype=torch.float64).pin_memory()

        def search_ivf(i):
            q_d.copy_(q_pin[i], non_blocking=True)
            index.search_dev(q_d.data_ptr(), nprobe, 10, rerank, loc.data_ptr(), st2.data_ptr())
            dist.all_gather_into_tensor(gat, loc)
            E.ctx.hits_merge_dev(gat.data_ptr(), E.world, 10, 10, mer.data_ptr())
            out_pin.copy_(mer, non_blocking=True)
            torch.cuda.synchronize(dev)
            h = np.ascontiguousarray(out_pin.numpy()).view(capi.HIT_DTYPE).reshape(-1).copy()
            return h[h["row"] != np.uint64(0xFFFFFFFFFFFFFFFF)], 0
    ivf_path = "stb_ivfpq_search_dev per rank -> nccl all_gather of k hits -> stb_hits_merge_dev -> one D2H"
    if E.world > 1:
        # the device-resident per-rank probe must return what the host call returns (ShardedCorpus.on_gpu_ivfpq:
        # stb_ivfpq_search per rank, all-gather, host merge); if it does not on ANY rank, every rank times the host form
        approx = ShardedCorpus.on_gpu_ivfpq(E.ctx, index, dist, dev, nprobe=nprobe, rerank=rerank)
        same = 1
        try:
            for i in range(3):
                a, b = search_ivf(i)[0], approx.search(qh[i], 10)
                same &= int(np.array_equal(a["row"], b["row"]) and np.array_equal(a["distance"], b["distance"]))
        except capi.StbError:
            same = 0
        flag = torch.tensor([same], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            search_ivf = lambda i: (approx.search(qh[i], 10), 0)
            ivf_path = "stb_ivfpq_search per rank (host hits) -> all_gather -> host merge (the device-resident form disagreed with it)"
    want = [search_exact(i) for i in range(64)]
    E.barrier()
    t0 = time.perf_counter()
    for i in range(64):
        search_exact(i)
    exact_ms = E.max_over_ranks(time.perf_counter() - t0) / 64 * 1e3
    rec, scanned = [], []
    for i in range(3):
        search_ivf(i)
    E.barrier()
    t0 = time.perf_counter()
    got = [search_ivf(i) for i in range(64)]
    ms = E.max_over_ranks(time.perf_counter() - t0) / 64 * 1e3
    for i in range(64):
        rec.append(len(set(got[i][0]["row"].tolist()) & set(want[i]["row"].tolist())) / 10.0)
        scanned.append(got[i][1])
    stt = index.stats()
    # local probe alone (no exchange): what one rank's ADC kernel pair costs per query
    t0 = time.perf_counter()
    loc = [index.search(qh[i], nprobe=nprobe, top_k=10, rerank=rerank) for i in range(64)]
    local_ms = E.max_over_ranks(time.perf_counter() - t0) / 64 * 1e3
    local_scanned = float(np.mean([x[1] for x in loc]))
    if xq is not None:
        xq.close()
    index.close(); c.close()
    torch.cuda.empty_cache()
    return {"workload": f"{rows} clustered rows{'' if E.world == 1 else f' row-sharded x{E.world}'}, nlist={nlist}{'' if E.world == 1 else ' per shard'}, nprobe={nprobe}, m=32x8bit, rerank={rerank}, top-k=10"
                        + (" (BASELINE configs[4])" if rows == 100_000_000 and E.world == 8 else ""),
            "parity": "unpinned (no IVF_PQ exists in the reference); quality = recall vs exact scan",
            "recall_at_10": float(np.mean(rec)), "min_recall": float(np.min(rec)), "build_s": build_s,
            "qps_e2e": 1e3 / ms, "ms_per_query_e2e": ms, "exact_scan_ms_per_query_e2e": exact_ms,
            "local_probe_ms_per_query": local_ms, "scanned_rows_per_query_per_gpu": local_scanned,
            "code_bytes_per_query_per_gpu": local_scanned * 32 + nlist * 1024 + 32768,
            "index_bytes_per_gpu": stt["index_bytes"], "max_list": stt["max_list"],
            "exchange": None if E.world == 1 else ivf_path + "; exact comparator: fused stb_search_xchg (q8 tier)"}


def side_embed(E, V=500_000, n_lines=1_000_000):
    """K3 on SURVEY 8d's synthetic ingestion batch: V=500k x 256 table (0.5 GB), line lengths ~
    clamp(round(LogNormal(2.5,0.8)),0,2048), ids ~ Zipf(1.1).  Algorithmic bytes = sum_i (1028*T_i + 1024)."""
    capi, torch, dev, stream = E.capi, E.torch, E.dev, E.stream
    rng = np.random.default_rng(SEED + 77)
    Emb = (rng.standard_normal((V, 256), dtype=np.float32) * np.float32(0.1))
    T = np.clip(np.round(rng.lognormal(2.5, 0.8, n_lines)), 0, 2048).astype(np.int64)
    offsets = np.concatenate([[0], np.cumsum(T)]).astype(np.uint64)
    ids = ((rng.zipf(1.1, int(T.sum())) - 1) % V).astype(np.uint32)
    table = capi.Table(E.ctx, Emb)
    off_d = torch.from_numpy(offsets.view(np.int64)).to(dev)
    ids_d = torch.from_numpy(ids.view(np.int32)).to(dev)
    out_d = torch.empty((n_lines, 256), dtype=torch.float32, device=dev)
    torch.cuda.synchronize(dev)
    for _ in range(3):
        capi.embed_dev(E.ctx, table, off_d.data_ptr(), ids_d.data_ptr(), n_lines, out_d.data_ptr())
    capi.embed_status(E.ctx)
    iters = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(iters):
        capi.embed_dev(E.ctx, table, off_d.data_ptr(), ids_d.data_ptr(), n_lines, out_d.data_ptr())
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / iters
    alg_bytes = float((1028 * T + 1024).sum())
    corpus = capi.Corpus(E.ctx, n_lines)
    t0 = time.perf_counter()
    capi.embed(E.ctx, table, offsets, ids, out=False, append_to=corpus)       # host CSR in, rows stay in HBM
    e2e_s = time.perf_counter() - t0
    import oracle
    n_chk = min(2000, n_lines)
    exp = oracle.embed_csr(Emb, offsets[:n_chk + 1], ids[:int(offsets[n_chk])])
    bit_exact = bool(np.array_equal(corpus.read(0, n_chk).view(np.uint32), exp.view(np.uint32)))
    corpus.close(); table.close()
    return {"kernel": "stb_embed_kernel", "lines": n_lines, "tokens": int(T.sum()), "table_rows": V,
            "ms": ms, "lines_per_s": n_lines / (ms * 1e-3), "achieved_GBps": alg_bytes / (ms * 1e-3) / 1e9,
            "frac_of_hbm_peak": alg_bytes / (ms * 1e-3) / 1e9 / E.peak_gbs,
            "bound": "hbm/l2 (random 1 KiB gathers, Zipf ids)", "e2e_lines_per_s": n_lines / e2e_s,
            "e2e_h2d_bytes": int(ids.nbytes + offsets.nbytes), "bit_exact_vs_oracle_first_2000": bit_exact}


def cpu_baseline_section(corpus, queries_h, rows, k):
    """oracle/cpu_baseline.c (the reference's scan restated) on the host cores over ALL rows of the
    benchmarked corpus (downloaded from HBM), 3 queries, 1 thread = faithful."""
    import oracle
    sample = corpus.read(0, rows)
    oracle.baseline_search(sample[:1000], queries_h[0], k, threads=1)
    ts = []
    for i in range(3):
        t0 = time.perf_counter()
        r1 = oracle.baseline_search(sample, queries_h[i], k, threads=1)
        ts.append(time.perf_counter() - t0)
    t = float(np.median(ts))
    nt = oracle.baseline_threads()
    t0 = time.perf_counter()
    oracle.baseline_search(sample, queries_h[0], k, threads=nt)
    tN = time.perf_counter() - t0
    got = corpus.search(queries_h[2], top_k=k)
    same_rows = bool(got["row"].tolist() == [int(x) for x in r1[0]])
    return {"value": float(f"{1.0 / t:.5g}"), "unit": "queries/s", "cores": 1, "kind": "port", "isa": oracle.baseline_isa(),
            "sample": f"all {rows} rows, 3 queries, median {t:.2f} s each",
            "host_cores": os.cpu_count(), "all_cores_value": float(f"{1.0 / tN:.5g}"), "all_cores_threads": nt,
            "gpu_rows_equal_cpu_rows": same_rows}


# ------------------------------------------------------------------ our arm ----------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from semtools_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    one_gpu = os.environ.get("STB_BENCH_ONE_GPU") == "1" and world > 1
    if one_gpu:
        local_rank = 0
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if one_gpu:
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=dev)
    dist = Dist(dist, torch, dev, one_gpu)
    # N > 1: deadlines from the first collective on (see Watchdog); until the headline exists a missed
    # deadline is an error exit, afterwards it costs the unfinished side sections only
    wd = Watchdog(rank, None) if world > 1 else None
    if wd is not None:
        wd.arm("corpus fill + headline measurements", 420.0)

    # a dedicated non-default stream shared by torch (events, NCCL ordering) and the library
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx = capi.Context(local_rank, stream.cuda_stream)
    assert ctx.stream == stream.cuda_stream != 0
    k = args.topk

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        if world == 1:
            return float(v)
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather_over_ranks(v):
        if world == 1:
            return [float(v)]
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        out = torch.zeros(world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(out, t)
        return [float(x) for x in out.cpu()]

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy, burst)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    E = Env(torch=torch, dist=dist, capi=capi, dev=dev, stream=stream, ctx=ctx, world=world, rank=rank,
            barrier=barrier, max_over_ranks=max_over_ranks, gather_over_ranks=gather_over_ranks, last_per_rank_ms=None,
            peak_gbs=peak, peak_tf=float(peaks.get("bf16_tflops", 1590.0)))

    # ---- corpus shard of this rank (strong scaling: the SAME global corpus) + candidate copies --------
    corpus, lo, hi = fill_shard(torch, dev, capi, ctx, args.rows, world, rank)
    torch.cuda.empty_cache()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream); corpus.prepare(1); e1.record(stream); torch.cuda.synchronize(dev)
    q8_build_ms = e0.elapsed_time(e1)

    n_q = 64
    queries_h = gen_queries(n_q)
    q_dev = torch.from_numpy(queries_h).to(dev)

    # ---- exchange wiring (N > 1) ---------------------------------------------------------
    exchange = "none"

    def make_xchg(max_nq=0):
        x = capi.Exchange(ctx, world, rank, k, max_nq=max_nq)
        handles = [None] * world
        dist.all_gather_object(handles, x.local_handle())
        x.connect(handles)
        return x

    xchg = None
    if world > 1:
        exchange = args.exchange
        if exchange == "p2p":
            try:
                xchg = make_xchg()
                ok = torch.ones(1, device=dev)
            except capi.StbError as e:
                print(f"[rank {rank}] p2p exchange unavailable ({e}); using nccl", file=sys.stderr)
                ok = torch.zeros(1, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if ok.item() == 0:
                xchg, exchange = None, "nccl"

    # ---- value: inputs resident in HBM, device-timed ---------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)
    launches0 = ctx.counters()["kernel_launches"]
    if world > 1 and xchg is None:                       # NCCL baseline: local K1 -> all_gather -> K4 merge kernel
        n_slots = args.steps + args.warmup
        local_hits = torch.zeros((n_slots, k, 2), dtype=torch.float64, device=dev)
        status = torch.zeros((n_slots, 4), dtype=torch.int32, device=dev)
        gathered = torch.zeros((world, k, 2), dtype=torch.float64, device=dev)
        final_hits = torch.zeros((n_slots, k, 2), dtype=torch.float64, device=dev)

        def step(i):
            corpus.search_topk_dev(q_dev[i % n_q].data_ptr(), k, local_hits[i].data_ptr(), status[i].data_ptr())
            dist.all_gather_into_tensor(gathered, local_hits[i])
            ctx.hits_merge_dev(gathered.data_ptr(), world, k, k, final_hits[i].data_ptr())
        for i in range(args.warmup):
            step(i)
        barrier()
        launches0 = ctx.counters()["kernel_launches"]
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for i in range(args.warmup, n_slots):
            step(i)
        ev1.record(stream)
        barrier()
        per_rank_ms = gather_over_ranks(ev0.elapsed_time(ev1) / args.steps)
        ms_step = max(per_rank_ms)
        st = status[args.warmup:].cpu().numpy()
        hits_t = final_hits[args.warmup:]
    else:
        # warm-up launches are counted out below
        ms_step, st, hits_t = timed_queries(E, corpus, q_dev, k, args.steps, args.warmup, xchg=xchg)
        per_rank_ms = E.last_per_rank_ms
    launches = ctx.counters()["kernel_launches"] - launches0 - (args.warmup if (world == 1 or xchg is not None) else 0)
    load_n = 0
    if (world == 1 or xchg is not None) and args.clock_load_queries > 0:
        load_n = args.clock_load_queries * world                   # same wall time at every N (shards shrink with N)
        clock_load(E, corpus, q_dev, k, load_n, xchg=xchg)
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = f"timed region + {load_n} untimed queries of the same kind"
    n_expect = min(k, args.rows) if xchg is not None else min(k, hi - lo)
    all_complete = bool((st[:, 1] == 1).all() and (st[:, 0] == n_expect).all())
    tier = TIER_NAMES[int(st[0, 3]) >> 16]
    if args.dump_outputs and rank == 0:
        last = np.ascontiguousarray(hits_t[-1].cpu().numpy()).view(capi.HIT_DTYPE).reshape(-1)
        dump_outputs(args.dump_outputs, last[last["row"] != np.uint64(0xFFFFFFFFFFFFFFFF)])   # unused tail: row = UINT64_MAX

    ranks_agree = None
    if world > 1:
        mine = hits_t[:min(args.steps, 16)].contiguous().view(torch.int64)
        ref = mine.clone()
        dist.broadcast(ref, src=0)
        agree = torch.tensor([int(torch.equal(ref, mine))], device=dev)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
        ranks_agree = bool(agree.item())

    # ---- e2e: host query in, host hits out, every step synchronous -------------------
    e2e_steps = max(10, min(args.steps, 100))
    if world > 1 and xchg is None:
        q_pin = torch.from_numpy(queries_h).pin_memory()
        out_pin = torch.zeros((k, 2), dtype=torch.float64).pin_memory()
        barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            q_dev[i % n_q].copy_(q_pin[i % n_q], non_blocking=True)
            step(i % n_slots)
            out_pin.copy_(final_hits[i % n_slots], non_blocking=True)
            torch.cuda.synchronize(dev)
        e2e_ms = max_over_ranks(time.perf_counter() - t0) / e2e_steps * 1e3
    else:
        e2e_ms = e2e_queries(E, corpus, queries_h, k, e2e_steps, xchg=xchg)
    # second e2e figure (stb_search_many, 16 queries per call): single-GPU runs only -- the sharded form of
    # that entry point has not been through a multi-GPU box yet and stays out of the scaling run
    e2e_many_ms = None
    if world == 1:
        try:
            e2e_many_ms = e2e_queries_many(E, corpus, queries_h, k, max(e2e_steps, 64))
        except Exception as e:                                         # noqa: BLE001 - the headline does not depend on it
            print(f"e2e many16 skipped: {type(e).__name__}: {e}", file=sys.stderr)

    # ---- the headline line: everything it needs is measured; side sections only add to it ----------
    rows_per_gpu = hi - lo
    sides = {}
    state = {"check": None, "cpu_base": None, "tier_stats": None}

    def make_line(truncated=None):
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
            ent = tr.get(f"stb_scan_topk_kernel/{tier}/{rows_per_gpu}/k{k}")
            if ent:
                traffic = ent["traffic_bytes"]           # dram read+write of one launch, ncu --set full capture of this kernel
        except (OSError, KeyError, ValueError):
            pass
        achieved = rows_per_gpu * 1024 / ms_step / 1e6
        read_gbs = rows_per_gpu * TIER_BYTES[tier] / ms_step / 1e6
        r5 = lambda v: float(f"{v:.5g}")
        line = {
            "metric": METRIC, "value": r5(1e3 / ms_step), "unit": "queries/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r5(ms_step),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": {"q8": "s8 dp4a scan + f64 exact re-rank", "h16": "f16 scan + f64 exact re-rank", "f32": "f32 scan + f64 exact re-rank"}[tier],
            "data": "synthetic",
            "config": {"workload": workload_name(args.rows, k), "rows": args.rows, "rows_per_gpu": rows_per_gpu, "top_k": k,
                       # the scanned copy is built ONCE per corpus, outside the timed region (like any index): its cost is stated here
                       "tier": tier, "tier_build_ms": float(f"{q8_build_ms:.4g}"),
                       "parallelism": f"row-shard x{world}" + (" ON ONE GPU (functional check, timings void)" if one_gpu else ""),
                       "exchange": exchange,
                       # timing rule: inputs larger than L2 (every query streams the whole copy from HBM) or a flush
                       "l2": (f"scanned copy {rows_per_gpu * TIER_BYTES[tier] / 1e6:.0f} MB = {rows_per_gpu * TIER_BYTES[tier] / 126e6:.1f}x the 126 MB L2, no flush"
                              if rows_per_gpu * TIER_BYTES[tier] > 126e6 else "WARNING: the scanned copy fits in L2 and is not flushed")},
            "clocks": clocks,
            # e2e.value: one synchronous host call per query (stb_search / stb_search_xchg).  many16 (N=1): the same
            # queries through stb_search_many, 16 per call (one H2D, 16 kernels, one sync): what a host holding
            # several queries calls; every query's input and result still cross PCIe inside the timed region
            "e2e": {"value": r5(1e3 / e2e_ms), "unit": "queries/s", "h2d_bytes_per_step": 1024, "d2h_bytes_per_step": 16 * k + 16,
                    "steps": e2e_steps, "ms_per_step": r5(e2e_ms),
                    "many16_value": r5(1e3 / e2e_many_ms) if e2e_many_ms else None},
            "gpu_launches": int(launches), "per_rank_ms_per_step": [r5(v) for v in per_rank_ms],
            "roofline": {"bound": "hbm", "kernel": f"stb_scan_topk_kernel/{tier}", "achieved": r5(achieved), "peak": peak, "unit": "GB/s",
                         "frac": r5(achieved / peak), "traffic": traffic, "peak_source": "measured" if "hbm_gbs" in peaks else "fallback",
                         "algorithmic_bytes": rows_per_gpu * 1024, "bytes_read": rows_per_gpu * TIER_BYTES[tier],
                         "frac_bytes_read": r5(read_gbs / peak)},
            "all_results_proven_exact": all_complete, "ranks_agree": ranks_agree, "parity_spot_check": state["check"],
        }
        if state["tier_stats"] is not None:
            line["tier_stats"] = {t: [v["tries"], v["proven"]] for t, v in state["tier_stats"].items()}
        if state["cpu_base"] is not None:
            line["cpu_baseline"] = state["cpu_base"]
        # one-number summaries of the side sections (details: the {"side": ...} lines above / --side-json)
        summ = {}
        if "batch1024" in sides and "value" in sides["batch1024"]:
            summ["batch1024_qps"] = round(sides["batch1024"]["value"]); summ["batch1024_ms"] = round(sides["batch1024"]["ms_per_batch"], 3)
        if "config2_1M" in sides and "q8" in sides["config2_1M"]:
            summ["config2_1M_us"] = round(sides["config2_1M"]["q8"]["us_per_query"], 1)
        if "config4_100M" in sides and "value" in sides["config4_100M"]:
            summ["config4_100M_qps"] = round(sides["config4_100M"]["value"], 1)
        for nm in ("ivfpq", "ivfpq_sharded"):
            if nm in sides and "recall_at_10" in sides[nm]:
                summ[nm + "_recall"] = round(sides[nm]["recall_at_10"], 3); summ[nm + "_qps"] = round(sides[nm]["qps_e2e"], 1)
        if "k3_embed" in sides and "lines_per_s" in sides["k3_embed"]:
            summ["k3_Mlines_s"] = round(sides["k3_embed"]["lines_per_s"] / 1e6, 1)
        line["side"] = summ
        if truncated:
            line["side_sections_truncated"] = truncated    # the headline figures above were complete before it happened
        return line

    def emit_line(truncated=None):
        full = make_line(truncated)
        line = shrink_line(full)
        if args.side_json:
            try:
                with open(args.side_json, "w") as f:
                    json.dump({"headline": full, "sides": sides}, f, indent=1)
            except OSError as e:
                print(f"--side-json: {e}", file=sys.stderr)
        print(json.dumps(line), flush=True)

    # N > 1: from here on a stalled or failed side section costs that section, not the line (see Watchdog)
    if wd is not None:
        with wd.lock:
            wd.emit = emit_line
        wd.disarm()

    # ---- parity spot-check of the benchmarked configuration (not timed) ----------------
    if rank == 0 and world == 1 and not args.no_side:
        try:
            import oracle
            n_s = min(1_000_000, hi - lo)
            sample = corpus.read(0, n_s)
            cs = capi.Corpus(ctx, n_s)
            cs.append(sample)
            cs.prepare()
            got = cs.search(queries_h[0], top_k=k)
            r, d = oracle.search_rows(sample, queries_h[0], top_k=k)
            state["check"] = bool(got["row"].tolist() == [int(x) for x in r] and np.array_equal(got["distance"], d)
                                  and cs.tier_stats()["q8"]["proven"] >= 1)
            cs.close()
        except Exception as e:                                         # noqa: BLE001 - reported, never fatal to the line
            state["check"] = f"error: {type(e).__name__}: {e}"

    # ---- side sections ------------------------------------------------------------------
    def side(name, fn, *a, collective=False, budget_s=240.0, **kw):
        """Side sections never take the headline line down with them.  Single-rank sections: errors are
        caught and reported.  Collective sections (N > 1): a deadline is armed (aligned by a barrier); a
        rank that raises cannot rejoin its peers, so rank 0 prints the line at once and the others leave at
        the deadline."""
        t0 = time.perf_counter()
        if collective and wd is not None:
            wd.arm(name + " (entry barrier)", 120.0)
            barrier()
            wd.arm(name, budget_s)
        try:
            res = fn(*a, **kw)
        except Exception as e:                                         # noqa: BLE001 - reported in the JSON
            res = {"error": f"{type(e).__name__}: {e}"}
            if collective and wd is not None:
                sides[name] = res
                if rank == 0:
                    wd.fire(f"section '{name}' failed on rank 0: {res['error']}")
                wd.park(f"section '{name}' failed: {res['error']}")
        if wd is not None:
            wd.disarm()
        res["section_s"] = round(time.perf_counter() - t0, 2)
        sides[name] = res
        if rank == 0:
            print(json.dumps({"side": name, **res}), flush=True)

    if not args.no_side:
        if world == 1:
            side("k1_tiers", side_k1_tiers, E, corpus, q_dev, queries_h, k, args.rows)
            side("config2_1M", side_config2, E, k, n=args.config2_rows)
            side("batch1024", side_batch, E, corpus, args.rows, k, nq=args.batch_queries)
            side("k3_embed", side_embed, E, V=args.embed_vocab, n_lines=args.embed_lines)
            side("ivfpq", side_ivfpq, E, args)
            try:
                state["cpu_base"] = cpu_baseline_section(corpus, queries_h, args.rows, k)
            except Exception as e:                                     # noqa: BLE001
                state["cpu_base"] = {"error": f"{type(e).__name__}: {e}"}
        else:
            # order: the section that shares the headline's code path first; the sharded K2 exchange last (its
            # N=8 run stalled once on the builder's box -- BASELINE.md section 6 -- and a stall must not cost the others)
            if args.config4_rows:
                side("config4_100M", side_config4, E, args, k, make_xchg if xchg is not None else None, collective=True, budget_s=240.0)
            if args.ivfpq_rows_per_gpu:
                side("ivfpq_sharded", side_ivfpq, E, args, make_xchg=make_xchg if exchange == "p2p" else None, collective=True, budget_s=360.0)
            side("batch1024", side_batch, E, corpus, args.rows, k, nq=args.batch_queries, make_xchg=make_xchg if xchg is not None else None,
                 collective=True, budget_s=120.0)
    try:                                                               # nothing after the measurements may cost the line
        state["tier_stats"] = corpus.tier_stats()
        corpus.close()
        torch.cuda.empty_cache()
    except Exception as e:                                             # noqa: BLE001
        print(f"[rank {rank}] closing the corpus: {type(e).__name__}: {e}", file=sys.stderr)
    if not args.no_side and world == 1 and args.config4_rows:
        side("config4_100M", side_config4, E, args, k, make_xchg)

    if wd is not None:
        wd.arm("teardown", 120.0)
        with wd.lock:
            wd.emit = lambda reason: None                               # the line is about to be printed here
    if rank == 0:
        emit_line()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
