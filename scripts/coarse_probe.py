"""K1 with and without the 4-bit coarse stage in front of the q8 tier, in one process.

At each corpus size (bench.py's row distribution: unit rows, 0.1 % duplicates, 0.01 % zero rows) the two
settings of STB_Q8_COARSE alternate over --rounds rounds of --queries pipelined stb_search_topk_dev calls,
timed with CUDA events.  Reports us/query (median and min..max over rounds), how many results proved
themselves, the bytes per row each setting streams (plus the coarse stage's q8 re-score gathers, an upper
bound from the CTA candidate count), and the card and its power limit.  Results must be identical.

    python scripts/coarse_probe.py [--rows 10000000,1000000] [--rounds 5] [--queries 200] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                  # noqa: BLE001 - report, do not guess
        return {"gpu": None, "error": repr(e)}


def fill(torch, dev, capi, ctx, n, seed):
    corpus = capi.Corpus(ctx, n)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    chunk = 1 << 22
    for lo in range(0, n, chunk):
        m = min(chunk, n - lo)
        x = torch.randn((m, 256), generator=g, device=dev, dtype=torch.float32)
        x /= x.norm(dim=1, keepdim=True)
        idx = torch.randint(0, m, (2 * max(m // 1000, 1) + max(m // 10000, 1),), generator=g, device=dev)
        nd = max(m // 1000, 1)
        x[idx[:nd]] = x[idx[nd:2 * nd]]
        x[idx[2 * nd:]] = 0.0
        torch.cuda.synchronize(dev)
        corpus.append_dev(x.data_ptr(), m)
        del x
    corpus.prepare(1)
    torch.cuda.synchronize(dev)
    return corpus


def run(torch, dev, corpus, q_dev, k, n_q):
    hits = torch.zeros((n_q, k, 2), dtype=torch.float64, device=dev)
    st = torch.zeros((n_q, 4), dtype=torch.int32, device=dev)
    for i in range(8):                                       # warm-up of this setting
        corpus.search_topk_dev(q_dev[i].data_ptr(), k, hits[i].data_ptr(), st[i].data_ptr())
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(torch.cuda.current_stream(dev))
    for i in range(n_q):
        corpus.search_topk_dev(q_dev[i].data_ptr(), k, hits[i].data_ptr(), st[i].data_ptr())
    e1.record(torch.cuda.current_stream(dev))
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) * 1e3 / n_q, st.cpu().numpy(), hits.cpu().numpy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="10000000,1000000")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--queries", type=int, default=200)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from semtools_b200 import capi
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(dev)                          # shared by the library and the timing events
    torch.cuda.set_stream(stream)
    ctx = capi.Context(0, stream.cuda_stream)
    result = {"card": card(), "k": args.k, "queries_per_round": args.queries, "rounds": args.rounds, "sizes": []}
    rng = np.random.default_rng(7)
    q = rng.standard_normal((args.queries, 256)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q_dev = torch.from_numpy(q).to(dev)
    for n in [int(x) for x in args.rows.split(",")]:
        corpus = fill(torch, dev, capi, ctx, n, seed=1234 + n)
        times = {"0": [], "1": []}
        proven = {"0": 0, "1": 0}
        outs = {}
        for _ in range(args.rounds):
            for setting in ("0", "1"):
                os.environ["STB_Q8_COARSE"] = setting
                us, st, hits = run(torch, dev, corpus, q_dev, args.k, args.queries)
                times[setting].append(us)
                proven[setting] += int((st[:, 1] == 1).sum())
                outs.setdefault(setting, hits)
                assert ((st[:, 3] >> 16) == 2).all(), st[:4]
        os.environ.pop("STB_Q8_COARSE", None)
        grid = 2 * torch.cuda.get_device_properties(dev).multi_processor_count
        entry = {
            "rows": n,
            "identical_hits": bool(np.array_equal(outs["0"], outs["1"])),
            "bytes_per_row": {"q8": 260, "coarse": 136},
            # each CTA re-scores at most 8 warps x 64 candidates with q8 codes (256 B + 4 B scale)
            "coarse_regather_bytes_per_query_max": grid * 512 * 260,
        }
        for setting, name in (("0", "q8"), ("1", "coarse+q8")):
            t = np.array(times[setting])
            bpr = 260 if setting == "0" else 136
            entry[name] = {"us_per_query_median": round(float(np.median(t)), 2),
                           "us_per_query_min_max": [round(float(t.min()), 2), round(float(t.max()), 2)],
                           "proven": f"{proven[setting]}/{args.rounds * args.queries}",
                           "scan_GBps_at_median": round(n * bpr / (np.median(t) * 1e-6) / 1e9, 1)}
        entry["speedup_median"] = round(entry["q8"]["us_per_query_median"] / entry["coarse+q8"]["us_per_query_median"], 3)
        result["sizes"].append(entry)
        print(json.dumps(entry), flush=True)
        corpus.close()
        torch.cuda.empty_cache()
    ctx.close()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
