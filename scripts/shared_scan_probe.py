"""Synchronized K1 scans: what pipelined stb_search_topk_dev calls cost when consecutive queries share one pass.

Back-to-back calls launch overlapped (two grids co-resident, one CTA per SM each) and every launch starts at
the running scan's front, so a line of the coarse copy is fetched from HBM once for two queries.  At each
corpus size (bench.py's row distribution, see coarse_probe.py) --rounds rounds of --queries calls are timed
with CUDA events.  Reports us/query (median and min..max over rounds), the HBM bytes per query that time
would allow at the 7.12 TB/s the q8 scan reached (BASELINE.md section 6) next to the bytes of one pass over
the coarse copy (136 B per row), how many results proved themselves, and the card and its power limit.
Near one pass per query the two grids are not sharing; well below it they are.

    python scripts/shared_scan_probe.py [--rows 1000000,10000000,100000000] [--rounds 5] [--queries 200] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from coarse_probe import card, fill, run  # noqa: E402

SCAN_TBPS = 7.12          # TB/s, the q8 scan's measured rate (BASELINE.md section 6)
COARSE_BYTES_PER_ROW = 136


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="1000000,10000000,100000000")
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
        times, proven, first = [], 0, None
        for _ in range(args.rounds):
            us, st, hits = run(torch, dev, corpus, q_dev, args.k, args.queries)
            times.append(us)
            proven += int((st[:, 1] == 1).sum())
            if first is None:
                first = hits
            assert np.array_equal(hits, first), "pipelined results changed between rounds"
        t = np.array(times)
        med = float(np.median(t))
        pass_bytes = n * COARSE_BYTES_PER_ROW
        implied = med * 1e-6 * SCAN_TBPS * 1e12
        entry = {"rows": n,
                 "us_per_query_median": round(med, 2),
                 "us_per_query_min_max": [round(float(t.min()), 2), round(float(t.max()), 2)],
                 "coarse_pass_GB": round(pass_bytes / 1e9, 3),
                 "hbm_GB_per_query_at_7.12TBps": round(implied / 1e9, 3),
                 "passes_per_query_at_7.12TBps": round(implied / pass_bytes, 3),
                 "proven": f"{proven}/{args.rounds * args.queries}",
                 "scan_front_after": ctx.scan_front()}
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
