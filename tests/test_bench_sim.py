"""bench.py's control flow, end to end, without a GPU (tests/bench_sim.py: torch.cuda stubbed, the C-ABI
binding replaced by an oracle-backed stand-in, NCCL replaced by gloo).  Pins what the driver depends on:
the run finishes, the LAST stdout line is the headline with every contract key, it stays below 1.5 kB,
side sections come first, and at N > 1 a stalled or failed side section costs that section only."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIM = os.path.join(ROOT, "tests", "bench_sim.py")
SMALL = ["--rows", "30000", "--steps", "5", "--warmup", "3", "--config4-rows", "40000", "--batch-queries", "32", "--clock-load-queries", "4"]
CONTRACT_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                 "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"}


def _lines(stdout):
    return [json.loads(x) for x in stdout.strip().splitlines() if x.startswith("{")]


def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _torchrun(n, port, extra, env=None):
    port = _free_port()                                  # the fixed numbers below only label the cases
    e = dict(os.environ, STB_BENCH_ONE_GPU="1", **(env or {}))
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
                           "--master-port", str(port), SIM, "--gpus", str(n)] + SMALL + extra,
                          capture_output=True, text=True, cwd=ROOT, env=e, timeout=600)


def test_single_gpu_flow_prints_sides_then_a_complete_headline(tmp_path):
    side_json, dump = tmp_path / "bench_side.json", tmp_path / "dump"
    r = subprocess.run([sys.executable, SIM, "--gpus", "1"] + SMALL + ["--ivfpq-rows", "20000", "--config2-rows", "20000", "--embed-lines", "3000",
                                                                        "--embed-vocab", "2000", "--side-json", str(side_json),
                                                                        "--dump-outputs", str(dump)],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    out = _lines(r.stdout)
    assert [d["side"] for d in out[:-1]] == ["k1_tiers", "config2_1M", "batch1024", "k3_embed", "ivfpq", "config4_100M"]
    assert all("error" not in d for d in out[:-1]), out
    head = out[-1]
    assert CONTRACT_KEYS | {"cpu_baseline"} <= set(head), sorted(CONTRACT_KEYS - set(head))
    assert len(r.stdout.strip().splitlines()[-1]) < 1500
    assert head["n_gpus"] == 1 and head["gpu_launches"] == 5 and head["parity_spot_check"] is True
    assert head["e2e"]["many16_value"] and {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(head["e2e"])
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(head["roofline"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(head["cpu_baseline"])
    assert {"batch1024_qps", "config2_1M_us", "config4_100M_qps", "ivfpq_recall", "k3_Mlines_s"} <= set(head["side"])
    full = json.load(open(side_json))                                          # the untrimmed line + every section
    assert full["headline"]["tier_stats"]["q8"][0] > 0 and set(full["sides"]) >= {"k1_tiers", "config4_100M"}
    # --dump-outputs: the hits of the last timed step (warm-up 3 + 5 steps -> query 7) over the generated corpus
    sys.path.insert(0, ROOT)
    import bench
    import oracle
    import torch
    rows = bench.gen_chunk_torch(torch, torch.device("cpu"), 0, 30000).numpy()
    want_rows, want_d = oracle.search_rows(rows, bench.gen_queries(64)[7], top_k=10)
    got_d, got_rows = np.load(dump / "hits_distance.npy"), np.load(dump / "hits_row.npy")
    assert got_d.dtype == got_rows.dtype == np.float64
    assert np.array_equal(got_rows, want_rows.astype(np.float64)) and np.array_equal(got_d, want_d)


def test_two_rank_flow_runs_the_sharded_sections_in_order():
    r = _torchrun(2, 29541, ["--ivfpq-rows-per-gpu", "8000"])
    assert r.returncode == 0, r.stderr[-2000:]
    out = _lines(r.stdout)
    assert [d["side"] for d in out[:-1]] == ["config4_100M", "ivfpq_sharded", "batch1024"]
    assert all("error" not in d for d in out[:-1]), out
    assert out[1]["recall_at_10"] == 1.0 and out[1]["exchange"].startswith("stb_ivfpq_search_dev")
    assert out[2]["ranks_agree"] is True and out[2]["agrees_with_single_query_path"] is True
    head = out[-1]
    assert CONTRACT_KEYS <= set(head) and head["n_gpus"] == 2 and head["ranks_agree"] is True
    assert head["config"]["exchange"] == "p2p" and len(head["per_rank_ms_per_step"]) == 2
    assert "side_sections_truncated" not in head and len(r.stdout.strip().splitlines()[-1]) < 1500


@pytest.mark.parametrize("fault,port", [({"FAKE_CAPI_STALL": "1:search_batch_dev"}, 29542), ({"FAKE_CAPI_RAISE": "0:search_batch_dev"}, 29543),
                                        ({"FAKE_CAPI_RAISE": "1:search_batch_dev"}, 29544)])
def test_a_stalled_or_failed_sharded_section_costs_that_section_only(fault, port):
    """The sharded K2 section hangs on one rank / raises on rank 0 / raises on another rank: the job still
    ends with exit code 0 and the headline (marked truncated) as the last stdout line, with the sections
    that had finished."""
    r = _torchrun(2, port, ["--ivfpq-rows-per-gpu", "0"], env=dict(fault, STB_BENCH_DEADLINE_SCALE="0.2"))
    assert r.returncode == 0, r.stderr[-2000:]
    out = _lines(r.stdout)
    head = out[-1]
    assert CONTRACT_KEYS <= set(head) and head["value"] > 0
    assert "batch1024" in head["side_sections_truncated"]
    assert [d["side"] for d in out[:-1]] == ["config4_100M"] and "config4_100M_qps" in head["side"]


def test_shrink_line_keeps_the_contract_keys_and_the_limit():
    sys.path.insert(0, ROOT)
    import bench
    full = {k: 1 for k in CONTRACT_KEYS}
    full.update({"config": {"workload": "w" * 150, "rows": 10_000_000, "rows_per_gpu": 10_000_000, "top_k": 10, "tier": "q8", "parallelism": "row-shard x1",
                            "exchange": "none", "l2": "scanned copy >> 126 MB L2, no flush"},
                 "roofline": {"bound": "hbm", "kernel": "stb_scan_topk_kernel/q8", "achieved": 28049.0, "peak": 6572.9, "unit": "GB/s", "frac": 4.2674,
                              "traffic": 2604123456, "peak_source": "measured", "algorithmic_bytes": 10240000000, "bytes_read": 2600000000, "frac_bytes_read": 1.08},
                 "cpu_baseline": {"value": 0.47, "unit": "queries/s", "cores": 1, "kind": "port", "isa": "avx512f", "sample": "s" * 60, "host_cores": 128,
                                  "all_cores_value": 0.58, "all_cores_threads": 128, "gpu_rows_equal_cpu_rows": True},
                 "e2e": {"value": 2432.8, "unit": "queries/s", "h2d_bytes_per_step": 1024, "d2h_bytes_per_step": 176, "steps": 100, "ms_per_step": 0.41, "many16_value": 2650.1},
                 "tier_stats": {"f32": [55, 55], "h16": [55, 55], "q8": [1161, 1161]}, "per_rank_ms_per_step": [0.365] * 8, "ranks_agree": None,
                 "side": {"x" * 20 + str(i): 123456.7 for i in range(12)}, "vs_baseline": None})
    line = bench.shrink_line(full)
    assert len(json.dumps(line)) <= bench.LINE_LIMIT < 1500
    assert CONTRACT_KEYS | {"cpu_baseline"} <= set(line) and "ranks_agree" not in line and line["vs_baseline"] is None
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(line["roofline"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"])
    assert full["tier_stats"] and "tier_stats" in full                      # the input is not modified


def test_a_timed_out_fused_exchange_makes_every_rank_switch_to_nccl():
    """One rank reports a peer time-out in the probe batch of the sharded K2 section: the exchange object is
    dead, all ranks agree (all-reduce) to measure with the NCCL exchange, and the section says so."""
    r = _torchrun(2, 29545, ["--ivfpq-rows-per-gpu", "0"], env={"FAKE_CAPI_TIMEOUT": "1:search_batch_dev"})
    assert r.returncode == 0, r.stderr[-2000:]
    out = _lines(r.stdout)
    assert [d["side"] for d in out[:-1]] == ["config4_100M", "batch1024"]
    b = out[1]
    assert "error" not in b and b["exchange"].startswith("nccl") and "timed out" in b["note"] and b["ranks_agree"] is True
    assert "side_sections_truncated" not in out[-1] and "batch1024_qps" in out[-1]["side"]


def test_the_stand_in_binding_has_the_real_binding_s_signatures():
    """The simulation is only worth something if bench.py calls the stand-in exactly as it calls
    semtools_b200.capi: every public method / function of tests/fake_capi.py must exist in the real binding
    with the same parameter names in the same order."""
    import inspect
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import fake_capi as fake
    from semtools_b200 import capi as real
    for cname in ("Context", "Corpus", "Exchange", "IvfPq", "Table"):
        fr, ff = getattr(real, cname), getattr(fake, cname)
        for name, fn in inspect.getmembers(ff, predicate=inspect.isfunction):
            if name.startswith("_") and name != "__init__":
                continue
            assert hasattr(fr, name), (cname, name)
            assert list(inspect.signature(getattr(fr, name)).parameters) == list(inspect.signature(fn).parameters), (cname, name)
    for name in ("embed", "embed_dev", "embed_status"):
        assert list(inspect.signature(getattr(real, name)).parameters) == list(inspect.signature(getattr(fake, name)).parameters), name
    assert fake.HIT_DTYPE is real.HIT_DTYPE and fake.StbError is real.StbError
