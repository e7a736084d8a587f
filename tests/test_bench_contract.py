"""bench.py contract checks that do not need a GPU: the reference arm runs on CPU and
prints the agreed JSON line; the argument surface and synthetic generators are stable."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--rows", "100000"],
                       capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("queries/sec over 10M-line corpus")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and d["config"]["rows"] == 100000
    assert d["steps"] == 1 and d["cpu_baseline"]["sample"].startswith("all 100000 rows")     # same workload, same step count
    assert len(r.stdout.strip().splitlines()[-1]) < 1500


def test_reference_arm_can_bound_its_sample(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "0", "--rows", "100000", "--ref-rows", "20000", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2 and "scaled x5" in d["cpu_baseline"]["sample"]
    # --dump-outputs: the hits of the last timed step (query 1) over the 20000 sampled rows
    sys.path.insert(0, ROOT)
    import bench
    import oracle
    want_rows, want_d = oracle.search_rows(bench.gen_chunk_numpy(0, 100000)[:20000], bench.gen_queries(64)[1], top_k=10)
    got_d, got_rows = np.load(tmp_path / "hits_distance.npy"), np.load(tmp_path / "hits_row.npy")
    assert got_d.dtype == got_rows.dtype == np.float64
    assert np.array_equal(got_rows, want_rows.astype(np.float64)) and np.allclose(got_d, want_d, rtol=0, atol=1e-6)


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, cwd=ROOT, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_reference_arm_non_zero_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, cwd=ROOT, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_synthetic_generators_are_deterministic():
    sys.path.insert(0, ROOT)
    import bench
    a, b = bench.gen_chunk_numpy(3, 5000), bench.gen_chunk_numpy(3, 5000)
    assert np.array_equal(a, b) and a.shape == (5000, 256) and a.dtype == np.float32
    norms = np.linalg.norm(a, axis=1)
    assert (norms == 0).sum() >= 1 and np.allclose(norms[norms > 0], 1.0, atol=1e-5)     # zero rows injected
    q = bench.gen_queries(8)
    assert np.array_equal(q, bench.gen_queries(8)) and np.allclose(np.linalg.norm(q, axis=1), 1.0, atol=1e-5)


_snippet_no = [0]


def _run_snippet(code):
    _snippet_no[0] += 1                                   # the watchdog's leave-flag file is named after parent pid + port
    env = dict(os.environ, MASTER_PORT=str(40000 + _snippet_no[0]))
    return subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=60, env=env)


def test_watchdog_prints_the_line_and_leaves_cleanly_when_a_phase_stalls():
    """bench.py's multi-rank deadline thread: a stalled phase costs the unfinished side sections, never
    the headline (rank 0 prints it, exit code 0); before a headline exists it is an error exit."""
    code = ("import sys, time, json; sys.path.insert(0, '.'); import bench\n"
            "wd = bench.Watchdog(0, lambda why: print(json.dumps({'value': 1.0, 'side_sections_truncated': why})))\n"
            "wd.arm('stuck section', 0.5); time.sleep(30)\n")
    r = _run_snippet(code)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["value"] == 1.0 and "stuck section" in d["side_sections_truncated"]
    # a non-zero rank leaves quietly (stdout stays rank 0's)
    r = _run_snippet(code.replace("bench.Watchdog(0,", "bench.Watchdog(3,"))
    assert r.returncode == 0 and r.stdout.strip() == "" and "rank 3" in r.stderr
    # nothing measured yet: error exit with an error object
    r = _run_snippet("import sys, time; sys.path.insert(0, '.'); import bench\n"
                     "wd = bench.Watchdog(0, None); wd.arm('fill', 0.3); time.sleep(30)\n")
    assert r.returncode == 1 and "error" in json.loads(r.stdout.strip().splitlines()[-1])
    # disarmed in time: nothing happens
    r = _run_snippet("import sys, time; sys.path.insert(0, '.'); import bench\n"
                     "wd = bench.Watchdog(0, None); wd.arm('quick', 0.5); wd.disarm(); time.sleep(1.2); print('alive')\n")
    assert r.returncode == 0 and r.stdout.strip() == "alive"
