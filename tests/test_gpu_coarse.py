"""The 4-bit coarse stage in front of the q8 tier (csrc/scan_topk.cu: stb_scan_q4, SRC 3): the warps rank
rows by a 4-bit upper bound, each CTA re-scores its candidates with the int8 copy, and everything above
(tree, exact re-rank, proof) is q8's.  Whether it runs (default) or not (STB_Q8_COARSE=0), the hits are
the oracle's.  A search that the coarse stage proves is one K1 launch; one it cannot prove is retried by
the single-stage q8 scan (a second launch) -- that is how these tests see which path ran."""
import numpy as np
import pytest

import oracle
from conftest import unit_rows
from semtools_b200 import capi

pytestmark = pytest.mark.gpu


def check(hits, rows_exp, d_exp):
    assert hits["row"].tolist() == [int(r) for r in rows_exp]
    assert np.array_equal(hits["distance"], np.asarray(d_exp, dtype=np.float64))


def make_corpus(ctx, rows):
    c = capi.Corpus(ctx, max(len(rows), 1))
    c.append(rows)
    return c


def launches_of(ctx, fn):
    before = ctx.counters()["kernel_launches"]
    out = fn()
    return out, ctx.counters()["kernel_launches"] - before


def bench_like_rows(rng, n):
    rows = unit_rows(rng, n)
    rows[rng.integers(0, n, n // 1000)] = rows[rng.integers(0, n, n // 1000)]
    rows[rng.integers(0, n, max(n // 10000, 1))] = 0.0
    return rows


@pytest.mark.parametrize("coarse", ["1", "0"])
def test_coarse_stage_on_and_off_give_the_oracle_hits(ctx, monkeypatch, coarse):
    monkeypatch.delenv("STB_SCAN_TIER", raising=False)
    monkeypatch.setenv("STB_Q8_COARSE", coarse)
    rng = np.random.default_rng(77)
    n = 300_000
    rows = bench_like_rows(rng, n)
    c = make_corpus(ctx, rows)
    c.prepare(1)
    qs = list(unit_rows(rng, 4)) + [rows[123].copy(), (rows[5] * np.float32(1e-3)).astype(np.float32)]
    for q in qs:
        for k in (1, 10, 16):
            r, d = oracle.search_rows(rows, q, top_k=k)
            hits, launches = launches_of(ctx, lambda: c.search(q, top_k=k))
            check(hits, r, d)
            if k <= 10:
                assert launches == 1                         # proven by the first K1 launch (coarse or q8)
    st = c.tier_stats()
    assert st["q8"]["proven"] >= 2 * len(qs), st


def test_coarse_stage_on_the_device_entry_point(ctx, monkeypatch):
    """stb_search_topk_dev has no ladder: it runs the coarse stage when the copies exist, reports the q8
    tier in the status word, and its proven results equal the single-stage q8 scan's."""
    torch = pytest.importorskip("torch")
    monkeypatch.delenv("STB_SCAN_TIER", raising=False)
    rng = np.random.default_rng(78)
    n = 1_000_003
    rows = bench_like_rows(rng, n)
    c = make_corpus(ctx, rows)
    c.prepare(1)
    qs = unit_rows(rng, 8)
    dev = torch.device("cuda:0")
    q_dev = torch.from_numpy(qs).to(dev)
    out = {}
    for coarse in ("1", "0"):
        monkeypatch.setenv("STB_Q8_COARSE", coarse)
        hits = torch.zeros((8, 10, 2), dtype=torch.float64, device=dev)
        status = torch.zeros((8, 4), dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        for i in range(8):
            c.search_topk_dev(q_dev[i].data_ptr(), 10, hits[i].data_ptr(), status[i].data_ptr())
        ctx.sync()
        st = status.cpu().numpy()
        assert (st[:, 1] == 1).all() and (st[:, 0] == 10).all(), st
        assert ((st[:, 3] >> 16) == 2).all(), st                 # tier field: q8 family
        out[coarse] = hits.cpu().numpy()
    assert np.array_equal(out["1"], out["0"])
    for i in range(2):
        r, d = oracle.search_rows(rows, qs[i], top_k=10)
        check(np.ascontiguousarray(out["1"][i]).view(capi.HIT_DTYPE).reshape(-1), r, d)


def test_appends_extend_both_copies(ctx, monkeypatch):
    """Rows appended after prepare() are converted for the int8 and the 4-bit copy alike: a new best row
    must be found (a stale coarse copy would drop it behind a bound that no longer covers it)."""
    monkeypatch.delenv("STB_SCAN_TIER", raising=False)
    monkeypatch.delenv("STB_Q8_COARSE", raising=False)
    rng = np.random.default_rng(79)
    rows = unit_rows(rng, 60_000)
    q = unit_rows(rng, 1)[0]
    c = make_corpus(ctx, rows)
    c.prepare(1)
    extra = unit_rows(rng, 3_000)
    extra[1234] = q                                           # the new best row lives in the appended part
    c.append(extra)
    all_rows = np.concatenate([rows, extra])
    r, d = oracle.search_rows(all_rows, q, top_k=10)
    for _ in range(2):                                         # the first search converts the new rows
        hits, launches = launches_of(ctx, lambda: c.search(q, top_k=10))
        check(hits, r, d)
    assert launches == 1 and hits["row"][0] == 60_000 + 1234
    assert c.tier_stats()["q8"]["built_rows"] == 63_000
    c.append(extra[:5])                                        # and through prepare(): same answer as the oracle
    c.prepare(1)
    all_rows = np.concatenate([all_rows, extra[:5]])
    r, d = oracle.search_rows(all_rows, q, top_k=16)
    check(c.search(q, top_k=16), r, d)


def decoy_corpus(rng, n, n_decoys, top_cos=0.9, decoy_cos=0.85):
    """Random rows, 10 rows at cosine `top_cos` to q scattered through the corpus and `n_decoys` rows at
    `decoy_cos` packed into the first tiles (more than a warp list holds): their 4-bit bounds (~0.1 wide)
    reach above the true 10th best, their int8 bounds (~0.01 wide) do not."""
    q = unit_rows(rng, 1)[0].astype(np.float64)
    rows = unit_rows(rng, n)

    def at_cos(m, cos):
        o = rng.standard_normal((m, 256))
        o -= (o @ q)[:, None] * q[None, :]
        o /= np.linalg.norm(o, axis=1, keepdims=True)
        return (cos * q[None, :] + np.sqrt(1 - cos * cos) * o).astype(np.float32)

    rows[:n_decoys] = at_cos(n_decoys, decoy_cos)
    rows[rng.choice(np.arange(n_decoys, n), 10, replace=False)] = at_cos(10, top_cos)
    return rows, q.astype(np.float32)


def test_a_corpus_that_defeats_the_coarse_proof_falls_to_q8_and_drops_the_stage(ctx, monkeypatch):
    monkeypatch.delenv("STB_SCAN_TIER", raising=False)
    monkeypatch.delenv("STB_Q8_COARSE", raising=False)
    rng = np.random.default_rng(80)
    rows, q = decoy_corpus(rng, 200_000, 256)
    c = make_corpus(ctx, rows)
    c.prepare(1)
    r, d = oracle.search_rows(rows, q, top_k=10)
    seen = []
    for _ in range(10):
        hits, launches = launches_of(ctx, lambda: c.search(q, top_k=10))
        check(hits, r, d)
        seen.append(launches)
    # coarse unproven -> single-stage q8 proves it; after 8 failing tries the stage is dropped for this corpus
    assert seen == [2] * 8 + [1] * 2, seen
    st = c.tier_stats()["q8"]
    assert st["tries"] == st["proven"] == 10, st
    monkeypatch.setenv("STB_Q8_COARSE", "0")
    hits, launches = launches_of(ctx, lambda: c.search(q, top_k=10))
    check(hits, r, d)
    assert launches == 1


def test_heavy_duplication_of_the_best_rows_still_ends_on_the_oracle(ctx, monkeypatch):
    """64 copies of each of the best rows: no warp list can prove anything, neither coarse nor q8;
    the ladder ends on the wider tiers / the collect path with the oracle's hits and tie order."""
    monkeypatch.delenv("STB_SCAN_TIER", raising=False)
    monkeypatch.delenv("STB_Q8_COARSE", raising=False)
    rng = np.random.default_rng(81)
    n = 120_000
    rows = unit_rows(rng, n)
    q = unit_rows(rng, 1)[0]
    best = np.argsort(-(rows @ q))[:3]
    for i, b in enumerate(best):
        rows[1000 + 64 * i: 1064 + 64 * i] = rows[b]
    c = make_corpus(ctx, rows)
    c.prepare(1)
    for k in (1, 10, 16):
        r, d = oracle.search_rows(rows, q, top_k=k)
        check(c.search(q, top_k=k), r, d)
