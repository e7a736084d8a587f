"""Synchronized scans (csrc/scan_topk.cu: stb_for_each_tile): every ticketed K1 launch starts at the context's
scan front -- a virtual row some earlier scan reached, possibly on another corpus, another tier (tile height)
or in row-ranges mode -- and wraps around to the tile before it.  A skipped tile does not show in the proof
(status[1] only covers the rows the scan saw), so exact copies of the queries are planted where a wrong start,
a wrong wrap or a lost ragged tile would drop them: next to row 0, next to the last row and on both sides of
the tile the scan starts at.  Every result must equal the oracle's and be proven; the ticket counters must
stay where the host booked them."""
import numpy as np
import pytest

import oracle
from conftest import unit_rows
from semtools_b200 import capi

pytestmark = pytest.mark.gpu

# STB_SCAN_TIER / STB_Q8_COARSE of each candidate copy, and the rows of one K1 tile on it
TIERS = {"f32": ("f32", "0", 8), "h16": ("h16", "0", 16), "q8": ("q8", "0", 32), "q4": ("q8", "1", 64)}


def use_tier(monkeypatch, name):
    tier, coarse, _ = TIERS[name]
    monkeypatch.setenv("STB_SCAN_TIER", tier)
    monkeypatch.setenv("STB_Q8_COARSE", coarse)


def check(hits, rows_exp, d_exp):
    assert hits["row"].tolist() == [int(r) for r in rows_exp]
    assert np.array_equal(hits["distance"], np.asarray(d_exp, dtype=np.float64))


def planted_corpus(ctx, rng, n, queries, places):
    rows = unit_rows(rng, n)
    for q, p in zip(queries, places):
        rows[p % n] = q
    c = capi.Corpus(ctx, n)
    c.append(rows)
    c.prepare()
    return c, rows


def test_interleaved_corpora_and_tiers_give_the_oracle_hits(ctx, monkeypatch):
    """Back-to-back device launches alternate between corpora of different sizes and between tiers, so each
    launch starts at a front left by another corpus or another tile height."""
    torch = pytest.importorskip("torch")
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(4242)
    corpora = []
    for n in (1, 33, 2_000, 150_000, 1_000_003):
        qs = unit_rows(rng, 3)
        mid = (n // 2) // 64 * 64                                  # the third query on both sides of a tile boundary
        c, rows = planted_corpus(ctx, rng, n, [qs[0], qs[1], qs[2], qs[2]], [0, n - 1, mid, mid - 1])
        corpora.append((c, rows, qs, torch.from_numpy(qs).to(dev)))
    names = list(TIERS)
    order = [(ci, qi, names[(ci + qi + rep) % len(names)]) for rep in range(2) for qi in range(3) for ci in range(len(corpora))]
    hits = torch.zeros((len(order), 10, 2), dtype=torch.float64, device=dev)
    status = torch.zeros((len(order), 4), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    for i, (ci, qi, name) in enumerate(order):                     # enqueued back to back, no synchronisation
        use_tier(monkeypatch, name)
        c, _, _, q_dev = corpora[ci]
        c.search_topk_dev(q_dev[qi].data_ptr(), 10, hits[i].data_ptr(), status[i].data_ptr())
    ctx.sync()
    d, h = ctx.ticket_check()
    assert d == h
    raw, st = hits.cpu().numpy(), status.cpu().numpy()
    for i, (ci, qi, name) in enumerate(order):
        _, rows, qs, _ = corpora[ci]
        r, dd = oracle.search_rows(rows, qs[qi], top_k=10)
        assert st[i, 1] == 1 and st[i, 0] == min(10, len(rows)), (name, len(rows), qi, st[i])
        check(np.ascontiguousarray(raw[i]).view(capi.HIT_DTYPE).reshape(-1)[: st[i, 0]], r, dd)


@pytest.mark.parametrize("name", list(TIERS))
def test_a_scan_started_anywhere_covers_every_tile(ctx, monkeypatch, name):
    """The front is steered to tile boundaries, into the ragged last tile and past the end of the corpus."""
    torch = pytest.importorskip("torch")
    dev = torch.device("cuda:0")
    use_tier(monkeypatch, name)
    tile = TIERS[name][2]
    rng = np.random.default_rng(4343)
    n = 150_001                                                    # a ragged last tile on every tier
    b = 1_000 * 64                                                 # a tile boundary on every tier
    qs = unit_rows(rng, 5)
    c, rows = planted_corpus(ctx, rng, n, qs, [0, n - 1, b - 1, b, b + tile])
    q_dev = torch.from_numpy(qs).to(dev)
    hits = torch.zeros((10, 2), dtype=torch.float64, device=dev)
    status = torch.zeros(4, dtype=torch.int32, device=dev)
    expect = [oracle.search_rows(rows, q, top_k=10) for q in qs]
    for front in (0, b, b - 1, b + tile, n - 1, n, n + b, 2**63 + 17):
        for qi in range(len(qs)):
            ctx.scan_front(front)
            c.search_topk_dev(q_dev[qi].data_ptr(), 10, hits.data_ptr(), status.data_ptr())
            ctx.sync()
            st = status.cpu().numpy()
            assert st[1] == 1 and st[0] == 10, (front, qi, st)
            check(np.ascontiguousarray(hits.cpu().numpy()).view(capi.HIT_DTYPE).reshape(-1), *expect[qi])
        f = ctx.scan_front()                                       # the launch moved the front: a tile start inside the corpus
        assert f < n and f % tile == 0, (front, f)
    d, h = ctx.ticket_check()
    assert d == h


def test_row_ranges_restart_the_row_map_at_the_wrap(ctx, monkeypatch):
    """Row-ranges mode walks its virtual -> local row map forward only; the wrap to virtual row 0 restarts it."""
    monkeypatch.delenv("STB_SCAN_TIER", raising=False)
    monkeypatch.delenv("STB_Q8_COARSE", raising=False)
    rng = np.random.default_rng(4444)
    n = 60_000
    qs = unit_rows(rng, 3)
    ranges = [[10, 20], [1_000, 9_000], [20_000, 20_001], [30_000, 59_990]]
    c, rows = planted_corpus(ctx, rng, n, qs, [10, 59_989, 8_999])
    virtual = sum(e - s for s, e in ranges)
    for front in (0, 8, 7_000, 8_010, virtual - 1, virtual + 5):
        for q in qs:
            ctx.scan_front(front)
            r, d32 = oracle.store_search(rows, ranges, q, 10)
            got = c.search(q, top_k=10, mode=capi.STB_MODE_STORE_QUERY, row_ranges=ranges)
            assert got["row"].tolist() == [int(x) for x in r], front
            assert np.array_equal(got["distance"].astype(np.float32), d32)
    d, h = ctx.ticket_check()
    assert d == h
