"""CPU model of the coarse stage in front of the q8 tier (csrc/scan_topk.cu: stb_q4_build_kernel,
stb_scan_q4).  The 4-bit score u4 only ranks rows inside a warp, but a row it drops is covered by the
warp's list minimum, so u4 must be an UPPER BOUND of the exact cosine, u4 >= c - 1e-5, like the q8 score
(test_q8_bound_model.py).  The kernels' arithmetic is restated in numpy float32 / int / f64 and checked
against the f64 cosine; a second test checks on bench-shaped data that the bound is tight enough for a
warp's 64-entry list to hold every row that can reach the k-th best cosine of a 10M-row corpus."""
import numpy as np
import pytest

F = np.float32
T_STEPS = (F(0.65) + F(0.05) * np.arange(8, dtype=F)).astype(F)


def normalise(rows):
    """stb_q8_build_kernel / stb_q4_build_kernel: x^ = x * rsqrt(sum x^2) in f32 (zero rows stay zero)."""
    rows = rows.astype(F)
    ss = (rows * rows).sum(axis=1, dtype=F)
    with np.errstate(divide="ignore"):
        inv = np.where(ss > 0, F(1) / np.sqrt(ss, dtype=F), F(0)).astype(F)
    return (rows * inv[:, None]).astype(F)


def _codes(xh, inv_s):
    with np.errstate(invalid="ignore"):                      # zero rows (inv_s = inf) are not used
        return np.clip(np.rint((xh * inv_s[:, None] + F(7.5)).astype(F)), 0, 15).astype(np.int64)


def build_q4(rows):
    """16 mid-rise levels x~ = s4 (c - 7.5); s4 = t max|x^| / 7.5 with the t of T_STEPS that minimises
    ||x^ - x~|| (first on ties); r = that norm in f64 for the stored s4, rounded up to f32."""
    xh = normalise(rows)
    am = np.abs(xh).max(axis=1).astype(F)
    best = np.full(len(xh), np.inf, dtype=F)
    s = np.zeros(len(xh), dtype=F)
    for t in T_STEPS:
        sk = (t * am * F(1.0 / 7.5)).astype(F)
        with np.errstate(divide="ignore"):
            inv_s = (F(1) / sk).astype(F)
        c = _codes(xh, inv_s)
        err = ((xh - sk[:, None] * (c.astype(F) - F(7.5))) ** 2).sum(axis=1, dtype=F)
        take = (am > 0) & (err < best)
        best[take] = err[take]
        s[take] = sk[take]
    with np.errstate(divide="ignore"):
        inv_s = np.where(s > 0, F(1) / s, F(0)).astype(F)
    c = np.where(s[:, None] > 0, _codes(xh, inv_s), 8)
    d = xh.astype(np.float64) - s.astype(np.float64)[:, None] * (c - 7.5)
    r64 = np.sqrt((d * d).sum(axis=1)) * (1 + 1e-9)
    r = r64.astype(F)
    r = np.where(r.astype(np.float64) < r64, np.nextafter(r, F(np.inf)), r).astype(F)   # round up
    r[s == 0] = 0
    return c, s, r


def pack_row_words(c):
    """Byte b of word l: low nibble c[8l+b], high nibble c[8l+4+b] -- lane j of a row group reads words 4j..4j+3."""
    c = c.reshape(len(c), 32, 2, 4)                          # [row][word l][lo/hi][byte b]
    return (c[:, :, 0, :] | (c[:, :, 1, :] << 4)).astype(np.uint8)


def quantise_query(q):
    """stb_scan_q4: q8 = rint(q^ S8), S8 = 127 / max|q^|; ||f|| with f = q^ - q8 / S8, inflated."""
    q = q.astype(F)
    rq = F(1) / np.sqrt((q * q).sum(dtype=F), dtype=F)
    amax = F(np.abs(q).max() * rq)
    S = F(127.0) / amax
    inv_S = F(1.0) / S
    qh = (q * rq).astype(F)
    q8 = np.clip(np.rint((q * F(rq * S)).astype(F)), -127, 127).astype(np.int64)
    f = (qh - q8.astype(F) * inv_S).astype(F)
    nf = F(F(np.sqrt((f * f).sum(dtype=F))) * F(1.001) + F(2e-6))
    return q8, inv_S, nf


def q4_scores(c, s, r, q):
    q8, inv_S, nf = quantise_query(q)
    dot = c @ q8                                             # int32 in the kernel: |2 dot| < 2^21
    assert np.abs(2 * dot).max() < 2 ** 24                   # exact as f32 too
    integ = (2 * dot - 15 * int(q8.sum())).astype(F)
    tail = (r * (F(1) + nf) + (nf + F(4e-6))).astype(F)
    return ((s * F(F(0.5) * inv_S)).astype(F) * integ + tail).astype(F)


def exact_cos(rows, q):
    r, qq = rows.astype(np.float64), q.astype(np.float64)
    n = np.sqrt((r * r).sum(axis=1)) * np.sqrt((qq * qq).sum())
    return np.divide(r @ qq, n, out=np.zeros(len(r)), where=n > 0)


def check(rows, q):
    c, s, r = build_q4(rows)
    u = q4_scores(c, s, r, q)
    slack = u.astype(np.float64) - exact_cos(rows, q)
    assert slack.min() >= -1e-5, (slack.min(), int(slack.argmin()))
    return slack


def unit(rng, n):
    x = rng.standard_normal((n, 256)).astype(F)
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(F)


def test_nibble_layout_gives_each_lane_one_contiguous_slice():
    """The packed words, read as nibble planes, hold elements 32j + 8i + {0..3} (low) and + {4..7} (high)
    in word i of lane j's 16-byte chunk, which is the order of the int8 query's bytes."""
    c = np.arange(256, dtype=np.int64)[None, :] % 16
    words = pack_row_words(c)[0]                             # [32 words][4 bytes]
    for j in range(8):
        for i in range(4):
            w = words[4 * j + i]
            assert (w & 15).tolist() == c[0, 32 * j + 8 * i: 32 * j + 8 * i + 4].tolist()
            assert (w >> 4).tolist() == c[0, 32 * j + 8 * i + 4: 32 * j + 8 * i + 8].tolist()


def test_upper_bound_holds_on_random_unit_rows_and_is_useful():
    rng = np.random.default_rng(11)
    rows = unit(rng, 20000)
    _, _, r = build_q4(rows)
    assert 0.09 < r.mean() < 0.115                           # MSE-chosen scale: ~0.103 on random unit rows
    for _ in range(6):
        slack = check(rows, unit(rng, 1)[0])
        assert np.median(slack) < 0.2


def test_upper_bound_holds_on_scaled_rows_and_scaled_queries():
    rng = np.random.default_rng(12)
    rows = (unit(rng, 5000) * rng.uniform(1e-3, 1e3, (5000, 1))).astype(F)
    for scale in (1e-4, 1.0, 37.5, 1e4):
        check(rows, (unit(rng, 1)[0] * F(scale)).astype(F))


def test_upper_bound_holds_on_adversarial_rows_and_queries():
    rng = np.random.default_rng(13)
    n = 4000
    rows = unit(rng, n)
    rows[:500, 0] += F(3.0)                                   # one dominant component: coarse grid for the rest
    # components parked on the nibble boundaries (midway between two levels) of the row's own grid
    base = unit(rng, 500)
    step = np.abs(base).max(axis=1, keepdims=True) * 0.8 / 7.5
    rows[500:1000] = ((np.floor(base / step) + 0.5 + rng.choice([-1e-4, 1e-4], base.shape)) * step).astype(F)
    rows[1000:1100] = 0.0                                     # zero rows: s4 = r = 0, bound = ||f||
    rows[1100:1200] *= F(1e-12)
    sparse = np.zeros((300, 256), dtype=F)                    # one-hot and two-hot rows
    sparse[np.arange(300), rng.integers(0, 256, 300)] = 1.0
    sparse[np.arange(300), rng.integers(0, 256, 300)] += F(0.5)
    rows[1200:1500] = sparse
    rows[1500:1600] = np.sign(unit(rng, 100)).astype(F)       # all components +-1
    queries = [unit(rng, 1)[0] for _ in range(4)]
    spike = unit(rng, 1)[0]; spike[7] = 40.0                  # dominant query component: ||f|| large
    queries.append(spike.astype(F))
    queries.append(np.sign(unit(rng, 1)[0]).astype(F))
    onehot = np.zeros(256, dtype=F); onehot[3] = 1.0
    queries.append(onehot)
    queries.append(rows[0].copy())
    queries.append((-rows[0]).astype(F))
    queries.append(rows[1550].copy())
    for q in queries:
        check(rows, q)


def test_zero_rows_store_nothing():
    rows = np.zeros((3, 256), dtype=F)
    c, s, r = build_q4(rows)
    assert np.all(s == 0) and np.all(r == 0)


@pytest.mark.parametrize("k", [1, 10, 16])
def test_room_in_the_warp_lists_on_bench_shaped_data(k):
    """bench.py: 10M random unit rows.  With 296 CTAs of 8 warps a warp scans ~4224 rows; a row whose u4
    reaches the k-th best exact cosine c_k must fit in the warp's 64-entry list, or the list minimum (which
    bounds every dropped row) exceeds c_k and the proof fails.  c_k of 10M rows from the exact
    distribution of the cosine of random unit vectors: (c + 1) / 2 ~ Beta(127.5, 127.5).  Measured here:
    mean / max per warp ~5 / 14 at k = 10 and ~12 / 21 at k = 16."""
    from scipy.stats import beta
    c_k = 2.0 * beta.isf(k / 10_000_000, 127.5, 127.5) - 1.0
    rng = np.random.default_rng(14)
    per_warp, n_warps = 4224, 48
    rows = unit(rng, per_warp * n_warps)
    c, s, r = build_q4(rows)
    for _ in range(2):
        u = q4_scores(c, s, r, unit(rng, 1)[0])
        counts = (u.astype(np.float64) >= c_k).reshape(n_warps, per_warp).sum(axis=1)
        assert counts.mean() <= 16 and counts.max() < 32, (c_k, counts.mean(), counts.max())   # half the list
