"""Model of K1's dynamic tile schedule with synchronized starts (csrc/scan_topk.cu: stb_for_each_tile and the
ticket booking in stb_launch_topk_t).  A launch scans tiles s, s+1, ..., n_tiles-1, 0, ..., s-1: ticket t
covers tiles (s + first_tile(t) + i) mod n_tiles.  Whatever s the scan front gives, every tile must be
scanned exactly once, the counter must advance by n_tickets + total_warps, and the row-ranges map (which
only walks forward) must be restarted wherever the virtual rows step back.  No GPU needed."""
import random

import pytest

TICKET_TILES = 4       # STB_TICKET_TILES
SCAN_WARPS = 8         # warps per CTA


def booking(n_tiles, warps_total):
    """Host side: bulk tickets of TICKET_TILES tiles, the last ~2 tiles per warp one by one."""
    single = min(n_tiles, 2 * warps_total)
    t_bulk = (n_tiles - single) // TICKET_TILES
    n_tickets = t_bulk + (n_tiles - t_bulk * TICKET_TILES)
    return t_bulk, n_tickets


def first_tile(t, t_bulk):
    return t * TICKET_TILES if t < t_bulk else t_bulk * TICKET_TILES + (t - t_bulk)


def start_tile(front, n_virtual, tile_rows):
    """What the warp that draws ticket 0 publishes: the front as a virtual row, reduced, rounded down."""
    return (front % n_virtual) // tile_rows


def ticket_tiles(t, s, n_tiles, t_bulk):
    """The device loop: (tile, restart) pairs of ticket t, with the incremental wrap of the kernel."""
    t0 = first_tile(t, t_bulk)
    t1 = t0 + TICKET_TILES if t < t_bulk else t0 + 1
    tile = s + t0
    if tile >= n_tiles:
        tile -= n_tiles
    out = []
    for i in range(t0, t1):
        out.append((tile, i == t0 or tile == 0))
        tile += 1
        if tile == n_tiles:
            tile = 0
    return out


def run_launch(n_tiles, warps_total, s, seed):
    """Warps draw from one counter in a random interleaving; each warp draws its next ticket before it
    processes the current one and stops at its first failing draw."""
    t_bulk, n_tickets = booking(n_tiles, warps_total)
    counter = 0
    rng = random.Random(seed)
    seen = []
    state = {}                      # warp -> current ticket (absent: not drawn yet)
    active = list(range(warps_total))
    while active:
        w = rng.choice(active)
        if w not in state:
            state[w] = counter
            counter += 1
            if first_tile(state[w], t_bulk) >= n_tiles:
                active.remove(w)
            continue
        cur = state[w]
        nxt = counter
        counter += 1
        seen.append(ticket_tiles(cur, s, n_tiles, t_bulk))
        state[w] = nxt
        if first_tile(nxt, t_bulk) >= n_tiles:
            active.remove(w)
    return seen, counter, n_tickets


CASES = []
for n_tiles in (1, 2, 3, 5, 17, 64, 1000, 3125, 20_011):
    for ctas in (1, 3, 148):
        warps = ctas * SCAN_WARPS
        t_bulk, _ = booking(n_tiles, warps)
        starts = {0, n_tiles - 1, n_tiles // 2}
        if t_bulk > 0:
            starts |= {1, 2, TICKET_TILES * t_bulk - 1, TICKET_TILES * t_bulk, min(TICKET_TILES * t_bulk + 1, n_tiles - 1)}
        CASES += [(n_tiles, warps, s) for s in sorted(x for x in starts if 0 <= x < n_tiles)]


@pytest.mark.parametrize("n_tiles,warps,s", CASES)
def test_every_tile_exactly_once_from_any_start(n_tiles, warps, s):
    seen, counter, n_tickets = run_launch(n_tiles, warps, s, seed=n_tiles * 7919 + s)
    tiles = [t for ticket in seen for t, _ in ticket]
    assert sorted(tiles) == list(range(n_tiles))
    assert len(seen) == n_tickets
    assert counter == n_tickets + warps                        # what the host books for the next launch
    for ticket in seen:
        assert ticket[0][1]                                     # restart at every ticket's first tile
        for (a, _), (b, restart) in zip(ticket, ticket[1:]):
            assert b == a + 1 or (a == n_tiles - 1 and b == 0 and restart)   # forward, or the wrap with a restart


def test_tickets_keep_the_rotated_row_order():
    """Tickets are issued in row order from s on: the grid streams one contiguous window that wraps."""
    n_tiles, warps, s = 20_011, 148 * SCAN_WARPS, 12_345
    t_bulk, n_tickets = booking(n_tiles, warps)
    flat = [t for k in range(n_tickets) for t, _ in ticket_tiles(k, s, n_tiles, t_bulk)]
    assert flat == [(s + i) % n_tiles for i in range(n_tiles)]


@pytest.mark.parametrize("tile_rows", [8, 16, 32, 64])
def test_the_start_tile_is_inside_the_scan_for_any_front(tile_rows):
    """The front may come from another corpus, another tier (tile height) or row-ranges mode: any u64."""
    rng = random.Random(tile_rows)
    for n_virtual in (1, 33, 2_000, 150_000, 1_000_003, 10_000_000):
        n_tiles = (n_virtual + tile_rows - 1) // tile_rows
        fronts = [0, n_virtual - 1, n_virtual, 2**64 - 1, (n_tiles - 1) * tile_rows] + [rng.randrange(2**64) for _ in range(50)]
        for f in fronts:
            s = start_tile(f, n_virtual, tile_rows)
            assert 0 <= s < n_tiles and s < 2**32                # packed into the low half of the start word


def test_the_ragged_last_tile_can_sit_mid_sequence():
    n_virtual, tile_rows = 1_000_003, 64
    n_tiles = (n_virtual + tile_rows - 1) // tile_rows
    s = start_tile(n_virtual - 1, n_virtual, tile_rows)
    assert s == n_tiles - 1                                     # a front on the last (ragged) tile starts there
    t_bulk, n_tickets = booking(n_tiles, 148 * SCAN_WARPS)
    first = ticket_tiles(0, s, n_tiles, t_bulk)
    assert first[0] == (n_tiles - 1, True) and first[1] == (0, True)

