"""Model checks (CPU, no GPU) of the peer-to-peer halo protocols on column slabs (SURVEY.md 8(e)).

Second half of this file: the flag-in-data ("LL") protocol the one-pass ring kernel runs since round 2
(prost_b200/csrc/pb_tile.cu SLAB, pb_stencil.cuh RingHalo, pb_pdhg.cu slab_ring_halo).  First half: the
sequence-word protocol with edge-tile counters (round 1's ring kernel; the two-pass slab kernels still publish a
whole column with one sequence word after all their edge CTAs are done, pb_stencil.cuh SlabHalo):

Per rank and iteration `it` (sequence numbers xs = ys = it, ys_in = it - 1) two groups of tiles run:
  left-edge tiles  : wait y_flag >= ys_in; read y slot ys_in (and, on residual-refresh iterations, slot
                     ys_in - 1); store the new x column 0 into the LEFT neighbour's x slot xs;
                     after ALL left-edge tiles: publish xs in the left neighbour's x flag;
  right-edge tiles : wait x_flag >= xs (the right neighbour's left-edge tiles of the SAME iteration); read x
                     slots xs and xs - 1; store the new y.gx column into the RIGHT neighbour's y slot ys;
                     after ALL right-edge tiles: publish ys in the right neighbour's y flag.
There are only two slots per direction (index = sequence number & 1); a slot is a whole column, tile j writes
segment j of it and reads segments j and j+1 (its halo rows belong to the next tile).  The model runs the ranks' tiles under a
random scheduler and checks that every read returns the column of exactly the expected (rank, iteration) -- i.e.
that no slot is overwritten before its last reader is done and no reader runs ahead of its writer -- and that the
schedule never deadlocks.  Locally, one launch runs per iteration: a rank's iteration it+1 starts after all its
tiles of iteration it."""
import random

import pytest


class Rank:
    def __init__(self, r, world, n_tiles):
        self.r, self.world = r, world
        self.has_left, self.has_right = r > 0, r + 1 < world
        # [slot][segment] -> (rank, iteration) tag of the writer; x slots are written by the right neighbour,
        # y slots by the left neighbour
        self.x_slot = [[None] * n_tiles for _ in range(2)]
        self.y_slot = [[None] * n_tiles for _ in range(2)]
        self.x_flag = self.y_flag = 0
        self.done = {"L": [0] * n_tiles, "R": [0] * n_tiles}     # iterations completed per tile
        self.edge_count = {}


def run_model(world, n_iters, n_tiles, check_every, seed):
    rng = random.Random(seed)
    ranks = [Rank(r, world, n_tiles) for r in range(world)]
    # pending work: (rank, group, tile) -> next iteration (1-based)
    steps = 0
    total = world * 2 * n_tiles * n_iters
    completed = 0
    while completed < total:
        enabled = []
        for rk in ranks:
            for grp in ("L", "R"):
                for j in range(n_tiles):
                    it = rk.done[grp][j] + 1
                    if it > n_iters:
                        continue
                    # local ordering
                    if any(rk.done[g][t] < it - 1 for g in ("L", "R") for t in range(n_tiles)):
                        continue
                    # halo waits (iteration 1 = the two-pass iteration 0 of the solver: K^T y := 0, no y halo)
                    if grp == "L" and rk.has_left and it > 1 and rk.y_flag < it - 1:
                        continue
                    if grp == "R" and rk.has_right and rk.x_flag < it:
                        continue
                    enabled.append((rk, grp, j, it))
        assert enabled, f"deadlock after {completed} of {total} tile steps (world={world}, seed={seed})"
        rk, grp, j, it = rng.choice(enabled)
        refresh = check_every and it % check_every == 0
        segs = [t for t in (j, j + 1) if t < n_tiles]
        if grp == "L" and rk.has_left:
            if it > 1:
                for t in segs:
                    assert rk.y_slot[(it - 1) & 1][t] == (rk.r - 1, it - 1), ("y halo", rk.r, it, t, rk.y_slot)
                    if refresh and it > 2:
                        assert rk.y_slot[(it - 2) & 1][t] == (rk.r - 1, it - 2), ("previous y halo", rk.r, it, t)
            ranks[rk.r - 1].x_slot[it & 1][j] = (rk.r, it)
        if grp == "R" and rk.has_right:
            for t in segs:
                assert rk.x_slot[it & 1][t] == (rk.r + 1, it), ("x halo", rk.r, it, t, rk.x_slot)
                if it > 1:
                    assert rk.x_slot[(it - 1) & 1][t] == (rk.r + 1, it - 1), ("previous x halo", rk.r, it, t)
            ranks[rk.r + 1].y_slot[it & 1][j] = (rk.r, it)
        rk.done[grp][j] = it
        completed += 1
        # the last tile of a group publishes the sequence number in the neighbour's flag
        key = (grp, it)
        rk.edge_count[key] = rk.edge_count.get(key, 0) + 1
        if rk.edge_count[key] == n_tiles:
            if grp == "L" and rk.has_left:
                assert ranks[rk.r - 1].x_flag == it - 1
                ranks[rk.r - 1].x_flag = it
            if grp == "R" and rk.has_right:
                assert ranks[rk.r + 1].y_flag == it - 1
                ranks[rk.r + 1].y_flag = it
        steps += 1
    return steps


@pytest.mark.parametrize("world", [2, 3, 4])
def test_two_slot_halo_protocol_is_safe_and_live(world):
    for seed in range(40):
        run_model(world, n_iters=7, n_tiles=3, check_every=3, seed=seed)


# Sanity of the model itself: if a group published its sequence number after its FIRST tile, a neighbour could
# overwrite a slot that other tiles still have to read (or a reader could see a half-written column) -- the model
# must notice.
def _broken_model(world, n_iters, n_tiles, seed):
    rng = random.Random(seed)
    ranks = [Rank(r, world, n_tiles) for r in range(world)]
    total = world * 2 * n_tiles * n_iters
    completed = 0
    while completed < total:
        enabled = []
        for rk in ranks:
            for grp in ("L", "R"):
                for j in range(n_tiles):
                    it = rk.done[grp][j] + 1
                    if it > n_iters:
                        continue
                    if any(rk.done[g][t] < it - 1 for g in ("L", "R") for t in range(n_tiles)):
                        continue
                    if grp == "L" and rk.has_left and it > 1 and rk.y_flag < it - 1:
                        continue
                    if grp == "R" and rk.has_right and rk.x_flag < it:
                        continue
                    enabled.append((rk, grp, j, it))
        if not enabled:
            return "deadlock"
        rk, grp, j, it = rng.choice(enabled)
        segs = [t for t in (j, j + 1) if t < n_tiles]
        if grp == "L" and rk.has_left:
            if it > 1 and any(rk.y_slot[(it - 1) & 1][t] != (rk.r - 1, it - 1) for t in segs):
                return "stale y halo"
            ranks[rk.r - 1].x_slot[it & 1][j] = (rk.r, it)
            ranks[rk.r - 1].x_flag = max(ranks[rk.r - 1].x_flag, it)          # BROKEN: published by the first tile
        if grp == "R" and rk.has_right:
            if any(rk.x_slot[it & 1][t] != (rk.r + 1, it) for t in segs) or \
                    (it > 1 and any(rk.x_slot[(it - 1) & 1][t] != (rk.r + 1, it - 1) for t in segs)):
                return "stale x halo"
            ranks[rk.r + 1].y_slot[it & 1][j] = (rk.r, it)
            ranks[rk.r + 1].y_flag = max(ranks[rk.r + 1].y_flag, it)          # BROKEN
        rk.done[grp][j] = it
        completed += 1
    return "ok"


def test_model_detects_a_broken_protocol():
    outcomes = {_broken_model(3, n_iters=7, n_tiles=3, seed=s) for s in range(200)}
    assert outcomes - {"ok"}, "the model never noticed that early publishing is unsafe"


# ---- flag-in-data protocol of the ring kernel (round 2) ----------------------------------------------------------
# Every segment of a column carries the tag (writer rank, iteration) itself; there is no separate flag and no
# counter.  Left-edge tile j of iteration `it` waits until segments j and j+1 of y slot (it-1) % Y carry the tag
# of the left neighbour's iteration it-1, reads (refresh iterations) the column before it from slot (it-2) % Y,
# then stores x segment j into the left neighbour's slot it & 1.  Right-edge tile j waits for x segment j of slot
# it & 1 (tag: right neighbour, iteration it), reads segment j of the other slot (iteration it-1) and stores y
# segment j into the right neighbour's slot it % Y.  Y = 3 in the product; the model shows that Y = 2 is NOT
# enough once refresh iterations read the column before the newest one.
class LLRank:
    def __init__(self, r, world, n_tiles, y_slots):
        self.r, self.world = r, world
        self.has_left, self.has_right = r > 0, r + 1 < world
        self.x_slot = [[None] * n_tiles for _ in range(2)]
        self.y_slot = [[None] * n_tiles for _ in range(y_slots)]
        self.done = {"L": [0] * n_tiles, "R": [0] * n_tiles}


def run_model_ll(world, n_iters, n_tiles, check_every, seed, y_slots=3):
    rng = random.Random(seed)
    ranks = [LLRank(r, world, n_tiles, y_slots) for r in range(world)]
    total = world * 2 * n_tiles * n_iters
    completed = 0
    while completed < total:
        enabled = []
        for rk in ranks:
            for grp in ("L", "R"):
                for j in range(n_tiles):
                    it = rk.done[grp][j] + 1
                    if it > n_iters:
                        continue
                    if any(rk.done[g][t] < it - 1 for g in ("L", "R") for t in range(n_tiles)):
                        continue
                    segs = [t for t in (j, j + 1) if t < n_tiles]
                    # the waits: tags in the data (iteration 1 = the two-pass iteration 0 of the solver, no y halo)
                    if grp == "L" and rk.has_left and it > 1 and \
                            any(rk.y_slot[(it - 1) % y_slots][t] != (rk.r - 1, it - 1) for t in segs):
                        continue
                    if grp == "R" and rk.has_right and rk.x_slot[it & 1][j] != (rk.r + 1, it):
                        continue
                    enabled.append((rk, grp, j, it, segs))
        if not enabled:
            return "deadlock"
        rk, grp, j, it, segs = rng.choice(enabled)
        refresh = check_every and it % check_every == 0
        if grp == "L" and rk.has_left:
            if refresh and it > 2 and any(rk.y_slot[(it - 2) % y_slots][t] != (rk.r - 1, it - 2) for t in segs):
                return "stale previous y halo"
            ranks[rk.r - 1].x_slot[it & 1][j] = (rk.r, it)
        if grp == "R" and rk.has_right:
            if it > 1 and rk.x_slot[(it - 1) & 1][j] != (rk.r + 1, it - 1):
                return "stale previous x halo"
            ranks[rk.r + 1].y_slot[it % y_slots][j] = (rk.r, it)
        rk.done[grp][j] = it
        completed += 1
    return "ok"


@pytest.mark.parametrize("world", [2, 3, 4])
def test_flag_in_data_halo_protocol_is_safe_and_live(world):
    for seed in range(60):
        assert run_model_ll(world, n_iters=8, n_tiles=3, check_every=3, seed=seed) == "ok"
        assert run_model_ll(world, n_iters=8, n_tiles=4, check_every=1, seed=seed) == "ok"


def test_flag_in_data_model_needs_the_third_y_slot():
    outcomes = {run_model_ll(3, n_iters=8, n_tiles=3, check_every=1, seed=s, y_slots=2) for s in range(300)}
    assert "stale previous y halo" in outcomes, "two y slots should be caught as unsafe under refresh reads"
    assert "deadlock" not in outcomes
