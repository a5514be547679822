"""CPU checks of the random placement restatement (tests/random_placement_ref.py): the draw rules, and the kernel's
32-candidate warp acceptance rule against the reference's sequential loop."""
import numpy as np
import pytest

from random_placement_ref import (Draws, border_walls, episode_placement, minstd_next, place_sequential, place_warp,
                                  whole_map)


def test_minstd_first_draws_from_seed_0():
    s, out = 1, []          # seed 0 -> state 1 (libstdc++ linear_congruential_engine::seed)
    for _ in range(4):
        s = minstd_next(s)
        out.append(s)
    assert out == [16807, 282475249, 1622650073, 984943658]


def test_whole_map_minstd_candidates_are_the_reference_formula():
    W, H = 40, 30
    occ = border_walls(W, H)
    d = Draws("minstd", W, H, rs=1)
    cells, short = place_sequential(d, occ.copy(), [(0, 1, whole_map(W, H))])
    # 16807 % 39 = 37, 282475249 % 29 = 1: blank, so the first candidate is taken
    assert cells == [[(16807 % 39, 282475249 % 29)]] and short == 0
    assert d.rs == 282475249


def test_philox_counter_and_mulhi():
    from philox_ref import philox4x32_10
    d = Draws("philox", 40, 40, seed=7, gid=3, episode=2, generation=5)
    xs, ys = d.philox_cells(1, [4], (2, 3, 10, 20))
    r = philox4x32_10([np.uint32(4), np.uint32(1), np.uint32(2), np.uint32(5 | 0x80000000)], [np.uint32(7), np.uint32(3)])
    assert xs[0] == 2 + (int(r[0]) * 10 >> 32) and ys[0] == 3 + (int(r[1]) * 20 >> 32)


def _fill(rng, W, H, frac):
    occ = border_walls(W, H)
    inner = rng.random_sample((H, W)) < frac
    return occ | inner


@pytest.mark.parametrize("mode", ["minstd", "philox"])
def test_warp_rule_equals_sequential_loop(mode):
    rng = np.random.RandomState(0)
    for trial in range(60):
        W, H = int(rng.randint(4, 14)), int(rng.randint(4, 14))
        occ = _fill(rng, W, H, rng.uniform(0, 0.9))
        ops = []
        for _ in range(int(rng.randint(1, 4))):
            w, h = int(rng.randint(1, W + 1)), int(rng.randint(1, H + 1))
            x0, y0 = int(rng.randint(0, W - w + 1)), int(rng.randint(0, H - h + 1))
            ops.append((int(rng.randint(0, 2)), int(rng.randint(0, 40)), (x0, y0, w, h)))
        args = dict(rs=int(rng.randint(1, 2**31 - 1)), seed=int(rng.randint(0, 2**32)), gid=trial, episode=trial % 3,
                    generation=trial % 5)
        a, b = Draws(mode, W, H, **args), Draws(mode, W, H, **args)
        oa, ob = occ.copy(), occ.copy()
        ca, sa = place_sequential(a, oa, ops)
        cb, sb = place_warp(b, ob, ops)
        assert ca == cb and sa == sb, trial
        assert a.rs == b.rs
        assert np.array_equal(oa, ob)


def test_warp_rule_with_nearly_full_rectangles_hits_the_cap_like_the_loop():
    # one blank cell in a small map: some seeds give up after W*H + 1 failed candidates
    W = H = 5
    occ = np.ones((H, W), dtype=bool)
    occ[2, 2] = False
    shorts = 0
    for s in range(1, 400):
        a, b = Draws("minstd", W, H, rs=s), Draws("minstd", W, H, rs=s)
        ca, sa = place_sequential(a, occ.copy(), [(0, 1, whole_map(W, H))])
        cb, sb = place_warp(b, occ.copy(), [(0, 1, whole_map(W, H))])
        assert (ca, sa, a.rs) == (cb, sb, b.rs)
        shorts += sa
    assert 0 < shorts < 399


def test_episode_placement_swaps_groups_and_ids():
    W = H = 12
    walls = border_walls(W, H)
    fixed = [[(1, 1, 0), (2, 1, 1)], [(9, 9, 2)]]
    ops = [(0, 3, (1, 1, 5, 10)), (1, 2, (6, 1, 5, 10))]
    p0, i0, s0, _ = episode_placement("philox", W, H, walls, fixed, ops, side=0, seed=1, gid=0)
    p1, i1, s1, _ = episode_placement("philox", W, H, walls, fixed, ops, side=1, seed=1, gid=0)
    assert s0 == s1 == 0
    assert i0 == [[0, 1, 3, 4, 5], [2, 6, 7]]
    assert i1 == [[2, 6, 7], [0, 1, 3, 4, 5]]
    assert p0[0] == p1[1] and p0[1] == p1[0]
