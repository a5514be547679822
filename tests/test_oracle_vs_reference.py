"""Pins the plain-C oracle (oracle/magent_oracle.c) against the reference engine itself
(oracle/_ref/libmagent_ref.so, built from /root/reference by oracle/Makefile, OMP_NUM_THREADS=1).
CPU only.  The tests that run the reference are skipped when its build is not present."""
import numpy as np
import pytest

from engines import OracleEngine, RefEngine, have_ref
from lockstep import assert_same, run_lockstep, setup_pair
from scenarios import c4_positions, generate_map_positions

needs_ref = pytest.mark.skipif(not have_ref(), reason="oracle/_ref/libmagent_ref.so not built")


@needs_ref
def test_spaces_and_action_table():
    ref, ora = RefEngine(40), OracleEngine(40)
    assert ref.env.view_space[0] == (ora.vs, ora.vs, ora.nc) == (13, 13, 7)
    assert ref.env.feature_space[0] == (ora.fs,) == (34,)
    assert ref.env.action_space[0] == (ora.n_action,) == (21,)
    table, base = ora.action_table()
    assert base == 13
    attack_base, v2a = ref.env.get_view2attack(ref.h[0])
    assert attack_base == 13
    # view2attack maps view cells to attack action numbers: same deltas as the oracle's table
    for k in range(8):
        dx, dy = table[13 + k]
        assert v2a[6 + dy, 6 + dx] == k
    assert (v2a >= 0).sum() == 8


def test_minstd_rand0_matches_libstdcxx():
    ora = OracleEngine(40)
    assert [ora.rng_next() for _ in range(4)] == [16807, 282475249, 1622650073, 984943658]


@needs_ref
@pytest.mark.parametrize("seed", [0, 1])
def test_battle40_fight_stream(seed):
    ref, ora = RefEngine(40), OracleEngine(40)
    left, right = generate_map_positions(40)
    pos = (left, right) if seed == 0 else (right, left)
    setup_pair([ref, ora], *pos)
    st = run_lockstep(ref, ora, steps=300, seed=seed, stream="fight")
    assert st["deaths"] > 20, st


@needs_ref
def test_battle40_uniform_stream():
    ref, ora = RefEngine(40), OracleEngine(40)
    setup_pair([ref, ora], *generate_map_positions(40))
    run_lockstep(ref, ora, steps=60, seed=3, stream="uniform")


@needs_ref
def test_battle80_512v512():
    ref, ora = RefEngine(80), OracleEngine(80)
    setup_pair([ref, ora], *c4_positions())
    st = run_lockstep(ref, ora, steps=60, seed=5, stream="fight", check_obs_every=5)
    assert st["deaths"] > 20, st


@needs_ref
def test_second_episode_keeps_rng_and_resets_ids():
    """reset() restarts ids at 0 but never reseeds the engine RNG (GridWorld.cc:76-124)."""
    ref, ora = RefEngine(40), OracleEngine(40)
    for ep in range(2):
        setup_pair([ref, ora], *generate_map_positions(40))
        run_lockstep(ref, ora, steps=40, seed=10 + ep, stream="fight", check_obs_every=10)


@needs_ref
def test_set_seed_and_occupied_positions_are_skipped():
    ref, ora = RefEngine(40), OracleEngine(40)
    for e in (ref, ora):
        e.set_seed(1234)
    left, right = generate_map_positions(40)
    # duplicates, a wall cell and an out-of-range cell are ignored (GridWorld.cc:180-187)
    dup = np.concatenate([left, left[:5], np.array([[0, 5, 0], [39, 39, 0]], np.int32)])
    setup_pair([ref, ora], dup, right)
    assert ref.get_num(0) == ora.get_num(0) == len(left)
    run_lockstep(ref, ora, steps=50, seed=7, stream="fight", check_obs_every=10)


@needs_ref
def test_inner_walls_and_observation_before_clear_dead():
    ref, ora = RefEngine(40), OracleEngine(40)
    walls = np.array([[20, y] for y in range(5, 35, 3)] + [[19, 20], [21, 20]], np.int32)
    left, right = generate_map_positions(40)
    setup_pair([ref, ora], left, right, walls=walls)
    # every 4th step clear_dead is skipped: the next observation/step sees dead agents in the lists
    run_lockstep(ref, ora, steps=120, seed=11, stream="fight", skip_clear_every=4)


@needs_ref
def test_mean_info_matches():
    ref, ora = RefEngine(40), OracleEngine(40)
    setup_pair([ref, ora], *generate_map_positions(40))

    def check(s, A, B, acts):
        for g in range(2):
            assert_same("mean_info", A.get_mean_info(g), B.get_mean_info(g), s)

    run_lockstep(ref, ora, steps=30, seed=2, stream="fight", check_obs_every=0, on_step=check)


@needs_ref
@pytest.mark.parametrize("size", [100, 104])
def test_large_map_mode_moves_run_band_by_band(size):
    """W*H > 99*99 switches the reference to large_map_mode (GridWorld.cc:79-88): moves are filed into x-band
    buffers at set_action (:443-463) and resolved band by band, then the boundary buffer (:662-672) -- a different
    collision order than plain set_action order.  Dense blocks that straddle several bands, crowded fight stream."""
    from scenarios import block_positions
    ref, ora = RefEngine(size), OracleEngine(size)
    left, right = block_positions(20, 30, 28, 20, stride=1), block_positions(size - 50, 30, 28, 20, stride=1)
    setup_pair([ref, ora], left, right)
    st = run_lockstep(ref, ora, steps=50, seed=size, stream="fight", check_obs_every=10)
    assert st["deaths"] > 20, st
