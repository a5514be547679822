"""GPU parity tests proper: the CUDA engine through the reference-facing C ABI (host buffers) against the
plain-C oracle on identical action streams -- every output compared bit for bit."""
import numpy as np
import pytest

from engines import CudaEngine, OracleEngine
from lockstep import assert_same, run_lockstep, setup_pair
from scenarios import c4_positions, generate_map_positions

pytestmark = pytest.mark.gpu


def test_spaces():
    cu = CudaEngine(40)
    assert cu.env.view_space[0] == (13, 13, 7)
    assert cu.env.feature_space[0] == (34,)
    assert cu.env.action_space[0] == (21,)
    base, v2a = cu.env.get_view2attack(cu.h[0])
    table, obase = OracleEngine(40).action_table()
    assert base == obase == 13
    for k in range(8):
        dx, dy = table[13 + k]
        assert v2a[6 + dy, 6 + dx] == k
    assert (v2a >= 0).sum() == 8


@pytest.mark.parametrize("seed", [0, 1])
def test_battle40_fight_stream(seed):
    ora, cu = OracleEngine(40), CudaEngine(40)
    left, right = generate_map_positions(40)
    pos = (left, right) if seed == 0 else (right, left)
    setup_pair([ora, cu], *pos)
    st = run_lockstep(ora, cu, steps=300, seed=seed, stream="fight")
    assert st["deaths"] > 20, st


def test_battle40_uniform_stream():
    ora, cu = OracleEngine(40), CudaEngine(40)
    setup_pair([ora, cu], *generate_map_positions(40))
    run_lockstep(ora, cu, steps=60, seed=3, stream="uniform")


def test_battle80_512v512():
    ora, cu = OracleEngine(80), CudaEngine(80)
    setup_pair([ora, cu], *c4_positions())
    st = run_lockstep(ora, cu, steps=60, seed=5, stream="fight", check_obs_every=5)
    assert st["deaths"] > 20, st


def test_second_episode_keeps_rng_and_resets_ids():
    ora, cu = OracleEngine(40), CudaEngine(40)
    for ep in range(2):
        setup_pair([ora, cu], *generate_map_positions(40))
        run_lockstep(ora, cu, steps=40, seed=10 + ep, stream="fight", check_obs_every=10)


def test_set_seed_and_occupied_positions_are_skipped():
    ora, cu = OracleEngine(40), CudaEngine(40)
    for e in (ora, cu):
        e.set_seed(1234)
    left, right = generate_map_positions(40)
    dup = np.concatenate([left, left[:5], np.array([[0, 5, 0], [39, 39, 0]], np.int32)])
    setup_pair([ora, cu], dup, right)
    assert ora.get_num(0) == cu.get_num(0) == len(left)
    run_lockstep(ora, cu, steps=50, seed=7, stream="fight", check_obs_every=10)


def test_inner_walls_and_observation_before_clear_dead():
    ora, cu = OracleEngine(40), CudaEngine(40)
    walls = np.array([[20, y] for y in range(5, 35, 3)] + [[19, 20], [21, 20]], np.int32)
    left, right = generate_map_positions(40)
    setup_pair([ora, cu], left, right, walls=walls)
    run_lockstep(ora, cu, steps=120, seed=11, stream="fight", skip_clear_every=4)


def test_ragged_group_sizes():
    """group sizes that are not multiples of the 8-agent store chunk nor of 4 (16-byte tail rounding)"""
    ora, cu = OracleEngine(40), CudaEngine(40)
    left, right = generate_map_positions(40)
    setup_pair([ora, cu], left[:13], right[:7])
    run_lockstep(ora, cu, steps=80, seed=4, stream="fight")


def test_mean_info_matches():
    ora, cu = OracleEngine(40), CudaEngine(40)
    setup_pair([ora, cu], *generate_map_positions(40))

    def check(s, A, B, acts):
        for g in range(2):
            assert_same("mean_info", A.get_mean_info(g), B.get_mean_info(g), s)

    run_lockstep(ora, cu, steps=30, seed=2, stream="fight", check_obs_every=0, on_step=check)


def test_injected_attack_order():
    """the test hook: both engines resolve attacks in one injected permutation instead of the RNG"""
    import ctypes
    ora, cu = OracleEngine(40), CudaEngine(40)
    setup_pair([ora, cu], *generate_map_positions(40))
    prng = np.random.RandomState(99)

    def inject(s, A, B, acts):
        n_att = int(sum((a >= 13).sum() for a in acts))
        perm = prng.permutation(n_att).astype(np.int32)
        A.inject_attack_order(perm)
        B.lib.mfmarl_inject_attack_order.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        B.lib.mfmarl_inject_attack_order(B.env.game, perm.ctypes.data_as(ctypes.c_void_p), n_att)

    st = run_lockstep(ora, cu, steps=150, seed=21, stream="fight", check_obs_every=10, on_step=inject)
    assert st["deaths"] > 10


def test_global_minimap_and_getters_match_the_reference_engine():
    """get_info keys the scripts can reach (GridWorld.cc:777-978): global_minimap, pos, id, alive, num -- CUDA engine
    against the unmodified reference engine mid-fight (dead agents still in the lists)."""
    from engines import RefEngine, have_ref
    from scenarios import fight_actions
    if not have_ref():
        pytest.skip("oracle/_ref not built")
    ref, cu = RefEngine(40), CudaEngine(40)
    left, right = generate_map_positions(40)
    for eng in (ref, cu):
        eng.reset(); eng.add_agents(0, left); eng.add_agents(1, right)
    rng = np.random.RandomState(3)
    for s in range(40):
        for g in range(2):
            a = fight_actions(rng, ref.get_pos(g), 40)
            ref.set_action(g, a); cu.set_action(g, a)
        assert ref.step() == cu.step()
        if s % 8 == 7:                      # between step and clear_dead: the dead are still listed
            for hw in ((10, 10), (13, 13), (7, 5)):
                a, b = ref.env.get_global_minimap(*hw), cu.env.get_global_minimap(*hw)
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (s, hw)
            for g in range(2):
                assert np.array_equal(ref.get_pos(g), cu.get_pos(g)) and np.array_equal(ref.get_agent_id(g), cu.get_agent_id(g))
                assert np.array_equal(ref.get_alive(g), cu.get_alive(g)) and ref.get_num(g) == cu.get_num(g)
        ref.clear_dead(); cu.clear_dead()
    assert ref.get_num(0) + ref.get_num(1) < 128


@pytest.mark.parametrize("size", [100, 104])
def test_large_map_mode_moves_run_band_by_band(size):
    """W*H > 99*99: the reference resolves moves x-band by x-band, then the band-boundary buffer
    (GridWorld.cc:79-88,443-463,662-672); k_step builds its move list in that order (ADVICE r1)."""
    from scenarios import block_positions
    ora, cu = OracleEngine(size), CudaEngine(size)
    left, right = block_positions(20, 30, 28, 20, stride=1), block_positions(size - 50, 30, 28, 20, stride=1)
    setup_pair([ora, cu], left, right)
    st = run_lockstep(ora, cu, steps=50, seed=size, stream="fight", check_obs_every=10)
    assert st["deaths"] > 20, st


def test_queries_after_a_late_or_random_add_see_the_new_agents():
    """add_agents after a step (late path) and method="random" rewrite the device state: the host mirror that answers
    get_pos / get_agent_id / get_observation must be refreshed (ADVICE r1, runtime_api.cu gridworld_add_agents)."""
    ora, cu = OracleEngine(40), CudaEngine(40)
    left, right = generate_map_positions(40)
    setup_pair([ora, cu], left[:20], right[:20])
    run_lockstep(ora, cu, steps=5, seed=1, stream="fight")
    for g in range(2):                         # warm the mirror, then add: the next getters must not answer from it
        cu.get_pos(g); cu.get_observation(g)
    extra0 = np.array([[30, 3, 0], [31, 3, 0], [32, 3, 0]], np.int32)
    extra1 = np.array([[30, 36, 0], [31, 36, 0]], np.int32)
    for eng in (ora, cu):
        eng.add_agents(0, extra0); eng.add_agents(1, extra1)
    for g in range(2):
        assert ora.get_num(g) == cu.get_num(g)
        assert_same("pos", ora.get_pos(g), cu.get_pos(g), 0)
        assert_same("id", ora.get_agent_id(g), cu.get_agent_id(g), 0)
        va, fa = ora.get_observation(g); vb, fb = cu.get_observation(g)
        assert_same("view", va, vb, 0); assert_same("feature", fa, fb, 0)
    run_lockstep(ora, cu, steps=20, seed=2, stream="fight")
    # method="random": positions come from the engine RNG; a getter between two random adds must see the first one
    cu2 = CudaEngine(40)
    cu2.reset()
    cu2.env.add_agents(cu2.h[0], method="random", n=10)
    p0 = cu2.get_pos(0).copy()
    assert len(p0) == 10 and (p0 > 0).all()
    cu2.env.add_agents(cu2.h[1], method="random", n=7)
    p1 = cu2.get_pos(1)
    assert len(p1) == 7 and (p1 > 0).all()
    assert len({tuple(p) for p in np.concatenate([p0, p1])}) == 17


def test_two_engine_shapes_interleaved_in_one_process():
    """cudaFuncAttributeMaxDynamicSharedMemorySize is per function and process wide: a small engine created after a
    large one must not lower the limit the large one still needs (ADVICE r1, engine.cu)."""
    big_o, big = OracleEngine(80), CudaEngine(80)
    setup_pair([big_o, big], *c4_positions())
    run_lockstep(big_o, big, steps=3, seed=5, stream="fight", check_obs_every=1)
    small_o, small = OracleEngine(40), CudaEngine(40)
    setup_pair([small_o, small], *generate_map_positions(40))
    run_lockstep(small_o, small, steps=3, seed=6, stream="fight", check_obs_every=1)
    run_lockstep(big_o, big, steps=3, seed=7, stream="fight", check_obs_every=1)
    run_lockstep(small_o, small, steps=3, seed=8, stream="fight", check_obs_every=1)


def test_speculation_rolls_back_when_the_caller_leaves_the_play_loop_order():
    """env_step enqueues clear_dead + both observations behind the step (runtime_api.cu).  Whatever the caller does
    next must see the reference's state: a second step without clear_dead, set_action / get_observation / add_agents
    between step and clear_dead (the dead still listed, GridWorld.cc:696-728 not run yet)."""
    ora, cu = OracleEngine(40), CudaEngine(40)
    setup_pair([ora, cu], *generate_map_positions(40))
    # (a) no observation at all and every 3rd clear_dead skipped: after a skipped one, set_action is the first call
    st = run_lockstep(ora, cu, steps=90, seed=31, stream="fight", check_obs_every=0, skip_clear_every=3)
    assert st["deaths"] > 5, st
    # (b) observation between step and clear_dead on every step
    rng = np.random.RandomState(5)
    from scenarios import fight_actions
    for s in range(30):
        for g in range(2):
            a = fight_actions(rng, ora.get_pos(g), 40)
            ora.set_action(g, a); cu.set_action(g, a)
        assert ora.step() == cu.step()
        for g in range(2):
            va, fa = ora.get_observation(g); vb, fb = cu.get_observation(g)
            assert_same("view before clear_dead", va, vb, s); assert_same("feature before clear_dead", fa, fb, s)
            assert_same("reward", ora.get_reward(g), cu.get_reward(g), s)
            assert_same("alive", ora.get_alive(g), cu.get_alive(g), s)
        if s % 7 == 3:                      # (c) a late add between step and clear_dead
            extra = np.array([[2 + s % 5, 2, 0], [3 + s % 5, 37, 0]], np.int32)
            for eng in (ora, cu):
                eng.add_agents(s % 2, extra)
        ora.clear_dead(); cu.clear_dead()
        for g in range(2):
            assert ora.get_num(g) == cu.get_num(g)
            assert_same("id", ora.get_agent_id(g), cu.get_agent_id(g), s)
            assert_same("pos", ora.get_pos(g), cu.get_pos(g), s)
    run_lockstep(ora, cu, steps=30, seed=32, stream="fight")


def test_step_graph_replay_follows_every_change_of_the_step_shape():
    """After two plain steps env_step replays the steady sequence (set_action x2 + step + speculative clear_dead +
    observe x2 + copies) as a CUDA graph (runtime_api.cu).  Everything baked into a graph changes here while it is in
    use: the order of the set_action calls, a group that does not act, a late add that grows the capacity (every
    buffer re-allocated), a new episode -- and the results stay the oracle's bit for bit."""
    from scenarios import fight_actions
    ora, cu = OracleEngine(40), CudaEngine(40)
    left, right = generate_map_positions(40)
    rng = np.random.RandomState(17)

    def check(s):
        for g in range(2):
            assert ora.get_num(g) == cu.get_num(g)
            assert_same("reward", ora.get_reward(g), cu.get_reward(g), s)
            assert_same("alive", ora.get_alive(g), cu.get_alive(g), s)
        ora.clear_dead(); cu.clear_dead()
        for g in range(2):
            va, fa = ora.get_observation(g); vb, fb = cu.get_observation(g)
            assert_same("view", va, vb, s); assert_same("feature", fa, fb, s)
            assert_same("id", ora.get_agent_id(g), cu.get_agent_id(g), s)
            assert_same("pos", ora.get_pos(g), cu.get_pos(g), s)

    import ctypes
    cu.lib.mfmarl_step_graph_replays.argtypes = [ctypes.c_void_p]
    replays = lambda: cu.lib.mfmarl_step_graph_replays(cu.env.game)
    for episode in range(2):
        setup_pair([ora, cu], left, right)
        for s in range(60):
            before = replays()
            order = (0, 1) if (s // 6) % 2 == 0 else (1, 0)          # the set_action order is part of the graph key
            if s % 17 == 16:
                order = order[:1]                                     # one group does not act this step
            acts = {g: fight_actions(rng, ora.get_pos(g), 40) for g in range(2)}
            for g in order:
                ora.set_action(g, acts[g]); cu.set_action(g, acts[g])
            assert ora.step() == cu.step()
            # late adds: 64 -> 66 agents in episode 0 (the capacity grows, every buffer moves); in episode 1 right after
            # its FIRST step, which was a graph replay (nothing but the replay tells the engine that it has stepped)
            if (s == 25 and episode == 0) or (s == 0 and episode == 1):
                assert replays() == before + 1, "this step was meant to be a graph replay"
                extra = np.array([[20, 3, 0], [21, 3, 0]], np.int32)
                check(s)
                for eng in (ora, cu):
                    eng.add_agents(0, extra)
                for g in range(2):
                    assert_same("pos after add", ora.get_pos(g), cu.get_pos(g), s)
            else:
                check(s)
    assert replays() > 80, replays()
