"""Battle maps and armies whose kernels do not fit in shared memory: k_step runs from a per-env HBM workspace, k_obs
and K7 read the observation record in HBM, and the record is built in place.  Each case asserts which kernels ran
from HBM (mfb_query "hbm_kernels": 1 k_step, 2 k_obs, 4 k_obs_record, 8 k_local_mean_action) and checks every output
bit against the C oracle (or, for K7, the numpy reference)."""
import importlib.util
import os

import numpy as np
import pytest

from engines import CudaEngine, OracleEngine
from lockstep import assert_same, run_lockstep, setup_pair
from scenarios import block_positions, generate_map_positions
from local_mean_ref import local_mean_action
from test_cuda_battle_batched import lockstep_batched, make, per_env_placements

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

STEP, OBS, RECORD, LOCAL = 1, 2, 4, 8


def density_cap(m):
    return max(64, int(m * m * 0.04))   # train_battle.py's capacity for --map_size m


@pytest.mark.parametrize("m, mask", [(176, STEP), (256, STEP | OBS)])
def test_scripts_density_against_the_oracle(m, mask):
    env, oracles = make(2, map_size=m, cap=density_cap(m))
    assert env.query("hbm_kernels") == mask
    lockstep_batched(env, oracles, steps=6, seed=m, check_obs_every=3)


def test_walls_at_340_run_the_record_from_hbm_too():
    m = 340
    left, right = generate_map_positions(m)
    walls = np.array([[m // 2, y, 0] for y in range(20, m - 20, 3)], np.int32)
    env, oracles = make(3, map_size=m, cap=density_cap(m), pos=(left, right))
    env.reset(); env.add_walls(walls); env.add_agents(0, left); env.add_agents(1, right)
    for o in oracles:
        o.reset(); o.add_walls(walls); o.add_agents(0, left); o.add_agents(1, right)
    assert env.query("hbm_kernels") == STEP | OBS | RECORD
    lockstep_batched(env, oracles, steps=4, seed=5, check_obs_every=2)


def sparse_600():
    # a few hundred agents on a 600x600 map, close enough to fight
    return block_positions(280, 280, 10, 12, stride=2), block_positions(301, 280, 10, 12, stride=2)


def test_sparse_600_runs_every_kernel_from_hbm():
    env, oracles = make(2, map_size=600, cap=128, pos=sparse_600())
    assert env.query("hbm_kernels") == STEP | OBS | RECORD | LOCAL
    lockstep_batched(env, oracles, steps=30, seed=6, check_obs_every=5, min_deaths=1)


def test_more_than_4095_attacks_in_one_step_minstd():
    """Two touching stride-1 blocks of 2304 per group, every agent attacking toward the other block: more than 4095
    attacks per step, so the minstd_rand0 jump needs the 13th and 14th bits of its table.  Agents on the front are hit
    several times a step and die, so the shuffled order decides who acts before being killed."""
    m, cols, rows = 200, 48, 48
    pos = (block_positions(52, 76, cols, rows, stride=1), block_positions(100, 76, cols, rows, stride=1))
    env, oracles = make(1, map_size=m, cap=cols * rows, pos=pos)
    assert env.query("hbm_kernels") & STEP
    o = oracles[0]
    table, base = o.action_table()
    toward = [[a for a in range(base, 21) if table[a][0] == (1 if g == 0 else -1)] for g in range(2)]
    assert all(len(t) == 3 for t in toward)
    rng = np.random.RandomState(0)
    kills = 0
    for s in range(20):
        num = env.get_num()
        acts = np.zeros((1, 2, env.capacity), np.int32)
        for g in range(2):
            acts[0, g, :num[0, g]] = rng.choice(toward[g], size=num[0, g])
            o.set_action(g, acts[0, g, :num[0, g]])
        assert o.attack_count() > 4095, o.attack_count()
        reward, alive, done, _ = env.step(torch.from_numpy(acts).cuda())
        reward, alive = reward.cpu().numpy(), alive.cpu().numpy()
        o.step()
        for g in range(2):
            n = num[0, g]
            assert_same("reward g%d" % g, o.get_reward(g), reward[0, g, :n], s)
            assert_same("alive g%d" % g, o.get_alive(g), alive[0, g, :n].astype(bool), s)
            kills += int((~o.get_alive(g)).sum())
        o.clear_dead()
        for g in range(2):
            assert_same("hp g%d" % g, o.get_hp(g), env.get("hp")[0, g, :env.get_num()[0, g]], s)
    assert kills > 20, kills


def test_bf16_rows_are_the_fp32_rows_rounded_at_a_big_geometry():
    m = 256
    env, _ = make(2, map_size=m, cap=density_cap(m))
    assert env.query("hbm_kernels") & OBS
    rng = np.random.RandomState(1)
    for _ in range(2):
        num = env.get_num()
        acts = np.zeros((2, 2, env.capacity), np.int32)
        for e in range(2):
            for g in range(2):
                acts[e, g, :num[e, g]] = rng.randint(0, 21, size=num[e, g])
        env.step(torch.from_numpy(acts).cuda())
    num = env.get_num()
    out32 = env.observe_groups(dtype=torch.float32)
    out16 = env.observe_groups(dtype=torch.bfloat16)
    for g in range(2):
        (v32, f32), (v16, f16) = out32[g], out16[g]
        for e in range(2):
            n = num[e, g]
            ref = v32[e, :n].to(torch.bfloat16).reshape(n, 169, 7)
            got = v16[e, :n].reshape(n, 169, 8)
            assert torch.equal(got[..., :7].view(torch.int16), ref.view(torch.int16)) and not got[..., 7].any()
            assert torch.equal(f16[e, :n], f32[e, :n])


@pytest.mark.parametrize("m, cap, pos", [(256, density_cap(256), None), (600, 128, sparse_600())])
def test_local_mean_action_at_a_big_geometry(m, cap, pos):
    env, oracles = make(2, map_size=m, cap=cap, pos=pos)
    assert bool(env.query("hbm_kernels") & LOCAL) == (m == 600)
    rng = np.random.RandomState(2)
    last = [[None, None] for _ in oracles]
    for s in range(4):
        num = env.get_num()
        acts = np.zeros((2, 2, env.capacity), np.int32)
        for e, o in enumerate(oracles):
            for g in range(2):
                acts[e, g, :num[e, g]] = rng.randint(0, 21, size=num[e, g])
                o.set_action(g, acts[e, g, :num[e, g]])
        _, alive, _, _ = env.step(torch.from_numpy(acts).cuda())
        alive = alive.cpu().numpy()
        for e, o in enumerate(oracles):
            o.step()
            for g in range(2):
                al = alive[e, g, :num[e, g]].astype(bool)
                last[e][g] = acts[e, g, :num[e, g]][al].astype(np.int64)
            o.clear_dead()
        num = env.get_num()
        for r in (6, 1.5):
            out = [t.cpu().numpy() for t in env.local_mean_action(radius=r)]
            for e, o in enumerate(oracles):
                for g in range(2):
                    n = num[e, g]
                    ref = local_mean_action(o.get_pos(g), last[e][g], np.ones(n, bool), r, 21)
                    assert_same("local r=%g e%d g%d" % (r, e, g), ref, out[g][e, :n], s)
                    assert not out[g][e, n:].any()


def test_auto_reset_and_random_sides_at_a_big_geometry():
    from mfmarl_b200 import BatchedGridWorld
    m = 200
    left, right = generate_map_positions(m)
    env = BatchedGridWorld(4, map_size=m, capacity=density_cap(m), rng="philox", seed=3, max_steps=3, auto_reset=True,
                           random_sides=True)
    env.reset(); env.add_agents(0, left); env.add_agents(1, right)
    assert env.query("hbm_kernels") & STEP
    pos0 = env.get("pos").copy()
    rng = np.random.RandomState(0)
    for _ in range(3):
        env.step(torch.from_numpy(rng.randint(0, 21, size=(4, 2, env.capacity)).astype(np.int32)).cuda())
    assert (env.get("step_ct") == 0).all()
    side = env.get("side")
    pos, num = env.get("pos"), env.get_num()
    for e in range(4):
        for g in range(2):
            src = (1 - g) if side[e] else g
            assert num[e, g] == len((left, right)[src])
            assert np.array_equal(pos[e, g, :num[e, g]], pos0[0, src, :num[e, g]])


def test_per_env_placements_at_a_big_geometry():
    from mfmarl_b200 import BatchedGridWorld
    E, m = 2, 180
    p0, p1 = per_env_placements(E, m, np.random.RandomState(4))
    env = BatchedGridWorld(E, map_size=m, capacity=density_cap(m))
    env.reset()
    added0, added1 = env.add_agents_per_env(0, p0), env.add_agents_per_env(1, p1)
    assert env.query("hbm_kernels") & STEP
    oracles = []
    for e in range(E):
        o = OracleEngine(m)
        o.reset()
        assert o.add_agents(0, np.c_[p0[e], np.zeros(len(p0[e]), np.int32)]) == added0[e]
        assert o.add_agents(1, np.c_[p1[e], np.zeros(len(p1[e]), np.int32)]) == added1[e]
        oracles.append(o)
    lockstep_batched(env, oracles, steps=5, seed=9, check_obs_every=2)


def test_single_env_abi_at_map_size_200():
    ora, cu = OracleEngine(200), CudaEngine(200)
    setup_pair([ora, cu], *generate_map_positions(200))
    run_lockstep(ora, cu, steps=8, seed=1, stream="fight", check_obs_every=4)


def test_record_off_is_refused_at_a_big_geometry():
    from mfmarl_b200 import BatchedGridWorld
    with pytest.raises(Exception, match="observation record"):
        BatchedGridWorld(1, map_size=256, capacity=density_cap(256), obs_record=0)


def _script(name):
    from conftest import PKG
    spec = importlib.util.spec_from_file_location(name, os.path.join(PKG, "python", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_train_and_battle_scripts_at_map_size_200(tmp_path):
    data = str(tmp_path / "data")
    runner = _script("train_battle").main(["--algo", "mfq", "--envs", "2", "--map_size", "200", "--n_round", "1",
                                           "--max_steps", "4", "--data_dir", data])
    assert runner is not None
    for side, model in enumerate(runner.models):   # (training saves only after a round the main model won)
        model.save(os.path.join(data, "models", "mfq-%d" % side), 0)
    _script("battle").main(["--algo", "mfq", "--oppo", "mfq", "--idx", "0", "0", "--map_size", "200", "--n_round", "1",
                            "--max_steps", "4", "--data_dir", data])
