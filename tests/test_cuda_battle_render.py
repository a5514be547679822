"""Observation rows rendered from state records (mfb_render_observations, kernel k_render_obs): bit for bit the rows
k_obs wrote for the same state at every geometry; out-of-range references and foreign records give zero rows and are
counted; the record-backed replay samples exactly what the row replay samples; train_battle.py --replay states trains
to the same parameters as --replay rows."""
import ctypes
import os

import numpy as np
import pytest

from scenarios import c4_positions, fight_actions, generate_map_positions

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def density_cap(m):
    return max(64, int(m * m * 0.04))   # train_battle.py's capacity for --map_size m


def make_engine(E, m, cap, walls=None, per_env=False, **kw):
    from mfmarl_b200 import BatchedGridWorld
    env = BatchedGridWorld(E, map_size=m, capacity=cap, **kw)
    env.reset()
    if walls is not None:
        env.add_walls(walls)
    left, right = c4_positions() if m == 80 else generate_map_positions(m)
    if per_env:                                        # every env its own placement: a few cells dropped per env
        rng = np.random.RandomState(11)
        for g, block in enumerate((left, right)):
            pos = np.repeat(block[None, :, :2], E, axis=0).copy()
            for e in range(E):
                pos[e, rng.choice(len(block), size=rng.randint(1, 6), replace=False)] = (-2, 5)
            env.add_agents_per_env(g, pos)
    else:
        env.add_agents(0, left); env.add_agents(1, right)
    return env


def fight(env, rng):
    num, pos = env.get_num(), env.get("pos")
    acts = np.zeros((env.n_envs, 2, env.capacity), np.int32)
    for e in range(env.n_envs):
        for g in range(2):
            acts[e, g, :num[e, g]] = fight_actions(rng, pos[e, g, :num[e, g]], env.map_size)
    return torch.from_numpy(acts).cuda()


def trajectory(env, steps, seed=0, clear_dead=True):
    """per step: (records [E, R], [(view, feature)] per group as k_obs wrote them, num [E, 2]) -- saved right after
    the observation, before the step"""
    rng = np.random.RandomState(seed)
    out = []
    for _ in range(steps):
        obs = env.observe_groups()
        rec = env.save_envs()
        out.append((rec, [(v.clone(), f.clone()) for v, f in obs], env.get_num()))
        env.step(fight(env, rng), clear_dead=clear_dead)
    return out


def check_render(env, traj, seed=1):
    """every listed slot of both groups of every env and step, rendered in one shuffled call, against k_obs's rows"""
    E = env.n_envs
    records = torch.cat([rec for rec, _, _ in traj])
    rows, want_v, want_f = [], [], []
    for t, (_, obs, num) in enumerate(traj):
        for e in range(E):
            for g in range(2):
                for i in range(num[e, g]):
                    rows.append((t * E + e, g, i))
    rows = np.array(rows, np.int32)
    rows = rows[np.random.RandomState(seed).permutation(len(rows))]
    for r, g, i in rows:
        t, e = divmod(int(r), E)
        want_v.append(traj[t][1][g][0][e, i]); want_f.append(traj[t][1][g][1][e, i])
    bad = torch.full((1,), -1, dtype=torch.int32, device="cuda")
    view, feat = env.render_observations(records, torch.from_numpy(rows).cuda(), bad_rows=bad)
    assert int(bad) == 0
    assert torch.equal(view.view(torch.int32), torch.stack(want_v).view(torch.int32)), "view rows differ"
    assert torch.equal(feat.view(torch.int32), torch.stack(want_f).view(torch.int32)), "feature rows differ"
    return len(rows)


@pytest.mark.parametrize("rng", ["minstd", "philox"])
def test_render_equals_k_obs_c3(rng):
    env = make_engine(4, 40, 64, rng=rng, seed=3)
    assert check_render(env, trajectory(env, 30)) > 1000


def test_render_equals_k_obs_c4_observation_record():
    env = make_engine(2, 80, 512, rng="philox", seed=5)
    assert check_render(env, trajectory(env, 8)) > 3000


def test_render_equals_k_obs_where_k_obs_runs_from_hbm():
    m = 256
    env = make_engine(1, m, density_cap(m), rng="philox", seed=2)
    assert env.capacity == 2624 and env.query("hbm_kernels") & 2
    check_render(env, trajectory(env, 3))


def test_render_equals_k_obs_with_walls_and_per_env_placements():
    walls = np.array([[20, y, 0] for y in range(8, 32)] + [[x, 10, 0] for x in range(5, 15)], np.int32)
    env = make_engine(3, 40, 64, walls=walls, per_env=True, rng="philox", seed=9)
    check_render(env, trajectory(env, 20))


def test_render_equals_k_obs_with_dead_agents_still_listed():
    env = make_engine(2, 40, 64, rng="philox", seed=4)
    traj = trajectory(env, 25, clear_dead=False)
    from mfmarl_b200.battle import decode_env_state
    d = decode_env_state(traj[-1][0][0], 64)            # dead agents are still listed in the last record
    assert any((d["alive"][g, :d["num"][g]] == 0).any() for g in range(2))
    check_render(env, traj)


def test_render_an_empty_group_has_zero_minimap():
    env = make_engine(1, 40, 64, rng="philox", seed=1)
    rec = env.save_envs()
    raw = rec.clone()
    raw.view(torch.int32)[0, 11] = 0                 # num[1] = 0: group 1 is empty, its minimap is 0 / 0 = 0
    env.load_envs(raw)
    obs = env.observe_groups()
    rec2 = env.save_envs()
    n0 = int(env.get_num()[0, 0])
    rows = torch.tensor([[0, 0, i] for i in range(n0)], dtype=torch.int32, device="cuda")
    view, feat = env.render_observations(rec2, rows)
    assert torch.equal(view.view(torch.int32), obs[0][0][0, :n0].view(torch.int32))
    assert torch.equal(feat.view(torch.int32), obs[0][1][0, :n0].view(torch.int32))
    assert torch.equal(view[..., 6].sum(dim=(1, 2)), torch.ones(n0, device="cuda"))   # the self marker alone


def test_zero_rows_and_the_counter():
    walls = np.array([[20, y, 0] for y in range(12, 28)], np.int32)
    env = make_engine(2, 40, 64, rng="philox", seed=7)
    other = make_engine(1, 40, 64, walls=walls, rng="philox", seed=7)
    env.step(fight(env, np.random.RandomState(0)))   # some agents die: num < cap
    rec = env.save_envs()
    num = env.get_num()
    foreign = other.save_envs()
    corrupt = rec[:1].clone()
    corrupt[0, 0] ^= 1                                 # magic
    off_map = rec[:1].clone()
    off_map.view(torch.int32)[0, 24 + 3] = 60000      # group 0 slot 3 off the map (x = 60000)
    records = torch.cat([rec, foreign, corrupt, off_map])   # 0, 1 = env; 2 foreign walls; 3 corrupt; 4 off-map slot 3
    good = [(0, 0, 0), (1, 1, 2), (4, 0, 0), (4, 1, 5)]
    bad = [(5, 0, 0), (-1, 0, 0), (0, 2, 0), (0, -1, 0), (0, 0, 64), (0, 0, -3), (0, 0, int(num[0, 0])),
           (1, 1, int(num[1, 1])), (2, 0, 0), (3, 0, 0), (4, 0, 3)]
    rows = torch.tensor(good + bad, dtype=torch.int32, device="cuda")
    counter = torch.full((1,), 99, dtype=torch.int32, device="cuda")
    view, feat = env.render_observations(records, rows, bad_rows=counter)
    assert int(counter) == len(bad)
    ng = len(good)
    assert not bool(view[ng:].any()) and not bool(feat[ng:].any())
    assert all(bool(view[k].any()) and bool(feat[k].any()) for k in range(ng))
    obs = env.observe_groups()
    for k in (0, 1):                                   # untouched records still render k_obs's rows
        r, g, i = good[k]
        assert torch.equal(view[k].view(torch.int32), obs[g][0][r, i].view(torch.int32))
    # the off-map agent is neither drawn nor counted: its group's minimap total is num - 1 agents' counts over num
    mini = view[2, :, :, 3].sum() - 1.0               # group 0's minimap without the self marker
    assert abs(float(mini) * int(num[0, 0]) - (int(num[0, 0]) - 1)) < 1e-3


def test_host_side_refusals():
    from mfmarl_b200.lib import load_library
    lib = load_library()
    env = make_engine(1, 40, 64)
    rec = env.save_envs()
    rows = torch.zeros((4, 3), dtype=torch.int32, device="cuda")
    view = torch.empty((4, 13, 13, 7), device="cuda")
    feat = torch.empty((4, 34), device="cuda")
    p = lambda t, off=0: ctypes.c_void_p(t.data_ptr() + off)
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    cases = [((1, p(rec), -1, p(rows), p(view), p(feat), None), "n_rows"),
             ((0, p(rec), 4, p(rows), p(view), p(feat), None), "n_records"),
             ((1, None, 4, p(rows), p(view), p(feat), None), "null records"),
             ((1, p(rec), 4, None, p(view), p(feat), None), "null rows"),
             ((1, p(rec), 4, p(rows), None, p(feat), None), "null view"),
             ((1, p(rec), 4, p(rows), p(view), None, None), "null feature"),
             ((1, p(rec, 4), 4, p(rows), p(view), p(feat), None), "records buffer must be 16-byte aligned"),
             ((1, p(rec), 4, p(rows), p(view, 4), p(feat), None), "view buffer must be 16-byte aligned")]
    for args, msg in cases:
        assert lib.mfb_render_observations(env._h, *args, s) == -1
        err = lib.mfb_last_error().decode()
        assert err.startswith("mfb_render_observations: ") and msg in err, err
    assert lib.mfb_render_observations(env._h, 1, p(rec), 0, p(rows), p(view), p(feat), None, s) == 0


def _pushes(env, steps, rng):
    """the arguments play_batched hands the main model's replay, per step: records and the group-0 rows"""
    E, cap = env.n_envs, env.capacity
    former = torch.zeros((E, 21), device="cuda")
    active = torch.ones((E,), dtype=torch.bool, device="cuda")
    for _ in range(steps):
        obs = env.observe_groups()
        rec = env.save_envs()
        num = torch.from_numpy(env.get_num()).cuda()
        ids = env.device_state("id").clone()
        acts = fight(env, rng)
        reward, alive, done, mean = env.step(acts)
        yield dict(acts=acts[:, 0], rewards=reward[:, 0].clone(), alives=alive[:, 0].clone(), ids=ids[:, 0],
                   prob=former.clone(), num=num[:, 0], active=active.clone()), \
            (obs[0][0].clone(), obs[0][1].clone()), rec
        former = mean[:, 0].clone()
        active = active & (done == 0)


@pytest.mark.parametrize("use_mean", [False, True])
def test_state_replay_samples_what_the_row_replay_samples(use_mean):
    from mfmarl_b200.algo.replay_device import DeviceMemoryGroup, DeviceStateMemoryGroup
    env = make_engine(3, 40, 64, rng="philox", seed=8)
    R = env.query("state_bytes")
    common = dict(use_mean=use_mean, device="cuda", stage_rows=3 * 64 * 12, seed=5)
    rows = DeviceMemoryGroup((13, 13, 7), (34,), 21, 2000, 256, 12, **common)
    states = DeviceStateMemoryGroup((13, 13, 7), (34,), 21, 2000, 256, 12, R, env.render_observations, **common)
    rng = np.random.RandomState(0)
    for rnd in range(4):                                # 4 rounds of <= 12 steps: the 2000-row ring wraps
        env.reset()
        left, right = generate_map_positions(40)
        env.add_agents(rnd % 2, left); env.add_agents(1 - rnd % 2, right)
        for kw, state, rec in _pushes(env, 12, rng):
            rows.push(state=state, **kw)
            states.push(records=rec, **kw)
        assert rows.tight() == states.tight()
        assert rows.nb_entries == states.nb_entries and rows.get_batch_num(False) == states.get_batch_num(False)
        assert torch.equal(rows.actions, states.actions) and torch.equal(rows.masks, states.masks)
        for _ in range(3):
            for a, b in zip(rows.sample(), states.sample()):
                assert a.dtype == b.dtype and torch.equal(a, b)
        idx = np.arange(rows.nb_entries - 5, rows.nb_entries)   # the ring's last rows and their wrapped successors
        for a, b in zip(rows.sample(idx=idx), states.sample(idx=idx)):
            assert torch.equal(a, b)
    assert states.head > 0                             # older rounds' records were freed
    assert states.tail - states.head <= 4 * 3 * 12


def test_state_replay_arena_full_error():
    from mfmarl_b200.algo.replay_device import DeviceStateMemoryGroup
    env = make_engine(2, 40, 64, rng="philox", seed=8)
    R = env.query("state_bytes")
    states = DeviceStateMemoryGroup((13, 13, 7), (34,), 21, 100000, 64, 12, R, env.render_observations,
                                    device="cuda", stage_rows=2 * 64 * 12, max_records=7)
    gen = _pushes(env, 12, np.random.RandomState(0))
    for _ in range(3):
        kw, _state, rec = next(gen)
        states.push(records=rec, **kw)
    kw, _state, rec = next(gen)
    with pytest.raises(RuntimeError, match=r"state-record arena full: 6 live records \+ 2 new need 8 records \(%d bytes\)" % (8 * R)):
        states.push(records=rec, **kw)


def _train(tmp_path, tag, extra):
    import importlib.util
    import random
    from conftest import PKG
    spec = importlib.util.spec_from_file_location("train_battle", os.path.join(PKG, "python", "train_battle.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    torch.manual_seed(0); random.seed(0); np.random.seed(0)
    data = str(tmp_path / tag)
    os.environ["MFMARL_SAVE_FINAL"] = "1"
    try:
        mod.main(["--algo", "mfq", "--save_every", "1000", "--data_dir", data] + extra)
    finally:
        del os.environ["MFMARL_SAVE_FINAL"]
    return torch.load(os.path.join(data, "final_rank0.pt"), map_location="cpu")


def test_train_battle_states_replay_trains_like_rows(tmp_path):
    deterministic = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    try:
        common = ["--envs", "8", "--max_steps", "50", "--n_round", "3"]
        a = _train(tmp_path, "rows", common + ["--replay", "rows"])
        b = _train(tmp_path, "states", common + ["--replay", "states"])
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = deterministic
    assert len(a) == len(b) > 0
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_train_battle_states_replay_records_every_env(tmp_path):
    _train(tmp_path, "big", ["--envs", "1024", "--max_steps", "20", "--n_round", "1", "--replay", "states"])
