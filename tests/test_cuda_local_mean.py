"""GPU: the neighbourhood mean action (mfb_local_mean_action, kernel K7) bit for bit against the numpy reference of
tests/local_mean_ref.py, on states driven in lockstep with the C oracle, and its use by play_batched / the learners."""
import importlib.util
import os

import numpy as np
import pytest

from engines import OracleEngine
from local_mean_ref import local_mean_action
from lockstep import assert_same
from scenarios import c4_positions, fight_actions, generate_map_positions

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

N_ACTION = 21
RADII = (1, 1.5, 6)


def make(E, map_size=40, cap=64, pos=None, **kw):
    from mfmarl_b200 import BatchedGridWorld
    env = BatchedGridWorld(E, map_size=map_size, capacity=cap, **kw)
    env.reset()
    left, right = pos if pos is not None else generate_map_positions(map_size)
    env.add_agents(0, left)
    env.add_agents(1, right)
    oracles = []
    for _ in range(E):
        o = OracleEngine(map_size)
        o.reset()
        o.add_agents(0, left)
        o.add_agents(1, right)
        oracles.append(o)
    return env, oracles


def check_rows(name, out, e, g, ref, n, s):
    assert_same("%s[e%d g%d]" % (name, e, g), ref, out[g][e, :n], s)
    assert not out[g][e, n:].any(), "%s[e%d g%d]: rows >= num are not zero at step %d" % (name, e, g, s)


def check_against_oracles(env, oracles, last, s):
    num = env.get_num()
    for r in RADII:
        out = [t.cpu().numpy() for t in env.local_mean_action(radius=r)]
        for e, o in enumerate(oracles):
            for g in range(2):
                n = num[e, g]
                assert n == o.get_num(g)
                ref = local_mean_action(o.get_pos(g), last[e][g], np.ones(n, bool), r, N_ACTION)
                check_rows("local r=%g" % r, out, e, g, ref, n, s)


def lockstep_local(env, oracles, steps, seed, min_deaths):
    """Step E envs with the fight stream, each against its own oracle; after the placement and after every
    step + clear_dead the local mean action of every radius must equal the reference built from the oracle's
    positions and the survivors' actions (the stable compaction keeps their order)."""
    E, cap = env.n_envs, env.capacity
    rngs = [np.random.RandomState(seed * 1000 + e) for e in range(E)]
    last = [[np.full(o.get_num(g), N_ACTION, np.int64) for g in range(2)] for o in oracles]
    deaths = 0
    check_against_oracles(env, oracles, last, -1)
    for s in range(steps):
        num = env.get_num()
        if num.min() == 0:
            break
        pos = env.get("pos")
        actions = np.zeros((E, 2, cap), np.int32)
        for e, o in enumerate(oracles):
            for g in range(2):
                n = num[e, g]
                assert_same("pos[e%d g%d]" % (e, g), o.get_pos(g), pos[e, g, :n], s)
                actions[e, g, :n] = fight_actions(rngs[e], pos[e, g, :n], env.map_size)
                o.set_action(g, actions[e, g, :n])
        _, alive, done, _ = env.step(torch.from_numpy(actions).cuda())
        alive, done = alive.cpu().numpy(), done.cpu().numpy()
        for e, o in enumerate(oracles):
            assert o.step() == bool(done[e])
            for g in range(2):
                n = num[e, g]
                al = o.get_alive(g)
                assert_same("alive[e%d g%d]" % (e, g), al, alive[e, g, :n].astype(bool), s)
                deaths += int((~al).sum())
                last[e][g] = actions[e, g, :n][al].astype(np.int64)
            o.clear_dead()
        check_against_oracles(env, oracles, last, s)
        if done.any():
            break
    assert deaths >= min_deaths, deaths
    return deaths


def test_local_mean_action_lockstep_40x40():
    env, oracles = make(4)
    lockstep_local(env, oracles, steps=150, seed=11, min_deaths=50)


def test_local_mean_action_lockstep_80x80_512v512_with_the_observation_record():
    env, oracles = make(2, map_size=80, cap=512, pos=c4_positions())
    assert env.capacity == 512
    lockstep_local(env, oracles, steps=40, seed=12, min_deaths=20)


def reference_from_state(env, r):
    """[E][2] reference rows from the engine's own state (mfb_get)"""
    num, pos, act, alive = env.get_num(), env.get("pos"), env.get("last_action"), env.get("alive")
    return [[local_mean_action(pos[e, g, :num[e, g]], act[e, g, :num[e, g]], alive[e, g, :num[e, g]].astype(bool), r,
                               N_ACTION) for g in range(2)] for e in range(env.n_envs)], num


def test_auto_reset_gives_zero_rows_and_leaves_the_other_envs_alone():
    """Env 0 holds one agent per group side by side and the first attacks the second every step, so it ends and
    auto-resets (random_sides: on either side) every few steps; envs 1 and 2 fight on with full armies."""
    from mfmarl_b200 import BatchedGridWorld
    E, cap = 3, 64
    env = BatchedGridWorld(E, map_size=40, capacity=cap, rng="philox", seed=5, auto_reset=True, random_sides=True)
    env.reset()
    left, right = generate_map_positions(40)
    for g, block, mine in ((0, left, [10, 10]), (1, right, [11, 10])):
        pos = np.full((E, len(block), 2), -1, np.int32)
        pos[0, 0] = mine
        pos[1:] = np.asarray(block, np.int32)[:, :2]
        env.add_agents_per_env(g, pos)
    table, base = OracleEngine(40).action_table()
    attack = {(int(dx), int(dy)): a for a, (dx, dy) in enumerate(table) if a >= base}
    rng = np.random.RandomState(3)
    resets = 0
    for s in range(40):
        num, pos = env.get_num(), env.get("pos")
        acts = np.zeros((E, 2, cap), np.int32)
        p0, p1 = pos[0, 0, 0], pos[0, 1, 0]
        acts[0, 0, 0] = attack[(int(p1[0] - p0[0]), int(p1[1] - p0[1]))]
        acts[0, 1, 0] = 6                                           # stays (move (0, 0))
        for e in (1, 2):
            for g in range(2):
                acts[e, g, :num[e, g]] = fight_actions(rng, pos[e, g, :num[e, g]], 40)
        env.step(torch.from_numpy(acts).cuda())
        step_ct = env.get("step_ct")
        for r in (1.5, 6):
            out = [t.cpu().numpy() for t in env.local_mean_action(radius=r)]
            ref, num = reference_from_state(env, r)
            for e in range(E):
                for g in range(2):
                    if step_ct[e] == 0:
                        assert not out[g][e].any(), "env %d just reset but has a nonzero row" % e
                    check_rows("local r=%g" % r, out, e, g, ref[e][g], num[e, g], s)
        resets += int(step_ct[0] == 0)
        assert step_ct[1] == step_ct[2] == s + 1
    assert resets >= 3, resets
    assert env.get("episode")[0] == resets


def test_null_group_repeat_calls_and_invalid_radii():
    env, _ = make(3)
    rng = np.random.RandomState(0)
    for _ in range(3):
        num, pos = env.get_num(), env.get("pos")
        acts = np.zeros((3, 2, 64), np.int32)
        for e in range(3):
            for g in range(2):
                acts[e, g, :num[e, g]] = fight_actions(rng, pos[e, g, :num[e, g]], 40)
        env.step(torch.from_numpy(acts).cuda())
    a0, a1 = [t.clone() for t in env.local_mean_action()]
    b0, b1 = env.local_mean_action(radius=6)
    assert torch.equal(a0, b0) and torch.equal(a1, b1) and a0.any() and a1.any()
    g1 = b1
    g1.fill_(-7.0)
    only0 = env.local_mean_action(groups=(0,), radius=1.5)
    assert only0[1] is None and only0[0].data_ptr() == b0.data_ptr()
    assert (g1 == -7.0).all(), "the group that was not asked for was written"
    g0 = only0[0].clone()
    only1 = env.local_mean_action(groups=(1,), radius=1.5)
    assert only1[0] is None and torch.equal(only0[0], g0)
    for bad in (0, -1, 6.5, float("nan"), float("inf")):
        with pytest.raises(RuntimeError, match="radius"):
            env.local_mean_action(radius=bad)
    assert torch.equal(only0[0], g0)


class Spaces:
    def get_view_space(self, h): return (13, 13, 7)
    def get_feature_space(self, h): return (34,)
    def get_action_space(self, h): return (21,)


def test_play_batched_local_mean_field_feeds_act_and_the_replay():
    from mfmarl_b200 import BatchedGridWorld
    from mfmarl_b200.algo import spawn_ai
    from mfmarl_b200.senario_battle import play_batched
    torch.manual_seed(0)
    E, cap, steps = 4, 64, 25
    env = BatchedGridWorld(E, map_size=40, capacity=cap, rng="philox", seed=1)
    seen, checked = {0: [], 1: []}, [0]

    def recording(g, act):
        def wrapped(**kw):
            prob = kw["prob"]
            assert tuple(prob.shape) == (E * cap, N_ACTION)
            seen[g].append(prob.clone())
            got = prob.view(E, cap, N_ACTION).cpu().numpy()
            ref, num = reference_from_state(env, 6.0)
            for e in range(E):
                check_rows("act prob", {g: got}, e, g, ref[e][g], num[e, g], len(seen[g]))
            checked[0] += 1
            return act(**kw)
        return wrapped

    class RandomPolicy:
        gen = torch.Generator(device="cuda").manual_seed(2)

        def act(self, state, prob, eps):
            return torch.randint(0, N_ACTION, (state[0].shape[0],), generator=self.gen, device="cuda", dtype=torch.int32)

    me = spawn_ai("mfq", Spaces(), 0, "mfq-me", steps, device="cuda")
    opp = RandomPolicy()
    me.act, opp.act = recording(0, me.act), recording(1, opp.act)
    flushed, inner_flush = [], me.flush_buffer_batched

    def flush(**kw):
        flushed.append({k: kw[k].clone() for k in ("prob", "num", "active")})
        inner_flush(**kw)
    me.flush_buffer_batched = flush
    me.train = lambda *a, **k: None            # keep the staged rows for the check below
    play_batched(env, 0, steps, [me, opp], eps=1.0, train=True, left_group=0, mean_field="local")
    assert checked[0] == 2 * len(flushed) and len(flushed) == steps
    assert any(bool(p.any()) for p in seen[0][1:]) and not seen[0][0].any()
    stage = me.device_replay._stage
    n_rec = me.device_replay.n_rec_envs(E, cap)
    want = []
    for t, f in enumerate(flushed):
        assert torch.equal(f["prob"], seen[0][t].view(E, cap, N_ACTION))
        for e in range(n_rec):
            if bool(f["active"][e]):
                want.append(f["prob"][e, :int(f["num"][e])])
    want = torch.cat(want)
    assert int(stage.cursor) == want.shape[0]
    assert torch.equal(stage.prob[:want.shape[0]], want)


@pytest.mark.parametrize("algo", ["mfq", "mfac"])
def test_learners_train_a_round_with_the_local_mean_field(algo):
    from mfmarl_b200 import BatchedGridWorld
    from mfmarl_b200.algo import spawn_ai
    from mfmarl_b200.senario_battle import play_batched
    torch.manual_seed(0)
    E, steps = 6, 10
    env = BatchedGridWorld(E, map_size=40, capacity=64, rng="philox", seed=3)
    models = [spawn_ai(algo, Spaces(), 0, algo + "-me", steps, device="cuda"),
              spawn_ai(algo, Spaces(), 1, algo + "-opponent", steps, device="cuda")]
    before = [p.detach().clone() for p in models[0].vars]
    max_nums, nums, mean_r, total_r = play_batched(env, 0, steps, models, eps=1.0, train=True, left_group=0,
                                                   mean_field="local", mf_radius=3)
    assert (max_nums == 64).all() and np.isfinite(mean_r).all() and np.isfinite(total_r).all()
    assert any(not torch.equal(a, b) for a, b in zip(before, models[0].vars))
    for p in models[0].vars:
        assert torch.isfinite(p).all()


def test_train_battle_local_mean_field_end_to_end(tmp_path):
    from conftest import PKG
    spec = importlib.util.spec_from_file_location("train_battle", os.path.join(PKG, "python", "train_battle.py"))
    train = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(train)
    runner = train.main(["--algo", "mfq", "--envs", "8", "--n_round", "1", "--max_steps", "20", "--mean_field", "local",
                         "--data_dir", str(tmp_path / "data")])
    assert runner is not None
