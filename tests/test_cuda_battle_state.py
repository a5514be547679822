"""Save, restore and fork the batched engine's environments (mfb_save_envs / mfb_load_envs): a restored env continues
bit for bit as its source would have -- outputs and state -- at every geometry, in both RNG modes, across auto-resets;
malformed records are refused before anything is written."""
import ctypes

import numpy as np
import pytest

from lockstep import assert_same
from scenarios import c4_positions, fight_actions, generate_map_positions

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

STATE_KEYS = ("num", "dead_ct", "pos", "hp", "id", "alive", "last_action", "step_ct", "rng", "side", "episode")


def density_cap(m):
    return max(64, int(m * m * 0.04))   # train_battle.py's capacity for --map_size m


def armies(m):
    return c4_positions() if m == 80 else generate_map_positions(m)


def per_env_armies(E, m, seed):
    """every env its own placement: which army takes the left block, and a few cells the engine skips (out of range)"""
    rng = np.random.RandomState(seed)
    left, right = armies(m)
    pos = [[], []]
    for _ in range(E):
        blocks = (right, left) if rng.randint(2) else (left, right)
        for g in range(2):
            p = blocks[g][:, :2].copy()
            p[rng.choice(len(p), size=rng.randint(1, 5), replace=False)] = (-2, 5)
            pos[g].append(p)
    return np.stack(pos[0]), np.stack(pos[1])


def engine(E, m, cap, placement=None, walls=None, **kw):
    from mfmarl_b200 import BatchedGridWorld
    env = BatchedGridWorld(E, map_size=m, capacity=cap, **kw)
    env.reset()
    if walls is not None:
        env.add_walls(walls)
    if placement is None:
        left, right = armies(m)
        env.add_agents(0, left); env.add_agents(1, right)
    elif placement != "none":
        env.add_agents_per_env(0, placement[0]); env.add_agents_per_env(1, placement[1])
    return env


def fight(env, rng):
    num, pos = env.get_num(), env.get("pos")
    acts = np.zeros((env.n_envs, 2, env.capacity), np.int32)
    for e in range(env.n_envs):
        for g in range(2):
            acts[e, g, :num[e, g]] = fight_actions(rng, pos[e, g, :num[e, g]], env.map_size)
    return torch.from_numpy(acts).cuda()


def moves_only(env, rng):
    return torch.from_numpy(rng.randint(0, 13, size=(env.n_envs, 2, env.capacity)).astype(np.int32)).cuda()


def same_rows(name, a, b, mask, step):
    if a.dtype == torch.bfloat16:
        a, b = a.view(torch.int16), b.view(torch.int16)
    elif a.dtype == torch.float32:
        a, b = a.view(torch.int32), b.view(torch.int32)
    a, b = a[mask], b[mask]
    if not torch.equal(a, b):
        bad = (a != b).nonzero()
        raise AssertionError("%s differs at step %d: %d mismatching values" % (name, step, len(bad)))


def compare_envs(A, ea, B, eb, step, outputs=True):
    """env ea of engine A against env eb of engine B: state (every mfb_get key but agent_steps) and, with outputs,
    the observations (fp32 both layouts, bf16) and the neighbourhood mean action of the listed rows"""
    ea, eb = np.atleast_1d(ea), np.atleast_1d(eb)
    for k in STATE_KEYS:
        assert_same(k, A.get(k)[ea], B.get(k)[eb], step)
    if not outputs:
        return
    cap = A.capacity
    num = torch.from_numpy(A.get_num()[ea]).cuda()
    ta, tb = torch.from_numpy(ea).cuda(), torch.from_numpy(eb).cuda()
    listed = torch.arange(cap, device="cuda")[None, None, :] < num[:, :, None]       # [n, 2, cap]
    (va, fa), (vb, fb) = A.observe(), B.observe()
    same_rows("view", va[ta], vb[tb], listed, step)
    same_rows("feature", fa[ta], fb[tb], listed, step)
    for dtype in (torch.float32, torch.bfloat16):
        ga, gb = A.observe_groups(dtype=dtype), B.observe_groups(dtype=dtype)
        for g in range(2):
            for j, what in enumerate(("view", "feature")):
                same_rows("groups %s %s g%d" % (dtype, what, g), ga[g][j][ta], gb[g][j][tb], listed[:, g], step)
    for g, (la, lb) in enumerate(zip(A.local_mean_action(), B.local_mean_action())):
        same_rows("local mean g%d" % g, la[ta], lb[tb], listed[:, g], step)


def stepped(env, acts):
    """step() -> (listed mask [E, 2, cap] before the step, reward, alive, done, mean action), copies"""
    num = torch.from_numpy(env.get_num()).cuda()
    listed = torch.arange(env.capacity, device="cuda")[None, None, :] < num[:, :, None]
    return (listed,) + tuple(t.clone() for t in env.step(acts))


def same_outputs(oa, ea, ob, eb, step):
    """step outputs of envs ea (of one engine) against envs eb (of another); returns the deaths among ea"""
    ta, tb = torch.from_numpy(np.atleast_1d(ea)).cuda(), torch.from_numpy(np.atleast_1d(eb)).cuda()
    listed = oa[0][ta]
    assert torch.equal(listed, ob[0][tb]), "num differs at step %d" % step
    same_rows("reward", oa[1][ta], ob[1][tb], listed, step)
    same_rows("alive", oa[2][ta], ob[2][tb], listed, step)
    assert torch.equal(oa[3][ta], ob[3][tb]), "done differs at step %d" % step
    assert torch.equal(oa[4][ta].view(torch.int32), ob[4][tb].view(torch.int32)), "mean action differs at step %d" % step
    return int((listed & (oa[2][ta] == 0)).sum())


def step_pair(A, ea, B, eb, acts_a, acts_b, step):
    return same_outputs(stepped(A, acts_a), ea, stepped(B, acts_b), eb, step)


# ---------------------------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize("rng_mode", ["minstd", "philox"])
@pytest.mark.parametrize("m, cap, E, K, max_steps", [(40, 64, 4, 40, 30), (80, 512, 2, 10, 7),
                                                      (256, density_cap(256), 2, 6, 4)])
def test_resume_continues_bit_for_bit(m, cap, E, K, max_steps, rng_mode):
    """A runs 2K steps; B runs K, saves every env, and a new engine C loads them and runs K more.  Episodes end on both
    sides of the save (auto_reset, random_sides, a per-env placement)."""
    cfg = dict(rng=rng_mode, seed=5, env_base=3, max_steps=max_steps, auto_reset=True, random_sides=True)
    place = per_env_armies(E, m, seed=m)
    A, B = engine(E, m, cap, place, **cfg), engine(E, m, cap, place, **cfg)
    if m == 256:
        assert A.query("hbm_kernels") & 1, "meant to run k_step from HBM"
    if m == 80:
        assert A.query("hbm_kernels") == 0
    rng = np.random.RandomState(m)
    every = list(range(E))
    deaths = 0
    for s in range(K):
        acts = fight(A, rng)
        deaths += step_pair(A, every, B, every, acts, acts, s)
    saved = B.save_envs()
    assert saved.shape == (E, 96 + 64 * A.capacity) and saved.device.type == "cuda"
    del B
    C = engine(E, m, cap, "none", **cfg)
    C.load_envs(saved)
    episodes = A.get("episode").copy()
    for s in range(K, 2 * K):
        compare_envs(A, every, C, every, s)
        acts = fight(A, rng)
        deaths += step_pair(A, every, C, every, acts, acts, s)
    compare_envs(A, every, C, every, 2 * K)
    assert (episodes > 0).all() and (A.get("episode") > episodes).all(), "episodes must end before and after the save"
    if m == 40:
        assert deaths > 0


# ---------------------------------------------------------------------------------------------------------------- 2
def test_fork_one_env_into_all_minstd():
    E, s = 5, 3
    S = engine(E, 40, 64, per_env_armies(E, 40, seed=1))
    rng = np.random.RandomState(2)
    for _ in range(8):
        S.step(fight(S, rng))
    F = engine(E, 40, 64, "none")
    F.load_envs(S.save_envs([s] * E))
    deaths = 0
    for t in range(25):
        compare_envs(S, [s] * E, F, list(range(E)), t, outputs=(t % 6 == 0))
        a = fight(S, rng)[s:s + 1].expand(E, -1, -1).contiguous()
        deaths += step_pair(S, [s], F, [0], a, a, t)
    compare_envs(S, [s] * E, F, list(range(E)), 25)
    assert deaths > 0


def test_fork_minstd_with_random_sides_is_exact_up_to_the_next_auto_reset():
    """The random_sides draw is Philox keyed by the global env id in every rng_mode: a MINSTD fork at another id equals
    its source up to the episode boundary, then draws its own side; where that side matches the source's, it stays
    equal (the attack shuffle's state travelled in the record)."""
    E, s, horizon, before = 8, 2, 12, 5
    cfg = dict(rng="minstd", seed=3, max_steps=horizon, auto_reset=True, random_sides=True)
    S = engine(E, 40, 64, **cfg)
    rng = np.random.RandomState(8)
    for _ in range(before):
        S.step(fight(S, rng))
    F = engine(E, 40, 64, "none", **cfg)
    F.load_envs(S.save_envs([s] * E))
    every = list(range(E))
    for t in range(horizon - before):           # the last of these steps ends the episode (the horizon)
        compare_envs(S, [s] * E, F, every, t, outputs=(t % 3 == 0))
        a = fight(S, rng)[s:s + 1].expand(E, -1, -1).contiguous()
        step_pair(S, [s] * E, F, every, a, a, t)
    assert (S.get("episode") == 1).all() and (F.get("episode") == 1).all()
    side_f, side_s = F.get("side"), S.get("side")
    assert np.array_equal(side_f, side_s), "each fork draws the side of its own global id"
    same = [d for d in every if side_f[d] == side_s[s]]
    assert 0 < len(same) < E, side_f
    pos_f, pos_s = F.get("pos"), S.get("pos")
    for d in every:
        if d not in same:
            assert not np.array_equal(pos_f[d], pos_s[s]), "env %d started its episode on the other side" % d
    for t in range(6):
        compare_envs(S, [s] * len(same), F, same, horizon + t, outputs=(t % 3 == 0))
        a = fight(S, rng)[s:s + 1].expand(E, -1, -1).contiguous()
        same_outputs(stepped(S, a), [s] * len(same), stepped(F, a), same, horizon + t)


# ---------------------------------------------------------------------------------------------------------------- 3
def test_fork_philox_reproduces_the_source_only_at_its_global_id():
    E, s = 4, 2
    cfg = dict(rng="philox", seed=9)
    S = engine(E, 40, 64, env_base=0, **cfg)
    rng = np.random.RandomState(3)
    for _ in range(30):
        S.step(fight(S, rng))
    rec = S.save_envs([s] * E)
    # env_base 1: index 1 has the source's global id 2
    T = engine(E, 40, 64, "none", env_base=1, **cfg)
    T.load_envs(rec)
    other = False
    for t in range(30):
        a = fight(S, rng)[s:s + 1].expand(E, -1, -1).contiguous()
        os_, ot = stepped(S, a), stepped(T, a)
        same_outputs(os_, [s], ot, [1], t)
        compare_envs(S, [s], T, [1], t, outputs=(t % 5 == 0))
        for d in (0, 2, 3):   # the kill reward goes to whoever lands the last hit: the order shows in the rewards
            other |= not torch.equal(os_[1][s].view(torch.int32), ot[1][d].view(torch.int32))
    assert other, "other global ids draw other attack orders"
    # moves only: no attack to shuffle, so every index equals the source (here: the record at its own global id)
    S2 = engine(E, 40, 64, "none", env_base=0, **cfg)
    S2.load_envs(rec[:1], envs=[s])
    T2 = engine(E, 40, 64, "none", env_base=1, **cfg)
    T2.load_envs(rec)
    for t in range(12):
        a = moves_only(S2, rng)[s:s + 1].expand(E, -1, -1).contiguous()
        step_pair(S2, [s] * E, T2, list(range(E)), a, a, t)
        compare_envs(S2, [s] * E, T2, list(range(E)), t, outputs=(t % 4 == 0))


# ---------------------------------------------------------------------------------------------------------------- 4
@pytest.mark.parametrize("rng_mode", ["minstd", "philox"])
def test_partial_reset_from_a_save_taken_after_placement(rng_mode):
    E, subset, rest = 4, [1, 3], [0, 2]
    cfg = dict(rng=rng_mode, seed=4)
    P, R = engine(E, 40, 64, **cfg), engine(E, 40, 64, **cfg)
    initial = P.save_envs()
    rng = np.random.RandomState(4)
    for s in range(50):
        a = fight(P, rng)
        P.step(a); R.step(a)
    P.load_envs(initial[subset], envs=subset)
    Q = engine(E, 40, 64, **cfg)
    for t in range(20):
        compare_envs(P, subset, Q, subset, t, outputs=(t % 5 == 0))
        compare_envs(P, rest, R, rest, t, outputs=(t % 5 == 0))
        a = fight(P, rng)
        op, oq, orr = stepped(P, a), stepped(Q, a), stepped(R, a)
        same_outputs(op, subset, oq, subset, t)
        same_outputs(op, rest, orr, rest, t)
    compare_envs(P, subset, Q, subset, 20)
    compare_envs(P, rest, R, rest, 20)


# ---------------------------------------------------------------------------------------------------------------- 5
def test_round_trip_decode_and_state_dict(tmp_path):
    from mfmarl_b200 import decode_env_state
    E = 3
    walls = np.array([[20, y, 0] for y in range(12, 28)], np.int32)
    cfg = dict(rng="philox", seed=8, max_steps=11, auto_reset=True, random_sides=True)
    A = engine(E, 40, 64, per_env_armies(E, 40, seed=5), walls=walls, **cfg)
    rng = np.random.RandomState(5)
    for _ in range(15):
        A.step(fight(A, rng))
    first = A.save_envs()
    A.load_envs(first)
    assert torch.equal(A.save_envs(), first)
    got = {k: A.get(k) for k in STATE_KEYS}
    for e in range(E):
        d = decode_env_state(first[e], A.capacity)
        assert d["magic"] == 0x5342464D and d["version"] == 1 and (d["W"], d["H"], d["cap"]) == (40, 40, 64)
        for k in STATE_KEYS:
            assert_same(k, np.asarray(d[k]), got[k][e], 0)
    path = str(tmp_path / "battle_state.pt")
    torch.save(A.state_dict(), path)
    B = engine(E, 40, 64, "none", **cfg)
    B.load_state_dict(torch.load(path))
    assert np.array_equal(B.get("walls"), A.get("walls")) and A.get("walls")[12:28, 20].all()
    every = list(range(E))
    for t in range(15):
        compare_envs(A, every, B, every, t, outputs=(t % 5 == 0))
        a = fight(A, rng)
        step_pair(A, every, B, every, a, a, t)


# ---------------------------------------------------------------------------------------------------------------- 6
def test_templates_travel_with_the_records():
    E = 4
    cfg = dict(seed=6, max_steps=8, auto_reset=True, random_sides=True)
    place = per_env_armies(E, 40, seed=6)
    P = engine(E, 40, 64, place, **cfg)
    rng = np.random.RandomState(6)
    for _ in range(3):
        P.step(fight(P, rng))
    S = engine(E, 40, 64, **cfg)                       # one shared template, unlike P's
    S.load_envs(P.save_envs())
    every = list(range(E))
    for t in range(12):                                # across the auto-reset at step 8
        compare_envs(P, every, S, every, t, outputs=(t % 4 == 0))
        a = fight(P, rng)
        step_pair(P, every, S, every, a, a, t)
    assert (S.get("episode") == 1).all()


# ---------------------------------------------------------------------------------------------------------------- 7
def _raw_load(env, n, envs, buf):
    idx = None if envs is None else np.ascontiguousarray(envs, dtype=np.int32)
    rc = env.lib.mfb_load_envs(env._h, n, None if idx is None else idx.ctypes.data,
                               None if buf is None else ctypes.c_void_p(buf.data_ptr()),
                               ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    return rc, env.lib.mfb_last_error().decode()


def test_refusals_leave_the_engine_unchanged():
    E = 4
    A = engine(E, 40, 64, seed=2)
    rng = np.random.RandomState(7)
    for _ in range(5):
        A.step(fight(A, rng))
    before = A.save_envs()
    cap = A.capacity

    def words(rec):
        return rec.view(torch.int32)

    def patched(k, fn):
        rec = before.clone()
        fn(words(rec[k]))
        return rec

    walled = engine(E, 40, 64, walls=np.array([[10, 10, 0]], np.int32), seed=2).save_envs()
    cases = [
        ("magic", patched(1, lambda w: w.__setitem__(0, 0x12345678)), "format version"),
        ("version", patched(0, lambda w: w.__setitem__(1, 2)), "format version"),
        ("width", patched(2, lambda w: w.__setitem__(2, 41)), "map size"),
        ("height", patched(2, lambda w: w.__setitem__(3, 39)), "map size"),
        ("capacity", patched(3, lambda w: w.__setitem__(4, 128)), "create the engine with the record's capacity"),
        ("wall hash", patched(0, lambda w: w.__setitem__(8, w[8] ^ 1)), "wall map"),
        ("other walls", walled, "wall map"),
        ("n_action", patched(3, lambda w: w.__setitem__(5, 20)), ": action count differs"),
        ("num > cap", patched(1, lambda w: w.__setitem__(11, cap + 1)), ": num outside"),
        ("dead_ct > cap", patched(1, lambda w: w.__setitem__(12, cap + 1)), ": dead_ct outside"),
        ("init_num < 0", patched(3, lambda w: w.__setitem__(20, -1)), ": template num outside"),
        ("pos off the map", patched(2, lambda w: w.__setitem__(24, 40)), ": agent position off the map"),
        ("pos y off the map", patched(2, lambda w: w.__setitem__(24 + 3, 45 << 16)), ": agent position off the map"),
        ("last action", patched(0, lambda w: w.__setitem__(24 + 3 * 2 * cap, 22 << 16)), ": last action"),
        ("template pos off the map", patched(1, lambda w: w.__setitem__(24 + 6 * 2 * cap + cap + 5, 40 << 16)),
         ": template position off the map (group 1, slot 5)"),
    ]
    for name, recs, reason in cases:
        rc, msg = _raw_load(A, E, None, recs)
        assert rc == -1 and msg.startswith("mfb_load_envs: record ") and reason in msg, (name, msg)
        assert torch.equal(A.save_envs(), before), name
    for name, n, envs, buf, reason in [("index out of range", 2, [0, E], before[:2], "out of range"),
                                       ("negative index", 1, [-1], before[:1], "out of range"),
                                       ("repeated target", 2, [1, 1], before[:2], "twice"),
                                       ("n = 0", 0, [], before, "outside"),
                                       ("n > n_envs", E + 1, None, before, "outside"),
                                       ("null buffer", E, None, None, "null")]:
        rc, msg = _raw_load(A, n, envs, buf)
        assert rc == -1 and msg.startswith("mfb_load_envs: ") and reason in msg, (name, msg)
        assert torch.equal(A.save_envs(), before), name
    with pytest.raises(ValueError, match="capacity"):
        A.load_envs(engine(E, 40, 128).save_envs())
    for other in (engine(E, 40, 128), engine(E, 48, 64), engine(E + 1, 40, 64)):
        with pytest.raises(ValueError, match="saved geometry"):
            A.load_state_dict(other.state_dict())
        assert torch.equal(A.save_envs(), before)
    A.load_envs(before.cpu())                                       # a valid CPU tensor is copied over and loaded
    assert torch.equal(A.save_envs(), before)
