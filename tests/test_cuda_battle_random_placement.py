"""Random placement on the GPU (mfb_add_agents_random): every env draws its own cells at commit and at every
auto-reset, exactly as the numpy restatement of tests/random_placement_ref.py says; at E = 1 in MINSTD mode it is the
single-env ABI's add_agents(method="random") cell for cell."""
import numpy as np
import pytest

from random_placement_ref import border_walls, episode_placement, whole_map
from scenarios import fight_actions

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def make(E, m, cap=64, rng="philox", seed=5, walls=(), fixed=((), ()), ops=(), **kw):
    from mfmarl_b200 import BatchedGridWorld
    env = BatchedGridWorld(E, map_size=m, capacity=cap, rng=rng, seed=seed, **kw)
    program(env, walls, fixed, ops)
    return env


def program(env, walls, fixed, ops):
    env.reset()
    if len(walls):
        env.add_walls(walls)
    for g in range(2):
        if len(fixed[g]):
            env.add_agents(g, fixed[g])
    for g, n, rect in ops:
        env.add_agents_random(g, n, rect)


def wall_map(m, walls):
    w = border_walls(m, m)
    for x, y in walls:
        w[y, x] = True
    return w


def fixed_with_ids(fixed):
    out, i = [[], []], 0
    for g in range(2):
        for x, y in fixed[g]:
            out[g].append((x, y, i)); i += 1
    return out


def snapshot(env):
    return {k: env.get(k) for k in ("num", "pos", "id", "placement_short", "rng", "episode", "side")}


def assert_env(st, e, expect, what=""):
    pos, ids, short, _ = expect
    for g in range(2):
        n = st["num"][e, g]
        assert n == len(pos[g]), "%s env %d group %d: %d agents, expected %d" % (what, e, g, n, len(pos[g]))
        assert [tuple(p) for p in st["pos"][e, g, :n].tolist()] == pos[g], "%s env %d group %d positions" % (what, e, g)
        assert st["id"][e, g, :n].tolist() == ids[g], "%s env %d group %d ids" % (what, e, g)
    assert st["placement_short"][e] == short, what


def resolved(m, ops):
    return [(g, n, whole_map(m, m) if rect is None else tuple(rect)) for g, n, rect in ops]


WALLS = [(x, 20) for x in range(5, 15)] + [(30, y) for y in range(8, 30)]
FIXED = ([(3, 3), (5, 3), (7, 3)], [(35, 35), (33, 35)])


# ---------------------------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize("seed", [0, 3, 123457])
@pytest.mark.parametrize("first", [0, 1])
def test_single_env_minstd_matches_the_single_env_abi(seed, first):
    from engines import CudaEngine
    m = 40
    ce = CudaEngine(m)
    ce.set_seed(seed); ce.reset()
    ce.add_walls(WALLS)
    for g in range(2):
        ce.add_agents(g, FIXED[g])
    ce.env.add_agents(ce.h[first], method="random", n=30)
    ce.env.add_agents(ce.h[1 - first], method="random", n=25)
    ops = [(first, 30, None), (1 - first, 25, None)]
    env = make(1, m, rng="minstd", seed=seed, walls=WALLS, fixed=FIXED, ops=ops)
    st = snapshot(env)
    expect = episode_placement("minstd", m, m, wall_map(m, WALLS), fixed_with_ids(FIXED), resolved(m, ops),
                               rs=seed % 2147483647 or 1)
    assert_env(st, 0, expect)
    assert st["rng"][0] == expect[3]
    for g in range(2):
        n = st["num"][0, g]
        assert np.array_equal(np.asarray(ce.get_pos(g))[:, :2], st["pos"][0, g, :n])
        assert np.array_equal(np.asarray(ce.get_agent_id(g)), st["id"][0, g, :n])
    rng = np.random.RandomState(seed)
    for step in range(50):
        num, pos = env.get_num(), env.get("pos")
        acts = np.zeros((1, 2, env.capacity), np.int32)
        for g in range(2):
            acts[0, g, :num[0, g]] = fight_actions(rng, pos[0, g, :num[0, g]], m)
            ce.set_action(g, acts[0, g, :num[0, g]])
        reward, alive, done, _ = env.step(torch.from_numpy(acts).cuda())
        ce.step()
        for g in range(2):
            n = num[0, g]
            assert np.array_equal(ce.get_reward(g).view(np.uint32), reward[0, g, :n].cpu().numpy().view(np.uint32)), step
            assert np.array_equal(ce.get_alive(g), alive[0, g, :n].cpu().numpy().astype(bool)), step
        ce.clear_dead()
        for g in range(2):
            assert np.array_equal(np.asarray(ce.get_pos(g))[:, :2], env.get("pos")[0, g, :env.get_num()[0, g]]), step


# ---------------------------------------------------------------------------------------------------------------- 2
def test_minstd_envs_draw_from_their_own_streams():
    m, E = 40, 8
    ops = [(0, 40, (1, 1, 19, 38)), (1, 40, (20, 1, 19, 38)), (0, 5, None)]
    env = make(E, m, rng="minstd", seed=1, fixed=FIXED, ops=ops)
    R = env.query("state_bytes")
    rec = env.save_envs()
    words = [int(s) for s in np.random.RandomState(7).randint(1, 2**31 - 1, size=E)]
    raw = rec.view(torch.int32).cpu().numpy().reshape(E, R // 4)
    raw[:, 14] = words
    env.load_envs(torch.from_numpy(raw).cuda().view(torch.uint8).reshape(E, R))
    program(env, (), FIXED, ops)                   # mfb_reset leaves the streams alone
    st = snapshot(env)
    for e in range(E):
        expect = episode_placement("minstd", m, m, border_walls(m, m), fixed_with_ids(FIXED), resolved(m, ops), rs=words[e])
        assert_env(st, e, expect)
        assert st["rng"][e] == expect[3]


# ---------------------------------------------------------------------------------------------------------------- 3
def test_philox_4096_envs():
    from scipy.stats import chisquare
    m, E, seed = 40, 4096, 11
    ops = [(0, 64, (1, 1, 16, 38)), (1, 64, (23, 1, 16, 38)), (1, 3, (17, 1, 6, 38))]
    env = make(E, m, rng="philox", seed=seed, walls=WALLS, fixed=FIXED, ops=ops)
    st = snapshot(env)
    walls = wall_map(m, WALLS)
    fixed = fixed_with_ids(FIXED)
    firsts = []
    for e in range(E):
        expect = episode_placement("philox", m, m, walls, fixed, resolved(m, ops), seed=seed, gid=e, generation=1)
        assert_env(st, e, expect)
        firsts.append(expect[0][0][len(fixed[0])])
    for e in range(0, E, 97):                  # cells distinct, inside their rectangles, off walls and fixed agents
        cells = set()
        for g in range(2):
            n = st["num"][e, g]
            for (x, y), i in zip(st["pos"][e, g, :n].tolist(), st["id"][e, g, :n].tolist()):
                assert (x, y) not in cells and not walls[y, x]
                cells.add((x, y))
                if i >= 5:                         # random agents: ids follow the call order of the ops
                    k = 0 if i < 5 + 64 else 1 if i < 5 + 128 else 2
                    x0, y0, w, h = ops[k][2]
                    assert x0 <= x < x0 + w and y0 <= y < y0 + h and g == ops[k][0]
    # the first random agent of env e is uniform over the blank cells of its rectangle
    blank = [(x, y) for x in range(1, 17) for y in range(1, 39) if not walls[y, x] and (x, y) not in FIXED[0]]
    counts = np.zeros(len(blank))
    index = {c: j for j, c in enumerate(blank)}
    for c in firsts:
        counts[index[c]] += 1
    assert chisquare(counts).pvalue > 1e-4


# ---------------------------------------------------------------------------------------------------------------- 4
@pytest.mark.parametrize("rng", ["minstd", "philox"])
def test_auto_reset_draws_every_episode(rng):
    m, E, K = 40, 6, 3
    ops = [(0, 20, (1, 1, 16, 38)), (1, 20, (23, 1, 16, 38))]
    env = make(E, m, rng=rng, seed=2, fixed=FIXED, ops=ops, auto_reset=True, max_steps=K)
    walls, fixed = border_walls(m, m), fixed_with_ids(FIXED)
    moves = np.random.RandomState(0)
    prev = snapshot(env)
    for step in range(1, 4 * K + 1):
        acts = torch.from_numpy(moves.randint(0, 13, size=(E, 2, env.capacity)).astype(np.int32)).cuda()
        env.step(acts)                             # moves only: the MINSTD stream is left to the placer
        st = snapshot(env)
        if step % K:
            continue
        for e in range(E):
            assert st["episode"][e] == step // K
            expect = episode_placement(rng, m, m, walls, fixed, resolved(m, ops), rs=prev["rng"][e], seed=2, gid=e,
                                       episode=step // K, generation=1)
            assert_env(st, e, expect, "episode %d" % (step // K))
        assert not np.array_equal(st["pos"], prev["pos"])
        prev = st


def test_philox_draws_do_not_depend_on_sharding_and_follow_the_generation():
    m, E = 40, 4
    ops = [(0, 30, (1, 1, 16, 38)), (1, 30, (23, 1, 16, 38))]
    kw = dict(rng="philox", seed=9, fixed=FIXED, ops=ops, auto_reset=True, max_steps=2)
    big, lo, hi = make(2 * E, m, **kw), make(E, m, env_base=0, **kw), make(E, m, env_base=E, **kw)
    moves = np.random.RandomState(1)
    for step in range(7):
        a = moves.randint(0, 13, size=(2 * E, 2, 64)).astype(np.int32)
        big.step(torch.from_numpy(a).cuda()); lo.step(torch.from_numpy(a[:E]).cuda()); hi.step(torch.from_numpy(a[E:]).cuda())
        for k in ("num", "pos", "id"):
            assert np.array_equal(big.get(k), np.concatenate([lo.get(k), hi.get(k)])), (k, step)
    first = snapshot(lo)["pos"]
    program(lo, (), FIXED, ops)                    # generation 2: new cells
    st = snapshot(lo)
    assert not np.array_equal(st["pos"], first)
    for e in range(E):
        expect = episode_placement("philox", m, m, border_walls(m, m), fixed_with_ids(FIXED), resolved(m, ops), seed=9,
                                   gid=e, episode=0, generation=2)
        assert_env(st, e, expect)


# ---------------------------------------------------------------------------------------------------------------- 5
def test_random_sides_swap_groups_and_ids():
    m, E = 40, 16
    ops = [(0, 20, (1, 1, 16, 38)), (1, 10, (23, 1, 16, 38))]
    env = make(E, m, rng="philox", seed=4, fixed=FIXED, ops=ops, auto_reset=True, max_steps=1, random_sides=True)
    moves = np.random.RandomState(2)
    sides = set()
    for ep in range(1, 4):
        env.step(torch.from_numpy(moves.randint(0, 13, size=(E, 2, 64)).astype(np.int32)).cuda())
        st = snapshot(env)
        for e in range(E):
            expect = episode_placement("philox", m, m, border_walls(m, m), fixed_with_ids(FIXED), resolved(m, ops),
                                       side=int(st["side"][e]), seed=4, gid=e, episode=ep, generation=1)
            assert_env(st, e, expect)
            sides.add(int(st["side"][e]))
    assert sides == {0, 1}


# ---------------------------------------------------------------------------------------------------------------- 6
@pytest.mark.parametrize("rng", ["minstd", "philox"])
def test_loaded_env_continues_through_auto_resets(rng):
    m, E = 40, 4
    ops = [(0, 24, (1, 1, 16, 38)), (1, 24, (23, 1, 16, 38))]
    kw = dict(rng=rng, seed=6, fixed=FIXED, ops=ops, auto_reset=True, max_steps=5)
    A, B = make(E, m, **kw), make(E, m, **kw)
    r = np.random.RandomState(3)

    def acts(env):
        num, pos = env.get_num(), env.get("pos")
        a = np.zeros((E, 2, 64), np.int32)
        for e in range(E):
            for g in range(2):
                a[e, g, :num[e, g]] = fight_actions(r, pos[e, g, :num[e, g]], m)
        return torch.from_numpy(a).cuda()

    for _ in range(3):
        A.step(acts(A))
    B.load_envs(A.save_envs())
    for step in range(12):                      # the episodes end at steps 5 and 10: two auto-resets
        a = acts(A)
        A.step(a); B.step(a)
        sa, sb = snapshot(A), snapshot(B)
        for k in ("num", "pos", "id", "rng", "episode", "placement_short"):
            assert np.array_equal(sa[k], sb[k]), (k, step)
    assert (sa["episode"] >= 2).all()


# ---------------------------------------------------------------------------------------------------------------- 7
def test_hbm_geometry_places_and_observes_like_the_oracle():
    from engines import OracleEngine
    m, E = 180, 2
    cap = max(64, int(m * m * 0.04))
    ops = [(0, 400, (1, 1, m // 2 - 4, m - 2)), (1, 400, (m // 2 + 3, 1, m // 2 - 4, m - 2))]
    env = make(E, m, cap=cap, rng="philox", seed=8, ops=ops, auto_reset=True, max_steps=1)
    assert env.query("hbm_kernels") & 1
    walls = border_walls(m, m)
    for ep in range(2):
        st = snapshot(env)
        view, feat = env.observe()
        view, feat = view.cpu().numpy(), feat.cpu().numpy()
        for e in range(E):
            expect = episode_placement("philox", m, m, walls, [[], []], resolved(m, ops), seed=8, gid=e, episode=ep,
                                       generation=1)
            assert_env(st, e, expect, "episode %d" % ep)
            o = OracleEngine(m); o.reset()
            for g in range(2):
                o.add_agents(g, expect[0][g])
            for g in range(2):
                n = st["num"][e, g]
                v, f = o.get_observation(g)
                assert np.array_equal(v.view(np.uint32), view[e, g, :n].view(np.uint32)), (ep, e, g)
                assert np.array_equal(f.view(np.uint32), feat[e, g, :n].view(np.uint32)), (ep, e, g)
        env.step(torch.zeros((E, 2, env.capacity), dtype=torch.int32, device="cuda") + 6)   # stand still, then re-place


# ---------------------------------------------------------------------------------------------------------------- 8
def test_shortfall_is_counted():
    from random_placement_ref import Draws, place_sequential
    m = 8
    inner = [(x, y) for x in range(1, m - 1) for y in range(1, m - 1) if (x, y) != (3, 4)]
    walls = wall_map(m, inner)
    outcome = {}
    for s in range(1, 200):
        d = Draws("minstd", m, m, rs=s)
        _, short = place_sequential(d, walls.copy(), [(0, 1, whole_map(m, m))])
        outcome.setdefault(short, (s, d.rs))
        if len(outcome) == 2:
            break
    for short, (s, rs) in outcome.items():
        env = make(1, m, cap=4, rng="minstd", seed=s, walls=inner, ops=[(0, 1, None)])
        st = snapshot(env)
        assert st["placement_short"][0] == short and st["num"][0, 0] == 1 - short and st["rng"][0] == rs
        if not short:
            assert st["pos"][0, 0, 0].tolist() == [3, 4]


# ---------------------------------------------------------------------------------------------------------------- 9
def test_refusals_change_nothing():
    m = 40
    env = make(2, m, rng="philox", fixed=FIXED, ops=[(0, 10, (1, 1, 10, 10))])
    before = snapshot(env)
    cases = [(lambda: env.add_agents_random(2, 5), "group = 2"),
             (lambda: env.add_agents_random(0, -1), "n = -1"),
             (lambda: env.add_agents_random(0, 5, (35, 1, 10, 5)), "leaves the 40x40 map"),
             (lambda: env.add_agents_random(0, 5, (0, 0, 1, 5)), "no interior cell"),
             (lambda: env.add_agents_random(0, 5, (5, 5, 0, 3)), "w and h must both be positive"),
             (lambda: env.add_agents_random(1, 95, (1, 1, 10, 10)), "n = 95 does not fit"),
             (lambda: env.add_agents(0, [[20, 20]]), "add_agents after add_agents_random"),
             (lambda: env.add_walls([[20, 20]]), "add_walls after add_agents_random")]
    for call, msg in cases:
        with pytest.raises(RuntimeError, match=msg):
            call()
        after = snapshot(env)
        for k in ("num", "pos", "id"):
            assert np.array_equal(before[k], after[k]), (msg, k)


# ---------------------------------------------------------------------------------------------------------------- 10
def test_play_batched_and_train_battle_with_random_placement(tmp_path):
    from mfmarl_b200 import BatchedGridWorld
    from mfmarl_b200.algo import spawn_ai
    from mfmarl_b200.senario_battle import play_batched

    class Spaces:
        def get_view_space(self, h): return (13, 13, 7)
        def get_feature_space(self, h): return (34,)
        def get_action_space(self, h): return (21,)

    env = BatchedGridWorld(6, map_size=40, capacity=64, rng="philox", seed=3)
    models = [spawn_ai("mfq", Spaces(), g, "mfq-%d" % g, 10, device="cuda") for g in range(2)]
    max_nums, nums, _, _ = play_batched(env, 0, 10, models, eps=1.0, train=True, left_group=1, placement="random")
    assert (max_nums == 64).all() and (env.get("placement_short") == 0).all()
    num, ids = env.get("num"), env.get("id")
    listed = np.arange(64)[None, :] < num[:, :, None]
    assert (ids[:, 1][listed[:, 1]] < 64).all() and (ids[:, 0][listed[:, 0]] >= 64).all()   # left_group 1: the low ids
    from test_cuda_battle_render import _train
    _train(tmp_path, "random", ["--envs", "64", "--placement", "random", "--n_round", "2", "--max_steps", "20"])
