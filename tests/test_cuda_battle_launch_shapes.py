"""Every launch class of the battle kernels k_step (K2) and k_obs (K1), each against the C oracle bit for bit.

The engine picks k_step's CTA width and k_obs's tile, grid and observation record from the env count and the capacity.
A test that lets it choose therefore runs only the shapes of its own env count: the small-E lockstep tests run 256-thread
k_step CTAs and 8-agent k_obs tiles, which production (hundreds of envs) never uses.  Each case below forces one class
(mfb_config step_threads / obs_tile_agents / obs_record, MFMARL_OBS_GRID) and asserts through mfb_query
("step_threads", "obs_tile", "obs_grid", "obs_record", "hbm_kernels") that it ran that class, so a change to the auto
rules cannot quietly move a case into another one.  Observations, features, rewards, alive flags, hp, positions and
mean actions are compared with the oracle bit for bit (mean actions to 1e-6); every k_obs case also checks that the bf16
rows are the fp32 rows rounded.

| kernel | class | what it reaches | case |
|---|---|---|---|
| k_step | 64 threads, 40x40, cap 64 | C3's production width at small E: loop scan (<= 4 warps), one pass | test_step_width[c3-64] |
| k_step | 64 / 96 / 128 threads, cap 512 | loop scan, several passes of list building and clear_dead compaction | test_step_width[c4-*] |
| k_step | 160 threads, cap 512 | shuffle scan (5 warps), several passes | test_step_width[c4-160] |
| k_step | 1024 threads, cap 36 | most threads idle, ragged capacity | test_step_width[ragged-1024] |
| k_step | 64 threads from HBM, 176x176 | k_step<true> (hbm_kernels & 1) with many passes | test_step_width[hbm-64] |
| k_step | 1..32, > 1024 | refused by mfb_create (one-warp CTAs leave group 1's mean action unset) | test_step_widths_k_step_cannot_serve_are_refused |
| k_obs | tile 8 .. 256 x record off / on | tiles per group, ragged last tile, tiles starting at or past num | test_obs_tile_and_record |
| k_obs | MFMARL_OBS_GRID = 1, 3 | one CTA takes many items: staging parity, minimap refresh and self markers carried over | test_obs_several_items_per_cta |
| k_obs | record forced on below cap 256 | k_obs<true> at 40x40 and an odd side | test_obs_record_forced[on-*] |
| k_obs | record forced off above cap 256 | kPre registers; above cap 512 the "rest from global" loop | test_obs_record_forced[off-*] |
| k_obs | group_mask 1 / 2 | one-group items; the other block and rows past num untouched | test_one_group_observe_*, test_one_group_bf16_* |
| k_obs | launches in flight on two streams | the ticket ring (kObsTicketRing = 8) wraps | test_observes_in_flight_on_two_streams |
| k_step | 16 move bands, 1001x1001 | band order and boundary buffer above W*H = 10^6 | test_sixteen_move_bands |
"""
import pytest

from lockstep import assert_same
from scenarios import block_positions, c4_positions, generate_map_positions
from test_cuda_battle_batched import lockstep_batched, make

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

STEP, OBS, RECORD, LOCAL = 1, 2, 4, 8


def density_cap(m):
    return max(64, int(m * m * 0.04))   # train_battle.py's capacity for --map_size m


def ragged_36():
    left, right = generate_map_positions(40)
    return left[:29], right[:33]


def pos_128x128():   # the 1024 v 1024 blocks of test_batched_largest_supported_shape_128x128_1024v1024
    return block_positions(48, 32, 16, 64, stride=1), block_positions(65, 32, 16, 64, stride=1)


def positions(kind):
    return {None: lambda: None, "c4": c4_positions, "ragged": ragged_36, "128": pos_128x128}[kind]()


def check_rows(env, oracles):
    """observe_groups in fp32 and bf16: the fp32 rows are the oracle's, the bf16 rows those rounded (zero channel 7),
    the features identical."""
    num = env.get_num()
    f32 = env.observe_groups()
    b16 = env.observe_groups(dtype=torch.bfloat16)
    for g in range(2):
        (v32, ft32), (v16, ft16) = f32[g], b16[g]
        for e, o in enumerate(oracles):
            n = int(num[e, g])
            ov, of = o.get_observation(g)
            assert_same("rows fp32 e%d g%d" % (e, g), ov, v32[e, :n].cpu().numpy(), -1)
            assert_same("features e%d g%d" % (e, g), of, ft32[e, :n].cpu().numpy(), -1)
            want = torch.zeros((n, 13, 13, 8), dtype=torch.bfloat16, device=v32.device)
            want[..., :7] = v32[e, :n].to(torch.bfloat16)
            assert torch.equal(v16[e, :n].view(torch.int16), want.view(torch.int16)), ("bf16 rows", e, g)
            assert torch.equal(ft16[e, :n], ft32[e, :n])


def run_rounds(env, oracles, rounds, steps, seed, check_obs_every=1, min_deaths=0):
    """lockstep_batched in rounds of `steps` (observations through mfb_observe), the fp32 / bf16 rows of
    mfb_observe_groups_* checked after each round."""
    deaths = 0
    for r in range(rounds):
        deaths += lockstep_batched(env, oracles, steps=steps, seed=seed + r, check_obs_every=check_obs_every)
        if (env.get_num() == 0).any():
            break
        check_rows(env, oracles)
    assert deaths >= min_deaths, deaths
    return deaths


# ---------------------------------------------------------------------------------------------------------------------
# k_step widths
# ---------------------------------------------------------------------------------------------------------------------
STEP_CASES = {
    # name: (map, cap, E, threads, positions, steps, check_obs_every, min_deaths, hbm mask)
    "c3-64": (40, 64, 4, 64, None, 80, 4, 10, 0),
    "c4-64": (80, 512, 2, 64, "c4", 40, 10, 5, 0),
    "c4-96": (80, 512, 2, 96, "c4", 40, 10, 5, 0),
    "c4-128": (80, 512, 2, 128, "c4", 40, 10, 5, 0),
    "c4-160": (80, 512, 2, 160, "c4", 40, 10, 5, 0),
    "ragged-1024": (40, 36, 2, 1024, "ragged", 100, 4, 1, 0),
    "hbm-64": (176, density_cap(176), 2, 64, None, 6, 3, 0, STEP),
}


@pytest.mark.parametrize("name", list(STEP_CASES))
def test_step_width(name):
    m, cap, E, threads, pos, steps, every, min_deaths, hbm = STEP_CASES[name]
    env, oracles = make(E, map_size=m, cap=cap, pos=positions(pos), step_threads=threads)
    assert env.query("step_threads") == threads
    assert env.query("hbm_kernels") & STEP == hbm
    lockstep_batched(env, oracles, steps=steps, seed=17, check_obs_every=every, min_deaths=min_deaths)


def test_step_widths_k_step_cannot_serve_are_refused():
    """1..32 would be a one-warp CTA: k_step's mean-action export zeroes and writes its [2][32] histogram with threads
    0..63, so group 1's bins would be uninitialised and its mean-action row never written.  Above 1024 no launch can
    succeed.  Both are refused by mfb_create, before anything is launched; 33 is rounded up to 64 and runs."""
    from mfmarl_b200 import BatchedGridWorld
    for bad in (1, 32, 1025, 4096):
        with pytest.raises(RuntimeError, match="step_threads = %d " % bad):
            BatchedGridWorld(2, map_size=40, capacity=64, step_threads=bad)
    for auto in (0, -5):
        env = BatchedGridWorld(2, map_size=40, capacity=64, step_threads=auto)
        assert env.query("step_threads") == 256          # auto: 2 envs cannot fill the GPU, so wide CTAs
    env, oracles = make(2, step_threads=33)
    assert env.query("step_threads") == 64
    lockstep_batched(env, oracles, steps=40, seed=3, check_obs_every=10, min_deaths=1)


# ---------------------------------------------------------------------------------------------------------------------
# k_obs tiles x record
# ---------------------------------------------------------------------------------------------------------------------
OBS_GEOMETRIES = {
    "40-cap64": (40, 64, 3, None, 8, 3),
    "40-cap36": (40, 36, 3, "ragged", 8, 3),
    "80-cap512": (80, 512, 2, "c4", 2, 6),
}
OBS_CASES = [(geo, tile, rec) for geo, tiles in (("40-cap64", (8, 16, 24, 64, 136, 256)),
                                                 ("40-cap36", (8, 16, 24)),
                                                 ("80-cap512", (24, 64, 136, 256)))
             for tile in tiles for rec in (0, 1)]


@pytest.mark.parametrize("geo, tile, record", OBS_CASES)
def test_obs_tile_and_record(geo, tile, record):
    m, cap, E, pos, rounds, steps = OBS_GEOMETRIES[geo]
    env, oracles = make(E, map_size=m, cap=cap, pos=positions(pos), obs_tile_agents=tile, obs_record=record)
    assert env.query("obs_record") == record and env.query("obs_tile") == 0
    num0 = env.get_num()
    if geo == "40-cap36":
        # several tiles per group, a ragged last tile (29 = 3 * 8 + 5), and for tiles 8 and 16 a tile that starts
        # at or past num from the first step on (32 >= 29): the skip path
        assert num0.min() == 29 and 29 % tile != 0
    run_rounds(env, oracles, rounds=rounds, steps=steps, seed=100 + tile, check_obs_every=1 if m == 40 else 3)
    assert env.query("obs_tile") == tile


# ---------------------------------------------------------------------------------------------------------------------
# several items per CTA
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("grid", [1, 3])
@pytest.mark.parametrize("record", [0, 1])
@pytest.mark.parametrize("tile", [24, 64])
def test_obs_several_items_per_cta(monkeypatch, grid, record, tile):
    """A persistent CTA carries its staging-buffer parity, the minimap refresh countdown and the self-marker positions
    from one item to the next.  Tile 24 is 3 chunks per item, so the parity flips across items; 3 envs x 2 groups x
    ceil(64 / tile) items over 1 or 3 CTAs, long enough for the self markers to move and for agents to die."""
    monkeypatch.setenv("MFMARL_OBS_GRID", str(grid))
    env, oracles = make(3, obs_tile_agents=tile, obs_record=record)
    run_rounds(env, oracles, rounds=10, steps=8, seed=300 + grid, min_deaths=5)
    assert env.query("obs_grid") == grid and env.query("obs_tile") == tile and env.query("obs_record") == record


# ---------------------------------------------------------------------------------------------------------------------
# record forced on / off
# ---------------------------------------------------------------------------------------------------------------------
RECORD_CASES = {
    # name: (map, cap, E, positions, record, rounds, steps, check_obs_every)
    "on-40-cap64": (40, 64, 3, None, 1, 4, 8, 1),
    "on-57-cap128": (57, 128, 3, None, 1, 4, 8, 1),
    "off-80-cap576": (80, 576, 2, "c4", 0, 5, 8, 4),
    "off-128-cap1024": (128, 1024, 2, "128", 0, 2, 6, 3),
}


@pytest.mark.parametrize("name", list(RECORD_CASES))
def test_obs_record_forced(name):
    """Auto keeps the record from cap 256 on, so without it k_obs never rebuilds its grid above cap 256: the kPre
    registers cover slots < 4 * 256, and above cap 512 the "rest from global" loop reads the others."""
    m, cap, E, pos, record, rounds, steps, every = RECORD_CASES[name]
    env, oracles = make(E, map_size=m, cap=cap, pos=positions(pos), obs_record=record)
    assert env.capacity == cap and env.query("obs_record") == record and env.query("hbm_kernels") == 0
    run_rounds(env, oracles, rounds=rounds, steps=steps, seed=cap, check_obs_every=every, min_deaths=1)


# ---------------------------------------------------------------------------------------------------------------------
# one group
# ---------------------------------------------------------------------------------------------------------------------
SENTINEL = 0xA5


def sentinel(shape, dtype):
    size = torch.empty((), dtype=dtype).element_size()
    t = torch.full(shape[:-1] + (shape[-1] * size,), SENTINEL, dtype=torch.uint8, device="cuda")
    return t.view(dtype)


def as_bytes(t):
    return t.contiguous().view(torch.uint8)


def one_group_env(geo, record):
    cap, pos = {"40-cap64": (64, None), "40-cap36": (36, ragged_36())}[geo]
    env, oracles = make(3, cap=cap, pos=pos, obs_record=record)
    lockstep_batched(env, oracles, steps=50, seed=5, check_obs_every=0, min_deaths=1)   # mid-fight, some agents gone
    return env, oracles


@pytest.mark.parametrize("geo", ["40-cap64", "40-cap36"])
@pytest.mark.parametrize("record", [0, 1])
def test_one_group_observe_leaves_the_rest_of_the_block_alone(geo, record):
    """mfb_observe with group_mask 1 or 2 into caller tensors full of a sentinel byte: the observed group's rows
    [:num] are the oracle's; the other group's block and the observed group's rows past num keep the sentinel, except
    that a ragged fp32 tail may spill up to 12 bytes into row num (the rows are 4732 B, 12 mod 16)."""
    env, oracles = one_group_env(geo, record)
    E, cap = env.n_envs, env.capacity
    num = env.get_num()
    row_bytes = 13 * 13 * 7 * 4
    for mask in (1, 2):
        g = mask >> 1
        view, feat = sentinel((E, 2, cap, 13, 13, 7), torch.float32), sentinel((E, 2, cap, 34), torch.float32)
        env.observe(group_mask=mask, out=(view, feat))
        torch.cuda.synchronize()
        vb = as_bytes(view).reshape(E, 2, cap, row_bytes).cpu().numpy()
        fb = as_bytes(feat).reshape(E, 2, cap, 34 * 4).cpu().numpy()
        for e, o in enumerate(oracles):
            n = int(num[e, g])
            ov, of = o.get_observation(g)
            assert_same("view mask %d e%d" % (mask, e), ov, view[e, g, :n].cpu().numpy(), -1)
            assert_same("feat mask %d e%d" % (mask, e), of, feat[e, g, :n].cpu().numpy(), -1)
            assert (vb[e, 1 - g] == SENTINEL).all() and (fb[e, 1 - g] == SENTINEL).all(), ("other group written", mask, e)
            assert (fb[e, g, n:] == SENTINEL).all(), ("features past num written", mask, e)
            if n < cap:
                assert (vb[e, g, n, 12:] == SENTINEL).all() and (vb[e, g, n + 1:] == SENTINEL).all(), ("rows past num", mask, e)
        assert env.query("obs_tile") > 0


@pytest.mark.parametrize("geo", ["40-cap64", "40-cap36"])
@pytest.mark.parametrize("record", [0, 1])
def test_one_group_bf16_observe_writes_rows_below_num_only(geo, record):
    """mfb_observe_groups_bf16 with one group into caller tensors: rows [:num] are the oracle's rows rounded to bf16
    with a zero eighth channel, features the oracle's; nothing past num changes (bf16 rows are whole 16-byte units)."""
    from mfmarl_b200.battle import _ptr, _stream
    env, oracles = one_group_env(geo, record)
    E, cap = env.n_envs, env.capacity
    num = env.get_num()
    for g in range(2):
        view, feat = sentinel((E, cap, 13, 13, 8), torch.bfloat16), sentinel((E, cap, 34), torch.float32)
        ptrs = [None] * 4
        ptrs[2 * g], ptrs[2 * g + 1] = _ptr(view), _ptr(feat)
        with torch.cuda.device(env.device):
            assert env.lib.mfb_observe_groups_bf16(env._h, *ptrs, _stream()) == 0, env.lib.mfb_last_error()
        torch.cuda.synchronize()
        vb, fb = as_bytes(view).reshape(E, cap, -1).cpu().numpy(), as_bytes(feat).reshape(E, cap, -1).cpu().numpy()
        for e, o in enumerate(oracles):
            n = int(num[e, g])
            ov, of = o.get_observation(g)
            want = torch.zeros((n, 13, 13, 8), dtype=torch.bfloat16)
            want[..., :7] = torch.from_numpy(ov).to(torch.bfloat16)
            assert torch.equal(view[e, :n].cpu().view(torch.int16), want.view(torch.int16)), ("bf16 rows", g, e)
            assert_same("feat g%d e%d" % (g, e), of, feat[e, :n].cpu().numpy(), -1)
            assert (vb[e, n:] == SENTINEL).all() and (fb[e, n:] == SENTINEL).all(), ("rows past num written", g, e)


# ---------------------------------------------------------------------------------------------------------------------
# observe launches in flight together
# ---------------------------------------------------------------------------------------------------------------------
def test_observes_in_flight_on_two_streams(monkeypatch):
    """Every observe launch takes its own ticket pair from a ring of 8, so launches of one engine may overlap on
    different streams.  Per step: one observe on the current stream, then one into each of two caller buffers on two
    side streams with no host synchronisation between them; 12 steps = 36 launches, so the ring wraps four times.
    MFMARL_OBS_GRID=16 keeps each launch small and long (128 items over 16 CTAs), and a spin on the current stream
    holds both side launches until both are enqueued, so that they can run at the same time.  Both side results equal the
    sequential one."""
    from mfmarl_b200 import BatchedGridWorld
    monkeypatch.setenv("MFMARL_OBS_GRID", "16")
    E, cap, steps = 64, 64, 12
    left, right = generate_map_positions(40)
    env = BatchedGridWorld(E, map_size=40, capacity=cap, rng="philox", seed=4)
    env.reset(); env.add_agents(0, left); env.add_agents(1, right)
    env.observe()
    main = torch.cuda.current_stream()
    side = [torch.cuda.Stream(), torch.cuda.Stream()]
    gen = torch.Generator(device="cuda"); gen.manual_seed(8)
    kept = []
    for s in range(steps):
        num = torch.from_numpy(env.get_num()).cuda()
        view, feat = env.observe()
        seq = (view.clone(), feat.clone())
        torch.cuda._sleep(200000)                 # holds both side launches until both are enqueued
        ready = main.record_event()
        outs = []
        for st in side:
            out = (torch.empty_like(view), torch.empty_like(feat))
            st.wait_event(ready)                  # (the buffers were allocated on the current stream)
            with torch.cuda.stream(st):
                env.observe(out=out)
            outs.append(out)
        for st in side:                           # k_step changes what k_obs reads: order it after both observes
            main.wait_stream(st)
        kept.append((num, seq, outs))
        actions = torch.randint(0, 21, (E, 2, cap), generator=gen, device="cuda", dtype=torch.int32)
        env.step(actions)
    torch.cuda.synchronize()
    assert env.query("obs_grid") == 16
    for s, (num, seq, outs) in enumerate(kept):
        num = num.cpu().numpy()
        for k, (view, feat) in enumerate(outs):
            for e in range(E):
                for g in range(2):
                    n = int(num[e, g])
                    assert torch.equal(view[e, g, :n], seq[0][e, g, :n]), ("view", s, k, e, g)
                    assert torch.equal(feat[e, g, :n], seq[1][e, g, :n]), ("feature", s, k, e, g)


# ---------------------------------------------------------------------------------------------------------------------
# 16 move bands
# ---------------------------------------------------------------------------------------------------------------------
def test_sixteen_move_bands():
    """Above W*H = 10^6 moves are filed into 16 x-bands instead of 8 (GridWorld.cc:79-88, :439).  At 1001 a band is
    ceil(1001 / 16) = 63 cells wide, with 8 it would be 126.  The armies are two touching strips stacked in y
    (x 437..500, y 496..497 and 498..499) that advance toward the centre (500, 500) into each other: their moves cross
    x = 441, a boundary of the 16 bands but not of the 8, and its boundary-buffer cells (x % 63 < 4 or > 59)."""
    m = 1001
    pos = block_positions(437, 496, 64, 2, stride=1), block_positions(437, 498, 64, 2, stride=1)
    env, oracles = make(2, map_size=m, cap=128, pos=pos)
    assert env.query("hbm_kernels") == STEP | OBS | RECORD | LOCAL
    lockstep_batched(env, oracles, steps=20, seed=16, check_obs_every=5, min_deaths=1)
