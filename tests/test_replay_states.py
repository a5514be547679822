"""CPU: the record-backed replay (DeviceStateMemoryGroup) with a fake renderer in place of k_render_obs -- it samples
what the row replay samples through ring wrap-around, frees a round's records once the ring has overwritten its rows,
moves and grows its arena without losing a live record, and refuses to outgrow max_records; and the command-line
refusals of --replay states."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

OBS, FEAT, ACT_N, R = (2,), (3,), 4, 32


def fake_renderer(records, rows):
    """view = (record stamp, slot), feature = (group, stamp + slot, record index): what the row replay stores below"""
    stamp = records[:, :4].contiguous().view(torch.int32)[:, 0].to(torch.float32)
    r, g, s = rows[:, 0].long(), rows[:, 1].to(torch.float32), rows[:, 2].to(torch.float32)
    st = stamp[r]
    return torch.stack([st, s], 1), torch.stack([g, st + s, st * 0 + 7], 1)


def step_inputs(rng, E, cap, stamp):
    records = torch.zeros((E, R), dtype=torch.uint8)
    stamps = torch.arange(stamp, stamp + E, dtype=torch.int32)
    records[:, :4] = stamps[:, None].view(torch.uint8).reshape(E, 4)
    slot = torch.arange(cap, dtype=torch.float32)
    st = stamps.to(torch.float32)[:, None].expand(E, cap)
    view = torch.stack([st, slot.expand(E, cap)], 2)
    feat = torch.stack([torch.zeros(E, cap), st + slot, torch.full((E, cap), 7.0)], 2)
    num = torch.from_numpy(rng.randint(0, cap + 1, size=E).astype(np.int32))
    kw = dict(acts=torch.from_numpy(rng.randint(0, ACT_N, size=(E, cap)).astype(np.int32)),
              rewards=torch.from_numpy(rng.rand(E, cap).astype(np.float32)),
              alives=torch.from_numpy((rng.rand(E, cap) > 0.1).astype(np.uint8)),
              ids=torch.arange(cap, dtype=torch.int32).expand(E, cap).contiguous(),
              prob=torch.from_numpy(rng.rand(E, ACT_N).astype(np.float32)), num=num,
              active=torch.from_numpy(rng.rand(E) > 0.2))
    return kw, (view, feat), records


def make_pair(max_len, E, cap, sub_len, **kw):
    from mfmarl_b200.algo.replay_device import DeviceMemoryGroup, DeviceStateMemoryGroup
    common = dict(use_mean=True, device="cpu", stage_rows=E * cap * sub_len, seed=3)
    rows = DeviceMemoryGroup(OBS, FEAT, ACT_N, max_len, 16, sub_len, **common)
    states = DeviceStateMemoryGroup(OBS, FEAT, ACT_N, max_len, 16, sub_len, R, fake_renderer, **common, **kw)
    return rows, states


def test_state_replay_matches_the_row_replay_and_frees_rounds():
    E, cap, sub_len, max_len = 3, 5, 4, 40
    rows, states = make_pair(max_len, E, cap, sub_len)
    rng, stamp, ends = np.random.RandomState(0), 1, []
    for rnd in range(12):
        for t in range(sub_len):
            kw, state, rec = step_inputs(rng, E, cap, stamp)
            stamp += E
            rows.push(state=state, **kw)
            states.push(records=rec, **kw)
        n = rows.tight()
        assert states.tight() == n
        ends.append(n)
        assert rows.nb_entries == states.nb_entries
        for _ in range(2):
            for a, b in zip(rows.sample(), states.sample()):
                assert torch.equal(a, b)
        # the live records: at most the rounds whose rows are not all overwritten yet (the ring holds the last max_len)
        live_rounds, held = 0, 0
        for m in reversed(ends):
            if held >= max_len:
                break
            live_rounds += 1
            held += m
        assert states.tail - states.head <= live_rounds * E * sub_len
        refs = states.obs0[:states.nb_entries, 0]
        assert bool((refs >= states.head).all()) and bool((refs < states.tail).all())
    assert states.arena.shape[0] < 12 * E * sub_len    # the arena was reused, not grown round after round


def test_state_replay_arena_moves_and_grows_by_round():
    E, cap, sub_len = 2, 4, 3
    rows, states = make_pair(10 ** 6, E, cap, sub_len)          # a ring that never wraps: nothing is freed
    rng, stamp = np.random.RandomState(1), 1
    sizes = []
    for rnd in range(5):
        for t in range(sub_len):
            kw, state, rec = step_inputs(rng, E, cap, stamp)
            stamp += E
            rows.push(state=state, **kw)
            slot = states.record_slice(E, cap)                   # the arena slice the next push uses
            slot.copy_(rec)
            states.push(records=slot, **kw)
        rows.tight(); states.tight()
        sizes.append(states.arena.shape[0])
        assert states.head == 0 and states.tail == (rnd + 1) * E * sub_len
    assert sizes[0] == E * sub_len and sizes[-1] >= 5 * E * sub_len and sizes == sorted(sizes)
    for a, b in zip(rows.sample(idx=np.arange(rows.nb_entries)), states.sample(idx=np.arange(states.nb_entries))):
        assert torch.equal(a, b)


def test_state_replay_compacts_the_live_records_to_the_front():
    E, cap, sub_len, max_len = 2, 4, 3, 12
    rows, states = make_pair(max_len, E, cap, sub_len, max_records=3 * E * sub_len)
    rng, stamp = np.random.RandomState(2), 1
    moved = False
    for rnd in range(10):
        for t in range(sub_len):
            kw, state, rec = step_inputs(rng, E, cap, stamp)
            kw["num"] = torch.full((E,), cap, dtype=torch.int32)   # full rounds: each round overwrites the last
            kw["active"] = torch.ones((E,), dtype=torch.bool)
            stamp += E
            head = states.head
            rows.push(state=state, **kw)
            states.push(records=rec, **kw)
            moved |= states.head < head
        rows.tight(); states.tight()
        assert states.arena.shape[0] <= 3 * E * sub_len
        for a, b in zip(rows.sample(), states.sample()):
            assert torch.equal(a, b)
    assert moved


def test_state_replay_refuses_to_outgrow_max_records():
    E, cap, sub_len = 2, 4, 3
    _rows, states = make_pair(10 ** 6, E, cap, sub_len, max_records=5)
    rng = np.random.RandomState(3)
    for stamp in (1, 3):
        kw, _state, rec = step_inputs(rng, E, cap, stamp)
        states.push(records=rec, **kw)
    kw, _state, rec = step_inputs(rng, E, cap, 5)
    with pytest.raises(RuntimeError, match=r"4 live records \+ 2 new need 6 records \(%d bytes\); max_records is 5" % (6 * R)):
        states.push(records=rec, **kw)


@pytest.mark.parametrize("argv, msg", [
    (["--algo", "mfac", "--envs", "4", "--replay", "states"], "Q learners"),
    (["--algo", "ac", "--envs", "4", "--replay", "states"], "Q learners"),
    (["--algo", "mfq", "--replay", "states"], "needs the batched engine"),
])
def test_replay_states_usage_errors(argv, msg, capsys):
    from mfmarl_b200.cli import battle_parser, check_battle_args
    ap = battle_parser("t", training=True)
    with pytest.raises(SystemExit):
        check_battle_args(ap, ap.parse_args(argv))
    assert msg in capsys.readouterr().err


def test_replay_states_is_accepted_for_the_q_learners():
    from mfmarl_b200.cli import battle_parser, check_battle_args
    ap = battle_parser("t", training=True)
    for algo in ("mfq", "il"):
        assert check_battle_args(ap, ap.parse_args(["--algo", algo, "--envs", "4", "--replay", "states"])).replay == "states"
    assert check_battle_args(ap, ap.parse_args(["--algo", "mfac"])).replay == "rows"
