"""CPU: the numpy reference of the neighbourhood mean action (tests/local_mean_ref.py) on hand-derived cases, its disc
pinned to the C oracle's view range, and the command-line check of --mean_field."""
import importlib.util
import os

import numpy as np
import pytest

from conftest import PKG
from engines import OracleEngine
from local_mean_ref import circle_offsets, local_mean_action

N_ACTION = 21


def test_radius_1_is_the_von_neumann_neighbourhood():
    assert sorted(circle_offsets(1)) == sorted([(0, -1), (-1, 0), (1, 0), (0, 1)])


def test_radius_1_5_is_the_moore_neighbourhood():
    want = [(dx, dy) for dy in (-1, 0, 1) for dx in (-1, 0, 1) if (dx, dy) != (0, 0)]
    assert circle_offsets(1.5) == want                       # row-major, as Range.h builds it


def test_radius_6_has_112_cells_besides_the_centre():
    offs = circle_offsets(6)
    assert len(offs) == 112 and len(set(offs)) == 112
    assert (6, 0) in offs and (0, -6) in offs and (4, 4) in offs and (5, 4) not in offs and (6, 1) not in offs


def test_three_agents_known_counts_and_quotients():
    pos = [[10, 10], [11, 10], [10, 12]]
    acts = [3, 5, 7]
    alive = [True, True, True]
    out = local_mean_action(pos, acts, alive, 1.5, N_ACTION)
    want = np.zeros((3, N_ACTION), np.float32)
    want[0, 5] = 1.0                                         # (1, 0) in the Moore disc; (0, 2) is not
    want[1, 3] = 1.0                                         # (-1, 0)
    assert np.array_equal(out, want)                         # agent 2 sees nobody at r = 1.5
    out = local_mean_action(pos, acts, alive, 2, N_ACTION)   # r = 2: (0, 2) is in, (-1, 2) is not
    want = np.zeros((3, N_ACTION), np.float32)
    want[0, 5] = want[0, 7] = np.float32(1) / np.float32(2)
    want[1, 3] = 1.0
    want[2, 3] = 1.0
    assert np.array_equal(out.view(np.uint32), want.view(np.uint32))
    out = local_mean_action(pos, [3, 3, 7], alive, 6, N_ACTION)
    assert np.array_equal(out[0], np.eye(N_ACTION, dtype=np.float32)[[3, 7]].mean(axis=0))
    assert out[2, 3] == 1.0 and out[1, 3] == np.float32(1) / np.float32(2) and out[1, 7] == np.float32(0.5)
    thirds = local_mean_action([[5, 5], [6, 5], [4, 5], [5, 6]], [0, 1, 1, 2], [True] * 4, 1, N_ACTION)
    assert thirds[0, 1] == np.float32(2) / np.float32(3) and thirds[0, 2] == np.float32(1) / np.float32(3)


def test_isolated_agent_gets_a_zero_row():
    out = local_mean_action([[5, 5], [20, 20]], [1, 2], [True, True], 6, N_ACTION)
    assert not out.any()


def test_agents_that_have_not_acted_or_are_dead_do_not_count():
    pos = [[5, 5], [6, 5], [5, 6]]
    out = local_mean_action(pos, [4, N_ACTION, 9], [True, True, True], 1.5, N_ACTION)
    assert out[0, 9] == 1.0 and out[0].sum() == 1.0          # agent 1 has not acted
    assert out[1, 4] == np.float32(0.5) and out[1, 9] == np.float32(0.5)   # agent 2 at (-1, 1) is in the Moore disc
    out = local_mean_action(pos, [4, 6, 9], [True, False, True], 1.5, N_ACTION)
    assert out[0, 9] == 1.0 and out[0].sum() == 1.0          # agent 1 is dead ...
    assert out[1, 4] == np.float32(0.5) and out[1, 9] == np.float32(0.5)   # ... but still observes


def test_a_dead_observer_counts_the_agent_standing_on_its_cell():
    out = local_mean_action([[5, 5], [5, 5]], [2, 8], [False, True], 1, N_ACTION)
    assert out[0, 8] == 1.0 and not out[1].any()


def test_radius_6_disc_is_the_oracle_view_disc():
    """One observer at (20, 20) of a 40x40 map with every other cell of its 13x13 window holding a group-mate: the
    oracle's own-group channel is the view disc, and it is circle_offsets(6) plus the centre."""
    o = OracleEngine(40)
    o.reset()
    window = [[20, 20]] + [[x, y] for y in range(14, 27) for x in range(14, 27) if (x, y) != (20, 20)]
    assert o.add_agents(0, window) == 169
    assert o.lib.mo_view_count(o.e) == 113
    view, _ = o.get_observation(0)
    pos = o.get_pos(0)
    assert tuple(pos[0]) == (20, 20)
    want = np.zeros((13, 13), np.float32)
    want[6, 6] = 1.0
    for dx, dy in circle_offsets(6):
        want[dy + 6, dx + 6] = 1.0
    assert np.array_equal(view[0, :, :, 1], want)


def _train_battle():
    spec = importlib.util.spec_from_file_location("train_battle", os.path.join(PKG, "python", "train_battle.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_train_battle_rejects_local_mean_field_without_envs(tmp_path, capsys):
    train = _train_battle()
    with pytest.raises(SystemExit) as ex:
        train.main(["--algo", "mfq", "--mean_field", "local", "--data_dir", str(tmp_path / "data")])
    assert ex.value.code == 2
    assert "--mean_field local" in capsys.readouterr().err
    assert not (tmp_path / "data").exists()
    with pytest.raises(SystemExit):
        train.main(["--algo", "mfq", "--mean_field", "nearby", "--envs", "4"])
