"""CPU: pins the numpy Ising oracle against the UNMODIFIED reference classes (run under the gym/imp shim
of oracle/ising_ref_shim) with injected uniforms -- exact float64 equality.  The comparison is skipped when the
reference tree is absent.  Without it only test_golden.py checks the oracle against the reference, on the one stored
20x20 run at T = 0.8 (tests/golden/ising20.npz); the other sizes and temperatures below are not covered then."""
import os
import sys

import numpy as np
import pytest

from conftest import REPO

sys.path.insert(0, os.path.join(REPO, "oracle"))
import ising_oracle  # noqa: E402

REF = "/root/reference"


def reference_env(n_agents, seed):
    for p in (os.path.join(REPO, "oracle", "ising_ref_shim"), REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    from examples.ising_model.multiagent.environment import IsingMultiAgentEnv
    import examples.ising_model as im
    sc = im.load("Ising.py").Scenario()
    np.random.seed(seed)
    env = IsingMultiAgentEnv(world=sc.make_world(num_agents=n_agents, agent_view=1),
                             reset_callback=sc.reset_world, reward_callback=sc.reward,
                             observation_callback=sc.observation, done_callback=sc.done)
    return env


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "examples", "ising_model")), reason="reference tree not present")
@pytest.mark.filterwarnings("ignore::DeprecationWarning")
@pytest.mark.parametrize("n,T,steps", [(400, 0.8, 25), (100, 0.297, 40), (49, 2.0, 30)])
def test_oracle_equals_reference_loop_body(n, T, steps):
    env = reference_env(n, seed=13)
    obs = np.stack(env.reset())
    spins = env.world.global_state.copy().astype(np.int64)[None]
    Qref, Qo = np.zeros((n, 5, 2)), np.zeros((1, 5, n, 2))
    rng = np.random.RandomState(5)
    lr = 0.1
    for t in range(steps):
        u = rng.random_sample(n)
        action = np.zeros(n, dtype=np.int32)
        for i in range(n):     # main_MFQ_Ising.py:114-116 with np.random.choice's draw injected
            s = np.count_nonzero(obs[i] == 1)
            vals = [np.exp(Qref[i, s, k] / T) for k in range(2)]
            denom = 0
            for v in vals:
                denom += v
            cdf = np.array([v / denom for v in vals]).cumsum()
            cdf /= cdf[-1]
            action[i] = cdf.searchsorted(u[i], side="right")
        obs_, reward, done, order, ups, downs = env.step(np.expand_dims(action, 1))
        for i in range(n):     # main_MFQ_Ising.py:127-131
            s = np.count_nonzero(obs[i] == 1)
            Qref[i, s, action[i]] = Qref[i, s, action[i]] + lr * (float(reward[i][0]) - Qref[i, s, action[i]])
        obs = np.stack(obs_)
        spins, Qo, info = ising_oracle.step(spins, Qo, T, lr, u[None])
        assert np.array_equal(info["action"][0], action)
        assert np.array_equal(info["reward"][0], np.array(reward).reshape(-1))
        assert np.array_equal(Qo[0].transpose(1, 0, 2), Qref)
        assert info["order"][0] == order and info["n_up"][0] == ups
        assert np.array_equal(spins[0], env.world.global_state.astype(np.int64))


def test_temperature_schedule():
    cur = 0.3
    seen = []
    for t in range(5):
        cur = ising_oracle.temperature_schedule(t, cur, 0.8)
        seen.append(cur)
    assert seen == [0.8] * 5
    cur = ising_oracle.temperature_schedule(0, 0.3, 0.1)
    assert abs(cur - 0.297) < 1e-12
