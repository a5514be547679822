"""How sparse are the fp32 observation rows k_obs writes?  A CPU estimate with the C oracle (oracle/magent_oracle.c),
uniform-random actions as bench.py drives them, episodes auto-reset at done / max steps.  Each snapshot lays one
environment's rows out as the engine does, [2 groups][cap][13][13][7] fp32, and counts non-zero words, all-zero 32-byte
sectors and 128-byte lines with at most a quarter of their words non-zero.  No GPU needed.

Rows at or past an agent count are taken as zeros, as --dump-outputs writes them.  In the engine's own blocks they are
stale rows that k_obs does not rewrite, so they cost no writes at all; counting them as zero words makes the figures
somewhat optimistic for the rows k_obs actually writes, more so late in an episode.  Only the two benchmark placements are known: 40x40
with 64 v 64 (C3) and 80x80 with 512 v 512 (C4).

    python profiles/obs_sparsity.py                      # C3: 40x40, 64 v 64
    python profiles/obs_sparsity.py --map 80 --cap 512   # C4: 80x80, 512 v 512
"""
import argparse
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "mean-field-multi-agent-reinforcement-learning_b200", "python"))
sys.path.insert(0, os.path.join(REPO, "tests"))
from engines import OracleEngine  # noqa: E402
from mfmarl_b200.scenarios import c4_positions, generate_map_positions  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--map", type=int, default=40)
    ap.add_argument("--cap", type=int, default=64)
    ap.add_argument("--episodes", type=int, default=3)
    ap.add_argument("--steps", type=int, default=200, help="snapshots at steps 0 .. steps-1 of each episode")
    ap.add_argument("--max-steps", type=int, default=400, help="episode length limit (auto-reset)")
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    if (a.map, a.cap) not in ((40, 64), (80, 512)):
        ap.error("--map/--cap: only the benchmark shapes 40/64 (C3) and 80/512 (C4) have a placement here")
    left, right = generate_map_positions(40) if a.map == 40 else c4_positions()
    rng = np.random.RandomState(a.seed)
    eng = OracleEngine(a.map)
    words = nz = sectors = zero_sectors = lines = sparse_lines = 0
    rows = np.zeros((2, a.cap, 13 * 13 * 7), np.float32)
    for _ in range(a.episodes):
        eng.reset(); eng.add_agents(0, left); eng.add_agents(1, right)
        for s in range(min(a.steps, a.max_steps)):
            n = [eng.get_num(g) for g in range(2)]
            rows[:] = 0.0
            for g in range(2):
                rows[g, :n[g]] = eng.get_observation(g)[0].reshape(n[g], -1)
            w = rows.reshape(-1).view(np.uint32) != 0
            words += w.size; nz += int(w.sum())
            sec = w.reshape(-1, 8).any(axis=1)
            sectors += sec.size; zero_sectors += int((~sec).sum())
            per_line = w.reshape(-1, 32).sum(axis=1)
            lines += per_line.size; sparse_lines += int((per_line <= 8).sum())
            for g in range(2):
                eng.set_action(g, rng.randint(0, 21, size=n[g]).astype(np.int32))
            done = eng.step()
            eng.clear_dead()
            if done:
                break
    print("map %dx%d, %d v %d, %d episodes, snapshots at steps 0..%d: %.1f %% of fp32 words non-zero, %.1f %% of 32-byte "
          "sectors all zero, %.1f %% of 128-byte lines with <= 1/4 of their words non-zero"
          % (a.map, a.map, a.cap, a.cap, a.episodes, a.steps - 1, 100.0 * nz / words, 100.0 * zero_sectors / sectors,
             100.0 * sparse_lines / lines))


if __name__ == "__main__":
    main()
