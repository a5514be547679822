"""Agent-steps/s of observe + step, and per-kernel time, for battle geometries on either side of the shared-memory
limit: M = 128 (every kernel in shared memory) and M = 176, 256, 400 at the training scripts' density
(capacity = 0.04 M^2), with enough envs that the observation rows exceed 1 GB per step.  k_obs's algorithmic bytes
(4868 per agent: view + feature row) over its time are printed beside C4's (80x80, 512 v 512, 128 envs).

    python profiles/large_map_probe.py [--steps 20] [--out large_map_probe.txt]

Kernel times are CUDA events around each launch; the card's name and power limit are read in the same run."""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "mean-field-multi-agent-reinforcement-learning_b200", "python"))
from mfmarl_b200 import BatchedGridWorld                               # noqa: E402
from mfmarl_b200.scenarios import c4_positions, generate_map_positions  # noqa: E402

BYTES_PER_AGENT_OBS = 13 * 13 * 7 * 4 + 34 * 4


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as ex:   # the probe still reports its numbers
        return "unknown (%s)" % ex


def run(m, E, steps, pos=None, cap=None):
    cap = cap or max(64, int(m * m * 0.04))
    left, right = pos if pos is not None else generate_map_positions(m)
    env = BatchedGridWorld(E, map_size=m, capacity=cap, rng="philox", seed=1)
    env.reset(); env.add_agents(0, left); env.add_agents(1, right)
    mask = env.query("hbm_kernels")
    rng = np.random.RandomState(0)
    acts = [torch.from_numpy(rng.randint(0, 21, size=(E, 2, env.capacity)).astype(np.int32)).cuda() for _ in range(4)]
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    agents = 0
    for s in range(2):                                               # warm-up
        env.observe(); env.step(acts[s % 4], clear_dead=False, want_mean_action=False)
    torch.cuda.synchronize()
    num0 = int(env.get_num().sum())
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for s in range(steps):
        ev[s][0].record(); env.observe(); ev[s][1].record()
        env.step(acts[s % 4], clear_dead=False, want_mean_action=False); ev[s][2].record()
    t1.record()
    torch.cuda.synchronize()
    agents = num0 * steps                                             # no clear_dead: the listed agents stay
    obs_ms = np.median([a.elapsed_time(b) for a, b, _ in ev])
    step_ms = np.median([b.elapsed_time(c) for _, b, c in ev])
    total_s = t0.elapsed_time(t1) / 1e3
    obs_gb = num0 * BYTES_PER_AGENT_OBS / 1e9
    line = ("M=%4d cap=%5d E=%4d hbm_kernels=%2d agents/step=%9d obs=%.2f GB/step  %.3e agent-steps/s  "
            "k_obs %.3f ms (%.0f GB/s algorithmic)  k_step %.3f ms" %
            (m, env.capacity, E, mask, num0, obs_gb, agents / total_s, obs_ms, obs_gb / (obs_ms / 1e3), step_ms))
    del env
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = ["card: " + card()]
    lines.append("C4 " + run(80, 128, a.steps, pos=c4_positions(), cap=512))
    for m in (128, 176, 256, 400):
        per_env = 2 * max(64, int(m * m * 0.04)) * BYTES_PER_AGENT_OBS
        E = max(2, -(-int(1.05e9) // per_env)) if m > 128 else 64
        lines.append(run(m, E, a.steps))
        print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        open(a.out, "w").write(text)


if __name__ == "__main__":
    main()
