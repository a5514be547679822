"""What random placement (mfb_add_agents_random) costs on the GPU, against the fixed blocks of map_positions:
  commit   host wall time of a placement commit (template upload, k_place, the read-back of the counts) for 4096 envs
           x 64 v 64 at 40x40, random halves (random_halves) against the blocks; every repetition is a fresh reset
  loop     agent-steps/s of a C3-shaped loop (4096 envs, 40x40, 64 v 64, Philox, uniform random actions, observe +
           step) with auto_reset and max_steps 20, so every env re-places itself every 20 steps
One JSON line per measurement.      python profiles/random_placement_probe.py > profiles/r13/random_placement_probe.txt"""
import json
import os
import subprocess
import sys
import time

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "mean-field-multi-agent-reinforcement-learning_b200", "python"))

from mfmarl_b200 import BatchedGridWorld  # noqa: E402
from mfmarl_b200.senario_battle import map_positions, random_halves  # noqa: E402

E, M, CAP = 4096, 40, 64


def program(env, placement):
    env.reset()
    if placement == "random":
        left, right = random_halves(M)
        env.add_agents_random(0, 64, left)
        env.add_agents_random(1, 64, right)
    else:
        left, right = map_positions(M)
        env.add_agents(0, left)
        env.add_agents(1, right)


def commit_ms(placement, reps=30):
    env = BatchedGridWorld(E, map_size=M, capacity=CAP, rng="philox", seed=1)
    times = []
    for i in range(reps + 5):
        program(env, placement)
        torch.cuda.synchronize()
        t = time.perf_counter()
        env.query("n_envs")                       # commits the placement (synchronous)
        if i >= 5:
            times.append((time.perf_counter() - t) * 1e3)
    assert (env.get("num") == 64).all()
    times.sort()
    return {"probe": "commit", "placement": placement, "envs": E, "median_ms": times[len(times) // 2],
            "min_ms": times[0], "max_ms": times[-1]}


def loop_rate(placement, steps=400, warmup=40):
    env = BatchedGridWorld(E, map_size=M, capacity=CAP, rng="philox", seed=1, auto_reset=True, max_steps=20)
    program(env, placement)
    gen = torch.Generator(device="cuda").manual_seed(0)
    acts = [torch.randint(0, 21, (E, 2, CAP), dtype=torch.int32, device="cuda", generator=gen) for _ in range(8)]
    for s in range(warmup):
        env.observe_groups(); env.step(acts[s % 8])
    torch.cuda.synchronize()
    before = int(env.get("agent_steps").sum())
    t = time.perf_counter()
    for s in range(steps):
        env.observe_groups(); env.step(acts[s % 8])
    torch.cuda.synchronize()
    dt = time.perf_counter() - t
    agents = int(env.get("agent_steps").sum()) - before
    return {"probe": "auto_reset_loop", "placement": placement, "envs": E, "max_steps": 20, "steps": steps,
            "seconds": dt, "agent_steps_per_s": agents / dt, "placement_short": int(env.get("placement_short").sum())}


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": gpu[0] if gpu else "unknown"}))
    for rep in range(3):                          # alternated, so drift shows up in both
        for placement in ("blocks", "random"):
            print(json.dumps(dict(commit_ms(placement), rep=rep)), flush=True)
    for rep in range(3):
        for placement in ("blocks", "random"):
            print(json.dumps(dict(loop_rate(placement), rep=rep)), flush=True)


if __name__ == "__main__":
    main()
