"""K7 (k_local_mean_action, BatchedGridWorld.local_mean_action) measured on its own and next to the lockstep step it
would run beside, plus the rollout rate of play_batched with the group and the local mean field.

    python profiles/local_mean_probe.py [--out profiles/r03/local_mean_probe.txt]

* K7 alone at the C3 shape (4096 envs x 64 v 64, 40x40) and the C4 shape (128 envs x 512 v 512, 80x80), radius 6 and
  1.5, after 50 steps of a fight-like action stream (groups mixed, partly dead).  Regions of >= 0.5 s of launches
  between CUDA events.  Reported: us per launch, agents/s (listed agents), the share of the 92 B/agent bound (8 B of
  pos + state read, 84 B of row written, at the 6.55 TB/s copy peak of DESIGN.md section 5) and the share of one
  lockstep step (observe_groups + step at the same shape, timed in the same run).
* play_batched at 1024 envs, bf16 observation rows, MF-Q and MF-AC, mean_field "group" and "local" alternated.
The GPU name and power limit are read in the same run and printed first."""
import argparse
import math
import os
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "mean-field-multi-agent-reinforcement-learning_b200", "python"))
from mfmarl_b200 import BatchedGridWorld  # noqa: E402
from mfmarl_b200.scenarios import c4_positions, generate_map_positions  # noqa: E402

COPY_PEAK = 6.55e12          # B/s, measured HBM copy peak (DESIGN.md section 5)
BYTES_READ, N_ACTION = 8, 21
MOVE_DELTAS = [(0, -2), (-1, -1), (0, -1), (1, -1), (-2, 0), (-1, 0), (0, 0), (1, 0), (2, 0),
               (-1, 1), (0, 1), (1, 1), (0, 2)]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else "nvidia-smi gave nothing"
    except Exception as ex:            # the name from torch is still worth printing
        return "%s (power limit not read: %s)" % (torch.cuda.get_device_name(), ex)


def fight_actions(env, gen):
    """device version of tests/scenarios.fight_actions: 50 % random attack, 35 % one move toward the map centre,
    15 % uniform"""
    E, cap = env.n_envs, env.capacity
    pos = env.device_state("pos")
    x, y = pos & 0xFFFF, (pos >> 16) & 0xFFFF
    c = env.map_size // 2
    lut = torch.full((3, 3), 6, dtype=torch.int32, device=pos.device)
    for k, (dx, dy) in enumerate(MOVE_DELTAS):
        if abs(dx) <= 1 and abs(dy) <= 1:
            lut[dy + 1, dx + 1] = k
    toward = lut[torch.sign(c - y).long() + 1, torch.sign(c - x).long() + 1]
    u = torch.rand((E, 2, cap), generator=gen, device=pos.device)
    attack = torch.randint(13, 21, (E, 2, cap), generator=gen, device=pos.device, dtype=torch.int32)
    uniform = torch.randint(0, 21, (E, 2, cap), generator=gen, device=pos.device, dtype=torch.int32)
    return torch.where(u < 0.5, attack, torch.where(u < 0.85, toward, uniform)).contiguous()


def timed(fn, min_seconds=0.5):
    """ms per call over a region of >= min_seconds (a 10-call calibration picks the count)"""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(10):
        fn()
    t1.record()
    torch.cuda.synchronize()
    reps = max(10, int(math.ceil(min_seconds * 1e3 / (t0.elapsed_time(t1) / 10))))
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps, reps


def kernel_shapes(out):
    gen = torch.Generator(device="cuda").manual_seed(0)
    for name, E, ms, cap, pos in (("C3 40x40 64v64 x4096", 4096, 40, 64, generate_map_positions(40)),
                                  ("C4 80x80 512v512 x128", 128, 80, 512, c4_positions())):
        env = BatchedGridWorld(E, map_size=ms, capacity=cap, rng="philox", seed=1)
        env.reset(); env.add_agents(0, pos[0]); env.add_agents(1, pos[1])
        for _ in range(50):
            env.step(fight_actions(env, gen))
        num = env.get_num()
        listed = int(num.sum())
        alive_acted = 0
        la, al = env.get("last_action"), env.get("alive")
        for e in range(E):
            for g in range(2):
                n = num[e, g]
                alive_acted += int(((la[e, g, :n] < N_ACTION) & (al[e, g, :n] > 0)).sum())
        bytes_moved = BYTES_READ * listed + 4 * N_ACTION * E * 2 * env.capacity
        out("%s: %d listed agents after 50 fight steps (%d alive and acted), %.1f MB per K7 launch" % (
            name, listed, alive_acted, bytes_moved / 1e6))
        # the lockstep step: observe both groups (per-group fp32 blocks) + step, fixed actions, armies re-placed when
        # an episode ends so that the state stays a battle
        step_env = BatchedGridWorld(E, map_size=ms, capacity=cap, rng="philox", seed=2, auto_reset=True, max_steps=100)
        step_env.reset(); step_env.add_agents(0, pos[0]); step_env.add_agents(1, pos[1])
        acts = fight_actions(step_env, gen)

        def lockstep():
            step_env.observe_groups()
            step_env.step(acts)
        step_ms, step_reps = timed(lockstep)
        out("%s: observe_groups + step  %9.1f us per step (%d steps timed)" % (name, step_ms * 1e3, step_reps))
        for r in (6.0, 1.5):
            k_ms, reps = timed(lambda: env.local_mean_action(radius=r))
            bound_ms = bytes_moved / COPY_PEAK * 1e3
            out("%s: K7 r=%-4g %9.1f us per launch  %.3e agents/s  %.2f of the 92 B/agent bound  %.3f of a lockstep "
                "step  (%d launches timed)" % (name, r, k_ms * 1e3, listed / (k_ms * 1e-3), bound_ms / k_ms,
                                                k_ms / step_ms, reps))
        del env, step_env
        torch.cuda.empty_cache()


def rollout(out, steps, repeats):
    from mfmarl_b200.algo import spawn_ai
    from mfmarl_b200.senario_battle import play_batched

    class Spaces:
        def get_view_space(self, h): return (13, 13, 7)
        def get_feature_space(self, h): return (34,)
        def get_action_space(self, h): return (21,)

    E = 1024
    for algo in ("mfq", "mfac"):
        torch.manual_seed(0)
        env = BatchedGridWorld(E, map_size=40, capacity=64, rng="philox", seed=0)
        models = [spawn_ai(algo, Spaces(), g, "%s-%d" % (algo, g), steps, device="cuda") for g in range(2)]
        rates = {"group": [], "local": []}
        for mf in ("group", "local"):        # warm-up of both paths (graph capture, cuDNN algorithm choice)
            play_batched(env, 0, 5, models, eps=1.0, train=False, left_group=0, obs_dtype=torch.bfloat16, mean_field=mf)
        for rep in range(repeats):
            for mf in ("group", "local"):
                torch.cuda.synchronize()
                a0 = int(env.get("agent_steps").sum())
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                play_batched(env, 1, steps, models, eps=1.0, train=False, left_group=0, obs_dtype=torch.bfloat16,
                             mean_field=mf)
                t1.record()
                torch.cuda.synchronize()
                ms = t0.elapsed_time(t1)
                rates[mf].append((int(env.get("agent_steps").sum()) - a0) / (ms * 1e-3))
        for mf in ("group", "local"):
            rs = sorted(rates[mf])
            out("play_batched %-4s 1024 envs bf16 rows, %d steps, mean_field=%-5s: %s agent-steps/s (median %.3e)" % (
                algo, steps, mf, " ".join("%.3e" % v for v in rates[mf]), rs[len(rs) // 2]))
        g, l = sorted(rates["group"])[repeats // 2], sorted(rates["local"])[repeats // 2]
        out("play_batched %-4s local / group = %.3f" % (algo, l / g))
        del env, models
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--steps", type=int, default=200, help="steps per play_batched round")
    ap.add_argument("--repeats", type=int, default=3, help="alternations of group / local per learner")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("local_mean_probe.py needs a CUDA device")
    lines = []

    def out(s):
        print(s, flush=True)
        lines.append(s)
    out("GPU: %s" % gpu_info())
    kernel_shapes(out)
    rollout(out, args.steps, args.repeats)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
