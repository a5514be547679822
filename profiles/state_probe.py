"""Time of saving, loading and forking every env of a battle engine (mfb_save_envs / mfb_load_envs), per call and as
GB/s of record bytes (n * R: what a save writes and a load reads; a save also reads as many bytes of state and a load
writes them, and a load reads its records twice -- check, then scatter).

    python profiles/state_probe.py [--calls 50] [--out state_probe.txt]

  save   save_envs() of every env: CUDA events around `calls` back-to-back calls (asynchronous on the stream)
  load   load_envs() of every env: host clock around each call, which ends in the check kernel's read-back (the one
         synchronisation of a load) and then enqueues the scatter; a synchronise closes each timed call
  fork   save_envs([0] * E) + load_envs(): env 0 copied into every env, host clock as for load

Geometries: C3 (40x40, 64 v 64, 4096 envs), C4 (80x80, 512 v 512, 128 envs), one whose kernels run from HBM (M = 256
at the scripts' density), and C3's geometry at 32768 envs, whose records (137 MB) do not fit the 126 MB L2.  The card's
name and power limit are read in the same run."""
import argparse
import ctypes
import os
import subprocess
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "mean-field-multi-agent-reinforcement-learning_b200", "python"))
from mfmarl_b200 import BatchedGridWorld                               # noqa: E402
from mfmarl_b200.scenarios import c4_positions, generate_map_positions  # noqa: E402

L2_BYTES = 126e6


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as ex:   # the probe still reports its numbers
        return "unknown (%s)" % ex


def host_timed(fn, calls):
    times = []
    for _ in range(calls):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return float(np.median(times)) * 1e6


def run(name, m, cap, E, calls, pos=None):
    left, right = pos if pos is not None else generate_map_positions(m)
    env = BatchedGridWorld(E, map_size=m, capacity=cap, rng="philox", seed=1, max_steps=50, auto_reset=True)
    env.reset(); env.add_agents(0, left); env.add_agents(1, right)
    rng = np.random.RandomState(0)
    for _ in range(3):   # a mid-game state
        env.step(torch.from_numpy(rng.randint(0, 21, size=(E, 2, env.capacity)).astype(np.int32)).cuda())
    R = env.query("state_bytes")
    rec = env.save_envs()
    for _ in range(3):   # warm-up of every path
        env.save_envs(); env.load_envs(rec); env.load_envs(env.save_envs([0] * E))
    rec = env.save_envs()
    torch.cuda.synchronize()
    out = torch.empty_like(rec)
    idx_all = None
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.current_stream().cuda_stream
    t0.record()
    for _ in range(calls):
        assert env.lib.mfb_save_envs(env._h, E, idx_all, ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(stream)) == 0
    t1.record()
    torch.cuda.synchronize()
    assert torch.equal(out, rec)
    save_us = t0.elapsed_time(t1) * 1e3 / calls
    load_us = host_timed(lambda: env.load_envs(rec), calls)
    fork_us = host_timed(lambda: env.load_envs(env.save_envs([0] * E)), calls)
    total = E * R
    gbs = lambda us: total / (us * 1e-6) / 1e9   # noqa: E731
    return ("%-28s hbm_kernels=%2d R=%7d B  n*R=%7.1f MB (%s L2)  save %8.1f us %6.0f GB/s  "
            "load %8.1f us %6.0f GB/s  fork %8.1f us %6.0f GB/s" % (
                name, env.query("hbm_kernels"), R, total / 1e6, "fits" if total < L2_BYTES else "exceeds",
                save_us, gbs(save_us), load_us, gbs(load_us), fork_us, gbs(fork_us)))


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    lines = ["card: " + card()]
    print(lines[0], flush=True)
    m256 = max(64, int(256 * 256 * 0.04))
    for name, m, cap, E, pos in [("C3 40x40 64v64 x4096", 40, 64, 4096, None),
                                 ("C4 80x80 512v512 x128", 80, 512, 128, c4_positions()),
                                 ("M=256 cap %d x42" % m256, 256, m256, 42, None),
                                 ("40x40 64v64 x32768", 40, 64, 32768, None)]:
        lines.append(run(name, m, cap, E, a.calls, pos))
        print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
