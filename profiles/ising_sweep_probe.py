"""Ising temperature sweeps on the GPU, measured (outputs in profiles/r05/):

  1. MF-Q at the C5 shape (16384 x 256^2, S = 100 sweeps per launch, K6s) with the shared schedule (mfi_run) and with
     a per-lattice table of the same values (mfi_run_lattices), alternated in one process;
  2. K8 Metropolis in site-sweeps/s at 16384 x 256^2 and 16384 x 20^2;
  3. the wall time of a 31-temperature x 8-replica sweep at 20 x 20 (one batch through the per-lattice tables) against
     31 separate IsingMFQ runs of 8 lattices each.

The card's name and power limit are read in the same run.  Timings: CUDA events around launches that are warmed up
first; the C5 working set (43 GB of Q) is far larger than the L2.

usage: python profiles/ising_sweep_probe.py [--rounds 3] [--lattices 16384]
"""
import argparse
import os
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "mean-field-multi-agent-reinforcement-learning_b200", "python"))

import torch  # noqa: E402

from mfmarl_b200 import IsingMetropolis, IsingMFQ  # noqa: E402
from mfmarl_b200 import ising_sweep  # noqa: E402
from mfmarl_b200.ising import temperature_schedule  # noqa: E402


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", default=3, type=int)
    ap.add_argument("--lattices", default=16384, type=int)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print("gpu: %s" % gpu, flush=True)
    B = args.lattices

    # 1. MF-Q C5: shared schedule vs per-lattice table, alternated
    S, L = 100, 256
    m = IsingMFQ(B, L, seed=13, lr=0.1)
    shared = torch.full((S,), 0.8, dtype=torch.float32, device=m.device)
    table = torch.full((S, B), 0.8, dtype=torch.float32, device=m.device)
    m.run(shared); m.run(table)                                         # warm-up of both kernels
    res = {"shared": [], "per-lattice": []}
    for r in range(args.rounds):
        for name, t in (("shared", shared), ("per-lattice", table)):
            ms = timed(lambda: m.run(t), 2)
            res[name].append(B * L * L * S / (ms * 1e-3))
    for name, v in res.items():
        print("mfq C5 %-11s %s site-steps/s (min %.4e max %.4e)" % (name, " ".join("%.4e" % x for x in v), min(v), max(v)),
              flush=True)
    del m, table
    torch.cuda.empty_cache()

    # 2. K8 Metropolis: the whole call (events; it includes the host's threshold table and its upload, with the
    # GPU idle meanwhile) and the kernel alone (torch.profiler's CUDA activity)
    for L, K in ((256, 100), (20, 1000)):
        chain = IsingMetropolis(B, L, seed=5)
        chain.run([1.0] * K)
        rates = []
        for r in range(args.rounds):
            ms = timed(lambda: chain.run([1.0] * K), 1)
            rates.append(B * L * L * K / (ms * 1e-3))
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for r in range(args.rounds):
                chain.run([1.0] * K)
            torch.cuda.synchronize()
        kern = [e.time_range.elapsed_us() for e in prof.events() if "k_ising_metropolis" in e.name]
        print("K8 %d x %d^2, %d sweeps per launch: call %s site-sweeps/s; kernel alone %s site-sweeps/s (%s ms)"
              % (B, L, K, " ".join("%.4e" % x for x in rates),
                 " ".join("%.4e" % (B * L * L * K / (t * 1e-6)) for t in kern), " ".join("%.2f" % (t * 1e-3) for t in kern)),
              flush=True)
        del chain
        torch.cuda.empty_cache()

    # 3. a 31-temperature sweep at 20 x 20: one batch vs 31 separate runs
    temps, R, L, K = ising_sweep.parse_grid("0.5:2.0:31"), 8, 20, 2000
    ising_sweep.run_mfq(temps[:2], R, L, 10)                             # warm-up
    for r in range(args.rounds):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        ising_sweep.run_mfq(temps, R, L, K)
        torch.cuda.synchronize(); t_batch = time.perf_counter() - t0
        t0 = time.perf_counter()
        for j, T in enumerate(temps):
            IsingMFQ(R, L, seed=13, lattice_base=j * R).run(temperature_schedule(0, K, 0.99, 2000, T))
        torch.cuda.synchronize(); t_sep = time.perf_counter() - t0
        print("sweep 31 T x %d replicas x %d^2, %d sweeps: one batch %.3f s, 31 separate runs %.3f s (%.1fx)"
              % (R, L, K, t_batch, t_sep, t_sep / t_batch), flush=True)


if __name__ == "__main__":
    main()
