"""Swendsen-Wang (K9) against checkerboard Metropolis (K8) on the GPU, measured (outputs in profiles/r07/):

  1. site-sweeps/s of each kernel at Tc, at 16384 x 20^2, 4096 x 64^2, 1024 x 128^2 and 296 x 256^2 (two waves of 148
     SMs): the kernel alone (torch.profiler's CUDA activity) and the whole call (CUDA events; it includes the host's
     threshold table and its upload);
  2. the integrated autocorrelation time at Tc of m^2 and of the bond energy for L = 16 .. 256, with Sokal's windowed
     estimator over many independent chains that start from equilibrium (200 K9 sweeps at Tc from random spins, the same
     spins for both methods);
  3. from the two, independent samples per second: lattice-sweeps/s of the timed series over 2 tau_int.

The card's name and power limit are read in the same run.

usage: python profiles/ising_cluster_probe.py [--rounds 3] [--quick]
"""
import argparse
import math
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "mean-field-multi-agent-reinforcement-learning_b200", "python"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from mfmarl_b200 import IsingMetropolis, IsingSwendsenWang  # noqa: E402

TC = 1.0 / math.log(1.0 + math.sqrt(2.0))
CHAINS = {"K9": IsingSwendsenWang, "K8": IsingMetropolis}
KERNELS = {"K9": "k_ising_swendsen_wang", "K8": "k_ising_metropolis"}


def rates(name, B, L, K, rounds):
    """(whole-call site-sweeps/s per round, kernel-alone site-sweeps/s per round) at Tc, K sweeps per launch"""
    chain = CHAINS[name](B, L, seed=5)
    chain.run([TC] * K)                                                # warm-up, and the chains reach Tc's clusters
    work = B * L * L * K
    call = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        chain.run([TC] * K)
        e1.record()
        torch.cuda.synchronize()
        call.append(work / (e0.elapsed_time(e1) * 1e-3))
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(rounds):
            chain.run([TC] * K)
        torch.cuda.synchronize()
    kern = [work / (e.time_range.elapsed_us() * 1e-6) for e in prof.events() if KERNELS[name] in e.name]
    return call, kern


def tau_int(series, c=6.0):
    """Sokal's windowed estimate of the integrated autocorrelation time of series [B, K] (B independent equilibrium
    chains): rho(t) from the chain-averaged autocovariance about the grand mean; the smallest window W >= c tau(W).
    -> (tau, its statistical error, W, True if the window was found before lag K / 4)"""
    x = series.to(torch.float64)
    x = x - x.mean()
    B, K = x.shape
    n = 1 << (2 * K - 1).bit_length()
    f = torch.fft.rfft(x, n=n, dim=1)
    acov = torch.fft.irfft(f * f.conj(), n=n, dim=1)[:, :K].sum(dim=0) / (B * torch.arange(K, 0, -1, device=x.device))
    rho = (acov / acov[0]).cpu().numpy()
    tau = 0.5 + np.cumsum(rho[1:])                                     # tau(W) for W = 1, 2, ...
    W = np.arange(1, K)
    ok = np.nonzero(W >= c * tau)[0]
    found = len(ok) > 0 and W[ok[0]] < K // 4
    w = int(W[ok[0]]) if len(ok) else K - 1
    t = float(tau[w - 1])
    return t, t * math.sqrt(2.0 * (2 * w + 1) / (B * K)), w, found


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", default=3, type=int)
    ap.add_argument("--quick", action="store_true", help="short series (a rehearsal, not a measurement)")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print("gpu: %s" % gpu, flush=True)
    q = 20 if args.quick else 1

    print("\n# 1. site-sweeps/s at T = Tc (call: CUDA events around the whole call; kernel: torch.profiler)", flush=True)
    for B, L, budget in ((16384, 20, 2e10), (4096, 64, 2e10), (1024, 128, 2e10), (296, 256, 2e10)):
        for name in ("K9", "K8"):
            K = max(10, int(budget / (B * L * L) / q / (10 if name == "K9" else 1)))
            call, kern = rates(name, B, L, K, args.rounds)
            print("%s %5d x %3d^2, %5d sweeps per launch: call %s  kernel %s site-sweeps/s"
                  % (name, B, L, K, " ".join("%.3e" % r for r in call), " ".join("%.3e" % r for r in kern)), flush=True)
            torch.cuda.empty_cache()

    print("\n# 2./3. tau_int at Tc (Sokal window, c = 6) and independent samples per second", flush=True)
    print("# method L chains sweeps | tau(m^2) +- err [W] | tau(e) +- err [W] | lattice-sweeps/s | indep. samples/s "
          "(m^2, e)", flush=True)
    # L: (chains, K9 sweeps, K8 sweeps); K8's series grow with its tau ~ L^2.17
    plan = {16: (2048, 5000, 40000), 32: (1024, 5000, 100000), 64: (1024, 5000, 200000), 128: (296, 5000, 400000),
            256: (148, 5000, 400000)}
    for L, (B, k9, k8) in plan.items():
        N = L * L
        eq = IsingSwendsenWang(B, L, seed=31)
        eq.run([TC] * 200)
        start = eq.spins.clone()
        for name, K in (("K9", k9 // q), ("K8", k8 // q)):
            chain = CHAINS[name](B, L, seed=41, spins=start)
            chunk = max(1, min(K, 20000))
            ups, bonds = [], []
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k0 in range(0, K, chunk):
                n_up, bond = chain.run([TC] * min(chunk, K - k0))
                ups.append(n_up); bonds.append(bond)
            e1.record()
            torch.cuda.synchronize()
            lsps = B * K / (e0.elapsed_time(e1) * 1e-3)
            m2 = ((2 * torch.cat(ups).to(torch.float64) - N) / N) ** 2
            en = -torch.cat(bonds).to(torch.float64) / N
            res = [tau_int(s.t().contiguous()) for s in (m2, en)]
            del ups, bonds, m2, en
            print("%s %3d %5d %7d | %9.3f +- %7.3f [%6d]%s | %9.3f +- %7.3f [%6d]%s | %.4e | %.4e %.4e"
                  % (name, L, B, K, res[0][0], res[0][1], res[0][2], "" if res[0][3] else " (window not found: "
                     "lower bound)", res[1][0], res[1][1], res[1][2], "" if res[1][3] else " (window not found: "
                     "lower bound)", lsps, lsps / (2 * res[0][0]), lsps / (2 * res[1][0])), flush=True)
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
