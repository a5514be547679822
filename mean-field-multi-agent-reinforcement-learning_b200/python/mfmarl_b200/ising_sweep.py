"""`python -m mfmarl_b200.ising_sweep`: the Ising curve -- order parameter and bond energy against temperature -- for
MF-Q and for MCMC chains of the same model, every (temperature, replica) lattice of a method in ONE batch.

MF-Q: lattice (j, r) follows main_MFQ_Ising.py's schedule (T from 0.3, times --decay_rate every --decay_gap sweeps)
with the floor T_j (that script's -t flag), through the per-lattice temperature tables of `mfi_run_lattices`.
MCMC (`--method mcmc`, CSV label mcmc): checkerboard Metropolis (K8, `mfi_metropolis`) at T_j for every sweep; even
sides only.
SW (`--method sw`, CSV label sw): Swendsen-Wang cluster updates (K9, `mfi_swendsen_wang`) at T_j for every sweep; any
side up to 256.  Near Tc its autocorrelation time is a few sweeps at any side, where Metropolis needs ~L^2 sweeps.
`--method both` is MF-Q and Metropolis.
Per temperature: mean and standard error over the replicas of each lattice's average, over the final --window sweeps,
of |2 up - N| / N and of the bond energy per site -sum_bonds sigma_i sigma_j / N (-2 when ordered; the energy of the
model, H = -1/2 sum_bonds sigma_i sigma_j, is half of it).  Lattice (j, r) is lattice j * replicas + r of the batch and
has lattice_base j * replicas + r, so it draws what it would draw in a run of its own.
"""
import argparse
import csv

import numpy as np
import torch

from .ising import IsingMetropolis, IsingMFQ, IsingSwendsenWang, temperature_schedule

COLUMNS = ["temperature", "order_mean", "order_sem", "energy_mean", "energy_sem"]


def parse_grid(text):
    """"lo:hi:n" -> n evenly spaced temperatures (both ends included); "a,b,c" -> those temperatures"""
    if ":" in text:
        lo, hi, n = text.split(":")
        return [float(t) for t in np.linspace(float(lo), float(hi), int(n))]
    return [float(t) for t in text.split(",")]


def summarise(temps, replicas, side, n_up, bond_sum, window):
    """n_up, bond_sum [K, B] (B = len(temps) * replicas) -> table [len(temps), 5] (COLUMNS)"""
    N = side * side
    up = n_up[-window:].to(torch.float64)
    order = ((2 * up - N).abs() / N).mean(dim=0).view(len(temps), replicas)        # per-lattice window averages
    energy = (-bond_sum[-window:].to(torch.float64) / N).mean(dim=0).view(len(temps), replicas)
    sem = lambda x: x.std(dim=1) / replicas ** 0.5 if replicas > 1 else torch.zeros_like(x[:, 0])  # noqa: E731
    table = torch.stack([torch.tensor(temps, dtype=torch.float64), order.mean(dim=1).cpu(), sem(order).cpu(),
                         energy.mean(dim=1).cpu(), sem(energy).cpu()], dim=1)
    return table.numpy()


def mfq_schedules(temps, replicas, sweeps, decay_rate, decay_gap):
    """[sweeps, len(temps) * replicas]: column j * replicas + r is main_MFQ_Ising.py's schedule with floor temps[j]"""
    cols = [temperature_schedule(0, sweeps, decay_rate, decay_gap, t) for t in temps for _ in range(replicas)]
    return torch.tensor(cols, dtype=torch.float64).t().contiguous()


def run_mfq(temps, replicas, side, sweeps, seed=13, lr=0.1, decay_rate=0.99, decay_gap=2000, spins=None, chunk=1000):
    """all lattices in one IsingMFQ, chunk sweeps per launch -> (n_up int32 [K, B], reward_sum [K, B])"""
    B = len(temps) * replicas
    model = IsingMFQ(B, side, seed=seed, lr=lr, spins=spins)
    sched = mfq_schedules(temps, replicas, sweeps, decay_rate, decay_gap).to(model.device)
    ups, rsums = [], []
    for k0 in range(0, sweeps, chunk):
        n_up, rsum = model.run(sched[k0:k0 + chunk].contiguous())
        ups.append(n_up); rsums.append(rsum)
    return torch.cat(ups), torch.cat(rsums)


def run_mcmc(temps, replicas, side, sweeps, seed=13, start="up", chunk=1000, chain_class=IsingMetropolis):
    """all lattices in one chain_class (IsingMetropolis or IsingSwendsenWang)
    -> (n_up int32 [K, B], bond_sum int32 [K, B])"""
    B = len(temps) * replicas
    spins = torch.ones((B, side, side), dtype=torch.int8) if start == "up" else None
    chain = chain_class(B, side, seed=seed, spins=spins)
    table = np.repeat(np.asarray(temps, np.float64), replicas)[None, :]
    ups, bonds = [], []
    for k0 in range(0, sweeps, chunk):
        n_up, bond = chain.run(np.repeat(table, min(chunk, sweeps - k0), axis=0))
        ups.append(n_up); bonds.append(bond)
    return torch.cat(ups), torch.cat(bonds)


def sweep(argv=None):
    """-> {method: table [n_temperatures, 5]} (COLUMNS), printed one line per temperature and written to --out"""
    ap = argparse.ArgumentParser(description="Ising order parameter and energy against temperature (B200)")
    ap.add_argument("--temperatures", default="0.5:2.0:31", help="lo:hi:n (n points, ends included) or a,b,c")
    ap.add_argument("--replicas", default=8, type=int, help="independent lattices per temperature")
    ap.add_argument("--side", default=20, type=int, help="lattice side (the paper's 20 x 20 by default)")
    ap.add_argument("--sweeps", default=5000, type=int)
    ap.add_argument("--window", default=1000, type=int, help="final sweeps the averages are taken over")
    ap.add_argument("--method", default="both", choices=["mfq", "mcmc", "sw", "both"],
                    help="mcmc: Metropolis (even sides); sw: Swendsen-Wang (any side <= 256); both: mfq and mcmc")
    ap.add_argument("--seed", default=13, type=int)
    ap.add_argument("-lr", "--learning_rate", default=0.1, type=float)
    ap.add_argument("-dr", "--decay_rate", default=0.99, type=float)
    ap.add_argument("-dg", "--decay_gap", default=2000, type=int)
    ap.add_argument("--mcmc_start", default="up", choices=["up", "random"],
                    help="start of the mcmc and sw chains: all up (reaches either phase fast) or Bernoulli(0.5)")
    ap.add_argument("--out", default=None, help="CSV file of the table (one row per method and temperature)")
    args = ap.parse_args(argv)
    temps = parse_grid(args.temperatures)
    assert 1 <= args.window <= args.sweeps, "--window must be in [1, --sweeps]"
    methods = ["mfq", "mcmc"] if args.method == "both" else [args.method]
    tables = {}
    for method in methods:
        if method == "mfq":
            n_up, rsum = run_mfq(temps, args.replicas, args.side, args.sweeps, seed=args.seed, lr=args.learning_rate,
                                 decay_rate=args.decay_rate, decay_gap=args.decay_gap)
        else:
            n_up, rsum = run_mcmc(temps, args.replicas, args.side, args.sweeps, seed=args.seed, start=args.mcmc_start,
                                  chain_class=IsingSwendsenWang if method == "sw" else IsingMetropolis)
        tables[method] = summarise(temps, args.replicas, args.side, n_up, rsum, args.window)
    for j, T in enumerate(temps):
        print("T = %.4f  " % T + "  ".join("%s |m| = %.4f +- %.4f  e = %.4f +- %.4f" % ((m,) + tuple(tables[m][j, 1:]))
                                          for m in methods))
    if args.out:
        with open(args.out, "w", newline="") as f:
            w = csv.writer(f)
            w.writerow(["method"] + COLUMNS)
            for m in methods:
                for row in tables[m]:
                    w.writerow([m] + ["%.9g" % v for v in row])
    return tables


if __name__ == "__main__":
    sweep()
