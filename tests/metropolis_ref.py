"""numpy restatement of K8 (`mfi_metropolis`, csrc/ising_mcmc.cu): checkerboard single-spin-flip Metropolis on L x L
tori, with the Philox keys, counters and integer thresholds documented in include/mfmarl_batched.h.  Test
infrastructure: the GPU kernel is compared with it bit for bit."""
import math

import numpy as np

from philox_ref import philox4x32_10

TAG = 2     # counter word 3 of K8's draws (MF-Q uses 0 and 1)


def threshold(h, T):
    """accept a flip with h in {2, 4} when the site's 32-bit Philox word is below this integer"""
    return min(int(math.floor(math.exp(-h / T) * 2 ** 32)), 2 ** 32 - 1)


def local_field(spins):
    """h_i = sigma_i sum_nbr sigma_j for int spins [..., L, L] in {0, 1}"""
    s = 2 * spins.astype(np.int64) - 1
    nb = np.roll(s, 1, -2) + np.roll(s, -1, -2) + np.roll(s, 1, -1) + np.roll(s, -1, -1)
    return s * nb


def accept(h, word, thr2, thr4):
    """the Metropolis decision for one site (all arguments broadcastable)"""
    word = np.asarray(word, dtype=np.uint64)
    return (h <= 0) | ((h == 2) & (word < np.uint64(thr2))) | ((h == 4) & (word < np.uint64(thr4)))


def words(B, L, seed, lattice_base, step, colour):
    """[B, L, L] uint32: the Philox word every site would draw in half-sweep (step, colour)"""
    wpr = (L + 31) // 32
    y = np.arange(L, dtype=np.uint64)[:, None]
    x = np.arange(L, dtype=np.uint64)[None, :]
    ctr0 = ((y * wpr + x // 32) * 4 + (x % 32) // 8).astype(np.uint32)
    comp = ((x % 32) // 2) % 4
    shape = (B, L, L)
    lat = (np.uint64(lattice_base) + np.arange(B, dtype=np.uint64))[:, None, None].astype(np.uint32)
    out = philox4x32_10([np.broadcast_to(ctr0, shape), np.full(shape, step, np.uint32),
                         np.full(shape, colour, np.uint32), np.full(shape, TAG, np.uint32)],
                        [np.full(shape, seed, np.uint32), np.broadcast_to(lat, shape)])
    return np.choose(np.broadcast_to(comp, shape).astype(np.int64), out)


def run(spins, temperatures, seed, lattice_base=0, step0=0):
    """spins int8 [B, L, L]; temperatures [K] or [K, B] -> (spins, n_up int32 [K, B], bond_sum int32 [K, B])"""
    spins = spins.astype(np.int8).copy()
    B, L, _ = spins.shape
    temps = np.asarray(temperatures, dtype=np.float64)
    if temps.ndim == 1:
        temps = np.repeat(temps[:, None], B, axis=1)
    K = temps.shape[0]
    colour = (np.arange(L)[:, None] + np.arange(L)[None, :]) % 2
    n_up = np.zeros((K, B), np.int32)
    bond_sum = np.zeros((K, B), np.int32)
    for k in range(K):
        thr2 = np.array([threshold(2, t) for t in temps[k]], np.uint64)[:, None, None]
        thr4 = np.array([threshold(4, t) for t in temps[k]], np.uint64)[:, None, None]
        for c in (0, 1):
            h = local_field(spins)
            flip = accept(h, words(B, L, seed, lattice_base, step0 + k, c), thr2, thr4) & (colour == c)
            spins = np.where(flip, 1 - spins, spins).astype(np.int8)
        n_up[k] = spins.reshape(B, -1).sum(axis=1)
        bond_sum[k] = local_field(spins).reshape(B, -1).sum(axis=1) // 2
    return spins, n_up, bond_sum
