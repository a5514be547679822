"""numpy restatement of K9 (`mfi_swendsen_wang`, csrc/ising_cluster.cu): Swendsen-Wang cluster updates on L x L tori,
with the Philox keys, counters and integer thresholds documented in include/mfmarl_batched.h.  Clusters come from
scipy's connected components of the block-diagonal bond graph of all lattices and are labelled by their smallest flat
site index, with no union-find involved: an independent statement of the kernel's canonical-label rule.  Test
infrastructure: the GPU kernel is compared with it bit for bit."""
import math

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from philox_ref import philox4x32_10

TAG = 3     # counter word 3 of K9's draws (MF-Q uses 0 and 1, K8 uses 2)


def threshold(T):
    """a bond between aligned spins is active when its 32-bit Philox word is below this integer"""
    return min(int(math.floor((1.0 - math.exp(-1.0 / T)) * 2 ** 32)), 2 ** 32 - 1)


def active(aligned, word, thr):
    """the Fortuin-Kasteleyn decision for one bond (all arguments broadcastable)"""
    return np.asarray(aligned, bool) & (np.asarray(word, np.uint64) < np.asarray(thr, np.uint64))


def neighbours(L):
    """flat indices of every site's right and down neighbour, each [L * L]"""
    i = np.arange(L * L)
    x, y = i % L, i // L
    return y * L + (x + 1) % L, ((y + 1) % L) * L + x


def _philox(B, n_ctr, ctr1, ctr2, seed, lattice_base):
    """the 4 output words [4, B, n_ctr] of counters (c, ctr1, ctr2, TAG), c < n_ctr, under lattice b's key"""
    shape = (B, n_ctr)
    c0 = np.broadcast_to(np.arange(n_ctr, dtype=np.uint32)[None, :], shape)
    lat = (np.uint64(lattice_base) + np.arange(B, dtype=np.uint64)).astype(np.uint32)[:, None]
    return np.stack(philox4x32_10([c0, np.full(shape, ctr1, np.uint32), np.full(shape, ctr2, np.uint32),
                                   np.full(shape, TAG, np.uint32)],
                                  [np.full(shape, seed, np.uint32), np.broadcast_to(lat, shape)]))


def bond_words(B, L, seed, lattice_base, step):
    """(right, down) [B, N] uint32: the Philox word of every site's right and down bond in sweep `step`"""
    N = L * L
    out = _philox(B, (N + 1) // 2, step, 0, seed, lattice_base)          # [4, B, ceil(N / 2)]
    i = np.arange(N)
    return out[2 * (i & 1), :, i >> 1].T, out[2 * (i & 1) + 1, :, i >> 1].T


def flip_words(B, L, seed, lattice_base, step):
    """[B, N] uint32: the flip word every site would draw as a root in sweep `step`"""
    N = L * L
    out = _philox(B, (N + 3) // 4, step, 1, seed, lattice_base)
    i = np.arange(N)
    return out[i & 3, :, i >> 2].T


def cluster_roots(active_right, active_down, L):
    """active_* bool [B, N] -> [B, N] int64: the smallest flat index of each site's cluster"""
    B, N = active_right.shape
    rt, dn = neighbours(L)
    off = (np.arange(B) * N)[:, None]
    src = np.concatenate([(np.arange(N)[None, :] + off)[active_right], (np.arange(N)[None, :] + off)[active_down]])
    dst = np.concatenate([(rt[None, :] + off)[active_right], (dn[None, :] + off)[active_down]])
    graph = coo_matrix((np.ones(len(src), np.int8), (src, dst)), shape=(B * N, B * N))
    n_comp, comp = connected_components(graph, directed=False)
    smallest = np.full(n_comp, B * N, np.int64)
    np.minimum.at(smallest, comp, np.arange(B * N))
    return (smallest[comp] - np.repeat(np.arange(B) * N, N)).reshape(B, N)


def bond_sum(spins):
    """sum over the 2N bonds of sigma_i sigma_j, int spins [B, L, L] in {0, 1} -> [B]"""
    s = 2 * spins.astype(np.int64) - 1
    return (s * np.roll(s, -1, -1) + s * np.roll(s, -1, -2)).reshape(len(s), -1).sum(axis=1)


def sweep(spins, thr, right_words, down_words, flip_words_):
    """one sweep from given words: spins int8 [B, L, L], thr [B] -> new spins.  Exposed for hand-derived tests."""
    B, L, _ = spins.shape
    flat = spins.reshape(B, -1).astype(np.int8)
    rt, dn = neighbours(L)
    thr = np.asarray(thr, np.uint64)[:, None]
    act_r = active(flat == flat[:, rt], right_words, thr)
    act_d = active(flat == flat[:, dn], down_words, thr)
    roots = cluster_roots(act_r, act_d, L)
    flip = (np.take_along_axis(flip_words_, roots, axis=1) >> np.uint32(31)).astype(np.int8)
    return (flat ^ flip).reshape(B, L, L)


def run(spins, temperatures, seed, lattice_base=0, step0=0):
    """spins int8 [B, L, L]; temperatures [K] or [K, B] -> (spins, n_up int32 [K, B], bond_sum int32 [K, B])"""
    spins = spins.astype(np.int8).copy()
    B, L, _ = spins.shape
    temps = np.asarray(temperatures, dtype=np.float64)
    if temps.ndim == 1:
        temps = np.repeat(temps[:, None], B, axis=1)
    K = temps.shape[0]
    n_up = np.zeros((K, B), np.int32)
    bonds = np.zeros((K, B), np.int32)
    for k in range(K):
        step = (step0 + k) & 0xFFFFFFFF
        right, down = bond_words(B, L, seed, lattice_base, step)
        spins = sweep(spins, [threshold(t) for t in temps[k]], right, down, flip_words(B, L, seed, lattice_base, step))
        n_up[k] = spins.reshape(B, -1).sum(axis=1)
        bonds[k] = bond_sum(spins)
    return spins, n_up, bonds
