"""CPU: the numpy Swendsen-Wang reference (tests/swendsen_wang_ref.py) that K9 is compared with on the GPU -- its
integer thresholds and bond decisions, hand-derived sweeps, the exact stationarity of the algorithm on the 2 x 2 torus,
and chains of the integer reference against exact enumeration of a 3 x 3 (odd) and a 4 x 4 torus."""
import itertools
import math

import numpy as np
import pytest

import swendsen_wang_ref as swr
from philox_ref import philox4x32_10

TC = 1.0 / math.log(1.0 + math.sqrt(2.0))
TOP = 2 ** 31


def test_threshold_is_the_floor_of_the_c_library_exp():
    for T in (0.05, 0.3, 0.8, 1.0, TC, 2.0, 7.5, 1e3, 1e17):
        want = min(math.floor((1.0 - math.exp(-1.0 / T)) * 2 ** 32), 2 ** 32 - 1)
        assert swr.threshold(T) == want and 0 <= want < 2 ** 32
    assert swr.threshold(1.0) == 2714937127                 # floor((1 - e^-1) * 2^32) = floor(2714937127.298)
    assert swr.threshold(1e-3) == 2 ** 32 - 1               # exp(-1000) = 0: clamped to the largest word
    assert swr.threshold(1e20) == 0                         # exp(-1e-20) rounds to 1: no bond is ever active


def test_bond_decision_at_the_threshold():
    for T in (0.5, TC, 3.0):
        thr = swr.threshold(T)
        assert swr.active(True, thr - 1, thr)
        assert not swr.active(True, thr, thr)
        assert swr.active(True, 0, thr)
        for word in (0, thr - 1, thr, 2 ** 32 - 1):          # anti-aligned: never
            assert not swr.active(False, word, thr)
    assert not swr.active(True, 2 ** 32 - 1, 2 ** 32 - 1)   # even at T -> 0 the largest word stays inactive


def test_counter_layout():
    """bond words: output 2 (i & 1) / 2 (i & 1) + 1 of counter (i >> 1, step, 0, 3); flip word: output i & 3 of counter
    (i >> 2, step, 1, 3); key (seed, lattice_base + lattice)"""
    B, L, seed, base, step = 2, 5, 77, 9, 123
    right, down = swr.bond_words(B, L, seed, base, step)
    flip = swr.flip_words(B, L, seed, base, step)
    for b in range(B):
        for i in (0, 1, 7, 24):
            r = [int(w) for w in philox4x32_10([i >> 1, step, 0, 3], [seed, base + b])]
            assert (right[b, i], down[b, i]) == (r[2 * (i & 1)], r[2 * (i & 1) + 1])
            f = [int(w) for w in philox4x32_10([i >> 2, step, 1, 3], [seed, base + b])]
            assert flip[b, i] == f[i & 3]


def _seed_whose_root_flips(flips, L=6, step=0):
    """first seed whose site-0 flip word in `step` has its top bit set (flips) or clear, with no bond word 2^32 - 1"""
    for seed in range(1000):
        right, down = swr.bond_words(1, L, seed, 0, step)
        if (right == 2 ** 32 - 1).any() or (down == 2 ** 32 - 1).any():
            continue
        if (swr.flip_words(1, L, seed, 0, step)[0, 0] >= TOP) == flips:
            return seed
    raise AssertionError("no seed")


@pytest.mark.parametrize("flips", [True, False])
def test_cold_aligned_lattice_is_one_cluster_flipping_on_root_zero(flips):
    """T = 1e-3 (threshold 2^32 - 1), all up: every bond is active, the lattice is one cluster rooted at 0, and it flips
    as a whole iff site 0's flip word has its top bit set"""
    L = 6
    seed = _seed_whose_root_flips(flips, L)
    spins, n_up, bond = swr.run(np.ones((1, L, L), np.int8), [1e-3], seed)
    want = 0 if flips else 1
    assert (spins == want).all()
    assert n_up.tolist() == [[want * L * L]] and bond.tolist() == [[2 * L * L]]
    right, down = swr.bond_words(1, L, seed, 0, 0)
    thr = swr.threshold(1e-3)
    roots = swr.cluster_roots(swr.active(True, right, thr), swr.active(True, down, thr), L)
    assert (roots == 0).all()


def test_hot_lattice_flips_every_site_on_its_own_word():
    """T = 1e20: no bond is active, every site is its own root and flips iff its own flip word has its top bit set"""
    B, L, seed = 3, 7, 5
    rng = np.random.RandomState(1)
    spins = rng.randint(0, 2, size=(B, L, L)).astype(np.int8)
    out, _, _ = swr.run(spins, [1e20], seed, lattice_base=4, step0=11)
    flip = (swr.flip_words(B, L, seed, 4, 11) >= TOP).astype(np.int8).reshape(B, L, L)
    assert np.array_equal(out, spins ^ flip)
    assert 0 < flip.sum() < flip.size


def test_side_2_doubled_bonds_are_separate_draws():
    """at L = 2, site 0's right bond and site 1's right bond join the same pair (0, 1) but are two bonds with their own
    words: either one alone joins the pair, and 0 and 1 flip together or apart accordingly"""
    spins = np.ones((1, 2, 2), np.int8)
    thr = [TOP]
    lo, hi = np.uint32(0), np.uint32(2 ** 32 - 1)
    no_down = np.full((1, 4), hi, np.uint32)
    flip = np.array([[TOP, 0, 0, 0]], np.uint32)            # only root 0 flips
    for right, joined in (([lo, hi, hi, hi], True), ([hi, lo, hi, hi], True), ([hi, hi, hi, hi], False)):
        out = swr.sweep(spins, thr, np.array([right], np.uint32), no_down, flip)
        assert out.reshape(-1).tolist() == ([0, 0, 1, 1] if joined else [0, 1, 1, 1]), right
    # and the two words of the pair's right bonds come from different output words of one counter
    r, _ = swr.bond_words(1, 2, 3, 0, 0)
    words = [int(w) for w in philox4x32_10([0, 0, 0, 3], [3, 0])]
    assert (r[0, 0], r[0, 1]) == (words[0], words[2]) and r[0, 0] != r[0, 1]


# ---- exact stationarity on the 2 x 2 torus --------------------------------------------------------------------------

def _bonds(L):
    rt, dn = swr.neighbours(L)
    return [(i, int(rt[i])) for i in range(L * L)] + [(i, int(dn[i])) for i in range(L * L)]


def _components(n, edges):
    parent = list(range(n))

    def find(x):
        while parent[x] != x:
            x = parent[x]
        return x
    for a, b in edges:
        ra, rb = find(a), find(b)
        if ra != rb:
            parent[max(ra, rb)] = min(ra, rb)
    return [find(i) for i in range(n)]


def sw_transition_matrix(L, T):
    """the exact Swendsen-Wang kernel with real-valued p = 1 - e^(-1/T) on the L x L torus (2^N states)"""
    N, p = L * L, 1.0 - math.exp(-1.0 / T)
    bonds = _bonds(L)
    P = np.zeros((2 ** N, 2 ** N))
    for s in range(2 ** N):
        spin = [(s >> i) & 1 for i in range(N)]
        aligned = [e for e in bonds if spin[e[0]] == spin[e[1]]]
        for mask in range(2 ** len(aligned)):
            on = [aligned[j] for j in range(len(aligned)) if (mask >> j) & 1]
            w_bonds = p ** len(on) * (1.0 - p) ** (len(aligned) - len(on))
            roots = _components(N, on)
            clusters = sorted(set(roots))
            for flips in range(2 ** len(clusters)):
                flipped = {c for j, c in enumerate(clusters) if (flips >> j) & 1}
                t = sum((spin[i] ^ (roots[i] in flipped)) << i for i in range(N))
                P[s, t] += w_bonds / 2 ** len(clusters)
    return P


def boltzmann(L, T):
    N = L * L
    states = np.array([[(s >> i) & 1 for i in range(N)] for s in range(2 ** N)], np.int8).reshape(-1, L, L)
    w = np.exp(swr.bond_sum(states) / (2.0 * T))
    return w / w.sum()


@pytest.mark.parametrize("T", [0.5, TC, 3.0])
def test_2x2_kernel_is_stationary_and_reversible(T):
    P = sw_transition_matrix(2, T)
    pi = boltzmann(2, T)
    assert np.allclose(P.sum(axis=1), 1.0, rtol=0, atol=1e-12)
    assert np.abs(pi @ P - pi).max() < 1e-12
    flow = pi[:, None] * P
    assert np.abs(flow - flow.T).max() < 1e-12


# ---- sampling: chains of the integer reference against exact enumeration ---------------------------------------------

def exact_averages(L, T):
    """Boltzmann averages of the bond sum and |m| over all 2^(L*L) states"""
    N = L * L
    states = np.array(list(itertools.product((0, 1), repeat=N)), np.int8).reshape(-1, L, L)
    bond = swr.bond_sum(states)
    absm = np.abs(2 * states.reshape(len(states), -1).sum(axis=1) - N) / N
    w = np.exp((bond - bond.max()) / (2.0 * T))
    return float((w * bond).sum() / w.sum()), float((w * absm).sum() / w.sum())


@pytest.mark.parametrize("L,T", [(3, 1.0), (3, TC), (3, 2.0), (4, 1.0), (4, TC), (4, 2.0)])
def test_chain_samples_the_boltzmann_distribution(L, T):
    """64 independent chains from random starts, 20 sweeps of burn-in, then 300 sweeps: the mean over chains of each
    chain's time average of the bond sum and of |m| lies within 5 standard errors of the exact average"""
    B, burn, K = 64, 20, 300
    rng = np.random.RandomState(5 + L)
    spins = rng.randint(0, 2, size=(B, L, L)).astype(np.int8)
    spins, _, _ = swr.run(spins, [T] * burn, seed=11)
    _, n_up, bond = swr.run(spins, [T] * K, seed=11, step0=burn)
    absm = np.abs(2 * n_up.astype(np.float64) - L * L) / (L * L)
    want_bond, want_m = exact_averages(L, T)
    for series, want in ((bond.astype(np.float64), want_bond), (absm, want_m)):
        per_chain = series.mean(axis=0)
        mean, se = per_chain.mean(), per_chain.std(ddof=1) / math.sqrt(B)
        assert abs(mean - want) < 5 * se, (L, T, mean, se, want)
