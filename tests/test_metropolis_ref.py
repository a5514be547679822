"""CPU: the numpy Metropolis reference (tests/metropolis_ref.py) that K8 is compared with on the GPU -- its single-site
decisions, its integer thresholds, and its stationary distribution against exact enumeration of a 4 x 4 torus."""
import itertools
import math

import numpy as np
import pytest

import metropolis_ref as mr


def test_single_site_decisions_at_both_thresholds():
    T = 1.0
    thr2, thr4 = mr.threshold(2, T), mr.threshold(4, T)
    assert thr2 == 581260615 and thr4 == 78665070          # floor(e^-2 * 2^32), floor(e^-4 * 2^32)
    for h, thr in ((2, thr2), (4, thr4)):
        assert mr.accept(h, thr - 1, thr2, thr4)
        assert not mr.accept(h, thr, thr2, thr4)
        assert not mr.accept(h, 2 ** 32 - 1, thr2, thr4)
        assert mr.accept(h, 0, thr2, thr4)
    for h in (-4, -2, 0):                                   # downhill and neutral flips: always
        assert mr.accept(h, 2 ** 32 - 1, thr2, thr4)
    # h = 2 uses thr2, h = 4 thr4: a word between them flips an h = 2 site and keeps an h = 4 one
    assert mr.accept(2, thr4, thr2, thr4) and not mr.accept(4, thr4, thr2, thr4)


def test_thresholds_are_the_floor_of_the_c_library_exp():
    for T in (0.05, 0.3, 0.8, 1.0, 1.1346, 2.0, 7.5, 1e3, 1e17):
        for h in (2, 4):
            want = min(math.floor(math.exp(-h / T) * 2 ** 32), 2 ** 32 - 1)
            assert mr.threshold(h, T) == want
            assert 0 <= want < 2 ** 32
    assert mr.threshold(2, 1e17) == 2 ** 32 - 1             # exp rounds to 1: clamped to the largest word
    assert mr.threshold(4, 0.05) == 0                        # exp(-80) * 2^32 < 1: never uphill


def test_one_sweep_by_hand():
    """2 x 2 torus, all up but site (0, 0): in the even half (0, 0) has h = -4 and flips whatever its draw; (1, 1) is
    even too, it sees (0, 1), (1, 0) twice each, all up, so h = 4 and at T -> 0 it stays.  The lattice is all up."""
    spins = np.array([[[0, 1], [1, 1]]], np.int8)
    out, n_up, bond = mr.run(spins, [0.01], seed=3)
    assert out.tolist() == [[[1, 1], [1, 1]]]
    assert n_up.tolist() == [[4]] and bond.tolist() == [[8]]          # 2N = 8 bonds, all aligned


def exact_averages(L, T):
    """Boltzmann averages of the bond sum and |m| over all 2^(L*L) states, weight exp(bond_sum / (2 T))"""
    N = L * L
    states = np.array(list(itertools.product((0, 1), repeat=N)), np.int8).reshape(-1, L, L)
    bond = mr.local_field(states).reshape(len(states), -1).sum(axis=1) // 2
    absm = np.abs(2 * states.reshape(len(states), -1).sum(axis=1) - N) / N
    w = np.exp((bond - bond.max()) / (2.0 * T))
    return float((w * bond).sum() / w.sum()), float((w * absm).sum() / w.sum())


@pytest.mark.parametrize("T", [1.0, 2.0])
def test_chain_samples_the_boltzmann_distribution_of_a_4x4_torus(T):
    """64 independent chains from random starts, 200 sweeps of burn-in, then 2500 sweeps: the mean over chains of each
    chain's time average of the bond sum and of |m| lies within 5 standard errors of the exact average"""
    L, B, burn, K = 4, 64, 200, 2500
    rng = np.random.RandomState(5)
    spins = rng.randint(0, 2, size=(B, L, L)).astype(np.int8)
    spins, _, _ = mr.run(spins, [T] * burn, seed=11)
    _, n_up, bond = mr.run(spins, [T] * K, seed=11, step0=burn)
    absm = np.abs(2 * n_up.astype(np.float64) - L * L) / (L * L)
    want_bond, want_m = exact_averages(L, T)
    for series, want in ((bond.astype(np.float64), want_bond), (absm, want_m)):
        per_chain = series.mean(axis=0)
        mean, se = per_chain.mean(), per_chain.std(ddof=1) / math.sqrt(B)
        assert abs(mean - want) < 5 * se, (T, mean, se, want)
