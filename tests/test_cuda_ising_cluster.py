"""GPU: the Swendsen-Wang chain K9 (`mfi_swendsen_wang`, `IsingSwendsenWang`) against its numpy restatement
(tests/swendsen_wang_ref.py) bit for bit at odd and even sides, its invariance to launch splits and sharding, its
refusal of bad input, its physics (Onsager's magnetisation; agreement with K8 at Tc), and the sweep command's `sw`
method."""
import ctypes
import math

import numpy as np
import pytest
import torch

import swendsen_wang_ref

pytestmark = pytest.mark.gpu

TC = 1.0 / math.log(1.0 + math.sqrt(2.0))


def _temps(K, B):
    grid = np.array([0.6, 1e-3, TC, 1.5, 1e20, 2.5, 1.0])
    return grid[(np.arange(K)[:, None] + 3 * np.arange(B)[None, :]) % len(grid)]


@pytest.mark.parametrize("L", [2, 3, 4, 5, 20, 21, 31, 32, 33, 64, 100, 128, 255, 256])
def test_swendsen_wang_equals_the_numpy_reference(L):
    """20 sweeps in two launches from step0 = 5, lattice_base 7, temperatures differing per lattice and per sweep
    (1e-3, Tc and 1e20 among them): spins after every launch, n_up and the bond sum of every sweep equal the reference
    bit for bit"""
    from mfmarl_b200 import IsingSwendsenWang
    B = 3 if L <= 128 else 2
    seed, base, step = 99, 7, 5
    rng = np.random.RandomState(L)
    spins = rng.randint(0, 2, size=(B, L, L)).astype(np.int8)
    temps = _temps(20, B)
    chain = IsingSwendsenWang(B, L, seed=seed, lattice_base=base, spins=torch.from_numpy(spins))
    chain.t = step
    for part in (temps[:9], temps[9:]):
        n_up, bond = chain.run(part)
        spins, want_up, want_bond = swendsen_wang_ref.run(spins, part, seed, base, step)
        step += len(part)
        assert np.array_equal(chain.spins.cpu().numpy(), spins)
        assert np.array_equal(n_up.cpu().numpy(), want_up)
        assert np.array_equal(bond.cpu().numpy(), want_bond)


def test_swendsen_wang_one_launch_equals_two():
    from mfmarl_b200 import IsingSwendsenWang
    temps = _temps(30, 5)
    a, b = IsingSwendsenWang(5, 63, seed=4), IsingSwendsenWang(5, 63, seed=4)
    n_a, e_a = a.run(temps)
    n_b1, e_b1 = b.run(temps[:13])
    n_b2, e_b2 = b.run(temps[13:])
    assert torch.equal(a.spins, b.spins)
    assert torch.equal(n_a, torch.cat([n_b1, n_b2])) and torch.equal(e_a, torch.cat([e_b1, e_b2]))


def test_swendsen_wang_does_not_depend_on_sharding():
    from mfmarl_b200 import IsingSwendsenWang
    rng = np.random.RandomState(2)
    spins = torch.from_numpy(rng.randint(0, 2, size=(4, 47, 47)).astype(np.int8))
    temps = _temps(25, 4)
    full = IsingSwendsenWang(4, 47, seed=6, spins=spins)
    shard = IsingSwendsenWang(2, 47, seed=6, lattice_base=2, spins=spins[2:])
    n_f, e_f = full.run(temps)
    n_s, e_s = shard.run(temps[:, 2:])
    assert torch.equal(full.spins[2:], shard.spins)
    assert torch.equal(n_f[:, 2:], n_s) and torch.equal(e_f[:, 2:], e_s)


@pytest.mark.parametrize("L", [21, 256])
def test_swendsen_wang_without_outputs_leaves_the_same_spins(L):
    from mfmarl_b200 import IsingSwendsenWang
    from mfmarl_b200.lib import load_library
    lib = load_library()
    B, K = 3, 12
    temps = np.ascontiguousarray(_temps(K, B))
    a = IsingSwendsenWang(B, L, seed=8)
    spins = a.spins.clone()
    a.run(temps)
    rc = lib.mfi_swendsen_wang(B, L, K, ctypes.c_void_p(spins.data_ptr()), temps.ctypes.data_as(ctypes.c_void_p),
                               8, 0, 0, None, None, None)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(a.spins, spins)


def _bad_call(lib, B, side, K, spins, temps, n_up, null_spins=False, null_temps=False):
    return lib.mfi_swendsen_wang(B, side, K, None if null_spins else ctypes.c_void_p(spins.data_ptr()),
                                 None if null_temps else temps.ctypes.data_as(ctypes.c_void_p), 1, 0, 0,
                                 ctypes.c_void_p(n_up.data_ptr()), ctypes.c_void_p(n_up.data_ptr()), None)


@pytest.mark.parametrize("case", ["side1", "side0", "side257", "T0", "Tneg", "Tinf", "Tnan", "null_spins",
                                  "null_temps", "no_lattice", "no_sweep"])
def test_swendsen_wang_rejects_bad_input_before_launching(case):
    """refused with rc -1 and a prefixed message naming the problem; spins and outputs untouched"""
    from mfmarl_b200 import IsingSwendsenWang
    from mfmarl_b200.lib import load_library
    lib = load_library()
    B, K, side = 3, 4, {"side1": 1, "side0": 0, "side257": 257}.get(case, 21)
    spins = torch.full((B, max(side, 1), max(side, 1)), 1, dtype=torch.int8, device="cuda")
    n_up = torch.full((K, B), -7, dtype=torch.int32, device="cuda")
    temps = np.full((K, B), 1.0)
    temps[2, 1] = {"T0": 0.0, "Tneg": -1.0, "Tinf": float("inf"), "Tnan": float("nan")}.get(case, 1.0)
    rc = _bad_call(lib, 0 if case == "no_lattice" else B, side, 0 if case == "no_sweep" else K, spins, temps, n_up,
                   null_spins=case == "null_spins", null_temps=case == "null_temps")
    assert rc == -1
    msg = lib.mfb_last_error().decode()
    # the bad temperature is entry [2][1] of the [K][B] table: flat index 2 B + 1 = 7
    want = "side" if case.startswith("side") else "at index 7" if case.startswith("T") else \
        "null" if case.startswith("null") else "at least one"
    assert msg.startswith("mfi_swendsen_wang: ") and want in msg, msg
    torch.cuda.synchronize()
    assert bool((spins == 1).all()) and bool((n_up == -7).all())
    if case.startswith("T") or case == "side257":
        with pytest.raises(RuntimeError, match="temperature" if case.startswith("T") else "side"):
            IsingSwendsenWang(B, side, spins=spins).run(temps)
        assert bool((spins == 1).all())


# ---- physics -----------------------------------------------------------------------------------------------------------

def onsager(T):
    """spontaneous magnetisation of the square-lattice Ising model with coupling 1/2 (Tc = 1 / ln(1 + sqrt 2))"""
    return (1.0 - math.sinh(1.0 / T) ** -4) ** 0.125 if T < TC else 0.0


@pytest.mark.parametrize("T", [0.8, 1.0, 2.0])
def test_swendsen_wang_magnetisation_follows_onsager(T, capsys):
    """64 lattices of 128 x 128 from all up, 300 sweeps of burn-in, then the mean of |m| over 1000 sweeps"""
    from mfmarl_b200 import IsingSwendsenWang
    B, L = 64, 128
    chain = IsingSwendsenWang(B, L, seed=17, spins=torch.ones((B, L, L), dtype=torch.int8))
    chain.run([T] * 300)
    n_up, bond = chain.run([T] * 1000)
    absm = float(((2 * n_up.to(torch.float64) - L * L).abs() / (L * L)).mean())
    with capsys.disabled():
        print("\n[K9 128^2 T=%.2f] <|m|> = %.5f, Onsager %.5f, bond energy per site %.4f"
              % (T, absm, onsager(T), -float(bond.to(torch.float64).mean()) / (L * L)))
    if T < TC:
        assert abs(absm - onsager(T)) < 0.005, (absm, onsager(T))
    else:
        assert absm < 0.05, absm


def test_swendsen_wang_agrees_with_metropolis_at_tc(capsys):
    """L = 16 at Tc, 512 chains from all up: <|m|> and the bond energy per site of K9 (300 + 2000 sweeps) and of K8
    (3000 + 20000 sweeps) agree within 5 combined standard errors of the per-chain means"""
    from mfmarl_b200 import IsingMetropolis, IsingSwendsenWang
    B, L = 512, 16
    N = L * L
    stats = {}
    for name, cls, burn, K in (("K9", IsingSwendsenWang, 300, 2000), ("K8", IsingMetropolis, 3000, 20000)):
        chain = cls(B, L, seed=23, spins=torch.ones((B, L, L), dtype=torch.int8))
        chain.run([TC] * burn)
        n_up, bond = chain.run([TC] * K)
        absm = ((2 * n_up.to(torch.float64) - N).abs() / N).mean(dim=0)
        energy = (-bond.to(torch.float64) / N).mean(dim=0)
        stats[name] = [(float(x.mean()), float(x.std()) / math.sqrt(B)) for x in (absm, energy)]
    with capsys.disabled():
        print("\n[Tc, 16^2] K9 |m| %.5f +- %.5f  e %.5f +- %.5f;  K8 |m| %.5f +- %.5f  e %.5f +- %.5f"
              % tuple(v for name in ("K9", "K8") for pair in stats[name] for v in pair))
    for (m9, s9), (m8, s8) in zip(stats["K9"], stats["K8"]):
        assert abs(m9 - m8) < 5 * math.hypot(s9, s8), (m9, s9, m8, s8)


# ---- the sweep command -------------------------------------------------------------------------------------------

def test_sweep_command_sw_at_an_odd_side_equals_a_run_by_hand(tmp_path):
    from mfmarl_b200 import IsingSwendsenWang, ising_sweep
    temps, R, L, K, W = [0.5, 1.0, TC, 2.0, 3.0], 6, 21, 400, 200
    out = tmp_path / "sweep.csv"
    tables = ising_sweep.sweep(["--temperatures", ",".join(repr(t) for t in temps), "--replicas", str(R),
                                "--side", str(L), "--sweeps", str(K), "--window", str(W), "--method", "sw",
                                "--out", str(out)])
    assert set(tables) == {"sw"}
    t = tables["sw"]
    assert t.shape == (len(temps), 5) and np.array_equal(t[:, 0], temps) and np.isfinite(t).all()
    assert t[0, 1] > 0.95 and t[-1, 1] < 0.3                        # ordered and disordered ends
    rows = [r for r in open(out).read().splitlines()[1:]]
    assert len(rows) == len(temps) and all(r.startswith("sw,") for r in rows)
    chain = IsingSwendsenWang(len(temps) * R, L, seed=13, spins=torch.ones((len(temps) * R, L, L), dtype=torch.int8))
    n_up, bond = chain.run(np.repeat(np.repeat(np.asarray(temps), R)[None, :], K, axis=0))
    assert np.array_equal(t, ising_sweep.summarise(temps, R, L, n_up, bond, W))


def test_sweep_command_both_is_still_mfq_and_metropolis():
    from mfmarl_b200 import ising_sweep
    tables = ising_sweep.sweep(["--temperatures", "0.5,2.0", "--replicas", "2", "--side", "8", "--sweeps", "20",
                                "--window", "10", "--method", "both"])
    assert set(tables) == {"mfq", "mcmc"}
