"""GPU: Ising temperature sweeps -- per-lattice temperature schedules for the MF-Q kernels (K6, the generic K6r, K6s),
the Metropolis chain K8 against its numpy restatement (tests/metropolis_ref.py) and Onsager's magnetisation, and the
`ising_sweep` command."""
import csv
import math
import os
import sys

import numpy as np
import pytest

from conftest import REPO

sys.path.insert(0, os.path.join(REPO, "oracle"))
import ising_oracle  # noqa: E402
import metropolis_ref  # noqa: E402

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _schedules(K, B):
    """[K, B]: a different, slowly changing schedule per lattice (float64; cast by IsingMFQ)"""
    k = np.arange(K, dtype=np.float64)[:, None]
    b = np.arange(B, dtype=np.float64)[None, :]
    return torch.from_numpy(0.45 + 0.35 * b + 0.4 * np.abs(np.sin(0.3 * k + b)))


def _batch_equals_singles(L, B, K, dtype, resident, masked, seed=21):
    from mfmarl_b200 import IsingMFQ
    rng = np.random.RandomState(L + B)
    spins = torch.from_numpy(rng.randint(0, 2, size=(B, L, L)).astype(np.int8))
    temps = _schedules(K, B)
    masks = None
    if masked:
        gen = torch.Generator(device="cuda"); gen.manual_seed(L)
        masks = (torch.rand((K, B, L * L), generator=gen, device="cuda") < 0.6).to(torch.uint8).contiguous()
    batch = IsingMFQ(B, L, dtype=dtype, seed=seed, spins=spins)
    n_up, rsum = batch.run(temps, resident=resident, update_mask=masks)
    for b in range(B):
        one = IsingMFQ(1, L, dtype=dtype, seed=seed, lattice_base=b, spins=spins[b:b + 1])
        n1, r1 = one.run(temps[:, b].tolist(), resident=resident,
                         update_mask=None if masks is None else masks[:, b:b + 1].contiguous())
        assert torch.equal(batch.spins[b:b + 1], one.spins), b
        assert torch.equal(batch.Q[b:b + 1], one.Q), b
        assert torch.equal(n_up[:, b:b + 1], n1), b
        assert torch.equal(rsum[:, b:b + 1], r1), b
    return batch


@pytest.mark.parametrize("L,dtype,resident,masked", [
    (20, torch.float32, False, False), (20, torch.float64, False, True), (33, torch.float32, False, True),
    (33, torch.float64, False, False),                                             # K6, streaming
    (20, torch.float32, True, False), (20, torch.float32, True, True), (48, torch.float32, True, False),
    (48, torch.float32, True, True), (20, torch.float64, True, True),               # generic K6r
    (64, torch.float32, True, False), (64, torch.float32, True, True), (128, torch.float32, True, False),
    (128, torch.float32, True, True), (256, torch.float32, True, False), (256, torch.float32, True, True),
    (512, torch.float32, True, False), (512, torch.float32, True, True),            # K6s
])
def test_per_lattice_schedules_equal_each_lattice_run_alone(L, dtype, resident, masked):
    """B lattices with B different schedules in one call == each lattice alone (lattice_base = b) with its own
    schedule, bit for bit: spins, Q, and n_up and reward_sum of every sweep"""
    B = 3 if L <= 256 else 2
    K = 9 if L <= 128 else 5
    batch = _batch_equals_singles(L, B, K, dtype, resident, masked)
    assert not torch.equal(batch.spins[0], batch.spins[1])


def _handover_batch(L):
    """a batch large enough that every K6s slot sweeps at least two lattices one after the other.  K6s runs
    n_slots <= n_SM * (co-resident CTAs per SM) / (strips per lattice) slots; the CTAs per SM are bounded by the
    threads per SM (2 L threads per CTA below side 512, 1024 at 512; 16 or 8 rows per strip)."""
    prop = torch.cuda.get_device_properties(0)
    threads, strips = (2 * L, L // 16) if L < 512 else (1024, 64)
    per_sm = min(32, getattr(prop, "max_threads_per_multi_processor", 2048) // threads)
    bound = prop.multi_processor_count * per_sm // strips
    return 2 * bound + 1


def _distinct_columns(K, B):
    """[K, B] with every column different from every other (the golden-ratio sequence never repeats)"""
    k = np.arange(K, dtype=np.float64)[:, None]
    b = np.arange(B, dtype=np.float64)[None, :]
    return torch.from_numpy(0.4 + 1.6 * ((b * 0.6180339887) % 1.0) + 0.2 * np.abs(np.sin(0.3 * k + b)))


def _handover_equals_streaming(L, K, masked):
    from mfmarl_b200 import IsingMFQ
    B = _handover_batch(L)
    gen = torch.Generator(device="cuda"); gen.manual_seed(L + K)
    spins = torch.randint(0, 2, (B, L, L), generator=gen, device="cuda", dtype=torch.int8)
    masks = (torch.rand((K, B, L * L), generator=gen, device="cuda") < 0.6).to(torch.uint8).contiguous() if masked else None
    temps = _distinct_columns(K, B)
    res, stream = IsingMFQ(B, L, seed=5, spins=spins), IsingMFQ(B, L, seed=5, spins=spins)
    n_r, r_r = res.run(temps, resident=True, update_mask=masks)
    n_s, r_s = stream.run(temps, resident=False, update_mask=masks)      # K6: one launch per sweep, [B] per launch
    assert torch.equal(res.spins, stream.spins) and torch.equal(res.Q, stream.Q)
    assert torch.equal(n_r, n_s) and torch.equal(r_r, r_s)
    for b in (B // 2 + 1, B - 1):                                          # handed-over lattices, each run alone
        one = IsingMFQ(1, L, seed=5, lattice_base=b, spins=spins[b:b + 1])
        n1, _ = one.run(temps[:, b].tolist(), resident=True,
                        update_mask=None if masks is None else masks[:, b:b + 1].contiguous())
        assert torch.equal(res.spins[b:b + 1], one.spins) and torch.equal(res.Q[b:b + 1], one.Q)
        assert torch.equal(n_r[:, b:b + 1], n1)


@pytest.mark.parametrize("L,masked", [(64, False), (128, True), (256, False), (256, True), (512, False)])
def test_per_lattice_schedules_across_lattice_hand_overs(L, masked):
    """K6s with more lattices than slots: every slot refills its temperature table from the column of each lattice it
    takes up.  The batch equals K streaming launches with the same table, and handed-over lattices equal themselves
    run alone."""
    _handover_equals_streaming(L, 7, masked)


def test_per_lattice_schedules_across_the_sweep_chunk_boundary():
    """K6s runs at most 4096 sweeps per launch: a 4100-sweep run is two launches, the second one's table offset by
    4096 rows of n_lattices temperatures -- here with hand-overs in both launches"""
    _handover_equals_streaming(512, 4100, False)


@pytest.mark.parametrize("L,resident", [(33, False), (20, True), (48, True), (64, True), (256, True), (512, True)])
def test_identical_rows_equal_the_shared_schedule(L, resident):
    from mfmarl_b200 import IsingMFQ
    B, K = 3, 6
    sched = [0.9, 0.8, 0.7, 1.5, 2.5, 0.6]
    a, b = IsingMFQ(B, L, seed=8), IsingMFQ(B, L, seed=8)
    n_a, r_a = a.run(torch.tensor(sched)[:, None].repeat(1, B), resident=resident)
    n_b, r_b = b.run(sched, resident=resident)
    assert torch.equal(a.spins, b.spins) and torch.equal(a.Q, b.Q)
    assert torch.equal(n_a, n_b) and torch.equal(r_a, r_b)


@pytest.mark.parametrize("resident", [False, True])
def test_fp64_per_lattice_matches_the_oracle(resident):
    """per-lattice temperatures through the fp64 kernels against ising_oracle.step with the same temperatures and
    injected uniforms"""
    from mfmarl_b200 import IsingMFQ
    B, L, K = 4, 20, 15
    rng = np.random.RandomState(3)
    spins = rng.randint(0, 2, size=(B, L, L)).astype(np.int8)
    temps = _schedules(K, B).numpy()
    u = rng.random_sample((K, B, L * L))
    m = IsingMFQ(B, L, dtype=torch.float64, spins=torch.from_numpy(spins))
    n_up, rsum = m.run(torch.from_numpy(temps), uniforms=torch.from_numpy(u).cuda(), resident=resident)
    Q = np.zeros((B, 5, L * L, 2))
    for k in range(K):
        spins, Q, info = ising_oracle.step(spins, Q, temps[k][:, None], 0.1, u[k])
        assert np.abs(u[k] - info["threshold"]).min() > 1e-12
        assert np.array_equal(n_up[k].cpu().numpy(), info["n_up"])
        assert np.array_equal(rsum[k].cpu().numpy(), info["reward_sum"])
    assert np.array_equal(m.spins.cpu().numpy(), spins)
    np.testing.assert_allclose(m.Q.cpu().numpy(), Q, rtol=1e-13, atol=1e-15)


@pytest.mark.parametrize("var,value", [("MFMARL_ISING_PERSIST", "1"), ("MFMARL_ISING_RPT", "4"),
                                       ("MFMARL_ISING_PERSIST", "0")])
def test_overrides_without_per_lattice_tables_refuse(var, value, monkeypatch):
    from mfmarl_b200 import IsingMFQ
    monkeypatch.setenv(var, value)
    m = IsingMFQ(2, 256, seed=3)
    before = (m.spins.clone(), m.Q.clone())
    with pytest.raises(RuntimeError, match="%s=%s" % (var, value)):
        m.run(_schedules(4, 2), resident=True)
    torch.cuda.synchronize()
    assert torch.equal(m.spins, before[0]) and torch.equal(m.Q, before[1]) and m.t == 0
    m.run([0.8] * 4, resident=True)                      # the shared schedule still takes the override


# ---- K8 --------------------------------------------------------------------------------------------------------------

def _mcmc_temps(K, B):
    grid = np.array([0.6, 1.0, 1.1346, 1.5, 2.5, 0.3])
    return grid[(np.arange(K)[:, None] + 2 * np.arange(B)[None, :]) % len(grid)]


@pytest.mark.parametrize("L,B", [(2, 3), (4, 3), (20, 4), (64, 3), (256, 2), (512, 2)])
def test_metropolis_equals_the_numpy_reference(L, B):
    """20 sweeps in two launches, temperatures differing per lattice and per sweep: spins after every launch, n_up and
    the bond sum of every sweep equal the reference bit for bit"""
    from mfmarl_b200 import IsingMetropolis
    seed, base = 99, 7
    rng = np.random.RandomState(L)
    spins = rng.randint(0, 2, size=(B, L, L)).astype(np.int8)
    temps = _mcmc_temps(20, B)
    chain = IsingMetropolis(B, L, seed=seed, lattice_base=base, spins=torch.from_numpy(spins))
    step = 0
    for part in (temps[:10], temps[10:]):
        n_up, bond = chain.run(part)
        spins, want_up, want_bond = metropolis_ref.run(spins, part, seed, base, step)
        step += len(part)
        assert np.array_equal(chain.spins.cpu().numpy(), spins)
        assert np.array_equal(n_up.cpu().numpy(), want_up)
        assert np.array_equal(bond.cpu().numpy(), want_bond)


def test_metropolis_one_launch_equals_two():
    from mfmarl_b200 import IsingMetropolis
    temps = _mcmc_temps(30, 5)
    a, b = IsingMetropolis(5, 64, seed=4), IsingMetropolis(5, 64, seed=4)
    n_a, e_a = a.run(temps)
    n_b1, e_b1 = b.run(temps[:13])
    n_b2, e_b2 = b.run(temps[13:])
    assert torch.equal(a.spins, b.spins)
    assert torch.equal(n_a, torch.cat([n_b1, n_b2])) and torch.equal(e_a, torch.cat([e_b1, e_b2]))


def test_metropolis_does_not_depend_on_sharding():
    from mfmarl_b200 import IsingMetropolis
    rng = np.random.RandomState(2)
    spins = torch.from_numpy(rng.randint(0, 2, size=(4, 48, 48)).astype(np.int8))
    temps = _mcmc_temps(25, 4)
    full = IsingMetropolis(4, 48, seed=6, spins=spins)
    shard = IsingMetropolis(2, 48, seed=6, lattice_base=2, spins=spins[2:])
    n_f, e_f = full.run(temps)
    n_s, e_s = shard.run(temps[:, 2:])
    assert torch.equal(full.spins[2:], shard.spins)
    assert torch.equal(n_f[:, 2:], n_s) and torch.equal(e_f[:, 2:], e_s)


def onsager(T):
    """spontaneous magnetisation of the square-lattice Ising model with coupling 1/2 (Tc = 1 / ln(1 + sqrt 2))"""
    return (1.0 - math.sinh(1.0 / T) ** -4) ** 0.125 if T < 1.0 / math.log(1 + math.sqrt(2)) else 0.0


@pytest.mark.parametrize("T", [0.8, 1.0, 2.0])
def test_metropolis_magnetisation_follows_onsager(T, capsys):
    """64 lattices of 256 x 256 from all up, 2000 sweeps of burn-in, then the mean of |m| over 2000 sweeps"""
    from mfmarl_b200 import IsingMetropolis
    B, L = 64, 256
    chain = IsingMetropolis(B, L, seed=17, spins=torch.ones((B, L, L), dtype=torch.int8))
    chain.run([T] * 2000)
    n_up, bond = chain.run([T] * 2000)
    absm = float(((2 * n_up.to(torch.float64) - L * L).abs() / (L * L)).mean())
    with capsys.disabled():
        print("\n[K8 256^2 T=%.2f] <|m|> = %.5f, Onsager %.5f, bond energy per site %.4f"
              % (T, absm, onsager(T), -float(bond.to(torch.float64).mean()) / (L * L)))
    if T < 1.1:
        assert abs(absm - onsager(T)) < 0.005, (absm, onsager(T))
    else:
        assert absm < 0.05, absm


@pytest.mark.parametrize("side,T", [(5, 1.0), (0, 1.0), (514, 1.0), (20, 0.0), (20, -1.0), (20, float("inf")),
                                    (20, float("nan"))])
def test_metropolis_rejects_bad_input_before_launching(side, T):
    from mfmarl_b200 import IsingMetropolis
    from mfmarl_b200.lib import load_library
    lib = load_library()
    B, K = 2, 3
    spins = torch.zeros((B, max(side, 1), max(side, 1)), dtype=torch.int8, device="cuda")
    n_up = torch.full((K, B), -7, dtype=torch.int32, device="cuda")
    temps = np.full((K, B), 1.0)
    temps[1, 1] = T
    import ctypes
    rc = lib.mfi_metropolis(B, side, K, ctypes.c_void_p(spins.data_ptr()), temps.ctypes.data_as(ctypes.c_void_p),
                            1, 0, 0, ctypes.c_void_p(n_up.data_ptr()), None, None)
    assert rc == -1
    msg = lib.mfb_last_error().decode()
    assert msg.startswith("mfi_metropolis: ") and ("side" in msg if side != 20 else "temperature" in msg), msg
    torch.cuda.synchronize()
    assert int(spins.abs().sum()) == 0 and bool((n_up == -7).all())
    if side == 20:
        with pytest.raises(RuntimeError, match="temperature"):
            IsingMetropolis(B, side, spins=spins).run(temps)


# ---- the sweep command -------------------------------------------------------------------------------------------

def test_sweep_table_and_its_mfq_column_equal_separate_runs(tmp_path):
    from mfmarl_b200 import IsingMFQ, ising_sweep
    from mfmarl_b200.ising import temperature_schedule
    temps, R, L, K, W = [0.5, 1.0, 2.0], 8, 20, 400, 100
    out = tmp_path / "sweep.csv"
    tables = ising_sweep.sweep(["--temperatures", "0.5,1.0,2.0", "--replicas", str(R), "--side", str(L),
                                "--sweeps", str(K), "--window", str(W), "--method", "both", "-dg", "20",
                                "-dr", "0.9", "--out", str(out)])
    assert set(tables) == {"mfq", "mcmc"}
    for t in tables.values():
        assert t.shape == (3, 5) and np.array_equal(t[:, 0], temps) and np.isfinite(t).all()
    rows = list(csv.reader(open(out)))
    assert rows[0] == ["method"] + ising_sweep.COLUMNS and len(rows) == 1 + 2 * 3
    # MF-Q: the batch == one IsingMFQ per temperature at that floor, R lattices each with their lattice_base
    spins0 = IsingMFQ(3 * R, L, seed=13).spins
    ups, rsums = [], []
    for j, T in enumerate(temps):
        m = IsingMFQ(R, L, seed=13, lattice_base=j * R, spins=spins0[j * R:(j + 1) * R])
        n_up, rsum = m.run(temperature_schedule(0, K, 0.9, 20, T))
        ups.append(n_up); rsums.append(rsum)
    want = ising_sweep.summarise(temps, R, L, torch.cat(ups, dim=1), torch.cat(rsums, dim=1), W)
    assert np.array_equal(tables["mfq"], want)
    # physics at the two ends: MCMC ordered at 0.5, disordered at 2.0
    assert tables["mcmc"][0, 1] > 0.95 and tables["mcmc"][2, 1] < 0.5
