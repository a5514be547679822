"""GPU: every shape class of the MF-Q Ising dispatch (tests/test_ising_shape_classes.py derives the classes from the
library and shares the representatives below) against the fp64 oracle (oracle/ising_oracle.py); the production
Philox draws, fp32 and fp64, pinned well below the top bit of each word; and K8 (Metropolis) on rows whose last word is
partial, at both threshold clamps, with K = 1 and without outputs, against tests/metropolis_ref.py."""
import ctypes
import math
import os
import sys

import numpy as np
import pytest

from conftest import REPO
from test_ising_shape_classes import (DRAW_SIDES, F32, F64, FP32_RESIDENT, FP32_STREAM, FP64_RESIDENT, FP64_STREAM)

sys.path.insert(0, os.path.join(REPO, "oracle"))
import ising_oracle  # noqa: E402
import metropolis_ref  # noqa: E402
from philox_ref import philox4x32_10  # noqa: E402

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TORCH_DTYPE = {F32: torch.float32, F64: torch.float64}


def _cluster(dtype, L):
    from mfmarl_b200.lib import load_library
    lib = load_library()
    lib.mfi_resident_cluster_size.argtypes = [ctypes.c_int, ctypes.c_int]
    return lib.mfi_resident_cluster_size(dtype, L)


def _schedules(K, B):
    """[K, B] float64: a different, slowly changing schedule per lattice, T in [0.45, 0.85 + 0.35 (B - 1)]"""
    k = np.arange(K, dtype=np.float64)[:, None]
    b = np.arange(B, dtype=np.float64)[None, :]
    return 0.45 + 0.35 * b + 0.4 * np.abs(np.sin(0.3 * k + b))


def _oracle_trajectory(dtype, L, B, K, per_lattice, masked, window):
    """the oracle's K sweeps from random spins with injected uniforms; every draw closer than `window` to its threshold
    is moved 1e-3 away first, so that the kernel and the oracle cannot part on a rounding tie.  The oracle runs at the
    temperatures the kernel sees (fp32-rounded in fp32).
    -> (spins0, temps [K, B], uniforms [K, B, N], masks [K, B, N] or None, infos, final spins, final Q)"""
    np_dtype = np.float32 if dtype == F32 else np.float64
    N = L * L
    rng = np.random.RandomState(1000 * dtype + L)
    spins0 = rng.randint(0, 2, size=(B, L, L)).astype(np.int8)
    temps = _schedules(K, B) if per_lattice else np.repeat(0.45 + 0.3 * np.abs(np.sin(0.4 * np.arange(K)))[:, None], B, 1)
    temps = temps.astype(np_dtype)
    masks = (rng.random_sample((K, B, N)) < 0.6).astype(np.uint8) if masked else None
    spins, Q = spins0.copy(), np.zeros((B, 5, N, 2))
    us, infos = [], []
    for k in range(K):
        T = temps[k].astype(np.float64)[:, None]
        mk = None if masks is None else masks[k]
        u = rng.random_sample((B, N)).astype(np_dtype)
        thr = ising_oracle.step(spins, Q, T, 0.1, u.astype(np.float64), update_mask=mk)[2]["threshold"]
        u = np.where(np.abs(u - thr) < window, np.where(thr < 0.5, thr + 1e-3, thr - 1e-3), u).astype(np_dtype)
        spins, Q, info = ising_oracle.step(spins, Q, T, 0.1, u.astype(np.float64), update_mask=mk)
        assert np.abs(u - info["threshold"]).min() > window
        us.append(u); infos.append(info)
    return spins0, temps, np.stack(us), masks, infos, spins, Q


def _run_against_oracle(dtype, L, B, K, per_lattice, masked, base):
    from mfmarl_b200 import IsingMFQ
    window = 1e-5 if dtype == F32 else 1e-10
    spins0, temps, us, masks, infos, spins, Q = _oracle_trajectory(dtype, L, B, K, per_lattice, masked, window)
    resident = _cluster(dtype, L) > 0
    m = IsingMFQ(B, L, dtype=TORCH_DTYPE[dtype], seed=9, lattice_base=base, spins=torch.from_numpy(spins0))
    n_up, rsum = m.run(torch.from_numpy(temps) if per_lattice else temps[:, 0].tolist(),
                       uniforms=torch.from_numpy(us).cuda().contiguous(), resident=resident,
                       update_mask=None if masks is None else torch.from_numpy(masks).cuda().contiguous())
    n_up, rsum = n_up.cpu().numpy(), rsum.cpu().numpy()
    for k, info in enumerate(infos):
        assert np.array_equal(n_up[k], info["n_up"]), "n_up differs after sweep %d" % k
        if dtype == F32:        # integer-valued rewards: the fp32 sums are exact
            assert np.array_equal(rsum[k], info["reward_sum"]), "reward_sum differs after sweep %d" % k
        else:
            np.testing.assert_allclose(rsum[k], info["reward_sum"], rtol=1e-13, atol=1e-15)
    assert np.array_equal(m.spins.cpu().numpy(), spins)
    if dtype == F32:
        np.testing.assert_allclose(m.Q.cpu().numpy(), Q, rtol=1e-6, atol=1e-7)
    else:
        np.testing.assert_allclose(m.Q.cpu().numpy(), Q, rtol=1e-13, atol=1e-15)
    return resident


# ---- 2. every class against the fp64 oracle --------------------------------------------------------------------------

@pytest.mark.parametrize("L", FP64_RESIDENT + FP64_STREAM)
@pytest.mark.parametrize("per_lattice,masked", [(False, False), (False, True), (True, False), (True, True)])
def test_fp64_follows_the_oracle_in_every_shape_class(L, per_lattice, masked):
    """12 sweeps in one resident launch (K streaming launches where the side has no resident kernel) with injected
    uniforms, B = 2 lattices at lattice_base 3: spins and n_up exact, reward_sum and Q to 1e-13"""
    resident = _run_against_oracle(F64, L, 2, 12, per_lattice, masked, base=3)
    assert resident == (L in FP64_RESIDENT)


def _fp32_cases():
    cases = []
    for L in FP32_RESIDENT + FP32_STREAM:
        if L <= 512:
            cases += [(L, 2, 12, False, False), (L, 2, 12, True, True)]
        else:                   # the oracle's cost at 896^2: one lattice, a few sweeps
            cases += [(L, 1, 3, False, False), (L, 1, 3, False, True)]
    return cases


@pytest.mark.parametrize("L,B,K,per_lattice,masked", _fp32_cases())
def test_fp32_follows_the_oracle_in_every_shape_class(L, B, K, per_lattice, masked):
    """fp32 with injected uniforms along the oracle's trajectory (draws within 1e-5 of the threshold moved away): spins,
    n_up and reward_sum equal, Q within 1e-6 relative, after K sweeps in one resident launch or K streaming launches"""
    resident = _run_against_oracle(F32, L, B, K, per_lattice, masked, base=3)
    assert resident == (L in FP32_RESIDENT)


@pytest.mark.parametrize("dtype,L", [(F32, L) for L in FP32_RESIDENT] + [(F64, L) for L in FP64_RESIDENT])
@pytest.mark.parametrize("per_lattice", [False, True])
def test_resident_production_draws_equal_streaming_in_every_shape_class(dtype, L, per_lattice):
    """production Philox draws: two resident launches equal the same sweeps as streaming launches bit for bit (spins,
    Q, n_up and reward_sum of every sweep), so the state carries over; lattice_base 4, act groups with per-lattice
    schedules"""
    from mfmarl_b200 import IsingMFQ
    B, K = 3, 6
    assert _cluster(dtype, L) > 0
    rng = np.random.RandomState(L)
    spins = torch.from_numpy(rng.randint(0, 2, size=(B, L, L)).astype(np.int8))
    a = IsingMFQ(B, L, dtype=TORCH_DTYPE[dtype], seed=21, lattice_base=4, spins=spins)
    b = IsingMFQ(B, L, dtype=TORCH_DTYPE[dtype], seed=21, lattice_base=4, spins=spins)
    for launch in range(2):
        temps = torch.from_numpy(_schedules(K, B)[::-1].copy() if launch else _schedules(K, B))
        if not per_lattice:
            temps = temps[:, 0].tolist()
        masks = None
        if per_lattice:
            masks = torch.from_numpy((rng.random_sample((K, B, L * L)) < 0.6).astype(np.uint8)).cuda()
        n_res, r_res = a.run(temps, resident=True, update_mask=masks)
        n_str, r_str = b.run(temps, resident=False, update_mask=masks)
        assert torch.equal(a.spins, b.spins), launch
        assert torch.equal(a.Q, b.Q), launch
        assert torch.equal(n_res, n_str) and torch.equal(r_res, r_str), launch
    assert not torch.equal(a.spins, spins.cuda())


# ---- 3. the production draws beyond the top bit ----------------------------------------------------------------------

def round_toward_zero_24(w):
    """uint32 words -> their value rounded toward zero to 24 significant bits (__uint2float_rz), as uint64"""
    w = np.asarray(w).astype(np.uint64)
    nbits = np.frexp(w.astype(np.float64))[1]                          # bit length (exact: w < 2^53)
    drop = np.maximum(nbits - 24, 0).astype(np.uint64)
    return (w >> drop) << drop


def production_uniforms(dtype, B, L, seed, lattice_base, step):
    """[B, L, L] float64: the uniform every site draws in the sweep with this step counter, from tests/philox_ref.py and
    the composition documented in include/mfmarl_batched.h (mfi_step).  Key (seed, lattice_base + lattice), counter
    (column, row / 4, step, w3).  fp32: w3 = 0, word row % 4 rounded toward zero to 24 significant bits, / 2^32.  fp64:
    w3 = 0 for rows 4j, 4j+1 and w3 = 1 for rows 4j+2, 4j+3; the pair (hi, lo) = output words (0, 1) for the even
    row and (2, 3) for the odd one; u = ((hi >> 5) 2^26 + (lo >> 6)) / 2^53."""
    shape = (B, L, L)
    x = np.broadcast_to(np.arange(L, dtype=np.uint32)[None, None, :], shape)
    band = np.broadcast_to((np.arange(L, dtype=np.uint32) // 4)[None, :, None], shape)
    lat = np.broadcast_to((lattice_base + np.arange(B, dtype=np.uint32))[:, None, None], shape).astype(np.uint32)
    key = [np.full(shape, seed, np.uint32), lat]
    row = np.broadcast_to(np.arange(L)[None, :, None], shape)

    def words(w3):
        return philox4x32_10([x, band, np.full(shape, step, np.uint32), np.full(shape, w3, np.uint32)], key)

    if dtype == F32:
        return round_toward_zero_24(np.choose(row % 4, words(0))).astype(np.float64) / 2.0 ** 32
    r1, r2 = words(0), words(1)
    pick = row % 4
    hi = np.choose(pick, [r1[0], r1[2], r2[0], r2[2]]).astype(np.uint64)
    lo = np.choose(pick, [r1[1], r1[3], r2[1], r2[3]]).astype(np.uint64)
    return ((hi >> np.uint64(5)).astype(np.float64) * 67108864.0 + (lo >> np.uint64(6)).astype(np.float64)) / 2.0 ** 53


def test_fp32_production_uniform_truncates_to_24_bits():
    """the numpy restatement of __uint2float_rz above, on words whose rounding direction matters"""
    w = np.array([0, 1, 2 ** 24 - 1, 2 ** 24 + 1, 2 ** 25 + 3, 2 ** 32 - 1, 0x89ABCDEF], dtype=np.uint32)
    assert round_toward_zero_24(w).tolist() == [0, 1, 2 ** 24 - 1, 2 ** 24, 2 ** 25, 2 ** 32 - 2 ** 8, 0x89ABCD00]


DRAW_TEMPS = (0.25, 1.1346, 5.0)


@pytest.mark.parametrize("dtype,L", DRAW_SIDES)
@pytest.mark.parametrize("T", DRAW_TEMPS + ("lattices",))
def test_production_draws_beyond_the_top_bit(dtype, L, T):
    """Every site gets the pair (0, q1) in all five planes, so its threshold 1 / (1 + exp(q1 / T)) does not depend on
    its neighbours.  q1 (|q1| <= 2) puts that threshold a set margin above or below the site's predicted production
    uniform -- 2e-5 in fp32, 1e-12 in fp64, about half the sites each way -- so the action of every site is known and
    one sweep checks the uniform to about 15 (fp32) or 40 (fp64) bits.  Step 3, lattice_base 5; "lattices" gives the
    three lattices the three temperatures in one per-lattice call."""
    from mfmarl_b200 import IsingMFQ
    seed, base, step0, B = 77, 5, 3, 3
    np_dtype = np.float32 if dtype == F32 else np.float64
    temps = np.array(DRAW_TEMPS if T == "lattices" else (T,) * B).astype(np_dtype)
    Tk = temps.astype(np.float64)[:, None, None]                      # the temperature the kernel sees
    u = production_uniforms(dtype, B, L, seed, base, step0)
    margin = 2.5e-5 if dtype == F32 else 2e-12
    lo, hi = 1.0 / (1.0 + np.exp(2.0 / Tk)), 1.0 / (1.0 + np.exp(-2.0 / Tk))     # thresholds with |q1| <= 2
    rng = np.random.RandomState(L + 10 * dtype)
    above = rng.randint(0, 2, size=u.shape).astype(bool)
    above = np.where(u + margin > hi, False, np.where(u - margin < lo, True, above))
    target = np.where(above, np.maximum(u + margin, lo), np.minimum(u - margin, hi))
    q1 = (Tk * np.log(1.0 / target - 1.0)).astype(np_dtype)
    thr = ising_oracle.action_threshold(0.0, q1.astype(np.float64), Tk)
    assert np.abs(u - thr).min() >= (2e-5 if dtype == F32 else 1e-12)
    assert np.abs(q1).max() <= 2.0 + 1e-6
    want = (u >= thr).astype(np.int8)
    assert 0.3 < want.mean() < 0.7

    m = IsingMFQ(B, L, dtype=TORCH_DTYPE[dtype], seed=seed, lattice_base=base)
    m.t = step0
    m.Q[..., 0] = 0
    m.Q[..., 1] = torch.from_numpy(q1.reshape(B, 1, L * L)).to(m.Q.device)
    per = torch.from_numpy(temps).cuda() if T == "lattices" else float(temps[0])
    if _cluster(dtype, L) > 0:
        m.run(per[None, :] if T == "lattices" else [per], resident=True)
    else:
        m.step(per)
    got = m.spins.cpu().numpy()
    bad = got != want
    assert not bad.any(), "%d of %d sites drew the other action, first at %r (u %.17g, threshold %.17g)" % (
        bad.sum(), bad.size, np.argwhere(bad)[0], u[bad][0], thr[bad][0])


# ---- 4. K8 edges -----------------------------------------------------------------------------------------------------

EDGE_GRID = np.array([0.6, 1e-3, 1.1346, 1e9, 2.5, 1e20])


def _edge_temps(K, B):
    """[K, B]: every lattice meets T = 1e-3 (both thresholds 0: no uphill flip) and 1e20 (exp(-h / T) rounds to 1, so
    floor(2^32 exp(-h / T)) = 2^32 and only the clamp to 2^32 - 1 keeps the threshold from wrapping to 0)"""
    return EDGE_GRID[(np.arange(K)[:, None] + 2 * np.arange(B)[None, :]) % len(EDGE_GRID)]


def test_edge_temperatures_reach_both_threshold_clamps():
    assert metropolis_ref.threshold(2, 1e-3) == 0 and metropolis_ref.threshold(4, 1e-3) == 0
    assert math.floor(math.exp(-2 / 1e20) * 2 ** 32) == 2 ** 32
    assert metropolis_ref.threshold(2, 1e20) == 2 ** 32 - 1 and metropolis_ref.threshold(4, 1e20) == 2 ** 32 - 1
    assert 2 ** 32 - 20 < metropolis_ref.threshold(4, 1e9) < 2 ** 32 - 1


@pytest.mark.parametrize("L,B,K", [(34, 3, 12), (48, 2, 12), (66, 2, 12), (94, 2, 10), (130, 2, 8), (510, 1, 6)])
def test_metropolis_rows_with_a_partial_last_word_equal_the_numpy_reference(L, B, K):
    """sides whose rows are several words with a partial last one, at the edge temperatures, in two launches: spins
    after each, n_up and the bond sum of every sweep equal the reference bit for bit"""
    from mfmarl_b200 import IsingMetropolis
    seed, base = 99, 7
    rng = np.random.RandomState(L)
    spins = rng.randint(0, 2, size=(B, L, L)).astype(np.int8)
    temps = _edge_temps(K, B)
    chain = IsingMetropolis(B, L, seed=seed, lattice_base=base, spins=torch.from_numpy(spins))
    step = 0
    for part in (temps[:K // 2], temps[K // 2:]):
        n_up, bond = chain.run(part)
        spins, want_up, want_bond = metropolis_ref.run(spins, part, seed, base, step)
        step += len(part)
        assert np.array_equal(chain.spins.cpu().numpy(), spins)
        assert np.array_equal(n_up.cpu().numpy(), want_up)
        assert np.array_equal(bond.cpu().numpy(), want_bond)


@pytest.mark.parametrize("L,B", [(2, 2), (34, 3), (64, 2), (130, 2)])
def test_metropolis_single_sweep_launches_equal_the_numpy_reference(L, B):
    """K = 1 per launch: the statistics of the only sweep are written after the loop"""
    from mfmarl_b200 import IsingMetropolis
    seed, base = 5, 2
    rng = np.random.RandomState(L + 1)
    spins = rng.randint(0, 2, size=(B, L, L)).astype(np.int8)
    chain = IsingMetropolis(B, L, seed=seed, lattice_base=base, spins=torch.from_numpy(spins))
    temps = _edge_temps(4, B)
    for k in range(4):
        n_up, bond = chain.run(temps[k:k + 1])
        spins, want_up, want_bond = metropolis_ref.run(spins, temps[k:k + 1], seed, base, k)
        assert n_up.shape == (1, B)
        assert np.array_equal(chain.spins.cpu().numpy(), spins)
        assert np.array_equal(n_up.cpu().numpy(), want_up) and np.array_equal(bond.cpu().numpy(), want_bond)


def test_metropolis_without_outputs_moves_the_same_spins():
    """d_n_up and d_bond_sum both NULL: the chain is the one of a run with outputs"""
    from mfmarl_b200 import IsingMetropolis
    from mfmarl_b200.lib import check, load_library
    B, L, K, seed = 3, 66, 7, 12
    rng = np.random.RandomState(3)
    spins = torch.from_numpy(rng.randint(0, 2, size=(B, L, L)).astype(np.int8))
    temps = np.ascontiguousarray(_edge_temps(K, B))
    with_out = IsingMetropolis(B, L, seed=seed, lattice_base=1, spins=spins)
    with_out.run(temps)
    bare = spins.cuda().contiguous()
    check(load_library().mfi_metropolis(B, L, K, ctypes.c_void_p(bare.data_ptr()), temps.ctypes.data_as(ctypes.c_void_p),
                                        seed, 1, 0, None, None,
                                        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert torch.equal(bare, with_out.spins)
    assert not torch.equal(bare, spins.cuda())
