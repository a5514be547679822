"""Ising-model tabular mean-field Q-learning on the GPU (kernel K6, C ABI `mfi_step`).

`IsingMFQ` holds a batch of B independent L x L tori (spins int8 [B, L, L], Q [B, 5, L*L, 2]) in HBM and
advances all of them by one fused step per call: Boltzmann action per site, spin update, reward, Q update
-- the loop body of the reference's main_MFQ_Ising.py:105-134.  `run` re-expresses that script's outer loop
(temperature schedule :108-112, order-parameter stagnation stop :149-156) over the fused step, with the
same command-line flags (:13-26).

The MCMC references of the same model: `IsingMetropolis` (checkerboard single-spin flips, kernel K8, `mfi_metropolis`)
and `IsingSwendsenWang` (cluster updates, kernel K9, `mfi_swendsen_wang`).
"""
import argparse
import ctypes
import time

import numpy as np
import torch

from .lib import check, load_library

_DTYPES = {torch.float32: 0, torch.float64: 1}


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class IsingMFQ:
    def __init__(self, n_lattices, side, dtype=torch.float32, device=None, seed=13, lr=0.1, lattice_base=0,
                 spins=None):
        if not torch.cuda.is_available():
            raise RuntimeError("IsingMFQ needs a CUDA device: there is no CPU fallback")
        self.lib = load_library()
        self.lib.mfi_step.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_double, ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_uint, ctypes.c_uint, ctypes.c_uint, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        self.lib.mfi_step.restype = ctypes.c_int
        self.lib.mfi_run.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double, ctypes.c_void_p,
                                     ctypes.c_void_p, ctypes.c_uint, ctypes.c_uint, ctypes.c_uint, ctypes.c_void_p,
                                     ctypes.c_void_p, ctypes.c_void_p]
        self.lib.mfi_run.restype = ctypes.c_int
        self.lib.mfi_resident_cluster_size.argtypes = [ctypes.c_int, ctypes.c_int]
        self.lib.mfi_resident_cluster_size.restype = ctypes.c_int
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.B, self.L, self.N = n_lattices, side, side * side
        self.dtype, self.seed, self.lr, self.lattice_base = dtype, seed, lr, lattice_base
        self.t = 0
        if spins is None:   # Bernoulli(0.5) spins (Ising.py:79-99 draws np.random.choice(2) per agent)
            gen = torch.Generator(device=self.device)
            gen.manual_seed(seed + 7919 * lattice_base)
            spins = torch.randint(0, 2, (n_lattices, side, side), generator=gen, device=self.device,
                                  dtype=torch.int8)
        self.spins = torch.as_tensor(spins, dtype=torch.int8, device=self.device).contiguous().clone()
        assert tuple(self.spins.shape) == (n_lattices, side, side)
        self.Q = torch.zeros((n_lattices, 5, self.N, 2), dtype=dtype, device=self.device)   # main_MFQ_Ising.py:92
        self.n_up = torch.zeros((n_lattices,), dtype=torch.int32, device=self.device)
        self.reward_sum = torch.zeros((n_lattices,), dtype=dtype, device=self.device)
        self.mse = torch.zeros((n_lattices,), dtype=dtype, device=self.device)

    def step(self, temperature, uniforms=None, update_mask=None, stats=True):
        """One fused sweep.  temperature: a number, or a [B] tensor with one temperature per lattice;
        uniforms [B, N] (same dtype) injects the Boltzmann draws (test hook);
        update_mask uint8 [B, N] restricts the Q update to the act group (act_rate < 1)."""
        if uniforms is not None:
            assert uniforms.dtype == self.dtype and uniforms.is_cuda and uniforms.is_contiguous()
        if update_mask is not None:
            assert update_mask.dtype == torch.uint8 and update_mask.is_cuda and update_mask.is_contiguous()
        # a one-element tensor stays the shared temperature it always was
        per_lattice = isinstance(temperature, torch.Tensor) and temperature.dim() == 1 and temperature.numel() > 1
        if per_lattice:
            assert tuple(temperature.shape) == (self.B,), "per-lattice temperatures must be [n_lattices]"
            temps = temperature.to(device=self.device, dtype=self.dtype).contiguous()
        with torch.cuda.device(self.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            if per_lattice:
                check(self.lib.mfi_step_lattices(_DTYPES[self.dtype], self.B, self.L, _ptr(self.spins), _ptr(self.Q),
                                                 _ptr(temps), float(self.lr), _ptr(uniforms), _ptr(update_mask),
                                                 self.seed, self.lattice_base, self.t, _ptr(self.n_up),
                                                 _ptr(self.reward_sum) if stats else None,
                                                 _ptr(self.mse) if stats else None, stream))
            else:
                check(self.lib.mfi_step(_DTYPES[self.dtype], self.B, self.L, _ptr(self.spins), _ptr(self.Q),
                                        float(temperature), float(self.lr), _ptr(uniforms), _ptr(update_mask),
                                        self.seed, self.lattice_base, self.t, _ptr(self.n_up),
                                        _ptr(self.reward_sum) if stats else None, _ptr(self.mse) if stats else None,
                                        stream))
        self.t += 1
        return self.n_up, self.reward_sum, self.mse

    @property
    def resident_cluster(self):
        """CTAs per lattice of the shared-memory-resident kernel, 0 if this shape only streams."""
        return self.lib.mfi_resident_cluster_size(_DTYPES[self.dtype], self.L)

    def run(self, temperatures, uniforms=None, resident=None, update_mask=None):
        """len(temperatures) sweeps.  With the resident kernel (default when the shape allows) they run in ONE
        launch with Q in shared memory; otherwise one streaming launch per sweep.  Both give the same bits.
        temperatures: a [K] schedule shared by every lattice, or a [K, B] tensor (column b = lattice b's schedule).
        update_mask uint8 [K, B, N]: the act group of every sweep (act_rate < 1).
        Returns (n_up int32 [K, B], reward_sum [K, B])."""
        temps = torch.as_tensor(temperatures, dtype=self.dtype, device=self.device).contiguous()
        per_lattice = temps.dim() == 2 and temps.shape[1] > 1          # ([K, 1] stays a shared schedule, as before)
        if per_lattice:
            assert temps.shape[1] == self.B, "per-lattice temperatures must be [n_sweeps, n_lattices]"
        K = int(temps.shape[0]) if per_lattice else int(temps.numel())
        if resident is None:
            resident = self.resident_cluster > 0
        n_up = torch.zeros((K, self.B), dtype=torch.int32, device=self.device)
        rsum = torch.zeros((K, self.B), dtype=self.dtype, device=self.device)
        if uniforms is not None:
            assert uniforms.dtype == self.dtype and uniforms.is_cuda and uniforms.is_contiguous()
            assert tuple(uniforms.shape) == (K, self.B, self.N)
        if update_mask is not None:
            assert update_mask.dtype == torch.uint8 and update_mask.is_cuda and update_mask.is_contiguous()
            assert tuple(update_mask.shape) == (K, self.B, self.N)
        if resident:
            run = self.lib.mfi_run_lattices if per_lattice else self.lib.mfi_run
            with torch.cuda.device(self.device):
                check(run(_DTYPES[self.dtype], self.B, self.L, K, _ptr(self.spins), _ptr(self.Q),
                          _ptr(temps), float(self.lr), _ptr(uniforms), _ptr(update_mask), self.seed,
                          self.lattice_base,
                          self.t, _ptr(n_up), _ptr(rsum),
                          ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
            self.t += K
            self.n_up.copy_(n_up[-1])
        else:
            host_t = temps if per_lattice else temps.cpu().tolist()
            for k in range(K):
                self.step(host_t[k], uniforms=None if uniforms is None else uniforms[k],
                          update_mask=None if update_mask is None else update_mask[k])
                n_up[k].copy_(self.n_up)
                rsum[k].copy_(self.reward_sum)
        return n_up, rsum

    def order_param(self):
        """|n_up - n_down| / N per lattice (core.py:106-110), from the last step's up counts."""
        up = self.n_up.to(torch.float64)
        # tensor / tensor: a true IEEE division (torch turns `/ python_scalar` into a reciprocal multiply)
        return (2 * up - self.N).abs() / torch.full_like(up, float(self.N))

    def q_table(self):
        """Q as the reference lays it out: [B, N, 5, 2]."""
        return self.Q.permute(0, 2, 1, 3).contiguous()


class _IsingChain:
    """B independent L x L tori of the model MF-Q learns on, H = -1/2 sum_bonds sigma_i sigma_j, on the same temperature
    axis (Tc ~ 1.1346), advanced by the MCMC kernel behind the C entry point `_entry` (which takes mfi_metropolis's
    arguments)."""
    _entry = None

    def __init__(self, n_lattices, side, seed=13, lattice_base=0, spins=None, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("%s needs a CUDA device: there is no CPU fallback" % type(self).__name__)
        self.lib = load_library()
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.B, self.L, self.N = n_lattices, side, side * side
        self.seed, self.lattice_base = seed, lattice_base
        self.t = 0
        if spins is None:   # Bernoulli(0.5) spins, as IsingMFQ
            gen = torch.Generator(device=self.device)
            gen.manual_seed(seed + 7919 * lattice_base)
            spins = torch.randint(0, 2, (n_lattices, side, side), generator=gen, device=self.device,
                                  dtype=torch.int8)
        self.spins = torch.as_tensor(spins, dtype=torch.int8, device=self.device).contiguous().clone()
        assert tuple(self.spins.shape) == (n_lattices, side, side)
        self.n_up = (self.spins != 0).sum(dim=(1, 2)).to(torch.int32)

    def run(self, temperatures):
        """K sweeps in one launch.  temperatures: [K] shared by every lattice, or [K, B] (column b = lattice b's).
        Returns (n_up int32 [K, B], bond_sum int32 [K, B]): up spins and sum over the 2N bonds of sigma_i sigma_j
        after every sweep (bond_sum = MF-Q's reward_sum; energy per site = -bond_sum / N)."""
        temps = np.asarray(temperatures.cpu() if isinstance(temperatures, torch.Tensor) else temperatures,
                           dtype=np.float64)
        if temps.ndim == 1:
            temps = np.repeat(temps[:, None], self.B, axis=1)
        assert temps.ndim == 2 and temps.shape[1] == self.B, "temperatures must be [K] or [K, n_lattices]"
        temps = np.ascontiguousarray(temps)
        K = temps.shape[0]
        n_up = torch.empty((K, self.B), dtype=torch.int32, device=self.device)
        bond_sum = torch.empty((K, self.B), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            check(getattr(self.lib, self._entry)(self.B, self.L, K, _ptr(self.spins),
                                                 temps.ctypes.data_as(ctypes.c_void_p), self.seed, self.lattice_base,
                                                 self.t, _ptr(n_up), _ptr(bond_sum),
                                                 ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        self.t += K
        self.n_up.copy_(n_up[-1])
        return n_up, bond_sum

    def order_param(self):
        """|n_up - n_down| / N per lattice after the last sweep"""
        up = self.n_up.to(torch.float64)
        return (2 * up - self.N).abs() / torch.full_like(up, float(self.N))


class IsingMetropolis(_IsingChain):
    """Checkerboard single-spin-flip Metropolis chains (kernel K8, C ABI `mfi_metropolis`) on B independent L x L tori
    of the model MF-Q learns on: H = -1/2 sum_i sigma_i sum_nbr sigma_j, the same temperature axis (Tc ~ 1.1346).
    The MCMC reference of the order-parameter-against-temperature curve.  L even, 2 <= L <= 512."""
    _entry = "mfi_metropolis"


class IsingSwendsenWang(_IsingChain):
    """Swendsen-Wang cluster chains (kernel K9, C ABI `mfi_swendsen_wang`) on B independent L x L tori of the same model
    and temperature axis as IsingMetropolis.  Its autocorrelation time near Tc is a few sweeps at any side, so it is
    the MCMC reference where single-spin flips decorrelate slowly; it needs no colouring.  2 <= L <= 256, odd or even."""
    _entry = "mfi_swendsen_wang"


def temperature_schedule(t0, n, decay_rate, decay_gap, floor, start=0.3):
    """main_MFQ_Ising.py:103-112: T starts at 0.3, is multiplied by decay_rate every decay_gap steps (first at step 0)
    and never drops below the -t flag.  -> (temperatures of steps t0 .. t0+n-1, as Python floats)."""
    temps, cur = [], start
    for t in range(t0 + n):
        if t % decay_gap == 0:
            cur *= decay_rate
        if cur < floor:
            cur = floor
        if t >= t0:
            temps.append(cur)
    return temps


def run(argv=None):
    """`python -m mfmarl_b200.ising -n 400 -t 0.8`: the experiment of main_MFQ_Ising.py on the GPU.

    Verbose (default): one fused step per launch, the per-step line of the reference printed for lattice 0.
    --quiet: `--chunk` sweeps per launch through the shared-memory-resident kernel when the shape allows (same bits as
    stepping one by one); the stagnation stop of main_MFQ_Ising.py:149-156 is evaluated on the per-sweep up counts of
    every chunk, so MaxO and its step are those of the step-by-step loop."""
    ap = argparse.ArgumentParser(description="Ising tabular MFQ (B200)")
    ap.add_argument("-n", "--num_agents", default=100, type=int)
    ap.add_argument("-t", "--temperature", default=1, type=float)
    ap.add_argument("-epi", "--episode", default=1, type=int)
    ap.add_argument("-ts", "--time_steps", default=10000, type=int)
    ap.add_argument("-lr", "--learning_rate", default=0.1, type=float)
    ap.add_argument("-dr", "--decay_rate", default=0.99, type=float)
    ap.add_argument("-dg", "--decay_gap", default=2000, type=int)
    ap.add_argument("-ac", "--act_rate", default=1.0, type=float)
    ap.add_argument("--lattices", default=1, type=int, help="independent lattices stepped together")
    ap.add_argument("--quiet", action="store_true")
    ap.add_argument("--chunk", default=100, type=int, help="sweeps per launch in --quiet mode")
    args = ap.parse_args(argv)
    side = int(np.ceil(np.sqrt(args.num_agents)))
    assert side * side == args.num_agents, "num_agents must be a perfect square"
    results = []
    for ep in range(args.episode):
        model = IsingMFQ(args.lattices, side, seed=13 + ep, lr=args.learning_rate)
        N = model.N
        gen = torch.Generator(device=model.device); gen.manual_seed(1000 + ep)
        max_order, max_step, done_, t0, t = 0.0, 0, 0, time.time(), 0
        chunked = args.quiet

        def act_groups(n):   # a random act group of int(act_rate * N) sites per sweep (main_MFQ_Ising.py:126)
            if args.act_rate >= 1.0:
                return None
            k = int(args.act_rate * N)
            order = torch.rand((n, args.lattices, N), generator=gen, device=model.device).argsort(dim=2)
            mask = torch.zeros((n, args.lattices, N), dtype=torch.uint8, device=model.device)
            mask.scatter_(2, order[:, :, :k], 1)
            return mask

        stop = False
        while t < args.time_steps and not stop:
            n = min(args.chunk, args.time_steps - t) if chunked else 1
            temps = temperature_schedule(t, n, args.decay_rate, args.decay_gap, args.temperature)
            masks = act_groups(n)
            if chunked:
                ups_seq = model.run(temps, update_mask=masks)[0][:, 0].cpu().tolist()   # up counts of lattice 0, per sweep
                rsum = mse = None
            else:
                n_up, rsum, mse = model.step(temps[0], update_mask=None if masks is None else masks[0])
                ups_seq = [int(n_up[0])]
            for ups in ups_seq:
                order_param = abs(2 * ups - N) / N                           # core.py:106-110
                if order_param > max_order:
                    max_order, max_step = order_param, t
                done_ = done_ + 1 if abs(max_order - order_param) < 0.001 else 0
                t += 1
                if done_ == 500:
                    stop = True
                    break
                if not args.quiet:
                    print("E: %d/%d, reward = %f, mse = %f, Order = %f, Up = %d, Down = %d"
                          % (ep, t - 1, float(rsum[0]), float(mse[0]), order_param, ups, N - ups))
        print("Episode: %d, MaxO = %f at %d (%.1f site-steps/s)"
              % (ep, max_order, max_step, t * N * args.lattices / (time.time() - t0)))
        results.append((max_order, max_step))
    return results


if __name__ == "__main__":
    run()
