#!/usr/bin/env python
"""bench.py -- battle agent-steps/s (observations + mean action included) on N B200s, with the roofline of
the dominant kernel and the reference CPU engine timed beside it.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA path (one process per GPU)
  python bench.py --impl reference [--gpus N] [--steps K] ...    the reference CPU engine on the host cores
  python bench.py --dump-outputs DIR ...                          also write the last timed step's outputs to DIR/*.npy

The headline figure is ONE timed region of exactly K steps after W warm-up steps, so the engines' state after it
depends on the arguments alone: two builds run with the same arguments can be compared output for output.

Workload (BASELINE.json configs[2], "C3"): 40x40 battle, 64 v 64 agents, 4096 lock-stepped environments per
GPU, synthetic uniform-random actions, episodes auto-reset at done / 400 steps.  One "step" = one lockstep
pass of the hot path over all environments of the GPU: k_obs (both groups' views + features) then k_step
(set_action x2, step, reward, alive, mean action, clear_dead).  By default the GPU's environments are split into
two engines on two streams (--pipeline 2), so that one half's latency-bound k_step runs under the other half's
bandwidth-bound k_obs -- what a double-buffered actor loop does.  Unit of work: agent-step (SURVEY.md 8d).
Inputs (actions) are resident in HBM for `value`; `e2e` feeds them from pinned host memory every step and
reads rewards / alive / done / mean actions back to the host inside the timed region.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "mean-field-multi-agent-reinforcement-learning_b200")
if os.path.join(PKG, "python") not in sys.path:
    sys.path.insert(0, os.path.join(PKG, "python"))
DUMP_BYTES = 64 << 20        # --dump-outputs: budget of the .npy files


def _checker_paths():
    """tests/ holds the adapters of the CPU engines (reference .so, C oracle): only the cpu_baseline / --impl reference
    legs put it on the path."""
    if os.path.join(REPO, "tests") not in sys.path:
        sys.path.insert(0, os.path.join(REPO, "tests"))

BYTES_PER_AGENT_OBS = 13 * 13 * 7 * 4 + 34 * 4          # 4868: view + feature rows written by k_obs
BYTES_PER_AGENT_STEP = BYTES_PER_AGENT_OBS + 4 + 4 + 1  # + action read, reward + alive written (SURVEY 8d)
WORKLOADS = {
    "c3": dict(name="battle_40x40_64v64_4096envs_per_gpu_uniform_actions (BASELINE configs[2])",
               map_size=40, cap=64, envs=4096, max_steps=400),
    "c4": dict(name="battle_80x80_512v512_128envs_per_gpu_uniform_actions (BASELINE configs[3] shard)",
               map_size=80, cap=512, envs=128, max_steps=400),
}
WORKLOADS["c2"] = dict(name="battle_40x40_64v64_single_env_through_the_reference_C_ABI (BASELINE configs[1])",
                       map_size=40, cap=64, envs=1, max_steps=400)
WORKLOADS["play"] = dict(name="battle_40x40_64v64_rollout_with_policy_networks (senario_battle.play, batched)",
                         map_size=40, cap=64, envs=1024, max_steps=400)
WORKLOADS["c5"] = dict(name="ising_256x256_x16384_lattices_mfq_T0.8 (BASELINE configs[4])", side=256,
                       lattices=16384, temperature=0.8, lr=0.1)
REF_SO = os.path.join(REPO, "oracle", "_ref", "libmagent_ref.so")
BYTES_PER_SITE = 14   # fp32 Q pair read 8 + Q write 4 + int8 spin read 1 + write 1 (SURVEY 8d)


def placement(wl):
    from mfmarl_b200.scenarios import c4_positions, generate_map_positions
    return generate_map_positions(40) if wl["map_size"] == 40 else c4_positions()


# ------------------------------------------------------------------------------------------------
# CPU side: the reference engine (or the C oracle port) on the host cores
# ------------------------------------------------------------------------------------------------
class SingleEnvThroughTheBinding:
    """magent.GridWorld('battle') over build/libmagent.so -- the calls senario_battle.play makes (group = 0 / 1)."""

    def __init__(self, map_size):
        import magent
        self.env = magent.GridWorld("battle", map_size=map_size)
        self.h = self.env.get_handles()

    def reset(self): self.env.reset()
    def add_agents(self, g, pos): self.env.add_agents(self.h[g], method="custom", pos=pos)
    def get_num(self, g): return self.env.get_num(self.h[g])
    def get_observation(self, g): return self.env.get_observation(self.h[g])
    def set_action(self, g, acts): self.env.set_action(self.h[g], acts)
    def step(self): return self.env.step()
    def get_reward(self, g): return self.env.get_reward(self.h[g])
    def get_alive(self, g): return self.env.get_alive(self.h[g])
    def clear_dead(self): self.env.clear_dead()


def cpu_worker(argv):
    """One single-threaded environment: `warm` untimed + `steps` timed lockstep steps of the hot loop
    (get_observation x2, set_action x2, step, get_reward/get_alive x2, mean action, clear_dead)."""
    kind, map_size, warm, steps, seed = argv[0], int(argv[1]), int(argv[2]), int(argv[3]), int(argv[4])
    os.environ["OMP_NUM_THREADS"] = argv[5] if len(argv) > 5 else "1"
    import numpy as np
    from mfmarl_b200.scenarios import c4_positions, generate_map_positions
    if kind == "cuda":            # --workload c2: the product through the reference-facing single-env C ABI
        eng = SingleEnvThroughTheBinding(map_size)
    else:
        _checker_paths()
        from engines import OracleEngine, RefEngine
        eng = RefEngine(map_size) if kind == "reference" else OracleEngine(map_size)
    left, right = generate_map_positions(40) if map_size == 40 else c4_positions()
    rng = np.random.RandomState(seed)
    eye = np.eye(21)

    def episode_reset():
        eng.reset(); eng.add_agents(0, left); eng.add_agents(1, right)

    episode_reset()
    agent_steps, t_start, ep_steps = 0, None, 0
    for s in range(warm + steps):
        if s == warm:
            t_start = time.perf_counter()
        n = [eng.get_num(0), eng.get_num(1)]
        for g in range(2):
            eng.get_observation(g)
        acts = [rng.randint(0, 21, size=n[g]).astype(np.int32) for g in range(2)]
        for g in range(2):
            eng.set_action(g, acts[g])
        done = eng.step()
        for g in range(2):
            eng.get_reward(g); eng.get_alive(g)
            np.mean(eye[acts[g]], axis=0, keepdims=True)      # senario_battle.py:141
        eng.clear_dead()
        if s >= warm:
            agent_steps += n[0] + n[1]
        ep_steps += 1
        if done or ep_steps >= 400:
            episode_reset(); ep_steps = 0
    print(json.dumps({"agent_steps": agent_steps, "seconds": time.perf_counter() - t_start}))


def run_cpu(kind, map_size, warm, steps, procs):
    """`procs` independent single-thread environments side by side (the fair throughput comparator:
    intra-env OpenMP scales ~1.4x at 8 threads and is nondeterministic, SURVEY.md F2 / section 6)."""
    cmds = [[sys.executable, os.path.abspath(__file__), "--_cpu_worker", kind, str(map_size), str(warm),
             str(steps), str(1000 + i)] for i in range(procs)]
    env = dict(os.environ, OMP_NUM_THREADS="1", CUDA_VISIBLE_DEVICES="")
    ps = [subprocess.Popen(c, stdout=subprocess.PIPE, env=env) for c in cmds]
    outs = [json.loads(p.communicate()[0].decode().strip().splitlines()[-1]) for p in ps]
    total = sum(o["agent_steps"] for o in outs)
    seconds = max(o["seconds"] for o in outs)
    return total / seconds, total, seconds


def run_cpu_openmp(kind, map_size, warm, steps, threads):
    """SURVEY.md 8d mode (ii): ONE environment with the reference's intra-env OpenMP on `threads` threads (its
    default is cpu_count // 2, c_lib.py:53-54).  Nondeterministic under OpenMP (SURVEY F2) -- timing only."""
    cmd = [sys.executable, os.path.abspath(__file__), "--_cpu_worker", kind, str(map_size), str(warm), str(steps),
           "999", str(threads)]
    env = dict(os.environ, OMP_NUM_THREADS=str(threads), CUDA_VISIBLE_DEVICES="")
    out = json.loads(subprocess.run(cmd, stdout=subprocess.PIPE, env=env).stdout.decode().strip().splitlines()[-1])
    return out["agent_steps"] / out["seconds"], out["seconds"]


def cpu_kind():
    return "reference" if os.path.exists(REF_SO) else "port"


# ------------------------------------------------------------------------------------------------
# clocks: sampled DURING the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake"}

    def __init__(self, device_index):
        self.samples, self.reason_bits, self.max_mhz = [], 0, None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(device_index).uuid)
                if not uuid.startswith("GPU-"):
                    uuid = "GPU-" + uuid
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.reason_bits |= nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            except Exception:
                pass
            time.sleep(0.005)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": [n for b, n in self.REASONS.items() if self.reason_bits & b],
                "samples": len(self.samples)}


def measured_peak():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload):
    """dram bytes per k_obs launch from the committed ncu --set full capture, if one exists."""
    try:
        with open(os.path.join(REPO, "profiles", "obs_traffic.json")) as f:
            return json.load(f).get(workload)
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Ctx:
    """process-wide set-up shared by the legs of one bench.py run (one process per GPU)"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def reduce(self, values, op):
        """element-wise MAX / SUM of a list of numbers over the ranks (float64)"""
        if self.world == 1:
            return [float(v) for v in values]
        t = self.torch.tensor([float(v) for v in values], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op={"max": self.dist.ReduceOp.MAX, "sum": self.dist.ReduceOp.SUM}[op])
        return [float(v) for v in t]

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def reduce_region(ctx, region_ms, region_work):
    """one timed region over the ranks: time = max, work = sum"""
    return ctx.reduce([region_ms], "max")[0], ctx.reduce([region_work], "sum")[0]


def pick_median(ctx, region_ms, region_work):
    """Per repeat: time = max over ranks, work = sum over ranks, throughput = work / time.  The repeat with the median
    THROUGHPUT is the one reported (the work per region varies a little with the phase of the episodes)."""
    t = ctx.reduce(region_ms, "max")
    w = ctx.reduce(region_work, "sum")
    order = sorted(range(len(t)), key=lambda i: w[i] / t[i])
    m = order[len(order) // 2]
    return t[m], w[m], {"repeats": len(t), "min": min(t), "median": sorted(t)[len(t) // 2], "max": max(t),
                        "reported": t[m]}


def dump_battle_outputs(out_dir, last, nums):
    """--dump-outputs: what the last timed step handed its caller, as float32 .npy files.  From k_step: reward, alive
    and mean_action per env and group, done per env; from k_obs: view and feature rows.  Rows at or past an env's agent
    count `num` (taken before the step) are stale in the engine's buffers and written as zeros.  The observations of a
    fixed, seeded sample of whole environments (obs_envs) fill half of the DUMP_BYTES budget; the step outputs cover
    every environment unless they would not fit the other half either (step_envs)."""
    import numpy as np
    import torch
    num = torch.cat(nums).long()                                        # [E, 2]
    reward, alive, done, mean = (torch.cat([l[1][i] for l in last]) for i in range(4))
    E, _, cap = reward.shape
    Eh = E // len(last)
    view_row, feat_row = last[0][0][0][0, 0, 0].numel(), last[0][0][1].shape[-1]
    rng = np.random.RandomState(0)

    def envs_within(per_env_bytes):
        n = min(E, max(1, (DUMP_BYTES // 2) // per_env_bytes))
        return np.arange(E) if n == E else np.sort(rng.choice(E, n, replace=False))

    obs_envs = envs_within(2 * cap * (view_row + feat_row) * 4)
    step_envs = envs_within(2 * cap * 8 + mean.shape[-1] * 8 + 12)
    live = torch.arange(cap, device=num.device) < num[..., None]       # [E, 2, cap]
    view = torch.stack([last[e // Eh][0][0][e % Eh] for e in obs_envs])
    feat = torch.stack([last[e // Eh][0][1][e % Eh] for e in obs_envs])
    lo, ls = live[torch.from_numpy(obs_envs).to(num.device)], torch.from_numpy(step_envs).to(num.device)
    out = {"num": num[ls], "reward": torch.where(live, reward, 0.0)[ls], "alive": torch.where(live, alive.float(), 0.0)[ls],
           "done": done[ls], "mean_action": mean[ls], "step_envs": torch.from_numpy(step_envs),
           "view": torch.where(lo[..., None, None, None], view, 0.0), "feature": torch.where(lo[..., None], feat, 0.0),
           "obs_envs": torch.from_numpy(obs_envs)}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def measure_battle(ctx, args, workload, K, W, envs_per_gpu=0, pipeline=None, obs_tile=None, extras=True, dump=None):
    """One battle workload on this rank's GPU: W warm-up steps, then ONE region of exactly K lockstep steps (bracketed
    by a barrier + synchronize; CUDA events on the launching streams), the e2e variant the same way.  With `dump` (a
    directory), rank 0 writes what the last timed step returned before anything else runs.  Returns the JSON fields of
    the workload (rank 0) -- every rank must call it."""
    torch = ctx.torch
    from mfmarl_b200 import BatchedGridWorld
    wl = WORKLOADS[workload]
    dev, world, rank, local = ctx.dev, ctx.world, ctx.rank, ctx.local
    E, cap = envs_per_gpu or wl["envs"], wl["cap"]
    left, right = placement(wl)
    # --pipeline P: the GPU's envs are split into P engines on P streams, so that the latency-bound k_step of one
    # part runs under the bandwidth-bound k_obs of the next (what a double-buffered actor loop does).  P = 1: one
    # engine, kernels back to back on one stream.
    P = max(1, args.pipeline if pipeline is None else pipeline)
    assert E % P == 0
    Eh = E // P
    tile = args.obs_tile if obs_tile is None else obs_tile
    envs = []
    for h in range(P):
        env = BatchedGridWorld(Eh, map_size=wl["map_size"], capacity=cap, device=dev, rng="philox", seed=0,
                               env_base=rank * E + h * Eh, max_steps=wl["max_steps"], auto_reset=True,
                               obs_tile_agents=tile, step_threads=args.step_threads,
                               concurrent_step_envs=Eh if P > 1 else 0)   # the sibling engine's k_step overlaps this k_obs
        env.reset(); env.add_agents(0, left); env.add_agents(1, right)
        envs.append(env)
    streams = [torch.cuda.current_stream()] if P == 1 else [torch.cuda.Stream(device=dev) for _ in range(P)]
    # synthetic actions, uniform{0..20} from torch's Philox generator, resident in HBM: a pool the steps cycle through
    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    POOL = 8
    pool = [[torch.randint(0, 21, (Eh, 2, cap), generator=gen, device=dev, dtype=torch.int32) for _ in range(POOL)]
            for _ in range(P)]
    for env in envs:
        env.observe()                 # allocates the observation block (E*2*cap*4868 B in total)

    def agent_steps_total():
        return sum(int(env.get("agent_steps").sum()) for env in envs)

    last = [None] * P                                  # per engine: (observe(), step()) of its latest step

    def one_step(h, env, k, events=None):
        st = streams[h]
        with torch.cuda.stream(st):
            if events: events[0].record(st)
            obs = env.observe()
            if events: events[1].record(st)
            last[h] = (obs, env.step(pool[h][k % POOL]))
            if events: events[2].record(st)

    for k in range(W):
        for h, env in enumerate(envs):
            one_step(h, env, k)
    ctx.barrier()

    dump = dump if rank == 0 else None
    num_alias = [env.device_state("num") for env in envs] if dump else None
    nums = [None] * P

    def timed_region(with_events, keep_num=False):
        ev = [[[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)] for _ in range(P)] if with_events else None
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = [torch.cuda.Event(enable_timing=True) for _ in range(P)]
        ctx.barrier()                              # (everything launched so far has run: the counter below is exact)
        a0 = agent_steps_total()
        ctx.barrier()
        t0.record()
        for h in range(P):
            streams[h].wait_event(t0)
        for k in range(K):
            for h, env in enumerate(envs):
                if keep_num and k == K - 1:            # agent counts the last step starts from (the dump's row mask)
                    with torch.cuda.stream(streams[h]):
                        nums[h] = num_alias[h].clone()
                one_step(h, env, k, ev[h][k] if ev else None)
        for h in range(P):
            t1[h].record(streams[h])
        ctx.barrier()
        return max(t0.elapsed_time(t) for t in t1), agent_steps_total() - a0, ev

    # ---- the timed region: exactly K steps ----
    with ClockSampler(local) as clocks:
        ms0, work0, _e = timed_region(False, keep_num=bool(dump))
    if dump:
        dump_battle_outputs(dump, last, nums)
    ms, agent_steps_all = reduce_region(ctx, ms0, work0)
    # ---- kernel attribution: the next K steps again, with event pairs around every launch ----
    _m, agent_steps, ev = timed_region(True)                                        # this rank
    obs_ms = sum(e[0].elapsed_time(e[1]) for evh in ev for e in evh) / (K * P)     # per k_obs launch
    step_ms = sum(e[1].elapsed_time(e[2]) for evh in ev for e in evh) / (K * P)    # per k_step launch

    # ---- the same region on FRESH episodes (armies at full strength), as round 1 measured it: reset, W warm-up steps,
    #      K timed steps, five times; the median and the spread of the five sit beside the single timed region. ----
    fresh = None
    if extras:
        f_ms, f_work = [], []
        for _ in range(5):
            for env in envs:
                env.reset(); env.add_agents(0, left); env.add_agents(1, right)
            for k in range(W):
                for h, env in enumerate(envs):
                    one_step(h, env, k)
            m, w_, _e = timed_region(False)
            f_ms.append(m); f_work.append(w_)
        fm, fw, fregions = pick_median(ctx, f_ms, f_work)
        fresh = {"value": fw / (fm * 1e-3), "unit": "agent-steps/s", "ms_per_step": fm / K, "region_ms": fregions,
                 "agents_per_step": fw / K,
                 "note": "steps %d..%d of fresh episodes (all %d agents of an env alive), the phase round 1 reported" % (W, W + K, 2 * cap)}

    # ---- attribution: with P > 1 the two kernels of different engines overlap, so the event pairs above contain
    #      the time a kernel shared the GPU with the other one.  A short extra run with the launches back to back on
    #      ONE stream gives each kernel's duration alone (what the ncu launch list also shows). ----
    alone = None
    if P > 1:
        n_alone = min(K, 20)
        as_a = agent_steps_total()
        eva = [[[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(n_alone)] for _ in range(P)]
        ctx.barrier()
        for k in range(n_alone):
            for h, env in enumerate(envs):
                eva[h][k][0].record(); env.observe(); eva[h][k][1].record()
                env.step(pool[h][k % POOL]); eva[h][k][2].record()
        ctx.barrier()
        alone = {"k_obs": sum(e[0].elapsed_time(e[1]) for evh in eva for e in evh) / (n_alone * P),
                 "k_step": sum(e[1].elapsed_time(e[2]) for evh in eva for e in evh) / (n_alone * P),
                 "agents_per_launch": (agent_steps_total() - as_a) / (n_alone * P), "launches": n_alone * P}

    # ---- e2e: actions from pinned host memory each step, results read back to pinned host memory each step.
    #      Pipelined like an actor loop: the upload of step t and the download of step t-1 ride on copy
    #      streams under k_obs; a step's results are consumed (waited for) before its buffers are reused ----
    h_act = [[p_.cpu().pin_memory() for p_ in pool[h]] for h in range(P)]
    n_act = envs[0].sizes["n_action"]

    def result_set():
        return (torch.empty((Eh, 2, cap), dtype=torch.float32).pin_memory(),
                torch.empty((Eh, 2, cap), dtype=torch.uint8).pin_memory(),
                torch.empty((Eh, 2, n_act), dtype=torch.float32).pin_memory(),
                torch.empty((Eh,), dtype=torch.int32).pin_memory())

    results = [[result_set(), result_set()] for _ in range(P)]
    for k in range(min(W, 4)):
        for h, env in enumerate(envs):
            with torch.cuda.stream(streams[h]):
                env.observe()
                env.host_wait(env.step_host_async(h_act[h][k % POOL], *results[h][k & 1]))
    checksum = [0.0]

    def e2e_region():
        ctx.barrier()
        a0 = agent_steps_total()
        ctx.barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = [torch.cuda.Event(enable_timing=True) for _ in range(P)]
        e0.record()
        for h in range(P):
            streams[h].wait_event(e0)
        tickets = [0] * P
        for k in range(K):
            for h, env in enumerate(envs):
                with torch.cuda.stream(streams[h]):
                    env.observe()
                    tickets[h] = env.step_host_async(h_act[h][k % POOL], *results[h][k & 1])   # H2D + k_step + D2H enqueued
                if k >= 1:                                                  # consume step k-1's results on the host
                    env.host_wait(tickets[h] ^ 1)
                    checksum[0] += float(results[h][(k - 1) & 1][0][0, 0, 0])
        for h, env in enumerate(envs):
            env.host_wait(tickets[h])
            checksum[0] += float(results[h][(K - 1) & 1][0][0, 0, 0])
            e1[h].record(streams[h])
        ctx.barrier()
        return max(e0.elapsed_time(t) for t in e1), agent_steps_total() - a0

    m0, w0 = e2e_region()
    e2e_ms, e2e_all = reduce_region(ctx, m0, w0)
    h2d = P * h_act[0][0].numel() * 4
    d2h = P * sum(t.numel() * t.element_size() for t in results[0][0])

    # ---- the same loop with the observations ALSO copied to pinned host memory every step, i.e. what a policy that
    #      lives on the host (the reference's own TF feed) would cost: PCIe-bound, reported for completeness ----
    obs_host = None
    if extras and args.obs_to_host_steps > 0 and world == 1:     # (a single-GPU figure: 2.5 GB of pinned memory per rank otherwise)
        view0, feat0 = envs[0].observe()
        h_view = torch.empty(view0.shape, dtype=torch.float32).pin_memory()
        h_feat = torch.empty(feat0.shape, dtype=torch.float32).pin_memory()
        ctx.barrier()
        as2 = agent_steps_total()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record()
        for k in range(args.obs_to_host_steps):
            for h, env in enumerate(envs):
                v, f = env.observe()
                h_view.copy_(v, non_blocking=True); h_feat.copy_(f, non_blocking=True)
                env.host_wait(env.step_host_async(h_act[h][k % POOL], *results[h][k & 1]))
        o1.record()
        ctx.barrier()
        obs_host = {"value": (agent_steps_total() - as2) / (o0.elapsed_time(o1) * 1e-3), "unit": "agent-steps/s",
                    "steps": args.obs_to_host_steps,
                    "d2h_bytes_per_step": d2h + P * (h_view.numel() + h_feat.numel()) * 4,
                    "note": "observations copied to pinned host memory as well (rank 0's figure): PCIe-bound"}
    del envs, pool, results, h_act
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    peak, peak_src = measured_peak()
    agents_per_launch = agent_steps / (K * P)
    # k_obs launch duration.  One stream: the event pair around each launch.  Several streams: launches of
    # different engines overlap (with each other and with k_step), so a launch's own event pair contains time it
    # shared the memory system; the duration charged per launch is then the timed region divided by the number of
    # k_obs launches -- conservative, since the region also contains every k_step.
    launch_ms = obs_ms if P == 1 else ms / (K * P)
    achieved = agents_per_launch * BYTES_PER_AGENT_OBS / (launch_ms * 1e-3) / 1e9
    return {
        "metric": "battle agent-steps/sec incl. obs+mean-action",
        "value": agent_steps_all / (ms * 1e-3), "unit": "agent-steps/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        # `config` is the workload, key for key what the --impl reference line carries; `setup` describes this arm's run
        "config": {"workload": wl["name"], "envs_per_gpu": E, "map": wl["map_size"], "agents_per_env": 2 * cap},
        "setup":  {"actions": "uniform{0..20}, torch Philox, pool of %d resident tensors" % POOL,
                   "rng": "philox(seed, env, step)", "auto_reset": "done or %d steps" % wl["max_steps"],
                   "l2": "outputs per step (%.2f GB) exceed the 126 MB L2; no explicit flush"
                         % (E * 2 * cap * BYTES_PER_AGENT_OBS / 1e9),
                   "sharding": "envs [r*E,(r+1)*E) on rank r, no collective on the env path",
                   "pipeline": "%d engine(s) x %d envs on %d stream(s)" % (P, Eh, P),
                   "obs_tile_agents": tile or "engine default",
                   "timed_region": "exactly %d steps, once, after %d warm-up steps" % (K, W)},
        "region_ms": ms,
        "agents_per_step": agent_steps_all / K,
        "fresh_episodes": fresh,
        "gpu_launches": 2 * K * P,
        "kernels_ms": {"k_obs": obs_ms, "k_step": step_ms,
                       "note": "event pairs on the launching streams, in a second region of K steps after the timed one" +
                               ("; with %d streams they include time shared with the other engine's kernel" % P
                                if P > 1 else "")},
        "kernels_alone_ms": alone,
        "roofline": {"bound": "hbm", "kernel": "k_obs", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak,
                     # per launch, like `achieved`: the ncu capture is one launch over the workload's full env count
                     "traffic": (lambda t: None if t is None else t * Eh / wl["envs"])(ncu_traffic(workload)),
                     "peak_source": peak_src,
                     "peak_note": "the measured peak is a COPY (read + write); k_obs only writes, and a pure fill_ of the "
                                  "same 2.55 GB reaches 7.47 TB/s on this part (profiles/write_probe.py), so frac can "
                                  "exceed 1 -- against that fill rate the one-stream kernel is at 0.92",
                     "bytes_per_agent": BYTES_PER_AGENT_OBS, "agents_per_launch": agents_per_launch,
                     "launch_ms": launch_ms,
                     "launch_ms_rule": "event pair around each k_obs launch" if P == 1 else
                                       "timed region / number of k_obs launches (the %d streams' launches overlap; "
                                       "their own event pairs, kernels_ms, include shared time)" % P,
                     "whole_step_frac": (agent_steps_all / world / K) * BYTES_PER_AGENT_STEP / (ms / K * 1e-3) / 1e9 / peak,
                     "alone": None if alone is None else {
                         "achieved": alone["agents_per_launch"] * BYTES_PER_AGENT_OBS / (alone["k_obs"] * 1e-3) / 1e9,
                         "frac": alone["agents_per_launch"] * BYTES_PER_AGENT_OBS / (alone["k_obs"] * 1e-3) / 1e9 / peak,
                         "note": "k_obs launched with nothing else on the GPU (short run after the timed regions)"}},
        "e2e": {"value": e2e_all / (e2e_ms * 1e-3), "unit": "agent-steps/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "region_ms": e2e_ms,
                "note": "mfb_step_host_async: actions from pinned host memory, rewards/alive/done/mean action "
                        "copied back to pinned host memory and waited for every step (copies pipelined under "
                        "k_obs); observations stay in HBM for the policy network",
                "with_observations_to_host": obs_host},
        "clocks": clocks.summary(),
        "dump_outputs": None if not dump else {
            "dir": dump, "note": "the timed region also held %d device copies of the agent counts (%d B each), "
                                 "enqueued before its last step for the dump's row mask" % (P, Eh * 2 * 4)},
    }


def measure_grad_allreduce(ctx, iters=20):
    """The one collective near the path (north star: optional shared-parameter gradient all-reduce over NVLink):
    algo.base.sync_gradients on the MF-Q network's real gradient set, timed on the device, max over ranks."""
    torch = ctx.torch
    from mfmarl_b200.algo.base import QNet, sync_gradients
    net = QNet((13, 13, 7), (34,), 21, use_mf=True).to(ctx.dev)
    gen = torch.Generator(device=ctx.dev); gen.manual_seed(77 + ctx.rank)
    params = list(net.parameters())
    for p_ in params:
        p_.grad = torch.randn(p_.shape, generator=gen, device=ctx.dev)
    want = ctx.reduce([float(sum(p_.grad.double().sum() for p_ in params))], "sum")[0] / ctx.world
    for _ in range(3):
        sync_gradients(params)
    for p_ in params:                       # fresh, rank-specific gradients for the checked call
        p_.grad = torch.randn(p_.shape, generator=gen, device=ctx.dev)
    want = ctx.reduce([float(sum(p_.grad.double().sum() for p_ in params))], "sum")[0] / ctx.world
    sync_gradients(params)
    got = float(sum(p_.grad.double().sum() for p_ in params))
    ctx.barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        sync_gradients(params)
    t1.record()
    ctx.barrier()
    ms = ctx.reduce([t0.elapsed_time(t1) / iters], "max")[0]
    n_bytes = sum(p_.numel() for p_ in params) * 4
    return {"what": "algo.base.sync_gradients on the MF-Q network's gradients (one flat NCCL all-reduce + average)",
            "bytes": n_bytes, "ms": ms, "algbw_GBs": n_bytes / (ms * 1e-3) / 1e9, "ranks": ctx.world,
            "mean_matches": abs(got - want) <= 1e-3 * max(1.0, abs(want))}


def run_ours(args):
    ctx = Ctx()
    main = measure_battle(ctx, args, args.workload, args.steps, args.warmup,
                          envs_per_gpu=args.envs, obs_tile=args.obs_tile, dump=args.dump_outputs)
    also = {}
    if args.workload == "c3" and not args.no_also:
        # the other two named shapes under the same clock (BASELINE configs[3] and [4]): shorter legs, same rules
        c4 = measure_battle(ctx, args, "c4", 200, max(3, min(args.warmup, 10)), pipeline=2, obs_tile=0, extras=False)
        c5 = measure_ising(ctx, args, min(max(args.steps, 100), 200), max(3, args.warmup))
        if ctx.rank == 0:
            keep = ("metric", "value", "unit", "ms_per_step", "scaling", "config", "region_ms", "roofline", "e2e",
                    "gpu_launches", "kernels_alone_ms", "sweeps_per_launch")
            also = {"c4": {k: c4[k] for k in keep if k in c4}, "c5": {k: c5[k] for k in keep if k in c5}}
    if ctx.world > 1 and not args.no_also:
        ar = measure_grad_allreduce(ctx)
        if ctx.rank == 0:
            also["grad_allreduce"] = ar
    if ctx.rank == 0:
        line = main
        if also:
            line["also"] = also
        wl = WORKLOADS[args.workload]
        if ctx.world == 1 and not args.no_cpu:
            kind = cpu_kind()
            procs = os.cpu_count() or 1
            v, total, secs = run_cpu(kind, wl["map_size"], 20, args.cpu_steps, procs)
            line["cpu_baseline"] = {"value": v, "unit": "agent-steps/s", "cores": procs, "kind": kind,
                                    "sample": "%d independent single-thread envs (OMP_NUM_THREADS=1) x %d lockstep steps "
                                              "of the same hot loop, %.1f s" % (procs, args.cpu_steps, secs)}
            if kind == "reference":
                v2, secs2 = run_cpu_openmp(kind, wl["map_size"], 20, max(2000, args.cpu_steps // 10), procs)
                line["cpu_baseline"]["one_env_openmp"] = {
                    "value": v2, "threads": procs,
                    "note": "one env, the reference's intra-env OpenMP on all cores (%.1f s); racy by construction" % secs2}
        print(json.dumps(line), flush=True)
    ctx.close()


# ------------------------------------------------------------------------------------------------
# Ising (BASELINE configs[4]): 16384 lattices of 256x256 in total, strong-scaled over the GPUs
# ------------------------------------------------------------------------------------------------
def ising_cpu_sample(side, lattices, sweeps, T, lr):
    """numpy restatement (oracle/ising_oracle.py) on one core: the reference itself is O(N^2) per step and
    cannot run 256x256 (SURVEY F5)."""
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import numpy as np
    import ising_oracle
    rng = np.random.RandomState(13)
    spins = rng.randint(0, 2, size=(lattices, side, side))
    Q = np.zeros((lattices, 5, side * side, 2))
    ising_oracle.step(spins, Q, T, lr, rng.random_sample((lattices, side * side)))
    t0 = time.perf_counter()
    for _ in range(sweeps):
        spins, Q, _info = ising_oracle.step(spins, Q, T, lr, rng.random_sample((lattices, side * side)))
    secs = time.perf_counter() - t0
    return lattices * side * side * sweeps / secs, secs


def measure_ising(ctx, args, K, W):
    """BASELINE configs[4] on this rank's shard of the lattices: one region of exactly K sweeps; every rank must call
    it, rank 0 gets the JSON fields."""
    torch = ctx.torch
    from mfmarl_b200 import IsingMFQ
    dev, world, rank, local = ctx.dev, ctx.world, ctx.rank, ctx.local
    wl = WORKLOADS["c5"]
    total = (args.envs if args.workload == "c5" else 0) or wl["lattices"]
    B, L, T = total // world, wl["side"], wl["temperature"]
    model = IsingMFQ(B, L, seed=13, lr=wl["lr"], lattice_base=rank * B, device=dev)

    # --sweeps-per-launch S: S > 1 runs S sweeps per launch with the Q strip resident in shared memory (K6s / K6p / K6r,
    # mfi_run; same bits as S streaming launches); S = 1 is the streaming kernel K6 (mfi_step), one launch per sweep.
    S = args.sweeps_per_launch
    if S == 0:
        S = 100 if model.resident_cluster > 0 else 1
    S = max(1, min(S, K))
    while K % S:
        S -= 1                      # exactly K sweeps are timed
    resident = S > 1
    temps = torch.full((S,), T, dtype=torch.float32, device=dev)

    def sweep_block():
        if resident:
            return model.run(temps, resident=True)[0][-1]
        return model.step(T)[0]

    for _ in range(max(W // S, 2) if resident else W):
        sweep_block()
    ctx.barrier()

    def region():
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.barrier()
        t0.record()
        for _ in range(K // S):
            sweep_block()
        t1.record()
        ctx.barrier()
        return t0.elapsed_time(t1)

    with ClockSampler(local) as clocks:
        m0 = region()
    ms = ctx.reduce([m0], "max")[0]
    # e2e: what the driver loop of main_MFQ_Ising.py reads every sweep (up counts -> order parameter) lands in
    # pinned host memory; the temperature schedule goes host -> device with every launch
    h_up = torch.empty((S, B), dtype=torch.int32).pin_memory()
    h_temps = torch.full((S,), T, dtype=torch.float32).pin_memory()

    def e2e_region():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.barrier()
        e0.record()
        for _ in range(K // S):
            if resident:
                temps.copy_(h_temps, non_blocking=True)
                n_up, _r = model.run(temps, resident=True)
                h_up.copy_(n_up, non_blocking=True)
            else:
                n_up, _r, _m = model.step(float(h_temps[0]))
                h_up[0].copy_(n_up, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        e1.record()
        ctx.barrier()
        return e0.elapsed_time(e1)

    e2e_ms = ctx.reduce([e2e_region()], "max")[0]
    order_mean = float(model.order_param().mean())
    del model
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    peak, peak_src = measured_peak()
    sites = B * world * L * L
    achieved = B * L * L * BYTES_PER_SITE / (ms / K * 1e-3) / 1e9
    kernel = {"0": "k_ising_resident_f32", "1": "k_ising_persist_f32"}.get(
        os.environ.get("MFMARL_ISING_PERSIST", ""), "k_ising_persist_swar_f32") if resident else "k_ising"
    return {
        "metric": "ising MFQ site-steps/sec", "value": sites * K / (ms * 1e-3), "unit": "site-steps/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"], "lattices_total": B * world, "lattices_per_gpu": B, "side": L,
                   "temperature": T, "lr": wl["lr"], "rng": "philox(seed, lattice, column, band, step)",
                   "l2": "Q + spins per GPU (%.1f GB) exceed the 126 MB L2" % (B * L * L * 41 / 1e9),
                   "timed_region": "exactly %d sweeps, once, after the warm-up" % K},
        "region_ms": ms,
        "gpu_launches": K // S,
        "sweeps_per_launch": S,
        "roofline": {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak,
                     "traffic": (lambda t: None if t is None else t * B * L * L)(ncu_traffic(
                         "c5_resident_bytes_per_site_per_launch" if resident else "c5_stream_bytes_per_site_per_launch")),
                     "peak_source": peak_src,
                     "bytes_per_site": BYTES_PER_SITE, "sites_per_launch": B * L * L * S,
                     "note": ("algorithmic bytes are the STREAMING formulation's 14 B per site-step; the resident "
                              "kernel keeps Q in shared memory for %d sweeps and really moves (80 + 2) / %d B per "
                              "site-step, so frac > 1 means it beats the streaming bound" % (S, S)) if resident else
                             "streaming kernel: Q pair read + one value written + spins per site-step"},
        "e2e": {"value": sites * K / (e2e_ms * 1e-3), "unit": "site-steps/s", "h2d_bytes_per_step": 4 if resident else 0,
                "d2h_bytes_per_step": B * 4, "region_ms": e2e_ms,
                "note": "temperatures from pinned host memory per launch (a scalar argument when streaming); the "
                        "per-sweep up counts (order parameter) are read back to pinned host memory and waited "
                        "for after every launch"},
        "clocks": clocks.summary(),
        "order_param_mean": order_mean,
    }


def run_ising(args):
    ctx = Ctx()
    line = measure_ising(ctx, args, args.steps, args.warmup)
    if ctx.rank == 0:
        wl = WORKLOADS["c5"]
        if ctx.world == 1 and not args.no_cpu:
            v, secs = ising_cpu_sample(wl["side"], 4, 3, wl["temperature"], wl["lr"])
            line["cpu_baseline"] = {"value": v, "unit": "site-steps/s", "cores": 1, "kind": "port",
                                    "sample": "numpy restatement, 4 lattices of %dx%d x 3 sweeps, %.1f s (the "
                                              "reference's own loop is O(N^2)/step: ~1e4 site-steps/s at 20x20)"
                                              % (wl["side"], wl["side"], secs)}
        print(json.dumps(line), flush=True)
    ctx.close()


# ------------------------------------------------------------------------------------------------
# BASELINE configs[1]: ONE environment through the reference's own C ABI (host numpy buffers, every call synchronous)
# ------------------------------------------------------------------------------------------------
def run_single_env(args):
    wl = WORKLOADS["c2"]
    steps = max(200, args.steps * 10)
    cmd = [sys.executable, os.path.abspath(__file__), "--_cpu_worker", "cuda", str(wl["map_size"]), "50", str(steps), "7"]
    out = json.loads(subprocess.run(cmd, stdout=subprocess.PIPE, env=dict(os.environ, OMP_NUM_THREADS="1"))
                     .stdout.decode().strip().splitlines()[-1])
    v = out["agent_steps"] / out["seconds"]
    line = {"metric": "battle agent-steps/sec incl. obs+mean-action, single env via the reference C ABI", "value": v,
            "unit": "agent-steps/s", "n_gpus": 1, "steps": steps, "warmup": 50, "ms_per_step": out["seconds"] * 1e3 / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"],
                       "note": "magent.GridWorld over build/libmagent.so: get_observation x2 (device->host copies of the "
                               "views), set_action x2, step, get_reward/get_alive x2, clear_dead; wall clock, every call "
                               "synchronises.  A latency figure: one 64 v 64 env cannot fill a GPU."},
            "e2e": {"value": v, "unit": "agent-steps/s", "h2d_bytes_per_step": 2 * wl["cap"] * 4,
                    "d2h_bytes_per_step": 2 * wl["cap"] * (BYTES_PER_AGENT_OBS + 5)}}
    if not args.no_cpu and os.path.exists(REF_SO):
        rv, _total, secs = run_cpu("reference", wl["map_size"], 50, steps, 1)
        line["cpu_baseline"] = {"value": rv, "unit": "agent-steps/s", "cores": 1, "kind": "reference",
                                "sample": "the same loop on the reference engine, one process, %.1f s" % secs}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# rollout with the policy networks in the loop (SURVEY.md 8f rows 1-3): an additional line, not the headline
# ------------------------------------------------------------------------------------------------
def run_play(args):
    import torch
    from mfmarl_b200 import BatchedGridWorld
    from mfmarl_b200.algo import spawn_ai
    from mfmarl_b200.senario_battle import play_batched
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    wl = WORKLOADS["play"]
    E, K = args.envs or wl["envs"], args.steps
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    env = BatchedGridWorld(E, map_size=wl["map_size"], capacity=wl["cap"], device=dev, rng="philox", seed=0)

    class Spaces:
        def get_view_space(self, h): return (13, 13, 7)
        def get_feature_space(self, h): return (34,)
        def get_action_space(self, h): return (21,)

    models = [spawn_ai(args.algo, Spaces(), g, "%s-%d" % (args.algo, g), K, device=dev) for g in range(2)]
    if args.policy_precision == "tf32":
        torch.backends.cuda.matmul.allow_tf32 = True
        torch.backends.cudnn.allow_tf32 = True
    elif args.policy_precision == "bf16":
        for m in models:
            m.act_autocast = torch.bfloat16
    obs_dtype = torch.bfloat16 if args.policy_precision == "bf16rows" else None   # the engine emits the policy's input format
    play_batched(env, 0, max(3, args.warmup), models, eps=1.0, train=False, left_group=0, obs_dtype=obs_dtype)
    torch.cuda.synchronize()
    a0 = int(env.get("agent_steps").sum())
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(dev.index or 0) as clocks:
        t0.record()
        play_batched(env, 1, K, models, eps=1.0, train=False, left_group=0, obs_dtype=obs_dtype)
        t1.record()
        torch.cuda.synchronize()
    ms = t0.elapsed_time(t1)
    agent_steps = int(env.get("agent_steps").sum()) - a0
    print(json.dumps({
        "metric": "battle rollout agent-steps/sec incl. policy networks", "value": agent_steps / (ms * 1e-3),
        "unit": "agent-steps/s", "n_gpus": 1, "steps": K, "warmup": max(3, args.warmup), "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"], "envs_per_gpu": E, "algo": args.algo, "policy_precision": args.policy_precision,
                   "note": "play_batched: k_obs (per-group blocks) -> two PyTorch policy forwards on the observation "
                           "block in place -> k_step; nothing leaves the device except one `any(active)` flag per step"},
        "clocks": clocks.summary()}), flush=True)


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU engine on the host cores, same metric / config
# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    if args.workload == "c5":
        v, secs = ising_cpu_sample(wl["side"], 4, max(1, min(args.steps, 5)), wl["temperature"], wl["lr"])
        print(json.dumps({"impl": "reference", "metric": "ising MFQ site-steps/sec", "value": v,
                          "unit": "site-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": secs * 1e3 / max(1, min(args.steps, 5)), "higher_is_better": True,
                          "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": wl["name"]},
                          "cpu_baseline": {"value": v, "unit": "site-steps/s", "cores": 1, "kind": "port",
                                           "sample": "numpy restatement, 4 lattices x %d sweeps" % min(args.steps, 5)},
                          "e2e": {"value": v, "unit": "site-steps/s", "h2d_bytes_per_step": 0,
                                  "d2h_bytes_per_step": 0}}), flush=True)
        return
    kind = cpu_kind()
    procs = os.cpu_count() or 1
    # one reference "step" = every worker advances its own env by CHUNK lockstep steps; CHUNK is sized so that the
    # timed part is at least ~30000 steps per worker (about 5 s) whatever --steps is -- shorter samples under-report
    CHUNK = max(32, -(-30000 // max(1, args.steps)))
    v, total, secs = run_cpu(kind, wl["map_size"], min(args.warmup * CHUNK, 500), args.steps * CHUNK, procs)
    sample = ("%d independent single-thread envs of the %s engine (OMP_NUM_THREADS=1), each step = %d lockstep "
              "steps per env (bounded sample of the %d-env workload), %.1f s"
              % (procs, "reference C++" if kind == "reference" else "C oracle port", CHUNK, wl["envs"], secs))
    line = {
        "impl": "reference",
        "metric": "battle agent-steps/sec incl. obs+mean-action", "value": v, "unit": "agent-steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs * 1e3 / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"], "envs_per_gpu": wl["envs"], "map": wl["map_size"],
                   "agents_per_env": 2 * wl["cap"]},
        "cpu_baseline": {"value": v, "unit": "agent-steps/s", "cores": procs, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "--_cpu_worker":
        return cpu_worker(sys.argv[2:])
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: the workload's)")
    ap.add_argument("--cpu-steps", type=int, default=60000, help="timed steps per CPU-baseline worker")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--algo", default="mfq", choices=["mfq", "il", "mfac", "ac"], help="--workload play: the learner")
    ap.add_argument("--policy-precision", default="fp32", choices=["fp32", "tf32", "bf16", "bf16rows"],
                    help="--workload play: precision of the rollout forward pass (training is always fp32)")
    ap.add_argument("--obs-to-host-steps", type=int, default=5,
                    help="extra e2e variant: steps timed with the observations copied to the host too (0 = skip)")
    ap.add_argument("--pipeline", type=int, default=2,
                    help="split the GPU's envs into this many engines on separate streams, so that the latency-bound "
                         "k_step of one half runs under the bandwidth-bound k_obs of the other (1 = one engine, one stream)")
    ap.add_argument("--sweeps-per-launch", type=int, default=0,
                    help="c5: Ising sweeps per launch (1 = streaming kernel, >1 = shared-memory-resident kernel, 0 = auto)")
    ap.add_argument("--obs-tile", type=int, default=0, help="agents per k_obs CTA (tuning; 0 = engine default)")
    ap.add_argument("--step-threads", type=int, default=0, help="threads per k_step CTA (tuning; 0 = auto)")
    ap.add_argument("--no-also", action="store_true",
                    help="skip the extra legs of the default line (C4, C5, and the gradient all-reduce when N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="battle workloads: write what the last timed step returned (rank 0's environments) to "
                         "DIR/<name>.npy, float32, at most 64 MB.  The row mask needs the agent counts the last step "
                         "starts from, so one small device copy per engine is enqueued inside the timed region")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("c3", "c4")):
        ap.error("--dump-outputs: only the battle workloads c3 and c4 of --impl ours")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: relaunch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000),
               os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.workload == "c5":
        return run_ising(args)
    if args.workload == "play":
        return run_play(args)
    if args.workload == "c2":
        return run_single_env(args)
    run_ours(args)


if __name__ == "__main__":
    main()
