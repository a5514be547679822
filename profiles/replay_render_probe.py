"""The record-backed replay (train_battle.py --replay states) against the row replay (--replay rows): the render
kernel k_render_obs, the memory of both replays, and train_battle round times.

    python profiles/replay_render_probe.py --part kernel [--out FILE]
    python profiles/replay_render_probe.py --part memory [--out FILE]
    python profiles/replay_render_probe.py --part train [--max_steps 400] [--out FILE]

kernel   k_render_obs over a round's records: E envs stepped T steps with uniform random actions (auto-reset), every
         env saved after every observation.  Batches of random rows (record, group, slot < num) are rendered: CUDA
         events around `calls` launches, each with its own row list.  Bytes per row: 4868 written; read: the record
         header (96 B), the listed agents' positions (4 B each) and the row's own slots (16 B) -- a lower bound (the
         window's agents add their state and hp, the 338-B wall window comes from L2).  Beside it the gather the render
         replaces: rows mode's obs0[idx], feat0[idx] from a 2^20-row ring (5.1 GB).  The records exceed the 126 MB L2.
memory   the replay's device memory at train_battle.py's defaults (--envs 1024, 40x40, cap 64, 400 steps), from the
         tensor shapes (ring + staging + record arena), no GPU needed.
train    wall time of one train_battle.py round (rollout + training, engine and model set-up included), rows and
         states at equal recorded envs (--envs 40: rows records all 40) alternated twice after a warm-up run, then
         states and rows at --envs 1024 (states records 1024 envs, rows 40).

The card's name and power limit are read in the same run."""
import argparse
import contextlib
import io
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PY = os.path.join(REPO, "mean-field-multi-agent-reinforcement-learning_b200", "python")
sys.path.insert(0, PY)

HBM_PEAK = 7.7e12          # HGX B200 data sheet, one GPU, 1000 W part
ROW_BYTES = (13 * 13 * 7 + 34) * 4   # 4868: one observation row (view + features)


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as ex:   # the probe still reports its numbers
        return "unknown (%s)" % ex


def kernel(out, calls=20):
    import torch
    from mfmarl_b200 import BatchedGridWorld
    from mfmarl_b200.scenarios import c4_positions, generate_map_positions
    torch.manual_seed(0)
    ring = torch.zeros((1 << 20, 13, 13, 7)), torch.zeros((1 << 20, 34))
    ring = ring[0].cuda(), ring[1].cuda()
    for name, m, cap, E, T, pos in [("C3 40x40 64v64", 40, 64, 1024, 40, None),
                                    ("C4 80x80 512v512", 80, 512, 128, 40, c4_positions())]:
        left, right = pos if pos is not None else generate_map_positions(m)
        env = BatchedGridWorld(E, map_size=m, capacity=cap, rng="philox", seed=1, max_steps=400, auto_reset=True)
        env.reset(); env.add_agents(0, left); env.add_agents(1, right)
        R = env.query("state_bytes")
        records = torch.empty((E * T, R), dtype=torch.uint8, device="cuda")
        for t in range(T):
            env.observe_groups()
            env.save_envs(out=records[t * E:(t + 1) * E])
            env.step(torch.randint(0, 21, (E, 2, env.capacity), dtype=torch.int32, device="cuda"))
        num = records[:, 40:48].contiguous().view(torch.int32).to(torch.int64)          # [n, 2]
        for B in (2560, 65536):
            lists, read = [], 0.0
            for _ in range(calls + 3):
                r = torch.randint(0, E * T, (B,), device="cuda")
                g = torch.randint(0, 2, (B,), device="cuda")
                n = num[r, g]
                s = (torch.rand(B, device="cuda") * n).long()
                lists.append(torch.stack([r, g, s], 1).to(torch.int32).contiguous())
                read += float((96 + 16 + 4 * num[r].sum(1)).double().mean()) / (calls + 3)
            bad = torch.zeros((1,), dtype=torch.int32, device="cuda")
            for k in range(3):
                env.render_observations(records, lists[k], bad_rows=bad)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(3, calls + 3):
                env.render_observations(records, lists[k])
            e1.record()
            torch.cuda.synchronize()
            t_render = e0.elapsed_time(e1) * 1e-3 / calls
            idx = [torch.randint(0, 1 << 20, (B,), device="cuda") for _ in range(calls + 3)]
            for k in range(3):
                ring[0][idx[k]]; ring[1][idx[k]]
            e0.record()
            for k in range(3, calls + 3):
                ring[0][idx[k]]; ring[1][idx[k]]
            e1.record()
            torch.cuda.synchronize()
            t_gather = e0.elapsed_time(e1) * 1e-3 / calls
            moved = B * (ROW_BYTES + read)
            out("%-17s records %6d x %5d B = %6.0f MB  batch %6d rows: render %8.1f us  %7.2f M rows/s  "
                "%5.0f B read/row  %6.0f GB/s = %4.2f of %.1f TB/s  (zero rows %d) | row gather %8.1f us  %6.0f GB/s  "
                "render/gather %.2f" % (
                    name, E * T, R, E * T * R / 1e6, B, t_render * 1e6, B / t_render / 1e6, read, moved / t_render / 1e9,
                    moved / t_render / HBM_PEAK, HBM_PEAK / 1e12, int(bad), t_gather * 1e6,
                    2 * B * ROW_BYTES / t_gather / 1e9, t_render / t_gather))
        del env, records


def memory(out):
    envs, cap, steps = 1024, 64, 400
    R = 96 + 64 * cap
    prob, common = 21 * 4, 4 + 4 + 1   # act + rew + term
    rows_ring = 1 << 20
    rows_row = ROW_BYTES + common + 1 + prob                 # + mask
    rows_stage = ROW_BYTES + common + 8 + 8 + prob            # + key, t
    st_ring = min(1 << 25, envs * cap * steps)
    st_row = 12 + common + 1 + prob
    st_stage = 12 + common + 8 + 8 + prob
    rec_rows = max(1, min(envs, rows_ring // (cap * steps)))
    rec_st = max(1, min(envs, st_ring // (cap * steps)))
    arena_round = rec_st * steps * R
    out("rows   ring %8d x %4d B = %5.2f GB, staging %8d x %4d B = %5.2f GB: %5.2f GB, records %4d of %d envs "
        "(%.0f B per row)" % (rows_ring, rows_row, rows_ring * rows_row / 1e9, rows_ring, rows_stage,
                              rows_ring * rows_stage / 1e9, rows_ring * (rows_row + rows_stage) / 1e9, rec_rows, envs,
                              rows_row))
    out("states ring %8d x %4d B = %5.2f GB, staging %8d x %4d B = %5.2f GB, arena %d B per recorded env-step: "
        "%5.2f GB per round of %d steps -> %5.2f GB with one round's records, %5.2f GB with two; records %4d of %d envs "
        "(%.0f B per row)" % (st_ring, st_row, st_ring * st_row / 1e9, st_ring, st_stage, st_ring * st_stage / 1e9, R,
                              arena_round / 1e9, steps, (st_ring * (st_row + st_stage) + arena_round) / 1e9,
                              (st_ring * (st_row + st_stage) + 2 * arena_round) / 1e9, rec_st, envs, st_row))


def train(out, max_steps):
    import importlib.util
    import random
    import tempfile
    import torch
    spec = importlib.util.spec_from_file_location("train_battle", os.path.join(PY, "train_battle.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    tmp = tempfile.mkdtemp(prefix="replay_probe_")

    def one(envs, replay, tag):
        torch.manual_seed(0); random.seed(0); np.random.seed(0)
        argv = ["--algo", "mfq", "--envs", str(envs), "--n_round", "1", "--max_steps", str(max_steps), "--save_every",
                "1000", "--replay", replay, "--data_dir", os.path.join(tmp, tag)]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        log = io.StringIO()
        with contextlib.redirect_stdout(log):
            runner = mod.main(argv)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        rep = runner.models[0].device_replay
        new_rows = int(rep.length)
        mem = torch.cuda.max_memory_allocated() / 1e9
        torch.cuda.reset_peak_memory_stats()
        out("%-6s --envs %4d --max_steps %d: round %7.2f s  (ring rows after the round %9d, recorded envs %4d, "
            "peak allocated %5.1f GB)" % (replay, envs, max_steps, dt, new_rows,
                                          rep.n_rec_envs(envs, 64), mem))
        del runner, rep
        torch.cuda.empty_cache()
        return dt

    one(40, "rows", "warm")
    for k in range(2):
        for replay in ("rows", "states"):
            one(40, replay, "%s%d" % (replay, k))
    one(1024, "states", "states1024")
    one(1024, "rows", "rows1024")


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--part", choices=("kernel", "memory", "train"), required=True)
    ap.add_argument("--max_steps", type=int, default=400)
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    f = open(a.out, "w") if a.out else None

    def out(line):
        print(line, flush=True)
        if f:
            f.write(line + "\n"); f.flush()
    if a.part != "memory":
        out("card: " + card())
    {"kernel": kernel, "memory": memory, "train": lambda o: train(o, a.max_steps)}[a.part](out)


if __name__ == "__main__":
    main()
