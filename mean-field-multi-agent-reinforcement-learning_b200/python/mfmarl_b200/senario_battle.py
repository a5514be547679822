"""The battle scenario of the reference (examples/battle_model/senario_battle.py): map generation and the rollout
loop, in two forms.

* `play` / `battle` drive ONE environment through the `magent.GridWorld` binding with exactly the reference's call
  order and bookkeeping (senario_battle.py:41-192 and :196-284), so the reference's `Runner`, `train_battle.py` and
  `battle.py` logic runs unchanged over the CUDA engine (models are the PyTorch ones of `mfmarl_b200.algo`).
* `play_batched` runs the same loop for E lock-stepped environments of a `BatchedGridWorld`: observations, mean
  actions, rewards and alive flags never leave the GPU; the policy networks consume the observation block in
  place and the replay buffers are device-resident (`algo.replay_device`).
"""
import math
import random

import numpy as np


def map_positions(map_size):
    """The two 8x8 (at 40x40) army blocks of senario_battle.py:8-38 -> (left, right) lists of [x, y, 0]."""
    width = height = map_size
    side = int(math.sqrt(map_size * map_size * 0.04)) * 2
    gap = 3
    y0 = (height - side) // 2
    left = [[x, y, 0] for x in range(width // 2 - gap - side, width // 2 - gap, 2) for y in range(y0, y0 + side, 2)]
    right = [[x, y, 0] for x in range(width // 2 + gap, width // 2 + gap + side, 2) for y in range(y0, y0 + side, 2)]
    return left, right


def generate_map(env, map_size, handles):
    """senario_battle.py:8-38: which handle gets the left block is one random.randint(0, 1) draw; the left block is
    added first (and therefore gets the lower agent ids)."""
    left, right = map_positions(map_size)
    left_id = random.randint(0, 1)
    env.add_agents(handles[left_id], method="custom", pos=left)
    env.add_agents(handles[1 - left_id], method="custom", pos=right)


def _rollout(env, n_round, map_size, max_steps, handles, models, print_every, eps, render, train):
    env.reset()
    generate_map(env, map_size, handles)
    n_group = len(handles)
    state, acts, ids = [None] * n_group, [None] * n_group, [None] * n_group
    alives, rewards = [None] * n_group, [None] * n_group
    nums = [env.get_num(handle) for handle in handles]
    max_nums = nums.copy()
    n_action = [env.get_action_space(handle)[0] for handle in handles]
    print("\n\n[*] ROUND #{0}, EPS: {1:.2f} NUMBER: {2}".format(n_round, eps, nums))
    mean_rewards = [[] for _ in range(n_group)]
    total_rewards = [[] for _ in range(n_group)]
    former_act_prob = [np.zeros((1, n)) for n in n_action]
    eye = [np.eye(n) for n in n_action]
    step_ct, done = 0, False
    while not done and step_ct < max_steps:
        for i in range(n_group):
            state[i] = list(env.get_observation(handles[i]))
            ids[i] = env.get_agent_id(handles[i])
        for i in range(n_group):
            former_act_prob[i] = np.tile(former_act_prob[i], (len(state[i][0]), 1))
            acts[i] = models[i].act(state=state[i], prob=former_act_prob[i], eps=eps)
        for i in range(n_group):
            env.set_action(handles[i], acts[i])
        done = env.step()
        for i in range(n_group):
            rewards[i] = env.get_reward(handles[i])
            alives[i] = env.get_alive(handles[i])
        if train:   # the main model's transition: the mean action it SAW goes in with it (senario_battle.py:125-130)
            models[0].flush_buffer(state=state[0], acts=acts[0], rewards=rewards[0], alives=alives[0], ids=ids[0],
                                   prob=former_act_prob[0])
        for i in range(n_group):   # group mean action of this step, over every agent that acted (:141)
            former_act_prob[i] = np.mean(eye[i][acts[i]], axis=0, keepdims=True)
        nums = [env.get_num(handle) for handle in handles]
        for i in range(n_group):
            sum_reward = sum(rewards[i])
            rewards[i] = sum_reward / nums[i]
            mean_rewards[i].append(rewards[i])
            total_rewards[i].append(sum_reward)
        if render:
            env.render()
        env.clear_dead()
        step_ct += 1
        if step_ct % print_every == 0:
            print("> step #{}, info: {}".format(step_ct, {"Ave-Reward": np.round(rewards, decimals=6), "NUM": nums}))
    if train:
        models[0].train()
    for i in range(n_group):
        mean_rewards[i] = sum(mean_rewards[i]) / len(mean_rewards[i])
        total_rewards[i] = sum(total_rewards[i])
    return max_nums, nums, mean_rewards, total_rewards


def play(env, n_round, map_size, max_steps, handles, models, print_every, eps=1.0, render=False, train=False):
    """One training round (senario_battle.py:41-192)."""
    return _rollout(env, n_round, map_size, max_steps, handles, models, print_every, eps, render, train)


def battle(env, n_round, map_size, max_steps, handles, models, print_every, eps=1.0, render=False, train=False):
    """One evaluation round (senario_battle.py:196-284): the same loop, nothing is stored or trained."""
    return _rollout(env, n_round, map_size, max_steps, handles, models, print_every, eps, render, False)


# ----------------------------------------------------------------------------------------------------------
# batched, device-resident form
# ----------------------------------------------------------------------------------------------------------
def play_batched(env, n_round, max_steps, models, eps=1.0, train=False, print_every=0, left_group=None,
                 positions=None, obs_dtype=None, host_lag=None, mean_field="group", mf_radius=None):
    """E episodes in lockstep on a `BatchedGridWorld` (one per environment), everything on the device.

    Per environment this is the loop of `play`: observe both groups -> models[g].act on the group's rows (with the
    group's previous mean action tiled per agent) -> step (set_action x2, step, reward, alive, mean action,
    clear_dead in one launch) -> statistics.  An environment stops contributing once it is done; the round ends when
    all are done or after max_steps.  With train=True the main model's transitions (group 0 rows of the active
    environments) go to its device replay buffer via `flush_buffer_batched`, and `train()` runs once at the end.

    obs_dtype=torch.bfloat16: the policies act on the engine's bf16 NHWC-8 observation rows (no cast, no padding pass,
    bf16 tensor cores; see algo.base.bf16_rollout_copy); the fp32 rows are still produced for the replay buffer when
    train=True.

    host_lag: how many steps the host may run ahead of the device before it looks at the "any environment still
    playing" flag (see below); None = 2 on a CUDA device, 0 = ask after every step.

    mean_field: which mean action the policies see.  "group" (the reference's, senario_battle.py:141): every agent of
    a group gets the one-hot mean of the whole group's previous actions.  "local": agent j gets the mean over its
    group-mates inside the disc of radius `mf_radius` (None = the view radius) that acted last step
    (`BatchedGridWorld.local_mean_action`), zeros before the first step; the replay then stores each agent's own row.

    Returns (max_nums [E, 2], nums [E, 2], mean_rewards [E, 2], total_rewards [E, 2]) as numpy arrays.
    """
    import torch
    if mean_field not in ("group", "local"):
        raise ValueError("mean_field must be 'group' or 'local', not %r" % (mean_field,))
    local = mean_field == "local"
    E, cap = env.n_envs, env.capacity
    dev = env.device
    if positions is None:
        positions = map_positions(env.map_size)
    if left_group is None:
        left_group = random.randint(0, 1)
    env.reset()
    env.add_agents(left_group, positions[0])
    env.add_agents(1 - left_group, positions[1])
    n_action = env.sizes["n_action"]
    if local:
        local_mean = env.local_mean_action(radius=mf_radius)    # nobody has acted yet: all rows zero
    live_num, live_id = env.device_state("num"), env.device_state("id")    # aliases of the engine's HBM state
    num = live_num.clone()                                                 # [E, 2] agents at observation time
    max_nums, final_nums = num.clone(), num.clone()
    former = torch.zeros((E, 2, n_action), dtype=torch.float32, device=dev)
    active = torch.ones((E,), dtype=torch.bool, device=dev)
    slot = torch.arange(cap, device=dev, dtype=torch.int32)
    sum_mean = torch.zeros((E, 2), dtype=torch.float64, device=dev)
    sum_total = torch.zeros((E, 2), dtype=torch.float64, device=dev)
    steps_run = torch.zeros((E,), dtype=torch.int64, device=dev)
    actions = torch.zeros((E, 2, cap), dtype=torch.int32, device=dev)
    step_ct = 0
    # "is any environment still playing" is the one thing the host has to learn from the device.  Asking after every
    # step would make the host wait for the step it has just enqueued before it can enqueue the next one (for the
    # dense MF-AC network the GPU then idles a quarter of the time, profiles/r02/play_busy_probe.txt), so the flag
    # travels to pinned memory behind each step and the host looks at the one from TWO steps back: it runs one step
    # ahead of the device.  After the last environment finishes, at most two more steps run with every environment
    # masked out (`active` gates the statistics and the replay rows), which changes nothing that is returned.
    lag = (2 if dev.type == "cuda" else 0) if host_lag is None else int(host_lag)
    flags = [torch.ones((1,), dtype=torch.bool).pin_memory() if lag else None for _ in range(max(lag, 1))]
    events = [torch.cuda.Event() if lag else None for _ in range(max(lag, 1))]

    def still_playing():
        if not lag:
            return bool(active.any())
        if step_ct < lag:
            return True
        events[step_ct % lag].synchronize()           # recorded behind step step_ct - lag
        return bool(flags[step_ct % lag][0])

    while step_ct < max_steps and still_playing():
        if obs_dtype is not None and obs_dtype != torch.float32:
            act_obs = env.observe_groups(dtype=obs_dtype)  # bf16 [E, cap, 13, 13, 8] rows for the policies
            obs = env.observe_groups(groups=(0,)) if train else act_obs
        else:
            obs = act_obs = env.observe_groups()           # per group: view [E, cap, 13, 13, 7], feature [E, cap, 34]
        num.copy_(live_num)
        ids = live_id.clone()                              # rows of this step, before clear_dead compacts them
        valid = (slot[None, None, :] < num[:, :, None]) & active[:, None, None]          # [E, 2, cap]
        for g in range(2):
            view, feat = act_obs[g]
            if local:
                prob = local_mean[g].view(E * cap, n_action)
            else:
                prob = former[:, g, None, :].expand(E, cap, n_action).reshape(E * cap, n_action)
            a = models[g].act(state=[view.view((E * cap,) + tuple(view.shape[2:])), feat.view(E * cap, -1)],
                              prob=prob, eps=eps)
            actions[:, g] = a.reshape(E, cap)
        actions.masked_fill_(~valid, 0)
        reward, alive, done, mean = env.step(actions, want_mean_action=not local)
        if train:
            models[0].flush_buffer_batched(state=obs[0], acts=actions[:, 0], rewards=reward[:, 0], alives=alive[:, 0],
                                           ids=ids[:, 0], prob=local_mean[0] if local else former[:, 0], num=num[:, 0],
                                           active=active)
        if local:
            # the next step's rows; enqueued after the flush above has read this step's on the same stream
            local_mean = env.local_mean_action(radius=mf_radius)
        # statistics (senario_battle.py:146-152): nums still include the agents that died this step
        r = torch.where(valid, reward, torch.zeros_like(reward)).to(torch.float64).sum(dim=2)   # [E, 2]
        act_f = active[:, None].to(torch.float64)
        sum_total += r * act_f
        sum_mean += r / num.clamp(min=1).to(torch.float64) * act_f
        steps_run += active.to(torch.int64)
        # the reference reads get_num BEFORE the step's clear_dead (senario_battle.py:146): the agents that died in an
        # environment's last step still count, which is what Runner's `kill` statistic is built on
        final_nums = torch.where(active[:, None], num, final_nums)
        if not local:
            former = torch.where(active[:, None, None], mean, former)
        active = active & (done == 0)
        if lag:
            flags[step_ct % lag].copy_(active.any().reshape(1), non_blocking=True)
            events[step_ct % lag].record()
        step_ct += 1
        if print_every and step_ct % print_every == 0:
            print("> step #{}, active envs: {}, agents: {}".format(step_ct, int(active.sum()),
                                                                   final_nums.sum(dim=0).tolist()))
    num = final_nums
    if train:
        models[0].train()
    steps = steps_run.clamp(min=1).to(torch.float64)[:, None]
    return (max_nums.cpu().numpy(), num.cpu().numpy(), (sum_mean / steps).cpu().numpy(), sum_total.cpu().numpy())
