"""Self-play training on the battle scenario -- the reference's train_battle.py with the same flags, over the CUDA
engine and the PyTorch learners.

    python train_battle.py --algo mfq                   one environment through the magent binding (reference loop)
    python train_battle.py --algo mfq --envs 1024       1024 lock-stepped environments on the GPU per round:
                                                         observations, mean actions and replay stay in HBM
    python train_battle.py --algo mfq --envs 1024 --mean_field local
                                                        the same with each agent's neighbourhood mean action
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

BASE_DIR = os.path.dirname(os.path.abspath(__file__))


def linear_decay(epoch, x, y):
    """piecewise-linear schedule through the points (x[i], y[i]) (train_battle.py:19-40)"""
    if epoch == x[0]:
        return y[0]
    eps = y[0]
    for i, x_i in enumerate(x):
        if epoch <= x_i:
            slope = (y[i] - y[i - 1]) / (x_i - x[i - 1])
            eps = slope * (epoch - x[i - 1]) + y[i - 1]
            break
    return eps


class BatchedEnvAdapter:
    """What Runner / spawn_ai ask of `env` (space queries) on top of a BatchedGridWorld, plus a `play` handle that
    reduces the per-environment statistics of play_batched to the scalars Runner logs (means over environments)."""

    def __init__(self, benv, rollout_bf16=False, mean_field="group"):
        self.benv, self.rollout_bf16, self.mean_field = benv, rollout_bf16, mean_field

    def get_view_space(self, handle):
        s = self.benv.sizes
        return (s["view_size"], s["view_size"], s["n_channel"])

    def get_feature_space(self, handle):
        return (self.benv.sizes["feature_size"],)

    def get_action_space(self, handle):
        return (self.benv.sizes["n_action"],)

    def play(self, env, n_round, map_size, max_steps, handles, models, print_every, eps=1.0, render=False, train=False):
        import numpy as np
        import torch
        from mfmarl_b200.senario_battle import play_batched
        print("\n\n[*] ROUND #{0}, EPS: {1:.2f} ENVS: {2}".format(n_round, eps, self.benv.n_envs))
        # every rank places the armies the same way round (the draw of senario_battle.py:14 comes from the round number)
        max_nums, nums, mean_r, total_r = play_batched(self.benv, n_round, max_steps, models, eps=eps, train=train,
                                                       print_every=print_every, left_group=n_round % 2,
                                                       obs_dtype=torch.bfloat16 if self.rollout_bf16 else None,
                                                       mean_field=self.mean_field)
        stats = np.stack([max_nums.mean(axis=0), nums.mean(axis=0), mean_r.mean(axis=0), total_r.mean(axis=0)])
        stats = all_ranks_mean(stats, self.benv.device)     # one decision (self-play update, win count) on every rank
        return tuple(list(row) for row in stats)


def all_ranks_mean(array, device):
    """mean over the torch.distributed ranks (a no-op for one process)"""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return array
    t = torch.as_tensor(array, dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return (t / dist.get_world_size()).cpu().numpy()


def init_distributed(device_arg):
    """One process per GPU under torchrun: rank r owns environments [r * E, (r + 1) * E) and the learners average their
    gradients (algo.base.sync_gradients) -- the only collective anywhere near the path (SURVEY.md section 8e)."""
    import torch
    import torch.distributed as dist
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    if world == 1:
        return 1, 0, device_arg
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if torch.cuda.is_available():
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return world, rank, "cuda:%d" % local
    dist.init_process_group("gloo")
    return world, rank, device_arg


def main(argv=None):
    from mfmarl_b200.cli import battle_parser, check_battle_args, data_dirs
    ap = battle_parser("self-play training on the battle scenario", training=True)
    args = check_battle_args(ap, ap.parse_args(argv))
    args.data_dir, render_dir = data_dirs(args, BASE_DIR)

    from mfmarl_b200.algo import spawn_ai, tools
    world, rank, args.device = init_distributed(args.device)
    if world > 1:
        import torch
        assert args.envs > 0, "multi-GPU training shards the lock-stepped environments: pass --envs"
        torch.manual_seed(0)                  # identical initial weights on every rank
    log_dir = os.path.join(args.data_dir, 'tmp')
    model_dir = os.path.join(args.data_dir, 'models/{}'.format(args.algo))
    if args.envs > 0:
        from mfmarl_b200 import BatchedGridWorld
        cap = max(64, int(args.map_size * args.map_size * 0.04))
        benv = BatchedGridWorld(args.envs, map_size=args.map_size, capacity=cap, device=args.device, rng="philox",
                                env_base=rank * args.envs)
        env = BatchedEnvAdapter(benv, rollout_bf16=args.rollout_bf16, mean_field=args.mean_field)
        handles, play = [0, 1], env.play
    else:
        import magent
        from mfmarl_b200.senario_battle import play
        env = magent.GridWorld('battle', map_size=args.map_size)
        env.set_render_dir(render_dir)
        handles = env.get_handles()
    # batched rounds produce envs x agents x steps rows: give the device replay room for up to 2^20 of them (5 GB)
    device_rows = min(1 << 20, args.envs * cap * args.max_steps) if args.envs > 0 else None
    # ... and scale the Q learners' minibatch with the number of recorded environments, so that a round keeps the
    # reference's number of gradient steps (new rows * 2 / batch, tools.py:352-360) instead of multiplying it
    rec_envs = max(1, min(args.envs, device_rows // (cap * args.max_steps))) if args.envs > 0 else 1
    models = [spawn_ai(args.algo, env, handles[0], args.algo + '-me', args.max_steps, device=args.device,
                       device_rows=device_rows, batch_size=64 * rec_envs),
              spawn_ai(args.algo, env, handles[1], args.algo + '-opponent', args.max_steps, device=args.device)]
    for m in models:
        m.grad_sync = world > 1
        if world > 1 and hasattr(m, "generator"):
            m.generator.manual_seed(1234 + rank)      # stochastic policies explore differently on every rank
    if rank > 0:                              # one rank writes checkpoints and logs
        model_dir, log_dir = os.path.join(model_dir, 'rank%d' % rank), os.path.join(log_dir, 'rank%d' % rank)
    runner = tools.Runner(env, handles, args.map_size, args.max_steps, models, play,
                          render_every=args.save_every if args.render else 0, save_every=args.save_every, tau=0.01,
                          log_name=args.algo, log_dir=log_dir, model_dir=model_dir, train=True)
    for k in range(0, args.n_round):
        eps = linear_decay(k, [0, int(args.n_round * 0.8), args.n_round], [1, 0.2, 0.1])
        runner.run(eps, k)
    if os.environ.get("MFMARL_SAVE_FINAL"):   # test hook: every rank dumps the main model's parameters
        import torch
        torch.save([p.detach().cpu() for p in models[0].vars], os.path.join(args.data_dir, "final_rank%d.pt" % rank))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return runner


if __name__ == '__main__':
    main()
