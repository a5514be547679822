"""Command-line plumbing shared by train_battle.py and battle.py: the reference scripts' flag names
(train_battle.py:44-77, battle.py:22-31) so existing command lines keep working, plus the options this package adds."""
import argparse
import os

ALGOS = ("ac", "mfac", "mfq", "il")


def battle_parser(description, training):
    ap = argparse.ArgumentParser(description=description)
    ap.add_argument("--algo", choices=ALGOS, required=True, help="learner of the main group")
    if training:
        ap.add_argument("--save_every", type=int, default=10, help="rounds between self-play checkpoints / renders")
        ap.add_argument("--update_every", type=int, default=5, help="target-network update interval of the Q learners")
        ap.add_argument("--n_round", type=int, default=2000, help="training rounds")
    else:
        ap.add_argument("--oppo", choices=ALGOS, help="learner of the opposing group")
        ap.add_argument("--n_round", type=int, default=50, help="evaluation rounds")
        ap.add_argument("--idx", nargs="*", required=True, help="checkpoint steps to load: main opponent")
    ap.add_argument("--render", action="store_true", help="write the render trace (config.json, video_N.txt)")
    ap.add_argument("--map_size", type=int, default=40, help="side of the square map (40 -> 64 agents per group)")
    ap.add_argument("--max_steps", type=int, default=400, help="episode horizon")
    ap.add_argument("--device", default=None, help="torch device of the learners (default: cuda)")
    ap.add_argument("--data_dir", default=None, help="where models, logs and render traces go (default: ./data)")
    if training:
        ap.add_argument("--envs", type=int, default=0,
                        help="lock-stepped environments on the GPU per round (0 = one environment via magent)")
        ap.add_argument("--rollout_bf16", action="store_true",
                        help="with --envs: the policies act on bf16 observation rows emitted by the engine (bf16 twins of "
                             "the networks; training stays fp32 on the fp32 rows)")
        ap.add_argument("--mean_field", choices=("group", "local"), default="group",
                        help="mean action of the mean-field learners: 'group' = over the whole group (the reference's), "
                             "'local' = over each agent's group-mates within its view radius (needs --envs)")
    return ap


def check_battle_args(ap, args):
    """combinations argparse cannot express; exits with a usage error like argparse itself"""
    if getattr(args, "mean_field", "group") == "local" and args.envs <= 0:
        ap.error("--mean_field local needs the batched engine: pass --envs N (N > 0)")
    return args


def data_dirs(args, base_dir):
    root = args.data_dir or os.path.join(base_dir, "data")
    render = os.path.join(root, "render")
    os.makedirs(render, exist_ok=True)
    return root, render
