"""PyTorch re-expression of the reference's learning algorithms (examples/battle_model/algo/), consuming the
engine's observations and the group mean action.  Same duck type as the TF1 models -- `act(state=, prob=, eps=)`,
`flush_buffer(**)`, `train()`, `save/load` -- so the reference's play loop can drive them unchanged.

    MFQ   mean-field Q-learning      algo/q_learning.py:74-143 + base.py (use_mf=True)
    IL    independent Q-learning     algo/q_learning.py:9-71   (DQN)
    AC    actor-critic               algo/ac.py:8-176
    MFAC  mean-field actor-critic    algo/ac.py:178-361
"""
from . import ac, q_learning, tools
from .ac import MFAC, ActorCritic
from .q_learning import DQN, MFQ

AC = ActorCritic
IL = DQN


def spawn_ai(algo_name, env, handle, human_name, max_steps, device=None, device_rows=None, batch_size=64, replay="rows"):
    """algo/__init__.py:10-19 without the TF session argument.  device_rows sizes the HBM-resident replay of the batched
    loop (rows of one agent-step, 4.9 KB each; default: the reference's 80000-row ring / 2^18 episode rows); batch_size is the Q learners' minibatch
    (q_learning.py:85: 64).  replay: the Q learners' device replay, "rows" (observation rows) or "states" (env state
    records, rows rendered when sampled: ~100 B per row); the actor-critic learners have "rows" only."""
    if replay != "rows" and algo_name not in ("mfq", "il"):
        raise ValueError("replay=%r needs a Q learner (mfq, il), not %r" % (replay, algo_name))
    if algo_name == "mfq":
        return MFQ(human_name, handle, env, max_steps, memory_size=80000, batch_size=batch_size, device=device,
                   device_memory_size=device_rows, replay=replay)
    if algo_name == "mfac":
        return MFAC(human_name, handle, env, device=device, sub_len=max_steps, **({"stage_rows": device_rows} if device_rows else {}))
    if algo_name == "ac":
        return AC(human_name, handle, env, device=device, sub_len=max_steps, **({"stage_rows": device_rows} if device_rows else {}))
    if algo_name == "il":
        return IL(human_name, handle, env, max_steps, memory_size=80000, batch_size=batch_size, device=device,
                  device_memory_size=device_rows, replay=replay)
    raise ValueError("unknown algorithm %r (choose from mfq, mfac, ac, il)" % (algo_name,))


__all__ = ["spawn_ai", "MFQ", "DQN", "IL", "ActorCritic", "AC", "MFAC", "tools", "ac", "q_learning"]
