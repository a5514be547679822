"""IL (DQN) and MF-Q on top of ValueNet, with the reference's MemoryGroup replay
(algo/q_learning.py:9-171)."""
from . import base, tools
from .replay_device import DeviceMemoryGroup, DeviceStateMemoryGroup


class _ReplayMixin:
    """Host replay (reference semantics, single-env binding) and device replay (batched engine) side by side:
    `flush_buffer` feeds the first, `flush_buffer_batched` the second; `train` drains whichever was fed.

    replay_kind "rows": the device replay stores every observation row (DeviceMemoryGroup); "states": it stores one env
    state record per recorded env and step and renders the rows when it samples (DeviceStateMemoryGroup) -- the play
    loop then saves the records into `record_slice(env)` and passes them to `flush_buffer_batched(records=...)`."""
    use_mean = False

    def _init_replay(self, memory_size, batch_size, sub_len, device_memory_size=None, stage_rows=None, replay="rows"):
        if replay not in ("rows", "states"):
            raise ValueError("replay must be 'rows' or 'states', not %r" % (replay,))
        self.replay_buffer = tools.MemoryGroup(self.view_space, self.feature_space, self.num_actions, memory_size,
                                               batch_size, sub_len, use_mean=self.use_mean)
        self._replay_cfg = (device_memory_size or memory_size, batch_size, sub_len, stage_rows)
        self.replay_kind = replay
        self.device_replay = None

    def flush_buffer(self, **kwargs):
        self.replay_buffer.push(**kwargs)

    def _make_device_replay(self, env=None):
        max_len, batch_size, sub_len, stage_rows = self._replay_cfg
        common = dict(use_mean=self.use_mean, device=self.device, stage_rows=stage_rows)
        if self.replay_kind == "states":
            self.device_replay = DeviceStateMemoryGroup(self.view_space, self.feature_space, self.num_actions, max_len,
                                                        batch_size, sub_len, env.query("state_bytes"),
                                                        env.render_observations, **common)
        else:
            self.device_replay = DeviceMemoryGroup(self.view_space, self.feature_space, self.num_actions, max_len,
                                                   batch_size, sub_len, **common)

    def record_slice(self, env):
        """replay_kind "states": the arena slice (uint8[n_rec, R]) where this step's records of `env`'s first n_rec
        envs go, before they are passed to flush_buffer_batched(records=...)."""
        if self.device_replay is None:
            self._make_device_replay(env)
        return self.device_replay.record_slice(env.n_envs, env.capacity)

    def flush_buffer_batched(self, **kwargs):
        if self.device_replay is None:
            self._make_device_replay()
        self.device_replay.push(**kwargs)

    def _active_replay(self):
        if self.device_replay is not None and self.device_replay.has_staged:
            return self.device_replay
        return self.replay_buffer


class DQN(_ReplayMixin, base.ValueNet):
    use_mean = False

    def __init__(self, name, handle, env, sub_len, memory_size=2 ** 10, batch_size=64, update_every=5, device=None,
                 device_memory_size=None, stage_rows=None, replay="rows"):
        base.ValueNet.__init__(self, env, handle, name, update_every=update_every, device=device)
        self._init_replay(memory_size, batch_size, sub_len, device_memory_size, stage_rows, replay)

    def train(self, verbose=True):
        replay = self._active_replay()
        replay.tight()
        losses = []
        n_batches = replay.get_batch_num(verbose)
        if self.grad_sync:
            n_batches = base.agree_on_count(n_batches, self.device)
        for i in range(n_batches):
            obs, feats, obs_next, feat_next, dones, rewards, actions, masks = replay.sample()
            target_q = self.calc_target_q(obs=obs_next, feature=feat_next, rewards=rewards, dones=dones)
            loss, q = base.ValueNet.train(self, state=[obs, feats], target_q=target_q, acts=actions, masks=masks)
            self.update()
            losses.append(loss)
            if verbose and i % 50 == 0:
                print("[*] LOSS:", loss, "/ Q:", q)
        return losses

    def save(self, dir_path, step=0):
        self._save(dir_path, "dqn", step)

    def load(self, dir_path, step=0):
        self._load(dir_path, "dqn", step)


class MFQ(_ReplayMixin, base.ValueNet):
    use_mean = True

    def __init__(self, name, handle, env, sub_len, eps=1.0, update_every=5, memory_size=2 ** 10, batch_size=64,
                 device=None, device_memory_size=None, stage_rows=None, replay="rows"):
        base.ValueNet.__init__(self, env, handle, name, use_mf=True, update_every=update_every, device=device)
        self.train_ct = 0
        self._init_replay(memory_size, batch_size, sub_len, device_memory_size, stage_rows, replay)

    def train(self, verbose=True):
        replay = self._active_replay()
        replay.tight()
        losses = []
        n_batches = replay.get_batch_num(verbose)
        if self.grad_sync:
            n_batches = base.agree_on_count(n_batches, self.device)
        for i in range(n_batches):
            (obs, feat, acts, act_prob, obs_next, feat_next, act_prob_next, rewards, dones,
             masks) = replay.sample()
            target_q = self.calc_target_q(obs=obs_next, feature=feat_next, rewards=rewards, dones=dones,
                                          prob=act_prob_next)
            loss, q = base.ValueNet.train(self, state=[obs, feat], target_q=target_q, prob=act_prob, acts=acts,
                                          masks=masks)
            self.update()
            losses.append(loss)
            if verbose and i % 50 == 0:
                print("[*] LOSS:", loss, "/ Q:", q)
        return losses

    def save(self, dir_path, step=0):
        self._save(dir_path, "mfq", step)

    def load(self, dir_path, step=0):
        self._load(dir_path, "mfq", step)
