"""Device-resident replay for the batched engine: the data structures of the reference's algo/tools.py with every
row kept in HBM, fed straight from the engine's observation / action / reward tensors.

`DeviceMemoryGroup`  = `MemoryGroup` (tools.py:223-362): per-agent trajectories are appended to a ring in a random
agent order, `mask = not terminal` with the last row of every trajectory masked out (its ring successor belongs
to another agent), `sample` draws idx uniformly and pairs it with (idx + 1) % nb_entries.
`DeviceEpisodesBuffer` = `EpisodesBuffer` (tools.py:122-173): whole trajectories per agent for the actor-critic
update, returned sorted by (agent, time) together with the segment structure.

An agent is identified by (environment, agent id); one call of `push` stores one lockstep step of group rows
[E, cap] and nothing is copied to the host.  Because a lockstep step of thousands of environments produces far more
rows than a replay ring holds, only the first `n_rec_envs` environments are recorded (all of them when the staging
area is large enough).
"""
import torch


class _Staging:
    """Time-major staging rows of the current round: fixed-capacity device tensors + a device-side cursor."""

    def __init__(self, rows, obs_shape, feat_shape, act_n, use_mean, device):
        self.rows, self.device, self.use_mean = rows, device, use_mean
        n = rows + 1                                     # the extra row swallows the writes of invalid slots
        self.obs = torch.empty((n,) + tuple(obs_shape), dtype=torch.float32, device=device)
        self.feat = torch.empty((n,) + tuple(feat_shape), dtype=torch.float32, device=device)
        self.act = torch.empty((n,), dtype=torch.int32, device=device)
        self.rew = torch.empty((n,), dtype=torch.float32, device=device)
        self.term = torch.empty((n,), dtype=torch.bool, device=device)
        self.key = torch.empty((n,), dtype=torch.int64, device=device)
        self.t = torch.empty((n,), dtype=torch.int64, device=device)
        self.prob = torch.empty((n, act_n), dtype=torch.float32, device=device) if use_mean else None
        self.cursor = torch.zeros((), dtype=torch.int64, device=device)
        self.upper = 0                                   # host-side upper bound of the cursor
        self.step = 0

    def reset(self):
        self.cursor.zero_()
        self.upper, self.step = 0, 0

    def push(self, n_rec, id_span, view, feat, acts, rewards, alives, ids, prob, num, active):
        """Append the valid rows (slot < num[e], env active) of the first n_rec envs; no host synchronisation."""
        E, cap = acts.shape
        n_rec = min(n_rec, E)
        if self.upper + n_rec * cap > self.rows:         # only now is the exact fill level needed
            self.upper = int(self.cursor)
            if self.upper + n_rec * cap > self.rows:
                raise RuntimeError("device replay staging full (%d rows): call tight()/train() once per round or "
                                   "raise stage_rows" % self.rows)
        dev = self.device
        slot = torch.arange(cap, device=dev)
        cnt = num[:n_rec].to(torch.int64)
        if active is not None:
            cnt = cnt * active[:n_rec].to(torch.int64)
        valid = slot[None, :] < cnt[:, None]                                    # [n_rec, cap]
        start = self.cursor + torch.cumsum(cnt, 0) - cnt                        # exclusive scan
        dest = torch.where(valid, start[:, None] + slot[None, :], torch.full_like(valid, self.rows, dtype=torch.int64))
        dest = dest.reshape(-1)
        self.obs.index_copy_(0, dest, view[:n_rec].reshape((n_rec * cap,) + tuple(view.shape[2:])))
        self.feat.index_copy_(0, dest, feat[:n_rec].reshape(n_rec * cap, -1))
        self.act.index_copy_(0, dest, acts[:n_rec].reshape(-1).to(torch.int32))
        self.rew.index_copy_(0, dest, rewards[:n_rec].reshape(-1))
        self.term.index_copy_(0, dest, (alives[:n_rec].reshape(-1) == 0))
        env = torch.arange(n_rec, device=dev, dtype=torch.int64)[:, None]
        self.key.index_copy_(0, dest, (env * id_span + ids[:n_rec].to(torch.int64)).reshape(-1))
        self.t.index_copy_(0, dest, torch.full((n_rec * cap,), self.step, dtype=torch.int64, device=dev))
        if self.use_mean:
            # [E, act_n]: one mean action per env (the group mean); [E, cap, act_n]: one per agent (the local mean)
            rows = prob[:n_rec] if prob.dim() == 3 else prob[:n_rec, None, :].expand(n_rec, cap, prob.shape[-1])
            self.prob.index_copy_(0, dest, rows.reshape(n_rec * cap, -1))
        self.cursor += cnt.sum()
        self.upper += n_rec * cap
        self.step += 1

    def sorted_rows(self, generator=None, agent_order=None):
        """-> (order, seg_last, n_agents): `order` lists the staged rows grouped by agent (agents in a random or
        injected order) and by time inside an agent; seg_last[i] marks the last row of a trajectory."""
        n = int(self.cursor)
        self.upper = n
        if n == 0:
            return None, None, 0
        keys, t = self.key[:n], self.t[:n]
        uniq, inv = torch.unique(keys, return_inverse=True)
        m = int(uniq.numel())
        if agent_order is not None:          # test hook: the flush order as a list of agent keys
            want = torch.as_tensor(agent_order, dtype=torch.int64, device=self.device)
            assert want.numel() == m
            pos = torch.searchsorted(uniq, want)
            assert bool((uniq[pos] == want).all())
            rank = torch.empty((m,), dtype=torch.int64, device=self.device)
            rank[pos] = torch.arange(m, device=self.device)
        else:
            rank = torch.randperm(m, generator=generator, device=self.device)
        agent_rank = rank[inv]
        order = torch.argsort(agent_rank * (self.step + 1) + t)
        sorted_rank = agent_rank[order]
        seg_last = torch.ones((n,), dtype=torch.bool, device=self.device)
        seg_last[:-1] = sorted_rank[1:] != sorted_rank[:-1]
        return order, seg_last, m


class DeviceMemoryGroup:
    def __init__(self, obs_shape, feat_shape, act_n, max_len, batch_size, sub_len, use_mean=False, device=None,
                 stage_rows=None, id_span=1 << 20, seed=None):
        self.device = torch.device(device if device is not None else "cuda")
        self.obs_shape, self.feat_shape, self.act_n = tuple(obs_shape), tuple(feat_shape), act_n
        self.max_len, self.batch_size, self.sub_len, self.use_mean = max_len, batch_size, sub_len, use_mean
        self.stage_rows = stage_rows if stage_rows is not None else max_len
        self.id_span = id_span
        dev = self.device
        self.obs0 = torch.zeros((max_len,) + self.obs_shape, dtype=torch.float32, device=dev)
        self.feat0 = torch.zeros((max_len,) + self.feat_shape, dtype=torch.float32, device=dev)
        self.actions = torch.zeros((max_len,), dtype=torch.int32, device=dev)
        self.rewards = torch.zeros((max_len,), dtype=torch.float32, device=dev)
        self.terminals = torch.zeros((max_len,), dtype=torch.bool, device=dev)
        self.masks = torch.zeros((max_len,), dtype=torch.bool, device=dev)
        self.prob = torch.zeros((max_len, act_n), dtype=torch.float32, device=dev) if use_mean else None
        self.length, self._flag, self._new_add = 0, 0, 0
        self._stage = None
        self.generator = torch.Generator(device=dev)
        if seed is not None:
            self.generator.manual_seed(seed)

    # -- push: one lockstep step of one group ------------------------------------------------------------
    def n_rec_envs(self, n_envs, capacity):
        return max(1, min(n_envs, self.stage_rows // max(1, capacity * self.sub_len)))

    def push(self, **kwargs):
        """state=(view [E, cap, 13, 13, 7], feature [E, cap, 34]), acts / rewards / alives / ids [E, cap],
        prob [E, act_n] (the mean action every agent of the env saw) or [E, cap, act_n] (each agent's own), num [E],
        active [E] bool or None."""
        view, feat = kwargs['state']
        if self._stage is None:
            self._stage = _Staging(self.stage_rows, self.obs_shape, self.feat_shape, self.act_n, self.use_mean,
                                   self.device)
        E, cap = kwargs['acts'].shape
        self._stage.push(self.n_rec_envs(E, cap), self.id_span, view, feat, kwargs['acts'], kwargs['rewards'],
                         kwargs['alives'], kwargs['ids'], kwargs.get('prob'), kwargs['num'], kwargs.get('active'))

    @property
    def has_staged(self):
        return self._stage is not None and self._stage.upper > 0

    # -- tight: trajectories -> ring ---------------------------------------------------------------------
    def tight(self, agent_order=None):
        st = self._stage
        if st is None:
            return
        order, seg_last, _m = st.sorted_rows(self.generator, agent_order)
        if order is None:
            return
        n = int(order.numel())
        self._new_add += n
        mask = ~st.term[order] & ~seg_last
        # sequential ring write with wrap (MetaBuffer.append, tools.py:62-78): row i lands at (flag + i) % max_len;
        # when n exceeds the ring only the last max_len rows survive
        first = max(0, n - self.max_len)
        src = order[first:]
        dest = (self._flag + first + torch.arange(n - first, device=self.device)) % self.max_len
        self.obs0.index_copy_(0, dest, st.obs[src])
        self.feat0.index_copy_(0, dest, st.feat[src])
        self.actions.index_copy_(0, dest, st.act[src])
        self.rewards.index_copy_(0, dest, st.rew[src])
        self.terminals.index_copy_(0, dest, st.term[src])
        self.masks.index_copy_(0, dest, mask[first:])
        if self.use_mean:
            self.prob.index_copy_(0, dest, st.prob[src])
        self._flag = (self._flag + n) % self.max_len
        self.length = min(self.length + n, self.max_len)
        st.reset()

    # -- sample ------------------------------------------------------------------------------------------
    def sample(self, idx=None):
        if idx is None:
            idx = torch.randint(self.nb_entries, (self.batch_size,), generator=self.generator, device=self.device)
        else:
            idx = torch.as_tensor(idx, dtype=torch.int64, device=self.device)
        nxt = (idx + 1) % self.nb_entries
        obs, obs_next = self.obs0[idx], self.obs0[nxt]
        feature, feature_next = self.feat0[idx], self.feat0[nxt]
        actions, rewards = self.actions[idx], self.rewards[idx]
        dones, masks = self.terminals[idx], self.masks[idx]
        if self.use_mean:
            return obs, feature, actions, self.prob[idx], obs_next, feature_next, self.prob[nxt], rewards, dones, masks
        return obs, feature, obs_next, feature_next, dones, rewards, actions, masks

    def get_batch_num(self, verbose=True):
        if verbose:
            print('\n[INFO] Length of buffer and new add:', self.length, self._new_add)
        res = self._new_add * 2 // self.batch_size
        self._new_add = 0
        return res

    @property
    def nb_entries(self):
        return self.length


class DeviceEpisodesBuffer:
    """Whole trajectories of one round for the actor-critic update (EpisodesBuffer, tools.py:122-173)."""

    def __init__(self, obs_shape, feat_shape, act_n, stage_rows, sub_len, use_mean=False, device=None,
                 id_span=1 << 20):
        self.device = torch.device(device if device is not None else "cuda")
        self.obs_shape, self.feat_shape, self.act_n = tuple(obs_shape), tuple(feat_shape), act_n
        self.stage_rows, self.sub_len, self.use_mean, self.id_span = stage_rows, sub_len, use_mean, id_span
        self._stage = None

    def n_rec_envs(self, n_envs, capacity):
        return max(1, min(n_envs, self.stage_rows // max(1, capacity * self.sub_len)))

    def push(self, **kwargs):
        view, feat = kwargs['state']
        if self._stage is None:
            self._stage = _Staging(self.stage_rows, self.obs_shape, self.feat_shape, self.act_n, self.use_mean,
                                   self.device)
        E, cap = kwargs['acts'].shape
        self._stage.push(self.n_rec_envs(E, cap), self.id_span, view, feat, kwargs['acts'], kwargs['rewards'],
                         kwargs['alives'], kwargs['ids'], kwargs.get('prob'), kwargs['num'], kwargs.get('active'))

    @property
    def has_staged(self):
        return self._stage is not None and self._stage.upper > 0

    def episodes(self):
        """-> dict(view, feature, action, reward, prob, seg_last, seg_id, n_agents): rows sorted by (agent, time)."""
        st = self._stage
        if st is None:
            return None
        order, seg_last, m = st.sorted_rows(None, None)
        if order is None:
            return None
        seg_id = torch.cumsum(seg_last.to(torch.int64), 0) - seg_last.to(torch.int64)
        out = dict(view=st.obs[order], feature=st.feat[order], action=st.act[order], reward=st.rew[order],
                   prob=st.prob[order] if self.use_mean else None, seg_last=seg_last, seg_id=seg_id, n_agents=m)
        st.reset()
        return out


def segmented_discounted_returns(reward, seg_last, seg_id, bootstrap, gamma):
    """Per trajectory (rows sorted by time, `seg_last` marks its end): keep = bootstrap[seg]; walking backwards
    keep = keep * gamma + r[i]; R[i] = keep -- ac.py:139-148 for all agents at once.  fp32 like the reference.
    The scan runs over time offsets (<= the longest trajectory) on [n_agents] vectors."""
    n = reward.numel()
    dev = reward.device
    idx = torch.arange(n, device=dev)
    last_idx = torch.zeros((int(seg_id.max()) + 1,), dtype=torch.int64, device=dev)
    last_idx[seg_id[seg_last]] = idx[seg_last]
    seg_len = torch.bincount(seg_id)
    first_idx = last_idx - seg_len + 1
    out = torch.empty_like(reward)
    keep = bootstrap.to(torch.float32).clone()
    for back in range(int(seg_len.max())):
        pos = last_idx - back
        live = pos >= first_idx
        p = torch.where(live, pos, last_idx)
        new_keep = keep * gamma + reward[p]
        keep = torch.where(live, new_keep, keep)
        out[p[live]] = keep[live]
    return out
