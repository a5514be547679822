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
`DeviceStateMemoryGroup` = `DeviceMemoryGroup` with a reference to an env state record in place of each observation
row: the observations are rendered again on the GPU when a batch is sampled, so a ring row costs ~100 B instead of
~4970 B and every environment can be recorded.
"""
import collections

import torch


class _Staging:
    """Time-major staging rows of the current round: fixed-capacity device tensors + a device-side cursor."""

    def __init__(self, rows, obs_shape, feat_shape, act_n, use_mean, device, row_refs=False):
        self.rows, self.device, self.use_mean = rows, device, use_mean
        n = rows + 1                                     # the extra row swallows the writes of invalid slots
        if row_refs:                                     # (record, group, slot) per row, no observation (feat = None)
            self.obs, self.feat = torch.empty((n, 3), dtype=torch.int32, device=device), None
        else:
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
        if self.feat is not None:
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
    _row_refs = False                                    # DeviceStateMemoryGroup: obs0 holds record references

    def __init__(self, obs_shape, feat_shape, act_n, max_len, batch_size, sub_len, use_mean=False, device=None,
                 stage_rows=None, id_span=1 << 20, seed=None):
        self.device = torch.device(device if device is not None else "cuda")
        self.obs_shape, self.feat_shape, self.act_n = tuple(obs_shape), tuple(feat_shape), act_n
        self.max_len, self.batch_size, self.sub_len, self.use_mean = max_len, batch_size, sub_len, use_mean
        self.stage_rows = stage_rows if stage_rows is not None else max_len
        self.id_span = id_span
        dev = self.device
        if self._row_refs:
            self.obs0, self.feat0 = torch.zeros((max_len, 3), dtype=torch.int32, device=dev), None
        else:
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
                                   self.device, self._row_refs)
        E, cap = kwargs['acts'].shape
        self._stage.push(self.n_rec_envs(E, cap), self.id_span, view, feat, kwargs['acts'], kwargs['rewards'],
                         kwargs['alives'], kwargs['ids'], kwargs.get('prob'), kwargs['num'], kwargs.get('active'))

    @property
    def has_staged(self):
        return self._stage is not None and self._stage.upper > 0

    # -- tight: trajectories -> ring ---------------------------------------------------------------------
    def tight(self, agent_order=None):
        """-> the number of rows the round appended to the ring (rows past max_len overwrite the round's first ones)."""
        st = self._stage
        if st is None:
            return 0
        order, seg_last, _m = st.sorted_rows(self.generator, agent_order)
        if order is None:
            return 0
        n = int(order.numel())
        self._new_add += n
        mask = ~st.term[order] & ~seg_last
        # sequential ring write with wrap (MetaBuffer.append, tools.py:62-78): row i lands at (flag + i) % max_len;
        # when n exceeds the ring only the last max_len rows survive
        first = max(0, n - self.max_len)
        src = order[first:]
        dest = (self._flag + first + torch.arange(n - first, device=self.device)) % self.max_len
        self.obs0.index_copy_(0, dest, st.obs[src])
        if self.feat0 is not None:
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
        return n

    # -- sample ------------------------------------------------------------------------------------------
    def sample(self, idx=None):
        if idx is None:
            idx = torch.randint(self.nb_entries, (self.batch_size,), generator=self.generator, device=self.device)
        else:
            idx = torch.as_tensor(idx, dtype=torch.int64, device=self.device)
        nxt = (idx + 1) % self.nb_entries
        obs, feature, obs_next, feature_next = self._observations(idx, nxt)
        actions, rewards = self.actions[idx], self.rewards[idx]
        dones, masks = self.terminals[idx], self.masks[idx]
        if self.use_mean:
            return obs, feature, actions, self.prob[idx], obs_next, feature_next, self.prob[nxt], rewards, dones, masks
        return obs, feature, obs_next, feature_next, dones, rewards, actions, masks

    def _observations(self, idx, nxt):
        return self.obs0[idx], self.feat0[idx], self.obs0[nxt], self.feat0[nxt]

    def get_batch_num(self, verbose=True):
        if verbose:
            print('\n[INFO] Length of buffer and new add:', self.length, self._new_add)
        res = self._new_add * 2 // self.batch_size
        self._new_add = 0
        return res

    @property
    def nb_entries(self):
        return self.length


class DeviceStateMemoryGroup(DeviceMemoryGroup):
    """`DeviceMemoryGroup` whose ring rows hold a reference (record, group, slot) into an arena of env state records
    (BatchedGridWorld.save_envs: R = 96 + 64 cap bytes per recorded env and step) instead of the observation row
    (4868 B).  `sample()` renders the rows with `renderer(records, rows) -> (view, feature)`
    (BatchedGridWorld.render_observations: bit for bit the rows observe_groups gave at that step).  Actions, rewards,
    terminals, masks, prob, the ring, the sampling and the generator calls are DeviceMemoryGroup's, so for the same
    pushes `sample()` returns the same tensors.

    Record arena: one record per recorded env and step (`push(records=...)`; `record_slice()` hands out the arena slice
    the next push uses, so that save_envs can write there directly).  The live records are [head, tail): the rows of
    round r reference only round r's records, and a round's records are freed once the ring has overwritten all of its
    rows.  When a push finds no room at the end, the live records move to the front (the references with them) and
    the arena grows if that is not enough -- up to `max_records` (None = no limit), past which push raises with the size
    it needs.  A live row's record is never dropped."""
    _row_refs = True

    def __init__(self, obs_shape, feat_shape, act_n, max_len, batch_size, sub_len, state_bytes, renderer, group=0,
                 max_records=None, **kwargs):
        super().__init__(obs_shape, feat_shape, act_n, max_len, batch_size, sub_len, **kwargs)
        self.state_bytes, self.renderer, self.group, self.max_records = state_bytes, renderer, group, max_records
        self.arena = torch.empty((0, state_bytes), dtype=torch.uint8, device=self.device)
        self.head = self.tail = 0               # live records
        self._rounds = collections.deque()      # per round in the ring: (end of its records, ring rows written after it, rows)
        self._written = 0                       # rows appended to the ring so far
        self._ref_base = None                   # (env, group, slot) per row of a push

    def _reserve(self, n):
        """Room for n more records at the tail (may move the live records, and the references to them, to the front)."""
        if self.tail + n <= self.arena.shape[0]:
            return
        live = self.tail - self.head
        need = live + n
        if self.max_records is not None and need > self.max_records:
            raise RuntimeError("state-record arena full: %d live records + %d new need %d records (%d bytes); "
                               "max_records is %d" % (live, n, need, need * self.state_bytes, self.max_records))
        if need <= self.arena.shape[0]:
            self.arena[:live] = self.arena[self.head:self.tail].clone()
        else:
            size = max(need, 2 * self.arena.shape[0], n * self.sub_len)
            if self.max_records is not None:
                size = min(size, self.max_records)
            arena = torch.empty((size, self.state_bytes), dtype=torch.uint8, device=self.device)
            arena[:live] = self.arena[self.head:self.tail]
            self.arena = arena
        shift = self.head
        if shift:
            self.obs0[:, 0] -= shift            # (the rows of freed rounds have all been overwritten)
            if self._stage is not None:
                self._stage.obs[:, 0] -= shift
            self._rounds = collections.deque((end - shift, w, rows) for end, w, rows in self._rounds)
            self.head, self.tail = 0, self.tail - shift

    def record_slice(self, n_envs, capacity):
        """uint8[n_rec, R] view of the arena where the next push's records go (n_rec = n_rec_envs(n_envs, capacity))."""
        n = self.n_rec_envs(n_envs, capacity)
        self._reserve(n)
        return self.arena[self.tail:self.tail + n]

    def push(self, **kwargs):
        """DeviceMemoryGroup.push with records=uint8[>= n_rec, R], the state of the first n_rec envs when this step's
        rows were observed (e.g. saved into record_slice()), in place of state=."""
        E, cap = kwargs['acts'].shape
        n = self.n_rec_envs(E, cap)
        records = kwargs.pop('records')[:n]
        self._reserve(n)
        base = self.tail
        dst = self.arena[base:base + n]
        if dst.data_ptr() != records.data_ptr():
            dst.copy_(records)
        self.tail += n
        if self._ref_base is None or tuple(self._ref_base.shape[:2]) != (n, cap):
            env = torch.arange(n, dtype=torch.int32, device=self.device)[:, None].expand(n, cap)
            slot = torch.arange(cap, dtype=torch.int32, device=self.device)[None, :].expand(n, cap)
            self._ref_base = torch.stack([env, torch.full_like(env, self.group), slot], dim=2)
        refs = self._ref_base.clone()
        refs[:, :, 0] += base
        kwargs['state'] = (refs, None)
        super().push(**kwargs)

    def tight(self, agent_order=None):
        n = super().tight(agent_order)
        self._written += n
        self._rounds.append((self.tail, self._written, n))
        while self._rounds and (self._rounds[0][2] == 0 or self._written - self._rounds[0][1] >= self.max_len):
            self.head = self._rounds.popleft()[0]    # every row of the oldest round has been overwritten
        return n

    def _observations(self, idx, nxt):
        b = idx.numel()
        view, feat = self.renderer(self.arena[:self.tail], torch.cat([self.obs0[idx], self.obs0[nxt]]))
        return view[:b], feat[:b], view[b:], feat[b:]


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
