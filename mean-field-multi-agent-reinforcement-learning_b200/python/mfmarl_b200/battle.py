"""BatchedGridWorld: E lock-stepped battle environments resident on one GPU.

Semantics per environment are those of magent.GridWorld('battle') driven by the play loop of the
reference (examples/battle_model/senario_battle.py:96-168): get_observation for both groups ->
set_action(g0), set_action(g1) -> step -> get_reward / get_alive -> mean action -> clear_dead; here one
`observe()` and one `step()` call do that for all E environments with two kernel launches.
"""
import ctypes

import numpy as np
import torch

from .lib import MfbConfig, check, load_library

RNG_MODES = {"minstd": 0, "philox": 1, "inject": 2}


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class BatchedGridWorld:
    def __init__(self, n_envs, map_size=40, capacity=64, device=None, rng="minstd", seed=0, env_base=0,
                 max_steps=0, auto_reset=False, step_threads=0, obs_tile_agents=0, obs_record=None, random_sides=False, concurrent_step_envs=0, **type_overrides):
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedGridWorld needs a CUDA device: there is no CPU fallback")
        self.lib = load_library()
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        cfg = MfbConfig()
        check(self.lib.mfb_default_config(ctypes.byref(cfg)))
        cfg.n_envs, cfg.map_width, cfg.map_height, cfg.capacity = n_envs, map_size, map_size, capacity
        cfg.rng_mode, cfg.seed, cfg.env_base = RNG_MODES[rng], seed, env_base
        cfg.max_steps, cfg.auto_reset, cfg.device = max_steps, int(auto_reset), self.device.index or 0
        cfg.step_threads, cfg.obs_tile_agents = step_threads, obs_tile_agents
        if obs_record is not None:          # None = the engine decides (on for capacity >= 256)
            cfg.obs_record = int(obs_record)
        cfg.random_sides = int(random_sides)
        cfg.concurrent_step_envs = int(concurrent_step_envs)   # pipelined use: a sibling engine's step() overlaps this observe()
        for key, value in type_overrides.items():
            if not hasattr(cfg, key):
                raise TypeError("unknown agent-type attribute %r" % key)
            setattr(cfg, key, value)
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            check(self.lib.mfb_create(ctypes.byref(cfg), ctypes.byref(self._h)))
        self.n_envs, self.map_size, self.rng = n_envs, map_size, rng
        self.view_radius = float(cfg.view_radius)
        self._bufs = {}
        self._sizes = None

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self.lib.mfb_destroy(h)
            self._h = None

    # ------------------------------------------------------------ set-up
    def reset(self):
        check(self.lib.mfb_reset(self._h))
        self._sizes = None

    def set_seed(self, seed):
        check(self.lib.mfb_set_seed(self._h, seed))

    def add_walls(self, pos):
        pos = np.asarray(pos, dtype=np.int32)
        xs, ys = np.ascontiguousarray(pos[:, 0]), np.ascontiguousarray(pos[:, 1])
        check(self.lib.mfb_add_walls(self._h, len(pos), xs.ctypes.data, ys.ctypes.data))
        self._sizes = None

    def add_agents(self, group, pos):
        """The same `pos` ([[x, y(, dir)], ...]) is placed in every environment; returns #added."""
        pos = np.asarray(pos, dtype=np.int32)
        xs, ys = np.ascontiguousarray(pos[:, 0]), np.ascontiguousarray(pos[:, 1])
        added = ctypes.c_int()
        check(self.lib.mfb_add_agents(self._h, group, len(pos), xs.ctypes.data, ys.ctypes.data,
                                      ctypes.byref(added)))
        self._sizes = None
        return added.value

    def add_agents_per_env(self, group, pos):
        """pos int[E, n, 2 or 3]: every environment gets its OWN placement; cells that are occupied, walls or out of
        range are skipped per environment (GridWorld.cc:180-187).  Returns the number added in each env, int32[E]."""
        pos = np.asarray(pos, dtype=np.int32)
        assert pos.ndim == 3 and pos.shape[0] == self.n_envs, pos.shape
        xs, ys = np.ascontiguousarray(pos[:, :, 0]), np.ascontiguousarray(pos[:, :, 1])
        added = np.zeros((self.n_envs,), np.int32)
        check(self.lib.mfb_add_agents_per_env(self._h, group, pos.shape[1], xs.ctypes.data, ys.ctypes.data,
                                              added.ctypes.data))
        self._sizes = None
        return added

    # ------------------------------------------------------------ sizes / buffers
    def query(self, key):
        out = ctypes.c_int()
        with torch.cuda.device(self.device):
            check(self.lib.mfb_query(self._h, key.encode(), ctypes.byref(out)))
        return out.value

    @property
    def sizes(self):
        if self._sizes is None:
            self._sizes = {k: self.query(k) for k in
                           ("capacity", "n_action", "view_size", "n_channel", "feature_size")}
        return self._sizes

    @property
    def capacity(self):
        return self.sizes["capacity"]

    def _buf(self, name, shape, dtype):
        t = self._bufs.get(name)
        if t is None or tuple(t.shape) != tuple(shape):
            t = self._bufs[name] = torch.zeros(shape, dtype=dtype, device=self.device)
        return t

    # ------------------------------------------------------------ the two launches
    def observe(self, group_mask=3, out=None):
        """-> (view float32[E, 2, cap, 13, 13, 7], feature float32[E, 2, cap, 34]); rows >= num are stale."""
        s = self.sizes
        E, cap, v = self.n_envs, s["capacity"], s["view_size"]
        if out is None:
            view = self._buf("view", (E, 2, cap, v, v, s["n_channel"]), torch.float32)
            feat = self._buf("feat", (E, 2, cap, s["feature_size"]), torch.float32)
        else:
            view, feat = out
        with torch.cuda.device(self.device):
            check(self.lib.mfb_observe(self._h, _ptr(view), _ptr(feat), group_mask, _stream()))
        return view, feat

    def observe_groups(self, groups=(0, 1), dtype=torch.float32):
        """Per-group observation blocks, each contiguous: -> [(view_g float32[E, cap, 13, 13, 7], feature_g
        float32[E, cap, 34]) for g in (0, 1)] (None for a group not asked for).  This is the layout a per-group
        policy network consumes in place (`view_g.view(E * cap, 13, 13, 7)` is free).

        dtype=torch.bfloat16: view_g is bfloat16[E, cap, 13, 13, 8] -- the same seven channels rounded to bf16 plus a
        zero eighth, i.e. exactly what a bf16 channels-last convolution wants (no cast, no padding pass, 42 % fewer
        bytes); features stay float32."""
        s = self.sizes
        E, cap, v = self.n_envs, s["capacity"], s["view_size"]
        bf16 = dtype == torch.bfloat16
        assert bf16 or dtype == torch.float32
        out, ptrs = [], []
        for g in (0, 1):
            if g in groups:
                view = self._buf("view%s_g%d" % ("16" if bf16 else "", g), (E, cap, v, v, 8 if bf16 else s["n_channel"]), dtype)
                feat = self._buf("feat_g%d" % g, (E, cap, s["feature_size"]), torch.float32)
                out.append((view, feat)); ptrs += [_ptr(view), _ptr(feat)]
            else:
                out.append(None); ptrs += [None, None]
        with torch.cuda.device(self.device):
            fn = self.lib.mfb_observe_groups_bf16 if bf16 else self.lib.mfb_observe_groups
            check(fn(self._h, *ptrs, _stream()))
        return out

    def local_mean_action(self, groups=(0, 1), radius=None):
        """Neighbourhood mean action of every listed agent (mfb_local_mean_action, kernel K7): per group a float32
        [E, cap, n_action] tensor (None for a group not asked for).  Row i is the one-hot mean of the last actions of
        agent i's living group-mates that have acted and stand inside the disc of `radius` around it (None = the
        view radius, the largest allowed), or zeros when there are none; rows >= num are zero.  Called after step(),
        its rows line up with the next observe_groups() rows.  The buffers belong to the engine and are reused by the
        next call; nothing in the engine state changes."""
        s = self.sizes
        E, cap, n_action = self.n_envs, s["capacity"], s["n_action"]
        radius = self.view_radius if radius is None else float(radius)
        out, ptrs = [], []
        for g in (0, 1):
            if g in groups:
                t = self._buf("local_mean_g%d" % g, (E, cap, n_action), torch.float32)
                out.append(t); ptrs.append(_ptr(t))
            else:
                out.append(None); ptrs.append(None)
        with torch.cuda.device(self.device):
            check(self.lib.mfb_local_mean_action(self._h, radius, *ptrs, _stream()))
        return out

    def device_state(self, key):
        """Live engine state as a torch tensor ALIASING the engine's HBM arrays (read-only by convention; contents
        change with every launch on the stream): "num" int32[E, 2], "id" int32[E, 2, cap], "pos" int32[E, 2, cap]
        (x | y << 16), "hp" float32[E, 2, cap], "step_ct" int32[E]."""
        E, cap = self.n_envs, self.capacity
        spec = {"num": ((E, 2), "<i4", torch.int32), "id": ((E, 2, cap), "<i4", torch.int32),
                "pos": ((E, 2, cap), "<i4", torch.int32), "hp": ((E, 2, cap), "<f4", torch.float32),
                "step_ct": ((E,), "<i4", torch.int32)}[key]
        self.get("num")                      # commits a pending placement and synchronises
        ptr = ctypes.c_void_p()
        check(self.lib.mfb_state_device_ptr(self._h, key.encode(), ctypes.byref(ptr)))

        class _Alias:
            __cuda_array_interface__ = {"shape": spec[0], "typestr": spec[1], "data": (ptr.value, False), "version": 2}
        with torch.cuda.device(self.device):
            return torch.as_tensor(_Alias(), device=self.device)

    def step(self, actions, attack_perm=None, clear_dead=True, want_mean_action=True):
        """actions int32[E, 2, cap] on the device -> (reward, alive, done, mean_action) device tensors."""
        s = self.sizes
        E, cap = self.n_envs, s["capacity"]
        assert actions.dtype == torch.int32 and actions.is_cuda and actions.is_contiguous()
        assert tuple(actions.shape) == (E, 2, cap), (tuple(actions.shape), (E, 2, cap))
        reward = self._buf("reward", (E, 2, cap), torch.float32)
        alive = self._buf("alive", (E, 2, cap), torch.uint8)
        done = self._buf("done", (E,), torch.int32)
        mean = self._buf("mean", (E, 2, s["n_action"]), torch.float32) if want_mean_action else None
        with torch.cuda.device(self.device):
            check(self.lib.mfb_step(self._h, _ptr(actions), _ptr(attack_perm), _ptr(reward), _ptr(alive),
                                    _ptr(mean), _ptr(done), int(clear_dead), _stream()))
        return reward, alive, done, mean

    def clear_dead(self):
        with torch.cuda.device(self.device):
            check(self.lib.mfb_clear_dead(self._h, _stream()))

    def step_host(self, h_actions, h_reward, h_alive, h_mean, h_done):
        """End-to-end variant: pinned host tensors in and out (H2D + kernels + D2H + sync in one call)."""
        with torch.cuda.device(self.device):
            check(self.lib.mfb_step_host(self._h, _ptr(h_actions), _ptr(h_reward), _ptr(h_alive),
                                         _ptr(h_mean), _ptr(h_done), _stream()))

    def step_host_async(self, h_actions, h_reward, h_alive, h_mean, h_done):
        """Pipelined end-to-end step: enqueue upload + k_step + download and return a ticket (0/1); the
        pinned result tensors are valid after host_wait(ticket)."""
        ticket = ctypes.c_int()
        with torch.cuda.device(self.device):
            check(self.lib.mfb_step_host_async(self._h, _ptr(h_actions), _ptr(h_reward), _ptr(h_alive),
                                               _ptr(h_mean), _ptr(h_done), _stream(), ctypes.byref(ticket)))
        return ticket.value

    def host_wait(self, ticket):
        check(self.lib.mfb_host_wait(self._h, ticket))

    # ------------------------------------------------------------ read-back
    _GET = {"num": ("i4", lambda E, c: (E, 2)), "dead_ct": ("i4", lambda E, c: (E, 2)),
            "pos": ("i4", lambda E, c: (E, 2, c, 2)), "hp": ("f4", lambda E, c: (E, 2, c)),
            "id": ("i4", lambda E, c: (E, 2, c)), "alive": ("u1", lambda E, c: (E, 2, c)),
            "last_action": ("i4", lambda E, c: (E, 2, c)), "step_ct": ("i4", lambda E, c: (E,)),
            "rng": ("u4", lambda E, c: (E,)), "agent_steps": ("u8", lambda E, c: (E,)),
            "side": ("i4", lambda E, c: (E,)), "episode": ("i4", lambda E, c: (E,))}

    def get(self, key):
        dtype, shape = self._GET[key]
        buf = np.empty(shape(self.n_envs, self.capacity), dtype=dtype)
        with torch.cuda.device(self.device):
            check(self.lib.mfb_get(self._h, key.encode(), buf.ctypes.data, _stream()))
        return buf

    def get_num(self):
        return self.get("num")


def mean_action(actions, num, n_action=21):
    """Group mean action (senario_battle.py:141): actions int32[rows, cap], num int32[rows] on the
    device -> float32[rows, n_action] = one-hot mean over the first num[r] agents of each row."""
    lib = load_library()
    assert actions.dtype == torch.int32 and num.dtype == torch.int32 and actions.is_cuda and num.is_cuda
    rows, cap = actions.shape
    out = torch.empty((rows, n_action), dtype=torch.float32, device=actions.device)
    with torch.cuda.device(actions.device):
        check(lib.mfb_mean_action(_ptr(actions.contiguous()), _ptr(num.contiguous()), _ptr(out), rows, cap,
                                  n_action, _stream()))
    return out
