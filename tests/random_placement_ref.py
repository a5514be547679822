"""Random placement (mfb_add_agents_random) restated in numpy: test infrastructure for place_random in
csrc/battle_kernels.cuh.

The draw rules:
  MINSTD  candidate t of an env is draws 2t+1, 2t+2 of its minstd_rand0 stream: x = x0 + r1 % w, y = y0 + r2 % h
          (the whole map: x = r1 % (W - 1), y = r2 % (H - 1), runtime_api.cu's add_agents(method="random")); the
          stream runs on through every op of the placement.
  PHILOX  candidate t of op k: Philox4x32-10, key (seed, env_base + e), counter (t, k, episode, generation | 2^31);
          x = x0 + mulhi(word0, w), y = y0 + mulhi(word1, h).  t restarts at 0 for every op.
A candidate is blank when x + 1 < W, y + 1 < H and the cell holds no wall, fixed agent or earlier random agent.  An
agent gives up after W*H + 1 failed candidates, and then the rest of its op is not placed either.

`place_sequential` is the reference's loop; `place_warp` is the kernel's 32-candidate batches with the match/ballot
acceptance rule and the lane-uniform scan, restated so the two can be compared.
"""
import numpy as np

from philox_ref import philox4x32_10

MINSTD_A, MINSTD_M = 16807, 2147483647
TOP = 0x80000000


def minstd_next(s):
    return (s * MINSTD_A) % MINSTD_M


def whole_map(W, H):
    return (0, 0, W - 1, H - 1)


class Draws:
    """the candidates of one env's placement; MINSTD keeps its stream in .rs"""

    def __init__(self, mode, W, H, rs=1, seed=0, gid=0, episode=0, generation=0):
        self.mode, self.W, self.H, self.rs = mode, W, H, int(rs)
        self.seed, self.gid, self.episode, self.generation = seed, gid, episode, generation

    def candidates(self, k, rect):
        """op k's candidates in order (MINSTD: advances .rs as they are taken)"""
        x0, y0, w, h = rect
        if self.mode == "minstd":
            while True:
                r1 = minstd_next(self.rs); r2 = minstd_next(r1); self.rs = r2
                yield x0 + r1 % w, y0 + r2 % h
        t = 0
        while True:
            xs, ys = self.philox_cells(k, np.arange(t, t + 64), rect)
            yield from zip(xs.tolist(), ys.tolist())
            t += 64

    def philox_cells(self, k, ts, rect):
        x0, y0, w, h = rect
        ts = np.asarray(ts, dtype=np.uint64).astype(np.uint32)
        r = philox4x32_10([ts, np.uint32(k), np.uint32(self.episode), np.uint32(self.generation | TOP)],
                          [np.uint32(self.seed), np.uint32(self.gid)])
        xs = x0 + ((r[0].astype(np.uint64) * np.uint64(w)) >> np.uint64(32)).astype(np.int64)
        ys = y0 + ((r[1].astype(np.uint64) * np.uint64(h)) >> np.uint64(32)).astype(np.int64)
        return xs, ys


def _blank(occ, x, y, W, H):
    return x + 1 < W and y + 1 < H and not occ[y, x]


def place_sequential(draws, occ, ops):
    """ops: [(group, n, rect)]; occ: bool[H, W] (walls and fixed agents), modified.  Returns per op the list of placed
    (x, y) and the number of agents not placed."""
    W, H = draws.W, draws.H
    max_fails = W * H + 1
    out, short = [], 0
    for k, (_, n, rect) in enumerate(ops):
        stream = draws.candidates(k, rect)
        cells = []
        for _ in range(n):
            fails, ok = 0, False
            while fails < max_fails:
                x, y = next(stream)
                if _blank(occ, x, y, W, H):
                    occ[y, x] = True
                    cells.append((x, y))
                    ok = True
                    break
                fails += 1
            if not ok:
                break
        short += n - len(cells)
        out.append(cells)
    return out, short


def place_warp(draws, occ, ops):
    """The kernel's rule: 32 candidates per batch, accepted when blank and first blank on their cell in lane order;
    a lane-uniform scan finds how far the sequential loop got in the batch."""
    W, H = draws.W, draws.H
    max_fails = W * H + 1
    out, short = [], 0
    for k, (_, n, rect) in enumerate(ops):
        x0, y0, w, h = rect
        cells, fails, t, gave_up = [], 0, 0, False
        while len(cells) < n and not gave_up:
            if draws.mode == "minstd":
                r, states = draws.rs, []
                for _ in range(32):
                    r1 = minstd_next(r); r2 = minstd_next(r1); r = r2
                    states.append((r1, r2))
                cand = [(x0 + r1 % w, y0 + r2 % h) for r1, r2 in states]
            else:
                xs, ys = draws.philox_cells(k, np.arange(t, t + 32), rect)
                cand = list(zip(xs.tolist(), ys.tolist()))
            blank = [_blank(occ, x, y, W, H) for x, y in cand]
            ok = [blank[l] and all(not (blank[j] and cand[j] == cand[l]) for j in range(l)) for l in range(32)]
            okm = [l for l in range(32) if ok[l]]
            acc, consumed, pos = [], 32, 0
            while True:
                nxt = okm[0] if okm else 32
                gap = nxt - pos
                if fails + gap >= max_fails:
                    consumed = pos + (max_fails - fails); gave_up = True; break
                if nxt == 32:
                    fails += gap; break
                acc.append(nxt); okm = okm[1:]; fails = 0; pos = nxt + 1
                if len(cells) + len(acc) == n:
                    consumed = pos; break
            for l in acc:
                x, y = cand[l]
                occ[y, x] = True
                cells.append((x, y))
            if draws.mode == "minstd":
                draws.rs = states[consumed - 1][1]
            t += consumed
        short += n - len(cells)
        out.append(cells)
    return out, short


def episode_placement(mode, W, H, walls, fixed, ops, side=0, **draw_args):
    """One env's episode start as the engine makes it.  walls: bool[H, W] (border ring included); fixed: [pos list of
    group 0, of group 1] in slot order with their ids (list of (x, y, id)); ops: [(group, n, rect)].  Returns
    (pos [2] lists of (x, y), id [2] lists, short, final minstd state)."""
    draws = Draws(mode, W, H, **draw_args)
    occ = np.array(walls, dtype=bool, copy=True)
    pos, ids = [[], []], [[], []]
    for g in range(2):
        src = fixed[1 - g] if side else fixed[g]
        for x, y, i in src:
            pos[g].append((x, y)); ids[g].append(i); occ[y, x] = True
    id_next = sum(len(f) for f in fixed)
    cells, short = place_sequential(draws, occ, ops)
    for (grp, n, _), c in zip(ops, cells):
        g = grp ^ side
        for j, (x, y) in enumerate(c):
            pos[g].append((x, y)); ids[g].append(id_next + j)
        id_next += n
    return pos, ids, short, draws.rs


def border_walls(W, H):
    w = np.zeros((H, W), dtype=bool)
    w[0, :] = w[-1, :] = True
    w[:, 0] = w[:, -1] = True
    return w
