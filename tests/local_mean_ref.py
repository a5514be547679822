"""numpy reference of the neighbourhood mean action (mfb_local_mean_action, kernel K7).  Pure numpy; no engine needed."""
import math

import numpy as np


def circle_offsets(radius):
    """(dx, dy) of the cells of CircleRange(radius, 0, parity 1) other than the centre, row-major -- the construction
    of magent_oracle.c:62-86 (Range.h:171-215): the radius is a float, the distances are computed in double."""
    r = float(np.float32(radius))
    eps = 1e-8
    width = 2 * int(r + eps) + 1
    center = int(r)
    if width % 2 != 1:
        width += 1
    out = []
    for i in range(width):
        for j in range(width):
            dis = math.sqrt(float(j - center) ** 2 + float(i - center) ** 2)
            if dis < r + eps and dis > 0.0 - eps and (i, j) != (center, center):
                out.append((j - center, i - center))
    return out


def local_mean_action(pos, last_action, alive, radius, n_action):
    """Brute force over all pairs of one group: pos int[n, 2] (x, y), last_action int[n], alive bool[n] ->
    float32[n, n_action].  Row i counts the agents j != i that are alive, have acted (last_action < n_action) and
    stand at an offset inside the disc (its centre included: a dead observer's cell may hold a living agent), and
    divides by their number in float32; zeros when there are none."""
    pos = np.asarray(pos, np.int64).reshape(-1, 2)
    last_action = np.asarray(last_action, np.int64).reshape(-1)
    alive = np.asarray(alive, bool).reshape(-1)
    n = len(pos)
    out = np.zeros((n, n_action), np.float32)
    if n == 0:
        return out
    offs = circle_offsets(radius)
    R = max([max(abs(dx), abs(dy)) for dx, dy in offs] + [0])
    table = np.zeros((2 * R + 1, 2 * R + 1), bool)
    table[R, R] = True
    for dx, dy in offs:
        table[dy + R, dx + R] = True
    dx = pos[None, :, 0] - pos[:, None, 0]                       # [observer, source]
    dy = pos[None, :, 1] - pos[:, None, 1]
    near = (np.abs(dx) <= R) & (np.abs(dy) <= R)
    near[near] = table[dy[near] + R, dx[near] + R]
    source = alive & (last_action >= 0) & (last_action < n_action)
    near &= source[None, :]
    np.fill_diagonal(near, False)
    onehot = np.zeros((n, n_action), np.int64)
    onehot[source, last_action[source]] = 1
    counts = near.astype(np.int64) @ onehot                     # [n, n_action]
    total = counts.sum(axis=1)
    has = total > 0
    out[has] = counts[has].astype(np.float32) / total[has, None].astype(np.float32)
    return out
