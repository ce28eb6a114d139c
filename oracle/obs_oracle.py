"""TEST INFRASTRUCTURE — float64 restatement of the reference's observation, ``WRSN.get_state``.

Follows ``rl_env/WRSN.py:130-186`` statement by statement, as ``orc_get_state`` in ``oracle/wrsn_oracle.c`` does: cell
centres from ``np.arange(unit / 2, 1.0, unit)``, one rank-1 term per source added in source order, ``(w * gx) * gy`` for the
nodes, the observer's own position and the charging chargers, ``((gx * gy) * w) / moving_time_max`` for the moving chargers
(with the observer's destination y, SURVEY Q5).  Its inputs are plain arrays, so a test can feed it whatever state the
device holds.  Only ``tests/`` may import this module: it is the checker of ``wrsn_observe`` (CUDA), never part of the
product path.

Pinned by ``tests/test_observe_raster.py`` against the golden episodes' observations and against ``orc_get_state``.
"""
import math

import numpy as np

# columns of the ``mc`` argument: one row per charger
MC_COLS = ("x", "y", "energy", "cpa0", "cpa1", "cpa2", "type")


def cell_centres(S):
    """np.arange(unit/2, 1.0, unit) (WRSN.py:135): numpy fills a[i] = start + i * ((start + unit) - start)."""
    unit = 1.0 / S
    c = np.arange(unit / 2, 1.0, unit)
    assert len(c) == S
    return c


def _g(c, x0, h):
    """WRSN.py:16-18, G(x; h) = exp(x^2 / (-2 h^2))."""
    u = c - x0
    return np.exp(u * u / (-2 * h ** 2))


def sources(frame, node_xy, status, energy, cs, mc, observer, consts):
    """The sources of the four channels, in the reference's order: a list per channel of (x0, y0, hx, hy, w, mode, tag),
    mode 0 = ``(w * gx) * gy``, mode 1 = ``((gx * gy) * w) / moving_time_max``; tag = node or charger index.
    ``mc``: [M, 7] with the columns of MC_COLS.  ``consts``: charging_range, alpha, beta, threshold, capacity (the nodes'),
    mc_capacity, velocity, charging_time_max, moving_time_max."""
    f = [float(v) for v in frame]
    W, H = f[1] - f[0], f[3] - f[2]
    R = float(consts["charging_range"])
    ab2 = consts["alpha"] / consts["beta"] ** 2
    thr, cap = float(consts["threshold"]), float(consts["capacity"])
    mc = np.asarray(mc, np.float64)
    me = mc[observer]
    out = [[], [], [], []]
    for n in range(len(status)):
        if status[n] == 0:
            continue
        w = (float(cs[n]) / ab2) / ((float(energy[n]) - thr) / (cap - thr))
        out[0].append(((node_xy[n][0] - f[0]) / W, (node_xy[n][1] - f[2]) / H, R / W, R / H, w, 0, n))
    tmp = min(H, W)
    out[1].append(((me[0] - f[0]) / W, (me[1] - f[2]) / H, 0.5 * tmp / W, 0.5 * tmp / H,
                   me[2] / consts["mc_capacity"], 0, observer))
    for a in range(len(mc)):
        an = mc[a]
        if a == observer or an[6] == 0:
            continue
        out[2].append(((an[3] - f[0]) / W, (an[4] - f[2]) / H, R / W, R / H, an[5] / consts["charging_time_max"], 0, a))
    for a in range(len(mc)):
        an = mc[a]
        if a == observer or an[6] != 0:
            continue
        dx, dy = float(an[0]) - float(an[3]), float(an[1]) - float(me[4])
        out[3].append(((an[3] - f[0]) / W, (an[4] - f[2]) / H, R / W, R / H, math.sqrt(dx * dx + dy * dy) / consts["velocity"], 1, a))
    return out


def term(S, src, moving_time_max):
    """One source's rank-1 term of an S x S channel."""
    x0, y0, hx, hy, w, mode = src[:6]
    c = cell_centres(S)
    gx, gy = _g(c, x0, hx), _g(c, y0, hy)
    if mode == 0:
        return np.outer(w * gx, gy)
    return np.outer(gx, gy) * w / moving_time_max


def raster(S, srcs, moving_time_max):
    """The 4 x S x S observation: every channel the sum of its sources' terms, added one by one in source order."""
    out = np.zeros((4, S, S))
    for ch in range(4):
        for s in srcs[ch]:
            out[ch] += term(S, s, moving_time_max)
    return out


def get_state(frame, node_xy, status, energy, cs, mc, observer, S, consts):
    """WRSN.get_state of charger ``observer``: float64 [4, S, S]."""
    return raster(S, sources(frame, node_xy, status, energy, cs, mc, observer, consts), consts["moving_time_max"])
