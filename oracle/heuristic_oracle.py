"""numpy restatement of the hand-written charging rules of ``wrsn_heuristic_action`` (include/wrsn_b200.h), for the tests.

Plain arrays in, one decision out.  Every quantity is computed with the IEEE operations the rule names (numpy rounds each
product, sum and quotient separately, as the kernels do), and every choice is ``np.lexsort`` on ``(id, key)``: the smallest key,
ties to the lowest id.
"""
import numpy as np

KINDS = ("min_lifetime", "nearest_urgent")


def euclid(ax, ay, bx, by):
    """scipy.spatial.distance.euclidean of 2-vectors: sqrt(dot(u - v, u - v)), products and sum rounded separately."""
    dx = np.subtract(ax, bx)
    dy = np.subtract(ay, by)
    return np.sqrt(dx * dx + dy * dy)


def choose(kind, a, n, x, y, energy, cs, status, mc_x, mc_y, mc_status, mc_dest_x, mc_dest_y, par):
    """The node charger ``a`` is sent to, or -1 when no node is alive.  ``n``: the scenario's own node count (ids >= n are
    padding); ``mc_*``: one entry per charger; ``par``: mapping with THR, MC_R, MTM and CTM."""
    if kind not in KINDS:
        raise ValueError(kind)
    ids = np.arange(n)
    x, y = np.asarray(x, np.float64)[:n], np.asarray(y, np.float64)[:n]
    energy, cs = np.asarray(energy, np.float64)[:n], np.asarray(cs, np.float64)[:n]
    alive = np.asarray(status)[:n] == 1
    with np.errstate(divide="ignore", invalid="ignore"):
        life = np.where(cs <= 0.0, np.inf, (energy - par["THR"]) / cs)
    claimed = np.zeros(n, bool)
    for j in range(len(mc_x)):
        if j != a and mc_status[j] != 0:
            claimed |= euclid(x, y, mc_dest_x[j], mc_dest_y[j]) <= par["MC_R"]
    cand = alive & ~claimed
    if not cand.any():
        cand = alive
    if not cand.any():
        return -1
    c = ids[cand]
    if kind == "nearest_urgent":
        u = c[life[c] < par["MTM"] + par["CTM"]]
        if u.size:
            d = euclid(mc_x[a], mc_y[a], x[u], y[u])
            return int(u[np.lexsort((u, d))[0]])
    return int(c[np.lexsort((c, life[c]))[0]])


def action(i, a, x, y, energy, mc_x, mc_y, par):
    """The 3-vector for node ``i`` (``i < 0``: charger ``a`` stays at its position, charge 0).  ``par``: F0..F3, CAP, CAPMTHR."""
    w, h = par["F1"] - par["F0"], par["F3"] - par["F2"]
    px, py = (float(x[i]), float(y[i])) if i >= 0 else (float(mc_x[a]), float(mc_y[a]))
    fx = 0.0 if w == 0.0 else (px - par["F0"]) / w
    fy = 0.0 if h == 0.0 else (py - par["F2"]) / h
    c = 0.0 if i < 0 else min(1.0, max(0.0, (par["CAP"] - float(energy[i])) / par["CAPMTHR"]))
    return np.array([fx, fy, c], np.float64)
