"""WRSN.get_network_fitness (rl_env/WRSN.py:188-220) restated with numpy (TEST INFRASTRUCTURE).

The reference gives every target the best lifetime with which some alive node covering it can still deliver to the base
station: over the paths of alive nodes from that node to one within communication range of the base station, the largest
bottleneck (minimum) of the nodes' lifetimes ``(energy - threshold) / energyCS`` (``+inf`` when ``energyCS == 0``).  A target
that no such node covers gets 0, and the fitness is the minimum over the targets (``+inf`` without targets).

Three implementations compute it by different algorithms: the C oracle (``orc_fitness``) by a label-correcting breadth-first
search from the direct nodes; the step kernel (``do_fitness``) by seeding each node with the bottleneck of its own routing
path and relaxing a max-min fixpoint; this file by label setting — a Dijkstra-style search that settles the nodes in
decreasing order of their widest-path value — over the static neighbour graph, built here from the coordinates with no
routing tree.  Only comparisons, minima and maxima touch the lifetimes after the one division, so all three must agree
bit for bit.
"""
import heapq

import numpy as np


def static_graph(nodes, targets, bs, com_range, sen_range):
    """``Node.probe_neighbors`` / ``probe_targets`` / ``BaseStation.probe_neighbors`` (Node.py:80-90, BaseStation.py:20-23):
    neighbour lists (within ``com_range``, in id order), the targets each node covers (within ``sen_range``) and the direct
    nodes (within ``com_range`` of the base station).  Distances are ``sqrt(dx * dx + dy * dy)`` with the products and the
    sum rounded separately (DESIGN §5)."""
    p = np.asarray(nodes, np.float64).reshape(-1, 2)
    t = np.asarray(targets, np.float64).reshape(-1, 2)
    bs = np.asarray(bs, np.float64).reshape(2)

    def dist(a, b):
        dx = a[:, None, 0] - b[None, :, 0]
        dy = a[:, None, 1] - b[None, :, 1]
        return np.sqrt(dx * dx + dy * dy)
    dnn = dist(p, p)
    near = (dnn <= com_range) & ~np.eye(len(p), dtype=bool)
    cover = dist(p, t) <= sen_range if len(t) else np.zeros((len(p), 0), bool)
    return dict(nbr=[np.nonzero(r)[0] for r in near], cover=[np.nonzero(r)[0] for r in cover],
                direct=dist(p, bs[None])[:, 0] <= com_range, T=len(t))


def lifetimes(energy, cs, status, threshold):
    """Per node ``(energy - threshold) / energyCS``, ``+inf`` where ``energyCS == 0``; NaN for dead nodes."""
    energy, cs = np.asarray(energy, np.float64), np.asarray(cs, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        lt = np.where(cs == 0.0, np.inf, (energy - threshold) / np.where(cs == 0.0, 1.0, cs))
    return np.where(np.asarray(status) == 1, lt, np.nan)


def widest_paths(graph, lt):
    """Per node the largest bottleneck of ``lt`` over the paths of alive nodes to a direct node (NaN where there is none)."""
    alive = ~np.isnan(lt)
    best = np.full(len(lt), np.nan)
    heap = [(-lt[i], int(i)) for i in np.nonzero(graph["direct"] & alive)[0]]
    heapq.heapify(heap)
    while heap:
        v, i = heapq.heappop(heap)
        if not np.isnan(best[i]):
            continue
        best[i] = -v
        for j in graph["nbr"][i]:
            if alive[j] and np.isnan(best[j]):
                heapq.heappush(heap, (-min(-v, lt[j]), int(j)))
    return best


def fitness(graph, energy, cs, status, threshold):
    """(minimum, per-target values [T], per-node widest-path values [N]) of ``WRSN.get_network_fitness``."""
    node = widest_paths(graph, lifetimes(energy, cs, status, threshold))
    per_target = np.zeros(graph["T"])
    for i in np.nonzero(node > 0.0)[0]:
        for t in graph["cover"][i]:
            per_target[t] = max(per_target[t], node[i])
    return (float(per_target.min()) if graph["T"] else np.inf), per_target, node
