"""Scenarios: the reference's YAML schema, the static communication graph, and a synthetic generator.

Mirrors ``physical_env/network/NetworkIO.py:15-34`` (YAML -> nodes / targets / base station /
``node_phy_spe`` / ``seed`` / ``max_time``), ``Network.__init__`` (``Network.py:16-27``: frame and node
density), ``Node.probe_neighbors`` / ``probe_targets`` (``Node.py:80-90``), ``BaseStation.probe_neighbors``
(``BaseStation.py:20-23``) and the per-hop transmit cost of ``Node.send_package`` (``Node.py:107-115``).

Everything here is *static* per scenario, so it is evaluated once on the host with the very arithmetic
the reference uses (numpy float64 ``sqrt(dx*dx+dy*dy)`` for ``scipy...euclidean``, Python ``**`` for the
powers) and shipped to the GPU as data; thresholds and constants are therefore bit-identical.
"""
import math
from dataclasses import dataclass, field

import numpy as np
import yaml

DEFAULT_NODE_PHY = dict(capacity=10800, com_range=80.1, efs=1.0e-08, emp=1.3e-12, er=0.0001, et=5.0e-05,
                        package_size=400, prob_gp=1, sen_range=40.1, threshold=540)   # hanoi1000n50.yaml:1-11
SHIPPED_MAX_TIME = 604800.0                          # max_time of hanoi1000n*.yaml / sonla1000n50.yaml (line 13 of each)
DEFAULT_MC = dict(capacity=108000, threshold=0, velocity=5, pm=1, charging_range=27, alpha=4500, beta=30,
                  epsilon=1e-10)                                                     # mc_types/default.yaml:2-9


@dataclass
class Scenario:
    nodes: np.ndarray                 # [N, 2] float64
    targets: np.ndarray               # [T, 2] float64
    base_station: np.ndarray          # [2]
    node_phy_spe: dict = field(default_factory=lambda: dict(DEFAULT_NODE_PHY))
    seed: int = 0
    max_time: float = 604800.0
    name: str = ""

    @property
    def N(self):
        return int(self.nodes.shape[0])

    @property
    def T(self):
        return int(self.targets.shape[0])

    # -- reference schema ------------------------------------------------------------------------
    @staticmethod
    def from_dict(d, name="", default_max_time=None):
        """``default_max_time``: the fix-up switch for scenarios that ship without ``max_time`` (the reference's four
        ``bacgiang_*.yaml``: ``NetworkIO.py:34`` raises ``KeyError`` on them, SURVEY Q10 / §8 f3).  ``None`` keeps the
        reference's behaviour (``KeyError``); a number — e.g. ``SHIPPED_MAX_TIME``, what the five loadable scenarios
        carry — is used where the key is missing."""
        if "max_time" not in d:
            if default_max_time is None:
                raise KeyError("scenario has no 'max_time' (NetworkIO.py:34 would raise too): pass default_max_time=... "
                               "(e.g. scenario.SHIPPED_MAX_TIME) to load it")
            d = dict(d, max_time=float(default_max_time))
        spe = dict(d["node_phy_spe"])
        if float(spe.get("prob_gp", 1)) < 1.0:
            raise ValueError("prob_gp < 1 needs the reference's MT19937 stream (SURVEY Q12); not supported")
        return Scenario(nodes=np.array(d["nodes"], np.float64).reshape(-1, 2),
                        targets=np.array(d["targets"], np.float64).reshape(-1, 2),
                        base_station=np.array(d["base_station"], np.float64).reshape(2),
                        node_phy_spe=spe, seed=int(d.get("seed", 0)), max_time=float(d["max_time"]), name=name)

    @staticmethod
    def load_yaml(path, default_max_time=None):
        with open(path) as f:
            return Scenario.from_dict(yaml.safe_load(f), name=str(path), default_max_time=default_max_time)

    def to_dict(self):
        """Reference-schema dict (``yaml.safe_dump`` of it loads in ``NetworkIO``)."""
        return dict(node_phy_spe={k: (float(v) if isinstance(v, float) else v) for k, v in self.node_phy_spe.items()},
                    seed=int(self.seed), max_time=float(self.max_time),
                    base_station=[float(self.base_station[0]), float(self.base_station[1])],
                    nodes=[[float(x), float(y)] for x, y in self.nodes],
                    targets=[[float(x), float(y)] for x, y in self.targets])

    def save_yaml(self, path):
        with open(path, "w") as f:
            yaml.safe_dump(self.to_dict(), f)


def load_mc_type(path_or_dict=None):
    if path_or_dict is None:
        return dict(DEFAULT_MC)
    if isinstance(path_or_dict, dict):
        return dict(path_or_dict)
    with open(path_or_dict) as f:
        return yaml.safe_load(f)


def _pairwise(ax, ay, bx, by):
    dx = ax[:, None] - bx[None, :]
    dy = ay[:, None] - by[None, :]
    return np.sqrt(dx * dx + dy * dy)


def _e_send(d, spe):
    """``Node.send_package`` :107-115 with Python floats (``**`` is libm ``pow`` exactly as in the reference)."""
    d = float(d)
    et, efs, emp, size = float(spe["et"]), float(spe["efs"]), float(spe["emp"]), spe["package_size"]
    d0 = (efs / emp) ** 0.5
    return float(((et + efs * d ** 2) if d <= d0 else (et + emp * d ** 4)) * size)


def build_static(sc, mc, warm_up_time=100.0):
    """Static graph + constants of one scenario as numpy arrays (see ``include/wrsn_b200.h`` WRSN_S_* / WRSN_P_*)."""
    spe = sc.node_phy_spe
    x = np.ascontiguousarray(sc.nodes[:, 0], np.float64)
    y = np.ascontiguousarray(sc.nodes[:, 1], np.float64)
    N, T = sc.N, sc.T
    bsx, bsy = float(sc.base_station[0]), float(sc.base_station[1])
    com, sen = float(spe["com_range"]), float(spe["sen_range"])
    dnn = _pairwise(x, y, x, y)                                   # dnn[i, j] = euclid(node j, node i)
    nbr = (dnn <= com) & ~np.eye(N, dtype=bool)
    nbr_ptr = np.zeros(N + 1, np.int32)
    nbr_ptr[1:] = np.cumsum(nbr.sum(1))
    ii, jj = np.nonzero(nbr)                                      # row-major: neighbours in id order
    nbr_idx = jj.astype(np.int32)
    nbr_dist = dnn[ii, jj].astype(np.float64)
    nbr_esend = np.array([_e_send(d, spe) for d in nbr_dist], np.float64)
    if T > 0:
        tx = np.ascontiguousarray(sc.targets[:, 0], np.float64)
        ty = np.ascontiguousarray(sc.targets[:, 1], np.float64)
        dnt = _pairwise(x, y, tx, ty)
        cov = dnt <= sen
    else:
        cov = np.zeros((N, 0), bool)
    tgt_ptr = np.zeros(N + 1, np.int32)
    tgt_ptr[1:] = np.cumsum(cov.sum(1))
    tgt_idx = np.nonzero(cov)[1].astype(np.int32)
    dbs = np.sqrt((x - bsx) * (x - bsx) + (y - bsy) * (y - bsy))  # euclid(BS, node): squares are sign-blind
    direct = (dbs <= com).astype(np.uint8)
    bs_esend = np.array([_e_send(d, spe) for d in dbs], np.float64)

    # Network.frame / nodes_density (Network.py:16-27)
    f0 = min(bsx, float(x.min())); f1 = max(bsx, float(x.max()))
    f2 = min(bsy, float(y.min())); f3 = max(bsy, float(y.max()))
    density = N / ((f1 - f0) * (f3 - f2))
    cap, thr = spe["capacity"], spe["threshold"]
    # WRSN.reset :50-52
    mtm = float(np.sqrt((f0 - f1) * (f0 - f1) + (f2 - f3) * (f2 - f3))) / mc["velocity"]
    ctm = (cap - thr) / (mc["alpha"] / (mc["beta"] ** 2))
    avgna = density * np.pi * (mc["charging_range"] ** 2)
    par = dict(CAP=cap, THR=thr, ERECV=spe["er"] * spe["package_size"], BSX=bsx, BSY=bsy, F0=f0, F1=f1, F2=f2, F3=f3,
               MAXTIME=sc.max_time, WARMUP=warm_up_time, MTM=mtm, CTM=ctm, AVGNA=avgna,
               MC_CAP=mc["capacity"], MC_THR=mc["threshold"], MC_V=mc["velocity"], MC_PM=mc["pm"],
               MC_R=mc["charging_range"], MC_ALPHA=mc["alpha"], MC_BETA=mc["beta"], MC_EPS=mc["epsilon"],
               MC_AB2=mc["alpha"] / (mc["beta"] ** 2), MC_CAP200=mc["capacity"] / 200.0, MC_PMV=mc["pm"] * mc["velocity"],
               EPSENV=1e-9, CAPMTHR=cap - thr,
               ESMAX=max([float(spe["er"] * spe["package_size"])] + list(nbr_esend) + list(bs_esend)),
               INVN=1.0 / float(N), NNODES=N, NTARGETS=T)
    return dict(N=N, T=T, x=x, y=y, nbr_ptr=nbr_ptr, nbr_idx=nbr_idx, nbr_dist=nbr_dist, nbr_esend=nbr_esend,
                tgt_ptr=tgt_ptr, tgt_idx=tgt_idx, direct=direct, bs_esend=bs_esend,
                par={k: float(v) for k, v in par.items()}, frame=np.array([f0, f1, f2, f3]), nodes_density=density)


def synthetic(num_nodes=100, num_targets=None, seed=0, num_gateways=3, node_phy_spe=None, max_time=604800.0):
    """Synthetic network in the reference's schema (SURVEY §8d).

    A sensor tree grown outward from ``num_gateways`` nodes on a ring inside the base station's
    communication range (hop length 0.60-0.95 com_range, no two nodes closer than 0.45 com_range, so the
    mean degree stays near the shipped scenarios' 2.1-2.3), in a square field of side 1000*sqrt(N/100) m
    with the base station at the centre; every target lies within 0.9 sen_range of some non-gateway node, so
    all targets are covered and connected at t = 0.
    """
    spe = dict(DEFAULT_NODE_PHY if node_phy_spe is None else node_phy_spe)
    N = int(num_nodes)
    T = N if num_targets is None else int(num_targets)
    rng = np.random.default_rng(seed)
    side = 1000.0 * math.sqrt(N / 100.0)
    bs = np.array([side / 2.0, side / 2.0])
    com, sen = float(spe["com_range"]), float(spe["sen_range"])
    g = max(1, min(int(num_gateways), N))
    pts = []
    a0 = rng.uniform(0, 2 * math.pi)
    for k in range(g):
        a = a0 + 2 * math.pi * k / g + rng.uniform(-0.15, 0.15)
        r = com * rng.uniform(0.70, 0.85)
        pts.append(bs + r * np.array([math.cos(a), math.sin(a)]))
    depth = [1] * g
    min_sep = 0.45 * com
    tries = 0
    while len(pts) < N:
        tries += 1
        if tries > 400000:
            raise RuntimeError("synthetic(): could not place all nodes")
        P = np.array(pts)
        # prefer shallow-ish frontier nodes so the tree spreads over the field instead of snaking
        w = 1.0 / (1.0 + np.array(depth, np.float64)) ** 0.5
        parent = int(rng.choice(len(pts), p=w / w.sum()))
        a = rng.uniform(0, 2 * math.pi)
        q = P[parent] + com * rng.uniform(0.60, 0.95) * np.array([math.cos(a), math.sin(a)])
        if not (0.0 <= q[0] <= side and 0.0 <= q[1] <= side):
            continue
        d = np.sqrt(((P - q) ** 2).sum(1))
        if d.min() < min_sep:
            continue
        if np.sqrt(((q - bs) ** 2).sum()) <= com * 1.02:      # keep the direct set to the gateways
            continue
        pts.append(q)
        depth.append(depth[parent] + 1)
    nodes = np.array(pts, np.float64)
    hosts = rng.integers(g if N > g else 0, N, size=T)
    ang = rng.uniform(0, 2 * math.pi, size=T)
    rad = sen * 0.9 * np.sqrt(rng.uniform(0, 1, size=T))
    targets = nodes[hosts] + np.stack([rad * np.cos(ang), rad * np.sin(ang)], 1)
    return Scenario(nodes=nodes, targets=targets.astype(np.float64), base_station=bs, node_phy_spe=spe,
                    seed=int(seed), max_time=float(max_time), name="synthetic_n%d_t%d_s%d" % (N, T, seed))
