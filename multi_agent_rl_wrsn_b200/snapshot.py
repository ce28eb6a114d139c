"""``EnvSnapshot`` — the continuation state of some environments of a ``BatchedWRSN``: what ``BatchedWRSN.restore`` needs to
continue each of them exactly where ``BatchedWRSN.snapshot`` took it.

A row's continuation state is its whole state record, its scenario and its request row (``include/wrsn_b200.h``:
``wrsn_copy_rows``).  A record is laid out by the batch's dims, so a snapshot also carries the layout it was taken under (the
ABI version, the layout-defining dims and the state-layout offset table) and one fingerprint per scenario of its batch;
``restore`` refuses a snapshot whose layout differs from the target batch's, and finds each row's scenario in the target batch
by fingerprint.
"""
import hashlib

import numpy as np
import torch

from . import _lib

LAYOUT_DIMS = ("N", "T", "M", "S", "Npad", "W", "Tw", "n_slot", "Emax", "TEmax", "state_bytes")
REQ_FIELDS = ("agent_id", "terminal", "reward", "now", "action", "detail", "flags", "stats", "sticky")
_REQ_SPEC = dict(agent_id=(torch.int32, ()), terminal=(torch.uint8, ()), reward=(torch.float64, ()), now=(torch.float64, ()),
                 action=(torch.float64, (3,)), detail=(torch.float64, (2,)), flags=(torch.int32, ()),
                 stats=(torch.float64, (3,)), sticky=(torch.int32, ()))


def scenario_fingerprint(static):
    """sha256 of one scenario's ``build_static`` arrays and ``par`` row.  It depends on the scenario alone (not on the batch
    it sits in), and ``par`` holds the warm-up time and the charger type, so a scenario simulated under other constants has
    another fingerprint."""
    h = hashlib.sha256()
    for k in sorted(static):
        v = static[k]
        if k == "par":
            names = sorted(v)
            h.update(("par:" + ",".join(names)).encode())
            v = np.array([v[p] for p in names], np.float64)
        a = np.ascontiguousarray(np.asarray(v))
        h.update(("%s:%s:%s;" % (k, a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def c_request(req):
    """The ``wrsn_request`` of a dict of request tensors (no ``order``: it is launch scratch, never part of a row's state)."""
    return _lib.Request(*[req[f].data_ptr() if f in req else None for f, _ in _lib.Request._fields_])


class EnvSnapshot:
    """Rows of one or several ``BatchedWRSN`` (shards of one job), with global row ids.

    ``ids`` int64 [n]: global row ids; ``scen`` int32 [n]: index of each row's scenario in ``meta["fingerprints"]``;
    ``state`` uint8 [n, state_bytes]: the state records; ``req``: the request rows, a dict of tensors (``REQ_FIELDS``).
    ``meta``: ``abi`` (ABI version), ``dims`` (``LAYOUT_DIMS``), ``offsets`` (the state-layout offset table) and
    ``fingerprints`` (one per scenario)."""

    def __init__(self, meta, ids, scen, state, req):
        self.meta, self.ids, self.scen, self.state, self.req = meta, ids, scen, state, req

    def __len__(self):
        return int(self.ids.shape[0])

    @property
    def device(self):
        return self.state.device

    def to(self, device):
        device = torch.device(device)
        return EnvSnapshot(self.meta, self.ids.to(device), self.scen.to(device), self.state.to(device),
                           {f: t.to(device) for f, t in self.req.items()})

    def _take(self, idx):
        i = torch.as_tensor(idx, dtype=torch.int64, device=self.device)
        return EnvSnapshot(self.meta, self.ids[i].contiguous(), self.scen[i].contiguous(), self.state[i].contiguous(),
                           {f: t[i].contiguous() for f, t in self.req.items()})

    def select(self, global_ids):
        """The rows with these global ids, in this order."""
        pos = {int(g): k for k, g in enumerate(self.ids.tolist())}
        want = [int(g) for g in np.asarray(global_ids, np.int64).reshape(-1)]
        missing = [g for g in want if g not in pos]
        if missing:
            raise ValueError("ids: rows %s are not in the snapshot" % missing[:8])
        return self._take([pos[g] for g in want])

    @staticmethod
    def cat(snaps):
        """One snapshot of the rows of several (the shards of one job): same ABI and layout; the scenario lists are merged."""
        snaps = list(snaps)
        if not snaps:
            raise ValueError("cat: no snapshots")
        first = snaps[0].meta
        fps = []
        scen = []
        for s in snaps:
            check_layout(s.meta, first["abi"], first["dims"], first["offsets"])
            remap = []
            for fp in s.meta["fingerprints"]:
                if fp not in fps:
                    fps.append(fp)
                remap.append(fps.index(fp))
            scen.append(torch.as_tensor(remap, dtype=torch.int32, device=s.device)[s.scen.long()].to(snaps[0].device))
        meta = dict(first, fingerprints=fps)
        dev = snaps[0].device
        return EnvSnapshot(meta, torch.cat([s.ids.to(dev) for s in snaps]), torch.cat(scen), torch.cat([s.state.to(dev) for s in snaps]),
                           {f: torch.cat([s.req[f].to(dev) for s in snaps]) for f in REQ_FIELDS})

    def save(self, path):
        torch.save(dict(meta=self.meta, ids=self.ids.cpu(), scen=self.scen.cpu(), state=self.state.cpu(),
                        req={f: t.cpu() for f, t in self.req.items()}), path)

    @staticmethod
    def load(path, device=None):
        """A snapshot written by ``save``, on ``device`` (default the CPU; ``restore`` moves it to the batch's device)."""
        d = torch.load(path, map_location=torch.device("cpu") if device is None else torch.device(device), weights_only=True)
        return EnvSnapshot(d["meta"], d["ids"], d["scen"], d["state"], d["req"])

    def validate(self):
        """Shapes and dtypes of the rows against the metadata (a snapshot read from a file is outside input)."""
        n = len(self)
        sb = int(self.meta["dims"]["state_bytes"])
        if self.ids.dtype != torch.int64 or tuple(self.ids.shape) != (n,):
            raise ValueError("ids: int64 [n] expected")
        if self.scen.dtype != torch.int32 or tuple(self.scen.shape) != (n,):
            raise ValueError("scen: int32 [n] expected")
        if n and (int(self.scen.min()) < 0 or int(self.scen.max()) >= len(self.meta["fingerprints"])):
            raise ValueError("scen: scenario index outside the snapshot's %d fingerprints" % len(self.meta["fingerprints"]))
        if self.state.dtype != torch.uint8 or tuple(self.state.shape) != (n, sb) or not self.state.is_contiguous():
            raise ValueError("state: contiguous uint8 [n, %d] expected" % sb)
        for f in REQ_FIELDS:
            dt, tail = _REQ_SPEC[f]
            t = self.req.get(f)
            if t is None or t.dtype != dt or tuple(t.shape) != (n,) + tail or not t.is_contiguous() or t.device != self.state.device:
                raise ValueError("req.%s: contiguous %s %s expected" % (f, dt, [n] + list(tail)))


def layout_meta(L, dims, offsets, fingerprints):
    return dict(abi=int(L.wrsn_abi_version()), dims={k: int(getattr(dims, k)) for k in LAYOUT_DIMS},
                offsets=[int(o) for o in offsets], fingerprints=list(fingerprints))


def check_layout(meta, abi, dims, offsets):
    """ValueError naming the first field of ``meta`` that differs from (abi, dims, offsets)."""
    if int(meta["abi"]) != int(abi):
        raise ValueError("abi: snapshot ABI version %d, this library %d" % (int(meta["abi"]), int(abi)))
    for k in LAYOUT_DIMS:
        if int(meta["dims"][k]) != int(dims[k]):
            raise ValueError("dims.%s: snapshot %d, this batch %d" % (k, int(meta["dims"][k]), int(dims[k])))
    if len(meta["offsets"]) != len(offsets):
        raise ValueError("offsets: snapshot has %d state fields, this batch %d" % (len(meta["offsets"]), len(offsets)))
    for k, (a, b) in enumerate(zip(meta["offsets"], offsets)):
        if int(a) != int(b):
            raise ValueError("offsets[%d]: snapshot %d, this batch %d" % (k, int(a), int(b)))
