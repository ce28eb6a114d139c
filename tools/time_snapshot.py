"""What copying running environments costs: BatchedWRSN.fork, snapshot, restore and EnvSnapshot files.

    python tools/time_snapshot.py [--envs 4096] [--preroll 200] [--reps 200]

Workload: the headline configuration of bench.py (--envs environments, 100-node / 100-target synthetic fields, three chargers, 64
topologies, step budget 60), pre-rolled --preroll steps under the reference's RandomController law decoded on the device, so the
records hold mid-episode state (steps in flight included).  Then, each timed with CUDA events over --reps repetitions after a
warm-up:

  fork          env.fork(first half, second half): host checks, one wrsn_copy_rows launch, the row counts refreshed;
  copy_kernel   the wrsn_copy_rows launch of that fork alone (row lists already on the device);
  index_copy    torch's index_copy_ of the same state bytes (state records only: no request rows, no scen_id), for comparison;
  snapshot      env.snapshot() of every row (allocation of the compact record included);
  restore       env.restore() of that snapshot into every row;

and save / load of the whole-batch snapshot to a file in a temporary directory with a host clock after a synchronise.  Bytes moved
count each state record and request row once read and once written; the state records of all rows (about 80 MB at 4096 rows)
fit the B200's 126 MB L2, so the rates may exceed what HBM alone would give.  Prints one JSON line per measurement and a summary
line with the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_agent_rl_wrsn_b200 import BatchedWRSN, EnvSnapshot, synthetic  # noqa: E402
from multi_agent_rl_wrsn_b200.controllers import BatchedRandomController  # noqa: E402

HBM_TBS = 7.7                                        # HGX B200 data sheet, one GPU
REQ_ROW_BYTES = 4 + 1 + 8 + 8 + 24 + 16 + 4 + 24 + 4 + 4   # request row fields and scen_id


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn, reps, warmup=10):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps          # us per call


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--envs", type=int, default=4096)
    p.add_argument("--topologies", type=int, default=64)
    p.add_argument("--preroll", type=int, default=200)
    p.add_argument("--reps", type=int, default=200)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_snapshot.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    scs = [synthetic(num_nodes=100, num_targets=100, seed=1000 + k) for k in range(a.topologies)]
    env = BatchedWRSN(scs, num_agent=3, num_envs=a.envs, device=dev, step_budget=60)
    obs = torch.zeros((env.B, 4, env.S, env.S), dtype=torch.float32, device=dev)
    act = torch.zeros((env.B, 3), dtype=torch.float64, device=dev)
    env.reset()
    env.get_state(out=obs)
    for _ in range(a.preroll):
        env.linear_controller_action(obs, BatchedRandomController.weights, out=act)
        env.rollout_step(act, obs)
    env.raise_on_error()
    torch.cuda.synchronize()
    B, half, sb = env.B, env.B // 2, env.dims.state_bytes
    in_flight = int((env.req.agent_id == -4).sum().item())
    src, dst = np.arange(half), np.arange(half, 2 * half)
    sr = torch.as_tensor(src.astype(np.int32), device=dev)
    dr = torch.as_tensor(dst.astype(np.int32), device=dev)
    me = (env.state, env.req.c, env.scen_id)
    idx = torch.as_tensor(dst, device=dev)
    rows_src = env.state[:half].clone()

    def copy_kernel():
        import ctypes as C
        env._call(env.L.wrsn_copy_rows, C.byref(env.dims), half, env.state.data_ptr(), C.byref(env.req.c), env.scen_id.data_ptr(),
                  sr.data_ptr(), B, env.state.data_ptr(), C.byref(env.req.c), env.scen_id.data_ptr(), dr.data_ptr(), B, env._stream())

    snap = env.snapshot()
    res = []

    def rec(name, us, rows):
        moved = 2 * rows * (sb + REQ_ROW_BYTES) if name != "index_copy" else 2 * rows * sb
        r = dict(measurement=name, rows=rows, us=round(us, 2), bytes_moved=moved, GBps=round(moved / us / 1e3, 1),
                 share_of_hbm_bound=round(moved / (HBM_TBS * 1e12) / (us * 1e-6), 3))
        res.append(r)
        print(json.dumps(r), flush=True)

    rec("fork", timed(lambda: env.fork(src, dst), a.reps), half)
    rec("copy_kernel", timed(copy_kernel, a.reps), half)
    rec("index_copy", timed(lambda: env.state.index_copy_(0, idx, rows_src), a.reps), half)
    rec("snapshot", timed(lambda: env.snapshot(), a.reps), B)
    rec("restore", timed(lambda: env.restore(snap), a.reps), B)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "rows.pt")
        saves, loads = [], []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            snap.save(path)
            saves.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            back = EnvSnapshot.load(path, device=dev)
            torch.cuda.synchronize()
            loads.append(time.perf_counter() - t0)
        size = os.path.getsize(path)
    assert torch.equal(back.state, snap.state)
    for name, ts in (("save", saves), ("load", loads)):
        r = dict(measurement=name, rows=B, file_bytes=size, ms_median=round(1e3 * float(np.median(ts)), 1),
                 ms_min=round(1e3 * min(ts), 1))
        res.append(r)
        print(json.dumps(r), flush=True)
    print(json.dumps(dict(summary=True, card=card(), envs=B, state_bytes=sb, rows_in_flight_at_preroll_end=in_flight,
                          preroll=a.preroll, reps=a.reps)), flush=True)


if __name__ == "__main__":
    main()
