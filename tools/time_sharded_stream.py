#!/usr/bin/env python
"""Timing of BASELINE config 5's stream-engine members (n_u = 9 and 10 at 1M x 256, K = 6, CLI defaults 10000 x 20, tol 1e-2),
CpG rows sharded over the GPUs of the run (torchrun; world size 1 runs without torchrun):
  python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port 29513 tools/time_sharded_stream.py
        [--outer K] [--full [--limit S]] [--nu 9,10] [--out path.jsonl]
Every rank generates the same problem on its GPU and keeps its rows.  For each member: ms per outer iteration over K timed outer
iterations (after one untimed), host clock around work that ends in a device synchronise; with --full also seconds for the whole
member (set-up + outer iterations to the termination test).  Rank 0 prints one JSON line per member with the card name and
power limit."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    name = torch.cuda.get_device_name()
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        power = f"unknown ({e!r})"
    return name, power


def main():
    args = sys.argv[1:]
    outer = int(args[args.index("--outer") + 1]) if "--outer" in args else 10
    out_path = args[args.index("--out") + 1] if "--out" in args else None
    limit = float(args[args.index("--limit") + 1]) if "--limit" in args else float("inf")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as g
    g.build()
    from demethify_b200.engine import DeviceProblem
    from demethify_b200.sharded import GpuShardBackend, RowShardedFit, row_range
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from time_fused import device_problem
    M, N, K, it1, it2, tol = 1_000_000, 256, 6, 10000, 20, 1e-2
    X, D, Rk = device_problem(torch, dev, M, N, K, 2, 55)
    lo, hi = row_range(M, rank, world)
    prob = DeviceProblem(X, D, Rk).row_slice(lo, hi)
    del X, D, Rk
    name, power = card()
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)
    for n_u in ([int(v) for v in args[args.index("--nu") + 1].split(",")] if "--nu" in args else (9, 10)):
        rs = np.random.RandomState(n_u)
        u0 = rs.uniform(size=(M, n_u))[lo:hi]
        a0 = rs.dirichlet(np.ones(K + n_u), N).T
        be = GpuShardBackend(prob, None, None, n_u, u0, a0)
        assert be.stream, be.batch.engine
        if world > 1:
            be.enable_peer_exchange()
        fit = RowShardedFit(be)
        fit.init()
        fit.outer(it2, 0.0)                            # untimed: first launches of every kernel
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for _ in range(outer):
            fit.outer(it2, 0.0)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) / outer * 1e3
        rec = {"config": "BASELINE c5 member, row-sharded stream engine", "M": M, "N": N, "K": K, "n_u": n_u, "gpus": world,
               "n_iter2": it2, "ms_per_outer": round(ms, 3), "timed_outer": outer, "peer_exchange": be.peer is not None,
               "collectives_per_outer": it2 + 2, "card": name, "power_limit": power}
        be.close()
        if "--full" in args:
            # the whole member as fit_row_sharded runs it (set-up, outer iterations, a poll of the done flags every 16), with a
            # progress line per poll; --limit S stops after S seconds and reports the outer iterations reached
            be = GpuShardBackend(prob, None, None, n_u, u0, a0)
            if world > 1:
                be.enable_peer_exchange()
            fit = RowShardedFit(be)
            barrier()
            t0 = time.perf_counter()
            fit.init()
            issued, done = 0, False
            while issued < it1 and not done and time.perf_counter() - t0 < limit:
                for _ in range(min(16, it1 - issued)):
                    fit.outer(it2, tol)
                issued += min(16, it1 - issued)
                done = be.all_done()
                if rank == 0:
                    print(f"n_u={n_u}: {issued} outer iterations issued, {time.perf_counter() - t0:.1f} s", file=sys.stderr, flush=True)
            (_u, _a, n_outer, cost), = be.results()
            rec.update(s_member=round(time.perf_counter() - t0, 2), n_outer=int(n_outer), cost=float(cost), converged=bool(done))
            be.close()
        if rank == 0:
            print(json.dumps(rec), flush=True)
            if out_path:
                with open(out_path, "a") as f:
                    f.write(json.dumps(rec) + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
