#!/usr/bin/env python
"""2+ GPU check of CpG-row sharding on the stream engine, i.e. for shapes the Gram form cannot run (run under torchrun on the GPU box):
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 tools/sharded_stream_check.py
1. A K = 6, n_u = 9 fit over NCCL and over the NVLink peer exchange (eager and as a replayed CUDA graph); rank 0 gathers u and
   compares alpha, u and the outer-iteration count with the CPU oracle on the full problem.
2. `demethify --shard rows --nbunknown 9` with K = 6 against a one-GPU run of the same command (CSV files).
3. evaluate_best_ic(shard="rows") for BIC and BCV over n_u = 7..10 at K = 6 (n_u = 7, 8 run on the Gram form, 9 and 10 on the stream
   engine) against the same sweep with shard="fits" on one GPU: criteria, the selected n_u, alpha and u.
With fewer GPUs than ranks the ranks share the GPUs: the collectives then go through gloo (NCCL refuses two ranks on one device),
and the NVLink peer exchange and the CUDA-graph case are left out (both need one GPU per rank)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    n_dev = torch.cuda.device_count()
    shared = n_dev < world
    dev = local % n_dev
    torch.cuda.set_device(dev)
    if shared:
        os.environ["LOCAL_RANK"] = str(dev)                # the CLI picks its device by local rank
        dist.init_process_group("gloo")
    else:
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    if rank == 0:
        print(f"sharded_stream_check: {world} ranks on {n_dev} x {torch.cuda.get_device_name()}, "
              f"{'gloo (ranks share GPUs)' if shared else 'NCCL'}", flush=True)
    import __graft_entry__ as g
    g.build()
    from demethify_b200 import sharded
    from demethify_b200.sharded import mdwbssmf_deconv_sharded, row_range
    from oracle import bssmf_numpy as orc
    from sharded_check import cli_check, ic_check
    rs = np.random.RandomState(6)
    M, N, K, n_u = 20011, 48, 6, 9
    a = rs.uniform(0.2, 1.0, size=K + 3)
    Rf = rs.beta(a, a, size=(M, K + 3))
    A = rs.dirichlet(np.ones(K + 3), N).T
    D = rs.poisson(50, size=(M, N)) + 1
    X = rs.binomial(D, np.clip(Rf @ A, 0, 1)) / D
    Rk = np.ascontiguousarray(Rf[:, :K])
    u0, R0, a0 = orc.draw_init("uniform_", X, D, Rk, n_u, seed=3)
    lo, hi = row_range(M, rank, world)
    ok = True
    # (iterations, tolerance, peer exchange, CUDA graph)
    cases = [(6, 10, 1e-9, "0", "0"), (200, 10, 30.0, "0", "0"), (6, 10, 1e-9, "1", "0"), (200, 10, 30.0, "1", "0"), (200, 10, 30.0, "1", "1")]
    for it1, it2, tol, peer, graph in [c for c in cases if not shared or c[3:] == ("0", "0")]:
        os.environ["DMF_PEER_XCHG"], os.environ["DMF_SHARDED_GRAPH"] = peer, graph
        if graph == "1":
            os.environ.setdefault("NCCL_GRAPH_REGISTER", "0")
        u, al, n_outer, cost = mdwbssmf_deconv_sharded(u0[lo:hi], a0, X[lo:hi], D[lo:hi], Rk[lo:hi], n_u, n_iter1=it1, n_iter2=it2, tol=tol)
        parts = [None] * world
        dist.all_gather_object(parts, (lo, u, al, n_outer))
        if rank == 0:
            tr = {}
            uo, ao = orc.solve_partial_reference(u0.copy(), R0, a0.copy(), X, D.astype(float), Rk, n_u, it1, it2, tol, trace=tr)
            ufull = np.vstack([p[1] for p in sorted(parts, key=lambda p: p[0])])
            same_alpha = all(np.array_equal(p[2], parts[0][2]) for p in parts)
            da, du = np.abs(al - ao).max(), np.abs(ufull - uo).max()
            good = same_alpha and all(p[3] == tr["n_outer"] for p in parts) and da <= 1e-6 and du <= 1e-6
            ok &= good
            print(f"sharded_stream_check world={world} K={K} n_u={n_u} peer_xchg={peer} graph={graph} it1={it1}: n_outer={n_outer} "
                  f"oracle={tr['n_outer']} max|d alpha|={da:.2e} max|d u|={du:.2e} alpha replicated={same_alpha} peer={sharded.last_info} "
                  f"-> {'OK' if good else 'FAIL'}", flush=True)
    os.environ["DMF_PEER_XCHG"], os.environ["DMF_SHARDED_GRAPH"] = "0" if shared else "1", "0"
    ok &= cli_check(rank, world, cases=[("uniform_", ["--nbunknown", "9"])], K=6)
    ok &= ic_check(rank, world, runs=(("BIC", "uniform_", 1), ("BCV", "uniform_", 4)), n_u_values=range(7, 11), K=6)
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
