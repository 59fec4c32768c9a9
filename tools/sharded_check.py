#!/usr/bin/env python
"""2+ GPU check of CpG-row sharding (run under torchrun on the GPU box):
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/sharded_check.py
Every rank fits its row range over NCCL; rank 0 gathers u and compares alpha, u and the outer-iteration count with the
CPU oracle on the full problem.  Then the `demethify` command runs its main fit with --shard rows for every init option (partial,
purity, reference-free, n_u = 0) and rank 0 compares the CSV files with a one-GPU run of the same seed.  Last, CCC and BCV
sweeps run row-sharded (evaluate_best_ic(shard="rows"), what `--shard rows --ic` runs) and rank 0 compares the criteria, the selected
n_u, alpha and u with the same sweep on one GPU."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import __graft_entry__ as g
    g.build()
    from demethify_b200 import sharded
    from demethify_b200.sharded import mdwbssmf_deconv_sharded, row_range
    from oracle import bssmf_numpy as orc
    rs = np.random.RandomState(5)
    M, N, K, n_u = 20011, 48, 6, 2
    a = rs.uniform(0.2, 1.0, size=K + n_u)
    Rf = rs.beta(a, a, size=(M, K + n_u))
    A = rs.dirichlet(np.ones(K + n_u), N).T
    D = rs.poisson(50, size=(M, N)) + 1
    X = rs.binomial(D, np.clip(Rf @ A, 0, 1)) / D
    Rk = np.ascontiguousarray(Rf[:, :K])
    u0, R0, a0 = orc.draw_init("uniform_", X, D, Rk, n_u, seed=3)
    lo, hi = row_range(M, rank, world)
    ok = True
    # (iterations, tolerance, peer exchange, CUDA graph): NCCL and the in-kernel NVLink exchange, eager and as a replayed graph
    # (the exchange count lives on the device, so replays advance it)
    cases = [(6, 20, 1e-9, "0", "0"), (400, 20, 1.0, "0", "0"), (6, 20, 1e-9, "1", "0"), (400, 20, 1.0, "1", "0"), (400, 20, 1.0, "1", "1"),
             (400, 20, 1.0, "0", "1")]
    for it1, it2, tol, peer, graph in cases:
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
            print(f"sharded_check world={world} peer_xchg={peer} graph={graph} it1={it1}: n_outer={n_outer} oracle={tr['n_outer']} max|d alpha|={da:.2e} max|d u|={du:.2e} "
                  f"alpha replicated={same_alpha} peer={sharded.last_info} -> {'OK' if good else 'FAIL'}", flush=True)
    ok &= cli_check(rank, world)
    ok &= ic_check(rank, world)
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


def cli_check(rank, world):
    import tempfile
    import pandas as pd
    from demethify_b200 import demethify
    rs = np.random.RandomState(8)
    M, N, K = 9001, 10, 5
    Rf = rs.beta(0.5, 0.5, size=(M, K + 2))
    D = rs.poisson(40, size=(M, N)) + 1
    X = rs.binomial(D, np.clip(Rf @ rs.dirichlet(np.ones(K + 2), N).T, 0, 1)) / D
    box = [tempfile.mkdtemp(prefix="dmf_cli_") if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    d = box[0]
    if rank == 0:
        pd.DataFrame(Rf[:, :K], columns=[f"ct{k}" for k in range(K)]).to_csv(f"{d}/ref.csv", index=False)
        for j in range(N):
            pd.DataFrame({"percent_modified": X[:, j], "valid_coverage": D[:, j]}).to_csv(f"{d}/s{j}.csv", index=False)
    dist.barrier()
    files = [f"{d}/s{j}.csv" for j in range(N)]
    cases = [("uniform_", ["--nbunknown", "2"]), ("uniform", ["--nbunknown", "2"]), ("beta", ["--nbunknown", "2"]),
             ("SVD", ["--nbunknown", "2"]), ("SVD", ["--nbunknown", "2", "--purity"] + ["60"] * N), ("SVD", ["--nbunknown", "2", "--noref"]),
             ("uniform_", ["--nbunknown", "0"])]
    ok = True
    for c, (init, extra) in enumerate(cases):
        ref = [] if "--noref" in extra else ["--ref", f"{d}/ref.csv"]
        extra = [e for e in extra if e != "--noref"]
        common = ["--methfreq"] + files + ref + ["--init", init, "--iterations", "300", "20", "--termination", "1e-2", "--seed", "3",
                                                  "--noprint"] + extra
        demethify.main(common + ["--outdir", f"{d}/rows{c}", "--shard", "rows"])
        dist.barrier()
        if rank == 0:
            env = os.environ["WORLD_SIZE"]
            os.environ["WORLD_SIZE"] = "1"                         # the same command on one GPU
            try:
                demethify.main(common + ["--outdir", f"{d}/one{c}"])
            finally:
                os.environ["WORLD_SIZE"] = env
            dev = 0.0
            for name in ("celltypes_proportions.csv", "methylation_profile_estimate.csv"):
                if os.path.exists(f"{d}/one{c}/{name}"):
                    a = pd.read_csv(f"{d}/rows{c}/{name}").select_dtypes("number").values
                    b = pd.read_csv(f"{d}/one{c}/{name}").select_dtypes("number").values
                    dev = max(dev, np.abs(a - b).max() if a.shape == b.shape else np.inf)
            good = dev <= 1e-6
            ok &= good
            print(f"sharded_check cli world={world} --init {init} {' '.join(extra[:3])}{' (reference-free)' if not ref else ''}: "
                  f"max|rows - one GPU|={dev:.2e} -> {'OK' if good else 'FAIL'}", flush=True)
        dist.barrier()
    box = [ok]
    dist.broadcast_object_list(box, src=0)
    return box[0]


def ic_check(rank, world):
    from demethify_b200.ic import evaluate_best_ic
    rs = np.random.RandomState(9)
    M, N, K = 30011, 12, 5
    Rf = rs.beta(0.5, 0.5, size=(M, K + 2))
    D = rs.poisson(40, size=(M, N)) + 1
    X = rs.binomial(D, np.clip(Rf @ rs.dirichlet(np.ones(K + 2), N).T, 0, 1)) / D
    one = dist.new_group([0])
    ok = True
    for crit, init, seed in (("CCC", "uniform_", 1), ("CCC", "SVD", 2), ("BCV", "uniform_", [3]), ("BCV", "uniform", 4), ("BCV", "SVD", 5)):
        u, a, best, values = evaluate_best_ic(X, Rf[:, :K], D, init, crit, seed, 300, 20, 1e-2, n_restarts=3, n_u_values=[1, 2, 3],
                                              shard="rows")
        if rank == 0:
            u1, a1, best1, values1 = evaluate_best_ic(X, Rf[:, :K], D, init, crit, seed, 300, 20, 1e-2, n_restarts=3, n_u_values=[1, 2, 3],
                                                      shard="fits", group=one)
            dv = np.abs(np.array(values) - np.array(values1)).max()
            da, du = np.abs(a - a1).max(), np.abs(u - u1).max()
            good = best == best1 and dv <= 1e-8 * max(1.0, np.abs(values1).max()) and da <= 1e-8 and du <= 1e-8
            ok &= good
            print(f"sharded_check ic world={world} {crit} --init {init} seed={seed}: best n_u {best} (one GPU {best1}) max|d criterion|={dv:.2e} "
                  f"max|d alpha|={da:.2e} max|d u|={du:.2e} -> {'OK' if good else 'FAIL'}", flush=True)
        dist.barrier()
    box = [ok]
    dist.broadcast_object_list(box, src=0)
    return box[0]


if __name__ == "__main__":
    main()
