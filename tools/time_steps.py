#!/usr/bin/env python
"""Wall time of the single solver steps deconvolution.update_u / update_alpha / frank_wolfe_nmf on a resident problem, next to
n_iter2 streaming passes of the same kind timed with CUDA events on a batch that already exists.  The difference is the per-call
cost of the step API: batch set-up, the upload of the iterates (and of R for update_alpha) and the read-back of the results.
Synthetic data drawn on the device; one JSON line.  Usage:
  python tools/time_steps.py [M N K n_u n_iter2]        (default 1000000 256 6 2 20, FP64)
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    import torch
    import __graft_entry__ as g
    g.build()
    from time_fused import device_problem
    from demethify_b200 import deconvolution as dec
    from demethify_b200.engine import DeviceProblem, FitBatch
    M, N, K, n_u, n_iter2 = (int(v) for v in sys.argv[1:6]) if len(sys.argv) > 5 else (1_000_000, 256, 6, 2, 20)
    dev = torch.device("cuda", 0)
    X, D, Rk = device_problem(torch, dev, M, N, K, n_u, 7)
    prob = DeviceProblem(X, D, Rk)
    dmax2 = float(D.max()) ** 2
    del X, D
    rs = np.random.RandomState(1)
    u = rs.uniform(size=(M, n_u))
    u_ = np.clip(u + 0.01 * rs.standard_normal((M, n_u)), 0, 1)
    A = rs.dirichlet(np.ones(K + n_u), N).T
    A_ = rs.dirichlet(np.ones(K + n_u), N).T
    R = np.hstack((Rk.cpu().numpy(), u))
    l_w = np.linalg.norm(A[-n_u:]) ** 2 * dmax2
    l_h = np.linalg.norm(R) ** 2 * dmax2
    pur = rs.uniform(size=N)
    H1, H2 = A[:K] * pur / A[:K].sum(0), A[K:] * (1 - pur) / A[K:].sum(0)

    def wall(fn, reps=5):
        fn()                                      # warm-up: module loads, allocator
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        return 1e3 * float(np.median(ts))

    out = {"M": M, "N": N, "K": K, "n_u": n_u, "n_iter2": n_iter2, "precision": "fp64", "problem": "resident"}
    out["update_u_ms"] = wall(lambda: dec.update_u(u, A, n_iter2, 2.5, 0.5 * l_w, l_w, u_, prob, None, n_u, None))
    out["update_alpha_ms"] = wall(lambda: dec.update_alpha(n_iter2, A, 2.5, 0.5 * l_h, l_h, A_, R, None, prob))
    out["frank_wolfe_nmf_ms"] = wall(lambda: dec.frank_wolfe_nmf(None, u, prob, H1, H2, pur, n_iter2, None))
    out["update_u_0_iter_ms"] = wall(lambda: dec.update_u(u, A, 0, 2.5, 0.5 * l_w, l_w, u_, prob, None, n_u, None))
    out["update_alpha_0_iter_ms"] = wall(lambda: dec.update_alpha(0, A, 2.5, 0.5 * l_h, l_h, A_, R, None, prob))
    out["batch_create_ms"] = wall(lambda: FitBatch(prob, n_u, [u], [A], engine="stream").close())

    # n_iter2 passes of each kind on one existing stream-engine batch, CUDA events
    b = FitBatch(prob, n_u, [u], [A], engine="stream")
    b.pass_init()
    for name, step in (("pass_u", b.pass_u), ("pass_alpha", b.pass_alpha)):
        for _ in range(3):
            step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record()
        for _ in range(reps * n_iter2):
            step()
        e1.record()
        torch.cuda.synchronize()
        out[f"{n_iter2}x_{name}_ms"] = e0.elapsed_time(e1) / reps
    b.close()
    out["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                capture_output=True, text=True).stdout.strip().splitlines()[0]
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
