"""GPU tests of the row-sharded CCC and BCV members on one device (world size 1, so every all-reduce is the identity): they must
give the criteria, the best n_u and the alpha of the single-process sweep (evaluate_best_ic with shard="fits"), and a row-sharded
batch of several fits must give every fit exactly what a one-fit row-sharded run gives.  Several processes are covered on CPU
(tests/test_sharded_ic_cpu.py, gloo) and on 2 GPUs by tools/sharded_check.py (torchrun)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
IT1, IT2, TOL = 10000, 20, 1e-2
N_RUNS = 3


@pytest.fixture(scope="module")
def lib():
    import torch
    assert torch.cuda.is_available()
    import __graft_entry__ as g
    g.build()
    from demethify_b200 import ic, sharded
    return ic, sharded


@pytest.mark.parametrize("criterion", ["CCC", "BCV"])
@pytest.mark.parametrize("init", ["uniform_", "uniform"])
def test_row_sharded_members_equal_single_process_sweep(lib, shipped, criterion, init):
    ic, _ = lib
    X, D, Rk = shipped["X"], shipped["D"], shipped["Rk"]
    M = X.shape[0]
    n_us, seed = [1, 2, 3], 2
    u1, a1, best1, values1 = ic.evaluate_best_ic(X, Rk, D, init, criterion, seed, IT1, IT2, TOL, n_restarts=N_RUNS, n_u_values=n_us,
                                                 shard="fits")
    values, payload = [], []
    for n_u in n_us:
        if criterion == "CCC":
            runs, u, a = ic.consensus_runs_sharded(X, D, Rk, M, 0, M, n_u, init, [seed + r for r in range(N_RUNS)], IT1, IT2, TOL)
            values.append(-ic.compute_ccc(runs))
        else:
            total, u, a, _errors = ic.bicross_validation_sharded(X, D, Rk, M, 0, M, n_u, init, seed, N_RUNS, IT1, IT2, TOL)
            values.append(total)
        payload.append((u, a))
    assert np.abs(np.array(values) - np.array(values1)).max() <= 1e-10 * max(1.0, np.abs(values1).max())
    best = int(np.argmin(values))
    assert n_us[best] == best1
    assert np.abs(payload[best][1] - a1).max() <= 1e-8 and np.abs(payload[best][0] - u1).max() <= 1e-8


@pytest.mark.parametrize("gram", [False, True])
def test_row_sharded_batch_equals_one_fit_runs(lib, shipped, gram):
    """R fits as ONE row-sharded batch (one statistics block, all-reduced copy and peer slot per fit) against R one-fit row-sharded
    runs: alpha bit for bit and the same outer-iteration count, on the fused engine and on the Gram-form engine."""
    from demethify_b200 import engine
    from demethify_b200.deconvolution import init_BSSMF_md
    _, sh = lib
    X, D, Rk = shipped["X"], shipped["D"], shipped["Rk"]
    n_u = 2
    inits = [init_BSSMF_md("uniform_", X, D, Rk, n_u, seed=s)[::2] for s in (3, 4, 5, 6)]
    engine.FUSED_SLOTS = not gram
    try:
        be = sh.GpuShardBackend(X, D, Rk, n_u, [i[0] for i in inits], [i[1] for i in inits])
        assert be.fused == (not gram)
        batch = sh.fit_row_sharded(be, 300, IT2, 1e-6)
        for (u0, a0), (u, a, n_outer, cost) in zip(inits, batch):
            u1, a1, n1, c1 = sh.mdwbssmf_deconv_sharded(u0, a0, X, D, Rk, n_u, n_iter1=300, n_iter2=IT2, tol=1e-6)
            assert n_outer == n1 and np.array_equal(a, a1) and np.array_equal(u, u1) and cost == c1
    finally:
        engine.FUSED_SLOTS = True
