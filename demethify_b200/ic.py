"""Mirror of the reference's demethify/ic.py: choosing the number of unknown cell types.

run_deconvolution / evaluate_best_ic / bicross_validation keep the reference signatures.  The fits of one n_u
(CCC restarts, BCV folds) are one batched launch set; the scalar criteria and the consensus clustering are the
reference's formulas on the host (SURVEY 2.1 row 6, Q9-Q11, Q15).
"""
import numpy as np
import torch.distributed as dist
import tqdm

from . import _lib
from .deconvolution import _initial_iterate, init_BSSMF_md, mdwbssmf_deconv, unsupervised_deconv, cost_f_w, last_fit_info
from .engine import DeviceProblem, FitBatch

__all__ = ["compute_bic", "compute_aic", "compute_consensus_matrix", "compute_ccc", "run_deconvolution", "bicross_validation",
           "evaluate_best_ic", "merge_sweep", "sweep_member_supported", "consensus_runs_sharded", "bicross_validation_sharded"]


def _world(group=None):
    return (dist.get_rank(group), dist.get_world_size(group)) if dist.is_available() and dist.is_initialized() else (0, 1)


def merge_sweep(local_results, local_payload, n_values, group=None):
    """Fit sharding of the n_u sweep (ic.py:192-216; every n_u re-seeds and is independent): rank r evaluated the positions
    r, r + world, ... of the sweep.  `local_results` maps position -> criterion, `local_payload` position -> (u, alpha) of this
    rank's candidates for the overall best.  Returns (criteria in sweep order, best position, (u, alpha) of the best) on every
    rank; the best is the reference's: the FIRST position whose criterion is strictly below everything before it."""
    rank, world = _world(group)
    gathered = [local_results]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, local_results, group=group)
    merged = {}
    for g in gathered:
        merged.update(g)
    values = [merged[p] for p in range(n_values)]
    best, best_pos = float("inf"), None
    for p, v in enumerate(values):
        if v < best:
            best, best_pos = v, p
    payload = local_payload.get(best_pos)
    if world > 1 and best_pos is not None:
        box = [payload if best_pos % world == rank else None]
        dist.broadcast_object_list(box, src=dist.get_global_rank(group, best_pos % world) if group is not None else best_pos % world, group=group)
        payload = box[0]
    return values, best_pos, payload


def compute_bic(cost, n_u, n_cpg, n_ct, n_samples):
    """ic.py:11-15 (the product form is the reference's, SURVEY Q10)."""
    l = n_samples * n_cpg
    k = n_u * n_cpg + (n_ct + n_u - 1) * n_samples
    return 2 * np.log(cost) * k * np.log(l) + (k * np.log(l) * (k + 1)) / (l - k - 1)


def compute_aic(cost, n_u, n_cpg, n_ct, n_samples):
    """ic.py:18-22."""
    l = n_samples * n_cpg
    k = n_u * n_cpg + (n_ct + n_u - 1) * n_samples
    return l * np.log(cost / l) + 2 * k + (2 * k * (k + 1)) / (l - k - 1)


def compute_consensus_matrix(alpha_runs):
    """ic.py:24-37: fraction of the runs in which two samples share their dominant cell type (argmax of the alpha column) - one
    kernel pair of the library (dmf_consensus) on the stacked runs."""
    import ctypes as C
    import torch
    from .engine import _stream_ptr, to_device
    stack = to_device(np.ascontiguousarray(np.stack([np.asarray(a, dtype=np.float64) for a in alpha_runs])), torch.float64)
    n_runs, kt, n = stack.shape
    labels = torch.empty((n_runs, n), dtype=torch.int32, device=stack.device)
    out = torch.empty((n, n), dtype=torch.float64, device=stack.device)
    _lib.check(_lib.lib().dmf_consensus(C.c_void_p(stack.data_ptr()), n_runs, kt, n, C.c_void_p(labels.data_ptr()),
                                        C.c_void_p(out.data_ptr()), _stream_ptr()))
    return out.cpu().numpy()


def compute_ccc(alpha_runs):
    """ic.py:40-45."""
    from scipy.cluster.hierarchy import linkage, cophenet
    from scipy.spatial.distance import pdist
    distance = pdist(compute_consensus_matrix(alpha_runs), metric="euclidean")
    ccc, _ = cophenet(linkage(distance, method="average"), distance)
    return ccc


def run_deconvolution(meth_f, counts, ref, n_u, init_option, seed, iter1, iter2, tol):
    """ic.py:47-55."""
    if ref is not None:
        u, R, alpha = init_BSSMF_md(init_option, meth_f, counts, ref, n_u, seed=seed)
        u, alpha = mdwbssmf_deconv(u, R, alpha, meth_f, counts, ref, n_u, n_iter1=iter1, n_iter2=iter2, tol=tol)
        R = np.hstack((ref, u.reshape(-1, n_u)))
    else:
        u, alpha = unsupervised_deconv(meth_f, n_u, counts, init_option, n_iter1=iter1, n_iter2=iter2, tol=tol, seed=seed)
        R = u
    return u, R, alpha


def _batched_fits(prob_list, ref, n_u, inits, iter1, iter2, tol):
    """Fits sharing one shape -> [(u, R, alpha, cost)]; partial-reference only (ref is not None)."""
    batch = FitBatch(prob_list, n_u, [i[0] for i in inits], [i[1] for i in inits], mode=_lib.DMF_MODE_PARTIAL)
    res = batch.results(batch.fit(iter1, iter2, tol))
    batch.close()
    return [(u, np.hstack((ref, u.reshape(-1, n_u))), a, c) for (u, a, _n, c) in res]


def bicross_validation(meth_f, n_u, counts, iter1, iter2, tol, n_folds=10, seed=None, ref=None, init_option="uniform_", fraction=0.3,
                       base=None):
    """ic.py:58-89.  The fold masks come from numpy's GLOBAL stream, which every fold's init re-seeds (SURVEY Q11):
    the same numpy calls are issued in the same order, then all folds are fitted as one batch."""
    np.random.seed(seed)
    total_press, best_u, best_alpha, min_error = 0, None, None, float("inf")
    meth_f = np.asarray(meth_f)
    counts = np.asarray(counts)
    folds = []
    for _ in range(n_folds):
        train_mask = np.random.rand(*meth_f.shape) < fraction
        test_mask = ~train_mask
        if np.sum(test_mask) == 0 or np.sum(train_mask) == 0:
            continue
        if ref is not None:
            u0, _, a0 = init_BSSMF_md(init_option, meth_f * train_mask, counts * train_mask, ref, n_u, seed=seed)
            folds.append((train_mask, test_mask, u0, a0))
        else:      # the reference-free solver draws its own init from the same re-seeded stream
            u, alpha = unsupervised_deconv(meth_f * train_mask, n_u, counts * train_mask, init_option, n_iter1=iter1, n_iter2=iter2,
                                           tol=tol, seed=seed)
            folds.append((train_mask, test_mask, u, alpha))
    if ref is not None and folds:
        base = base if base is not None else DeviceProblem(meth_f, counts, ref)
        probs = [base.masked(f[0]) for f in folds]
        fits = _batched_fits(probs, np.asarray(ref), n_u, [(f[2], f[3]) for f in folds], iter1, iter2, tol)
    else:
        fits = [(f[2], f[2], f[3], None) for f in folds]
    for (train_mask, test_mask, _u0, _a0), (u, R, alpha, _c) in zip(folds, fits):
        # ||(X - R alpha) o test_mask||_F^2 == weighted cost with 0/1 weights: one more streaming pass
        test_error = cost_f_w(meth_f, R, alpha, test_mask.astype(np.float64)) / np.sum(test_mask)
        total_press += test_error
        if test_error < min_error:
            min_error, best_u, best_alpha = test_error, u, alpha
    return total_press, best_u, best_alpha       # the reference returns total, not mean (Q15)


def sweep_member_supported(K, n_u):
    """The library pads the known and the unknown block to even widths and needs their sum <= 32 (include/demethify_b200.h)."""
    return n_u >= 0 and (K + (K & 1)) + (n_u + (n_u & 1)) <= 32


def _sharded_initial_iterate(X_loc, D_loc, R_loc, M, K, N, lo, hi, n_u, init_option, seed, group, init_backend, rng=None):
    """init_BSSMF_md on the rows [lo, hi) of an M x N problem whose rows are sharded over `group` -> (u_local, alpha).  `uniform_` /
    `beta` draw from `rng`, by default RandomState(seed) (== the reference's set_seed(seed) + global stream: int -> init_genrand,
    list -> init_by_array, Q1); `uniform` / `SVD` re-seed the global stream and all-reduce their row sums (sharded.ShardedInit) on
    `init_backend(X_loc, D_loc, R_loc)`."""
    from .sharded import GpuInitBackend, init_BSSMF_md_sharded
    if init_option in ("uniform_", "beta"):
        return _initial_iterate("partial", init_option, M, N, K, n_u, rows=(lo, hi), rng=np.random.RandomState(seed) if rng is None else rng)
    if init_option in ("uniform", "SVD"):
        return init_BSSMF_md_sharded(init_option, None, None, None, n_u, seed=seed, group=group,
                                     backend=(init_backend or GpuInitBackend)(X_loc, D_loc, R_loc))
    raise NotImplementedError("row-sharded sweeps: --init uniform_, beta, uniform or SVD")


def _gpu_fit_backend(problems, n_u, U0s, A0s):
    """The sharded fits of one member as one batch: `problems` holds one (X, d_x, R_trunc) of this rank's rows per fit, or one
    that all fits share; X may be a resident DeviceProblem."""
    from .sharded import GpuShardBackend
    probs = [p[0] if isinstance(p[0], DeviceProblem) else DeviceProblem(*p) for p in problems]
    return GpuShardBackend(probs, None, None, n_u, [np.asarray(u).reshape(-1, n_u) for u in U0s], [np.asarray(a) for a in A0s])


def _sum_over_ranks(values, group):
    """Sum of the float64 `values` over the ranks of `group` (one all-reduce) -> ndarray."""
    import torch
    t = torch.tensor(np.asarray(values, dtype=np.float64))
    if _world(group)[1] > 1:
        if dist.get_backend(group) == "nccl":
            t = t.cuda()
        dist.all_reduce(t, group=group)
    return t.cpu().numpy()


def _row_sharded_member(prob_local, lo, hi, M, K, N, n_u, init_option, seed, iter1, iter2, tol, group):
    """One sweep member with the CpG rows sharded over the ranks of `group` (BASELINE config 5): every rank draws the same
    initial iterate from the same seed, keeps its rows of u and runs the row-sharded solver -> (u_local, alpha, cost)."""
    from .sharded import mdwbssmf_deconv_sharded
    u0, a0 = _sharded_initial_iterate(prob_local, None, None, M, K, N, lo, hi, n_u, init_option, seed, group, None)
    u_loc, alpha, _n, cost = mdwbssmf_deconv_sharded(u0, a0, prob_local, None, None, n_u, n_iter1=iter1, n_iter2=iter2, tol=tol,
                                                     group=group)
    return u_loc, alpha, cost


def consensus_runs_sharded(X_loc, D_loc, R_loc, M, lo, hi, n_u, init_option, seeds, iter1, iter2, tol, group=None, init_backend=None,
                           fit_backend=None):
    """The restarts of a CCC member (ic.py:195-200) with the CpG rows [lo, hi) of this rank: one initial iterate per seed by the
    rules of the row-sharded sweep, then all restarts as ONE row-sharded batch (one all-reduce per step covers every restart) ->
    (alpha of every restart, u_local and alpha of the last restart).  `init_backend(X, d_x, R)` (sharded.GpuInitBackend) and
    `fit_backend(problems, n_u, U0s, A0s)` (a GpuShardBackend batch) do this rank's arithmetic; X_loc may be a resident
    DeviceProblem of the rows (then D_loc and R_loc are None)."""
    from .sharded import fit_row_sharded
    K, N = (X_loc.K, X_loc.N) if isinstance(X_loc, DeviceProblem) else (np.shape(R_loc)[1], np.shape(X_loc)[1])
    inits = [_sharded_initial_iterate(X_loc, D_loc, R_loc, M, K, N, lo, hi, n_u, init_option, s, group, init_backend) for s in seeds]
    fits = fit_row_sharded((fit_backend or _gpu_fit_backend)([(X_loc, D_loc, R_loc)], n_u, [i[0] for i in inits], [i[1] for i in inits]),
                           iter1, iter2, tol, group)
    return [f[1] for f in fits], fits[-1][0], fits[-1][1]


def _state_key(state):
    return (np.asarray(state[1], dtype=np.uint32).tobytes(), int(state[2]), int(state[3]), float(state[4]))


def bicross_validation_sharded(X_loc, D_loc, R_loc, M, lo, hi, n_u, init_option, seed, n_folds, iter1, iter2, tol, fraction=0.3, group=None,
                               init_backend=None, fit_backend=None, cost=None):
    """bicross_validation (ic.py:58-89) with a reference matrix and the CpG rows [lo, hi) of an M x N problem on this rank ->
    (total PRESS, u_local and alpha of the best fold, test error of every fold (None where the reference skips it)).

    Every fold draws its mask from numpy's global stream and then re-seeds it in its init, so a fold's mask starts either where the
    seeding put the stream (the first fold), or after the init's draws (every later fold), or 2 M N words after a skipped fold's
    mask (a mask with no train or no test entry over all rows, :119-120).  The planner replays those stream positions: each rank
    draws only its rows of each distinct mask (mt_jump.mask_rows), the train counts are all-reduced for the skip test, and a fold
    whose start state was seen before repeats that fold.  Only the distinct folds are fitted - at most two when no fold is skipped
    - as one row-sharded batch of masked problems, each from its own initial iterate.  The test error ||(X - R alpha) o test||^2
    is summed over the ranks and divided by the global test count; errors add to the total in fold order, the best fold is the
    first strict minimum, and the global stream is left where the reference leaves it.  `init_backend` and `fit_backend` as in
    consensus_runs_sharded; `cost(X, R, alpha, W)` is cost_f_w on this rank's rows."""
    from .deconvolution import set_seed
    from .mt_jump import mask_rows
    from .sharded import fit_row_sharded
    if seed is None and _world(group)[1] > 1:
        raise ValueError("row-sharded bicross-validation needs a seed: every rank draws its rows of the same fold masks")
    K, N = np.shape(R_loc)[1], np.shape(X_loc)[1]
    X_loc, D_loc, R_loc = (np.asarray(a, dtype=np.float64) for a in (X_loc, D_loc, R_loc))
    set_seed(seed)
    state, after_init = np.random.get_state(), None
    masks, distinct, order = {}, [], []          # start state -> (train rows, global train count, state after the mask); fitted folds
    for _ in range(n_folds):
        key = _state_key(state)
        if key not in masks:
            train, end = mask_rows(state, M, N, lo, hi, fraction)
            masks[key] = (train, _sum_over_ranks([train.sum()], group)[0], end)
        train, n_train, end = masks[key]
        if n_train == 0 or n_train == M * N:         # no train or no test entry: the reference skips the fold without re-seeding
            order.append(None)
            state = end
            continue
        hit = [i for i, d in enumerate(distinct) if d["key"] == key]
        if not hit:
            Xm, Dm = X_loc * train, D_loc * train
            set_seed(seed)                            # the fold's init (:75) re-seeds the global stream and draws from it
            u0, a0 = _sharded_initial_iterate(Xm, Dm, R_loc, M, K, N, lo, hi, n_u, init_option, seed, group, init_backend, rng=np.random)
            after_init = np.random.get_state()
            distinct.append(dict(key=key, test=~train, n_test=M * N - n_train, prob=(Xm, Dm, R_loc), u0=u0, a0=a0))
            hit = [len(distinct) - 1]
        order.append(hit[0])
        state = after_init
    np.random.set_state(state)
    if not distinct:
        return 0, None, None, order
    fits = fit_row_sharded((fit_backend or _gpu_fit_backend)([d["prob"] for d in distinct], n_u, [d["u0"] for d in distinct],
                                                             [d["a0"] for d in distinct]), iter1, iter2, tol, group)
    cost = cost or cost_f_w
    sse = _sum_over_ranks([cost(X_loc, np.hstack((R_loc, u.reshape(-1, n_u))), a, d["test"].astype(np.float64))
                           for d, (u, a, _n, _c) in zip(distinct, fits)], group)
    errors = [None if i is None else sse[i] / distinct[i]["n_test"] for i in order]
    total_press, best, min_error = 0, None, float("inf")
    for i, e in zip(order, errors):
        if i is not None:
            total_press += e
            if e < min_error:
                min_error, best = e, i
    return total_press, fits[best][0], fits[best][1], errors


def evaluate_best_ic(meth_f, ref, counts, init_option, ic, seed, iter1, iter2, tol, n_restarts=5, n_u_values=None, shard="fits",
                     group=None):
    """ic.py:169-218.  n_u_values defaults to the reference's hard-coded range(1, 26) (Q9); 0 may be listed explicitly (AIC / BIC):
    it is the reference-based fit of demethify.py:209-213 (the reference's own loop breaks at 0, SURVEY Q9).

    X, d_x and R_trunc are uploaded ONCE and stay resident in HBM for the whole sweep; the criterion of a member comes from the
    cost the solver finished with (the reference recomputes the same number with cost_f_w, ic.py:206).  Members whose shape the
    library cannot run (known + unknown types, each padded to even, > 32) are reported up front, skipped and recorded as inf.

    Under torch.distributed: shard="fits" (default) gives position p of the sweep to rank p mod world (every member re-seeds and
    is independent); shard="rows" runs EVERY member with the CpG rows sharded over the ranks (one all-reduce per outer
    iteration, sharded.py) - the partitioning for matrices that are large per member (every criterion with a reference matrix;
    every init but ICA, and the reference-based member n_u = 0).  A CCC member's restarts and a BCV member's distinct folds are
    then one row-sharded batch (consensus_runs_sharded, bicross_validation_sharded)."""
    n_u_values = range(1, 25 + 1) if n_u_values is None else n_u_values
    meth_f = np.asarray(meth_f)
    n_cpg, n_samples = meth_f.shape
    n_ct = ref.shape[1] if ref is not None else 0
    best_n_u, best_u_overall, best_alpha_overall = None, None, None
    if ic == "minka":
        # the reference raises here: run_deconvolution() is called with three arguments missing (ic.py:189, Q7)
        raise TypeError("run_deconvolution() missing 3 required positional arguments: 'iter1', 'iter2', and 'tol'")
    if isinstance(seed, (list, tuple)) and ic == "CCC":
        raise TypeError("can only concatenate list (not \"int\") to list")      # ic.py:196 with `--seed S` (Q1)
    n_u_values = list(n_u_values)
    unsupported = [n for n in n_u_values if not sweep_member_supported(n_ct, n)]
    if unsupported:
        import warnings
        warnings.warn(f"n_u = {unsupported} with {n_ct} known cell types exceed the library limit (known + unknown types, each padded "
                      "to even, <= 32): these members are skipped and recorded as inf", RuntimeWarning, stacklevel=2)
    if 0 in n_u_values and (ic not in ("AIC", "BIC") or ref is None):
        raise ValueError("n_u = 0 (reference-based fit) is available for AIC / BIC with a reference matrix only")
    rank, world = _world(group)
    rows_mode = shard == "rows" and world > 1
    if rows_mode and ref is None:
        raise NotImplementedError("row-sharded sweeps need a reference matrix")
    if rows_mode:
        from .sharded import row_range
        lo, hi = row_range(n_cpg, rank, world)
        prob = DeviceProblem(meth_f[lo:hi], np.asarray(counts)[lo:hi], np.asarray(ref)[lo:hi])
    else:
        lo, hi = 0, n_cpg
        prob = DeviceProblem(meth_f, counts, ref)                       # resident for the whole sweep
    src = prob if init_option in ("uniform_", "uniform", "beta") else meth_f      # the SVD init reads the host matrix
    local_results, local_payload, local_best = {}, {}, float("inf")
    positions = list(range(len(n_u_values))) if rows_mode else list(range(len(n_u_values)))[rank::world]
    for pos in tqdm.tqdm(positions, disable=rank != 0):
        n_u = n_u_values[pos]
        if n_u in unsupported:
            local_results[pos] = float("inf")
            continue
        if n_u == 0:
            from .init_func import wls_all_samples
            if rows_mode:
                from .sharded import wls_all_samples_sharded
                alpha = wls_all_samples_sharded(prob, None, None, y_is_dx=True, group=group)
                u = np.zeros((hi - lo, 0))
                import torch
                cost_t = torch.tensor([cost_f_w(meth_f[lo:hi], np.asarray(ref)[lo:hi], alpha, np.asarray(counts)[lo:hi])],
                                      dtype=torch.float64, device=prob.device)
                dist.all_reduce(cost_t, group=group)                          # the cost over all rows
                cost = float(cost_t.item())
            else:
                alpha = wls_all_samples(prob, None, None, y_is_dx=True)          # demethify.py:209-213
                u = np.zeros((n_cpg, 0))
                cost = cost_f_w(meth_f, np.asarray(ref), alpha, counts)
            ic_result = compute_bic(cost, 0, n_cpg, n_ct, n_samples) if ic == "BIC" else compute_aic(cost, 0, n_cpg, n_ct, n_samples)
        elif ic == "CCC":
            if rows_mode:
                alpha_runs, u, alpha = consensus_runs_sharded(prob, None, None, n_cpg, lo, hi, n_u, init_option,
                                                              [seed + r for r in range(n_restarts)], iter1, iter2, tol, group)
            elif ref is not None:
                inits = [init_BSSMF_md(init_option, src, counts, ref, n_u, seed=seed + r) for r in range(n_restarts)]
                fits = _batched_fits(prob, np.asarray(ref), n_u, [(i[0], i[2]) for i in inits], iter1, iter2, tol)
                alpha_runs = [f[2] for f in fits]
                u, alpha = fits[-1][0], fits[-1][2]
            else:
                alpha_runs = []
                for r in range(n_restarts):
                    u, alpha = unsupervised_deconv(src, n_u, counts, init_option, n_iter1=iter1, n_iter2=iter2, tol=tol, seed=seed + r)
                    alpha_runs.append(alpha)
            ic_result = -compute_ccc(alpha_runs)
        elif ic == "BCV" and rows_mode:
            ic_result, u, alpha, _errors = bicross_validation_sharded(meth_f[lo:hi], np.asarray(counts)[lo:hi], np.asarray(ref)[lo:hi],
                                                                      n_cpg, lo, hi, n_u, init_option, seed, n_restarts, iter1, iter2, tol,
                                                                      group=group)
        elif ic == "BCV":
            ic_result, u, alpha = bicross_validation(meth_f, n_u, counts, iter1, iter2, tol, fraction=0.3, n_folds=n_restarts, seed=seed,
                                                     ref=ref, init_option=init_option, base=prob)
        else:
            if rows_mode:
                u, alpha, cost = _row_sharded_member(prob, lo, hi, n_cpg, n_ct, n_samples, n_u, init_option, seed, iter1, iter2, tol, group)
            elif ref is not None:
                u0, R0, a0 = init_BSSMF_md(init_option, src, counts, ref, n_u, seed=seed)
                u, alpha = mdwbssmf_deconv(u0, R0, a0, prob, None, None, n_u, n_iter1=iter1, n_iter2=iter2, tol=tol)
                cost = last_fit_info()["cost"]
            else:
                u, alpha = unsupervised_deconv(src, n_u, counts, init_option, n_iter1=iter1, n_iter2=iter2, tol=tol, seed=seed)
                cost = last_fit_info()["cost"]
            ic_result = compute_bic(cost, n_u, n_cpg, n_ct, n_samples) if ic == "BIC" else compute_aic(cost, n_u, n_cpg, n_ct, n_samples)
        local_results[pos] = ic_result
        if ic_result < local_best:                 # the overall best (first position of the minimum) is the LAST strict improvement
            local_best = ic_result                 # inside its rank's share: keep only that one
            local_payload = {pos: (u, alpha)}
    if rows_mode:
        # every rank evaluated every member on its rows: criteria are replicated, u of the winner is gathered row range by row range
        values = [local_results[p] for p in range(len(n_u_values))]
        best_pos = min(local_payload) if local_payload else None
        payload = None
        if best_pos is not None:
            u_loc, alpha = local_payload[best_pos]
            parts = [None] * world
            dist.all_gather_object(parts, np.asarray(u_loc), group=group)
            payload = (np.concatenate(parts, axis=0), alpha)
        list_result = values
    else:
        list_result, best_pos, payload = merge_sweep(local_results, local_payload, len(n_u_values), group)
    if best_pos is not None:
        best_n_u, (best_u_overall, best_alpha_overall) = n_u_values[best_pos], payload
    return best_u_overall, best_alpha_overall, best_n_u, list_result
