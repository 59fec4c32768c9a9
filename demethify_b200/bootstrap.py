"""Mirror of the reference's demethify/bootstrap.py: bootstrap confidence intervals.

The reference fits the resamples one after another (bootstrap.py:26-46); here all resamples of a wave are ONE
batched launch set that shares X, d_x, R_trunc in HBM.  Where the library supports it the resamples run in
MULTIPLICITY FORM: a resample is the source matrix with per-row multiplicities, its u rows (one per resampled position,
the reference's per-position semantics, SURVEY Q6) are ordered by source row and addressed through a CSR, so the
streaming passes read the shared matrices contiguously and, with a fit-major grid, mostly out of L2.  Otherwise
(K > 6, n_u > 4) every fit carries a row index and the kernels gather rows.  Seeds, resampling indices, init draws and
the percentile arithmetic follow the reference exactly (SURVEY Q3-Q6): seed_i = seed_{i-1} + i,
sklearn.utils.resample == RandomState(seed).randint.
"""
import os

import numpy as np
import pandas as pd
import torch
import torch.distributed as dist

from . import _lib
from .deconvolution import _init_option, _initial_iterate, _quiet, _zero_guard, init_BSSMF_md, init_BSSMF_md_p
from .engine import DeviceProblem, FitBatch, device_free_bytes
from .init_func import wls_all_samples

__all__ = ["bt_ci", "bootstrap_seeds", "resample_indices", "resample_layout", "bootstrap_fits", "shard_of", "merge_resample_stacks",
           "percentile_bounds_device"]


def _world(group):
    return (dist.get_rank(group), dist.get_world_size(group)) if dist.is_available() and dist.is_initialized() else (0, 1)


def shard_of(items, rank, world):
    """Fit sharding (SURVEY 8 e1 (i)): resample b runs on rank b mod world — the resamples are independent (bootstrap.py:26)."""
    return list(items[rank::world])


def merge_resample_stacks(local, n_total, group=None):
    """All-gather the per-rank stacks (B_r, ...) of a fit-sharded bootstrap into the full (n_total, ...) stack on every rank.
    The order along the fit axis is rank-major; the percentiles of bt_ci do not depend on it."""
    rank, world = _world(group)
    if world == 1:
        return local
    counts = [len(range(r, n_total, world)) for r in range(world)]
    bmax = max(counts)
    pad = torch.zeros((bmax,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[:local.shape[0]] = local
    out = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(out, pad, group=group)
    return torch.cat([out[r][:counts[r]] for r in range(world)], dim=0)


def bootstrap_seeds(seed, n_bootstrap):
    """bootstrap.py:27 — the seed accumulates: seed, seed+1, seed+3, seed+6, ..."""
    if isinstance(seed, (list, tuple, np.ndarray)):
        # `--seed S` reaches bt_ci as [S] in the reference and `seed + i` raises TypeError (SURVEY Q1)
        raise TypeError("can only concatenate list (not \"int\") to list")
    out, s = [], seed
    for i in range(n_bootstrap):
        s = s + i if s is not None else None
        out.append(s)
    return out


def resample_indices(seed, M):
    """sklearn.utils.resample(X, counts, ref, random_state=seed) (bootstrap.py:28) draws
    RandomState(seed).randint(0, M, size=(M,)) once and indexes every array with it."""
    return np.random.RandomState(seed).randint(0, M, size=(M,))


def _shape_only_init(seed, init_option, M, K, N, n_u, with_zero_guard):
    """uniform_ / beta inits (deconvolution.py:54-61, :246-253) from a PRIVATE legacy stream: RandomState(seed) produces
    exactly what the reference's set_seed(seed) + global numpy.random calls produce, and is safe to use from worker threads."""
    return _initial_iterate("partial" if with_zero_guard else "purity", init_option, M, N, K, n_u, rng=np.random.RandomState(seed),
                            say=_quiet)


def device_draws(chunk, M, n_u, K, N, dev, with_zero_guard):
    """The draws of one wave of (resample seed, init seed) jobs with the `uniform_` init, on the device (dmf_rng_legacy_streams):
    idx (B, M) int32 = RandomState(resample seed).randint(0, M, M) (bootstrap.py:28), u0 (B, M, n_u) = the first M n_u uniforms of
    RandomState(init seed) (deconvolution.py:54-55); alpha_0 (B, Kt, N) numpy: the dirichlet draw that follows in the same stream,
    taken by numpy itself from the generator state the kernel hands back (Kt N values; its -log(1 - U) must round like glibc's)."""
    import ctypes as C
    from .engine import _stream_ptr
    lib = _lib.lib()
    B = len(chunk)
    row_seeds = sorted({j[0] for j in chunk})
    pos = {sd: i for i, sd in enumerate(row_seeds)}
    sr = torch.from_numpy(np.array(row_seeds, dtype=np.uint32).view(np.int32)).to(dev)        # (uint32 bits in an int32 tensor)
    idx_u = torch.empty((len(row_seeds), M), dtype=torch.int32, device=dev)
    _lib.check(lib.dmf_rng_legacy_streams(C.c_void_p(sr.data_ptr()), len(row_seeds), M, C.c_void_p(idx_u.data_ptr()), M, 0, None, 0, None,
                                          _stream_ptr()))
    idx_d = idx_u if len(row_seeds) == B else idx_u[torch.tensor([pos[j[0]] for j in chunk], device=dev)]
    si = torch.from_numpy(np.array([j[1] for j in chunk], dtype=np.uint32).view(np.int32)).to(dev)
    u0_d = torch.empty((B, M, n_u), dtype=torch.float64, device=dev)
    state = torch.empty((B, 625), dtype=torch.int32, device=dev)
    _lib.check(lib.dmf_rng_legacy_streams(C.c_void_p(si.data_ptr()), B, 0, None, 0, M * n_u, C.c_void_p(u0_d.data_ptr()), M * n_u,
                                          C.c_void_p(state.data_ptr()), _stream_ptr()))
    st = state.cpu().numpy().view(np.uint32)
    A0 = np.empty((B, K + n_u, N))
    rs = np.random.RandomState(0)
    for k in range(B):
        rs.set_state(("MT19937", st[k, :624], int(st[k, 624]), 0, 0.0))
        alpha = rs.dirichlet(np.ones(K + n_u), N).T
        A0[k] = _zero_guard(alpha, n_u) if with_zero_guard else alpha      # init_BSSMF_md only
    return idx_d, u0_d, A0


def percentile_bounds_device(stack, lower_percentile, upper_percentile):
    """np.percentile(stack, [lo, hi], axis=0) (bootstrap.py:53-54, :77-78; default linear interpolation) on the device, by the
    library's selection kernel (dmf_percentile_bounds: one thread per entry keeps the few smallest / largest of the B values, no
    sort of the B x P stack).  Confidence levels so low that more than dmf_percentile_max_keep() order statistics per tail are
    needed fall back to torch.quantile (same linear rule)."""
    import ctypes as C
    from .engine import _stream_ptr
    lib = _lib.lib()
    B = stack.shape[0]
    flat = stack.reshape(B, -1).to(torch.float64).contiguous()          # (host tensors - the gloo tests - take the torch.quantile branch)
    P = flat.shape[1]
    out = torch.empty((2, P), dtype=torch.float64, device=stack.device)
    klo, khi = int(np.floor((B - 1) * (lower_percentile / 100.0))), int(np.floor((B - 1) * (upper_percentile / 100.0)))
    if stack.is_cuda and max(min(klo + 2, B), min(B - khi, B)) <= lib.dmf_percentile_max_keep():
        _lib.check(lib.dmf_percentile_bounds(C.c_void_p(flat.data_ptr()), B, P, float(lower_percentile), float(upper_percentile),
                                             C.c_void_p(out[0].data_ptr()), C.c_void_p(out[1].data_ptr()), _stream_ptr()))
    else:
        q = torch.tensor([lower_percentile / 100.0, upper_percentile / 100.0], dtype=torch.float64, device=stack.device)
        step = max(1, (1 << 24) // max(B, 1))          # torch.quantile caps the size of its input
        for c0 in range(0, P, step):
            out[:, c0:c0 + step] = torch.quantile(flat[:, c0:c0 + step], q, dim=0, interpolation="linear")
    shape = stack.shape[1:]
    return out[0].reshape(shape).cpu().numpy(), out[1].reshape(shape).cpu().numpy()


def resample_layout(idx, M, with_csr=True):
    """Stacked resample indices (B, M) (sklearn.utils.resample, bootstrap.py:28) -> the layout the library wants:
    order (B, M): stable argsort of every resample by source row (position p of the sorted resample was position order[p] of the
    reference's), rows (B, M) int32: the sorted source rows, and — multiplicity form — mult (B, M) int32: how often every source
    row was drawn (16-byte aligned rows), offs (B, M + 1) int32: CSR offsets of the positions of every source row."""
    B = idx.shape[0]
    order = torch.sort(idx, dim=1, stable=True).indices
    rows = torch.gather(idx, 1, order).to(torch.int32)
    if not with_csr:
        return order, rows, None, None
    Mp = (M + 3) // 4 * 4                             # the multiplicities are streamed with 16-byte bulk copies: aligned rows
    mult = torch.zeros((B, Mp), dtype=torch.int32, device=idx.device)[:, :M]
    mult.scatter_add_(1, idx, torch.ones_like(idx, dtype=torch.int32))
    offs = torch.zeros((B, M + 1), dtype=torch.int32, device=idx.device)
    offs[:, 1:] = torch.cumsum(mult, 1)
    return order, rows, mult, offs


def bootstrap_fits(n_bootstrap, n_u, meth_f, counts, ref, init_option, n_iter1, n_iter2, tol, purity, seed, prob=None,
                   keep_u=True, on_device=False, seeds=None, restarts=1):
    """All resample fits -> (alphas (B, Kt, N), us (B, M, n_u) or None, n_outer list).
    restarts = R > 1 (extension; BASELINE config 4, SURVEY Q5): every resample is fitted R times from the initial iterates of the
    seeds s, s + 1, ..., s + R - 1 (the convention of ic.py:196; the rows are those of seed s) in the same batch, and the fit with
    the lowest final cost is kept (the selection rule of demethify.py:199-203).
    `purity` is the internal vector (already divided by 100, bootstrap.py:18) or None.  With on_device the two stacks
    stay torch tensors in HBM (the percentiles of bt_ci are then taken there, SURVEY 8 f4).  `seeds` restricts the run to a
    sub-list of the reference's seed sequence (one rank's share of a fit-sharded bootstrap)."""
    meth_f = np.asarray(meth_f)
    M, N = meth_f.shape
    if n_u > 0:
        # the reference falls back to uniform_ when n_u > N (deconvolution.py:44-45, :234-239), then dispatches on the option;
        # anything it would run that this path does not have is refused BEFORE a resample is drawn (never silently replaced)
        init_option = _init_option("partial" if purity is None else "purity", init_option, n_u, N, say=_quiet)
    seeds = bootstrap_seeds(seed, n_bootstrap) if seeds is None else list(seeds)
    n_bootstrap = len(seeds)
    restarts = max(1, int(restarts))
    if restarts > 1 and n_u == 0:
        raise ValueError("restarts apply to the iterative fits (n_u >= 1)")
    prob = prob or DeviceProblem(meth_f, counts, ref)
    alphas = np.zeros((n_bootstrap, prob.K + n_u, N))
    if on_device and n_u > 0:
        need = n_bootstrap * (M * n_u + (prob.K + n_u) * N) * 8
        on_device = need < device_free_bytes(prob.device) // 3        # else fall back to host stacks
    if n_u == 0:
        for b, s in enumerate(seeds):          # bootstrap.py:40-43: per-sample NNLS on the resampled rows
            idx = resample_indices(s, M)
            alphas[b] = wls_all_samples(prob.gathered(idx), None, None, y_is_dx=True)
        return alphas, None, [0] * n_bootstrap
    if on_device:
        alphas = torch.zeros((n_bootstrap, prob.K + n_u, N), dtype=torch.float64, device=prob.device)
        us = torch.zeros((n_bootstrap, M, n_u), dtype=torch.float64, device=prob.device) if keep_u else None
    else:
        us = np.zeros((n_bootstrap, M, n_u)) if keep_u else None
    n_outer = []
    data_dependent_init = init_option in ("uniform", "SVD")
    # fits per wave: bounded by device memory (two u slots + partials per fit)
    ng = {1: 2, 2: 5}.get(n_u, 14)                            # Gram engine: per-row statistics, one record per warp of a row
    ntc = 1 << max(0, ((N + 3) // 4 - 1).bit_length())
    per_fit = (2 * M * (n_u + (n_u & 1)) * (8 if prob.precision == "fp64" else 4) + M * ng * ((ntc + 31) // 32) * 8 * (n_u <= 4)
               + 64 * (prob.K + n_u) * N * 8 + 4096
               + M * (44 + 24 * n_u))                          # wave-level stacks: resample index, order, rows, mult, offs, u0 / results
    wave = int(max(1, min(n_bootstrap * restarts, (device_free_bytes(prob.device) // 2) // max(per_fit, 1), 4096)))
    wave = max(restarts, wave // restarts * restarts)           # the restarts of a resample stay in one wave
    jobs = [(s, s + r) for s in seeds for r in range(restarts)]  # (resample seed, init seed)
    mode = _lib.DMF_MODE_PURITY if purity is not None else _lib.DMF_MODE_PARTIAL
    use_mult = prob.K <= 6 and n_u <= 4 and prob.K + (prob.K & 1) + n_u + (n_u & 1) <= 8
    dev = prob.device
    # MATERIALISED form: where the fused one-pass engine applies (FP64, n_u <= 2, K <= 8, N <= 256, n_iter2 <= 64) every resample of
    # a wave gets its own gathered copy of X, d_x, R_trunc (one row-gather kernel per matrix) and runs the same single streaming pass
    # per outer iteration as a plain fit: half the FP64 work per outer iteration of the two-pass multiplicity form, positions stay in
    # the reference's order (no sort / CSR), at the price of HBM traffic instead of L2 hits and of gigabytes of scratch per wave.
    from . import get_engine
    use_fused = (get_engine() in ("auto", "fused") and prob.precision == "fp64" and n_u <= 2 and prob.K <= 8 and N <= 256 and 1 <= n_iter2 <= 64
                 and M >= 4096)
    if use_fused:
        row_bytes = prob.X.shape[1] * prob.X.element_size() + prob.D.shape[1] * prob.D.element_size() + \
            (prob.Rk.shape[1] * prob.Rk.element_size() if prob.Rk is not None else 0)
        per_fit = M * (row_bytes + 4 * (n_u + (n_u & 1)) * 8 + 8 + 8 * n_u * 3) + 64 * (prob.K + n_u) * N * 8 + (1 << 20)
        wave = int(max(1, min(n_bootstrap * restarts, (device_free_bytes(prob.device) * 2 // 3) // max(per_fit, 1), 1024)))
        wave = max(restarts, wave // restarts * restarts)
    device_rng = (init_option == "uniform_" and prob.X.is_cuda and all(isinstance(t, (int, np.integer)) and 0 <= t < 2 ** 32 for j in jobs for t in j)
                  and os.environ.get("DMF_HOST_RNG") != "1")
    for w0 in range(0, len(jobs), wave):
        chunk = jobs[w0:w0 + wave]

        Bw = len(chunk)
        if device_rng:
            # SURVEY 8 f2: the two large draws of every resample come from the library's MT19937 kernel (bit-identical to numpy's
            # legacy streams); the host only continues each stream for the Kt x N dirichlet draw of alpha_0
            idx_d, u0_d, A0 = device_draws(chunk, M, n_u, prob.K, N, dev, with_zero_guard=purity is None)
        else:
            # host staging for the wave: the worker threads draw straight into it, one H2D copy per array (pageable on purpose:
            # page-locking gigabytes per wave costs more than the copy saves)
            idx_np = np.empty((Bw, M), dtype=np.int64)
            u0_np = np.empty((Bw, M, n_u), dtype=np.float64)
            A0 = np.empty((Bw, prob.K + n_u, N))

            def prepare(k):
                s_rows, s = chunk[k]
                idx = resample_indices(s_rows, M)
                if data_dependent_init:      # `uniform` / SVD look at the resampled data and use the global stream: sequential
                    Xb, Db, Rb = meth_f[idx], np.asarray(counts)[idx], np.asarray(ref)[idx]
                    if purity is not None:
                        u0, _, a0 = init_BSSMF_md_p(init_option, Xb, Db, Rb, n_u, purity, seed=s)
                    else:
                        u0, _, a0 = init_BSSMF_md(init_option, Xb, Db, Rb, n_u, seed=s)
                else:                        # uniform_ / beta draws depend on shapes only (deconvolution.py:54-61)
                    u0, a0 = _shape_only_init(s, init_option, M, prob.K, N, n_u, with_zero_guard=purity is None)
                idx_np[k], u0_np[k], A0[k] = idx, np.asarray(u0).reshape(M, n_u), a0
            if data_dependent_init:
                for k in range(Bw):
                    prepare(k)
            else:                            # numpy's legacy generators release the GIL: draw the resamples of the wave in parallel
                from concurrent.futures import ThreadPoolExecutor
                with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
                    list(ex.map(prepare, range(Bw)))
            # batched device ops: order the resampled positions of every fit by source row (stable sort); u is position-indexed, so it is
            # permuted along; multiplicities and CSR offsets per source row
            idx_d = torch.from_numpy(idx_np).to(dev)                                                    # (Bw, M) int64
            u0_d = torch.from_numpy(u0_np).to(dev)                                                      # (Bw, M, n_u)
        if use_fused:
            probs = prob.gathered_many(idx_d)                                                       # this wave's resampled matrices
            del idx_d
            batch = FitBatch(probs, n_u, u0_d, A0, mode=mode, purity=purity)
            del u0_d
            states = batch.fit(n_iter1, n_iter2, tol)
            U_d, A_d = batch.stacked_current(states)
            if restarts > 1:
                cost = torch.tensor([st.cost for st in states], dtype=torch.float64, device=dev).view(-1, restarts)
                best = torch.argmin(cost, dim=1) + torch.arange(cost.shape[0], device=dev) * restarts
                U_d, A_d = U_d[best], A_d[best]
                n_outer.extend(states[int(i)].n_outer for i in best.cpu())
            else:
                n_outer.extend(st.n_outer for st in states)
            b0, nb = w0 // restarts, Bw // restarts
            if on_device:
                alphas[b0:b0 + nb] = A_d.to(torch.float64)
                if keep_u:
                    us[b0:b0 + nb] = U_d.to(torch.float64)
            else:
                alphas[b0:b0 + nb] = A_d.to(torch.float64).cpu().numpy()
                if keep_u:
                    us[b0:b0 + nb] = U_d.to(torch.float64).cpu().numpy()
            batch.close()
            del batch, probs, U_d, A_d
            continue
        order_d, rows_d, cnt, offs_d = resample_layout(idx_d.long(), M, with_csr=use_mult)
        U0 = torch.gather(u0_d, 1, order_d.unsqueeze(-1).expand(-1, -1, n_u))
        del u0_d
        batch = None
        if use_mult:
            try:
                batch = FitBatch(prob, n_u, U0, A0, mode=mode, purity=purity, rows=rows_d, mult=cnt, offs=offs_d)
            except _lib.DmfError:                     # shape outside the multiplicity form (tile geometry): gather form from now on
                use_mult = False
        if batch is None:
            batch = FitBatch(prob, n_u, U0, A0, mode=mode, purity=purity, rows=rows_d)
        del idx_d
        states = batch.fit(n_iter1, n_iter2, tol)
        U_d, A_d = batch.stacked_current(states)
        if restarts > 1:                             # best of the R restarts of every resample: lowest final cost, first on ties
            cost = torch.tensor([st.cost for st in states], dtype=torch.float64, device=dev).view(-1, restarts)
            best = torch.argmin(cost, dim=1) + torch.arange(cost.shape[0], device=dev) * restarts
            U_d, A_d, order_d = U_d[best], A_d[best], order_d[best]
            n_outer.extend(states[int(i)].n_outer for i in best.cpu())
        else:
            n_outer.extend(st.n_outer for st in states)
        b0, nb = w0 // restarts, Bw // restarts
        if on_device:
            alphas[b0:b0 + nb] = A_d.to(torch.float64)
            if keep_u:                               # back to the resampled-position order of the reference (Q6)
                us[b0:b0 + nb].scatter_(1, order_d.unsqueeze(-1).expand(-1, -1, n_u), U_d.to(torch.float64))
        else:
            alphas[b0:b0 + nb] = A_d.to(torch.float64).cpu().numpy()
            if keep_u:
                back = torch.empty((nb, M, n_u), dtype=torch.float64, device=dev)
                back.scatter_(1, order_d.unsqueeze(-1).expand(-1, -1, n_u), U_d.to(torch.float64))
                us[b0:b0 + nb] = back.cpu().numpy()
        batch.close()
    return alphas, us, n_outer


def bt_ci(confidence_level, n_bootstrap, n_u, meth_f, counts, ref, init_option, n_iter1, n_iter2, tol, header, outdir, samples,
          purity, seed, restarts=1):
    """bootstrap.py:10-93 — same arguments, same two CSV files, same return value (list of DataFrames).  `restarts` (additive):
    see bootstrap_fits."""
    supervised = n_u == 0
    a = 1 - confidence_level / 100
    lower_percentile = 100 * (a / 2)
    upper_percentile = 100 * (1 - (a / 2))
    pur = None
    if purity:
        pur = np.array(purity) / 100.0                      # bootstrap.py:18 (NOT 1 - p/100, SURVEY Q4)
    rank, world = _world(None)
    if world > 1:
        # fit sharding over the GPUs of the job (one process per GPU; every rank calls bt_ci): rank r fits resamples r, r + world, ...,
        # the stacks are all-gathered over NCCL, every rank takes the percentiles, rank 0 writes the files
        mine = shard_of(bootstrap_seeds(seed, n_bootstrap), rank, world)
        alphas, us, _ = bootstrap_fits(len(mine), n_u, meth_f, counts, ref, init_option, n_iter1, n_iter2, tol, pur, seed, on_device=True,
                                       seeds=mine, restarts=restarts)
        if not isinstance(alphas, torch.Tensor):        # supervised path / host stacks: move to the device for the all-gather
            from .engine import current_device
            alphas = torch.from_numpy(np.ascontiguousarray(alphas)).to(current_device())
            us = torch.from_numpy(np.ascontiguousarray(us)).to(current_device()) if us is not None else None
        alphas = merge_resample_stacks(alphas, n_bootstrap)
        us = merge_resample_stacks(us, n_bootstrap) if us is not None else None
    else:
        alphas, us, _ = bootstrap_fits(n_bootstrap, n_u, meth_f, counts, ref, init_option, n_iter1, n_iter2, tol, pur, seed, on_device=True,
                                       restarts=restarts)
    if isinstance(alphas, torch.Tensor):
        lo, hi = percentile_bounds_device(alphas, lower_percentile, upper_percentile)
    else:
        lo = np.percentile(alphas, lower_percentile, axis=0)    # (Kt, N); bootstrap.py:53-54
        hi = np.percentile(alphas, upper_percentile, axis=0)
    results = []
    unknown_header = [] if supervised else ["unknown_cell_" + str(i + 1) for i in range(n_u)]
    cell_types = list(header) + unknown_header
    n_ct = np.asarray(ref).shape[1] + n_u
    cols = {}
    for i in range(np.asarray(meth_f).shape[1]):
        cols[f"Sample_{i + 1}"] = [(float(lo[k, i]), float(hi[k, i])) for k in range(n_ct)]
    proportions_df = pd.DataFrame(cols, index=cell_types)
    proportions_df.columns = samples
    proportions_df.index.name = "Cell Type"
    if rank == 0:
        proportions_df.to_csv(outdir + "/confidence_interval_celltypes_proportions.csv", index=True)
    results.append(proportions_df)
    if not supervised:
        if isinstance(us, torch.Tensor):
            ulo, uhi = percentile_bounds_device(us, lower_percentile, upper_percentile)
        else:
            ulo = np.percentile(us, lower_percentile, axis=0)   # (M, n_u); bootstrap.py:77-78
            uhi = np.percentile(us, upper_percentile, axis=0)
        ref_cols = {unknown_header[k]: [(float(ulo[j, k]), float(uhi[j, k])) for j in range(us.shape[1])] for k in range(n_u)}
        ref_estimate_df = pd.DataFrame(ref_cols)
        if rank == 0:
            ref_estimate_df.to_csv(outdir + "/confidence_interval_methylation_estimate.csv", index=False)
        results.append(ref_estimate_df)
    return results
