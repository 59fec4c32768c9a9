"""Drop-in mirror of the reference's demethify/deconvolution.py on top of the sm_100a kernel library.

Same function names, argument order, defaults and numpy-in / numpy-out contract as the reference
(file:line cited per function); the arithmetic of every solver step runs in libdemethify_sm100.so.
Initial draws use numpy's legacy MT19937 stream exactly as the reference does (set_seed -> numpy.random),
so that u0 / alpha0 are bit-identical for a given seed.
"""
import numpy as np
import numpy.random as rd
import torch

from . import _lib
from .engine import DeviceProblem, FitBatch, to_device
from .init_func import wls_intercept, wls_all_samples, nndsvd_initialize

__all__ = ["set_seed", "cost_f_w", "projection_simplex_sort_2d", "init_BSSMF_md", "init_BSSMF_md_p", "update_u", "update_alpha",
           "frank_wolfe_nmf", "mdwbssmf_deconv", "mdwbssmf_deconv_p", "unsupervised_deconv", "last_fit_info", "best_of_restarts"]

_last = {}


def last_fit_info():
    """{'n_outer', 'cost', 'launches'} of the most recent solver call (the reference exposes no such hook;
    needed for the identical-iteration-count parity check)."""
    return dict(_last)


def set_seed(seed=None):
    """deconvolution.py:9-11 — seeds numpy's global legacy stream (int -> init_genrand, list -> init_by_array)."""
    if seed is not None:
        rd.seed(seed)


def _split_r(R):
    """A full R (M x Kt) as the kernels take it, [R_trunc | u] -> (R_trunc or None, u, n_u, mode).  The library pads both blocks to
    even widths and needs their sum <= 32: the last TWO columns are "u" when Kt is even, the last one when it is odd (works up to
    Kt = 32).  For the cost and the alpha step, which see R only as a whole, any split is equivalent."""
    Kt = R.shape[1]
    nu = 2 if (Kt % 2 == 0 and Kt >= 2) else 1
    if Kt > nu:
        return R[:, :Kt - nu], R[:, Kt - nu:], nu, _lib.DMF_MODE_PARTIAL
    return None, R, nu, _lib.DMF_MODE_UNSUPERVISED


def cost_f_w(y, R, alpha, d_x):
    """deconvolution.py:15-17 — sum d_x * (y - R @ alpha)^2, one streaming pass on the GPU."""
    R = np.asarray(R)
    alpha = np.asarray(alpha)
    Rk, u, nu, mode = _split_r(R)
    prob = DeviceProblem(y, d_x, Rk)
    batch = FitBatch(prob, nu, [u], [alpha], mode=mode, engine="stream")
    batch.pass_init()
    cost = batch.states()[0].cost
    batch.close()
    return cost


def projection_simplex_sort_2d(v, z=1):
    """deconvolution.py:21-37 — column-wise Euclidean projection onto the simplex.  On the solver path this
    runs inside the alpha-step kernel; this standalone form (used only by the SVD init on a Kt x N matrix)
    is host-side glue."""
    v = np.asarray(v, dtype=np.float64)
    p, n = v.shape
    srt = -np.sort(-v, axis=0)
    pi = np.cumsum(srt, axis=0) - z
    ok = (srt - pi / np.arange(1, p + 1)[:, None]) > 0
    if not ok.any(axis=0).all():
        raise ZeroDivisionError("division by zero")
    rho = p - 1 - np.argmax(ok[::-1], axis=0)
    theta = pi[rho, np.arange(n)] / (rho + 1)
    return np.maximum(v - theta, 0)


def _quiet(message):
    pass


def _init_option(variant, init_option, n_u, N, say=print):
    """The option the reference dispatches on for `variant` ("partial", "purity" or "free", see _initial_iterate).  With more
    unknowns than samples the purity variant first falls back to `uniform` and says so (:232-234), then every variant falls back to
    `uniform_` (:44-45); an option this path does not run raises what the reference raises, or NotImplementedError."""
    if variant == "purity" and init_option != "uniform" and n_u > N:
        say("The number of unknowns is greater than the number of samples, we'll go with a uniform initialisation. ")
        init_option = "uniform"
    if init_option != "uniform_" and n_u > N:
        init_option = "uniform_"
    if variant == "free":
        if init_option == "uniform":
            raise NameError("name 'R_trunc' is not defined")   # what the reference does (deconvolution.py:117, SURVEY Q8)
        if init_option not in ("uniform_", "beta", "SVD"):
            raise NotImplementedError(f"init option {init_option!r} is not available on the B200 path")
    elif init_option == "ICA":
        raise NotImplementedError("--init ICA forms an M x M covariance (init_func.py:120) and is out of scope of the "
                                  "B200 path (SURVEY.md 2.1 row 4); use uniform_, uniform, beta or SVD")
    elif init_option not in ("uniform_", "uniform", "beta", "SVD"):
        raise ValueError(f"unknown init option {init_option!r}")
    return init_option


def _zero_guard(alpha, n_u):
    """:74-76 (init_BSSMF_md only): a zero in the first unknown row of alpha sets that row to 1e-10 and scales the known rows by
    1 - 1e-10, in place."""
    if alpha[-n_u:][0].all() == 0.0:
        alpha[-n_u:][0] = 1e-10
        alpha[:-n_u] = (1 - 1e-10) * alpha[:-n_u]
    return alpha


def _initial_iterate(variant, init_option, M, N, K, n_u, rows=None, wls=None, nndsvd=None, purity=None, rng=rd, say=print):
    """The reference's initial iterate of an M x N problem with K known and n_u unknown types -> (rows [lo, hi) = `rows` of u0, all M
    rows when None; alpha0).  `variant` is "partial" (init_BSSMF_md, :40-78), "purity" (init_BSSMF_md_p, :228-267) or "free"
    (unsupervised_deconv, :107-150, K = 0).  `rng` is numpy's legacy stream: the numpy.random module after set_seed, or a private
    RandomState(seed); the draws are issued in the reference's order, so u0 and alpha0 are bit-identical to it.  The data-dependent
    options call `wls(extra=None)`, the reference-based fit of every sample over all rows with the caller's rows of u as an extra
    regressor block, and `nndsvd(rank, H1=None)`, the NNDSVD (flag 0) of max(X - R_trunc H1, 1e-8), or of X, -> (the caller's rows of
    W, H).  `say` prints the purity fallback message."""
    init_option = _init_option(variant, init_option, n_u, N, say)
    if init_option == "SVD":
        if variant == "free":
            u, alpha = nndsvd(n_u)
            return u.clip(0, 1), projection_simplex_sort_2d(alpha)
        H1 = wls()                                         # constrained_nndsvd (init_func.py:17-37)
        W2, H2 = nndsvd(n_u, H1)
        u, alpha = np.clip(W2, 0, 1), np.vstack([H1, H2])
        if variant == "purity":                            # :262
            return u, np.vstack((purity * projection_simplex_sort_2d(alpha[:-n_u]), projection_simplex_sort_2d(alpha[-n_u:])))
        alpha = projection_simplex_sort_2d(alpha)
    else:
        if init_option == "beta":
            temp = np.ones((M, n_u))
            u = rng.beta(temp * 0.5, temp * 0.5)
        else:
            u = rng.uniform(size=(M, n_u))
        if rows is not None:
            u = u[rows[0]:rows[1]]
        # `uniform`: per-sample wls_intercept on [R_trunc | u] (:49-52)
        alpha = wls(extra=u) if init_option == "uniform" else rng.dirichlet(np.ones(K + n_u), N).T
    return u, (_zero_guard(alpha, n_u) if variant == "partial" else alpha)


def _host_steps(meth_frequency, d_x, R_trunc):
    """`wls` and `nndsvd` of _initial_iterate on one process: wls_all_samples of the caller's data (a resident DeviceProblem too), and
    nndsvd_initialize of the float64 host residual that constrained_nndsvd forms."""
    def wls(extra=None):
        return wls_all_samples(meth_frequency, d_x, R_trunc, extra=extra)

    def nndsvd(rank, H1=None):
        Y = np.asarray(meth_frequency, dtype=np.float64)
        if H1 is not None:
            Y = np.maximum(Y - np.asarray(R_trunc, dtype=np.float64) @ H1, 1e-8)
        return nndsvd_initialize(Y, rank=rank)
    return dict(wls=wls, nndsvd=nndsvd)


def init_BSSMF_md(init_option, meth_frequency, d_x, R_trunc, n_u, seed=None, rb_alg=wls_intercept):
    """deconvolution.py:40-78."""
    set_seed(seed)
    M, K = R_trunc.shape
    u, alpha = _initial_iterate("partial", init_option, M, meth_frequency.shape[1], K, n_u, **_host_steps(meth_frequency, d_x, R_trunc))
    return u, np.c_[R_trunc, u], alpha


def _problem(meth_frequency, d_x, R_trunc):
    # `meth_frequency` may be a DeviceProblem that is already resident in HBM (the n_u sweep of ic.py fits the same data many times,
    # a user's own outer loop calls the solver steps on the same data every iteration); it brings its own d_x and R_trunc
    return meth_frequency if isinstance(meth_frequency, DeviceProblem) else DeviceProblem(meth_frequency, d_x, R_trunc)


def _check_shape(name, a, shape):
    if tuple(np.shape(a)) != shape:
        raise ValueError(f"{name} must be {shape[0]} x {shape[1]}, got shape {tuple(np.shape(a))}")


def _host(t):
    return t.to(torch.float64).contiguous().cpu().numpy()


def update_u(u, alpha, n_iter2, a1, l_w_, l_w, u_, meth_frequency, R_trunc, n_u, d_x):
    """deconvolution.py:81-90 — n_iter2 accelerated projected-gradient steps on u, one streaming pass each, from the caller's
    iterates (u, u_) and momentum state (a1, and l_w_ = the l_w of the previous step).  -> (u, u_, a1, l_w_).  A resident DeviceProblem
    in place of meth_frequency supplies X, d_x and R_trunc."""
    prob = _problem(meth_frequency, d_x, R_trunc)
    n_u = int(n_u)
    _check_shape("u", u, (prob.M, n_u))
    _check_shape("u_", u_, (prob.M, n_u))
    _check_shape("alpha", alpha, (prob.K + n_u, prob.N))
    steps = max(int(n_iter2), 0)
    batch = FitBatch(prob, n_u, [u], [alpha], engine="stream")
    batch.u_view(0, 1).copy_(to_device(u_, prob.dtype, prob.device))      # u_prev: the U pass reads slot u_cur ^ 1 (FitBatch put u there)
    batch.set_step_state(0, [a1], [l_w], [l_w_])
    for _ in range(steps):
        batch.pass_u()
    st, = batch.states()
    out = _host(batch.u_view(0, st.u_slot)), _host(batch.u_view(0, st.u_slot ^ 1)), st.a1, float(l_w if steps else l_w_)
    batch.close()
    return out


def update_alpha(n_iter2, alpha, a2, l_h_, l_h, alpha_, R, d_x, meth_frequency):
    """deconvolution.py:93-102 — n_iter2 accelerated projected-gradient steps on alpha incl. the simplex projection, one streaming
    pass each, from the caller's iterates (alpha, alpha_) and momentum state (a2, and l_h_ = the l_h of the previous step).
    -> (alpha, alpha_, a2, l_h_).  A resident DeviceProblem in place of meth_frequency supplies X and d_x; R = [R_trunc | u] changes
    every outer iteration and is uploaded on every call."""
    R = np.asarray(R)
    if R.ndim != 2 or R.shape[1] < 1:
        raise ValueError("R must be M x Kt")
    Rk, u, nu, mode = _split_r(R)
    prob = meth_frequency.with_reference(Rk) if isinstance(meth_frequency, DeviceProblem) else DeviceProblem(meth_frequency, d_x, Rk)
    Kt = R.shape[1]
    _check_shape("R", R, (prob.M, Kt))
    _check_shape("alpha", alpha, (Kt, prob.N))
    _check_shape("alpha_", alpha_, (Kt, prob.N))
    steps = max(int(n_iter2), 0)
    batch = FitBatch(prob, nu, [u], [alpha], mode=mode, engine="stream")
    batch.A[0, 1].copy_(to_device(alpha_, prob.dtype, prob.device))       # alpha_prev: slot a_cur ^ 1
    batch.set_step_state(1, [a2], [l_h], [l_h_])
    for _ in range(steps):
        batch.pass_alpha()
    st, = batch.states()
    if st.done == 3:
        batch.close()
        raise _lib.DmfError("non-finite values reached the simplex projection")
    out = _host(batch.A[0, st.a_slot]), _host(batch.A[0, st.a_slot ^ 1]), st.a2, float(l_h if steps else l_h_)
    batch.close()
    return out


def init_BSSMF_md_p(init_option, meth_frequency, d_x, R_trunc, n_u, purity, rb_alg=wls_intercept, seed=None):
    """deconvolution.py:228-267."""
    set_seed(seed)
    M, K = R_trunc.shape
    u, alpha = _initial_iterate("purity", init_option, M, meth_frequency.shape[1], K, n_u, purity=purity,
                                **_host_steps(meth_frequency, d_x, R_trunc))
    return u, np.c_[R_trunc, u], alpha


def frank_wolfe_nmf(W1, W2, meth_frequency, H1, H2, purity, n_iter2, d_x):
    """deconvolution.py:280-302 — n_iter2 Frank-Wolfe steps k = 0 .. n_iter2-1 on (H1, H2) with W1 = R_trunc and W2 = u fixed, one
    streaming pass each.  -> (H1, H2).  A resident DeviceProblem in place of meth_frequency supplies X, d_x and W1 (its R_trunc)."""
    prob = _problem(meth_frequency, d_x, W1)
    if np.ndim(W2) != 2:
        raise ValueError("W2 must be M x n_u")
    n_u = np.shape(W2)[1]
    if W1 is not None:
        _check_shape("W1", W1, (prob.M, prob.K))
    _check_shape("W2", W2, (prob.M, n_u))
    _check_shape("H1", H1, (prob.K, prob.N))
    _check_shape("H2", H2, (n_u, prob.N))
    batch = FitBatch(prob, n_u, [W2], [np.vstack((H1, H2))], mode=_lib.DMF_MODE_PURITY, purity=purity, engine="stream")
    for k in range(int(n_iter2)):
        batch.pass_fw(k)
    st, = batch.states()
    H = _host(batch.A[0, st.a_slot])
    batch.close()
    return H[:prob.K], H[prob.K:]


def _solve(mode, u, alpha, meth_frequency, d_x, R_trunc, n_u, n_iter1, n_iter2, tol, purity=None):
    prob = _problem(meth_frequency, d_x, R_trunc)
    batch = FitBatch(prob, n_u, [np.asarray(u).reshape(-1, n_u)], [np.asarray(alpha)], mode=mode, purity=purity)
    states = batch.fit(n_iter1, n_iter2, tol)
    (u_out, a_out, n_outer, cost), = batch.results(states)
    _last.update(n_outer=n_outer, cost=cost, launches=batch.launch_count(), geometry=batch.geometry(), engine=batch.engine)
    batch.close()
    return u_out, a_out


def mdwbssmf_deconv(u, R, alpha, meth_frequency, d_x, R_trunc, n_u, n_iter1=100000, n_iter2=50, tol=1e-3):
    """deconvolution.py:190-223 — partial-reference accelerated projected gradient; returns (u, alpha)."""
    return _solve(_lib.DMF_MODE_PARTIAL, u, alpha, meth_frequency, d_x, R_trunc, n_u, n_iter1, n_iter2, tol)


def mdwbssmf_deconv_p(u, R, alpha, meth_frequency, d_x, R_trunc, n_u, purity, n_iter1=100, n_iter2=500, tol=1e-3):
    """deconvolution.py:305-337 — purity-constrained variant (U step + Frank-Wolfe alpha step)."""
    return _solve(_lib.DMF_MODE_PURITY, u, alpha, meth_frequency, d_x, R_trunc, n_u, n_iter1, n_iter2, tol, purity=purity)


def unsupervised_deconv(meth_frequency, n_u, d_x, init_option, n_iter1=100000, n_iter2=20, tol=1e-3, seed=None):
    """deconvolution.py:107-184 — reference-free variant (no R_trunc)."""
    set_seed(seed)
    M, nb = meth_frequency.shape
    u, alpha = _initial_iterate("free", init_option, M, nb, 0, n_u, **_host_steps(meth_frequency, d_x, None))
    return _solve(_lib.DMF_MODE_UNSUPERVISED, u, alpha, meth_frequency, d_x, None, n_u, n_iter1, n_iter2, tol)


def best_of_restarts(meth_frequency, d_x, R_trunc, n_u, init_option, seed, n_restarts, n_iter1, n_iter2, tol, purity=None,
                     distinct_seeds=True):
    """The restart loops of demethify.py:167-203 as ONE batched launch set: n_restarts fits, the one with the lowest final cost
    wins (first on ties, `cost < best_cost` at :199-203).  The reference re-seeds every restart with the same seed, so its
    restarts are one and the same fit (SURVEY Q2): distinct_seeds=False reproduces that (a single fit is run);
    distinct_seeds=True draws restart r from seed + r, the convention ic.py:196 uses.  -> (u, alpha, best restart, costs)."""
    if not distinct_seeds or n_restarts <= 1:
        seeds = [seed]
    else:
        base = seed[0] if isinstance(seed, (list, tuple)) else seed
        seeds = [base + r for r in range(n_restarts)]
    prob = _problem(meth_frequency, d_x, R_trunc)
    src = prob if init_option in ("uniform_", "uniform", "beta") else meth_frequency
    inits = []
    for s in seeds:
        if R_trunc is None:
            raise NotImplementedError("best_of_restarts: reference-free fits go through unsupervised_deconv one seed at a time")
        if purity is not None:
            u0, _, a0 = init_BSSMF_md_p(init_option, src, d_x, R_trunc, n_u, purity, seed=s)
        else:
            u0, _, a0 = init_BSSMF_md(init_option, src, d_x, R_trunc, n_u, seed=s)
        inits.append((np.asarray(u0).reshape(-1, n_u), np.asarray(a0)))
    mode = _lib.DMF_MODE_PURITY if purity is not None else _lib.DMF_MODE_PARTIAL
    batch = FitBatch(prob, n_u, [i[0] for i in inits], [i[1] for i in inits], mode=mode, purity=purity)
    res = batch.results(batch.fit(n_iter1, n_iter2, tol))
    costs = [r[3] for r in res]
    best = int(np.argmin(costs))
    _last.update(n_outer=res[best][2], cost=costs[best], launches=batch.launch_count(), geometry=batch.geometry(), engine=batch.engine)
    batch.close()
    return res[best][0], res[best][1], best, costs
