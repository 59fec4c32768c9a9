"""Exact references of the kernels around the fit: the WLS moment matrix and its NNLS, the residual Gram matrix, the NNDSVD
sign-split rule, and an fp64 mirror of the device NNLS.

The moment references work on dyadic inputs: values on multiples of 2^-bits in [0, 1] and integer weights.  Every product the
moment kernel forms is then an integer multiple of 2^-2 bits (2^-3 bits for y = d x), and as long as the largest possible sum
stays below 2^53 units every partial sum is exact in fp64, whatever the order of accumulation.  `moment_bit_budget` computes
that bound; a test asserts it before it asks for bit-for-bit equality.

CPU only, numpy / fractions / mpmath (a dependency of the scipy stack already installed).
"""
import itertools
from fractions import Fraction

import mpmath
import numpy as np

EPS = 2.0 ** -52


def dyadic(rs, shape, bits, lo=0, hi=None):
    """Random multiples of 2^-bits in [lo, hi] (integer numerators) as float64."""
    hi = (1 << bits) if hi is None else hi
    return rs.randint(lo, hi + 1, size=shape).astype(np.float64) / (1 << bits)


def _units(a, scale_bits):
    """a * 2^scale_bits as int64, asserting that it is an integer (the value is dyadic at that scale)."""
    s = np.asarray(a, dtype=np.float64) * float(1 << scale_bits)
    i = s.astype(np.int64)
    assert np.array_equal(i.astype(np.float64), s), "input is not dyadic at the declared scale"
    return i


def moment_scale_bits(bits, y_is_dx):
    """Fixed-point scale (power of two) at which every product d z_p z_q of the moment kernel is an integer: z carries 2^-bits
    (1, x, R), so z_p z_q carries 2^-2bits; y = d x keeps the same unit (d is an integer)."""
    return 2 * bits


def moment_bit_budget(M, bits, w_max, y_is_dx):
    """Bits of the largest value a partial sum of the moment kernel can reach, in units of 2^-2bits.  With non-negative inputs
    every partial sum is at most the full sum, so one bound covers every accumulation order."""
    z_max = (1 << bits) * (w_max if y_is_dx else 1)              # units of 2^-bits: 1 -> 2^bits, y = d x <= w_max 2^bits
    term = w_max * z_max * z_max
    return int(M * term).bit_length()


def wls_moments_exact(X, D, R, y_is_dx, bits):
    """Z_j = sum_m d_mj z z^T, z = [1, y_mj, R_m0 .. R_m,K-1] (dmf_wls.cuh) as int64 (Kz, Kz, N) in units of 2^-2bits.
    R holds every regressor column (the kernel's R1 and R2 blocks side by side)."""
    M, N = X.shape
    K = R.shape[1]
    d = _units(D, 0)
    x = _units(X, bits)
    r = _units(R, bits) if K else np.zeros((M, 0), np.int64)
    y = d * x if y_is_dx else x
    z = np.empty((M, N, K + 2), dtype=np.int64)
    z[:, :, 0] = 1 << bits
    z[:, :, 1] = y
    z[:, :, 2:] = r[:, None, :]
    assert moment_bit_budget(M, bits, int(d.max()) if d.size else 1, y_is_dx) <= 62      # int64 itself must not overflow
    return np.einsum("mj,mjp,mjq->pqj", d, z, z)


def centred_normal_equations(mom, j):
    """(G, b) of sample j from an exact moment matrix, in Fractions: G_pq = Z_{2+p,2+q} - Z_{0,2+p} Z_{0,2+q} / Z_00,
    b_p = Z_{1,2+p} - Z_{0,2+p} Z_{0,1} / Z_00 (the centring of sklearn's LinearRegression with fit_intercept)."""
    Kz = mom.shape[0]
    K = Kz - 2
    Z = [[Fraction(int(mom[p, q, j])) for q in range(Kz)] for p in range(Kz)]
    sw = Z[0][0]
    G = [[Z[2 + p][2 + q] - Z[0][2 + p] * Z[0][2 + q] / sw for q in range(K)] for p in range(K)]
    b = [Z[1][2 + p] - Z[0][2 + p] * Z[0][1] / sw for p in range(K)]
    return G, b


def _solve(G, b, P):
    """Exact solve of G_PP s_P = b_P (Gauss-Jordan in Fractions); None if G_PP is singular."""
    n = len(P)
    A = [[G[P[i]][P[k]] for k in range(n)] + [b[P[i]]] for i in range(n)]
    for c in range(n):
        piv = next((r for r in range(c, n) if A[r][c] != 0), None)
        if piv is None:
            return None
        A[c], A[piv] = A[piv], A[c]
        for r in range(n):
            if r != c and A[r][c] != 0:
                f = A[r][c] / A[c][c]
                A[r] = [a - f * e for a, e in zip(A[r], A[c])]
    return [A[i][n] / A[i][i] for i in range(n)]


def kkt_certificate(G, b, x):
    """Exact KKT check of min_{x >= 0} 1/2 x^T G x - b^T x: x >= 0, w = b - G x, w_p = 0 where x_p > 0, w_p <= 0 where x_p = 0.
    Returns (ok, min positive x, max w over the active set (<= 0), max |w| over the passive set (0 when exact))."""
    K = len(b)
    w = [b[p] - sum(G[p][q] * x[q] for q in range(K)) for p in range(K)]
    pas = [p for p in range(K) if x[p] != 0]
    act = [p for p in range(K) if x[p] == 0]
    xmin = min((x[p] for p in pas), default=None)
    wmax = max((w[p] for p in act), default=None)
    stat = max((abs(w[p]) for p in pas), default=Fraction(0))
    ok = all(v >= 0 for v in x) and stat == 0 and (wmax is None or wmax <= 0)
    return ok, xmin, wmax, stat


def cond_mp(G, P, dps=50):
    """2-norm condition number of G_PP at `dps` digits (symmetric: ratio of the extreme eigenvalues' magnitudes)."""
    if not P:
        return mpmath.mpf(1)
    with mpmath.workdps(dps):
        A = mpmath.matrix([[mpmath.mpf(G[i][k].numerator) / G[i][k].denominator for k in P] for i in P])
        ev = mpmath.eigsy(A, eigvals_only=True)
        ev = [abs(e) for e in ev]
        return max(ev) / min(ev)


def nnls_exact(G, b):
    """The NNLS of the centred normal equations, exactly: Lawson-Hanson in Fractions (finite in exact arithmetic), then an
    exact KKT certificate.  Returns dict(x (Fractions), passive (sorted indices), cond (mpmath), removals (inner-loop steps),
    kkt (kkt_certificate tuple))."""
    K = len(b)
    x = [Fraction(0)] * K
    pas = set()
    removals = 0
    while True:
        w = [b[p] - sum(G[p][q] * x[q] for q in range(K)) for p in range(K)]
        cand = [p for p in range(K) if p not in pas and w[p] > 0]
        if not cand:
            break
        pas.add(max(cand, key=lambda p: (w[p], -p)))
        while True:
            P = sorted(pas)
            sP = _solve(G, b, P)
            assert sP is not None, "singular passive set"
            s = [Fraction(0)] * K
            for i, p in enumerate(P):
                s[p] = sP[i]
            if all(s[p] > 0 for p in P):
                x = s
                break
            step = min(x[p] / (x[p] - s[p]) for p in P if s[p] <= 0)
            x = [x[p] + step * (s[p] - x[p]) for p in range(K)]
            for p in P:
                if x[p] <= 0:
                    pas.discard(p)
                    x[p] = Fraction(0)
            removals += 1
    kkt = kkt_certificate(G, b, x)
    assert kkt[0], "exact Lawson-Hanson result fails its KKT certificate"
    P = sorted(pas)
    return dict(x=x, passive=P, cond=cond_mp(G, P), removals=removals, kkt=kkt)


def nnls_brute_force(G, b):
    """Every passive set: the one whose exact solve is positive and whose dual is non-positive (the unique minimiser when G is
    positive definite)."""
    K = len(b)
    for n in range(K + 1):
        for P in itertools.combinations(range(K), n):
            sP = _solve(G, b, list(P))
            if sP is None or any(v <= 0 for v in sP):
                continue
            x = [Fraction(0)] * K
            for i, p in enumerate(P):
                x[p] = sP[i]
            if kkt_certificate(G, b, x)[0]:
                return x, list(P)
    raise AssertionError("no passive set satisfies the KKT conditions")


def objective(G, b, x):
    """1/2 x^T G x - b^T x, exactly (x in Fractions or floats converted exactly)."""
    x = [Fraction(v) for v in x]
    K = len(b)
    return sum(x[p] * G[p][q] * x[q] for p in range(K) for q in range(K)) / 2 - sum(b[p] * x[p] for p in range(K))


def wls_nnls_mirror(mom, j, K, M):
    """Line-by-line fp64 mirror of wls_nnls_kernel (dmf_wls.cuh) for sample j of a float64 (Kz, Kz, N) moment matrix.  The
    library is compiled with -fmad=false and the kernel has no explicit fma, so every operation here rounds as on the device.
    Returns (normalised x, status bits, raw x, number of inner-loop steps, whether the inner loop hit its 3 K limit)."""
    Kz = K + 2
    Z = lambda p, q: float(mom[p, q, j])            # noqa: E731
    sw = Z(0, 0)
    G = [[0.0] * K for _ in range(K)]
    b = [0.0] * K
    for p in range(K):
        rp = Z(0, 2 + p) / sw
        b[p] = Z(1, 2 + p) - rp * Z(0, 1)
        for q in range(K):
            G[p][q] = Z(2 + p, 2 + q) - rp * Z(0, 2 + q)
    x = [0.0] * K
    pas = [False] * K
    nb = 0.0
    for p in range(K):
        nb += abs(b[p])
    tolx = 10.0 * float(M if M > K else K) * 2.220446049250313e-16
    tol = tolx * nb
    st = dict(singular=False, capped=False)
    s = [0.0] * K

    def solve():
        idx = [p for p in range(K) if pas[p]]
        for p in range(K):
            s[p] = 0.0
        n = len(idx)
        L = [[0.0] * n for _ in range(n)]
        for i in range(n):
            for k in range(i + 1):
                v = G[idx[i]][idx[k]]
                for t in range(k):
                    v -= L[i][t] * L[k][t]
                if i == k and not (v > 0.0):
                    st["singular"] = True
                L[i][k] = np.sqrt(v if v > 0.0 else 1e-300) if i == k else v / L[k][k]
        y = [0.0] * n
        for i in range(n):
            v = b[idx[i]]
            for t in range(i):
                v -= L[i][t] * y[t]
            y[i] = v / L[i][i]
        for i in range(n - 1, -1, -1):
            v = y[i]
            for t in range(i + 1, n):
                v -= L[t][i] * s[idx[t]]
            s[idx[i]] = v / L[i][i]

    def grad():
        w = [0.0] * K
        for p in range(K):
            v = b[p]
            for q in range(K):
                v -= G[p][q] * x[q]
            w[p] = v
        return w

    w = grad()
    it, max_it = 0, 3 * K
    while True:
        best, wb = -1, tol
        for p in range(K):
            if not pas[p] and w[p] > wb:
                wb, best = w[p], p
        if best < 0:
            break
        pas[best] = True
        solve()
        while True:
            smin = min((s[p] for p in range(K) if pas[p]), default=1e300)
            if smin > 0.0:
                break
            if it >= max_it:
                st["capped"] = True
                break
            it += 1
            step = 1e300
            for p in range(K):
                if pas[p] and s[p] <= 0.0:
                    t = x[p] / (x[p] - s[p])
                    step = min(step, t)
            for p in range(K):
                x[p] = x[p] * (1.0 - step) + step * s[p]
            for p in range(K):
                if x[p] <= tolx:
                    pas[p] = False
            for p in range(K):
                if not pas[p]:
                    x[p] = 0.0
            solve()
        for p in range(K):
            x[p] = s[p]
        w = grad()
    tot = 0.0
    for p in range(K):
        tot += x[p]
    den = tot if tot > 1e-10 else 1e-10
    status = (0 if tot == tot else 1) | (2 if st["singular"] else 0) | (4 if st["capped"] else 0)
    return np.array([v / den for v in x]), status, np.array(x), it, st["capped"]


def _sumsq_mp(a):
    """sum a_i^2 exactly (as mpf at the working precision): Python integers when the values are multiples of 2^-64 below 2^10,
    mpmath otherwise."""
    a = np.asarray(a, dtype=np.float64)
    s = a * 2.0 ** 52
    if a.size and np.abs(a).max() < 2 ** 10 and np.array_equal(np.floor(s), s):
        t = sum(int(v) * int(v) for v in s.astype(np.int64).tolist())
        return mpmath.mpf(t) / mpmath.mpf(2) ** 104
    return mpmath.fsum(mpmath.mpf(float(v)) ** 2 for v in a)


def nndsvd_scales_mp(U, S, Vh, rank, dps=50):
    """Per component i of init_func.py:46-69 (the rule of nndsvd_split_kernel / nndsvd_apply_kernel), in mpmath on the given
    factors: (positive, fu, fv) with W[:, i] = fu * (the chosen sign part of u_i), H[i] = fv * (that of v_i).  Component 0 is
    sqrt(S_0) |u_0|, sqrt(S_0) |v_0| (positive = True); component i >= 1 takes the sign pattern with the larger product of norms,
    the positive one on a tie, scaled by sqrt(S_i term) / norm.  A chosen pattern with a zero norm is 0 / 0 in the reference too:
    NaN."""
    out = []
    with mpmath.workdps(dps):
        for i in range(rank):
            s = mpmath.mpf(float(S[i]))
            if i == 0:
                out.append((True, mpmath.sqrt(s), mpmath.sqrt(s)))
                continue
            u, v = np.asarray(U[:, i], dtype=np.float64), np.asarray(Vh[i, :], dtype=np.float64)
            sq = _sumsq_mp
            nup, nun = mpmath.sqrt(sq(u[u > 0])), mpmath.sqrt(sq(u[u < 0]))
            nvp, nvn = mpmath.sqrt(sq(v[v > 0])), mpmath.sqrt(sq(v[v < 0]))
            termp, termn = nup * nvp, nun * nvn
            positive = termp >= termn
            term = termp if positive else termn
            nu_, nv_ = (nup, nvp) if positive else (nun, nvn)
            out.append((positive, mpmath.sqrt(s * term) / nu_ if nu_ else mpmath.nan, mpmath.sqrt(s * term) / nv_ if nv_ else mpmath.nan))
    return out


def nndsvd_rule_mp(U, S, Vh, rank, dps=50):
    """W (M x rank) and H (rank x N) of the NNDSVD rule (nndsvd_scales_mp) as lists of mpf, before the kernels' 1e-11 threshold
    (that is applied to rounded values, so a test applies it to the rounded reference), and the chosen patterns."""
    M, N = U.shape[0], Vh.shape[1]
    sc = nndsvd_scales_mp(U, S, Vh, rank, dps)
    with mpmath.workdps(dps):
        W = [[mpmath.mpf(0)] * rank for _ in range(M)]
        H = [[mpmath.mpf(0)] * N for _ in range(rank)]
        for i, (positive, fu, fv) in enumerate(sc):
            part = (lambda t: abs(t)) if i == 0 else ((lambda t: max(t, 0.0)) if positive else (lambda t: max(-t, 0.0)))
            for m in range(M):
                W[m][i] = fu * mpmath.mpf(part(float(U[m, i])))
            for j in range(N):
                H[i][j] = fv * mpmath.mpf(part(float(Vh[i, j])))
        return W, H, [p for p, _, _ in sc]


def gamma(n):
    """gamma_n = n u / (1 - n u), u = 2^-53: the bound of n successive fp64 roundings."""
    u = 2.0 ** -53
    return n * u / (1.0 - n * u)
