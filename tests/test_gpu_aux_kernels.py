"""The kernels that produce the fit's input and post-process its output, against exact references (oracle/exact.py).

Where the inputs make every sum the kernel forms exact in fp64 (dyadic values, small integer weights, a bit budget asserted by
the test), the kernel must agree bit for bit with an integer-arithmetic reference, whatever its accumulation order.  Elsewhere
the bar is componentwise, from the operation's error analysis.  The C ABI is called through ctypes so that padded pitches, M = 0
and raw moment matrices can be expressed."""
import ctypes as C
import os
from fractions import Fraction

import numpy as np
import pytest

from oracle import exact as ex

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DMF_E_STATE = 4
BITS = 10                      # X and R on multiples of 2^-10 in [0, 1]


@pytest.fixture(scope="module")
def env():
    import torch
    assert torch.cuda.is_available()
    import __graft_entry__ as g
    g.build()
    from demethify_b200 import _lib
    from demethify_b200.engine import _handle, _stream_ptr
    return dict(torch=torch, lib=_lib.lib(), L=_lib, h=_handle(torch.cuda.current_device()), st=_stream_ptr)


def _dev(env, a, dtype, ld=None):
    """Row-major device copy of a 2-D array with row pitch ld (zero padded)."""
    torch = env["torch"]
    a = np.atleast_2d(a)
    ld = a.shape[1] if ld is None else ld
    if dtype == "u16":
        buf = np.zeros((a.shape[0], ld), np.uint16)
        buf[:, :a.shape[1]] = a
        return torch.from_numpy(buf.view(np.int16)).cuda()
    buf = np.zeros((a.shape[0], ld), np.float64 if dtype == "f64" else np.float32)
    buf[:, :a.shape[1]] = a
    return torch.from_numpy(buf).cuda()


def _ws(env, nbytes):
    torch = env["torch"]
    t = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    return t, C.c_void_p((t.data_ptr() + 255) // 256 * 256)


def _err(env):
    return env["lib"].dmf_last_error().decode()


# ================================================================================================= WLS moments
def _even(n):
    return n + (n & 1)


def wls_call(env, fn, X, D, R1, R2, y_is_dx, dt, wt, pad=0, out=None, mom=None):
    """dmf_wls_fit / dmf_wls_moments on one storage pair with row pitches padded by `pad` (even) elements -> (rc, tensors)."""
    torch, L, lib = env["torch"], env["L"], env["lib"]
    M, N = X.shape
    K, K2 = R1.shape[1], R2.shape[1]
    ldx, ldd = _even(N) + pad, _even(N) + pad
    ldr, ldr2 = _even(K) + pad, _even(K2) + pad
    keep = [_dev(env, X, dt, ldx), _dev(env, D, "u16" if wt == "u16" else dt, ldd)]
    keep += [_dev(env, R1, dt, ldr) if K else None, _dev(env, R2, dt, ldr2) if K2 else None]
    out = torch.zeros((K + K2, N), dtype=torch.float64, device="cuda") if out is None else out
    desc = L.WlsDesc(M=M, N=N, K=K, K2=K2, dtype=L.DMF_F64 if dt == "f64" else L.DMF_F32,
                     wtype=L.DMF_W_U16 if wt == "u16" else L.DMF_W_FLOAT, y_is_dx=int(y_is_dx), ldx=ldx, ldd=ldd, ldr=ldr if K else 0,
                     ldr2=ldr2 if K2 else 0, X=keep[0].data_ptr(), D=keep[1].data_ptr(), R1=keep[2].data_ptr() if K else None,
                     R2=keep[3].data_ptr() if K2 else None, out=out.data_ptr())
    nb = C.c_size_t()
    assert lib.dmf_wls_workspace_bytes(env["h"], C.byref(desc), C.byref(nb)) == 0, _err(env)
    ws, wp = _ws(env, nb.value)
    if fn == "fit":
        rc = lib.dmf_wls_fit(env["h"], C.byref(desc), wp, nb.value, env["st"]())
        torch.cuda.synchronize()
        return rc, out
    Kz = K + K2 + 2
    mom = torch.full((Kz * Kz * N,), np.nan, dtype=torch.float64, device="cuda")
    rc = lib.dmf_wls_moments(env["h"], C.byref(desc), C.c_void_p(mom.data_ptr()), wp, nb.value, env["st"]())
    torch.cuda.synchronize()
    return rc, mom.cpu().numpy().reshape(Kz, Kz, N)


def wls_solve(env, mom, K, K2, M):
    torch, L = env["torch"], env["L"]
    N = mom.shape[2]
    out = torch.full((K + K2, N), np.nan, dtype=torch.float64, device="cuda")
    m = torch.from_numpy(np.ascontiguousarray(mom, dtype=np.float64)).cuda()
    desc = L.WlsDesc(M=M, N=N, K=K, K2=K2, out=out.data_ptr())
    ws, wp = _ws(env, 256)
    rc = env["lib"].dmf_wls_solve(env["h"], C.byref(desc), C.c_void_p(m.data_ptr()), wp, 256, env["st"]())
    torch.cuda.synchronize()
    return rc, out.cpu().numpy()


def _moment_inputs(seed, M, N, Kt, w_max):
    rs = np.random.RandomState(seed)
    X = ex.dyadic(rs, (M, N), BITS)
    R = ex.dyadic(rs, (M, Kt), BITS)
    D = rs.randint(0, w_max + 1, size=(M, N)).astype(np.float64)
    D[0] = np.maximum(D[0], 1)
    return X, D, R


# (M, N, K + K2, y_is_dx, pitch padding): the 8 x 8 block boundaries of K + K2, the slabs / pow2ceil / row groups of N, one row,
# two rows, a row tile +- 1 and enough tiles for more than 16 CTAs (two-level hier_reduce), padded pitches, odd K
MOMENT_CASES = ([(300, 3, kt, False, 0) for kt in (1, 6, 7, 14, 15, 22, 31, 32)] +
                [(300, 5, 32, True, 2)] +
                [(700, n, 5, False, 2 * (n % 2)) for n in (1, 2, 255, 256, 257, 513)] +
                [(m, 4, 3, dx, 0) for m in (1, 2) for dx in (False, True)] +
                [(m, 7, 9, False, 4) for m in (255, 256, 257, 511, 512, 513)] +
                [(40000, 6, 5, False, 0), (40000, 6, 5, True, 2)])


@pytest.mark.parametrize("M,N,Kt,y_is_dx,pad", MOMENT_CASES, ids=[f"M{c[0]}-N{c[1]}-Kt{c[2]}-{'dx' if c[3] else 'x'}-pad{c[4]}"
                                                                  for c in MOMENT_CASES])
def test_wls_moments_bitwise_vs_exact(env, M, N, Kt, y_is_dx, pad):
    """Every storage pair returns exactly the integer reference: the moments are identical across fp64 / fp32 values and float /
    u16 weights, the K2 block included."""
    w_max = 15 if (y_is_dx and M > 512) else 255
    budget = ex.moment_bit_budget(M, BITS, w_max, y_is_dx)
    assert budget <= 53, budget                      # every partial sum is an integer below 2^53 units: exact in any order
    X, D, R = _moment_inputs(M + N + Kt, M, N, Kt, w_max)
    K2 = Kt // 3
    K = Kt - K2
    want = ex.wls_moments_exact(X, D, R, y_is_dx, BITS).astype(np.float64) / float(1 << (2 * BITS))
    for dt, wt in (("f64", "f"), ("f64", "u16"), ("f32", "f"), ("f32", "u16")):
        rc, got = wls_call(env, "moments", X, D, R[:, :K], R[:, K:], y_is_dx, dt, wt, pad)
        assert rc == 0, _err(env)
        assert np.array_equal(got, want), (dt, wt, np.argwhere(got != want)[:5])


def test_wls_moments_without_rows_are_zero(env):
    torch, L = env["torch"], env["L"]
    Kz, N = 7, 5
    mom = torch.full((Kz * Kz * N,), np.nan, dtype=torch.float64, device="cuda")
    out = torch.zeros((5, N), dtype=torch.float64, device="cuda")
    desc = L.WlsDesc(M=0, N=N, K=3, K2=2, dtype=L.DMF_F64, wtype=L.DMF_W_FLOAT, ldx=6, ldd=6, ldr=4, ldr2=2, out=out.data_ptr())
    ws, wp = _ws(env, 256)
    assert env["lib"].dmf_wls_moments(env["h"], C.byref(desc), C.c_void_p(mom.data_ptr()), wp, 256, env["st"]()) == 0, _err(env)
    assert (mom.cpu().numpy() == 0).all()


@pytest.mark.parametrize("M,N,K,K2", [(3000, 257, 29, 3), (1500, 513, 32, 0), (999, 40, 7, 8)])
def test_wls_moments_then_solve_equals_fit_bitwise(env, M, N, K, K2):
    rs = np.random.RandomState(N)
    R = ex.dyadic(rs, (M, K + K2), BITS)
    A = rs.dirichlet(np.ones(K + K2), N).T
    X = np.round(np.clip(R @ A + rs.normal(0, 0.02, (M, N)), 0, 1) * 1024) / 1024
    D = rs.randint(1, 60, size=(M, N)).astype(np.float64)
    rc, fit = wls_call(env, "fit", X, D, R[:, :K], R[:, K:], True, "f64", "f")
    assert rc == 0, _err(env)
    rc, mom = wls_call(env, "moments", X, D, R[:, :K], R[:, K:], True, "f64", "f")
    assert rc == 0, _err(env)
    rc, sol = wls_solve(env, mom, K, K2, M)
    assert rc == 0, _err(env)
    assert np.array_equal(sol, fit.cpu().numpy())


# ================================================================================================= WLS NNLS
def _exact_props(r):
    x = r["x"]
    s = sum(x)
    return np.array([float(v / s) if s else 0.0 for v in x])


def _check_nnls(env, X, D, R, c_max, record, bits=BITS):
    """dmf_wls_fit against the exact NNLS of every sample: active set (when the KKT margins are clear), componentwise error
    |x - x*| <= c K cond(G_PP) eps |x*|_inf (c recorded), non-negativity."""
    M, N = X.shape
    K = R.shape[1]
    rc, out = wls_call(env, "fit", X, D, R, np.zeros((M, 0)), False, "f64", "f")
    assert rc == 0, _err(env)
    got = out.cpu().numpy()
    assert (got >= 0).all()
    mom = ex.wls_moments_exact(X, D, R, False, bits)
    for j in range(N):
        G, b = ex.centred_normal_equations(mom, j)
        r = ex.nnls_exact(G, b)
        want = _exact_props(r)
        ok, xmin, wmax, _ = r["kkt"]
        clear = (xmin is None or float(xmin) > 1e-6 * max(1.0, float(max(r["x"])))) and (wmax is None or float(wmax) < -1e-9 * float(sum(abs(v) for v in b)))
        if clear:
            assert [p for p in range(K) if got[p, j] > 0] == r["passive"], j
        c = np.abs(got[:, j] - want).max() / (K * float(r["cond"]) * ex.EPS * np.abs(want).max())
        record.append(c)
        assert c <= c_max, (j, c, float(r["cond"]))


def test_wls_nnls_vs_exact(env, capsys):
    rs = np.random.RandomState(3)
    consts = []
    # active constraints: true proportions with several exact zeros
    M, N, K = 600, 12, 8
    R = ex.dyadic(rs, (M, K), BITS)
    A = rs.dirichlet(np.ones(K), N).T
    A[rs.rand(K, N) < 0.4] = 0.0
    A /= np.maximum(A.sum(0), 1e-12)
    X = np.round(np.clip(R @ A + rs.normal(0, 0.01, (M, N)), 0, 1) * 1024) / 1024
    D = rs.randint(1, 30, size=(M, N)).astype(np.float64)
    _check_nnls(env, X, D, R, 64, consts)
    # correlated references: a shared profile plus cell-specific deviations of size delta, cond(G) ~ 1e2 .. 1e8
    conds = []
    for delta_bits in (3, 6, 9, 13):
        M, N, K = 1024, 4, 5
        shared = rs.randint(0, 1 << 15, size=(M, 1))
        dev = rs.randint(0, 1 << (16 - delta_bits), size=(M, K))
        R = (shared + dev).astype(np.float64) / (1 << 16)
        A = rs.dirichlet(np.ones(K), N).T
        X = np.round(np.clip(R @ A + rs.normal(0, 1e-3, (M, N)), 0, 1) * (1 << 16)) / (1 << 16)
        D = np.ones((M, N))
        mom = ex.wls_moments_exact(X, D, R, False, 16)
        conds.append(float(ex.cond_mp(ex.centred_normal_equations(mom, 0)[0], list(range(K)))))
        rc, out = wls_call(env, "fit", X, D, R, np.zeros((M, 0)), False, "f64", "f")
        assert rc == 0, _err(env)
        got = out.cpu().numpy()
        assert (got >= 0).all()
        for j in range(N):
            r = ex.nnls_exact(*ex.centred_normal_equations(mom, j))
            want = _exact_props(r)
            c = np.abs(got[:, j] - want).max() / (K * float(r["cond"]) * ex.EPS * np.abs(want).max())
            consts.append(c)
            assert c <= 64, (delta_bits, j, c, float(r["cond"]))
    assert conds[0] < 1e3 and conds[-1] > 1e7, conds
    with capsys.disabled():
        print(f"\nwls nnls: max c = {max(consts):.3g} over {len(consts)} samples, cond(G) swept {conds[0]:.2g} .. {conds[-1]:.2g}")


def test_wls_nnls_removal_duplicates_and_degenerate_weights(env):
    # a problem whose Lawson-Hanson run drops a variable it added (tests/test_exact_oracle_cpu.py REMOVAL_CASE): exact result
    G3, b3 = [[57, 32, 45], [32, 26, 26], [45, 26, 38]], [31, 20, 28]
    mom = np.zeros((5, 5, 1))
    mom[0, 0, 0] = 1.0
    mom[2:, 2:, 0] = G3
    mom[1, 2:, 0] = mom[2:, 1, 0] = b3
    rc, got = wls_solve(env, mom, 3, 0, 1)
    assert rc == 0, _err(env)
    x = [Fraction(0), Fraction(4, 39), Fraction(2, 3)]
    want = np.array([float(v / sum(x)) for v in x])
    assert got[0, 0] == 0.0 and np.abs(got[:, 0] - want).max() <= 64 * ex.EPS
    # duplicated reference columns: the pair's combined proportion is the exact one (the split is not determined)
    rs = np.random.RandomState(5)
    M, N, K = 800, 6, 4
    R = ex.dyadic(rs, (M, K), BITS)
    R[:, 3] = R[:, 1]
    A = rs.dirichlet(np.ones(K), N).T
    X = np.round(np.clip(R @ A + rs.normal(0, 0.01, (M, N)), 0, 1) * 1024) / 1024
    D = rs.randint(1, 30, size=(M, N)).astype(np.float64)
    rc, out = wls_call(env, "fit", X, D, R, np.zeros((M, 0)), False, "f64", "f")
    assert rc == 0, _err(env)
    got = out.cpu().numpy()
    assert (got >= 0).all()
    mom = ex.wls_moments_exact(X, D, R[:, :3], False, BITS)
    for j in range(N):
        r = ex.nnls_exact(*ex.centred_normal_equations(mom, j))
        want = _exact_props(r)
        merged = np.array([got[0, j], got[1, j] + got[3, j], got[2, j]])
        assert np.abs(merged - want).max() <= 1e-9, (j, merged, want)
    # one row with a non-zero weight: the centred G is 0, every proportion 0
    D1 = np.zeros((M, N))
    D1[17] = 3.0
    rc, out = wls_call(env, "fit", X, D1, R[:, :3], np.zeros((M, 0)), False, "f64", "f")
    assert rc == 0, _err(env)
    assert (out.cpu().numpy() == 0).all()
    # a sample whose weights are all zero (masked out completely): all its proportions are 0, the other samples are untouched
    D0 = D.copy()
    D0[:, 2] = 0
    rc, out0 = wls_call(env, "fit", X, D0, R[:, :3], np.zeros((M, 0)), False, "f64", "f")
    rc1, out1 = wls_call(env, "fit", X, D, R[:, :3], np.zeros((M, 0)), False, "f64", "f")
    assert rc == 0 and rc1 == 0, _err(env)
    o0, o1 = out0.cpu().numpy(), out1.cpu().numpy()
    assert (o0[:, 2] == 0).all() and np.array_equal(np.delete(o0, 2, 1), np.delete(o1, 2, 1))



def test_wls_nnls_iteration_limit_is_an_error(env):
    """Normal equations on which the 3 K inner steps of the active-set loop run out with a negative coefficient (the fp64 mirror,
    tests/test_exact_oracle_cpu.py): DMF_E_STATE, not a negative proportion with status OK."""
    mom = np.load(os.path.join(GOLDEN, "wls_nnls_iteration_cap.npy"))
    rc, got = wls_solve(env, mom, mom.shape[0] - 2, 0, 1)
    assert rc == DMF_E_STATE and "iteration" in _err(env), (rc, got[:, 0])


# ================================================================================================= residual Gram / projection
def resid_desc(env, X, R, H1, ldx, ldr):
    torch, L = env["torch"], env["L"]
    M, N = X.shape
    K = 0 if R is None else R.shape[1]
    keep = [_dev(env, X, "f64", ldx) if M else torch.zeros(2, dtype=torch.float64, device="cuda")]
    d = L.ResidDesc(M=M, N=N, K=K, ldx=ldx, ldr=ldr if K else 0, X=keep[0].data_ptr())
    if K:
        keep += [_dev(env, R, "f64", ldr) if M else torch.zeros(2, dtype=torch.float64, device="cuda"),
                 torch.from_numpy(np.ascontiguousarray(H1)).cuda()]
        d.R, d.H1 = keep[1].data_ptr(), keep[2].data_ptr()
    nb = C.c_size_t()
    assert env["lib"].dmf_resid_workspace_bytes(env["h"], C.byref(d), C.byref(nb)) == 0, _err(env)
    ws, wp = _ws(env, nb.value)
    keep.append(ws)
    return d, wp, nb.value, keep


def resid_gram(env, X, R, H1, pad=0):
    torch = env["torch"]
    N = X.shape[1]
    K = 0 if R is None else R.shape[1]
    d, wp, nb, keep = resid_desc(env, X, R, H1, _even(N) + pad, _even(K) + pad)
    G = torch.full((N, N), np.nan, dtype=torch.float64, device="cuda")
    neg = torch.full((1,), 7, dtype=torch.int32, device="cuda")
    rc = env["lib"].dmf_resid_gram(env["h"], C.byref(d), C.c_void_p(G.data_ptr()), C.c_void_p(neg.data_ptr()), wp, nb, env["st"]())
    assert rc == 0, _err(env)
    torch.cuda.synchronize()
    return G.cpu().numpy(), int(neg.item())


def _residual_inputs(seed, M, N, K, clamp=0.0, e_bits=BITS):
    """X = R H1 + E with dyadic R, H1, E (E on multiples of 2^-e_bits in (0, 1]): r = max(X - R H1, 1e-8) is E exactly where
    E > 0; E = 0 entries (a share `clamp`) are floored to exactly 1e-8."""
    rs = np.random.RandomState(seed)
    E = ex.dyadic(rs, (M, N), e_bits, lo=1)
    if clamp:
        E[rs.rand(M, N) < clamp] = 0.0
    if K == 0:
        return E, None, None, E
    R = ex.dyadic(rs, (M, K), BITS)
    H1 = ex.dyadic(rs, (K, N), BITS)
    X = R @ H1 + E                                      # every product and sum is exact (units of 2^-20, far below 2^53)
    assert np.array_equal(X - R @ H1, E)
    return X, R, H1, np.where(E > 0, E, 1e-8)


GRAM_CASES = ([(1001, n, 0, 0) for n in (1, 63, 64, 65, 127, 128, 129, 511, 512)] +
              [(1001, 129, k, 2) for k in (1, 31, 32)] +
              [(m, 65, 1, 0) for m in (0, 1, 3, 31, 33)] + [(20000, 65, 3, 4), (5000, 200, 0, 2)])


@pytest.mark.parametrize("M,N,K,pad", GRAM_CASES, ids=[f"M{c[0]}-N{c[1]}-K{c[2]}-pad{c[3]}" for c in GRAM_CASES])
def test_resid_gram_bitwise_vs_exact(env, M, N, K, pad):
    X, R, H1, r = _residual_inputs(M * 7 + N + K, M, N, K)
    assert (M * (1 << 2 * BITS)).bit_length() <= 53          # sum of M products of 2^-10 multiples in [0, 1]: exact in fp64
    want = r.T @ r if M else np.zeros((N, N))                # exact: every partial sum is an integer number of 2^-20 units
    G1, neg = resid_gram(env, X, R, H1, pad)
    G2, _ = resid_gram(env, X, R, H1, pad)
    assert neg == 0
    assert np.array_equal(G1, want), np.argwhere(G1 != want)[:5]
    assert np.array_equal(G1, G1.T) and np.array_equal(G1.view(np.int64), G2.view(np.int64))


def test_resid_gram_floor_componentwise(env):
    """Entries floored to exactly 1e-8: G is no longer dyadic; |G^ - G| <= gamma_M sum_m |r_mi r_mj| entry by entry against the
    exact rational G."""
    M, N, K = 3001, 65, 4
    X, R, H1, r = _residual_inputs(11, M, N, K, clamp=0.3)
    got, _ = resid_gram(env, X, R, H1, 2)
    E = np.where(r == 1e-8, 0.0, r)
    Z = (r == 1e-8).astype(np.float64)
    EE, EZ, ZZ = E.T @ E, E.T @ Z, Z.T @ Z                   # exact (small dyadic sums)
    c = Fraction(1e-8)
    g = ex.gamma(M)
    for i in range(N):
        for j in range(N):
            exact = Fraction(EE[i, j]) + c * (Fraction(EZ[i, j]) + Fraction(EZ[j, i])) + c * c * Fraction(ZZ[i, j])
            assert abs(Fraction(got[i, j]) - exact) <= Fraction(g) * exact, (i, j)
    assert np.array_equal(got, got.T)


PROJ_CASES = [(4749, 20, 0, 1), (4749, 20, 0, 20), (4749, 65, 3, 31), (4749, 200, 0, 32), (37, 33, 2, 5), (4751, 40, 32, 7)]


@pytest.mark.parametrize("M,N,K,rank", PROJ_CASES, ids=[f"M{c[0]}-N{c[1]}-K{c[2]}-rank{c[3]}" for c in PROJ_CASES])
def test_resid_project_bitwise_vs_exact(env, M, N, K, rank):
    """U = r Vh^T diag(inv_sigma) and the sums of its squared positive / negative parts, exact: dyadic residual and Vh (4 bits),
    power-of-two inv_sigma.  M > 8 rows x 4 CTAs per SM x 148 SMs, so every warp takes several rows."""
    torch = env["torch"]
    rs = np.random.RandomState(M + N + rank)
    X, R, H1, r = _residual_inputs(rs.randint(1 << 30), M, N, K, e_bits=4)
    Vh = rs.randint(-16, 17, size=(rank, N)).astype(np.float64) / 16
    inv_s = 2.0 ** rs.randint(-3, 4, size=rank)
    U_want = (r @ Vh.T) * inv_s
    sums_want = np.concatenate([(np.maximum(U_want, 0) ** 2).sum(0), (np.maximum(-U_want, 0) ** 2).sum(0)])
    # U in units of 2^-11 (r, Vh on 2^-4, inv_sigma >= 2^-3), U^2 in 2^-22: the non-negative partial sums stay below their total
    assert (int(np.abs(r).sum(1).max() * 2 ** 8)).bit_length() <= 53 and int(sums_want.max() * 2.0 ** 22).bit_length() <= 53
    d, wp, nb, keep = resid_desc(env, X, R, H1, _even(N) + 2, _even(K) + 2)
    Vt, it = torch.from_numpy(Vh).cuda(), torch.from_numpy(inv_s).cuda()
    U = torch.full((M, rank), np.nan, dtype=torch.float64, device="cuda")
    sums = torch.full((2 * rank,), np.nan, dtype=torch.float64, device="cuda")
    rc = env["lib"].dmf_resid_project(env["h"], C.byref(d), C.c_void_p(Vt.data_ptr()), C.c_void_p(it.data_ptr()), rank,
                                      C.c_void_p(U.data_ptr()), C.c_void_p(sums.data_ptr()), wp, nb, env["st"]())
    assert rc == 0, _err(env)
    assert np.array_equal(U.cpu().numpy(), U_want)
    assert np.array_equal(sums.cpu().numpy(), sums_want)


# ================================================================================================= NNDSVD
def _nndsvd_factors(rs, M, N, rank):
    """U, Vh on multiples of 2^-8 (norms exact in fp64), with: component 1 a sign tie (|u+||v+| == |u-||v-|), component 2
    single-signed (u >= 0), component 3 sigma = 0; column 0 holds values exactly at and just below the 1e-11 threshold."""
    U = rs.randint(-256, 257, size=(M, rank)).astype(np.float64) / 256
    Vh = rs.randint(-256, 257, size=(rank, N)).astype(np.float64) / 256
    S = np.sort(rs.randint(1, 1 << 12, size=rank).astype(np.float64) / 16)[::-1].copy()
    if rank > 1:
        h = M // 2
        U[:h, 1] = np.abs(U[:h, 1])
        U[h:2 * h, 1] = -U[:h, 1]
        if M % 2:
            U[-1, 1] = 0.0
        hn = N // 2
        Vh[1, :hn] = np.abs(Vh[1, :hn])
        Vh[1, hn:2 * hn] = -Vh[1, :hn]
        if N % 2:
            Vh[1, -1] = 0.0
    if rank > 2:
        U[:, 2] = np.abs(U[:, 2])
    if rank > 3:
        S[3] = 0.0
    S[0] = 1.0
    U[:2, 0] = [1e-11, np.nextafter(1e-11, 0)]
    return U, S, Vh


def _check_nndsvd(W, H, U, S, Vh, rank, scales):
    """W, H against the mpmath scales: the chosen pattern exactly, values within 8 eps (a handful of correctly rounded operations
    on exact norms), and the 1e-11 threshold on the rounded value."""
    for i, (positive, fu, fv) in enumerate(scales):
        for F, a, f in ((W[:, i], U[:, i], fu), (H[i, :], Vh[i, :], fv)):
            part = np.abs(a) if i == 0 else (np.maximum(a, 0) if positive else np.maximum(-a, 0))
            want = float(f) * part
            big = want >= 1e-11 * (1 + 16 * ex.EPS)
            small = want < 1e-11 * (1 - 16 * ex.EPS)
            assert (F[small] == 0).all(), i
            assert (np.abs(F[big] - want[big]) <= 8 * ex.EPS * want[big]).all(), i
            assert (F >= 0).all()


@pytest.mark.parametrize("M,N,rank", [(1000, 40, 5), (300000, 30, 4), (77, 9, 1)])
def test_nndsvd_apply_and_split_vs_rule(env, M, N, rank):
    torch, lib = env["torch"], env["lib"]
    rs = np.random.RandomState(M + rank)
    U, S, Vh = _nndsvd_factors(rs, M, N, rank)
    scales = ex.nndsvd_scales_mp(U, S, Vh, rank)
    if rank > 1:
        assert scales[1][0] and scales[2][0]            # the tie and the single-signed component take the positive pattern
    sums = np.concatenate([(np.maximum(U, 0) ** 2).sum(0), (np.maximum(-U, 0) ** 2).sum(0)])     # exact: 2^-16 units
    Ut, Vt, St, sm = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (U, Vh, S, sums))
    W = torch.full((M, rank), np.nan, dtype=torch.float64, device="cuda")
    H = torch.full((rank, N), np.nan, dtype=torch.float64, device="cuda")
    assert lib.dmf_nndsvd_apply(C.c_void_p(Ut.data_ptr()), M, C.c_void_p(Vt.data_ptr()), C.c_void_p(St.data_ptr()), C.c_void_p(sm.data_ptr()),
                                N, rank, C.c_void_p(W.data_ptr()), C.c_void_p(H.data_ptr()), env["st"]()) == 0, _err(env)
    torch.cuda.synchronize()
    Wa, Ha = W.cpu().numpy(), H.cpu().numpy()
    _check_nndsvd(Wa, Ha, U, S, Vh, rank, scales)
    assert Wa[0, 0] == 1e-11 and Wa[1, 0] == 0.0
    if M <= 1000:                                        # the single-process kernel on padded factors: the same W and H
        Up = torch.zeros((M, rank + 3), dtype=torch.float64, device="cuda")
        Up[:, :rank] = Ut
        Vp = torch.zeros((rank, N + 5), dtype=torch.float64, device="cuda")
        Vp[:, :N] = Vt
        W2 = torch.full((M, rank), np.nan, dtype=torch.float64, device="cuda")
        H2 = torch.full((rank, N), np.nan, dtype=torch.float64, device="cuda")
        assert lib.dmf_nndsvd_split(C.c_void_p(Up.data_ptr()), rank + 3, C.c_void_p(St.data_ptr()), C.c_void_p(Vp.data_ptr()), N + 5, M, N,
                                    rank, C.c_void_p(W2.data_ptr()), C.c_void_p(H2.data_ptr()), env["st"]()) == 0, _err(env)
        torch.cuda.synchronize()
        _check_nndsvd(W2.cpu().numpy(), H2.cpu().numpy(), U, S, Vh, rank, scales)


# ================================================================================================= percentiles
def _keep(B, qlo, qhi):
    klo, khi = int(np.floor((B - 1) * (qlo / 100.0))), int(np.floor((B - 1) * (qhi / 100.0)))
    return max(min(klo + 2, B), min(B - khi, B))


def _same(got, want):
    """Bit for bit, except that the sign of a zero follows numpy's partition order among tied +-0 (unspecified): equal as values."""
    gi, wi = got.view(np.int64), want.view(np.int64)
    return np.array_equal(got, want, equal_nan=True) and bool(((gi == wi) | (got == 0) | np.isnan(want)).all())


PCT_CASES = [(1, 0, 100, 129), (2, 0, 100, 127), (3, 25, 75, 1_000_000), (3, 50, 50, 128), (200, 15.1, 85, 129),
             (200, 15.6, 85, 128), (1000, 12.66, 90, 1), (1000, 12.76, 90, 127), (40, 2.5, 97.5, 5000)]


@pytest.mark.parametrize("B,qlo,qhi,P", PCT_CASES, ids=[f"B{c[0]}-q{c[1]}-{c[2]}-P{c[3]}" for c in PCT_CASES])
def test_percentile_bitwise_vs_numpy(env, B, qlo, qhi, P):
    """q = 0 / 100, q_lo = q_hi, B in {1, 2, 3}, keep exactly 32 / 33 / 128 (kernel) and 129 (torch.quantile fallback), g = 0.5
    exactly (B = 3, q = 25 / 75)."""
    torch = env["torch"]
    from demethify_b200.bootstrap import percentile_bounds_device
    expected_keep = {(200, 15.1): 32, (200, 15.6): 33, (1000, 12.66): 128, (1000, 12.76): 129}
    if (B, qlo) in expected_keep:
        assert _keep(B, qlo, qhi) == expected_keep[(B, qlo)]
    rs = np.random.RandomState(B + P)
    stack = rs.uniform(-1, 1, size=(B, P))
    stack[:, ::7] = np.round(stack[:, ::7] * 4) / 4              # ties
    lo, hi = percentile_bounds_device(torch.from_numpy(stack).cuda(), qlo, qhi)
    assert _same(lo, np.percentile(stack, qlo, axis=0)) and _same(hi, np.percentile(stack, qhi, axis=0))


@pytest.mark.parametrize("B,qlo,qhi", [(5, 0, 100), (41, 2.5, 97.5), (300, 20, 80), (1000, 12.76, 90)])
def test_percentile_special_values(env, B, qlo, qhi):
    """Constant columns, +-0 ties, +-inf and NaN (np.percentile: NaN for a column that holds one) - in the kernel and in the
    torch.quantile fallback (keep > 128)."""
    torch = env["torch"]
    from demethify_b200.bootstrap import percentile_bounds_device
    rs = np.random.RandomState(B)
    P = 300
    stack = rs.uniform(-1, 1, size=(B, P))
    stack[:, 0] = 0.25                                              # constant
    stack[:, 1] = np.where(rs.rand(B) < 0.5, 0.0, -0.0)             # +-0 only
    stack[:, 2] = np.where(rs.rand(B) < 0.3, np.inf, stack[:, 2])
    stack[:, 3] = np.where(rs.rand(B) < 0.3, -np.inf, stack[:, 3])
    stack[:, 4] = np.inf
    stack[B // 2, 5] = np.nan                                       # one NaN in the middle
    stack[0, 6] = np.nan                                            # first
    stack[-1, 7] = np.nan                                           # last
    stack[:, 8] = np.nan
    stack[:, 9] = np.where(rs.rand(B) < 0.5, np.inf, -np.inf)
    stack[rs.rand(B, P) < 0.01] = np.nan
    with np.errstate(invalid="ignore"):
        want_lo, want_hi = np.percentile(stack, qlo, axis=0), np.percentile(stack, qhi, axis=0)
    lo, hi = percentile_bounds_device(torch.from_numpy(stack).cuda(), qlo, qhi)
    assert _same(lo, want_lo), np.argwhere(~np.isclose(lo, want_lo, equal_nan=True))[:5]
    assert _same(hi, want_hi), np.argwhere(~np.isclose(hi, want_hi, equal_nan=True))[:5]


# ================================================================================================= consensus
@pytest.mark.parametrize("n_runs,Kt,N", [(7, 1, 30), (5, 4, 1), (3, 6, 512), (1000, 3, 40)])
def test_consensus_bitwise_vs_numpy(env, n_runs, Kt, N):
    """labels = np.argmax (first maximum; ties include -0.0 / 0.0; the first NaN wins), consensus = mean over runs."""
    from demethify_b200.ic import compute_consensus_matrix
    rs = np.random.RandomState(n_runs + N)
    runs = rs.randint(0, 3, size=(n_runs, Kt, N)).astype(np.float64) / 2        # many exact ties
    runs[rs.rand(n_runs, Kt, N) < 0.1] = -0.0
    if Kt > 1:
        runs[0, :, 0] = [0.0, -0.0] + [-1.0] * (Kt - 2)
        runs[0, :, -1] = [-0.0, 0.0] + [-1.0] * (Kt - 2)
        runs[rs.rand(n_runs, Kt, N) < 0.02] = np.nan
        runs[1 % n_runs, :, 0] = [np.nan] * Kt
        runs[0, 1, N // 2] = np.nan
    labels = np.argmax(runs, axis=1)
    want = (labels[:, :, None] == labels[:, None, :]).sum(0) / n_runs
    got = compute_consensus_matrix(list(runs))
    assert np.array_equal(got, want)
