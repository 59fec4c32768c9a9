"""Every kernel the library can launch, run against the oracle.

The library is a set of lookup tables (dmf_inst_body.cuh): each streaming and Gram-form kernel exists once per storage pair
(fp64 / fp32 values, float / uint16 weights), the fused kernels once per weight type.  A *dispatch entry* is one (lookup function,
storage tag, arguments) triple that resolves to a kernel; tests/plan_probe.cu lists them all ("universe") and names the entries a
fit of a given shape launches on each engine.  CASES is the test matrix: the CPU test below checks that it reaches every entry,
the GPU tests run every case with its exact memory layout and compare with the fp64 oracle.

Pitch styles: `device` is DeviceProblem's rule (16-byte multiples), `minimal` the smallest even pitches (ldx = ldd = even(N), the
layout of INTEGRATION.md's stub: rows that are not a multiple of 16 bytes, so the tile copies have tails and the gathered form
copies rows byte by byte), `padded` every pitch a few elements larger than the row and a gap behind M*ldu in every U slot."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from demethify_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBE = os.path.join(ROOT, "tests", "plan_probe.cu")
TAGS = ("f64_f64", "f64_u16", "f32_f32", "f32_u16")
MODES = {"partial": _lib.DMF_MODE_PARTIAL, "purity": _lib.DMF_MODE_PURITY, "unsup": _lib.DMF_MODE_UNSUPERVISED}
ENGINES = {"stream": _lib.DMF_ENGINE_STREAM, "gram": _lib.DMF_ENGINE_GRAM, "fused": _lib.DMF_ENGINE_FUSED}
FORMS = {"plain": 0, "mult": 1, "rows": 2}          # the probe's form codes
DMF_E_ARG = 1                                        # include/demethify_b200.h
IT1, IT2 = 3, 6                                      # outer / inner iterations of a matrix case (tol = 0: exactly IT1 outer ones)
TRACE_CAP = 2                                        # fewer than IT1 + 1 costs: the entries behind the cap must stay untouched


def even(n):
    return n + (n & 1)


def _cases():
    """(M, N, K, n_u, dtype, wtype, mode, engine, form, pitch style, max_ctas_per_fit, n_fits), deterministic."""
    # stream engine: one shape per U-pass table entry (kUTable, first entry covering even(K), even(n_u)); cost / alpha buckets 8, 16, 32
    stream = [(1237, 33, 5, 2, "partial"),     # u[kb=6,nub=2], ktb 8
              (1500, 20, 7, 1, "purity"),      # u[8,2], ktb 16
              (900, 64, 3, 3, "partial"),      # u[8,8]
              (1100, 17, 12, 2, "partial"),    # u[16,2]
              (800, 40, 10, 5, "purity"),      # u[16,8]
              (700, 24, 4, 9, "partial"),      # u[16,16]
              (600, 100, 20, 2, "partial"),    # u[32,2], ktb 32
              (500, 9, 17, 7, "partial"),      # u[32,8]
              (650, 30, 0, 18, "unsup")]       # u[32,32]
    # Gram-form engine: one shape per rowgram table entry (kRowgramTable: first entry covering even(K), n_u); panels 8 and 16 wide,
    # u_inner for 1, 2, 4, 8 unknown types, alpha_inner 8, 16, 32 lanes
    gram = [(1500, 16, 0, 1, "unsup"), (1300, 65, 0, 2, "unsup"), (1000, 40, 0, 3, "unsup"), (900, 24, 0, 6, "unsup"),
            (1237, 33, 5, 1, "partial"), (1111, 48, 6, 2, "purity"), (800, 100, 3, 4, "partial"), (700, 20, 4, 7, "partial"),
            (600, 130, 7, 1, "purity"), (900, 17, 12, 2, "partial"), (750, 64, 9, 3, "partial"),
            (640, 12, 19, 1, "partial"), (560, 36, 20, 2, "purity"), (500, 120, 17, 4, "partial")]
    # multiplicity form (Gram-form engine only): 1 (its own panel), 2 and 4 unknown-type buckets
    mult = [(1200, 24, 5, 1, "partial"), (1000, 40, 4, 2, "purity"), (900, 17, 3, 4, "partial")]
    # fused engine (fp64 only): known bucket 0 / 4 / 6 / 8 x 1 / 2 unknown types x width class N <= 64 / 128 / 256
    fused = [(K, n_u) for K in (0, 3, 5, 8) for n_u in (1, 2)]
    styles = ("device", "minimal", "padded")
    out = []
    for t, tag in enumerate(TAGS):
        dt, wt = tag.split("_")
        wt = "u16" if wt == "u16" else "f"
        for i, (M, N, K, n_u, mode) in enumerate(stream):
            form = "rows" if i in (0, 3) else "plain"
            out.append((M, N, K, n_u, dt, wt, mode, "stream", form, styles[(i + t) % 3], 17 if i == 2 else 0, 2 if i == 3 else 1))
        for i, (M, N, K, n_u, mode) in enumerate(gram):
            form = "rows" if i in (5, 9) else "plain"
            out.append((M, N, K, n_u, dt, wt, mode, "gram", form, styles[(i + t + 1) % 3], 1 if i == 4 else 0, 2 if i == 10 else 1))
        for i, (M, N, K, n_u, mode) in enumerate(mult):
            out.append((M, N, K, n_u, dt, wt, mode, "gram", "mult", styles[(i + t + 2) % 3], 0, 2 if i == 1 else 1))
        if dt == "f64":
            for i, (N, (K, n_u)) in enumerate((N, f) for N in ((40, 104, 200) if wt == "u16" else (33, 72, 129)) for f in fused):
                mode = "unsup" if K == 0 else ("purity" if i % 3 == 1 else "partial")
                out.append((900 + 37 * i, N, K, n_u, dt, wt, mode, "fused", "plain", styles[(i + t) % 3], 17 if i % 7 == 3 else 0,
                            3 if i == 10 else 1))
    return out


CASES = _cases()

# Dispatch entries no shape of the planner's domain launches, with the reason.  The scan in
# test_matrix_reaches_every_dispatch_entry keeps this list exact: an entry belongs here if and only if the scan cannot reach it.
UNREACHABLE = {}


def case_id(c):
    M, N, K, n_u, dt, wt, mode, eng, form, style, mc, nf = c
    return f"{dt}_{wt}-{eng}-{mode}-{form}-{style}-M{M}N{N}K{K}u{n_u}" + (f"-ctas{mc}" if mc else "") + (f"-fits{nf}" if nf > 1 else "")


def layout(c):
    """Pitches of a case (elements): ldx, ldd, ldr, ldu, u_slot, u_slots."""
    M, N, K, n_u, dt, wt, mode, eng, form, style, mc, nf = c
    es = 8 if dt == "f64" else 4
    if style == "device":                                   # DeviceProblem / FitBatch
        wide = N * es >= 512
        ldx = ((N * es + 127) // 128 * 128 + 16) // es if wide else (N + 7) // 8 * 8
        ldd = (((N * 2 + 127) // 128 * 128 + 16) // 2 if wide else (N + 7) // 8 * 8) if wt == "u16" else ldx
        ldu = even(n_u)
        u_slot = (M * ldu + 31) // 32 * 32
        u_slots = 4 if dt == "f64" and n_u <= 2 and form == "plain" else 2
        return ldx, ldd, even(K), ldu, u_slot, u_slots
    al16 = lambda n: (n * es + 15) // 16 * 16 // es         # noqa: E731
    if style == "minimal":
        ldx = ldd = even(N)
        ldr, ldu = even(K), even(n_u)
        u_slot = al16(M * ldu)
    else:                                                   # padded; u16 weights keep 16-byte rows so the fused engine still applies
        ldx = even(N) + 6
        ldd = (N + 7) // 8 * 8 + 8 if wt == "u16" else even(N) + 4
        ldr, ldu = even(K) + 2, even(n_u) + 2
        u_slot = al16(M * ldu) + 16
    return ldx, ldd, ldr, ldu, u_slot, 4 if eng == "fused" else 2


def probe_line(c):
    M, N, K, n_u, dt, wt, mode, eng, form, style, mc, nf = c
    ldx, ldd, ldr, ldu, u_slot, u_slots = layout(c)
    return (M, N, K, n_u, _lib.DMF_F64 if dt == "f64" else _lib.DMF_F32, _lib.DMF_W_U16 if wt == "u16" else _lib.DMF_W_FLOAT, MODES[mode],
            nf, mc, u_slots, ldx, ldd, ldr, ldu, u_slot, FORMS[form])


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    import __graft_entry__ as g
    from demethify_b200 import _build
    g.build()
    exe = str(tmp_path_factory.mktemp("matrix") / "plan_probe")
    objs = sorted(os.path.join(_build.OBJ, f) for f in os.listdir(_build.OBJ) if f.startswith("dmf_inst_") and f.endswith(".o"))
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    res = subprocess.run([nvcc] + _build.NVCC_FLAGS + ["-I", _build.CSRC, PROBE] + objs + ["-o", exe], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr

    def run(shapes=None, mode=None):
        if mode:
            return subprocess.run([exe, mode], capture_output=True, text=True, check=True).stdout.splitlines()
        lines = "".join(" ".join(str(v) for v in s) + "\n" for s in shapes)
        out = subprocess.run([exe], input=lines, capture_output=True, text=True, check=True).stdout.splitlines()
        assert len(out) == len(shapes)
        return [json.loads(line) for line in out]
    return run


WLS_CASES = [(tag, integer) for tag in TAGS for integer in (True, False) if integer or not tag.endswith("u16")]


def test_matrix_reaches_every_dispatch_entry(probe):
    """CASES launches every dispatch entry that some shape can launch, on every (storage tag, engine, mode) the planner offers,
    with every pitch style per storage tag, and the planner accepts every case."""
    universe = probe(mode="universe")
    assert len(universe) == len(set(universe))
    scan = probe(mode="scan")
    reached_anywhere = {s for s in scan if not s.startswith("combo ")}
    combos = {tuple(s.split()[1:]) for s in scan if s.startswith("combo ")}
    wls = {f"wls<{tag}>" for tag, _ in WLS_CASES}
    assert set(UNREACHABLE) == set(universe) - reached_anywhere - wls, "UNREACHABLE must list exactly what no shape launches"

    plans = probe([probe_line(c) for c in CASES])
    launched, seen_combos, seen_styles = set(), set(), set()
    for c, p in zip(CASES, plans):
        assert p["rc"] == 0, (case_id(c), p.get("err"))
        assert p["mult_ok"] or c[8] != "mult", case_id(c)
        eng = c[7]
        assert eng in p["launch"], (case_id(c), "engine not offered")
        assert "null" not in p["launch"][eng], case_id(c)
        launched |= set(p["launch"][eng])
        tag = f"{c[4]}_{'u16' if c[5] == 'u16' else c[4]}"
        seen_combos.add((tag, eng, c[6]))
        seen_styles.add((tag, c[9]))
    missing = set(universe) - set(UNREACHABLE) - wls - launched
    assert not missing, f"dispatch entries no case launches: {sorted(missing)}"
    assert launched <= set(universe)
    allowed = combos
    assert allowed - seen_combos == set(), f"(storage, engine, mode) the planner offers that no case runs: {sorted(allowed - seen_combos)}"
    assert seen_styles == {(t, s) for t in TAGS for s in ("device", "minimal", "padded")}


# ================================================================================================= GPU
@pytest.fixture(scope="module")
def pkg():
    import torch
    assert torch.cuda.is_available()
    import __graft_entry__ as g
    g.build()
    import demethify_b200
    demethify_b200.set_precision("fp64")
    demethify_b200.set_engine("auto")
    return demethify_b200


def synth(seed, M, N, K, n_true, float_weights, depth=40):
    rs = np.random.RandomState(seed)
    a = rs.uniform(0.2, 1.0, size=K + n_true)
    Rf = rs.beta(a, a, size=(M, K + n_true))
    A = rs.dirichlet(np.ones(K + n_true), N).T
    D = rs.poisson(depth, size=(M, N)) + 1
    X = rs.binomial(D, np.clip(Rf @ A, 0, 1)) / D
    D = D * 0.37 if float_weights else D.astype(np.int64)
    return X, D, np.ascontiguousarray(Rf[:, :K])


class Problem:
    """The inputs of one case (host, float64 values of what the device holds) and the initial iterates of its fits."""

    def __init__(self, c, seed=0):
        M, N, K, n_u, dt, wt, mode, eng, form, style, mc, nf = c
        self.c = c
        rs = np.random.RandomState(seed + M + 7 * N + 31 * K + n_u)
        X, D, Rk = synth(seed + M + N + K, M, N, K, max(n_u, 1), wt == "f")
        r32 = (lambda a: a.astype(np.float32).astype(np.float64)) if dt == "f32" else (lambda a: a)
        self.X, self.D, self.Rk = r32(X), (r32(D) if wt == "f" else D), r32(Rk)
        self.pur = rs.uniform(0.3, 0.9, size=N) if mode == "purity" else None
        self.rows = [np.sort(rs.randint(0, M, size=M)).astype(np.int32) if form != "plain" else None for _ in range(nf)]
        self.U0, self.A0 = [], []
        for i in range(nf):
            if mode == "unsup":           # the draws of oracle.solve_unsupervised("uniform_", seed)
                d = np.random.RandomState(100 * seed + i)
                u0, a0 = d.uniform(size=(M, n_u)), d.dirichlet(np.ones(n_u), N).T
            else:
                u0, a0 = rs.uniform(size=(M, n_u)), rs.dirichlet(np.ones(K + n_u), N).T
                if mode == "purity":
                    a0 = np.vstack([a0[:K] / a0[:K].sum(0) * self.pur, a0[K:] / a0[K:].sum(0) * (1 - self.pur)])
            self.U0.append(r32(u0)); self.A0.append(r32(a0))
        self.seed = seed

    def fit_inputs(self, i):
        r = self.rows[i]
        return (self.X, self.D, self.Rk) if r is None else (self.X[r], self.D[r], self.Rk[r])

    def oracle(self, i, it1=IT1, it2=IT2, tol=0.0):
        from oracle import bssmf_numpy as orc
        n_u, mode = self.c[3], self.c[6]
        X, D, Rk = self.fit_inputs(i)
        D = D.astype(float)
        tr = {}
        if mode == "unsup":
            u, a = orc.solve_unsupervised(X, n_u, D, "uniform_", it1, it2, tol, seed=100 * self.seed + i, trace=tr)
            assert np.array_equal(u.shape, self.U0[i].shape)
        elif mode == "purity":
            u, a = orc.solve_purity(self.U0[i].copy(), np.c_[Rk, self.U0[i]], self.A0[i].copy(), X, D, Rk, n_u, self.pur, it1, it2, tol,
                                    trace=tr)
        else:
            u, a = orc.solve_partial_reference(self.U0[i].copy(), np.c_[Rk, self.U0[i]], self.A0[i].copy(), X, D, Rk, n_u, it1, it2,
                                               tol, trace=tr)
        return u, a, tr["n_outer"], tr["costs"]


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def run_device(prob, it1=IT1, it2=IT2, tol=0.0, engine=None, max_ctas=None, wtype=None):
    """A `device`-style case through DeviceProblem / FitBatch -> (results, geometry, engine)."""
    import torch
    from demethify_b200.engine import DeviceProblem, FitBatch
    M, N, K, n_u, dt, wt, mode, eng, form, style, mc, nf = prob.c
    wt = wtype or wt
    precision = "fp64" if dt == "f64" else "fp32"
    Rk = prob.Rk if K else None
    dp = DeviceProblem(prob.X, prob.D, Rk, precision=precision, narrow_weights=wt == "u16")
    assert dp.wtype == (_lib.DMF_W_U16 if wt == "u16" else _lib.DMF_W_FLOAT)
    kw = dict(mode=MODES[mode], purity=prob.pur, max_ctas_per_fit=mc if max_ctas is None else max_ctas, engine=engine or eng,
              trace_cap=TRACE_CAP)
    dev = dp.device
    if form == "rows":
        kw["rows"] = [torch.from_numpy(r).to(dev) for r in prob.rows]
    elif form == "mult":
        kw["rows"] = [torch.from_numpy(r).to(dev) for r in prob.rows]
        kw["mult"] = [torch.from_numpy(np.bincount(r, minlength=M).astype(np.int32)).to(dev) for r in prob.rows]
        kw["offs"] = [torch.from_numpy(np.r_[0, np.cumsum(np.bincount(r, minlength=M))].astype(np.int32)).to(dev) for r in prob.rows]
    b = FitBatch(dp, n_u, prob.U0, prob.A0, **kw)
    try:
        res = b.results(b.fit(it1, it2, tol))
        return res, b.geometry(), b.engine, b.trace.cpu().numpy()
    finally:
        b.close()


def run_raw(prob, it1=IT1, it2=IT2, tol=0.0, canaries=True):
    """A case with its exact pitches through the C ABI (ctypes on _lib.Shape / _lib.FitDesc, the recipe of INTEGRATION.md).
    U slot gaps and the trace entries behind trace_cap are NaN canaries; U padding columns start at zero."""
    import torch
    from demethify_b200 import engine as E
    M, N, K, n_u, dt, wt, mode, eng, form, style, mc, nf = prob.c
    ldx, ldd, ldr, ldu, u_slot, u_slots = layout(prob.c)
    npt = np.float64 if dt == "f64" else np.float32
    dev = E.current_device()
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)       # noqa: E731
    Xh = np.zeros((M, ldx), npt); Xh[:, :N] = prob.X
    Dh = np.zeros((M, ldd), np.uint16 if wt == "u16" else npt); Dh[:, :N] = prob.D
    Rh = np.zeros((M, ldr), npt); Rh[:, :K] = prob.Rk
    Uh = np.full((nf, u_slots, u_slot), np.nan, npt)
    for i in range(nf):
        for s in range(u_slots):
            blk = np.zeros((M, ldu), npt)
            if s < 2:
                blk[:, :n_u] = prob.U0[i]
            Uh[i, s, :M * ldu] = blk.reshape(-1)
    Ah = np.stack([np.stack([a, a]) for a in prob.A0]).astype(npt)
    Th = np.full((nf, TRACE_CAP + 3), np.nan)
    Xd, Dd, Rd, Ud, Ad, Td = up(Xh), up(Dh), up(Rh), up(Uh), up(Ah), up(Th)
    keep = [Xd, Dd, Rd, Ud, Ad, Td]
    pur = up(prob.pur) if prob.pur is not None else None
    lib = _lib.lib()
    h = E._handle(dev.index)
    shape = _lib.Shape(M=M, N=N, K=K, n_u=n_u, dtype=_lib.DMF_F64 if dt == "f64" else _lib.DMF_F32,
                       wtype=_lib.DMF_W_U16 if wt == "u16" else _lib.DMF_W_FLOAT, mode=MODES[mode], n_fits=nf, max_ctas_per_fit=mc,
                       ldx=ldx, ldd=ldd, ldr=ldr, ldu=ldu, u_slot=u_slot, u_slots=u_slots)
    nbytes = C.c_size_t()
    _lib.check(lib.dmf_batch_workspace_bytes(h, C.byref(shape), C.byref(nbytes)))
    ws = torch.empty(nbytes.value + 256, dtype=torch.uint8, device=dev)
    descs = (_lib.FitDesc * nf)()
    for i in range(nf):
        d = descs[i]
        d.X, d.D, d.Rk = Xd.data_ptr(), Dd.data_ptr(), Rd.data_ptr() if K else None
        if form != "plain":
            r = up(prob.rows[i]); keep.append(r)
            d.rows = r.data_ptr()
        if form == "mult":
            cnt = np.bincount(prob.rows[i], minlength=M)
            m, o = up(cnt.astype(np.int32)), up(np.r_[0, np.cumsum(cnt)].astype(np.int32)); keep += [m, o]
            d.mult, d.offs = m.data_ptr(), o.data_ptr()
        d.U, d.A = Ud[i].data_ptr(), Ad[i].data_ptr()
        d.purity = pur.data_ptr() if pur is not None else None
        d.cost_trace, d.trace_cap = Td[i].data_ptr(), TRACE_CAP
    b = C.c_void_p()
    _lib.check(lib.dmf_batch_create(h, C.byref(shape), descs, C.c_void_p((ws.data_ptr() + 255) // 256 * 256), nbytes.value, _stream(),
                                    C.byref(b)))
    try:
        _lib.check(lib.dmf_batch_set_engine(b, ENGINES[eng]))
        g = [C.c_int32() for _ in range(3)]
        _lib.check(lib.dmf_batch_geometry(b, *[C.byref(v) for v in g]))
        _lib.check(lib.dmf_fit_batched(b, it1, it2, tol, _stream()))
        st = (_lib.FitState * nf)()
        _lib.check(lib.dmf_batch_read_state(b, st, nf, _stream()))
    finally:
        lib.dmf_batch_destroy(b)
    Uo, Ao, To = Ud.cpu().numpy(), Ad.cpu().numpy(), Td.cpu().numpy()
    res = [(Uo[i, s.u_slot, :M * ldu].reshape(M, ldu)[:, :n_u].astype(np.float64), Ao[i, s.a_slot].astype(np.float64), s.n_outer, s.cost)
           for i, s in enumerate(st)]
    if canaries:
        assert np.isnan(Uo[:, :, M * ldu:]).all(), "a kernel wrote into the gap behind M*ldu of a U slot"
        assert (Uo[:, :, :M * ldu].reshape(nf, u_slots, M, ldu)[..., n_u:] == 0).all(), "a kernel wrote a U padding column"
        assert np.isnan(To[:, TRACE_CAP:]).all(), "a kernel wrote beyond trace_cap"
    geom = {"ctas_per_fit": g[0].value, "tile_rows": g[1].value, "smem_bytes": g[2].value}
    return res, geom, eng, To


def run_case(prob, **kw):
    return (run_device if prob.c[9] == "device" else run_raw)(prob, **kw)


def bars(dt):
    # fp64: |d alpha|, |d u| and the relative cost difference after IT1 outer iterations (DESIGN reports ~1e-14 after full fits);
    # fp32: the suite's fp32 bars against the fp64 oracle on the fp32-rounded inputs
    return (1e-10, 1e-10, 1e-12) if dt == "f64" else (1e-4, 1e-3, 1e-5)


def check_vs_oracle(prob, res, trace=None, it1=IT1, it2=IT2, tol=0.0):
    ta, tu, tc = bars(prob.c[4])
    for i, (u, a, n_outer, cost) in enumerate(res):
        uo, ao, no, costs = prob.oracle(i, it1, it2, tol)
        assert n_outer == no, (i, n_outer, no)
        assert np.abs(a - ao).max() <= ta, (i, np.abs(a - ao).max())
        assert np.abs(u - uo).max() <= tu, (i, np.abs(u - uo).max())
        assert abs(cost - costs[-1]) <= tc * costs[-1], (i, cost, costs[-1])
        if trace is not None:
            assert np.all(np.abs(trace[i, :TRACE_CAP] - costs[:TRACE_CAP]) <= tc * costs[0]), (i, trace[i], costs)


@pytest.fixture(scope="module")
def predicted(probe):
    plans = probe([probe_line(c) for c in CASES])
    return {case_id(c): p for c, p in zip(CASES, plans)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_case_vs_oracle(pkg, predicted, case):
    """The case's layout on its engine: the geometry the probe predicts, the oracle's iterate and cost, untouched canaries."""
    prob = Problem(case)
    res, geom, eng, trace = run_case(prob)
    assert eng == case[7]
    e = predicted[case_id(case)]["engines"][eng]
    assert (geom["ctas_per_fit"], geom["tile_rows"], geom["smem_bytes"]) == (e["ctas"], e["tile_rows"], e["smem"])
    check_vs_oracle(prob, res, trace)


# (M, N, K, n_u, mode, engine, tol): fits that stop on the cost test before n_iter1
CONVERGED = [(1400, 24, 5, 2, "partial", "stream", 2e-2), (1400, 24, 5, 2, "partial", "gram", 2e-2),
             (1400, 24, 5, 2, "partial", "fused", 2e-2), (1300, 40, 3, 1, "purity", "gram", 150.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K,n_u,mode,eng,tol", CONVERGED, ids=lambda v: str(v))
def test_converged_fit_stops_with_oracle(pkg, M, N, K, n_u, mode, eng, tol):
    prob = Problem((M, N, K, n_u, "f64", "u16", mode, eng, "plain", "minimal" if eng != "fused" else "padded", 0, 1))
    res, _, _, trace = run_case(prob, it1=200, it2=10, tol=tol)
    _, _, no, _ = prob.oracle(0, 200, 10, tol)
    assert 1 < no < 200
    check_vs_oracle(prob, res, trace, 200, 10, tol)


def _same(r1, r2):
    for (u1, a1, n1, c1), (u2, a2, n2, c2) in zip(r1, r2):
        assert n1 == n2 and c1 == c2 and np.array_equal(a1, a2) and np.array_equal(u1, u2)


@pytest.mark.gpu
@pytest.mark.parametrize("eng", ["stream", "gram", "fused"])
def test_u16_and_float_weights_bit_identical(pkg, probe, eng):
    """Integer coverage stored as uint16 or as fp64: the same arithmetic wherever the tile geometry is the same."""
    N = {"stream": 16, "gram": 40, "fused": 40}[eng]         # sample counts at which both weight types get the same tiles
    c16 = (1301, N, 5, 2, "f64", "u16", "partial", eng, "plain", "device", 0, 1)
    cf = c16[:5] + ("f",) + c16[6:]
    p16, pf = probe([probe_line(c16), probe_line(cf)])
    g16, gf = p16["engines"][eng], pf["engines"][eng]
    assert (g16["ctas"], g16["tile_rows"]) == (gf["ctas"], gf["tile_rows"])
    prob = Problem(c16)
    r16, *_ = run_device(prob)
    rf, *_ = run_device(prob, wtype="f")
    _same(r16, rf)


@pytest.mark.gpu
@pytest.mark.parametrize("tag,eng", [("f64_u16", "stream"), ("f64_u16", "gram"), ("f64_u16", "fused"), ("f32_f32", "stream"),
                                     ("f32_f32", "gram")])
def test_pitch_styles_bit_identical(pkg, probe, eng, tag):
    """minimal and padded pitches against DeviceProblem's: bit for bit wherever the probe reports the same CTAs and tile rows (the
    fused engine needs 16-byte weight rows, which the minimal pitch of 46 u16 weights is not)."""
    dt, wt = tag.split("_")
    base = (1203, 46, 5, 2, dt, "u16" if wt == "u16" else "f", "partial", eng, "plain")
    cs = {s: base + (s, 0, 1) for s in ("device", "minimal", "padded")}
    plans = dict(zip(cs, probe([probe_line(c) for c in cs.values()])))
    ref = Problem(cs["device"])
    rd, *_ = run_device(ref)
    n_same = 0
    for s in ("minimal", "padded"):
        e, ed = plans[s]["engines"].get(eng), plans["device"]["engines"][eng]
        if e is None or (e["ctas"], e["tile_rows"]) != (ed["ctas"], ed["tile_rows"]):
            continue
        prob = Problem(cs[s])
        rs_, *_ = run_raw(prob)
        _same(rd, rs_)
        n_same += 1
    assert n_same >= 1


@pytest.mark.gpu
@pytest.mark.parametrize("eng", ["stream", "gram"])
@pytest.mark.parametrize("style", ["device", "minimal"])
def test_gathered_form_matches_materialised_gather(pkg, eng, style):
    """A fit on rows gathered by the kernels' tile producer against the same fit on a copy of those rows."""
    c = (1407, 26, 5, 2, "f32", "u16", "partial", eng, "rows", style, 0, 1)
    prob = Problem(c)
    rg, *_ = run_case(prob)
    mat = Problem(c[:8] + ("plain",) + c[9:])
    r = prob.rows[0]
    mat.X, mat.D, mat.Rk, mat.U0, mat.A0 = prob.X[r], prob.D[r], prob.Rk[r], prob.U0, prob.A0
    rm, *_ = run_case(mat)
    _same(rg, rm)


@pytest.mark.gpu
@pytest.mark.parametrize("eng", ["stream", "gram", "fused"])
def test_batch_matches_single_fits(pkg, eng):
    """Three fits that stop at different outer iterations: the batch (its descriptor array compacted to the running fits) returns
    what each fit returns alone with the same CTAs per fit."""
    from demethify_b200.engine import DeviceProblem, FitBatch
    M, N, K, n_u, tol = 9001, 24, 5, 2, 20.0
    probs, inits = [], []
    for s in range(3):
        X, D, Rk = synth(500 + s, M, N, K, n_u, False)
        rs = np.random.RandomState(600 + s)
        probs.append((X, D, Rk))
        inits.append((rs.uniform(size=(M, n_u)), rs.dirichlet(np.ones(K + n_u), N).T))
    dps = [DeviceProblem(X, D, Rk) for X, D, Rk in probs]
    b = FitBatch(dps, n_u, [i[0] for i in inits], [i[1] for i in inits], max_ctas_per_fit=17, engine=eng)
    assert b.geometry()["ctas_per_fit"] == 17
    rb = b.results(b.fit(60, 10, tol))
    b.close()
    assert len({r[2] for r in rb}) == 3, [r[2] for r in rb]
    for dp, (u0, a0), r in zip(dps, inits, rb):
        s = FitBatch(dp, n_u, [u0], [a0], max_ctas_per_fit=17, engine=eng)
        rs_ = s.results(s.fit(60, 10, tol))
        s.close()
        _same([r], rs_)


@pytest.mark.gpu
@pytest.mark.parametrize("eng", ["stream", "gram", "fused"])
def test_run_to_run_bit_identical(pkg, eng):
    c = (2111, 40, 6, 2, "f64", "u16", "partial", eng, "plain", "padded", 0, 1)
    prob = Problem(c)
    r1, *_ = run_raw(prob)
    r2, *_ = run_raw(prob)
    _same(r1, r2)


@pytest.mark.gpu
@pytest.mark.parametrize("eng", ["stream", "gram", "fused"])
def test_forced_grids(pkg, probe, eng):
    """One CTA per fit, and 17 CTAs (a second reduction level holding a one-CTA group), against the default grid."""
    base = (20011, 48, 5, 2, "f64", "u16", "partial", eng, "plain", "device")
    default = probe([probe_line(base + (0, 1))])[0]["engines"][eng]
    assert default["tiles"] >= 17 and default["ctas"] > 17
    prob = Problem(base + (0, 1))
    r0, g0, *_ = run_device(prob)
    assert g0["ctas_per_fit"] == default["ctas"]
    for mc in (1, 17):
        r, g, *_ = run_device(prob, max_ctas=mc)
        assert g["ctas_per_fit"] == mc
        for (u, a, n, c), (u0, a0, n0, c0) in zip(r, r0):
            assert n == n0 and np.abs(a - a0).max() <= 1e-12 and np.abs(u - u0).max() <= 1e-12 and abs(c - c0) <= 1e-12 * c0


@pytest.mark.gpu
@pytest.mark.parametrize("tag,integer", WLS_CASES, ids=lambda v: str(v))
def test_wls_each_storage_pair(pkg, tag, integer):
    """wls_all_samples (dmf_wls_fit) on every storage pair, integer and non-integer weights, against the oracle's NNLS fit."""
    from demethify_b200.init_func import wls_all_samples
    from oracle import bssmf_numpy as orc
    dt, wt = tag.split("_")
    M, N, K = 2003, 37, 5
    X, D, Rk = synth(71 + N, M, N, K, 2, not integer)
    if dt == "f32":
        X, Rk = X.astype(np.float32).astype(np.float64), Rk.astype(np.float32).astype(np.float64)
        if not integer:
            D = D.astype(np.float32).astype(np.float64)
    from demethify_b200.engine import DeviceProblem
    prob = DeviceProblem(X, D, Rk, precision="fp64" if dt == "f64" else "fp32", narrow_weights=wt == "u16")
    assert prob.wtype == (_lib.DMF_W_U16 if wt == "u16" else _lib.DMF_W_FLOAT)
    got = wls_all_samples(prob, None, None)
    want = np.stack([orc.wls_simplex_fit(X[:, j], D[:, j].astype(float), Rk) for j in range(N)], axis=1)
    assert np.abs(got - want).max() <= (1e-8 if dt == "f64" else 1e-4)


# ------------------------------------------------------------------------------------------------- dmf_pack_weights_u16
PACK_VALUES = [0.0, -0.0, 65535.0, 65535.5, 65536.0, -1.0, np.nan, np.inf, -np.inf, 1.0, 12345.0, 0.5]
PACK_I64 = [0, 65535, 65536, -1, 2 ** 32 + 5, 2 ** 53 + 1, 7]


def _pack(src_np, kind):
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    src = torch.from_numpy(src_np).to(dev)
    dst = torch.full((len(src_np),), 0xBEEF, dtype=torch.int32, device=dev).to(torch.int16).view(torch.uint16)
    bad = torch.full((1,), -7, dtype=torch.int32, device=dev)
    _lib.check(_lib.lib().dmf_pack_weights_u16(C.c_void_p(src.data_ptr()), kind, len(src_np), C.c_void_p(dst.data_ptr()),
                                               C.c_void_p(bad.data_ptr()), _stream()))
    return dst.view(torch.int16).cpu().numpy().view(np.uint16), int(bad.item())


def _want(vals):
    v = np.asarray(vals, dtype=np.float64)
    ok = (v >= 0) & (v <= 65535) & (v == np.floor(np.where(np.isfinite(v), v, 0.5)))
    return np.where(ok, v, 0).astype(np.uint16), int((~ok).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_pack_weights_boundaries(pkg, kind):
    if kind == 2:
        src = np.array(PACK_I64, dtype=np.int64)
        ok = (src >= 0) & (src <= 65535)
        want, nbad = np.where(ok, src, 0).astype(np.uint16), int((~ok).sum())
    else:
        src = np.array(PACK_VALUES, dtype=np.float64 if kind == 0 else np.float32)
        want, nbad = _want(src)
    got, bad = _pack(src, kind)
    assert np.array_equal(got, want) and bad == nbad


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_pack_weights_counts_every_bad_entry(pkg, kind):
    """More entries than the grid has threads (148 * 16 blocks of 256): one thread visits several; two bad entries one grid stride
    apart fall on the same thread and must count twice."""
    stride = 148 * 16 * 256
    n = 3 * stride + 11
    src = (np.arange(n) % 60000).astype({0: np.float64, 1: np.float32, 2: np.int64}[kind])
    src[5] = -3
    src[5 + stride] = 70000
    src[n - 1] = 65536
    got, bad = _pack(src, kind)
    want = np.where((src >= 0) & (src <= 65535), src, 0).astype(np.uint16)
    assert bad == 3 and np.array_equal(got, want)


def test_pack_weights_argument_errors():
    import __graft_entry__ as g
    g.build()
    lib = _lib.lib()
    one = (C.c_double * 1)(1.0)
    out = (C.c_uint16 * 1)()
    bad = (C.c_int32 * 1)()
    assert lib.dmf_pack_weights_u16(None, 0, 1, out, bad, None) == DMF_E_ARG
    assert lib.dmf_pack_weights_u16(one, 0, -1, out, bad, None) == DMF_E_ARG


# ------------------------------------------------------------------------------------------------- dmf_gather_rows
GATHER = [(1, 16, 50), (1, 13, 50), (2, 8, 40), (2, 21, 40), (4, 4, 33), (4, 7, 33), (8, 2, 70), (8, 9, 70), (8, 64, 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("elem,row_elems,n_rows", GATHER, ids=lambda v: str(v))
@pytest.mark.parametrize("dst_offset", [0, 1])
def test_gather_rows_bit_exact(pkg, elem, row_elems, n_rows, dst_offset):
    """Rows of 16-byte multiples (vector copies) and of other lengths (byte copies), a destination view that starts off its
    allocation's alignment, repeated rows: bit for bit what numpy fancy indexing returns."""
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    rs = np.random.RandomState(elem * 100 + row_elems)
    src = rs.randint(0, 256, size=(97, row_elems * elem)).astype(np.uint8)
    rows = rs.randint(0, 97, size=n_rows).astype(np.int32)
    rows[1] = rows[0]
    s = torch.from_numpy(src).to(dev)
    r = torch.from_numpy(rows).to(dev)
    buf = torch.full((n_rows * row_elems * elem + 64,), 0xA5, dtype=torch.uint8, device=dev)
    off = dst_offset * elem
    _lib.check(_lib.lib().dmf_gather_rows(C.c_void_p(s.data_ptr()), C.c_void_p(r.data_ptr()), n_rows, row_elems, elem,
                                          C.c_void_p(buf.data_ptr() + off), _stream()))
    out = buf.cpu().numpy()
    assert np.array_equal(out[off:off + n_rows * row_elems * elem].reshape(n_rows, -1), src[rows])
    assert (out[:off] == 0xA5).all() and (out[off + n_rows * row_elems * elem:] == 0xA5).all()


@pytest.mark.gpu
def test_gather_rows_zero_rows_and_argument_errors(pkg):
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    s = torch.zeros(64, dtype=torch.uint8, device=dev)
    r = torch.zeros(4, dtype=torch.int32, device=dev)
    d = torch.full((64,), 7, dtype=torch.uint8, device=dev)
    lib = _lib.lib()
    p = lambda t: C.c_void_p(t.data_ptr())       # noqa: E731
    assert lib.dmf_gather_rows(p(s), p(r), 0, 8, 8, p(d), _stream()) == 0
    torch.cuda.synchronize()
    assert (d.cpu().numpy() == 7).all()
    assert lib.dmf_gather_rows(None, p(r), 1, 8, 8, p(d), _stream()) == DMF_E_ARG
    assert lib.dmf_gather_rows(p(s), None, 1, 8, 8, p(d), _stream()) == DMF_E_ARG
    assert lib.dmf_gather_rows(p(s), p(r), 1, 8, 8, None, _stream()) == DMF_E_ARG
    assert lib.dmf_gather_rows(p(s), p(r), -1, 8, 8, p(d), _stream()) == DMF_E_ARG
    assert lib.dmf_gather_rows(p(s), p(r), 1, 0, 8, p(d), _stream()) == DMF_E_ARG
    assert lib.dmf_gather_rows(p(s), p(r), 1, 8, 3, p(d), _stream()) == DMF_E_ARG
