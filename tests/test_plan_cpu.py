"""CPU checks of the launch planner (make_plan in dmf_api.cu): tests/plan_probe.cu is compiled against the library's instantiation
objects and prints the plan of every shape of a grid.  Every engine the planner offers must resolve to a kernel for every launch it
makes, stage layouts must suit the bulk copies and fit shared memory, workspace regions must be aligned and disjoint, and the geometry
of the benchmark shape and of BASELINE configs 2 and 4 is pinned."""
import itertools
import json
import os
import subprocess

import pytest

from demethify_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBE = os.path.join(ROOT, "tests", "plan_probe.cu")
F64, F32, WF, W16 = _lib.DMF_F64, _lib.DMF_F32, _lib.DMF_W_FLOAT, _lib.DMF_W_U16
PARTIAL, PURITY, UNSUP = _lib.DMF_MODE_PARTIAL, _lib.DMF_MODE_PURITY, _lib.DMF_MODE_UNSUPERVISED
PLAIN, MULT, GATHER = 0, 1, 2
DMF_E_SHAPE = 3           # include/demethify_b200.h


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    import __graft_entry__ as g
    from demethify_b200 import _build
    g.build()
    exe = str(tmp_path_factory.mktemp("plan") / "plan_probe")
    objs = sorted(os.path.join(_build.OBJ, f) for f in os.listdir(_build.OBJ) if f.startswith("dmf_inst_") and f.endswith(".o"))
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    res = subprocess.run([nvcc] + _build.NVCC_FLAGS + ["-I", _build.CSRC, PROBE] + objs + ["-o", exe], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr

    def run(shapes):
        lines = "".join(" ".join(str(v) for v in s) + "\n" for s in shapes)
        out = subprocess.run([exe], input=lines, capture_output=True, text=True, check=True).stdout.splitlines()
        assert len(out) == len(shapes)
        return [json.loads(line) for line in out]
    return run


def shape(M, N, K, n_u, dtype=F64, wtype=W16, mode=PARTIAL, n_fits=1, max_ctas=0, u_slots=4, form=PLAIN, wide=None):
    """One probe line with the pitches the Python layer (engine.py) chooses."""
    es = 8 if dtype == F64 else 4
    wide = N * es >= 512 if wide is None else wide
    pitch = (lambda b: ((N * b + 127) // 128 * 128 + 16) // b) if wide else (lambda b: (N + 7) // 8 * 8)
    ldx = pitch(es)
    ldd = pitch(2) if wtype == W16 else ldx
    ldu = n_u + (n_u & 1)
    return (M, N, K, n_u, dtype, wtype, mode, n_fits, max_ctas, u_slots, ldx, ldd, K + (K & 1), ldu, (M * ldu + 31) // 32 * 32, form)


def grid():
    out = []
    for K, n_u, N, dtype, wtype, form in itertools.product((0, 1, 4, 6, 7, 8, 12, 20, 26), (1, 2, 3, 4, 5, 8, 10, 16), (16, 64, 100, 256, 300, 512),
                                                          (F64, F32), (WF, W16), (PLAIN, MULT, GATHER)):
        out.append(shape(100_000, N, K, n_u, dtype, wtype, UNSUP if K == 0 else PARTIAL, u_slots=2 if form == MULT else 4, form=form))
    for K, n_u, N, form in itertools.product((1, 6, 8), (1, 2, 4), (16, 64, 128, 256), (PLAIN, MULT)):
        out.append(shape(200_000, N, K, n_u, mode=PURITY, form=form))
        out.append(shape(1_000, N, K, n_u, form=form, wide=True))
        out.append(shape(1_000_000, N, K, n_u, n_fits=64, u_slots=2 if form == MULT else 4, form=form))
        out.append(shape(1_000_000, N, K, n_u, n_fits=3, max_ctas=7, form=form))
    return out


def test_plan_grid(probe):
    shapes = grid()
    plans = probe(shapes)
    seen = {k: set() for k in ("engine", "s_f", "nub", "kb", "ktb", "nub_g", "kb_g", "types", "form")}
    for s, p in zip(shapes, plans):
        if p["rc"] or not p.get("mult_ok", 1) and s[-1] == MULT:
            continue
        assert not p["null_kernels"], (s, p["null_kernels"])
        for name, e in p["engines"].items():
            if not isinstance(e, dict):
                continue
            seen["engine"].add(name)
            assert all(o % 128 == 0 for o in e["offs"]), (s, name, e)
            assert all(t % 16 == 0 for t in e.get("tx", [])), (s, name, e)
            assert e["ring"] <= e["smem"] <= p["cap"], (s, name, e)
            assert 1 <= e["ctas"] <= e["tiles"] and e["groups"] == (e["ctas"] + 15) // 16, (s, name, e)
            if name == "fused":
                assert e["ring"] <= e["stats"], (s, e)
        regions = sorted((o, n) for o, n in p["ws"] if n)
        assert all(o % 256 == 0 for o, _ in p["ws"]), (s, p["ws"])
        assert all(a + n <= b for (a, n), (b, _) in zip(regions, regions[1:])), (s, p["ws"])
        assert regions[-1][0] + regions[-1][1] <= p["ws_bytes"] and p["ws_bytes"] % 256 == 0, (s, p["ws"])
        b = p["buckets"]
        seen["nub"].add(b["nub"]); seen["kb"].add(b["kb"]); seen["ktb"].add(b["ktb"])
        if "gram" in p["engines"]:
            seen["nub_g"].add(b["nub_g"]); seen["kb_g"].add(b["kb_g"]); seen["types"].add((s[4], s[5])); seen["form"].add(s[-1])
        if "fused" in p["engines"]:
            seen["s_f"].add(b["s_f"])
    # the grid reaches every engine and every bucket the planner can choose
    assert seen["engine"] == {"stream", "gram", "p1", "fused"}
    assert seen["s_f"] == {1, 2, 4}
    assert seen["nub"] == {2, 8, 16, 32} and seen["kb"] == {6, 8, 16, 32} and seen["ktb"] == {8, 16, 32}
    assert seen["nub_g"] == {1, 2, 4, 8} and seen["kb_g"] == {0, 6, 16, 32}
    assert seen["types"] == {(F64, WF), (F64, W16), (F32, WF), (F32, W16)} and seen["form"] == {PLAIN, MULT, GATHER}


def test_plan_rejects_shapes_with_their_messages(probe):
    bad = [shape(1000, 16, 20, 16), shape(1000, 600, 6, 2), shape(1000, 16, 2, 2, mode=UNSUP), shape(1000, 16, 0, 2, mode=PURITY)]
    got = [(p["rc"], p["err"]) for p in probe(bad)]
    assert got[0] == (DMF_E_SHAPE, "K + n_u (even padded) > 32 is not supported by this build")
    assert got[1] == (DMF_E_SHAPE, "N too large for this K + n_u in this build (N <= 512 for small K + n_u, <= 256 otherwise)")
    assert got[2] == (DMF_E_SHAPE, "unsupervised mode requires K = 0")
    assert got[3] == (DMF_E_SHAPE, "purity mode requires K >= 1")


# (ctas per fit, tile rows, dynamic shared memory) per engine and workspace bytes, as computed before the planner was consolidated
PINNED = {
    "bench 1M x 256, K 6, n_u 2": (
        shape(1_000_000, 256, 6, 2),
        {"stream": (296, 8, 108160), "gram": (148, 16, 215296), "fused": (148, 16, 225664)}, 133972992),
    "BASELINE config 2: 100k x 16, K 6, n_u 2": (
        shape(100_000, 16, 6, 2),
        {"stream": (296, 64, 77056), "gram": (148, 256, 193792), "fused": (148, 32, 86016)}, 8761600),
    "BASELINE config 4: 64 resamples of 500k x 64, K 6, n_u 1, multiplicity form": (
        shape(500_000, 64, 6, 1, n_fits=64, u_slots=2, form=MULT),
        {"stream": (32, 16, 60416), "gram": (32, 64, 189696), "p1": (32, 32, 94976)}, 1048375808),
    "BASELINE config 4: 64 resamples of 500k x 64, K 6, n_u 1, materialised": (
        shape(500_000, 64, 6, 1, n_fits=64),
        {"stream": (32, 16, 60416), "gram": (32, 64, 189696), "fused": (32, 32, 204288)}, 1048375808),
}


def test_plan_pinned_geometry(probe):
    names = list(PINNED)
    plans = probe([PINNED[n][0] for n in names])
    for name, p in zip(names, plans):
        got = {e: (v["ctas"], v["tile_rows"], v["smem"]) for e, v in p["engines"].items() if isinstance(v, dict)}
        assert (got, p["ws_bytes"]) == PINNED[name][1:], name
