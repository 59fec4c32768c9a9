"""Host-side logic that needs no GPU: sweep validation, refusal of initialisations the path does not have, seed lists."""
import numpy as np
import pytest


def test_sweep_member_supported_limits():
    from demethify_b200.ic import sweep_member_supported
    assert sweep_member_supported(5, 25)             # the fixture: 5 known types, the reference's whole 1..25 sweep
    assert sweep_member_supported(6, 26)
    assert not sweep_member_supported(7, 25)         # even(7) + even(25) = 34 > 32
    assert sweep_member_supported(7, 24)
    assert sweep_member_supported(25, 6) and not sweep_member_supported(25, 7)
    assert sweep_member_supported(6, 0)


@pytest.mark.parametrize("option,exc", [("ICA", NotImplementedError), ("svd", ValueError), ("typo", ValueError)])
def test_bootstrap_refuses_inits_it_does_not_have(option, exc):
    """bootstrap_fits must not silently replace an initialisation (it used to fall back to uniform_): the same errors as the
    point-estimate path, raised before any resample is drawn or any device is touched."""
    from demethify_b200.bootstrap import bootstrap_fits
    X = np.random.RandomState(0).uniform(size=(20, 6))
    with pytest.raises(exc):
        bootstrap_fits(3, 1, X, np.ones_like(X), np.zeros((20, 2)), option, 5, 5, 1e-3, None, 1)


def test_bootstrap_n_u_above_samples_falls_back_like_the_reference():
    """n_u > N turns every option into uniform_ (deconvolution.py:44-45) before the dispatch: no error for ICA then; the call goes
    on to the device layer, which refuses without a GPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from demethify_b200 import _lib
    from demethify_b200.bootstrap import bootstrap_fits
    X = np.random.RandomState(0).uniform(size=(20, 2))
    with pytest.raises(_lib.DmfError):
        bootstrap_fits(2, 3, X, np.ones_like(X), np.zeros((20, 2)), "ICA", 5, 5, 1e-3, None, 1)


def test_bootstrap_seed_sequence_and_restart_jobs():
    from demethify_b200.bootstrap import bootstrap_seeds
    assert bootstrap_seeds(1, 6) == [1, 2, 4, 7, 11, 16]          # bootstrap.py:27, SURVEY Q3
    with pytest.raises(TypeError):
        bootstrap_seeds([5], 3)                                    # `--seed 5` reaches bt_ci as a list (Q1)


def _bench_module():
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_clock_sampler_window():
    """bench.py's nvidia-smi sampler: only samples inside the timed region count; a region shorter than the sampling period falls
    back to all samples (warm-up ran the same kernels) and says so."""
    import time
    bench = _bench_module()

    class FakeProc:
        def terminate(self):
            pass
    row = lambda mhz, cap: [str(mhz), "1965", "0x4", "Not Active", "Not Active", "Not Active", cap]
    s = bench.ClockSampler(0)
    s.proc = FakeProc()
    t = time.perf_counter()
    s.rows = [(t - 2.0, row(500, "Not Active")), (t - 1.0, row(1200, "Not Active"))]      # before the timed region
    s.mark_begin()
    s.rows += [(time.perf_counter(), row(1950, "Active")), (time.perf_counter(), row(1965, "Not Active"))]
    out = s.stop()
    assert out["samples"] == 2 and out["sm_mhz"] == 1957.5 and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["sw_power_cap"] and out["window"] == "timed region"
    s2 = bench.ClockSampler(0)
    s2.proc = FakeProc()
    s2.rows = [(time.perf_counter() - 1.0, row(1900, "Not Active"))]
    s2.mark_begin()
    out2 = s2.stop()
    assert out2["samples"] == 1 and out2["sm_mhz"] == 1900.0 and out2["window"].startswith("warm-up")


def test_bench_dump_outputs_budget(tmp_path):
    """bench.py --dump-outputs: float64 .npy files under 64 MB in all; an array over its share becomes the same seeded sample of
    its rows on every run, with the row indices beside it."""
    import os
    bench = _bench_module()
    u = np.random.RandomState(0).uniform(size=(4_000_000, 2))         # 64 MB on its own
    alpha = np.random.RandomState(1).uniform(size=(8, 256)).astype(np.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"u": u, "alpha": alpha, "cost": 2.5})
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["alpha.npy", "cost.npy", "u.npy", "u_rows.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) < 64 * 2 ** 20
    got = {n: np.load(tmp_path / "a" / n) for n in names}
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["alpha.npy"], alpha) and got["cost.npy"] == 2.5
    rows = got["u_rows.npy"].astype(np.int64)
    assert np.all(np.diff(rows) > 0) and np.array_equal(got["u.npy"], u[rows])
    assert rows[-1] > 3 * len(rows) and len(rows) * (u[0].nbytes + 8) > 0.99 * bench.DUMP_BYTES / 3    # spread over u, fills its share
    assert all(np.array_equal(got[n], np.load(tmp_path / "b" / n)) for n in names)
    u_headline = u[:1_000_000]                                         # the default workload's u (1M x 2) is written whole
    bench.dump_outputs(str(tmp_path / "c"), {"u": u_headline, "alpha": alpha, "cost": 2.5})
    assert not (tmp_path / "c" / "u_rows.npy").exists() and np.array_equal(np.load(tmp_path / "c" / "u.npy"), u_headline)


def test_bench_reference_arm_dumps_its_last_step(tmp_path, monkeypatch, capsys):
    """--impl reference --dump-outputs writes the oracle's (u, alpha, cost) of its last timed step."""
    import argparse
    bench = _bench_module()
    u, a = np.arange(6.0).reshape(3, 2), np.full((8, 4), 0.125)
    leg = {"result": (u, a, {"costs": [9.0, 7.5]}), "value": 1.0, "unit": bench.UNIT, "cores": 1, "kind": "port", "sample": "",
           "s_per_step_sample": 1.0}
    monkeypatch.setattr(bench, "cpu_reference_leg", lambda steps, warmup: leg)
    bench.run_reference(argparse.Namespace(steps=1, warmup=0, gpus=1, dump_outputs=str(tmp_path)), 0, 1)
    assert '"impl": "reference"' in capsys.readouterr().out
    assert np.array_equal(np.load(tmp_path / "u.npy"), u) and np.array_equal(np.load(tmp_path / "alpha.npy"), a)
    assert np.load(tmp_path / "cost.npy") == 7.5


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"]])
def test_bench_refuses_bad_step_counts(monkeypatch, argv):
    bench = _bench_module()
    monkeypatch.setattr("sys.argv", ["bench.py", *argv])
    with pytest.raises(SystemExit):
        bench.parse()
