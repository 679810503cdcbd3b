"""bench.py's one-line JSON contract: the reference arm and the no-GPU behaviour on the CPU, our arm on a B200."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT, have_gpu

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config"}


def run_bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=ROOT)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    return r, (json.loads(lines[-1]) if lines else None)


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "sipnet_ref")), reason="oracle/_ref not built")
def test_reference_arm_line():
    r, line = run_bench("--impl", "reference", "--steps", "1", "--warmup", "1", "--members", "64", "--years", "1")
    assert r.returncode == 0 and line is not None, r.stderr[-2000:]
    assert BASE_KEYS <= set(line) and line["impl"] == "reference"
    assert line["metric"] == "ensemble member-timesteps/sec" and line["unit"] == "member-timesteps/s"
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["dtype"] == "f64"
    assert "workload" in line["config"] and "model" not in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["value"] > 1e4


@pytest.mark.skipif(have_gpu(), reason="needs a machine WITHOUT a GPU")
def test_our_arm_refuses_to_run_without_a_gpu():
    r, line = run_bench("--steps", "1", "--warmup", "1", "--members", "64", "--years", "1")
    assert r.returncode != 0 and line is None
    assert "no CPU fallback" in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_our_arm_line():
    r, line = run_bench("--steps", "2", "--warmup", "3", "--members", "2048", "--years", "1", "--no-cpu-baseline")
    assert r.returncode == 0 and line is not None, r.stderr[-2000:]
    assert BASE_KEYS <= set(line) and "impl" not in line
    assert line["n_gpus"] == 1 and line["steps"] == 2 and line["warmup"] == 3 and line["scaling"] == "weak"
    assert line["comm_nranks"] == 1 and "C4" in line["config"]["workload"]
    roof = line["roofline"]
    assert roof["bound"] in ("fp64", "hbm") and roof["unit"] in ("TFLOP/s", "GB/s")
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-12 and 0 < roof["frac"] < 1
    assert set(line["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert line["gpu_launches"] >= 4 * line["steps"]              # init_state, step kernel, replay, summary kernels per pass
    e2e = line["e2e"]
    T = line["config"]["model_steps"]
    assert e2e["h2d_bytes_per_step"] == 80 * 2048 * 8 and e2e["d2h_bytes_per_step"] == (2 + 2 + 6) * T * 8
    assert 0 < e2e["value"] < line["value"]                       # the copies are inside the timed region
    assert line["oracle_spot_check"]["bit_identical_to_oracle"] is True
    assert line["c5"]["comm_nranks"] == 1 and line["c5"]["value"] > 0
    assert line["c2"]["e2e"]["d2h_bytes_per_step"] == 32 * T * 4096 * 8
    assert line["c2"]["d2h_probe"]["gb_s_all_ranks"] >= line["c2"]["e2e"]["d2h_gb_s_all_ranks"] > 0   # the ceiling beside it


@pytest.mark.gpu
def test_dumped_outputs_repeat_run_to_run_and_are_the_pass_results(tmp_path):
    """--dump-outputs writes what the last timed pass returned; the same arguments give the same inputs, so two runs
    write the same arrays.  They are the C4 pass's results: the members' NEE / GPP columns of a fresh run, bit for
    bit and equal to the oracle, and the ensemble summaries of those columns."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from oracle.pyoracle import Oracle
    from sipnet_b200 import _abi as A, api, synth
    M = 2048
    names = ("mean", "variance", "quantiles", "member_nee_gpp")
    dumps = []
    for k in range(2):
        d = tmp_path / str(k)
        r, line = run_bench("--steps", "2", "--warmup", "1", "--members", str(M), "--years", "1", "--no-cpu-baseline",
                            "--no-extras", "--dump-outputs", str(d))
        assert r.returncode == 0 and line is not None, r.stderr[-2000:]
        assert sorted(p.name for p in d.iterdir()) == sorted(n + ".npy" for n in names)
        dumps.append({n: np.load(d / (n + ".npy")) for n in names})
    T = line["config"]["model_steps"]
    a, b = dumps
    assert a["mean"].shape == a["variance"].shape == (1, 2, T) and a["quantiles"].shape == (1, 2, 3, T)
    assert a["member_nee_gpp"].shape == (2, T, 64)
    for n in names:
        assert a[n].dtype == np.float64 and np.isfinite(a[n]).all(), n
        assert np.array_equal(a[n], b[n]), n

    site = synth.synth_site(0, 1, "half-daily")
    params = synth.synth_params(M, stream=100)
    with api.Ensemble([site], params, None, dict(synth.SYNTH_FLAGS), math=A.MATH_FAST, summary_cols=[A.O["nee"], A.O["gpp"]],
                      outputs=A.OUT_MOMENTS | A.OUT_QUANTILES, quantiles=bench.QUANTILES) as ens:
        ens.run()
        ens.sync()
        x = bench.kept_columns(ens, M, T).cpu().numpy()         # [2][T][M]: NEE, GPP of every member
    pick = bench.dump_members(M)
    assert np.array_equal(a["member_nee_gpp"], x[:, :, pick])
    scale = np.abs(x).max()
    np.testing.assert_allclose(a["mean"][0], x.mean(axis=2), rtol=1e-12, atol=1e-12 * scale)
    np.testing.assert_allclose(a["variance"][0], x.var(axis=2), rtol=1e-9, atol=1e-9 * scale ** 2)
    np.testing.assert_allclose(a["quantiles"][0], np.quantile(x, bench.QUANTILES, axis=2).transpose(1, 0, 2), rtol=4e-16,
                               atol=1e-300)
    orc = Oracle()
    for j in (0, pick.size - 1):
        rc, done, o_out, _, _ = orc.run(synth.SYNTH_FLAGS, params[:, pick[j]], site, want_debug=False)
        assert rc == 0 and done == T
        assert np.array_equal(a["member_nee_gpp"][:, :, j], o_out[:, [A.O["nee"], A.O["gpp"]]].T)


def test_dump_stays_under_64_mb_for_long_runs():
    """Past DUMP_BYTES the dump keeps evenly spaced steps, the first and the last included."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    assert np.array_equal(bench.dump_steps(7306, 10 + 2 * 64), np.arange(7306))
    for T in (58440, 365 * 2 * 1000, 10 ** 7):
        per_step = 10 + 2 * bench.dump_members(131072).size
        s = bench.dump_steps(T, per_step)
        assert s[0] == 0 and s[-1] == T - 1 and (np.diff(s) > 0).all()
        assert 8 * per_step * s.size <= bench.DUMP_BYTES < 64_000_000 - 4096


@pytest.mark.parametrize("args", [("--steps", "0"), ("--impl", "reference", "--dump-outputs", "d"),
                                  ("--workload", "c3", "--dump-outputs", "d")])
def test_bad_arguments_are_refused(args):
    r, line = run_bench(*args)
    assert r.returncode == 2 and line is None and "bench.py: error:" in r.stderr


def test_both_arms_share_one_config_object():
    """`config` must be the same dict in both arms (the driver compares them)."""
    import argparse
    sys.path.insert(0, ROOT)
    import bench
    args = argparse.Namespace(members=131072, years=10)
    a = bench.bench_config(args, 7306)
    assert a == bench.bench_config(args, 7306) and set(a) >= {"workload", "members_per_gpu", "model_steps"}
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"config": bench_config(args, T)') == 2      # our arm and the reference arm


def test_host_writer_section_runs_without_a_gpu():
    """bench.py's informational `host_writer` section is host C only (the drop-in driver's main-output writer)."""
    sys.path.insert(0, ROOT)
    import bench
    r = bench.host_writer_rate(300, members=19)
    assert r["value"] > 0 and r["text_gb_s"] > 0 and r["threads"] >= 1 and "19 members x 300 steps" in r["sample"]
