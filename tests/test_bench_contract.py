"""bench.py's output contract (the keys the driver and the judge read), checked on the CPU:
the committed B200 line under profiles/ has every required key with sane values, and the
reference arm (`--impl reference`, the oracle port on the host cores) runs here and prints a
conforming line.  `--dump-outputs`: its size cap and sampling on the CPU, the dumped outputs on the GPU."""
import glob
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BASE_KEYS = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"]


def _check_common(line):
    for k in BASE_KEYS:
        assert k in line, k
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert line["metric"] == "audio_hours_aligned_per_second" and "audio-hours" in base["metric"]
    assert line["unit"] == "audio-hours/s" and line["higher_is_better"] is True and line["scaling"] == "weak"
    assert line["vs_baseline"] is None and base["published"] == {}          # nothing published to divide by
    assert line["data"] == "synthetic" and "workload" in line["config"] and "model" not in line["config"]
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in line["e2e"], k


def test_committed_b200_line_has_the_contract_keys():
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r1_v*_bench*.json")),
                   key=lambda p: int(os.path.basename(p).split("_")[1][1:]))
    newest_full = [p for p in files if "gpu" not in os.path.basename(p) and "reference" not in os.path.basename(p)][-1]
    text = open(newest_full).read()
    line = json.loads(text[text.index("{"):])
    _check_common(line)
    assert line["n_gpus"] == 1 and line["warmup"] >= 3 and line["value"] > 0 and line["gpu_launches"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert 0 < line["e2e"]["value"] < line["value"]                           # the copies cost something
    roof = line["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in roof, k
    assert roof["bound"] in ("hbm", "tensor") and abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-12
    cpu = line["cpu_baseline"]
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in cpu, k
    assert cpu["kind"] in ("port", "reference") and cpu["cores"] >= 1
    clocks = line["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(clocks)
    assert not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(clocks["reasons"]))
    par = line["parity"]
    assert par["features_f32_identical"] and par["path1_identical"] and par["path2_int_identical"]
    assert par["nodes_max_abs_diff_s"] <= 1e-9


def test_reference_arm_runs_on_the_host_cores():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--scale", "0.03"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1                                                    # ONE JSON line on stdout
    line = json.loads(lines[0])
    _check_common(line)
    assert line["impl"] == "reference" and line["gpu_launches"] == 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["e2e"]["value"] == line["value"] == line["cpu_baseline"]["value"]
    installed = os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "describealign.py"))
    # the unmodified reference where tools/install_reference.sh put it (with the port beside it), else the port
    assert line["cpu_baseline"]["kind"] == ("reference" if installed else "port") and line["cpu_baseline"]["cores"] >= 1
    if installed:
        assert line["cpu_baseline"]["oracle_port_beside_it"]["kind"] == "port"


def test_steps_and_warmup_are_checked():
    for bad in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *bad], capture_output=True, text=True,
                             timeout=60, cwd=ROOT)
        assert res.returncode == 2 and res.stdout == "", (bad, res.stderr[-500:])


DUMP_SAMPLE = r'''
import sys
import numpy as np
sys.path.insert(0, %(root)r)
import bench
rng = np.random.default_rng(5)
bench.dump_outputs(%(out)r, {"rows": rng.standard_normal((1500000, 5)), "feature": rng.standard_normal(6000000).astype(np.float32),
                             "scalar": np.array([0.25])})
'''


def test_dump_outputs_keeps_a_seeded_sample_under_64_mb(tmp_path):
    """Outputs beyond the budget: every large array keeps the same seeded, ordered sample of its rows with their
    indices, small ones stay whole, and the same arrays give the same files."""
    import numpy as np
    rng = np.random.default_rng(5)
    rows, feature = rng.standard_normal((1500000, 5)), rng.standard_normal(6000000).astype(np.float32)
    for out in (tmp_path / "a", tmp_path / "b"):
        res = subprocess.run([sys.executable, "-c", DUMP_SAMPLE % dict(root=ROOT, out=str(out))], capture_output=True,
                             text=True, timeout=300)
        assert res.returncode == 0, res.stderr[-2000:]
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["feature.npy", "feature_rows.npy", "rows.npy", "rows_rows.npy", "scalar.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64e6
    for name, full in (("rows", rows), ("feature", feature)):
        idx = np.load(tmp_path / "a" / f"{name}_rows.npy")
        assert idx.dtype == np.float64 and 0.25 * len(full) < len(idx) < len(full) and np.all(np.diff(idx) > 0)
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f"{name}.npy"), full[idx.astype(np.int64)])
    assert np.load(tmp_path / "a" / "scalar.npy").tolist() == [0.25]
    for f in files:
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f


@pytest.mark.gpu
def test_dump_outputs_are_what_the_api_computes(tmp_path):
    """bench.py --dump-outputs: the last timed step's paths of each distinct pair equal what the synchronous API
    computes on the same synthetic PCM, and --steps is the number of timed steps the line reports."""
    import numpy as np
    from describealign_b200 import api, synth
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--scale", "0.05",
                          "--pairs", "5", "--workers", "2", "--distinct", "2", "--no-cpu-baseline", "--no-numa-bind",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 2 and line["config"]["pairs_per_gpu_per_step"] == 5
    files = sorted(os.listdir(tmp_path))
    assert len(files) == 2 * 8 and sum(os.path.getsize(tmp_path / f) for f in files) <= 64e6
    for k in range(2):
        v, a = synth.config_pair("C2", k, 0.05)
        det = {}
        path = api.align_pcm(v, a, details=det)[3]
        got = {f[len(f"pair{k}_"):-len(".npy")]: np.load(tmp_path / f) for f in files if f.startswith(f"pair{k}_")}
        assert all(x.dtype in (np.float32, np.float64) for x in got.values())
        # the engine hands back the rows (video j, audio i, cluster, qual, cum) in frames; align_pcm returns them
        # with j and i divided by 210 (host_fit.build_nodes)
        np.testing.assert_array_equal(got["path2"][:, 2:], path[:, 2:])
        np.testing.assert_array_equal(got["path2"][:, :2] / 210., path[:, :2])
        np.testing.assert_array_equal(got["path1"], np.stack(det["path1"], axis=1))
        for f in range(3):      # energy, zero crossings, band 0: what the host fit reads
            np.testing.assert_array_equal(got[f"video_feature{f}"], det["video_features"][f])
            np.testing.assert_array_equal(got[f"audio_feature{f}"], det["audio_features"][f])


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0", "--scale", "0.03"], capture_output=True, text=True,
                         timeout=300, cwd=ROOT, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""
