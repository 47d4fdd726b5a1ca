"""The bench.py contract that can be checked without a GPU: the reference arm prints ONE JSON line with the agreed keys
(it times the reference's own host-compiled device programs, or the oracle port where those are not built), and the clock
sampler degrades gracefully where neither NVML nor nvidia-smi can see a GPU."""
import json
import os
import subprocess
import sys

import helpers as H


def test_reference_arm_prints_the_contract_line(built):
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.run([sys.executable, os.path.join(H.ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--resolution", "192 108"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "rtigo3_geometry_192x108_samples_per_s" and d["unit"] == "Msamples/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "192x108" in d["config"]["workload"]
    # both arms build `config` with the same function: same keys, same spp per step (the driver compares the two lines)
    sys.path.insert(0, H.ROOT)
    import bench
    args = bench.parse_args(["--resolution", "192 108"])
    assert d["config"] == bench.path_config(args, 1)
    assert bench.metric_name(bench.parse_args([])) == "rtigo3_geometry_1080p_samples_per_s"
    assert bench.parse_args(["--config", "c1"]).resolution == "512 512" and bench.parse_args(["--config", "c4"]).scene == "rtigo3_instances"


def test_reference_arm_is_silent_on_other_ranks(built):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(H.ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path, monkeypatch):
    """--dump-outputs: float32 arrays as they are, integer arrays as float64; over the limit, every array keeps the same seeded
    sample of its rows, identical from run to run."""
    import numpy as np
    import pytest
    sys.path.insert(0, H.ROOT)
    import bench
    with pytest.raises(SystemExit):
        bench.parse_args(["--impl", "reference", "--dump-outputs", str(tmp_path)])
    t = np.arange(4000, dtype=np.float32) * np.float32(0.25)
    prim = np.arange(4000, dtype=np.uint32) + np.uint32(4000000000)
    bench.dump_outputs(str(tmp_path / "all"), {"hit_t": t, "hit_primitive": prim})
    assert np.load(str(tmp_path / "all" / "hit_t.npy")).tobytes() == t.tobytes()
    whole = np.load(str(tmp_path / "all" / "hit_primitive.npy"))
    assert whole.dtype == np.float64 and np.array_equal(whole, prim)
    monkeypatch.setattr(bench, "DUMP_LIMIT", 12000)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"hit_t": t, "hit_primitive": prim})
    got = {name: np.load(str(tmp_path / "a" / (name + ".npy"))) for name in ("hit_t", "hit_primitive")}
    assert sum(a.nbytes for a in got.values()) <= 12000 and len(got["hit_t"]) > 500
    assert np.array_equal(got["hit_t"] * 4, got["hit_primitive"] - 4000000000)          # the same rows of both arrays
    assert np.all(np.diff(got["hit_t"]) > 0)                                             # in order, no row twice
    for name, a in got.items():
        assert np.load(str(tmp_path / "b" / (name + ".npy"))).tobytes() == a.tobytes()


def test_clock_sampler_without_a_gpu():
    sys.path.insert(0, H.ROOT)
    import bench
    s = bench.ClockSampler(0)
    s.start()
    s.stop_flag.set()
    s.join(timeout=10)
    summary = s.summary()
    assert set(summary) >= {"sm_mhz", "sm_max_mhz", "reasons", "samples", "source"}
    assert summary["source"] in ("nvml", "nvidia-smi")


def test_parity_check_of_the_multi_gpu_arm_accepts_the_oracle_mean_and_rejects_a_wrong_frame(built, tmp_path):
    """bench.py's untimed N > 1 parity step: the combined frame must be the mean over the ranks of the raw radiance of each
    rank's first seed iteration (every rank accumulates from sample 0).  Exercised here with frames made by the oracle."""
    import numpy as np
    sys.path.insert(0, H.ROOT)
    import bench
    from tweeker_raytracer_b200 import host
    app = host.App(H.write_system(tmp_path, "rtigo3_cornell_box", resolution="96 128", samplesSqrt=4), H.scene_path("rtigo3_cornell_box"), host_only=True)
    world, local = 2, 8
    w, h = app.resolution
    ref, sysd = H.oracle_scene(app), H.oracle_sys(app)
    xy = np.array([(x, y) for y in range(h) for x in range(w)], dtype=np.uint32)
    frame = np.zeros((h, w, 4), dtype=np.float32)
    frame[..., :3] = ((ref.path_radiance(sysd, app.info.miss, w, xy, 0) + ref.path_radiance(sysd, app.info.miss, w, xy, local)) * np.float32(0.5)).reshape(h, w, 3)
    good = bench.parity_check(app, frame, world, local)
    assert good["result"] == "pass" and good["rows"] == 2 and good["mismatches"] == 0
    frame[64, 5, 1] += 0.01
    assert bench.parity_check(app, frame, world, local)["result"] == "fail"
    # the wrong partition (rank 1 starting at iteration 1 instead of `local`) is caught as well
    assert bench.parity_check(app, frame, world, 1)["result"] == "fail"
    app.close()
