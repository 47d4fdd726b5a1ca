"""bench.py --dump-outputs on the GPU: the frame the timed steps leave behind is the oracle's frame of the same iterations,
bit for bit, so the file a build writes can be compared with another build's output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers as H
from tweeker_raytracer_b200 import host

pytestmark = pytest.mark.gpu


def run_bench(out_dir, flags):
    env = dict(os.environ, RANK="0", LOCAL_RANK="0", WORLD_SIZE="1")
    run = subprocess.run([sys.executable, os.path.join(H.ROOT, "bench.py")] + flags
                         + ["--no-cpu-baseline", "--no-ncu", "--no-probes", "--dump-outputs", out_dir],
                         capture_output=True, text=True, timeout=600, env=env)
    assert run.returncode == 0, run.stderr[-2000:]
    return json.loads([l for l in run.stdout.splitlines() if l.startswith("{")][-1])


def test_dump_outputs_hold_the_frame_of_the_last_timed_step(cuda_device, tmp_path):
    sys.path.insert(0, H.ROOT)
    import bench
    flags = ["--resolution", "64 36", "--spp-per-step", "2", "--warmup", "1", "--steps", "3"]
    out_dir = os.path.join(str(tmp_path), "outputs")
    line = run_bench(out_dir, flags)
    assert line["steps"] == 3 and line["warmup"] == 1
    assert os.listdir(out_dir) == ["frame.npy"]
    got = np.load(os.path.join(out_dir, "frame.npy"))
    assert got.dtype == np.float32 and got.shape == (36, 64, 4)
    # one warm-up and three timed steps of 2 iterations each, accumulated into one running average: 8 iterations
    args = bench.parse_args(flags)
    app = host.App(bench.system_file(str(tmp_path), args, 0), bench.scene_file(str(tmp_path), args), host_only=True)
    try:
        want = H.oracle_scene(app).render(H.oracle_sys(app), app.info.miss, 64, 36, iter_count=8).reshape(36, 64, 4)
    finally:
        app.close()
    assert got.tobytes() == want.tobytes()


@pytest.mark.parametrize("config", ["c3-1M-coh-closest", "c3-1M-incoh-any"])
def test_dump_outputs_hold_the_hits_of_the_ray_configs(cuda_device, tmp_path, config):
    """Config 3: the dumped fields are the hits (or occlusion flags) of the same rays traced against the same soup through the
    library's query interface, field for field."""
    sys.path.insert(0, H.ROOT)
    import bench
    from tweeker_raytracer_b200 import core
    out_dir = os.path.join(str(tmp_path), "outputs")
    run_bench(out_dir, ["--config", config, "--rays", "4096", "--warmup", "1", "--steps", "2"])
    ntris, kind, mode = bench.c3_parse(config)
    rays = bench.rays_numpy(4096, kind, mode)
    ctx = core.Context(0)
    try:
        verts = bench.soup_numpy(ntris)
        idx = np.arange(3 * ntris, dtype=np.uint32)
        d_verts, d_idx = ctx.to_device(verts), ctx.to_device(idx)
        inst = np.zeros(1, dtype=core.INSTANCE_DTYPE)
        inst[0]["transform"] = [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0]
        inst[0]["gas"] = ctx.gas_build(d_verts, 12, 3 * ntris, d_idx, ntris, core.BUILD_GPU_LBVH)
        top = ctx.ias_build(inst)
        if mode == "closest":
            hits = ctx.trace_closest_host(top, rays)
            want = {"hit_t": hits["t"], "hit_u": hits["u"], "hit_v": hits["v"], "hit_instance": hits["inst"].astype(np.float64),
                    "hit_primitive": hits["prim"].astype(np.float64)}
        else:
            want = {"occluded": ctx.trace_any_host(top, rays).astype(np.float64)}
    finally:
        ctx.close()
    assert sorted(os.listdir(out_dir)) == sorted(name + ".npy" for name in want)
    for name, w in want.items():
        got = np.load(os.path.join(out_dir, name + ".npy"))
        assert got.dtype == w.dtype and got.shape == (len(rays),), name
        assert got.tobytes() == np.ascontiguousarray(w).tobytes(), name
    if mode == "closest":
        assert 0 < int((want["hit_primitive"] != 0xFFFFFFFF).sum()) < len(rays)      # some rays hit, some miss
