"""GPU parity, part 8: launch shapes and path lengths at the edges -- resolutions that do not tile into 8x4 warps, a single
pixel, paths of length 0 and 1, Russian roulette from the first vertex, an empty scene, more samples than one batch holds.
All frames bit-exact against the oracle."""
import os

import numpy as np
import pytest

import helpers as H
from tweeker_raytracer_b200 import host

pytestmark = pytest.mark.gpu


def _check(tmp_path, scene="rtigo3_cornell_box", iterations=3, scene_file=None, **overrides):
    with host.App(H.write_system(tmp_path, scene, **overrides), scene_file or H.scene_path(scene)) as app:
        w, h = app.resolution
        assert app.render(iterations) == iterations
        got = app.frame()
        want = H.oracle_scene(app).render(H.oracle_sys(app), app.info.miss, w, h, iter_count=iterations).reshape(h, w, 4)
        assert got.tobytes() == want.tobytes()
        assert app.stats().stackOverflows == 0
        return got


@pytest.mark.parametrize("resolution", ["1 1", "7 5", "33 17", "130 3", "8 4", "64 36"])
def test_launch_shapes(cuda_device, tmp_path, resolution):
    _check(tmp_path, resolution=resolution, samplesSqrt=2, iterations=4)


@pytest.mark.parametrize("lengths", ["0 0", "0 1", "1 1", "0 2", "3 3", "0 16"])
def test_path_lengths(cuda_device, tmp_path, lengths):
    frame = _check(tmp_path, scene="rtigo3_geometry", resolution="72 40", samplesSqrt=2, pathLengths=lengths, iterations=3)
    if lengths == "0 0":
        assert not frame[..., :3].any() and np.all(frame[..., 3] == 1.0)     # no segment is traced: black, alpha 1


def test_empty_scene_shows_the_environment(cuda_device, tmp_path):
    scene = os.path.join(str(tmp_path), "scene_empty.txt")
    with open(scene, "w") as f:
        f.write("albedo 1 1 1\nmaterial default brdf_diffuse\n")
    frame = _check(tmp_path, scene="rtigo3_geometry", scene_file=scene, resolution="40 24", samplesSqrt=2, light=0, miss=1, iterations=2)
    assert np.all(frame[..., :3] == 1.0)                                     # constant white environment, nothing in front of it


def test_more_paths_than_one_batch(cuda_device, tmp_path, monkeypatch):
    """RTC_MAX_PATHS forces several batches per enqueue; the running average must not depend on the batching."""
    monkeypatch.setenv("RTC_MAX_PATHS", str(64 * 36 * 3))
    a = _check(tmp_path, scene="rtigo3_geometry", resolution="64 36", samplesSqrt=4, iterations=10)
    monkeypatch.delenv("RTC_MAX_PATHS")
    b = _check(tmp_path, scene="rtigo3_geometry", resolution="64 36", samplesSqrt=4, iterations=10)
    assert a.tobytes() == b.tobytes()


def test_roofline_probes(cuda_device):
    """The denominators bench.py reports fractions against are measured by kernels of this library: they must be in the range
    a B200 can deliver."""
    from tweeker_raytracer_b200 import core
    ctx = core.Context(0)
    try:
        l2 = ctx.probe_gather(32 << 20, 64)
        fp32 = ctx.probe_pipes(0)
        issue = ctx.probe_pipes(1)
        assert 500.0 < l2 < 20000.0          # GB/s of random 16-byte gathers out of L2
        assert 20.0 < fp32 < 90.0            # TFLOP/s: 148 SMs x 128 lanes x 2 x ~1.9 GHz = 72
        assert 400.0 < issue < 1300.0        # 1e9 warp instructions per second: 148 SMs x 4 schedulers x ~1.9 GHz = 1125
    finally:
        ctx.close()


def test_shading_arithmetic_bit_identical_to_the_host_build(cuda_device, tmp_path):
    """include/rt_portable_math.h is shared by the oracle and the shading kernels: a frame comparison alone would not notice
    the two compilers disagreeing on an input no test scene produces.  Here the device evaluates every pinned transcendental,
    IEEE division / square root and an uncontracted multiply-add (rtc_probe_math: the shading translation unit's flags) over
    dense and random inputs, and every result must carry the bits gcc's build of the same header produces.  (The header is
    checked against float64 libm independently, tests/test_cpu_portable_math.py.)"""
    from tweeker_raytracer_b200 import core
    pm = H.portable_math_lib(tmp_path)
    rng = np.random.default_rng(2024)
    n = 1 << 20
    wide = (rng.normal(size=n) * 10.0 ** rng.integers(-12, 12, size=n)).astype(np.float32)
    wide2 = (rng.normal(size=n) * 10.0 ** rng.integers(-12, 12, size=n)).astype(np.float32)
    unit = rng.uniform(-1.0, 1.0, size=n).astype(np.float32)
    cases = {
        "sin": [(np.linspace(-4 * np.pi, 4 * np.pi, n), None), (rng.uniform(-1e5, 1e5, size=n), None), (wide[np.abs(wide) < 1e8], None)],
        "cos": [(np.linspace(-4 * np.pi, 4 * np.pi, n), None), (rng.uniform(-1e5, 1e5, size=n), None), (wide[np.abs(wide) < 1e8], None)],
        "atan": [(np.linspace(-50, 50, n), None), (wide, None), (np.array([0.0, -0.0, 1.0, -1.0, 2.414213562373095, 0.4142135623730950]), None)],
        "atan2": [(wide, wide2), (unit, rng.uniform(-1.0, 1.0, size=n)), (np.array([0.0, 1.0, -1.0, 0.0, 0.0]), np.array([0.0, 0.0, 0.0, -1.0, 1.0]))],
        "acos": [(np.linspace(-1, 1, n), None), (unit, None), (np.array([1.0000001, -1.0000001, 1.0, -1.0, 0.5, -0.5, 0.0, 1e-5]), None)],
        "exp": [(np.linspace(-85, 88.7, n), None), (rng.normal(size=n), None), (np.array([0.0, -0.0, 100.0, -200.0, 88.72283, -103.0]), None)],
        "log": [(np.abs(wide) + 1e-30, None), (np.linspace(0.5, 2.0, n), None), (np.array([1.0, 0.0, -1.0, np.inf, 1e-40, 3.4e38]), None)],
        "pow": [(rng.uniform(0, 4, size=n), np.full(n, 1.0 / 2.2)), (rng.uniform(0, 4, size=n), rng.uniform(0.1, 3.0, size=n)), (np.array([0.0, -1.0, 1.0]), np.array([2.0, 2.0, 2.2]))],
        "div": [(wide, np.where(wide2 == 0, 1.0, wide2)), (unit, rng.uniform(0.5, 2.0, size=n))],
        "sqrt": [(np.abs(wide), None), (np.linspace(0, 4, n), None)],
        "muladd": [(wide, wide2), (unit, rng.uniform(-1.0, 1.0, size=n))],
    }
    assert sorted(cases) == sorted(core.MATH_FUNCTIONS)
    ctx = core.Context(0)
    try:
        for name, inputs in cases.items():
            for x, y in inputs:
                x = np.ascontiguousarray(x, dtype=np.float32)
                y = None if y is None else np.ascontiguousarray(y, dtype=np.float32)
                got = ctx.probe_math(name, x, y)
                want = H.portable_math_call(pm, name, x, y)
                same = got.view(np.uint32) == want.view(np.uint32)
                assert same.all(), (name, x[~same][:4], got[~same][:4], want[~same][:4])
    finally:
        ctx.close()
