"""Pins of the oracle (no GPU).  The oracle is only trusted because it reproduces THE REFERENCE'S OWN arithmetic:
tests/golden/reference_frames.npz and reference_rng.json were produced by the reference's shader sources compiled for
the host (tests/golden/make_golden.py, oracle/ref_driver.cpp); where oracle/_ref/libref.so is available the comparison
is also made live.  The libm build of the oracle must match bit for bit; the pinned-arithmetic build (the one the GPU is
compared with) differs from it only in the last bits of sin/cos/atan/acos/exp and must agree statistically."""
import json
import os

import numpy as np
import pytest

import helpers as H
from golden import make_golden
from oracle import orc
from tweeker_raytracer_b200 import host, partition

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def golden_frames():
    return np.load(os.path.join(GOLDEN, "reference_frames.npz"))


def render_case(tmp, key, variant):
    name, overrides, iterations = make_golden.CASES[key]
    app = host.App(H.write_system(tmp, name, **overrides), H.scene_path(name), host_only=True)
    scene = H.oracle_scene(app, variant)
    sysd = H.oracle_sys(app)
    w, h = app.resolution
    out = {}
    if "tiled" in key:
        lw = partition.tiled_launch_width(w, 3, sysd.tileSize.x)
        for index in range(3):
            sysd.deviceCount, sysd.deviceIndex, sysd.distribution = 3, index, 1
            out["%s_dev%d" % (key, index)] = scene.render(sysd, app.info.miss, lw, h, local_copy=True, iter_count=iterations, threads=2).reshape(h, lw, 4)
    else:
        out[key] = scene.render(sysd, app.info.miss, w, h, iter_count=iterations, threads=2).reshape(h, w, 4)
    return out, app, scene, sysd


@pytest.mark.parametrize("key", sorted(make_golden.CASES))
def test_libm_oracle_reproduces_reference_frames(built, tmp_path, golden_frames, key):
    got, app, _, _ = render_case(tmp_path, key, "libm")
    for k, frame in got.items():
        want = golden_frames[k]
        assert frame.shape == want.shape
        # same libm, same operation order -> identical bits; a different glibc may move the last bit of a transcendental
        identical = float((frame.view(np.uint32) == want.view(np.uint32)).mean())
        assert identical > 0.999, "%s: only %.4f of the values are bit-identical to the reference" % (k, identical)
        assert np.allclose(frame, want, rtol=1e-5, atol=1e-6)
    app.close()


@pytest.mark.parametrize("key", ["cornell_32x32_4spp", "geometry_env_48x27_4spp", "textures_64x36_4spp", "textures_rr_env_48x27_3spp"])
def test_libm_oracle_equals_reference_frames_bit_for_bit(built, tmp_path, golden_frames, key):
    """Bit for bit against the frames the reference's own device programs rendered for these cases (orc.Reference.render,
    stored by tests/golden/make_golden.py): the libm oracle and the host-compiled reference share arithmetic and libm, so no
    last bit may move (a C library whose transcendentals round differently shows up here first)."""
    got, app, _, _ = render_case(tmp_path, key, "libm")
    assert got[key].tobytes() == golden_frames[key].tobytes()
    app.close()


def test_rng_known_answers_from_reference(built):
    with open(os.path.join(GOLDEN, "reference_rng.json")) as f:
        g = json.load(f)
    for a, b, want in g["tea4"]:
        assert orc.tea4(a, b) == want
    for row in g["lcg"]:
        seq, state = orc.rng_sequence(row["seed"], len(row["samples_hex"]))
        assert state == row["state"]
        assert [float(np.float32(x)).hex() for x in seq] == row["samples_hex"]
        assert all(0.0 <= x < 1.0 for x in seq)


def test_pinned_oracle_agrees_with_libm_oracle(built, tmp_path):
    # the GPU is compared with the pinned build; the reference with the libm build: tie the two together
    name, overrides = "rtigo3_cornell_box", dict(resolution="48 48", samplesSqrt=8)
    app = host.App(H.write_system(tmp_path, name, **overrides), H.scene_path(name), host_only=True)
    sysd = H.oracle_sys(app)
    a = H.oracle_scene(app, "pinned").render(sysd, app.info.miss, 48, 48, iter_count=64)
    b = H.oracle_scene(app, "libm").render(sysd, app.info.miss, 48, 48, iter_count=64)
    same = float((a.view(np.uint32) == b.view(np.uint32)).all(axis=1).mean())
    assert same > 0.5                        # most pixels never see a differing transcendental bit
    assert H.psnr(np.clip(a[:, :3], 0, 1), np.clip(b[:, :3], 0, 1)) > 40.0
    assert abs(float(a[:, :3].mean()) - float(b[:, :3].mean())) < 2e-3
    app.close()


def test_geometry_scene_pinned_vs_libm_psnr(built, tmp_path):
    name, overrides = "rtigo3_geometry", dict(resolution="64 36", samplesSqrt=6)
    app = host.App(H.write_system(tmp_path, name, **overrides), H.scene_path(name), host_only=True)
    sysd = H.oracle_sys(app)
    a = H.oracle_scene(app, "pinned").render(sysd, app.info.miss, 64, 36, iter_count=36)
    b = H.oracle_scene(app, "libm").render(sysd, app.info.miss, 64, 36, iter_count=36)
    assert H.psnr(np.clip(a[:, :3], 0, 1), np.clip(b[:, :3], 0, 1)) > 40.0
    app.close()


@pytest.mark.parametrize("key", ["geometry_converged_96x54_256spp", "cornell_converged_64x64_256spp"])
def test_converged_frames_reach_40_db_against_the_reference(built, tmp_path, golden_frames, key):
    """BASELINE.json's image check: converged frames at PSNR >= 40 dB against the reference's output.  The reference here is its
    own device code compiled for the host (libm transcendentals); the frame compared is the pinned-arithmetic oracle's, which
    the GPU reproduces bit for bit (tests/test_gpu_render_parity.py), so this bounds the GPU image as well."""
    got, app, _, _ = render_case(tmp_path, key, "pinned")
    want = golden_frames[key]
    a, b = np.clip(got[key][..., :3], 0.0, 1.0), np.clip(want[..., :3], 0.0, 1.0)
    assert H.psnr(a, b) >= 40.0, H.psnr(a, b)
    assert abs(float(a.mean()) - float(b.mean())) < 2e-3
    app.close()


@pytest.mark.skipif(not (os.path.exists(orc.REF_LIB) or os.path.isdir(orc.REFERENCE_SHADERS)), reason="host-compiled reference not available")
@pytest.mark.parametrize("seed", [0, 1, 2, 3, 4, 5])
def test_random_scenes_equal_live_reference(built, tmp_path, seed):
    """Randomly generated scenes (the generator of tests/test_gpu_fuzz.py), half of them with albedo and cutout textures: the
    libm oracle must reproduce the reference's own device programs bit for bit, any-hit programs included."""
    import test_gpu_fuzz as fuzz
    rng = np.random.default_rng(7000 + seed)
    scene_file = os.path.join(str(tmp_path), "scene_fuzz.txt")
    fuzz.random_scene(scene_file, rng, textures=bool(seed & 1))
    miss = int(rng.integers(0, 3))
    overrides = dict(resolution="40 24", samplesSqrt=2, miss=miss, light=int(rng.integers(0 if miss else 1, 3)),
                     lensShader=int(rng.integers(0, 3)), pathLengths="%d %d" % (int(rng.integers(0, 3)), int(rng.integers(2, 9))),
                     envMap="procedural 64 32", envRotation="%.3f" % rng.uniform(0, 1))
    app = host.App(H.write_system(tmp_path, "rtigo3_textures", **overrides), scene_file, host_only=True)
    scene = H.oracle_scene(app, "libm")
    sysd = H.oracle_sys(app)
    got = scene.render(sysd, app.info.miss, 40, 24, iter_count=3, threads=2)
    want = orc.Reference(scene, app.info.miss).render(sysd, 40, 24, iter_count=3)
    assert got.tobytes() == want.tobytes()
    app.close()
