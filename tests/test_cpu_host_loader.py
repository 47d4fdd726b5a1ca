"""Host side (no GPU): tokenizer, the two description formats, tessellators, index semantics, tile partition."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers as H
from oracle import orc
from tweeker_raytracer_b200 import core, host, partition


def load(tmp, scene_text=None, name="rtigo3_cornell_box", **overrides):
    sysfile = H.write_system(tmp, name, **overrides)
    if scene_text is None:
        scene = H.scene_path(name)
    else:
        scene = os.path.join(str(tmp), "scene.txt")
        with open(scene, "w") as f:
            f.write(scene_text)
    return host.App(sysfile, scene, host_only=True)


def test_libraries_export_every_declared_symbol(built):
    L = core.lib()
    missing = [s for s in core.SYMBOLS if not hasattr(L, s)]
    assert not missing
    # every function rtc_core.h declares is in the list (the header is the contract)
    import re
    with open(os.path.join(H.ROOT, "include", "rtc_core.h")) as f:
        declared = set(re.findall(r"\b(rtc_[a-z_0-9]+)\s*\(", f.read()))
    declared -= {"rtc_trace"}
    assert declared <= set(core.SYMBOLS), declared - set(core.SYMBOLS)
    Hh = host.lib()
    assert not [s for s in host.SYMBOLS if not hasattr(Hh, s)]
    assert L.rtc_version() == 102


def test_stats_layout_matches_the_header(tmp_path):
    """core.Stats is read through rtc_stats_get, which writes sizeof(rtc_stats) bytes: the binding must have the C compiler's
    layout of include/rtc_core.h, field for field."""
    import subprocess
    names = [name for name, _ in core.Stats._fields_]
    src = os.path.join(str(tmp_path), "layout.c")
    with open(src, "w") as f:
        f.write('#include <stdio.h>\n#include "rtc_core.h"\nint main(void) {\n  printf("%zu\\n", sizeof(rtc_stats));\n')
        f.writelines('  printf("%%zu\\n", offsetof(rtc_stats, %s));\n' % n for n in names)
        f.write("  return 0;\n}\n")
    exe = os.path.join(str(tmp_path), "layout")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I" + os.path.join(H.ROOT, "include"), "-o", exe, src])
    got = [int(v) for v in subprocess.check_output([exe]).split()]
    assert got == [C.sizeof(core.Stats)] + [getattr(core.Stats, n).offset for n in names]
    assert names[-1] == "cutoutGraphBuilds" and C.sizeof(core.Stats) == 56


def test_struct_layouts_match_the_reference_contract(built):
    assert C.sizeof(host.SystemData) == 192 and host.SystemData.topObject.offset == 16 and host.SystemData.resolution.offset == 96
    assert host.SystemData.iterationIndex.offset == 140 and host.SystemData.envRotation.offset == 184
    assert C.sizeof(host.CompositorData) == 56
    assert host.ATTR_DTYPE.itemsize == 48 and host.MATERIAL_DTYPE.itemsize == 64 and host.LIGHT_DTYPE.itemsize == 80
    assert host.MATERIAL_DTYPE.fields["albedo"][1] == 28 and host.MATERIAL_DTYPE.fields["flags"][1] == 56
    assert host.LIGHT_DTYPE.fields["area"][1] == 52 and host.LIGHT_DTYPE.fields["emission"][1] == 56
    assert core.INSTANCE_DTYPE.itemsize == 64 and core.RAY_DTYPE.itemsize == 32 and core.HIT_DTYPE.itemsize == 20


def test_no_gpu_means_loud_failure_not_fallback(built, tmp_path):
    if core.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(core.RtcError):
        core.Context(0)
    with pytest.raises(core.RtcError):
        host.App(H.write_system(tmp_path, "rtigo3_cornell_box"), H.scene_path("rtigo3_cornell_box"))


def test_cornell_box_index_semantics(built, tmp_path):
    app = load(tmp_path)
    i = app.info
    assert (i.resolutionX, i.resolutionY, i.samplesSqrt, i.miss, i.lightMode, i.strategy) == (512, 512, 4, 0, 1, 0)
    # the area light is created before the scene file is read: material 0, geometry 0, instance 0 (Application.cpp:636-676)
    assert (i.numGeometries, i.numInstances, i.numMaterials, i.numLights) == (5, 8, 7, 1)
    t, g, m, l = app.instance(0)
    assert (g, m, l) == (0, 0, 0) and np.array_equal(t, np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], dtype=np.float32))
    mats = app.materials()
    assert mats["indexBSDF"].tolist() == [1, 0, 0, 0, 0, 1, 2]              # area light, white, default, red, green, mirror, glass
    assert mats["flags"][0] == 0x20 and np.all(mats["albedo"][0] == 0)     # thin-walled black specular
    assert np.allclose(mats["albedo"][3], (0.8, 0.05, 0.05)) and mats["ior"][6] == 1.5
    lights = app.lights()
    assert lights["type"][0] == 1 and lights["area"][0] == 1.0 and np.allclose(lights["normal"][0], (0, -1, 0))
    assert np.allclose(lights["position"][0], (-0.5, 1.95, -0.5)) and np.allclose(lights["emission"][0], 10)
    # both spheres share one geometry (cache key sphere_180_90_1), 2*180*89 triangles
    assert app.instance(6)[1] == app.instance(7)[1] == 4
    attrs, idx = app.geometry(4)
    assert len(attrs) == 181 * 90 and len(idx) == 2 * 180 * 89 == 32040
    s = app.system_data()
    assert abs(s.sceneEpsilon - 500 * 1e-7) < 1e-10 and (s.pathLengths.x, s.pathLengths.y) == (2, 5) and s.numLights == 1
    assert (s.tileShift.x, s.tileShift.y) == (3, 3) and s.distribution == 0
    cam = app.camera()
    assert np.allclose(cam["P"][0], (0, 1, 3.6), atol=1e-6) and np.allclose(cam["W"][0], (0, 0, -1), atol=1e-6)
    app.close()


def test_light_and_miss_combinations(built, tmp_path):
    # miss 1|2 put the environment light at index 0 and the quad at 1; miss 0 + light 0 leaves no lights at all
    app = load(tmp_path, miss=1)
    assert app.lights()["type"].tolist() == [0, 1] and app.instance(0)[3] == 1
    app.close()
    app = load(tmp_path, miss=0, light=0)
    assert app.info.numLights == 0 and app.info.numInstances == 7 and app.materials()["indexBSDF"].tolist() == [0, 0, 0, 0, 1, 2]
    app.close()
    app = load(tmp_path, light=7)            # clamped to 2: the 4x4 quad at y = 4
    l = app.lights()
    assert l["area"][0] == 16.0 and np.allclose(l["position"][0], (-2, 4, -2))
    app.close()


def test_tessellator_counts_and_order(built, tmp_path):
    text = ("material default brdf_diffuse\nmodel box default\nmodel plane 3 2 1 default\nmodel plane 1 1 0 default\n"
            "model sphere 8 5 1.0 default\nmodel sphere 8 5 0.5 default\nmodel torus 6 4 0.75 0.25 default\nmodel box default\n")
    app = load(tmp_path, text, light=0)
    assert app.info.numGeometries == 6 and app.info.numInstances == 7     # the second box reuses box_1_1
    a, i = app.geometry(0)
    assert len(a) == 24 and len(i) == 12
    assert i[:2].tolist() == [[0, 1, 2], [2, 3, 0]] and np.allclose(a["normal"][0], (-1, 0, 0)) and np.allclose(a["normal"][20], (0, 1, 0))
    assert np.allclose(a["vertex"][:4], [(-1, -1, -1), (-1, -1, 1), (-1, 1, 1), (-1, 1, -1)])
    a, i = app.geometry(1)
    assert len(a) == 4 * 3 and len(i) == 2 * 3 * 2 and i[0].tolist() == [0, 1, 5] and i[1].tolist() == [5, 4, 0]
    assert np.allclose(a["vertex"][0], (-1, 0, 1)) and np.allclose(a["vertex"][-1], (1, 0, -1)) and np.allclose(a["normal"][0], (0, 1, 0))
    a, i = app.geometry(2)
    assert np.allclose(a["vertex"][0], (0, -1, 1)) and np.allclose(a["tangent"][0], (0, 0, -1))
    a, i = app.geometry(3)
    assert len(a) == 9 * 5 and len(i) == 2 * 8 * 4 and np.allclose(a["vertex"][0], (0, -1, 0), atol=1e-6)     # south pole first
    assert np.allclose(np.linalg.norm(a["vertex"], axis=1), 1, atol=1e-6)
    a, _ = app.geometry(4)
    assert a["vertex"][:, 1].max() < 1e-6                                    # thetaMax 0.5: lower hemisphere only
    a, i = app.geometry(5)
    assert len(a) == 7 * 5 and len(i) == 2 * 6 * 4 and np.allclose(a["vertex"][0], (1.0, 0, 0), atol=1e-6)
    app.close()


def test_transform_stack_applies_in_file_order(built, tmp_path):
    text = ("material default brdf_diffuse\nidentity\npush scale 2 2 2 translate 1 0 0 model box default pop\n"
            "push translate 1 0 0 scale 2 2 2 model box default pop\npush rotate 0 1 0 90 translate 0 0 5 model box default pop\n"
            "pop model box default\n")
    app = load(tmp_path, text, light=0)
    assert np.allclose(app.instance(0)[0], [2, 0, 0, 1, 0, 2, 0, 0, 0, 0, 2, 0])        # scale first, then translate
    assert np.allclose(app.instance(1)[0], [2, 0, 0, 2, 0, 2, 0, 0, 0, 0, 2, 0])        # translate first, then scale
    t = app.instance(2)[0].reshape(3, 4)
    assert np.allclose(t[:, :3] @ np.array([1, 0, 0]), (0, 0, -1), atol=1e-6) and np.allclose(t[:, 3], (0, 0, 5))
    assert np.allclose(app.instance(3)[0], [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0])        # pop on an empty stack resets to identity
    app.close()


def test_parser_comments_values_and_unknown_tokens(built, tmp_path):
    text = ("# comment line\nalbedo 0.25 .5 +1e0   # trailing comment\nmaterial a brdf_ggx_smith\nfoo bar\nroughness 0.3 0.2\r\n"
            "absorption 0.5 0.5 0.5 absorptionScale 2 ior 1.33 thinwalled 1 material b bsdf_specular material a brdf_diffuse\n"
            "model box nosuchmaterial\nmodel box b\n")
    app = load(tmp_path, text, light=0)
    m = app.materials()
    assert len(m) == 3 and np.allclose(m["albedo"][0], (0.25, 0.5, 1.0)) and m["indexBSDF"].tolist() == [3, 2, 0]
    assert np.allclose(m["roughness"][1], (0.3, 0.2)) and m["flags"][1] == 0x20 and abs(m["ior"][1] - 1.33) < 1e-6
    assert np.allclose(m["absorption"][1], -np.log(0.5) * 2, rtol=1e-6) and np.all(m["absorption"][0] == 0)
    assert app.instance(0)[2] == -1         # unknown reference and no `default` material: stays -1 as in the reference
    assert app.instance(1)[2] == 1
    app.close()


def test_system_description_fallbacks(built, tmp_path):
    app = load(tmp_path, tileSize="12 16", lensShader=9, strategy=7, resolution="0 -3", samplesSqrt=0)
    s = app.system_data()
    assert (s.tileSize.x, s.tileSize.y) == (8, 16) and (s.tileShift.x, s.tileShift.y) == (3, 4)
    assert s.lensShader == 0 and app.info.strategy == 0 and app.resolution == (1, 1) and app.info.samplesSqrt == 1
    app.close()
    with pytest.raises(core.RtcError):
        host.App(os.path.join(str(tmp_path), "does_not_exist.txt"), H.scene_path("rtigo3_cornell_box"), host_only=True)


@pytest.mark.parametrize("count,width,tile", [(2, 100, 8), (3, 100, 8), (4, 1920, 16), (8, 3840, 8), (5, 37, 4)])
def test_tile_partition_owns_every_pixel_exactly_once(count, width, tile):
    shift = partition.tile_shift(tile)
    lw = partition.tiled_launch_width(width, count, tile)
    assert lw % tile == 0 and lw * count >= width
    for y in (0, tile - 1, tile, 5 * tile + 1):
        owners = np.zeros(width, dtype=int)
        for d in range(count):
            for x in range(lw):
                col = partition.distribute(x, y, d, count, tile, shift, shift)
                if col < width:
                    owners[col] += 1
        assert (owners == 1).all()


def test_oracle_generate_primary_follows_the_partition(built, tmp_path):
    app = load(tmp_path, resolution="40 16", tileSize="8 8")
    scene = H.oracle_scene(app)
    sysd = H.oracle_sys(app)
    lw = partition.tiled_launch_width(40, 3, 8)
    skipped = 0
    for d in range(3):
        sysd.deviceCount, sysd.deviceIndex, sysd.distribution = 3, d, 1
        rays = scene.generate_primary(sysd, lw, 16, 0).reshape(16, lw)
        for y in range(16):
            for x in range(lw):
                col = partition.distribute(x, y, d, 3, 8, 3, 3)
                assert (rays[y, x]["tmax"] < 0) == (col >= 40)
                skipped += col >= 40
    assert skipped == (3 * lw - 40) * 16
    app.close()


def test_environment_cdfs_are_distributions(built, tmp_path):
    app = load(tmp_path, name="rtigo3_geometry", miss=2, envMap="procedural 64 32", resolution="8 8")
    texels, cdf_u, cdf_v, integral = app.environment()
    assert texels.shape == (32, 64, 4) and cdf_u.shape == (32, 65) and cdf_v.shape == (33,)
    assert np.all(cdf_u[:, 0] == 0) and np.allclose(cdf_u[:, -1], 1) and cdf_v[0] == 0 and abs(cdf_v[-1] - 1) < 1e-6
    assert np.all(np.diff(cdf_u, axis=1) >= 0) and np.all(np.diff(cdf_v) >= 0) and integral > 0
    # integral = mean over the sphere of (r+g+b)/3 times 4 pi, by the reference's quadrature
    sin_t = np.sin(np.pi * (np.arange(32) + 0.5) / 32)[:, None]
    want = float((texels[..., :3].sum(axis=2) / 3 * sin_t).sum() * 2 * np.pi * np.pi / (64 * 32))
    assert abs(integral - want) / want < 1e-4
    assert app.system_data().envWidth == 64
    app.close()


def test_radiance_hdr_file_round_trip(built, tmp_path):
    # flat RGBE file, 8 x 4, written here; the loader flips it so row 0 is the south pole
    w, h = 8, 4
    img = np.zeros((h, w, 3), dtype=np.float32)
    img[0, :, 0] = 2.0      # top row of the file = up = last row in memory
    img[3, :, 2] = 0.5
    path = os.path.join(str(tmp_path), "env.hdr")
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n-Y %d +X %d\n" % (h, w))
        for y in range(h):
            for x in range(w):
                m = img[y, x].max()
                if m < 1e-32:
                    f.write(bytes(4))
                else:
                    e = int(np.floor(np.log2(m))) + 1
                    s = 256.0 / (2.0 ** e)
                    f.write(bytes([int(img[y, x, 0] * s), int(img[y, x, 1] * s), int(img[y, x, 2] * s), e + 128]))
    app = load(tmp_path, name="rtigo3_geometry", miss=2, envMap=path, resolution="8 8")
    texels = app.environment()[0]
    assert texels.shape == (4, 8, 4)
    assert np.allclose(texels[3, :, 0], 2.0) and np.allclose(texels[0, :, 2], 0.5) and np.allclose(texels[1], [0, 0, 0, 1])
    app.close()


def test_save_system_description_round_trip(built, tmp_path):
    app = load(tmp_path, name="rtigo3_geometry", resolution="320 180", envRotation=0.25, composite=1, textureCutout="./my_slots.png")
    app.set_camera(0.6, 0.4, 35.0, 7.5, (0.5, 1.5, -0.25))
    path = app.save_system(os.path.join(str(tmp_path), "saved_system.txt"))
    assert path and os.path.exists(path)
    text = open(path).read()
    for line in ("strategy 0", "resolution 320 180", "samplesSqrt 16", "miss 1", "light 2", "pathLengths 2 6", "envRotation 0.25",
                 "camera 0.6 0.4 35 7.5", "center 0.5 1.5 -0.25", "composite 1", "batchIterations 32", "textureCutout ./my_slots.png"):
        assert line in text, line
    assert "textureAlbedo" not in text          # the reference's hard-coded default is not written out
    again = host.App(path, H.scene_path("rtigo3_geometry"), host_only=True)
    a, b = app.system_data(), again.system_data()
    assert bytes(a) == bytes(b)
    assert app.camera().tobytes() == again.camera().tobytes()
    assert bytes(app.tonemapper()) == bytes(again.tonemapper())
    app.close()
    again.close()


# ---- the environment CDF builder against the reference's own Texture::calculateSphericalCDF ------------------------------
def _env_case(tmp_path, key):
    if key.startswith("procedural"):
        spec = "procedural " + key.split("_")[1].replace("x", " ")
    else:
        spec = H.write_rgbe_hdr(os.path.join(str(tmp_path), "random.hdr"), H.random_rgbe(48, 24, 20261018))
    app = load(tmp_path, name="rtigo3_geometry", miss=2, envMap=spec, resolution="8 8")
    env = app.environment()
    app.close()
    return env


@pytest.mark.parametrize("key", ["procedural_64x32", "procedural_256x128", "random_48x24"])
def test_environment_cdf_equals_reference_golden(built, tmp_path, key):
    """host/EnvMap.cpp restates Texture.cpp:1500-1645; tests/golden/reference_envcdf.npz holds the outputs of the reference's own
    function (compiled where it lies, tests/golden/make_golden_envcdf.py) on the same texels: bit-exact."""
    gold = np.load(os.path.join(H.ROOT, "tests", "golden", "reference_envcdf.npz"))
    texels, cdf_u, cdf_v, integral = _env_case(tmp_path, key)
    assert texels.tobytes() == gold[key + "_texels"].tobytes()          # same input (procedural sky / .hdr reader)
    assert cdf_u.tobytes() == gold[key + "_cdf_u"].tobytes()
    assert cdf_v.tobytes() == gold[key + "_cdf_v"].tobytes()
    assert np.float32(integral).tobytes() == gold[key + "_integral"].tobytes()
    if key == "random_48x24":
        equal = np.arange(49, dtype=np.float32) / np.float32(48)                # a row that is black after filtering: equal distribution
        assert any(np.array_equal(row, equal) for row in cdf_u)


def test_environment_cdf_of_a_run_length_encoded_hdr_equals_reference_golden(built, tmp_path):
    """The random map of the test above written with run-length encoded scanlines: the reader's RLE path must give the same
    texels, and the CDFs must equal what the reference's own function returned for them (tests/golden/reference_envcdf.npz)."""
    gold = np.load(os.path.join(H.ROOT, "tests", "golden", "reference_envcdf.npz"))
    spec = H.write_rgbe_hdr(os.path.join(str(tmp_path), "random_rle.hdr"), H.random_rgbe(48, 24, 20261018), rle=True)
    app = load(tmp_path, name="rtigo3_geometry", miss=2, envMap=spec, resolution="8 8")
    texels, cdf_u, cdf_v, integral = app.environment()
    app.close()
    assert texels.tobytes() == gold["random_48x24_texels"].tobytes()
    u, v, i = gold["random_48x24_cdf_u"], gold["random_48x24_cdf_v"], gold["random_48x24_integral"]
    assert cdf_u.tobytes() == u.tobytes() and cdf_v.tobytes() == v.tobytes() and np.float32(integral).tobytes() == np.float32(i).tobytes()
