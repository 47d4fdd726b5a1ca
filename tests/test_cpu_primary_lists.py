"""Tile lists of the primary rays (csrc/primary_lists.cuh) on the CPU: the list builder and the list pass compiled unchanged by g++
together with the ray generation (csrc/shade.cuh) and the traversal (csrc/trace.cuh) -- tests/native/primary_lists_host.cpp --
and held to the traversal bit for bit.

For every primary ray of a pinhole launch, the split depth-0 extend (the list pass on a tile whose list fits, the traversal on a
tile that overflowed) must give the traversal's (t, u, v, instance, primitive): on the geometry scene at 1920x1080 with the
benchmark's camera, on random cameras (grazing views of the floor among them), at a field of view of a few degrees (the tile's
own angle is then tiny), with instances squashed to the conditioning limit the builder accepts and beyond it, on the Cornell box
and on a small instanced scene, and with the list capacity forced down to 4 so that both kinds of tile occur in every scene."""
import os
import sys

import numpy as np
import pytest

import helpers as H
from tile_lists import OVERFLOW, lists_lib, load, primary


def check(app, export, w, h, iteration=0, k=None):
    got, want, counts, _ = primary(app, export, w, h, iteration, k)
    assert H.hits_equal(got, want)
    return counts, want


def test_geometry_scene_at_1080p_with_the_benchmark_camera(built, tmp_path):
    app, export = load(tmp_path, "rtigo3_geometry", "1920 1080")
    counts, hits = check(app, export, 1920, 1080, iteration=5)
    listed = counts != OVERFLOW
    assert listed.mean() > 0.9                               # most tiles are traced through their list
    assert (counts[listed] == 0).any() and (counts[listed] > 2).any()
    assert (hits["inst"] != 0xFFFFFFFF).mean() > 0.3
    app.close()


@pytest.mark.parametrize("seed", range(6))
def test_geometry_scene_from_random_cameras(built, tmp_path, seed):
    """Cameras all around the scene; seeds 0 and 1 look along the floor from just above it (the floor is seen edge-on at the
    horizon), the others from anywhere within the scene's reach."""
    rng = np.random.default_rng(seed)
    app, export = load(tmp_path, "rtigo3_geometry", "320 180")
    phi = float(rng.uniform(0.0, 1.0))
    if seed < 2:
        theta, distance, center = 0.5 + float(rng.uniform(-1e-3, 1e-3)), float(rng.uniform(3.0, 12.0)), (float(rng.uniform(-1, 1)), 1e-3 * (seed + 1), 0.0)
    else:
        theta, distance, center = float(rng.uniform(0.05, 0.95)), float(rng.uniform(0.5, 15.0)), tuple(float(v) for v in rng.uniform(-2.0, 2.0, 3))
    app.set_camera(phi, theta, float(rng.uniform(20.0, 90.0)), distance, center)
    check(app, export, 320, 180, iteration=seed)
    check(app, export, 320, 180, iteration=seed, k=4)
    app.close()


@pytest.mark.parametrize("fov", [3.0, 1.0])
def test_narrow_field_of_view_at_1080p(built, tmp_path, fov):
    """A tile then spans a few arc seconds: its side planes must still be exact to far below the padding."""
    app, export = load(tmp_path, "rtigo3_geometry", "1920 1080")
    app.set_camera(0.81, 0.55, fov, 10.0, (1.2, 0.5, -0.4))
    counts, hits = check(app, export, 1920, 1080, iteration=2)
    assert (counts != OVERFLOW).mean() > 0.5 and (hits["inst"] != 0xFFFFFFFF).mean() > 0.3
    app.close()


def squashed(transform, scale, rot):
    """transform (3x4 object->world, 12 floats) applied after squashing object space along z by `scale` and rotating it by rot."""
    t = np.asarray(transform, dtype=np.float64).reshape(3, 4)
    a = t[:, :3] @ rot @ np.diag([1.0, 1.0, scale]) @ rot.T
    return np.concatenate([a, t[:, 3:]], axis=1).astype(np.float32).ravel()


@pytest.mark.parametrize("scale", [1.0 / 40.0, 1.0 / 200.0])
def test_squashed_instances_at_1080p(built, tmp_path, scale):
    """Every instance of the geometry scene squashed by `scale` along a random object-space axis: |M|_F |M^-1|_F about 57 (the
    builder lists such instances) and 280 (beyond its limit of 64: tiles that meet one are traced by the traversal)."""
    from tweeker_raytracer_b200 import core
    app, _ = load(tmp_path, "rtigo3_geometry", "1920 1080")
    rng = np.random.default_rng(7)
    rot, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    geos = [app.geometry(g) for g in range(app.info.numGeometries)]
    insts = [(squashed(t, scale, rot), g) for t, g in (app.instance(i)[:2] for i in range(app.info.numInstances))]
    export, _ = core.host_scene_export(geos, insts)
    counts, hits = check(app, export, 1920, 1080)
    assert (hits["inst"] != 0xFFFFFFFF).mean() > 0.02
    if scale > 1.0 / 64.0:
        assert ((counts != OVERFLOW) & (counts > 0)).any()
    app.close()


def test_cornell_box(built, tmp_path):
    app, export = load(tmp_path, "rtigo3_cornell_box", "256 256")
    counts, _ = check(app, export, 256, 256)
    assert (counts != OVERFLOW).mean() > 0.5
    app.close()


def test_small_instanced_scene(built, tmp_path):
    sys.path.insert(0, os.path.join(H.ROOT, "tools"))
    import make_instances_scene
    scene = os.path.join(str(tmp_path), "scene_lattice.txt")
    make_instances_scene.write_scene(scene, count=64, tess=(24, 12))
    app, export = load(tmp_path, "rtigo3_instances", "320 240", scene=scene)
    counts, hits = check(app, export, 320, 240)
    assert (counts != OVERFLOW).any() and (hits["inst"] != 0xFFFFFFFF).any()
    app.close()


def test_small_capacity_splits_every_scene_into_listed_and_overflowed_tiles(built, tmp_path):
    assert lists_lib(4).pl_list_capacity() == 4
    for name, res in (("rtigo3_geometry", "480 272"), ("rtigo3_cornell_box", "128 128")):
        app, export = load(tmp_path, name, res)
        w, h = (int(v) for v in res.split())
        counts, _ = check(app, export, w, h, k=4)
        assert (counts == OVERFLOW).any() and ((counts != OVERFLOW) & (counts > 0)).any()
        app.close()
