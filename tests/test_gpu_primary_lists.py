"""Tile lists of the primary rays on a B200: frames of pinhole launches, whose depth-0 extend runs through the per-tile candidate
lists (csrc/primary_lists.cuh) and the traversal of the overflowed tiles, equal the scalar oracle's frames bit for bit -- at full
HD, where the lists are used, and after the camera moved between two launches of one context, which makes the device rebuild its
lists from the new camera."""
import numpy as np
import pytest

import helpers as H
from tweeker_raytracer_b200 import host

pytestmark = pytest.mark.gpu


def assert_rows_identical(got, want, rows):
    same = got[rows].view(np.uint32) == want[rows].view(np.uint32)
    assert same.all(), "%d of %d pixels differ" % (int((~same.all(axis=2)).sum()), same.shape[0] * same.shape[1])


def render(app, iterations):
    done = 0
    while done < iterations:
        done = app.render(iterations - done)
    return app.frame()


@pytest.mark.parametrize("name", ["rtigo3_geometry", "rtigo3_cornell_box"])
def test_one_iteration_at_full_hd(cuda_device, tmp_path, name):
    app = host.App(H.write_system(tmp_path, name, resolution="1920 1080"), H.scene_path(name))
    try:
        got = render(app, 1)
        ref = H.oracle_scene(app)
        want = ref.render(H.oracle_sys(app), app.info.miss, 1920, 1080, iter_count=1, row_step=36, row_offset=3).reshape(1080, 1920, 4)
        assert_rows_identical(got, want, slice(3, 1080, 36))
        assert got[3::36, :, :3].mean() > 0.01
    finally:
        app.close()


def test_camera_moved_between_launches(cuda_device, tmp_path):
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="1920 1080", samplesSqrt=2), H.scene_path("rtigo3_geometry"))
    try:
        render(app, 2)
        first = app.frame().copy()
        app.set_camera(0.3, 0.35, 45.0, 6.0, (0.5, 0.8, -0.5))
        got = render(app, 2)
        ref = H.oracle_scene(app)                      # takes the moved camera
        want = ref.render(H.oracle_sys(app), app.info.miss, 1920, 1080, iter_count=2, row_step=45, row_offset=7).reshape(1080, 1920, 4)
        assert_rows_identical(got, want, slice(7, 1080, 45))
        assert not np.array_equal(first.view(np.uint32), got.view(np.uint32))
    finally:
        app.close()
