"""GPU tests of rtc_ias_rebuild, the device rebuild of a scene's instance level.  Closest hits do not depend on the BVH and any-hit
is a boolean, so a rebuilt scene must give BIT-IDENTICAL hits and frames to the scene as built; its nodes and leaves must equal
the host twin (rtc_host_ias_rebuild) byte for byte, and it must not block the host once the scene has been rebuilt before."""
import ctypes as C
import os
import sys
import time

import numpy as np
import pytest

import helpers as H
from oracle import orc
from test_cpu_ias_rebuild import random_instances
from test_cpu_refit import deform, moved
from test_gpu_builder import soup
from tweeker_raytracer_b200 import core, host

sys.path.insert(0, os.path.join(H.ROOT, "tools"))
import make_instances_scene  # noqa: E402

pytestmark = pytest.mark.gpu


class Scene:
    """geometries and instances uploaded to one context: GAS built by the host SAH builder (as the host twin builds them)"""

    def __init__(self, ctx, geos, insts):
        self.ctx, self.geos, self.insts, self.keep, self.gas = ctx, list(geos), list(insts), [], []
        for a, ix in geos:
            d_a, d_i = ctx.to_device(a), ctx.to_device(ix)
            self.keep += [d_a, d_i]
            self.gas.append(ctx.gas_build(d_a, a.dtype.itemsize, len(a), d_i, len(ix), core.BUILD_HOST_SAH))

    def descs(self, transforms):
        out = np.zeros(len(self.insts), dtype=core.INSTANCE_DTYPE)
        out["transform"] = np.asarray(transforms, dtype=np.float32).reshape(-1, 12)
        out["instanceId"] = np.arange(len(self.insts))
        out["gas"] = [self.gas[g] for _, g in self.insts]
        out["lightIndex"] = -1
        return out

    def build(self, transforms=None):
        return self.ctx.ias_build(self.descs([t for t, _ in self.insts] if transforms is None else transforms))


def same_tlas(a, b):
    return a["tlas_nodes"].tobytes() == b["tlas_nodes"].tobytes() and a["tlas_leaves"].tobytes() == b["tlas_leaves"].tobytes()


def check_hits(ctx, top, fresh, rays, export):
    """closest hits and occlusion of `top` equal those of the freshly built `fresh`, and rtc_trace_count equals the oracle's
    traversal of top's export"""
    got = ctx.trace_closest_host(top, rays)
    assert H.hits_equal(got, ctx.trace_closest_host(fresh, rays))
    short = rays.copy(); short["tmax"] = 0.5
    assert np.array_equal(ctx.trace_any_host(top, short), ctx.trace_any_host(fresh, short))
    d_r = ctx.to_device(rays)
    try:
        counts = ctx.trace_count(top, d_r, len(rays))
    finally:
        ctx.free(d_r)
    hits, want = orc.wide_trace(export, rays)
    assert H.hits_equal(hits, got)
    assert (counts.nodes, counts.tris, counts.instances) == want
    return got


@pytest.mark.parametrize("n", [1, 2, 8, 9, 1000, 10001, 1_000_000])
def test_device_rebuild_equals_the_host_twin(cuda_device, n):
    geos, insts = random_instances(n, seed=n, spread=max(2.0, 0.5 * n ** (1 / 3)))
    twin, _ = core.host_scene_rebuild_export(geos, insts, ["rebuild"])
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, insts)
        top, fresh = s.build(), s.build()
        ctx.ias_rebuild(top)
        export = ctx.scene_export(top)
        assert same_tlas(export, twin)
        assert ctx.scene_info(top).numTlasNodes == len(twin["tlas_nodes"])
        ctx.ias_rebuild(top)
        assert same_tlas(ctx.scene_export(top), twin)                       # a second rebuild: the same bytes
        if n <= 10001:
            half = max(2.0, 0.5 * n ** (1 / 3)) / 2 + 0.5
            got = check_hits(ctx, top, fresh, H.random_rays(100000, seed=1, lo=(-half,) * 3, hi=(half,) * 3, tmin=1e-5), export)
            assert n < 100 or (got["inst"] != 0xffffffff).mean() > 0.05
        else:
            half = 0.25 * n ** (1 / 3) + 0.5
            rays = H.random_rays(1_000_000, seed=2, lo=(-half,) * 3, hi=(half,) * 3, tmin=1e-5)
            assert H.hits_equal(ctx.trace_closest_host(top, rays), ctx.trace_closest_host(fresh, rays))


def test_sequences_of_updates_and_rebuilds(cuda_device):
    attrs, idx = soup(3000, seed=4, extent=0.04)
    rng = np.random.default_rng(8)
    xf0 = [moved([0.3, 0, 0, x, 0, 0.3, 0, y, 0, 0, 0.3, z], seed=k) for k, (x, y, z) in enumerate(rng.uniform(-2, 2, size=(300, 3)))]
    insts = [(t, 0) for t in xf0]
    new_attrs = deform(attrs, 0.03, seed=2)
    xf1 = [moved(t, seed=1000 + k) for k, t in enumerate(xf0)]
    xf2 = [xf1[p] for p in rng.permutation(len(xf1))]                        # large motion: the instances swap places
    rays = H.random_rays(100000, seed=6, lo=(-2.5, -2.5, -2.5), hi=(2.5, 2.5, 2.5), tmin=1e-5)
    with core.Context(0) as ctx:
        s = Scene(ctx, [(attrs, idx)], insts)
        top = s.build()
        d_a = s.keep[0]
        ctx.upload(d_a, new_attrs)
        ctx.gas_refit(s.gas[0])
        with pytest.raises(core.RtcError, match="rtc_ias_update"):
            ctx.ias_rebuild(top)
        ctx.ias_update(top, np.asarray(xf1, dtype=np.float32))
        steps, current = [([new_attrs], xf1)], xf1
        fresh_geo = Scene(ctx, [(new_attrs, idx)], insts)
        for step in ("rebuild", "update", "rebuild"):
            if step == "rebuild":
                ctx.ias_rebuild(top)
                steps.append("rebuild")
            else:
                ctx.ias_update(top, np.asarray(xf2, dtype=np.float32))
                steps.append(([None], xf2))
                current = xf2
            export = ctx.scene_export(top)
            twin, _ = core.host_scene_rebuild_export([(attrs, idx)], insts, steps)
            assert same_tlas(export, twin), step
            assert export["world_to_object"].tobytes() == twin["world_to_object"].tobytes()
            fresh = fresh_geo.build(current)
            got = check_hits(ctx, top, fresh, rays, export)
            assert (got["inst"] != 0xffffffff).mean() > 0.05
            ctx.scene_destroy(fresh)


def test_refusals(cuda_device):
    attrs, idx = soup(500, seed=3, extent=0.05)
    with core.Context(0) as ctx:
        s = Scene(ctx, [(attrs, idx)], [([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], 0)] * 3)
        top = s.build()
        with pytest.raises(core.RtcError, match="unknown topObject"):
            ctx.ias_rebuild(12345)
        ctx.gas_refit(s.gas[0])
        with pytest.raises(core.RtcError, match="rtc_ias_update"):
            ctx.ias_rebuild(top)
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        ctx.ias_rebuild(top)
        ctx.gas_destroy(s.gas[0])
        with pytest.raises(core.RtcError, match="a GAS of this scene was destroyed"):
            ctx.ias_rebuild(top)


def stream_busy(stream):
    """cudaStreamQuery of the CUDA runtime the library runs on: True while work enqueued on `stream` has not finished"""
    cudart = C.CDLL("libcudart.so.12")
    cudart.cudaStreamQuery.argtypes = [C.c_void_p]
    rc = cudart.cudaStreamQuery(C.c_void_p(stream))
    assert rc in (0, 600), rc                                            # cudaSuccess, cudaErrorNotReady
    return rc == 600


def test_rebuild_does_not_block_the_host(cuda_device, tmp_path):
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="1920 1080", samplesSqrt=1), H.scene_path("rtigo3_geometry"))
    try:
        app.render(1)
        app.frame()                                                      # the App's output buffer exists
        ctx = app.context(0)
        ctx.set_trace_schedule("group")                                  # no timed batch, so no launch waits for the schedule tuner
        sys_data = app.system_data()
        top = sys_data.topObject
        ctx.ias_rebuild(top)                                             # the first rebuild allocates and may synchronise
        ctx.synchronize()
        t0 = time.perf_counter()
        ctx.launch(sys_data, 1920, 1080, core.RAYGEN_FULL_FRAME, app.info.miss, 0, 4)
        ctx.synchronize()
        per_iteration = (time.perf_counter() - t0) / 4
        iterations = int(min(2000, max(8, 0.5 / per_iteration)))         # about half a second of work
        ctx.launch(sys_data, 1920, 1080, core.RAYGEN_FULL_FRAME, app.info.miss, 0, iterations)
        ctx.ias_rebuild(top)
        pending = stream_busy(ctx.stream)
        ctx.synchronize()
        assert pending, "rtc_ias_rebuild returned after the launch before it had finished: it synchronised the host"
    finally:
        app.close()


def _oracle_frame(app, iterations):
    w, h = app.resolution
    return H.oracle_scene(app).render(H.oracle_sys(app), app.info.miss, w, h, iter_count=iterations).reshape(h, w, 4)


def _stress(tmp_path):
    scene = str(tmp_path / "stress.txt")
    make_instances_scene.write_scene(scene, count=300, tess=(24, 12))
    return H.write_system(tmp_path, "rtigo3_instances", resolution="96 64", samplesSqrt=2), scene


@pytest.mark.parametrize("scene", ["rtigo3_geometry", "rtigo3_textures", "stress"])
def test_frames_through_a_rebuild(cuda_device, tmp_path, scene):
    """render(k), rebuild_instance_level(), render(k) gives the frame of render(2k) and of the oracle.  The textured scene has
    cutout materials, so the ordered any-hit rounds and their cached graph run across the rebuild."""
    files = _stress(tmp_path) if scene == "stress" else (H.write_system(tmp_path, scene, resolution="96 64", samplesSqrt=2), H.scene_path(scene))
    k = 2
    b = host.App(*files)
    try:
        assert b.render(2 * k) == 2 * k
        want = b.frame()
        assert want.tobytes() == _oracle_frame(b, 2 * k).tobytes()
    finally:
        b.close()
    a = host.App(*files)
    try:
        assert a.render(k) == k
        a.frame()                                                        # the iterations held back so far have run
        builds = [a.context(0).stats().cutoutGraphBuilds]
        a.rebuild_instance_level()
        assert a.render(k) == 2 * k
        assert a.frame().tobytes() == want.tobytes()
        builds.append(a.context(0).stats().cutoutGraphBuilds)
        a.rebuild_instance_level()
        a.render(1)
        a.frame()
        builds.append(a.context(0).stats().cutoutGraphBuilds)
        assert builds[1] - builds[0] <= 1 and builds[2] == builds[1], builds
    finally:
        a.close()
