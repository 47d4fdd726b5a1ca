"""GPU tests of the in-place updates rtc_gas_refit / rtc_ias_update.  Closest hits are defined independently of the BVH, any-hit is a
boolean and the cutout rounds use a canonical candidate order, so a refitted scene must give BIT-IDENTICAL hits and frames to a
scene built from scratch on the same vertices and transforms; for host-built GAS the device refit must also equal the host twin
(rtc_host_gas_refit / rtc_host_ias_refit) byte for byte."""
import os
import sys

import numpy as np
import pytest

import helpers as H
from oracle import orc
from test_cpu_host_accel import check_structure, tri_boxes
from test_cpu_refit import deform, moved, topology
from test_gpu_builder import IDENTITY, soup
from tweeker_raytracer_b200 import core, host

sys.path.insert(0, os.path.join(H.ROOT, "tools"))
import make_instances_scene  # noqa: E402

pytestmark = pytest.mark.gpu

XF = [IDENTITY, [0.5, 0, 0, 1.2, 0, 0.5, 0, 0.1, 0, 0, 0.5, 0.3], [0, -0.6, 0, 0.4, 0.6, 0, 0, 1.1, 0, 0, 0.6, -0.4]]


def instances(gas, transforms):
    inst = np.zeros(len(transforms), dtype=core.INSTANCE_DTYPE)
    for k, t in enumerate(transforms):
        inst[k]["transform"], inst[k]["instanceId"], inst[k]["gas"], inst[k]["materialIndex"], inst[k]["lightIndex"] = t, k, gas, 0, -1
    return inst


def build(ctx, attrs, idx, transforms, flags):
    d_a, d_i = ctx.to_device(attrs), ctx.to_device(idx)
    gas = ctx.gas_build(d_a, 48, len(attrs), d_i, len(idx), flags)
    return gas, ctx.ias_build(instances(gas, transforms)), d_a


def exports_equal(a, b):
    return (a["tlas_nodes"].tobytes() == b["tlas_nodes"].tobytes() and a["tlas_leaves"].tobytes() == b["tlas_leaves"].tobytes()
            and a["world_to_object"].tobytes() == b["world_to_object"].tobytes()
            and all(x[0].tobytes() == y[0].tobytes() and x[1].tobytes() == y[1].tobytes() for x, y in zip(a["gas"].values(), b["gas"].values())))


@pytest.mark.parametrize("flags", [core.BUILD_HOST_SAH, core.BUILD_GPU_LBVH])
@pytest.mark.parametrize("n", [1, 1000, 200000])
def test_refit_with_unchanged_inputs_leaves_the_export_unchanged(cuda_device, flags, n):
    attrs, idx = soup(n, seed=n, extent=0.3 if n == 1 else 0.01 if n > 1000 else 0.08)
    with core.Context(0) as ctx:
        gas, top, _ = build(ctx, attrs, idx, XF, flags)
        before = ctx.scene_export(top)
        ctx.gas_refit(gas)
        ctx.ias_update(top, np.asarray(XF, dtype=np.float32))
        assert exports_equal(ctx.scene_export(top), before)


@pytest.mark.parametrize("flags", [core.BUILD_HOST_SAH, core.BUILD_GPU_LBVH])
def test_refit_equals_rebuild_and_host_twin(cuda_device, flags):
    attrs, idx = soup(20000, seed=11, extent=0.03)
    new = deform(attrs, 0.02, seed=5)
    new_xf = [moved(t, seed=40 + k) for k, t in enumerate(XF)]
    rays = H.random_rays(200000, seed=3, lo=(-0.5, -0.5, -0.5), hi=(1.9, 1.6, 1.3), tmin=1e-5)
    with core.Context(0) as ctx:
        gas, top, d_a = build(ctx, attrs, idx, XF, flags)
        built_nodes = ctx.scene_export(top)["gas"][gas][0]
        ctx.upload(d_a, new)                                       # vertices updated in place
        ctx.gas_refit(gas)
        with pytest.raises(core.RtcError, match="rtc_ias_update"):
            ctx.trace_closest_host(top, rays[:10])
        ctx.ias_update(top, np.asarray(new_xf, dtype=np.float32))
        export = ctx.scene_export(top)
        _, fresh_top, _ = build(ctx, new, idx, new_xf, flags)
        got = ctx.trace_closest_host(top, rays)
        assert H.hits_equal(got, ctx.trace_closest_host(fresh_top, rays))
        short = rays.copy(); short["tmax"] = 0.3
        assert np.array_equal(ctx.trace_any_host(top, short), ctx.trace_any_host(fresh_top, short))
        d_r = ctx.to_device(rays)
        try:
            counts = ctx.trace_count(top, d_r, len(rays))
        finally:
            ctx.free(d_r)
        hits, want = orc.wide_trace(export, rays)
        assert H.hits_equal(hits, got)
        assert (counts.nodes, counts.tris, counts.instances) == want
        assert (got["inst"] != 0xffffffff).mean() > 0.1
        (nodes, tris), = export["gas"].values()
        if flags == core.BUILD_HOST_SAH:
            twin, _ = core.host_scene_refit_export([(attrs, idx)], [(t, 0) for t in XF], [new], new_xf)
            assert exports_equal(export, twin)
        else:
            assert topology(nodes) == topology(built_nodes)
            check_structure(nodes, len(tris), tri_boxes(tris), 3)
        check_structure(export["tlas_nodes"], len(export["tlas_leaves"]), None, 1)


def test_stale_scene_and_new_attribute_buffer(cuda_device):
    attrs, idx = soup(5000, seed=2, extent=0.03)
    new = deform(attrs, 0.05, seed=9)
    rays = H.random_rays(50000, seed=4, lo=(-0.5, -0.5, -0.5), hi=(1.9, 1.6, 1.3), tmin=1e-5)
    with core.Context(0) as ctx:
        gas, top, d_a = build(ctx, attrs, idx, XF[:2], core.BUILD_HOST_SAH)
        d_new = ctx.to_device(new)
        ctx.gas_refit(gas, d_new)
        for call in (lambda: ctx.trace_closest_host(top, rays[:10]), lambda: ctx.trace_any_host(top, rays[:10])):
            with pytest.raises(core.RtcError, match="rtc_ias_update"):
                call()
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        ctx.free(d_a)                                              # the build's buffer is gone: nothing may read it any more
        got = ctx.trace_closest_host(top, rays)
        _, fresh_top, _ = build(ctx, new, idx, XF[:2], core.BUILD_HOST_SAH)
        assert H.hits_equal(got, ctx.trace_closest_host(fresh_top, rays))
        with pytest.raises(core.RtcError, match="out of bounds"):
            ctx.ias_update(top, np.zeros((3, 12), dtype=np.float32))
        with pytest.raises(core.RtcError, match="unknown topObject"):
            ctx.ias_update(12345, np.zeros((0, 12), dtype=np.float32))
        with pytest.raises(core.RtcError, match="bad gas handle"):
            ctx.gas_refit(999)


def _oracle_frame(app, iterations):
    w, h = app.resolution
    return H.oracle_scene(app).render(H.oracle_sys(app), app.info.miss, w, h, iter_count=iterations).reshape(h, w, 4)


@pytest.mark.parametrize("scene", ["rtigo3_geometry", "rtigo3_textures"])
def test_moved_instances_render_the_frame_of_a_scene_built_there(cuda_device, tmp_path, scene):
    """The oracle renders the scene from the App's (updated) instance list with its own BVH: the frame of the refitted scene must
    equal it bit for bit.  The textured scene has cutout materials active, so the ordered any-hit rounds run on the refit."""
    app = host.App(H.write_system(tmp_path, scene, resolution="160 90", samplesSqrt=2), H.scene_path(scene))
    try:
        app.set_coalesce(64)
        app.render(2)                                              # pending: must be rendered with the old positions
        old = [app.instance(i)[0].copy() for i in range(app.info.numInstances)]
        for i in (0, app.info.numInstances - 1):
            m = old[i].reshape(3, 4).copy()
            m[:, :3] = m[:, :3] @ np.array([[0.8, -0.6, 0], [0.6, 0.8, 0], [0, 0, 1]], dtype=np.float32)
            m[:, 3] += (0.1, 0.05, -0.1)
            app.update_instance_transform(i, m.reshape(12))
        app.set_coalesce(1)
        app.render(4)
        moved_frame = app.frame()
        assert moved_frame.tobytes() == _oracle_frame(app, 4).tobytes()
        assert app.stats().stackOverflows == 0
        with pytest.raises(core.RtcError):
            app.update_instance_transform(app.info.numInstances, old[0])
    finally:
        app.close()


def test_launch_on_a_stale_scene_fails_until_it_is_updated(cuda_device, tmp_path):
    app = host.App(H.write_system(tmp_path, "rtigo3_cornell_box", resolution="64 64", samplesSqrt=1), H.scene_path("rtigo3_cornell_box"))
    try:
        app.render(1)
        app.frame()                                                # the first launch allocated the App's output buffer
        ctx = app.context(0)
        sys_data = app.system_data()
        ctx.gas_refit(0)                                           # the App's first geometry, vertices unchanged
        with pytest.raises(core.RtcError, match="rtc_ias_update"):
            ctx.launch(sys_data, 64, 64, core.RAYGEN_FULL_FRAME, app.info.miss, 0, 1)
        ctx.ias_update(sys_data.topObject, np.zeros((0, 12), dtype=np.float32))
        ctx.launch(sys_data, 64, 64, core.RAYGEN_FULL_FRAME, app.info.miss, 0, 1)
        ctx.synchronize()
    finally:
        app.close()


def test_pending_render_uses_the_old_positions(cuda_device, tmp_path):
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="96 64", samplesSqrt=2), H.scene_path("rtigo3_geometry"))
    try:
        want = _oracle_frame(app, 3)
        app.set_coalesce(64)
        app.render(3)                                              # held back by the Raytracer
        m = app.instance(0)[0].copy()
        m[3] += 0.25
        app.update_instance_transform(0, m)                        # flushes the pending iterations first
        assert app.frame().tobytes() == want.tobytes()
    finally:
        app.close()


def test_scale_ten_million_triangles_and_ten_thousand_instances(cuda_device, tmp_path):
    attrs, idx = soup(10_000_000, seed=1, extent=0.002)
    new = deform(attrs, 0.002, seed=3)
    rays = H.random_rays(1_000_000, seed=5, lo=(-0.2, -0.2, -0.2), hi=(1.2, 1.2, 1.2), tmin=1e-5)
    with core.Context(0) as ctx:
        gas, top, d_a = build(ctx, attrs, idx, [IDENTITY], core.BUILD_GPU_LBVH)
        ctx.upload(d_a, new)
        ctx.gas_refit(gas)
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        got = ctx.trace_closest_host(top, rays)
        _, fresh, _ = build(ctx, new, idx, [IDENTITY], core.BUILD_GPU_LBVH)
        assert H.hits_equal(got, ctx.trace_closest_host(fresh, rays))
        assert ctx.stats().stackOverflows == 0
    del attrs, new

    scene = str(tmp_path / "instances.txt")
    make_instances_scene.write_scene(scene, count=10000)
    app = host.App(H.write_system(tmp_path, "rtigo3_instances", resolution="64 64", samplesSqrt=1), scene, host_only=True)
    try:
        geos = [app.geometry(g) for g in range(app.info.numGeometries)]
        insts = [app.instance(i)[:2] for i in range(app.info.numInstances)]
    finally:
        app.close()
    assert len(insts) >= 10000
    new_xf = np.asarray([moved(t, seed=i) for i, (t, _) in enumerate(insts)], dtype=np.float32)
    with core.Context(0) as ctx:
        handles = []
        for a, ix in geos:
            d_a, d_i = ctx.to_device(a), ctx.to_device(ix)
            handles.append(ctx.gas_build(d_a, a.dtype.itemsize, len(a), d_i, len(ix), core.BUILD_HOST_SAH))
        def inst(xf):
            out = np.zeros(len(insts), dtype=core.INSTANCE_DTYPE)
            for k, (t, g) in enumerate(insts):
                out[k]["transform"], out[k]["instanceId"], out[k]["gas"], out[k]["lightIndex"] = xf[k], k, handles[g], -1
            return out
        top = ctx.ias_build(inst([t for t, _ in insts]))
        ctx.ias_update(top, new_xf)
        fresh = ctx.ias_build(inst(new_xf))
        lo, hi = new_xf[:, [3, 7, 11]].min(axis=0), new_xf[:, [3, 7, 11]].max(axis=0)
        rays = H.random_rays(1_000_000, seed=8, lo=tuple(lo), hi=tuple(hi), tmin=1e-4)
        got = ctx.trace_closest_host(top, rays)
        assert H.hits_equal(got, ctx.trace_closest_host(fresh, rays))
        assert (got["inst"] != 0xffffffff).mean() > 0.05
        assert ctx.stats().stackOverflows == 0
