"""GPU tests of instance visibility masks and triangle face culling: rtc_scene_set_instance_masks and rtc_trace_closest_ex /
rtc_trace_any_ex / rtc_trace_count_ex, under all three schedules of the triangle tests.

  * the filtered kernels with everything visible equal the plain kernels bit for bit, counters included;
  * with random instance and ray masks and every cull flag they equal the oracle's brute force (closest and any hit) and the
    counters equal the restatement of oracle/wide_bvh.inc's traversal with the two tests (tests/mask_oracle.py) on the exported BVH;
  * closed meshes seen from outside and inside, and a mirrored instance, agree with the oracle;
  * masks of created scenes belong to positions and survive builds, updates and rebuilds;
  * masks are stream-ordered; the plain entry points equal the _ex calls with (0xFF, 0); rendering refuses a masked scene;
  * every refusal enqueues nothing."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import helpers as H
from mask_oracle import MaskedScene, wide_trace_ex
from oracle import orc
from test_cpu_ias_rebuild import mesh
from test_cpu_trace_masks import FLAG_SETS
from test_gpu_builder import soup
from test_gpu_ias_rebuild import Scene
from tweeker_raytracer_b200 import core, host

sys.path.insert(0, os.path.join(H.ROOT, "tools"))
import make_instances_scene  # noqa: E402

pytestmark = pytest.mark.gpu

SCHEDULES = ["group", "one_tri", "two_tri"]


def counts(ctx, top, rays, any_hit=False, mask=0xFF, flags=0):
    d_r = ctx.to_device(rays)
    try:
        c = ctx.trace_count(top, d_r, len(rays), any_hit=any_hit, mask=mask, flags=flags)
    finally:
        ctx.free(d_r)
    assert c.rays == len(rays)
    return (c.nodes, c.tris, c.instances)


def app_scene(tmp_path, name):
    """(App, top, oracle scene, rays) of one test scene"""
    if name == "instances":
        path = os.path.join(str(tmp_path), "scene_lattice.txt")
        make_instances_scene.write_scene(path, count=343, tess=(24, 12))
        app = host.App(H.write_system(tmp_path, "rtigo3_instances", resolution="64 64", samplesSqrt=1), path)
        rays = H.random_rays(20000, 5, lo=(-12.0, 0.0, -12.0), hi=(12.0, 12.0, 12.0))
    else:
        system = {"cornell": "rtigo3_cornell_box", "geometry": "rtigo3_geometry"}[name]
        app = host.App(H.write_system(tmp_path, system, resolution="64 64", samplesSqrt=1), H.scene_path(system))
        rays = H.random_rays(20000, 5)
    ref = MaskedScene(H.oracle_scene(app), app.info.numInstances)
    w, h = app.resolution
    primary = ref.scene.generate_primary(H.oracle_sys(app), w, h, 0)
    rays = np.concatenate([primary[primary["tmax"] > 0], rays])
    return app, app.system_data(0).topObject, ref, rays


def soup_scene(ctx, n=200000):
    attrs, idx = soup(n, seed=11, extent=float(n) ** (-1.0 / 3.0))
    s = Scene(ctx, [(attrs, idx)], [([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], 0)])
    rng = np.random.default_rng(3)
    rays = np.zeros(50000, dtype=core.RAY_DTYPE)
    o, d = rng.random((len(rays), 3)), rng.normal(size=(len(rays), 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays["ox"], rays["oy"], rays["oz"], rays["tmin"] = o[:, 0], o[:, 1], o[:, 2], 1e-5
    rays["dx"], rays["dy"], rays["dz"], rays["tmax"] = d[:, 0], d[:, 1], d[:, 2], 1e27
    return s, s.build(), rays


def check_everything_visible(ctx, top, n, rays):
    short = rays.copy(); short["tmax"] = np.minimum(short["tmax"], 0.5)
    for schedule in SCHEDULES:
        ctx.set_trace_schedule(schedule)
        ctx.set_instance_masks(top, 0, np.full(n, 0xFF, dtype=np.uint8))
        plain = (ctx.trace_closest_host(top, rays), ctx.trace_any_host(top, short), counts(ctx, top, rays), counts(ctx, top, short, True))
        ctx.set_instance_masks(top, 0, np.full(n, 0x01, dtype=np.uint8))
        assert H.hits_equal(ctx.trace_closest_host(top, rays, mask=0x01), plain[0]), schedule
        assert np.array_equal(ctx.trace_any_host(top, short, mask=0x01), plain[1]), schedule
        assert counts(ctx, top, rays, mask=0x01) == plain[2], schedule
        assert counts(ctx, top, short, True, mask=0x01) == plain[3], schedule
        # the plain entry points on the masked scene take the filtered kernels: the same results
        assert H.hits_equal(ctx.trace_closest_host(top, rays), plain[0]), schedule
        ctx.set_instance_masks(top, 0, np.full(n, 0xFF, dtype=np.uint8))
    assert (plain[0]["inst"] != 0xffffffff).mean() > 0.05


@pytest.mark.parametrize("name", ["cornell", "geometry", "instances"])
def test_filtered_kernels_with_everything_visible(cuda_device, tmp_path, name):
    app, top, ref, rays = app_scene(tmp_path, name)
    check_everything_visible(app.context(0), top, app.info.numInstances, rays)
    app.close()


def test_filtered_kernels_with_everything_visible_on_a_soup(cuda_device):
    with core.Context(0) as ctx:
        _, top, rays = soup_scene(ctx)
        check_everything_visible(ctx, top, 1, rays)


def check_filtered(ctx, top, ref, rays, masks, ray_mask, flags, label, brute=1500):
    """closest and any hit against the oracle's brute force (the first `brute` rays) and its BVH, counters against the restatement"""
    export = ctx.scene_export(top)
    got = ctx.trace_closest_host(top, rays, mask=ray_mask, flags=flags)
    assert H.hits_equal(got[:brute], ref.trace_closest_ex(rays[:brute], ray_mask, flags)), label
    model, model_counts = wide_trace_ex(export, rays, masks=masks, ray_mask=ray_mask, flags=flags)
    assert H.hits_equal(got, model), label
    assert counts(ctx, top, rays, mask=ray_mask, flags=flags) == model_counts, label
    short = rays.copy(); short["tmax"] = np.minimum(short["tmax"], 0.5)
    occl = ctx.trace_any_host(top, short, mask=ray_mask, flags=flags).astype(bool)
    assert np.array_equal(occl[:brute], ref.trace_any_ex(short[:brute], ray_mask, flags).astype(bool)), label
    assert counts(ctx, top, short, True, mask=ray_mask, flags=flags) == wide_trace_ex(export, short, any_hit=True, masks=masks,
                                                                                    ray_mask=ray_mask, flags=flags)[1], label
    return got


@pytest.mark.parametrize("name", ["cornell", "geometry", "instances"])
def test_random_masks_and_flags_equal_the_oracle(cuda_device, tmp_path, name):
    app, top, ref, rays = app_scene(tmp_path, name)
    ctx = app.context(0)
    rng = np.random.default_rng(len(name))
    n = app.info.numInstances
    for schedule in SCHEDULES:
        ctx.set_trace_schedule(schedule)
        masks = rng.integers(0, 256, size=n).astype(np.uint8)
        ctx.set_instance_masks(top, 0, masks)
        ref.set_instance_masks(0, masks)
        for flags in FLAG_SETS:
            ray_mask = int(rng.integers(1, 256))
            check_filtered(ctx, top, ref, rays, masks, ray_mask, flags, (name, schedule, flags, ray_mask))
    app.close()


def closed_box():
    v = np.array([[x, y, z] for x in (-1, 1) for y in (-1, 1) for z in (-1, 1)], dtype=np.float32)
    quads = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    idx = [[a, b, c] for (a, b, c, d) in quads] + [[a, c, d] for (a, b, c, d) in quads]
    return mesh(v, idx)


def test_culling_of_closed_meshes_and_a_mirrored_instance(cuda_device):
    """boxes of 12 outward-wound triangles, placed plainly, rotated and scaled, and mirrored; rays from outside and from inside"""
    box = closed_box()
    transforms = [[1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0],
                  [0.0, -1.5, 0.0, 4.0, 1.2, 0.0, 0.0, 0.0, 0.0, 0.0, 0.8, 0.5],
                  [-1, 0, 0, -4.0, 0, 1, 0, 0.5, 0, 0, 1, 0.0],                          # mirrored
                  [1, 0, 0, 0, 0, 1, 0, 4.0, 0, 0, -1.3, 0]]                             # mirrored and scaled
    insts = [(np.array(t, dtype=np.float32), 0) for t in transforms]
    with core.Context(0) as ctx:
        s = Scene(ctx, [box], insts)
        top = s.build()
        ref = orc.Scene()
        ref.add_geometry(*box)
        for t, _ in insts:
            ref.add_instance(t, 0, 0)
        ref.commit()
        ref = MaskedScene(ref, len(insts))
        inside = H.random_rays(3000, 1, lo=(-0.9, -0.9, -0.9), hi=(0.9, 0.9, 0.9))
        around = H.random_rays(6000, 2, lo=(-7, -3, -3), hi=(7, 7, 3))
        rays = np.concatenate([inside, around])
        masks = np.full(len(insts), 0xFF, dtype=np.uint8)
        for schedule in SCHEDULES:
            ctx.set_trace_schedule(schedule)
            for flags in FLAG_SETS:
                got = check_filtered(ctx, top, ref, rays, masks, 0xFF, flags, (schedule, flags), brute=len(rays))
                if flags == core.RAY_CULL_BACK_FACING:
                    assert (got[:len(inside)]["inst"] != 0).all()                 # never the box the ray starts in
        ref.close()


def build_device(ctx, top, records):
    d = ctx.to_device(records)
    try:
        ctx.ias_build_device(top, d, len(records))
    finally:
        ctx.free(d)


def test_created_scene_masks_persist(cuda_device):
    rng = np.random.default_rng(9)
    attrs, idx = soup(2000, seed=5, extent=0.05)
    quad = mesh(np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0]], dtype=np.float32), [[0, 1, 2], [0, 2, 3]])
    cap = 64
    xf = [np.array([0.5, 0, 0, x, 0, 0.5, 0, y, 0, 0, 0.5, z], dtype=np.float32) for x, y, z in rng.uniform(-2, 2, size=(cap, 3))]
    rays = H.random_rays(20000, 4, lo=(-2.5, -2.5, -2.5), hi=(2.5, 2.5, 2.5), tmin=1e-5)
    masks = rng.integers(0, 256, size=cap).astype(np.uint8)
    with core.Context(0) as ctx:
        s = Scene(ctx, [(attrs, idx), quad], [(t, k % 2) for k, t in enumerate(xf)])
        top = ctx.ias_create(cap)
        ctx.set_instance_masks(top, 0, masks)

        def same_as_fresh(records, label):
            fresh = ctx.ias_build(records)
            ctx.set_instance_masks(fresh, 0, masks[:len(records)])
            for flags in (0, core.RAY_CULL_BACK_FACING):
                for ray_mask in (0x01, 0x5A, 0xFF):
                    got = ctx.trace_closest_host(top, rays, mask=ray_mask, flags=flags)
                    assert H.hits_equal(got, ctx.trace_closest_host(fresh, rays, mask=ray_mask, flags=flags)), (label, flags, ray_mask)
                    assert counts(ctx, top, rays, mask=ray_mask, flags=flags) == wide_trace_ex(
                        ctx.scene_export(top), rays, masks=masks[:len(records)], ray_mask=ray_mask, flags=flags)[1], (label, flags, ray_mask)
            ctx.scene_destroy(fresh)

        all_records = s.descs(xf)
        build_device(ctx, top, all_records[:40])
        same_as_fresh(all_records[:40], "first build")
        other = all_records[:25].copy()
        other["gas"] = s.gas[1]                                            # a different count and GAS
        build_device(ctx, top, other)
        same_as_fresh(other, "second build")
        moved = np.array([t + np.float32(0.1) * np.array([0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0], dtype=np.float32) for t in xf[:25]])
        d_m = ctx.to_device(moved)
        ctx.ias_update_device(top, d_m, 25)
        ctx.ias_rebuild(top)
        ctx.synchronize()
        ctx.free(d_m)
        after = other.copy(); after["transform"] = moved
        same_as_fresh(after, "update and rebuild")
        build_device(ctx, top, all_records)                                # positions past 25 kept their masks
        same_as_fresh(all_records, "full build")


def test_masks_are_stream_ordered(cuda_device, tmp_path):
    app, top, ref, rays = app_scene(tmp_path, "instances")
    ctx = app.context(0)
    n = app.info.numInstances
    rng = np.random.default_rng(2)
    masks_a, masks_b = (rng.integers(0, 4, size=n).astype(np.uint8) for _ in range(2))
    d_r = ctx.to_device(rays)
    d_ha, d_hb = ctx.malloc(len(rays) * 20), ctx.malloc(len(rays) * 20)
    for _ in range(2):                                                     # no synchronisation between the four calls
        ctx.set_instance_masks(top, 0, masks_a)
        ctx.trace_closest(top, d_r, len(rays), d_ha, mask=0x01)
        ctx.set_instance_masks(top, 0, masks_b)
        ctx.trace_closest(top, d_r, len(rays), d_hb, mask=0x01)
        got_a, got_b = ctx.download(d_ha, core.HIT_DTYPE, len(rays)), ctx.download(d_hb, core.HIT_DTYPE, len(rays))
        for masks, got in ((masks_a, got_a), (masks_b, got_b)):
            assert H.hits_equal(got, wide_trace_ex(ctx.scene_export(top), rays, masks=masks, ray_mask=0x01)[0])
    assert not H.hits_equal(got_a, got_b)
    for p in (d_r, d_ha, d_hb):
        ctx.free(p)
    app.close()


def test_plain_entry_points_on_a_masked_scene(cuda_device, tmp_path):
    app, top, ref, rays = app_scene(tmp_path, "geometry")
    ctx = app.context(0)
    masks = np.random.default_rng(4).integers(0, 256, size=app.info.numInstances).astype(np.uint8)
    ctx.set_instance_masks(top, 0, masks)
    ref.set_instance_masks(0, masks)
    d_r = ctx.to_device(rays)
    d_h, d_o = ctx.malloc(len(rays) * 20), ctx.malloc(len(rays) * 4)
    for schedule in SCHEDULES:
        ctx.set_trace_schedule(schedule)
        core._check(ctx.L.rtc_trace_closest_ex(ctx.h, int(top), int(d_r), len(rays), int(d_h), 0xFF, 0))
        ex = ctx.download(d_h, core.HIT_DTYPE, len(rays))
        core._check(ctx.L.rtc_trace_any_ex(ctx.h, int(top), int(d_r), len(rays), int(d_o), 0xFF, 0))
        ex_any = ctx.download(d_o, np.uint32, len(rays))
        assert H.hits_equal(ctx.trace_closest_host(top, rays), ex)
        assert np.array_equal(ctx.trace_any_host(top, rays), ex_any)
        assert H.hits_equal(ex[:1500], ref.trace_closest_ex(rays[:1500], 0xFF, 0))
        out = core.TraceCounts()
        core._check(ctx.L.rtc_trace_count_ex(ctx.h, int(top), int(d_r), len(rays), 0, 0xFF, 0, C.byref(out)))
        assert (out.nodes, out.tris, out.instances) == counts(ctx, top, rays)
    for p in (d_r, d_h, d_o):
        ctx.free(p)
    app.close()


def test_rendering_refuses_a_masked_scene(cuda_device, tmp_path):
    def render(app):
        while app.render(1) < app.spp:
            pass
        return app.frame()

    sysfile = H.write_system(tmp_path, "rtigo3_cornell_box", resolution="64 64", samplesSqrt=2)
    clean = host.App(sysfile, H.scene_path("rtigo3_cornell_box"))
    want = render(clean)
    clean.close()
    app = host.App(sysfile, H.scene_path("rtigo3_cornell_box"))
    ctx, sys_data = app.context(0), app.system_data(0)
    top, n = sys_data.topObject, app.info.numInstances
    w, h = app.resolution
    launches = ctx.stats().kernelLaunches
    masks = np.full(n, 0xFF, dtype=np.uint8); masks[n - 1] = 0xFE
    ctx.set_instance_masks(top, 0, masks)
    with pytest.raises(core.RtcError, match="does not evaluate instance masks"):
        ctx.launch(sys_data, w, h, core.RAYGEN_FULL_FRAME, app.info.miss, 0, 1)
    with pytest.raises(core.RtcError, match="does not evaluate instance masks"):
        ctx.launch_ex(sys_data, w, h, core.RAYGEN_FULL_FRAME, app.info.miss, 0, 1, 0)
    assert ctx.stats().kernelLaunches == launches
    ctx.set_instance_masks(top, n - 1, [0xFF])
    got = render(app)
    assert got.tobytes() == want.tobytes()
    app.close()


def test_refusals_enqueue_nothing(cuda_device):
    attrs, idx = soup(500, seed=3, extent=0.05)
    with core.Context(0) as ctx:
        s = Scene(ctx, [(attrs, idx)], [([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], 0)] * 3)
        top = s.build()
        created = ctx.ias_create(8)
        rays = H.random_rays(100, 1)
        d_r, d_h = ctx.to_device(rays), ctx.malloc(100 * 20)
        ctx.synchronize()
        before = ctx.stats().kernelLaunches
        L, h = ctx.L, ctx.h
        out = core.TraceCounts()
        calls = [lambda m, f, t=top, n=100: L.rtc_trace_closest_ex(h, int(t), int(d_r), n, int(d_h), m, f),
                 lambda m, f, t=top, n=100: L.rtc_trace_any_ex(h, int(t), int(d_r), n, int(d_h), m, f),
                 lambda m, f, t=top, n=100: L.rtc_trace_count_ex(h, int(t), int(d_r), n, 0, m, f, C.byref(out))]
        for call in calls:
            for args, text in (((0x100, 0), b"visibilityMask"), ((0xFF, 4), b"rayFlags"), ((0xFF, 0x80000000), b"rayFlags")):
                assert call(*args) != 0 and text in L.rtc_last_error()
            assert call(0xFF, 0, t=12345) != 0 and b"unknown topObject" in L.rtc_last_error()
            assert call(0x01, 1, n=2 ** 32) != 0 and b"2^32" in L.rtc_last_error()
        with pytest.raises(core.RtcError, match="instance range out of bounds"):
            ctx.set_instance_masks(top, 2, [1, 2])
        with pytest.raises(core.RtcError, match="instance range out of bounds"):
            ctx.set_instance_masks(created, 0, np.zeros(9, dtype=np.uint8))
        with pytest.raises(core.RtcError, match="unknown topObject"):
            ctx.set_instance_masks(12345, 0, [1])
        assert L.rtc_scene_set_instance_masks(h, int(top), 0, 1, None) != 0 and b"masks is null" in L.rtc_last_error()
        assert L.rtc_scene_set_instance_masks(h, int(top), 3, 0, None) == 0        # empty range at the end: nothing to do
        ctx.set_instance_masks(created, 0, np.zeros(8, dtype=np.uint8))           # up to the capacity
        assert ctx.stats().kernelLaunches == before
        ctx.gas_refit(s.gas[0])                                                   # stale scene: refused like rtc_trace_closest
        ctx.synchronize()
        before = ctx.stats().kernelLaunches
        for call in calls:
            assert call(0x01, 0) != 0 and b"rtc_ias_update" in L.rtc_last_error()
        assert ctx.stats().kernelLaunches == before
        ctx.free(d_r); ctx.free(d_h)
