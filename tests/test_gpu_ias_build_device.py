"""GPU tests of rtc_ias_create / rtc_ias_build_device: a scene whose instance set is read from device memory and whose instance level
is built in place on the device.  Its nodes, leaves, world->object matrices and instance -> GAS map must equal the host twin
(host_scene_export + rtc_host_ias_rebuild) byte for byte; its hits, any-hit results, work counts and frames must equal those of a
scene rtc_ias_build makes from the same records; it must never block the host, nor capture the cutout graph again."""
import subprocess
import sys
import time

import numpy as np
import pytest

import helpers as H
from test_cpu_ias_rebuild import mesh, random_instances
from test_cpu_refit import deform
from test_gpu_builder import soup
from test_gpu_ias_rebuild import Scene, check_hits, stream_busy
from tweeker_raytracer_b200 import core, host

pytestmark = pytest.mark.gpu


def same_export(export, twin):
    for key in ("tlas_nodes", "tlas_leaves", "world_to_object"):
        assert export[key].tobytes() == twin[key].tobytes(), key
    assert export["instance_gas"][:len(twin["instance_gas"])].tolist() == list(twin["instance_gas"])


def build_device(ctx, top, records):
    """ias_build_device of host records staged in device memory (freed once the build has run)"""
    d = ctx.to_device(records)
    try:
        ctx.ias_build_device(top, d, len(records))
    finally:
        ctx.free(d)                                                      # rtc_free synchronises the stream first


@pytest.mark.parametrize("n", [0, 1, 2, 8, 9, 1000, 10001, 1_000_000])
def test_build_equals_the_host_twin(cuda_device, n):
    geos, insts = random_instances(max(n, 1), seed=n, spread=max(2.0, 0.5 * n ** (1 / 3)))
    insts = insts[:n]
    twin, _ = core.host_scene_rebuild_export(geos, insts, ["rebuild"])
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, insts)
        records = s.descs([t for t, _ in insts])
        top = ctx.ias_create(n)
        build_device(ctx, top, records)
        export = ctx.scene_export(top)
        same_export(export, twin)
        info = ctx.scene_info(top)
        assert (info.numInstances, info.numTlasNodes, info.numTlasLeaves) == (n, len(twin["tlas_nodes"]), n)
        assert info.numGas == (1 if n else 0) and ctx.scene_rejected_instances(top) == 0
        build_device(ctx, top, records)
        same_export(ctx.scene_export(top), twin)                        # a second build: the same bytes
        fresh = ctx.ias_build(records)
        half = max(2.0, 0.5 * n ** (1 / 3)) / 2 + 0.5
        if n == 0:
            rays = H.random_rays(10000, seed=1, lo=(-half,) * 3, hi=(half,) * 3, tmin=1e-5)
            assert (ctx.trace_closest_host(top, rays)["inst"] == 0xffffffff).all()
        elif n <= 10001:
            got = check_hits(ctx, top, fresh, H.random_rays(100000, seed=1, lo=(-half,) * 3, hi=(half,) * 3, tmin=1e-5), export)
            assert n < 100 or (got["inst"] != 0xffffffff).mean() > 0.05
        else:
            half = 0.25 * n ** (1 / 3) + 0.5
            rays = H.random_rays(1_000_000, seed=2, lo=(-half,) * 3, hi=(half,) * 3, tmin=1e-5)
            assert H.hits_equal(ctx.trace_closest_host(top, rays), ctx.trace_closest_host(fresh, rays))


def three_geometries():
    a, ia = soup(400, seed=1, extent=0.08)
    b, ib = soup(900, seed=2, extent=0.05)
    empty = mesh(np.zeros((0, 3), dtype=np.float32), np.zeros((0, 3), dtype=np.uint32))
    return [(a, ia), (b, ib), empty]


def test_changing_instance_sets(cuda_device):
    """one created scene of capacity 1000 through 1000 -> 10 -> 0 -> 500 -> 1000 instances with different GAS mixes"""
    geos = three_geometries()
    _, base = random_instances(1000, seed=7, spread=6.0)
    rng = np.random.default_rng(5)
    rays = H.random_rays(100000, seed=6, lo=(-3.5,) * 3, hi=(3.5,) * 3, tmin=1e-5)
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, [])
        top = ctx.ias_create(1000)
        for count in (1000, 10, 0, 500, 1000):
            insts = [(base[i][0], int(rng.integers(0, 3))) for i in range(count)]
            s.insts = insts
            records = s.descs([t for t, _ in insts])
            records["materialIndex"] = rng.integers(0, 4, size=count)
            build_device(ctx, top, records)
            twin, _ = core.host_scene_rebuild_export(geos, insts, ["rebuild"])
            export = ctx.scene_export(top)
            same_export(export, twin)
            assert ctx.scene_info(top).numInstances == count
            fresh = ctx.ias_build(records)
            if count:
                check_hits(ctx, top, fresh, rays, export)
            else:
                assert (ctx.trace_closest_host(top, rays)["inst"] == 0xffffffff).all()
            ctx.scene_destroy(fresh)


def test_updates_rebuilds_refits_and_destroy(cuda_device):
    geos = three_geometries()[:2]
    _, base = random_instances(300, seed=9, spread=5.0)
    insts = [(t, k % 2) for k, (t, _) in enumerate(base)]
    xf0 = [t for t, _ in insts]
    xf1 = [np.asarray(t) + np.float32(0.25) * np.array([0, 0, 0, 1] * 3, dtype=np.float32) for t in xf0]
    rays = H.random_rays(100000, seed=3, lo=(-3,) * 3, hi=(3,) * 3, tmin=1e-5)
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, insts)
        top = ctx.ias_create(400)
        build_device(ctx, top, s.descs(xf0))
        steps = ["rebuild"]

        def check(current):
            twin, _ = core.host_scene_rebuild_export(geos, insts, steps)
            export = ctx.scene_export(top)
            same_export(export, twin)
            fresh = s.build(current)
            check_hits(ctx, top, fresh, rays, export)
            ctx.scene_destroy(fresh)

        ctx.ias_update(top, np.asarray(xf1[:100], dtype=np.float32))
        steps.append(([None, None], xf1[:100] + xf0[100:]))
        check(xf1[:100] + xf0[100:])
        d_x = ctx.to_device(np.asarray(xf1, dtype=np.float32))
        ctx.ias_update_device(top, d_x, 300)
        ctx.synchronize()
        ctx.free(d_x)
        steps.append(([None, None], xf1))
        check(xf1)
        ctx.ias_rebuild(top)
        steps.append("rebuild")
        check(xf1)
        # a refit of any GAS of the context makes the scene stale until an update
        new_attrs = deform(geos[1][0], 0.02, seed=4)
        ctx.upload(s.keep[2], new_attrs)
        ctx.gas_refit(s.gas[1])
        with pytest.raises(core.RtcError, match="rtc_ias_update"):
            ctx.trace_closest_host(top, rays[:10])
        with pytest.raises(core.RtcError, match="rtc_ias_update"):
            ctx.ias_rebuild(top)
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        steps.append(([None, new_attrs], xf1))
        geos_now = [geos[0], (new_attrs, geos[1][1])]
        twin, _ = core.host_scene_rebuild_export(geos, insts, steps)
        export = ctx.scene_export(top)
        same_export(export, twin)
        fresh = Scene(ctx, geos_now, insts).build(xf1)
        check_hits(ctx, top, fresh, rays, export)
        # a destroyed GAS: refused until the next build, whose records naming it are rejected
        ctx.gas_destroy(s.gas[1])
        with pytest.raises(core.RtcError, match="a GAS of this scene was destroyed"):
            ctx.trace_closest_host(top, rays[:10])
        with pytest.raises(core.RtcError, match="a GAS of this scene was destroyed"):
            ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        build_device(ctx, top, s.descs(xf1))
        assert ctx.scene_rejected_instances(top) == 150
        hits = ctx.trace_closest_host(top, rays)
        assert not np.isin(hits["inst"], np.arange(1, 300, 2)).any() and (hits["inst"] != 0xffffffff).any()


def test_rejected_records(cuda_device):
    """a bad handle, a destroyed handle and a wrong instanceId: counted, never hit, the other instances as built"""
    geos = three_geometries()
    _, base = random_instances(200, seed=12, spread=4.0)
    insts = [(t, k % 2) for k, (t, _) in enumerate(base)]
    rays = H.random_rays(100000, seed=5, lo=(-2.5,) * 3, hi=(2.5,) * 3, tmin=1e-5)
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, insts)
        doomed = Scene(ctx, geos[:1], []).gas[0]
        ctx.gas_destroy(doomed)
        records = s.descs([t for t, _ in insts])
        bad = [3, 40, 77]
        records["gas"][3] = 999
        records["gas"][40] = doomed
        records["instanceId"][77] = 5
        top = ctx.ias_create(200)
        build_device(ctx, top, records)
        assert ctx.scene_rejected_instances(top) == 3
        assert ctx.scene_export(top)["instance_gas"][bad].tolist() == [core.REJECTED_INSTANCE] * 3
        # the reference: the same scene with the rejected positions as instances of the empty mesh
        ref = records.copy()
        ref["gas"][bad] = s.gas[2]
        ref["instanceId"][77] = 77
        fresh = ctx.ias_build(ref)
        got = ctx.trace_closest_host(top, rays)
        assert H.hits_equal(got, ctx.trace_closest_host(fresh, rays))
        assert not np.isin(got["inst"], bad).any() and (got["inst"] != 0xffffffff).mean() > 0.05
        short = rays.copy(); short["tmax"] = 0.5
        assert np.array_equal(ctx.trace_any_host(top, short), ctx.trace_any_host(fresh, short))


def test_refusals(cuda_device):
    geos = three_geometries()[:1]
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, [([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], 0)] * 3)
        built = s.build()
        top = ctx.ias_create(3)
        d = ctx.to_device(s.descs([t for t, _ in s.insts]))
        try:
            for args, msg in [((12345, d, 3), "unknown topObject"), ((built, d, 3), "rtc_ias_create"),
                              ((top, d, 4), "capacity"), ((top, 0, 3), "instances is null"),
                              ((top, d + 2, 3), "4-byte aligned")]:
                with pytest.raises(core.RtcError, match=msg):
                    ctx.ias_build_device(*args)
            for stride in (0, 60, 66):
                with pytest.raises(core.RtcError, match="strideBytes"):
                    ctx.ias_build_device(top, d, 3, stride)
            with pytest.raises(core.RtcError, match="rtc_ias_create"):
                ctx.scene_rejected_instances(built)
            ctx.ias_build_device(top, 0, 0, 0)                           # no record: nothing to read
            ctx.ias_build_device(top, d, 3, 64)
            ctx.set_instance_flags(top, 0, [0, 0, 0])
            with pytest.raises(core.RtcError, match="out of bounds"):
                ctx.set_instance_flags(top, 2, [0, 0])
            ctx.synchronize()
        finally:
            ctx.free(d)


def _app_records(app, ctx):
    """the App's instances as rtc_instance_desc records, with the GAS handles of its own scene, and its per-instance flags"""
    sys_data = app.system_data()
    gas = ctx.scene_export(sys_data.topObject)["instance_gas"]
    n = app.info.numInstances
    records = np.zeros(n, dtype=core.INSTANCE_DTYPE)
    for i in range(n):
        t, _, m, light = app.instance(i)
        records[i] = (t, i, gas[i], m, light)
    return records


def _flags(app, records):
    mats = app.materials()
    cut = [1 if 0 <= m < len(mats) and mats[m]["textureCutout"] != 0 else 0 for m in records["materialIndex"]]
    return cut, bool((mats["textureAlbedo"] != 0).any())


def _render(ctx, sys_data, w, h, miss, top, iterations):
    sys_data.topObject = top
    ctx.launch(sys_data, w, h, core.RAYGEN_FULL_FRAME, miss, 0, iterations)
    return ctx.download(sys_data.outputBuffer, np.float32, w * h * 4)


def _scene(ctx, top, app, records, build):
    cut, albedo = _flags(app, records)
    if build:
        top = ctx.ias_build(records)
    else:
        build_device(ctx, top, records)
    ctx.set_instance_flags(top, 0, cut)
    ctx.set_albedo_textures(top, albedo)
    return top


@pytest.mark.parametrize("scene", ["rtigo3_geometry", "rtigo3_textures"])
def test_frames(cuda_device, tmp_path, scene):
    """the App's SystemData with topObject replaced by a created scene renders the App's frame bit for bit; the cutout graph is
    not captured again across builds; a material reassignment written on the device renders as rtc_ias_build of it"""
    app = host.App(H.write_system(tmp_path, scene, resolution="96 64", samplesSqrt=2), H.scene_path(scene))
    try:
        app.render(1)
        app.frame()
        ctx = app.context(0)
        w, h = app.resolution
        sys_data = app.system_data()
        own = sys_data.topObject
        records = _app_records(app, ctx)
        top = _scene(ctx, ctx.ias_create(len(records)), app, records, False)
        want = _render(ctx, sys_data, w, h, app.info.miss, own, 4)
        assert _render(ctx, sys_data, w, h, app.info.miss, top, 4).tobytes() == want.tobytes()
        builds = ctx.stats().cutoutGraphBuilds
        for _ in range(3):
            _scene(ctx, top, app, records, False)
            assert _render(ctx, sys_data, w, h, app.info.miss, top, 4).tobytes() == want.tobytes()
        assert ctx.stats().cutoutGraphBuilds == builds
        # a material reassignment written on the device
        other = records.copy()
        other["materialIndex"] = np.roll(records["materialIndex"], 1)
        _scene(ctx, top, app, other, False)
        ref = _scene(ctx, 0, app, other, True)
        got = _render(ctx, sys_data, w, h, app.info.miss, top, 4)
        expect = _render(ctx, sys_data, w, h, app.info.miss, ref, 4)
        assert got.tobytes() == expect.tobytes() and got.tobytes() != want.tobytes()
        ctx.synchronize()
        ctx.scene_destroy(ref)
        ctx.scene_destroy(top)
        sys_data.topObject = own
    finally:
        app.close()


def test_build_does_not_block_the_host(cuda_device, tmp_path):
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="1920 1080", samplesSqrt=1), H.scene_path("rtigo3_geometry"))
    try:
        app.render(1)
        app.frame()
        ctx = app.context(0)
        ctx.set_trace_schedule("group")
        sys_data = app.system_data()
        records = _app_records(app, ctx)
        top = ctx.ias_create(len(records))
        d = ctx.to_device(records)
        ctx.ias_build_device(top, d, len(records))                       # warm: the pool holds the build's scratch
        ctx.synchronize()
        t0 = time.perf_counter()
        ctx.launch(sys_data, 1920, 1080, core.RAYGEN_FULL_FRAME, app.info.miss, 0, 4)
        ctx.synchronize()
        per_iteration = (time.perf_counter() - t0) / 4
        iterations = int(min(2000, max(8, 0.5 / per_iteration)))
        ctx.launch(sys_data, 1920, 1080, core.RAYGEN_FULL_FRAME, app.info.miss, 0, iterations)
        ctx.ias_build_device(top, d, len(records))
        pending = stream_busy(ctx.stream)
        ctx.synchronize()
        assert pending, "rtc_ias_build_device returned after the launch before it had finished: it synchronised the host"
        ctx.free(d)
        ctx.scene_destroy(top)
    finally:
        app.close()


_TORCH_RECORDS = """
import sys
import numpy as np
import torch
sys.path.insert(0, "tests")
from test_cpu_ias_rebuild import random_instances
from test_gpu_ias_build_device import same_export
from test_gpu_ias_rebuild import Scene
from tweeker_raytracer_b200 import core

geos, insts = random_instances(5000, seed=21, spread=10.0)
twin, _ = core.host_scene_rebuild_export(geos, insts, ["rebuild"])
with core.Context(0) as ctx:
    s = Scene(ctx, geos, insts)
    top = ctx.ias_create(5000)
    ctx.synchronize()
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))
    with torch.cuda.stream(stream):
        xf = torch.from_numpy(np.asarray([t for t, _ in insts], dtype=np.float32)).to("cuda")
        rec = torch.zeros((5000, 16), dtype=torch.int32, device="cuda")
        rec.view(torch.float32)[:, :12] = xf * 2.0 - xf                  # a kernel of torch's writes the transforms
        rec[:, 12] = torch.arange(5000, dtype=torch.int32, device="cuda")
        rec[:, 13] = s.gas[0]
        rec[:, 15] = -1
        ctx.ias_build_device(top, rec.data_ptr(), 5000)                  # no host synchronisation in between
    ctx.synchronize()
    same_export(ctx.scene_export(top), twin)
print("torch records ok")
"""


def test_records_written_by_torch_on_the_context_stream(cuda_device):
    """records a torch kernel writes on torch.cuda.ExternalStream(rtc_context_stream) are consumed in stream order.  In a fresh
    interpreter: torch must be imported before the host library brings in its own NCCL."""
    out = subprocess.run([sys.executable, "-c", _TORCH_RECORDS], cwd=H.ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "torch records ok" in out.stdout, out.stdout + out.stderr
