"""GPU tests of rtc_ias_update_device, the instance update whose object->world matrices are read from device memory on the context
stream.  Its results must equal rtc_ias_update with the same matrices from host memory and the host twin byte for byte
(instance level, leaves, world->object rows), frames must be bit-identical to the host update's, it must not block the host, and
it must read its buffer when the stream reaches it, not during the call."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import helpers as H
from test_cpu_ias_rebuild import random_instances
from test_cpu_refit import deform, moved
from test_gpu_builder import soup
from test_gpu_ias_rebuild import Scene, _stress, check_hits, stream_busy
from tweeker_raytracer_b200 import core, host

pytestmark = pytest.mark.gpu


def mixed(transforms, seed):
    """New object->world matrices: moved() (rotation, non-uniform scale, mirror) for every fourth instance (the first 2000 of
    them), and for the others shears, rotations with per-axis scales from 1e-3 to 1e3, or such a matrix translated up to 1e4."""
    x = np.asarray(transforms, dtype=np.float64).reshape(-1, 3, 4).copy()
    n = len(x)
    rng = np.random.default_rng(seed)
    kind = np.arange(n) % 4
    q, _ = np.linalg.qr(rng.normal(size=(n, 3, 3)))
    scaled = q * 10.0 ** rng.uniform(-3, 3, size=(n, 1, 3))
    shear = np.eye(3) + np.triu(rng.uniform(-2, 2, size=(n, 3, 3)), 1)
    a = np.where((kind == 1)[:, None, None], shear, scaled)
    x[kind >= 1, :, :3] = (x[:, :, :3] @ a)[kind >= 1]
    far = kind == 3
    x[far, :, 3] = rng.uniform(-1e4, 1e4, size=(int(far.sum()), 3))
    out = x.astype(np.float32).reshape(n, 12)
    for k in range(0, min(n, 8000), 4):
        out[k] = moved(out[k], seed=seed + k)
    return out


def same_export(a, b):
    return (a["tlas_nodes"].tobytes() == b["tlas_nodes"].tobytes() and a["tlas_leaves"].tobytes() == b["tlas_leaves"].tobytes()
            and a["world_to_object"].tobytes() == b["world_to_object"].tobytes())


def rays_for(n, count, seed):
    half = max(2.0, 0.5 * n ** (1 / 3)) / 2 + 0.5
    return H.random_rays(count, seed=seed, lo=(-half,) * 3, hi=(half,) * 3, tmin=1e-5)


@pytest.mark.parametrize("n", [1, 9, 1000, 10001, 1_000_000])
def test_equals_the_host_update_and_the_twin(cuda_device, n):
    geos, insts = random_instances(n, seed=n, spread=max(2.0, 0.5 * n ** (1 / 3)))
    x = mixed([t for t, _ in insts], seed=n + 1)
    twin, _ = core.host_scene_rebuild_export(geos, insts, [([None], x)])
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, insts)
        by_host, by_device = s.build(), s.build()
        d_x = ctx.to_device(x)
        ctx.ias_update(by_host, x)
        ctx.ias_update_device(by_device, d_x, n)
        got, want = ctx.scene_export(by_device), ctx.scene_export(by_host)
        assert same_export(got, want)
        assert same_export(got, twin)
        for i in sorted(set(np.linspace(0, n - 1, min(n, 64)).astype(int))):
            inv = ctx.instance_inverse(by_device, int(i))
            assert inv.tobytes() == ctx.instance_inverse(by_host, int(i)).tobytes() == twin["world_to_object"][i].tobytes()
        # a build from the same matrices writes its instance records with the update kernels: the host twin's build, byte for byte
        fresh = s.build(x)
        built, _ = core.host_scene_export(geos, [(x[i], g) for i, (_, g) in enumerate(insts)])
        assert same_export(ctx.scene_export(fresh), built)
        if n <= 10001:
            check_hits(ctx, by_device, fresh, rays_for(n, 20000, seed=3), got)
        ctx.free(d_x)


def test_ranges_strides_and_determinism(cuda_device):
    n = 2000
    geos, insts = random_instances(n, seed=5, spread=12.0)
    x0 = np.asarray([t for t, _ in insts], dtype=np.float32)
    x = mixed(x0, seed=6)
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, insts)
        for first, count in [(0, 0), (0, n), (777, 1), (123, 1001)]:
            by_host, by_device = s.build(), s.build()
            ctx.ias_update(by_host, x[first:first + count], first)
            d_x = ctx.to_device(x[first:first + count] if count else np.zeros(12, dtype=np.float32))
            ctx.ias_update_device(by_device, d_x, count, first)
            current = x0.copy()
            current[first:first + count] = x[first:first + count]
            twin, _ = core.host_scene_rebuild_export(geos, insts, [([None], current)])
            got = ctx.scene_export(by_device)
            assert same_export(got, ctx.scene_export(by_host)), (first, count)
            assert same_export(got, twin), (first, count)
            ctx.free(d_x)
            ctx.scene_destroy(by_host)
            ctx.scene_destroy(by_device)
        # OptixInstance-sized records: the 32 bytes behind each transform are NaN garbage and must be ignored
        records = np.full((n, 20), np.nan, dtype=np.float32)
        records.view(np.uint32)[:, 12:] = 0x7fc0dead
        records[:, :12] = x
        d_rec, d_x = ctx.to_device(records), ctx.to_device(x)
        by_host, strided, dense, again = s.build(), s.build(), s.build(), s.build()
        ctx.ias_update(by_host, x)
        ctx.ias_update_device(strided, d_rec, n, stride=80)
        ctx.ias_update_device(dense, d_x, n)
        ctx.ias_update_device(again, d_x, n)
        want = ctx.scene_export(by_host)
        for top in (strided, dense, again):
            assert same_export(ctx.scene_export(top), want)
        ctx.ias_update_device(again, d_x, n)                              # the same inputs once more: the same bytes
        assert same_export(ctx.scene_export(again), want)
        ctx.free(d_rec)
        ctx.free(d_x)


@pytest.mark.parametrize("bounds", ["tight", "box"])
def test_interleavings(cuda_device, monkeypatch, bounds):
    """Two GAS, each instanced 150 times; every step is compared with the host twin taken through the same steps.  With
    RTC_INSTANCE_BOUNDS=box the boxes come from the GAS bounds (the build's, or the refitted ones on the device) instead of
    the transformed vertices."""
    monkeypatch.setenv("RTC_INSTANCE_BOUNDS", bounds)
    geo0, geo1 = soup(2000, seed=4, extent=0.04), soup(1500, seed=5, extent=0.05)
    rng = np.random.default_rng(9)
    xf0 = np.asarray([moved([0.3, 0, 0, a, 0, 0.3, 0, b, 0, 0, 0.3, c], seed=k) for k, (a, b, c) in enumerate(rng.uniform(-2, 2, size=(300, 3)))],
                     dtype=np.float32)
    insts = [(t, 0 if k < 150 else 1) for k, t in enumerate(xf0)]
    geos = [geo0, geo1]
    new0 = deform(geo0[0], 0.03, seed=2)
    rays = H.random_rays(50000, seed=6, lo=(-2.5,) * 3, hi=(2.5,) * 3, tmin=1e-5)
    xs = [np.asarray([moved(t, seed=100 * j + k) for k, t in enumerate(xf0)], dtype=np.float32) for j in range(1, 5)]
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, insts)
        top = s.build()
        assert same_export(ctx.scene_export(top), core.host_scene_export(geos, insts)[0])
        d_xs = [ctx.to_device(x) for x in xs]
        steps, current = [], xf0.copy()

        def check(step, hits=True):
            steps.append(step)
            twin, _ = core.host_scene_rebuild_export(geos, insts, steps)
            export = ctx.scene_export(top)
            assert same_export(export, twin), len(steps)
            if hits:
                fresh_scene = Scene(ctx, [(new0, geo0[1]), geo1], insts)
                fresh = fresh_scene.build(current)
                check_hits(ctx, top, fresh, rays, export)
                ctx.scene_destroy(fresh)

        # a GAS refit, then a device update of a sub-range: instances of the refitted GAS outside it keep their matrices
        ctx.upload(s.keep[0], new0)
        ctx.gas_refit(s.gas[0])
        on_refitted = s.build()                                           # reads GAS 0's refitted bounds on the device
        assert same_export(ctx.scene_export(on_refitted), core.host_scene_export([(new0, geo0[1]), geo1], insts)[0])
        ctx.scene_destroy(on_refitted)
        ctx.ias_update_device(top, d_xs[0] + 48 * 100, 100, first=100)
        current[100:200] = xs[0][100:200]
        check(([new0, None], current.copy()))
        ctx.ias_update(top, xs[1])                                        # host update
        current = xs[1].copy()
        check(([None, None], current.copy()))
        ctx.ias_update_device(top, d_xs[2], 300)
        current = xs[2].copy()
        check(([None, None], current.copy()))
        ctx.ias_rebuild(top)
        check("rebuild")
        ctx.ias_update_device(top, d_xs[3] + 48 * 10, 50, first=10)
        current[10:60] = xs[3][10:60]
        check(([None, None], current.copy()))
        # GAS 1's vertex buffer rewritten in place but not refitted, GAS 0 refitted: a device update of GAS 0 instances only
        # recomputes GAS 0's instances, and GAS 1's keep their bytes
        ctx.upload(s.keep[2], deform(geo1[0], 0.2, seed=3))
        ctx.gas_refit(s.gas[0])
        ctx.ias_update_device(top, d_xs[0] + 48 * 20, 30, first=20)
        current[20:50] = xs[0][20:50]
        check(([new0, None], current.copy()), hits=False)
        for d in d_xs:
            ctx.free(d)


def _frame_after_update(files, k, device):
    """render(k), move every instance (moved()) with ias_update_device or ias_update, render(k) more"""
    app = host.App(*files)
    try:
        assert app.render(k) == k
        app.frame()                                                      # the iterations held back so far have run
        ctx = app.context(0)
        top = app.system_data().topObject
        n = app.info.numInstances
        x = np.asarray([moved(app.instance(i)[0], seed=i) for i in range(n)], dtype=np.float32)
        d_x = ctx.to_device(x)
        if device:
            ctx.ias_update_device(top, d_x, n)
        else:
            ctx.ias_update(top, x)
        assert app.render(k) == 2 * k
        frame = app.frame()
        ctx.free(d_x)
        return frame
    finally:
        app.close()


@pytest.mark.parametrize("scene", ["rtigo3_geometry", "rtigo3_textures", "stress"])
def test_frames_equal_the_host_update(cuda_device, tmp_path, scene):
    """The textured scene has cutout materials: the cached graph of the ordered any-hit rounds runs across the update."""
    files = _stress(tmp_path) if scene == "stress" else (H.write_system(tmp_path, scene, resolution="96 64", samplesSqrt=2), H.scene_path(scene))
    want = _frame_after_update(files, 2, device=False)
    got = _frame_after_update(files, 2, device=True)
    assert got.tobytes() == want.tobytes()


def _long_launch(ctx, sys_data, app):
    """enqueues about half a second of rendering"""
    ctx.synchronize()
    t0 = time.perf_counter()
    ctx.launch(sys_data, 1920, 1080, core.RAYGEN_FULL_FRAME, app.info.miss, 0, 4)
    ctx.synchronize()
    per_iteration = (time.perf_counter() - t0) / 4
    ctx.launch(sys_data, 1920, 1080, core.RAYGEN_FULL_FRAME, app.info.miss, 0, int(min(2000, max(8, 0.5 / per_iteration))))


def _big_app(tmp_path):
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="1920 1080", samplesSqrt=1), H.scene_path("rtigo3_geometry"))
    app.render(1)
    app.frame()                                                          # the App's output buffer exists
    ctx = app.context(0)
    ctx.set_trace_schedule("group")                                      # no timed batch, so no launch waits for the schedule tuner
    return app, ctx


def test_does_not_block_the_host(cuda_device, tmp_path):
    app, ctx = _big_app(tmp_path)
    try:
        sys_data = app.system_data()
        top = sys_data.topObject
        n = app.info.numInstances
        x = np.asarray([app.instance(i)[0] for i in range(n)], dtype=np.float32)
        d_x = ctx.to_device(x)
        gas = int(ctx.scene_export(top)["instance_gas"][0])
        # load the update's kernels once, on a scene of its own: the first launch of a kernel may load its module
        side = ctx.ias_build(np.array([(x[0], 0, gas, 0, -1)], dtype=core.INSTANCE_DTYPE))
        ctx.ias_update_device(side, d_x, 1)
        ctx.synchronize()
        _long_launch(ctx, sys_data, app)
        ctx.ias_update_device(top, d_x, n)                               # the scene's very first update
        pending = stream_busy(ctx.stream)
        ctx.synchronize()
        assert pending, "the first rtc_ias_update_device of a scene returned after the launch had finished: it synchronised the host"
        ctx.gas_refit(gas)                                               # the GAS's refit scratch is allocated here, not below
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        ctx.ias_update(side, np.zeros((0, 12), dtype=np.float32))
        _long_launch(ctx, sys_data, app)
        ctx.gas_refit(gas)
        ctx.ias_update_device(top, d_x, 1)                               # a refitted GAS is pending: the candidate list
        pending = stream_busy(ctx.stream)
        ctx.synchronize()
        assert pending, "rtc_ias_update_device with a refitted GAS returned after the launch had finished: it synchronised the host"
        ctx.scene_destroy(side)
        ctx.free(d_x)
    finally:
        app.close()


def test_reads_the_buffer_in_stream_order(cuda_device, tmp_path):
    app, ctx = _big_app(tmp_path)
    try:
        sys_data = app.system_data()
        top = sys_data.topObject
        n = app.info.numInstances
        x0 = np.asarray([app.instance(i)[0] for i in range(n)], dtype=np.float32)
        x1 = np.asarray([moved(t, seed=i) for i, t in enumerate(x0)], dtype=np.float32)
        x2 = np.asarray([moved(t, seed=1000 + i) for i, t in enumerate(x0)], dtype=np.float32)
        d_x = ctx.to_device(x0)
        ctx.ias_update_device(top, d_x, n)                               # kernels loaded, scratch allocated
        ctx.synchronize()
        _long_launch(ctx, sys_data, app)
        ctx.upload_async(d_x, x1.ctypes.data, x1.nbytes)
        ctx.ias_update_device(top, d_x, n)
        ctx.upload_async(d_x, x2.ctypes.data, x2.nbytes)
        ctx.synchronize()
        got = ctx.scene_export(top)
        ctx.ias_update(top, x1)
        assert same_export(got, ctx.scene_export(top))
        ctx.ias_update(top, x2)
        assert not same_export(got, ctx.scene_export(top))
        ctx.free(d_x)
    finally:
        app.close()


def test_host_update_reads_page_locked_memory_during_the_call(cuda_device, tmp_path):
    """rtc_ias_update's `transforms` may be reused on return, also when it is page-locked (rtc_host_alloc), which a copy engine
    would read only when the stream gets there: refilled behind a long launch, the scene must still get the call's matrices."""
    app, ctx = _big_app(tmp_path)
    try:
        sys_data = app.system_data()
        top = sys_data.topObject
        n = app.info.numInstances
        x0 = np.asarray([app.instance(i)[0] for i in range(n)], dtype=np.float32)
        x1 = np.asarray([moved(t, seed=i) for i, t in enumerate(x0)], dtype=np.float32)
        x2 = np.asarray([moved(t, seed=1000 + i) for i, t in enumerate(x0)], dtype=np.float32)
        p = ctx.host_alloc(x1.nbytes)
        pinned = np.ctypeslib.as_array((C.c_float * x1.size).from_address(p)).reshape(n, 12)
        pinned[:] = x0
        ctx.ias_update(top, pinned)                                      # kernels loaded, scratch allocated
        ctx.synchronize()
        pinned[:] = x1
        _long_launch(ctx, sys_data, app)
        ctx.ias_update(top, pinned)
        pinned[:] = x2                                                   # the caller refills the buffer for its next frame
        pending = stream_busy(ctx.stream)
        ctx.synchronize()
        assert pending, "the launch had finished before the buffer was refilled: the test did not test anything"
        got = ctx.scene_export(top)
        ctx.ias_update(top, x1)
        assert same_export(got, ctx.scene_export(top))
        ctx.host_free(p)
    finally:
        app.close()


_TORCH_PRODUCER = r"""
import sys
import torch                                   # first: a host library loaded before it may bring another NCCL into the process
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[2]]
from test_cpu_ias_rebuild import random_instances
from test_gpu_ias_rebuild import Scene
from tweeker_raytracer_b200 import core
n = 1000
geos, insts = random_instances(n, seed=11, spread=10.0)
x = np.asarray([t for t, _ in insts], dtype=np.float32)
with core.Context(0) as ctx:
    s = Scene(ctx, geos, insts)
    by_device, by_host = s.build(), s.build()
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))
    with torch.cuda.stream(stream):
        src = torch.from_numpy(x).to("cuda:0")
        t = (src.view(n, 3, 4) * torch.tensor([1.5, 0.5, 2.0], device="cuda:0").view(1, 3, 1)).reshape(n, 12).contiguous()
        ctx.ias_update_device(by_device, t.data_ptr(), n)
    ctx.synchronize()
    ctx.ias_update(by_host, t.cpu().numpy())
    a, b = ctx.scene_export(by_device), ctx.scene_export(by_host)
    for k in ("tlas_nodes", "tlas_leaves", "world_to_object"):
        assert a[k].tobytes() == b[k].tobytes(), k
print("same bytes")
"""


def test_torch_producer_on_the_context_stream(cuda_device):
    """A PyTorch producer writes the matrices on the context stream (torch.cuda.ExternalStream); the update reads them in order.
    In an interpreter of its own, which imports torch before the library."""
    r = subprocess.run([sys.executable, "-c", _TORCH_PRODUCER, H.ROOT, os.path.join(H.ROOT, "tests")], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "same bytes" in r.stdout, r.stdout + r.stderr


def test_refusals(cuda_device):
    attrs, idx = soup(500, seed=3, extent=0.05)
    n = 4
    with core.Context(0) as ctx:
        s = Scene(ctx, [(attrs, idx)], [([1, 0, 0, k, 0, 1, 0, 0, 0, 0, 1, 0], 0) for k in range(n)])
        top = s.build()
        x = np.asarray([moved([1, 0, 0, k, 0, 1, 0, 0, 0, 0, 1, 0], seed=k) for k in range(n)], dtype=np.float32)
        d_x = ctx.to_device(x)
        before = ctx.scene_export(top)
        cases = [
            (dict(top=12345, d_transforms=d_x, count=1), "unknown topObject"),
            (dict(top=top, d_transforms=d_x, count=1, first=n), "out of bounds"),
            (dict(top=top, d_transforms=d_x, count=n, first=1), "out of bounds"),
            (dict(top=top, d_transforms=0, count=1), "null"),
            (dict(top=top, d_transforms=d_x + 2, count=1), "aligned"),
            (dict(top=top, d_transforms=d_x, count=1, stride=44), "strideBytes"),
            (dict(top=top, d_transforms=d_x, count=1, stride=50), "strideBytes"),
            (dict(top=top, d_transforms=d_x, count=0, stride=0), "strideBytes"),
        ]
        for kw, why in cases:
            with pytest.raises(core.RtcError, match=why):
                ctx.ias_update_device(**kw)
            ctx.synchronize()
            assert same_export(ctx.scene_export(top), before), kw
        ctx.ias_update_device(top, 0, 0)                                  # count == 0 with a null pointer is allowed
        assert ctx.L.rtc_ias_update(ctx.h, top, 0, 1, C.c_void_p(d_x)) != 0   # rtc_ias_update reads host memory only
        assert "rtc_ias_update_device" in ctx.L.rtc_last_error().decode()
        assert same_export(ctx.scene_export(top), before)
        ctx.gas_destroy(s.gas[0])
        with pytest.raises(core.RtcError, match="a GAS of this scene was destroyed"):
            ctx.ias_update_device(top, d_x, n)
        ctx.free(d_x)
