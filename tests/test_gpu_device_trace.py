"""GPU tests of the device-side queries of include/rtc_device.cuh: user kernels (tests/native/device_trace_kernels.cu, built here by
nvcc with -Iinclude alone, once with the default flags and once with -fmad=false) that call rtc_device_trace_closest /
rtc_device_trace_any on a scene's topObject.

  * bit-identical to rtc_trace_closest / rtc_trace_any, and to the _ex calls with one mask and flag set, on a 1 M-triangle soup
    (coherent and incoherent rays), the host app's geometry scene and a small instanced scene with mirrored and scaled instances;
  * per-ray masks and flags equal the _ex calls run once per distinct (mask, flags) on the rays that have it;
  * both builds of the module agree; odd lanes only, blocks of 32 / 96 / 1024 threads and empty intervals;
  * a fused ambient-occlusion kernel equals rtc_trace_closest + a ray-writing kernel + rtc_trace_any;
  * in a created scene, user kernels interleaved with device builds, updates and rebuilds on the context stream, without a host
    synchronisation, equal rtc_trace_closest enqueued at the same points;
  * after a GAS rebuild, refit or destroy the queries refuse the scene (RTC_DEVICE_SCENE_UNUSABLE) until the update that cures it."""
import numpy as np
import pytest

import helpers as H
from device_trace import Module
from test_gpu_builder import soup
from test_gpu_ias_rebuild import Scene
from tweeker_raytracer_b200 import core, host

pytestmark = pytest.mark.gpu

OK, UNUSABLE, BAD_ARGUMENT = 0, 1, 2
FLAG_SETS = [0, core.RAY_CULL_BACK_FACING, core.RAY_CULL_FRONT_FACING, core.RAY_CULL_BACK_FACING | core.RAY_CULL_FRONT_FACING]
IDENTITY = [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0]


@pytest.fixture(scope="module")
def modules(cuda_device, tmp_path_factory):
    d = tmp_path_factory.mktemp("device_trace")
    return Module(d), Module(d, ["-fmad=false"])


def coherent_rays(n, origin, lo, hi, seed):
    """a pinhole bundle: one origin, directions to a grid over the box [lo, hi] (z of the box's far side)"""
    side = int(np.sqrt(n))
    ys, xs = np.divmod(np.arange(side * side), side)
    target = np.stack([lo[0] + (xs + 0.5) / side * (hi[0] - lo[0]), lo[1] + (ys + 0.5) / side * (hi[1] - lo[1]),
                       np.full(side * side, lo[2])], axis=1)
    d = target - np.asarray(origin)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.zeros(side * side, dtype=core.RAY_DTYPE)
    rays["ox"], rays["oy"], rays["oz"] = origin
    rays["dx"], rays["dy"], rays["dz"] = d[:, 0], d[:, 1], d[:, 2]
    rays["tmin"], rays["tmax"] = 1e-5, 1e27
    return rays


def check_equal_to_batch(ctx, modules, top, rays, label, mask=0xFF, flags=0, short_tmax=0.5):
    """both module builds against rtc_trace_closest(_ex) and rtc_trace_any(_ex) with (mask, flags); returns the closest hits"""
    want = ctx.trace_closest_host(top, rays, mask=mask, flags=flags)
    short = rays.copy(); short["tmax"] = np.minimum(short["tmax"], short_tmax)
    want_any = ctx.trace_any_host(top, short, mask=mask, flags=flags)
    for m in modules:
        got, status = m.trace_host(ctx, top, rays, mask=mask, fl=flags)
        assert (status == OK).all() and H.hits_equal(got, want), label
        occ, status = m.trace_host(ctx, top, short, any_hit=True, mask=mask, fl=flags)
        assert (status == OK).all() and np.array_equal(occ, want_any), label
    return want


def soup_scene(ctx, n):
    attrs, idx = soup(n, seed=21, extent=float(n) ** (-1.0 / 3.0))
    keep = [ctx.to_device(attrs), ctx.to_device(idx)]
    gas = ctx.gas_build(keep[0], attrs.dtype.itemsize, len(attrs), keep[1], n, core.BUILD_GPU_LBVH)
    inst = np.zeros(1, dtype=core.INSTANCE_DTYPE)
    inst["transform"], inst["gas"], inst["lightIndex"] = IDENTITY, gas, -1
    return ctx.ias_build(inst), keep


def test_million_triangle_soup(modules):
    with core.Context(0) as ctx:
        top, keep = soup_scene(ctx, 1_000_000)
        coh = coherent_rays(400_000, (0.5, 0.5, 2.5), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), seed=1)
        incoh = H.random_rays(400_000, seed=2, lo=(0, 0, 0), hi=(1, 1, 1), tmin=1e-5)
        for label, rays in (("coherent", coh), ("incoherent", incoh)):
            hits = check_equal_to_batch(ctx, modules, top, rays, label, short_tmax=0.02)
            assert (hits["inst"] != 0xffffffff).mean() > 0.3, label
            for mask, flags in ((0x01, core.RAY_CULL_BACK_FACING), (0xFF, core.RAY_CULL_FRONT_FACING)):
                check_equal_to_batch(ctx, modules, top, rays[:100_000], (label, mask, flags), mask, flags, short_tmax=0.02)
        for m in modules:
            assert m.stack_overflows(ctx) == 0
        for p in keep:
            ctx.free(p)


def test_geometry_scene(modules, tmp_path):
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="256 256", samplesSqrt=1), H.scene_path("rtigo3_geometry"))
    try:
        ctx, top = app.context(0), app.system_data(0).topObject
        ref = H.oracle_scene(app)
        primary = ref.generate_primary(H.oracle_sys(app), 256, 256, 0)
        ref.close()
        for label, rays in (("primary", primary[primary["tmax"] > 0]), ("random", H.random_rays(200_000, 7))):
            hits = check_equal_to_batch(ctx, modules, top, rays, label)
            assert (hits["inst"] != 0xffffffff).mean() > 0.2, label
            check_equal_to_batch(ctx, modules, top, rays, (label, "cull back"), 0xFF, core.RAY_CULL_BACK_FACING)
    finally:
        app.close()


def instanced_scene(ctx):
    """a soup instanced five times: identity, mirrored and non-uniformly scaled, uniformly scaled, mirrored in one axis, rotated"""
    attrs, idx = soup(20_000, seed=4, extent=0.04)
    transforms = [IDENTITY, [-0.7, 0.2, 0, 1.5, 0.1, 1.3, 0.3, -0.5, 0, -0.4, 0.6, 2.0], [2.5, 0, 0, -1, 0, 2.5, 0, 0.5, 0, 0, 2.5, 1],
                  [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, -1, 0.25], [0, -1, 0, 2, 1, 0, 0, -1, 0, 0, 1, -2]]
    s = Scene(ctx, [(attrs, idx)], [(np.asarray(t, dtype=np.float32), 0) for t in transforms])
    return s, s.build(), H.random_rays(200_000, seed=9, lo=(-2, -2, -2), hi=(3.5, 3, 3.5), tmin=1e-5)


def test_small_instanced_scene(modules):
    with core.Context(0) as ctx:
        s, top, rays = instanced_scene(ctx)
        hits = check_equal_to_batch(ctx, modules, top, rays, "all visible")
        assert len(set(hits["inst"][hits["inst"] != 0xffffffff].tolist())) == 5
        ctx.set_instance_masks(top, 0, np.array([0x01, 0x02, 0x03, 0x00, 0x80], dtype=np.uint8))
        for flags in FLAG_SETS:
            for mask in (0xFF, 0x01, 0x82):
                check_equal_to_batch(ctx, modules, top, rays[:50_000], (mask, flags), mask, flags)


def test_per_ray_masks_equal_ex_per_distinct_mask(modules):
    with core.Context(0) as ctx:
        s, top, rays = instanced_scene(ctx)
        ctx.set_instance_masks(top, 0, np.array([0x01, 0x02, 0x04, 0x08, 0x10], dtype=np.uint8))
        rng = np.random.default_rng(3)
        palette = np.array([0x00, 0x01, 0x03, 0x06, 0x0C, 0x10, 0x15, 0xFF], dtype=np.uint32)
        masks = palette[rng.integers(0, len(palette), size=len(rays))]
        flags = np.asarray(FLAG_SETS, dtype=np.uint32)[rng.integers(0, 4, size=len(rays))]
        short = rays.copy(); short["tmax"] = 0.5
        results = [(m.trace_host(ctx, top, rays, masks=masks, flags=flags), m.trace_host(ctx, top, short, True, masks=masks, flags=flags))
                   for m in modules]
        for (hits, st), (occ, st_any) in results:
            assert (st == OK).all() and (st_any == OK).all()
            for mk, fl in sorted(set(zip(masks.tolist(), flags.tolist()))):
                sel = np.flatnonzero((masks == mk) & (flags == fl))
                assert H.hits_equal(hits[sel], ctx.trace_closest_host(top, rays[sel], mask=mk, flags=fl)), (mk, fl)
                assert np.array_equal(occ[sel], ctx.trace_any_host(top, short[sel], mask=mk, flags=fl)), (mk, fl)
        # per-ray refusals in the same launch: a miss for those rays only
        bad = masks.copy(); bad[::7] = 0x100
        hits, st = modules[0].trace_host(ctx, top, rays, masks=bad, flags=flags)
        assert (st[::7] == BAD_ARGUMENT).all() and (hits["inst"][::7] == 0xffffffff).all() and (hits["t"][::7] == -1).all()
        keep = np.ones(len(rays), dtype=bool); keep[::7] = False
        assert (st[keep] == OK).all() and H.hits_equal(hits[keep], results[0][0][0][keep])


@pytest.mark.parametrize("block", [32, 96, 1024])
def test_odd_lanes_block_sizes_and_empty_intervals(modules, block):
    with core.Context(0) as ctx:
        s, top, rays = instanced_scene(ctx)
        rays = rays[:100_000].copy()
        rays["tmax"][5::11] = rays["tmin"][5::11]                  # empty intervals
        rays["tmax"][9::13] = -1.0
        want = ctx.trace_closest_host(top, rays)
        want_any = ctx.trace_any_host(top, rays)
        odd = np.arange(len(rays)) % 2 == 1
        for m in modules:
            got, st = m.trace_host(ctx, top, rays, block=block, odd_only=True)
            assert (st[odd] == OK).all() and (st[~odd] == -1).all()
            assert H.hits_equal(got[odd], want[odd])
            assert (got.view(np.uint8).reshape(len(rays), 20)[~odd] == 0xAB).all()      # the even lanes wrote nothing
            occ, st = m.trace_host(ctx, top, rays, any_hit=True, block=block, odd_only=True)
            assert (st[odd] == OK).all() and np.array_equal(occ[odd], want_any[odd]) and (occ[~odd] == 0xABABABAB).all()
            got, st = m.trace_host(ctx, top, rays, block=block)
            assert (st == OK).all() and H.hits_equal(got, want)
        assert (want["inst"][5::11] == 0xffffffff).all() and (want["inst"][9::13] == 0xffffffff).all()


def test_fused_ambient_occlusion_equals_the_three_call_pipeline(modules, tmp_path):
    w, h, samples, radius = 512, 384, 8, 0.5
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="%d %d" % (w, h), samplesSqrt=1), H.scene_path("rtigo3_geometry"))
    try:
        ctx, top = app.context(0), app.system_data(0).topObject
        n = w * h
        d_primary = ctx.malloc(n * 32)
        ctx.generate_primary(app.system_data(0), w, h, 0, d_primary)
        bufs = [ctx.malloc(n * 20), ctx.malloc(n * 4), ctx.malloc(n * 20), ctx.malloc(n * samples * 32), ctx.malloc(n * samples * 4),
                ctx.malloc(n * 4)]
        fused_hits, fused_counts, hits, ao, occ, counts = bufs
        for m in modules:
            m.ao_fused(ctx, top, d_primary, n, samples, radius, fused_hits, fused_counts)
            m.ao_pipeline(ctx, top, d_primary, n, samples, radius, hits, ao, occ, counts)
            a, b = ctx.download(fused_hits, core.HIT_DTYPE, n), ctx.download(hits, core.HIT_DTYPE, n)
            ca, cb = ctx.download(fused_counts, np.uint32, n), ctx.download(counts, np.uint32, n)
            assert H.hits_equal(a, b) and np.array_equal(ca, cb)
            assert (a["inst"] != 0xffffffff).mean() > 0.3 and 0 < ca.mean() < samples
        for p in [d_primary] + bufs:
            ctx.free(p)
    finally:
        app.close()


def records(gas, transforms):
    out = np.zeros(len(transforms), dtype=core.INSTANCE_DTYPE)
    out["transform"] = np.asarray(transforms, dtype=np.float32).reshape(-1, 12)
    out["instanceId"], out["gas"], out["lightIndex"] = np.arange(len(transforms)), gas, -1
    return out


def test_created_scene_interleaved_with_device_builds(modules):
    """every stage: a user kernel and rtc_trace_closest enqueued back to back, with no host synchronisation from the first build
    to the last query"""
    m = modules[0]
    with core.Context(0) as ctx:
        a1, i1 = soup(30_000, seed=5, extent=0.05)
        a2, i2 = soup(10_000, seed=6, extent=0.1)
        rng = np.random.default_rng(8)
        t1 = [np.c_[np.eye(3) * rng.uniform(0.5, 1.5), rng.uniform(-1, 1, size=3)].reshape(-1) for _ in range(40)]
        t2 = [t + np.array([0, 0, 0, 0.3, 0, 0, 0, -0.2, 0, 0, 0, 0.1]) for t in t1]
        rays = H.random_rays(100_000, seed=10, lo=(-1.5, -1.5, -1.5), hi=(2.5, 2.5, 2.5), tmin=1e-5)
        n = len(rays)
        d_a1, d_i1, d_a2, d_i2 = ctx.to_device(a1), ctx.to_device(i1), ctx.to_device(a2), ctx.to_device(i2)
        gas = ctx.gas_create(40_000)
        top = ctx.ias_create(64)
        d_rec = ctx.to_device(records(gas, t1))
        d_t2 = ctx.to_device(np.asarray(t2, dtype=np.float32).reshape(-1, 12))
        d_rays = ctx.to_device(rays)
        stages = 6
        user = [ctx.malloc(n * 20) for _ in range(stages)]
        batch = [ctx.malloc(n * 20) for _ in range(stages)]
        d_st = [ctx.malloc(n * 4) for _ in range(stages)]
        ctx.synchronize()

        def probe(k):
            m.query(ctx, top, d_rays, n, user[k], d_status=d_st[k])
            ctx.trace_closest(top, d_rays, n, batch[k])

        ctx.gas_build_device(gas, d_a1, a1.dtype.itemsize, len(a1), d_i1, len(i1))
        ctx.ias_build_device(top, d_rec, 40)
        probe(0)
        ctx.ias_update_device(top, d_t2, 40)
        probe(1)
        ctx.ias_rebuild(top)
        probe(2)
        ctx.ias_update_device(top, d_rec, 20, first=0, stride=64)
        probe(3)
        ctx.gas_build_device(gas, d_a2, a2.dtype.itemsize, len(a2), d_i2, len(i2))
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        probe(4)
        ctx.ias_build_device(top, d_rec, 25)
        probe(5)
        results = []
        for k in range(stages):
            got, want = ctx.download(user[k], core.HIT_DTYPE, n), ctx.download(batch[k], core.HIT_DTYPE, n)
            assert (ctx.download(d_st[k], np.int32, n) == OK).all(), k
            assert H.hits_equal(got, want), k
            assert (got["inst"] != 0xffffffff).mean() > 0.05, k
            results.append(got)
        assert not H.hits_equal(results[0], results[1]) and not H.hits_equal(results[3], results[4])
        for p in [d_a1, d_i1, d_a2, d_i2, d_rec, d_t2, d_rays] + user + batch + d_st:
            ctx.free(p)


def statuses(m, ctx, top, rays):
    hits, st = m.trace_host(ctx, top, rays)
    occ, st_any = m.trace_host(ctx, top, rays, any_hit=True)
    return hits, occ, st, st_any


def check_refused(m, ctx, top, rays, label):
    hits, occ, st, st_any = statuses(m, ctx, top, rays)
    assert (st == UNUSABLE).all() and (st_any == UNUSABLE).all(), label
    assert (hits["inst"] == 0xffffffff).all() and (hits["t"] == -1).all() and (occ == 0).all(), label


def check_usable(m, ctx, top, rays, label):
    hits, occ, st, st_any = statuses(m, ctx, top, rays)
    assert (st == OK).all() and (st_any == OK).all(), label
    assert H.hits_equal(hits, ctx.trace_closest_host(top, rays)), label
    assert (hits["inst"] != 0xffffffff).any(), label


def test_unusable_after_gas_changes_until_the_update(modules):
    m = modules[0]
    with core.Context(0) as ctx:
        a, ix = soup(20_000, seed=12, extent=0.05)
        b, ib = soup(5_000, seed=13, extent=0.08)
        s = Scene(ctx, [(a, ix), (b, ib)], [(np.asarray(IDENTITY, dtype=np.float32), 0), (np.asarray(IDENTITY, dtype=np.float32), 1)])
        top = s.build()
        other = Scene(ctx, [(b, ib)], [(np.asarray(IDENTITY, dtype=np.float32), 0)])
        top_other = other.build()
        rays = H.random_rays(20_000, seed=14, lo=(0, 0, 0), hi=(1, 1, 1), tmin=1e-5)
        check_usable(m, ctx, top, rays, "built")
        ctx.gas_rebuild(s.gas[0])                                   # the first rebuild of a referenced GAS
        check_refused(m, ctx, top, rays, "after the first rebuild")
        check_usable(m, ctx, top_other, rays, "a scene that does not reference it")
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        check_usable(m, ctx, top, rays, "after the update")
        ctx.gas_refit(s.gas[0])
        check_refused(m, ctx, top, rays, "after a refit")
        ctx.ias_update_device(top, 0, 0)
        check_usable(m, ctx, top, rays, "after the device update")
        ctx.gas_destroy(s.gas[1])
        check_refused(m, ctx, top, rays, "after the destroy")
        check_usable(m, ctx, top_other, rays, "the other scene")

        # a created scene: stale after any GAS change of the context, refused after the destroy of a handle it references
        gas = ctx.gas_create(20_000)
        d_a, d_i = ctx.to_device(a), ctx.to_device(ix)
        ctx.gas_build_device(gas, d_a, a.dtype.itemsize, len(a), d_i, len(ix))
        created = ctx.ias_create(4)
        d_rec = ctx.to_device(records(gas, [IDENTITY]))
        d_rec_other = ctx.to_device(records(s.gas[0], [IDENTITY]))
        ctx.ias_build_device(created, d_rec, 1)
        check_usable(m, ctx, created, rays, "created")
        ctx.gas_rebuild(s.gas[0])                                   # not referenced, but the created scene cannot know
        check_refused(m, ctx, created, rays, "created, after a rebuild of another GAS")
        ctx.ias_update(created, np.zeros((0, 12), dtype=np.float32))
        check_usable(m, ctx, created, rays, "created, after the update")
        ctx.gas_destroy(gas)
        check_refused(m, ctx, created, rays, "created, after the destroy")
        ctx.ias_build_device(created, d_rec_other, 1)
        check_usable(m, ctx, created, rays, "created, rebuilt over a live GAS")
        for p in (d_a, d_i, d_rec, d_rec_other):
            ctx.free(p)
        assert m.stack_overflows(ctx) == 0
