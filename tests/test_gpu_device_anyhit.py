"""GPU tests of the any-hit callbacks of include/rtc_device.cuh: user kernels (tests/native/device_anyhit_kernels.cu, built here by
nvcc with -Iinclude alone, once with the default flags and once with -fmad=false) whose lambdas decide with
tests/native/anyhit_predicates.h.

  * the always-accept callback equals rtc_trace_closest_ex / rtc_trace_any_ex on a 1 M-triangle soup (coherent and incoherent
    rays), the geometry scene and an instanced scene with mirrored and scaled instances;
  * every predicate, the all-hits enumeration and accept-and-end equal the host build of the header over the same exported
    structure, bit for bit, call counts and digests included; on the geometry scene also brute force;
  * the self-skip kernel equals the host build and brute force without the primary's triangle;
  * blocks of 32, 96 and 1024 threads, odd lanes only, empty intervals;
  * a created scene with device builds, updates and rebuilds interleaved on the stream;
  * after a GAS rebuild the queries refuse the scene and the callback is never called."""
import numpy as np
import pytest

import helpers as H
from device_anyhit import ACCEPT, ALPHA, FRONT, IGNORE, NOT_SELF, Args, Module, brute_any, brute_candidates, brute_closest, host_trace, per_ray
from mask_oracle import MaskedScene
from test_gpu_builder import soup
from test_gpu_device_trace import IDENTITY, coherent_rays, instanced_scene, records, soup_scene
from test_gpu_ias_rebuild import Scene
from tweeker_raytracer_b200 import core, host

pytestmark = pytest.mark.gpu

OK, UNUSABLE = 0, 1
ALPHA_TRANSPARENT = 96
PREDICATES = [(ACCEPT, 0), (ALPHA, ALPHA_TRANSPARENT), (FRONT, 0)]


@pytest.fixture(scope="module")
def modules(cuda_device, tmp_path_factory):
    d = tmp_path_factory.mktemp("device_anyhit")
    return Module(d), Module(d, ["-fmad=false"])


def check_accept_equals_batch(ctx, modules, top, rays, label, mask=0xFF, flags=0, short_tmax=0.5):
    want = ctx.trace_closest_host(top, rays, mask=mask, flags=flags)
    short = rays.copy(); short["tmax"] = np.minimum(short["tmax"], short_tmax)
    want_any = ctx.trace_any_host(top, short, mask=mask, flags=flags)
    for m in modules:
        got = m.trace_host(ctx, top, rays, mask=mask, fl=flags)
        assert (got["status"] == OK).all() and H.hits_equal(got["out"], want), label
        got = m.trace_host(ctx, top, short, any_hit=True, mask=mask, fl=flags)
        assert (got["status"] == OK).all() and np.array_equal(got["out"], want_any), label
    return want


def check_against_host(ctx, modules, top, rays, inst_masks, ray_masks, ray_flags, label):
    """every predicate (closest and any), all hits and accept-and-end against the host build over the exported structure"""
    export = ctx.scene_export(top)
    n = len(rays)
    rm, rf = per_ray(ray_masks, n), per_ray(ray_flags, n)
    cases = [("closest", p, q, False) for p, q in PREDICATES] + [("any", p, q, False) for p, q in PREDICATES]
    cases += [("any", IGNORE, 0, False), ("closest", ALPHA, ALPHA_TRANSPARENT, True)]
    for mode, pred, p0, end in cases:
        want = host_trace(export, inst_masks, rays, rm, rf, mode=mode, pred=pred, p0=p0, end=end, k=1)
        assert (want["status"] == OK).all() and want["duplicates"] == 0
        for m in modules:
            got = m.trace_host(ctx, top, rays, any_hit=mode == "any", pred=pred, p0=per_ray(p0, n), end=end, masks=rm, flags=rf)
            same = H.hits_equal(got["out"], want["out"]) if mode == "closest" else np.array_equal(got["out"], want["out"])
            assert (got["status"] == OK).all() and same, (label, mode, pred, end)
            assert np.array_equal(got["calls"], want["calls"]) and np.array_equal(got["digest"], want["digest"]), (label, mode, pred, end)
    return export


def test_million_triangle_soup(modules):
    with core.Context(0) as ctx:
        top, keep = soup_scene(ctx, 1_000_000)
        coh = coherent_rays(400_000, (0.5, 0.5, 2.5), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), seed=1)
        incoh = H.random_rays(400_000, seed=2, lo=(0, 0, 0), hi=(1, 1, 1), tmin=1e-5)
        rng = np.random.default_rng(3)
        for label, rays in (("coherent", coh), ("incoherent", incoh)):
            hits = check_accept_equals_batch(ctx, modules, top, rays, label, short_tmax=0.02)
            assert (hits["inst"] != 0xffffffff).mean() > 0.3, label
            check_accept_equals_batch(ctx, modules, top, rays[:100_000], label, 0x01, core.RAY_CULL_BACK_FACING, short_tmax=0.02)
            sub = rays[::40].copy()
            check_against_host(ctx, modules, top, sub, np.full(1, 0xFF, np.uint8), 0xFF,
                               np.asarray([0, 1, 2], dtype=np.uint32)[rng.integers(0, 3, size=len(sub))], label)
        for m in modules:
            assert m.stack_overflows(ctx) == 0
        for p in keep:
            ctx.free(p)


def test_geometry_scene_and_self_skip(modules, tmp_path):
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="256 256", samplesSqrt=1), H.scene_path("rtigo3_geometry"))
    try:
        ctx, top = app.context(0), app.system_data(0).topObject
        ref = MaskedScene(H.oracle_scene(app), app.info.numInstances)
        primary = ref.scene.generate_primary(H.oracle_sys(app), 256, 256, 0)
        primary = primary[primary["tmax"] > 0]
        random = H.random_rays(100_000, 7)
        for label, rays in (("primary", primary), ("random", random)):
            check_accept_equals_batch(ctx, modules, top, rays, label)
            check_accept_equals_batch(ctx, modules, top, rays, label, 0xFF, core.RAY_CULL_BACK_FACING)
        rays = np.concatenate([primary[::4], random[:20_000]])
        inst_masks = np.full(app.info.numInstances, 0xFF, np.uint8)
        check_against_host(ctx, modules, top, rays, inst_masks, 0xFF, 0, "geometry")
        # brute force on a subset
        few = rays[::300].copy()
        for pred, p0 in PREDICATES:
            got = modules[0].trace_host(ctx, top, few, pred=pred, p0=per_ray(p0, len(few)))["out"]
            assert H.hits_equal(got, brute_closest(ref, few, pred=pred, p0=p0)), pred
            occ = modules[0].trace_host(ctx, top, few, any_hit=True, pred=pred, p0=per_ray(p0, len(few)))["out"]
            assert np.array_equal(occ.astype(bool), brute_any(ref, few, pred=pred, p0=p0).astype(bool)), pred
        got = modules[0].trace_host(ctx, top, few, any_hit=True, pred=IGNORE)
        _, counts = brute_candidates(ref, few)
        assert np.array_equal(got["calls"], counts) and counts.sum() > len(few)

        # self-skip: a secondary ray from the primary hit with tmin = 0 that ignores the primary's triangle
        n = len(primary)
        d_p = ctx.to_device(primary)
        bufs = [ctx.malloc(n * 20), ctx.malloc(n * 32), ctx.malloc(n * 20)]
        export = ctx.scene_export(top)
        for m in modules:
            m.self_skip(ctx, top, d_p, n, *bufs)
            first = ctx.download(bufs[0], core.HIT_DTYPE, n)
            sec = ctx.download(bufs[1], core.RAY_DTYPE, n)
            second = ctx.download(bufs[2], core.HIT_DTYPE, n)
            assert H.hits_equal(first, ctx.trace_closest_host(top, primary))
            want = host_trace(export, inst_masks, sec, mode="closest", pred=NOT_SELF, p0=first["inst"], p1=first["prim"], k=1)["out"]
            assert H.hits_equal(second, want)
            assert not ((second["inst"] == first["inst"]) & (second["prim"] == first["prim"]) & (first["inst"] != 0xffffffff)).any()
            sel = np.flatnonzero(first["inst"] != 0xffffffff)[::400]
            assert H.hits_equal(second[sel], brute_closest(ref, sec[sel], pred=NOT_SELF, p0=first["inst"][sel], p1=first["prim"][sel]))
        for p in [d_p] + bufs:
            ctx.free(p)
        for m in modules:
            assert m.stack_overflows(ctx) == 0
        ref.close()
    finally:
        app.close()


def test_small_instanced_scene(modules):
    with core.Context(0) as ctx:
        s, top, rays = instanced_scene(ctx)
        check_accept_equals_batch(ctx, modules, top, rays, "all visible")
        inst_masks = np.array([0x01, 0x02, 0x03, 0x00, 0x80], dtype=np.uint8)
        ctx.set_instance_masks(top, 0, inst_masks)
        for flags in (0, core.RAY_CULL_BACK_FACING, core.RAY_CULL_FRONT_FACING):
            check_accept_equals_batch(ctx, modules, top, rays[:50_000], (0x82, flags), 0x82, flags)
        rng = np.random.default_rng(5)
        sub = rays[:40_000]
        ray_masks = np.array([0x00, 0x01, 0x03, 0x82, 0xFF], dtype=np.uint32)[rng.integers(0, 5, size=len(sub))]
        ray_flags = np.array([0, 1, 2, 3], dtype=np.uint32)[rng.integers(0, 4, size=len(sub))]
        check_against_host(ctx, modules, top, sub, inst_masks, ray_masks, ray_flags, "instanced")


@pytest.mark.parametrize("block", [32, 96, 1024])
def test_odd_lanes_block_sizes_and_empty_intervals(modules, block):
    with core.Context(0) as ctx:
        s, top, rays = instanced_scene(ctx)
        rays = rays[:100_000].copy()
        rays["tmax"][5::11] = rays["tmin"][5::11]
        rays["tmax"][9::13] = -1.0
        n = len(rays)
        odd = np.arange(n) % 2 == 1
        for any_hit, pred in ((False, ALPHA), (True, IGNORE)):
            full = modules[0].trace_host(ctx, top, rays, any_hit=any_hit, pred=pred, p0=per_ray(ALPHA_TRANSPARENT, n))
            assert (full["status"] == OK).all() and (full["calls"][5::11] == 0).all() and (full["calls"][9::13] == 0).all()
            assert full["calls"].sum() > n // 10
            for m in modules:
                got = m.trace_host(ctx, top, rays, any_hit=any_hit, pred=pred, p0=per_ray(ALPHA_TRANSPARENT, n), block=block, odd_only=True)
                assert (got["status"][odd] == OK).all() and (got["status"][~odd] == -1).all()
                assert (got["calls"][~odd] == 0xffffffff).all() and np.array_equal(got["calls"][odd], full["calls"][odd])
                assert np.array_equal(got["digest"][odd], full["digest"][odd])
                if any_hit:
                    assert np.array_equal(got["out"][odd], full["out"][odd]) and (got["out"][~odd] == 0xABABABAB).all()
                else:
                    assert H.hits_equal(got["out"][odd], full["out"][odd])
                    assert (got["out"].view(np.uint8).reshape(n, 20)[~odd] == 0xAB).all()
                got = m.trace_host(ctx, top, rays, any_hit=any_hit, pred=pred, p0=per_ray(ALPHA_TRANSPARENT, n), block=block)
                assert np.array_equal(got["calls"], full["calls"]) and np.array_equal(got["digest"], full["digest"])


def enqueue(m, ctx, top, d_rays, n, d_out, d_status, d_calls, pred=ACCEPT, any_hit=False):
    a = Args(top=int(top), rays=int(d_rays), out=int(d_out), status=int(d_status), calls=int(d_calls), n=n, mask=0xFF, fl=0, pred=pred)
    m._check(m.L.da_query(1 if any_hit else 0, a, 128, ctx.stream))


def test_created_scene_interleaved_with_device_builds(modules):
    """every stage: the always-accept and the alpha kernels and rtc_trace_closest enqueued back to back, with no host
    synchronisation from the first build to the last query"""
    m = modules[0]
    with core.Context(0) as ctx:
        a1, i1 = soup(30_000, seed=5, extent=0.05)
        a2, i2 = soup(10_000, seed=6, extent=0.1)
        rng = np.random.default_rng(8)
        t1 = [np.c_[np.eye(3) * rng.uniform(0.5, 1.5), rng.uniform(-1, 1, size=3)].reshape(-1) for _ in range(40)]
        t2 = [t + np.array([0, 0, 0, 0.3, 0, 0, 0, -0.2, 0, 0, 0, 0.1]) for t in t1]
        rays = H.random_rays(50_000, seed=10, lo=(-1.5, -1.5, -1.5), hi=(2.5, 2.5, 2.5), tmin=1e-5)
        n = len(rays)
        d_a1, d_i1, d_a2, d_i2 = ctx.to_device(a1), ctx.to_device(i1), ctx.to_device(a2), ctx.to_device(i2)
        gas = ctx.gas_create(40_000)
        top = ctx.ias_create(64)
        d_rec = ctx.to_device(records(gas, t1))
        d_t2 = ctx.to_device(np.asarray(t2, dtype=np.float32).reshape(-1, 12))
        d_rays = ctx.to_device(rays)
        stages = 5
        bufs = [[ctx.malloc(n * 20) for _ in range(3)] + [ctx.malloc(n * 4) for _ in range(4)] for _ in range(stages)]
        ctx.synchronize()

        def probe(k):
            accept, alpha, batch, st0, st1, c0, c1 = bufs[k]
            enqueue(m, ctx, top, d_rays, n, accept, st0, c0)
            enqueue(m, ctx, top, d_rays, n, alpha, st1, c1, pred=ALPHA)
            ctx.trace_closest(top, d_rays, n, batch)

        ctx.gas_build_device(gas, d_a1, a1.dtype.itemsize, len(a1), d_i1, len(i1))
        ctx.ias_build_device(top, d_rec, 40)
        probe(0)
        ctx.ias_update_device(top, d_t2, 40)
        probe(1)
        ctx.ias_rebuild(top)
        probe(2)
        ctx.gas_build_device(gas, d_a2, a2.dtype.itemsize, len(a2), d_i2, len(i2))
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        probe(3)
        ctx.ias_build_device(top, d_rec, 25)
        probe(4)
        export = ctx.scene_export(top)
        for k in range(stages):
            accept, alpha, batch, st0, st1, c0, c1 = bufs[k]
            want = ctx.download(batch, core.HIT_DTYPE, n)
            assert (ctx.download(st0, np.int32, n) == OK).all() and (ctx.download(st1, np.int32, n) == OK).all(), k
            assert H.hits_equal(ctx.download(accept, core.HIT_DTYPE, n), want), k
            assert (want["inst"] != 0xffffffff).mean() > 0.05, k
            got_alpha = ctx.download(alpha, core.HIT_DTYPE, n)
            assert not H.hits_equal(got_alpha, want), k
        host = host_trace(export, np.full(25, 0xFF, np.uint8), rays, mode="closest", pred=ALPHA, k=1)
        assert H.hits_equal(got_alpha, host["out"]) and np.array_equal(ctx.download(bufs[-1][6], np.uint32, n), host["calls"])
        for p in [d_a1, d_i1, d_a2, d_i2, d_rec, d_t2, d_rays] + [b for s in bufs for b in s]:
            ctx.free(p)
        assert m.stack_overflows(ctx) == 0


def test_refused_after_a_gas_rebuild_without_a_callback_call(modules):
    m = modules[0]
    with core.Context(0) as ctx:
        a, ix = soup(20_000, seed=12, extent=0.05)
        s = Scene(ctx, [(a, ix)], [(np.asarray(IDENTITY, dtype=np.float32), 0)])
        top = s.build()
        rays = H.random_rays(20_000, seed=14, lo=(0, 0, 0), hi=(1, 1, 1), tmin=1e-5)
        for any_hit in (False, True):
            got = m.trace_host(ctx, top, rays, any_hit=any_hit, pred=IGNORE)
            assert (got["status"] == OK).all() and got["calls"].sum() > 0
        ctx.gas_rebuild(s.gas[0])
        for any_hit in (False, True):
            got = m.trace_host(ctx, top, rays, any_hit=any_hit, pred=IGNORE)
            assert (got["status"] == UNUSABLE).all() and (got["calls"] == 0).all() and (got["digest"] == 0).all(), any_hit
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        got = m.trace_host(ctx, top, rays, any_hit=True, pred=IGNORE)
        assert (got["status"] == OK).all() and got["calls"].sum() > 0
        assert m.stack_overflows(ctx) == 0
