#!/usr/bin/env python
"""Refit against rebuild on one GPU; prints one JSON line per measurement, the first one naming the card and its power limit.

  python tools/refit_bench.py [--sizes 1M,10M,100M] [--rays 8M] [--repeats 5]

  * device-LBVH soups of bench.py's config 3 (centres uniform in the unit cube, edge n^(-1/3)): rtc_gas_build ms against
    rtc_gas_refit ms, and incoherent closest-hit Mrays/s after a smooth per-vertex displacement of 0, 0.5 and 2 mean edge lengths,
    refitted against rebuilt (the hits of the two are checked to be equal in the same run);
  * the same soups with their vertex triplets traded among the triangles (a random permutation: the refit's topology is
    useless): rtc_gas_rebuild ms (the first call, which allocates and synchronises, and the median of later ones), the device
    memory the first rebuild leaves resident, and incoherent closest-hit Mrays/s refitted (over the first thousandth of the rays),
    rebuilt on the device (rtc_gas_rebuild) and built anew by rtc_gas_build, whose hits are checked to be equal in the same run;
  * the 10 001-instance scene (tools/make_instances_scene.py): rtc_ias_build ms against rtc_ias_update ms with every instance and
    with 1 % of them moved, rtc_ias_update_device ms with every instance moved (matrices uploaded once, outside the timed call)
    and rtc_ias_rebuild ms, and incoherent closest-hit Mrays/s through the scene after 1, 10 and 100
    animation steps of small rotations and after a random permutation of the tori's transforms (same boxes, no spatial coherence
    left in the built topology): refitted, rebuilt on the device (rtc_ias_rebuild) and rebuilt by rtc_ias_build, whose hits are
    checked to be equal in the same run;
  * about a million small instances (a 12-triangle box on a jittered lattice): rtc_ias_build ms (one run) against
    rtc_ias_update ms and rtc_ias_update_device ms of every instance, and rtc_ias_rebuild ms;
  * an instance set that changes every step, on 10 001 and 1 M of those boxes (two meshes: a box and a smaller one, its level
    of detail): the whole set, a tenth of it despawned, and a tenth of the instances swapped to the other mesh with new
    materials.  Each is built into one scene of rtc_ias_create by rtc_ias_build_device from records already in device memory
    (device ms between events, and host ms of the call and its synchronisation), against rtc_ias_build of the same records and,
    for the counts a scene of rtc_ias_build can hold, rtc_ias_update_device + rtc_ias_rebuild; incoherent closest-hit Mrays/s of
    the created and the built scene after each, whose hits are checked to be equal in the same run.
  * --device-geometry: the traded soups above, built into one GAS of rtc_gas_create by rtc_gas_build_device from vertices and
    indices already in device memory: device ms between events and host ms of the call alone (its enqueue), against
    rtc_gas_build(RTC_BUILD_DEFAULT) host wall ms and rtc_gas_rebuild device ms of the same triangles; the device memory the
    created GAS holds per triangle of capacity; incoherent closest-hit Mrays/s of the result against the default build (the host
    SAH builder below 2^20 triangles), whose hits are checked to be equal in the same run; a count that changes between calls
    (0.9 n, n, 0.1 n into capacity n); and a build of n / 100 triangles into capacity n against the same build into a GAS of
    capacity n / 100 (the collapse graph's grids are sized for the capacity).
Builds are timed on the host clock (they end in a synchronisation); refits, updates and traces between CUDA events on the
context stream, each the median of `repeats` runs after one warm-up.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
import helpers as H  # noqa: E402
import make_instances_scene  # noqa: E402
from tweeker_raytracer_b200 import core, host  # noqa: E402


def emit(**kw):
    print(json.dumps(kw), flush=True)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = "nvidia-smi unavailable: %s" % e
    return out


def timed(ctx, fn, repeats):
    fn()
    ms = []
    for _ in range(repeats):
        ctx.timer_start()
        fn()
        ms.append(ctx.timer_stop())
    return float(np.median(ms))


def wall(ctx, fn, repeats):
    ms = []
    for _ in range(repeats):
        ctx.synchronize()
        t0 = time.perf_counter()
        fn()
        ctx.synchronize()
        ms.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ms))


def displace(verts, amount, edge, seed=7):
    """Smooth per-vertex displacement of `amount` mean edge lengths (a sine field over the position), float32, in chunks."""
    rng = np.random.default_rng(seed)
    k = rng.normal(size=(3, 3)).astype(np.float32) * np.float32(6.0)
    phase = rng.uniform(0, 2 * np.pi, size=3).astype(np.float32)
    out = np.empty_like(verts)
    chunk = 1 << 24
    for a in range(0, len(verts), chunk):
        v = verts[a:a + chunk]
        out[a:a + chunk] = v + np.float32(amount * edge) * np.sin(v @ k + phase)
    return out


def mem_free():
    """free bytes of the current device (cudaMemGetInfo of the runtime the library runs on)"""
    import ctypes as C
    cudart = C.CDLL("libcudart.so.12")
    free, total = C.c_size_t(0), C.c_size_t(0)
    assert cudart.cudaMemGetInfo(C.byref(free), C.byref(total)) == 0
    return free.value


def mrays(ctx, top, d_rays, nrays, d_hits, repeats):
    ms = timed(ctx, lambda: ctx.trace_closest(top, d_rays, nrays, d_hits), repeats)
    return nrays / ms / 1e3


def soup_runs(ctx, n, nrays, repeats):
    verts = bench.soup_numpy(n)
    edge = float(n) ** (-1.0 / 3.0)
    idx = np.arange(3 * n, dtype=np.uint32)
    d_v, d_i = ctx.malloc(verts.nbytes), ctx.malloc(idx.nbytes)
    ctx.upload(d_v, verts)
    ctx.upload(d_i, idx)
    del idx
    inst = np.zeros(1, dtype=core.INSTANCE_DTYPE)
    inst[0]["transform"] = [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0]
    def build():
        return ctx.gas_build(d_v, 12, 3 * n, d_i, n, core.BUILD_GPU_LBVH)

    build_ms = wall(ctx, lambda: ctx.gas_destroy(build()), repeats + 1)
    gas = build()
    inst[0]["gas"] = gas
    top = ctx.ias_build(inst)
    refit_ms = timed(ctx, lambda: ctx.gas_refit(gas), repeats)
    update_ms = timed(ctx, lambda: ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32)), repeats)
    emit(what="gas_build_vs_refit", triangles=n, builder="gpu_lbvh", build_ms=build_ms, refit_ms=refit_ms, ias_update_after_refit_ms=update_ms,
         speedup=build_ms / refit_ms)
    rays = bench.rays_numpy(nrays, "incoh", "closest")
    d_rays, d_hits, d_hits2 = ctx.malloc(rays.nbytes), ctx.malloc(20 * nrays), ctx.malloc(20 * nrays)
    ctx.upload(d_rays, rays)
    del rays
    for amount in (0.0, 0.5, 2.0):
        ctx.upload(d_v, displace(verts, amount, edge) if amount else verts)
        ctx.gas_refit(gas)
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        refit_rate = mrays(ctx, top, d_rays, nrays, d_hits, repeats)
        fresh = build()
        inst[0]["gas"] = fresh
        fresh_top = ctx.ias_build(inst)
        rebuilt_rate = mrays(ctx, fresh_top, d_rays, nrays, d_hits2, repeats)
        a = ctx.download(d_hits, np.uint8, 20 * nrays)
        b = ctx.download(d_hits2, np.uint8, 20 * nrays)
        emit(what="soup_trace_after_displacement", triangles=n, displacement_edges=amount, rays=nrays, refitted_mrays=refit_rate,
             rebuilt_mrays=rebuilt_rate, refitted_over_rebuilt=refit_rate / rebuilt_rate, hits_equal=bool(np.array_equal(a, b)))
        ctx.scene_destroy(fresh_top)
        ctx.gas_destroy(fresh)
    # the vertex triplets traded among the triangles: refitted, rebuilt on the device, built anew
    ctx.upload(d_v, verts.reshape(n, 9)[np.random.default_rng(3).permutation(n)].reshape(-1, 3))
    ctx.gas_refit(gas)
    ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
    # the refitted GAS traces three orders of magnitude slower: a thousandth of the rays (the first ones, whose hits are compared)
    nslow = max(1, nrays // 1000)
    refit_rate = mrays(ctx, top, d_rays, nslow, d_hits, repeats)
    ctx.synchronize()
    free0 = mem_free()
    first_ms = wall(ctx, lambda: ctx.gas_rebuild(gas), 1)
    resident = free0 - mem_free()
    rebuild_ms = timed(ctx, lambda: ctx.gas_rebuild(gas), repeats)
    ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
    rebuilt_rate = mrays(ctx, top, d_rays, nrays, d_hits2, repeats)
    fresh = build()
    inst[0]["gas"] = fresh
    fresh_top = ctx.ias_build(inst)
    d_hits3 = ctx.malloc(20 * nrays)
    built_rate = mrays(ctx, fresh_top, d_rays, nrays, d_hits3, repeats)
    a, b, c = (ctx.download(d, np.uint8, 20 * nrays) for d in (d_hits, d_hits2, d_hits3))
    a, b_head = a[:20 * nslow], b[:20 * nslow]
    emit(what="gas_rebuild", triangles=n, build_ms=build_ms, refit_ms=refit_ms, first_rebuild_ms=first_ms, rebuild_ms=rebuild_ms,
         resident_bytes_after_first_rebuild=resident, resident_bytes_per_triangle=resident / n)
    emit(what="soup_trace_after_trading_places", triangles=n, rays=nrays, refitted_rays=nslow, refitted_mrays=refit_rate, rebuilt_mrays=rebuilt_rate,
         built_mrays=built_rate, hits_equal=bool(np.array_equal(a, b_head) and np.array_equal(b, c)))
    ctx.scene_destroy(fresh_top)
    ctx.gas_destroy(fresh)
    ctx.scene_destroy(top)
    ctx.gas_destroy(gas)
    for p in (d_v, d_i, d_rays, d_hits, d_hits2, d_hits3):
        ctx.free(p)


def device_geometry_runs(ctx, n, nrays, repeats):
    verts = bench.soup_numpy(n)
    verts = verts.reshape(n, 9)[np.random.default_rng(3).permutation(n)].reshape(-1, 3)        # the traded soup
    idx = np.arange(3 * n, dtype=np.uint32)
    d_v, d_i = ctx.malloc(verts.nbytes), ctx.malloc(idx.nbytes)
    ctx.upload(d_v, verts)
    ctx.upload(d_i, idx)
    del verts, idx
    inst = np.zeros(1, dtype=core.INSTANCE_DTYPE)
    inst[0]["transform"] = [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0]
    default_ms = wall(ctx, lambda: ctx.gas_destroy(ctx.gas_build(d_v, 12, 3 * n, d_i, n)), 3)
    built = ctx.gas_build(d_v, 12, 3 * n, d_i, n)
    ctx.gas_rebuild(built)                                                  # the first rebuild allocates
    rebuild_ms = timed(ctx, lambda: ctx.gas_rebuild(built), repeats)
    ctx.gas_destroy(built)
    ctx.synchronize()
    free0 = mem_free()
    g = ctx.gas_create(n)
    resident = free0 - mem_free()
    device_ms = timed(ctx, lambda: ctx.gas_build_device(g, d_v, 12, 3 * n, d_i, n), repeats)
    call_ms = []
    for _ in range(repeats):
        ctx.synchronize()
        t0 = time.perf_counter()
        ctx.gas_build_device(g, d_v, 12, 3 * n, d_i, n)
        call_ms.append((time.perf_counter() - t0) * 1e3)
    inst[0]["gas"] = g
    top = ctx.ias_build(inst)
    default = ctx.gas_build(d_v, 12, 3 * n, d_i, n)
    inst[0]["gas"] = default
    default_top = ctx.ias_build(inst)
    rays = bench.rays_numpy(nrays, "incoh", "closest")
    d_rays, d_hits, d_hits2 = ctx.malloc(rays.nbytes), ctx.malloc(20 * nrays), ctx.malloc(20 * nrays)
    ctx.upload(d_rays, rays)
    del rays
    created_rate = mrays(ctx, top, d_rays, nrays, d_hits, repeats)
    default_rate = mrays(ctx, default_top, d_rays, nrays, d_hits2, repeats)
    a = ctx.download(d_hits, np.uint8, 20 * nrays)
    b = ctx.download(d_hits2, np.uint8, 20 * nrays)
    emit(what="gas_build_device", triangles=n, build_device_ms=device_ms, build_device_call_host_ms=float(np.median(call_ms)),
         gas_rebuild_ms=rebuild_ms, gas_build_default_wall_ms=default_ms,
         default_builder="host_sah" if n <= (1 << 20) else "gpu_lbvh", resident_bytes_of_create=resident,
         resident_bytes_per_triangle_of_capacity=resident / n, rays=nrays, created_mrays=created_rate, default_mrays=default_rate,
         created_over_default=created_rate / default_rate, hits_equal=bool(np.array_equal(a, b)))
    ctx.scene_destroy(top)
    ctx.scene_destroy(default_top)
    ctx.gas_destroy(default)
    # a count that changes from call to call, into the same GAS
    counts = [(9 * n) // 10, n, n // 10]
    ms = [timed(ctx, lambda: ctx.gas_build_device(g, d_v, 12, 3 * n, d_i, m), repeats) for m in counts]
    emit(what="gas_build_device_changing_count", capacity=n, triangles=counts, build_device_ms=ms)
    # n / 100 triangles into capacity n, against a GAS whose capacity is n / 100
    m = max(1, n // 100)
    big_ms = timed(ctx, lambda: ctx.gas_build_device(g, d_v, 12, 3 * n, d_i, m), repeats)
    small = ctx.gas_create(m)
    small_ms = timed(ctx, lambda: ctx.gas_build_device(small, d_v, 12, 3 * n, d_i, m), repeats)
    emit(what="gas_build_device_small_in_large", capacity=n, triangles=m, build_device_ms=big_ms, capacity_equal_ms=small_ms,
         idle_capacity_ms=big_ms - small_ms)
    ctx.gas_destroy(small)
    ctx.gas_destroy(g)
    for p in (d_v, d_i, d_rays, d_hits, d_hits2):
        ctx.free(p)


def rotation(angle, axis):
    c, s = np.cos(angle), np.sin(angle)
    r = np.eye(3)
    i, j = [(1, 2), (0, 2), (0, 1)][axis]
    r[i, i], r[i, j], r[j, i], r[j, j] = c, -s, s, c
    return r


def instance_runs(ctx, nrays, repeats):
    with tempfile.TemporaryDirectory() as tmp:
        scene = os.path.join(tmp, "instances.txt")
        make_instances_scene.write_scene(scene, count=10000)
        app = host.App(H.write_system(tmp, "rtigo3_instances", resolution="64 64", samplesSqrt=1), scene, host_only=True)
        try:
            geos = [app.geometry(g) for g in range(app.info.numGeometries)]
            insts = [app.instance(i)[:2] for i in range(app.info.numInstances)]
        finally:
            app.close()
    keep, handles = [], []
    for a, ix in geos:
        d_a, d_i = ctx.to_device(a), ctx.to_device(ix)
        keep += [d_a, d_i]
        handles.append(ctx.gas_build(d_a, a.dtype.itemsize, len(a), d_i, len(ix), core.BUILD_HOST_SAH))
    xf0 = np.asarray([t for t, _ in insts], dtype=np.float32).reshape(-1, 12)
    n = len(insts)

    def descs(xf):
        out = np.zeros(n, dtype=core.INSTANCE_DTYPE)
        out["transform"] = xf
        out["instanceId"] = np.arange(n)
        out["gas"] = [handles[g] for _, g in insts]
        out["lightIndex"] = -1
        return out

    tops = []
    build_ms = wall(ctx, lambda: tops.append(ctx.ias_build(descs(xf0))), repeats)
    for t in tops[1:]:
        ctx.scene_destroy(t)
    top = tops[0]

    def step(xf, k):
        """one animation step: every instance turns by a small angle about its own centre"""
        out = xf.reshape(n, 3, 4).astype(np.float64)
        out[:, :, :3] = out[:, :, :3] @ rotation(0.02 * (1 + k % 3), k % 3)
        return out.astype(np.float32).reshape(n, 12)

    moved = step(xf0, 0)
    all_ms = timed(ctx, lambda: ctx.ias_update(top, moved), repeats)
    few = max(1, n // 100)
    few_ms = timed(ctx, lambda: ctx.ias_update(top, moved[:few]), repeats)
    d_moved = ctx.to_device(moved)
    all_device_ms = timed(ctx, lambda: ctx.ias_update_device(top, d_moved, n), repeats)
    ctx.free(d_moved)
    spare = ctx.ias_build(descs(xf0))
    rebuild_ms = timed(ctx, lambda: ctx.ias_rebuild(spare), repeats)             # the warm-up is the scene's first rebuild
    ctx.scene_destroy(spare)
    emit(what="ias_build_vs_update", instances=n, build_ms=build_ms, update_all_ms=all_ms, update_1pct_ms=few_ms,
         update_all_device_ms=all_device_ms, rebuild_ms=rebuild_ms,
         speedup_all=build_ms / all_ms, speedup_1pct=build_ms / few_ms, build_over_rebuild=build_ms / rebuild_ms)

    lo, hi = xf0[:, [3, 7, 11]].min(axis=0) - 1.0, xf0[:, [3, 7, 11]].max(axis=0) + 1.0
    rays = bench.rays_numpy(nrays, "incoh", "closest")
    for c, k in zip("xyz", range(3)):
        rays["o" + c] = lo[k] + rays["o" + c] * (hi[k] - lo[k])
    d_rays, d_hits, d_hits2 = ctx.to_device(rays), ctx.malloc(20 * nrays), ctx.malloc(20 * nrays)
    d_hits3 = ctx.malloc(20 * nrays)

    def three_ways(refitted, xf, **row):
        """Mrays/s of the refitted scene, of a scene rebuilt on the device over the same boxes and of one rtc_ias_build built"""
        refit_rate = mrays(ctx, refitted, d_rays, nrays, d_hits, repeats)
        device = ctx.ias_build(descs(xf))
        ctx.ias_rebuild(device)
        device_rate = mrays(ctx, device, d_rays, nrays, d_hits3, repeats)
        fresh = ctx.ias_build(descs(xf))
        rebuilt_rate = mrays(ctx, fresh, d_rays, nrays, d_hits2, repeats)
        a = ctx.download(d_hits, np.uint8, 20 * nrays)
        b = ctx.download(d_hits2, np.uint8, 20 * nrays)
        c = ctx.download(d_hits3, np.uint8, 20 * nrays)
        emit(instances=n, rays=nrays, refitted_mrays=refit_rate, device_rebuilt_mrays=device_rate, rebuilt_mrays=rebuilt_rate,
             refitted_over_rebuilt=refit_rate / rebuilt_rate, device_rebuilt_over_rebuilt=device_rate / rebuilt_rate,
             hits_equal=bool(np.array_equal(a, b) and np.array_equal(a, c)), **row)
        ctx.scene_destroy(device)
        ctx.scene_destroy(fresh)

    xf = xf0.copy()
    ctx.ias_update(top, xf)
    done = 0
    for steps in (1, 10, 100):
        while done < steps:
            xf = step(xf, done)
            ctx.ias_update(top, xf)
            done += 1
        three_ways(top, xf, what="instances_trace_after_steps", steps=steps)
    # the tori trade places: every box keeps its size, the built topology no longer groups neighbours
    tori = np.array([i for i, (_, g) in enumerate(insts) if g == insts[-1][1]])
    permuted = xf0.copy()
    permuted[tori] = xf0[np.random.default_rng(1).permutation(tori)]
    ctx.ias_update(top, xf0)
    ctx.ias_update(top, permuted)
    three_ways(top, permuted, what="instances_trace_after_permutation")
    ctx.scene_destroy(top)
    for p in keep + [d_rays, d_hits, d_hits2, d_hits3]:
        ctx.free(p)


def box_mesh(size):
    v = np.array([[x, y, z] for x in (0, size) for y in (0, size) for z in (0, size)], dtype=np.float32)
    faces = [(0, 1, 3), (0, 3, 2), (4, 6, 7), (4, 7, 5), (0, 4, 5), (0, 5, 1), (2, 3, 7), (2, 7, 6), (0, 2, 6), (0, 6, 4), (1, 5, 7), (1, 7, 3)]
    attrs = np.zeros(8, dtype=[("vertex", "f4", 3), ("tangent", "f4", 3), ("normal", "f4", 3), ("texcoord", "f4", 3)])
    attrs["vertex"] = v
    return attrs, np.asarray(faces, dtype=np.uint32)


def many_instance_runs(ctx, count, repeats):
    side = int(round(count ** (1.0 / 3.0)))
    n = side ** 3
    rng = np.random.default_rng(3)
    attrs, idx = box_mesh(0.4)
    d_a, d_i = ctx.to_device(attrs), ctx.to_device(idx)
    gas = ctx.gas_build(d_a, attrs.dtype.itemsize, len(attrs), d_i, len(idx), core.BUILD_HOST_SAH)
    g = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), axis=-1).reshape(-1, 3).astype(np.float64)
    xf = np.zeros((n, 3, 4))
    xf[:, :, :3] = np.eye(3)
    xf[:, :, 3] = g + rng.uniform(-0.3, 0.3, size=(n, 3))
    xf = xf.astype(np.float32).reshape(n, 12)
    inst = np.zeros(n, dtype=core.INSTANCE_DTYPE)
    inst["transform"], inst["instanceId"], inst["gas"], inst["lightIndex"] = xf, np.arange(n), gas, -1
    tops = []
    build_ms = wall(ctx, lambda: tops.append(ctx.ias_build(inst)), 1)
    top = tops[0]
    update_ms = timed(ctx, lambda: ctx.ias_update(top, xf), repeats)
    d_xf = ctx.to_device(xf)
    update_device_ms = timed(ctx, lambda: ctx.ias_update_device(top, d_xf, n), repeats)
    ctx.free(d_xf)
    rebuild_ms = timed(ctx, lambda: ctx.ias_rebuild(top), repeats)
    emit(what="many_instances_build_vs_update_vs_rebuild", instances=n, build_ms=build_ms, build_runs=1, update_all_ms=update_ms,
         update_all_device_ms=update_device_ms, rebuild_ms=rebuild_ms, build_over_rebuild=build_ms / rebuild_ms)
    ctx.scene_destroy(top)
    ctx.gas_destroy(gas)
    ctx.free(d_a)
    ctx.free(d_i)


def changing_instance_runs(ctx, count, nrays, repeats):
    side = int(np.ceil(count ** (1.0 / 3.0)))
    n = count
    rng = np.random.default_rng(5)
    keep, gas = [], []
    for size in (0.4, 0.25):
        attrs, idx = box_mesh(size)
        d_a, d_i = ctx.to_device(attrs), ctx.to_device(idx)
        keep += [d_a, d_i]
        gas.append(ctx.gas_build(d_a, attrs.dtype.itemsize, len(attrs), d_i, len(idx), core.BUILD_HOST_SAH))
    g = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), axis=-1).reshape(-1, 3)[:n].astype(np.float64)
    xf = np.zeros((n, 3, 4))
    xf[:, :, :3] = np.eye(3)
    xf[:, :, 3] = g + rng.uniform(-0.3, 0.3, size=(n, 3))
    xf = xf.astype(np.float32).reshape(n, 12)
    full = np.zeros(n, dtype=core.INSTANCE_DTYPE)
    full["transform"], full["instanceId"], full["gas"], full["lightIndex"] = xf, np.arange(n), gas[0], -1
    swapped = full.copy()
    pick = rng.choice(n, n // 10, replace=False)
    swapped["gas"][pick] = gas[1]
    swapped["materialIndex"][pick] = 1
    variants = [("full", full), ("despawned", full[:n - n // 10].copy()), ("swapped", swapped)]
    rays = bench.rays_numpy(nrays, "incoh", "closest")
    for c, k in zip("xyz", range(3)):
        rays["o" + c] = -1.0 + rays["o" + c] * (side + 1.0)
    d_rays, d_hits, d_hits2 = ctx.to_device(rays), ctx.malloc(20 * nrays), ctx.malloc(20 * nrays)
    top = ctx.ias_create(n)
    for what, records in variants:
        d_rec = ctx.to_device(records)
        m = len(records)
        device_ms = timed(ctx, lambda: ctx.ias_build_device(top, d_rec, m), repeats)
        device_wall_ms = wall(ctx, lambda: ctx.ias_build_device(top, d_rec, m), repeats)
        tops = []
        build_ms = wall(ctx, lambda: tops.append(ctx.ias_build(records)), 1 if n > 100000 else repeats)
        for t in tops[1:]:
            ctx.scene_destroy(t)
        built = tops[0]
        d_xf = ctx.to_device(np.ascontiguousarray(records["transform"]))
        ctx.ias_rebuild(built)                                            # the scene's first rebuild allocates
        update_rebuild_ms = timed(ctx, lambda: (ctx.ias_update_device(built, d_xf, m), ctx.ias_rebuild(built)), repeats)
        ctx.free(d_xf)
        ctx.ias_build_device(top, d_rec, m)
        created_rate = mrays(ctx, top, d_rays, nrays, d_hits, repeats)
        built_fresh = ctx.ias_build(records)
        built_rate = mrays(ctx, built_fresh, d_rays, nrays, d_hits2, repeats)
        a = ctx.download(d_hits, np.uint8, 20 * nrays)
        b = ctx.download(d_hits2, np.uint8, 20 * nrays)
        emit(what="changing_instances_" + what, capacity=n, instances=m, build_device_ms=device_ms, build_device_wall_ms=device_wall_ms,
             ias_build_ms=build_ms, update_device_plus_rebuild_ms=update_rebuild_ms, ias_build_over_build_device=build_ms / device_ms,
             rays=nrays, created_mrays=created_rate, built_mrays=built_rate, hits_equal=bool(np.array_equal(a, b)),
             rejected=ctx.scene_rejected_instances(top))
        ctx.scene_destroy(built)
        ctx.scene_destroy(built_fresh)
        ctx.free(d_rec)
    ctx.scene_destroy(top)
    for h in gas:
        ctx.gas_destroy(h)
    for p in keep + [d_rays, d_hits, d_hits2]:
        ctx.free(p)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--sizes", default="1M,10M,100M")
    ap.add_argument("--rays", default="8M")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--no-instances", action="store_true")
    ap.add_argument("--many-instances", default="1M", help="instance count of the small-instance scene (0: skip)")
    ap.add_argument("--changing-instances", default="10001,1M", help="capacities of the changing instance sets (0: skip)")
    ap.add_argument("--device-geometry", default="", help="triangle counts of the rtc_gas_build_device runs, e.g. 1M,10M,100M")
    args = ap.parse_args()
    scale = {"K": 10 ** 3, "M": 10 ** 6}
    count = lambda s: int(float(s[:-1]) * scale[s[-1]]) if s[-1] in scale else int(s)    # noqa: E731
    if core.device_count() < 1:
        raise SystemExit("refit_bench needs a CUDA device: " + core.lib().rtc_last_error().decode())
    emit(what="card", nvidia_smi=card(), rtc_version=core.lib().rtc_version())
    with core.Context(0) as ctx:
        for s in filter(None, args.sizes.split(",")):
            soup_runs(ctx, count(s), count(args.rays), args.repeats)
        for s in filter(None, args.device_geometry.split(",")):
            device_geometry_runs(ctx, count(s), count(args.rays), args.repeats)
        if not args.no_instances:
            instance_runs(ctx, count(args.rays), args.repeats)
            if count(args.many_instances):
                many_instance_runs(ctx, count(args.many_instances), args.repeats)
            for c in args.changing_instances.split(","):
                if count(c):
                    changing_instance_runs(ctx, count(c), count(args.rays), args.repeats)


if __name__ == "__main__":
    main()
