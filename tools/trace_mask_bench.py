#!/usr/bin/env python
"""Visibility masks and face culling of the ray queries (rtc_trace_*_ex) against the plain kernels.

  (a) everything visible: every instance mask 0x01 and ray mask 0x01 through the filtered kernels, against rtc_trace_closest /
      rtc_trace_any (the plain kernels) on the same rays -- the c3 soups (coherent and incoherent, closest and any hit) and the
      10 001-instance scene of tools/make_instances_scene.py;
  (b) the instanced scene with every second instance masked out;
  (c) back-face culling on the instanced scene's closed tori.
Each row: Mrays/s (median of --repeats timed calls after one warm-up call, CUDA events on the context stream), instances entered
per ray (rtc_trace_count / rtc_trace_count_ex over the same rays), and the card's name and power limit read in the same run.
The filtered results are checked against the plain ones where they must be equal.  One JSON line per row.

  python tools/trace_mask_bench.py [--tris 1e7] [--rays 4e6] [--repeats 9]
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
import helpers as H  # noqa: E402
import make_instances_scene  # noqa: E402
from refit_bench import card, timed  # noqa: E402
from tweeker_raytracer_b200 import core, host  # noqa: E402


def measure(ctx, top, rays, mode, repeats, mask=0xFF, flags=0, label="", **row):
    """Mrays/s and instances entered per ray of one query; returns the results for comparisons"""
    n = len(rays)
    d_r = ctx.to_device(rays)
    d_out = ctx.malloc(n * (20 if mode == "closest" else 4))
    if mode == "closest":
        fn = lambda: ctx.trace_closest(top, d_r, n, d_out, mask=mask, flags=flags)  # noqa: E731
    else:
        fn = lambda: ctx.trace_any(top, d_r, n, d_out, mask=mask, flags=flags)  # noqa: E731
    ms = timed(ctx, fn, repeats)
    out = ctx.download(d_out, core.HIT_DTYPE if mode == "closest" else np.uint32, n)
    c = ctx.trace_count(top, d_r, n, any_hit=mode == "any", mask=mask, flags=flags)
    ctx.free(d_r)
    ctx.free(d_out)
    print(json.dumps(dict(row, label=label, mode=mode, rays=n, ms=round(ms, 4), mrays_per_s=round(n / ms / 1e3, 2),
                          instances_per_ray=round(c.instances / max(c.rays, 1), 4), nodes_per_ray=round(c.nodes / max(c.rays, 1), 3),
                          ray_mask=mask, flags=flags)), flush=True)
    return out


def same(a, b):
    return H.hits_equal(a, b) if a.dtype == core.HIT_DTYPE else np.array_equal(a, b)


def soup_runs(ctx, ntris, nrays, repeats):
    verts = bench.soup_numpy(ntris)
    d_v = ctx.to_device(verts)
    d_i = ctx.to_device(np.arange(3 * ntris, dtype=np.uint32))
    gas = ctx.gas_build(d_v, 12, 3 * ntris, d_i, ntris, core.BUILD_GPU_LBVH)
    inst = np.zeros(1, dtype=core.INSTANCE_DTYPE)
    inst["transform"] = [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0]
    inst["gas"], inst["lightIndex"] = gas, -1
    top = ctx.ias_build(inst)
    for kind in ("coh", "incoh"):
        for mode in ("closest", "any"):
            rays = bench.rays_numpy(nrays, kind, mode)
            cfg = "c3-%dM-%s-%s" % (ntris // 10 ** 6, kind, mode)
            plain = measure(ctx, top, rays, mode, repeats, label="(a) plain", workload=cfg)
            ctx.set_instance_masks(top, 0, [0x01])
            filt = measure(ctx, top, rays, mode, repeats, mask=0x01, label="(a) filtered, all visible", workload=cfg)
            ctx.set_instance_masks(top, 0, [0xFF])
            assert same(plain, filt), cfg
    ctx.scene_destroy(top)
    ctx.gas_destroy(gas)
    ctx.free(d_v)
    ctx.free(d_i)


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
    n = len(insts)
    xf = np.asarray([t for t, _ in insts], dtype=np.float32).reshape(n, 12)
    recs = np.zeros(n, dtype=core.INSTANCE_DTYPE)
    recs["transform"], recs["instanceId"], recs["lightIndex"] = xf, np.arange(n), -1
    recs["gas"] = [handles[g] for _, g in insts]
    top = ctx.ias_build(recs)
    lo, hi = xf[:, [3, 7, 11]].min(axis=0), xf[:, [3, 7, 11]].max(axis=0)
    rays = H.random_rays(nrays, seed=3, lo=tuple(lo), hi=tuple(hi), tmin=1e-5)
    short = rays.copy(); short["tmax"] = 2.0
    wl = "instanced scene, %d instances" % n
    for mode, r in (("closest", rays), ("any", short)):
        plain = measure(ctx, top, r, mode, repeats, label="(a) plain", workload=wl)
        ctx.set_instance_masks(top, 0, np.full(n, 0x01, dtype=np.uint8))
        filt = measure(ctx, top, r, mode, repeats, mask=0x01, label="(a) filtered, all visible", workload=wl)
        assert same(plain, filt), mode
        half = np.full(n, 0x01, dtype=np.uint8); half[1::2] = 0x02
        ctx.set_instance_masks(top, 0, half)
        measure(ctx, top, r, mode, repeats, mask=0x01, label="(b) every second instance masked out", workload=wl)
        ctx.set_instance_masks(top, 0, np.full(n, 0xFF, dtype=np.uint8))
        measure(ctx, top, r, mode, repeats, flags=core.RAY_CULL_BACK_FACING, label="(c) back faces culled (closed tori)", workload=wl)
    ctx.scene_destroy(top)
    for h in handles:
        ctx.gas_destroy(h)
    for p in keep:
        ctx.free(p)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tris", default="1e7")
    ap.add_argument("--rays", default="4e6")
    ap.add_argument("--repeats", type=int, default=9)
    args = ap.parse_args()
    print(json.dumps({"card": card()}), flush=True)
    with core.Context(0) as ctx:
        ctx.set_trace_schedule("group")
        soup_runs(ctx, int(float(args.tris)), int(float(args.rays)), args.repeats)
        instance_runs(ctx, int(float(args.rays)), args.repeats)
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
