#!/usr/bin/env python
"""The device-side queries of include/rtc_device.cuh (a user kernel, one ray per thread) against the batch queries.

  (a) rtc_device_trace_closest / rtc_device_trace_any in a user kernel against rtc_trace_closest / rtc_trace_any on the c3 soups
      (10 M triangles, 100 M coherent and incoherent rays, bench.py's generators);
  (b) a fused ambient-occlusion kernel (one primary ray and 8 occlusion rays per pixel, the count reduced in a register) against the
      three-call pipeline (rtc_trace_closest, a kernel that writes the occlusion rays, rtc_trace_any, a reduction kernel) on the
      geometry scene at 1920x1080.
The user kernels are tests/native/device_trace_kernels.cu, built with nvcc into a temporary directory.  Each row: the median of
--repeats timed calls after one warm-up call (CUDA events on the context stream); every pair of results is checked bit for bit.
The card's name and power limit are read in the same run.  One JSON line per row.

  python tools/device_trace_bench.py [--tris 1e7] [--rays 1e8] [--repeats 5]
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
from device_trace import Module  # noqa: E402
from refit_bench import card, timed  # noqa: E402
from tweeker_raytracer_b200 import core, host  # noqa: E402


def row(**kw):
    print(json.dumps(kw), flush=True)


def soup_runs(ctx, m, ntris, nrays, repeats):
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
            n = len(rays)
            d_r = ctx.to_device(rays)
            del rays
            size = 20 if mode == "closest" else 4
            dtype = core.HIT_DTYPE if mode == "closest" else np.uint32
            d_batch, d_inline = ctx.malloc(n * size), ctx.malloc(n * size)
            wl = "c3-%dM-%s-%s" % (ntris // 10 ** 6, kind, mode)
            fn = ctx.trace_closest if mode == "closest" else ctx.trace_any
            ms = timed(ctx, lambda: fn(top, d_r, n, d_batch), repeats)
            row(workload=wl, path="batch (rtc_trace_%s)" % mode, rays=n, ms=round(ms, 3), mrays_per_s=round(n / ms / 1e3, 1))
            want = ctx.download(d_batch, dtype, n)
            for block in (128, 256):
                ms = timed(ctx, lambda: m.query(ctx, top, d_r, n, d_inline, any_hit=mode == "any", block=block), repeats)
                got = ctx.download(d_inline, dtype, n)
                same = H.hits_equal(got, want) if mode == "closest" else np.array_equal(got, want)
                row(workload=wl, path="user kernel (rtc_device_trace_%s), %d threads per block" % (mode, block), rays=n, ms=round(ms, 3),
                    mrays_per_s=round(n / ms / 1e3, 1), bit_identical=bool(same))
                assert same, (wl, block)
            del want, got
            for p in (d_r, d_batch, d_inline):
                ctx.free(p)
    ctx.scene_destroy(top)
    ctx.gas_destroy(gas)
    ctx.free(d_v)
    ctx.free(d_i)


def ao_runs(m, repeats, w=1920, h=1080, samples=8, radius=0.5):
    with tempfile.TemporaryDirectory() as tmp:
        app = host.App(H.write_system(tmp, "rtigo3_geometry", resolution="%d %d" % (w, h), samplesSqrt=1), H.scene_path("rtigo3_geometry"))
        try:
            ctx, top = app.context(0), app.system_data(0).topObject
            n = w * h
            d_primary = ctx.malloc(n * 32)
            ctx.generate_primary(app.system_data(0), w, h, 0, d_primary)
            bufs = [ctx.malloc(n * 20), ctx.malloc(n * 4), ctx.malloc(n * 20), ctx.malloc(n * samples * 32), ctx.malloc(n * samples * 4),
                    ctx.malloc(n * 4)]
            fused_hits, fused_counts, hits, ao, occ, counts = bufs
            wl = "geometry scene %dx%d, 1 primary + %d occlusion rays per pixel" % (w, h, samples)
            ms = timed(ctx, lambda: m.ao_pipeline(ctx, top, d_primary, n, samples, radius, hits, ao, occ, counts), repeats)
            row(workload=wl, path="three calls: rtc_trace_closest, ray-writing kernel, rtc_trace_any, reduction", ms=round(ms, 3),
                mrays_per_s=round(n * (1 + samples) / ms / 1e3, 1))
            ms = timed(ctx, lambda: m.ao_fused(ctx, top, d_primary, n, samples, radius, fused_hits, fused_counts), repeats)
            same = (H.hits_equal(ctx.download(fused_hits, core.HIT_DTYPE, n), ctx.download(hits, core.HIT_DTYPE, n))
                    and np.array_equal(ctx.download(fused_counts, np.uint32, n), ctx.download(counts, np.uint32, n)))
            row(workload=wl, path="fused user kernel", ms=round(ms, 3), mrays_per_s=round(n * (1 + samples) / ms / 1e3, 1), bit_identical=bool(same))
            assert same
            for p in [d_primary] + bufs:
                ctx.free(p)
        finally:
            app.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tris", default="1e7")
    ap.add_argument("--rays", default="1e8")
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    row(card=card())
    with tempfile.TemporaryDirectory() as tmp:
        m = Module(tmp)
        with core.Context(0) as ctx:
            ctx.set_trace_schedule("group")
            soup_runs(ctx, m, int(float(args.tris)), int(float(args.rays)), args.repeats)
        ao_runs(m, args.repeats)
    row(card=card())


if __name__ == "__main__":
    main()
