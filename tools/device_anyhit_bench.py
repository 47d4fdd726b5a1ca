#!/usr/bin/env python
"""The any-hit callbacks of include/rtc_device.cuh in user kernels (tests/native/device_anyhit_kernels.cu, one ray per thread).

  (a) cost of the hook: the always-accept callback against rtc_device_trace_closest / _any on the c3 soup (10 M triangles, 100 M
      coherent and incoherent rays, bench.py's generators), every pair of results checked bit for bit;
  (b) alpha-tested closest rays on the geometry scene at 1920x1080: the primary rays of rtc_generate_primary plus one hashed
      secondary ray per pixel from its alpha-tested hit; about half of the triangles are transparent by the hash of
      tests/native/anyhit_predicates.h (128 of 256, a quarter of the rest checkered).  One callback traversal against the restart
      loop a caller writes without callbacks (trace again from tmin = t of each transparent hit): rays/s, mean restarts per ray,
      and the rays on which the restart loop returns another hit than the callback (it skips candidates at the t it restarts from);
  (c) all hits: an any query whose callback ignores, counts and digests every candidate, on the rays of (b).
Each row: the median of --repeats timed calls after one warm-up call (CUDA events on the context stream).  The card's name and
power limit are read in the same run.  One JSON line per row.

  python tools/device_anyhit_bench.py [--tris 1e7] [--rays 1e8] [--repeats 5]
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
from device_anyhit import Module  # noqa: E402
from refit_bench import card, timed  # noqa: E402
from tweeker_raytracer_b200 import core, host  # noqa: E402

PLAIN, ACCEPT_ALL, ALPHA, ALL_HITS = range(4)


def row(**kw):
    print(json.dumps(kw), flush=True)


def hook_cost(ctx, m, ntris, nrays, repeats):
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
            d_plain, d_cb = ctx.malloc(n * size), ctx.malloc(n * size)
            wl = "c3-%dM-%s-%s" % (ntris // 10 ** 6, kind, mode)
            any_hit = mode == "any"
            # alternate the two kernels so that clock drift hits both
            ms = {PLAIN: [], ACCEPT_ALL: []}
            for _ in range(3):
                for k, d in ((PLAIN, d_plain), (ACCEPT_ALL, d_cb)):
                    ms[k].append(timed(ctx, lambda: m.lean(ctx, k, any_hit, top, d_r, n, d), repeats))
            a, b = ctx.download(d_plain, dtype, n), ctx.download(d_cb, dtype, n)
            same = H.hits_equal(a, b) if mode == "closest" else np.array_equal(a, b)
            p, c = float(np.median(ms[PLAIN])), float(np.median(ms[ACCEPT_ALL]))
            row(workload=wl, path="rtc_device_trace_%s" % mode, rays=n, ms=round(p, 3), mrays_per_s=round(n / p / 1e3, 1))
            row(workload=wl, path="rtc_device_trace_%s_anyhit, always-accept lambda" % mode, rays=n, ms=round(c, 3),
                mrays_per_s=round(n / c / 1e3, 1), cost_vs_plain_pct=round(100.0 * (c / p - 1.0), 2), bit_identical=bool(same))
            assert same, wl
            del a, b
            for q in (d_r, d_plain, d_cb):
                ctx.free(q)
    ctx.scene_destroy(top)
    ctx.gas_destroy(gas)
    ctx.free(d_v)
    ctx.free(d_i)


def alpha_and_all_hits(m, repeats, w=1920, h=1080, alpha=128):
    with tempfile.TemporaryDirectory() as tmp:
        app = host.App(H.write_system(tmp, "rtigo3_geometry", resolution="%d %d" % (w, h), samplesSqrt=1), H.scene_path("rtigo3_geometry"))
        try:
            ctx, top = app.context(0), app.system_data(0).topObject
            n = w * h
            d_rays = ctx.malloc(2 * n * 32)
            d_hits, d_restart_hits, d_restarts = ctx.malloc(2 * n * 20), ctx.malloc(2 * n * 20), ctx.malloc(2 * n * 4)
            d_count, d_digest = ctx.malloc(2 * n * 4), ctx.malloc(2 * n * 8)
            ctx.generate_primary(app.system_data(0), w, h, 0, d_rays)
            m.lean(ctx, ALPHA, False, top, d_rays, n, d_hits, alpha)
            m.secondary_rays(ctx, d_rays, d_hits, n, d_rays + n * 32)
            total = 2 * n
            wl = "geometry scene %dx%d, primary + 1 secondary ray per pixel, %d/256 triangles transparent" % (w, h, alpha)
            ms_cb = timed(ctx, lambda: m.lean(ctx, ALPHA, False, top, d_rays, total, d_hits, alpha), repeats)
            ms_rs = timed(ctx, lambda: m.alpha_restart(ctx, top, d_rays, total, alpha, d_restart_hits, d_restarts), repeats)
            cb = ctx.download(d_hits, core.HIT_DTYPE, total)
            rs = ctx.download(d_restart_hits, core.HIT_DTYPE, total)
            restarts = ctx.download(d_restarts, np.uint32, total)
            differ = ~((cb["t"].view(np.uint32) == rs["t"].view(np.uint32)) & (cb["inst"] == rs["inst"]) & (cb["prim"] == rs["prim"]))
            row(workload=wl, path="closest query with the alpha lambda (one traversal)", rays=total, ms=round(ms_cb, 3),
                mrays_per_s=round(total / ms_cb / 1e3, 1), hit_fraction=round(float((cb["inst"] != 0xffffffff).mean()), 4))
            row(workload=wl, path="restart loop: rtc_device_trace_closest again from tmin = t of each transparent hit", rays=total,
                ms=round(ms_rs, 3), mrays_per_s=round(total / ms_rs / 1e3, 1), mean_restarts_per_ray=round(float(restarts.mean()), 4),
                max_restarts=int(restarts.max()), rays_differing_from_callback=int(differ.sum()),
                callback_speedup=round(ms_rs / ms_cb, 3))
            ms_all = timed(ctx, lambda: m.lean(ctx, ALL_HITS, True, top, d_rays, total, d_count, 0, d_digest), repeats)
            counts = ctx.download(d_count, np.uint32, total)
            cand = int(counts.astype(np.int64).sum())
            row(workload="geometry scene %dx%d, the rays above" % (w, h), path="all hits: any query, callback ignores and counts every candidate",
                rays=total, ms=round(ms_all, 3), mrays_per_s=round(total / ms_all / 1e3, 1), candidates=cand,
                mcandidates_per_s=round(cand / ms_all / 1e3, 1), mean_candidates_per_ray=round(cand / total, 3))
            for p in (d_rays, d_hits, d_restart_hits, d_restarts, d_count, d_digest):
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
            hook_cost(ctx, m, int(float(args.tris)), int(float(args.rays)), args.repeats)
        alpha_and_all_hits(m, args.repeats)
    row(card=card())


if __name__ == "__main__":
    main()
