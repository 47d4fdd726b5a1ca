#!/usr/bin/env python
"""The two instance levels of a scene compared WITHOUT a GPU: the SAH level rtc_ias_build builds and the LBVH level
rtc_ias_rebuild builds over the same instance boxes, both made by the host twins (rtc_host_ias_build, rtc_host_ias_rebuild).
Prints one JSON line per level with the work per ray of tests/tools/bvh_quality.py (nodes, triangles, instances entered, for
primary and bounce rays, every hit checked against the oracle) and the warp cost of tests/tools/simd_cost.py (primary, bounce
and shadow rays).  Both are models: they predict, a B200 run (tools/refit_bench.py) measures.

  python tools/ias_level_quality.py [--config c2|c4] [--width 240 --height 136] [--instances 10000]
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests", "tools"))

import bvh_quality                                 # noqa: E402
import helpers as H                                # noqa: E402
import simd_cost                                   # noqa: E402
from tweeker_raytracer_b200 import core            # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--config", default="c4", choices=sorted(bvh_quality.CONFIGS))
    ap.add_argument("--width", type=int, default=240)
    ap.add_argument("--height", type=int, default=136)
    ap.add_argument("--instances", type=int, default=10000)
    args = ap.parse_args()
    assert args.width % 8 == 0 and args.height % 4 == 0
    with tempfile.TemporaryDirectory() as tmp:
        app = bvh_quality.load(args.config, args.width, args.height, args.instances, tmp)
        try:
            geos = [app.geometry(g) for g in range(app.info.numGeometries)]
            insts = [app.instance(i)[:2] for i in range(app.info.numInstances)]
            ref = H.oracle_scene(app)
            w, h = app.resolution
            primary = ref.generate_primary(H.oracle_sys(app), w, h, 0)[simd_cost.tile_order(w, h)]
            bounce = simd_cost.octant_runs(bvh_quality.bounce_rays(primary, ref.trace_closest(primary), 7))
            for level, steps in (("sah", []), ("lbvh", ["rebuild"])):
                export, info = core.host_scene_rebuild_export(geos, insts, steps)
                result = {"config": args.config, "instance_level": level, "resolution": [w, h], "instances": len(insts),
                          "tlas_nodes": info["tlas_nodes"], "per_ray": bvh_quality.measure(app, export, False)}
                result["warp_cost"] = {name: simd_cost.summarise(H.product_simd_cost(export, rays, any_hit))["warp_cost_per_ray"]
                                       for name, rays, any_hit in (("primary", primary, False), ("bounce", bounce, False), ("shadow", bounce, True))}
                print(json.dumps(result), flush=True)
        finally:
            app.close()


if __name__ == "__main__":
    main()
