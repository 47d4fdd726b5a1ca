"""GPU tests of the device builders, refits, rebuilds and instance updates on non-finite, huge and out-of-range inputs (the catalogue of
test_cpu_extreme_inputs.py on the device).  A triangle with a non-finite vertex coordinate and an instance whose transform has a
non-finite entry are inactive, and so is anything beyond B = 2^126 (DESIGN.md section 3): the timed traversal kernels (rcp.approx box test) under every schedule must
give the oracle's brute-force hits over the active inputs, the device export must equal the host twin byte for byte where one
exists, and the counting kernels must equal the scalar traversal of the exported structure."""
import numpy as np
import pytest

import helpers as H
from oracle import orc
from test_cpu_extreme_inputs import NONFINITE, changed_transform, gas_rays, instance_rays, instance_scene, with_vertex
from test_cpu_gas_rebuild import IDENT, oracle_of, soup
from test_gpu_gas_rebuild import _largest_mesh, _oracle_frame, gas_export, same_gas
from test_gpu_ias_build_device import build_device
from test_gpu_ias_rebuild import Scene
from tweeker_raytracer_b200 import core, host

pytestmark = pytest.mark.gpu

SCHEDULES = ["group", "one_tri", "two_tri"]
VALUES = dict(NONFINITE, **{"1e35": 1e35, "beyond_B": 1e38})            # finite within B, and beyond B = 2^126


def check_device_hits(ctx, top, geos, insts, rays):
    """closest and any hits of the timed kernels under each schedule against brute force; counters against the oracle's
    traversal of the exported structure"""
    ref = oracle_of(geos, insts)
    want = ref.trace_closest(rays, brute_force=True)
    want_any = ref.trace_any(rays, brute_force=True).astype(bool)
    assert (want["inst"] != 0xffffffff).sum() > 0
    for schedule in SCHEDULES:
        ctx.set_trace_schedule(schedule)
        assert H.hits_equal(ctx.trace_closest_host(top, rays), want), schedule
        assert np.array_equal(ctx.trace_any_host(top, rays).astype(bool), want_any), schedule
    export = ctx.scene_export(top)
    d_r = ctx.to_device(rays)
    try:
        counts = ctx.trace_count(top, d_r, len(rays))
    finally:
        ctx.free(d_r)
    hits, wide = orc.wide_trace(export, rays)
    assert H.hits_equal(hits, want)
    assert (counts.nodes, counts.tris, counts.instances) == wide
    return export


@pytest.mark.parametrize("value", sorted(VALUES))
@pytest.mark.parametrize("path", ["sah", "lbvh", "refit", "rebuild"])
def test_extreme_vertex(cuda_device, path, value):
    attrs, idx = soup(2000, seed=1)
    rays = gas_rays(attrs, seed=11)
    with core.Context(0) as ctx:
        d_a, d_i = ctx.to_device(attrs), ctx.to_device(idx)
        for where, axis in [(w, a) for w in ("vertex7", "first_triangle", "last_triangle", "all_three") for a in range(3)]:
            new = with_vertex(attrs, idx, where, axis, np.float32(VALUES[value]))
            d_n = ctx.to_device(new)
            if path in ("sah", "lbvh"):
                g = ctx.gas_build(d_n, attrs.dtype.itemsize, len(attrs), d_i, len(idx), core.BUILD_HOST_SAH if path == "sah" else core.BUILD_GPU_LBVH)
                twin = core.host_scene_export([(new, idx)], [(IDENT, 0)])[0] if path == "sah" else None
            else:
                g = ctx.gas_build(d_a, attrs.dtype.itemsize, len(attrs), d_i, len(idx), core.BUILD_HOST_SAH)
                if path == "refit":
                    ctx.gas_refit(g, d_n)
                    twin = core.host_scene_rebuild_export([(attrs, idx)], [(IDENT, 0)], [([new], [IDENT])])[0]
                else:
                    ctx.gas_rebuild(g, d_n)
                    twin = core.host_scene_rebuild_export([(attrs, idx)], [(IDENT, 0)], [("gas_rebuild", 0, new)])[0]
            if twin is not None:
                assert same_gas(gas_export(ctx, g), twin["gas"][0]), (where, axis)
            desc = np.zeros(1, dtype=core.INSTANCE_DTYPE)
            desc["transform"], desc["gas"], desc["lightIndex"] = IDENT, g, -1
            top = ctx.ias_build(desc)
            check_device_hits(ctx, top, [(new, idx)], [(IDENT, 0)], rays)
            ctx.scene_destroy(top)
            ctx.gas_destroy(g)
            ctx.free(d_n)


@pytest.mark.parametrize("kind", ["nan", "inf", "-inf"])
@pytest.mark.parametrize("path", ["build", "update", "update_device", "update_device_optix_stride", "rebuild", "build_device"])
def test_nonfinite_instance_transform(cuda_device, path, kind):
    geos, xf = instance_scene()
    insts = [(t, 0) for t in xf]
    rays = instance_rays(21)
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, insts)
        for entry in (0, 5, 11):
            new = list(xf)
            new[17] = changed_transform(kind, entry)
            twin = None
            if path == "build":
                top = s.build(new)
                twin = core.host_scene_export(geos, [(t, 0) for t in new])[0]
            elif path == "build_device":
                top = ctx.ias_create(len(new))
                build_device(ctx, top, s.descs(new))
                twin = core.host_scene_rebuild_export(geos, [(t, 0) for t in new], ["rebuild"])[0]
            else:
                top = s.build()
                if path == "update":
                    ctx.ias_update(top, np.asarray(new, dtype=np.float32))
                elif path == "rebuild":
                    ctx.ias_update(top, np.asarray(new, dtype=np.float32))
                    ctx.ias_rebuild(top)
                    twin = core.host_scene_rebuild_export(geos, insts, [([None], new), "rebuild"])[0]
                else:
                    stride = 48 if path == "update_device" else 80         # OptixInstance: the matrix, then 32 bytes of other fields
                    buf = np.zeros((len(new), stride // 4), dtype=np.float32)
                    buf[:, :12] = np.asarray(new, dtype=np.float32)
                    d = ctx.to_device(buf)
                    ctx.ias_update_device(top, d, len(new), stride=stride)
                    ctx.synchronize()
                    ctx.free(d)
                if path != "rebuild":
                    twin = core.host_scene_rebuild_export(geos, insts, [([None], new)])[0]
            export = check_device_hits(ctx, top, geos, [(t, 0) for t in new], rays)
            if twin is not None:
                assert export["tlas_nodes"].tobytes() == twin["tlas_nodes"].tobytes(), entry
                assert export["tlas_leaves"].tobytes() == twin["tlas_leaves"].tobytes(), entry
            ctx.scene_destroy(top)


@pytest.mark.parametrize("kind", ["zero_scale", "scale_1e-30", "scale_1e30", "rotated_mirrored", "translate_1e36", "translate_1e38"])
def test_singular_scaled_and_mirrored_instances(cuda_device, kind):
    geos, xf = instance_scene()
    new = list(xf)
    new[17] = changed_transform(kind)
    with core.Context(0) as ctx:
        s = Scene(ctx, geos, [(t, 0) for t in xf])
        top = s.build()
        ctx.ias_update(top, np.asarray(new, dtype=np.float32))
        check_device_hits(ctx, top, geos, [(t, 0) for t in new], instance_rays(23))


@pytest.mark.parametrize("value", ["nan", "inf"])
@pytest.mark.parametrize("scene", ["rtigo3_geometry", "rtigo3_textures"])
def test_mesh_update_with_a_nonfinite_vertex(cuda_device, tmp_path, scene, value):
    """App.update_geometry with one non-finite vertex, refitted and rebuilt: the frame equals the oracle's frame, in which the
    triangles that use the vertex are inactive.  The textured scene has cutout materials, so the ordered any-hit rounds run
    over the inactive triangles too."""
    frames = []
    for rebuild in (False, True):
        app = host.App(H.write_system(tmp_path, scene, resolution="96 64", samplesSqrt=2), H.scene_path(scene))
        try:
            g = _largest_mesh(app)
            attrs, idx = app.geometry(g)
            new = attrs.copy()
            new["vertex"][idx[len(idx) // 2, 0], 1] = np.float32(NONFINITE[value])
            app.update_geometry(g, new, rebuild=rebuild)
            app.render(4)
            frame = app.frame()
            assert frame.tobytes() == _oracle_frame(app, 4).tobytes()
            frames.append(frame)
        finally:
            app.close()
    assert frames[0].tobytes() == frames[1].tobytes()
