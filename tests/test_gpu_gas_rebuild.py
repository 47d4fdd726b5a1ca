"""GPU tests of rtc_gas_rebuild, the device rebuild of a geometry's topology from its current vertex positions.  Its nodes and
triangle records must equal the host twin (rtc_host_gas_rebuild) byte for byte whichever builder made the GAS, a scene updated
after the rebuild must give the hits of a scene built from the same vertices, and the rebuild must not block the host once the
GAS has been rebuilt before.  The host application deforms meshes through App.update_geometry, refitted or rebuilt."""
import ctypes as C
import time

import numpy as np
import pytest

import helpers as H
from oracle import orc
from test_cpu_refit import deform, moved
from test_gpu_builder import soup
from test_gpu_ias_rebuild import Scene, check_hits, stream_busy
from tweeker_raytracer_b200 import core, host

pytestmark = pytest.mark.gpu

IDENT = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], dtype=np.float32)


def gas_export(ctx, g):
    """(nodes [m, 80] u1, triangle records [t, 12] f4) of one GAS"""
    nn, nt = C.c_uint64(0), C.c_uint64(0)
    core._check(ctx.L.rtc_gas_info(ctx.h, g, C.byref(nn), C.byref(nt)))
    nodes = np.zeros((nn.value, 80), dtype=np.uint8)
    tris = np.zeros((max(nt.value, 1), 12), dtype=np.float32)
    core._check(ctx.L.rtc_gas_export(ctx.h, g, nodes.ctypes.data_as(C.c_void_p), tris.ctypes.data_as(C.c_void_p)))
    return nodes, tris[:nt.value]


def same_gas(a, b):
    return a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes()


def traded(attrs, seed):
    """the vertex triplets of a soup permuted among its triangles: every triangle moves far, the refit's topology is useless"""
    out = attrs.copy()
    out["vertex"] = attrs["vertex"].reshape(-1, 3, 3)[np.random.default_rng(seed).permutation(len(attrs) // 3)].reshape(-1, 3)
    return out


@pytest.mark.parametrize("n", [1, 2, 8, 9, 1000, 100_000, 1_000_000, 10_000_000])
def test_device_rebuild_equals_the_host_twin(cuda_device, n):
    attrs, idx = soup(n, seed=n, extent=0.5 / max(n, 8) ** (1 / 3))
    twin = core.host_scene_rebuild_export([(attrs, idx)], [(IDENT, 0)], [("gas_rebuild", 0, None)])[0]["gas"][0]
    builders = [core.BUILD_GPU_LBVH] if n > 1_000_000 else [core.BUILD_HOST_SAH, core.BUILD_GPU_LBVH]
    with core.Context(0) as ctx:
        d_a, d_i = ctx.to_device(attrs), ctx.to_device(idx)
        for flags in builders:
            g = ctx.gas_build(d_a, attrs.dtype.itemsize, len(attrs), d_i, n, flags)
            ctx.gas_rebuild(g)
            assert same_gas(gas_export(ctx, g), twin), flags
            ctx.gas_rebuild(g)                                               # a second rebuild: the same bytes
            assert same_gas(gas_export(ctx, g), twin), flags
            ctx.gas_destroy(g)


def test_rebuilt_scene_hits_counters_and_export(cuda_device):
    attrs, idx = soup(20000, seed=3, extent=0.02)
    xf = [moved([0.5, 0, 0, x, 0, 0.5, 0, y, 0, 0, 0.5, z], seed=k) for k, (x, y, z) in enumerate(np.random.default_rng(1).uniform(-1, 1, size=(12, 3)))]
    insts = [(t, 0) for t in xf]
    new = traded(attrs, seed=5)
    rays = H.random_rays(100000, seed=6, lo=(-1.5, -1.5, -1.5), hi=(1.5, 1.5, 1.5), tmin=1e-5)
    with core.Context(0) as ctx:
        s = Scene(ctx, [(attrs, idx)], insts)
        top = s.build()
        d_new = ctx.to_device(new)
        ctx.gas_rebuild(s.gas[0], d_new)
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        export = ctx.scene_export(top)
        twin, _ = core.host_scene_rebuild_export([(attrs, idx)], insts, [("gas_rebuild", 0, new), ([None], xf)])
        assert same_gas(export["gas"][s.gas[0]], twin["gas"][0])
        assert export["tlas_nodes"].tobytes() == twin["tlas_nodes"].tobytes()        # instance boxes and the refitted level
        assert export["tlas_leaves"].tobytes() == twin["tlas_leaves"].tobytes()
        assert export["world_to_object"].tobytes() == twin["world_to_object"].tobytes()
        fresh = Scene(ctx, [(new, idx)], insts).build()
        got = check_hits(ctx, top, fresh, rays, export)
        assert (got["inst"] != 0xffffffff).mean() > 0.05
        info = ctx.scene_info(top)
        assert info.numNodes == len(export["gas"][s.gas[0]][0]) + info.numTlasNodes


def test_seeded_programs_of_refits_rebuilds_and_updates(cuda_device):
    """Refits and rebuilds of two GAS, instance updates and instance-level rebuilds in seeded orders: after every step the export
    equals the host twin's replay of the same program."""
    geos = [soup(4000, seed=11, extent=0.03), soup(2500, seed=12, extent=0.04)]
    rng = np.random.default_rng(21)
    insts = [(moved([0.4, 0, 0, x, 0, 0.4, 0, y, 0, 0, 0.4, z], seed=k), k % 2) for k, (x, y, z) in enumerate(rng.uniform(-1, 1, size=(9, 3)))]
    rays = H.random_rays(30000, seed=2, lo=(-1.5, -1.5, -1.5), hi=(1.5, 1.5, 1.5), tmin=1e-5)
    for seed in range(3):
        prog = np.random.default_rng(seed)
        with core.Context(0) as ctx:
            s = Scene(ctx, geos, insts)
            top = s.build()
            cur_attrs = [a for a, _ in geos]
            cur_xf = [t for t, _ in insts]
            cur_buf = [s.keep[0], s.keep[2]]                                         # each GAS's vertex buffer
            steps = []
            for k in range(8):
                op = ["gas_refit", "gas_rebuild", "ias_update", "ias_rebuild"][prog.integers(4)]
                if op in ("gas_refit", "gas_rebuild"):
                    g = int(prog.integers(2))
                    new = traded(cur_attrs[g], seed=100 * seed + k) if op == "gas_rebuild" else deform(cur_attrs[g], 0.02, seed=100 * seed + k)
                    cur_attrs[g] = new
                    if prog.integers(2):
                        ctx.upload(cur_buf[g], new)                                  # the GAS's own buffer, updated in place
                        d = 0
                    else:
                        d = cur_buf[g] = ctx.to_device(new)                          # a new buffer replaces it
                        s.keep.append(d)
                    (ctx.gas_rebuild if op == "gas_rebuild" else ctx.gas_refit)(s.gas[g], d)
                    ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
                    refit = [None, None]
                    if op == "gas_rebuild":
                        steps.append(("gas_rebuild", g, new))
                    else:
                        refit[g] = new
                    steps.append((refit, list(cur_xf)))
                elif op == "ias_update":
                    cur_xf = [moved(t, seed=1000 * seed + 10 * k + i) for i, t in enumerate(cur_xf)]
                    ctx.ias_update(top, np.asarray(cur_xf, dtype=np.float32))
                    steps.append(([None, None], list(cur_xf)))
                else:
                    ctx.ias_rebuild(top)
                    steps.append("rebuild")
                export = ctx.scene_export(top)
                twin, _ = core.host_scene_rebuild_export(geos, insts, steps)
                for g in range(2):
                    assert same_gas(export["gas"][s.gas[g]], twin["gas"][g]), (seed, k, op, g)
                assert export["tlas_nodes"].tobytes() == twin["tlas_nodes"].tobytes(), (seed, k, op)
                assert export["tlas_leaves"].tobytes() == twin["tlas_leaves"].tobytes(), (seed, k, op)
                assert export["world_to_object"].tobytes() == twin["world_to_object"].tobytes(), (seed, k, op)
            hits, _ = orc.wide_trace(twin, rays)
            assert H.hits_equal(ctx.trace_closest_host(top, rays), hits)


def test_refusals_and_a_new_attribute_buffer(cuda_device):
    attrs, idx = soup(3000, seed=7, extent=0.03)
    new = traded(attrs, seed=1)
    rays = H.random_rays(20000, seed=4, lo=(-0.5, -0.5, -0.5), hi=(1.5, 1.5, 1.5), tmin=1e-5)
    with core.Context(0) as ctx:
        s = Scene(ctx, [(attrs, idx)], [(IDENT, 0), (moved(IDENT, seed=3), 0)])
        top = s.build()
        d_new = ctx.to_device(new)
        ctx.gas_rebuild(s.gas[0], d_new)
        for call in (lambda: ctx.trace_closest_host(top, rays[:10]), lambda: ctx.trace_any_host(top, rays[:10])):
            with pytest.raises(core.RtcError, match="rtc_ias_update"):
                call()
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        ctx.free(s.keep[0])                                                  # the build's buffer is gone: nothing may read it
        ctx.gas_rebuild(s.gas[0])                                            # the GAS's buffer is now d_new
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        fresh = Scene(ctx, [(new, idx)], s.insts).build()
        assert H.hits_equal(ctx.trace_closest_host(top, rays), ctx.trace_closest_host(fresh, rays))
        with pytest.raises(core.RtcError, match="bad gas handle"):
            ctx.gas_rebuild(999)
        ctx.gas_destroy(s.gas[0])
        with pytest.raises(core.RtcError, match="bad gas handle"):
            ctx.gas_rebuild(s.gas[0])
        empty = ctx.gas_build(ctx.to_device(attrs[:3]), attrs.dtype.itemsize, 3, ctx.to_device(idx[:0].reshape(-1)), 0, core.BUILD_HOST_SAH)
        ctx.gas_rebuild(empty)                                               # no triangles: nothing to do


def test_rebuild_does_not_block_the_host(cuda_device, tmp_path):
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="1920 1080", samplesSqrt=1), H.scene_path("rtigo3_geometry"))
    try:
        app.render(1)
        app.frame()                                                          # the App's output buffer exists
        ctx = app.context(0)
        ctx.set_trace_schedule("group")                                      # no timed batch, so no launch waits for the tuner
        sys_data = app.system_data()
        top = sys_data.topObject
        g = app.info.numGeometries - 1
        ctx.gas_rebuild(g)                                                   # the first rebuild allocates and may synchronise
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        ctx.synchronize()
        t0 = time.perf_counter()
        ctx.launch(sys_data, 1920, 1080, core.RAYGEN_FULL_FRAME, app.info.miss, 0, 4)
        ctx.synchronize()
        per_iteration = (time.perf_counter() - t0) / 4
        iterations = int(min(2000, max(8, 0.5 / per_iteration)))             # about half a second of work
        ctx.launch(sys_data, 1920, 1080, core.RAYGEN_FULL_FRAME, app.info.miss, 0, iterations)
        ctx.gas_rebuild(g)
        pending = stream_busy(ctx.stream)
        ctx.synchronize()
        assert pending, "rtc_gas_rebuild returned after the launch before it had finished: it synchronised the host"
        ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))
        ctx.synchronize()
    finally:
        app.close()


def _oracle_frame(app, iterations):
    w, h = app.resolution
    return H.oracle_scene(app).render(H.oracle_sys(app), app.info.miss, w, h, iter_count=iterations).reshape(h, w, 4)


def _largest_mesh(app):
    """the geometry with the most triangles (not the area light's parallelogram)"""
    return int(np.argmax([len(app.geometry(g)[1]) for g in range(app.info.numGeometries)]))


@pytest.mark.parametrize("scene", ["rtigo3_geometry", "rtigo3_textures"])
def test_deformed_mesh_frames(cuda_device, tmp_path, scene):
    """App.update_geometry, refitted and rebuilt: iterations held back before the update render the old mesh, and the frames
    after it equal the oracle's frame of the deformed scene and each other.  The textured scene has cutout materials, so the
    ordered any-hit rounds run on the deformed mesh; their cached graph captures no GAS pointer, so an update of the GAS alone
    does not capture it again."""
    frames = []
    for rebuild in (False, True):
        app = host.App(H.write_system(tmp_path, scene, resolution="96 64", samplesSqrt=2), H.scene_path(scene))
        try:
            g = _largest_mesh(app)
            attrs, idx = app.geometry(g)
            new = deform(attrs, 0.5, seed=g)
            v0, v1 = attrs["vertex"][idx].astype(np.float64), new["vertex"][idx].astype(np.float64)
            size = np.linalg.norm(v0[:, 1] - v0[:, 0], axis=1)
            assert np.median(np.linalg.norm(v1.mean(axis=1) - v0.mean(axis=1), axis=1)) > 2 * np.median(size)   # moved far
            old = _oracle_frame(app, 3)
            app.set_coalesce(64)
            app.render(3)                                                    # held back by the Raytracer
            app.update_geometry(g, new, rebuild=rebuild)                     # flushes them first: they render the old mesh
            assert app.frame().tobytes() == old.tobytes()
            assert app.geometry(g)[0].tobytes() == new.tobytes()
            app.set_coalesce(1)
            app.render(4)
            frame = app.frame()
            assert frame.tobytes() == _oracle_frame(app, 4).tobytes()
            assert app.stats().stackOverflows == 0
            # The cutout graph is captured again when the launch shape or the any-hit scratch changes (the deformed mesh may ignore
            # more candidates), never for a GAS: the same update again, with launches of the same shape, captures nothing.
            builds = app.context(0).stats().cutoutGraphBuilds
            app.update_geometry(g, new, rebuild=rebuild)
            app.render(4)
            assert app.frame().tobytes() == frame.tobytes()
            assert app.context(0).stats().cutoutGraphBuilds == builds
            with pytest.raises(core.RtcError):
                app.update_geometry(g, new[:-1], rebuild=rebuild)
            frames.append(frame)
        finally:
            app.close()
    assert frames[0].tobytes() == frames[1].tobytes()
