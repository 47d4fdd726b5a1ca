"""CPU tests of the refit through its host-only twin (rtc_host_gas_refit / rtc_host_ias_refit, csrc/accel_host.cpp): the node
routine of rtc_gas_refit / rtc_ias_update (csrc/bvh_rules.h) run on host arrays, no CUDA call.

  * identity: refitting with unchanged positions and transforms reproduces the build byte for byte (nodes, triangle records,
    instance-level leaves, world->object matrices), for every leaf size and both collapses, on the Cornell box and the
    geometry scene;
  * after a smooth deformation of every mesh and new transforms (rotation, non-uniform scale, mirror): every structural
    invariant of the node format holds, the topology bytes are those of the build, and the scalar traversal of the refitted
    structure finds the hits and occlusion of brute force over the deformed scene and of a fresh build of it;
  * edge cases (empty geometry, one triangle, an instance of an empty mesh, a mesh collapsed to a point) and the error paths.
"""
import ctypes as C

import numpy as np
import pytest

import helpers as H
from oracle import orc
from test_cpu_host_accel import check_structure, decode, scene_arrays, tri_boxes
from tweeker_raytracer_b200 import core

IDENT = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], dtype=np.float32)
SCENES = ["rtigo3_cornell_box", "rtigo3_geometry"]


def topology(nodes):
    """The bytes a refit must not touch: imask (byte 15), childBase, triBase, meta (bytes 16..31)."""
    return np.ascontiguousarray(nodes)[:, 15:32].tobytes()


def deform(attrs, amplitude, seed):
    """Smooth per-vertex displacement: a sine field over the position, `amplitude` times the mesh extent."""
    out = np.array(attrs, copy=True)
    v = out["vertex"].astype(np.float64)
    if len(v) == 0:
        return out
    rng = np.random.default_rng(seed)
    ext = float(np.max(v.max(axis=0) - v.min(axis=0))) or 1.0
    k = rng.normal(size=(3, 3)) * 2.0 / ext
    phase = rng.uniform(0, 2 * np.pi, size=3)
    out["vertex"] = (v + amplitude * ext * np.sin(v @ k + phase)).astype(np.float32)
    return out


def moved(transform, seed):
    """transform followed (in object space) by a random rotation, a non-uniform scale and a mirror."""
    rng = np.random.default_rng(seed)
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    a = q @ np.diag(rng.uniform(0.6, 1.4, size=3) * np.array([-1.0, 1.0, 1.0]))
    m = np.asarray(transform, dtype=np.float64).reshape(3, 4)
    out = np.zeros((3, 4))
    out[:, :3] = m[:, :3] @ a
    out[:, 3] = m[:, 3] + rng.uniform(-0.05, 0.05, size=3)
    return out.astype(np.float32).reshape(12)


def assert_same_export(a, b):
    assert a["tlas_nodes"].tobytes() == b["tlas_nodes"].tobytes()
    assert a["tlas_leaves"].tobytes() == b["tlas_leaves"].tobytes()
    assert a["world_to_object"].tobytes() == b["world_to_object"].tobytes()
    for g in b["gas"]:
        assert a["gas"][g][0].tobytes() == b["gas"][g][0].tobytes(), g
        assert a["gas"][g][1].tobytes() == b["gas"][g][1].tobytes(), g


@pytest.mark.parametrize("scene", SCENES)
@pytest.mark.parametrize("leaf_max", [1, 2, 3])
@pytest.mark.parametrize("collapse", ["optimal", "greedy"])
def test_refit_with_unchanged_inputs_reproduces_the_build(built, tmp_path, monkeypatch, scene, leaf_max, collapse):
    monkeypatch.setenv("RTC_HOST_LEAF_MAX", str(leaf_max))
    monkeypatch.setenv("RTC_HOST_COLLAPSE", collapse)
    monkeypatch.setenv("RTC_TLAS_COLLAPSE", collapse)
    app, geos, insts = scene_arrays(tmp_path, H.scene_path(scene), scene)
    app.close()
    built_export, _ = core.host_scene_export(geos, insts)
    refit_export, _ = core.host_scene_refit_export(geos, insts, [a for a, _ in geos], [t for t, _ in insts])
    assert_same_export(refit_export, built_export)


@pytest.mark.parametrize("scene", SCENES)
@pytest.mark.parametrize("bounds", ["tight", "box"])
def test_refit_after_deformation_keeps_the_structure_and_the_hits(built, tmp_path, monkeypatch, scene, bounds):
    monkeypatch.setenv("RTC_INSTANCE_BOUNDS", bounds)
    app, geos, insts = scene_arrays(tmp_path, H.scene_path(scene), scene)
    ref_app = H.oracle_scene(app)
    app.close()
    new_attrs = [deform(a, 0.05, seed=g) for g, (a, _) in enumerate(geos)]
    new_xf = [moved(t, seed=100 + i) for i, (t, _) in enumerate(insts)]
    built_export, _ = core.host_scene_export(geos, insts)
    export, _ = core.host_scene_refit_export(geos, insts, new_attrs, new_xf)

    assert topology(export["tlas_nodes"]) == topology(built_export["tlas_nodes"])
    assert export["tlas_leaves"].tobytes() == built_export["tlas_leaves"].tobytes()
    check_structure(export["tlas_nodes"], len(export["tlas_leaves"]), None, 1)
    for g, (nodes, tris) in export["gas"].items():
        assert topology(nodes) == topology(built_export["gas"][g][0])
        assert tris[:, 3].tobytes() == built_export["gas"][g][1][:, 3].tobytes()        # primitive ids: leaf order kept
        check_structure(nodes, len(tris), tri_boxes(tris), 3)
        ids = tris[:, 3].view(np.uint32)
        verts = new_attrs[g]["vertex"][geos[g][1].reshape(-1, 3)[ids]]
        assert np.array_equal(tris.reshape(-1, 3, 4)[:, :, :3], verts)                  # the new positions, gathered

    # hits: the oracle's own BVH and brute force over the deformed scene
    s = orc.Scene()
    for (a, idx), na in zip(geos, new_attrs):
        s.add_geometry(na, idx)
    for (t, g), nt in zip(insts, new_xf):
        s.add_instance(nt, g, 0, -1)
    s.set_materials(np.zeros(1, dtype=orc.MATERIAL_DTYPE))
    s.set_lights(np.zeros(0, dtype=orc.LIGHT_DTYPE))
    s.set_camera(np.zeros(1, dtype=orc.CAMERA_DTYPE))
    s.commit()
    rays = H.random_rays(4000, seed=7)
    hits, _ = orc.wide_trace(export, rays)
    assert H.hits_equal(hits, s.trace_closest(rays))
    assert H.hits_equal(hits[:400], s.trace_closest(rays[:400], brute_force=True))
    occl, _ = orc.wide_trace(export, rays, any_hit=True)
    assert np.array_equal(occl["inst"] != 0xffffffff, s.trace_any(rays).astype(bool))
    fresh, _ = core.host_scene_export([(na, idx) for (_, idx), na in zip(geos, new_attrs)], [(nt, g) for (_, g), nt in zip(insts, new_xf)])
    assert H.hits_equal(hits, orc.wide_trace(fresh, rays)[0])
    assert (hits["inst"] != 0xffffffff).mean() > 0.2
    assert not H.hits_equal(hits, ref_app.trace_closest(rays))                        # the scene did move


def one_triangle(offset=0.0):
    return np.array([[offset, 0, 0], [offset + 1, 0, 0], [offset, 1, 0]], dtype=np.float32), np.array([[0, 1, 2]], dtype=np.uint32)


def test_refit_edge_cases(built):
    empty = (np.zeros((0, 3), dtype=np.float32), np.zeros((0, 3), dtype=np.uint32))
    one = one_triangle()
    rng = np.random.default_rng(3)
    mesh = (rng.uniform(0, 1, size=(30, 3)).astype(np.float32), np.arange(30, dtype=np.uint32).reshape(10, 3))
    shifted = IDENT.copy(); shifted[3] = 5.0
    geos, insts = [empty, one, mesh], [(IDENT, 0), (IDENT, 1), (IDENT, 2)]
    point = np.full_like(mesh[0], 0.25)                             # every vertex of the mesh collapsed to one point
    new_attrs = [empty[0], one_triangle(0.5)[0], point]
    new_xf = [IDENT, shifted, IDENT]
    export, info = core.host_scene_refit_export(geos, insts, new_attrs, new_xf)
    fresh, _ = core.host_scene_export([(a, g[1]) for a, g in zip(new_attrs, geos)], [(t, g) for t, (_, g) in zip(new_xf, insts)])
    assert info["gas_nodes"][0] == 1 and export["gas"][0][0].tobytes() == fresh["gas"][0][0].tobytes()   # the empty node stays
    check_structure(export["gas"][1][0], 1, tri_boxes(export["gas"][1][1]), 3)
    # a box of zero extent: its planes contain the point in the kernels' arithmetic, fmaf(q, step, p) (one rounding of the exact
    # value), though not always exactly -- the same holds for a fresh build of the collapsed mesh
    check_structure(export["gas"][2][0], 10, None, 3)
    n = decode(export["gas"][2][0])
    step = np.ldexp(1.0, n["e"].astype(np.int64) - 127)[:, :, None]
    used = (n["meta"] != 0)[:, None, :]
    lo = (n["p"][:, :, None].astype(np.float64) + n["qlo"] * step).astype(np.float32)
    hi = (n["p"][:, :, None].astype(np.float64) + n["qhi"] * step).astype(np.float32)
    assert np.all(np.where(used, lo, 0.0) <= 0.25) and np.all(np.where(used, hi, 1.0) >= 0.25)
    check_structure(export["tlas_nodes"], 3, None, 1)
    rays = np.zeros(4, dtype=orc.RAY_DTYPE)
    rays["oz"], rays["dz"], rays["tmax"] = 1.0, -1.0, 1e27
    rays["ox"] = [0.75, 5.75, 0.25, 0.1]
    rays["oy"] = [0.25, 0.25, 0.25, 0.25]
    hits, _ = orc.wide_trace(export, rays)
    assert hits["inst"].tolist()[:2] == [0xffffffff, 1]             # the triangle moved: x = 0.5 + 5 .. 6.5 in world space
    assert H.hits_equal(hits, orc.wide_trace(fresh, rays)[0])


def test_refit_error_paths(built):
    L = core.lib()
    verts, idx = one_triangle()
    g = C.c_void_p()
    assert L.rtc_host_gas_build(verts.ctypes.data_as(C.c_void_p), 12, 3, idx.ctypes.data_as(C.c_void_p), 1, C.byref(g)) == 0
    top = C.c_void_p()
    handles = (C.c_void_p * 1)(g)
    assert L.rtc_host_ias_build(IDENT.ctypes.data_as(C.c_void_p), C.cast(handles, C.c_void_p), 1, C.byref(top)) == 0
    try:
        wide = np.zeros((3, 4), dtype=np.float32)
        assert L.rtc_host_gas_refit(g, wide.ctypes.data_as(C.c_void_p), 16) != 0 and b"stride" in L.rtc_last_error()
        assert L.rtc_host_gas_refit(g, None, 12) != 0 and b"null" in L.rtc_last_error()
        assert L.rtc_host_gas_refit(top, verts.ctypes.data_as(C.c_void_p), 12) != 0 and b"geometry-level" in L.rtc_last_error()
        assert L.rtc_host_gas_refit(None, verts.ctypes.data_as(C.c_void_p), 12) != 0
        two = np.tile(IDENT, 2)
        handles2 = (C.c_void_p * 2)(g, g)
        assert L.rtc_host_ias_refit(top, two.ctypes.data_as(C.c_void_p), C.cast(handles2, C.c_void_p), 2) != 0
        assert b"instance count" in L.rtc_last_error()
        assert L.rtc_host_ias_refit(top, None, C.cast(handles, C.c_void_p), 1) != 0 and b"null" in L.rtc_last_error()
        assert L.rtc_host_ias_refit(g, IDENT.ctypes.data_as(C.c_void_p), C.cast(handles, C.c_void_p), 1) != 0
        assert b"instance-level" in L.rtc_last_error()
        bad = (C.c_void_p * 1)(top)
        assert L.rtc_host_ias_refit(top, IDENT.ctypes.data_as(C.c_void_p), C.cast(bad, C.c_void_p), 1) != 0
        assert b"bad geometry handle" in L.rtc_last_error()
        # a refused refit leaves the structure usable: refitting with the build's inputs still reproduces it
        assert L.rtc_host_ias_refit(top, IDENT.ctypes.data_as(C.c_void_p), C.cast(handles, C.c_void_p), 1) == 0
    finally:
        L.rtc_host_accel_destroy(top)
        L.rtc_host_accel_destroy(g)
