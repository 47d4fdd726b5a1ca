"""CPU tests of the geometry rebuild through its host twin (rtc_host_gas_rebuild, csrc/accel_host.cpp): the LBVH of
rtc_gas_rebuild (csrc/bvh_build_gas_rebuild_gpu.cu) over the triangles' current positions, in the same arithmetic, no CUDA call.

  * structure: every invariant of the node format with one triangle per leaf slot, every triangle in exactly one slot, children
    above their parent, conservative child boxes, and the triangle records (positions and primitive id bits) in leaf order;
  * hits: the scalar traversal of a scene whose geometry was rebuilt finds the hits and occlusion of the SAH-built scene and of
    brute force, on the refit tests' scenes, deformed meshes of the geometry scene and random soups;
  * edge cases: 1, 2, 8 and 9 triangles, duplicate and zero-area triangles, identical centres (Morton ties), far coordinates;
  * determinism: the bytes depend only on positions and indices (not on the leaf size of the build, earlier refits or
    rebuilds), and a refit with unchanged inputs reproduces a rebuild byte for byte;
  * the error paths, the exported symbols, and no spills in the new kernels.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as H
from oracle import orc
from test_cpu_host_accel import check_structure, decode, scene_arrays, tri_boxes
from test_cpu_refit import deform
from tweeker_raytracer_b200 import core

IDENT = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], dtype=np.float32)


def mesh(verts, idx):
    a = np.zeros(len(verts), dtype=orc.ATTR_DTYPE)
    a["vertex"] = verts
    return a, np.ascontiguousarray(idx, dtype=np.uint32).reshape(-1, 3)


def soup(n, seed, spread=10.0, size=0.3, offset=0.0):
    """n independent triangles of edge length ~size, centres uniform in a cube of side `spread` around `offset`."""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-spread / 2, spread / 2, size=(n, 1, 3)) + offset
    v = (c + rng.uniform(-size, size, size=(n, 3, 3))).astype(np.float32).reshape(-1, 3)
    return mesh(v, np.arange(3 * n).reshape(-1, 3))


def oracle_of(geos, insts):
    s = orc.Scene()
    for attrs, idx in geos:
        s.add_geometry(attrs, idx)
    for t, g in insts:
        s.add_instance(t, g, 0, -1)
    s.set_materials(np.zeros(1, dtype=orc.MATERIAL_DTYPE))
    s.set_lights(np.zeros(0, dtype=orc.LIGHT_DTYPE))
    s.set_camera(np.zeros(1, dtype=orc.CAMERA_DTYPE))
    s.commit()
    return s


def check_gas(nodes, tris, attrs, idx):
    """The structure of a rebuilt geometry and its triangle records against the mesh (attrs, idx)."""
    n = len(idx)
    check_structure(nodes, n, tri_boxes(tris), 1)
    for i, node in enumerate(decode(nodes)):
        if node["imask"]:
            assert node["childBase"] > i                                   # children above their parent (the refit's order)
    prim = tris[:, 3].view(np.uint32)
    assert sorted(prim.tolist()) == list(range(n))                        # every triangle exactly once
    v = attrs["vertex"][idx[prim]].reshape(n, 9)
    assert np.array_equal(tris.reshape(n, 3, 4)[:, :, :3].reshape(n, 9).view(np.uint32), v.view(np.uint32))
    assert not tris.reshape(n, 3, 4)[:, 1:, 3].any()


def check_rebuilt(geos, insts, rays, brute=200, rebuilt=None):
    """Every geometry of (geos, insts) rebuilt, then the instances updated: structure, and hits against the SAH build and brute
    force.  `rebuilt`: the geometries to rebuild (all by default).  Returns the export."""
    rebuilt = range(len(geos)) if rebuilt is None else rebuilt
    sah, _ = core.host_scene_export(geos, insts)
    steps = [("gas_rebuild", g, None) for g in rebuilt] + [([None] * len(geos), [t for t, _ in insts])]
    export, info = core.host_scene_rebuild_export(geos, insts, steps)
    for g in rebuilt:
        nodes, tris = export["gas"][g]
        assert info["gas_nodes"][g] == len(nodes) < max(len(geos[g][1]), 1) + 16
        if len(geos[g][1]):
            check_gas(nodes, tris, *geos[g])
    assert export["world_to_object"].tobytes() == sah["world_to_object"].tobytes()
    hits, _ = orc.wide_trace(export, rays)
    assert H.hits_equal(hits, orc.wide_trace(sah, rays)[0])
    occl, _ = orc.wide_trace(export, rays, any_hit=True)
    assert np.array_equal(occl["inst"] != 0xffffffff, orc.wide_trace(sah, rays, any_hit=True)[0]["inst"] != 0xffffffff)
    ref = oracle_of(geos, insts)
    assert H.hits_equal(hits[:brute], ref.trace_closest(rays[:brute], brute_force=True))
    assert np.array_equal(occl["inst"][:brute] != 0xffffffff, ref.trace_any(rays[:brute]).astype(bool))
    return export


@pytest.mark.parametrize("scene", ["rtigo3_cornell_box", "rtigo3_geometry"])
def test_rebuild_of_the_refit_scenes(built, tmp_path, scene):
    app, geos, insts = scene_arrays(tmp_path, H.scene_path(scene), scene)
    app.close()
    check_rebuilt(geos, insts, H.random_rays(3000, seed=7))


def test_rebuild_of_deformed_meshes_of_the_geometry_scene(built, tmp_path):
    """The meshes deformed far (half their extent) and rebuilt from the new positions equal the rebuild of the deformed scene
    built anew, and find its hits."""
    app, geos, insts = scene_arrays(tmp_path, H.scene_path("rtigo3_geometry"), "rtigo3_geometry")
    app.close()
    new = [deform(a, 0.5, seed=g) for g, (a, _) in enumerate(geos)]
    moved = [(a, i) for a, (_, i) in zip(new, geos)]
    rays = H.random_rays(3000, seed=8)
    steps = [("gas_rebuild", g, a) for g, a in enumerate(new)] + [([None] * len(geos), [t for t, _ in insts])]
    export, _ = core.host_scene_rebuild_export(geos, insts, steps)
    fresh = check_rebuilt(moved, insts, rays)
    for g in range(len(geos)):
        assert export["gas"][g][0].tobytes() == fresh["gas"][g][0].tobytes(), g
        assert export["gas"][g][1].tobytes() == fresh["gas"][g][1].tobytes(), g
    # the instance level keeps the topology of the original scene's build, refitted: same hits
    assert H.hits_equal(orc.wide_trace(export, rays)[0], orc.wide_trace(fresh, rays)[0])


@pytest.mark.parametrize("n", [1000, 20000])
def test_rebuild_of_random_soups(built, n):
    geos = [soup(n, seed=n)]
    rays = H.random_rays(4000, seed=3, lo=(-5, -5, -5), hi=(5, 5, 5))
    export = check_rebuilt(geos, [(IDENT, 0)], rays, brute=100)
    assert (orc.wide_trace(export, rays)[0]["inst"] != 0xffffffff).mean() > 0.1


def test_rebuild_of_a_soup_whose_triangles_traded_places(built):
    """Vertex triplets permuted among the triangles: the rebuild equals the rebuild of the permuted soup built anew."""
    attrs, idx = soup(5000, seed=4)
    perm = np.random.default_rng(1).permutation(len(idx))
    traded = attrs.copy()
    traded["vertex"] = attrs["vertex"].reshape(-1, 3, 3)[perm].reshape(-1, 3)
    export, _ = core.host_scene_rebuild_export([(attrs, idx)], [(IDENT, 0)], [("gas_rebuild", 0, traded), ([None], [IDENT])])
    fresh, _ = core.host_scene_rebuild_export([(traded, idx)], [(IDENT, 0)], [("gas_rebuild", 0, None), ([None], [IDENT])])
    assert export["gas"][0][0].tobytes() == fresh["gas"][0][0].tobytes()
    assert export["gas"][0][1].tobytes() == fresh["gas"][0][1].tobytes()
    check_rebuilt([(traded, idx)], [(IDENT, 0)], H.random_rays(2000, seed=5, lo=(-5, -5, -5), hi=(5, 5, 5)), brute=100)


def edge_mesh(case):
    tri = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=np.float32)
    if case in ("1", "2", "8", "9"):
        n = int(case)
        return mesh(np.concatenate([tri + [1.1 * (t % 3), 1.1 * (t // 3), 0.0] for t in range(n)]), np.arange(3 * n).reshape(-1, 3))
    if case == "duplicates":                                              # the same triangle five times, and shared vertices
        return mesh(np.concatenate([tri, tri + [2, 0, 0]]), [[0, 1, 2]] * 5 + [[3, 4, 5], [3, 4, 5], [0, 4, 5]])
    if case == "zero_area":                                               # degenerate: a point, and collinear vertices
        v = np.array([[0.5, 0.5, 0], [0.5, 0.5, 0], [0.5, 0.5, 0], [0, 0, 0], [1, 0, 0], [2, 0, 0]], dtype=np.float32)
        return mesh(np.concatenate([v, tri + [0, 0, 0.5]]), [[0, 1, 2], [3, 4, 5], [6, 7, 8], [0, 7, 8]])
    if case == "same_centre":                                             # one Morton code: the index bits order the tree
        rng = np.random.default_rng(2)
        d = rng.uniform(0.1, 1.0, size=(40, 3))
        c = np.full((40, 3), 0.5)                                         # every box [c - d, c + d]: its centre is c
        v = np.stack([c - d, c + d, c + d * rng.uniform(-1, 1, size=(40, 3))], axis=1)
        return mesh(v.astype(np.float32).reshape(-1, 3), np.arange(120).reshape(-1, 3))
    if case == "far":                                                     # coordinates near 3e4: coarse float grid in the frames
        return soup(300, seed=6, spread=4.0, size=0.5, offset=3.0e4)
    raise ValueError(case)


@pytest.mark.parametrize("case", ["1", "2", "8", "9", "duplicates", "zero_area", "same_centre", "far"])
def test_rebuild_edge_cases(built, case):
    attrs, idx = edge_mesh(case)
    v = attrs["vertex"].astype(np.float64)
    lo, hi = v.min(axis=0), v.max(axis=0)
    rng = np.random.default_rng(1)
    rays = np.zeros(256, dtype=orc.RAY_DTYPE)
    rays["ox"], rays["oy"] = rng.uniform(lo[0] - 0.2, hi[0] + 0.2, 256), rng.uniform(lo[1] - 0.2, hi[1] + 0.2, 256)
    rays["oz"], rays["dz"], rays["tmax"] = hi[2] + 1.0, -1.0, 1e27
    rays["dx"] = rng.uniform(-0.05, 0.05, 256)
    export = check_rebuilt([(attrs, idx)], [(IDENT, 0)], rays, brute=256)
    assert (orc.wide_trace(export, rays)[0]["inst"] != 0xffffffff).any()
    if case == "1":
        assert len(export["gas"][0][0]) == 1


def test_rebuild_of_an_empty_geometry_is_a_no_op(built):
    empty = mesh(np.zeros((0, 3), dtype=np.float32), np.zeros((0, 3), dtype=np.uint32))
    tri = edge_mesh("1")
    before, _ = core.host_scene_export([empty, tri], [(IDENT, 0), (IDENT, 1)])
    after, _ = core.host_scene_rebuild_export([empty, tri], [(IDENT, 0), (IDENT, 1)], [("gas_rebuild", 0, None), ([None, None], [IDENT, IDENT])])
    assert after["gas"][0][0].tobytes() == before["gas"][0][0].tobytes()


def gas_bytes(export, g=0):
    return export["gas"][g][0].tobytes(), export["gas"][g][1].tobytes()


def test_rebuild_bytes_depend_only_on_positions_and_indices(built, tmp_path, monkeypatch):
    app, geos, insts = scene_arrays(tmp_path, H.scene_path("rtigo3_geometry"), "rtigo3_geometry")
    app.close()
    xf = [t for t, _ in insts]
    g = max(range(len(geos)), key=lambda k: len(geos[k][1]))
    attrs = geos[g][0]
    once, _ = core.host_scene_rebuild_export(geos, insts, [("gas_rebuild", g, None)])
    twice, _ = core.host_scene_rebuild_export(geos, insts, [("gas_rebuild", g, None), ("gas_rebuild", g, None)])
    assert gas_bytes(once, g) == gas_bytes(twice, g)
    # a build with leaves of 2 (the default), refitted away and back, then rebuilt
    refits = [[None] * len(geos) for _ in range(2)]
    refits[0][g], refits[1][g] = deform(attrs, 0.3, seed=1), attrs
    after_refits, _ = core.host_scene_rebuild_export(geos, insts, [(refits[0], xf), (refits[1], xf), ("gas_rebuild", g, None)])
    assert gas_bytes(after_refits, g) == gas_bytes(once, g)
    # after a rebuild over other positions
    after_rebuild, _ = core.host_scene_rebuild_export(geos, insts, [("gas_rebuild", g, refits[0][g]), ("gas_rebuild", g, attrs)])
    assert gas_bytes(after_rebuild, g) == gas_bytes(once, g)
    # a build with leaves of 3
    monkeypatch.setenv("RTC_HOST_LEAF_MAX", "3")
    leaves3, _ = core.host_scene_rebuild_export(geos, insts, [("gas_rebuild", g, None)])
    assert gas_bytes(leaves3, g) == gas_bytes(once, g)
    assert gas_bytes(core.host_scene_export(geos, insts)[0], g) != gas_bytes(once, g)      # a different topology


def test_refit_with_unchanged_inputs_reproduces_the_rebuild(built, tmp_path):
    app, geos, insts = scene_arrays(tmp_path, H.scene_path("rtigo3_geometry"), "rtigo3_geometry")
    app.close()
    xf = [t for t, _ in insts]
    rebuild = [("gas_rebuild", g, None) for g in range(len(geos))] + [([None] * len(geos), xf)]
    once, _ = core.host_scene_rebuild_export(geos, insts, rebuild)
    refit, _ = core.host_scene_rebuild_export(geos, insts, rebuild + [([a for a, _ in geos], xf)])
    for g in range(len(geos)):
        assert gas_bytes(refit, g) == gas_bytes(once, g), g
    assert refit["tlas_nodes"].tobytes() == once["tlas_nodes"].tobytes()
    assert refit["world_to_object"].tobytes() == once["world_to_object"].tobytes()


def test_rebuild_error_paths(built):
    L = core.lib()
    attrs, idx = edge_mesh("2")
    g, top = C.c_void_p(), C.c_void_p()
    assert L.rtc_host_gas_build(attrs.ctypes.data_as(C.c_void_p), attrs.dtype.itemsize, len(attrs), idx.ctypes.data_as(C.c_void_p), len(idx), C.byref(g)) == 0
    handles = (C.c_void_p * 1)(g)
    assert L.rtc_host_ias_build(IDENT.ctypes.data_as(C.c_void_p), C.cast(handles, C.c_void_p), 1, C.byref(top)) == 0
    try:
        assert L.rtc_host_gas_rebuild(None, None, 0) != 0 and b"geometry-level" in L.rtc_last_error()
        assert L.rtc_host_gas_rebuild(top, None, 0) != 0 and b"geometry-level" in L.rtc_last_error()
        assert L.rtc_host_gas_rebuild(g, attrs.ctypes.data_as(C.c_void_p), 12) != 0 and b"stride" in L.rtc_last_error()
        assert L.rtc_host_gas_rebuild(g, attrs.ctypes.data_as(C.c_void_p), attrs.dtype.itemsize) == 0
        assert L.rtc_host_gas_rebuild(g, None, 0) == 0
    finally:
        L.rtc_host_accel_destroy(top)
        L.rtc_host_accel_destroy(g)


def test_symbols_are_exported(built):
    L = core.lib()
    for name in ("rtc_gas_rebuild", "rtc_host_gas_rebuild"):
        assert name in core.SYMBOLS and hasattr(L, name)


def test_rebuild_kernels_do_not_spill(tmp_path):
    """-Xptxas -v of csrc/bvh_build_gas_rebuild_gpu.cu, compiled as the Makefile compiles it: no kernel spills."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    csrc = os.path.join(H.ROOT, "tweeker_raytracer_b200", "csrc")
    out = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC",
                          "-I" + os.path.join(H.ROOT, "include"), "-I" + csrc, "-fmad=false", "-Xptxas", "-v", "-c",
                          os.path.join(csrc, "bvh_build_gas_rebuild_gpu.cu"), "-o", str(tmp_path / "gas_rebuild.o")],
                         capture_output=True, text=True, check=True).stderr
    kernels = re.findall(r"Compiling entry function '(\w+)'.*?(\d+) bytes spill stores, (\d+) bytes spill loads", out, re.S)
    assert len({k for k, _, _ in kernels if "k_gas_" in k}) == 6, out
    assert all(s == "0" and l == "0" for _, s, l in kernels), kernels
