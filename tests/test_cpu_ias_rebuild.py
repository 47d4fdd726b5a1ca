"""CPU tests of the instance-level rebuild through its host twin (rtc_host_ias_rebuild, csrc/accel_host.cpp): the LBVH of
rtc_ias_rebuild (csrc/bvh_build_ias_gpu.cu) over the instance boxes of the last build / refit, in the same arithmetic, no CUDA call.

  * structure: every invariant of the node format with one instance per leaf slot, every instance in exactly one slot, children
    above their parent, and every conservative child box containing the instances below it;
  * hits: the scalar traversal of the rebuilt structure finds the hits and occlusion of the SAH-built structure and of brute force,
    on the stress scene (reduced), the geometry scene, 100 000 random instances, one and two instances, identical transforms
    (Morton ties), instances of an empty mesh and RTC_INSTANCE_BOUNDS=box;
  * determinism, and a refit with unchanged inputs after a rebuild reproduces the rebuild byte for byte;
  * the error paths.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import helpers as H
from oracle import orc
from test_cpu_host_accel import check_structure, decode, scene_arrays
from tweeker_raytracer_b200 import core

IDENT = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], dtype=np.float32)


def mesh(verts, idx):
    a = np.zeros(len(verts), dtype=orc.ATTR_DTYPE)
    a["vertex"] = verts
    return a, np.ascontiguousarray(idx, dtype=np.uint32).reshape(-1, 3)


def random_instances(n, seed, spread=50.0):
    """n instances of one small triangle, randomly rotated, scaled and placed in a cube of side `spread`."""
    rng = np.random.default_rng(seed)
    geo = mesh(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=np.float32), [[0, 1, 2]])
    q, _ = np.linalg.qr(rng.normal(size=(n, 3, 3)))
    m = np.zeros((n, 3, 4))
    m[:, :, :3] = q * rng.uniform(0.05, 0.3, size=(n, 1, 1))
    m[:, :, 3] = rng.uniform(-spread / 2, spread / 2, size=(n, 3))
    return [geo], [(t, 0) for t in m.astype(np.float32).reshape(n, 12)]


def stress_scene(tmp_path, count):
    sys.path.insert(0, os.path.join(H.ROOT, "tools"))
    import make_instances_scene
    path = os.path.join(str(tmp_path), "scene_stress.txt")
    make_instances_scene.write_scene(path, count=count, tess=(24, 12))
    return path


def vertex_bounds(geos, insts):
    """[n, 2, 3] float64 bounds of every instance's transformed vertices (the origin for an empty mesh): the padded boxes the
    instance level is built over contain them."""
    out = np.zeros((len(insts), 2, 3))
    for i, (t, g) in enumerate(insts):
        attrs, idx = geos[g]
        if len(idx) == 0:
            continue
        m = np.asarray(t, dtype=np.float64).reshape(3, 4)
        w = attrs["vertex"].astype(np.float64) @ m[:, :3].T + m[:, 3]
        out[i] = w.min(axis=0), w.max(axis=0)
    return out


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


def scene_bounds(geos, insts):
    b = vertex_bounds(geos, insts)
    return b[:, 0].min(axis=0) - 0.1, b[:, 1].max(axis=0) + 0.1


def check_rebuilt(geos, insts, rays, brute=200):
    """The rebuild of (geos, insts): its structure, and its hits against the SAH build and brute force.  Returns the export."""
    sah, _ = core.host_scene_export(geos, insts)
    export, info = core.host_scene_rebuild_export(geos, insts, ["rebuild"])
    n = len(insts)
    assert info["tlas_nodes"] == len(export["tlas_nodes"]) < n + 16
    assert sorted(export["tlas_leaves"].tolist()) == list(range(n))
    check_structure(export["tlas_nodes"], n, vertex_bounds(geos, insts)[export["tlas_leaves"]], 1)
    nodes = decode(export["tlas_nodes"])
    for i, node in enumerate(nodes):
        if node["imask"]:
            assert node["childBase"] > i                                   # children above their parent (the refit's order)
    assert export["world_to_object"].tobytes() == sah["world_to_object"].tobytes()
    hits, _ = orc.wide_trace(export, rays)
    assert H.hits_equal(hits, orc.wide_trace(sah, rays)[0])
    occl, _ = orc.wide_trace(export, rays, any_hit=True)
    assert np.array_equal(occl["inst"] != 0xffffffff, orc.wide_trace(sah, rays, any_hit=True)[0]["inst"] != 0xffffffff)
    ref = oracle_of(geos, insts)
    assert H.hits_equal(hits[:brute], ref.trace_closest(rays[:brute], brute_force=True))
    assert np.array_equal(occl["inst"][:brute] != 0xffffffff, ref.trace_any(rays[:brute]).astype(bool))
    return export


@pytest.mark.parametrize("bounds", ["tight", "box"])
def test_rebuild_of_the_stress_scene(built, tmp_path, monkeypatch, bounds):
    monkeypatch.setenv("RTC_INSTANCE_BOUNDS", bounds)
    app, geos, insts = scene_arrays(tmp_path, stress_scene(tmp_path, 1000), "rtigo3_instances")
    app.close()
    lo, hi = scene_bounds(geos, insts)
    export = check_rebuilt(geos, insts, H.random_rays(3000, seed=11, lo=lo, hi=hi))
    assert len(export["tlas_leaves"]) == 1001


def test_rebuild_of_the_geometry_scene(built, tmp_path):
    app, geos, insts = scene_arrays(tmp_path, H.scene_path("rtigo3_geometry"), "rtigo3_geometry")
    app.close()
    check_rebuilt(geos, insts, H.random_rays(4000, seed=7))


def test_rebuild_of_100000_random_instances(built):
    geos, insts = random_instances(100_000, seed=5)
    rays = H.random_rays(20000, seed=3, lo=(-25, -25, -25), hi=(25, 25, 25))
    export = check_rebuilt(geos, insts, rays, brute=100)
    assert (orc.wide_trace(export, rays)[0]["inst"] != 0xffffffff).mean() > 0.1


@pytest.mark.parametrize("case", ["one", "two", "identical", "empty_mesh"])
def test_rebuild_edge_cases(built, case):
    tri = mesh(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=np.float32), [[0, 1, 2]])
    empty = mesh(np.zeros((0, 3), dtype=np.float32), np.zeros((0, 3), dtype=np.uint32))
    shifted = IDENT.copy(); shifted[3] = 3.0
    geos = [tri, empty]
    insts = {"one": [(IDENT, 0)],
             "two": [(IDENT, 0), (shifted, 0)],
             "identical": [(IDENT, 0)] * 37,                                 # one Morton code: the index bits order the tree
             "empty_mesh": [(IDENT, 1), (shifted, 0), (IDENT, 1), (IDENT, 0)]}[case]
    rays = np.zeros(64, dtype=orc.RAY_DTYPE)
    rng = np.random.default_rng(1)
    rays["ox"], rays["oy"] = rng.uniform(-0.5, 4.5, 64), rng.uniform(-0.5, 1.5, 64)
    rays["oz"], rays["dz"], rays["tmax"] = 1.0, -1.0, 1e27
    export = check_rebuilt(geos, insts, rays, brute=64)
    hits, _ = orc.wide_trace(export, rays)
    assert (hits["inst"] != 0xffffffff).any()
    if case == "one":
        assert len(export["tlas_nodes"]) == 1 and export["tlas_leaves"].tolist() == [0]


def test_rebuild_is_deterministic_and_a_refit_reproduces_it(built, tmp_path):
    app, geos, insts = scene_arrays(tmp_path, stress_scene(tmp_path, 500), "rtigo3_instances")
    app.close()
    xf = [t for t, _ in insts]
    once, _ = core.host_scene_rebuild_export(geos, insts, ["rebuild"])
    twice, _ = core.host_scene_rebuild_export(geos, insts, ["rebuild", "rebuild"])
    assert once["tlas_nodes"].tobytes() == twice["tlas_nodes"].tobytes()
    assert once["tlas_leaves"].tobytes() == twice["tlas_leaves"].tobytes()
    refit, _ = core.host_scene_rebuild_export(geos, insts, ["rebuild", ([None] * len(geos), xf)])
    assert refit["tlas_nodes"].tobytes() == once["tlas_nodes"].tobytes()
    assert refit["tlas_leaves"].tobytes() == once["tlas_leaves"].tobytes()
    sah, _ = core.host_scene_export(geos, insts)
    assert once["tlas_nodes"].tobytes() != sah["tlas_nodes"].tobytes()        # a different topology over the same boxes


def test_rebuild_after_a_refit_uses_the_refitted_boxes(built):
    geos, insts = random_instances(2000, seed=9)
    rng = np.random.default_rng(2)
    perm = rng.permutation(len(insts))
    moved = [insts[p][0] for p in perm]                                       # the lattice permuted: same boxes, new places
    export, _ = core.host_scene_rebuild_export(geos, insts, [([None], moved), "rebuild"])
    fresh, _ = core.host_scene_rebuild_export(geos, [(t, 0) for t in moved], ["rebuild"])
    assert export["tlas_nodes"].tobytes() == fresh["tlas_nodes"].tobytes()
    assert export["tlas_leaves"].tobytes() == fresh["tlas_leaves"].tobytes()


def test_rebuild_error_paths(built):
    L = core.lib()
    tri = mesh(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=np.float32), [[0, 1, 2]])
    g = C.c_void_p()
    assert L.rtc_host_gas_build(tri[0].ctypes.data_as(C.c_void_p), tri[0].dtype.itemsize, 3, tri[1].ctypes.data_as(C.c_void_p), 1, C.byref(g)) == 0
    try:
        assert L.rtc_host_ias_rebuild(g) != 0 and b"instance-level" in L.rtc_last_error()
        assert L.rtc_host_ias_rebuild(None) != 0 and b"instance-level" in L.rtc_last_error()
    finally:
        L.rtc_host_accel_destroy(g)
    assert "rtc_ias_rebuild" in core.SYMBOLS and "rtc_host_ias_rebuild" in core.SYMBOLS


def test_rebuild_kernels_do_not_spill(tmp_path):
    """-Xptxas -v of csrc/bvh_build_ias_gpu.cu, compiled as the Makefile compiles it: no kernel of the rebuild spills."""
    import re
    import subprocess
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    csrc = os.path.join(H.ROOT, "tweeker_raytracer_b200", "csrc")
    out = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                          "-I" + os.path.join(H.ROOT, "include"), "-I" + csrc, "-fmad=false", "-Xptxas", "-v", "-c",
                          os.path.join(csrc, "bvh_build_ias_gpu.cu"), "-o", str(tmp_path / "ias.o")],
                         capture_output=True, text=True, check=True).stderr
    kernels = re.findall(r"Compiling entry function '(\w*k_ias_\w+)'.*?(\d+) bytes spill stores, (\d+) bytes spill loads", out, re.S)
    assert len({k for k, _, _ in kernels}) == 5, out
    assert all(s == "0" and l == "0" for _, s, l in kernels), kernels
