"""CPU tests of rtc_gas_create / rtc_gas_build_device / rtc_gas_rejected_triangles: the exports and their ctypes signatures, and
the host twin the GPU tests compare a created GAS against -- the ("gas_build_device", g, attributes, indices) step of
host_scene_rebuild_export: rtc_host_gas_build + rtc_host_gas_rebuild over the vertices with one NaN vertex appended, which every
out-of-range index is replaced by.  Such triangles are inactive: the oracle's traversal of the twin finds exactly the brute-force
hits of the valid triangles.  The refit kernel, which now reads the same NaN vertex for such an index, does not spill."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as H
from oracle import orc
from test_cpu_gas_rebuild import IDENT, check_gas, mesh, oracle_of, soup
from test_cpu_refit import deform
from tweeker_raytracer_b200 import core

NEW = ("rtc_gas_create", "rtc_gas_build_device", "rtc_gas_rejected_triangles")
CTYPES = {"rtc_context*": C.c_void_p, "uint64_t": C.c_uint64, "uint32_t": C.c_uint32, "uint32_t*": C.POINTER(C.c_uint32)}


def test_exports_and_signatures(built):
    L = core.lib()
    nm = subprocess.run(["nm", "-D", "--defined-only", core.LIB_PATH], capture_output=True, text=True, check=True).stdout
    header = open(os.path.join(H.ROOT, "include", "rtc_core.h")).read()
    for name in NEW:
        assert name in core.SYMBOLS and re.search(r"\bT %s\b" % name, nm), name
        proto = re.search(r"int %s\(([^)]*)\);" % name, header)
        assert proto, name
        params = [re.sub(r"\s*\w+$", "", p.strip()).replace(" *", "*") for p in proto.group(1).split(",")]
        assert [CTYPES[p] for p in params] == list(getattr(L, name).argtypes), name


def with_bad_indices(n, seed, num_bad):
    """a soup of n triangles, num_bad of them with one index >= the vertex count (in any corner), and the reference mesh in
    which those triangles lie far outside the rays' reach instead"""
    attrs, idx = soup(n, seed=seed, spread=4.0)
    rng = np.random.default_rng(seed)
    bad = np.sort(rng.choice(n, size=num_bad, replace=False))
    idx = idx.copy()
    idx[bad, rng.integers(0, 3, size=num_bad)] = len(attrs) + rng.integers(0, 1 << 31, size=num_bad).astype(np.uint32)
    far = np.concatenate([attrs, attrs[:1]])                             # one more vertex for the out-of-range corners
    ref_idx = idx.copy()
    ref_idx[ref_idx >= len(attrs)] = len(attrs)
    far["vertex"][ref_idx[bad].reshape(-1)] = 1.0e6                       # every corner of a bad triangle goes far away
    return attrs, idx, bad, (far, ref_idx)


def test_out_of_range_indices_are_inactive(built):
    attrs, idx, bad, (far, ref_idx) = with_bad_indices(3000, seed=5, num_bad=300)
    # the bad triangles share no vertex with good ones (a soup), so moving their corners away changes nothing else
    assert not np.isin(ref_idx[bad], np.delete(idx, bad, axis=0)).any()
    twin, info = core.host_scene_rebuild_export([soup(10, seed=1)], [(IDENT, 0)], [("gas_build_device", 0, attrs, idx), ([None], [IDENT])])
    nodes, tris = twin["gas"][0]
    assert info["gas_tris"][0] == len(tris) == 3000 and len(nodes) < 3000 + 16
    prim = tris[:, 3].view(np.uint32)
    assert sorted(prim.tolist()) == list(range(3000))
    v0 = tris.reshape(-1, 3, 4)[:, 0, :3]
    assert np.isnan(v0[np.isin(prim, bad)]).all() and not np.isnan(v0[~np.isin(prim, bad)]).any()
    rays = H.random_rays(4000, seed=3, lo=(-2.5,) * 3, hi=(2.5,) * 3, tmax=100.0)
    hits, _ = orc.wide_trace(twin, rays)
    ref = oracle_of([(far, ref_idx)], [(IDENT, 0)])
    assert H.hits_equal(hits, ref.trace_closest(rays, brute_force=True))
    assert not np.isin(hits["prim"][hits["inst"] != 0xffffffff], bad).any() and (hits["inst"] != 0xffffffff).mean() > 0.1
    occl, _ = orc.wide_trace(twin, rays, any_hit=True)
    assert np.array_equal(occl["inst"] != 0xffffffff, ref.trace_any(rays).astype(bool))


def test_twin_of_valid_indices_is_the_rebuild(built):
    """without a bad index the appended NaN vertex changes nothing: the twin equals rtc_host_gas_rebuild of the same mesh"""
    attrs, idx = soup(2000, seed=8)
    twin, _ = core.host_scene_rebuild_export([soup(10, seed=1)], [(IDENT, 0)], [("gas_build_device", 0, attrs, idx), ([None], [IDENT])])
    rebuilt, _ = core.host_scene_rebuild_export([(attrs, idx)], [(IDENT, 0)], [("gas_rebuild", 0, None), ([None], [IDENT])])
    for key in ("tlas_nodes", "world_to_object"):
        assert twin[key].tobytes() == rebuilt[key].tobytes(), key
    assert twin["gas"][0][0].tobytes() == rebuilt["gas"][0][0].tobytes()
    assert twin["gas"][0][1].tobytes() == rebuilt["gas"][0][1].tobytes()
    check_gas(*twin["gas"][0], attrs, idx)
    # refits and rebuilds after it read the GAS's vertex records (the NaN vertex stays behind them)
    new = deform(attrs, 0.2, seed=2)
    steps = [("gas_build_device", 0, attrs, idx), ("gas_rebuild", 0, new), ([None], [IDENT])]
    after, _ = core.host_scene_rebuild_export([soup(10, seed=1)], [(IDENT, 0)], steps)
    fresh, _ = core.host_scene_rebuild_export([(new, idx)], [(IDENT, 0)], [("gas_rebuild", 0, None), ([None], [IDENT])])
    assert after["gas"][0][0].tobytes() == fresh["gas"][0][0].tobytes()
    refit, _ = core.host_scene_rebuild_export([soup(10, seed=1)], [(IDENT, 0)], steps + [([attrs], [IDENT])])
    refit_fresh, _ = core.host_scene_rebuild_export([(new, idx)], [(IDENT, 0)], [("gas_rebuild", 0, None), ([attrs], [IDENT])])
    assert refit["gas"][0][1].tobytes() == refit_fresh["gas"][0][1].tobytes()


def test_twin_of_no_triangles(built):
    """a build of no triangle leaves the one empty node rtc_host_gas_build writes for none"""
    empty = mesh(np.zeros((0, 3), dtype=np.float32), np.zeros((0, 3), dtype=np.uint32))
    built0, _ = core.host_scene_export([empty], [(IDENT, 0)])
    attrs, _ = soup(5, seed=1)
    for verts in (empty[0], attrs):
        twin, info = core.host_scene_rebuild_export([soup(50, seed=2)], [(IDENT, 0)],
                                                    [("gas_build_device", 0, verts, np.zeros((0, 3), dtype=np.uint32)), ([None], [IDENT])])
        assert info["gas_nodes"][0] == 1 and info["gas_tris"][0] == 0
        assert twin["gas"][0][0].tobytes() == built0["gas"][0][0].tobytes()
        assert twin["tlas_nodes"].tobytes() == built0["tlas_nodes"].tobytes()


@pytest.mark.parametrize("source", ["bvh_build_gas_rebuild_gpu.cu", "bvh_refit.cu"])
def test_changed_kernels_do_not_spill(tmp_path, source):
    """-Xptxas -v of the files whose kernels read vertices through an index, compiled as the Makefile compiles them"""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    csrc = os.path.join(H.ROOT, "tweeker_raytracer_b200", "csrc")
    out = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC",
                          "-I" + os.path.join(H.ROOT, "include"), "-I" + csrc, "-fmad=false", "-Xptxas", "-v", "-c",
                          os.path.join(csrc, source), "-o", str(tmp_path / "k.o")], capture_output=True, text=True, check=True).stderr
    kernels = re.findall(r"Compiling entry function '(\w+)'.*?(\d+) bytes spill stores, (\d+) bytes spill loads", out, re.S)
    assert kernels and all(s == "0" and l == "0" for _, s, l in kernels), kernels
