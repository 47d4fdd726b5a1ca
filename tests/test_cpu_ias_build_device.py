"""CPU tests of rtc_ias_create / rtc_ias_build_device / rtc_scene_rejected_instances: the exports and their ctypes signatures, and
the host twin the GPU tests compare a created scene against -- host_scene_export of the instance set followed by one
rtc_host_ias_rebuild, which is what rtc_ias_build_device computes over the same records (the LBVH of rtc_ias_rebuild over the
instance boxes of the build)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as H
from test_cpu_ias_rebuild import check_rebuilt, mesh, random_instances
from tweeker_raytracer_b200 import core

NEW = ("rtc_ias_create", "rtc_ias_build_device", "rtc_scene_rejected_instances")
CTYPES = {"rtc_context*": C.c_void_p, "uint64_t": C.c_uint64, "uint32_t": C.c_uint32, "uint64_t*": C.POINTER(C.c_uint64),
          "uint32_t*": C.POINTER(C.c_uint32)}


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


def test_twin_of_no_instances(built):
    """rtc_ias_build_device of no record leaves the one empty root node rtc_ias_build writes for none"""
    geos, _ = random_instances(1, seed=0)
    built0, _ = core.host_scene_export(geos, [])
    twin, info = core.host_scene_rebuild_export(geos, [], ["rebuild"])
    assert info["tlas_nodes"] == 1 and len(twin["tlas_leaves"]) == 0
    assert twin["tlas_nodes"].tobytes() == built0["tlas_nodes"].tobytes()


@pytest.mark.parametrize("n", [1, 2, 9, 1000])
def test_twin_of_n_instances(built, n):
    geos, insts = random_instances(n, seed=n, spread=max(2.0, 0.5 * n ** (1 / 3)))
    half = max(2.0, 0.5 * n ** (1 / 3)) / 2 + 0.5
    export = check_rebuilt(geos, insts, H.random_rays(2000, seed=n, lo=(-half,) * 3, hi=(half,) * 3, tmin=1e-5))
    assert export["instance_gas"].tolist() == [0] * n


def test_twin_of_changing_instance_sets(built):
    """count and GAS assignment change from step to step: every step's twin is the rebuild of that step's set alone"""
    tri = mesh(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=np.float32), [[0, 1, 2]])
    quad = mesh(np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0]], dtype=np.float32), [[0, 1, 2], [0, 2, 3]])
    empty = mesh(np.zeros((0, 3), dtype=np.float32), np.zeros((0, 3), dtype=np.uint32))
    geos = [tri, quad, empty]
    _, base = random_instances(1000, seed=3, spread=8.0)
    rng = np.random.default_rng(4)
    for count in (1000, 10, 0, 500, 1000):
        insts = [(base[i][0], int(rng.integers(0, 3))) for i in range(count)]
        if count == 0:
            twin, _ = core.host_scene_rebuild_export(geos, insts, ["rebuild"])
            assert len(twin["tlas_nodes"]) == 1
            continue
        twin = check_rebuilt(geos, insts, H.random_rays(2000, seed=count, lo=(-4.5,) * 3, hi=(4.5,) * 3, tmin=1e-5))
        assert twin["instance_gas"].tolist() == [g for _, g in insts]
