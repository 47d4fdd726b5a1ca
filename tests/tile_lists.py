"""Host build of the tile lists of the primary rays (tests/native/primary_lists_host.cpp: csrc/primary_lists.cuh with the ray
generation of csrc/shade.cuh and the traversal of csrc/trace.cuh, compiled by g++) and its loader: shared by
tests/test_cpu_primary_lists.py and tools/tile_list_counts.py."""
import ctypes as C
import os
import subprocess

import numpy as np

import helpers as H
from oracle import orc
from tweeker_raytracer_b200 import core, host

OVERFLOW = 0xFFFFFFFF
_libs = {}


def lists_lib(k=None):
    """The host build of the tile lists; k overrides the list capacity (RTC_TILE_LIST_K)."""
    if k not in _libs:
        src = os.path.join(H.ROOT, "tests", "native", "primary_lists_host.cpp")
        out_dir = os.path.join(H.ROOT, "oracle", "_build")
        os.makedirs(out_dir, exist_ok=True)
        so = os.path.join(out_dir, "libprimary_lists_host%s.so" % ("" if k is None else "_k%d" % k))
        csrc = os.path.join(H.ROOT, "tweeker_raytracer_b200", "csrc")
        deps = [src, os.path.join(H.ROOT, "tests", "native", "trace_host.cpp")] + [os.path.join(csrc, f) for f in ("primary_lists.cuh", "trace.cuh", "shade.cuh", "rtc_internal.h")]
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I" + os.path.join(H.ROOT, "include"), "-I" + csrc,
                                   "-I/usr/local/cuda/include"] + ([] if k is None else ["-DRTC_TILE_LIST_K=%d" % k]) + ["-o", so, src])
        L = C.CDLL(so)
        L.pl_primary.argtypes = [C.POINTER(orc.WideScene), C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.pl_list_capacity.restype = C.c_uint32
        _libs[k] = L
    return _libs[k]


def primary(app, export, w, h, iteration=0, k=None):
    """(list-path hits, traversal hits, per-tile counts, per-tile traversal work counters) of one iteration."""
    L = lists_lib(k)
    ws, sizes, keep = H._wide_scene(export)
    sysd = app.system_data(0)
    camera = np.ascontiguousarray(app.camera())
    sysd.cameraDefinitions = camera.ctypes.data          # host_only: the host copy stands in for the device array
    n, tiles = w * h, (w // 8) * (h // 4)
    got, want = np.zeros(n, dtype=orc.HIT_DTYPE), np.zeros(n, dtype=orc.HIT_DTYPE)
    counts, work = np.zeros(tiles, dtype=np.uint32), np.zeros((tiles, 3), dtype=np.uint64)
    rc = L.pl_primary(C.byref(ws), *sizes, C.byref(sysd), w, h, iteration, got.ctypes.data, want.ctypes.data,
                      counts.ctypes.data, work.ctypes.data)
    assert rc == 0
    return got, want, counts, work


def load(tmp_path, name, resolution, scene=None, **overrides):
    app = host.App(H.write_system(tmp_path, name, resolution=resolution, samplesSqrt=1, **overrides), scene or H.scene_path(name), host_only=True)
    geos = [app.geometry(g) for g in range(app.info.numGeometries)]
    insts = [app.instance(i)[:2] for i in range(app.info.numInstances)]
    export, _ = core.host_scene_export(geos, insts)
    return app, export
