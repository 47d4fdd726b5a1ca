"""Test infrastructure of the visibility masks and face culling of rtc_trace_*_ex (RTC_RAY_CULL_*):

  * product_trace_ex: the FILTER traversal of csrc/trace.cuh compiled for the host (tests/native/trace_host_ex.cpp);
  * MaskedScene: an oracle scene (oracle/orc.py Scene) with per-instance masks, traced by brute force
    (tests/native/oracle_masks.c) with facing decided by the sign of det, as the kernels do ("det"), or by
    dot((v1 - v0) x (v2 - v0), d_obj) < 0 in double ("normal");
  * wide_trace_ex: oracle/wide_bvh.inc's restatement of the traversal with the two tests, whose counters the counting kernels of
    rtc_trace_count_ex must equal.
Both libraries are built on first use into oracle/_build (git-ignored), next to the oracle and the host build of the traversal."""
import ctypes as C
import os
import subprocess

import numpy as np

import helpers as H
from oracle import orc

_BUILD = os.path.join(H.ROOT, "oracle", "_build")
_libs = {}


def _build(name, cmd, src, deps, libs=()):
    if name not in _libs:
        os.makedirs(_BUILD, exist_ok=True)
        so = os.path.join(_BUILD, name)
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in [src] + deps):
            subprocess.check_call(cmd + ["-o", so, src] + list(libs))
        _libs[name] = C.CDLL(so)
    return _libs[name]


def trace_host_ex_lib():
    csrc = os.path.join(H.ROOT, "tweeker_raytracer_b200", "csrc")
    native = os.path.join(H.ROOT, "tests", "native")
    return _build("libtrace_host_ex.so",
                  ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I" + os.path.join(H.ROOT, "include"), "-I" + csrc,
                   "-I/usr/local/cuda/include"],
                  os.path.join(native, "trace_host_ex.cpp"),
                  [os.path.join(native, "trace_host.cpp"), os.path.join(csrc, "trace.cuh"), os.path.join(csrc, "rtc_internal.h")])


def oracle_masks_lib():
    odir = os.path.join(H.ROOT, "oracle")
    L = _build("liborc_masks.so",
               ["gcc", "-O2", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-I" + os.path.join(H.ROOT, "include"), "-I" + odir],
               os.path.join(H.ROOT, "tests", "native", "oracle_masks.c"),
               [os.path.join(odir, f) for f in ("rt_oracle.c", "rt_oracle.h", "wide_bvh.inc")], ["-lm", "-lpthread"])
    for fn in (L.mk_trace_closest, L.mk_trace_any):
        fn.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p]
        fn.restype = None
    L.mk_wide_trace.argtypes = [C.POINTER(orc.WideScene), C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p,
                                C.POINTER(C.c_uint64)]
    L.mk_wide_trace.restype = None
    return L


def product_trace_ex(export, rays, masks, ray_mask=0xFF, flags=0, any_hit=False, cap=0):
    """The FILTER traversal of csrc/trace.cuh on the host over an exported (or host-built) wide BVH: (hits, (nodes, tris, instances),
    stack overflows).  masks: one byte per instance; cap: the triangle schedule (0 group, 1 or 2 triangles per step)."""
    L = trace_host_ex_lib()
    ws, sizes, keep = H._wide_scene(export)
    rays = np.ascontiguousarray(rays, dtype=orc.RAY_DTYPE)
    m = np.ascontiguousarray(masks, dtype=np.uint8)
    assert len(m) == len(export["instance_gas"])
    hits = np.zeros(len(rays), dtype=orc.HIT_DTYPE)
    counts = (C.c_uint64 * 3)()
    overflows = C.c_uint64(0)
    L.th_trace_ex.argtypes = [C.POINTER(orc.WideScene), C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int,
                              C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    rc = L.th_trace_ex(C.byref(ws), *sizes, rays.ctypes.data_as(C.c_void_p), len(rays), 1 if any_hit else 0, m.ctypes.data_as(C.c_void_p),
                       int(ray_mask), int(flags), int(cap), hits.ctypes.data_as(C.c_void_p), counts, C.byref(overflows))
    assert rc == 0
    return hits, (int(counts[0]), int(counts[1]), int(counts[2])), int(overflows.value)


class MaskedScene:
    """An oracle scene (orc.Scene, committed) of `n` instances with 8-bit visibility masks, 0xFF by default."""

    def __init__(self, scene, n):
        self.scene, self.masks = scene, np.full(n, 0xFF, dtype=np.uint8)
        self.L = oracle_masks_lib()

    def set_instance_masks(self, first, masks):
        m = np.asarray(masks, dtype=np.uint8)
        self.masks[first:first + len(m)] = m

    def _args(self, rays, ray_mask, flags, rule):
        rays = np.ascontiguousarray(rays, dtype=orc.RAY_DTYPE)
        mode = {"det": 1, "normal": 0}[rule]
        return rays, (self.scene.h, self.masks.ctypes.data_as(C.c_void_p), int(ray_mask), int(flags), mode,
                      rays.ctypes.data_as(C.c_void_p), len(rays))

    def trace_closest_ex(self, rays, ray_mask=0xFF, flags=0, rule="det"):
        rays, args = self._args(rays, ray_mask, flags, rule)
        hits = np.zeros(len(rays), dtype=orc.HIT_DTYPE)
        self.L.mk_trace_closest(*args, hits.ctypes.data_as(C.c_void_p))
        return hits

    def trace_any_ex(self, rays, ray_mask=0xFF, flags=0, rule="det"):
        rays, args = self._args(rays, ray_mask, flags, rule)
        occ = np.zeros(len(rays), dtype=np.uint8)
        self.L.mk_trace_any(*args, occ.ctypes.data_as(C.c_void_p))
        return occ

    def close(self):
        self.scene.close()


def wide_trace_ex(export, rays, masks=None, ray_mask=0xFF, flags=0, any_hit=False):
    """oracle/wide_bvh.inc's traversal of the exported wide BVH with the mask and facing tests: (hits, (nodes, tris, instances))."""
    L = oracle_masks_lib()
    ws, _, keep = H._wide_scene(export)
    m = np.ascontiguousarray(masks if masks is not None else np.full(len(export["instance_gas"]), 0xFF), dtype=np.uint8)
    rays = np.ascontiguousarray(rays, dtype=orc.RAY_DTYPE)
    hits = np.zeros(len(rays), dtype=orc.HIT_DTYPE)
    counts = (C.c_uint64 * 3)()
    L.mk_wide_trace(C.byref(ws), rays.ctypes.data_as(C.c_void_p), len(rays), 1 if any_hit else 0, m.ctypes.data_as(C.c_void_p),
                    int(ray_mask), int(flags), hits.ctypes.data_as(C.c_void_p), counts)
    return hits, (int(counts[0]), int(counts[1]), int(counts[2]))
