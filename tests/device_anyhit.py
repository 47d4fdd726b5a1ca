"""Test infrastructure of the any-hit callbacks of include/rtc_device.cuh (rtc_device_trace_closest_anyhit / _any_anyhit):

  * host_trace: the header compiled by g++ over an exported wide BVH (tests/native/device_anyhit_host.cpp), with a recording callback;
  * brute force (tests/native/oracle_anyhit.c) on a MaskedScene of tests/mask_oracle.py;
  * Module: the user kernels of tests/native/device_anyhit_kernels.cu, built by nvcc with -Iinclude as the only include path into a
    directory of the caller's and loaded with ctypes.
The decisions (ACCEPT, IGNORE, ALPHA, FRONT, NOT_SELF) are those of tests/native/anyhit_predicates.h.  Shared by
tests/test_cpu_device_anyhit.py, tests/test_gpu_device_anyhit.py and tools/device_anyhit_bench.py."""
import ctypes as C
import os
import subprocess

import numpy as np

import helpers as H
from mask_oracle import _build
from oracle import orc

ACCEPT, IGNORE, ALPHA, FRONT, NOT_SELF = range(5)
RECORD_DTYPE = np.dtype([("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("inst", "<u4"), ("prim", "<u4"), ("frontFacing", "<u4")])
INCLUDE = os.path.join(H.ROOT, "include")
CSRC = os.path.join(H.ROOT, "tweeker_raytracer_b200", "csrc")
NATIVE = os.path.join(H.ROOT, "tests", "native")
SOURCE = os.path.join(NATIVE, "device_anyhit_kernels.cu")
u64, u32 = C.c_uint64, C.c_uint32


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def per_ray(v, n, dtype=np.uint32):
    return np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=dtype), n))


def host_lib():
    L = _build("libdevice_anyhit_host.so",
               ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I" + INCLUDE, "-I" + CSRC, "-I/usr/local/cuda/include"],
               os.path.join(NATIVE, "device_anyhit_host.cpp"),
               [os.path.join(NATIVE, f) for f in ("trace_host.cpp", "anyhit_predicates.h")]
               + [os.path.join(INCLUDE, "rtc_device.cuh"), os.path.join(CSRC, "trace.cuh"), os.path.join(CSRC, "rtc_internal.h")])
    L.dah_trace.argtypes = ([C.POINTER(orc.WideScene), u32, u32, u32, C.c_void_p, C.c_void_p, C.c_void_p, u32, u32, C.c_void_p, u64,
                             C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, u32]
                            + [C.c_void_p] * 6 + [C.POINTER(u64), C.POINTER(u64)])
    return L


def host_constants():
    out = (C.c_int * 4)()
    host_lib().dah_constants(out)
    return dict(zip(("IGNORE", "ACCEPT", "ACCEPT_AND_END", "CANDIDATE_BYTES"), list(out)))


def host_trace(export, inst_masks, rays, ray_masks=0xFF, ray_flags=0, mode="closest", pred=ACCEPT, p0=0, p1=0, end=False, k=256,
               usable=1, abi=None):
    """The header on the host.  mode: closest / any (the any-hit queries), plain_closest / plain_any (rtc_device_trace_closest /
    _any).  Returns a dict: out (hits or occluded), status, calls, records (n x k), digest (n x 3), duplicates, reads."""
    from test_cpu_device_trace import constants
    L = host_lib()
    ws, sizes, keep = H._wide_scene(export)
    rays = np.ascontiguousarray(rays, dtype=orc.RAY_DTYPE)
    n = len(rays)
    im = np.ascontiguousarray(inst_masks, dtype=np.uint8)
    rm, rf, q0, q1 = per_ray(ray_masks, n), per_ray(ray_flags, n), per_ray(p0, n), per_ray(p1, n)
    hits = np.zeros(n, dtype=orc.HIT_DTYPE)
    occ = np.full(n, 7, dtype=np.uint32)
    status = np.full(n, -1, dtype=np.int32)
    calls = np.zeros(n, dtype=np.uint32)
    records = np.zeros((n, k), dtype=RECORD_DTYPE)
    digest = np.zeros((n, 3), dtype=np.uint32)
    dup, reads = u64(0), u64(0)
    m = {"closest": 0, "any": 1, "plain_closest": 2, "plain_any": 3}[mode]
    rc = L.dah_trace(C.byref(ws), *sizes, _ptr(im), usable, constants()["ABI"] if abi is None else abi, _ptr(rays), n, _ptr(rm), _ptr(rf), m,
                     pred, _ptr(q0), _ptr(q1), 1 if end else 0, k, _ptr(hits), _ptr(occ), _ptr(status), _ptr(calls), _ptr(records),
                     _ptr(digest), C.byref(dup), C.byref(reads))
    assert rc == 0
    return dict(out=occ if m in (1, 3) else hits, status=status, calls=calls, records=records, digest=digest, duplicates=int(dup.value),
                reads=int(reads.value))


def oracle_lib():
    odir = os.path.join(H.ROOT, "oracle")
    L = _build("liborc_anyhit.so",
               ["gcc", "-O2", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-I" + INCLUDE, "-I" + odir, "-I" + NATIVE],
               os.path.join(NATIVE, "oracle_anyhit.c"),
               [os.path.join(NATIVE, f) for f in ("oracle_masks.c", "anyhit_predicates.h")]
               + [os.path.join(odir, f) for f in ("rt_oracle.c", "rt_oracle.h", "wide_bvh.inc")], ["-lm", "-lpthread"])
    for fn in (L.ah_closest, L.ah_any):
        fn.argtypes = [C.c_void_p] * 3 + [u64] + [C.c_void_p] * 2 + [C.c_int] + [C.c_void_p] * 3
        fn.restype = None
    L.ah_candidates.argtypes = [C.c_void_p] * 3 + [u64] + [C.c_void_p] * 2 + [u32] + [C.c_void_p] * 2
    L.ah_candidates.restype = None
    return L


def _oracle_args(ref, rays, ray_masks, ray_flags):
    rays = np.ascontiguousarray(rays, dtype=orc.RAY_DTYPE)
    n = len(rays)
    rm, rf = per_ray(ray_masks, n), per_ray(ray_flags, n)
    return rays, [rm, rf], (ref.scene.h, _ptr(ref.masks), _ptr(rays), n, _ptr(rm), _ptr(rf))


def brute_closest(ref, rays, ray_masks=0xFF, ray_flags=0, pred=ACCEPT, p0=0, p1=0):
    """the smallest accepted candidate in (t, instance, primitive) order; ref: a MaskedScene"""
    rays, keep, args = _oracle_args(ref, rays, ray_masks, ray_flags)
    q0, q1 = per_ray(p0, len(rays)), per_ray(p1, len(rays))
    hits = np.zeros(len(rays), dtype=orc.HIT_DTYPE)
    oracle_lib().ah_closest(*args, pred, _ptr(q0), _ptr(q1), _ptr(hits))
    return hits


def brute_any(ref, rays, ray_masks=0xFF, ray_flags=0, pred=ACCEPT, p0=0, p1=0):
    rays, keep, args = _oracle_args(ref, rays, ray_masks, ray_flags)
    q0, q1 = per_ray(p0, len(rays)), per_ray(p1, len(rays))
    occ = np.zeros(len(rays), dtype=np.uint8)
    oracle_lib().ah_any(*args, pred, _ptr(q0), _ptr(q1), _ptr(occ))
    return occ


def brute_candidates(ref, rays, ray_masks=0xFF, ray_flags=0, k=256):
    """(records n x k, counts): every candidate of each ray after masks, culling and (tmin, tmax)"""
    rays, keep, args = _oracle_args(ref, rays, ray_masks, ray_flags)
    out = np.zeros((len(rays), k), dtype=RECORD_DTYPE)
    counts = np.zeros(len(rays), dtype=np.uint32)
    oracle_lib().ah_candidates(*args, k, _ptr(out), _ptr(counts))
    return out, counts


def record_keys(records, count):
    """the sorted candidate list of one ray as (t bits, inst, prim, u bits, v bits, frontFacing) tuples"""
    r = records[:count]
    return sorted(zip(r["t"].view(np.uint32).tolist(), r["inst"].tolist(), r["prim"].tolist(), r["u"].view(np.uint32).tolist(),
                      r["v"].view(np.uint32).tolist(), r["frontFacing"].tolist()))


class Args(C.Structure):
    """da_args of device_anyhit_kernels.cu"""
    _fields_ = [(f, u64) for f in ("top", "rays", "masks", "flags", "p0", "p1", "out", "status", "calls", "records", "digest")] + \
               [(f, u32) for f in ("n", "mask", "fl", "k")] + [(f, C.c_int) for f in ("pred", "end", "oddOnly", "pad")]


class Module:
    """one build of the user kernels; flags: extra nvcc flags (e.g. ["-fmad=false"])"""

    def __init__(self, out_dir, flags=()):
        so = os.path.join(str(out_dir), "libdevice_anyhit%s.so" % "".join(f.replace("=", "_") for f in flags))
        subprocess.check_call(["/usr/local/cuda/bin/nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a"] + list(flags)
                              + ["-I" + INCLUDE, "-Xcompiler", "-fPIC", "-shared", "-cudart", "shared", "-o", so, SOURCE])
        self.L = C.CDLL(so)
        self.L.da_query.argtypes = [C.c_int, C.POINTER(Args), C.c_int, u64]
        self.L.da_lean.argtypes = [C.c_int, C.c_int, u64, u64, u32, u32, u64, u64, u64]
        self.L.da_alpha_restart.argtypes = [u64, u64, u32, u32, u64, u64, u64]
        self.L.da_secondary_rays.argtypes = [u64, u64, u32, u64, u64]
        self.L.da_self_skip.argtypes = [u64] * 2 + [u32] + [u64] * 4
        self.L.da_stack_overflows.argtypes = [u64, u64]

    @staticmethod
    def _check(rc):
        assert rc == 0, "CUDA error %d" % rc

    def lean(self, ctx, mode, any_hit, top, d_rays, n, d_out, alpha=0, d_digest=0):
        self._check(self.L.da_lean(1 if any_hit else 0, mode, int(top), int(d_rays), n, alpha, int(d_out), int(d_digest), ctx.stream))

    def alpha_restart(self, ctx, top, d_rays, n, alpha, d_hits, d_restarts):
        self._check(self.L.da_alpha_restart(int(top), int(d_rays), n, alpha, int(d_hits), int(d_restarts), ctx.stream))

    def secondary_rays(self, ctx, d_primary, d_hits, n, d_out):
        self._check(self.L.da_secondary_rays(int(d_primary), int(d_hits), n, int(d_out), ctx.stream))

    def self_skip(self, ctx, top, d_primary, n, d_hits, d_secondary, d_second_hits):
        self._check(self.L.da_self_skip(int(top), int(d_primary), n, int(d_hits), int(d_secondary), int(d_second_hits), ctx.stream))

    def stack_overflows(self, ctx):
        d = ctx.malloc(16)
        try:
            self._check(self.L.da_stack_overflows(d, ctx.stream))
            return int(ctx.download(d, np.uint32, 1)[0])
        finally:
            ctx.free(d)

    def trace_host(self, ctx, top, rays, any_hit=False, pred=ACCEPT, p0=None, p1=None, end=False, masks=None, flags=None, mask=0xFF, fl=0,
                   k=0, block=128, odd_only=False):
        """host rays in, dict(out, status, calls, records, digest) out; masks / flags / p0 / p1: per ray (uint32) or None"""
        from tweeker_raytracer_b200 import core
        rays = np.ascontiguousarray(rays, dtype=core.RAY_DTYPE)
        n = len(rays)
        keep = []

        def dev(a):
            if a is None:
                return 0
            keep.append(ctx.to_device(np.ascontiguousarray(a, dtype=np.uint32)))
            return keep[-1]

        out_bytes = n * (4 if any_hit else 20)
        a = Args(top=int(top), rays=0, masks=dev(masks), flags=dev(flags), p0=dev(p0), p1=dev(p1), n=n, mask=mask, fl=fl, k=k, pred=pred,
                 end=1 if end else 0, oddOnly=1 if odd_only else 0)
        keep.append(ctx.to_device(rays)); a.rays = keep[-1]
        for name, nbytes, fill in (("out", out_bytes, 0xAB), ("status", 4 * n, 0xFF), ("calls", 4 * n, 0xFF), ("digest", 12 * n, 0),
                                   ("records", 24 * n * k, 0)):
            if nbytes == 0:
                continue
            keep.append(ctx.malloc(max(nbytes, 16)))
            ctx.memset(keep[-1], fill, nbytes)
            setattr(a, name, keep[-1])
        try:
            self._check(self.L.da_query(1 if any_hit else 0, C.byref(a), block, ctx.stream))
            res = dict(out=ctx.download(a.out, np.uint32 if any_hit else core.HIT_DTYPE, n), status=ctx.download(a.status, np.int32, n),
                       calls=ctx.download(a.calls, np.uint32, n), digest=ctx.download(a.digest, np.uint32, 3 * n).reshape(n, 3))
            if k:
                res["records"] = ctx.download(a.records, RECORD_DTYPE, n * k).reshape(n, k)
            return res
        finally:
            for p in keep:
                ctx.free(p)
