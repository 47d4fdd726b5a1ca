"""Test infrastructure of the device-side queries (include/rtc_device.cuh): tests/native/device_trace_kernels.cu, user kernels that
call them, built by nvcc with -Iinclude as the only include path into a directory of the caller's and loaded with ctypes.  Shared
by tests/test_gpu_device_trace.py and tools/device_trace_bench.py."""
import ctypes as C
import os
import subprocess

import numpy as np

import helpers as H
from tweeker_raytracer_b200 import core

SOURCE = os.path.join(H.ROOT, "tests", "native", "device_trace_kernels.cu")


class Module:
    """one build of the user kernels; flags: extra nvcc flags (e.g. ["-fmad=false"])"""

    def __init__(self, out_dir, flags=()):
        so = os.path.join(str(out_dir), "libdevice_trace%s.so" % "".join(f.replace("=", "_") for f in flags))
        subprocess.check_call(["/usr/local/cuda/bin/nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a"] + list(flags)
                              + ["-I" + os.path.join(H.ROOT, "include"), "-Xcompiler", "-fPIC", "-shared", "-cudart", "shared", "-o", so, SOURCE])
        self.L = C.CDLL(so)
        u64, u32 = C.c_uint64, C.c_uint32
        self.L.dt_query.argtypes = [C.c_int, u64, u64, u32, u64, u64, u32, u32, u64, u64, C.c_int, C.c_int, u64]
        self.L.dt_ao_fused.argtypes = [u64, u64, u32, u32, C.c_float, u64, u64, u64]
        self.L.dt_ao_rays.argtypes = [u64, u64, u32, u32, C.c_float, u64, u64]
        self.L.dt_ao_reduce.argtypes = [u64, u32, u32, u64, u64]
        self.L.dt_stack_overflows.argtypes = [u64, u64]

    @staticmethod
    def _check(rc):
        assert rc == 0, "CUDA error %d" % rc

    def query(self, ctx, top, d_rays, n, d_out, any_hit=False, d_masks=0, d_flags=0, mask=0xFF, flags=0, d_status=0, block=128, odd_only=False):
        """enqueues one user kernel on the context stream: closest (d_out: rtc_hit[n]) or any hit (uint32[n])"""
        self._check(self.L.dt_query(1 if any_hit else 0, int(top), int(d_rays), int(n), int(d_masks), int(d_flags), int(mask), int(flags),
                                    int(d_out), int(d_status), int(block), 1 if odd_only else 0, ctx.stream))

    def ao_fused(self, ctx, top, d_primary, n, samples, radius, d_hits, d_counts):
        self._check(self.L.dt_ao_fused(int(top), int(d_primary), n, samples, radius, int(d_hits), int(d_counts), ctx.stream))

    def ao_rays(self, ctx, d_primary, d_hits, n, samples, radius, d_ao):
        self._check(self.L.dt_ao_rays(int(d_primary), int(d_hits), n, samples, radius, int(d_ao), ctx.stream))

    def ao_reduce(self, ctx, d_occluded, n, samples, d_counts):
        self._check(self.L.dt_ao_reduce(int(d_occluded), n, samples, int(d_counts), ctx.stream))

    def ao_pipeline(self, ctx, top, d_primary, n, samples, radius, d_hits, d_ao, d_occluded, d_counts):
        """the same occlusion counts through the batch queries: rtc_trace_closest, a ray-writing kernel, rtc_trace_any, a reduction"""
        ctx.trace_closest(top, d_primary, n, d_hits)
        self.ao_rays(ctx, d_primary, d_hits, n, samples, radius, d_ao)
        ctx.trace_any(top, d_ao, n * samples, d_occluded)
        self.ao_reduce(ctx, d_occluded, n, samples, d_counts)

    def stack_overflows(self, ctx):
        d = ctx.malloc(16)
        try:
            self._check(self.L.dt_stack_overflows(d, ctx.stream))
            return int(ctx.download(d, np.uint32, 1)[0])
        finally:
            ctx.free(d)

    def trace_host(self, ctx, top, rays, any_hit=False, masks=None, flags=None, mask=0xFF, fl=0, block=128, odd_only=False):
        """host rays in, (hits or occluded, status) out; masks / flags: per ray (uint32) or None"""
        rays = np.ascontiguousarray(rays, dtype=core.RAY_DTYPE)
        n = len(rays)
        keep = [ctx.to_device(rays)]
        d_m = 0
        if masks is not None:
            keep.append(ctx.to_device(np.ascontiguousarray(masks, dtype=np.uint32))); d_m = keep[-1]
        d_f = 0
        if flags is not None:
            keep.append(ctx.to_device(np.ascontiguousarray(flags, dtype=np.uint32))); d_f = keep[-1]
        out_bytes = n * (4 if any_hit else 20)
        d_out, d_st = ctx.malloc(max(out_bytes, 16)), ctx.malloc(max(4 * n, 16))
        keep += [d_out, d_st]
        try:
            ctx.memset(d_out, 0xAB, out_bytes)
            ctx.memset(d_st, 0xFF, 4 * n)
            self.query(ctx, top, keep[0], n, d_out, any_hit, d_m, d_f, mask, fl, d_st, block, odd_only)
            out = ctx.download(d_out, np.uint32 if any_hit else core.HIT_DTYPE, n)
            return out, ctx.download(d_st, np.int32, n)
        finally:
            for p in keep:
                ctx.free(p)
