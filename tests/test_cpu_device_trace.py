"""CPU tests of the device-side queries of include/rtc_device.cuh (rtc_device_trace_closest / rtc_device_trace_any).

The header is compiled by g++ (tests/native/device_trace_host.cpp, with the intrinsic shims of tests/native/trace_host.cpp) and held
  * with a random mask and flag set per ray, to the oracle's masks brute force (tests/native/oracle_masks.c), bit for bit, on the
    fuzz scenes and the degenerate soups of tests/test_cpu_trace_masks.py;
  * with one mask and flag set for all rays, to the filtered traversal of rtc_trace_*_ex on the host (trace_host_ex.cpp);
  * on every refusal, to a miss without a single node, leaf, instance-record or mask read.
nvcc compiles the header for sm_100a with -Iinclude as the only include path, with the default flags and with -fmad=false, and
device-links two translation units of one -rdc=true program.  The storage hook the header uses changes no instruction of the
library's kernels."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import helpers as H
from mask_oracle import _build, product_trace_ex
from oracle import orc
from test_cpu_trace_masks import FLAG_SETS, fuzz_scene, soup_scene

NVCC = "/usr/local/cuda/bin/nvcc"
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
INCLUDE = os.path.join(H.ROOT, "include")
CSRC = os.path.join(H.ROOT, "tweeker_raytracer_b200", "csrc")
NATIVE = os.path.join(H.ROOT, "tests", "native")
KERNELS = os.path.join(NATIVE, "device_trace_kernels.cu")


def device_trace_host_lib():
    L = _build("libdevice_trace_host.so",
               ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I" + INCLUDE, "-I" + CSRC, "-I/usr/local/cuda/include"],
               os.path.join(NATIVE, "device_trace_host.cpp"),
               [os.path.join(NATIVE, "trace_host.cpp"), os.path.join(INCLUDE, "rtc_device.cuh"), os.path.join(CSRC, "trace.cuh"),
                os.path.join(CSRC, "rtc_internal.h")])
    L.dth_trace.argtypes = [C.POINTER(orc.WideScene), C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                            C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                            C.POINTER(C.c_uint64)]
    return L


def constants():
    out = (C.c_int * 5)()
    device_trace_host_lib().dth_constants(out)
    return dict(zip(("OK", "SCENE_UNUSABLE", "BAD_ARGUMENT", "ABI_MISMATCH", "ABI"), [int(v) & 0xffffffff for v in out]))


def device_trace(export, inst_masks, rays, ray_masks, ray_flags, any_hit=False, usable=1, abi=None):
    """The header on the host over an exported wide BVH laid out as the library lays it out behind topObject: (hits or occluded,
    status per ray, scene reads)."""
    L = device_trace_host_lib()
    ws, sizes, keep = H._wide_scene(export)
    rays = np.ascontiguousarray(rays, dtype=orc.RAY_DTYPE)
    im = np.ascontiguousarray(inst_masks, dtype=np.uint8)
    rm = np.ascontiguousarray(np.broadcast_to(ray_masks, len(rays)), dtype=np.uint32)
    rf = np.ascontiguousarray(np.broadcast_to(ray_flags, len(rays)), dtype=np.uint32)
    hits = np.zeros(len(rays), dtype=orc.HIT_DTYPE)
    occ = np.full(len(rays), 7, dtype=np.uint32)
    status = np.full(len(rays), -1, dtype=np.int32)
    reads = C.c_uint64(0)
    rc = L.dth_trace(C.byref(ws), *sizes, im.ctypes.data_as(C.c_void_p), usable, constants()["ABI"] if abi is None else abi,
                     rays.ctypes.data_as(C.c_void_p), len(rays), rm.ctypes.data_as(C.c_void_p), rf.ctypes.data_as(C.c_void_p),
                     1 if any_hit else 0, hits.ctypes.data_as(C.c_void_p), occ.ctypes.data_as(C.c_void_p), status.ctypes.data_as(C.c_void_p),
                     C.byref(reads))
    assert rc == 0
    return (occ if any_hit else hits), status, int(reads.value)


def per_ray_filters(rng, n):
    """a mask and a flag set per ray: ten random masks plus 0 and 0xFF, every flag set"""
    palette = np.concatenate([rng.integers(1, 255, size=10), [0, 0xFF]]).astype(np.uint32)
    return palette[rng.integers(0, len(palette), size=n)], np.asarray(FLAG_SETS, dtype=np.uint32)[rng.integers(0, len(FLAG_SETS), size=n)]


def check_per_ray_against_brute_force(export, ref, rays, inst_masks, rng, label):
    ref.set_instance_masks(0, inst_masks)
    ray_masks, ray_flags = per_ray_filters(rng, len(rays))
    hits, status, _ = device_trace(export, inst_masks, rays, ray_masks, ray_flags)
    occ, status_any, _ = device_trace(export, inst_masks, rays, ray_masks, ray_flags, any_hit=True)
    assert (status == 0).all() and (status_any == 0).all()
    groups = 0
    for m, f in sorted(set(zip(ray_masks.tolist(), ray_flags.tolist()))):
        sel = np.flatnonzero((ray_masks == m) & (ray_flags == f))
        assert H.hits_equal(hits[sel], ref.trace_closest_ex(rays[sel], m, f)), (label, m, f)
        assert np.array_equal(occ[sel].astype(bool), ref.trace_any_ex(rays[sel], m, f).astype(bool)), (label, m, f)
        groups += 1
    assert groups >= 30
    assert (hits["inst"] != 0xffffffff).mean() > 0.02, label


@pytest.mark.parametrize("seed", list(range(4)))
def test_per_ray_masks_and_flags_equal_brute_force_on_fuzz_scenes(built, tmp_path, seed):
    app, export, ref = fuzz_scene(tmp_path, seed)
    rng = np.random.default_rng(500 + seed)
    masks = rng.integers(0, 256, size=len(export["instance_gas"])).astype(np.uint8)
    rays = H.random_rays(4000, seed=seed, lo=(-5, 0.05, -5), hi=(5, 4, 5))
    check_per_ray_against_brute_force(export, ref, rays, masks, rng, "fuzz %d" % seed)
    app.close()


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_per_ray_masks_and_flags_equal_brute_force_on_degenerate_soups(built, seed):
    export, ref, rays = soup_scene(seed)
    rng = np.random.default_rng(600 + seed)
    masks = rng.integers(0, 256, size=len(export["instance_gas"])).astype(np.uint8)
    check_per_ray_against_brute_force(export, ref, rays, masks, rng, "soup %d" % seed)
    ref.close()


@pytest.mark.parametrize("seed", [0, 5])
def test_one_mask_for_all_rays_equals_the_ex_traversal(built, tmp_path, seed):
    app, export, ref = fuzz_scene(tmp_path, seed)
    rng = np.random.default_rng(700 + seed)
    masks = rng.integers(0, 256, size=len(export["instance_gas"])).astype(np.uint8)
    masks[0] = 0                                  # never entered, even by (0xFF, 0)
    rays = H.random_rays(3000, seed=seed, lo=(-5, 0.05, -5), hi=(5, 4, 5))
    for flags in FLAG_SETS:
        for ray_mask in (0xFF, int(rng.integers(1, 255)), 0):
            want, _, _ = product_trace_ex(export, rays, masks, ray_mask, flags)
            got, status, _ = device_trace(export, masks, rays, ray_mask, flags)
            assert (status == 0).all() and H.hits_equal(got, want), (flags, ray_mask)
            want_any, _, _ = product_trace_ex(export, rays, masks, ray_mask, flags, any_hit=True)
            got_any, status, _ = device_trace(export, masks, rays, ray_mask, flags, any_hit=True)
            assert (status == 0).all() and np.array_equal(got_any, (want_any["inst"] != 0xffffffff).astype(np.uint32)), (flags, ray_mask)
    app.close()


def test_every_refusal_is_a_miss_without_a_scene_read(built):
    export, _, rays = soup_scene(1)
    k = constants()
    rays = rays[:500]
    masks = np.full(len(export["instance_gas"]), 0xFF, dtype=np.uint8)
    hits, status, reads = device_trace(export, masks, rays, 0xFF, 0)
    assert (status == k["OK"]).all() and reads > 0 and (hits["inst"] != 0xffffffff).any()
    cases = [("mask 0x100", dict(ray_masks=0x100, ray_flags=0), k["BAD_ARGUMENT"]),
             ("mask 0xFFFFFFFF", dict(ray_masks=0xFFFFFFFF, ray_flags=0), k["BAD_ARGUMENT"]),
             ("flag 4", dict(ray_masks=0xFF, ray_flags=4), k["BAD_ARGUMENT"]),
             ("flag bit 31", dict(ray_masks=0xFF, ray_flags=0x80000001), k["BAD_ARGUMENT"]),
             ("usable 0", dict(ray_masks=0xFF, ray_flags=0, usable=0), k["SCENE_UNUSABLE"]),
             ("abi", dict(ray_masks=0xFF, ray_flags=0, abi=k["ABI"] ^ 1), k["ABI_MISMATCH"]),
             ("abi of no record", dict(ray_masks=0xFF, ray_flags=0, abi=0), k["ABI_MISMATCH"])]
    for label, kw, want in cases:
        hits, status, reads = device_trace(export, masks, rays, **kw)
        assert (status == want).all() and reads == 0, label
        assert (hits["t"] == -1).all() and (hits["inst"] == 0xffffffff).all() and (hits["prim"] == 0xffffffff).all(), label
        assert (hits["u"] == 0).all() and (hits["v"] == 0).all(), label
        occ, status, reads = device_trace(export, masks, rays, any_hit=True, **kw)
        assert (status == want).all() and reads == 0 and (occ == 0).all(), label
    assert (k["OK"], k["SCENE_UNUSABLE"], k["BAD_ARGUMENT"], k["ABI_MISMATCH"]) == (0, 1, 2, 3)


def ptxas_report(text):
    """{kernel: (registers, stack frame bytes, spill store bytes)} from -Xptxas -v"""
    out, name = {}, None
    for line in text.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores", line)
        if m and name:
            out[name] = [None, int(m.group(1)), int(m.group(2))]
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and name in out:
            out[name][0] = int(m.group(1))
    return {k: tuple(v) for k, v in out.items()}


@pytest.mark.parametrize("flags", [[], ["-fmad=false"]], ids=["default", "fmad-false"])
def test_header_compiles_for_sm100a_with_the_include_directory_alone(tmp_path, flags):
    r = subprocess.run([NVCC, "-O3", "-std=c++17"] + ARCH + flags + ["-I" + INCLUDE, "-Xptxas", "-v", "-c", KERNELS,
                        "-o", str(tmp_path / "k.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    report = ptxas_report(r.stderr)
    queries = {k: v for k, v in report.items() if "k_query" in k or "k_ao_fused" in k}
    assert len(queries) == 5
    for name, (regs, stack, spills) in sorted(queries.items()):
        print("%-12s %-90s %3d registers, %3d B stack, %3d B spilled" % (" ".join(flags) or "default", name, regs, stack, spills))
        if "ILb0EEEv" in name or "k_ao_fused" in name:       # the kernels not squeezed into 64 registers for 1024-thread blocks
            assert spills == 0 and stack == 320, name


def test_two_translation_units_device_link(tmp_path):
    srcs = {"a.cu": "__global__ void ka(uint64_t top, const rtc_ray* r, rtc_hit* h) { rtc_device_trace_closest(top, r[threadIdx.x], h + threadIdx.x); }",
            "b.cu": "__global__ void kb(uint64_t top, const rtc_ray* r, uint32_t* o) { rtc_device_trace_any(top, r[threadIdx.x], o + threadIdx.x, 1u, "
                    "RTC_RAY_CULL_BACK_FACING); }"}
    objs = []
    for name, body in srcs.items():
        src = tmp_path / name
        src.write_text('#include "rtc_device.cuh"\n' + body + "\n")
        obj = str(tmp_path / (name + ".o"))
        subprocess.run([NVCC, "-std=c++17"] + ARCH + ["-rdc=true", "-I" + INCLUDE, "-c", str(src), "-o", obj], check=True)
        objs.append(obj)
    r = subprocess.run([NVCC] + ARCH + ["-dlink"] + objs + ["-o", str(tmp_path / "link.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def normalized_sass(obj):
    """cuobjdump -sass without what depends on the source path: the identifier line and the per-file hash of anonymous-namespace
    names"""
    text = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    text = re.sub(r"(?m)^.*identifier = .*$", "", text)
    return re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", text)


def test_overflow_storage_hook_changes_no_kernel(built, tmp_path):
    """kernels_trace.o and kernels_shade.o as built equal a build whose trace.cuh defines the overflow counter without the hook"""
    src = tmp_path / "csrc"
    shutil.copytree(CSRC, src)
    text = (src / "trace.cuh").read_text()
    plain = re.sub(r"#ifndef RTC_STACK_OVERFLOW_STORAGE\n#define RTC_STACK_OVERFLOW_STORAGE\n#endif\n", "", text)
    plain = plain.replace("RTC_STACK_OVERFLOW_STORAGE __device__", "__device__")
    assert plain != text and "RTC_STACK_OVERFLOW_STORAGE __device__" not in plain
    (src / "trace.cuh").write_text(plain)
    common = [NVCC, "-O3", "-std=c++17"] + ARCH + ["-lineinfo", "-Xcompiler", "-fPIC", "-I" + INCLUDE, "-I" + str(src)]
    jobs = {"kernels_trace": subprocess.Popen(common + ["-c", str(src / "kernels_trace.cu"), "-o", str(tmp_path / "kernels_trace.o")]),
            "kernels_shade": subprocess.Popen(common + ["-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-c", str(src / "kernels_shade.cu"),
                                                        "-o", str(tmp_path / "kernels_shade.o")])}
    for name, job in jobs.items():
        assert job.wait() == 0, name
    for name in jobs:
        built_obj = os.path.join(H.ROOT, "tweeker_raytracer_b200", "lib", name + ".o")
        assert normalized_sass(built_obj) == normalized_sass(str(tmp_path / (name + ".o"))), name
