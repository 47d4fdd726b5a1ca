"""Shared helpers of the test-suite: scene files in temp dirs, App -> oracle scene conversion, ray sets."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import orc  # noqa: E402  (test infrastructure)

SCENES = os.path.join(ROOT, "scenes")


def system_text(name, **overrides):
    """Reads scenes/system_<name>.txt and replaces/appends `keyword value` lines."""
    with open(os.path.join(SCENES, "system_%s.txt" % name)) as f:
        lines = f.read().splitlines()
    out = []
    seen = set()
    for line in lines:
        key = line.split()[0] if line.split() else ""
        if key in overrides:
            out.append("%s %s" % (key, overrides[key]))
            seen.add(key)
        else:
            out.append(line)
    for k, v in overrides.items():
        if k not in seen:
            out.append("%s %s" % (k, v))
    return "\n".join(out) + "\n"


def write_system(tmpdir, name, **overrides):
    path = os.path.join(str(tmpdir), "system_%s.txt" % name)
    with open(path, "w") as f:
        f.write(system_text(name, **overrides))
    return path


def scene_path(name):
    return os.path.join(SCENES, "scene_%s.txt" % name)


def oracle_scene(app, variant="pinned", instances=None):
    """Feeds the scene an App loaded (geometries, flattened instances, materials, lights, camera, environment) to the oracle.
    instances: [(transform, geometry, material, light)] replaces the App's instance list."""
    s = orc.Scene(variant)
    for g in range(app.info.numGeometries):
        attrs, idx = app.geometry(g)
        s.add_geometry(attrs, idx)
    if instances is None:
        instances = [app.instance(i) for i in range(app.info.numInstances)]
    for t, g, m, l in instances:
        s.add_instance(t, g, m, l)
    s.set_materials(app.materials())
    s.set_lights(app.lights())
    s.set_camera(app.camera())
    env = app.environment()
    if env is not None:
        s.set_env(env[0], env[1], env[2], env[3])
    s.commit()
    return s


def oracle_sys(app, device_index=0):
    """SystemData in the oracle's ctypes type, copied field by field from the host's."""
    src = app.system_data(device_index)
    dst = orc.SystemData()
    for name, _ in orc.SystemData._fields_:
        v = getattr(src, name)
        if name in ("resolution", "tileSize", "tileShift", "pathLengths"):
            getattr(dst, name).x, getattr(dst, name).y = v.x, v.y
        elif name == "rect":
            for k in range(4):
                dst.rect[k] = v[k]
        else:
            setattr(dst, name, v)
    return dst


def random_rays(n, seed, lo=(-1.2, -0.2, -1.2), hi=(1.2, 2.2, 1.2), tmin=5e-5, tmax=1e27):
    """Incoherent rays: origins uniform in a box, directions uniform on the sphere."""
    rng = np.random.default_rng(seed)
    rays = np.zeros(n, dtype=orc.RAY_DTYPE)
    o = rng.uniform(lo, hi, size=(n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    rays["ox"], rays["oy"], rays["oz"] = o[:, 0], o[:, 1], o[:, 2]
    rays["dx"], rays["dy"], rays["dz"] = d[:, 0], d[:, 1], d[:, 2]
    rays["tmin"] = tmin
    rays["tmax"] = tmax
    return rays


def hits_equal(a, b):
    """Bit-exact comparison of two hit arrays (t, u, v as raw bits; instance and primitive ids)."""
    return (np.array_equal(a["inst"], b["inst"]) and np.array_equal(a["prim"], b["prim"])
            and np.array_equal(a["t"].view(np.uint32), b["t"].view(np.uint32))
            and np.array_equal(a["u"].view(np.uint32), b["u"].view(np.uint32))
            and np.array_equal(a["v"].view(np.uint32), b["v"].view(np.uint32)))


def psnr(a, b, peak=1.0):
    mse = float(np.mean((np.asarray(a, dtype=np.float64) - np.asarray(b, dtype=np.float64)) ** 2))
    return 99.0 if mse == 0 else 10.0 * np.log10(peak * peak / mse)


def random_rgbe(w, h, seed):
    """Seeded Radiance RGBE texels [h, w, 4] uint8: mostly dark, a few very bright, three black rows and a black column band."""
    rng = np.random.default_rng(seed)
    img = np.zeros((h, w, 4), dtype=np.uint8)
    img[..., :3] = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    img[..., 3] = (128 + np.round(rng.random((h, w)) ** 4 * 6 - 3)).astype(np.uint8)       # exponents 2^-3 .. 2^3
    img[h // 3 - 1:h // 3 + 2] = 0                # three black rows: the middle one stays black after the 3x3 filter -> "equal distribution" branch
    img[:, w // 2:w // 2 + 3] = 0                 # a black band next to bright texels: what its Gaussian filter is there for
    return img


def write_rgbe_hdr(path, rgbe, rle=False):
    """Radiance .hdr file, top row first, from RGBE bytes [h, w, 4]: flat, or with rle=True adaptive run-length encoded
    scanlines (each channel as runs of one repeated byte and literal stretches)."""
    h, w = rgbe.shape[:2]
    rgbe = np.ascontiguousarray(rgbe, dtype=np.uint8)
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n-Y %d +X %d\n" % (h, w))
        if not rle:
            f.write(rgbe.tobytes())
        else:
            for row in rgbe:
                f.write(bytes((2, 2, w >> 8, w & 255)))
                for c in range(4):
                    f.write(_rle_bytes(row[:, c].tolist()))
    return path


def _rle_bytes(vals):
    """One channel of a scanline: a run of n >= 3 equal bytes is (128 + n, byte), anything else literal (n, n bytes)."""
    out, i, n = bytearray(), 0, len(vals)
    while i < n:
        run = 1
        while i + run < n and run < 127 and vals[i + run] == vals[i]:
            run += 1
        if run >= 3:
            out += bytes((128 + run, vals[i]))
            i += run
            continue
        j = i
        while j < n and j - i < 128 and not (j + 2 < n and vals[j] == vals[j + 1] == vals[j + 2]):
            j += 1
        out += bytes([j - i] + vals[i:j])
        i = j
    return bytes(out)


PORTABLE_MATH_SRC = r"""
#include "rt_portable_math.h"
#include <math.h>
#define W(name, expr) void name(const float* x, const float* y, float* o, int n) { for (int i = 0; i < n; ++i) o[i] = expr; }
W(p_sin, rt_sinf(x[i])) W(p_cos, rt_cosf(x[i])) W(p_atan, rt_atanf(x[i])) W(p_atan2, rt_atan2f(x[i], y[i]))
W(p_acos, rt_acosf(x[i])) W(p_exp, rt_expf(x[i])) W(p_log, rt_logf(x[i])) W(p_pow, rt_powf(x[i], y[i]))
W(p_div, x[i] / y[i]) W(p_sqrt, sqrtf(x[i])) W(p_muladd, x[i] * y[i] + x[i])
"""


def portable_math_lib(tmpdir):
    """include/rt_portable_math.h compiled for the host with the oracle's flags: the CPU side of the arithmetic both the oracle
    and the shading kernels are defined by (tests/test_cpu_portable_math.py, tests/test_gpu_edge_cases.py)."""
    import ctypes
    import subprocess
    src = os.path.join(str(tmpdir), "pm.c")
    with open(src, "w") as f:
        f.write(PORTABLE_MATH_SRC)
    so = os.path.join(str(tmpdir), "pm.so")
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-I" + os.path.join(ROOT, "include"), "-o", so, src, "-lm"])
    return ctypes.CDLL(so)


def portable_math_call(lib, name, x, y=None):
    import ctypes
    x = np.ascontiguousarray(x, dtype=np.float32)
    y = np.ascontiguousarray(y if y is not None else np.zeros_like(x), dtype=np.float32)
    o = np.zeros_like(x)
    getattr(lib, "p_" + name)(x.ctypes.data_as(ctypes.c_void_p), y.ctypes.data_as(ctypes.c_void_p), o.ctypes.data_as(ctypes.c_void_p), len(x))
    return o


_trace_host = {}


def product_trace_lib(defs=()):
    """tests/native/trace_host.cpp: the PRODUCT's traversal source (csrc/trace.cuh) compiled for the host by g++; built once per
    session into oracle/_build (git-ignored) next to the oracle.  defs: extra -D switches of trace.cuh (e.g.
    "RTC_ONE_TRI_PER_STEP=1"), each combination its own library."""
    key = tuple(defs)
    if key not in _trace_host:
        import ctypes
        import subprocess
        src = os.path.join(ROOT, "tests", "native", "trace_host.cpp")
        out_dir = os.path.join(ROOT, "oracle", "_build")
        os.makedirs(out_dir, exist_ok=True)
        tag = "".join("_" + "".join(ch if ch.isalnum() else "-" for ch in d) for d in key)
        so = os.path.join(out_dir, "libtrace_host%s.so" % tag)
        deps = [src, os.path.join(ROOT, "tweeker_raytracer_b200", "csrc", "trace.cuh"), os.path.join(ROOT, "tweeker_raytracer_b200", "csrc", "rtc_internal.h")]
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include"),
                                   "-I" + os.path.join(ROOT, "tweeker_raytracer_b200", "csrc"), "-I/usr/local/cuda/include"]
                                  + ["-D" + d for d in key] + ["-o", so, src])
        _trace_host[key] = ctypes.CDLL(so)
    return _trace_host[key]


def _wide_scene(export):
    """An exported (or host-built) wide BVH marshalled for tests/native/trace_host.cpp: (WideScene, the scalar / size arguments that
    follow it, the arrays that must stay alive during the call)."""
    import ctypes as C
    handles = sorted(export["gas"])
    slot = {g: k for k, g in enumerate(handles)}
    inst_gas = np.ascontiguousarray([slot[int(g)] for g in export["instance_gas"]], dtype=np.uint32)
    keep_n = [np.ascontiguousarray(export["gas"][g][0]) for g in handles]
    keep_t = [np.ascontiguousarray(export["gas"][g][1], dtype=np.float32) for g in handles]
    node_ptrs = (C.c_void_p * max(len(handles), 1))(*[a.ctypes.data for a in keep_n])
    tri_ptrs = (C.c_void_p * max(len(handles), 1))(*[a.ctypes.data for a in keep_t])
    n_nodes = np.ascontiguousarray([len(a) for a in keep_n], dtype=np.uint32)
    n_tris = np.ascontiguousarray([len(a) for a in keep_t], dtype=np.uint32)
    tn, tl, w2o = (np.ascontiguousarray(export[k]) for k in ("tlas_nodes", "tlas_leaves", "world_to_object"))
    ws = orc.WideScene(tn.ctypes.data, tl.ctypes.data, w2o.ctypes.data, inst_gas.ctypes.data, C.cast(node_ptrs, C.c_void_p), C.cast(tri_ptrs, C.c_void_p),
                       len(export["instance_gas"]))
    sizes = (len(tn), len(tl), len(handles), n_nodes.ctypes.data_as(C.c_void_p), n_tris.ctypes.data_as(C.c_void_p))
    return ws, sizes, (inst_gas, keep_n, keep_t, node_ptrs, tri_ptrs, n_nodes, n_tris, tn, tl, w2o)


def product_trace(export, rays, any_hit=False, skip=None, defs=()):
    """Runs the host build of csrc/trace.cuh over an exported (or host-built) wide BVH: (hits, (nodes, tris, instances), stack
    overflows).  skip: [n, 3] uint32 keys (t bits, instance, primitive) -> the closest candidate AFTER the key (SKIP variant)."""
    import ctypes as C
    L = product_trace_lib(defs)
    ws, sizes, keep = _wide_scene(export)
    rays = np.ascontiguousarray(rays, dtype=orc.RAY_DTYPE)
    hits = np.zeros(len(rays), dtype=orc.HIT_DTYPE)
    counts = (C.c_uint64 * 3)()
    overflows = C.c_uint64(0)
    skip_ptr = None
    if skip is not None:
        skip = np.ascontiguousarray(skip, dtype=np.uint32).reshape(len(rays), 3)
        skip_ptr = skip.ctypes.data_as(C.c_void_p)
    L.th_trace.argtypes = [C.POINTER(orc.WideScene), C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int,
                           C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    rc = L.th_trace(C.byref(ws), *sizes, rays.ctypes.data_as(C.c_void_p), len(rays), 1 if any_hit else 0, skip_ptr, hits.ctypes.data_as(C.c_void_p), counts, C.byref(overflows))
    assert rc == 0
    return hits, (int(counts[0]), int(counts[1]), int(counts[2])), int(overflows.value)


SIMD_COST_FIELDS = ["iterations", "node_passes", "tri_passes_max", "inst_passes", "lane_steps", "nodes", "tris", "instances", "refills", "rays"]


def product_simd_cost(export, rays, any_hit=False, fetch_threshold=12, defs=(), leaf_threshold=0):
    """Lock-step emulation of one persistent warp of trace_stream over `rays` in list order (tests/native/trace_host.cpp
    th_simd_cost): dict of SIMD_COST_FIELDS.  A model of what a warp pays (the maximum over its lanes per iteration)."""
    import ctypes as C
    L = product_trace_lib(defs)
    ws, sizes, keep = _wide_scene(export)
    rays = np.ascontiguousarray(rays, dtype=orc.RAY_DTYPE)
    out = (C.c_uint64 * 10)()
    L.th_simd_cost.argtypes = [C.POINTER(orc.WideScene), C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int,
                               C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64)]
    rc = L.th_simd_cost(C.byref(ws), *sizes, rays.ctypes.data_as(C.c_void_p), len(rays), 1 if any_hit else 0, fetch_threshold, leaf_threshold, out)
    assert rc == 0
    return {k: int(out[i]) for i, k in enumerate(SIMD_COST_FIELDS)}
