"""ctypes binding of librtcore.so -- the C ABI declared in include/rtc_core.h.

Thin by design: one Python method per C entry point, device addresses as plain ints.  The library is the
product; if it is missing this module raises (there is no fallback of any kind).
"""
import ctypes as C
import os

import numpy as np

_LIBDIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib")
LIB_PATH = os.path.join(_LIBDIR, "librtcore.so")

RAY_DTYPE = np.dtype([("ox", "f4"), ("oy", "f4"), ("oz", "f4"), ("tmin", "f4"), ("dx", "f4"), ("dy", "f4"), ("dz", "f4"), ("tmax", "f4")])
HIT_DTYPE = np.dtype([("t", "f4"), ("u", "f4"), ("v", "f4"), ("inst", "u4"), ("prim", "u4")])
INSTANCE_DTYPE = np.dtype([("transform", "f4", 12), ("instanceId", "u4"), ("gas", "u4"), ("materialIndex", "i4"), ("lightIndex", "i4")])
assert RAY_DTYPE.itemsize == 32 and HIT_DTYPE.itemsize == 20 and INSTANCE_DTYPE.itemsize == 64

RAYGEN_FULL_FRAME, RAYGEN_LOCAL_COPY = 0, 1
BUILD_DEFAULT, BUILD_HOST_SAH, BUILD_GPU_LBVH = 0, 1, 2
REJECTED_INSTANCE = 0xFFFFFFFF      # instance_gas of a record rtc_ias_build_device rejected

# every symbol include/rtc_core.h declares (tests check that the built library exports all of them)
SYMBOLS = [
    "rtc_version", "rtc_last_error", "rtc_context_create", "rtc_context_destroy", "rtc_synchronize", "rtc_context_stream",
    "rtc_device_count", "rtc_device_name", "rtc_peer_can_access", "rtc_peer_enable", "rtc_peer_disable", "rtc_memcpy_peer",
    "rtc_malloc", "rtc_free", "rtc_upload", "rtc_download", "rtc_memset", "rtc_host_alloc", "rtc_host_free",
    "rtc_gas_build", "rtc_gas_destroy", "rtc_ias_build", "rtc_scene_info_get", "rtc_scene_destroy", "rtc_instance_inverse",
    "rtc_scene_set_instance_flags", "rtc_scene_set_albedo_textures", "rtc_texture_create", "rtc_texture_destroy",
    "rtc_launch", "rtc_launch_ex", "rtc_launch_counts_get", "rtc_launch_counts_reset", "rtc_timer_start", "rtc_timer_stop",
    "rtc_profile_enable", "rtc_profile_get", "rtc_trace_closest", "rtc_trace_any", "rtc_trace_count", "rtc_generate_primary",
    "rtc_composite", "rtc_tonemap", "rtc_stats_get", "rtc_stats_reset",
    "rtc_probe_gather", "rtc_probe_pipes", "rtc_scene_export", "rtc_gas_info", "rtc_gas_export",
    "rtc_probe_math",
    "rtc_host_gas_build", "rtc_host_ias_build", "rtc_host_accel_info", "rtc_host_accel_export", "rtc_host_accel_destroy",
    "rtc_trace_schedule_get", "rtc_trace_schedule_set",
    "rtc_gas_refit", "rtc_ias_update", "rtc_host_gas_refit", "rtc_host_ias_refit",
    "rtc_ias_rebuild", "rtc_host_ias_rebuild", "rtc_ias_update_device",
    "rtc_gas_rebuild", "rtc_host_gas_rebuild",
    "rtc_ias_create", "rtc_ias_build_device", "rtc_scene_rejected_instances",
    "rtc_gas_create", "rtc_gas_build_device", "rtc_gas_rejected_triangles",
    "rtc_scene_set_instance_masks", "rtc_trace_closest_ex", "rtc_trace_any_ex", "rtc_trace_count_ex",
]

MATH_FUNCTIONS = ["sin", "cos", "atan", "atan2", "acos", "exp", "log", "pow", "div", "sqrt", "muladd"]     # enum rtc_math_fn


class Stats(C.Structure):
    _fields_ = [("radianceRays", C.c_uint64), ("shadowRays", C.c_uint64), ("pathSamples", C.c_uint64),
                ("kernelLaunches", C.c_uint64), ("lastTraceMs", C.c_double), ("stackOverflows", C.c_uint64),
                ("cutoutGraphBuilds", C.c_uint64)]


class SceneInfo(C.Structure):
    _fields_ = [("numNodes", C.c_uint64), ("numTris", C.c_uint64), ("numInstances", C.c_uint32), ("numTlasNodes", C.c_uint32),
                ("numGas", C.c_uint32), ("numTlasLeaves", C.c_uint32), ("gasBuildMs", C.c_double), ("iasBuildMs", C.c_double)]


class TraceCounts(C.Structure):
    _fields_ = [("nodes", C.c_uint64), ("tris", C.c_uint64), ("instances", C.c_uint64), ("rays", C.c_uint64)]


SCHEDULE_GROUP, SCHEDULE_ONE_TRI, SCHEDULE_TWO_TRI = 0, 1, 2
RAY_CULL_BACK_FACING, RAY_CULL_FRONT_FACING = 1, 2      # rayFlags of rtc_trace_*_ex
SCHEDULE_NAMES = ["group", "one_tri", "two_tri"]


class TraceSchedule(C.Structure):
    _fields_ = [("schedule", C.c_int), ("decided", C.c_int), ("measured", C.c_int), ("pathsPerBatch", C.c_uint64),
                ("groupMs", C.c_float * 2), ("oneTriMs", C.c_float), ("twoTriMs", C.c_float)]


KERNEL_CLASSES = ["generate", "extend", "shade", "connect", "accumulate", "other"]


class Profile(C.Structure):
    _fields_ = [("ms", C.c_double * 6), ("launches", C.c_uint64 * 6)]


class RtcError(RuntimeError):
    pass


_lib = None


def lib():
    """Loads librtcore.so; raises when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RtcError("%s is missing: run `make` (or __graft_entry__.build()); there is no fallback path" % LIB_PATH)
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        L.rtc_last_error.restype = C.c_char_p
        L.rtc_context_stream.restype = C.c_uint64
        L.rtc_context_stream.argtypes = [C.c_void_p]
        L.rtc_context_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        for name in ("rtc_context_destroy", "rtc_synchronize", "rtc_stats_reset"):
            getattr(L, name).argtypes = [C.c_void_p]
        L.rtc_device_count.argtypes = [C.POINTER(C.c_int)]
        L.rtc_malloc.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.rtc_free.argtypes = [C.c_void_p, C.c_uint64]
        L.rtc_upload.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]
        L.rtc_download.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]
        L.rtc_memset.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_uint64]
        L.rtc_host_alloc.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
        L.rtc_host_free.argtypes = [C.c_void_p, C.c_void_p]
        L.rtc_gas_build.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]
        L.rtc_gas_destroy.argtypes = [C.c_void_p, C.c_uint32]
        L.rtc_ias_build.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64)]
        L.rtc_gas_refit.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64]
        L.rtc_ias_update.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]
        L.rtc_ias_update_device.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32]
        L.rtc_ias_rebuild.argtypes = [C.c_void_p, C.c_uint64]
        L.rtc_gas_rebuild.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64]
        L.rtc_ias_create.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64)]
        L.rtc_ias_build_device.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
        L.rtc_scene_rejected_instances.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32)]
        L.rtc_gas_create.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
        L.rtc_gas_build_device.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32]
        L.rtc_gas_rejected_triangles.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
        L.rtc_scene_info_get.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(SceneInfo)]
        L.rtc_scene_destroy.argtypes = [C.c_void_p, C.c_uint64]
        L.rtc_scene_set_instance_flags.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]
        L.rtc_scene_set_albedo_textures.argtypes = [C.c_void_p, C.c_uint64, C.c_int]
        L.rtc_texture_create.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint64)]
        L.rtc_texture_destroy.argtypes = [C.c_void_p, C.c_uint64]
        L.rtc_instance_inverse.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
        L.rtc_launch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int]
        L.rtc_launch_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.rtc_launch_counts_get.argtypes = [C.c_void_p, C.POINTER(TraceCounts)]
        L.rtc_launch_counts_reset.argtypes = [C.c_void_p]
        L.rtc_timer_start.argtypes = [C.c_void_p]
        L.rtc_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.rtc_profile_enable.argtypes = [C.c_void_p, C.c_int]
        L.rtc_profile_get.argtypes = [C.c_void_p, C.POINTER(Profile)]
        L.rtc_trace_closest.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64]
        L.rtc_trace_any.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64]
        L.rtc_trace_count.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(TraceCounts)]
        L.rtc_scene_set_instance_masks.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]
        L.rtc_trace_closest_ex.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
        L.rtc_trace_any_ex.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
        L.rtc_trace_count_ex.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_uint32, C.c_uint32, C.POINTER(TraceCounts)]
        L.rtc_generate_primary.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_uint64]
        L.rtc_composite.argtypes = [C.c_void_p, C.c_void_p]
        L.rtc_tonemap.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]
        L.rtc_stats_get.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.rtc_scene_export.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.rtc_gas_info.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.rtc_gas_export.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
        L.rtc_probe_gather.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(C.c_double)]
        L.rtc_probe_pipes.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
        L.rtc_probe_math.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
        L.rtc_trace_schedule_get.argtypes = [C.c_void_p, C.POINTER(TraceSchedule)]
        L.rtc_trace_schedule_set.argtypes = [C.c_void_p, C.c_int]
        L.rtc_host_gas_build.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
        L.rtc_host_ias_build.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
        L.rtc_host_gas_refit.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.rtc_host_ias_refit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
        L.rtc_host_ias_rebuild.argtypes = [C.c_void_p]
        L.rtc_host_gas_rebuild.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.rtc_host_accel_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_void_p]
        L.rtc_host_accel_export.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.rtc_host_accel_destroy.argtypes = [C.c_void_p]
        L.rtc_host_accel_destroy.restype = None
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise RtcError(lib().rtc_last_error().decode("utf-8", "replace"))


def _vertex_records(attrs):
    attrs = np.ascontiguousarray(attrs)
    return attrs, attrs.dtype.itemsize * int(np.prod(attrs.shape[1:], dtype=np.int64))      # records, bytes per vertex record


def _transforms(instances):
    n = len(instances)
    transforms = np.ascontiguousarray([np.asarray(t, dtype=np.float32).reshape(12) for t, _ in instances], dtype=np.float32).reshape(n, 12)
    return transforms, np.ascontiguousarray([g for _, g in instances], dtype=np.uint32)


def _host_export(L, accels, top, inst_gas, info):
    """Context.scene_export's layout of host-twin accels (accels[g] = geometry g, top = the instance level)."""
    gas = {}
    info["gas_nodes"], info["gas_tris"] = [], []
    for g, h in enumerate(accels):
        nn, npr = C.c_uint64(0), C.c_uint64(0)
        _check(L.rtc_host_accel_info(h, C.byref(nn), C.byref(npr), None))
        nodes = np.zeros((nn.value, 80), dtype=np.uint8)
        tris = np.zeros((max(npr.value, 1), 12), dtype=np.float32)
        _check(L.rtc_host_accel_export(h, nodes.ctypes.data_as(C.c_void_p), None, tris.ctypes.data_as(C.c_void_p), None))
        gas[g] = (nodes, tris[:npr.value])
        info["gas_nodes"].append(int(nn.value)); info["gas_tris"].append(int(npr.value))
    n = len(inst_gas)
    nn, npr = C.c_uint64(0), C.c_uint64(0)
    _check(L.rtc_host_accel_info(top, C.byref(nn), C.byref(npr), None))
    nodes = np.zeros((nn.value, 80), dtype=np.uint8)
    leaves = np.zeros(max(npr.value, 1), dtype=np.uint32)
    w2o = np.zeros((n, 12), dtype=np.float32)
    _check(L.rtc_host_accel_export(top, nodes.ctypes.data_as(C.c_void_p), leaves.ctypes.data_as(C.c_void_p), None, w2o.ctypes.data_as(C.c_void_p)))
    info["tlas_nodes"] = int(nn.value)
    return {"tlas_nodes": nodes, "tlas_leaves": leaves[:npr.value], "world_to_object": w2o, "instance_gas": inst_gas, "gas": gas}


def _host_build(L, geometries, instances, accels):
    for attrs, idx in geometries:
        attrs, stride = _vertex_records(attrs)
        idx = np.ascontiguousarray(idx, dtype=np.uint32).reshape(-1, 3)
        h = C.c_void_p()
        _check(L.rtc_host_gas_build(attrs.ctypes.data_as(C.c_void_p), stride, len(attrs), idx.ctypes.data_as(C.c_void_p), len(idx), C.byref(h)))
        accels.append(h)
    transforms, inst_gas = _transforms(instances)
    n = len(inst_gas)
    handles = (C.c_void_p * max(n, 1))(*[accels[int(g)] for g in inst_gas])
    top = C.c_void_p()
    _check(L.rtc_host_ias_build(transforms.ctypes.data_as(C.c_void_p), C.cast(handles, C.c_void_p), n, C.byref(top)))
    return top, inst_gas


def host_scene_export(geometries, instances):
    """The acceleration structure rtc_gas_build(BUILD_HOST_SAH) + rtc_ias_build would upload for this scene, built WITHOUT a GPU
    (rtc_host_gas_build / rtc_host_ias_build: the same builder code fed from host arrays), in the layout of Context.scene_export.
    geometries: [(attributes structured array or [n, k] float32 with the position first, indices [m, 3] uint32)];
    instances: [(transform 12 floats, geometry index)].  Also returns the build statistics per level."""
    L = lib()
    accels, info = [], {}
    try:
        top, inst_gas = _host_build(L, geometries, instances, accels)
        accels.append(top)
        export = _host_export(L, accels[:-1], top, inst_gas, info)
    finally:
        for h in accels:
            L.rtc_host_accel_destroy(h)
    return export, info


def host_scene_refit_export(geometries, instances, new_attributes, new_transforms):
    """host_scene_export of the scene built from (geometries, instances), then refitted WITHOUT a GPU (rtc_host_gas_refit /
    rtc_host_ias_refit, the twin of rtc_gas_refit / rtc_ias_update): new_attributes[g] replaces geometry g's vertex records (None:
    unchanged, not refitted), new_transforms the 12 floats of every instance.  Topology stays the build's."""
    L = lib()
    accels, info = [], {}
    try:
        top, inst_gas = _host_build(L, geometries, instances, accels)
        accels.append(top)
        for g, attrs in enumerate(new_attributes):
            if attrs is not None:
                attrs, stride = _vertex_records(attrs)
                _check(L.rtc_host_gas_refit(accels[g], attrs.ctypes.data_as(C.c_void_p), stride))
        transforms = np.ascontiguousarray(new_transforms, dtype=np.float32).reshape(len(inst_gas), 12)
        handles = (C.c_void_p * max(len(inst_gas), 1))(*[accels[int(g)] for g in inst_gas])
        _check(L.rtc_host_ias_refit(top, transforms.ctypes.data_as(C.c_void_p), C.cast(handles, C.c_void_p), len(inst_gas)))
        export = _host_export(L, accels[:-1], top, inst_gas, info)
    finally:
        for h in accels:
            L.rtc_host_accel_destroy(h)
    return export, info


def _nan_padded(attrs):
    """vertex records as bytes [n + 1, stride] with one record appended whose position is (NaN, NaN, NaN): the vertex an
    out-of-range index of rtc_gas_build_device reads"""
    attrs, stride = _vertex_records(attrs)
    rows = attrs.view(np.uint8).reshape(len(attrs), stride)
    pad = np.zeros((1, stride), dtype=np.uint8)
    pad[0, :12] = np.full(3, np.nan, dtype=np.float32).view(np.uint8)
    return np.ascontiguousarray(np.concatenate([rows, pad])), stride


def _host_gas_build_device(L, attrs, idx):
    """the twin of rtc_gas_build_device: rtc_host_gas_build + rtc_host_gas_rebuild over the vertices with one NaN vertex appended,
    which every index >= the vertex count is replaced by"""
    n = len(np.ascontiguousarray(attrs))
    padded, stride = _nan_padded(attrs)
    idx = np.array(idx, dtype=np.uint32).reshape(-1, 3)
    idx[idx >= n] = n
    h = C.c_void_p()
    _check(L.rtc_host_gas_build(padded.ctypes.data_as(C.c_void_p), stride, n + 1, idx.ctypes.data_as(C.c_void_p), len(idx), C.byref(h)))
    rc = L.rtc_host_gas_rebuild(h, None, 0)
    if rc != 0:
        L.rtc_host_accel_destroy(h)
        _check(rc)
    return h


def host_scene_rebuild_export(geometries, instances, steps):
    """host_scene_export of the scene built from (geometries, instances), then taken WITHOUT a GPU through `steps`, in order:
    "rebuild" (rtc_host_ias_rebuild, the twin of rtc_ias_rebuild), ("gas_rebuild", g, attributes) (rtc_host_gas_rebuild, the
    twin of rtc_gas_rebuild of geometry g: attributes = its new vertex records, or None for its current positions),
    ("gas_build_device", g, attributes, indices) (the twin of rtc_gas_build_device of geometry g: its triangle set becomes
    (attributes, indices), out-of-range indices included) or (new_attributes, new_transforms), a refit as in
    host_scene_refit_export (rtc_gas_refit of the geometries given, then rtc_ias_update of every instance).  A device program of
    rtc_gas_build_device / rtc_gas_rebuild / rtc_gas_refit calls followed by rtc_ias_update is ("gas_build_device", ...) and
    ("gas_rebuild", ...) steps and then one refit step that refits the other geometries."""
    L = lib()
    accels, info = [], {}
    padded = set()              # geometries replaced by a gas_build_device step: their twin holds one NaN vertex more
    try:
        top, inst_gas = _host_build(L, geometries, instances, accels)
        accels.append(top)
        handles = (C.c_void_p * max(len(inst_gas), 1))(*[accels[int(g)] for g in inst_gas])

        def records(g, attrs):
            return _nan_padded(attrs) if g in padded else _vertex_records(attrs)

        for step in steps:
            if isinstance(step, str) and step == "rebuild":
                _check(L.rtc_host_ias_rebuild(top))
                continue
            if isinstance(step, tuple) and len(step) == 4 and step[0] == "gas_build_device":
                _, g, attrs, idx = step
                h = _host_gas_build_device(L, attrs, idx)
                L.rtc_host_accel_destroy(accels[g])
                accels[g] = h
                padded.add(g)
                handles = (C.c_void_p * max(len(inst_gas), 1))(*[accels[int(k)] for k in inst_gas])
                continue
            if isinstance(step, tuple) and len(step) == 3 and step[0] == "gas_rebuild":
                _, g, attrs = step
                if attrs is None:
                    _check(L.rtc_host_gas_rebuild(accels[g], None, 0))
                else:
                    attrs, stride = records(g, attrs)
                    _check(L.rtc_host_gas_rebuild(accels[g], attrs.ctypes.data_as(C.c_void_p), stride))
                continue
            new_attributes, new_transforms = step
            for g, attrs in enumerate(new_attributes):
                if attrs is not None:
                    attrs, stride = records(g, attrs)
                    _check(L.rtc_host_gas_refit(accels[g], attrs.ctypes.data_as(C.c_void_p), stride))
            transforms = np.ascontiguousarray(new_transforms, dtype=np.float32).reshape(len(inst_gas), 12)
            _check(L.rtc_host_ias_refit(top, transforms.ctypes.data_as(C.c_void_p), C.cast(handles, C.c_void_p), len(inst_gas)))
        export = _host_export(L, accels[:-1], top, inst_gas, info)
    finally:
        for h in accels:
            L.rtc_host_accel_destroy(h)
    return export, info


def device_count():
    n = C.c_int(0)
    rc = lib().rtc_device_count(C.byref(n))
    return n.value if rc == 0 else 0


class Context:
    """rtc_context: one GPU, one stream.  `handle` may wrap a context owned by the C++ host (owned=False)."""

    def __init__(self, device=0, handle=None):
        self.L = lib()
        self.owned = handle is None
        if handle is None:
            h = C.c_void_p()
            _check(self.L.rtc_context_create(device, C.byref(h)))
            self.h = h
        else:
            self.h = C.c_void_p(handle)

    def close(self):
        if self.h and self.owned:
            self.L.rtc_context_destroy(self.h)
        self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def stream(self):
        return self.L.rtc_context_stream(self.h)

    def synchronize(self):
        _check(self.L.rtc_synchronize(self.h))

    def malloc(self, nbytes):
        p = C.c_uint64(0)
        _check(self.L.rtc_malloc(self.h, int(nbytes), C.byref(p)))
        return p.value

    def free(self, dptr):
        _check(self.L.rtc_free(self.h, int(dptr)))

    def memset(self, dptr, value, nbytes):
        _check(self.L.rtc_memset(self.h, int(dptr), int(value), int(nbytes)))

    def upload(self, dptr, array):
        a = np.ascontiguousarray(array)
        _check(self.L.rtc_upload(self.h, int(dptr), a.ctypes.data_as(C.c_void_p), a.nbytes))
        self.synchronize()   # `a` may be a temporary

    def upload_async(self, dptr, host_ptr, nbytes):
        _check(self.L.rtc_upload(self.h, int(dptr), C.c_void_p(host_ptr), int(nbytes)))

    def download_async(self, host_ptr, dptr, nbytes):
        _check(self.L.rtc_download(self.h, C.c_void_p(host_ptr), int(dptr), int(nbytes)))

    def to_device(self, array):
        a = np.ascontiguousarray(array)
        p = self.malloc(max(a.nbytes, 16))
        self.upload(p, a)
        return p

    def download(self, dptr, dtype, count):
        out = np.zeros(count, dtype=dtype)
        _check(self.L.rtc_download(self.h, out.ctypes.data_as(C.c_void_p), int(dptr), out.nbytes))
        self.synchronize()
        return out

    def host_alloc(self, nbytes):
        p = C.c_void_p()
        _check(self.L.rtc_host_alloc(self.h, int(nbytes), C.byref(p)))
        return p.value

    def host_free(self, ptr):
        _check(self.L.rtc_host_free(self.h, C.c_void_p(ptr)))

    def gas_build(self, d_attributes, stride, num_verts, d_indices, num_tris, flags=BUILD_DEFAULT):
        g = C.c_uint32(0)
        _check(self.L.rtc_gas_build(self.h, int(d_attributes), stride, num_verts, int(d_indices), num_tris, flags, C.byref(g)))
        return g.value

    def gas_refit(self, gas, d_attributes=0):
        """rtc_gas_refit: the GAS's vertex positions changed (in place, or d_attributes = new records of the build's stride).
        Every scene instancing it must then get ias_update before it is traced."""
        _check(self.L.rtc_gas_refit(self.h, gas, int(d_attributes)))

    def gas_rebuild(self, gas, d_attributes=0):
        """rtc_gas_rebuild: a new topology for the GAS from its current vertex positions (its own buffer, updated in place, or
        d_attributes = new records of the build's stride), on the device and in place (the handle stays valid).  Asynchronous,
        except for the first rebuild of a GAS.  Every scene instancing it must then get ias_update before it is traced."""
        _check(self.L.rtc_gas_rebuild(self.h, gas, int(d_attributes)))

    def gas_create(self, capacity):
        """rtc_gas_create: a GAS without triangles (every ray misses it) with room for `capacity` triangles, whose triangle set
        gas_build_device replaces in place.  Synchronises once."""
        g = C.c_uint32(0)
        _check(self.L.rtc_gas_create(self.h, int(capacity), C.byref(g)))
        return g.value

    def gas_build_device(self, gas, d_attributes, stride, num_verts, d_indices, num_tris):
        """rtc_gas_build_device: the GAS's triangles become the num_tris index triplets at the device address d_indices over the
        num_verts vertex records (stride bytes each) at d_attributes (ints, e.g. tensor.data_ptr()), built on the device in place.
        Both buffers are read on the context stream when the build runs and become the GAS's own, as in gas_build: keep them alive.
        Never blocks the host.  Every scene instancing the GAS must then get ias_update (or ias_build_device) before it is traced."""
        _check(self.L.rtc_gas_build_device(self.h, int(gas), int(d_attributes), int(stride), int(num_verts), int(d_indices), int(num_tris)))

    def gas_rejected_triangles(self, gas):
        """rtc_gas_rejected_triangles: triangles of the last gas_build_device with an index >= num_verts (synchronises)."""
        n = C.c_uint32(0)
        _check(self.L.rtc_gas_rejected_triangles(self.h, int(gas), C.byref(n)))
        return n.value

    def ias_update(self, top, transforms, first=0):
        """rtc_ias_update: transforms [count, 12] (object -> world) of instances first .. first + count - 1 (count may be 0: only
        bring the scene up to date with refitted GAS)."""
        t = np.ascontiguousarray(transforms, dtype=np.float32).reshape(-1, 12)
        _check(self.L.rtc_ias_update(self.h, int(top), first, len(t), t.ctypes.data_as(C.c_void_p) if len(t) else None))

    def ias_update_device(self, top, d_transforms, count, first=0, stride=48):
        """rtc_ias_update_device: the object -> world matrices of instances first .. first + count - 1 are the 12 floats at the
        device address d_transforms + i * stride (an int, e.g. tensor.data_ptr() of a CUDA tensor; stride 48: dense [count, 12],
        80: OptixInstance records).  The buffer is read on the context stream when the update runs, not during the call: write
        it on `self.stream` (or order the writer with events) and keep it unchanged until the update has run."""
        _check(self.L.rtc_ias_update_device(self.h, int(top), first, count, int(d_transforms), stride))

    def ias_rebuild(self, top):
        """rtc_ias_rebuild: a new instance-level topology over the instance boxes of the last build / update, on the device and
        in place (`top` stays valid, hits do not change).  Asynchronous, except for the first rebuild of a scene."""
        _check(self.L.rtc_ias_rebuild(self.h, int(top)))

    def gas_destroy(self, gas):
        _check(self.L.rtc_gas_destroy(self.h, gas))

    def ias_build(self, instances):
        inst = np.ascontiguousarray(instances, dtype=INSTANCE_DTYPE)
        top = C.c_uint64(0)
        _check(self.L.rtc_ias_build(self.h, inst.ctypes.data_as(C.c_void_p), len(inst), C.byref(top)))
        return top.value

    def ias_create(self, capacity):
        """rtc_ias_create: an empty scene (every ray misses) with room for `capacity` instances, whose instance set
        ias_build_device replaces in place.  Synchronises once."""
        top = C.c_uint64(0)
        _check(self.L.rtc_ias_create(self.h, int(capacity), C.byref(top)))
        return top.value

    def ias_build_device(self, top, d_records, count, stride=64):
        """rtc_ias_build_device: the scene's instances become the `count` INSTANCE_DTYPE records at the device address
        d_records + i * stride (an int, e.g. tensor.data_ptr() of a CUDA uint8 tensor), and its instance level is rebuilt in place.
        The records are read on the context stream when the build runs, as in ias_update_device.  Never blocks the host."""
        _check(self.L.rtc_ias_build_device(self.h, int(top), int(d_records), int(stride), int(count)))

    def scene_rejected_instances(self, top):
        """rtc_scene_rejected_instances: records the last ias_build_device rejected (synchronises)."""
        n = C.c_uint32(0)
        _check(self.L.rtc_scene_rejected_instances(self.h, int(top), C.byref(n)))
        return n.value

    def scene_info(self, top):
        info = SceneInfo()
        _check(self.L.rtc_scene_info_get(self.h, int(top), C.byref(info)))
        return info

    def scene_destroy(self, top):
        _check(self.L.rtc_scene_destroy(self.h, int(top)))

    def set_instance_flags(self, top, first, flags):
        f = np.ascontiguousarray(flags, dtype=np.uint32)
        _check(self.L.rtc_scene_set_instance_flags(self.h, int(top), first, len(f), f.ctypes.data_as(C.c_void_p)))

    def set_instance_masks(self, top, first, masks):
        """8-bit visibility masks of instances first .. first + len(masks) - 1 (rtc_scene_set_instance_masks; 0xFF by default)."""
        m = np.ascontiguousarray(masks, dtype=np.uint8)
        _check(self.L.rtc_scene_set_instance_masks(self.h, int(top), first, len(m), m.ctypes.data_as(C.c_void_p)))

    def set_albedo_textures(self, top, enable):
        _check(self.L.rtc_scene_set_albedo_textures(self.h, int(top), 1 if enable else 0))

    def texture_create(self, rgba):
        """rgba: float32 [height, width, 4] -> handle for MaterialDefinition.textureAlbedo / textureCutout."""
        t = np.ascontiguousarray(rgba, dtype=np.float32)
        h = C.c_uint64(0)
        _check(self.L.rtc_texture_create(self.h, t.shape[1], t.shape[0], t.ctypes.data_as(C.c_void_p), C.byref(h)))
        return h.value

    def texture_destroy(self, handle):
        _check(self.L.rtc_texture_destroy(self.h, int(handle)))

    def instance_inverse(self, top, instance):
        out = np.zeros(12, dtype=np.float32)
        _check(self.L.rtc_instance_inverse(self.h, int(top), instance, out.ctypes.data_as(C.c_void_p)))
        return out

    def launch(self, sys, launch_width, launch_height, raygen, miss, iter_first, iter_count):
        _check(self.L.rtc_launch(self.h, C.byref(sys), launch_width, launch_height, raygen, miss, iter_first, iter_count))

    def launch_ex(self, sys, launch_width, launch_height, raygen, miss, iter_first, iter_count, accum_first, count_work=False):
        _check(self.L.rtc_launch_ex(self.h, C.byref(sys), launch_width, launch_height, raygen, miss, iter_first, iter_count, accum_first,
                                    1 if count_work else 0))

    def launch_counts(self):
        """(extend, connect) TraceCounts of the launches made with count_work since the last reset."""
        out = (TraceCounts * 2)()
        _check(self.L.rtc_launch_counts_get(self.h, out))
        return out[0], out[1]

    def scene_export(self, top):
        """The acceleration structure as host arrays: dict(tlas_nodes [n, 80] u1, tlas_leaves u4, world_to_object [n, 12] f4,
        instance_gas u4, gas {handle: (nodes [m, 80] u1, tris [t, 12] f4)})."""
        info = self.scene_info(top)
        nodes = np.zeros((info.numTlasNodes, 80), dtype=np.uint8)
        leaves = np.zeros(max(info.numTlasLeaves, 1), dtype=np.uint32)
        w2o = np.zeros((info.numInstances, 12), dtype=np.float32)
        inst_gas = np.zeros(max(info.numInstances, 1), dtype=np.uint32)
        _check(self.L.rtc_scene_export(self.h, int(top), nodes.ctypes.data_as(C.c_void_p), leaves.ctypes.data_as(C.c_void_p),
                                       w2o.ctypes.data_as(C.c_void_p), inst_gas.ctypes.data_as(C.c_void_p)))
        gas = {}
        for g in sorted(set(int(v) for v in inst_gas[:info.numInstances]) - {REJECTED_INSTANCE}):
            nn, nt = C.c_uint64(0), C.c_uint64(0)
            _check(self.L.rtc_gas_info(self.h, g, C.byref(nn), C.byref(nt)))
            gn = np.zeros((nn.value, 80), dtype=np.uint8)
            gt = np.zeros((max(nt.value, 1), 12), dtype=np.float32)
            _check(self.L.rtc_gas_export(self.h, g, gn.ctypes.data_as(C.c_void_p), gt.ctypes.data_as(C.c_void_p)))
            gas[g] = (gn, gt[:nt.value])
        return {"tlas_nodes": nodes, "tlas_leaves": leaves[:info.numTlasLeaves], "world_to_object": w2o,
                "instance_gas": inst_gas[:info.numInstances], "gas": gas}

    def trace_schedule(self):
        """Which schedule of the triangle tests the next launch uses and how it was chosen (rtc_trace_schedule_get): dict with
        schedule ("group" | "one_tri" | "two_tri"), decided, measured, paths_per_batch, group_ms [first, second], one_tri_ms, two_tri_ms."""
        t = TraceSchedule()
        _check(self.L.rtc_trace_schedule_get(self.h, C.byref(t)))
        return {"schedule": SCHEDULE_NAMES[t.schedule], "decided": bool(t.decided), "measured": bool(t.measured), "paths_per_batch": int(t.pathsPerBatch),
                "group_ms": [float(t.groupMs[0]), float(t.groupMs[1])], "one_tri_ms": float(t.oneTriMs), "two_tri_ms": float(t.twoTriMs)}

    def set_trace_schedule(self, schedule):
        """schedule: "group", "one_tri", "two_tri", or "auto" (measure again)."""
        _check(self.L.rtc_trace_schedule_set(self.h, {"group": 0, "one_tri": 1, "two_tri": 2, "auto": -1}[schedule]))

    def probe_gather(self, nbytes, loads_per_thread=256):
        """GB/s of random 16-byte gathers over a working set of nbytes (L2-resident when it fits)."""
        v = C.c_double(0.0)
        _check(self.L.rtc_probe_gather(self.h, nbytes, loads_per_thread, C.byref(v)))
        return v.value

    def probe_pipes(self, mode):
        """mode 0: FP32 TFLOP/s (FFMA); mode 1: 1e9 warp instructions per second (FFMA + LOP3 alternating)."""
        v = C.c_double(0.0)
        _check(self.L.rtc_probe_pipes(self.h, mode, C.byref(v)))
        return v.value

    def probe_math(self, name, x, y=None):
        """name(x, y) element-wise on the device with the shading kernels' arithmetic (include/rt_portable_math.h, IEEE / and sqrt)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        y = np.ascontiguousarray(y if y is not None else np.zeros_like(x), dtype=np.float32)
        out = np.zeros_like(x)
        _check(self.L.rtc_probe_math(self.h, MATH_FUNCTIONS.index(name), x.ctypes.data_as(C.c_void_p), y.ctypes.data_as(C.c_void_p),
                                     out.ctypes.data_as(C.c_void_p), x.size))
        return out

    def launch_counts_reset(self):
        _check(self.L.rtc_launch_counts_reset(self.h))

    def timer_start(self):
        _check(self.L.rtc_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(self.L.rtc_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def profile_enable(self, enable=True):
        _check(self.L.rtc_profile_enable(self.h, 1 if enable else 0))

    def profile(self):
        p = Profile()
        _check(self.L.rtc_profile_get(self.h, C.byref(p)))
        return {name: (p.ms[i], p.launches[i]) for i, name in enumerate(KERNEL_CLASSES)}

    # mask: the ray's visibility mask, flags: RAY_CULL_*; the _ex exports are called only when either is not the default
    def trace_closest(self, top, d_rays, n, d_hits, mask=0xFF, flags=0):
        if mask == 0xFF and flags == 0:
            _check(self.L.rtc_trace_closest(self.h, int(top), int(d_rays), int(n), int(d_hits)))
        else:
            _check(self.L.rtc_trace_closest_ex(self.h, int(top), int(d_rays), int(n), int(d_hits), int(mask), int(flags)))

    def trace_any(self, top, d_rays, n, d_occluded, mask=0xFF, flags=0):
        if mask == 0xFF and flags == 0:
            _check(self.L.rtc_trace_any(self.h, int(top), int(d_rays), int(n), int(d_occluded)))
        else:
            _check(self.L.rtc_trace_any_ex(self.h, int(top), int(d_rays), int(n), int(d_occluded), int(mask), int(flags)))

    def trace_count(self, top, d_rays, n, any_hit=False, mask=0xFF, flags=0):
        out = TraceCounts()
        if mask == 0xFF and flags == 0:
            _check(self.L.rtc_trace_count(self.h, int(top), int(d_rays), int(n), 1 if any_hit else 0, C.byref(out)))
        else:
            _check(self.L.rtc_trace_count_ex(self.h, int(top), int(d_rays), int(n), 1 if any_hit else 0, int(mask), int(flags), C.byref(out)))
        return out

    def generate_primary(self, sys, launch_width, launch_height, iteration, d_rays):
        _check(self.L.rtc_generate_primary(self.h, C.byref(sys), launch_width, launch_height, iteration, int(d_rays)))

    def composite(self, args):
        _check(self.L.rtc_composite(self.h, C.byref(args)))

    def tonemap(self, params, d_rgba, d_rgb, num_pixels):
        _check(self.L.rtc_tonemap(self.h, C.byref(params), int(d_rgba), int(d_rgb), int(num_pixels)))

    def stats(self):
        s = Stats()
        _check(self.L.rtc_stats_get(self.h, C.byref(s)))
        return s

    def stats_reset(self):
        _check(self.L.rtc_stats_reset(self.h))

    # convenience for host-resident ray sets
    def trace_closest_host(self, top, rays, mask=0xFF, flags=0):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        d_r = self.to_device(rays)
        d_h = self.malloc(max(len(rays) * HIT_DTYPE.itemsize, 16))
        try:
            self.trace_closest(top, d_r, len(rays), d_h, mask=mask, flags=flags)
            return self.download(d_h, HIT_DTYPE, len(rays))
        finally:
            self.free(d_r)
            self.free(d_h)

    def trace_any_host(self, top, rays, mask=0xFF, flags=0):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        d_r = self.to_device(rays)
        d_o = self.malloc(max(len(rays) * 4, 16))
        try:
            self.trace_any(top, d_r, len(rays), d_o, mask=mask, flags=flags)
            return self.download(d_o, np.uint32, len(rays))
        finally:
            self.free(d_r)
            self.free(d_o)
