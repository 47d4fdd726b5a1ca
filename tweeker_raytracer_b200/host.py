"""ctypes binding of librtigo3host.so -- the C++ mirror of rtigo3's Application / Raytracer / Device classes.

`App(system_file, scene_file)` does what `rtigo3 -s system -d scene` does up to the first render call: parses the two
description files, tessellates the models, creates the Raytracer of the chosen strategy and uploads the scene through
the C ABI of librtcore.  `host_only=True` stops before any device is touched (scene inspection without a GPU).
"""
import ctypes as C
import os

import numpy as np

from . import core

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "librtigo3host.so")

ATTR_DTYPE = np.dtype([("vertex", "f4", 3), ("tangent", "f4", 3), ("normal", "f4", 3), ("texcoord", "f4", 3)])
MATERIAL_DTYPE = np.dtype([("textureAlbedo", "u8"), ("textureCutout", "u8"), ("roughness", "f4", 2), ("indexBSDF", "i4"),
                           ("albedo", "f4", 3), ("absorption", "f4", 3), ("ior", "f4"), ("flags", "u4"), ("pad0", "i4")])
LIGHT_DTYPE = np.dtype([("type", "i4"), ("position", "f4", 3), ("vecU", "f4", 3), ("vecV", "f4", 3), ("normal", "f4", 3),
                        ("area", "f4"), ("emission", "f4", 3), ("unused", "f4", 3)])
CAMERA_DTYPE = np.dtype([("P", "f4", 3), ("U", "f4", 3), ("V", "f4", 3), ("W", "f4", 3)])


class Int2(C.Structure):
    _fields_ = [("x", C.c_int), ("y", C.c_int)]


class SystemData(C.Structure):
    """rt_SystemData (include/rtigo3_abi.h), 192 bytes."""
    _fields_ = [("rect", C.c_int * 4), ("topObject", C.c_uint64), ("outputBuffer", C.c_uint64), ("tileBuffer", C.c_uint64),
                ("texelBuffer", C.c_uint64), ("cameraDefinitions", C.c_uint64), ("lightDefinitions", C.c_uint64),
                ("materialDefinitions", C.c_uint64), ("envTexture", C.c_uint64), ("envCDF_U", C.c_uint64), ("envCDF_V", C.c_uint64),
                ("resolution", Int2), ("tileSize", Int2), ("tileShift", Int2), ("pathLengths", Int2),
                ("deviceCount", C.c_int), ("deviceIndex", C.c_int), ("distribution", C.c_int), ("iterationIndex", C.c_int),
                ("samplesSqrt", C.c_int), ("sceneEpsilon", C.c_float), ("clockScale", C.c_float), ("lensShader", C.c_int),
                ("numCameras", C.c_int), ("numMaterials", C.c_int), ("numLights", C.c_int), ("envWidth", C.c_uint),
                ("envHeight", C.c_uint), ("envIntegral", C.c_float), ("envRotation", C.c_float), ("_pad", C.c_int)]


class CompositorData(C.Structure):
    _fields_ = [("outputBuffer", C.c_uint64), ("tileBuffer", C.c_uint64), ("resolution", Int2), ("tileSize", Int2),
                ("tileShift", Int2), ("launchWidth", C.c_int), ("deviceCount", C.c_int), ("deviceIndex", C.c_int), ("_pad", C.c_int)]


class TonemapperParams(C.Structure):
    _fields_ = [("gamma", C.c_float), ("colorBalance", C.c_float * 3), ("whitePoint", C.c_float), ("burnHighlights", C.c_float),
                ("crushBlacks", C.c_float), ("saturation", C.c_float), ("brightness", C.c_float)]


class Info(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("resolutionX", "resolutionY", "samplesSqrt", "miss", "lightMode", "strategy", "numDevices",
                                       "numGeometries", "numInstances", "numMaterials", "numLights", "hasEnvironment")]


assert C.sizeof(SystemData) == 192 and C.sizeof(CompositorData) == 56

SYMBOLS = ["rth_last_error", "rth_app_create", "rth_app_destroy", "rth_app_info", "rth_app_geometry", "rth_app_instance",
           "rth_app_materials", "rth_app_lights", "rth_app_camera", "rth_app_system_data", "rth_app_tonemapper",
           "rth_app_environment", "rth_app_render", "rth_app_render_calls", "rth_app_set_coalesce", "rth_app_synchronize", "rth_app_frame", "rth_app_local_frame", "rth_app_restart",
           "rth_app_set_composite", "rth_app_save_system", "rth_app_set_camera", "rth_app_update_material", "rth_app_update_light_emission", "rth_app_benchmark", "rth_app_screenshot", "rth_app_tonemap", "rth_app_context", "rth_app_stats",
           "rth_app_update_material_textures", "rth_app_picture", "rth_process_group_id", "rth_app_join_group", "rth_app_group_reduce_mean", "rth_sample_range",
           "rth_app_update_instance_transform", "rth_app_rebuild_instance_level", "rth_app_update_geometry"]

_lib = None


def lib():
    global _lib
    if _lib is None:
        core.lib()   # librtcore.so first (RTLD_GLOBAL), so the host library binds to the in-tree build
        if not os.path.exists(LIB_PATH):
            raise core.RtcError("%s is missing: run `make`" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.rth_last_error.restype = C.c_char_p
        L.rth_app_create.restype = C.c_void_p
        L.rth_app_create.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        L.rth_app_destroy.argtypes = [C.c_void_p]
        L.rth_app_info.argtypes = [C.c_void_p, C.POINTER(Info)]
        L.rth_app_geometry.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint), C.POINTER(C.c_void_p), C.POINTER(C.c_uint)]
        L.rth_app_instance.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.rth_app_materials.argtypes = [C.c_void_p, C.c_void_p]
        L.rth_app_lights.argtypes = [C.c_void_p, C.c_void_p]
        L.rth_app_camera.argtypes = [C.c_void_p, C.c_void_p]
        L.rth_app_system_data.argtypes = [C.c_void_p, C.c_int, C.POINTER(SystemData)]
        L.rth_app_tonemapper.argtypes = [C.c_void_p, C.POINTER(TonemapperParams)]
        L.rth_app_environment.argtypes = [C.c_void_p, C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                          C.POINTER(C.c_void_p), C.POINTER(C.c_float)]
        L.rth_app_render.argtypes = [C.c_void_p, C.c_uint]
        L.rth_app_render.restype = C.c_uint
        L.rth_app_synchronize.argtypes = [C.c_void_p]
        L.rth_app_frame.argtypes = [C.c_void_p]
        L.rth_app_frame.restype = C.c_void_p
        L.rth_app_local_frame.argtypes = [C.c_void_p]
        L.rth_app_local_frame.restype = C.c_void_p
        L.rth_app_restart.argtypes = [C.c_void_p]
        L.rth_app_set_composite.argtypes = [C.c_void_p, C.c_int]
        L.rth_app_save_system.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int]
        L.rth_app_set_camera.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]
        L.rth_app_update_material.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_int]
        L.rth_app_update_material_textures.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rth_app_picture.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(C.c_void_p)]
        L.rth_app_update_light_emission.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.rth_app_update_instance_transform.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.rth_app_rebuild_instance_level.argtypes = [C.c_void_p]
        L.rth_app_update_geometry.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint, C.c_int]
        L.rth_app_render.argtypes = [C.c_void_p, C.c_uint]
        L.rth_app_render.restype = C.c_uint
        L.rth_app_render_calls.argtypes = [C.c_void_p, C.c_uint]
        L.rth_app_render_calls.restype = C.c_uint
        L.rth_app_set_coalesce.argtypes = [C.c_void_p, C.c_uint]
        L.rth_app_set_coalesce.restype = C.c_uint
        L.rth_app_benchmark.argtypes = [C.c_void_p]
        L.rth_app_benchmark.restype = C.c_double
        L.rth_app_screenshot.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int]
        L.rth_app_tonemap.argtypes = [C.c_void_p, C.c_void_p]
        L.rth_app_context.argtypes = [C.c_void_p, C.c_int]
        L.rth_app_context.restype = C.c_void_p
        L.rth_app_stats.argtypes = [C.c_void_p, C.POINTER(core.Stats)]
        L.rth_process_group_id.argtypes = [C.c_char_p]
        L.rth_app_join_group.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_char_p]
        L.rth_app_group_reduce_mean.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]
        L.rth_sample_range.argtypes = [C.c_uint, C.c_int, C.c_int, C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
        L.rth_sample_range.restype = None
        _lib = L
    return _lib


def process_group_id():
    """128 bytes identifying a new process group (made on rank 0; broadcast them to the other ranks out of band)."""
    buf = C.create_string_buffer(128)
    if lib().rth_process_group_id(buf) != 0:
        raise core.RtcError(lib().rth_last_error().decode())
    return buf.raw


def sample_range(samples_per_pixel, rank, world):
    """(first iteration, count) rank `rank` of `world` renders: Raytracer::samplesPerRank, no device needed."""
    first, count = C.c_uint(), C.c_uint()
    lib().rth_sample_range(samples_per_pixel, rank, world, C.byref(first), C.byref(count))
    return first.value, count.value


def _copy(ptr, dtype, count):
    if count == 0:
        return np.zeros(0, dtype=dtype)
    buf = (C.c_char * (np.dtype(dtype).itemsize * count)).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype, count=count).copy()


class App:
    """rtigo3's Application: system description + scene description -> renderer."""

    def __init__(self, system_file, scene_file, host_only=False):
        self.L = lib()
        self.h = self.L.rth_app_create(os.fsencode(system_file), os.fsencode(scene_file), 1 if host_only else 0)
        if not self.h:
            raise core.RtcError("Application failed to initialize: " + self.L.rth_last_error().decode("utf-8", "replace"))
        self.h = C.c_void_p(self.h)
        self.info = Info()
        self.L.rth_app_info(self.h, C.byref(self.info))
        self.group_rank = 0

    def close(self):
        if self.h:
            self.L.rth_app_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def group_reduce_mean(self, src, dst, count):
        """Collective: mean over the ranks of `count` floats at device address src -> dst on rank 0 (pass 0 elsewhere),
        enqueued on the render stream (ncclReduce over NVLink)."""
        if self.L.rth_app_group_reduce_mean(self.h, src, dst, count) != 0:
            raise core.RtcError(self.L.rth_last_error().decode())

    # ---- host-side scene (valid in host_only mode too)
    @property
    def resolution(self):
        return self.info.resolutionX, self.info.resolutionY

    @property
    def spp(self):
        return self.info.samplesSqrt * self.info.samplesSqrt

    def geometry(self, g):
        a, nv, i, nt = C.c_void_p(), C.c_uint(), C.c_void_p(), C.c_uint()
        if self.L.rth_app_geometry(self.h, g, C.byref(a), C.byref(nv), C.byref(i), C.byref(nt)) != 0:
            raise IndexError(g)
        return _copy(a.value, ATTR_DTYPE, nv.value), _copy(i.value, np.uint32, 3 * nt.value).reshape(-1, 3)

    def instance(self, i):
        t = np.zeros(12, dtype=np.float32)
        g, m, l = C.c_int(), C.c_int(), C.c_int()
        if self.L.rth_app_instance(self.h, i, t.ctypes.data_as(C.c_void_p), C.byref(g), C.byref(m), C.byref(l)) != 0:
            raise IndexError(i)
        return t, g.value, m.value, l.value

    def materials(self):
        out = np.zeros(self.info.numMaterials, dtype=MATERIAL_DTYPE)
        self.L.rth_app_materials(self.h, out.ctypes.data_as(C.c_void_p))
        return out

    def lights(self):
        out = np.zeros(max(self.info.numLights, 1), dtype=LIGHT_DTYPE)
        n = self.L.rth_app_lights(self.h, out.ctypes.data_as(C.c_void_p))
        return out[:n]

    def camera(self):
        out = np.zeros(1, dtype=CAMERA_DTYPE)
        self.L.rth_app_camera(self.h, out.ctypes.data_as(C.c_void_p))
        return out

    def system_data(self, device_index=0):
        s = SystemData()
        self.L.rth_app_system_data(self.h, device_index, C.byref(s))
        return s

    def tonemapper(self):
        t = TonemapperParams()
        self.L.rth_app_tonemapper(self.h, C.byref(t))
        return t

    def environment(self):
        w, h, integral = C.c_uint(), C.c_uint(), C.c_float()
        t, cu, cv = C.c_void_p(), C.c_void_p(), C.c_void_p()
        if self.L.rth_app_environment(self.h, C.byref(w), C.byref(h), C.byref(t), C.byref(cu), C.byref(cv), C.byref(integral)) != 0:
            return None
        W, H = w.value, h.value
        return (_copy(t.value, np.float32, 4 * W * H).reshape(H, W, 4), _copy(cu.value, np.float32, (W + 1) * H).reshape(H, W + 1),
                _copy(cv.value, np.float32, H + 1), integral.value)

    def save_system(self, filename=""):
        """Application::saveSystemDescription: returns the path written."""
        buf = C.create_string_buffer(1024)
        rc = self.L.rth_app_save_system(self.h, os.fsencode(filename) if filename else None, buf, 1024)
        return buf.value.decode() if rc == 0 else None

    def set_camera(self, phi, theta, fov, distance, center):
        c = np.asarray(center, dtype=np.float32)
        self.L.rth_app_set_camera(self.h, phi, theta, fov, distance, c.ctypes.data_as(C.c_void_p))

    def update_material(self, index, index_bsdf, albedo, roughness=(0.1, 0.1), absorption_color=(1, 1, 1), absorption_scale=0.0, ior=1.5, thinwalled=False):
        a, r, c = (np.asarray(v, dtype=np.float32) for v in (albedo, roughness, absorption_color))
        rc = self.L.rth_app_update_material(self.h, index, index_bsdf, a.ctypes.data_as(C.c_void_p), r.ctypes.data_as(C.c_void_p),
                                            c.ctypes.data_as(C.c_void_p), absorption_scale, ior, 1 if thinwalled else 0)
        if rc != 0:
            raise core.RtcError("updateMaterial(%d) failed" % index)

    def update_material_textures(self, index, use_albedo, use_cutout):
        """The GUI's texture check boxes of one material (switches the instances' hit records like Device::updateMaterial)."""
        if self.L.rth_app_update_material_textures(self.h, index, 1 if use_albedo else 0, 1 if use_cutout else 0) != 0:
            raise core.RtcError("updateMaterial(%d) failed" % index)

    def picture(self, name):
        """float32 [height, width, 4] texels of the "albedo" / "cutout" picture (row 0 = v 0), or None."""
        w, h, t = C.c_uint(), C.c_uint(), C.c_void_p()
        if self.L.rth_app_picture(self.h, name.encode(), C.byref(w), C.byref(h), C.byref(t)) != 0:
            return None
        return _copy(t.value, np.float32, 4 * w.value * h.value).reshape(h.value, w.value, 4)

    def update_light_emission(self, index, emission):
        e = np.asarray(emission, dtype=np.float32)
        if self.L.rth_app_update_light_emission(self.h, index, e.ctypes.data_as(C.c_void_p)) != 0:
            raise core.RtcError("updateLight(%d) failed" % index)

    def update_instance_transform(self, i, m):
        """Moves instance i (the numbering of instance(i)) to the object -> world matrix m (12 floats, row-major 3x4): the instance
        level is refitted on every device and the accumulation restarts.  Frames already requested are rendered at the old place."""
        t = np.ascontiguousarray(m, dtype=np.float32).reshape(12)
        rc = self.L.rth_app_update_instance_transform(self.h, i, t.ctypes.data_as(C.c_void_p))
        if rc != 0:
            raise core.RtcError("updateInstanceTransform(%d) failed: %s" % (i, self.L.rth_last_error().decode() if rc == -2 else "index out of range"))

    def rebuild_instance_level(self):
        """Rebuilds the instance level's topology on every device, over the instance boxes of the last update (after large motion,
        which the refit of update_instance_transform handles badly).  Hits do not change, so the accumulation goes on; iterations
        already requested are rendered first."""
        if self.L.rth_app_rebuild_instance_level(self.h) != 0:
            raise core.RtcError("rebuildInstanceLevel failed: %s" % self.L.rth_last_error().decode())

    def update_geometry(self, g, attributes, rebuild=False):
        """Deforms geometry g (the numbering of geometry(g)): `attributes` are its new vertex records (ATTR_DTYPE, the same count;
        geometry(g) returns them from then on).  Its GAS is refitted on every device, or rebuilt with rebuild=True (after large
        deformation, which a refit handles badly), the instances are updated and the accumulation restarts.  Frames already
        requested are rendered with the old mesh.  A light's definition does not follow a deformed light geometry."""
        a = np.ascontiguousarray(attributes, dtype=ATTR_DTYPE)
        rc = self.L.rth_app_update_geometry(self.h, g, a.ctypes.data_as(C.c_void_p), len(a), 1 if rebuild else 0)
        if rc != 0:
            raise core.RtcError("updateGeometry(%d) failed: %s" % (g, self.L.rth_last_error().decode() if rc == -2 else "bad index or vertex count"))

    # ---- device side
    def render(self, count=1):
        return self.L.rth_app_render(self.h, count)

    def render_calls(self, calls):
        """`calls` times the reference's `unsigned int Raytracer::render()` (one iteration per call; coalesced by the Raytracer)."""
        return self.L.rth_app_render_calls(self.h, calls)

    def set_coalesce(self, limit):
        """Raytracer::setCoalesceLimit: iterations render() may hold back before one batched launch (1 = none); returns the previous limit."""
        return self.L.rth_app_set_coalesce(self.h, limit)

    def synchronize(self):
        if self.L.rth_app_synchronize(self.h) != 0:
            raise core.RtcError(self.L.rth_last_error().decode())

    def local_frame(self):
        """This process's own running average (no collective), float32 [height, width, 4]."""
        p = self.L.rth_app_local_frame(self.h)
        if not p:
            raise core.RtcError("getLocalOutputBufferHost failed")
        w, h = self.resolution
        return _copy(p, np.float32, 4 * w * h).reshape(h, w, 4)

    def frame(self):
        """float32 [height, width, 4], row 0 = bottom of the image.  In a process group this is a collective and only rank 0
        receives the (mean) frame: the other ranks get None."""
        p = self.L.rth_app_frame(self.h)
        if not p:
            if self.group_rank > 0:
                return None
            raise core.RtcError("getOutputBufferHost failed")
        w, h = self.resolution
        return _copy(p, np.float32, 4 * w * h).reshape(h, w, 4)

    def frame_view(self):
        """Like frame() but a zero-copy view of the host staging buffer (valid until the next frame call)."""
        p = self.L.rth_app_frame(self.h)
        if not p:
            if self.group_rank > 0:
                return None
            raise core.RtcError("getOutputBufferHost failed")
        w, h = self.resolution
        buf = (C.c_float * (4 * w * h)).from_address(p)
        return np.frombuffer(buf, dtype=np.float32).reshape(h, w, 4)

    def restart(self):
        self.L.rth_app_restart(self.h)

    def join_group(self, rank, world, group_id):
        """Raytracer::joinProcessGroup: this process becomes rank `rank` of a sample-range partition over `world`
        processes (one GPU each).  Afterwards frame()/frame_view() are collectives; rank 0 receives the mean frame."""
        if len(group_id) != 128:
            raise ValueError("group_id must be the 128 bytes of process_group_id()")
        if self.L.rth_app_join_group(self.h, rank, world, group_id) != 0:
            raise core.RtcError(self.L.rth_last_error().decode())
        self.group_rank = rank

    def set_composite(self, mode):
        self.L.rth_app_set_composite(self.h, mode)

    def benchmark(self):
        return self.L.rth_app_benchmark(self.h)

    def screenshot(self, tonemap=True):
        buf = C.create_string_buffer(1024)
        rc = self.L.rth_app_screenshot(self.h, 1 if tonemap else 0, buf, 1024)
        return buf.value.decode() if rc == 0 else None

    def tonemap(self):
        w, h = self.resolution
        out = np.zeros((h, w, 3), dtype=np.uint8)
        if self.L.rth_app_tonemap(self.h, out.ctypes.data_as(C.c_void_p)) != 0:
            raise core.RtcError(self.L.rth_last_error().decode())
        return out

    def context(self, device_index=0):
        p = self.L.rth_app_context(self.h, device_index)
        if not p:
            raise core.RtcError("no such device")
        return core.Context(handle=p)

    def stats(self):
        s = core.Stats()
        if self.L.rth_app_stats(self.h, C.byref(s)) != 0:
            raise core.RtcError(self.L.rth_last_error().decode())
        return s
