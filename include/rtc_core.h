/*
 * rtc_core.h -- C ABI of the B200-native rtigo3 path-tracing core (librtcore.so).
 *
 * This is the drop-in boundary: the fourteen OptiX host entry points the reference's Device class
 * calls (SURVEY.md section 8b) are replaced by the functions below.  Plain pointers and sizes only;
 * device addresses travel as uint64_t exactly like CUdeviceptr does in the reference.  Every
 * function returns 0 on success and a non-zero code on failure; rtc_last_error() then holds
 * "ERROR: file(line): call (code) text", the CU_CHECK format of apps/rtigo3/inc/CheckMacros.h:39-79.
 * Not thread-safe by contract (the reference drives each Device from one host thread).
 *
 *   reference call site (apps/rtigo3/src/...)                         replacement
 *   ---------------------------------------------------------------  -------------------------------
 *   Device.cpp:245-316  cuCtxCreate, cuStreamCreate,                  rtc_context_create
 *                       optixDeviceContextCreate, initPipeline
 *   Device.cpp:320-358  ~Device                                       rtc_context_destroy
 *   Device.cpp:1391-1405 optixAccelComputeMemoryUsage+optixAccelBuild rtc_gas_build
 *                       (OPTIX_BUILD_INPUT_TYPE_TRIANGLES)
 *   Device.cpp:1427-1443 createInstance, :1471-1482 optixAccelBuild   rtc_ias_build
 *                       (INSTANCES), :1492-1532 createHitGroupRecords
 *   DeviceSingleGPU.cpp:164, DeviceMultiGPUZeroCopy.cpp:141,          rtc_launch
 *   DeviceMultiGPUPeerAccess.cpp:180, DeviceMultiGPULocalCopy.cpp:190
 *                       optixLaunch
 *   DeviceMultiGPULocalCopy.cpp:279-337 compositor kernel launch      rtc_composite
 *   Application.cpp:2262-2295 CPU tonemapper ("PERF Add a native CUDA rtc_tonemap
 *                       kernel doing this", :2275)
 *   Device.cpp:1503-1513, :1141-1160 hit-record (SBT header) choice   rtc_scene_set_instance_flags
 *                       per instance: plain or cutout programs
 *   Texture.cpp:640-760 Texture::create (2D image -> CUtexObject)     rtc_texture_create / rtc_texture_destroy
 *   Device.cpp synchronizeStream (cuStreamSynchronize)                rtc_synchronize
 *   cuMemAlloc / cuMemFree / cuMemcpyHtoDAsync / cuMemcpyDtoHAsync    rtc_malloc / rtc_free / rtc_upload / rtc_download
 *
 * Program selection that OptiX did through entry-function names (raygen variant by strategy,
 * Device.cpp:634-648; miss program by m_miss, :660-672; environment light callable, :705) is an
 * argument of rtc_launch.
 */
#ifndef RTC_CORE_H
#define RTC_CORE_H

#include "rtigo3_abi.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rtc_context rtc_context;

/* One instance = Device::createInstance + the per-instance hit record (GeometryInstanceData). */
typedef struct {
  float    transform[12];   /* object -> world, row-major 3x4 (OptixInstance::transform) */
  uint32_t instanceId;      /* OptixInstance::instanceId; must equal the array position */
  uint32_t gas;             /* handle returned by rtc_gas_build */
  int      materialIndex;
  int      lightIndex;      /* < 0: not a light */
} rtc_instance_desc;

/* One ray / one hit of the query interface (BASELINE config 3 and the parity hook). 32 B and 20 B. */
typedef struct { float ox, oy, oz, tmin, dx, dy, dz, tmax; } rtc_ray;
typedef struct { float t, u, v; uint32_t inst; uint32_t prim; } rtc_hit;   /* miss: t = -1, inst = prim = 0xffffffff */

typedef struct {
  uint64_t radianceRays;     /* closest-hit rays traced by extend since the last reset */
  uint64_t shadowRays;       /* any-hit rays traced by connect */
  uint64_t pathSamples;      /* paths started by generate */
  uint64_t kernelLaunches;   /* kernels of this library launched */
  double   lastTraceMs;      /* device time of the last rtc_trace_* call (CUDA events on the context stream) */
  uint64_t stackOverflows;   /* rays whose traversal stack overflowed since the library was loaded; must be 0 */
  uint64_t cutoutGraphBuilds; /* CUDA graphs of the cutout any-hit rounds captured since the last reset (one per pair) */
} rtc_stats;

/* BVH statistics of a built scene. */
typedef struct {
  uint64_t numNodes;         /* 80 B wide nodes: every distinct GAS referenced + the instance level */
  uint64_t numTris;          /* 48 B triangle records of every distinct GAS referenced */
  uint32_t numInstances;
  uint32_t numTlasNodes;
  uint32_t numGas;           /* distinct GAS referenced */
  uint32_t numTlasLeaves;    /* instance-level leaf slots (one instance id each) */
  double   gasBuildMs;       /* sum of the build times of the referenced GAS */
  double   iasBuildMs;
} rtc_scene_info;

/* Work one traversal did, summed over a ray set (the algorithmic-bytes figure of DESIGN.md):
 * wide nodes popped (80 B each), triangles tested (48 B each), instances entered (64 B each). */
typedef struct {
  uint64_t nodes, tris, instances, rays;
} rtc_trace_counts;

enum { RTC_RAYGEN_FULL_FRAME = 0,      /* __raygen__path_tracer            (raygeneration.cu:167) */
       RTC_RAYGEN_LOCAL_COPY = 1 };    /* __raygen__path_tracer_local_copy (raygeneration.cu:259) */

enum { RTC_BUILD_DEFAULT = 0,          /* GPU LBVH for large inputs, host SAH for small ones */
       RTC_BUILD_HOST_SAH = 1,
       RTC_BUILD_GPU_LBVH = 2 };

int         rtc_version(void);
const char* rtc_last_error(void);

int rtc_context_create(int deviceOrdinal, rtc_context** out);
int rtc_context_destroy(rtc_context* ctx);
int rtc_synchronize(rtc_context* ctx);
/* The context's stream as a cudaStream_t value (for callers that enqueue their own work, e.g. NCCL). */
uint64_t rtc_context_stream(rtc_context* ctx);

/* Device enumeration and peer-to-peer plumbing of the multi-GPU strategies
 * (cuDeviceGetCount / cuDeviceGetName, Raytracer.cpp:53-64; cuDeviceCanAccessPeer / cuCtxEnablePeerAccess,
 * Raytracer.cpp:127-132; cuMemcpyPeerAsync, DeviceMultiGPULocalCopy.cpp:289-295). */
int rtc_device_count(int* count);
int rtc_device_name(int deviceOrdinal, char* name, int length);
int rtc_peer_can_access(int deviceOrdinal, int peerOrdinal, int* canAccess);
int rtc_peer_enable(rtc_context* ctx, rtc_context* peer);      /* ctx may then dereference peer's allocations */
int rtc_peer_disable(rtc_context* ctx, rtc_context* peer);
/* dst (on dstCtx) <- src (on srcCtx): waits for srcCtx's stream, then copies asynchronously on dstCtx's stream. */
int rtc_memcpy_peer(rtc_context* dstCtx, uint64_t dst, rtc_context* srcCtx, uint64_t src, uint64_t bytes);

int rtc_malloc(rtc_context* ctx, uint64_t bytes, uint64_t* dptr);
int rtc_free(rtc_context* ctx, uint64_t dptr);
int rtc_upload(rtc_context* ctx, uint64_t dst, const void* src, uint64_t bytes);     /* async on the context stream */
int rtc_download(rtc_context* ctx, void* dst, uint64_t src, uint64_t bytes);         /* async on the context stream */
int rtc_memset(rtc_context* ctx, uint64_t dst, int value, uint64_t bytes);
int rtc_host_alloc(rtc_context* ctx, uint64_t bytes, void** ptr);                    /* pinned, portable, device-mapped (UVA: same pointer on every GPU) */
int rtc_host_free(rtc_context* ctx, void* ptr);

/* attributes: device pointer to vertex records, position = 3 floats at offset 0, strideBytes apart
 * (48 for TriangleAttributes); indices: device pointer to numTris uint32 triplets.
 * Inactive inputs (every build, refit, rebuild and update below; DESIGN.md section 3): a triangle with a vertex coordinate that
 * is NaN, +-inf or beyond B = 2^126 in magnitude, and an instance whose transform has such an entry or whose transformed vertices
 * reach beyond B, are never hit and bound nothing; every other triangle and instance gives exactly the brute-force hits. */
int rtc_gas_build(rtc_context* ctx, uint64_t attributes, uint32_t strideBytes, uint32_t numVerts,
                  uint64_t indices, uint32_t numTris, uint32_t buildFlags, uint32_t* gas);
/* Builds the instance level, the per-instance tables and returns SystemData::topObject. */
int rtc_ias_build(rtc_context* ctx, const rtc_instance_desc* instances, uint32_t numInstances, uint64_t* topObject);
/*
 * In-place updates (optixAccelBuild with OPTIX_BUILD_OPERATION_UPDATE).  All are asynchronous on the context stream and do not
 * synchronise the host, except for a one-time allocation of refit scratch on a GAS's first refit: work enqueued before
 * sees the old structure, work enqueued after sees the new one.  Topology is never changed -- vertex and triangle counts,
 * indices, instance count, the GAS of an instance and materials stay as built; changing them is a rebuild.  Node topology and
 * leaf order stay as built, so traversal cost grows with the size of the deformation (DESIGN.md section 3, "Refit").
 *
 * rtc_gas_refit: refit a GAS after its vertex POSITIONS changed; numVerts, numTris, indices and stride must be the build's.
 *   attributes: the new vertex records (same stride as the build), or 0 = the build's buffer, updated in place by the caller.
 *   Only boxes and triangle records are rewritten.  Every scene that instances this GAS must then be brought up to date with
 *   rtc_ias_update before it is traced: until then rtc_launch, rtc_launch_ex and rtc_trace_* on such a scene fail.
 * rtc_ias_update: transforms of instances first .. first+count-1 are replaced (count x 12 floats, object->world, row-major; may
 *   be null when count == 0), world->object matrices and shading tables follow, the bounds of every instance whose transform
 *   changed or whose GAS was refitted since the last build / update are recomputed, and the instance level is refitted.
 *   `transforms` is host memory, pageable or page-locked (rtc_host_alloc, registered or managed memory), and may be reused on
 *   return: the call has read it by then.  Device memory is refused: that is rtc_ias_update_device.
 * rtc_ias_update_device: rtc_ias_update with the matrices in memory the context's GPU can read (its device memory, or mapped
 *   host memory) -- the counterpart of optixAccelBuild reading OptixInstance records from device memory.  The matrix of instance
 *   first + i is the 12 floats (object->world, row-major 3x4) at transforms + i * strideBytes; strideBytes is a multiple of 4
 *   and at least 48: 48 for a dense [count, 12] float array, 80 for an OptixInstance array (its transform[12] is at offset 0,
 *   the other bytes are ignored).  `transforms` must be 4-byte aligned; it may be 0 when count == 0.
 *   The buffer is read ON THE CONTEXT STREAM, when the stream reaches the update, not during the call -- the opposite of
 *   rtc_ias_update.  The caller must have finished writing it by then and must not overwrite it until the update has run: write
 *   it on the same stream (rtc_context_stream) or order the writer and later writers with events.
 *   The results are those of rtc_ias_update with the same matrices, byte for byte; everything else is as there (refitted GAS,
 *   count == 0, refusals).  Never synchronises the host and allocates only from the stream-ordered pool.
 */
int rtc_gas_refit(rtc_context* ctx, uint32_t gas, uint64_t attributes);
int rtc_ias_update(rtc_context* ctx, uint64_t topObject, uint32_t first, uint32_t count, const float* transforms);
int rtc_ias_update_device(rtc_context* ctx, uint64_t topObject, uint32_t first, uint32_t count, uint64_t transforms, uint32_t strideBytes);
/*
 * rtc_ias_rebuild: a new TOPOLOGY for the scene's instance level, built on the device (LBVH, one instance per leaf slot) over the
 *   instance boxes of the last rtc_ias_build / rtc_ias_update, written in place: topObject, the tables, instance flags and every
 *   SystemData that holds topObject stay valid, and hits are bit-identical (closest hit does not depend on the node order, any
 *   hit is a boolean); only the nodes, the leaf order and the traversal cost change.  Use it after large motion, which a refit
 *   handles badly (DESIGN.md section 3): animate with rtc_ias_update, then rtc_ias_rebuild.  Asynchronous on the context stream,
 *   like the refits; the first rebuild of a scene allocates its build arrays and a node array of the worst-case size and
 *   synchronises once.  Two rebuilds of the same boxes give the same bytes (rtc_host_ias_rebuild reproduces them).  Refused, as
 *   launches are, for a scene with a GAS refitted since its last update and for a scene that instances a destroyed GAS.
 *   After a rebuild the instance level's node count lives on the device: rtc_scene_info_get and rtc_scene_export read it back
 *   and therefore synchronise the stream.
 */
int rtc_ias_rebuild(rtc_context* ctx, uint64_t topObject);
/*
 * rtc_gas_rebuild: a new TOPOLOGY for a GAS, built on the device (LBVH, one triangle per leaf slot) from its current vertex
 *   positions and written in place: the handle stays valid.  Use it after large deformation, which rtc_gas_refit handles badly
 *   (DESIGN.md section 3).  attributes: as in rtc_gas_refit (the new vertex records, same stride as the build, which replace the
 *   GAS's buffer; or 0 = its own buffer, updated in place by the caller); numVerts, numTris, indices and stride stay as built.
 *   Asynchronous on the context stream: the vertices are read when the stream reaches the rebuild, work enqueued before sees the
 *   old structure and work enqueued after the new one.  The first rebuild of a GAS allocates its build arrays and a node array of
 *   the worst-case size and synchronises once; later rebuilds never block the host.  Like a refit it makes every scene that
 *   instances the GAS stale until rtc_ias_update.  Two rebuilds of the same positions give the same bytes, whichever builder
 *   made the GAS and whatever refits or rebuilds came before (rtc_host_gas_rebuild reproduces them).  A GAS without triangles
 *   is left as it is.  After a rebuild the node count lives on the device: rtc_gas_info, rtc_gas_export and rtc_scene_info_get
 *   read it back and therefore synchronise the stream.  Detect the feature by this export (rtc_version is unchanged).
 */
int rtc_gas_rebuild(rtc_context* ctx, uint32_t gas, uint64_t attributes);
/*
 * Geometry whose triangle set lives on the device (optixAccelBuild over OPTIX_BUILD_INPUT_TYPE_TRIANGLES with inputs in device
 * memory, called every frame into the same output buffers): meshes whose triangle count or connectivity changes from frame to
 * frame -- isosurfaces, fracture, level of detail, streamed terrain tiles -- without a host stall and without a new handle.
 *
 * rtc_gas_create: a GAS with room for `capacity` triangles (0 is treated as 1) and no triangle yet (the nodes and bounds
 *   rtc_gas_build writes for numTris == 0: every ray misses it).  Allocates everything its builds will use -- a node array for
 *   capacity + 16 nodes, 48 B of triangle records per triangle, refit scratch, the LBVH arrays and the collapse graph -- and
 *   synchronises once.  The handle works wherever one of rtc_gas_build does (rtc_ias_build, records of rtc_ias_build_device,
 *   rtc_gas_refit, rtc_gas_rebuild, rtc_gas_info, rtc_gas_export, rtc_gas_destroy).
 * rtc_gas_build_device: replaces the GAS's whole triangle set with numTris <= capacity triangles (uint3 index triplets at
 *   `indices`) over numVerts vertex records of strideBytes bytes at `attributes` (the position is their first 12 bytes), and
 *   builds a new LBVH over them in place: same handle, same node array.
 *   - Stream order: vertices and indices are read ON THE CONTEXT STREAM, when the stream reaches the call, as rtc_ias_build_device
 *     reads its records.  Never synchronises the host; allocates only from the stream-ordered pool.  Work enqueued before sees the
 *     old triangles, work enqueued after sees the new ones.
 *   - Ownership: `attributes` and `indices` become the GAS's buffers, as if rtc_gas_build had been given them: shading reads
 *     them, rtc_gas_refit(gas, 0) and rtc_gas_rebuild(gas, 0) work on them.  Keep them alive and unchanged (apart from refits)
 *     until the next build or rtc_gas_destroy.  numVerts and numTris may differ from call to call.
 *   - Bad indices: an index >= numVerts reads the vertex (NaN, NaN, NaN), so its triangle is inactive (never hit, bounds
 *     nothing, NaN in v0 of its record), and is counted for rtc_gas_rejected_triangles.  No index makes a kernel read outside
 *     [attributes, attributes + numVerts * strideBytes).
 *   - Result bytes: nodes and triangle records equal rtc_host_gas_build + rtc_host_gas_rebuild(accel, NULL) over the same
 *     triangles, with every out-of-range index replaced by the index of one NaN vertex appended to the vertices.  Two builds of
 *     the same input give the same bytes, whatever the GAS held before.
 *   - Staleness: as after rtc_gas_rebuild, every scene that instances the GAS is stale until rtc_ias_update or
 *     rtc_ias_build_device runs on it; launches and rtc_trace_* on it are refused until then.
 *   - Refused (synchronously, nothing enqueued, the GAS unchanged): an unknown or destroyed handle, a GAS of rtc_gas_build,
 *     numTris > capacity, a stride below 12 or not a multiple of 4, `attributes` or `indices` not 4-byte aligned, null buffers
 *     with numTris > 0.
 *   rtc_gas_info, rtc_gas_export and rtc_scene_info_get report the current triangle count.
 * rtc_gas_rejected_triangles: the triangles with an out-of-range index in the last build of the GAS (0 for a GAS of
 *   rtc_gas_build, which refuses such indices).  Synchronises.
 * Detect the feature by these exports (rtc_version is unchanged).
 */
int rtc_gas_create(rtc_context* ctx, uint32_t capacity, uint32_t* gas);
int rtc_gas_build_device(rtc_context* ctx, uint32_t gas, uint64_t attributes, uint32_t strideBytes, uint32_t numVerts,
                         uint64_t indices, uint32_t numTris);
int rtc_gas_rejected_triangles(rtc_context* ctx, uint32_t gas, uint32_t* count);
/*
 * Scenes whose instance set lives on the device (optixAccelBuild over OPTIX_BUILD_INPUT_TYPE_INSTANCES, called every frame into
 * the same buffers): spawn and despawn objects, swap an instance's GAS (level of detail, a broken variant) or reassign its
 * material without a host stall and without a new topObject.
 *
 * rtc_ias_create: an empty scene with room for `capacity` instances (0 instances: every ray misses).  Allocates everything its
 *   builds will use -- tables, boxes, a node array for the capacity, the LBVH arrays and the collapse graph -- and synchronises
 *   once.  topObject stays valid until rtc_scene_destroy.
 * rtc_ias_build_device: replaces the scene's whole instance set with numInstances <= capacity rtc_instance_desc records at
 *   instances + i * strideBytes (device memory or mapped host memory; strideBytes >= 64 and a multiple of 4; 4-byte aligned;
 *   `instances` and strideBytes may be 0 when numInstances == 0), and builds a new LBVH instance level over them in place.
 *   - Stream order: the records are read ON THE CONTEXT STREAM, as rtc_ias_update_device reads its matrices: written before the
 *     stream reaches the call and left unchanged until it has run.  Never synchronises the host; allocates only from the
 *     stream-ordered pool.  Work enqueued before sees the old instance set, work enqueued after sees the new one.
 *   - What stays valid: topObject, the SceneDesc it points at, instance flags (they belong to positions and persist across
 *     builds) and every SystemData that holds the scene.  The cutout any-hit graph is not captured again.
 *   - Per record: transform, gas, materialIndex and lightIndex come from device memory; the shading table's indices and
 *     attributes come from the GAS.
 *   - Rejected records: a record whose gas is out of range or destroyed, or whose instanceId differs from its position, becomes
 *     an empty instance -- the box and root node of a GAS without triangles, so nothing of it is ever hit or shaded -- and is
 *     counted for rtc_scene_rejected_instances.  No record can make the traversal read freed or foreign memory.
 *   - Result bytes: nodes, leaves and world->object matrices equal rtc_host_ias_build + rtc_host_ias_rebuild (and rtc_ias_build
 *     + rtc_ias_rebuild) of the same records; hits and frames equal those of rtc_ias_build of the same records, bit for bit.
 *   - Refused (synchronously, nothing enqueued): an unknown topObject, a scene of rtc_ias_build, numInstances > capacity, a bad
 *     stride or alignment, null records with numInstances > 0.
 *   rtc_ias_update, rtc_ias_update_device, rtc_ias_rebuild, rtc_scene_set_instance_flags (range checked against the capacity),
 *   rtc_scene_info_get, rtc_scene_export and rtc_instance_inverse accept created scenes, over the current instance count.
 *   rtc_scene_info_get and rtc_scene_export read the device's instance -> GAS map (rejected records: 0xffffffff) and node count
 *   back, and so synchronise.
 *   Staleness: the host does not know which GAS a created scene references, so it is stale after a refit or rebuild of ANY GAS of
 *   the context until rtc_ias_update (count 0 is enough) or rtc_ias_build_device runs on it -- conservative: the update then
 *   recomputes exactly the instances whose GAS changed, selected on the device.  rtc_gas_destroy of a GAS the last build
 *   references makes the scene unusable ("a GAS of this scene was destroyed") until the next rtc_ias_build_device.
 * rtc_scene_rejected_instances: the records the last rtc_ias_build_device of the scene rejected.  Synchronises.
 * Detect the feature by these exports (rtc_version is unchanged).
 */
int rtc_ias_create(rtc_context* ctx, uint32_t capacity, uint64_t* topObject);
int rtc_ias_build_device(rtc_context* ctx, uint64_t topObject, uint64_t instances, uint32_t strideBytes, uint32_t numInstances);
int rtc_scene_rejected_instances(rtc_context* ctx, uint64_t topObject, uint32_t* count);
int rtc_scene_info_get(rtc_context* ctx, uint64_t topObject, rtc_scene_info* info);
/* Frees one scene (the instance level and its tables; GAS stay alive until rtc_gas_destroy / context destroy). */
int rtc_scene_destroy(rtc_context* ctx, uint64_t topObject);
/* A scene that instances a destroyed GAS can only be destroyed: launches, rtc_trace_* and rtc_ias_update on it fail. */
int rtc_gas_destroy(rtc_context* ctx, uint32_t gas);
/*
 * Which hit records an instance uses.  The reference writes the cutout program group (__anyhit__radiance_cutout,
 * __anyhit__shadow_cutout; shaders/anyhit.cu:46-80, :94-132) into the two SBT records of every instance whose material
 * has a cutout texture (src/Device.cpp:1503-1513) and rewrites those headers when the GUI toggles it (:1141-1160).
 * flags[i] applies to instance first + i.  Stream-ordered on the context stream; every instance starts at 0.
 * While at least one instance carries RTC_INSTANCE_CUTOUT, launches process the candidate intersections of a ray in the
 * canonical order (t, instance, primitive) -- closest candidate first, an ignored candidate is followed by the next one --
 * which is the order this library DEFINES for the reference's order-dependent stochastic alpha test.
 */
#define RTC_INSTANCE_CUTOUT 1u
int rtc_scene_set_instance_flags(rtc_context* ctx, uint64_t topObject, uint32_t first, uint32_t count, const uint32_t* flags);
/* Tells the core that MaterialDefinition.textureAlbedo may be non-zero for this scene (closesthit.cu:233-240); selects
 * the shading kernels that interpolate texture coordinates.  Off by default, like the reference's GUI toggle. */
int rtc_scene_set_albedo_textures(rtc_context* ctx, uint64_t topObject, int enable);
/*
 * Material textures.  Replaces Texture::create for 2D images (src/Texture.cpp:640-760, cuTexObjectCreate with wrap/wrap
 * addressing, linear filter, normalised coordinates): rgba = width*height RGBA32F texels, row 0 first.  The returned
 * handle goes into MaterialDefinition.textureAlbedo / textureCutout (0 = no texture).  The fetch is a software bilinear
 * filter (wrap in u and v, texel centres at (i+0.5)/size) so that it is reproducible on a CPU.
 */
int rtc_texture_create(rtc_context* ctx, uint32_t width, uint32_t height, const float* rgba, uint64_t* handle);
int rtc_texture_destroy(rtc_context* ctx, uint64_t handle);
/*
 * Export of the acceleration structure to host memory, for tools and for the test oracle, which traverses the IDENTICAL wide BVH
 * to reproduce the work counters of rtc_trace_count / rtc_launch_counts_get (SURVEY.md section 8d).  Synchronous.
 *   rtc_scene_export: tlasNodes = numTlasNodes x 80 B wide nodes, tlasLeaves = numTlasLeaves instance ids,
 *                     worldToObject = numInstances x 12 floats, instanceGas = numInstances GAS handles; any pointer may be null.
 *   rtc_gas_info / rtc_gas_export: nodes = numNodes x 80 B, tris = numTris x 12 floats in leaf order
 *                     (v0.xyz, primitive id bits, v1.xyz, 0, v2.xyz, 0).
 * Node layout: csrc/rtc_internal.h Node8.
 */
int rtc_scene_export(rtc_context* ctx, uint64_t topObject, void* tlasNodes, uint32_t* tlasLeaves, float* worldToObject, uint32_t* instanceGas);
int rtc_gas_info(rtc_context* ctx, uint32_t gas, uint64_t* numNodes, uint64_t* numTris);
int rtc_gas_export(rtc_context* ctx, uint32_t gas, void* nodes, float* tris);
/* Copies out the 3x4 world->object matrix of one instance.  The matrices live on the device (the builds and updates compute them there), so
 * this reads one row set back and synchronises the context stream. */
int rtc_instance_inverse(rtc_context* ctx, uint64_t topObject, uint32_t instance, float out[12]);

/*
 * Host-only twin of rtc_gas_build(RTC_BUILD_HOST_SAH) + rtc_ias_build: the same builder code (csrc/accel_host.cpp,
 * csrc/bvh_build_host.cpp) fed from HOST arrays, returning the arrays the two functions would upload -- no CUDA call, no
 * context.  For tools (tests/tools/bvh_quality.py) and for the CPU tests of the builder: the test oracle traverses the result in the
 * kernels' order of operations, so node / triangle / instance counts per ray of a B200 run are known before it happens.
 *   geometry level: nodes = numNodes x 80 B, primOrder = numPrims triangle indices in leaf order, tris = numPrims x 12 floats
 *   instance level: nodes, primOrder = the instance-level leaf slots (instance ids), worldToObject = numInstances x 12 floats
 * transforms: 12 floats per instance (object -> world, rtc_instance_desc::transform); geometry[i]: the accel of instance i's mesh.
 * Any pointer of rtc_host_accel_export may be null.
 */
typedef struct rtc_host_accel rtc_host_accel;
int  rtc_host_gas_build(const void* attributes, uint32_t strideBytes, uint32_t numVerts, const uint32_t* indices, uint32_t numTris,
                        rtc_host_accel** out);
int  rtc_host_ias_build(const float* transforms, const rtc_host_accel* const* geometry, uint32_t numInstances, rtc_host_accel** out);
/* Host-only twin of rtc_gas_refit / rtc_ias_update, on what rtc_host_gas_build / rtc_host_ias_build returned: the same node
 * routine (csrc/bvh_rules.h), visiting the nodes in descending index order (children always sit above their parent).
 * rtc_host_gas_refit: attributes = the new vertex records, strideBytes = the build's.
 * rtc_host_ias_refit: every instance's transform and geometry (numInstances = the build's; geometry[i] may have been refitted). */
int  rtc_host_gas_refit(rtc_host_accel* accel, const void* attributes, uint32_t strideBytes);
int  rtc_host_ias_refit(rtc_host_accel* accel, const float* transforms, const rtc_host_accel* const* geometry, uint32_t numInstances);
/* Host-only twin of rtc_ias_rebuild, on an instance-level accel (after rtc_host_ias_build or rtc_host_ias_refit): the same LBVH
 * over the same boxes in the same float arithmetic, so nodes and leaves equal the device rebuild's byte for byte. */
int  rtc_host_ias_rebuild(rtc_host_accel* accel);
/* Host-only twin of rtc_gas_rebuild, on a geometry accel from rtc_host_gas_build: the same LBVH over the same triangles in the
 * same float arithmetic, so nodes and triangle records equal the device rebuild's byte for byte.  attributes: the new vertex
 * records (strideBytes = the build's), or null to rebuild over the positions of the last build, refit or rebuild. */
int  rtc_host_gas_rebuild(rtc_host_accel* accel, const void* attributes, uint32_t strideBytes);
int  rtc_host_accel_info(const rtc_host_accel* accel, uint64_t* numNodes, uint64_t* numPrims, float bounds[6]);
int  rtc_host_accel_export(const rtc_host_accel* accel, void* nodes, uint32_t* primOrder, float* tris, float* worldToObject);
void rtc_host_accel_destroy(rtc_host_accel* accel);

/*
 * One optixLaunch-equivalent per iteration in [iterationFirst, iterationFirst + iterationCount):
 * sys is the HOST copy of SystemData (pointers inside are device pointers owned by the caller);
 * sys->iterationIndex is ignored in favour of the range.  raygen = RTC_RAYGEN_*, miss = RT_MISS_*.
 * Asynchronous on the context stream.
 */
int rtc_launch(rtc_context* ctx, const rt_SystemData* sys, uint32_t launchWidth, uint32_t launchHeight,
               int raygen, int miss, int iterationFirst, int iterationCount);

/* rtc_launch with the accumulation index decoupled from the seed index: iteration b of the call draws its seeds from
 * iterationFirst + b and is blended into the frame as sample number accumulationFirst + b (running average weight
 * 1 / (accumulationFirst + b + 1)).  rtc_launch == rtc_launch_ex with accumulationFirst = iterationFirst.  Used by the
 * sample-range partition across GPUs (each GPU averages its own disjoint iteration indices from zero).
 * countWork != 0 additionally accumulates the traversal work counters read by rtc_launch_counts_get (slower; for
 * the algorithmic-bytes figure only, never for a timed run). */
int rtc_launch_ex(rtc_context* ctx, const rt_SystemData* sys, uint32_t launchWidth, uint32_t launchHeight,
                  int raygen, int miss, int iterationFirst, int iterationCount, int accumulationFirst, int countWork);
/*
 * Schedule of the triangle tests in the traversal kernels (csrc/trace.cuh Traversal::step).  Three are compiled; hits, frames and
 * work counters are bit-identical under all of them, only the timing inside a warp differs:
 *   RTC_SCHEDULE_GROUP    a step tests every triangle of the leaves its node visit found (what rounds 1 and 2 measured);
 *   RTC_SCHEDULE_ONE_TRI  a step tests at most one triangle, and a lane with more pending skips its node visit;
 *   RTC_SCHEDULE_TWO_TRI  the same with at most two (one leaf of the host builder).
 * By default every context MEASURES: of its first rtc_launch batches of >= 1 Mi paths one is a warm-up and the next four run
 * group / one triangle / two triangles / group between events; a capped schedule serves the later launches only if it beats
 * the faster group batch by 3 % (the faster capped one if both do).  The environment variable
 * RTC_TRACE_SCHEDULE=group|onetri|twotri, or rtc_trace_schedule_set, fixes the schedule; rtc_trace_schedule_set(ctx, -1) measures
 * again.  rtc_trace_schedule_get reports the schedule in use and the four batch times (it takes a pending decision first,
 * which waits for the last timed batch).
 */
enum { RTC_SCHEDULE_GROUP = 0, RTC_SCHEDULE_ONE_TRI = 1, RTC_SCHEDULE_TWO_TRI = 2 };
typedef struct {
  int      schedule;         /* RTC_SCHEDULE_* the next launch uses */
  int      decided;          /* 0 while the measurement is still running */
  int      measured;         /* 1 when the decision came from the timed batches (not from the environment / _set) */
  uint64_t pathsPerBatch;    /* size of the timed batches */
  float    groupMs[2];       /* device time of the first and the second RTC_SCHEDULE_GROUP batch */
  float    oneTriMs;         /* device time of the RTC_SCHEDULE_ONE_TRI batch */
  float    twoTriMs;         /* device time of the RTC_SCHEDULE_TWO_TRI batch */
} rtc_trace_schedule;
int rtc_trace_schedule_get(rtc_context* ctx, rtc_trace_schedule* out);
int rtc_trace_schedule_set(rtc_context* ctx, int schedule);

/* Work counters of the launches made with countWork since the last reset: [0] extend (radiance rays), [1] connect (shadow rays). */
int rtc_launch_counts_get(rtc_context* ctx, rtc_trace_counts out[2]);
int rtc_launch_counts_reset(rtc_context* ctx);

/* Device-side timing on the context stream (CUDA events). */
int rtc_timer_start(rtc_context* ctx);
int rtc_timer_stop(rtc_context* ctx, float* milliseconds);     /* synchronises the stream */
/* Per-kernel-class timing: while enabled every launch of the wavefront is bracketed by an event pair. */
enum { RTC_KERNEL_GENERATE = 0, RTC_KERNEL_EXTEND = 1, RTC_KERNEL_SHADE = 2, RTC_KERNEL_CONNECT = 3,
       RTC_KERNEL_ACCUMULATE = 4, RTC_KERNEL_OTHER = 5, RTC_NUM_KERNEL_CLASSES = 6 };
typedef struct {
  double   ms[RTC_NUM_KERNEL_CLASSES];        /* summed device time per class */
  uint64_t launches[RTC_NUM_KERNEL_CLASSES];
} rtc_profile;
int rtc_profile_enable(rtc_context* ctx, int enable);          /* enabling resets the accumulated profile */
int rtc_profile_get(rtc_context* ctx, rtc_profile* out);        /* synchronises the stream */

/* Ray queries against a built scene; rays/hits/occluded are device pointers.  occluded: one uint32 per ray.
 * The same queries from the caller's own CUDA kernels, one ray per call with its own mask and flags: include/rtc_device.cuh
 * (rtc_device_trace_closest / rtc_device_trace_any on topObject), whose comment is their contract. */
int rtc_trace_closest(rtc_context* ctx, uint64_t topObject, uint64_t rays, uint64_t numRays, uint64_t hits);
int rtc_trace_any(rtc_context* ctx, uint64_t topObject, uint64_t rays, uint64_t numRays, uint64_t occluded);
/* Same traversal as rtc_trace_closest (anyHit = 0) / rtc_trace_any (anyHit = 1) with work counters; synchronous. */
int rtc_trace_count(rtc_context* ctx, uint64_t topObject, uint64_t rays, uint64_t numRays, int anyHit, rtc_trace_counts* out);
/*
 * Visibility masks and face culling of the ray queries (OptixInstance::visibilityMask, the visibilityMask argument of optixTrace,
 * OPTIX_RAY_FLAG_CULL_{BACK,FRONT}_FACING_TRIANGLES).
 *   - Instance masks are 8 bits; every instance starts at 0xFF.  rtc_scene_set_instance_masks sets masks[i] on instance
 *     first + i, stream-ordered on the context stream like rtc_scene_set_instance_flags; `masks` may be reused on return.  In a
 *     scene of rtc_ias_create the masks belong to positions up to the capacity and persist across rtc_ias_build_device, like
 *     flags.  rtc_ias_update, rtc_ias_update_device and rtc_ias_rebuild never touch them.
 *   - Mask test: a ray of mask m never enters an instance of mask k with (k & m) == 0, and nothing of that instance is hit.  In
 *     the counters of rtc_trace_count_ex such an instance is not entered; the instance-level node visits that found it count.
 *   - Facing is decided in the instance's object space: a hit is front-facing when dot((v1 - v0) x (v2 - v0), d) < 0, d the
 *     object-space ray direction.  A mirrored instance (transform of negative determinant) therefore culls the opposite
 *     world-space side.  A culled candidate is not a hit: the closest-hit query goes on to the next candidate, the any-hit query
 *     does not stop.  Both flags together cull every triangle.
 *   - rtc_trace_closest, rtc_trace_any and rtc_trace_count are the _ex calls with (0xFF, 0).
 *   - Refused (synchronously, nothing enqueued): visibilityMask > 0xFF, unknown rayFlags bits, and what the plain calls refuse
 *     (an unknown or unusable scene, more than 2^32 rays); for the setter an unknown scene, first + count out of range, or null
 *     masks with count > 0.
 *   - Rendering does not evaluate masks: while an instance mask of a scene is not 0xFF, rtc_launch / rtc_launch_ex on that scene
 *     fail, and they work again once the masks are 0xFF.
 * Detect the feature by these exports (rtc_version is unchanged).
 */
#define RTC_RAY_CULL_BACK_FACING   1u
#define RTC_RAY_CULL_FRONT_FACING  2u
int rtc_scene_set_instance_masks(rtc_context* ctx, uint64_t topObject, uint32_t first, uint32_t count, const uint8_t* masks);
int rtc_trace_closest_ex(rtc_context* ctx, uint64_t topObject, uint64_t rays, uint64_t numRays, uint64_t hits,
                         uint32_t visibilityMask, uint32_t rayFlags);
int rtc_trace_any_ex(rtc_context* ctx, uint64_t topObject, uint64_t rays, uint64_t numRays, uint64_t occluded,
                     uint32_t visibilityMask, uint32_t rayFlags);
int rtc_trace_count_ex(rtc_context* ctx, uint64_t topObject, uint64_t rays, uint64_t numRays, int anyHit,
                       uint32_t visibilityMask, uint32_t rayFlags, rtc_trace_counts* out);
/* Primary rays of one iteration, one rtc_ray per launch index (skipped indices get tmax = -1). */
int rtc_generate_primary(rtc_context* ctx, const rt_SystemData* sys, uint32_t launchWidth, uint32_t launchHeight,
                         int iteration, uint64_t rays);

int rtc_composite(rtc_context* ctx, const rt_CompositorData* args);
int rtc_tonemap(rtc_context* ctx, const rt_TonemapperParams* params, uint64_t rgba, uint64_t rgb8, uint64_t numPixels);

/*
 * Roofline denominators measured on this GPU (csrc/probes.cu), for the fractions bench.py reports next to the HBM one
 * (SURVEY.md section 8d: L2 and FP32 peaks are not in MEASURED_PEAKS.json).  Synchronous.
 *   rtc_probe_gather: random 16-byte gathers (the access pattern of node / triangle fetches) over a working set of
 *                     `bytes` (rounded down to a power of two): L2-resident below the L2 size, HBM gathers above it.
 *   rtc_probe_pipes : mode 0 -> FP32 TFLOP/s of independent FFMA chains; mode 1 -> 1e9 warp instructions issued per
 *                     second with FFMA and LOP3 alternating (fma pipe + alu pipe), the issue-slot peak.
 */
int rtc_probe_gather(rtc_context* ctx, uint64_t bytes, uint32_t loadsPerThread, double* gigabytesPerSecond);
int rtc_probe_pipes(rtc_context* ctx, int mode, double* rate);

/*
 * Test hook: out[i] = fn(x[i], y[i]) evaluated on the device by the shading translation unit, i.e. with the arithmetic the
 * closest-hit / BSDF / light / miss replacements are compiled with (pinned transcendentals of include/rt_portable_math.h,
 * IEEE division and square root, no FMA contraction).  The bits must equal the same header compiled for the host -- the
 * definition the "bit-identical to the CPU oracle" parity claim rests on.  x, y, out: HOST arrays of n floats.  Synchronous.
 */
enum rtc_math_fn { RTC_MATH_SIN = 0, RTC_MATH_COS, RTC_MATH_ATAN, RTC_MATH_ATAN2, RTC_MATH_ACOS, RTC_MATH_EXP, RTC_MATH_LOG,
                   RTC_MATH_POW, RTC_MATH_DIV, RTC_MATH_SQRT, RTC_MATH_MULADD, RTC_MATH_COUNT };
int rtc_probe_math(rtc_context* ctx, int fn, const float* x, const float* y, float* out, uint32_t n);

int rtc_stats_get(rtc_context* ctx, rtc_stats* out);   /* synchronises the context stream */
int rtc_stats_reset(rtc_context* ctx);

#ifdef __cplusplus
}
#endif
#endif /* RTC_CORE_H */
