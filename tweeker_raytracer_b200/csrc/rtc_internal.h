// rtc_internal.h -- structures shared by the host side of librtcore and its sm_100a kernels.
//
// HBM layout of one scene (everything the traversal touches is 16-byte addressable so every
// fetch is one LDG.128):
//   per GAS    nodes  uint4[5] per wide node (80 B): 8 children, quantised boxes    -> Node8 below (root = node 0)
//              tris   float4[3] per triangle (48 B): v0.xyz|prim id, v1.xyz|0, v2.xyz|0   (leaf order)
//   per scene  tlasNodes  the same 80 B nodes over instance bounds (root = node 0)
//              tlasLeaves uint32 per instance-level leaf slot -> instance id
//              instances  float4[4] per instance (64 B): world->object rows 0..2, {GAS nodes ptr, GAS tris ptr}
//   shading tables (used by shade only): objectToWorld float4[3], rt_GeometryInstanceData per instance
// Node and triangle indices are relative to their own GAS, so a GAS is built once (on the host or by the
// GPU builder, straight into device memory) and shared by any number of instances and scenes.
#pragma once

#include <cstdint>
#include <string>
#include <utility>
#include <vector>

#include <cuda_runtime.h>

#include "rtc_core.h"

// 8-wide node with child boxes quantised to 8 bits per plane on a per-node power-of-two grid
// (after Ylitie, Karras, Laine, "Efficient Incoherent Ray Traversal on GPUs Through Compressed
// Wide BVHs", HPG 2017).  Child i occupies slot i; slots are assigned by octant so that
// slot ^ (7 ^ rayOctant) is a front-to-back priority.
//   empty slot : imask bit clear, meta == 0
//   inner child: imask bit set; its node is childBase + popc(imask & ((1 << slot) - 1))
//   leaf child : imask bit clear, meta = (count << 5) | offset; primitives triBase + offset .. + count - 1
struct Node8
{
  float    px, py, pz;
  uint8_t  ex, ey, ez;      // biased exponents: grid step = 2^(e - 127)
  uint8_t  imask;
  uint32_t childBase;
  uint32_t triBase;
  uint8_t  meta[8];
  uint8_t  qlox[8], qloy[8];
  uint8_t  qloz[8], qhix[8];
  uint8_t  qhiy[8], qhiz[8];
};
static_assert(sizeof(Node8) == 80, "wide node is 80 bytes");

// Device-visible scene descriptor; SystemData::topObject points at one of these (in device memory).
struct SceneDesc
{
  const uint4*    tlasNodes;
  const uint32_t* tlasLeaves;
  const float4*   instances;
  const float4*   objectToWorld;
  const rt_GeometryInstanceData* geomInst;
  const uint32_t* instFlags;      // RTC_INSTANCE_* per instance (which hit records the instance uses)
  uint32_t        numInstances;
  uint32_t        numTlasNodes;
  uint32_t        numTlasLeaves;
  uint32_t        pad0;
};

// Host-side result of a BVH build over generic primitive boxes.
struct WideBvh
{
  std::vector<Node8>    nodes;      // nodes[0] is the root
  std::vector<uint32_t> primOrder;  // leaf order -> input primitive index
  float lo[3], hi[3];               // bounds of everything
};

struct PrimBox { float lo[3], hi[3]; };

// bvh_build_host.cpp: binned-SAH binary build, greedy collapse to 8-wide, octant slot assignment, quantisation.
// leafMax: primitives per leaf child (1..3).  Triangles: 2 (rtc_gas_build).  Instances: 1 -- entering an instance costs about three node
// visits (transform, shear constants, the GAS root), so a leaf box shared by two or three instances is never worth it
// (geometry scene: 1.30 -> 1.06 instance entries per ray, +7.5 % samples/s).
void build_wide_bvh_host(const PrimBox* prims, uint32_t numPrims, WideBvh& out, uint32_t leafMax = 3, bool instanceLevel = false);

// accel_host.cpp: the host halves of rtc_gas_build (host SAH builder) and rtc_ias_build (the instance level's SAH build) -- no
// CUDA call in any of them -- shared with the host-only twin of the two builds (rtc_host_gas_build / rtc_host_ias_build,
// include/rtc_core.h).  The twin's instance boxes and world->object matrices are the reference for the device's instance records
// (bvh_refit.cu): the same bvh_rules.h arithmetic, compiled for the host and the device.
bool gas_assemble_host(const uint8_t* verts, uint32_t strideBytes, uint32_t numVerts, const uint32_t* idx, uint32_t numTris,
                       WideBvh& bvh, std::vector<float4>& tris);
void instance_bounds_host(const float transform[12], const uint8_t* verts, uint32_t strideBytes, uint32_t numVerts, PrimBox& out);
bool instance_bounds_tight();      // false with RTC_INSTANCE_BOUNDS=box
void tlas_build_host(const PrimBox* boxes, uint32_t numInstances, WideBvh& bvh);

// Refit scratch of one wide BVH (bvh_refit.cu): the parent and an arrival counter per node, and the float box each node computed
// for itself (6 floats; node 0's box bounds the whole structure).  One allocation, made on the structure's first refit.
struct RefitScratch
{
  void*     base = nullptr;
  uint32_t* parent = nullptr;
  uint32_t* arrivals = nullptr;
  float*    box = nullptr;
  bool      pooled = false;          // base came from the stream-ordered pool (cudaMallocAsync)
};

struct LbvhRebuild;

struct GasRecord
{
  void*    d_nodes = nullptr;              // Node8[numNodes]
  void*    d_tris = nullptr;               // float4[3 * numTris]
  uint32_t numNodes = 0, numTris = 0;
  float    lo[3] = { 0, 0, 0 }, hi[3] = { 0, 0, 0 };
  uint64_t attributes = 0, indices = 0;    // caller-owned inputs (kept for the per-instance shading table)
  uint32_t strideBytes = 0, numVerts = 0;
  double   buildMs = 0.0;
  int      builder = 0;                    // RTC_BUILD_HOST_SAH or RTC_BUILD_GPU_LBVH
  uint64_t generation = 0;                 // rtc_gas_refit / rtc_gas_rebuild / rtc_gas_build_device count: scenes built / updated at an older generation are stale
  RefitScratch refit;
  bool     boundsOnDevice = false;         // lo / hi are stale: the refitted or rebuilt bounds are refit.box[0..5] on the device
  // rtc_gas_rebuild (bvh_build_gas_rebuild_gpu.cu): its arrays, made by the first rebuild, and from then on the node count on the
  // device -- numNodes is then only brought up to date by sync_gas_node_count (rtc_api.cpp) -- and the triangles the last build
  // rejected (rtc_gas_rejected_triangles)
  LbvhRebuild* rebuild = nullptr;
  const uint32_t* d_numNodes = nullptr;
  const uint32_t* d_rejected = nullptr;
  // rtc_gas_create: the triangles its arrays hold (the most rtc_gas_build_device accepts); 0 for a GAS of rtc_gas_build
  uint32_t capacity = 0;
};

struct SceneRecord
{
  SceneDesc desc{};          // host copy
  SceneDesc* d_desc = nullptr;
  void *d_tlasNodes = nullptr, *d_instances = nullptr, *d_tlasLeaves = nullptr, *d_o2w = nullptr, *d_geomInst = nullptr, *d_instFlags = nullptr;
  std::vector<uint32_t> instFlags;         // host copy of the per-instance flags
  uint32_t numCutout = 0;                  // instances using the cutout hit records: > 0 selects the ordered any-hit path
  bool     albedoTextures = false;         // MaterialDefinition.textureAlbedo may be non-zero: selects the textured shade kernels
  // The current object->world and world->object matrices live on the device only (d_o2w, d_instances): the instance records of
  // rtc_ias_build, rtc_ias_update and rtc_ias_update_device write them there, rtc_scene_export and rtc_instance_inverse read them back.
  std::vector<uint32_t> instGas;           // GAS handle per instance
  std::vector<std::pair<uint32_t, uint64_t>> gasGeneration;   // each distinct GAS and its generation at the last build / update
  // per instance: the position of its GAS in gasGeneration (the instance records' per-GAS table); in a created scene its GAS handle
  // (an index of the context's GAS table), or kRejectedInstance
  uint32_t* d_instGasSlot = nullptr;
  // rtc_ias_create / rtc_ias_build_device: the instance set lives on the device, in arrays sized for `capacity`.  instGas and
  // gasGeneration stay empty; the device holds what they hold for a built scene.
  bool     created = false;
  uint32_t capacity = 0;
  uint64_t* d_instGen = nullptr;           // per instance: its GAS's generation when its record was written
  uint32_t* d_words = nullptr;             // [kRejectedWord] records the last build rejected, [kCandidateWord] records written by a call
  uint32_t* d_gasRefs = nullptr;           // per GAS handle: instances of the last build that reference it (pooled)
  uint32_t  gasRefsCount = 0;              // handles d_gasRefs covers (the context's GAS count at the last build)
  uint32_t  gasRefsCapacity = 0;
  void*     d_emptyGas = nullptr;          // an empty GAS root node (and room for its triangles): the geometry of a rejected record
  uint64_t  gasEpoch = 0;                  // rtc_context::gasEpoch at the last build / update: a created scene is stale when it differs
  bool      gasDestroyed = false;          // rtc_gas_destroy of a handle the last build references
  PrimBox* d_instBoxes = nullptr;          // the padded world box of every instance (leaf boxes of the instance level)
  RefitScratch refit;
  // rtc_ias_rebuild (bvh_build_ias_gpu.cu): its arrays, made by the first rebuild, and from then on the instance level's node count
  // on the device -- desc.numTlasNodes is then only brought up to date by sync_tlas_node_count (rtc_api.cpp)
  LbvhRebuild* rebuild = nullptr;
  const uint32_t* d_numTlasNodes = nullptr;
  uint64_t totalNodes = 0, totalTris = 0;  // unique GAS nodes / triangles referenced + instance level
  uint32_t numGas = 0;
  double   gasBuildMs = 0.0, iasBuildMs = 0.0;
};

// Wavefront state of one launch batch (device pointers, SoA, sized for `capacity` paths).
struct WavefrontBuffers
{
  uint64_t capacity = 0;
  float4 *rayOrg = nullptr, *rayDir = nullptr;     // per path: next radiance ray (org.xyz,tmin) (dir.xyz,tmax)
  float4 *hit = nullptr;                           // per path: t,u,v,prim bits
  uint32_t *hitInst = nullptr;                     // per path
  float4 *throughput = nullptr;                    // per path: T.xyz, pdf
  float4 *radiance = nullptr;                      // per path: L.xyz, flags bits
  uint4  *misc = nullptr;                          // per path: seed, depth, stackIdx, pixel index
  float4 *absStack = nullptr;                      // per path x 4: nested-volume stack
  float4 *shadowOrg = nullptr, *shadowDir = nullptr, *shadowContrib = nullptr;  // per path
  uint32_t *queueA = nullptr, *queueB = nullptr, *shadowQueue = nullptr;
  uint32_t *bins = nullptr; uint32_t binStride = 0;  // per shade class: path ids binned after extend (class c at bins + c * binStride)
  uint32_t *counters = nullptr;                    // [0..63] extend counts per depth, [64..127] shadow counts per depth,
                                                   // [128..191] extend ray cursors, [192..255] connect ray cursors
  void* base = nullptr;
  // ordered any-hit processing (scenes with cutout materials only): two ping-pong queues of paths whose closest candidate
  // was ignored, and their counters {count A, count B, cursor}; allocated on first use
  uint32_t *cutQueue[2] = { nullptr, nullptr };
  uint32_t *cutCounters = nullptr;
  uint64_t cutCapacity = 0;
  void* cutBase = nullptr;
};

// RTC_SCHEDULE_GROUP / RTC_SCHEDULE_ONE_TRI / RTC_SCHEDULE_TWO_TRI (rtc_core.h): how the lane-owned traversal driver times its triangle tests
// (trace.cuh Traversal::step); hits and work counters do not depend on it.
// Run-time choice between the schedules.  The capped ones were written when no GPU was left to measure them on, so the library
// measures them itself: of the first batches of a context that are large enough to time (>= 1 Mi paths), one is a warm-up and
// the next four run group / one triangle / two triangles / group, each between two events; a capped schedule serves every later
// launch only if it beats the FASTER of the two group batches by 3 % (the faster capped one if both do).  Results are
// bit-identical under all of them, so the choice never shows in a frame.  RTC_TRACE_SCHEDULE=group|onetri|twotri fixes it (auto
// is the default); rtc_trace_schedule_get reports what happened.
struct ScheduleTuner
{
  enum State { WARMUP = 0, TIMING = 1, PENDING = 2, DONE = 3 };
  static constexpr int kSlots = 4;  // timed batches: group, one triangle, two triangles, group again
  int         state = WARMUP;
  int         slot = 0;             // TIMING: the next timed batch
  cudaEvent_t ev[2 * kSlots] = {};  // begin / end of each timed batch
  uint64_t    paths = 0;            // size of the timed batches (all must be the same)
  int         restarts = 0;         // a batch of another size restarts the measurement; bounded
  float       ms[kSlots] = { 0.0f, 0.0f, 0.0f, 0.0f };
  bool        fixedByEnv = false;
};

struct rtc_context
{
  int device = 0;
  cudaStream_t stream = nullptr;
  int numSMs = 0;
  std::vector<GasRecord> gas;
  std::vector<SceneRecord*> scenes;
  WavefrontBuffers wf;
  uint64_t* d_stats = nullptr;        // device counters: radiance rays, shadow rays, path samples
  uint64_t kernelLaunches = 0;
  double lastTraceMs = 0.0;
  bool traceTimed = false;
  cudaEvent_t evA = nullptr, evB = nullptr;
  cudaEvent_t evTimerA = nullptr, evTimerB = nullptr;
  // per-kernel-class profile (rtc_profile_enable): pending event pairs are resolved at rtc_profile_get
  bool profiling = false;
  struct ProfileSpan { int cls; cudaEvent_t a, b; };
  std::vector<ProfileSpan> spans;
  std::vector<cudaEvent_t> eventPool;
  rtc_profile profile{};
  std::vector<void*> textures;                    // rtc_texture_create allocations still alive
  // side streams of the shade stage: the class-specialised kernels of one depth are independent of each other and mostly
  // small, so they run concurrently (fork from `stream` after k_bin, join before connect); created on first use
  cudaStream_t shadeStreams[6] = {};
  cudaEvent_t  shadeFork = nullptr, shadeJoin[6] = {};
  unsigned long long* d_launchCounts = nullptr;   // 3 x kTraceCountWords: extend, connect, rtc_trace_count
  uint32_t* d_cursor = nullptr;                   // ray cursor of the query kernels (rtc_trace_*)
  int    traceSchedule = 0;                       // RTC_SCHEDULE_*: how the lane-owned driver times its triangle tests (what the NEXT launch uses)
  ScheduleTuner tuner;                            // picks traceSchedule by timing one batch with each (kernels_shade.cu, "schedule tuner")
  void*  cutoutGraph = nullptr;                   // CutoutGraph (kernels_shade.cu): the device-side loop of the ordered any-hit rounds
  uint64_t cutoutGraphBuilds = 0;                 // graph pairs captured since the last rtc_stats_reset (rtc_stats)
  // The device GAS table, indexed by handle: the instance records of created scenes read it.  Kept up to date on the stream by
  // rtc_gas_build, rtc_gas_create, rtc_gas_build_device, rtc_gas_refit, rtc_gas_rebuild and rtc_gas_destroy (a destroyed GAS has null nodes); grown from the pool.
  struct GasUpdateInput* d_gasTable = nullptr;
  uint64_t* d_gasGen = nullptr;                   // per handle: GasRecord::generation
  uint32_t gasTableCapacity = 0;
  uint64_t gasEpoch = 0;                          // refits and rebuilds of any GAS of the context
};

// work counters of one traversal kernel: {nodes, tris, insts, rays}
constexpr int kTraceCountWords = 4;

// RAII-less helpers used by the launchers: bracket one kernel launch with an event pair when profiling is on
int profile_begin(rtc_context* ctx, int cls);
int profile_end(rtc_context* ctx);

// RTC_BUILD_DEFAULT picks the GPU LBVH builder above this many triangles (host SAH quality below it)
constexpr uint32_t kGpuBuildThreshold = 1u << 20;
// bvh_build_gpu.cu: Morton LBVH on the device, straight into rec.d_nodes / rec.d_tris; fills numNodes, lo, hi
int build_gas_gpu(rtc_context* ctx, GasRecord& rec);

// bvh_refit.cu: refits and instance records, all enqueued on ctx->stream without a host synchronisation (except the one-time
// scratch allocation of a GAS refit).  refit_gas_gpu rewrites the triangle records from rec.attributes and re-quantises every
// node bottom-up.
int refit_gas_gpu(rtc_context* ctx, GasRecord& rec);
// One distinct GAS of a scene as its instance records read it (SceneRecord::gasGeneration order).
struct GasUpdateInput
{
  const void*    nodes;            // the GAS's node and triangle arrays: row 3 of the traversal record of each of its instances
  const void*    tris;
  const uint8_t* verts;            // the GAS's vertex records (tight bounds)
  uint32_t stride, numVerts;       // numVerts = 0 for an empty GAS
  const float* gasBox;             // device lo[3], hi[3] of a refitted GAS, or null: gasLoHi
  float    gasLoHi[6];
  uint64_t attributes;             // rt_GeometryInstanceData::attributes
  uint32_t emptyGas, pad;
  uint64_t indices;                // rt_GeometryInstanceData::indices
};
// d_instGasSlot of a created scene for a record rtc_ias_build_device rejected
constexpr uint32_t kRejectedInstance = 0xffffffffu;
enum { kRejectedWord = 0, kCandidateWord = 1, kSceneWords = 2 };
// The records of the candidate instances (rtc_ias_build: every instance; rtc_ias_update, rtc_ias_update_device: the recomputed
// ones): candidate j is instance candidates[j], or first + j when `candidates` is empty.  Instance i in [first, first + count)
// takes the object->world matrix at transforms + (i - first) * strideBytes (device-readable memory, read when the stream gets
// there), every other candidate keeps its current one (d_o2w).  Writes the 64 B traversal records (world->object rows, GAS
// pointers), the object->world rows, shading-table attributes and padded boxes of the candidates; allocates only from the
// stream-ordered pool.
int write_instance_records_gpu(rtc_context* ctx, SceneRecord& s, const uint8_t* transforms, uint32_t strideBytes, uint32_t first,
                               uint32_t count, const std::vector<uint32_t>& candidates, const std::vector<GasUpdateInput>& gas, bool tight);
// The same kernels for a created scene, over the context's GAS table, with the candidates selected on the device.  records
// non-null (rtc_ias_build_device): every instance i < s.desc.numInstances takes the rtc_instance_desc at records + i * strideBytes,
// which is validated; its GAS handle, generation, shading-table row and the per-handle reference counts are written, rejected
// records counted.  records null (the updates): the instances of [first, first + count) take the matrices at transforms, and every
// instance whose GAS's generation changed is recomputed with its current one.
int write_created_records_gpu(rtc_context* ctx, SceneRecord& s, const uint8_t* records, const uint8_t* transforms, uint32_t strideBytes,
                              uint32_t first, uint32_t count, bool tight);
// The updates' refit of the instance level's nodes over s.d_instBoxes; a scene's first refit allocates its scratch from the
// stream-ordered pool.
int refit_instance_level_gpu(rtc_context* ctx, SceneRecord& s);
// stream: the one the structure's work runs on (a pooled scratch is freed behind it)
void free_refit_scratch(RefitScratch& r, cudaStream_t stream);

// bvh_build_ias_gpu.cu: a new LBVH topology of the instance level over s.d_instBoxes, in place and stream-ordered; the first call
// on a scene allocates (and synchronises once), later calls never block the host
int rebuild_instances_gpu(rtc_context* ctx, SceneRecord& s);
// rtc_ias_create: the rebuild's arrays for `capacity` instances, set up at once (synchronises); the scene starts with no instance
int create_instance_level_gpu(rtc_context* ctx, SceneRecord& s, uint32_t capacity);
// bvh_build_gas_rebuild_gpu.cu: the same for a geometry, over the rec.numTris triangles of rec.attributes / rec.indices (an index
// >= rec.numVerts reads a NaN vertex); writes the triangle records in leaf order and the root box into rec.refit.box[0..5]
int rebuild_gas_gpu(rtc_context* ctx, GasRecord& rec);
// rtc_gas_create: the rebuild's arrays for `capacity` triangles (rec.d_tris already holds them), set up at once (synchronises);
// the GAS starts with rec.numTris == 0
int create_gas_gpu(rtc_context* ctx, GasRecord& rec, uint32_t capacity);
// the wide nodes a rebuilt node array holds: every wide node but the root has a sibling-group parent, so one-primitive leaves give
// < n + 16 (the same bound as build_gas_gpu's)
inline uint32_t ias_rebuild_capacity(uint32_t numPrims) { return numPrims + 16u; }
void free_lbvh_rebuild(LbvhRebuild* r);

// error plumbing (rtc_api.cpp)
int rtc_set_error(const char* file, int line, const char* call, int code, const char* text);
#define RTC_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return rtc_set_error(__FILE__, __LINE__, #call, (int)e_, cudaGetErrorString(e_)); } while (0)
#define RTC_FAIL(text) return rtc_set_error(__FILE__, __LINE__, __func__, -1, text)

// kernel launchers (kernels_trace.cu / kernels_shade.cu); all enqueue on ctx->stream
int launch_trace_closest(rtc_context* ctx, const SceneDesc* d_scene, const rtc_ray* rays, uint64_t n, rtc_hit* hits);
int launch_trace_any(rtc_context* ctx, const SceneDesc* d_scene, const rtc_ray* rays, uint64_t n, uint32_t* occluded);
// counting variant: adds {nodes popped, triangles tested, instances entered, rays} to d_counts[0..3]
int launch_trace_count(rtc_context* ctx, const SceneDesc* d_scene, const rtc_ray* rays, uint64_t n, int anyHit, unsigned long long* d_counts);
// cursor: zero-initialised device counter the persistent warps hand rays out from (one per launch)
int launch_extend(rtc_context* ctx, const SceneDesc* d_scene, const WavefrontBuffers& wf, const uint32_t* queue, const uint32_t* count,
                  uint32_t* cursor, bool countWork);
int launch_connect(rtc_context* ctx, const SceneDesc* d_scene, const WavefrontBuffers& wf, const uint32_t* count, uint32_t* cursor, bool countWork);
// ordered any-hit processing (cutout materials): re-trace past an ignored candidate / shadow rays as closest-hit queries
int launch_extend_after(rtc_context* ctx, const SceneDesc* d_scene, const WavefrontBuffers& wf, const uint32_t* queue, const uint32_t* count, uint32_t* cursor);
int launch_connect_closest(rtc_context* ctx, const SceneDesc* d_scene, const WavefrontBuffers& wf, const uint32_t* queue, const uint32_t* count,
                           uint32_t* cursor, bool after);
int launch_generate_primary(rtc_context* ctx, const rt_SystemData& sys, uint32_t w, uint32_t h, int iteration, rtc_ray* rays);
int launch_wavefront(rtc_context* ctx, const rt_SystemData& sys, uint32_t w, uint32_t h, int raygen, int miss, int iterFirst, int iterCount,
                     int accumFirst, bool countWork);
int launch_composite(rtc_context* ctx, const rt_CompositorData& args);
int launch_tonemap(rtc_context* ctx, const rt_TonemapperParams& p, const float4* rgba, uint8_t* rgb, uint64_t n);
int launch_probe_math(rtc_context* ctx, int fn, const float* x, const float* y, float* out, uint32_t n);   // device pointers
int ensure_wavefront(rtc_context* ctx, uint64_t capacity, bool* outOfMemory = nullptr);
void release_cutout_graph(rtc_context* ctx);
int read_stack_overflows(rtc_context* ctx, uint64_t* out);
// schedule tuner (kernels_shade.cu); tuner_finish blocks for the last timed batch when a decision is pending
void tuner_finish(rtc_context* ctx);
void tuner_release(rtc_context* ctx);
void preload_capped_trace_kernels();       // kernels_trace.cu: loads the capped-schedule kernels before they are timed (lazy module loading)
int read_stack_overflows_primary(rtc_context* ctx, uint64_t* out);   // the counter of the primary-ray extend kernel (kernels_shade.cu)
