// rtc_api.cpp -- the C ABI of librtcore (include/rtc_core.h): contexts, memory, acceleration-structure
// builds, launches.  This file replaces the OptiX host calls of apps/rtigo3/src/Device.cpp (see the table
// at the top of rtc_core.h); there is no CPU rendering path here: every entry point that produces
// rays, hits or pixels ends in a kernel launch on the context's stream.
#include "rtc_internal.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iterator>
#include <limits>
#include <set>

namespace {

thread_local std::string g_lastError;

double now_ms()
{
  using namespace std::chrono;
  return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

SceneRecord* find_scene(rtc_context* ctx, uint64_t topObject)
{
  for (SceneRecord* s : ctx->scenes) if ((uint64_t)(uintptr_t)s->d_desc == topObject) return s;
  return nullptr;
}

void free_scene(SceneRecord* s, cudaStream_t stream)
{
  cudaFree(s->d_desc); cudaFree(s->d_tlasNodes); cudaFree(s->d_instances); cudaFree(s->d_tlasLeaves); cudaFree(s->d_o2w); cudaFree(s->d_geomInst); cudaFree(s->d_instFlags);
  cudaFree(s->d_instBoxes); cudaFree(s->d_instGasSlot); free_refit_scratch(s->refit, stream); free_lbvh_rebuild(s->rebuild);
  cudaFree(s->d_instGen); cudaFree(s->d_words); cudaFree(s->d_emptyGas);
  if (s->d_gasRefs) cudaFreeAsync(s->d_gasRefs, stream);
  delete s;
}

constexpr const char* kDestroyedGas = "a GAS of this scene was destroyed";
constexpr const char* kStaleScene = "a GAS of this scene was refitted after the scene was built or updated: call rtc_ias_update on the scene first";
constexpr const char* kStaleCreatedScene = "a GAS of the context was refitted or rebuilt after this scene of rtc_ias_create was built or updated: "
                                           "call rtc_ias_update on the scene first";

// Why the scene cannot be traced, or nullptr.  A GAS it instances was destroyed: its nodes and triangles are freed, and the
// scene's instance records still point at them.  Or (unless `refitAllowed`, for the instance updates, which cure it) the scene is
// stale: a GAS was refitted after the scene was built or last updated, so its instance boxes and instance level no longer
// bound the triangles, and its shading table may point at a vertex buffer the caller has since freed.
// A created scene does not know on the host which GAS it references: it is stale after a refit or rebuild of any GAS of the
// context (conservative; the update then recomputes exactly the instances whose GAS changed), and rtc_gas_destroy marks it when
// its last build references the handle.
const char* scene_unusable(const rtc_context* ctx, const SceneRecord* s, bool refitAllowed = false)
{
  if (s->created)
  {
    if (s->gasDestroyed) return kDestroyedGas;
    return (s->gasEpoch != ctx->gasEpoch && !refitAllowed) ? kStaleCreatedScene : nullptr;
  }
  bool stale = false;
  for (const std::pair<uint32_t, uint64_t>& g : s->gasGeneration)
  {
    if (ctx->gas[g.first].d_nodes == nullptr) return kDestroyedGas;
    stale = stale || ctx->gas[g.first].generation != g.second;
  }
  return (stale && !refitAllowed) ? kStaleScene : nullptr;
}

// After rtc_ias_rebuild the instance level's node count is only on the device: bring the host copy (desc.numTlasNodes and the
// scene's node total) up to date.  Synchronises the stream.
int sync_tlas_node_count(rtc_context* ctx, SceneRecord* s)
{
  if (!s->d_numTlasNodes) return 0;
  uint32_t count = 0;
  RTC_CUDA(cudaMemcpyAsync(&count, s->d_numTlasNodes, sizeof(count), cudaMemcpyDeviceToHost, ctx->stream));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  s->totalNodes = s->totalNodes - s->desc.numTlasNodes + count;
  s->desc.numTlasNodes = count;
  return 0;
}

// After rtc_gas_rebuild a GAS's node count is only on the device: bring the host copy (numNodes, and the node total of every
// scene that instances the GAS) up to date.  Synchronises the stream.
int sync_gas_node_count(rtc_context* ctx, uint32_t gas)
{
  GasRecord& g = ctx->gas[gas];
  if (!g.d_numNodes) return 0;
  uint32_t count = 0;
  RTC_CUDA(cudaMemcpyAsync(&count, g.d_numNodes, sizeof(count), cudaMemcpyDeviceToHost, ctx->stream));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  for (SceneRecord* s : ctx->scenes)
    for (const std::pair<uint32_t, uint64_t>& e : s->gasGeneration)
      if (e.first == gas) s->totalNodes = s->totalNodes - g.numNodes + count;
  g.numNodes = count;
  return 0;
}

// One GAS as its instance records read it.  A refitted GAS's bounds are read on the device; a destroyed one has null nodes.
GasUpdateInput gas_entry(const GasRecord& g)
{
  GasUpdateInput u;
  u.nodes = g.d_nodes; u.tris = g.d_tris;
  u.verts = reinterpret_cast<const uint8_t*>((uintptr_t)g.attributes); u.stride = g.strideBytes; u.numVerts = g.numTris ? g.numVerts : 0u;
  u.gasBox = g.boundsOnDevice ? g.refit.box : nullptr;
  for (int c = 0; c < 3; ++c) { u.gasLoHi[c] = g.lo[c]; u.gasLoHi[3 + c] = g.hi[c]; }
  u.attributes = g.attributes;
  u.emptyGas = g.numTris == 0 ? 1u : 0u; u.pad = 0u;
  u.indices = g.indices;
  return u;
}

// The per-GAS table of the scene's instance records, in gasGeneration order.
std::vector<GasUpdateInput> gas_update_inputs(const rtc_context* ctx, const SceneRecord* s)
{
  std::vector<GasUpdateInput> gas(s->gasGeneration.size());
  for (size_t k = 0; k < gas.size(); ++k) gas[k] = gas_entry(ctx->gas[s->gasGeneration[k].first]);
  return gas;
}

// Writes GAS h's entry and generation into the context's device GAS table, stream-ordered; a handle past the table grows it from
// the pool behind the stream (work already enqueued keeps reading the old table until it is freed behind it).
int write_gas_table(rtc_context* ctx, uint32_t h)
{
  if (h >= ctx->gasTableCapacity)
  {
    const uint32_t cap = std::max(std::max(64u, h + 1u), 2u * ctx->gasTableCapacity);
    GasUpdateInput* table = nullptr;
    uint64_t* gen = nullptr;
    RTC_CUDA(cudaMallocAsync((void**)&table, (size_t)cap * sizeof(GasUpdateInput), ctx->stream));
    const cudaError_t e = cudaMallocAsync((void**)&gen, (size_t)cap * sizeof(uint64_t), ctx->stream);
    if (e != cudaSuccess) { cudaFreeAsync(table, ctx->stream); return rtc_set_error(__FILE__, __LINE__, "cudaMallocAsync(GAS table)", (int)e, cudaGetErrorString(e)); }
    if (ctx->gasTableCapacity)
    {
      RTC_CUDA(cudaMemcpyAsync(table, ctx->d_gasTable, (size_t)ctx->gasTableCapacity * sizeof(GasUpdateInput), cudaMemcpyDeviceToDevice, ctx->stream));
      RTC_CUDA(cudaMemcpyAsync(gen, ctx->d_gasGen, (size_t)ctx->gasTableCapacity * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream));
      cudaFreeAsync(ctx->d_gasTable, ctx->stream);
      cudaFreeAsync(ctx->d_gasGen, ctx->stream);
    }
    ctx->d_gasTable = table; ctx->d_gasGen = gen; ctx->gasTableCapacity = cap;
  }
  const GasRecord& g = ctx->gas[h];
  const GasUpdateInput entry = gas_entry(g);
  RTC_CUDA(cudaMemcpyAsync(ctx->d_gasTable + h, &entry, sizeof(entry), cudaMemcpyHostToDevice, ctx->stream));
  RTC_CUDA(cudaMemcpyAsync(ctx->d_gasGen + h, &g.generation, sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}

// instances of a created scene are at most its capacity; flags of positions past the instance count wait for a later build
void count_cutout(SceneRecord* s)
{
  s->numCutout = 0;
  for (uint32_t i = 0; i < s->desc.numInstances && i < s->instFlags.size(); ++i) if (s->instFlags[i] & RTC_INSTANCE_CUTOUT) s->numCutout++;
}

// rtc_ias_update and rtc_ias_update_device (arguments checked): instance first + i takes the matrix at transforms + i * strideBytes
// (device-readable).  Recomputes exactly the instances of the range and those of every GAS refitted since the last build / update
// -- no other: the vertex buffer of a GAS that was not refitted may already hold positions its boxes do not bound yet.
int update_instances(rtc_context* ctx, SceneRecord* s, uint32_t first, uint32_t count, const uint8_t* transforms, uint32_t strideBytes)
{
  if (s->created)
  {
    // the candidates are selected on the device (the range, and the instances whose GAS's generation changed)
    if (s->desc.numInstances)
    {
      if (int rc = write_created_records_gpu(ctx, *s, nullptr, transforms, strideBytes, first, count, instance_bounds_tight())) return rc;
      if (int rc = refit_instance_level_gpu(ctx, *s)) return rc;
    }
    s->gasEpoch = ctx->gasEpoch;
    return 0;
  }
  std::vector<uint8_t> refitted(ctx->gas.size(), 0u);
  bool anyRefitted = false;
  for (const std::pair<uint32_t, uint64_t>& g : s->gasGeneration)
    if (ctx->gas[g.first].generation != g.second) { refitted[g.first] = 1u; anyRefitted = true; }
  std::vector<uint32_t> candidates;           // empty: the range
  if (anyRefitted)
    for (uint32_t i = 0; i < s->desc.numInstances; ++i)
      if ((first <= i && i < first + count) || refitted[s->instGas[i]]) candidates.push_back(i);
  if (count || !candidates.empty())
  {
    if (int rc = write_instance_records_gpu(ctx, *s, transforms, strideBytes, first, count, candidates, gas_update_inputs(ctx, s),
                                            instance_bounds_tight())) return rc;
    if (int rc = refit_instance_level_gpu(ctx, *s)) return rc;
  }
  for (std::pair<uint32_t, uint64_t>& g : s->gasGeneration) g.second = ctx->gas[g.first].generation;
  return 0;
}

} // namespace

int rtc_set_error(const char* file, int line, const char* call, int code, const char* text)
{
  char buf[1024];
  std::snprintf(buf, sizeof(buf), "ERROR: %s(%d): %s (%d) %s", file, line, call, code, text ? text : "");
  g_lastError = buf;
  return code ? code : -1;
}

static int take_event(rtc_context* ctx, cudaEvent_t* e)
{
  if (!ctx->eventPool.empty()) { *e = ctx->eventPool.back(); ctx->eventPool.pop_back(); return 0; }
  RTC_CUDA(cudaEventCreate(e));
  return 0;
}

int profile_begin(rtc_context* ctx, int cls)
{
  if (!ctx->profiling) return 0;
  // bound the number of pending events: resolve (synchronise) every 4096 launches
  if (ctx->spans.size() >= 4096)
  {
    RTC_CUDA(cudaStreamSynchronize(ctx->stream));
    for (rtc_context::ProfileSpan& sp : ctx->spans)
    {
      float ms = 0.0f;
      RTC_CUDA(cudaEventElapsedTime(&ms, sp.a, sp.b));
      ctx->profile.ms[sp.cls] += ms; ctx->profile.launches[sp.cls] += 1;
      ctx->eventPool.push_back(sp.a); ctx->eventPool.push_back(sp.b);
    }
    ctx->spans.clear();
  }
  rtc_context::ProfileSpan sp; sp.cls = cls;
  if (int rc = take_event(ctx, &sp.a)) return rc;
  if (int rc = take_event(ctx, &sp.b)) return rc;
  RTC_CUDA(cudaEventRecord(sp.a, ctx->stream));
  ctx->spans.push_back(sp);
  return 0;
}

int profile_end(rtc_context* ctx)
{
  if (!ctx->profiling) return 0;
  RTC_CUDA(cudaEventRecord(ctx->spans.back().b, ctx->stream));
  return 0;
}

extern "C" {

int rtc_version(void) { return 102; }

const char* rtc_last_error(void) { return g_lastError.c_str(); }

int rtc_context_destroy(rtc_context* ctx);

static int context_init(rtc_context* ctx, int deviceOrdinal)
{
  ctx->device = deviceOrdinal;
  cudaDeviceProp prop;
  RTC_CUDA(cudaGetDeviceProperties(&prop, deviceOrdinal));
  ctx->numSMs = prop.multiProcessorCount;
  // schedule of the lane-owned driver's triangle tests: measured per context (auto) unless RTC_TRACE_SCHEDULE=group|onetri|twotri fixes it
  if (const char* e = getenv("RTC_TRACE_SCHEDULE"))
  {
    if (e[0] == 'g' || e[0] == '0') { ctx->traceSchedule = RTC_SCHEDULE_GROUP; ctx->tuner.state = ScheduleTuner::DONE; ctx->tuner.fixedByEnv = true; }
    else if (e[0] == 'o' || e[0] == '1') { ctx->traceSchedule = RTC_SCHEDULE_ONE_TRI; ctx->tuner.state = ScheduleTuner::DONE; ctx->tuner.fixedByEnv = true; }
    else if (e[0] == 't' || e[0] == '2') { ctx->traceSchedule = RTC_SCHEDULE_TWO_TRI; ctx->tuner.state = ScheduleTuner::DONE; ctx->tuner.fixedByEnv = true; }
  }
  RTC_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  {
    // keep freed build scratch in the device's default memory pool instead of returning it to the OS at every synchronise
    cudaMemPool_t pool = nullptr;
    if (cudaDeviceGetDefaultMemPool(&pool, deviceOrdinal) == cudaSuccess)
    {
      uint64_t threshold = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
    }
    cudaGetLastError();
  }
  RTC_CUDA(cudaEventCreate(&ctx->evA));
  RTC_CUDA(cudaEventCreate(&ctx->evB));
  RTC_CUDA(cudaEventCreate(&ctx->evTimerA));
  RTC_CUDA(cudaEventCreate(&ctx->evTimerB));
  RTC_CUDA(cudaMalloc(&ctx->d_stats, 8 * sizeof(uint64_t)));
  RTC_CUDA(cudaMemset(ctx->d_stats, 0, 8 * sizeof(uint64_t)));
  RTC_CUDA(cudaMalloc(&ctx->d_cursor, 4 * sizeof(uint32_t)));
  RTC_CUDA(cudaMalloc(&ctx->d_launchCounts, 3 * kTraceCountWords * sizeof(unsigned long long)));
  RTC_CUDA(cudaMemset(ctx->d_launchCounts, 0, 3 * kTraceCountWords * sizeof(unsigned long long)));
  return 0;
}

int rtc_context_create(int deviceOrdinal, rtc_context** out)
{
  if (!out) RTC_FAIL("out is null");
  *out = nullptr;
  int count = 0;
  RTC_CUDA(cudaGetDeviceCount(&count));
  if (deviceOrdinal < 0 || deviceOrdinal >= count) RTC_FAIL("device ordinal out of range (no CUDA device, no rendering: this core has no CPU path)");
  RTC_CUDA(cudaSetDevice(deviceOrdinal));
  rtc_context* ctx = new rtc_context();
  if (const int rc = context_init(ctx, deviceOrdinal))
  {
    const std::string why = rtc_last_error();      // the destroy below must not clobber the reason
    rtc_context_destroy(ctx);
    g_lastError = why;
    return rc;
  }
  *out = ctx;
  return 0;
}


int rtc_context_destroy(rtc_context* ctx)
{
  if (!ctx) return 0;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  release_cutout_graph(ctx);
  tuner_release(ctx);
  for (SceneRecord* s : ctx->scenes) free_scene(s, ctx->stream);
  for (GasRecord& g : ctx->gas) { cudaFree(g.d_nodes); cudaFree(g.d_tris); free_refit_scratch(g.refit, ctx->stream); free_lbvh_rebuild(g.rebuild); }
  if (ctx->wf.base) cudaFree(ctx->wf.base);
  if (ctx->wf.cutBase) cudaFree(ctx->wf.cutBase);
  for (void* t : ctx->textures) cudaFree(t);
  cudaFree(ctx->d_gasTable);
  cudaFree(ctx->d_gasGen);
  cudaFree(ctx->d_stats);
  cudaFree(ctx->d_launchCounts);
  cudaFree(ctx->d_cursor);
  for (rtc_context::ProfileSpan& sp : ctx->spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
  for (cudaEvent_t e : ctx->eventPool) cudaEventDestroy(e);
  for (cudaEvent_t e : { ctx->evA, ctx->evB, ctx->evTimerA, ctx->evTimerB }) if (e) cudaEventDestroy(e);
  for (int k = 0; k < 6; ++k) { if (ctx->shadeStreams[k]) cudaStreamDestroy(ctx->shadeStreams[k]); if (ctx->shadeJoin[k]) cudaEventDestroy(ctx->shadeJoin[k]); }
  if (ctx->shadeFork) cudaEventDestroy(ctx->shadeFork);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  cudaGetLastError();
  delete ctx;
  return 0;
}

int rtc_synchronize(rtc_context* ctx)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

uint64_t rtc_context_stream(rtc_context* ctx) { return (uint64_t)(uintptr_t)ctx->stream; }

int rtc_device_count(int* count)
{
  if (!count) RTC_FAIL("count is null");
  *count = 0;
  RTC_CUDA(cudaGetDeviceCount(count));
  return 0;
}

int rtc_device_name(int deviceOrdinal, char* name, int length)
{
  if (!name || length <= 0) RTC_FAIL("bad name buffer");
  cudaDeviceProp prop;
  RTC_CUDA(cudaGetDeviceProperties(&prop, deviceOrdinal));
  std::snprintf(name, (size_t)length, "%s", prop.name);
  return 0;
}

int rtc_peer_can_access(int deviceOrdinal, int peerOrdinal, int* canAccess)
{
  if (!canAccess) RTC_FAIL("canAccess is null");
  if (deviceOrdinal == peerOrdinal) { *canAccess = 1; return 0; }
  RTC_CUDA(cudaDeviceCanAccessPeer(canAccess, deviceOrdinal, peerOrdinal));
  return 0;
}

int rtc_peer_enable(rtc_context* ctx, rtc_context* peer)
{
  if (ctx->device == peer->device) return 0;
  RTC_CUDA(cudaSetDevice(ctx->device));
  const cudaError_t e = cudaDeviceEnablePeerAccess(peer->device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return 0; }
  RTC_CUDA(e);
  return 0;
}

int rtc_peer_disable(rtc_context* ctx, rtc_context* peer)
{
  if (ctx->device == peer->device) return 0;
  RTC_CUDA(cudaSetDevice(ctx->device));
  const cudaError_t e = cudaDeviceDisablePeerAccess(peer->device);
  if (e == cudaErrorPeerAccessNotEnabled) { cudaGetLastError(); return 0; }
  RTC_CUDA(e);
  return 0;
}

int rtc_memcpy_peer(rtc_context* dstCtx, uint64_t dst, rtc_context* srcCtx, uint64_t src, uint64_t bytes)
{
  RTC_CUDA(cudaSetDevice(srcCtx->device));
  RTC_CUDA(cudaStreamSynchronize(srcCtx->stream));
  RTC_CUDA(cudaSetDevice(dstCtx->device));
  if (bytes == 0) return 0;
  if (dstCtx->device == srcCtx->device)
    RTC_CUDA(cudaMemcpyAsync((void*)(uintptr_t)dst, (const void*)(uintptr_t)src, bytes, cudaMemcpyDeviceToDevice, dstCtx->stream));
  else
    RTC_CUDA(cudaMemcpyPeerAsync((void*)(uintptr_t)dst, dstCtx->device, (const void*)(uintptr_t)src, srcCtx->device, bytes, dstCtx->stream));
  return 0;
}

int rtc_malloc(rtc_context* ctx, uint64_t bytes, uint64_t* dptr)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  void* p = nullptr;
  RTC_CUDA(cudaMalloc(&p, bytes ? bytes : 1));
  *dptr = (uint64_t)(uintptr_t)p;
  return 0;
}

int rtc_free(rtc_context* ctx, uint64_t dptr)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  RTC_CUDA(cudaFree((void*)(uintptr_t)dptr));
  return 0;
}

int rtc_upload(rtc_context* ctx, uint64_t dst, const void* src, uint64_t bytes)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  if (bytes) RTC_CUDA(cudaMemcpyAsync((void*)(uintptr_t)dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}

int rtc_download(rtc_context* ctx, void* dst, uint64_t src, uint64_t bytes)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  if (bytes) RTC_CUDA(cudaMemcpyAsync(dst, (const void*)(uintptr_t)src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return 0;
}

int rtc_memset(rtc_context* ctx, uint64_t dst, int value, uint64_t bytes)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  if (bytes) RTC_CUDA(cudaMemsetAsync((void*)(uintptr_t)dst, value, bytes, ctx->stream));
  return 0;
}

int rtc_host_alloc(rtc_context* ctx, uint64_t bytes, void** ptr)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocPortable | cudaHostAllocMapped));
  return 0;
}

int rtc_host_free(rtc_context* ctx, void* ptr)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaFreeHost(ptr));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Geometry acceleration structure (replaces optixAccelBuild over OPTIX_BUILD_INPUT_TYPE_TRIANGLES,
// Device.cpp:1362-1405: vertex stride sizeof(TriangleAttributes), uint3 indices, flags NONE).
// ------------------------------------------------------------------------------------------------
int rtc_gas_build(rtc_context* ctx, uint64_t attributes, uint32_t strideBytes, uint32_t numVerts,
                  uint64_t indices, uint32_t numTris, uint32_t buildFlags, uint32_t* gas)
{
  if (!gas) RTC_FAIL("gas is null");
  if (strideBytes < 12 || (strideBytes & 3u)) RTC_FAIL("vertex stride must be a multiple of 4 and at least 12");
  RTC_CUDA(cudaSetDevice(ctx->device));
  const double t0 = now_ms();
  GasRecord rec;
  rec.attributes = attributes; rec.indices = indices; rec.strideBytes = strideBytes; rec.numVerts = numVerts; rec.numTris = numTris;

  int builder = (int)buildFlags;
  if (builder == RTC_BUILD_DEFAULT)
  {
    builder = (numTris > kGpuBuildThreshold) ? RTC_BUILD_GPU_LBVH : RTC_BUILD_HOST_SAH;
    // RTC_FORCE_BUILDER=gpu|host overrides the size rule (used by the tests to run whole scenes through either builder)
    if (const char* force = std::getenv("RTC_FORCE_BUILDER"))
    {
      if (std::strcmp(force, "gpu") == 0) builder = RTC_BUILD_GPU_LBVH;
      else if (std::strcmp(force, "host") == 0) builder = RTC_BUILD_HOST_SAH;
    }
  }
  if (builder != RTC_BUILD_GPU_LBVH && builder != RTC_BUILD_HOST_SAH) RTC_FAIL("bad build flags");
  rec.builder = builder;

  if (builder == RTC_BUILD_GPU_LBVH && numTris > 0)
  {
    if (int rc = build_gas_gpu(ctx, rec)) return rc;
  }
  else
  {
    // host quality build: fetch positions and indices, bin-SAH, collapse, quantise, upload
    std::vector<uint8_t> verts((size_t)numVerts * strideBytes);
    std::vector<uint32_t> idx((size_t)numTris * 3u);
    RTC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (!verts.empty()) RTC_CUDA(cudaMemcpy(verts.data(), (const void*)(uintptr_t)attributes, verts.size(), cudaMemcpyDeviceToHost));
    if (!idx.empty()) RTC_CUDA(cudaMemcpy(idx.data(), (const void*)(uintptr_t)indices, idx.size() * 4u, cudaMemcpyDeviceToHost));
    WideBvh bvh;
    std::vector<float4> tris;
    if (!gas_assemble_host(verts.data(), strideBytes, numVerts, idx.data(), numTris, bvh, tris)) RTC_FAIL("triangle index out of range");
    rec.numNodes = (uint32_t)bvh.nodes.size();
    for (int k = 0; k < 3; ++k) { rec.lo[k] = bvh.lo[k]; rec.hi[k] = bvh.hi[k]; }
    RTC_CUDA(cudaMalloc(&rec.d_nodes, bvh.nodes.size() * sizeof(Node8)));
    RTC_CUDA(cudaMemcpy(rec.d_nodes, bvh.nodes.data(), bvh.nodes.size() * sizeof(Node8), cudaMemcpyHostToDevice));
    RTC_CUDA(cudaMalloc(&rec.d_tris, tris.empty() ? 16 : tris.size() * sizeof(float4)));
    if (!tris.empty()) RTC_CUDA(cudaMemcpy(rec.d_tris, tris.data(), tris.size() * sizeof(float4), cudaMemcpyHostToDevice));
  }
  rec.buildMs = now_ms() - t0;
  ctx->gas.push_back(rec);
  *gas = (uint32_t)(ctx->gas.size() - 1);
  return write_gas_table(ctx, *gas);
}

int rtc_gas_destroy(rtc_context* ctx, uint32_t gas)
{
  if (gas >= ctx->gas.size()) RTC_FAIL("bad gas handle");
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  GasRecord& g = ctx->gas[gas];
  // created scenes whose last build references the handle (the device's reference counts, read now that the stream is drained)
  for (SceneRecord* s : ctx->scenes)
    if (s->created && gas < s->gasRefsCount && g.d_nodes)
    {
      uint32_t refs = 0;
      RTC_CUDA(cudaMemcpy(&refs, s->d_gasRefs + gas, sizeof(refs), cudaMemcpyDeviceToHost));
      if (refs) s->gasDestroyed = true;
    }
  cudaFree(g.d_nodes); cudaFree(g.d_tris); free_refit_scratch(g.refit, ctx->stream); free_lbvh_rebuild(g.rebuild);
  g.d_nodes = nullptr; g.d_tris = nullptr; g.numNodes = 0; g.numTris = 0; g.boundsOnDevice = false;
  g.rebuild = nullptr; g.d_numNodes = nullptr; g.d_rejected = nullptr; g.capacity = 0;
  return write_gas_table(ctx, gas);
}

int rtc_gas_refit(rtc_context* ctx, uint32_t gas, uint64_t attributes)
{
  if (gas >= ctx->gas.size() || ctx->gas[gas].d_nodes == nullptr) RTC_FAIL("bad gas handle");
  RTC_CUDA(cudaSetDevice(ctx->device));
  GasRecord& g = ctx->gas[gas];
  if (attributes) g.attributes = attributes;
  g.generation++;
  ctx->gasEpoch++;
  if (int rc = refit_gas_gpu(ctx, g)) return rc;
  return write_gas_table(ctx, gas);
}

int rtc_gas_rebuild(rtc_context* ctx, uint32_t gas, uint64_t attributes)
{
  if (gas >= ctx->gas.size() || ctx->gas[gas].d_nodes == nullptr) RTC_FAIL("bad gas handle");
  RTC_CUDA(cudaSetDevice(ctx->device));
  GasRecord& g = ctx->gas[gas];
  if (attributes) g.attributes = attributes;
  g.generation++;
  ctx->gasEpoch++;
  if (int rc = rebuild_gas_gpu(ctx, g)) return rc;
  return write_gas_table(ctx, gas);
}

// A GAS whose triangle set rtc_gas_build_device replaces in place: node array, triangle records, refit scratch, LBVH arrays and
// collapse graph for `capacity` triangles, allocated now; no triangle yet (the empty node of rtc_gas_build for none).
int rtc_gas_create(rtc_context* ctx, uint32_t capacity, uint32_t* gas)
{
  if (!gas) RTC_FAIL("gas is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  const double t0 = now_ms();
  GasRecord rec;
  rec.capacity = capacity ? capacity : 1u;
  rec.strideBytes = 12;
  rec.builder = RTC_BUILD_GPU_LBVH;
  RTC_CUDA(cudaMalloc(&rec.d_tris, (size_t)rec.capacity * 3u * sizeof(float4)));
  int rc = create_gas_gpu(ctx, rec, rec.capacity);
  if (rc == 0) { const cudaError_t e = cudaStreamSynchronize(ctx->stream); if (e != cudaSuccess) rc = rtc_set_error(__FILE__, __LINE__, "rtc_gas_create", (int)e, cudaGetErrorString(e)); }
  if (rc)
  {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(rec.d_nodes); cudaFree(rec.d_tris); free_refit_scratch(rec.refit, ctx->stream); free_lbvh_rebuild(rec.rebuild);
    cudaGetLastError();
    return rc;
  }
  rec.numNodes = 1;
  rec.buildMs = now_ms() - t0;
  ctx->gas.push_back(rec);
  *gas = (uint32_t)(ctx->gas.size() - 1);
  return write_gas_table(ctx, *gas);
}

int rtc_gas_build_device(rtc_context* ctx, uint32_t gas, uint64_t attributes, uint32_t strideBytes, uint32_t numVerts,
                         uint64_t indices, uint32_t numTris)
{
  if (gas >= ctx->gas.size() || ctx->gas[gas].d_nodes == nullptr) RTC_FAIL("bad gas handle");
  GasRecord& g = ctx->gas[gas];
  if (!g.capacity) RTC_FAIL("rtc_gas_build_device needs a GAS of rtc_gas_create (this one was built by rtc_gas_build)");
  if (numTris > g.capacity) RTC_FAIL("numTris exceeds the GAS's capacity");
  if (strideBytes < 12 || (strideBytes & 3u)) RTC_FAIL("vertex stride must be a multiple of 4 and at least 12");
  if (attributes & 3u) RTC_FAIL("attributes is not 4-byte aligned");
  if (indices & 3u) RTC_FAIL("indices is not 4-byte aligned");
  if (numTris && (!attributes || !indices)) RTC_FAIL("attributes or indices is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  const double t0 = now_ms();
  // the triangle totals of the scenes of rtc_ias_build that instance it (created scenes count theirs from the GAS records)
  for (SceneRecord* s : ctx->scenes)
    for (const std::pair<uint32_t, uint64_t>& e : s->gasGeneration)
      if (e.first == gas) s->totalTris = s->totalTris - g.numTris + numTris;
  g.attributes = attributes; g.indices = indices; g.strideBytes = strideBytes; g.numVerts = numVerts; g.numTris = numTris;
  g.generation++;
  ctx->gasEpoch++;
  if (int rc = rebuild_gas_gpu(ctx, g)) return rc;
  g.buildMs = now_ms() - t0;
  return write_gas_table(ctx, gas);
}

int rtc_gas_rejected_triangles(rtc_context* ctx, uint32_t gas, uint32_t* count)
{
  if (gas >= ctx->gas.size() || ctx->gas[gas].d_nodes == nullptr) RTC_FAIL("bad gas handle");
  if (!count) RTC_FAIL("count is null");
  *count = 0;
  const GasRecord& g = ctx->gas[gas];
  if (!g.d_rejected || !g.numTris) return 0;      // rtc_gas_build checked every index
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaMemcpyAsync(count, g.d_rejected, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Instance level (replaces createInstance + optixAccelBuild INSTANCES + createHitGroupRecords,
// Device.cpp:1427-1532).  Single-level instancing, as the reference's pipeline (Device.cpp:560).
// ------------------------------------------------------------------------------------------------
int rtc_ias_build(rtc_context* ctx, const rtc_instance_desc* instances, uint32_t numInstances, uint64_t* topObject)
{
  if (!topObject) RTC_FAIL("topObject is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  const double t0 = now_ms();
  std::vector<float4> o2w((size_t)numInstances * 3u);
  std::vector<rt_GeometryInstanceData> gi(numInstances);
  SceneRecord* rec = new SceneRecord();
  rec->instGas.resize(numInstances);
  std::set<uint32_t> distinct;
  for (uint32_t i = 0; i < numInstances; ++i)
  {
    const rtc_instance_desc& d = instances[i];
    if (d.instanceId != i) { delete rec; RTC_FAIL("instanceId must equal the array position"); }
    if (d.gas >= ctx->gas.size() || ctx->gas[d.gas].d_nodes == nullptr) { delete rec; RTC_FAIL("bad gas handle in instance"); }
    distinct.insert(d.gas);
    rec->instGas[i] = d.gas;
    for (int r = 0; r < 3; ++r)
      o2w[3u * i + r] = make_float4(d.transform[4 * r], d.transform[4 * r + 1], d.transform[4 * r + 2], d.transform[4 * r + 3]);
    gi[i].indices = ctx->gas[d.gas].indices; gi[i].materialIndex = d.materialIndex; gi[i].lightIndex = d.lightIndex;
  }
  rec->numGas = (uint32_t)distinct.size();
  for (uint32_t g : distinct)
  {
    if (int rc = sync_gas_node_count(ctx, g)) { delete rec; return rc; }
    rec->totalNodes += ctx->gas[g].numNodes; rec->totalTris += ctx->gas[g].numTris; rec->gasBuildMs += ctx->gas[g].buildMs;
    rec->gasGeneration.emplace_back(g, ctx->gas[g].generation);
  }
  // the instance -> GAS table entry of the instance records (the position of the GAS in gasGeneration, which follows `distinct`)
  std::vector<uint32_t> slot(numInstances);
  for (uint32_t i = 0; i < numInstances; ++i) slot[i] = (uint32_t)std::distance(distinct.begin(), distinct.find(rec->instGas[i]));
  rec->instFlags.assign(numInstances, 0u);

  auto alloc = [](void** dst, size_t bytes) { return cudaMalloc(dst, bytes ? bytes : 16); };
  // stream-ordered: the kernels that write the instance records read what is staged here
  auto upload = [&](void** dst, const void* src, size_t bytes) -> cudaError_t {
    cudaError_t e = alloc(dst, bytes);
    if (e != cudaSuccess) return e;
    return bytes ? cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream) : cudaSuccess;
  };
  cudaError_t e = cudaSuccess;
  if (e == cudaSuccess) e = alloc(&rec->d_instances, (size_t)numInstances * 4u * sizeof(float4));
  if (e == cudaSuccess) e = upload(&rec->d_o2w, o2w.data(), o2w.size() * sizeof(float4));
  if (e == cudaSuccess) e = upload(&rec->d_geomInst, gi.data(), gi.size() * sizeof(rt_GeometryInstanceData));
  if (e == cudaSuccess) e = upload(&rec->d_instFlags, rec->instFlags.data(), rec->instFlags.size() * 4u);
  if (e == cudaSuccess) e = alloc((void**)&rec->d_instBoxes, (size_t)numInstances * sizeof(PrimBox));
  if (e == cudaSuccess) e = upload((void**)&rec->d_instGasSlot, slot.data(), slot.size() * 4u);
  if (e != cudaSuccess) { free_scene(rec, ctx->stream); return rtc_set_error(__FILE__, __LINE__, "rtc_ias_build upload", (int)e, cudaGetErrorString(e)); }
  // Every instance's records from the object->world rows staged above; the instance level is built on the host over the boxes
  // they hold.  RTC_INSTANCE_BOUNDS=box bounds the eight transformed corners of the GAS box instead of the transformed vertices.
  std::vector<PrimBox> boxes(numInstances);
  if (numInstances)
  {
    if (int rc = write_instance_records_gpu(ctx, *rec, static_cast<const uint8_t*>(rec->d_o2w), 48u, 0u, numInstances, {},
                                            gas_update_inputs(ctx, rec), instance_bounds_tight()))
    {
      free_scene(rec, ctx->stream);
      return rc;
    }
    e = cudaMemcpyAsync(boxes.data(), rec->d_instBoxes, boxes.size() * sizeof(PrimBox), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { free_scene(rec, ctx->stream); return rtc_set_error(__FILE__, __LINE__, "rtc_ias_build instance boxes", (int)e, cudaGetErrorString(e)); }
  }
  WideBvh bvh;
  tlas_build_host(boxes.data(), numInstances, bvh);

  if (e == cudaSuccess) e = upload(&rec->d_tlasNodes, bvh.nodes.data(), bvh.nodes.size() * sizeof(Node8));
  if (e == cudaSuccess) e = upload(&rec->d_tlasLeaves, bvh.primOrder.data(), bvh.primOrder.size() * 4u);
  rec->desc.instFlags = (const uint32_t*)rec->d_instFlags;
  rec->desc.tlasNodes = (const uint4*)rec->d_tlasNodes;
  rec->desc.tlasLeaves = (const uint32_t*)rec->d_tlasLeaves;
  rec->desc.instances = (const float4*)rec->d_instances;
  rec->desc.objectToWorld = (const float4*)rec->d_o2w;
  rec->desc.geomInst = (const rt_GeometryInstanceData*)rec->d_geomInst;
  rec->desc.numInstances = numInstances;
  rec->desc.numTlasNodes = (uint32_t)bvh.nodes.size();
  rec->desc.numTlasLeaves = (uint32_t)bvh.primOrder.size();
  if (e == cudaSuccess) e = upload((void**)&rec->d_desc, &rec->desc, sizeof(SceneDesc));
  if (e != cudaSuccess) { free_scene(rec, ctx->stream); return rtc_set_error(__FILE__, __LINE__, "rtc_ias_build upload", (int)e, cudaGetErrorString(e)); }
  rec->totalNodes += bvh.nodes.size();
  rec->iasBuildMs = now_ms() - t0;
  ctx->scenes.push_back(rec);
  *topObject = (uint64_t)(uintptr_t)rec->d_desc;
  return 0;
}

int rtc_ias_update(rtc_context* ctx, uint64_t topObject, uint32_t first, uint32_t count, const float* transforms)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  const uint32_t n = s->desc.numInstances;
  if ((uint64_t)first + count > n) RTC_FAIL("instance range out of bounds");
  if (count && !transforms) RTC_FAIL("transforms is null");
  if (const char* why = scene_unusable(ctx, s, true)) RTC_FAIL(why);
  RTC_CUDA(cudaSetDevice(ctx->device));
  // The device path on a stream-ordered device copy of the matrices, freed behind the update.  `transforms` may be reused on
  // return, so the call must have read it by then.  A copy from pageable memory is staged before cudaMemcpyAsync returns; one
  // from page-locked memory (rtc_host_alloc, cudaHostRegister, pinned tensors) or managed memory reads it only when the stream
  // gets there, so such a source is first copied into pageable memory of the library's.
  const float* src = transforms;
  std::vector<float> pageable;
  if (count)
  {
    cudaPointerAttributes attr{};
    if (cudaPointerGetAttributes(&attr, transforms) != cudaSuccess) { cudaGetLastError(); attr.type = cudaMemoryTypeUnregistered; }
    if (attr.type == cudaMemoryTypeDevice) RTC_FAIL("transforms is device memory: use rtc_ias_update_device");
    if (attr.type != cudaMemoryTypeUnregistered) { pageable.assign(transforms, transforms + (size_t)count * 12u); src = pageable.data(); }
  }
  uint8_t* staged = nullptr;
  if (count)
  {
    RTC_CUDA(cudaMallocAsync((void**)&staged, (size_t)count * 48u, ctx->stream));
    const cudaError_t e = cudaMemcpyAsync(staged, src, (size_t)count * 48u, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) { cudaFreeAsync(staged, ctx->stream); return rtc_set_error(__FILE__, __LINE__, "rtc_ias_update upload", (int)e, cudaGetErrorString(e)); }
  }
  const int rc = update_instances(ctx, s, first, count, staged, 48u);
  if (staged) cudaFreeAsync(staged, ctx->stream);
  return rc;
}

int rtc_ias_update_device(rtc_context* ctx, uint64_t topObject, uint32_t first, uint32_t count, uint64_t transforms, uint32_t strideBytes)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  if ((uint64_t)first + count > s->desc.numInstances) RTC_FAIL("instance range out of bounds");
  if (count && !transforms) RTC_FAIL("transforms is null");
  if (count && (transforms & 3u)) RTC_FAIL("transforms is not 4-byte aligned");
  if (strideBytes < 48 || (strideBytes & 3u)) RTC_FAIL("strideBytes must be a multiple of 4 and at least 48");
  if (const char* why = scene_unusable(ctx, s, true)) RTC_FAIL(why);
  RTC_CUDA(cudaSetDevice(ctx->device));
  return update_instances(ctx, s, first, count, reinterpret_cast<const uint8_t*>((uintptr_t)transforms), strideBytes);
}

int rtc_ias_rebuild(rtc_context* ctx, uint64_t topObject)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  if (const char* why = scene_unusable(ctx, s)) RTC_FAIL(why);
  RTC_CUDA(cudaSetDevice(ctx->device));
  return rebuild_instances_gpu(ctx, *s);
}

// A created scene's GAS totals from the device's per-handle reference counts.  Synchronises the stream.
int sync_created_scene_totals(rtc_context* ctx, SceneRecord* s)
{
  std::vector<uint32_t> refs(s->gasRefsCount);
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  if (!refs.empty()) RTC_CUDA(cudaMemcpy(refs.data(), s->d_gasRefs, refs.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  s->numGas = 0; s->totalNodes = s->desc.numTlasNodes; s->totalTris = 0; s->gasBuildMs = 0.0;
  for (uint32_t h = 0; h < refs.size(); ++h)
  {
    if (!refs[h] || !ctx->gas[h].d_nodes) continue;
    if (int rc = sync_gas_node_count(ctx, h)) return rc;
    const GasRecord& g = ctx->gas[h];
    s->numGas++; s->totalNodes += g.numNodes; s->totalTris += g.numTris; s->gasBuildMs += g.buildMs;
  }
  return 0;
}

int rtc_ias_create(rtc_context* ctx, uint32_t capacity, uint64_t* topObject)
{
  if (!topObject) RTC_FAIL("topObject is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  SceneRecord* s = new SceneRecord();
  s->created = true;
  s->capacity = capacity;
  s->instFlags.assign(capacity, 0u);
  const size_t cap = capacity ? capacity : 1u;
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void** dst, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(dst, bytes); };
  alloc((void**)&s->d_desc, sizeof(SceneDesc));
  alloc(&s->d_instances, cap * 4u * sizeof(float4));
  alloc(&s->d_tlasLeaves, cap * sizeof(uint32_t));
  alloc(&s->d_o2w, cap * 3u * sizeof(float4));
  alloc(&s->d_geomInst, cap * sizeof(rt_GeometryInstanceData));
  alloc(&s->d_instFlags, cap * sizeof(uint32_t));
  alloc((void**)&s->d_instBoxes, cap * sizeof(PrimBox));
  alloc((void**)&s->d_instGasSlot, cap * sizeof(uint32_t));
  alloc((void**)&s->d_instGen, cap * sizeof(uint64_t));
  alloc((void**)&s->d_words, kSceneWords * sizeof(uint32_t));
  alloc(&s->d_emptyGas, sizeof(Node8) + 3u * sizeof(float4));
  // the empty GAS of rejected records: every slot of its root empty (imask 0, meta 0)
  if (e == cudaSuccess) e = cudaMemsetAsync(s->d_emptyGas, 0, sizeof(Node8) + 3u * sizeof(float4), ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(s->d_instFlags, 0, cap * sizeof(uint32_t), ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(s->d_words, 0, kSceneWords * sizeof(uint32_t), ctx->stream);
  if (e != cudaSuccess) { free_scene(s, ctx->stream); return rtc_set_error(__FILE__, __LINE__, "rtc_ias_create", (int)e, cudaGetErrorString(e)); }
  s->desc.instFlags = (const uint32_t*)s->d_instFlags;
  s->desc.tlasLeaves = (const uint32_t*)s->d_tlasLeaves;
  s->desc.instances = (const float4*)s->d_instances;
  s->desc.objectToWorld = (const float4*)s->d_o2w;
  s->desc.geomInst = (const rt_GeometryInstanceData*)s->d_geomInst;
  s->desc.numInstances = 0; s->desc.numTlasLeaves = 0; s->desc.numTlasNodes = 1;
  // the node array, refit scratch, LBVH arrays and collapse graph for the capacity; the one empty root node of no instances
  if (int rc = create_instance_level_gpu(ctx, *s, capacity)) { cudaStreamSynchronize(ctx->stream); free_scene(s, ctx->stream); return rc; }
  e = cudaMemcpyAsync(s->d_desc, &s->desc, sizeof(SceneDesc), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) { free_scene(s, ctx->stream); return rtc_set_error(__FILE__, __LINE__, "rtc_ias_create", (int)e, cudaGetErrorString(e)); }
  s->totalNodes = 1;
  s->gasEpoch = ctx->gasEpoch;
  ctx->scenes.push_back(s);
  *topObject = (uint64_t)(uintptr_t)s->d_desc;
  return 0;
}

int rtc_ias_build_device(rtc_context* ctx, uint64_t topObject, uint64_t instances, uint32_t strideBytes, uint32_t numInstances)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  if (!s->created) RTC_FAIL("rtc_ias_build_device needs a scene of rtc_ias_create (this one was built by rtc_ias_build)");
  if (numInstances > s->capacity) RTC_FAIL("numInstances exceeds the scene's capacity");
  if (numInstances && !instances) RTC_FAIL("instances is null");
  if (numInstances && (instances & 3u)) RTC_FAIL("instances is not 4-byte aligned");
  if (numInstances && (strideBytes < 64 || (strideBytes & 3u))) RTC_FAIL("strideBytes must be a multiple of 4 and at least 64");
  RTC_CUDA(cudaSetDevice(ctx->device));
  const double t0 = now_ms();
  // the per-handle reference counts cover every handle of the context (pooled, grown behind the stream)
  const uint32_t numGas = (uint32_t)ctx->gas.size();
  if (numGas > s->gasRefsCapacity)
  {
    if (s->d_gasRefs) RTC_CUDA(cudaFreeAsync(s->d_gasRefs, ctx->stream));
    s->d_gasRefs = nullptr; s->gasRefsCapacity = 0; s->gasRefsCount = 0;
    const uint32_t cap = std::max(numGas, ctx->gasTableCapacity);
    RTC_CUDA(cudaMallocAsync((void**)&s->d_gasRefs, (size_t)cap * sizeof(uint32_t), ctx->stream));
    s->gasRefsCapacity = cap;
  }
  s->gasRefsCount = numGas;
  if (numGas) RTC_CUDA(cudaMemsetAsync(s->d_gasRefs, 0, (size_t)numGas * sizeof(uint32_t), ctx->stream));
  RTC_CUDA(cudaMemsetAsync(s->d_words + kRejectedWord, 0, sizeof(uint32_t), ctx->stream));
  s->desc.numInstances = numInstances;
  s->desc.numTlasLeaves = numInstances;
  RTC_CUDA(cudaMemcpyAsync(s->d_desc, &s->desc, sizeof(SceneDesc), cudaMemcpyHostToDevice, ctx->stream));
  if (int rc = write_created_records_gpu(ctx, *s, reinterpret_cast<const uint8_t*>((uintptr_t)instances), nullptr, strideBytes, 0u, 0u,
                                         instance_bounds_tight())) return rc;
  if (int rc = rebuild_instances_gpu(ctx, *s)) return rc;
  count_cutout(s);
  s->gasEpoch = ctx->gasEpoch;
  s->gasDestroyed = false;
  s->iasBuildMs = now_ms() - t0;
  return 0;
}

int rtc_scene_rejected_instances(rtc_context* ctx, uint64_t topObject, uint32_t* count)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  if (!count) RTC_FAIL("count is null");
  if (!s->created) RTC_FAIL("not a scene of rtc_ias_create");
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaMemcpyAsync(count, s->d_words + kRejectedWord, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int rtc_scene_info_get(rtc_context* ctx, uint64_t topObject, rtc_scene_info* info)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  RTC_CUDA(cudaSetDevice(ctx->device));
  if (int rc = sync_tlas_node_count(ctx, s)) return rc;
  if (s->created) { if (int rc = sync_created_scene_totals(ctx, s)) return rc; }
  for (const std::pair<uint32_t, uint64_t>& g : s->gasGeneration) if (int rc = sync_gas_node_count(ctx, g.first)) return rc;
  std::memset(info, 0, sizeof(*info));
  info->numNodes = s->totalNodes; info->numTris = s->totalTris; info->numInstances = s->desc.numInstances;
  info->numTlasNodes = s->desc.numTlasNodes; info->numTlasLeaves = s->desc.numTlasLeaves; info->numGas = s->numGas; info->gasBuildMs = s->gasBuildMs; info->iasBuildMs = s->iasBuildMs;
  return 0;
}

int rtc_scene_destroy(rtc_context* ctx, uint64_t topObject)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  for (size_t i = 0; i < ctx->scenes.size(); ++i)
    if ((uint64_t)(uintptr_t)ctx->scenes[i]->d_desc == topObject)
    {
      RTC_CUDA(cudaStreamSynchronize(ctx->stream));
      release_cutout_graph(ctx);          // it may have captured this scene's tables; a later scene can get the same addresses
      free_scene(ctx->scenes[i], ctx->stream);
      ctx->scenes.erase(ctx->scenes.begin() + (long)i);
      return 0;
    }
  RTC_FAIL("unknown topObject");
}

// Per-instance hit-record selection (Device.cpp:1503-1513; updateMaterial :1141-1160 rewrites the SBT headers).
int rtc_scene_set_instance_flags(rtc_context* ctx, uint64_t topObject, uint32_t first, uint32_t count, const uint32_t* flags)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  // a created scene's flags belong to positions up to its capacity and persist across its builds
  if ((uint64_t)first + count > (s->created ? s->capacity : s->desc.numInstances)) RTC_FAIL("instance range out of bounds");
  if (count == 0) return 0;
  if (!flags) RTC_FAIL("flags is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  for (uint32_t i = 0; i < count; ++i) s->instFlags[first + i] = flags[i];
  count_cutout(s);
  // stream-ordered behind the launches already enqueued; `flags` may be reused by the caller at once (pageable source: staged copy)
  RTC_CUDA(cudaMemcpyAsync((uint32_t*)s->d_instFlags + first, &s->instFlags[first], (size_t)count * 4u, cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}

int rtc_scene_set_albedo_textures(rtc_context* ctx, uint64_t topObject, int enable)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  s->albedoTextures = enable != 0;
  return 0;
}

// Material textures: 16-byte header {width, height, 0, 0} + RGBA32F texels in one allocation; the handle is its address.
int rtc_texture_create(rtc_context* ctx, uint32_t width, uint32_t height, const float* rgba, uint64_t* handle)
{
  if (!handle) RTC_FAIL("handle is null");
  if (width == 0 || height == 0 || !rgba) RTC_FAIL("empty texture");
  RTC_CUDA(cudaSetDevice(ctx->device));
  const size_t texelBytes = (size_t)width * height * 16u;
  void* d = nullptr;
  RTC_CUDA(cudaMalloc(&d, 16u + texelBytes));
  const uint32_t header[4] = { width, height, 0u, 0u };
  cudaError_t e = cudaMemcpy(d, header, 16u, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy((char*)d + 16, rgba, texelBytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(d); return rtc_set_error(__FILE__, __LINE__, "rtc_texture_create upload", (int)e, cudaGetErrorString(e)); }
  ctx->textures.push_back(d);
  *handle = (uint64_t)(uintptr_t)d;
  return 0;
}

int rtc_texture_destroy(rtc_context* ctx, uint64_t handle)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  for (size_t i = 0; i < ctx->textures.size(); ++i)
    if ((uint64_t)(uintptr_t)ctx->textures[i] == handle)
    {
      RTC_CUDA(cudaStreamSynchronize(ctx->stream));
      RTC_CUDA(cudaFree(ctx->textures[i]));
      ctx->textures.erase(ctx->textures.begin() + (long)i);
      return 0;
    }
  RTC_FAIL("unknown texture handle");
}

int rtc_scene_export(rtc_context* ctx, uint64_t topObject, void* tlasNodes, uint32_t* tlasLeaves, float* worldToObject, uint32_t* instanceGas)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  if (int rc = sync_tlas_node_count(ctx, s)) return rc;
  if (tlasNodes) RTC_CUDA(cudaMemcpy(tlasNodes, s->d_tlasNodes, (size_t)s->desc.numTlasNodes * sizeof(Node8), cudaMemcpyDeviceToHost));
  if (tlasLeaves && s->desc.numTlasLeaves) RTC_CUDA(cudaMemcpy(tlasLeaves, s->d_tlasLeaves, (size_t)s->desc.numTlasLeaves * 4u, cudaMemcpyDeviceToHost));
  // world->object rows 0..2 of each 64-byte instance record, where the updates computed them
  if (worldToObject && s->desc.numInstances)
    RTC_CUDA(cudaMemcpy2D(worldToObject, 48, s->d_instances, 64, 48, s->desc.numInstances, cudaMemcpyDeviceToHost));
  if (instanceGas && s->created && s->desc.numInstances)
    RTC_CUDA(cudaMemcpy(instanceGas, s->d_instGasSlot, (size_t)s->desc.numInstances * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  else if (instanceGas) std::memcpy(instanceGas, s->instGas.data(), s->instGas.size() * sizeof(uint32_t));
  return 0;
}

int rtc_gas_info(rtc_context* ctx, uint32_t gas, uint64_t* numNodes, uint64_t* numTris)
{
  if (gas >= ctx->gas.size() || ctx->gas[gas].d_nodes == nullptr) RTC_FAIL("bad gas handle");
  if (ctx->gas[gas].d_numNodes)
  {
    RTC_CUDA(cudaSetDevice(ctx->device));
    if (int rc = sync_gas_node_count(ctx, gas)) return rc;
  }
  if (numNodes) *numNodes = ctx->gas[gas].numNodes;
  if (numTris) *numTris = ctx->gas[gas].numTris;
  return 0;
}

int rtc_gas_export(rtc_context* ctx, uint32_t gas, void* nodes, float* tris)
{
  if (gas >= ctx->gas.size() || ctx->gas[gas].d_nodes == nullptr) RTC_FAIL("bad gas handle");
  const GasRecord& g = ctx->gas[gas];
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  if (int rc = sync_gas_node_count(ctx, gas)) return rc;
  if (nodes) RTC_CUDA(cudaMemcpy(nodes, g.d_nodes, (size_t)g.numNodes * sizeof(Node8), cudaMemcpyDeviceToHost));
  if (tris && g.numTris) RTC_CUDA(cudaMemcpy(tris, g.d_tris, (size_t)g.numTris * 12u * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

int rtc_instance_inverse(rtc_context* ctx, uint64_t topObject, uint32_t instance, float out[12])
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  if (instance >= s->desc.numInstances) RTC_FAIL("instance out of range");
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaMemcpyAsync(out, static_cast<const float4*>(s->d_instances) + 4u * (size_t)instance, 48, cudaMemcpyDeviceToHost, ctx->stream));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Launches
// ------------------------------------------------------------------------------------------------
int rtc_launch(rtc_context* ctx, const rt_SystemData* sys, uint32_t launchWidth, uint32_t launchHeight,
               int raygen, int miss, int iterationFirst, int iterationCount)
{
  if (!sys) RTC_FAIL("sys is null");
  if (raygen != RTC_RAYGEN_FULL_FRAME && raygen != RTC_RAYGEN_LOCAL_COPY) RTC_FAIL("bad raygen selector");
  if (miss < RT_MISS_NULL || miss > RT_MISS_SPHERE) RTC_FAIL("bad miss selector");
  if (miss == RT_MISS_SPHERE && (sys->envTexture == 0 || sys->envCDF_U == 0 || sys->envCDF_V == 0)) RTC_FAIL("miss 2 needs envTexture/envCDF_U/envCDF_V");
  if (const SceneRecord* s = find_scene(ctx, sys->topObject)) { if (const char* why = scene_unusable(ctx, s)) RTC_FAIL(why); }
  RTC_CUDA(cudaSetDevice(ctx->device));
  return launch_wavefront(ctx, *sys, launchWidth, launchHeight, raygen, miss, iterationFirst, iterationCount, iterationFirst, false);
}

int rtc_launch_ex(rtc_context* ctx, const rt_SystemData* sys, uint32_t launchWidth, uint32_t launchHeight,
                  int raygen, int miss, int iterationFirst, int iterationCount, int accumulationFirst, int countWork)
{
  if (!sys) RTC_FAIL("sys is null");
  if (raygen != RTC_RAYGEN_FULL_FRAME && raygen != RTC_RAYGEN_LOCAL_COPY) RTC_FAIL("bad raygen selector");
  if (miss < RT_MISS_NULL || miss > RT_MISS_SPHERE) RTC_FAIL("bad miss selector");
  if (miss == RT_MISS_SPHERE && (sys->envTexture == 0 || sys->envCDF_U == 0 || sys->envCDF_V == 0)) RTC_FAIL("miss 2 needs envTexture/envCDF_U/envCDF_V");
  if (accumulationFirst < 0) RTC_FAIL("accumulationFirst < 0");
  if (const SceneRecord* s = find_scene(ctx, sys->topObject)) { if (const char* why = scene_unusable(ctx, s)) RTC_FAIL(why); }
  RTC_CUDA(cudaSetDevice(ctx->device));
  return launch_wavefront(ctx, *sys, launchWidth, launchHeight, raygen, miss, iterationFirst, iterationCount, accumulationFirst, countWork != 0);
}

int rtc_trace_schedule_get(rtc_context* ctx, rtc_trace_schedule* out)
{
  if (!out) RTC_FAIL("out is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  tuner_finish(ctx);        // a pending decision is taken now (waits for the last timed batch)
  const ScheduleTuner& t = ctx->tuner;
  out->schedule = ctx->traceSchedule;
  out->decided = t.state == ScheduleTuner::DONE ? 1 : 0;
  out->measured = (t.state == ScheduleTuner::DONE && t.ms[1] > 0.0f) ? 1 : 0;
  out->pathsPerBatch = t.paths;
  out->groupMs[0] = t.ms[0]; out->oneTriMs = t.ms[1]; out->twoTriMs = t.ms[2]; out->groupMs[1] = t.ms[3];
  return 0;
}

int rtc_trace_schedule_set(rtc_context* ctx, int schedule)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  if (schedule == RTC_SCHEDULE_GROUP || schedule == RTC_SCHEDULE_ONE_TRI || schedule == RTC_SCHEDULE_TWO_TRI)
  {
    ctx->traceSchedule = schedule;
    ctx->tuner.state = ScheduleTuner::DONE;
    return 0;
  }
  if (schedule != -1) RTC_FAIL("schedule must be one of RTC_SCHEDULE_* or -1 (measure again)");
  ctx->traceSchedule = RTC_SCHEDULE_GROUP;
  ctx->tuner.state = ScheduleTuner::WARMUP;
  ctx->tuner.slot = 0; ctx->tuner.restarts = 0; ctx->tuner.paths = 0;
  for (float& ms : ctx->tuner.ms) ms = 0.0f;
  return 0;
}

int rtc_launch_counts_get(rtc_context* ctx, rtc_trace_counts out[2])
{
  if (!out) RTC_FAIL("out is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  unsigned long long h[2 * kTraceCountWords];
  RTC_CUDA(cudaMemcpyAsync(h, ctx->d_launchCounts, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < 2; ++k)
  {
    const unsigned long long* c = h + kTraceCountWords * k;
    out[k].nodes = c[0]; out[k].tris = c[1]; out[k].instances = c[2]; out[k].rays = c[3];
  }
  return 0;
}

int rtc_launch_counts_reset(rtc_context* ctx)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaMemsetAsync(ctx->d_launchCounts, 0, 2 * kTraceCountWords * sizeof(unsigned long long), ctx->stream));
  return 0;
}

int rtc_timer_start(rtc_context* ctx)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaEventRecord(ctx->evTimerA, ctx->stream));
  return 0;
}

int rtc_timer_stop(rtc_context* ctx, float* milliseconds)
{
  if (!milliseconds) RTC_FAIL("milliseconds is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaEventRecord(ctx->evTimerB, ctx->stream));
  RTC_CUDA(cudaEventSynchronize(ctx->evTimerB));
  RTC_CUDA(cudaEventElapsedTime(milliseconds, ctx->evTimerA, ctx->evTimerB));
  return 0;
}

static int profile_resolve(rtc_context* ctx)
{
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  for (rtc_context::ProfileSpan& sp : ctx->spans)
  {
    float ms = 0.0f;
    RTC_CUDA(cudaEventElapsedTime(&ms, sp.a, sp.b));
    ctx->profile.ms[sp.cls] += ms;
    ctx->profile.launches[sp.cls] += 1;
    ctx->eventPool.push_back(sp.a); ctx->eventPool.push_back(sp.b);
  }
  ctx->spans.clear();
  return 0;
}

int rtc_profile_enable(rtc_context* ctx, int enable)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  if (int rc = profile_resolve(ctx)) return rc;
  if (enable) std::memset(&ctx->profile, 0, sizeof(ctx->profile));
  ctx->profiling = enable != 0;
  return 0;
}

int rtc_profile_get(rtc_context* ctx, rtc_profile* out)
{
  if (!out) RTC_FAIL("out is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  if (int rc = profile_resolve(ctx)) return rc;
  *out = ctx->profile;
  return 0;
}

int rtc_trace_closest(rtc_context* ctx, uint64_t topObject, uint64_t rays, uint64_t numRays, uint64_t hits)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  if (const char* why = scene_unusable(ctx, s)) RTC_FAIL(why);
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaEventRecord(ctx->evA, ctx->stream));
  if (int rc = launch_trace_closest(ctx, &s->desc, (const rtc_ray*)(uintptr_t)rays, numRays, (rtc_hit*)(uintptr_t)hits)) return rc;
  RTC_CUDA(cudaEventRecord(ctx->evB, ctx->stream));
  ctx->traceTimed = true;
  return 0;
}

int rtc_trace_any(rtc_context* ctx, uint64_t topObject, uint64_t rays, uint64_t numRays, uint64_t occluded)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  if (const char* why = scene_unusable(ctx, s)) RTC_FAIL(why);
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaEventRecord(ctx->evA, ctx->stream));
  if (int rc = launch_trace_any(ctx, &s->desc, (const rtc_ray*)(uintptr_t)rays, numRays, (uint32_t*)(uintptr_t)occluded)) return rc;
  RTC_CUDA(cudaEventRecord(ctx->evB, ctx->stream));
  ctx->traceTimed = true;
  return 0;
}

int rtc_trace_count(rtc_context* ctx, uint64_t topObject, uint64_t rays, uint64_t numRays, int anyHit, rtc_trace_counts* out)
{
  SceneRecord* s = find_scene(ctx, topObject);
  if (!s) RTC_FAIL("unknown topObject");
  if (!out) RTC_FAIL("out is null");
  if (const char* why = scene_unusable(ctx, s)) RTC_FAIL(why);
  RTC_CUDA(cudaSetDevice(ctx->device));
  unsigned long long* d = ctx->d_launchCounts + 2 * kTraceCountWords;
  RTC_CUDA(cudaMemsetAsync(d, 0, kTraceCountWords * sizeof(uint64_t), ctx->stream));
  if (int rc = launch_trace_count(ctx, &s->desc, (const rtc_ray*)(uintptr_t)rays, numRays, anyHit, d)) return rc;
  uint64_t h[4];
  RTC_CUDA(cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  out->nodes = h[0]; out->tris = h[1]; out->instances = h[2]; out->rays = h[3];
  return 0;
}

int rtc_generate_primary(rtc_context* ctx, const rt_SystemData* sys, uint32_t launchWidth, uint32_t launchHeight,
                         int iteration, uint64_t rays)
{
  if (!sys) RTC_FAIL("sys is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  return launch_generate_primary(ctx, *sys, launchWidth, launchHeight, iteration, (rtc_ray*)(uintptr_t)rays);
}

int rtc_composite(rtc_context* ctx, const rt_CompositorData* args)
{
  if (!args) RTC_FAIL("args is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  return launch_composite(ctx, *args);
}

int rtc_tonemap(rtc_context* ctx, const rt_TonemapperParams* params, uint64_t rgba, uint64_t rgb8, uint64_t numPixels)
{
  if (!params) RTC_FAIL("params is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  return launch_tonemap(ctx, *params, (const float4*)(uintptr_t)rgba, (uint8_t*)(uintptr_t)rgb8, numPixels);
}

int rtc_probe_math(rtc_context* ctx, int fn, const float* x, const float* y, float* out, uint32_t n)
{
  if (!ctx || !x || !y || !out) RTC_FAIL("null argument");
  if (fn < 0 || fn >= RTC_MATH_COUNT) RTC_FAIL("unknown function");
  if (n == 0) return 0;
  RTC_CUDA(cudaSetDevice(ctx->device));
  float* d = nullptr;
  RTC_CUDA(cudaMalloc(&d, (size_t)n * 3 * sizeof(float)));
  const bool ok = cudaMemcpyAsync(d, x, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream) == cudaSuccess &&
                  cudaMemcpyAsync(d + n, y, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream) == cudaSuccess &&
                  launch_probe_math(ctx, fn, d, d + n, d + 2 * (size_t)n, n) == 0 &&
                  cudaMemcpyAsync(out, d + 2 * (size_t)n, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream) == cudaSuccess &&
                  cudaStreamSynchronize(ctx->stream) == cudaSuccess;
  cudaFree(d);
  if (!ok) RTC_FAIL("device error");
  return 0;
}

int rtc_stats_get(rtc_context* ctx, rtc_stats* out)
{
  if (!out) RTC_FAIL("out is null");
  RTC_CUDA(cudaSetDevice(ctx->device));
  uint64_t h[4];
  RTC_CUDA(cudaMemcpyAsync(h, ctx->d_stats, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  if (ctx->traceTimed)
  {
    float ms = 0.0f;
    RTC_CUDA(cudaEventElapsedTime(&ms, ctx->evA, ctx->evB));
    ctx->lastTraceMs = ms;
  }
  out->radianceRays = h[0]; out->shadowRays = h[1]; out->pathSamples = h[2];
  out->kernelLaunches = ctx->kernelLaunches; out->lastTraceMs = ctx->lastTraceMs; out->cutoutGraphBuilds = ctx->cutoutGraphBuilds;
  return read_stack_overflows(ctx, &out->stackOverflows);
}

int rtc_stats_reset(rtc_context* ctx)
{
  RTC_CUDA(cudaSetDevice(ctx->device));
  RTC_CUDA(cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(uint64_t), ctx->stream));
  ctx->kernelLaunches = 0;
  ctx->cutoutGraphBuilds = 0;
  return 0;
}

} // extern "C"
