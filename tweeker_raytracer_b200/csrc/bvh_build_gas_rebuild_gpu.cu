// bvh_build_gas_rebuild_gpu.cu -- rtc_gas_rebuild and rtc_gas_build_device: a new topology for a geometry, built on the device
// from its current vertex and index buffers and written in place into its node and triangle arrays (the handle stays valid).
//
//   1. exact triangle boxes, exact min / max of their centres                    k_gas_boxes
//   2. Morton codes, sort, radix tree, fit                                        lbvh_rebuild_tail (lbvh_collapse.cuh)
//   3. collapse to 8-wide nodes, one triangle per leaf slot, level by level       k_gas_pick, k_gas_scan, k_gas_emit
//   4. triangle records in leaf order (v0.xyz | primitive id bits, v1, v2), the refit's parent index and zeroed arrival
//      counters (in k_gas_emit); the root box for the instance records            k_gas_bounds
//
// The pipeline, its deterministic bytes and its one-time synchronisation are those of lbvh_collapse.cuh, which the instance-level
// rebuild (bvh_build_ias_gpu.cu) shares.  The bytes depend only on positions and indices: the collapse reads neither the nodes
// nor the triangle records the GAS held before, so the builder that made it and earlier refits or rebuilds do not show.
//
// Every input of a build -- triangle count, vertex and index buffers, vertex count and stride -- is written by k_gas_begin into
// the words of LbvhRebuild::counters from kInput on, where the collapse graph (captured once) reads it.  So a GAS of
// rtc_gas_create, whose arrays are sized for its capacity, builds any triangle set up to it with the same graph, and
// rtc_gas_rebuild of any GAS is a build over its current buffers.  An index past the vertex records reads the vertex
// kMissingVertexBits (bvh_rules.h): its triangle is inactive, and k_gas_boxes counts it.
//
// Compiled with -fmad=false: the collapse's surface areas and slot costs (bvh_rules.h) must round like the host twin
// (rtc_host_gas_rebuild, accel_host.cpp), which is compiled with -ffp-contract=off.
#include "rtc_internal.h"
#include "bvh_rules.h"
#include "lbvh_collapse.cuh"

namespace {

// the geometry's words of LbvhRebuild::counters (counters[kInput] is the triangle count); the buffers are 8-byte aligned words
enum { kGasNumVerts = kInput + 1, kGasStride = kInput + 2, kGasRejected = kInput + 3, kGasVerts = kInput + 4, kGasIndices = kInput + 6 };
static_assert(kGasIndices + 2 <= kNumCounters && (kGasVerts & 1) == 0 && (kGasIndices & 1) == 0, "geometry input words");

struct GasInput
{
  const uint8_t* verts;
  const uint32_t* idx;
  uint32_t numVerts, stride;
};

__device__ __forceinline__ GasInput gas_input(const uint32_t* counters)
{
  GasInput in;
  in.verts = reinterpret_cast<const uint8_t*>(*reinterpret_cast<const unsigned long long*>(counters + kGasVerts));
  in.idx = reinterpret_cast<const uint32_t*>(*reinterpret_cast<const unsigned long long*>(counters + kGasIndices));
  in.numVerts = counters[kGasNumVerts]; in.stride = counters[kGasStride];
  return in;
}

// Corner c of triangle t; false for an index past the vertex records, which reads kMissingVertexBits and is never dereferenced.
__device__ __forceinline__ bool gas_vertex(const GasInput& in, uint32_t t, int c, float x[3])
{
  const uint32_t vi = __ldg(in.idx + 3u * (size_t)t + c);
  if (vi >= in.numVerts)
  {
    x[0] = x[1] = x[2] = __uint_as_float(kMissingVertexBits);
    return false;
  }
  const float* p = reinterpret_cast<const float*>(in.verts + (size_t)vi * in.stride);
  x[0] = __ldg(p); x[1] = __ldg(p + 1); x[2] = __ldg(p + 2);
  return true;
}

// One thread per triangle: its exact box (the arithmetic of rtc_host_gas_rebuild), and the block's share of the centre box.
// Triangles with an index past the vertex records are counted into *rejected.
__global__ void __launch_bounds__(kLbvhBlock)
k_gas_boxes(const GasInput in, uint32_t n, float4* __restrict__ lo, float4* __restrict__ hi, float* __restrict__ centreBox,
            uint32_t* __restrict__ rejected)
{
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  float cLo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, cHi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  bool bad = false;
  if (t < n)
  {
    float bLo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, bHi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
    bool active = true;
    for (int c = 0; c < 3; ++c)
    {
      float x[3];
      bad = !gas_vertex(in, t, c, x) || bad;
      active = active && rules_in_range3(x);
      for (int k = 0; k < 3; ++k) { bLo[k] = fminf(bLo[k], x[k]); bHi[k] = fmaxf(bHi[k], x[k]); }
    }
    if (!active) rules_empty_box(bLo, bHi);
    lo[t] = make_float4(bLo[0], bLo[1], bLo[2], 0.0f);
    hi[t] = make_float4(bHi[0], bHi[1], bHi[2], 0.0f);
    if (active) for (int k = 0; k < 3; ++k) { cLo[k] = 0.5f * (bLo[k] + bHi[k]); cHi[k] = cLo[k]; }
  }
  const unsigned badLanes = __ballot_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && badLanes) atomicAdd(rejected, (uint32_t)__popc(badLanes));
  lbvh_reduce_centre_box(cLo, cHi, centreBox);
}

// The state of one build and its inputs.  No triangle: the one empty node rtc_gas_build writes for none (bvh_build_host.cpp),
// counted by collapse_begin, and the bounds (0, 0) it reports.
__global__ void k_gas_begin(float* __restrict__ centreBox, uint32_t* __restrict__ counters, int2* __restrict__ work, const GasInput in,
                            uint32_t n, uint4* __restrict__ nodes, float* __restrict__ box)
{
  collapse_begin(centreBox, counters, work);
  counters[kInput] = n;
  counters[kGasNumVerts] = in.numVerts; counters[kGasStride] = in.stride; counters[kGasRejected] = 0u;
  *reinterpret_cast<unsigned long long*>(counters + kGasVerts) = (unsigned long long)(uintptr_t)in.verts;
  *reinterpret_cast<unsigned long long*>(counters + kGasIndices) = (unsigned long long)(uintptr_t)in.idx;
  if (n == 0)
  {
    union { Node8 n; uint4 v[5]; } e;
    for (int j = 0; j < 5; ++j) e.v[j] = make_uint4(0u, 0u, 0u, 0u);
    e.n.ex = e.n.ey = e.n.ez = 127;
    for (int s = 0; s < 8; ++s) e.n.qlox[s] = e.n.qloy[s] = e.n.qloz[s] = 255;
    for (int j = 0; j < 5; ++j) nodes[j] = e.v[j];
    for (int k = 0; k < 6; ++k) box[k] = 0.0f;
  }
}

// the bounds of the GAS (the fitted box of the binary root), where the instance records read a refitted GAS's bounds
__global__ void k_gas_bounds(const float4* __restrict__ boxLo, const float4* __restrict__ boxHi, float* __restrict__ box)
{
  const float4 a = boxLo[0], b = boxHi[0];
  box[0] = a.x; box[1] = a.y; box[2] = a.z; box[3] = b.x; box[4] = b.y; box[5] = b.z;
}

__global__ void __launch_bounds__(kCollapseBlock, 4)
k_gas_pick(const CollapseArgs A, const int2* __restrict__ work, const uint32_t* __restrict__ workCount)
{
  collapse_pick(A, (int)A.counters[kInput], work, workCount);
}

__global__ void __launch_bounds__(kScanThreads)
k_gas_scan(const CollapseArgs A, const uint32_t* __restrict__ workCount, uint32_t* __restrict__ nextCount,
           cudaGraphConditionalHandle handle, int setCondition)
{
  collapse_scan(A, workCount, nextCount, handle, setCondition);
}

// the leaf slot holds the triangle record, as the builders and the refit write it
__global__ void __launch_bounds__(kCollapseBlock)
k_gas_emit(const CollapseArgs A, float4* __restrict__ tris, const int2* __restrict__ work, const uint32_t* __restrict__ workCount,
           int2* __restrict__ nextWork)
{
  collapse_emit(A, (int)A.counters[kInput], work, workCount, nextWork, [&](uint32_t slot, uint32_t p) {
    const GasInput in = gas_input(A.counters);
    const uint32_t prim = A.order[p];
    float x[3][3];
    for (int c = 0; c < 3; ++c) gas_vertex(in, prim, c, x[c]);
    float4 rec[3];
    rules_tri_record(x[0], x[1], x[2], prim, rec);
    float4* out = tris + 3u * (size_t)slot;
    for (int c = 0; c < 3; ++c) out[c] = rec[c];
  });
}

// The arrays of lbvh_rebuild_alloc for n triangles and the collapse graph.  Only then does the GAS switch to the new node array
// and refit scratch: a failure leaves it as it was.  Its instance records still point at the old node array, which is freed here;
// every scene that instances the GAS is stale (a new generation) until rtc_ias_update rewrites them.
int setup_gas_rebuild(rtc_context* ctx, GasRecord& rec, LbvhRebuild& R, uint32_t n)
{
  if (int rc = lbvh_rebuild_alloc(ctx, R, n, nullptr)) return rc;
  const CollapseArgs& A = R.args;
  float4* tris = static_cast<float4*>(rec.d_tris);
  if (int rc = build_collapse_graph(ctx, R, [&](int level, unsigned grid, int2* work, const uint32_t* count, uint32_t* nextCount, int2* nextWork,
                                                cudaGraphConditionalHandle handle) {
        k_gas_pick<<<grid, kCollapseBlock, 0, ctx->stream>>>(A, work, count);
        k_gas_scan<<<1, kScanThreads, 0, ctx->stream>>>(A, count, nextCount, handle, level);
        k_gas_emit<<<grid, kCollapseBlock, 0, ctx->stream>>>(A, tris, work, count, nextWork);
      })) return rc;
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));

  cudaFree(rec.d_nodes);
  free_refit_scratch(rec.refit, ctx->stream);
  rec.d_nodes = R.nodes; R.nodes = nullptr;
  rec.refit = R.refit; R.refit = RefitScratch();
  rec.d_numNodes = A.counters + kNodeCount;
  rec.d_rejected = A.counters + kGasRejected;
  return 0;
}

int setup_gas(rtc_context* ctx, GasRecord& rec, uint32_t n)
{
  LbvhRebuild* r = new LbvhRebuild();
  if (int rc = setup_gas_rebuild(ctx, rec, *r, n))
  {
    cudaStreamSynchronize(ctx->stream);
    free_lbvh_rebuild(r);
    cudaGetLastError();
    return rc;
  }
  rec.rebuild = r;
  return 0;
}

} // namespace

int rebuild_gas_gpu(rtc_context* ctx, GasRecord& rec)
{
  const uint32_t n = rec.numTris;
  if (n == 0 && !rec.rebuild) return 0;          // a built GAS without triangles: one empty node, nothing to rebuild
  if (!rec.rebuild)
    if (int rc = setup_gas(ctx, rec, n)) return rc;
  LbvhRebuild& R = *rec.rebuild;
  cudaStream_t st = ctx->stream;
  GasInput in;
  in.verts = reinterpret_cast<const uint8_t*>((uintptr_t)rec.attributes);
  in.idx = reinterpret_cast<const uint32_t*>((uintptr_t)rec.indices);
  in.numVerts = rec.numVerts; in.stride = rec.strideBytes;
  k_gas_begin<<<1, 1, 0, st>>>(R.centreBox, R.args.counters, R.work[0], in, n, static_cast<uint4*>(rec.d_nodes), rec.refit.box);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  rec.boundsOnDevice = true;
  if (n == 0) return 0;
  RTC_CUDA(cudaMemsetAsync(R.flags, 0, (size_t)n * sizeof(uint32_t), st));
  k_gas_boxes<<<(n + kLbvhBlock - 1) / kLbvhBlock, kLbvhBlock, 0, st>>>(in, n, R.lo, R.hi, R.centreBox, R.args.counters + kGasRejected);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  if (int rc = lbvh_rebuild_tail(ctx, R, n)) return rc;
  k_gas_bounds<<<1, 1, 0, st>>>(R.boxLo, R.boxHi, rec.refit.box);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  return 0;
}

int create_gas_gpu(rtc_context* ctx, GasRecord& rec, uint32_t capacity)
{
  if (int rc = setup_gas(ctx, rec, capacity)) return rc;
  return rebuild_gas_gpu(ctx, rec);
}
