// bvh_build_gas_rebuild_gpu.cu -- rtc_gas_rebuild: a new topology for a geometry, built on the device from its current vertex
// positions and written in place into its node and triangle arrays (the handle stays valid).
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
// Compiled with -fmad=false: the collapse's surface areas and slot costs (bvh_rules.h) must round like the host twin
// (rtc_host_gas_rebuild, accel_host.cpp), which is compiled with -ffp-contract=off.
#include "rtc_internal.h"
#include "bvh_rules.h"
#include "lbvh_collapse.cuh"

namespace {

// the vertex buffer of the call, which the collapse graph (captured once) reads from the counters
__device__ __forceinline__ const uint8_t* rebuild_verts(const CollapseArgs& A)
{
  return reinterpret_cast<const uint8_t*>(*reinterpret_cast<const unsigned long long*>(A.counters + kInput));
}

struct TriangleLeaves
{
  uint32_t stride, numVerts;
  const uint32_t* idx;
  float4* tris;
};

// One thread per triangle: its exact box (the arithmetic of rtc_host_gas_rebuild), and the block's share of the centre box.
__global__ void __launch_bounds__(kLbvhBlock)
k_gas_boxes(const uint8_t* __restrict__ verts, const TriangleLeaves L, uint32_t n, float4* __restrict__ lo, float4* __restrict__ hi,
            float* __restrict__ centreBox)
{
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  float cLo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, cHi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  if (t < n)
  {
    float bLo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, bHi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
    bool active = true;
    for (int c = 0; c < 3; ++c)
    {
      const uint32_t vi = __ldg(L.idx + 3u * (size_t)t + c);
      if (vi >= L.numVerts) continue;                   // indices are the build's, which checked them
      const float* p = reinterpret_cast<const float*>(verts + (size_t)vi * L.stride);
      const float x[3] = { __ldg(p), __ldg(p + 1), __ldg(p + 2) };
      active = active && rules_in_range3(x);
      for (int k = 0; k < 3; ++k) { bLo[k] = fminf(bLo[k], x[k]); bHi[k] = fmaxf(bHi[k], x[k]); }
    }
    if (!active) rules_empty_box(bLo, bHi);
    lo[t] = make_float4(bLo[0], bLo[1], bLo[2], 0.0f);
    hi[t] = make_float4(bHi[0], bHi[1], bHi[2], 0.0f);
    if (active) for (int k = 0; k < 3; ++k) { cLo[k] = 0.5f * (bLo[k] + bHi[k]); cHi[k] = cLo[k]; }
  }
  lbvh_reduce_centre_box(cLo, cHi, centreBox);
}

__global__ void k_gas_begin(float* __restrict__ centreBox, uint32_t* __restrict__ counters, int2* __restrict__ work, const uint8_t* verts)
{
  collapse_begin(centreBox, counters, work);
  *reinterpret_cast<unsigned long long*>(counters + kInput) = (unsigned long long)(uintptr_t)verts;
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
  collapse_pick(A, A.n, work, workCount);
}

__global__ void __launch_bounds__(kScanThreads)
k_gas_scan(const CollapseArgs A, const uint32_t* __restrict__ workCount, uint32_t* __restrict__ nextCount,
           cudaGraphConditionalHandle handle, int setCondition)
{
  collapse_scan(A, workCount, nextCount, handle, setCondition);
}

// the leaf slot holds the triangle record, as the builders and the refit write it
__global__ void __launch_bounds__(kCollapseBlock)
k_gas_emit(const CollapseArgs A, const TriangleLeaves L, const int2* __restrict__ work, const uint32_t* __restrict__ workCount,
           int2* __restrict__ nextWork)
{
  collapse_emit(A, A.n, work, workCount, nextWork, [&](uint32_t slot, uint32_t p) {
    const uint8_t* verts = rebuild_verts(A);
    const uint32_t prim = A.order[p];
    float x[3][3];
    for (int c = 0; c < 3; ++c)
    {
      const uint32_t vi = __ldg(L.idx + 3u * (size_t)prim + c);
      if (vi >= L.numVerts) return;                     // indices are the build's, which checked them
      const float* v = reinterpret_cast<const float*>(verts + (size_t)vi * L.stride);
      x[c][0] = __ldg(v); x[c][1] = __ldg(v + 1); x[c][2] = __ldg(v + 2);
    }
    float4 rec[3];
    rules_tri_record(x[0], x[1], x[2], prim, rec);
    float4* out = L.tris + 3u * (size_t)slot;
    for (int c = 0; c < 3; ++c) out[c] = rec[c];
  });
}

TriangleLeaves triangle_leaves(const GasRecord& rec)
{
  TriangleLeaves L;
  L.stride = rec.strideBytes; L.numVerts = rec.numVerts;
  L.idx = reinterpret_cast<const uint32_t*>((uintptr_t)rec.indices);
  L.tris = static_cast<float4*>(rec.d_tris);
  return L;
}

// First call on a GAS: the arrays of lbvh_rebuild_alloc and the collapse graph.  Only then does the GAS switch to the new node
// array and refit scratch: a failure leaves it as it was.  Its instance records still point at the old node array, which is
// freed here; every scene that instances the GAS is stale (a new generation) until rtc_ias_update rewrites them.
int setup_gas_rebuild(rtc_context* ctx, GasRecord& rec, LbvhRebuild& R)
{
  if (int rc = lbvh_rebuild_alloc(ctx, R, rec.numTris, nullptr)) return rc;
  const CollapseArgs& A = R.args;
  const TriangleLeaves L = triangle_leaves(rec);
  if (int rc = build_collapse_graph(ctx, R, [&](int level, unsigned grid, int2* work, const uint32_t* count, uint32_t* nextCount, int2* nextWork,
                                                cudaGraphConditionalHandle handle) {
        k_gas_pick<<<grid, kCollapseBlock, 0, ctx->stream>>>(A, work, count);
        k_gas_scan<<<1, kScanThreads, 0, ctx->stream>>>(A, count, nextCount, handle, level);
        k_gas_emit<<<grid, kCollapseBlock, 0, ctx->stream>>>(A, L, work, count, nextWork);
      })) return rc;
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));

  cudaFree(rec.d_nodes);
  free_refit_scratch(rec.refit, ctx->stream);
  rec.d_nodes = R.nodes; R.nodes = nullptr;
  rec.refit = R.refit; R.refit = RefitScratch();
  rec.d_numNodes = A.counters + kNodeCount;
  return 0;
}

} // namespace

int rebuild_gas_gpu(rtc_context* ctx, GasRecord& rec)
{
  const uint32_t n = rec.numTris;
  if (n == 0) return 0;                          // one empty node: nothing to rebuild
  if (!rec.rebuild)
  {
    LbvhRebuild* r = new LbvhRebuild();
    if (int rc = setup_gas_rebuild(ctx, rec, *r))
    {
      cudaStreamSynchronize(ctx->stream);
      free_lbvh_rebuild(r);
      cudaGetLastError();
      return rc;
    }
    rec.rebuild = r;
  }
  LbvhRebuild& R = *rec.rebuild;
  cudaStream_t st = ctx->stream;
  const uint8_t* verts = reinterpret_cast<const uint8_t*>((uintptr_t)rec.attributes);
  k_gas_begin<<<1, 1, 0, st>>>(R.centreBox, R.args.counters, R.work[0], verts);
  RTC_CUDA(cudaMemsetAsync(R.flags, 0, (size_t)n * sizeof(uint32_t), st));
  k_gas_boxes<<<(n + kLbvhBlock - 1) / kLbvhBlock, kLbvhBlock, 0, st>>>(verts, triangle_leaves(rec), n, R.lo, R.hi, R.centreBox);
  ctx->kernelLaunches += 2;
  RTC_CUDA(cudaGetLastError());
  if (int rc = lbvh_rebuild_tail(ctx, R, n)) return rc;
  k_gas_bounds<<<1, 1, 0, st>>>(R.boxLo, R.boxHi, rec.refit.box);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  rec.boundsOnDevice = true;
  return 0;
}
