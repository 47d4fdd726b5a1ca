// bvh_build_ias_gpu.cu -- rtc_ias_rebuild: a new topology for a scene's instance level, built on the device from the padded
// instance boxes the scene holds (SceneRecord::d_instBoxes) and written in place into its node and leaf arrays.
//
//   1. instance boxes -> float4 boxes, exact min / max of their centres          k_ias_boxes
//   2. Morton codes, sort, radix tree, fit                                        lbvh_rebuild_tail (lbvh_collapse.cuh)
//   3. collapse to 8-wide nodes, one instance per leaf slot, level by level       k_ias_pick, k_ias_scan, k_ias_emit
//   4. instance-level leaves in leaf order, the refit's parent index and zeroed arrival counters (in k_ias_emit)
//
// The pipeline, its deterministic bytes and its one-time synchronisation are those of lbvh_collapse.cuh, which the geometry
// rebuild (bvh_build_gas_rebuild_gpu.cu) shares; the leaf slot here holds an instance id.  The instance count of a build is a
// launch argument outside the collapse graph and the device word counters[kInput] inside it, so a scene of rtc_ias_create, whose
// arrays are sized for its capacity, builds any count up to it with the same graph.
//
// Compiled with -fmad=false: the collapse's surface areas and slot costs (bvh_rules.h) must round like the host twin, which is
// compiled with -ffp-contract=off.
#include "rtc_internal.h"
#include "bvh_rules.h"
#include "lbvh_collapse.cuh"

#include <cstring>

namespace {

__global__ void __launch_bounds__(kLbvhBlock)
k_ias_boxes(const PrimBox* __restrict__ boxes, uint32_t n, float4* __restrict__ lo, float4* __restrict__ hi, float* __restrict__ centreBox)
{
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  float cLo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, cHi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  if (t < n)
  {
    const PrimBox b = boxes[t];
    lo[t] = make_float4(b.lo[0], b.lo[1], b.lo[2], 0.0f);
    hi[t] = make_float4(b.hi[0], b.hi[1], b.hi[2], 0.0f);
    for (int k = 0; k < 3; ++k) { cLo[k] = 0.5f * (b.lo[k] + b.hi[k]); cHi[k] = cLo[k]; }
  }
  lbvh_reduce_centre_box(cLo, cHi, centreBox);
}

__global__ void k_ias_begin(float* __restrict__ centreBox, uint32_t* __restrict__ counters, int2* __restrict__ work, uint32_t n)
{
  collapse_begin(centreBox, counters, work);
  counters[kInput] = n;
}

// (Four blocks per SM in the launch bounds: with the bound on threads alone ptxas keeps it at 64 registers and spills.)
__global__ void __launch_bounds__(kCollapseBlock, 4)
k_ias_pick(const CollapseArgs A, const int2* __restrict__ work, const uint32_t* __restrict__ workCount)
{
  collapse_pick(A, (int)A.counters[kInput], work, workCount);
}

__global__ void __launch_bounds__(kScanThreads)
k_ias_scan(const CollapseArgs A, const uint32_t* __restrict__ workCount, uint32_t* __restrict__ nextCount,
           cudaGraphConditionalHandle handle, int setCondition)
{
  collapse_scan(A, workCount, nextCount, handle, setCondition);
}

// the leaf slot holds the instance
__global__ void __launch_bounds__(kCollapseBlock)
k_ias_emit(const CollapseArgs A, const int2* __restrict__ work, const uint32_t* __restrict__ workCount, int2* __restrict__ nextWork)
{
  collapse_emit(A, (int)A.counters[kInput], work, workCount, nextWork, [&](uint32_t slot, uint32_t p) { A.leaves[slot] = A.order[p]; });
}

// First call on a scene: the arrays of lbvh_rebuild_alloc for n instances and the collapse graph.  Only then does the scene switch
// to the new node array: a failure leaves it as it was.
int setup_rebuild(rtc_context* ctx, SceneRecord& s, LbvhRebuild& R, uint32_t n)
{
  if (int rc = lbvh_rebuild_alloc(ctx, R, n, static_cast<uint32_t*>(s.d_tlasLeaves))) return rc;
  const CollapseArgs& A = R.args;
  if (int rc = build_collapse_graph(ctx, R, [&](int level, unsigned grid, int2* work, const uint32_t* count, uint32_t* nextCount, int2* nextWork,
                                                cudaGraphConditionalHandle handle) {
        k_ias_pick<<<grid, kCollapseBlock, 0, ctx->stream>>>(A, work, count);
        k_ias_scan<<<1, kScanThreads, 0, ctx->stream>>>(A, count, nextCount, handle, level);
        k_ias_emit<<<grid, kCollapseBlock, 0, ctx->stream>>>(A, work, count, nextWork);
      })) return rc;
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));

  // switch the scene to the new arrays; the cutout graph captured its SceneDesc, and with it the node array freed here (a created
  // scene has none yet)
  if (s.d_tlasNodes) release_cutout_graph(ctx);
  cudaFree(s.d_tlasNodes);
  free_refit_scratch(s.refit, ctx->stream);
  s.d_tlasNodes = R.nodes; R.nodes = nullptr;
  s.refit = R.refit; R.refit = RefitScratch();
  s.desc.tlasNodes = static_cast<const uint4*>(s.d_tlasNodes);
  RTC_CUDA(cudaMemcpyAsync(s.d_desc, &s.desc, sizeof(SceneDesc), cudaMemcpyHostToDevice, ctx->stream));
  s.d_numTlasNodes = A.counters + kNodeCount;
  return 0;
}

} // namespace

void free_lbvh_rebuild(LbvhRebuild* r)
{
  if (!r) return;
  if (r->exec) cudaGraphExecDestroy(r->exec);
  if (r->graph) cudaGraphDestroy(r->graph);
  cudaFree(r->base); cudaFree(r->nodes); free_refit_scratch(r->refit, nullptr);      // allocated with cudaMalloc by lbvh_rebuild_alloc
  delete r;
}

int setup_scene_rebuild(rtc_context* ctx, SceneRecord& s, uint32_t n)
{
  LbvhRebuild* r = new LbvhRebuild();
  if (int rc = setup_rebuild(ctx, s, *r, n))
  {
    cudaStreamSynchronize(ctx->stream);
    free_lbvh_rebuild(r);
    cudaGetLastError();
    return rc;
  }
  s.rebuild = r;
  return 0;
}

int rebuild_instances_gpu(rtc_context* ctx, SceneRecord& s)
{
  const uint32_t n = s.desc.numInstances;
  if (n == 0 && !s.rebuild) return 0;           // one empty node: nothing to rebuild
  if (!s.rebuild)
    if (int rc = setup_scene_rebuild(ctx, s, n)) return rc;
  LbvhRebuild& R = *s.rebuild;
  cudaStream_t st = ctx->stream;
  k_ias_begin<<<1, 1, 0, st>>>(R.centreBox, R.args.counters, R.work[0], n);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  if (n == 0)
  {
    // a created scene without instances: the one empty node rtc_ias_build writes for none (bvh_build_host.cpp), one node counted
    // by k_ias_begin
    static Node8 empty = [] {
      Node8 e; std::memset(&e, 0, sizeof(e));
      e.ex = e.ey = e.ez = 127;
      for (int k = 0; k < 8; ++k) e.qlox[k] = e.qloy[k] = e.qloz[k] = 255;
      return e;
    }();
    RTC_CUDA(cudaMemcpyAsync(s.d_tlasNodes, &empty, sizeof(Node8), cudaMemcpyHostToDevice, st));
    return 0;
  }
  RTC_CUDA(cudaMemsetAsync(R.flags, 0, (size_t)n * sizeof(uint32_t), st));
  k_ias_boxes<<<(n + kLbvhBlock - 1) / kLbvhBlock, kLbvhBlock, 0, st>>>(s.d_instBoxes, n, R.lo, R.hi, R.centreBox);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  return lbvh_rebuild_tail(ctx, R, n);
}

int create_instance_level_gpu(rtc_context* ctx, SceneRecord& s, uint32_t capacity)
{
  if (int rc = setup_scene_rebuild(ctx, s, capacity > 0 ? capacity : 1u)) return rc;
  return rebuild_instances_gpu(ctx, s);
}
