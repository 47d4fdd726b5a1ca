// lbvh_collapse.cuh -- the device LBVH rebuild both levels share: one primitive per leaf slot, deterministic bytes, and no host
// synchronisation after the first call.  bvh_build_ias_gpu.cu (rtc_ias_rebuild, rtc_ias_build_device: instance leaves) and
// bvh_build_gas_rebuild_gpu.cu (rtc_gas_rebuild, rtc_gas_build_device: triangle leaves) wrap the device bodies below in their own
// kernels and hand them the leaf write.
//
//   primitive boxes and the exact min / max of their centres                     the caller's kernel, lbvh_reduce_centre_box
//   63-bit Morton codes, stable radix sort (key, then index)                      k_morton, cub::DeviceRadixSort    (lbvh.cuh)
//   binary radix tree (Karras 2012), bottom-up fit                                k_radix_tree, k_fit_boxes         (lbvh.cuh)
//   collapse to 8-wide nodes, one primitive per leaf slot, level by level         collapse_pick, collapse_scan, collapse_emit
//   leaves in leaf order (the caller's leaf write), the refit's parent index and zeroed arrival counters   (collapse_emit)
//
// Deterministic bytes: the geometry builder's collapse hands out child blocks with atomicAdd, so its node order depends on the
// order threads arrive in.  Here every level's child blocks and leaf runs come from an exclusive scan over the level's work
// items, so the nodes are in breadth-first order, slot by slot: two rebuilds of the same boxes give the same bytes, and the host
// twins (rtc_host_ias_rebuild, rtc_host_gas_rebuild, accel_host.cpp) reproduce them.  Children still sit above their parent (the
// refit relies on it).
//
// No host synchronisation after the first call: the geometry builder reads every level's work count back to the host to size
// the next launch.  Here the levels are a CUDA graph with a conditional WHILE node (as the cutout any-hit rounds in
// kernels_shade.cu): the kernels read the level's work count from device memory, and the scan kernel sets the loop condition
// when the next level is empty.  Everything the graph captures is allocated on the first call, so it stays valid for the
// structure.  The grids are sized for the capacity; blocks past the level's work return at once.
//
// Compile with -fmad=false: the collapse's surface areas and slot costs (bvh_rules.h) must round like the host twins, which are
// compiled with -ffp-contract=off.
#pragma once

#include "lbvh.cuh"

#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>

#include <cfloat>

namespace {

constexpr int kCollapseBlock = 128;
constexpr int kScanThreads = 256;
// words of LbvhRebuild::counters; from kInput on they hold the inputs of the call, which the collapse graph (captured once) reads:
// counters[kInput] is the primitive count of the call (a created structure's count changes from build to build), the words
// after it are the caller's (a geometry keeps its vertex and index buffers there, bvh_build_gas_rebuild_gpu.cu)
enum { kNodeCount = 0, kLeafCount = 1, kWorkCount = 2 /* two: ping-pong */, kLevelNodeBase = 4, kLevelLeafBase = 5, kInput = 6, kNumCounters = 14 };

struct CollapseArgs
{
  const int2* child; const float4* boxLo; const float4* boxHi;
  const uint32_t* order;          // sorted position -> primitive
  uint4* nodes; uint32_t* leaves; // leaves: the instance level's leaf slots (null for a geometry, whose leaf write is its own)
  uint32_t* parent; uint32_t* arrivals;
  int* kidAt;                     // 8 per work item: the binary node in each slot, -1 empty
  uint32_t* local;                // per work item: exclusive prefix in its block, inner count | leaf count << 16
  uint32_t* blockSums;            // per block: the same packing
  uint2* blockPrefix;             // per block: exclusive prefix of the level (inner, leaves)
  uint32_t* counters;
};

// The block's share of the exact min / max of the centres (cLo = cHi = the centre of this thread's box, or +-FLT_MAX).
__device__ __forceinline__ void lbvh_reduce_centre_box(float cLo[3], float cHi[3], float* __restrict__ centreBox)
{
  __shared__ float sLo[3][kLbvhBlock / 32], sHi[3][kLbvhBlock / 32];
  for (int k = 0; k < 3; ++k)
  {
    float a = cLo[k], b = cHi[k];
    for (int off = 16; off; off >>= 1) { a = fminf(a, __shfl_down_sync(0xffffffffu, a, off)); b = fmaxf(b, __shfl_down_sync(0xffffffffu, b, off)); }
    if ((threadIdx.x & 31) == 0) { sLo[k][threadIdx.x >> 5] = a; sHi[k][threadIdx.x >> 5] = b; }
  }
  __syncthreads();
  if (threadIdx.x < 3)
  {
    float a = FLT_MAX, b = -FLT_MAX;
    for (int w = 0; w < kLbvhBlock / 32; ++w) { a = fminf(a, sLo[threadIdx.x][w]); b = fmaxf(b, sHi[threadIdx.x][w]); }
    if (a <= b) { atomicMinF(centreBox + threadIdx.x, a); atomicMaxF(centreBox + 3 + threadIdx.x, b); }
  }
}

// the state of one rebuild: the centre box to reduce into, one wide node (the root, over binary node 0) to collapse
__device__ __forceinline__ void collapse_begin(float* __restrict__ centreBox, uint32_t* __restrict__ counters, int2* __restrict__ work)
{
  for (int k = 0; k < 3; ++k) { centreBox[k] = FLT_MAX; centreBox[3 + k] = -FLT_MAX; }
  counters[kNodeCount] = 1u; counters[kLeafCount] = 0u;
  counters[kWorkCount] = 1u; counters[kWorkCount + 1] = 0u;
  work[0] = make_int2(0, 0);
}

// One thread per work item (binary node, wide node index) of the level: the wide node without its childBase / triBase, its
// slots' binary nodes, and the exclusive scan of (inner children, leaf slots) within the block.  n: the primitives of this build.
__device__ __forceinline__ void collapse_pick(const CollapseArgs& A, int n, const int2* __restrict__ work, const uint32_t* __restrict__ workCount)
{
  const uint32_t count = *workCount;
  if (blockIdx.x * kCollapseBlock >= count) return;             // the whole block: no thread reaches the scan
  const uint32_t w = blockIdx.x * kCollapseBlock + threadIdx.x;
  uint32_t packed = 0;
  if (w < count)
  {
    const int2 item = work[w];
    int kidAt[8];
    union { Node8 n; uint4 v[5]; } node;
    uint32_t numInner, numLeaves;
    lbvh_instance_node(item.x, n,
                       [&](int id, float lo[3], float hi[3]) {
                         const float4 a = A.boxLo[id], b = A.boxHi[id];
                         lo[0] = a.x; lo[1] = a.y; lo[2] = a.z; hi[0] = b.x; hi[1] = b.y; hi[2] = b.z;
                       },
                       [&](int id) { return A.child[id]; }, kidAt, node.n, numInner, numLeaves);
    for (int j = 0; j < 5; ++j) A.nodes[5u * (size_t)item.y + j] = node.v[j];
    for (int s = 0; s < 8; ++s) A.kidAt[8u * (size_t)w + s] = kidAt[s];
    packed = numInner | (numLeaves << 16);
  }
  using Scan = cub::BlockScan<uint32_t, kCollapseBlock>;
  __shared__ typename Scan::TempStorage tmp;
  uint32_t prefix, total;
  Scan(tmp).ExclusiveSum(packed, prefix, total);
  if (w < count) A.local[w] = prefix;
  if (threadIdx.x == 0) A.blockSums[blockIdx.x] = total;
}

// One block: the exclusive scan of the level's block sums, the level's bases in the node and leaf arrays, the next level's work
// count, and (setCondition) the loop condition: run again while the next level has work.
__device__ __forceinline__ void collapse_scan(const CollapseArgs& A, const uint32_t* __restrict__ workCount, uint32_t* __restrict__ nextCount,
                                              cudaGraphConditionalHandle handle, int setCondition)
{
  const uint32_t numBlocks = (*workCount + kCollapseBlock - 1) / kCollapseBlock;
  const uint32_t per = (numBlocks + kScanThreads - 1) / kScanThreads;
  const uint32_t first = threadIdx.x * per, last = min(first + per, numBlocks);
  unsigned long long sum = 0;                                  // inner children in the low word, leaf slots in the high word
  for (uint32_t b = first; b < last; ++b) { const uint32_t v = A.blockSums[b]; sum += (v & 0xffffu) | ((unsigned long long)(v >> 16) << 32); }
  using Scan = cub::BlockScan<unsigned long long, kScanThreads>;
  __shared__ typename Scan::TempStorage tmp;
  unsigned long long prefix, total;
  Scan(tmp).ExclusiveSum(sum, prefix, total);
  for (uint32_t b = first; b < last; ++b)
  {
    A.blockPrefix[b] = make_uint2((uint32_t)prefix, (uint32_t)(prefix >> 32));
    const uint32_t v = A.blockSums[b];
    prefix += (v & 0xffffu) | ((unsigned long long)(v >> 16) << 32);
  }
  if (threadIdx.x == 0)
  {
    const uint32_t inner = (uint32_t)total, leaves = (uint32_t)(total >> 32);
    A.counters[kLevelNodeBase] = A.counters[kNodeCount];
    A.counters[kLevelLeafBase] = A.counters[kLeafCount];
    A.counters[kNodeCount] += inner;
    A.counters[kLeafCount] += leaves;
    *nextCount = inner;
    if (setCondition) cudaGraphSetConditional(handle, inner != 0u ? 1u : 0u);
  }
}

// One thread per work item: childBase / triBase from the scans, the next level's work items, the leaves, the parent of every
// child and a zero arrival counter for the refit (bvh_refit.cu).  leaf(slot, p) writes leaf slot `slot`, which holds the
// primitive at sorted position p.
template <class Leaf>
__device__ __forceinline__ void collapse_emit(const CollapseArgs& A, int n, const int2* __restrict__ work, const uint32_t* __restrict__ workCount,
                                              int2* __restrict__ nextWork, const Leaf& leaf)
{
  const uint32_t w = blockIdx.x * kCollapseBlock + threadIdx.x;
  if (w >= *workCount) return;
  const uint32_t dst = (uint32_t)work[w].y;
  const uint2 bp = A.blockPrefix[blockIdx.x];
  const uint32_t loc = A.local[w];
  const uint32_t innerOff = bp.x + (loc & 0xffffu), leafOff = bp.y + (loc >> 16);
  const uint32_t childBase = A.counters[kLevelNodeBase] + innerOff, triBase = A.counters[kLevelLeafBase] + leafOff;
  uint32_t inner = 0, numLeaves = 0;
  for (int s = 0; s < 8; ++s)
  {
    const int kid = A.kidAt[8u * (size_t)w + s];
    if (kid < 0) continue;
    if (kid >= n - 1) { leaf(triBase + numLeaves, (uint32_t)(kid - (n - 1))); ++numLeaves; }
    else
    {
      nextWork[innerOff + inner] = make_int2(kid, (int)(childBase + inner));
      A.parent[childBase + inner] = dst;
      ++inner;
    }
  }
  uint32_t* words = reinterpret_cast<uint32_t*>(A.nodes + 5u * (size_t)dst);
  words[4] = inner ? childBase : 0u;
  words[5] = numLeaves ? triBase : 0u;
  A.arrivals[dst] = 0u;
}

} // namespace

// Everything one structure's rebuilds use, allocated by the first (free_lbvh_rebuild releases it).
struct LbvhRebuild
{
  uint32_t n = 0, capacity = 0;                 // primitives the arrays hold (at most), wide nodes the node array holds
  void* base = nullptr;
  void* nodes = nullptr; RefitScratch refit;     // the structure's new node array and refit scratch until setup has succeeded
  float4 *lo = nullptr, *hi = nullptr, *boxLo = nullptr, *boxHi = nullptr;
  unsigned long long *keys = nullptr, *keysAlt = nullptr;
  uint32_t *order = nullptr, *orderAlt = nullptr, *flags = nullptr;
  int2 *child = nullptr, *range = nullptr, *work[2] = { nullptr, nullptr };
  int* parent = nullptr;
  float* centreBox = nullptr;
  void* sortTemp = nullptr; size_t sortBytes = 0;
  const unsigned long long* sortedKeys = nullptr; const uint32_t* sortedOrder = nullptr;
  CollapseArgs args{};
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
};

namespace {

// First call on a structure of n primitives: drains the stream once (launches in flight may still read the old nodes), then
// allocates a node array of the worst-case size, refit scratch sized for it (the layout of alloc_refit_scratch, bvh_refit.cu) and
// the build arrays in one allocation.  `leaves`: CollapseArgs::leaves.
int lbvh_rebuild_alloc(rtc_context* ctx, LbvhRebuild& R, uint32_t n, uint32_t* leaves)
{
  R.n = n;
  R.capacity = ias_rebuild_capacity(n);
  const size_t cap = R.capacity, nBin = 2 * (size_t)n;
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));

  RTC_CUDA(cudaMalloc(&R.nodes, cap * sizeof(Node8)));
  RTC_CUDA(cudaMalloc(&R.refit.base, cap * (2 * sizeof(uint32_t) + 6 * sizeof(float))));
  R.refit.box = static_cast<float*>(R.refit.base);
  R.refit.parent = reinterpret_cast<uint32_t*>(R.refit.box + 6 * cap);
  R.refit.arrivals = R.refit.parent + cap;

  {
    cub::DoubleBuffer<unsigned long long> k(nullptr, nullptr);
    cub::DoubleBuffer<uint32_t> v(nullptr, nullptr);
    RTC_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, R.sortBytes, k, v, (int)n, 0, 63, ctx->stream));
  }
  const size_t numBlocks = (cap + kCollapseBlock - 1) / kCollapseBlock;
  size_t offset = 0;
  auto carve = [&](size_t bytes) { const size_t at = offset; offset += (bytes + 255) & ~(size_t)255; return at; };
  const size_t oLo = carve(n * sizeof(float4)), oHi = carve(n * sizeof(float4));
  const size_t oBoxLo = carve(nBin * sizeof(float4)), oBoxHi = carve(nBin * sizeof(float4));
  const size_t oKeys = carve(n * 8u), oKeysAlt = carve(n * 8u), oOrder = carve(n * 4u), oOrderAlt = carve(n * 4u), oFlags = carve(n * 4u);
  const size_t oChild = carve(n * sizeof(int2)), oRange = carve(n * sizeof(int2)), oParent = carve(nBin * 4u);
  const size_t oWork0 = carve(cap * sizeof(int2)), oWork1 = carve(cap * sizeof(int2));
  const size_t oCentre = carve(6 * sizeof(float)), oSort = carve(R.sortBytes);
  const size_t oKidAt = carve(cap * 8u * sizeof(int)), oLocal = carve(cap * 4u), oBlockSums = carve(numBlocks * 4u);
  const size_t oBlockPrefix = carve(numBlocks * sizeof(uint2)), oCounters = carve(kNumCounters * 4u);
  RTC_CUDA(cudaMalloc(&R.base, offset));
  uint8_t* b = static_cast<uint8_t*>(R.base);
  R.lo = reinterpret_cast<float4*>(b + oLo); R.hi = reinterpret_cast<float4*>(b + oHi);
  R.boxLo = reinterpret_cast<float4*>(b + oBoxLo); R.boxHi = reinterpret_cast<float4*>(b + oBoxHi);
  R.keys = reinterpret_cast<unsigned long long*>(b + oKeys); R.keysAlt = reinterpret_cast<unsigned long long*>(b + oKeysAlt);
  R.order = reinterpret_cast<uint32_t*>(b + oOrder); R.orderAlt = reinterpret_cast<uint32_t*>(b + oOrderAlt);
  R.flags = reinterpret_cast<uint32_t*>(b + oFlags);
  R.child = reinterpret_cast<int2*>(b + oChild); R.range = reinterpret_cast<int2*>(b + oRange);
  R.parent = reinterpret_cast<int*>(b + oParent);
  R.work[0] = reinterpret_cast<int2*>(b + oWork0); R.work[1] = reinterpret_cast<int2*>(b + oWork1);
  R.centreBox = reinterpret_cast<float*>(b + oCentre);
  R.sortTemp = b + oSort;
  {
    // which buffer the sort leaves its result in depends only on n and the key bits: found once (over the still unwritten
    // arrays), the collapse graph captures it; a build of fewer primitives copies its result there (lbvh_rebuild_tail)
    cub::DoubleBuffer<unsigned long long> k(R.keys, R.keysAlt);
    cub::DoubleBuffer<uint32_t> v(R.order, R.orderAlt);
    RTC_CUDA(cub::DeviceRadixSort::SortPairs(R.sortTemp, R.sortBytes, k, v, (int)n, 0, 63, ctx->stream));
    R.sortedKeys = k.Current(); R.sortedOrder = v.Current();
  }
  CollapseArgs& A = R.args;
  A.child = R.child; A.boxLo = R.boxLo; A.boxHi = R.boxHi; A.order = R.sortedOrder;
  A.nodes = static_cast<uint4*>(R.nodes); A.leaves = leaves;
  A.parent = R.refit.parent; A.arrivals = R.refit.arrivals;
  A.kidAt = reinterpret_cast<int*>(b + oKidAt); A.local = reinterpret_cast<uint32_t*>(b + oLocal);
  A.blockSums = reinterpret_cast<uint32_t*>(b + oBlockSums); A.blockPrefix = reinterpret_cast<uint2*>(b + oBlockPrefix);
  A.counters = reinterpret_cast<uint32_t*>(b + oCounters);
  return 0;
}

// The WHILE loop of the collapse: its body holds two levels (work[0] -> work[1] -> work[0]), so every kernel argument is static.
// level(level, grid, work, count, nextCount, nextWork, handle) enqueues one level's pick, scan and emit kernels on ctx->stream.
template <class Level>
int build_collapse_graph(rtc_context* ctx, LbvhRebuild& R, const Level& level)
{
  RTC_CUDA(cudaGraphCreate(&R.graph, 0));
  cudaGraphConditionalHandle handle;
  RTC_CUDA(cudaGraphConditionalHandleCreate(&handle, R.graph, 1u, cudaGraphCondAssignDefault));   // the root level always runs
  cudaGraphNodeParams wp{};
  wp.type = cudaGraphNodeTypeConditional;
  wp.conditional.handle = handle; wp.conditional.type = cudaGraphCondTypeWhile; wp.conditional.size = 1;
  cudaGraphNode_t whileNode = nullptr;
  RTC_CUDA(cudaGraphAddNode(&whileNode, R.graph, nullptr, 0, &wp));
  cudaGraph_t body = wp.conditional.phGraph_out[0];
  RTC_CUDA(cudaStreamBeginCaptureToGraph(ctx->stream, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
  const unsigned grid = (R.capacity + kCollapseBlock - 1) / kCollapseBlock;
  for (int l = 0; l < 2; ++l)
    level(l, grid, R.work[l], R.args.counters + kWorkCount + l, R.args.counters + kWorkCount + (l ^ 1), R.work[l ^ 1], handle);
  cudaGraph_t captured = nullptr;
  const cudaError_t launchError = cudaGetLastError();
  RTC_CUDA(cudaStreamEndCapture(ctx->stream, &captured));
  RTC_CUDA(launchError);
  RTC_CUDA(cudaGraphInstantiate(&R.exec, R.graph, 0));
  return 0;
}

// Every step after the primitive boxes (R.lo, R.hi, R.centreBox) of n <= R.n primitives: Morton codes, the sort, the radix
// tree, the fit and the collapse graph, all enqueued on ctx->stream.
int lbvh_rebuild_tail(rtc_context* ctx, LbvhRebuild& R, uint32_t n)
{
  cudaStream_t st = ctx->stream;
  const unsigned gridN = (n + kLbvhBlock - 1) / kLbvhBlock;
  k_morton<<<gridN, kLbvhBlock, 0, st>>>(R.lo, R.hi, n, R.centreBox, R.keys, R.order);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  {
    cub::DoubleBuffer<unsigned long long> k(R.keys, R.keysAlt);
    cub::DoubleBuffer<uint32_t> v(R.order, R.orderAlt);
    if (n != R.n)
    {
      size_t bytes = 0;
      RTC_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, k, v, (int)n, 0, 63, st));
      if (bytes > R.sortBytes) RTC_FAIL("radix sort needs more temporary storage for fewer items (internal error)");
    }
    RTC_CUDA(cub::DeviceRadixSort::SortPairs(R.sortTemp, R.sortBytes, k, v, (int)n, 0, 63, st));
    // the sort's output buffer depends on n: the captured kernels read the one found for R.n
    if (k.Current() != R.sortedKeys) RTC_CUDA(cudaMemcpyAsync((void*)R.sortedKeys, k.Current(), (size_t)n * 8u, cudaMemcpyDeviceToDevice, st));
    if (v.Current() != R.sortedOrder) RTC_CUDA(cudaMemcpyAsync((void*)R.sortedOrder, v.Current(), (size_t)n * 4u, cudaMemcpyDeviceToDevice, st));
  }
  if (n > 1)
  {
    k_radix_tree<<<(n - 1 + kLbvhBlock - 1) / kLbvhBlock, kLbvhBlock, 0, st>>>(R.sortedKeys, (int)n, R.child, R.parent, R.range);
    ctx->kernelLaunches++;
  }
  k_fit_boxes<<<gridN, kLbvhBlock, 0, st>>>((int)n, R.sortedOrder, R.lo, R.hi, R.child, R.parent, R.boxLo, R.boxHi, R.flags);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  RTC_CUDA(cudaGraphLaunch(R.exec, st));
  ctx->kernelLaunches += 6;                      // one body execution; further levels are not counted
  return 0;
}

} // namespace
