// bvh_build_gpu.cu -- device builder for geometry acceleration structures (replaces optixAccelBuild over
// OPTIX_BUILD_INPUT_TYPE_TRIANGLES, apps/rtigo3/src/Device.cpp:1391-1405, for inputs too large for the host builder).
//
//   1. triangle bounds + scene bounds                                   k_tri_bounds
//   2. 63-bit Morton codes of the box centres, radix sort               k_morton, cub::DeviceRadixSort (library sort; build path only)
//   3. binary radix tree over the sorted codes (Karras 2012)            k_radix_tree
//   4. bottom-up box fit                                                k_fit_boxes
//   5. SAH-binned top levels: the subtrees of a cut of ~4096 nodes are re-linked by a binned-SAH
//      build over their boxes (the cut is tiny, so it runs on the host) k_mark_cut, build_binary_sah_host
//   6. collapse to 8-wide nodes with quantised child boxes, level by    k_collapse_level
//      level, emitting triangles in leaf order
// Everything stays in device memory; the result is written straight into GasRecord::d_nodes / d_tris.
// The node format is that of bvh_build_host.cpp; both builders quantise through bvh_rules.h.
#include "rtc_internal.h"
#include "bvh_rules.h"
#include "lbvh.cuh"

#include <cub/device/device_radix_sort.cuh>

#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>

namespace {

constexpr int kB = 256;
constexpr uint32_t kLeafMax = 3;      // a wide leaf child holds 1..3 triangles

struct BuildArrays
{
  // per triangle (input order)
  float4* triLo; float4* triHi;
  // sort
  unsigned long long* keys; unsigned long long* keysAlt; uint32_t* order; uint32_t* orderAlt;
  // binary tree: node ids 0..n-2 internal, n-1..2n-2 leaves (sorted position p -> n-1+p); ids >= 2n-1: SAH top nodes
  int2* child;            // children of internal / top nodes
  int*  parent;
  int2* range;            // sorted positions [first, last] covered by a node
  float4* boxLo; float4* boxHi;
  uint32_t* flags;        // arrival counters of the bottom-up fit
  float* sceneBox;        // lo[3], hi[3]
};

__global__ void __launch_bounds__(kB)
k_tri_bounds(const uint8_t* __restrict__ verts, uint32_t stride, const uint32_t* __restrict__ idx, uint32_t n, uint32_t numVerts,
             float4* __restrict__ triLo, float4* __restrict__ triHi, float* __restrict__ sceneBox, uint32_t* __restrict__ badIndex)
{
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  if (t < n)
  {
    for (int c = 0; c < 3; ++c)
    {
      const uint32_t vi = __ldg(idx + 3u * (size_t)t + c);
      if (vi >= numVerts) { atomicExch(badIndex, 1u); continue; }
      const float* p = reinterpret_cast<const float*>(verts + (size_t)vi * stride);
      for (int k = 0; k < 3; ++k) { const float v = __ldg(p + k); lo[k] = fminf(lo[k], v); hi[k] = fmaxf(hi[k], v); }
    }
    triLo[t] = make_float4(lo[0], lo[1], lo[2], 0.0f);
    triHi[t] = make_float4(hi[0], hi[1], hi[2], 0.0f);
  }
  // block reduction of the scene box, then one atomic per block and plane
  __shared__ float sLo[3][kB / 32], sHi[3][kB / 32];
  for (int k = 0; k < 3; ++k)
  {
    float a = lo[k], b = hi[k];
    for (int off = 16; off; off >>= 1) { a = fminf(a, __shfl_down_sync(0xffffffffu, a, off)); b = fmaxf(b, __shfl_down_sync(0xffffffffu, b, off)); }
    if ((threadIdx.x & 31) == 0) { sLo[k][threadIdx.x >> 5] = a; sHi[k][threadIdx.x >> 5] = b; }
  }
  __syncthreads();
  if (threadIdx.x < 3)
  {
    float a = FLT_MAX, b = -FLT_MAX;
    for (int w = 0; w < kB / 32; ++w) { a = fminf(a, sLo[threadIdx.x][w]); b = fmaxf(b, sHi[threadIdx.x][w]); }
    if (a <= b) { atomicMinF(sceneBox + threadIdx.x, a); atomicMaxF(sceneBox + 3 + threadIdx.x, b); }
  }
}

// nodes of the cut: subtree size <= limit while the parent's is larger
__global__ void __launch_bounds__(kB)
k_mark_cut(int n, int limit, const int* __restrict__ parent, const int2* __restrict__ range, int* __restrict__ cutNodes, uint32_t* __restrict__ cutCount, uint32_t cutCapacity)
{
  const int node = blockIdx.x * blockDim.x + threadIdx.x;
  if (node >= 2 * n - 1 || node == 0) return;
  const int size = (node < n - 1) ? (range[node].y - range[node].x + 1) : 1;
  const int2 pr = range[parent[node]];
  if (size <= limit && (pr.y - pr.x + 1) > limit)
  {
    const uint32_t slot = atomicAdd(cutCount, 1u);
    if (slot < cutCapacity) cutNodes[slot] = node;
  }
}

__global__ void k_gather_boxes(const int* __restrict__ nodes, uint32_t count, const float4* __restrict__ boxLo, const float4* __restrict__ boxHi, PrimBox* __restrict__ out)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const float4 lo = boxLo[nodes[i]], hi = boxHi[nodes[i]];
  PrimBox b; b.lo[0] = lo.x; b.lo[1] = lo.y; b.lo[2] = lo.z; b.hi[0] = hi.x; b.hi[1] = hi.y; b.hi[2] = hi.z;
  out[i] = b;
}

struct CollapseParams
{
  int n;                      // triangles
  const int2* child; const int2* range; const float4* boxLo; const float4* boxHi;
  const uint32_t* order;      // sorted position -> triangle
  const uint8_t* verts; uint32_t stride; const uint32_t* idx;
  Node8* nodes; float4* tris;
  uint32_t* nodeCount; uint32_t* triCount;
  int leafMax;                // triangles per leaf child, 1..kLeafMax
};

__device__ __forceinline__ float half_area(const float4 lo, const float4 hi)
{
  const float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z;
  return dx * dy + dy * dz + dz * dx;
}

// One thread = one wide node of the current level: opens the largest children of its binary subtree until eight remain,
// assigns octant slots, quantises conservatively, allocates its children contiguously and queues them for the next level.
__global__ void __launch_bounds__(128)
k_collapse_level(const CollapseParams P, const int2* __restrict__ work, uint32_t workCount, int2* __restrict__ nextWork, uint32_t* __restrict__ nextCount)
{
  const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= workCount) return;
  const int src = work[w].x;
  const uint32_t dst = (uint32_t)work[w].y;
  const int n = P.n;
  auto size_of = [&](int node) { return (node >= n - 1 && node < 2 * n - 1) ? 1 : (P.range[node].y - P.range[node].x + 1); };
  auto is_leaf = [&](int node) { return size_of(node) <= P.leafMax; };

  int kids[8]; int nk = 0;
  if (is_leaf(src)) kids[nk++] = src;
  else { const int2 c = P.child[src]; kids[nk++] = c.x; kids[nk++] = c.y; }
  while (nk < 8)
  {
    int best = -1; float bestArea = -1.0f;
    for (int i = 0; i < nk; ++i)
      if (!is_leaf(kids[i])) { const float a = half_area(P.boxLo[kids[i]], P.boxHi[kids[i]]); if (a > bestArea) { bestArea = a; best = i; } }
    if (best < 0) break;
    const int2 c = P.child[kids[best]];
    kids[best] = c.x; kids[nk++] = c.y;
  }

  const float4 blo = P.boxLo[src], bhi = P.boxHi[src];
  const float boxLo[3] = { blo.x, blo.y, blo.z }, boxHi[3] = { bhi.x, bhi.y, bhi.z };
  float kLo[8][3], kHi[8][3];
  for (int i = 0; i < nk; ++i)
  {
    const float4 a = P.boxLo[kids[i]], b = P.boxHi[kids[i]];
    kLo[i][0] = a.x; kLo[i][1] = a.y; kLo[i][2] = a.z; kHi[i][0] = b.x; kHi[i][1] = b.y; kHi[i][2] = b.z;
  }

  // octant slots: greedy maximum of dot(child centre - node centre, slot sign vector)
  int kidAt[8]; for (int s = 0; s < 8; ++s) kidAt[s] = -1;
  {
    float centre[3]; for (int k = 0; k < 3; ++k) centre[k] = 0.5f * (boxLo[k] + boxHi[k]);
    uint32_t slotUsed = 0, kidDone = 0;
    for (int round = 0; round < nk; ++round)
    {
      int bi = -1, bs = -1; float bc = -FLT_MAX;
      for (int i = 0; i < nk; ++i)
      {
        if (kidDone & (1u << i)) continue;
        const float d0 = 0.5f * (kLo[i][0] + kHi[i][0]) - centre[0], d1 = 0.5f * (kLo[i][1] + kHi[i][1]) - centre[1], d2 = 0.5f * (kLo[i][2] + kHi[i][2]) - centre[2];
        for (int s = 0; s < 8; ++s)
        {
          if (slotUsed & (1u << s)) continue;
          const float c = ((s & 4) ? d0 : -d0) + ((s & 2) ? d1 : -d1) + ((s & 1) ? d2 : -d2);
          if (c > bc || bi < 0) { bc = c; bi = i; bs = s; }
        }
      }
      kidAt[bs] = bi; slotUsed |= 1u << bs; kidDone |= 1u << bi;
    }
  }

  // quantisation frame and conservative child planes (bvh_rules.h)
  Node8 node;
  {
    uint32_t occupied = 0;
    for (int s = 0; s < 8; ++s) if (kidAt[s] >= 0) occupied |= 1u << s;
    float nodeLo[3], nodeHi[3];
    quantise_node(occupied, [&](int s, float lo[3], float hi[3]) {
      for (int k = 0; k < 3; ++k) { lo[k] = kLo[kidAt[s]][k]; hi[k] = kHi[kidAt[s]][k]; }
    }, node, nodeLo, nodeHi);
  }
  node.imask = 0;
  uint32_t numInner = 0, numLeafTris = 0;
  for (int s = 0; s < 8; ++s)
  {
    node.meta[s] = 0;
    if (kidAt[s] < 0) continue;
    const int kid = kids[kidAt[s]];
    if (!is_leaf(kid)) { node.imask |= (uint8_t)(1u << s); ++numInner; }
    else numLeafTris += (uint32_t)size_of(kid);
  }
  node.childBase = numInner ? atomicAdd(P.nodeCount, numInner) : 0u;
  node.triBase = numLeafTris ? atomicAdd(P.triCount, numLeafTris) : 0u;
  const uint32_t nextBase = numInner ? atomicAdd(nextCount, numInner) : 0u;

  uint32_t triOffset = 0, rel = 0;
  for (int s = 0; s < 8; ++s)
  {
    if (kidAt[s] < 0) continue;
    const int kid = kids[kidAt[s]];
    if (node.imask & (1u << s))
    {
      nextWork[nextBase + rel] = make_int2(kid, (int)(node.childBase + rel));
      ++rel;
    }
    else
    {
      const int cnt = size_of(kid);
      const int first = (kid >= n - 1 && kid < 2 * n - 1) ? kid - (n - 1) : P.range[kid].x;
      node.meta[s] = (uint8_t)(((uint32_t)cnt << 5) | triOffset);
      for (int i = 0; i < cnt; ++i)
      {
        const uint32_t prim = P.order[first + i];
        float4* out = P.tris + (size_t)(node.triBase + triOffset + (uint32_t)i) * 3u;
        for (int c = 0; c < 3; ++c)
        {
          const uint32_t vi = __ldg(P.idx + 3u * (size_t)prim + c);
          const float* v = reinterpret_cast<const float*>(P.verts + (size_t)vi * P.stride);
          out[c] = make_float4(__ldg(v), __ldg(v + 1), __ldg(v + 2), c == 0 ? __uint_as_float(prim) : 0.0f);
        }
      }
      triOffset += (uint32_t)cnt;
    }
  }
  P.nodes[dst] = node;
}

// Build scratch comes from the stream-ordered pool (cudaMallocAsync): a synchronous cudaMalloc/cudaFree of a dozen
// multi-gigabyte arrays costs far more wall time than the build kernels themselves (100 M triangles: 57 ms of kernels).
struct DeviceFree
{
  cudaStream_t stream = nullptr;
  std::vector<void*> ptrs;
  ~DeviceFree() { for (void* p : ptrs) cudaFreeAsync(p, stream); }
  template <class T> cudaError_t alloc(T** p, size_t count)
  {
    cudaError_t e = cudaMallocAsync((void**)p, count * sizeof(T) + 16, stream);
    if (e == cudaSuccess) ptrs.push_back(*p);
    return e;
  }
};

} // namespace

// Binned-SAH binary build over a few thousand boxes on the host (bvh_build_host.cpp); returns nodes as (left, right)
// with negative values ~leafIndex, root first.
void build_binary_sah_host(const PrimBox* prims, uint32_t numPrims, std::vector<int2>& children, std::vector<PrimBox>& boxes);

static int build_gas_gpu_impl(rtc_context* ctx, GasRecord& rec)
{
  const uint32_t n = rec.numTris;
  if (n == 0) RTC_FAIL("build_gas_gpu needs at least one triangle");
  if (n > 0x3fffffffu) RTC_FAIL("too many triangles for one GAS");
  cudaStream_t st = ctx->stream;
  const bool verbose = std::getenv("RTC_BUILD_VERBOSE") != nullptr;     // phase timings on stderr
  auto tick = std::chrono::steady_clock::now();
  auto phase = [&](const char* name) {
    if (!verbose) return;
    cudaStreamSynchronize(st);
    const auto now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "build_gas_gpu[%u tris] %-10s %8.3f ms\n", n, name, std::chrono::duration<double, std::milli>(now - tick).count());
    tick = now;
  };
  DeviceFree scratch;
  scratch.stream = st;
  BuildArrays A{};
  uint32_t* d_counters = nullptr;       // [0] bad index, [1] cut count, [2] wide nodes, [3] tris, [4..5] level queue counts
  int* d_cut = nullptr; PrimBox* d_cutBoxes = nullptr;
  const uint32_t cutCapacity = 1u << 16;
  const size_t numBinary = 2 * (size_t)n - 1;
  const size_t topCapacity = 2 * (size_t)cutCapacity;      // SAH top nodes appended behind the radix tree
  RTC_CUDA(scratch.alloc(&A.triLo, n)); RTC_CUDA(scratch.alloc(&A.triHi, n));
  RTC_CUDA(scratch.alloc(&A.keys, n)); RTC_CUDA(scratch.alloc(&A.keysAlt, n));
  RTC_CUDA(scratch.alloc(&A.order, n)); RTC_CUDA(scratch.alloc(&A.orderAlt, n));
  RTC_CUDA(scratch.alloc(&A.child, numBinary + topCapacity)); RTC_CUDA(scratch.alloc(&A.parent, numBinary));
  RTC_CUDA(scratch.alloc(&A.range, numBinary + topCapacity));
  RTC_CUDA(scratch.alloc(&A.boxLo, numBinary + topCapacity)); RTC_CUDA(scratch.alloc(&A.boxHi, numBinary + topCapacity));
  RTC_CUDA(scratch.alloc(&A.flags, n)); RTC_CUDA(scratch.alloc(&A.sceneBox, 8));
  RTC_CUDA(scratch.alloc(&d_counters, 8)); RTC_CUDA(scratch.alloc(&d_cut, cutCapacity)); RTC_CUDA(scratch.alloc(&d_cutBoxes, cutCapacity));

  phase("alloc");
  const float initBox[6] = { FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX };
  RTC_CUDA(cudaMemcpyAsync(A.sceneBox, initBox, sizeof(initBox), cudaMemcpyHostToDevice, st));
  RTC_CUDA(cudaMemsetAsync(d_counters, 0, 8 * sizeof(uint32_t), st));
  RTC_CUDA(cudaMemsetAsync(A.flags, 0, (size_t)n * sizeof(uint32_t), st));
  const unsigned gridN = (n + kB - 1) / kB;
  k_tri_bounds<<<gridN, kB, 0, st>>>((const uint8_t*)(uintptr_t)rec.attributes, rec.strideBytes, (const uint32_t*)(uintptr_t)rec.indices, n, rec.numVerts,
                                      A.triLo, A.triHi, A.sceneBox, d_counters);
  k_morton<<<gridN, kB, 0, st>>>(A.triLo, A.triHi, n, A.sceneBox, A.keys, A.order);
  ctx->kernelLaunches += 2;
  {
    cub::DoubleBuffer<unsigned long long> k(A.keys, A.keysAlt);
    cub::DoubleBuffer<uint32_t> v(A.order, A.orderAlt);
    size_t tempBytes = 0;
    RTC_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tempBytes, k, v, (int)n, 0, 63, st));
    void* temp = nullptr;
    RTC_CUDA(scratch.alloc((uint8_t**)&temp, tempBytes));
    RTC_CUDA(cub::DeviceRadixSort::SortPairs(temp, tempBytes, k, v, (int)n, 0, 63, st));
    A.keys = k.Current(); A.order = v.Current();
  }
  phase("sort");
  if (n > 1)
  {
    k_radix_tree<<<(n - 1 + kB - 1) / kB, kB, 0, st>>>(A.keys, (int)n, A.child, A.parent, A.range);
    ctx->kernelLaunches++;
  }
  k_fit_boxes<<<gridN, kB, 0, st>>>((int)n, A.order, A.triLo, A.triHi, A.child, A.parent, A.boxLo, A.boxHi, A.flags);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());

  float hostBox[6]; uint32_t hostCounters[8];
  RTC_CUDA(cudaMemcpyAsync(hostBox, A.sceneBox, sizeof(hostBox), cudaMemcpyDeviceToHost, st));
  RTC_CUDA(cudaMemcpyAsync(hostCounters, d_counters, sizeof(hostCounters), cudaMemcpyDeviceToHost, st));
  RTC_CUDA(cudaStreamSynchronize(st));
  if (hostCounters[0]) RTC_FAIL("triangle index out of range");
  for (int k = 0; k < 3; ++k) { rec.lo[k] = hostBox[k]; rec.hi[k] = hostBox[3 + k]; }

  phase("tree+fit");
  // ---- SAH-binned top levels over a cut of the radix tree
  int rootNode = (n == 1) ? 0 : 0;            // binary root (for n == 1 the single leaf has id n-1 = 0)
  if (n > 8 * kLeafMax * 64)
  {
    // subtrees of at most n / kCutDivisor triangles form the cut whose top is rebuilt with binned SAH on the host
    uint32_t cutDivisor = 2048u;
    if (const char* e = std::getenv("RTC_GPU_CUT_DIVISOR")) { const long v = atol(e); if (64 <= v && v <= 32768) cutDivisor = (uint32_t)v; }
    int limit = (int)(n / cutDivisor); if (limit < (int)kLeafMax) limit = (int)kLeafMax;
    k_mark_cut<<<(unsigned)((numBinary + kB - 1) / kB), kB, 0, st>>>((int)n, limit, A.parent, A.range, d_cut, d_counters + 1, cutCapacity);
    RTC_CUDA(cudaMemcpyAsync(hostCounters, d_counters, sizeof(hostCounters), cudaMemcpyDeviceToHost, st));
    RTC_CUDA(cudaStreamSynchronize(st));
    const uint32_t cutCount = hostCounters[1];
    if (verbose) std::fprintf(stderr, "build_gas_gpu[%u tris] cut of %u subtrees (<= %d triangles each, capacity %u)\n", n, cutCount, limit, cutCapacity);
    if (cutCount >= 2 && cutCount <= cutCapacity)
    {
      k_gather_boxes<<<(cutCount + kB - 1) / kB, kB, 0, st>>>(d_cut, cutCount, A.boxLo, A.boxHi, d_cutBoxes);
      std::vector<PrimBox> cutBoxes(cutCount); std::vector<int> cutNodes(cutCount);
      RTC_CUDA(cudaMemcpyAsync(cutBoxes.data(), d_cutBoxes, cutCount * sizeof(PrimBox), cudaMemcpyDeviceToHost, st));
      RTC_CUDA(cudaMemcpyAsync(cutNodes.data(), d_cut, cutCount * sizeof(int), cudaMemcpyDeviceToHost, st));
      RTC_CUDA(cudaStreamSynchronize(st));
      std::vector<int2> topChildren; std::vector<PrimBox> topBoxes;
      build_binary_sah_host(cutBoxes.data(), cutCount, topChildren, topBoxes);
      // append: top node t -> id numBinary + t; its leaves are the cut's radix-tree nodes
      const size_t m = topChildren.size();
      std::vector<int2> hc(m), hr(m); std::vector<float4> hlo(m), hhi(m);
      for (size_t t = 0; t < m; ++t)
      {
        auto map = [&](int c) { return c < 0 ? cutNodes[(size_t)(~c)] : (int)(numBinary + (size_t)c); };
        hc[t] = make_int2(map(topChildren[t].x), map(topChildren[t].y));
        hr[t] = make_int2(0, (int)n - 1);        // only the size matters to the collapse: a top node is never a leaf cluster
        hlo[t] = make_float4(topBoxes[t].lo[0], topBoxes[t].lo[1], topBoxes[t].lo[2], 0.0f);
        hhi[t] = make_float4(topBoxes[t].hi[0], topBoxes[t].hi[1], topBoxes[t].hi[2], 0.0f);
      }
      RTC_CUDA(cudaMemcpyAsync(A.child + numBinary, hc.data(), m * sizeof(int2), cudaMemcpyHostToDevice, st));
      RTC_CUDA(cudaMemcpyAsync(A.range + numBinary, hr.data(), m * sizeof(int2), cudaMemcpyHostToDevice, st));
      RTC_CUDA(cudaMemcpyAsync(A.boxLo + numBinary, hlo.data(), m * sizeof(float4), cudaMemcpyHostToDevice, st));
      RTC_CUDA(cudaMemcpyAsync(A.boxHi + numBinary, hhi.data(), m * sizeof(float4), cudaMemcpyHostToDevice, st));
      RTC_CUDA(cudaStreamSynchronize(st));
      rootNode = (int)numBinary;
    }
  }

  phase("sah-top");
  // ---- collapse, level by level
  const size_t maxWide = (size_t)n + 16;          // every wide node but the root has a sibling group parent: < n nodes
  RTC_CUDA(cudaMalloc(&rec.d_nodes, maxWide * sizeof(Node8)));
  RTC_CUDA(cudaMalloc(&rec.d_tris, (size_t)n * 3u * sizeof(float4)));
  int2* d_work[2] = { nullptr, nullptr };
  RTC_CUDA(scratch.alloc(&d_work[0], maxWide)); RTC_CUDA(scratch.alloc(&d_work[1], maxWide));
  CollapseParams P;
  P.n = (int)n; P.child = A.child; P.range = A.range; P.boxLo = A.boxLo; P.boxHi = A.boxHi; P.order = A.order;
  P.verts = (const uint8_t*)(uintptr_t)rec.attributes; P.stride = rec.strideBytes; P.idx = (const uint32_t*)(uintptr_t)rec.indices;
  P.nodes = (Node8*)rec.d_nodes; P.tris = (float4*)rec.d_tris; P.nodeCount = d_counters + 2; P.triCount = d_counters + 3;
  // One triangle per leaf child.  A triangle test costs a warp ~2.7x what a node visit costs (it runs for the 3-4 lanes that
  // have just found a leaf, the node visit for 26-29), and the leaves of an LBVH over unstructured triangles are loose: single-
  // triangle leaves trade 18 triangle tests per ray for a few more node visits -- 1 M / 10 M-triangle soups, incoherent closest
  // hit: 1069 -> 1358 and 818 -> 1090 Mrays/s (leaves of <= 2: 1196 / 920).  RTC_GPU_LEAF_MAX=2|3 restores larger leaves.
  P.leafMax = 1;
  if (const char* e = std::getenv("RTC_GPU_LEAF_MAX")) { const int v = atoi(e); if (1 <= v && v <= (int)kLeafMax) P.leafMax = v; }
  const uint32_t one = 1u, zero = 0u;
  const int2 rootWork = make_int2(rootNode, 0);
  RTC_CUDA(cudaMemcpyAsync(d_counters + 2, &one, sizeof(uint32_t), cudaMemcpyHostToDevice, st));     // wide node 0 = root
  RTC_CUDA(cudaMemcpyAsync(d_counters + 3, &zero, sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  RTC_CUDA(cudaMemcpyAsync(d_work[0], &rootWork, sizeof(int2), cudaMemcpyHostToDevice, st));
  uint32_t workCount = 1;
  int cur = 0, levels = 0;
  while (workCount)
  {
    ++levels;
    RTC_CUDA(cudaMemcpyAsync(d_counters + 4, &zero, sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    k_collapse_level<<<(workCount + 127) / 128, 128, 0, st>>>(P, d_work[cur], workCount, d_work[cur ^ 1], d_counters + 4);
    ctx->kernelLaunches++;
    RTC_CUDA(cudaMemcpyAsync(&workCount, d_counters + 4, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    RTC_CUDA(cudaStreamSynchronize(st));
    cur ^= 1;
  }
  RTC_CUDA(cudaMemcpyAsync(hostCounters, d_counters, sizeof(hostCounters), cudaMemcpyDeviceToHost, st));
  RTC_CUDA(cudaStreamSynchronize(st));
  RTC_CUDA(cudaGetLastError());
  phase("collapse");
  if (verbose) std::fprintf(stderr, "build_gas_gpu[%u tris] %d collapse levels, %u wide nodes\n", n, levels, hostCounters[2]);
  if (hostCounters[3] != n) RTC_FAIL("GPU build lost triangles (internal error)");
  rec.numNodes = hostCounters[2];
  // the node array was sized for the worst case (one wide node per triangle): shrink it to what the collapse produced
  if ((size_t)rec.numNodes * 2 < maxWide)
  {
    void* exact = nullptr;
    RTC_CUDA(cudaMalloc(&exact, (size_t)rec.numNodes * sizeof(Node8)));
    cudaError_t e = cudaMemcpyAsync(exact, rec.d_nodes, (size_t)rec.numNodes * sizeof(Node8), cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { cudaFree(exact); return rtc_set_error(__FILE__, __LINE__, "shrink node array", (int)e, cudaGetErrorString(e)); }
    RTC_CUDA(cudaFree(rec.d_nodes));
    rec.d_nodes = exact;
  }
  return 0;
}

// The outputs are allocated half-way through the build: a failure after that point must not leak them.
int build_gas_gpu(rtc_context* ctx, GasRecord& rec)
{
  const int rc = build_gas_gpu_impl(ctx, rec);
  if (rc != 0)
  {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(rec.d_nodes); cudaFree(rec.d_tris);
    rec.d_nodes = nullptr; rec.d_tris = nullptr;
    cudaGetLastError();
  }
  return rc;
}
