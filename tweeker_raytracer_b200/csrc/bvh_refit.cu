// bvh_refit.cu -- in-place update of built acceleration structures (the counterpart of optixAccelBuild with
// OPTIX_BUILD_OPERATION_UPDATE), and the instance records the instance level is built and updated over.
//
//   GAS refit (rtc_gas_refit)        k_refit_tris   one pass over the leaf-ordered triangle records: new positions, id bits kept
//                                    k_refit_nodes  bottom-up over the wide nodes (Karras-style arrival counters: the last child
//                                                   to arrive processes the parent), re-quantised through bvh_rules.h
//   instance records                 k_instance_gather  one record per written instance: its matrix (device memory: the
//   (rtc_ias_build,                                     caller's for rtc_ias_update_device, staged by rtc_ias_update, the
//    rtc_ias_update,                                    scene's own object->world rows for rtc_ias_build, the caller's
//    rtc_ias_update_device,                             rtc_instance_desc records for rtc_ias_build_device), the inverse, its
//    rtc_ias_build_device)                              GAS's entry of the per-GAS table (of a created scene: the context's
//                                                       table, indexed by handle; the records written are selected here)
//                                    k_instance_bounds, k_instance_finish: the padded world box, the traversal and shading rows
//   instance-level refit             k_refit_nodes over the instance level (rtc_ias_build builds its nodes on the host instead,
//   (the updates)                                   over the boxes the records hold)
// Node topology (imask, childBase, triBase, meta) and leaf order stay as built; only the frame, the quantised planes and the
// triangle positions are rewritten.  Min / max are order-independent, so the result does not depend on the arrival order and
// equals the host twin (accel_host.cpp), which visits the nodes in descending index order.
//
// Compiled with -fmad=false: invert_3x4 and instance_box_finish (bvh_rules.h) must round like the host twin, which compiles them
// with -ffp-contract=off.
#include "rtc_internal.h"
#include "bvh_rules.h"

#include <cfloat>

namespace {

constexpr int kB = 256;

union NodeWords
{
  uint4 v[5];
  Node8 n;
};

__global__ void __launch_bounds__(kB)
k_refit_parents(const uint4* __restrict__ nodes, uint32_t numNodes, uint32_t* __restrict__ parent)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= numNodes) return;
  const uint32_t imask = nodes[5u * (size_t)i].w >> 24;
  const uint32_t childBase = nodes[5u * (size_t)i + 1].x;
  for (uint32_t r = 0; r < (uint32_t)__popc(imask); ++r) parent[childBase + r] = i;
}

__global__ void __launch_bounds__(kB)
k_refit_tris(float4* __restrict__ tris, uint32_t numTris, const uint8_t* __restrict__ verts, uint32_t stride, uint32_t numVerts,
             const uint32_t* __restrict__ idx)
{
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= numTris) return;
  float4* rec = tris + 3u * (size_t)t;
  const uint32_t prim = __float_as_uint(rec[0].w);
  float x[3][3];
  for (int c = 0; c < 3; ++c)
  {
    const uint32_t vi = __ldg(idx + 3u * (size_t)prim + c);
    if (vi >= numVerts)                                 // only rtc_gas_build_device leaves such an index: an inactive triangle
    {
      x[c][0] = x[c][1] = x[c][2] = __uint_as_float(kMissingVertexBits);
      continue;
    }
    const float* p = reinterpret_cast<const float*>(verts + (size_t)vi * stride);
    x[c][0] = __ldg(p); x[c][1] = __ldg(p + 1); x[c][2] = __ldg(p + 2);
  }
  float4 r[3];
  rules_tri_record(x[0], x[1], x[2], prim, r);
  for (int c = 0; c < 3; ++c) rec[c] = r[c];
}

struct RefitParams
{
  uint4* nodes; uint32_t numNodes;
  const float4* tris;                                   // geometry level: leaf-ordered triangle records
  const uint32_t* leaves; const PrimBox* primBoxes;     // instance level: leaf slot -> instance, instance boxes
  const uint32_t* parent; uint32_t* arrivals; float* box;
};

__device__ void refit_one(const RefitParams& P, uint32_t idx)
{
  NodeWords w;
  for (int j = 0; j < 5; ++j) w.v[j] = P.nodes[5u * (size_t)idx + j];
  auto leafBox = [&](uint32_t first, uint32_t count, float lo[3], float hi[3]) {
    for (int k = 0; k < 3; ++k) { lo[k] = INFINITY; hi[k] = -INFINITY; }
    for (uint32_t t = first; t < first + count; ++t)
    {
      if (P.tris)
      {
        float x[3][3];
        for (int c = 0; c < 3; ++c)
        {
          const float4 v = P.tris[3u * (size_t)t + c];
          x[c][0] = v.x; x[c][1] = v.y; x[c][2] = v.z;
        }
        if (!rules_in_range3(x[0]) || !rules_in_range3(x[1]) || !rules_in_range3(x[2])) continue;     // inactive triangle
        for (int c = 0; c < 3; ++c)
          for (int k = 0; k < 3; ++k) { lo[k] = x[c][k] < lo[k] ? x[c][k] : lo[k]; hi[k] = hi[k] < x[c][k] ? x[c][k] : hi[k]; }
      }
      else
      {
        const PrimBox b = P.primBoxes[P.leaves[t]];
        for (int k = 0; k < 3; ++k) { lo[k] = b.lo[k] < lo[k] ? b.lo[k] : lo[k]; hi[k] = hi[k] < b.hi[k] ? b.hi[k] : hi[k]; }
      }
    }
  };
  // boxes of inner children were written by other threads: read them from L2, behind the fence of the arrival protocol
  auto innerBox = [&](uint32_t child, float lo[3], float hi[3]) {
    for (int k = 0; k < 3; ++k) { lo[k] = __ldcg(P.box + 6u * (size_t)child + k); hi[k] = __ldcg(P.box + 6u * (size_t)child + 3 + k); }
  };
  float lo[3], hi[3];
  refit_node(w.n, leafBox, innerBox, lo, hi);
  for (int j = 0; j < 5; ++j) P.nodes[5u * (size_t)idx + j] = w.v[j];
  for (int k = 0; k < 3; ++k) { __stcg(P.box + 6u * (size_t)idx + k, lo[k]); __stcg(P.box + 6u * (size_t)idx + 3 + k, hi[k]); }
}

// One thread per node without inner children; after each node it climbs to the parent, which the LAST child to arrive refits.
// The arrival counter is reset by that thread, so the next refit starts from zero without a memset.
__device__ __forceinline__ void refit_from(const RefitParams& P, uint32_t i)
{
  if (P.nodes[5u * (size_t)i].w >> 24) return;          // imask != 0: reached from below
  uint32_t node = i;
  for (;;)
  {
    refit_one(P, node);
    if (node == 0) return;
    __threadfence();
    const uint32_t parent = P.parent[node];
    const uint32_t expected = (uint32_t)__popc(P.nodes[5u * (size_t)parent].w >> 24);
    if (atomicAdd(P.arrivals + parent, 1u) != expected - 1u) return;
    P.arrivals[parent] = 0u;
    __threadfence();
    node = parent;
  }
}

__global__ void __launch_bounds__(kB)
k_refit_nodes(const RefitParams P)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.numNodes) return;
  refit_from(P, i);
}

// A structure rtc_ias_rebuild or rtc_gas_rebuild wrote: its node count is on the device, and the nodes above it are not part of
// the structure.
__global__ void __launch_bounds__(kB)
k_refit_nodes_live(const RefitParams P, const uint32_t* __restrict__ numNodes)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *numNodes) return;
  refit_from(P, i);
}

// One instance whose records are written, as k_instance_gather assembles it.
struct InstanceUpdate
{
  float    transform[12];          // object -> world
  float    inverse[12];            // world -> object (invert_3x4)
  GasUpdateInput gas;              // its GAS's entry of the per-GAS table
  uint32_t instance, pad;
  int32_t  materialIndex, lightIndex;   // rtc_ias_build_device: the record's (written with the GAS's indices)
};

// ---- instance level: tight world bounds of every instance from its transformed vertices -------------------------
// The reference hands OptiX the instance transform and lets the driver bound the instance (Device.cpp:1427-1443,
// optixAccelBuild over OPTIX_BUILD_INPUT_TYPE_INSTANCES :1471-1482).  The first version here bounded the eight transformed
// corners of the GAS box, which is loose for rotated instances (a torus rotated by 45 degrees: +40 % per axis) and made
// rays enter instances they cannot hit; an instance entry costs about three node visits.  One CTA per instance now
// transforms every vertex of the instance's GAS and reduces min/max.
// numUp: the records k_instance_gather selected on the device (created scenes; the grid is their upper bound), or null
__global__ void __launch_bounds__(kB)
k_instance_bounds(const InstanceUpdate* __restrict__ up, PrimBox* __restrict__ out, const uint32_t* __restrict__ numUp)
{
  if (numUp && blockIdx.x >= *numUp) return;
  const InstanceUpdate& I = up[blockIdx.x];
  const GasUpdateInput& g = I.gas;
  float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  for (uint32_t v = threadIdx.x; v < g.numVerts; v += blockDim.x)
  {
    const float* p = reinterpret_cast<const float*>(g.verts + (size_t)v * g.stride);
    const float x = p[0], y = p[1], z = p[2];
    if (!rules_in_range(x) || !rules_in_range(y) || !rules_in_range(z)) continue;      // only inactive triangles use it
#pragma unroll
    for (int r = 0; r < 3; ++r)
    {
      const float* m = I.transform + 4 * r;
      const float w = fmaf(m[0], x, fmaf(m[1], y, fmaf(m[2], z, m[3])));
      lo[r] = fminf(lo[r], w); hi[r] = fmaxf(hi[r], w);
    }
  }
  __shared__ float sLo[3][kB / 32], sHi[3][kB / 32];
#pragma unroll
  for (int r = 0; r < 3; ++r)
  {
    for (int off = 16; off; off >>= 1)
    {
      lo[r] = fminf(lo[r], __shfl_down_sync(0xffffffffu, lo[r], off));
      hi[r] = fmaxf(hi[r], __shfl_down_sync(0xffffffffu, hi[r], off));
    }
    if ((threadIdx.x & 31) == 0) { sLo[r][threadIdx.x >> 5] = lo[r]; sHi[r][threadIdx.x >> 5] = hi[r]; }
  }
  __syncthreads();
  if (threadIdx.x < 3)
  {
    float a = sLo[threadIdx.x][0], b = sHi[threadIdx.x][0];
    for (int w = 1; w < kB / 32; ++w) { a = fminf(a, sLo[threadIdx.x][w]); b = fmaxf(b, sHi[threadIdx.x][w]); }
    out[blockIdx.x].lo[threadIdx.x] = a; out[blockIdx.x].hi[threadIdx.x] = b;
  }
}

struct GatherParams
{
  const uint32_t* candidates;      // candidate -> instance, or null: candidate j is instance first + j
  uint32_t numCandidates, first, count, stride;
  const uint8_t* transforms;       // the object->world matrices of instances first .. first + count - 1, `stride` bytes apart
  const float4* o2w;               // the scene's current object->world rows (3 per instance)
  uint32_t* gasSlot;               // instance -> its entry of `gas` (written from the records by rtc_ias_build_device)
  const GasUpdateInput* gas;
  InstanceUpdate* up;
  // created scenes (null otherwise): thread j looks at instance j < numCandidates and appends the records it writes to `up`,
  // counting them in words[kCandidateWord]
  uint32_t* words;
  const uint8_t* records;          // rtc_ias_build_device: rtc_instance_desc of instance i at records + i * stride
  uint32_t numGas;                 // handles in `gas` (the context's table)
  const uint64_t* gasGen;          // per handle: the GAS's generation
  uint64_t* instGen;               // per instance: the generation its record was written at
  uint32_t* gasRefs;               // per handle: instances referencing it (rtc_ias_build_device)
  const void* emptyGas;            // the geometry of a rejected record: one empty node
};

// A created scene's instance j: whether its record is written and, if so, its matrix, GAS entry and (build) material.
__device__ __forceinline__ bool gather_created(const GatherParams& P, uint32_t i, InstanceUpdate& u)
{
  uint32_t h;
  if (P.records)
  {
    const uint8_t* r = P.records + (size_t)i * P.stride;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(r);
    for (int k = 0; k < 12; ++k) u.transform[k] = __uint_as_float(w[k]);
    h = w[13];
    if (w[12] != i || h >= P.numGas || P.gas[h].nodes == nullptr) { h = kRejectedInstance; atomicAdd(P.words + kRejectedWord, 1u); }
    else { atomicAdd(P.gasRefs + h, 1u); P.instGen[i] = P.gasGen[h]; }
    P.gasSlot[i] = h;
    u.materialIndex = (int32_t)w[14]; u.lightIndex = (int32_t)w[15];
  }
  else
  {
    h = P.gasSlot[i];
    const bool changed = h != kRejectedInstance && P.gasGen[h] != P.instGen[i];
    if (i - P.first >= P.count && !changed) return false;
    if (changed) P.instGen[i] = P.gasGen[h];
    if (i - P.first < P.count)
    {
      const float* t = reinterpret_cast<const float*>(P.transforms + (size_t)(i - P.first) * P.stride);
      for (int k = 0; k < 12; ++k) u.transform[k] = t[k];
    }
    else
      for (int r = 0; r < 3; ++r)
      {
        const float4 v = P.o2w[3u * (size_t)i + r];
        u.transform[4 * r] = v.x; u.transform[4 * r + 1] = v.y; u.transform[4 * r + 2] = v.z; u.transform[4 * r + 3] = v.w;
      }
    u.materialIndex = 0; u.lightIndex = 0;
  }
  if (h != kRejectedInstance) u.gas = P.gas[h];
  else
  {
    // an empty GAS: a point box at the origin, and nothing to hit if a ray enters it
    u.gas = GasUpdateInput{};
    u.gas.nodes = P.emptyGas; u.gas.tris = static_cast<const uint8_t*>(P.emptyGas) + sizeof(Node8); u.gas.emptyGas = 1u;
  }
  return true;
}

// One thread per candidate: its matrix (new from `transforms`, or the current one), the inverse (bvh_rules.h, the bits of the
// host's invert_3x4: this file is compiled with -fmad=false) and its GAS's table entry, as the records the two kernels below read.
__global__ void __launch_bounds__(128)
k_instance_gather(const GatherParams P)
{
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= P.numCandidates) return;
  InstanceUpdate u;
  if (P.words)
  {
    if (!gather_created(P, j, u)) return;
    invert_3x4(u.transform, u.inverse);
    u.instance = j; u.pad = 0u;
    P.up[atomicAdd(P.words + kCandidateWord, 1u)] = u;
    return;
  }
  const uint32_t i = P.candidates ? P.candidates[j] : P.first + j;
  if (i - P.first < P.count)                            // unsigned: first <= i < first + count
  {
    const float* t = reinterpret_cast<const float*>(P.transforms + (size_t)(i - P.first) * P.stride);
    for (int k = 0; k < 12; ++k) u.transform[k] = t[k];
  }
  else
  {
    for (int r = 0; r < 3; ++r)
    {
      const float4 v = P.o2w[3u * (size_t)i + r];
      u.transform[4 * r] = v.x; u.transform[4 * r + 1] = v.y; u.transform[4 * r + 2] = v.z; u.transform[4 * r + 3] = v.w;
    }
  }
  invert_3x4(u.transform, u.inverse);
  u.gas = P.gas[P.gasSlot[i]];
  u.instance = i; u.pad = 0u;
  P.up[j] = u;
}

// One thread per written instance: the padded box (instance_box_finish, bvh_rules.h), the instance's 64 B traversal record
// (world->object rows 0..2, row 3 = {GAS nodes, GAS triangles}) and its rows of the shading tables (object->world, the GAS's
// vertex attributes and indices -- rtc_gas_build_device replaces both; with `material` also the record's material and light).
// numUp as in k_instance_bounds.
__global__ void __launch_bounds__(128)
k_instance_finish(const InstanceUpdate* __restrict__ up, uint32_t count, const uint32_t* __restrict__ numUp, const PrimBox* __restrict__ exact,
                  int tight, int material, PrimBox* __restrict__ instBoxes, float4* __restrict__ instances, float4* __restrict__ o2w,
                  rt_GeometryInstanceData* __restrict__ gi)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (numUp ? *numUp : count)) return;
  const InstanceUpdate& u = up[i];
  const GasUpdateInput& g = u.gas;
  float gas[6];
  for (int k = 0; k < 6; ++k) gas[k] = g.gasBox ? g.gasBox[k] : g.gasLoHi[k];
  PrimBox b = {};
  if (tight) b = exact[i];
  instance_box_finish(u.transform, gas, gas + 3, tight != 0, g.emptyGas != 0, b);
  const uint32_t inst = u.instance;
  instBoxes[inst] = b;
  for (int r = 0; r < 3; ++r)
  {
    instances[4u * inst + r] = make_float4(u.inverse[4 * r], u.inverse[4 * r + 1], u.inverse[4 * r + 2], u.inverse[4 * r + 3]);
    o2w[3u * inst + r] = make_float4(u.transform[4 * r], u.transform[4 * r + 1], u.transform[4 * r + 2], u.transform[4 * r + 3]);
  }
  *reinterpret_cast<ulonglong2*>(instances + 4u * inst + 3) = make_ulonglong2((uintptr_t)g.nodes, (uintptr_t)g.tris);
  gi[inst].attributes = g.attributes;
  gi[inst].indices = g.indices;
  if (material) { gi[inst].materialIndex = u.materialIndex; gi[inst].lightIndex = u.lightIndex; }
}

// pooled: from the stream-ordered pool (the instance level: its updates never allocate with a call that may block)
int alloc_refit_scratch(rtc_context* ctx, RefitScratch& r, const uint4* nodes, uint32_t numNodes, bool pooled = false)
{
  if (r.base) return 0;
  const size_t n = numNodes;
  if (pooled) RTC_CUDA(cudaMallocAsync(&r.base, n * (2 * sizeof(uint32_t) + 6 * sizeof(float)), ctx->stream));
  else        RTC_CUDA(cudaMalloc(&r.base, n * (2 * sizeof(uint32_t) + 6 * sizeof(float))));
  r.pooled = pooled;
  r.box = static_cast<float*>(r.base);
  r.parent = reinterpret_cast<uint32_t*>(r.box + 6 * n);
  r.arrivals = r.parent + n;
  RTC_CUDA(cudaMemsetAsync(r.arrivals, 0, n * sizeof(uint32_t), ctx->stream));
  k_refit_parents<<<(numNodes + kB - 1) / kB, kB, 0, ctx->stream>>>(nodes, numNodes, r.parent);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  return 0;
}

// liveCount: the device word that holds the node count (numNodes is then the capacity), or null
int launch_refit_nodes(rtc_context* ctx, const RefitScratch& r, uint4* nodes, uint32_t numNodes, const float4* tris,
                       const uint32_t* leaves, const PrimBox* primBoxes, const uint32_t* liveCount = nullptr)
{
  RefitParams P;
  P.nodes = nodes; P.numNodes = numNodes; P.tris = tris; P.leaves = leaves; P.primBoxes = primBoxes;
  P.parent = r.parent; P.arrivals = r.arrivals; P.box = r.box;
  if (liveCount) k_refit_nodes_live<<<(numNodes + kB - 1) / kB, kB, 0, ctx->stream>>>(P, liveCount);
  else           k_refit_nodes<<<(numNodes + kB - 1) / kB, kB, 0, ctx->stream>>>(P);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  return 0;
}

} // namespace

void free_refit_scratch(RefitScratch& r, cudaStream_t stream)
{
  if (r.pooled) cudaFreeAsync(r.base, stream);
  else cudaFree(r.base);
  r = RefitScratch();
}

int refit_gas_gpu(rtc_context* ctx, GasRecord& rec)
{
  if (rec.numTris == 0) return 0;                       // one empty node: nothing to refit, the bounds stay (0, 0)
  uint4* nodes = static_cast<uint4*>(rec.d_nodes);
  if (int rc = alloc_refit_scratch(ctx, rec.refit, nodes, rec.numNodes)) return rc;
  k_refit_tris<<<(rec.numTris + kB - 1) / kB, kB, 0, ctx->stream>>>(static_cast<float4*>(rec.d_tris), rec.numTris,
                                                                    (const uint8_t*)(uintptr_t)rec.attributes, rec.strideBytes, rec.numVerts,
                                                                    (const uint32_t*)(uintptr_t)rec.indices);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  // after rtc_gas_rebuild the scratch is the rebuild's (sized for the node capacity, parents kept up to date by every rebuild) and
  // the live node count is on the device
  const int rc = rec.rebuild ? launch_refit_nodes(ctx, rec.refit, nodes, ias_rebuild_capacity(rec.numTris), static_cast<const float4*>(rec.d_tris),
                                                  nullptr, nullptr, rec.d_numNodes)
                             : launch_refit_nodes(ctx, rec.refit, nodes, rec.numNodes, static_cast<const float4*>(rec.d_tris), nullptr, nullptr);
  if (rc) return rc;
  rec.boundsOnDevice = true;
  return 0;
}

int write_instance_records_gpu(rtc_context* ctx, SceneRecord& s, const uint8_t* transforms, uint32_t strideBytes, uint32_t first,
                               uint32_t count, const std::vector<uint32_t>& candidates, const std::vector<GasUpdateInput>& gas, bool tight)
{
  const uint32_t m = candidates.empty() ? count : (uint32_t)candidates.size();
  if (m == 0) return 0;
  // the records, exact bounds, per-GAS table and candidate list, one stream-ordered allocation freed behind the kernels; the two
  // host arrays are small (nothing per instance unless a GAS was refitted) and staged by the copies themselves
  const size_t upBytes = m * sizeof(InstanceUpdate), exactBytes = m * sizeof(PrimBox);
  const size_t gasBytes = gas.size() * sizeof(GasUpdateInput), listBytes = candidates.size() * sizeof(uint32_t);
  uint8_t* d = nullptr;
  RTC_CUDA(cudaMallocAsync((void**)&d, upBytes + exactBytes + gasBytes + listBytes, ctx->stream));
  GatherParams P;
  P.up = reinterpret_cast<InstanceUpdate*>(d);
  PrimBox* d_exact = reinterpret_cast<PrimBox*>(d + upBytes);
  GasUpdateInput* d_gas = reinterpret_cast<GasUpdateInput*>(d + upBytes + exactBytes);
  uint32_t* d_list = reinterpret_cast<uint32_t*>(d + upBytes + exactBytes + gasBytes);
  P.candidates = candidates.empty() ? nullptr : d_list;
  P.numCandidates = m; P.first = first; P.count = count; P.stride = strideBytes; P.transforms = transforms;
  P.o2w = static_cast<const float4*>(s.d_o2w); P.gasSlot = s.d_instGasSlot; P.gas = d_gas;
  P.words = nullptr; P.records = nullptr; P.numGas = 0; P.gasGen = nullptr; P.instGen = nullptr; P.gasRefs = nullptr; P.emptyGas = nullptr;
  cudaError_t e = cudaMemcpyAsync(d_gas, gas.data(), gasBytes, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess && listBytes) e = cudaMemcpyAsync(d_list, candidates.data(), listBytes, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess)
  {
    k_instance_gather<<<(m + 127) / 128, 128, 0, ctx->stream>>>(P);
    ctx->kernelLaunches++;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess && tight)
  {
    k_instance_bounds<<<m, kB, 0, ctx->stream>>>(P.up, d_exact, nullptr);
    ctx->kernelLaunches++;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess)
  {
    k_instance_finish<<<(m + 127) / 128, 128, 0, ctx->stream>>>(P.up, m, nullptr, d_exact, tight ? 1 : 0, 0, s.d_instBoxes,
                                                                static_cast<float4*>(s.d_instances), static_cast<float4*>(s.d_o2w),
                                                                static_cast<rt_GeometryInstanceData*>(s.d_geomInst));
    ctx->kernelLaunches++;
    e = cudaGetLastError();
  }
  cudaFreeAsync(d, ctx->stream);
  if (e != cudaSuccess) return rtc_set_error(__FILE__, __LINE__, "write_instance_records_gpu", (int)e, cudaGetErrorString(e));
  return 0;
}

int write_created_records_gpu(rtc_context* ctx, SceneRecord& s, const uint8_t* records, const uint8_t* transforms, uint32_t strideBytes,
                              uint32_t first, uint32_t count, bool tight)
{
  const uint32_t m = s.desc.numInstances;          // every instance may be written: the device selects them
  if (m == 0) return 0;
  const size_t upBytes = m * sizeof(InstanceUpdate);
  uint8_t* d = nullptr;
  RTC_CUDA(cudaMallocAsync((void**)&d, upBytes + m * sizeof(PrimBox), ctx->stream));
  GatherParams P;
  P.candidates = nullptr; P.numCandidates = m; P.first = first; P.count = count; P.stride = strideBytes; P.transforms = transforms;
  P.o2w = static_cast<const float4*>(s.d_o2w); P.gasSlot = s.d_instGasSlot; P.gas = ctx->d_gasTable;
  P.up = reinterpret_cast<InstanceUpdate*>(d);
  P.words = s.d_words; P.records = records; P.numGas = (uint32_t)ctx->gas.size(); P.gasGen = ctx->d_gasGen; P.instGen = s.d_instGen;
  P.gasRefs = s.d_gasRefs; P.emptyGas = s.d_emptyGas;
  PrimBox* d_exact = reinterpret_cast<PrimBox*>(d + upBytes);
  const uint32_t* numUp = s.d_words + kCandidateWord;
  cudaError_t e = cudaMemsetAsync(s.d_words + kCandidateWord, 0, sizeof(uint32_t), ctx->stream);
  if (e == cudaSuccess)
  {
    k_instance_gather<<<(m + 127) / 128, 128, 0, ctx->stream>>>(P);
    ctx->kernelLaunches++;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess && tight)
  {
    k_instance_bounds<<<m, kB, 0, ctx->stream>>>(P.up, d_exact, numUp);
    ctx->kernelLaunches++;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess)
  {
    k_instance_finish<<<(m + 127) / 128, 128, 0, ctx->stream>>>(P.up, m, numUp, d_exact, tight ? 1 : 0, records ? 1 : 0, s.d_instBoxes,
                                                                static_cast<float4*>(s.d_instances), static_cast<float4*>(s.d_o2w),
                                                                static_cast<rt_GeometryInstanceData*>(s.d_geomInst));
    ctx->kernelLaunches++;
    e = cudaGetLastError();
  }
  cudaFreeAsync(d, ctx->stream);
  if (e != cudaSuccess) return rtc_set_error(__FILE__, __LINE__, "write_created_records_gpu", (int)e, cudaGetErrorString(e));
  return 0;
}

// The built node array, or the one rtc_ias_rebuild rebuilt, whose live node count is on the device.
int refit_instance_level_gpu(rtc_context* ctx, SceneRecord& s)
{
  uint4* tlas = static_cast<uint4*>(s.d_tlasNodes);
  // after a rebuild the scratch exists (bvh_build_ias_gpu.cu sized it for the node capacity and keeps its parents up to date)
  if (int rc = alloc_refit_scratch(ctx, s.refit, tlas, s.desc.numTlasNodes, true)) return rc;
  const uint32_t* leaves = static_cast<const uint32_t*>(s.d_tlasLeaves);
  if (s.rebuild)
    return launch_refit_nodes(ctx, s.refit, tlas, ias_rebuild_capacity(s.desc.numInstances), nullptr, leaves, s.d_instBoxes, s.d_numTlasNodes);
  return launch_refit_nodes(ctx, s.refit, tlas, s.desc.numTlasNodes, nullptr, leaves, s.d_instBoxes);
}
