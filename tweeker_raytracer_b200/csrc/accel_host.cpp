// accel_host.cpp -- the host halves of the acceleration-structure builds, free of CUDA calls.
//
// rtc_gas_build (host SAH builder) and rtc_ias_build in rtc_api.cpp fetch their inputs from the device, call the functions
// below and upload what they return.  The same functions sit behind rtc_host_gas_build / rtc_host_ias_build
// (include/rtc_core.h), the host-only twin of the two builds: tools and the CPU tests build exactly the arrays a B200 would
// be handed -- wide nodes, leaf-ordered triangles, instance-level leaves, world->object matrices -- and the scalar oracle
// traverses them in the kernels' order of operations (oracle/wide_bvh.inc).  Nothing here renders or intersects anything.
#include "rtc_internal.h"
#include "bvh_rules.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>

// Host quality build of one geometry: triangle boxes, binned SAH, collapse, quantisation, triangles in leaf order
// (v0.xyz | primitive id bits, v1.xyz | 0, v2.xyz | 0).  Returns false when an index is out of range.
bool gas_assemble_host(const uint8_t* verts, uint32_t strideBytes, uint32_t numVerts, const uint32_t* idx, uint32_t numTris,
                       WideBvh& bvh, std::vector<float4>& tris)
{
  std::vector<PrimBox> boxes(numTris);
  auto vertex = [&](uint32_t i) { return reinterpret_cast<const float*>(verts + (size_t)i * strideBytes); };
  for (uint32_t t = 0; t < numTris; ++t)
  {
    PrimBox& b = boxes[t];
    for (int k = 0; k < 3; ++k) { b.lo[k] = std::numeric_limits<float>::infinity(); b.hi[k] = -b.lo[k]; }
    for (int c = 0; c < 3; ++c)
    {
      const uint32_t vi = idx[3u * t + c];
      if (vi >= numVerts) return false;
      const float* p = vertex(vi);
      for (int k = 0; k < 3; ++k) { b.lo[k] = std::fmin(b.lo[k], p[k]); b.hi[k] = std::fmax(b.hi[k], p[k]); }
    }
  }
  // triangles per leaf child of the host SAH build.  2: geometry scene 2526 -> 2545 Msamples/s, Cornell box 809 -> 820 against
  // leaves of up to 3; 1 is better only for the instanced scene (355 -> 368) and loses 2 % elsewhere.  RTC_HOST_LEAF_MAX overrides.
  uint32_t leafMax = 2;
  if (const char* e = getenv("RTC_HOST_LEAF_MAX")) { const int v = atoi(e); if (1 <= v && v <= 3) leafMax = (uint32_t)v; }
  build_wide_bvh_host(boxes.data(), numTris, bvh, leafMax);
  tris.resize((size_t)numTris * 3u);
  for (uint32_t s = 0; s < numTris; ++s)
  {
    const uint32_t prim = bvh.primOrder[s];
    for (int c = 0; c < 3; ++c)
    {
      const float* p = vertex(idx[3u * prim + c]);
      float w = 0.0f;
      if (c == 0) std::memcpy(&w, &prim, 4);
      tris[3u * (size_t)s + c] = make_float4(p[0], p[1], p[2], w);
    }
  }
  return true;
}

// Exact world bounds of the transformed vertices of one instance, in the arithmetic of k_instance_bounds (bvh_refit.cu):
// one fmaf chain per row, min / max are order-independent, so the device reduction and this loop agree bit for bit.
void instance_bounds_host(const float transform[12], const uint8_t* verts, uint32_t strideBytes, uint32_t numVerts, PrimBox& out)
{
  float lo[3] = { std::numeric_limits<float>::max(), std::numeric_limits<float>::max(), std::numeric_limits<float>::max() };
  float hi[3] = { -lo[0], -lo[1], -lo[2] };
  for (uint32_t v = 0; v < numVerts; ++v)
  {
    const float* p = reinterpret_cast<const float*>(verts + (size_t)v * strideBytes);
    for (int r = 0; r < 3; ++r)
    {
      const float* m = transform + 4 * r;
      const float w = std::fmaf(m[0], p[0], std::fmaf(m[1], p[1], std::fmaf(m[2], p[2], m[3])));
      lo[r] = std::fmin(lo[r], w); hi[r] = std::fmax(hi[r], w);
    }
  }
  for (int r = 0; r < 3; ++r) { out.lo[r] = lo[r]; out.hi[r] = hi[r]; }
}

bool instance_bounds_tight()
{
  const char* e = getenv("RTC_INSTANCE_BOUNDS");
  return !(e && e[0] == 'b');
}

void tlas_build_host(const PrimBox* boxes, uint32_t numInstances, WideBvh& bvh)
{
  build_wide_bvh_host(boxes, numInstances, bvh, getenv("RTC_TLAS_LEAF") ? (uint32_t)atoi(getenv("RTC_TLAS_LEAF")) : 1u, true);
}

// ------------------------------------------------------------------------------------------------
// Host-only twin of rtc_gas_build(RTC_BUILD_HOST_SAH) + rtc_ias_build (include/rtc_core.h)
// ------------------------------------------------------------------------------------------------
struct rtc_host_accel;

namespace {

// The node refit of bvh_refit.cu on host arrays: descending node index is bottom-up, because both builders place every child
// above its parent.  The root's box becomes the bounds of the structure.
template <class LeafBox>
void refit_host(WideBvh& bvh, const LeafBox& leafBox)
{
  std::vector<float> box(bvh.nodes.size() * 6u);
  for (size_t i = bvh.nodes.size(); i-- > 0;)
    refit_node(bvh.nodes[i], leafBox, [&](uint32_t child, float lo[3], float hi[3]) {
      for (int k = 0; k < 3; ++k) { lo[k] = box[6u * child + k]; hi[k] = box[6u * child + 3 + k]; }
    }, &box[6u * i], &box[6u * i + 3]);
  for (int k = 0; k < 3; ++k) { bvh.lo[k] = box[k]; bvh.hi[k] = box[3 + k]; }
}

} // namespace

struct rtc_host_accel
{
  bool isInstanceLevel = false;
  WideBvh bvh;
  std::vector<float4> tris;             // geometry level
  std::vector<uint8_t> positions;       // geometry level: vertex positions, 12 B apart (for the instance bounds and the rebuild)
  std::vector<uint32_t> indices;        // geometry level: the build's index triplets (for the refit)
  uint32_t numVerts = 0, numTris = 0, strideBytes = 0;
  std::vector<float> inverses;          // instance level: 12 floats per instance
  std::vector<PrimBox> boxes;           // instance level: the padded instance boxes of the last build / refit (for the rebuild)
};

// world->object matrices and padded world boxes of every instance, as rtc_ias_build computes them; false on a bad geometry handle
static bool instance_boxes_host(const float* transforms, const rtc_host_accel* const* geometry, uint32_t numInstances,
                                std::vector<float>& inverses, std::vector<PrimBox>& boxes)
{
  for (uint32_t i = 0; i < numInstances; ++i) if (!geometry[i] || geometry[i]->isInstanceLevel) return false;
  boxes.assign(numInstances, PrimBox());
  const bool tight = instance_bounds_tight();
  for (uint32_t i = 0; i < numInstances; ++i)
  {
    const rtc_host_accel* g = geometry[i];
    const float* m = transforms + 12u * (size_t)i;
    invert_3x4(m, &inverses[(size_t)i * 12u]);
    if (tight) instance_bounds_host(m, g->positions.data(), 12u, g->numTris ? g->numVerts : 0u, boxes[i]);
    instance_box_finish(m, g->bvh.lo, g->bvh.hi, tight, g->numTris == 0, boxes[i]);
  }
  return true;
}

extern "C" {

int rtc_host_gas_build(const void* attributes, uint32_t strideBytes, uint32_t numVerts, const uint32_t* indices, uint32_t numTris,
                       rtc_host_accel** out)
{
  if (!out) RTC_FAIL("out is null");
  if (strideBytes < 12 || (strideBytes & 3u)) RTC_FAIL("vertex stride must be a multiple of 4 and at least 12");
  if ((numVerts && !attributes) || (numTris && !indices)) RTC_FAIL("null input array");
  rtc_host_accel* a = new rtc_host_accel();
  a->numVerts = numVerts; a->numTris = numTris; a->strideBytes = strideBytes;
  if (!gas_assemble_host(static_cast<const uint8_t*>(attributes), strideBytes, numVerts, indices, numTris, a->bvh, a->tris))
  {
    delete a;
    RTC_FAIL("triangle index out of range");
  }
  a->positions.resize((size_t)numVerts * 12u);
  for (uint32_t v = 0; v < numVerts; ++v) std::memcpy(&a->positions[(size_t)v * 12u], static_cast<const uint8_t*>(attributes) + (size_t)v * strideBytes, 12);
  a->indices.assign(indices, indices + 3u * (size_t)numTris);
  *out = a;
  return 0;
}

int rtc_host_ias_build(const float* transforms, const rtc_host_accel* const* geometry, uint32_t numInstances, rtc_host_accel** out)
{
  if (!out) RTC_FAIL("out is null");
  if (numInstances && (!transforms || !geometry)) RTC_FAIL("null input array");
  rtc_host_accel* a = new rtc_host_accel();
  a->isInstanceLevel = true;
  a->inverses.resize((size_t)numInstances * 12u);
  std::vector<PrimBox> boxes;
  if (!instance_boxes_host(transforms, geometry, numInstances, a->inverses, boxes)) { delete a; RTC_FAIL("bad geometry handle in instance"); }
  tlas_build_host(boxes.data(), numInstances, a->bvh);
  a->boxes = std::move(boxes);
  *out = a;
  return 0;
}

int rtc_host_gas_refit(rtc_host_accel* accel, const void* attributes, uint32_t strideBytes)
{
  if (!accel || accel->isInstanceLevel) RTC_FAIL("not a geometry-level accel");
  if (strideBytes != accel->strideBytes) RTC_FAIL("vertex stride differs from the build's");
  if (accel->numVerts && !attributes) RTC_FAIL("null input array");
  const uint8_t* verts = static_cast<const uint8_t*>(attributes);
  for (uint32_t v = 0; v < accel->numVerts; ++v) std::memcpy(&accel->positions[(size_t)v * 12u], verts + (size_t)v * strideBytes, 12);
  for (uint32_t s = 0; s < accel->numTris; ++s)
  {
    const uint32_t prim = accel->bvh.primOrder[s];
    for (int c = 0; c < 3; ++c)
    {
      const float* p = reinterpret_cast<const float*>(verts + (size_t)accel->indices[3u * prim + c] * strideBytes);
      float4& r = accel->tris[3u * (size_t)s + c];
      r.x = p[0]; r.y = p[1]; r.z = p[2];
    }
  }
  if (accel->numTris == 0) return 0;
  const std::vector<float4>& tris = accel->tris;
  refit_host(accel->bvh, [&](uint32_t first, uint32_t count, float lo[3], float hi[3]) {
    for (int k = 0; k < 3; ++k) { lo[k] = INFINITY; hi[k] = -INFINITY; }
    for (uint32_t t = first; t < first + count; ++t)
      for (int c = 0; c < 3; ++c)
      {
        const float4& v = tris[3u * (size_t)t + c];
        const float x[3] = { v.x, v.y, v.z };
        for (int k = 0; k < 3; ++k) { lo[k] = x[k] < lo[k] ? x[k] : lo[k]; hi[k] = hi[k] < x[k] ? x[k] : hi[k]; }
      }
  });
  return 0;
}

int rtc_host_ias_refit(rtc_host_accel* accel, const float* transforms, const rtc_host_accel* const* geometry, uint32_t numInstances)
{
  if (!accel || !accel->isInstanceLevel) RTC_FAIL("not an instance-level accel");
  if ((size_t)numInstances * 12u != accel->inverses.size()) RTC_FAIL("instance count differs from the build's");
  if (numInstances && (!transforms || !geometry)) RTC_FAIL("null input array");
  std::vector<PrimBox> boxes;
  if (!instance_boxes_host(transforms, geometry, numInstances, accel->inverses, boxes)) RTC_FAIL("bad geometry handle in instance");
  accel->boxes = boxes;
  if (numInstances == 0) return 0;
  const std::vector<uint32_t>& leaves = accel->bvh.primOrder;
  refit_host(accel->bvh, [&](uint32_t first, uint32_t count, float lo[3], float hi[3]) {
    for (int k = 0; k < 3; ++k) { lo[k] = INFINITY; hi[k] = -INFINITY; }
    for (uint32_t t = first; t < first + count; ++t)
    {
      const PrimBox& b = boxes[leaves[t]];
      for (int k = 0; k < 3; ++k) { lo[k] = b.lo[k] < lo[k] ? b.lo[k] : lo[k]; hi[k] = hi[k] < b.hi[k] ? b.hi[k] : hi[k]; }
    }
  });
  return 0;
}

} // extern "C"

// The steps of the device rebuilds (lbvh_collapse.cuh) on host arrays: centre bounds, Morton codes, a stable sort, the radix tree,
// the fit (min / max, exact in any order) and the breadth-first collapse, whose running counters are the device's per-level
// exclusive scans.  out.primOrder: leaf slot -> primitive; out.lo / hi: the fitted box of the root.
static void lbvh_rebuild_host(const std::vector<PrimBox>& boxes, WideBvh& out)
{
  const int n = (int)boxes.size();
  std::vector<float4> lo(n), hi(n);
  float centreBox[6] = { FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX };
  for (int i = 0; i < n; ++i)
  {
    const PrimBox& b = boxes[i];
    lo[i] = make_float4(b.lo[0], b.lo[1], b.lo[2], 0.0f);
    hi[i] = make_float4(b.hi[0], b.hi[1], b.hi[2], 0.0f);
    for (int k = 0; k < 3; ++k)
    {
      const float c = 0.5f * (b.lo[k] + b.hi[k]);
      centreBox[k] = std::fmin(centreBox[k], c); centreBox[3 + k] = std::fmax(centreBox[3 + k], c);
    }
  }
  std::vector<unsigned long long> code(n);
  std::vector<uint32_t> order(n);
  for (int i = 0; i < n; ++i) { code[i] = lbvh_morton(lo[i], hi[i], centreBox); order[i] = (uint32_t)i; }
  std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return code[a] < code[b]; });
  std::vector<unsigned long long> keys(n);
  for (int p = 0; p < n; ++p) keys[p] = code[order[p]];

  // binary tree: ids 0..n-2 internal, n-1..2n-2 leaves; the fit climbs from every leaf, the second child to arrive carries on
  std::vector<int2> child(n > 1 ? n - 1 : 1), range(n > 1 ? n - 1 : 1);
  std::vector<int> parent(2 * (size_t)n, -1);
  for (int i = 0; i < n - 1; ++i) lbvh_radix_node(keys.data(), n, i, child.data(), parent.data(), range.data());
  std::vector<PrimBox> box(2 * (size_t)n);
  std::vector<uint8_t> arrived(n, 0);
  for (int p = 0; p < n; ++p)
  {
    box[n - 1 + p] = boxes[order[p]];
    if (n == 1) break;
    for (int node = parent[n - 1 + p]; node >= 0; node = parent[node])
    {
      if (!arrived[node]++) break;
      const PrimBox &a = box[child[node].x], &b = box[child[node].y];
      for (int k = 0; k < 3; ++k) { box[node].lo[k] = std::fmin(a.lo[k], b.lo[k]); box[node].hi[k] = std::fmax(a.hi[k], b.hi[k]); }
    }
  }

  out.nodes.assign(1, Node8());
  out.primOrder.assign(n, 0u);
  std::vector<int2> work(1, make_int2(0, 0)), next;
  uint32_t numNodes = 1, numLeaves = 0;
  while (!work.empty())
  {
    next.clear();
    for (const int2& item : work)
    {
      int kidAt[8];
      Node8 node;
      uint32_t numInner, nodeLeaves;
      lbvh_instance_node(item.x, n,
                         [&](int id, float l[3], float h[3]) { for (int k = 0; k < 3; ++k) { l[k] = box[id].lo[k]; h[k] = box[id].hi[k]; } },
                         [&](int id) { return child[id]; }, kidAt, node, numInner, nodeLeaves);
      if (numInner) node.childBase = numNodes;
      if (nodeLeaves) node.triBase = numLeaves;
      for (int s = 0; s < 8; ++s)
      {
        if (kidAt[s] < 0) continue;
        if (kidAt[s] >= n - 1) out.primOrder[numLeaves++] = order[kidAt[s] - (n - 1)];
        else next.push_back(make_int2(kidAt[s], (int)numNodes++));
      }
      out.nodes[item.y] = node;
    }
    out.nodes.resize(numNodes);
    work.swap(next);
  }
  for (int k = 0; k < 3; ++k) { out.lo[k] = box[0].lo[k]; out.hi[k] = box[0].hi[k]; }
}

extern "C" {

int rtc_host_ias_rebuild(rtc_host_accel* accel)
{
  if (!accel || !accel->isInstanceLevel) RTC_FAIL("not an instance-level accel");
  if (accel->boxes.empty()) return 0;
  lbvh_rebuild_host(accel->boxes, accel->bvh);
  return 0;
}

// rtc_gas_rebuild (bvh_build_gas_rebuild_gpu.cu): triangle boxes as k_gas_boxes computes them, the LBVH over them, the triangle
// records in leaf order
int rtc_host_gas_rebuild(rtc_host_accel* accel, const void* attributes, uint32_t strideBytes)
{
  if (!accel || accel->isInstanceLevel) RTC_FAIL("not a geometry-level accel");
  if (attributes)
  {
    if (strideBytes != accel->strideBytes) RTC_FAIL("vertex stride differs from the build's");
    const uint8_t* verts = static_cast<const uint8_t*>(attributes);
    for (uint32_t v = 0; v < accel->numVerts; ++v) std::memcpy(&accel->positions[(size_t)v * 12u], verts + (size_t)v * strideBytes, 12);
  }
  const uint32_t n = accel->numTris;
  if (n == 0) return 0;
  auto vertex = [&](uint32_t prim, int c) { return reinterpret_cast<const float*>(&accel->positions[(size_t)accel->indices[3u * prim + c] * 12u]); };
  std::vector<PrimBox> boxes(n);
  for (uint32_t t = 0; t < n; ++t)
  {
    PrimBox& b = boxes[t];
    for (int k = 0; k < 3; ++k) { b.lo[k] = FLT_MAX; b.hi[k] = -FLT_MAX; }
    for (int c = 0; c < 3; ++c)
    {
      const float* p = vertex(t, c);
      for (int k = 0; k < 3; ++k) { b.lo[k] = std::fmin(b.lo[k], p[k]); b.hi[k] = std::fmax(b.hi[k], p[k]); }
    }
  }
  lbvh_rebuild_host(boxes, accel->bvh);
  for (uint32_t s = 0; s < n; ++s)
  {
    const uint32_t prim = accel->bvh.primOrder[s];
    for (int c = 0; c < 3; ++c)
    {
      const float* p = vertex(prim, c);
      float w = 0.0f;
      if (c == 0) std::memcpy(&w, &prim, 4);
      accel->tris[3u * (size_t)s + c] = make_float4(p[0], p[1], p[2], w);
    }
  }
  return 0;
}

int rtc_host_accel_info(const rtc_host_accel* accel, uint64_t* numNodes, uint64_t* numPrims, float bounds[6])
{
  if (!accel) RTC_FAIL("accel is null");
  if (numNodes) *numNodes = accel->bvh.nodes.size();
  if (numPrims) *numPrims = accel->bvh.primOrder.size();
  if (bounds) for (int k = 0; k < 3; ++k) { bounds[k] = accel->bvh.lo[k]; bounds[3 + k] = accel->bvh.hi[k]; }
  return 0;
}

int rtc_host_accel_export(const rtc_host_accel* accel, void* nodes, uint32_t* primOrder, float* tris, float* worldToObject)
{
  if (!accel) RTC_FAIL("accel is null");
  if (nodes) std::memcpy(nodes, accel->bvh.nodes.data(), accel->bvh.nodes.size() * sizeof(Node8));
  if (primOrder && !accel->bvh.primOrder.empty()) std::memcpy(primOrder, accel->bvh.primOrder.data(), accel->bvh.primOrder.size() * 4u);
  if (tris && !accel->tris.empty()) std::memcpy(tris, accel->tris.data(), accel->tris.size() * sizeof(float4));
  if (worldToObject && !accel->inverses.empty()) std::memcpy(worldToObject, accel->inverses.data(), accel->inverses.size() * sizeof(float));
  return 0;
}

void rtc_host_accel_destroy(rtc_host_accel* accel) { delete accel; }

} // extern "C"
