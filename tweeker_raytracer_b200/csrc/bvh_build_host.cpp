// bvh_build_host.cpp -- quality builder for the wide BVH: binned-SAH binary tree on the host,
// greedy surface-area collapse to 8 children, octant slot assignment, conservative quantisation.
//
// Replaces optixAccelBuild (apps/rtigo3/src/Device.cpp:1401 triangles, :1478 instances), which has no
// source in the reference.  Used for the instance level and for small / medium geometry; the GPU LBVH
// builder (bvh_build_gpu.cu) takes over for large inputs and emits the same node format through
// emit_wide_from_binary().
#include "rtc_internal.h"
#include "bvh_rules.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>

namespace {

struct Box
{
  float lo[3], hi[3];
  void clear() { for (int k = 0; k < 3; ++k) { lo[k] = std::numeric_limits<float>::infinity(); hi[k] = -lo[k]; } }
  void grow(const float* l, const float* h) { for (int k = 0; k < 3; ++k) { lo[k] = std::min(lo[k], l[k]); hi[k] = std::max(hi[k], h[k]); } }
  float halfArea() const
  {
    if (rules_box_empty(lo, hi)) return 0.0f;       // only inactive primitives (bvh_rules.h): nothing to intersect
    const float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    return dx * dy + dy * dz + dz * dx;
  }
};

struct BinNode
{
  Box      box;
  int32_t  left = -1, right = -1;   // -1: leaf
  uint32_t first = 0, count = 0;    // leaf range in the ordered primitive list
};

constexpr int kBins = 32;
constexpr uint32_t kLeafMax = 3;    // a leaf child of a wide node carries 1..3 primitives (3 bits of meta)

// SAH bin of a centre; clamped in float before the conversion, because centres of boxes near the float limit overflow to
// infinity and the conversion of a NaN or an out-of-range value is undefined
inline int bin_of(float centre, float lo, float scale)
{
  const float f = (centre - lo) * scale;
  return f >= (float)(kBins - 1) ? kBins - 1 : (f > 0.0f ? (int)f : 0);
}

struct Builder
{
  const PrimBox* prims;
  uint32_t leafMax = kLeafMax;
  float splitCost = 1.2f;           // cost of one more node level relative to one triangle test (SAH termination of small leaves)
  std::vector<uint32_t> order;
  std::vector<BinNode> nodes;

  int build(uint32_t first, uint32_t count)
  {
    const int idx = (int)nodes.size();
    nodes.emplace_back();
    Box box, cbox; box.clear(); cbox.clear();
    for (uint32_t i = first; i < first + count; ++i)
    {
      const PrimBox& p = prims[order[i]];
      box.grow(p.lo, p.hi);
      float c[3]; for (int k = 0; k < 3; ++k) c[k] = 0.5f * (p.lo[k] + p.hi[k]);
      cbox.grow(c, c);
    }
    nodes[idx].box = box;
    nodes[idx].first = first; nodes[idx].count = count;
    if (count <= 1) return idx;

    int bestAxis = -1, bestSplit = 0; float bestCost = std::numeric_limits<float>::infinity();
    for (int axis = 0; axis < 3; ++axis)
    {
      const float ext = cbox.hi[axis] - cbox.lo[axis];
      if (!(ext > 0.0f)) continue;
      Box bb[kBins]; uint32_t bc[kBins];
      for (int b = 0; b < kBins; ++b) { bb[b].clear(); bc[b] = 0; }
      const float scale = (float)kBins / ext;
      for (uint32_t i = first; i < first + count; ++i)
      {
        const PrimBox& p = prims[order[i]];
        const int b = bin_of(0.5f * (p.lo[axis] + p.hi[axis]), cbox.lo[axis], scale);
        bb[b].grow(p.lo, p.hi); bc[b]++;
      }
      float rightArea[kBins]; uint32_t rightCount[kBins]; Box acc; acc.clear(); uint32_t n = 0;
      for (int b = kBins - 1; b > 0; --b) { if (bc[b]) acc.grow(bb[b].lo, bb[b].hi); n += bc[b]; rightArea[b] = n ? acc.halfArea() : 0.0f; rightCount[b] = n; }
      acc.clear(); n = 0;
      for (int b = 0; b < kBins - 1; ++b)
      {
        if (bc[b]) acc.grow(bb[b].lo, bb[b].hi);
        n += bc[b];
        if (n == 0 || rightCount[b + 1] == 0) continue;
        const float cost = acc.halfArea() * (float)n + rightArea[b + 1] * (float)rightCount[b + 1];
        if (cost < bestCost) { bestCost = cost; bestAxis = axis; bestSplit = b; }
      }
    }
    // SAH termination for small leaves: intersecting `count` primitives vs. one more node level
    if (count <= leafMax)
    {
      const float leafCost = box.halfArea() * (float)count;
      if (bestAxis < 0 || bestCost + splitCost * box.halfArea() >= leafCost) return idx;
    }
    uint32_t mid;
    if (bestAxis < 0)
    {
      mid = first + count / 2;
    }
    else
    {
      const float ext = cbox.hi[bestAxis] - cbox.lo[bestAxis];
      const float scale = (float)kBins / ext;
      const float clo = cbox.lo[bestAxis];
      auto it = std::partition(order.begin() + first, order.begin() + first + count, [&](uint32_t pi) {
        const PrimBox& p = prims[pi];
        return bin_of(0.5f * (p.lo[bestAxis] + p.hi[bestAxis]), clo, scale) <= bestSplit;
      });
      mid = (uint32_t)(it - order.begin());
      if (mid == first || mid == first + count) mid = first + count / 2;
    }
    const int l = build(first, mid - first);
    const int r = build(mid, first + count - mid);
    nodes[idx].left = l; nodes[idx].right = r;
    return idx;
  }
};

// SAH-optimal collapse of the binary tree into 8-wide nodes (after Ylitie, Karras, Laine, HPG 2017, section 4.1).  The
// leaves are given, so the cost that is left to minimise is the summed surface area of the wide nodes.  For every binary node
// n: t[n][i] = the smallest such sum when the subtree of n is represented by a forest of at most i roots, each root a leaf or a
// wide node.
//   leaf n : t[n][i] = 0
//   inner n: t[n][1] = area(n) + D(n, 8)                       one wide node whose <= 8 children cover the subtree
//            t[n][i] = min(D(n, i), t[n][i - 1])               2 <= i <= 7
//            D(n, j) = min over 0 < k < j of t[left][k] + t[right][j - k]
// The greedy rule (open the child with the largest area until there are eight) fills the upper levels well but leaves the
// bottom of the tree with two- and three-child nodes: 3.6 children per node on the instanced stress scene.
struct Collapse
{
  struct Entry
  {
    double  t[8];          // t[i - 1] = cost with at most i roots
    uint8_t split[9];      // split[j]: roots given to the left child in D(n, j), j = 2..8
    uint8_t take[8];       // take[i - 1]: the budget t[n][i] actually uses (<= i); 1 means "n is one root"
  };
  const std::vector<BinNode>& bn;
  std::vector<Entry> e;

  explicit Collapse(const std::vector<BinNode>& nodes) : bn(nodes) {}

  // children are created after their parent (Builder::build), so a reverse sweep is bottom-up
  void run()
  {
    e.resize(bn.size());
    for (size_t n = bn.size(); n-- > 0;)
    {
      Entry& x = e[n];
      if (bn[n].left < 0)
      {
        for (int i = 0; i < 8; ++i) { x.t[i] = 0.0; x.take[i] = 1; }
        continue;
      }
      const Entry& l = e[(size_t)bn[n].left];
      const Entry& r = e[(size_t)bn[n].right];
      double D[9];
      for (int j = 2; j <= 8; ++j)
      {
        D[j] = std::numeric_limits<double>::infinity();
        for (int k = 1; k < j; ++k)
        {
          const double c = l.t[k - 1] + r.t[j - k - 1];
          if (c < D[j]) { D[j] = c; x.split[j] = (uint8_t)k; }
        }
      }
      x.t[0] = (double)bn[n].box.halfArea() + D[8]; x.take[0] = 1;
      for (int i = 2; i <= 8; ++i)
      {
        if (i == 8) break;
        if (D[i] < x.t[i - 2]) { x.t[i - 1] = D[i]; x.take[i - 1] = (uint8_t)i; }
        else                   { x.t[i - 1] = x.t[i - 2]; x.take[i - 1] = x.take[i - 2]; }
      }
    }
  }

  // appends the roots of the optimal forest of subtree n with at most `budget` roots
  void roots(int n, int budget, int* kids, int& count) const
  {
    const int use = (bn[n].left < 0) ? 1 : (int)e[(size_t)n].take[budget - 1];
    if (use == 1) { kids[count++] = n; return; }
    const int k = (int)e[(size_t)n].split[use];
    roots(bn[n].left, k, kids, count);
    roots(bn[n].right, use - k, kids, count);
  }

  // the children of the wide node rooted at inner binary node n
  int children(int n, int* kids) const
  {
    int count = 0;
    const int k = (int)e[(size_t)n].split[8];
    roots(bn[n].left, k, kids, count);
    roots(bn[n].right, 8 - k, kids, count);
    return count;
  }
};

struct Emitter
{
  const std::vector<BinNode>& bn;
  const std::vector<uint32_t>& order;
  WideBvh& out;
  const Collapse* collapse;     // null: the greedy collapse (the default)

  // writes wide node `dst` for the binary subtree `src`
  void emit(uint32_t dst, int src)
  {
    // 1. collect up to 8 children
    int kids[8]; int n = 0;
    if (bn[src].left < 0) { kids[n++] = src; }
    else if (collapse) { n = collapse->children(src, kids); }
    else
    {
      // greedy: open the inner child with the largest surface area first
      kids[n++] = bn[src].left; kids[n++] = bn[src].right;
      while (n < 8)
      {
        int best = -1; float bestArea = -1.0f;
        for (int i = 0; i < n; ++i)
          if (bn[kids[i]].left >= 0) { const float a = bn[kids[i]].box.halfArea(); if (a > bestArea) { bestArea = a; best = i; } }
        if (best < 0) break;
        const int k = kids[best];
        kids[best] = bn[k].left;
        kids[n++] = bn[k].right;
      }
    }

    // 2. assign children to octant slots: greedy max of dot(child centre - node centre, slot sign vector)
    const Box& box = bn[src].box;
    float centre[3]; for (int k = 0; k < 3; ++k) centre[k] = 0.5f * (box.lo[k] + box.hi[k]);
    float cost[8][8];
    for (int i = 0; i < n; ++i)
    {
      const Box& cb = bn[kids[i]].box;
      float d[3]; for (int k = 0; k < 3; ++k) d[k] = 0.5f * (cb.lo[k] + cb.hi[k]) - centre[k];
      for (int s = 0; s < 8; ++s)
        cost[i][s] = ((s & 4) ? d[0] : -d[0]) + ((s & 2) ? d[1] : -d[1]) + ((s & 1) ? d[2] : -d[2]);
    }
    int slotOf[8]; bool slotUsed[8] = {}; bool kidDone[8] = {};
    for (int round = 0; round < n; ++round)
    {
      int bi = -1, bs = -1; float bc = -std::numeric_limits<float>::infinity();
      for (int i = 0; i < n; ++i) if (!kidDone[i])
        for (int s = 0; s < 8; ++s) if (!slotUsed[s] && (cost[i][s] > bc || bi < 0)) { bc = cost[i][s]; bi = i; bs = s; }
      slotOf[bi] = bs; slotUsed[bs] = true; kidDone[bi] = true;
    }
    int kidAt[8]; for (int s = 0; s < 8; ++s) kidAt[s] = -1;
    for (int i = 0; i < n; ++i) kidAt[slotOf[i]] = kids[i];

    // 3. quantisation frame and conservative child planes (bvh_rules.h)
    Node8 node; std::memset(&node, 0, sizeof(node));
    uint32_t occupied = 0;
    for (int s = 0; s < 8; ++s) if (kidAt[s] >= 0) occupied |= 1u << s;
    float nodeLo[3], nodeHi[3];
    quantise_node(occupied, [&](int s, float lo[3], float hi[3]) {
      const Box& cb = bn[kidAt[s]].box;
      for (int k = 0; k < 3; ++k) { lo[k] = cb.lo[k]; hi[k] = cb.hi[k]; }
    }, node, nodeLo, nodeHi);

    // 4. children: inner ones get one contiguous block of wide nodes, leaf primitives one contiguous run
    uint32_t numInner = 0;
    for (int s = 0; s < 8; ++s) if (kidAt[s] >= 0 && bn[kidAt[s]].left >= 0) { node.imask |= (uint8_t)(1u << s); ++numInner; }
    node.childBase = (uint32_t)out.nodes.size();
    out.nodes.resize(out.nodes.size() + numInner);
    node.triBase = (uint32_t)out.primOrder.size();
    uint32_t triOffset = 0;
    for (int s = 0; s < 8; ++s)
    {
      if (kidAt[s] < 0) continue;
      const BinNode& c = bn[kidAt[s]];
      if (c.left < 0)
      {
        node.meta[s] = (uint8_t)((c.count << 5) | triOffset);
        for (uint32_t i = 0; i < c.count; ++i) out.primOrder.push_back(order[c.first + i]);
        triOffset += c.count;
      }
    }
    out.nodes[dst] = node;
    uint32_t rel = 0;
    for (int s = 0; s < 8; ++s)
      if (node.imask & (1u << s)) { emit(node.childBase + rel, kidAt[s]); ++rel; }
  }
};

} // namespace

void build_wide_bvh_host(const PrimBox* prims, uint32_t numPrims, WideBvh& out, uint32_t leafMax, bool instanceLevel)
{
  out.nodes.clear(); out.primOrder.clear();
  for (int k = 0; k < 3; ++k) { out.lo[k] = 0.0f; out.hi[k] = 0.0f; }
  if (numPrims == 0)
  {
    // one empty node: every slot is empty, traversal falls straight through
    Node8 node; std::memset(&node, 0, sizeof(node));
    node.ex = node.ey = node.ez = 127;
    for (int s = 0; s < 8; ++s) { node.qlox[s] = node.qloy[s] = node.qloz[s] = 255; }
    out.nodes.push_back(node);
    return;
  }
  Builder b; b.prims = prims;
  b.leafMax = std::min(std::max(leafMax, 1u), kLeafMax);
  b.order.resize(numPrims);
  for (uint32_t i = 0; i < numPrims; ++i) b.order[i] = i;
  b.nodes.reserve(2 * (size_t)numPrims);
  const int root = b.build(0, numPrims);
  for (int k = 0; k < 3; ++k) { out.lo[k] = b.nodes[root].box.lo[k]; out.hi[k] = b.nodes[root].box.hi[k]; }
  out.nodes.reserve(numPrims / 2 + 8);
  out.primOrder.reserve(numPrims);
  out.nodes.emplace_back();
  // Collapse: greedy (open the largest child first) unless RTC_HOST_COLLAPSE=optimal (geometry level) / RTC_TLAS_COLLAPSE=optimal
  // (instance level) selects the SAH-optimal dynamic programme.  The optimal collapse needs 30-48 % fewer nodes and visits 3-7 %
  // fewer of them per ray, but a warp pays per iteration for the lane with the MOST triangles, and full bottom nodes hand one
  // lane more triangles at a time; instance-level leaves of one node are entered without a new box test, so a fuller
  // instance-level node culls less.  The lock-step warp model of tests/tools/simd_cost.py (which reproduces the sign and size of
  // six A/Bs round 2 measured on a B200) puts it at -3 % on the geometry scene, -2 % on the Cornell box, +2 % on the instanced
  // stress scene (profiles/bvh_quality_r2.md); no GPU measurement of it exists, so the measured collapse stays the default.
  const char* mode = getenv(instanceLevel ? "RTC_TLAS_COLLAPSE" : "RTC_HOST_COLLAPSE");
  const bool greedy = !(mode && mode[0] == 'o');
  Collapse collapse(b.nodes);
  if (!greedy) collapse.run();
  Emitter em{ b.nodes, b.order, out, greedy ? nullptr : &collapse };
  em.emit(0, root);
}

// Binned-SAH binary tree with single-primitive leaves; used by the GPU builder for the top levels over a cut of its
// radix tree.  children[i] = (left, right), a negative value ~k means primitive k; node 0 is the root.
void build_binary_sah_host(const PrimBox* prims, uint32_t numPrims, std::vector<int2>& children, std::vector<PrimBox>& boxes)
{
  Builder b; b.prims = prims; b.leafMax = 1;
  b.order.resize(numPrims);
  for (uint32_t i = 0; i < numPrims; ++i) b.order[i] = i;
  b.nodes.reserve(2 * (size_t)numPrims);
  b.build(0, numPrims);
  // renumber: internal nodes get consecutive ids in creation order (the root was created first)
  std::vector<int> id(b.nodes.size(), -1);
  int next = 0;
  for (size_t i = 0; i < b.nodes.size(); ++i) if (b.nodes[i].left >= 0) id[i] = next++;
  children.assign((size_t)next, make_int2(0, 0));
  boxes.assign((size_t)next, PrimBox());
  auto ref = [&](int node) { return b.nodes[node].left >= 0 ? id[node] : ~(int)b.order[b.nodes[node].first]; };
  for (size_t i = 0; i < b.nodes.size(); ++i)
  {
    if (b.nodes[i].left < 0) continue;
    children[(size_t)id[i]] = make_int2(ref(b.nodes[i].left), ref(b.nodes[i].right));
    PrimBox pb;
    for (int k = 0; k < 3; ++k) { pb.lo[k] = b.nodes[i].box.lo[k]; pb.hi[k] = b.nodes[i].box.hi[k]; }
    boxes[(size_t)id[i]] = pb;
  }
}
