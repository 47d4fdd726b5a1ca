// bvh_rules.h -- arithmetic that the host builder (bvh_build_host.cpp), the device builders (bvh_build_gpu.cu,
// bvh_build_ias_gpu.cu), the device instance records and refit (bvh_refit.cu) and the host-only twins (accel_host.cpp) must apply
// bit for bit: the world->object matrix of an instance, the quantisation of one wide node, the padding of an instance's world box,
// and the Morton codes, radix tree and wide nodes of the LBVH.  One definition, compiled for the host and for sm_100a.
//
// FMA contraction: every product in quantise_node is by a power of two (step * 2^-4, step * 2^-6 with step >= 2^-120, which
// stays a normal float) and is therefore exact, so a contracted multiply-add rounds exactly like the separate operations.
// invert_3x4 and instance_box_finish multiply in double by values that are not powers of two: the host twin compiles them with
// -ffp-contract=off and bvh_refit.cu with -fmad=false.
#pragma once

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>

#include "rtc_internal.h"

#if defined(__CUDACC__)
#define RTC_HD __host__ __device__ __forceinline__
#else
#define RTC_HD inline
#endif

RTC_HD float rules_pow2f(int e)
{
  const uint32_t u = (uint32_t)(e + 127) << 23;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

// Inactive inputs (DESIGN.md section 3).  B = 2^126: coordinates of magnitude up to B keep every node extent within the
// 254 grid steps of 2^120 that quantise_node can represent, so finite inputs up to B are exact.  A triangle with a vertex
// coordinate that is NaN, infinite or beyond B, and an instance whose transform has a non-finite entry or whose world bounds
// reach beyond B, is inactive: its box is the empty box lo = FLT_MAX, hi = -FLT_MAX (centre 0, so the builders' binning and
// Morton codes stay finite; unions skip it and quantise_node gives it an empty slot), and an inactive triangle's leaf record
// holds NaN for v0 (rules_tri_record), so the triangle test never reports it when it shares a leaf with active ones.
#define RTC_COORD_BOUND 0x1p126f

RTC_HD bool rules_in_range(float x) { return fabsf(x) <= RTC_COORD_BOUND; }      // false for NaN, +-inf and beyond B

RTC_HD bool rules_in_range3(const float* p) { return rules_in_range(p[0]) && rules_in_range(p[1]) && rules_in_range(p[2]); }

RTC_HD void rules_empty_box(float lo[3], float hi[3])
{
  for (int k = 0; k < 3; ++k) { lo[k] = 3.402823466e38f; hi[k] = -3.402823466e38f; }
}

// The leaf record of a triangle (v0.xyz | primitive id bits, v1.xyz | 0, v2.xyz | 0).  An inactive triangle's v0 is NaN: that
// makes two edge functions, the determinant and t NaN in the triangle test, so it is never reported.
RTC_HD void rules_tri_record(const float* v0, const float* v1, const float* v2, uint32_t prim, float4 rec[3])
{
  const bool active = rules_in_range3(v0) && rules_in_range3(v1) && rules_in_range3(v2);
  float w;
  memcpy(&w, &prim, 4);
  rec[0] = active ? make_float4(v0[0], v0[1], v0[2], w) : make_float4(__builtin_nanf(""), __builtin_nanf(""), __builtin_nanf(""), w);
  rec[1] = make_float4(v1[0], v1[1], v1[2], 0.0f);
  rec[2] = make_float4(v2[0], v2[1], v2[2], 0.0f);
}

// The position an index past the vertex records reads in rtc_gas_build_device (and the refit and rebuild of its GAS): (NaN, NaN,
// NaN), the quiet NaN of rules_tri_record, so its triangle is inactive.  The host twin appends one such vertex instead.
constexpr uint32_t kMissingVertexBits = 0x7fc00000u;

RTC_HD bool rules_box_empty(const float lo[3], const float hi[3])
{
  return !(lo[0] <= hi[0] && lo[1] <= hi[1] && lo[2] <= hi[2]);
}

// World->object matrix of an instance.  DEFINED here (OptiX computed it inside optixAccelBuild,
// Device.cpp:1478, read back by closesthit.cu:49-52): adjugate / determinant of the upper 3x3 in double,
// rounded once to float; translation -(Minv * t) in double.  The oracle states the same definition.
// rtc_ias_build, rtc_ias_update and rtc_ias_update_device compute it on the device (bvh_refit.cu k_instance_gather), the host twin
// (accel_host.cpp) on the host; IEEE double division and no contraction give the same bits on both.
RTC_HD void invert_3x4(const float m[12], float out[12])
{
  const double a = m[0], b = m[1], c = m[2],  tx = m[3];
  const double d = m[4], e = m[5], f = m[6],  ty = m[7];
  const double g = m[8], h = m[9], i = m[10], tz = m[11];
  const double c00 = e * i - f * h, c01 = c * h - b * i, c02 = b * f - c * e;
  const double c10 = f * g - d * i, c11 = a * i - c * g, c12 = c * d - a * f;
  const double c20 = d * h - e * g, c21 = b * g - a * h, c22 = a * e - b * d;
  const double det = a * c00 + b * c10 + c * c20;
  const double r = 1.0 / det;
  const double i00 = c00 * r, i01 = c01 * r, i02 = c02 * r;
  const double i10 = c10 * r, i11 = c11 * r, i12 = c12 * r;
  const double i20 = c20 * r, i21 = c21 * r, i22 = c22 * r;
  out[0] = (float)i00; out[1] = (float)i01; out[2]  = (float)i02; out[3]  = (float)(-(i00 * tx + i01 * ty + i02 * tz));
  out[4] = (float)i10; out[5] = (float)i11; out[6]  = (float)i12; out[7]  = (float)(-(i10 * tx + i11 * ty + i12 * tz));
  out[8] = (float)i20; out[9] = (float)i21; out[10] = (float)i22; out[11] = (float)(-(i20 * tx + i21 * ty + i22 * tz));
}

// Quantisation frame and conservative planes of one wide node.  child(s, lo, hi) yields the float box of the child in slot s for
// every slot set in `occupied`; the frame is derived from the union of those boxes, which is returned in nodeLo / nodeHi.
// Writes p, e, qlo, qhi; empty slots and slots whose box is empty (rules_box_empty) get qlo = 255, qhi = 0 and stay out of the
// node box.  When every box is empty the node box is empty (lo = INFINITY, hi = -INFINITY) and the frame is p = 0, e = 0.
// imask, childBase, triBase and meta are left alone.
// Per axis: grid step 2^e with (hi - p) <= 254 steps, origin p a sixteenth of a step below the box, so every child plane keeps
// slack on the grid (see DESIGN.md "conservative boxes").
template <class ChildBox>
RTC_HD void quantise_node(uint32_t occupied, const ChildBox& child, Node8& node, float nodeLo[3], float nodeHi[3])
{
  for (int k = 0; k < 3; ++k) { nodeLo[k] = INFINITY; nodeHi[k] = -INFINITY; }
  uint32_t live = 0;
  for (int s = 0; s < 8; ++s)
  {
    if (!(occupied & (1u << s))) continue;
    float lo[3], hi[3];
    child(s, lo, hi);
    if (rules_box_empty(lo, hi)) continue;
    live |= 1u << s;
    for (int k = 0; k < 3; ++k) { nodeLo[k] = lo[k] < nodeLo[k] ? lo[k] : nodeLo[k]; nodeHi[k] = nodeHi[k] < hi[k] ? hi[k] : nodeHi[k]; }
  }
  occupied = live;
  if (!occupied)
  {
    node.px = node.py = node.pz = 0.0f;
    node.ex = node.ey = node.ez = 127;
    uint8_t* q[6] = { node.qlox, node.qloy, node.qloz, node.qhix, node.qhiy, node.qhiz };
    for (int k = 0; k < 6; ++k) for (int s = 0; s < 8; ++s) q[k][s] = k < 3 ? 255 : 0;
    return;
  }
  float maxExt = 0.0f;
  for (int k = 0; k < 3; ++k) { const float d = nodeHi[k] - nodeLo[k]; maxExt = maxExt < d ? d : maxExt; }
  int e[3]; float p[3], step[3];
  for (int k = 0; k < 3; ++k)
  {
    const float floorExt = maxExt * 0x1p-20f < 1.0e-30f ? 1.0e-30f : maxExt * 0x1p-20f;
    const float ext = nodeHi[k] - nodeLo[k] < floorExt ? floorExt : nodeHi[k] - nodeLo[k];
    int ek; frexpf(ext / 253.0f, &ek);            // 2^ek > ext/253
    ek = ek < -120 ? -120 : (ek > 120 ? 120 : ek);
    for (;;)
    {
      step[k] = rules_pow2f(ek);
      p[k] = nodeLo[k] - step[k] * 0.0625f;
      if (!(p[k] < nodeLo[k])) p[k] = nextafterf(nodeLo[k], -INFINITY);
      if (fmaf(254.0f, step[k], p[k]) >= nodeHi[k] || ek >= 120) break;
      ++ek;
    }
    e[k] = ek;
  }
  node.px = p[0]; node.py = p[1]; node.pz = p[2];
  node.ex = (uint8_t)(e[0] + 127); node.ey = (uint8_t)(e[1] + 127); node.ez = (uint8_t)(e[2] + 127);
  uint8_t* qlo[3] = { node.qlox, node.qloy, node.qloz };
  uint8_t* qhi[3] = { node.qhix, node.qhiy, node.qhiz };
  for (int s = 0; s < 8; ++s)
  {
    if (!(occupied & (1u << s))) { for (int k = 0; k < 3; ++k) { qlo[k][s] = 255; qhi[k][s] = 0; } continue; }
    float lo[3], hi[3];
    child(s, lo, hi);
    for (int k = 0; k < 3; ++k)
    {
      int ql = (int)floor(((double)lo[k] - (double)p[k]) / (double)step[k]);
      int qh = (int)ceil(((double)hi[k] - (double)p[k]) / (double)step[k]);
      ql = ql < 0 ? 0 : (ql > 255 ? 255 : ql); qh = qh < 0 ? 0 : (qh > 255 ? 255 : qh);
      // keep at least 1/64 step of slack, evaluated with the arithmetic the kernels use (q * step + p)
      while (ql > 0 && !(fmaf((float)ql, step[k], p[k]) <= lo[k] - step[k] * 0.015625f)) --ql;
      while (qh < 255 && !(fmaf((float)qh, step[k], p[k]) >= hi[k] + step[k] * 0.015625f)) ++qh;
      qlo[k][s] = (uint8_t)ql; qhi[k][s] = (uint8_t)qh;
    }
  }
}

// Refit of one built wide node: the child boxes are re-derived (leaf slots: leafBox(first, count, lo, hi) over primitives
// triBase + offset ..; inner slots: innerBox(childIndex, lo, hi)) and the node is re-quantised.  Topology bytes stay as built.
template <class LeafBox, class InnerBox>
RTC_HD void refit_node(Node8& node, const LeafBox& leafBox, const InnerBox& innerBox, float nodeLo[3], float nodeHi[3])
{
  float cLo[8][3], cHi[8][3];
  uint32_t occupied = 0, inner = 0;
  for (int s = 0; s < 8; ++s)
  {
    if (node.imask & (1u << s)) { innerBox(node.childBase + inner, cLo[s], cHi[s]); ++inner; }
    else if (node.meta[s]) leafBox(node.triBase + (node.meta[s] & 31u), (uint32_t)node.meta[s] >> 5, cLo[s], cHi[s]);
    else continue;
    occupied |= 1u << s;
  }
  quantise_node(occupied, [&](int s, float lo[3], float hi[3]) { for (int k = 0; k < 3; ++k) { lo[k] = cLo[s][k]; hi[k] = cHi[s][k]; } },
                node, nodeLo, nodeHi);
}

// The box the instance level is built over.  tight: b holds the exact bounds of the transformed vertices on entry and is padded
// -- the object-space ray is a ROUNDED transform of the world ray, so a hit found in object space may lie a few ulps outside
// the exact world-space box.  Otherwise b becomes the padded bounds of the eight transformed corners of the GAS box (the
// round-1 bounds, looser for rotated instances).  Instances of an empty GAS, or of one whose triangles are all inactive, get a
// point box at the origin.  An instance whose transform has a non-finite entry, or whose world bounds reach beyond B (tight: the
// exact bounds on entry; otherwise the padded corner box), is inactive: it gets the empty box, which no ray enters.
RTC_HD void instance_box_finish(const float transform[12], const float gasLo[3], const float gasHi[3], bool tight, bool emptyGas, PrimBox& b)
{
  bool active = true;
  for (int k = 0; k < 12; ++k) active = active && rules_in_range(transform[k]);
  if (!active) { rules_empty_box(b.lo, b.hi); return; }
  if (emptyGas || rules_box_empty(gasLo, gasHi)) { for (int k = 0; k < 3; ++k) { b.lo[k] = 0.0f; b.hi[k] = 0.0f; } return; }
  const double ext = fabs((double)gasHi[0] - gasLo[0]) + fabs((double)gasHi[1] - gasLo[1]) + fabs((double)gasHi[2] - gasLo[2]);
  if (tight)
  {
    if (!rules_in_range3(b.lo) || !rules_in_range3(b.hi)) { rules_empty_box(b.lo, b.hi); return; }
    for (int r = 0; r < 3; ++r)
    {
      const float* m = &transform[4 * r];
      const double scale = fabs((double)m[0]) + fabs((double)m[1]) + fabs((double)m[2]);
      // the pad is capped at 2^116 so that exact bounds within B stay finite however large ext * scale is
      const double padLo = fmin((fabs((double)b.lo[r]) + ext * scale) * 1.0e-5, 0x1p116);
      const double padHi = fmin((fabs((double)b.hi[r]) + ext * scale) * 1.0e-5, 0x1p116);
      b.lo[r] = nextafterf((float)((double)b.lo[r] - padLo), -INFINITY);
      b.hi[r] = nextafterf((float)((double)b.hi[r] + padHi), INFINITY);
    }
  }
  else
  {
    for (int k = 0; k < 3; ++k) { b.lo[k] = INFINITY; b.hi[k] = -INFINITY; }
    for (int corner = 0; corner < 8; ++corner)
    {
      const double x = (corner & 1) ? gasHi[0] : gasLo[0], y = (corner & 2) ? gasHi[1] : gasLo[1], z = (corner & 4) ? gasHi[2] : gasLo[2];
      for (int r = 0; r < 3; ++r)
      {
        const float* m = &transform[4 * r];
        const double wv = m[0] * x + m[1] * y + m[2] * z + m[3];
        const double scale = fabs((double)m[0]) + fabs((double)m[1]) + fabs((double)m[2]);
        const double pad = (fabs(wv) + ext * scale) * 1.0e-5;
        const float lo = nextafterf((float)(wv - pad), -INFINITY);
        const float hi = nextafterf((float)(wv + pad), INFINITY);
        b.lo[r] = fminf(b.lo[r], lo); b.hi[r] = fmaxf(b.hi[r], hi);
      }
    }
    if (!rules_in_range3(b.lo) || !rules_in_range3(b.hi)) rules_empty_box(b.lo, b.hi);
  }
}

// ---- LBVH (Karras 2012) ---------------------------------------------------------------------------------------------------------
RTC_HD unsigned long long lbvh_spread21(uint32_t v)
{
  unsigned long long x = v & 0x1fffffull;
  x = (x | (x << 32)) & 0x1f00000000ffffull;
  x = (x | (x << 16)) & 0x1f0000ff0000ffull;
  x = (x | (x << 8))  & 0x100f00f00f00f00full;
  x = (x | (x << 4))  & 0x10c30c30c30c30c3ull;
  x = (x | (x << 2))  & 0x1249249249249249ull;
  return x;
}

// 63-bit Morton code of the centre of the box (lo, hi) in the frame sceneBox = {lo[3], hi[3]}
RTC_HD unsigned long long lbvh_morton(const float4 lo, const float4 hi, const float* sceneBox)
{
  const float c[3] = { 0.5f * (lo.x + hi.x), 0.5f * (lo.y + hi.y), 0.5f * (lo.z + hi.z) };
  uint32_t q[3];
  for (int k = 0; k < 3; ++k)
  {
    const float ext = sceneBox[3 + k] - sceneBox[k];
    float u = ext > 0.0f ? (c[k] - sceneBox[k]) / ext : 0.5f;
    u = fminf(fmaxf(u, 0.0f), 1.0f);
    q[k] = (uint32_t)fminf(u * 2097152.0f, 2097151.0f);
  }
  return (lbvh_spread21(q[0]) << 2) | (lbvh_spread21(q[1]) << 1) | lbvh_spread21(q[2]);
}

// common prefix length of sorted keys i and j, index bits break ties between equal codes
RTC_HD int lbvh_delta(const unsigned long long* __restrict__ keys, int n, int i, int j)
{
  if (j < 0 || j >= n) return -1;
  const unsigned long long a = keys[i], b = keys[j];
#if defined(__CUDA_ARCH__)
  if (a != b) return __clzll((long long)(a ^ b));
  return 64 + __clz(i ^ j);
#else
  if (a != b) return __builtin_clzll(a ^ b);
  return 64 + __builtin_clz((unsigned)(i ^ j));
#endif
}

// Internal node i (0 <= i < n - 1) of the binary radix tree over n sorted keys: node ids 0..n-2 are internal (0 = root),
// n-1..2n-2 the leaves (sorted position p -> n-1+p).
RTC_HD void lbvh_radix_node(const unsigned long long* __restrict__ keys, int n, int i, int2* __restrict__ child, int* __restrict__ parent,
                            int2* __restrict__ range)
{
  const int d = (lbvh_delta(keys, n, i, i + 1) - lbvh_delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
  const int dmin = lbvh_delta(keys, n, i, i - d);
  int lmax = 2;
  while (lbvh_delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
  int l = 0;
  for (int t = lmax >> 1; t >= 1; t >>= 1) if (lbvh_delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
  const int j = i + l * d;
  const int dnode = lbvh_delta(keys, n, i, j);
  int s = 0;
  for (int t = (l + 1) >> 1; ; t = (t + 1) >> 1)
  {
    if (lbvh_delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    if (t == 1) break;
  }
#if defined(__CUDA_ARCH__)
  const int gamma = i + s * d + min(d, 0);
  const int first = min(i, j), last = max(i, j);
#else
  const int gamma = i + s * d + std::min(d, 0);
  const int first = std::min(i, j), last = std::max(i, j);
#endif
  const int left = (first == gamma) ? (n - 1 + gamma) : gamma;
  const int right = (last == gamma + 1) ? (n - 1 + gamma + 1) : (gamma + 1);
  child[i] = make_int2(left, right);
  range[i] = make_int2(first, last);
  parent[left] = i;
  parent[right] = i;
  if (i == 0) parent[0] = -1;
}

// One wide node of the instance-level LBVH (one instance per leaf slot) over binary node src of the radix tree: the greedy
// collapse of the geometry builder's k_collapse_level (open the child with the largest surface area until eight remain, octant
// slots, bvh_rules quantisation).  box(id, lo, hi) yields a binary node's box, child(id) its children.  kidAt[s] = the binary
// node in slot s or -1; the node gets imask and meta (leaf offsets in slot order), childBase = triBase = 0.
template <class Box, class Child>
RTC_HD void lbvh_instance_node(int src, int n, const Box& box, const Child& child, int kidAt[8], Node8& node, uint32_t& numInner,
                               uint32_t& numLeaves)
{
  auto is_leaf = [&](int id) { return id >= n - 1; };
  auto half_area = [](const float lo[3], const float hi[3]) {
    const float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    return dx * dy + dy * dz + dz * dx;
  };
  int kids[8]; int nk = 0;
  float kLo[8][3], kHi[8][3];
  if (is_leaf(src)) kids[nk++] = src;
  else { const int2 c = child(src); kids[nk++] = c.x; kids[nk++] = c.y; }
  for (int i = 0; i < nk; ++i) box(kids[i], kLo[i], kHi[i]);
  while (nk < 8)
  {
    int best = -1; float bestArea = -1.0f;
    for (int i = 0; i < nk; ++i)
      if (!is_leaf(kids[i])) { const float a = half_area(kLo[i], kHi[i]); if (a > bestArea) { bestArea = a; best = i; } }
    if (best < 0) break;
    const int2 c = child(kids[best]);
    kids[best] = c.x; kids[nk] = c.y;
    box(c.x, kLo[best], kHi[best]); box(c.y, kLo[nk], kHi[nk]);
    ++nk;
  }
  float sLo[3], sHi[3];
  box(src, sLo, sHi);
  int slotKid[8]; for (int s = 0; s < 8; ++s) slotKid[s] = -1;
  {
    float centre[3]; for (int k = 0; k < 3; ++k) centre[k] = 0.5f * (sLo[k] + sHi[k]);
    uint32_t slotUsed = 0, kidDone = 0;
    for (int round = 0; round < nk; ++round)
    {
      int bi = -1, bs = -1; float bc = -3.402823466e38f;
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
      slotKid[bs] = bi; slotUsed |= 1u << bs; kidDone |= 1u << bi;
    }
  }
  uint32_t occupied = 0;
  for (int s = 0; s < 8; ++s) if (slotKid[s] >= 0) occupied |= 1u << s;
  float nodeLo[3], nodeHi[3];
  quantise_node(occupied, [&](int s, float lo[3], float hi[3]) {
    for (int k = 0; k < 3; ++k) { lo[k] = kLo[slotKid[s]][k]; hi[k] = kHi[slotKid[s]][k]; }
  }, node, nodeLo, nodeHi);
  node.imask = 0; node.childBase = 0; node.triBase = 0;
  numInner = 0; numLeaves = 0;
  for (int s = 0; s < 8; ++s)
  {
    node.meta[s] = 0;
    kidAt[s] = slotKid[s] >= 0 ? kids[slotKid[s]] : -1;
    if (kidAt[s] < 0) continue;
    if (is_leaf(kidAt[s])) { node.meta[s] = (uint8_t)((1u << 5) | numLeaves); ++numLeaves; }
    else { node.imask |= (uint8_t)(1u << s); ++numInner; }
  }
}
