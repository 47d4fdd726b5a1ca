// bvh_rules.h -- arithmetic that the host builder (bvh_build_host.cpp), the device builder (bvh_build_gpu.cu), the device refit
// (bvh_refit.cu) and the host-only refit twin (accel_host.cpp) must apply bit for bit: the quantisation of one wide node and the
// padding of an instance's world box.  One definition, compiled for the host and for sm_100a.
//
// FMA contraction: every product in quantise_node is by a power of two (step * 2^-4, step * 2^-6 with step >= 2^-120, which
// stays a normal float) and is therefore exact, so a contracted multiply-add rounds exactly like the separate operations.
// instance_box_finish multiplies in double by values that are not powers of two: the host compiles it with
// -ffp-contract=off and bvh_refit.cu with -fmad=false.
#pragma once

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

// Quantisation frame and conservative planes of one wide node.  child(s, lo, hi) yields the float box of the child in slot s for
// every slot set in `occupied`; the frame is derived from the union of those boxes, which is returned in nodeLo / nodeHi.
// Writes p, e, qlo, qhi; empty slots get qlo = 255, qhi = 0.  imask, childBase, triBase and meta are left alone.
// Per axis: grid step 2^e with (hi - p) <= 254 steps, origin p a sixteenth of a step below the box, so every child plane keeps
// slack on the grid (see DESIGN.md "conservative boxes").
template <class ChildBox>
RTC_HD void quantise_node(uint32_t occupied, const ChildBox& child, Node8& node, float nodeLo[3], float nodeHi[3])
{
  for (int k = 0; k < 3; ++k) { nodeLo[k] = INFINITY; nodeHi[k] = -INFINITY; }
  for (int s = 0; s < 8; ++s)
  {
    if (!(occupied & (1u << s))) continue;
    float lo[3], hi[3];
    child(s, lo, hi);
    for (int k = 0; k < 3; ++k) { nodeLo[k] = lo[k] < nodeLo[k] ? lo[k] : nodeLo[k]; nodeHi[k] = nodeHi[k] < hi[k] ? hi[k] : nodeHi[k]; }
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
// round-1 bounds, looser for rotated instances).  Instances of an empty GAS get a point box at the origin.
RTC_HD void instance_box_finish(const float transform[12], const float gasLo[3], const float gasHi[3], bool tight, bool emptyGas, PrimBox& b)
{
  const double ext = fabs((double)gasHi[0] - gasLo[0]) + fabs((double)gasHi[1] - gasLo[1]) + fabs((double)gasHi[2] - gasLo[2]);
  if (tight)
  {
    for (int r = 0; r < 3; ++r)
    {
      const float* m = &transform[4 * r];
      const double scale = fabs((double)m[0]) + fabs((double)m[1]) + fabs((double)m[2]);
      const double padLo = (fabs((double)b.lo[r]) + ext * scale) * 1.0e-5, padHi = (fabs((double)b.hi[r]) + ext * scale) * 1.0e-5;
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
  }
  if (emptyGas) { for (int k = 0; k < 3; ++k) { b.lo[k] = 0.0f; b.hi[k] = 0.0f; } }
}
