/* tests/native/anyhit_predicates.h -- TEST INFRASTRUCTURE: the any-hit decisions the tests of include/rtc_device.cuh use, compiled
 * by nvcc (the user kernels of device_anyhit_kernels.cu), by g++ (the host build of the header, device_anyhit_host.cpp) and by gcc
 * (the brute force of oracle_anyhit.c).  Every decision is an exact function of the candidate's bits, so the three agree.
 *
 * ahp_decide(pred, candidate, p0, p1, end):
 *   AHP_ACCEPT       every candidate
 *   AHP_IGNORE       no candidate (an any query then visits every candidate of the ray)
 *   AHP_ALPHA        (inst, prim) hashed: transparent with probability p0 / 256, else checkered with probability 1/4 (opaque where
 *                    floor(u * 8) + floor(v * 8) is even), else opaque
 *   AHP_FRONT        front-facing candidates only
 *   AHP_NOT_SELF     every candidate but (inst, prim) = (p0, p1)
 * end != 0: an accept is RTC_ANYHIT_ACCEPT_AND_END (2).
 */
#ifndef ANYHIT_PREDICATES_H
#define ANYHIT_PREDICATES_H

#include <stdint.h>
#include <string.h>
#include <math.h>

#if defined(__CUDACC__)
#define AHP_FN static __host__ __device__ __forceinline__
#else
#define AHP_FN static inline
#endif

enum { AHP_ACCEPT = 0, AHP_IGNORE = 1, AHP_ALPHA = 2, AHP_FRONT = 3, AHP_NOT_SELF = 4 };

AHP_FN uint32_t ahp_hash(uint32_t x)
{
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}

AHP_FN uint32_t ahp_bits(float f)
{
  uint32_t u;
  memcpy(&u, &f, 4);
  return u;
}

/* 0 transparent, 1 opaque */
AHP_FN int ahp_alpha(uint32_t inst, uint32_t prim, float u, float v, uint32_t transparentPer256)
{
  const uint32_t h = ahp_hash(ahp_hash(inst ^ 0x9e3779b9u) ^ prim);
  if ((h & 0xffu) < transparentPer256) return 0;
  if (((h >> 8) & 3u) == 0u) return (((int)floorf(u * 8.0f) + (int)floorf(v * 8.0f)) & 1) == 0;
  return 1;
}

AHP_FN int ahp_decide(int pred, float t, float u, float v, uint32_t inst, uint32_t prim, uint32_t frontFacing, uint32_t p0, uint32_t p1,
                      int end)
{
  int accept;
  (void)t;
  switch (pred)
  {
  case AHP_ACCEPT:   accept = 1; break;
  case AHP_ALPHA:    accept = ahp_alpha(inst, prim, u, v, p0); break;
  case AHP_FRONT:    accept = frontFacing != 0u; break;
  case AHP_NOT_SELF: accept = !(inst == p0 && prim == p1); break;
  default:           accept = 0; break;
  }
  return accept ? (end ? 2 : 1) : 0;
}

/* order-independent digest of a set of candidates: d[0] count, d[1] sum, d[2] XOR of a hash of (t, u, v, inst, prim, frontFacing) */
AHP_FN uint32_t ahp_candidate_hash(float t, float u, float v, uint32_t inst, uint32_t prim, uint32_t frontFacing)
{
  uint32_t h = ahp_hash(ahp_bits(t) ^ 0x85ebca6bu);
  h = ahp_hash(h ^ ahp_bits(u)); h = ahp_hash(h ^ ahp_bits(v));
  h = ahp_hash(h ^ inst); h = ahp_hash(h ^ prim);
  return ahp_hash(h ^ frontFacing);
}

AHP_FN void ahp_digest_add(uint32_t d[3], float t, float u, float v, uint32_t inst, uint32_t prim, uint32_t frontFacing)
{
  const uint32_t h = ahp_candidate_hash(t, u, v, inst, prim, frontFacing);
  d[0] += 1u; d[1] += h; d[2] ^= h;
}

/* one candidate as the tests record it (the layout of rtc_candidate) */
typedef struct { float t, u, v; uint32_t inst, prim, frontFacing; } ahp_record;

#endif
