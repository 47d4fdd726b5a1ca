// tests/native/primary_lists_host.cpp -- TEST INFRASTRUCTURE: the PRODUCT's tile lists of the primary rays compiled for the host.
//
// csrc/primary_lists.cuh (tile frustum, list builder, list pass) together with csrc/shade.cuh (start_path, the pinhole lens
// shader) and csrc/trace.cuh (through trace_host.cpp, which gives the CUDA intrinsics their IEEE meaning), compiled unchanged by
// g++ with -ffp-contract=off.  pl_primary plays the depth-0 extend of one iteration of a pinhole launch the way the kernels do:
// a list per 8x4 tile, the list pass for the 32 rays of a listed tile, the traversal for an overflowed one -- and, for every
// ray, the traversal alone, so that tests/test_cpu_primary_lists.py can compare the two bit for bit.
#include "trace_host.cpp"
#include "shade.cuh"
#include "primary_lists.cuh"

extern "C" {

uint32_t pl_list_capacity() { return kTileListK; }

// sys.cameraDefinitions points at a host copy of the camera.  Per launch index (tile-major, 32 per tile, as the kernels number paths): listHits
// (what the split extend stores), travHits (the traversal alone).  Per tile: tileCounts (entries or kTileOverflow) and
// travCounts[3] (the traversal's nodes, triangles, instance entries over the tile's 32 rays).
int pl_primary(const th_scene* ws, uint32_t numTlasNodes, uint32_t numTlasLeaves, uint32_t numGas, const uint32_t* numGasNodes,
               const uint32_t* numGasTris, const rt_SystemData* sys, uint32_t w, uint32_t h, int iteration,
               rtc_hit* listHits, rtc_hit* travHits, uint32_t* tileCounts, uint64_t* travCounts)
{
  if ((w & 7u) || (h & 3u)) return -1;
  HostScene hs;
  build_host_scene(hs, ws, numTlasNodes, numTlasLeaves, numGas, numGasNodes, numGasTris);
  const SceneDesc& sc = hs.sc;

  const uint32_t tilesPerRow = w >> 3, tiles = (w >> 3) * (h >> 2);
  std::vector<uint2> list(kTileListK);
  uint2 smStack[RTC_SM_STACK]; float smRay[RTC_SM_RAY_WORDS]; uint2 lmStack[RTC_LM_STACK];
  for (uint32_t tile = 0; tile < tiles; ++tile)
  {
    const uint32_t ty = tile / tilesPerRow, tx = tile - ty * tilesPerRow;
    float P[3], n[4][3], c[3];
    const uint32_t count = tile_planes(*sys, tx << 3, ty << 2, P, n, c) ? build_tile_list(sc, P, n, c, list.data()) : kTileOverflow;
    tileCounts[tile] = count;
    uint64_t* tc = travCounts + 3 * (size_t)tile;
    tc[0] = tc[1] = tc[2] = 0;
    for (uint32_t lane = 0; lane < 32u; ++lane)
    {
      const uint32_t idx = tile * 32u + lane, x = (tx << 3) + (lane & 7u), y = (ty << 2) + (lane >> 3);
      uint32_t seed = 0, col = 0; float3 pos, wi;
      if (!start_path(*sys, w, x, y, iteration, seed, pos, wi, col)) return -2;
      const float4 o = make_float4(pos.x, pos.y, pos.z, sys->sceneEpsilon), dir = make_float4(wi.x, wi.y, wi.z, RT_DEFAULT_MAX);
      Traversal<false, true, 1, false> tr;
      tr.smStack = smStack; tr.smRay = smRay; tr.lmStack = lmStack;
      if (tr.begin(sc, o, dir))
      {
        while (tr.step(sc)) {}
        tc[0] += tr.counts.nodes; tc[1] += tr.counts.tris; tc[2] += tr.counts.insts;
      }
      const TraceHit a = tr.result();
      const TraceHit b = count == kTileOverflow ? a : trace_tile_list(sc, list.data(), count, o, dir);
      travHits[idx].t = a.t; travHits[idx].u = a.u; travHits[idx].v = a.v; travHits[idx].inst = a.inst; travHits[idx].prim = a.prim;
      listHits[idx].t = b.t; listHits[idx].u = b.u; listHits[idx].v = b.v; listHits[idx].inst = b.inst; listHits[idx].prim = b.prim;
    }
  }
  return 0;
}

} // extern "C"
