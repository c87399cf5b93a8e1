// host_refit_check.cpp — the device refit source (refit.cuh: child boxes -> node box -> re-quantised node, bottom-up by level)
// compiled for the host through host_shim.h: build the tree with the product's builder, move a third of the triangles (rigid
// offset + squash), refit level by level, then check nearest hits against brute force over the MOVED triangles with the device
// traversal source (traverse.cuh).  Exit code 0 iff every ray agrees bit for bit.
//   host_refit_check dump.bin [maxRays]
#include "host_shim.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../refit.cuh"

using namespace pt;

int main(int argc, char** argv)
{
  if(argc < 2) { std::fprintf(stderr, "usage: host_refit_check dump.bin [maxRays]\n"); return 2; }
  FILE* f = std::fopen(argv[1], "rb");
  uint32_t nT, nR;
  if(!f || std::fread(&nT, 4, 1, f) != 1 || std::fread(&nR, 4, 1, f) != 1) return 2;
  std::vector<float> tv((size_t)nT * 9), rv((size_t)nR * 8);
  if(std::fread(tv.data(), 4, tv.size(), f) != tv.size() || std::fread(rv.data(), 4, rv.size(), f) != rv.size()) return 2;
  std::fclose(f);
  if(argc > 2) nR = std::min<uint32_t>(nR, (uint32_t)std::atoi(argv[2]));
  std::vector<FlatTri>  tris(nT);
  std::vector<uint32_t> gids(nT);
  for(uint32_t i = 0; i < nT; i++)
  {
    std::memcpy(tris[i].v0, &tv[i * 9], 12); std::memcpy(tris[i].e1, &tv[i * 9 + 3], 12); std::memcpy(tris[i].e2, &tv[i * 9 + 6], 12);
    tris[i].rnode = 0; tris[i].prim = i; tris[i].flags = TRI_NOCULL | TRI_OPAQUE; gids[i] = i;
  }
  WideBvh B;
  buildWideBvh(tris, gids, 0, B);
  // move every third triangle (by global id): the records of the tree are rewritten in place, like k_refit_tris does
  for(uint32_t s = 0; s < B.numTris; s++)
  {
    float*   T = &B.tris[(size_t)s * 12];
    uint32_t gid; std::memcpy(&gid, &T[11], 4);
    if(gid % 3u) continue;
    T[0] += 0.37f; T[1] = T[1] * 0.8f + 0.11f; T[2] -= 0.23f;
    T[5] *= 0.8f; T[9] *= 0.8f;
  }
  // level ranges (breadth-first emission)
  std::vector<std::pair<uint32_t, uint32_t>> levels;
  for(uint32_t first = 0, count = 1; count;)
  {
    levels.push_back({first, count});
    uint32_t next = 0;
    for(uint32_t n = first; n < first + count; n++) next += (uint32_t)__builtin_popcount(__float_as_uint(B.nodes[(size_t)n * 20 + 3]) >> 24);
    first += count; count = next;
  }
  std::vector<float4> nodeBox((size_t)B.numNodes * 2);
  for(size_t l = levels.size(); l-- > 0;)
    for(uint32_t i = 0; i < levels[l].second; i++)
      refitNode(levels[l].first + i, B.nodes.data(), B.tris.data(), nodeBox.data());
  std::printf("tris %u nodes %u levels %zu rays %u, root box (%.3f %.3f %.3f)-(%.3f %.3f %.3f)\n", B.numTris, B.numNodes, levels.size(), nR, nodeBox[0].x, nodeBox[0].y,
              nodeBox[0].z, nodeBox[1].x, nodeBox[1].y, nodeBox[1].z);
  BvhView view{reinterpret_cast<const float4*>(B.nodes.data()), reinterpret_cast<const float4*>(B.tris.data())};
  uint64_t bad = 0, hits = 0;
  for(uint32_t r = 0; r < nR; r++)
  {
    const float* R = &rv[(size_t)r * 8];
    const float3 org = f3(R[0], R[1], R[2]), dir = f3(R[4], R[5], R[6]);
    float bt = R[7]; uint32_t bg = 0xFFFFFFFFu;
    for(uint32_t s = 0; s < B.numTris; s++)
    {
      const float* T = &B.tris[(size_t)s * 12];
      const float3 v0 = f3(T[0], T[1], T[2]), e1 = f3(T[4], T[5], T[6]), e2 = f3(T[8], T[9], T[10]);
      const float3 pvec = crossFma(dir, e2);
      const float  det = dotFma(e1, pvec), inv = 1.0f / det;
      const float3 tvec = org - v0;
      const float  u = dotFma(tvec, pvec) * inv;
      const float3 qvec = crossFma(tvec, e1);
      const float  v = dotFma(dir, qvec) * inv, t = dotFma(e2, qvec) * inv;
      uint32_t gid; std::memcpy(&gid, &T[11], 4);
      if((det != 0.0f) & (u >= 0.0f) & (u <= 1.0f) & (v >= 0.0f) & (u + v <= 1.0f) & (t > 0.0f) & (t < R[7]) && (t < bt || (t == bt && gid < bg))) { bt = t; bg = gid; }
    }
    Cand     cand[kCand];
    TraceHit opq; opq.slot = 0xFFFFFFFFu;
    walkCollect(view, org, dir, 0.0f, R[7], false, false, true, false, 0.f, 0u, opq, cand);
    const bool ok = (bg == 0xFFFFFFFFu) ? (opq.slot == 0xFFFFFFFFu) : (opq.slot != 0xFFFFFFFFu && opq.gid == bg && __float_as_uint(opq.t) == __float_as_uint(bt));
    bad += !ok; hits += bg != 0xFFFFFFFFu;
  }
  std::printf("hit rate %.3f, mismatches after refit: %llu\n", (double)hits / nR, (unsigned long long)bad);
  return bad ? 1 : 0;
}
