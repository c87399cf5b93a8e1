// host_lbvh_check.cpp — the DEVICE LBVH build source (lbvh.cuh: Morton keys, bitonic sort, Karras hierarchy, bottom-up fit, level-
// by-level collapse into compressed 8-wide nodes) run on the host, "thread" after "thread", through host_shim.h, then walked by
// the device traversal source (traverse.cuh) and checked against brute force: nearest hit in (t, id) order, bit for bit; plus
// structural checks (every triangle emitted exactly once, node / triangle counters consistent).
//   host_lbvh_check dump.bin [maxRays]
#include "host_shim.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../lbvh.cuh"

using namespace pt;

int main(int argc, char** argv)
{
  if(argc < 2) { std::fprintf(stderr, "usage: host_lbvh_check dump.bin [maxRays]\n"); return 2; }
  FILE* f = std::fopen(argv[1], "rb");
  uint32_t nT, nR;
  if(!f || std::fread(&nT, 4, 1, f) != 1 || std::fread(&nR, 4, 1, f) != 1) return 2;
  std::vector<float> tv((size_t)nT * 9), rv((size_t)nR * 8);
  if(std::fread(tv.data(), 4, tv.size(), f) != tv.size() || std::fread(rv.data(), 4, rv.size(), f) != rv.size()) return 2;
  std::fclose(f);
  if(argc > 2) nR = std::min<uint32_t>(nR, (uint32_t)std::atoi(argv[2]));
  // records in flatten order; the tree is built over every second triangle + a few (a subset, like the opaque-only tree)
  std::vector<float> rec((size_t)nT * 12);
  for(uint32_t i = 0; i < nT; i++)
  {
    float* R = &rec[(size_t)i * 12];
    std::memcpy(R, &tv[i * 9], 12); std::memcpy(R + 4, &tv[i * 9 + 3], 12); std::memcpy(R + 8, &tv[i * 9 + 6], 12);
    R[3] = __uint_as_float(0u | ((TRI_NOCULL | TRI_OPAQUE) << 28)); R[7] = __uint_as_float(i); R[11] = __uint_as_float(i);
  }
  std::vector<uint32_t> subset;
  for(uint32_t i = 0; i < nT; i++) if(i % 2 == 0 || i % 7 == 0) subset.push_back(i);
  const uint32_t m = (uint32_t)subset.size();
  uint32_t M = 1; while(M < m) M <<= 1;
  std::vector<float4> primLo(m), primHi(m), boxLo(m), boxHi(m);
  std::vector<unsigned long long> keys(M);
  std::vector<int> left(m), right(m), parentI(m), parentL(m);
  std::vector<uint32_t> first(m), last(m), visits(m, 0), triMeta((size_t)m * 2), counters(3, 0);
  std::vector<float> nodes((size_t)m * 20 + 20, 0.f), tris((size_t)m * 12);
  int cb[6] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int)0x80000000, (int)0x80000000, (int)0x80000000};
  LbvhWork W{m, M, rec.data(), subset.data(), primLo.data(), primHi.data(), keys.data(), left.data(), right.data(), parentI.data(), parentL.data(), first.data(),
             last.data(), boxLo.data(), boxHi.data(), visits.data(), cb, nodes.data(), tris.data(), triMeta.data(), 0u, counters.data()};
  for(uint32_t i = 0; i < m; i++) lbvhBounds(i, W);
  for(uint32_t i = 0; i < M; i++) lbvhMorton(i, W);
  for(uint32_t k = 2; k <= M; k <<= 1)
    for(uint32_t j = k >> 1; j > 0; j >>= 1)
      for(uint32_t t = 0; t < M; t++) bitonicStep(t, keys.data(), j, k);
  for(uint32_t i = 1; i < m; i++) if(!(keys[i - 1] < keys[i])) { std::printf("sort broken at %u\n", i); return 1; }
  for(uint32_t i = 0; i + 1 < m; i++) lbvhHierarchy(i, W);
  for(uint32_t i = 0; i < m; i++) lbvhFit(i, W);
  // level loop
  std::vector<int2> qa(m + 1), qb(m + 1);
  qa[0] = make_int2(m >= 2 ? 0 : ~0, 0);
  uint32_t count = 1, levels = 0;
  counters[0] = 1;
  while(count)
  {
    counters[2] = 0;
    for(uint32_t q = 0; q < count; q++) lbvhEmit(q, W, qa.data(), qb.data());
    count = counters[2];
    std::swap(qa, qb);
    levels++;
  }
  const uint32_t numNodes = counters[0];
  std::printf("subset %u of %u triangles -> %u wide nodes, %u triangles emitted, %u levels\n", m, nT, numNodes, counters[1], levels);
  if(counters[1] != m) return 1;
  std::vector<int> seen(nT, 0);
  for(uint32_t s = 0; s < m; s++) seen[__float_as_uint(tris[(size_t)s * 12 + 11])]++;
  for(uint32_t i = 0; i < nT; i++) if(seen[i] != ((i % 2 == 0 || i % 7 == 0) ? 1 : 0)) { std::printf("triangle %u emitted %d times\n", i, seen[i]); return 1; }
  BvhView  view{reinterpret_cast<const float4*>(nodes.data()), reinterpret_cast<const float4*>(tris.data())};
  uint64_t bad = 0, hits = 0;
  int      maxSp = 0;
  for(uint32_t r = 0; r < nR; r++)
  {
    const float* R = &rv[(size_t)r * 8];
    const float3 org = f3(R[0], R[1], R[2]), dir = f3(R[4], R[5], R[6]);
    float bt = R[7]; uint32_t bg = 0xFFFFFFFFu;
    for(uint32_t k = 0; k < m; k++)
    {
      const float* T = &rec[(size_t)subset[k] * 12];
      const float3 v0 = f3(T[0], T[1], T[2]), e1 = f3(T[4], T[5], T[6]), e2 = f3(T[8], T[9], T[10]);
      const float3 pvec = crossFma(dir, e2);
      const float  det = dotFma(e1, pvec), inv = 1.0f / det;
      const float3 tvec = org - v0;
      const float  u = dotFma(tvec, pvec) * inv;
      const float3 qvec = crossFma(tvec, e1);
      const float  v = dotFma(dir, qvec) * inv, t = dotFma(e2, qvec) * inv;
      const uint32_t gid = subset[k];
      if((det != 0.0f) & (u >= 0.0f) & (u <= 1.0f) & (v >= 0.0f) & (u + v <= 1.0f) & (t > 0.0f) & (t < R[7]) && (t < bt || (t == bt && gid < bg))) { bt = t; bg = gid; }
    }
    Cand     cand[kCand];
    TraceHit opq; opq.slot = 0xFFFFFFFFu;
    bool     ovf = false;
    walkCollect(view, org, dir, 0.0f, R[7], false, false, true, false, 0.f, 0u, opq, cand, &ovf, &maxSp);
    const bool ok = !ovf && ((bg == 0xFFFFFFFFu) ? (opq.slot == 0xFFFFFFFFu) : (opq.slot != 0xFFFFFFFFu && opq.gid == bg && __float_as_uint(opq.t) == __float_as_uint(bt)));
    bad += !ok; hits += bg != 0xFFFFFFFFu;
  }
  std::printf("hit rate %.3f, deepest stack %d of %d, mismatches: %llu\n", (double)hits / nR, maxSp, TravState::kStackSize, (unsigned long long)bad);
  return bad ? 1 : 0;
}
