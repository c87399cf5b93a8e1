// host_traverse_check.cpp — the device traversal source (traverse.cuh: node decode with the PRMT plane conversion, octant
// order, compressed stack, postponed groups, single-tree closest / shadow walks with candidate lists, lower bounds, refinement
// of the opaque hit in continuation walks) compiled for the host through host_shim.h and checked against brute force over all
// triangles, on the tree the product's builder (bvh.cpp) makes.  A third of the triangles is flagged non-opaque.
//
//   host_traverse_check dump.bin [maxRays] [opaqueMod] [ommLevel]   (dump format of scripts/dump_bvh_input.py: triangles + rays)
//
// ommLevel > 0: every non-opaque triangle gets an opacity micromap of that subdivision level (4-state format, states from a hash of
// triangle and micro-triangle index; every 7th triangle a FULLY_TRANSPARENT / FULLY_OPAQUE special state instead) and the walks run
// with the lookup of omm.cuh: an OPAQUE micro-triangle must behave like an opaque triangle, a TRANSPARENT one like no triangle.
//
// Checks, per ray, against the sorted brute-force hit list (the triangle test is the same fma chain, so bit for bit):
// (1) closest protocol of k_trace / k_alpha with every candidate rejected: walks resumed behind the last candidate until a walk
//     returns fewer than kCand; the candidates enumerated must be exactly the non-opaque hits in front of the nearest opaque hit,
//     in (t, id) order, and the opaque hit the last walk reports must be the nearest opaque hit;
// (2) shadow protocol of k_shadow / k_alpha: the first walk reports an occluder iff an opaque triangle is on the segment,
//     otherwise the walks enumerate every non-opaque hit of the segment in order.
// Exit code 0 iff everything matches and no walk came near the stack limit.
#include "host_shim.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../traverse.cuh"

using namespace pt;

struct BF
{
  float    t;
  uint32_t gid;
  int      kind;  // 1 opaque / committed, 2 any-hit candidate (hits on TRANSPARENT micro-triangles are not listed)
};

int main(int argc, char** argv)
{
  if(argc < 2) { std::fprintf(stderr, "usage: host_traverse_check dump.bin [maxRays]\n"); return 2; }
  FILE* f = std::fopen(argv[1], "rb");
  uint32_t nT, nR;
  if(!f || std::fread(&nT, 4, 1, f) != 1 || std::fread(&nR, 4, 1, f) != 1) return 2;
  std::vector<float> tv((size_t)nT * 9), rv((size_t)nR * 8);
  if(std::fread(tv.data(), 4, tv.size(), f) != tv.size() || std::fread(rv.data(), 4, rv.size(), f) != rv.size()) return 2;
  std::fclose(f);
  if(argc > 2) nR = std::min<uint32_t>(nR, (uint32_t)std::atoi(argv[2]));
  // triangle i is opaque iff i % opaqueMod != 0 (default 3: a third non-opaque); a negative value flips it (|mod| 8: 7/8 non-opaque,
  // deep candidate lists and many continuation walks)
  const int opaqueMod = argc > 3 ? std::atoi(argv[3]) : 3;
  auto isOpaque = [&](uint32_t i) { return opaqueMod > 0 ? (i % (uint32_t)opaqueMod) != 0 : (i % (uint32_t)(-opaqueMod)) == 0; };
  std::vector<FlatTri>  tris(nT);
  std::vector<uint32_t> gids(nT);
  for(uint32_t i = 0; i < nT; i++)
  {
    std::memcpy(tris[i].v0, &tv[i * 9], 12); std::memcpy(tris[i].e1, &tv[i * 9 + 3], 12); std::memcpy(tris[i].e2, &tv[i * 9 + 6], 12);
    tris[i].rnode = 0; tris[i].prim = i; tris[i].flags = TRI_NOCULL | (isOpaque(i) ? TRI_OPAQUE : 0u); gids[i] = i;
  }
  WideBvh B;
  buildWideBvh(tris, gids, 0, B);
  BvhView view{reinterpret_cast<const float4*>(B.nodes.data()), reinterpret_cast<const float4*>(B.tris.data())};
  // synthetic micromaps
  const uint32_t        ommLevel = argc > 4 ? (uint32_t)std::atoi(argv[4]) : 0u;
  std::vector<uint8_t>  ommData;
  std::vector<uint32_t> ommRefOfGid(nT, kOmmNoLookup | (uint32_t)OMM_UNKNOWN), ommRef;
  auto                  hash = [](uint32_t a, uint32_t b) {
    uint32_t h = a * 2654435761u ^ (b + 0x9e3779b9u) * 2246822519u;
    h ^= h >> 15;
    h *= 3266489917u;
    h ^= h >> 13;
    return h;
  };
  if(ommLevel)
  {
    const uint32_t micro = 1u << (2 * ommLevel), bytes = (micro * 2 + 7) / 8;
    for(uint32_t i = 0; i < nT; i++)
    {
      if(isOpaque(i))
        continue;
      if(i % 7 == 0)
      {
        ommRefOfGid[i] = kOmmNoLookup | (uint32_t)((i / 7) & 1u ? OMM_OPAQUE : OMM_TRANSPARENT);
        continue;
      }
      ommRefOfGid[i] = (ommLevel << 28) | (1u << 27) | (uint32_t)ommData.size();
      const size_t at = ommData.size();
      ommData.resize(at + bytes, 0);
      for(uint32_t m = 0; m < micro; m++)
        ommData[at + (m >> 2)] |= (uint8_t)((hash(i, m) & 3u) << ((m & 3u) * 2u));
    }
    ommData.resize(ommData.size() + 4, 0);
    ommRef.resize(B.numTris);
    for(uint32_t k = 0; k < B.numTris; k++)
    {
      uint32_t gid;
      std::memcpy(&gid, &B.tris[(size_t)k * 12 + 11], 4);
      ommRef[k] = ommRefOfGid[gid];
    }
    view.ommRef = ommRef.data();
    view.ommData = ommData.data();
  }
  // how the walk must see a hit: 1 opaque (committed), 0 absent, 2 any-hit candidate
  auto effective = [&](uint32_t gid, float u, float v) -> int {
    if(isOpaque(gid))
      return 1;
    if(!ommLevel)
      return 2;
    return ommStateOf(ommRefOfGid[gid], u, v, [&](uint32_t o) { return (uint32_t)ommData[o]; });
  };
  std::printf("tris %u nodes %u rays %u kCand %d\n", B.numTris, B.numNodes, nR, kCand);

  uint64_t bad1 = 0, bad2 = 0, bad3 = 0, hits = 0, listed = 0;
  int      maxSp = 0;
  std::vector<BF> bf;
  for(uint32_t r = 0; r < nR; r++)
  {
    const float* R = &rv[(size_t)r * 8];
    const float3 org = f3(R[0], R[1], R[2]), dir = f3(R[4], R[5], R[6]);
    const float  tmin = 0.0f, tmax = (r & 1) ? R[7] : 3.0f;  // half the rays as bounded segments
    // brute force with the kernel's own triangle arithmetic
    bf.clear();
    for(uint32_t i = 0; i < nT; i++)
    {
      const float3 v0 = f3(tris[i].v0[0], tris[i].v0[1], tris[i].v0[2]), e1 = f3(tris[i].e1[0], tris[i].e1[1], tris[i].e1[2]),
                   e2 = f3(tris[i].e2[0], tris[i].e2[1], tris[i].e2[2]);
      const float3 pvec = crossFma(dir, e2);
      const float  det = dotFma(e1, pvec);
      const float  inv = 1.0f / det;
      const float3 tvec = org - v0;
      const float  u = dotFma(tvec, pvec) * inv;
      const float3 qvec = crossFma(tvec, e1);
      const float  v = dotFma(dir, qvec) * inv;
      const float  t = dotFma(e2, qvec) * inv;
      if((det != 0.0f) & (u >= 0.0f) & (u <= 1.0f) & (v >= 0.0f) & (u + v <= 1.0f) & (t > tmin) & (t < tmax))
      {
        const int kind = effective(i, u, v);
        if(kind != OMM_TRANSPARENT)
          bf.push_back(BF{t, i, kind});
      }
    }
    std::sort(bf.begin(), bf.end(), [](const BF& a, const BF& b) { return a.t < b.t || (a.t == b.t && a.gid < b.gid); });
    // expected: nearest opaque hit, non-opaque hits strictly in front of it
    size_t firstOpaque = bf.size();
    for(size_t k = 0; k < bf.size(); k++)
      if(bf[k].kind == 1)
      {
        firstOpaque = k;
        break;
      }
    hits += !bf.empty();
    // (1) closest protocol
    {
      std::vector<BF> expect;
      for(size_t k = 0; k < bf.size(); k++)
        if(bf[k].kind == 2 && (firstOpaque == bf.size() || bf[k].t < bf[firstOpaque].t))
          expect.push_back(bf[k]);
      Cand     cand[kCand];
      TraceHit opq;
      opq.slot = 0xFFFFFFFFu;
      size_t   k = 0;
      bool     haveLo = false, ok = true, ovf = false;
      float    loT = 0.f;
      uint32_t loId = 0;
      for(;;)
      {
        const int m = walkCollect(view, org, dir, tmin, tmax, false, false, true, haveLo, loT, loId, opq, cand, &ovf, &maxSp);
        for(int i = 0; i < m && ok; i++, k++)
          ok = k < expect.size() && __float_as_uint(cand[i].t) == __float_as_uint(expect[k].t) && cand[i].gid == expect[k].gid;
        if(!ok || m < kCand)
          break;
        haveLo = true;
        loT = cand[kCand - 1].t;
        loId = cand[kCand - 1].gid;
      }
      if(!ok || k != expect.size() || ovf)
        bad3++;
      listed += k;
      if(firstOpaque == bf.size() ? (opq.slot != 0xFFFFFFFFu)
                                  : (opq.slot == 0xFFFFFFFFu || __float_as_uint(opq.t) != __float_as_uint(bf[firstOpaque].t) || opq.gid != bf[firstOpaque].gid))
        bad1++;
    }
    // (2) shadow protocol
    {
      Cand     cand[kCand];
      TraceHit opq;
      opq.slot = 0xFFFFFFFFu;
      bool     ovf = false;
      int      m = walkCollect(view, org, dir, tmin, tmax, false, true, false, false, 0.f, 0u, opq, cand, &ovf, &maxSp);
      if((opq.slot != 0xFFFFFFFFu) != (firstOpaque != bf.size()) || ovf)
        bad2++;
      else if(opq.slot == 0xFFFFFFFFu)
      {
        size_t k = 0;
        bool   ok = true;
        for(;;)
        {
          for(int i = 0; i < m && ok; i++, k++)
            ok = k < bf.size() && __float_as_uint(cand[i].t) == __float_as_uint(bf[k].t) && cand[i].gid == bf[k].gid;
          if(!ok || m < kCand)
            break;
          const float    loT = cand[kCand - 1].t;
          const uint32_t loId = cand[kCand - 1].gid;
          opq.slot = 0xFFFFFFFFu;
          m = walkCollect(view, org, dir, tmin, tmax, false, true, false, true, loT, loId, opq, cand, &ovf, &maxSp);
          if(opq.slot != 0xFFFFFFFFu)
            ok = false;
        }
        if(!ok || k != bf.size() || ovf)
          bad2++;
      }
    }
  }
  std::printf("hit rate %.3f, %.2f candidates per ray, deepest stack %d of %d | mismatches: nearest opaque %llu, shadow %llu, candidates %llu\n", (double)hits / nR,
              (double)listed / nR, maxSp, TravState::kStackSize, (unsigned long long)bad1, (unsigned long long)bad2, (unsigned long long)bad3);
  if(maxSp >= TravState::kStackSize)
    return 1;
  return (bad1 | bad2 | bad3) ? 1 : 0;
}
