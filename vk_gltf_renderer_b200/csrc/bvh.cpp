// bvh.cpp — SAH BVH2 (binned) -> 8-wide collapse -> compressed wide nodes.  See bvh.h.
#include "bvh.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <cstring>

namespace pt {
namespace {

struct Box
{
  float lo[3], hi[3];
  void  reset()
  {
    for(int a = 0; a < 3; a++)
    {
      lo[a] = FLT_MAX;
      hi[a] = -FLT_MAX;
    }
  }
  void grow(const Box& b)
  {
    for(int a = 0; a < 3; a++)
    {
      lo[a] = std::min(lo[a], b.lo[a]);
      hi[a] = std::max(hi[a], b.hi[a]);
    }
  }
  float halfArea() const
  {
    float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    return dx * dy + dy * dz + dz * dx;
  }
};

struct Node2
{
  Box      box;
  uint32_t left = 0, right = 0;   // inner
  uint32_t first = 0, count = 0;  // BVH2 leaf when count > 0 (one triangle unless the centroids coincide)
  uint32_t nprims = 0;            // triangles below this node: order[first .. first + nprims)
  // SAH-optimal collapse (Ylitie, Karras, Laine 2017, section 3): cost[i-1] = cheapest forest of <= i wide-BVH
  // roots for this subtree; asLeaf = the single-root optimum is a leaf; splitK[i-1] = roots given to the left
  // child (0 = "use i-1 roots instead")
  float   cost[7];
  uint8_t splitK[8];
  bool    asLeaf = false;
};

struct Builder
{
  const std::vector<FlatTri>& tris;
  std::vector<Box>            tbox;
  std::vector<float>          cen;  // 3 per tri
  std::vector<uint32_t>       order;
  std::vector<Node2>          n2;

  explicit Builder(const std::vector<FlatTri>& t)
      : tris(t)
  {
  }

  void prepare()
  {
    const size_t n = tris.size();
    tbox.resize(n);
    cen.resize(n * 3);
    order.resize(n);
    for(size_t i = 0; i < n; i++)
    {
      const FlatTri& T = tris[i];
      Box&           b = tbox[i];
      for(int a = 0; a < 3; a++)
      {
        // the kernel intersects (v0, v0+e1, v0+e2): bound exactly that, padded a few ulp
        float v1 = T.v0[a] + T.e1[a], v2 = T.v0[a] + T.e2[a];
        float lo = std::min(T.v0[a], std::min(v1, v2)), hi = std::max(T.v0[a], std::max(v1, v2));
        float pad = std::max(std::fabs(lo), std::fabs(hi)) * 4e-7f + 1e-30f;
        b.lo[a] = lo - pad;
        b.hi[a] = hi + pad;
        cen[i * 3 + a] = 0.5f * (b.lo[a] + b.hi[a]);
      }
      order[i] = (uint32_t)i;
    }
  }

  // binned SAH down to single triangles; leaves of <= 3 triangles are formed by the collapse below
  void build2()
  {
    struct Job
    {
      uint32_t node, first, count;
    };
    n2.clear();
    n2.reserve(tris.size() * 2);
    n2.push_back(Node2());
    std::vector<Job> stack;
    stack.push_back({0, 0, (uint32_t)tris.size()});
    // SAH bins per axis (16 is what every measurement in profiles/ used unless it says otherwise)
    constexpr int NB = 16;
    while(!stack.empty())
    {
      Job j = stack.back();
      stack.pop_back();
      Box bb, cb;
      bb.reset();
      cb.reset();
      for(uint32_t i = j.first; i < j.first + j.count; i++)
      {
        uint32_t t = order[i];
        bb.grow(tbox[t]);
        for(int a = 0; a < 3; a++)
        {
          cb.lo[a] = std::min(cb.lo[a], cen[t * 3 + a]);
          cb.hi[a] = std::max(cb.hi[a], cen[t * 3 + a]);
        }
      }
      n2[j.node].box = bb;
      n2[j.node].first = j.first;
      n2[j.node].count = j.count;
      n2[j.node].nprims = j.count;
      if(j.count <= 1)
        continue;
      float bestCost = FLT_MAX;
      int   bestAxis = -1, bestBin = -1;
      for(int ax = 0; ax < 3; ax++)
      {
        float e = cb.hi[ax] - cb.lo[ax];
        if(!(e > 0.f))
          continue;
        Box      bins[NB];
        uint32_t cnt[NB];
        for(int b = 0; b < NB; b++)
        {
          bins[b].reset();
          cnt[b] = 0;
        }
        const float scale = (float)NB / e, c0 = cb.lo[ax];
        for(uint32_t i = j.first; i < j.first + j.count; i++)
        {
          uint32_t t = order[i];
          int      b = std::min(NB - 1, (int)((cen[t * 3 + ax] - c0) * scale));
          cnt[b]++;
          bins[b].grow(tbox[t]);
        }
        float    rArea[NB];
        uint32_t rCnt[NB];
        Box      acc;
        acc.reset();
        uint32_t c = 0;
        for(int b = NB - 1; b > 0; b--)
        {
          acc.grow(bins[b]);
          c += cnt[b];
          rArea[b] = c ? acc.halfArea() : 0.f;
          rCnt[b] = c;
        }
        acc.reset();
        c = 0;
        for(int b = 0; b < NB - 1; b++)
        {
          acc.grow(bins[b]);
          c += cnt[b];
          if(c == 0 || rCnt[b + 1] == 0)
            continue;
          // cost in units of "triangle slots": leaves hold up to 3 triangles per slot
          float cost = acc.halfArea() * (float)c + rArea[b + 1] * (float)rCnt[b + 1];
          if(cost < bestCost)
          {
            bestCost = cost;
            bestAxis = ax;
            bestBin = b;
          }
        }
      }
      uint32_t mid;
      if(bestAxis < 0)
        mid = j.first + j.count / 2;
      else
      {
        const float e = cb.hi[bestAxis] - cb.lo[bestAxis], scale = (float)NB / e, c0 = cb.lo[bestAxis];
        auto        it = std::partition(order.begin() + j.first, order.begin() + j.first + j.count, [&](uint32_t t) {
          int b = std::min(NB - 1, (int)((cen[t * 3 + bestAxis] - c0) * scale));
          return b <= bestBin;
        });
        mid = (uint32_t)(it - order.begin());
        if(mid == j.first || mid == j.first + j.count)
          mid = j.first + j.count / 2;
      }
      uint32_t l = (uint32_t)n2.size();
      n2.push_back(Node2());
      n2.push_back(Node2());
      n2[j.node].left = l;
      n2[j.node].right = l + 1;
      n2[j.node].count = 0;
      stack.push_back({l, j.first, mid - j.first});
      stack.push_back({l + 1, mid, j.first + j.count - mid});
    }
  }
};

static inline uint32_t f2u(float f)
{
  uint32_t u;
  memcpy(&u, &f, 4);
  return u;
}
static inline float u2f(uint32_t u)
{
  float f;
  memcpy(&f, &u, 4);
  return f;
}

}  // namespace

void buildWideBvh(const std::vector<FlatTri>& tris, const std::vector<uint32_t>& gids, uint32_t triBaseOffset, WideBvh& out)
{
  out = WideBvh();
  out.numTris = (uint32_t)tris.size();
  for(int a = 0; a < 3; a++)
  {
    out.boundsLo[a] = 0.f;
    out.boundsHi[a] = 0.f;
  }
  if(tris.empty())
  {
    // a single empty node keeps the traversal kernels branch-free about "no scene"
    out.nodes.assign(20, 0.f);
    out.numNodes = 1;
    return;
  }
  Builder B(tris);
  B.prepare();
  B.build2();
  for(int a = 0; a < 3; a++)
  {
    out.boundsLo[a] = B.n2[0].box.lo[a];
    out.boundsHi[a] = B.n2[0].box.hi[a];
  }

  // ---- SAH-optimal collapse: dynamic programme over the binary tree, children before parents -----------------
  // (children are always created after their parent, so a reverse sweep sees them first)
  const float kCostNode = 1.0f, kCostPrim = 0.7f;  // one node step ~ 250 SASS instructions, one triangle test ~ 125, but at fewer lanes (ncu r02c): measured on the bench scene (r02x, one box) 0.4 -> 970.9 / 976.4, 0.5 -> 982.1, 0.6 -> 984.1, 0.7 -> 986.1 Mray/s (17.39 / 12.41 -> 18.03 / 11.12 nodes / triangle tests per ray)
  const float invRootArea = 1.0f / std::max(B.n2[0].box.halfArea(), 1e-30f);
  for(size_t ni = B.n2.size(); ni-- > 0;)
  {
    Node2&      n = B.n2[ni];
    const float area = n.box.halfArea() * invRootArea;
    const float leafCost = (n.nprims <= 3) ? area * (float)n.nprims * kCostPrim : FLT_MAX;
    for(int i = 0; i < 8; i++)
      n.splitK[i] = 0;
    if(n.count > 0)
    {
      // BVH2 leaf (normally one triangle; coincident centroids can leave up to 3, larger groups were split in half)
      for(int i = 0; i < 7; i++)
        n.cost[i] = leafCost;
      n.asLeaf = true;
      continue;
    }
    const Node2 &L = B.n2[n.left], &R = B.n2[n.right];
    auto         distribute = [&](int j, uint8_t& bestK) {
      float best = FLT_MAX;
      bestK = 1;
      for(int k = 1; k < j; k++)
      {
        const float c = L.cost[std::min(k, 7) - 1] + R.cost[std::min(j - k, 7) - 1];
        if(c < best)
        {
          best = c;
          bestK = (uint8_t)k;
        }
      }
      return best;
    };
    uint8_t     k8;
    const float internalCost = distribute(8, k8) + area * kCostNode;
    n.splitK[7] = k8;
    n.asLeaf = leafCost <= internalCost;
    n.cost[0] = std::min(leafCost, internalCost);
    for(int i = 2; i <= 7; i++)
    {
      uint8_t     k;
      const float d = distribute(i, k);
      if(d < n.cost[i - 2])
      {
        n.cost[i - 1] = d;
        n.splitK[i - 1] = k;
      }
      else
      {
        n.cost[i - 1] = n.cost[i - 2];
        n.splitK[i - 1] = 0;
      }
    }
  }
  // roots of the cheapest forest of <= j wide nodes / leaves covering subtree n
  struct Gather
  {
    const std::vector<Node2>& n2;
    void run(uint32_t n, int j, uint32_t* out, int& cnt) const
    {
      const Node2& N = n2[n];
      if(j <= 1 || N.count > 0)
      {
        out[cnt++] = n;
        return;
      }
      const int k = N.splitK[j - 1];
      if(k == 0)
      {
        run(n, j - 1, out, cnt);
        return;
      }
      run(N.left, k, out, cnt);
      run(N.right, j - k, out, cnt);
    }
  } gather{B.n2};

  // ---- emit the wide nodes ----------------------------------------------------------------------
  struct Pending
  {
    uint32_t n2;     // BVH2 node this wide node covers
    uint32_t index;  // index of the wide node in out.nodes
    uint32_t depth;
  };
  std::vector<Pending> queue;
  out.nodes.assign(20, 0.f);
  queue.push_back({0, 0, 1});
  out.tris.reserve(tris.size() * 12);
  out.triMeta.reserve(tris.size() * 2);
  size_t qi = 0;
  // a root that is itself a leaf: wrap it in a wide node with one leaf child (handled by the generic path
  // because a leaf BVH2 node is simply a child that cannot be opened)
  while(qi < queue.size())
  {
    Pending pn = queue[qi++];
    out.maxDepth = std::max(out.maxDepth, pn.depth);
    const Node2& root = B.n2[pn.n2];
    // children of this wide node = the optimal forest of <= 8 roots of the subtree (a root that is a single
    // BVH2 leaf is wrapped in a wide node with one leaf child)
    uint32_t ch[8];
    int      nch = 0;
    if(root.count > 0)
      ch[nch++] = pn.n2;
    else
    {
      gather.run(root.left, root.splitK[7], ch, nch);
      gather.run(root.right, 8 - root.splitK[7], ch, nch);
    }
    // Slot assignment + per-node AXIS MAP.  The kernel visits the inner children of a node in descending (slot ^ oct) order,
    // where bit k of `oct` is the sign of the ray direction along the axis that bit k of the slot index stands for.  Ylitie et
    // al. fix that to (x, y, z); here every node chooses which axis each of its three slot bits follows (27 maps, two or three
    // bits may share an axis and then rank the children along it), which orders children that are spread along one or two axes
    // correctly for every ray (offline, tools/order_exp.cpp on the bench scene: 15.4 -> 14.0 nodes and 8.4 -> 7.5 triangle tests
    // per ray).  For each map the children are assigned to slots by the optimal assignment of centroid offsets (subset DP), and
    // the map whose order agrees best with the true front-to-back order over 26 sample directions wins.  6 bits per node (axis of
    // bit 0 | bit 1 << 2 | bit 2 << 4), stored above the 26-bit child base.  Round 1 used the fixed (z, y, x) map.
    int               childAt[8];
    for(int s = 0; s < 8; s++)
      childAt[s] = -1;
    uint32_t axisMap = 2u | (1u << 2) | (0u << 4);  // bit 0 -> z, bit 1 -> y, bit 2 -> x
    {
      float cen[8][3], mid[3];
      for(int i = 0; i < nch; i++)
        for(int a3 = 0; a3 < 3; a3++)
          cen[i][a3] = 0.5f * (B.n2[ch[i]].box.lo[a3] + B.n2[ch[i]].box.hi[a3]);
      for(int a3 = 0; a3 < 3; a3++)
      {
        float lo = FLT_MAX, hi = -FLT_MAX;
        for(int i = 0; i < nch; i++)
        {
          lo = std::min(lo, cen[i][a3]);
          hi = std::max(hi, cen[i][a3]);
        }
        mid[a3] = 0.5f * (lo + hi);
      }
      double bestScore = -1.0;
      int    bestCode[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      for(int map = 0; map < 27; map++)
      {
        const int ax[3] = {map % 3, (map / 3) % 3, map / 9};  // axis of slot bit 0, 1, 2
        // bits on the same axis form a binary rank along it: the higher bit is the more significant one
        float w[3];
        for(int bt = 0; bt < 3; bt++)
        {
          int lower = 0;
          for(int b2 = 0; b2 < bt; b2++)
            lower += ax[b2] == ax[bt];
          w[bt] = (float)(1 << lower);
        }
        float cost[8][8];
        for(int i = 0; i < nch; i++)
          for(int sl = 0; sl < 8; sl++)
          {
            float v = 0.f;
            for(int bt = 0; bt < 3; bt++)
              v += (((sl >> bt) & 1) ? 1.f : -1.f) * w[bt] * (cen[i][ax[bt]] - mid[ax[bt]]);
            cost[i][sl] = v;
          }
        // optimal assignment of the children (in order) to distinct slots: DP over the set of used slots
        float   best[256];
        uint8_t from[8][256];
        for(int m = 0; m < 256; m++)
          best[m] = -FLT_MAX;
        best[0] = 0.f;
        for(int m = 0; m < 256; m++)
        {
          const int i = __builtin_popcount((unsigned)m);
          if(i >= nch || best[m] == -FLT_MAX)
            continue;
          for(int sl = 0; sl < 8; sl++)
          {
            if(m & (1 << sl))
              continue;
            const int   nm = m | (1 << sl);
            const float v = best[m] + cost[i][sl];
            if(v > best[nm])
            {
              best[nm] = v;
              from[i][nm] = (uint8_t)sl;
            }
          }
        }
        int   bm = -1;
        float bv = -FLT_MAX;
        for(int m = 0; m < 256; m++)
          if(__builtin_popcount((unsigned)m) == nch && best[m] > bv)
          {
            bv = best[m];
            bm = m;
          }
        int code[8];
        for(int i = nch - 1, m = bm; i >= 0; i--)
        {
          code[i] = from[i][m];
          m &= ~(1 << code[i]);
        }
        // agreement of the visiting order with the front-to-back order of the centroids over the 26 directions of the cube
        double score = 0.0;
        for(int dxi = -1; dxi <= 1; dxi++)
          for(int dyi = -1; dyi <= 1; dyi++)
            for(int dzi = -1; dzi <= 1; dzi++)
            {
              if(!dxi && !dyi && !dzi)
                continue;
              const float d[3] = {(float)dxi, (float)dyi, (float)dzi};
              int         eff = 0;
              for(int bt = 0; bt < 3; bt++)
                if(d[ax[bt]] >= 0.f)
                  eff |= 1 << bt;
              for(int i = 0; i < nch; i++)
                for(int j = i + 1; j < nch; j++)
                {
                  const float pi = cen[i][0] * d[0] + cen[i][1] * d[1] + cen[i][2] * d[2], pj = cen[j][0] * d[0] + cen[j][1] * d[1] + cen[j][2] * d[2];
                  if(pi == pj)
                  {
                    score += 0.5;
                    continue;
                  }
                  const bool iFirst = (code[i] ^ eff) > (code[j] ^ eff);  // visited first = larger (slot ^ oct)
                  score += ((pi < pj) == iFirst) ? 1.0 : 0.0;
                }
            }
        if(ax[0] == 2 && ax[1] == 1 && ax[2] == 0)
          score *= 1.0000001;  // ties go to the standard map
        if(score > bestScore)
        {
          bestScore = score;
          axisMap = (uint32_t)ax[0] | ((uint32_t)ax[1] << 2) | ((uint32_t)ax[2] << 4);
          memcpy(bestCode, code, sizeof(code));
        }
      }
      for(int i = 0; i < nch; i++)
        childAt[bestCode[i]] = i;
    }
    const Box& nb = root.box;

    // quantisation frame
    float    p[3] = {nb.lo[0], nb.lo[1], nb.lo[2]};
    uint32_t eb[3];
    double   scale[3];
    for(int a = 0; a < 3; a++)
    {
      double ext = (double)nb.hi[a] - (double)nb.lo[a];
      int    e = (ext > 0.0) ? (int)std::ceil(std::log2(ext / 255.0)) : -126;
      // make sure 255 * 2^e really covers the extent after float rounding
      while(std::ldexp(255.0, e) < ext)
        e++;
      e = std::max(-126, std::min(127, e));
      eb[a] = (uint32_t)(e + 127);
      scale[a] = std::ldexp(1.0, e);
    }
    uint8_t  imask = 0, meta[8], qlo[3][8], qhi[3][8];
    uint32_t childBase = (uint32_t)(out.nodes.size() / 20);  // internal children appended below
    uint32_t triBase = triBaseOffset + (uint32_t)(out.tris.size() / 12);
    uint32_t triCount = 0, innerCount = 0;
    for(int s = 0; s < 8; s++)
    {
      meta[s] = 0;
      for(int a = 0; a < 3; a++)
      {
        qlo[a][s] = 255;  // empty slot: inverted box never hits
        qhi[a][s] = 0;
      }
      if(childAt[s] < 0)
        continue;
      const Node2& c = B.n2[ch[childAt[s]]];
      for(int a = 0; a < 3; a++)
      {
        double lo = ((double)c.box.lo[a] - (double)p[a]) / scale[a];
        double hi = ((double)c.box.hi[a] - (double)p[a]) / scale[a];
        int    ql = (int)std::floor(lo - 1e-3), qh = (int)std::ceil(hi + 1e-3);
        qlo[a][s] = (uint8_t)std::max(0, std::min(255, ql));
        qhi[a][s] = (uint8_t)std::max(0, std::min(255, qh));
      }
      if(!c.asLeaf)
      {
        imask |= (uint8_t)(1u << s);
        meta[s] = (uint8_t)((1u << 5) | (24u + (uint32_t)s));
        innerCount++;
      }
      else
      {
        // unary count in the high 3 bits, triangle offset in the low 5
        uint32_t bits = (c.nprims == 1) ? 1u : (c.nprims == 2 ? 3u : 7u);
        meta[s] = (uint8_t)((bits << 5) | triCount);
        for(uint32_t k = 0; k < c.nprims; k++)
        {
          const uint32_t local = B.order[c.first + k];
          const uint32_t gid = gids[local];
          const FlatTri& T = tris[local];
          float          rec[12] = {T.v0[0], T.v0[1], T.v0[2], u2f(T.rnode | (T.flags << 28)), T.e1[0], T.e1[1], T.e1[2], u2f(T.prim), T.e2[0], T.e2[1], T.e2[2], u2f(gid)};
          out.tris.insert(out.tris.end(), rec, rec + 12);
          out.triMeta.push_back(T.rnode | (T.flags << 28));
          out.triMeta.push_back(T.prim);
        }
        triCount += c.nprims;
      }
    }
    // reserve the internal children (ascending slot order) and queue them
    out.nodes.resize(out.nodes.size() + (size_t)innerCount * 20, 0.f);
    uint32_t k = 0;
    for(int s = 0; s < 8; s++)
    {
      if(childAt[s] < 0)
        continue;
      const uint32_t cn = ch[childAt[s]];
      if(!B.n2[cn].asLeaf)
        queue.push_back({cn, childBase + k++, pn.depth + 1});
    }
    float* N = &out.nodes[(size_t)pn.index * 20];
    N[0] = p[0];
    N[1] = p[1];
    N[2] = p[2];
    N[3] = u2f(eb[0] | (eb[1] << 8) | (eb[2] << 16) | ((uint32_t)imask << 24));
    N[4] = u2f(childBase | (axisMap << 26));  // child base (26 bits) | axis map (6 bits)
    N[5] = u2f(triBase);
    N[6] = u2f((uint32_t)meta[0] | ((uint32_t)meta[1] << 8) | ((uint32_t)meta[2] << 16) | ((uint32_t)meta[3] << 24));
    N[7] = u2f((uint32_t)meta[4] | ((uint32_t)meta[5] << 8) | ((uint32_t)meta[6] << 16) | ((uint32_t)meta[7] << 24));
    auto pack4 = [](const uint8_t* q) { return (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24); };
    for(int a = 0; a < 3; a++)
    {
      N[8 + a * 4 + 0] = u2f(pack4(&qlo[a][0]));
      N[8 + a * 4 + 1] = u2f(pack4(&qlo[a][4]));
      N[8 + a * 4 + 2] = u2f(pack4(&qhi[a][0]));
      N[8 + a * 4 + 3] = u2f(pack4(&qhi[a][4]));
    }
  }
  out.numNodes = (uint32_t)(out.nodes.size() / 20);
}

}  // namespace pt
