// bvh_build.cpp — host builder of the compressed 8-wide BVH the `extend` kernel traverses.
// Replaces the reference's binary BVHNode (bvh.rs:74-130), whose construction sorts the whole object vector instead
// of the [start,end) range and so drops objects (bvh.rs:86,108) — it is not replicated.  Closest-hit semantics stay
// those of the linear HittableList scan (hittable_list.rs:39-51); the BVH only culls.
//
// Pipeline: per primitive type a binned-SAH binary tree (1 primitive per leaf, 2 for triangles)  ->  collapse to 8-wide nodes by
// repeatedly opening the child with the largest surface area  ->  children assigned to octant-ordered slots (so the
// traversal visits near children first by XOR-ing the slot with the ray octant)  ->  child boxes quantised to 7 bits
// per plane relative to the node origin with a power-of-two step, rounded outward (conservative).
// The per-type trees hang under one root, so every node's leaf children share one primitive type.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <cstdio>
#include <atomic>
#include <future>
#include <thread>
#include <cstdlib>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <new>
#include <numeric>

#include "rtb_internal.hpp"

namespace rtb {
namespace {

// Four floats at a time for the bounds / binning passes: SSE2 on x86-64, a plain array elsewhere (aarch64 hosts such as
// Grace-based GB200 nodes; the compiler vectorises the loops over the four lanes itself).
#if defined(__SSE2__)
typedef __m128 v4f;
inline v4f v4_set1(float x) { return _mm_set1_ps(x); }
inline v4f v4_set(float x, float y, float z, float w) { return _mm_set_ps(w, z, y, x); }
inline v4f v4_load(const float* p) { return _mm_load_ps(p); }
inline void v4_store(float* p, v4f a) { _mm_store_ps(p, a); }
inline v4f v4_min(v4f a, v4f b) { return _mm_min_ps(a, b); }
inline v4f v4_max(v4f a, v4f b) { return _mm_max_ps(a, b); }
inline v4f v4_add(v4f a, v4f b) { return _mm_add_ps(a, b); }
inline v4f v4_sub(v4f a, v4f b) { return _mm_sub_ps(a, b); }
inline v4f v4_mul(v4f a, v4f b) { return _mm_mul_ps(a, b); }
inline void v4_trunc_store(int32_t* p, v4f a) { _mm_store_si128(reinterpret_cast<__m128i*>(p), _mm_cvttps_epi32(a)); }
#else
struct v4f { float v[4]; };
inline v4f v4_set1(float x) { return v4f{{x, x, x, x}}; }
inline v4f v4_set(float x, float y, float z, float w) { return v4f{{x, y, z, w}}; }
inline v4f v4_load(const float* p) { return v4f{{p[0], p[1], p[2], p[3]}}; }
inline void v4_store(float* p, v4f a) { for (int i = 0; i < 4; ++i) p[i] = a.v[i]; }
inline v4f v4_min(v4f a, v4f b) { v4f r; for (int i = 0; i < 4; ++i) r.v[i] = b.v[i] < a.v[i] ? b.v[i] : a.v[i]; return r; }
inline v4f v4_max(v4f a, v4f b) { v4f r; for (int i = 0; i < 4; ++i) r.v[i] = b.v[i] > a.v[i] ? b.v[i] : a.v[i]; return r; }
inline v4f v4_add(v4f a, v4f b) { v4f r; for (int i = 0; i < 4; ++i) r.v[i] = a.v[i] + b.v[i]; return r; }
inline v4f v4_sub(v4f a, v4f b) { v4f r; for (int i = 0; i < 4; ++i) r.v[i] = a.v[i] - b.v[i]; return r; }
inline v4f v4_mul(v4f a, v4f b) { v4f r; for (int i = 0; i < 4; ++i) r.v[i] = a.v[i] * b.v[i]; return r; }
inline void v4_trunc_store(int32_t* p, v4f a) {  // lane 3 carries an integer bit pattern: any finite-or-not value may appear
  for (int i = 0; i < 4; ++i) p[i] = (a.v[i] > -2.0e9f && a.v[i] < 2.0e9f) ? (int32_t)a.v[i] : INT32_MIN;
}
#endif

struct Box3 {
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  void grow(const float l[3], const float h[3]) {
    for (int a = 0; a < 3; ++a) {  // plain compares: std::fmin/fmax carry NaN semantics and do not inline to min/max
      lo[a] = l[a] < lo[a] ? l[a] : lo[a];
      hi[a] = h[a] > hi[a] ? h[a] : hi[a];
    }
  }
  void grow(const Box3& b) { grow(b.lo, b.hi); }
  void grow_pt(const float p[3]) { grow(p, p); }
  float area() const {
    float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    if (dx < 0 || dy < 0 || dz < 0) return 0.f;
    return 2.f * (dx * dy + dy * dz + dz * dx);
  }
};

struct BinNode {  // binary tree node
  Box3 box;
  int left = -1, right = -1;  // children, or -1 for a leaf
  uint32_t first = 0, count = 0;
  uint32_t nleaves = 1;       // leaf nodes in this subtree
};

struct alignas(16) Rec {  // one primitive's padded bounds; the records themselves are partitioned, so every range the
  float lo[3];             // builder touches is contiguous in memory (index-only partitioning made the build
  uint32_t prim_enc;       // DRAM-latency-bound).  Two 16-byte halves: (lo, prim) and (hi, 0) load as SSE vectors; the
  float hi[3];             // primitive index carries bit 30 so that, read as a float, lane 3 is a normal number (no
  uint32_t _pad;           // denormal assists in the vector arithmetic that ignores it)
  float centroid(int a) const { return 0.5f * (lo[a] + hi[a]); }
  uint32_t prim() const { return prim_enc & 0x3FFFFFFFu; }
};
static_assert(sizeof(Rec) == 32, "Rec must be two SSE vectors");

// SSE accumulation of bounds: lanes 0-2 = x, y, z; lane 3 carries the record's integer fields and is ignored
struct Box4 {
  v4f lo = v4_set1(INFINITY), hi = v4_set1(-INFINITY);
  void grow(v4f l, v4f h) { lo = v4_min(lo, l); hi = v4_max(hi, h); }
  void grow(const Box4& b) { grow(b.lo, b.hi); }
  Box3 box3() const {
    alignas(16) float l[4], h[4];
    v4_store(l, lo);
    v4_store(h, hi);
    Box3 b;
    for (int a = 0; a < 3; ++a) { b.lo[a] = l[a]; b.hi[a] = h[a]; }
    return b;
  }
};

struct Builder {
  explicit Builder(const HostScene& h) : hs(h) {}
  const HostScene& hs;
  std::vector<Rec> recs;            // the current type's primitives, partitioned in place
  // binary nodes, indexed by the ranges build_at() hands out; raw storage: only reachable nodes are ever written, so the
  // 2n-node array (104 MB for 1 M triangles) is not initialised
  BinNode* bin = nullptr;
  ~Builder() { std::free(bin); }
  Builder(const Builder&) = delete;
  Builder& operator=(const Builder&) = delete;
  uint32_t max_leaf = 1;            // primitives per leaf slot (1..3)
  int par_depth = 5;                // levels of the tree whose halves are built concurrently

  // bounds of the records [a, b) and of their centroids (SSE: one min + one max per record and box)
  void range_bounds(uint32_t a, uint32_t b, Box3& box, Box3& cbox) const {
    Box4 bx, cb;
    const v4f half = v4_set1(0.5f);
    for (uint32_t i = a; i < b; ++i) {
      const v4f l = v4_load(recs[i].lo), h = v4_load(recs[i].hi);
      bx.grow(l, h);
      const v4f c = v4_mul(half, v4_add(l, h));
      cb.grow(c, c);
    }
    box = bx.box3();
    cbox = cb.box3();
  }

  // 16-bin histograms of the records [a, b) on the three axes: bin = clamp(int((centroid - lo) * k)), exactly the
  // expression the partition step evaluates
  void range_bins(uint32_t a, uint32_t b, const float lo[3], const float k[3], const bool valid[3], Box3 (&bb)[3][16],
                  uint32_t (&bc)[3][16]) const {
    const int NB = 16;
    Box4 acc[3][NB];
    const v4f half = v4_set1(0.5f);
    const v4f lo4 = v4_set(lo[0], lo[1], lo[2], 0.f), k4 = v4_set(k[0], k[1], k[2], 0.f);
    for (uint32_t i = a; i < b; ++i) {
      const v4f l = v4_load(recs[i].lo), h = v4_load(recs[i].hi);
      const v4f c = v4_mul(half, v4_add(l, h));
      alignas(16) int32_t bi[4];
      v4_trunc_store(bi, v4_mul(v4_sub(c, lo4), k4));
      for (int ax = 0; ax < 3; ++ax) {
        if (!valid[ax]) continue;
        int q = bi[ax];
        q = q < 0 ? 0 : (q >= NB ? NB - 1 : q);
        acc[ax][q].grow(l, h);
        bc[ax][q]++;
      }
    }
    for (int ax = 0; ax < 3; ++ax)
      for (int q = 0; q < NB; ++q) bb[ax][q] = acc[ax][q].box3();
  }

  // SAH sweep over the 16 bins of every valid axis
  static void best_split(const Box3 (&bb)[3][16], const uint32_t (&bc)[3][16], const bool (&valid)[3], int& best_axis,
                         int& best_bin) {
    const int NB = 16;
    float best_cost = INFINITY;
    best_axis = best_bin = -1;
    for (int a = 0; a < 3; ++a) {
      if (!valid[a]) continue;
      float right_area[NB];
      uint32_t right_cnt[NB];
      Box3 acc;
      uint32_t cnt = 0;
      for (int b = NB - 1; b > 0; --b) {
        acc.grow(bb[a][b]);
        cnt += bc[a][b];
        right_area[b] = acc.area();
        right_cnt[b] = cnt;
      }
      Box3 accl;
      uint32_t cl = 0;
      for (int b = 0; b < NB - 1; ++b) {
        accl.grow(bb[a][b]);
        cl += bc[a][b];
        if (cl == 0 || right_cnt[b + 1] == 0) continue;
        const float cost = accl.area() * (float)cl + right_area[b + 1] * (float)right_cnt[b + 1];
        if (cost < best_cost) { best_cost = cost; best_axis = a; best_bin = b; }
      }
    }
  }

  // binned SAH split of order[first, first+count): fills the node's bounds; returns false for a leaf
  bool split(uint32_t first, uint32_t count, BinNode& node, uint32_t& mid) {
    Box3 box, cbox;
    range_bounds(first, first + count, box, cbox);
    node.box = box;
    node.first = first;
    node.count = count;
    node.left = node.right = -1;
    node.nleaves = 1;
    if (count <= max_leaf) return false;
    // 16 bins per axis, all three axes binned in one pass over the primitives
    const int NB = 16;
    Box3 bb[3][NB];
    uint32_t bc[3][NB] = {{0}};
    float k[3], lo[3];
    bool valid[3];
    for (int a = 0; a < 3; ++a) {
      const float ext = cbox.hi[a] - cbox.lo[a];
      valid[a] = ext > 0.f;
      k[a] = valid[a] ? NB / ext : 0.f;
      lo[a] = cbox.lo[a];
    }
    range_bins(first, first + count, lo, k, valid, bb, bc);
    int best_axis = -1, best_bin = -1;
    best_split(bb, bc, valid, best_axis, best_bin);
    if (best_axis < 0) {
      mid = first + count / 2;  // all centroids coincide: split the range
    } else {
      const float kk = k[best_axis], l0 = lo[best_axis];
      const int ba = best_axis;
      auto it = std::partition(recs.begin() + first, recs.begin() + first + count, [&](const Rec& p) {
        int b = (int)((p.centroid(ba) - l0) * kk);
        b = b < 0 ? 0 : (b >= NB ? NB - 1 : b);
        return b <= best_bin;
      });
      mid = (uint32_t)(it - recs.begin());
      if (mid == first || mid == first + count) mid = first + count / 2;
    }
    return true;
  }

  // Multi-threaded version of split() for the few huge ranges at the top of the tree (the serial passes over 1 M
  // records made the first three levels cost as much as all the others together): per-thread partial bounds / bins are
  // merged, and the partition is a stable two-way scatter through `tmp` with per-thread prefix offsets.
  std::vector<Rec> tmp;
  bool split_par(uint32_t first, uint32_t count, BinNode& node, uint32_t& mid, unsigned T) {
    const int NB = 16;
    struct Part { Box3 box, cbox; Box3 bb[3][16]; uint32_t bc[3][16]; uint32_t n_left; };
    std::vector<Part> part(T);
    const uint32_t per = (count + T - 1) / T;
    auto run = [&](auto&& fn) {
      std::vector<std::thread> pool;
      for (unsigned t = 1; t < T; ++t) pool.emplace_back([&, t]() { fn(t); });
      fn(0u);
      for (std::thread& th : pool) th.join();
    };
    auto range = [&](unsigned t, uint32_t& a, uint32_t& b) {
      a = first + std::min(count, t * per);
      b = first + std::min(count, t * per + per);
    };
    run([&](unsigned t) {
      uint32_t a, b;
      range(t, a, b);
      range_bounds(a, b, part[t].box, part[t].cbox);
    });
    Box3 box, cbox;
    for (unsigned t = 0; t < T; ++t) { box.grow(part[t].box); cbox.grow(part[t].cbox); }
    node.box = box;
    node.first = first;
    node.count = count;
    node.left = node.right = -1;
    node.nleaves = 1;
    if (count <= max_leaf) return false;
    float k[3], lo[3];
    bool valid[3];
    for (int a = 0; a < 3; ++a) {
      const float ext = cbox.hi[a] - cbox.lo[a];
      valid[a] = ext > 0.f;
      k[a] = valid[a] ? NB / ext : 0.f;
      lo[a] = cbox.lo[a];
    }
    run([&](unsigned t) {
      uint32_t a0, b0;
      range(t, a0, b0);
      Part& P = part[t];
      std::memset(P.bc, 0, sizeof(P.bc));
      range_bins(a0, b0, lo, k, valid, P.bb, P.bc);
    });
    Box3 bb[3][NB];
    uint32_t bc[3][NB] = {{0}};
    for (unsigned t = 0; t < T; ++t)
      for (int a = 0; a < 3; ++a)
        for (int b = 0; b < NB; ++b) { bb[a][b].grow(part[t].bb[a][b]); bc[a][b] += part[t].bc[a][b]; }
    int best_axis = -1, best_bin = -1;
    best_split(bb, bc, valid, best_axis, best_bin);
    if (best_axis < 0) {
      mid = first + count / 2;  // all centroids coincide: split the range
      return true;
    }
    const float kk = k[best_axis], l0 = lo[best_axis];
    const int ba = best_axis;
    auto goes_left = [&](const Rec& p) {
      int b = (int)((p.centroid(ba) - l0) * kk);
      b = b < 0 ? 0 : (b >= NB ? NB - 1 : b);
      return b <= best_bin;
    };
    run([&](unsigned t) {
      uint32_t a, b;
      range(t, a, b);
      uint32_t n = 0;
      for (uint32_t i = a; i < b; ++i) n += goes_left(recs[i]) ? 1u : 0u;
      part[t].n_left = n;
    });
    uint32_t total_left = 0;
    for (unsigned t = 0; t < T; ++t) total_left += part[t].n_left;
    if (total_left == 0 || total_left == count) {
      mid = first + count / 2;
      return true;
    }
    // `tmp` mirrors `recs` index for index: concurrent splits work on disjoint ranges of both
    std::vector<uint32_t> loff(T), roff(T);
    uint32_t l = 0, r = total_left;
    for (unsigned t = 0; t < T; ++t) {
      uint32_t a, b;
      range(t, a, b);
      loff[t] = l; roff[t] = r;
      l += part[t].n_left;
      r += (b - a) - part[t].n_left;
    }
    run([&](unsigned t) {
      uint32_t a, b;
      range(t, a, b);
      uint32_t li = first + loff[t], ri = first + roff[t];
      for (uint32_t i = a; i < b; ++i) {
        if (goes_left(recs[i])) tmp[li++] = recs[i];
        else tmp[ri++] = recs[i];
      }
    });
    run([&](unsigned t) {
      uint32_t a, b;
      range(t, a, b);
      if (b > a) std::memcpy(&recs[a], &tmp[a], (size_t)(b - a) * sizeof(Rec));
    });
    mid = first + total_left;
    return true;
  }

  // Builds the subtree of recs[first, first+count) with its root at bin[me].  A subtree of n records has at most 2n-1
  // nodes, so it owns the index range [me, me + 2n - 1): the left child is bin[me+1], the right child starts after the
  // left subtree's range.  Ranges of concurrently built subtrees are disjoint — no splicing, no reallocation (`bin` is
  // sized 2n up front; unused slots stay empty).  Large subtrees near the top are built concurrently and their splits
  // are themselves multi-threaded.
  void build_at(int me, uint32_t first, uint32_t count, int depth) {
    BinNode nd;
    uint32_t mid = 0;
    unsigned T = 1;
    if (count >= 131072 && par_depth > 0) {
      const unsigned hw = std::max(1u, std::min(std::thread::hardware_concurrency(), 32u));
      T = std::max(1u, hw >> std::min(depth, 5));
    }
    const bool inner = T > 1 ? split_par(first, count, nd, mid, T) : split(first, count, nd, mid);
    bin[me] = nd;
    if (!inner) return;
    const int l = me + 1, r = me + 2 * (int)(mid - first);
    if (count >= 32768 && depth < par_depth) {
      auto fut = std::async(std::launch::async, [&]() { build_at(l, first, mid - first, depth + 1); });
      build_at(r, mid, first + count - mid, depth + 1);
      fut.get();
    } else {
      build_at(l, first, mid - first, depth + 1);
      build_at(r, mid, first + count - mid, depth + 1);
    }
    bin[me].left = l;
    bin[me].right = r;
    bin[me].nleaves = bin[l].nleaves + bin[r].nleaves;
  }

  int build_range(uint32_t first, uint32_t count) {
    std::free(bin);
    bin = static_cast<BinNode*>(std::malloc(2 * (size_t)count * sizeof(BinNode)));
    if (!bin) throw std::bad_alloc();
    if (count >= 131072 && par_depth > 0) tmp.resize(recs.size());
    build_at(0, first, count, 0);
    std::vector<Rec>().swap(tmp);
    return 0;
  }
};

struct WideChild {
  Box3 box;
  int bin_node;   // binary node index (leaf or internal) in the type's tree; -1 for typed-root links
  int link_node;  // for the root joining node: wide node index to link to
  bool leaf;
};

// child planes are quantised to 7 bits: the device turns a byte into the float 128+q with ONE byte-permute
// (0x43000000 | q << 16) and no int->float conversion; 8 bits would need an extra FADD per plane (48 per node visit)
const int QMAX = 127;

uint8_t exp_byte_for(float extent) {
  // smallest power-of-two step s = 2^(e-127) with QMAX*s >= extent
  if (!(extent > 0.f)) return 1;
  int e;
  std::frexp(extent / (float)QMAX, &e);  // extent/QMAX = m * 2^e, m in [0.5,1)  ->  2^e >= extent/QMAX
  int biased = e + 127;
  if (biased < 1) biased = 1;
  if (biased > 254) biased = 254;
  return (uint8_t)biased;
}
float step_from_byte(uint8_t b) {
  uint32_t bits = (uint32_t)b << 23;
  float f;
  std::memcpy(&f, &bits, 4);
  return f;
}

struct Assembler {
  const HostScene& hs;
  HostBvh& out;
  uint32_t max_depth = 0;

  // quantise children into node `ni`
  void quantise(Node8& n, const WideChild* ch, const int* slot_of, int nch) {
    Box3 nb;
    for (int i = 0; i < nch; ++i) nb.grow(ch[i].box);
    n.ox = nb.lo[0]; n.oy = nb.lo[1]; n.oz = nb.lo[2];
    uint8_t eb[3];
    float step[3];
    for (int a = 0; a < 3; ++a) {
      eb[a] = exp_byte_for(nb.hi[a] - nb.lo[a]);
      for (;;) {  // make sure 255 steps really cover the extent in float arithmetic
        step[a] = step_from_byte(eb[a]);
        if (nb.lo[a] + (float)QMAX * step[a] >= nb.hi[a] || eb[a] >= 254) break;
        ++eb[a];
      }
    }
    n.ex = eb[0]; n.ey = eb[1]; n.ez = eb[2];
    for (int s = 0; s < 8; ++s)
      for (int a = 0; a < 3; ++a) { n.qlo[a][s] = QMAX; n.qhi[a][s] = 0; }  // empty: inverted box, never hit
    for (int i = 0; i < nch; ++i) {
      int s = slot_of[i];
      for (int a = 0; a < 3; ++a) {
        double o = nb.lo[a], st = step[a];
        int ql = (int)std::floor(((double)ch[i].box.lo[a] - o) / st);
        int qh = (int)std::ceil(((double)ch[i].box.hi[a] - o) / st);
        ql = ql < 0 ? 0 : (ql > QMAX ? QMAX : ql);
        qh = qh < 0 ? 0 : (qh > QMAX ? QMAX : qh);
        // verify in float, the arithmetic the device uses (o + q*step is exact or rounded; widen if needed)
        while (ql > 0 && nb.lo[a] + (float)ql * step[a] > ch[i].box.lo[a]) --ql;
        while (qh < QMAX && nb.lo[a] + (float)qh * step[a] < ch[i].box.hi[a]) ++qh;
        n.qlo[a][s] = (uint8_t)ql;
        n.qhi[a][s] = (uint8_t)qh;
      }
    }
  }

  // octant-ordered slot assignment: slot bit a set = child lies on the + side of axis a
  void assign_slots(const WideChild* ch, int nch, int* slot_of) {
    Box3 nb;
    for (int i = 0; i < nch; ++i) nb.grow(ch[i].box);
    float pc[3];
    for (int a = 0; a < 3; ++a) pc[a] = 0.5f * (nb.lo[a] + nb.hi[a]);
    float cost[8][8];
    for (int i = 0; i < nch; ++i) {
      float d[3];
      for (int a = 0; a < 3; ++a) d[a] = 0.5f * (ch[i].box.lo[a] + ch[i].box.hi[a]) - pc[a];
      for (int s = 0; s < 8; ++s)
        cost[i][s] = ((s & 1) ? d[0] : -d[0]) + ((s & 2) ? d[1] : -d[1]) + ((s & 4) ? d[2] : -d[2]);
    }
    bool child_done[8] = {false}, slot_used[8] = {false};
    for (int i = 0; i < nch; ++i) slot_of[i] = -1;
    for (int round = 0; round < nch; ++round) {
      float best = -INFINITY;
      int bi = -1, bs = -1;
      for (int i = 0; i < nch; ++i) {
        if (child_done[i]) continue;
        for (int s = 0; s < 8; ++s) {
          if (slot_used[s]) continue;
          if (cost[i][s] > best) { best = cost[i][s]; bi = i; bs = s; }
        }
      }
      child_done[bi] = true;
      slot_used[bs] = true;
      slot_of[bi] = bs;
    }
  }
};

}  // namespace

int build_bvh8(const HostScene& hs, HostBvh& out, std::string& err) {
  out.nodes.clear();
  for (int t = 0; t < (int)PT_COUNT; ++t) { out.geom[t].clear(); out.info[t].clear(); }
  out.attr.clear();
  out.max_depth = 0;
  out.global_refs.clear();
  const size_t np = hs.prims.size();
  // malformed input (NaN / inf / 1e308 constructor arguments) must come back as an error, not as a builder that sorts NaNs
  for (size_t i = 0; i < np; ++i) {
    const HostPrim& p = hs.prims[i];
    bool ok = p.type < PT_COUNT;
    for (int a = 0; a < 3 && ok; ++a) ok = std::isfinite(p.lo[a]) && std::isfinite(p.hi[a]) && p.lo[a] <= p.hi[a] && std::fabs(p.lo[a]) < 1e30f && std::fabs(p.hi[a]) < 1e30f;
    for (int w = 0; w < 12 && ok; ++w) ok = std::isfinite(p.g[w]);
    if (!ok) {
      err = "primitive " + std::to_string(p.prim_id) + " has non-finite or out-of-range geometry";
      return RTB_ERR_INVALID;
    }
  }

  // Leaf entries: geometry words, (prim id, material word) and — when some triangle has vertex normals or texture
  // coordinates — a shading record per triangle (all zero for the flat ones).  Info bit 31 marks a quad with an exact
  // plane or a triangle with a shading record.
  bool with_attr = false;
  for (size_t i = 0; i < np && !with_attr; ++i) with_attr = hs.prims[i].type == PT_TRI && hs.prims[i].attr != RTB_NONE;
  for (size_t i = 0; i < np; ++i)
    if (hs.prims[i].type == PT_TRI && hs.prims[i].attr != RTB_NONE && hs.prims[i].attr >= hs.attrs.size()) {
      err = "internal: triangle shading record out of range";
      return RTB_ERR_INVALID;
    }
  auto emit_leaf = [&](const HostPrim& p, std::vector<float>* geom, std::vector<uint32_t>* info, std::vector<float>& attr) {
    for (uint32_t w = 0; w < geom_words(p.type); ++w) geom[p.type].push_back(p.g[w]);
    const bool has_attr = p.type == PT_TRI && p.attr != RTB_NONE;
    info[p.type].push_back(p.prim_id);
    info[p.type].push_back((p.material & 0xFFFFFFu) | (p.face_mode << 24) |
                           ((p.type == PT_QUAD && p.plane_exact) || has_attr ? 0x80000000u : 0u));
    if (with_attr && p.type == PT_TRI) {
      static const AttrRec flat{};
      const AttrRec& r = has_attr ? hs.attrs[p.attr] : flat;
      attr.insert(attr.end(), r.f, r.f + RTB_ATTR_FLOATS);
    }
  };

  // --- "global" primitives: a primitive whose box is (nearly) the whole scene box (the r=1000 ground sphere of
  // book 1) cannot be culled by any node and only coarsens the quantisation grid of the node that holds
  // it.  Up to RTB_MAX_GLOBALS of them are kept out of the tree and tested first for every ray (which also gives an
  // early t_max that culls nodes behind them).
  std::vector<char> is_global(np, 0);
  {
    Box3 scene;
    for (size_t i = 0; i < np; ++i) scene.grow(hs.prims[i].lo, hs.prims[i].hi);
    const float scene_area = scene.area();
    const bool enabled = hs.opt_globals != 0 && !(getenv("RTB_GLOBALS") && atoi(getenv("RTB_GLOBALS")) == 0);
    const size_t tiny = getenv("RTB_TINY_SCENE") ? (size_t)atoi(getenv("RTB_TINY_SCENE")) : 16;
    if (enabled && np <= tiny && np <= RTB_MAX_GLOBALS) {
      // a scene this small (the 13-primitive Cornell box) is cheaper to scan than to traverse: one node visit decodes
      // 48 planes, about as much work as ten quad tests
      for (size_t i = 0; i < np; ++i) is_global[i] = 1;
    } else if (enabled && scene_area > 0.f) {
      std::vector<std::pair<float, uint32_t>> big;
      for (size_t i = 0; i < np; ++i) {
        Box3 b;
        b.grow(hs.prims[i].lo, hs.prims[i].hi);
        const float a = b.area();
        if (a >= 0.8f * scene_area) big.emplace_back(-a, (uint32_t)i);  // dominates the scene box (walls at 1/3 do not pay)
      }
      std::sort(big.begin(), big.end());
      for (size_t k = 0; k < big.size() && k < 4; ++k) is_global[big[k].second] = 1;
      // A handful of LARGE primitives of a type of their own (the six walls around the 1 M-triangle height field: their
      // boxes add up to twice the scene box, nearly every ray reaches one anyway): in the tree they cost a typed subtree
      // whose leaf tests split every leaf-test round of the deep-tree extend kernel in two (one type at a time); out of
      // it they cost a few full-width quad tests per ray.  C4: 4120 -> 4400 Mrays/s, one node visit less per segment.
      // (A SMALL lone primitive — the one moving sphere of the final scene — stays in the tree: testing it for every ray
      // costs 3 %.)
      if (!(getenv("RTB_GLOBAL_MINORITY") && atoi(getenv("RTB_GLOBAL_MINORITY")) == 0)) {
        size_t cnt[PT_COUNT] = {0, 0, 0, 0};
        float area[PT_COUNT] = {0.f, 0.f, 0.f, 0.f};
        for (size_t i = 0; i < np; ++i)
          if (hs.prims[i].type < PT_COUNT && !is_global[i]) {
            Box3 b;
            b.grow(hs.prims[i].lo, hs.prims[i].hi);
            cnt[hs.prims[i].type]++;
            area[hs.prims[i].type] += b.area();
          }
        size_t n_glob = 0, n_types = 0;
        for (size_t i = 0; i < np; ++i) n_glob += is_global[i];
        for (uint32_t t = 0; t < PT_COUNT; ++t) n_types += cnt[t] ? 1u : 0u;
        for (uint32_t t = 0; t < PT_COUNT && n_types > 1; ++t)
          if (cnt[t] && cnt[t] <= 8 && area[t] >= scene_area && n_glob + cnt[t] <= RTB_MAX_GLOBALS) {
            for (size_t i = 0; i < np; ++i)
              if (hs.prims[i].type == t && !is_global[i]) { is_global[i] = 1; ++n_glob; }
            --n_types;
          }
      }
    }
  }

  const bool timing = getenv("RTB_BVH_TIMING") != nullptr;
  auto now = []() { return std::chrono::steady_clock::now(); };
  auto t_start = now();
  // --- per-type binary trees ---------------------------------------------------------------------------------
  struct TypedTree { Builder* b; int root; uint32_t type; };
  size_t type_count[PT_COUNT] = {0, 0, 0, 0};
  for (size_t i = 0; i < np; ++i)
    if (!is_global[i] && hs.prims[i].type < PT_COUNT) type_count[hs.prims[i].type]++;
  std::vector<Builder*> builders;
  std::vector<TypedTree> trees;
  for (uint32_t t = 0; t < PT_COUNT; ++t) {
    Builder* b = new Builder(hs);
    // one primitive per leaf slot: a sphere/quad test costs more than a (quantised) box test and single-primitive
    // leaves fill the 8 slots of a node; triangles keep up to 2 per slot to bound the node count of large meshes
    b->max_leaf = (t == PT_TRI) ? std::max(1u, std::min(3u, hs.opt_max_leaf_tris)) : 1u;
    if (const char* e = getenv("RTB_MAX_LEAF")) b->max_leaf = (uint32_t)std::max(1, std::min(3, atoi(e)));
    builders.push_back(b);
    if (type_count[t] == 0) continue;
    b->recs.reserve(type_count[t]);
    for (size_t i = 0; i < np; ++i)
      if (hs.prims[i].type == t && !is_global[i]) {
        Rec r{};
        for (int a = 0; a < 3; ++a) { r.lo[a] = hs.prims[i].lo[a]; r.hi[a] = hs.prims[i].hi[a]; }
        r.prim_enc = (uint32_t)i | 0x40000000u;
        b->recs.push_back(r);
      }
    if (timing) std::fprintf(stderr, "[rtb200]   type %u: %zu records filled at %.3f s\n", t, b->recs.size(),
                             std::chrono::duration<double>(now() - t_start).count());
    if (const char* e = getenv("RTB_BVH_PAR")) b->par_depth = atoi(e);
    int root = b->build_range(0, (uint32_t)b->recs.size());
    trees.push_back(TypedTree{b, root, t});
  }
  auto cleanup = [&]() {
    for (Builder* b : builders) delete b;
    // global primitives live at the end of their type's leaf-ordered arrays; no node references them
    for (size_t i = 0; i < np; ++i) {
      if (!is_global[i]) continue;
      const HostPrim& p = hs.prims[i];
      const uint32_t idx = (uint32_t)(out.info[p.type].size() / 2);
      emit_leaf(p, out.geom, out.info, out.attr);
      out.global_refs.push_back((p.type << REF_TYPE_SHIFT) | idx);
    }
  };

  auto t_binary = now();
  Assembler as{hs, out};
  if (trees.empty()) {  // empty scene: a single node with no children (every ray misses)
    Node8 n;
    std::memset(&n, 0, sizeof(n));
    n.ex = n.ey = n.ez = 1;
    for (int s = 0; s < 8; ++s)
      for (int a = 0; a < 3; ++a) { n.qlo[a][s] = QMAX; n.qhi[a][s] = 0; }
    out.nodes.push_back(n);
    cleanup();
    return RTB_OK;
  }

  // --- breadth-first collapse into wide nodes -------------------------------------------------------------------
  struct Pending { uint32_t node; int tree; int bin_node; uint32_t depth; };
  std::vector<Pending> queue;
  size_t qhead = 0;
  const bool joined = trees.size() > 1;
  out.nodes.emplace_back();
  if (joined) {
    // The root joins the typed trees.  Its children are all internal nodes and may come from different trees (only the LEAF
    // children of a node share a type), so the typed roots are opened — largest box first — until the eight slots are used:
    // a ray does not spend one visit on a 2-3-child join node plus one per typed root before it reaches real branching
    // (final scene: 5.6 -> 4.x node visits per segment).  RTB_JOIN_OPEN=0: the plain join of round 1.
    struct Cand { int tree, bin; };
    Cand cand[8];
    int nch = (int)trees.size();
    for (int i = 0; i < nch; ++i) cand[i] = Cand{i, trees[i].root};
    const bool open_join = !(getenv("RTB_JOIN_OPEN") && atoi(getenv("RTB_JOIN_OPEN")) == 0);
    while (open_join && nch < 8) {
      int best = -1;
      float best_area = -1.f;
      for (int i = 0; i < nch; ++i) {
        const BinNode& c = trees[cand[i].tree].b->bin[cand[i].bin];
        if (c.left < 0) continue;
        const float a = c.box.area();
        if (a > best_area) { best_area = a; best = i; }
      }
      if (best < 0) break;
      const Cand o = cand[best];
      const BinNode& ob = trees[o.tree].b->bin[o.bin];
      cand[best] = Cand{o.tree, ob.left};
      cand[nch++] = Cand{o.tree, ob.right};
    }
    WideChild ch[8];
    uint32_t base = (uint32_t)out.nodes.size();
    for (int i = 0; i < nch; ++i) {
      ch[i].box = trees[cand[i].tree].b->bin[cand[i].bin].box;
      ch[i].leaf = false;  // (a one-primitive tree becomes a node with one leaf child, process())
      out.nodes.emplace_back();
    }
    int slot_of[8];
    as.assign_slots(ch, nch, slot_of);
    // internal children must be stored in ascending slot order
    int idx[8];
    std::iota(idx, idx + nch, 0);
    std::sort(idx, idx + nch, [&](int a, int b) { return slot_of[a] < slot_of[b]; });
    Node8 n;
    std::memset(&n, 0, sizeof(n));
    as.quantise(n, ch, slot_of, nch);
    n.child_base = base;
    n.prim_base = 0;
    for (int k = 0; k < nch; ++k) {
      int i = idx[k];
      n.imask |= (uint8_t)(1u << slot_of[i]);
      queue.push_back(Pending{base + (uint32_t)k, cand[i].tree, cand[i].bin, 2});
    }
    out.nodes[0] = n;
  } else {
    queue.push_back(Pending{0, 0, trees[0].root, 1});
  }

  float open_min_rel = hs.opt_open_min_rel;
  if (const char* e = getenv("RTB_OPEN_MIN_REL")) open_min_rel = (float)atof(e);

  // One wide node: gather up to 8 children of binary node pd.bin_node, assign slots, quantise, append its leaf
  // primitives and allocate its internal children — into `sk` (the global arrays, or a subtree-local set).
  struct Sink {
    std::vector<Node8>* nodes;
    std::vector<float>* geom;      // [PT_COUNT]
    std::vector<uint32_t>* info;   // [PT_COUNT]
    std::vector<float>* attr;      // triangle shading records
    std::vector<Pending>* queue;
    uint32_t max_depth = 0;
  };
  auto process = [&](const Pending& pd, Sink& sk, std::string& perr) -> bool {
    Builder& b = *trees[pd.tree].b;
    const uint32_t type = trees[pd.tree].type;
    if (pd.depth > sk.max_depth) sk.max_depth = pd.depth;
    // gather up to 8 children by opening the largest internal child
    int cand[8];
    int nc = 0;
    const BinNode& rootbn = b.bin[pd.bin_node];
    if (rootbn.left < 0) {
      cand[nc++] = pd.bin_node;  // typed root that is itself a leaf: node with one leaf child
    } else {
      cand[nc++] = rootbn.left;
      cand[nc++] = rootbn.right;
      while (nc < 8) {
        int best = -1;
        float best_area = -1.f;
        for (int i = 0; i < nc; ++i) {
          const BinNode& c = b.bin[cand[i]];
          if (c.left < 0) continue;
          // child planes are quantised relative to THIS node's extent: do not pull the children of a subtree that is
          // tiny next to the node (the 22-unit sphere field beside the r=1000 ground sphere) up into its coarse grid
          float rel = 0.f;
          for (int a = 0; a < 3; ++a) {
            const float E = rootbn.box.hi[a] - rootbn.box.lo[a];
            if (E > 0.f) rel = std::fmax(rel, (c.box.hi[a] - c.box.lo[a]) / E);
          }
          if (rel < open_min_rel) continue;
          float a = c.box.area();
          if (a > best_area) { best_area = a; best = i; }
        }
        if (best < 0) break;
        int open = cand[best];
        cand[best] = b.bin[open].left;
        cand[nc++] = b.bin[open].right;
      }
    }
    WideChild ch[8];
    for (int i = 0; i < nc; ++i) {
      ch[i].box = b.bin[cand[i]].box;
      ch[i].bin_node = cand[i];
      ch[i].leaf = b.bin[cand[i]].left < 0;
    }
    int slot_of[8];
    as.assign_slots(ch, nc, slot_of);
    int idx[8];
    std::iota(idx, idx + nc, 0);
    std::sort(idx, idx + nc, [&](int x, int y) { return slot_of[x] < slot_of[y]; });
    Node8 n;
    std::memset(&n, 0, sizeof(n));
    as.quantise(n, ch, slot_of, nc);
    const uint32_t prim_base = (uint32_t)(sk.info[type].size() / 2);
    if (prim_base > REF_INDEX_MASK) { perr = "too many primitives of one type"; return false; }
    n.prim_base = (type << REF_TYPE_SHIFT) | prim_base;
    n.child_base = (uint32_t)sk.nodes->size();
    uint32_t off = 0;
    for (int k = 0; k < nc; ++k) {
      int i = idx[k];
      int s = slot_of[i];
      if (ch[i].leaf) {
        const BinNode& lf = b.bin[ch[i].bin_node];
        if (lf.count > 3 || off + lf.count > 24) { perr = "internal: leaf too large"; return false; }
        n.meta[s] = (uint8_t)((lf.count << 5) | off);
        for (uint32_t q = 0; q < lf.count; ++q) {
          emit_leaf(hs.prims[b.recs[lf.first + q].prim()], sk.geom, sk.info, *sk.attr);
        }
        off += lf.count;
      } else {
        n.imask |= (uint8_t)(1u << s);
        uint32_t child_node = (uint32_t)sk.nodes->size();
        sk.nodes->emplace_back();
        sk.queue->push_back(Pending{child_node, pd.tree, ch[i].bin_node, pd.depth + 1});
      }
    }
    (*sk.nodes)[pd.node] = n;
    return true;
  };

  // Serial breadth-first phase: the top of the tree (at least the prefix the extend kernel stages in shared memory)
  // stays in pure breadth-first order.  Large trees then hand the pending subtrees to worker threads.
  Sink top{&out.nodes, out.geom, out.info, &out.attr, &queue, 0};
  const bool parallel = np >= 50000 && !(getenv("RTB_BVH_PAR") && atoi(getenv("RTB_BVH_PAR")) == 0);
  while (qhead < queue.size()) {
    if (parallel && out.nodes.size() >= 1024 && queue.size() - qhead >= 64) break;
    Pending pd = queue[qhead++];
    if (!process(pd, top, err)) { cleanup(); return RTB_ERR_INVALID; }
  }
  out.max_depth = top.max_depth;
  if (qhead < queue.size()) {
    // Parallel phase: every pending subtree is collapsed into its own node / primitive arrays (breadth-first inside the
    // subtree, indices local), then the subtrees are appended in pending order with their indices rebased, so the
    // layout does not depend on thread timing.  Deep nodes of one subtree end up contiguous in memory.
    struct Sub {
      std::vector<Node8> nodes;
      std::vector<float> geom[PT_COUNT];
      std::vector<uint32_t> info[PT_COUNT];
      std::vector<float> attr;
      uint32_t max_depth = 0;
      std::string err;
      bool ok = true;
    };
    const size_t n_sub = queue.size() - qhead;
    std::vector<Sub> subs(n_sub);
    std::atomic<size_t> next{0};
    auto worker = [&]() {
      std::vector<Pending> lq;
      for (;;) {
        const size_t k = next.fetch_add(1);
        if (k >= n_sub) break;
        Sub& sb = subs[k];
        const Pending root = queue[qhead + k];
        sb.nodes.emplace_back();  // local node 0 = the subtree root (its global index was allocated by its parent)
        lq.clear();
        lq.push_back(Pending{0u, root.tree, root.bin_node, root.depth});
        Sink sk{&sb.nodes, sb.geom, sb.info, &sb.attr, &lq, 0};
        for (size_t h = 0; h < lq.size() && sb.ok; ++h) {
          const Pending pd = lq[h];  // copy: process() appends to lq
          sb.ok = process(pd, sk, sb.err);
        }
        sb.max_depth = sk.max_depth;
      }
    };
    unsigned n_thr = std::max(1u, std::min(std::thread::hardware_concurrency(), 32u));
    if (const char* e = getenv("RTB_BVH_THREADS")) n_thr = (unsigned)std::max(1, atoi(e));
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < n_thr; ++t) pool.emplace_back(worker);
    worker();
    for (std::thread& t : pool) t.join();
    for (size_t k = 0; k < n_sub; ++k) {
      Sub& sb = subs[k];
      if (!sb.ok) { err = sb.err; cleanup(); return RTB_ERR_INVALID; }
      const Pending root = queue[qhead + k];
      const uint32_t type = trees[root.tree].type;
      const uint32_t node_base = (uint32_t)out.nodes.size();          // local node i >= 1  ->  node_base + i - 1
      const uint32_t prim_off = (uint32_t)(out.info[type].size() / 2);  // local primitive j ->  prim_off + j
      if ((uint64_t)prim_off + sb.info[type].size() / 2 > REF_INDEX_MASK) { err = "too many primitives of one type"; cleanup(); return RTB_ERR_INVALID; }
      for (size_t i = 0; i < sb.nodes.size(); ++i) {
        Node8 n = sb.nodes[i];
        n.child_base = node_base + n.child_base - 1u;  // a local child index is always >= 1
        n.prim_base = (type << REF_TYPE_SHIFT) | ((n.prim_base & REF_INDEX_MASK) + prim_off);
        if (i == 0) out.nodes[root.node] = n;
        else out.nodes.push_back(n);
      }
      out.geom[type].insert(out.geom[type].end(), sb.geom[type].begin(), sb.geom[type].end());
      out.info[type].insert(out.info[type].end(), sb.info[type].begin(), sb.info[type].end());
      out.attr.insert(out.attr.end(), sb.attr.begin(), sb.attr.end());  // (triangle subtrees only)
      if (sb.max_depth > out.max_depth) out.max_depth = sb.max_depth;
    }
  }
  cleanup();
  if (timing) {
    auto t_end = now();
    std::fprintf(stderr, "[rtb200] BVH build: binary SAH %.3f s, collapse + quantise %.3f s, %zu nodes\n",
                 std::chrono::duration<double>(t_binary - t_start).count(),
                 std::chrono::duration<double>(t_end - t_binary).count(), out.nodes.size());
  }
  if (out.max_depth > 28) { err = "BVH too deep for the traversal stack"; return RTB_ERR_INVALID; }
  return RTB_OK;
}

}  // namespace rtb
