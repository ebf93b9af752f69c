// rtb_kernels.cu — the wavefront path-tracing pipeline (sm_100a) over a SLOT-STABLE path pool.  One iteration =
//   extend (wide-BVH closest hit + media; writes the hit record and the slot's shade class)
//   shade_terminal / shade_lambert / shade_specular / shade_isotropic (one kernel per material family; a finished
//   path's slot is restarted in place with the next camera path)  ->  advance (rotates the iteration counters)
// replacing the reference's recursive ray_color (main.rs:63-139) and its per-pixel sample loop (main.rs:731-784).
// There are no global work queues: every kernel walks the pool in 256-slot chunks, one warp per chunk, and compacts the
// slots it wants warp-locally (byte compares + warp scan into a shared-memory list).  No kernel issues a contended
// atomic.  Tensor cores are not used: nothing here is a dense contraction.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "rtb_device.cuh"
#include "rtb_launch.hpp"

namespace rtb {

// ---- helpers ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ray_octant(float3 d) {
  return (d.x < 0.0f ? 1u : 0u) | (d.y < 0.0f ? 2u : 0u) | (d.z < 0.0f ? 4u : 0u);
}

__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ void red_add_v4(float4* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// accumulate + write_color's NaN policy moved to per-sample rejection (SURVEY App. A #10)
__device__ __forceinline__ void deposit(const DevParams& prm, DevCounters* c, uint32_t pixel, float3 L) {
  if (!(isfinite(L.x) && isfinite(L.y) && isfinite(L.z))) {
    atomicAdd(&c->rejected, 1ull);
    return;
  }
  const float Y = 0.2126f * L.x + 0.7152f * L.y + 0.0722f * L.z;
  red_add_v4(prm.accum + pixel, L.x, L.y, L.z, Y * Y);
}

// the ray records of a chunk (8 KB, contiguous) start their way from HBM to L2 when a warp claims the chunk (+1 %)
__device__ __forceinline__ void prefetch_chunk_rays(const DevPool& pool, uint32_t chunk_base, uint32_t lane) {
  const char* rp = reinterpret_cast<const char*>(pool.ray + 2 * (size_t)chunk_base);
  prefetch_l2(rp + 128u * lane);
  prefetch_l2(rp + 128u * (lane + 32u));
}

// ---- stage the top of the BVH in shared memory -------------------------------------------------------------------
__device__ __forceinline__ void stage_nodes(const DevScene& sc, uint4* snodes, uint32_t n_snodes) {
  const uint32_t words = n_snodes * 5u;
  for (uint32_t i = threadIdx.x; i < words; i += blockDim.x) snodes[i] = __ldg(sc.nodes + i);  // coalesced 128-bit
  __syncthreads();
}

// the octant remap table of trav_step<..., OCTMAP = true> (rtb_device.cuh), filled before stage_nodes()' barrier
__device__ __forceinline__ void octmap_fill() {
  for (uint32_t i = threadIdx.x; i < 8u * 256u; i += blockDim.x) s_octmap[i] = (uint8_t)octant_remap(i & 0xFFu, i >> 8);
}

// media + classification + result write of one finished ray (Material trait dispatch, material.rs:11-21): the info word
// carries material | face mode | shade queue, resolved on the host, so no material fetch is needed here
__device__ __forceinline__ void finish_ray(const DevScene& sc, const DevPool& pool, const DevParams& prm, uint32_t slot,
                                           float3 o, float3 d, Closest best) {
  if (sc.n_media) {
    const uint32_t pixel = __float_as_uint(pool.st[2 * slot].w);
    const uint32_t st = __float_as_uint(pool.st[2 * slot + 1].w);
    intersect_media(sc, o, d, RTB_TMIN, best, pixel, st >> 8, (st & 0xFFu) + 1u, prm.seed, !(prm.opt & RTB_OPT_PROBE));
  }
  uint32_t queue = Q_TERMINAL, minfo = 0;
  if (best.ref != REF_MISS) {
    const uint32_t type = best.ref >> REF_TYPE_SHIFT, idx = best.ref & REF_INDEX_MASK;
    minfo = type == PT_MEDIUM ? sc.media[idx].minfo : __ldg(&sc.info[type][idx].y);
    queue = RTB_MINFO_QUEUE(minfo);
  }
  RTB_CHECK(CHK_SLOT, slot < pool.n);
  pool.hit[slot] = make_float4(best.t, __uint_as_float(best.ref), __uint_as_float(minfo), 0.f);
  pool.cls[slot] = (uint8_t)queue;
}

// a ray whose closest hit the f32 tests could not decide: queued for the exact pass (rare: 0.03-0.3 % of the rays, so
// the one atomic per entry is uncontended in practice)
__device__ __forceinline__ void queue_fix(const DevPool& pool, uint32_t slot, uint32_t kind, float lo, float hi) {
  const uint32_t qi = atomicAdd(&pool.c->redo_count[0], 1u);
  RTB_CHECK(CHK_QUEUE, qi < pool.n && slot < pool.n);
  pool.redo[0][qi] =
      make_uint4(slot | (kind == FIX_REFINE ? RTB_REDO_REFINE : 0u), __float_as_uint(lo), __float_as_uint(hi), 0u);
}

// ---- the exact pass (out of line: it must not cost the hot kernels a register) -----------------------------------------
// One queue entry: FIX_RETRACE = the ray is traced again with traverse_exact() inside the slab the hot kernel handed
// over; FIX_REFINE = the (certain) hit's distance is recomputed in f64 (returns 1).  The hit record and the slot's class
// are rewritten before the shade kernels of the iteration run.
// `dsc` is the scene struct in DEVICE memory (DevScene::self): passing the kernel parameter by reference would force the
// compiler to copy the whole parameter block into every thread's local memory.
__device__ __forceinline__ void finish_ray(const DevScene& sc, const DevPool& pool, const DevParams& prm, uint32_t slot,
                                           float3 o, float3 d, Closest best);
static __device__ __noinline__ uint32_t fix_one(const DevScene* __restrict__ dsc, float4* ray, float4* st, float4* hit, uint8_t* cls,
                                                DevCounters* c, uint4 q, uint32_t seed, uint32_t opt) {
  const DevScene& sc = *dsc;
  DevPool pool;
  pool.n = 0xFFFFFFFFu; pool.n_chunks = 0;
  pool.ray = ray; pool.st = st; pool.hit = hit; pool.cls = cls;
  pool.redo[0] = pool.redo[1] = nullptr; pool.cursor = nullptr; pool.c = c;
  DevParams prm;
  prm.seed = seed; prm.opt = opt;
  const uint32_t slot = q.x & ~RTB_REDO_REFINE;
  const float4 ro = ray[2 * slot], rd = ray[2 * slot + 1];
  if (q.x & RTB_REDO_REFINE) {
    const float4 h = hit[slot];
    hit[slot].x = refine_hit(sc, __float_as_uint(h.y), xyz(ro), xyz(rd), ro.w, h.x);
    return 1u;
  }
  const Closest best = traverse_exact(sc, xyz(ro), xyz(rd), ro.w, __uint_as_float(q.y), __uint_as_float(q.z));
  finish_ray(sc, pool, prm, slot, xyz(ro), xyz(rd), best);
  return 0u;
}

// The entries the last extend launch queued, one per lane, spread over all warps of the grid.  Returns (entries handled, of
// which refinements) of this thread.
// (Measured and not kept: running this as the PROLOGUE of the next extend launch instead of its own kernel — the queued
// hits are then shaded one iteration late (C1 217 -> 257 iterations) and a 20 us single-lane exact trace stalls a warp
// whose chunks are statically assigned: C1 7997 -> 7390, C3 3711 -> 3438 Mrays/s, profiles/r3_ab.md.)
__device__ __forceinline__ uint2 fix_prologue(const DevScene& sc, const DevPool& pool, const DevParams& prm, uint32_t warp_in_grid,
                                              uint32_t n_warps_in_grid, uint32_t lane) {
  const uint32_t n = pool.c->redo_count[0];
  uint2 done = make_uint2(0u, 0u);
  for (uint32_t i = warp_in_grid * 32u + lane; i < n; i += n_warps_in_grid * 32u) {
    done.y += fix_one(sc.self, pool.ray, pool.st, pool.hit, pool.cls, pool.c, pool.redo[0][i], prm.seed, prm.opt);
    ++done.x;
  }
  return done;
}

// ---- warp-local chunk lists -------------------------------------------------------------------------------------------
// A warp owns RTB_CHUNK consecutive slots; lane l holds the class bytes of slots 8l..8l+7 (`cw`).  append_class() appends
// the chunk-relative indices of the slots whose class is `key` to the warp's shared-memory list (ascending slot order)
// and returns the new list length.  Must be executed by all 32 lanes.
__device__ __forceinline__ uint32_t append_class(uint2 cw, uint32_t key, uint8_t* list, uint32_t len, uint32_t lane) {
  // bytes equal to key -> 0xFF (SIMD-in-a-word compare), one bit per matching slot
  // (bits 0-2 of a class byte = the class; bits 3-5 = the direction octant of the slot's ray when octant ordering is on)
  const uint32_t e0 = __vcmpeq4(cw.x & 0x07070707u, key * 0x01010101u), e1 = __vcmpeq4(cw.y & 0x07070707u, key * 0x01010101u);
  const uint32_t cnt = (__popc(e0) + __popc(e1)) >> 3;
  uint32_t incl = cnt;
#pragma unroll
  for (uint32_t d = 1; d < 32; d <<= 1) {
    const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += v;
  }
  const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
  if (total) {
    uint32_t pos = len + incl - cnt;
#pragma unroll
    for (uint32_t j = 0; j < 8; ++j)
      if (((j < 4 ? e0 : e1) >> (8 * (j & 3))) & 1u) {
        RTB_CHECK(CHK_LIST, pos < RTB_CHUNK);
        list[pos++] = (uint8_t)(8u * lane + j);
      }
  }
  return len + total;
}

// extend's order of a chunk: the live slots sorted by the kernel that produced their ray — restarted slots (new camera
// rays: consecutive path numbers = neighbouring pixels of one tile) first, then the Lambertian bounces, metal, glass,
// media.  Rays of one kind share warps, so the coherent primary rays are not diluted by incoherent bounce rays
// (slot order alone: C1 extend 27.2 -> 32.3 ms, C3 68.6 -> 86.0 ms, profiles/r2_ab.md §4).
__device__ __forceinline__ uint32_t build_extend_list(const DevPool& pool, uint32_t chunk, uint8_t* list, uint32_t lane) {
  const uint2 cw = *reinterpret_cast<const uint2*>(pool.cls + chunk * RTB_CHUNK + 8u * lane);
  uint32_t len = 0;
  len = append_class(cw, CLS_NEW, list, len, lane);
  len = append_class(cw, Q_TERMINAL, list, len, lane);
  len = append_class(cw, Q_LAMBERT, list, len, lane);
  len = append_class(cw, Q_METAL, list, len, lane);
  len = append_class(cw, Q_DIELECTRIC, list, len, lane);
  len = append_class(cw, Q_ISOTROPIC, list, len, lane);
  __syncwarp();
  return len;
}

// The same list ordered by (ray kind, direction octant): a counting sort over 6 x 8 buckets in shared memory.  Rays of one
// octant descend the tree in the same child order (slot ^ octant), so a warp's lanes visit the same nodes for longer and
// their node / primitive fetches hit the same cache lines (bounce rays of one chunk start from neighbouring surfaces but
// scatter in all directions).  `cnt` = 64 per-warp counters.
__device__ __forceinline__ uint32_t build_extend_list_sorted(const DevPool& pool, uint32_t chunk, uint8_t* list, uint32_t* cnt, uint32_t lane) {
  const uint2 cw = *reinterpret_cast<const uint2*>(pool.cls + chunk * RTB_CHUNK + 8u * lane);
  cnt[lane] = 0u;
  cnt[lane + 32u] = 0u;
  __syncwarp();
  uint32_t key[8], rank[8];
#pragma unroll
  for (uint32_t j = 0; j < 8; ++j) {
    const uint32_t b = ((j < 4 ? cw.x : cw.y) >> (8 * (j & 3))) & 0xFFu, cls = b & 7u;
    // kind rank: restarted camera rays first (coherent), then the bounce kinds; dead slots are skipped
    key[j] = cls == CLS_DEAD ? 64u : ((cls == CLS_NEW ? 0u : cls + 1u) << 3) | ((b >> 3) & 7u);
    rank[j] = key[j] < 64u ? atomicAdd(&cnt[key[j]], 1u) : 0u;
  }
  __syncwarp();
  // exclusive scan of the 48 bucket counts (lane l: buckets l and 32 + l)
  const uint32_t v0 = cnt[lane], v1 = lane < 16u ? cnt[32u + lane] : 0u;
  uint32_t i0 = v0, i1 = v1;
#pragma unroll
  for (uint32_t d = 1; d < 32; d <<= 1) {
    const uint32_t a = __shfl_up_sync(0xffffffffu, i0, d), b2 = __shfl_up_sync(0xffffffffu, i1, d);
    if (lane >= d) { i0 += a; i1 += b2; }
  }
  const uint32_t t0 = __shfl_sync(0xffffffffu, i0, 31), total = t0 + __shfl_sync(0xffffffffu, i1, 15);
  __syncwarp();
  cnt[lane] = i0 - v0;
  if (lane < 16u) cnt[32u + lane] = t0 + i1 - v1;
  __syncwarp();
#pragma unroll
  for (uint32_t j = 0; j < 8; ++j)
    if (key[j] < 64u) {
      RTB_CHECK(CHK_LIST, cnt[key[j]] + rank[j] < RTB_CHUNK);
      list[cnt[key[j]] + rank[j]] = (uint8_t)(8u * lane + j);
    }
  __syncwarp();
  return total;
}

// instrumented build (COUNT): a warp's node visits / primitive tests per type go to the lane's counters
__device__ __forceinline__ void report_counts(DevCounters* c, uint32_t nv, TestCount nt, uint32_t lane) {
  nv = __reduce_add_sync(0xffffffffu, nv);
  uint32_t tot = 0;
#pragma unroll
  for (uint32_t t = 0; t < PT_COUNT; ++t) {
    nt.n[t] = __reduce_add_sync(0xffffffffu, nt.n[t]);
    tot += nt.n[t];
  }
  if (lane == 0) {
    atomicAdd(&c->nodes_visited, (unsigned long long)nv);
    atomicAdd(&c->prims_tested, (unsigned long long)tot);
    for (uint32_t t = 0; t < PT_COUNT; ++t)
      if (nt.n[t]) atomicAdd(&c->prims_tested_type[t], (unsigned long long)nt.n[t]);
  }
}

// ---- extend ------------------------------------------------------------------------------------------------------
// Dynamic-fetch variant (deep trees).  Persistent warps: every lane owns one in-flight ray and advances it by ONE node
// visit per loop iteration, so the 32 lanes execute the node-decode code together.  Rays finish after different
// numbers of visits; instead of idling until the slowest lane of the warp is done a finished lane immediately swaps
// its ray:
//   * rays are PREFETCHED 32 slots at a time by the whole warp (coalesced class + ray loads, 1/d, the scene's global
//     primitives) into a per-warp shared-memory buffer; an idle lane takes the next prepared ray with four LDS.128;
//   * results are pushed to a per-warp shared-memory buffer and WRITTEN OUT 32 at a time by the whole warp.
// So the set-up / tear-down code always runs with full warps and only the swap itself is divergent.
// Work is claimed from a device-side cursor one chunk (RTB_CHUNK slots) at a time; the chunk's live slots are ordered by
// ray kind (build_extend_list) and handed out 32 at a time.
// COUNT = true: the instrumented build used for the roofline's algorithmic work (nodes visited / primitives tested per
// segment); the timed path runs COUNT = false.
// Register caps.  The one-ray-per-thread kernels run 2 CTAs/SM (configure_launch) with at most 80 registers: 2 x 256 x 80 =
// 41 K of the 64 K registers, so a 256-thread shade CTA of another lane fits beside them.  Measured (C1, Mrays/s): cap 72:
// 4476, 80: 4497, 88: 4326, 96: 3947 — the extend kernel alone is fastest at 88+, the overlapped pipeline at 80.
// The dynamic-fetch kernel (deep trees) is latency-bound on its dependent node -> primitive fetches and wants WARPS: at 64
// registers (no spills) four extend CTAs — of four wavefront lanes — share an SM, 32 warps instead of 24: C4 3706 -> 4096
// Mrays/s (profiles/r3_ab.md §9).
#ifndef RTB_EXTEND_MAXREG
#define RTB_EXTEND_MAXREG 80
#endif
#ifndef RTB_EXTEND_DYN_MAXREG
#define RTB_EXTEND_DYN_MAXREG 64
#endif
struct ExtIn { float4 o_time, d_slot, idir_oct, best; };  // best = (t, ref, group word, t upper bound) after the global primitives
struct ExtOut { float t; uint32_t ref, slot, redo; float lo, hi; uint32_t _pad[2]; };
#define RTB_EXTEND_WARPS (RTB_EXTEND_THREADS / 32)

// Leaf primitives are always PARKED here (drain_parked; threshold = DevParams::opt bits 8-13, default 14 lanes): testing
// them at the node visit instead costs 7 % on the 1 M-triangle mesh (profiles/r3_ab.md §2).
template <bool COUNT>
__global__ void __maxnreg__(RTB_EXTEND_DYN_MAXREG)
k_extend(DevScene sc, DevPool pool, DevParams prm, uint32_t n_snodes) {
  extern __shared__ uint4 snodes[];
  __shared__ ExtIn s_in[RTB_EXTEND_WARPS][32];
  __shared__ ExtOut s_out[RTB_EXTEND_WARPS][32];
  __shared__ uint8_t s_list[RTB_EXTEND_WARPS][RTB_CHUNK];
  __shared__ uint4 s_park[RTB_EXTEND_WARPS][32];
  DevCounters* c = pool.c;
  stage_nodes(sc, snodes, n_snodes);
  uint32_t sbase = (uint32_t)__cvta_generic_to_shared(snodes);
  asm volatile("mov.u32 %0, %0;" : "+r"(sbase));  // opaque: keep it in a register instead of re-deriving it per node visit
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t lt_mask = (1u << lane) - 1u;
  const uint32_t park_min = max(1u, (prm.opt >> RTB_OPT_PARK_SHIFT) & RTB_OPT_PARK_MASK);  // lanes that must wait before a drain
  uint4* park = &s_park[warp][lane];
  uint32_t parked_mask = 0;  // warp-uniform: lanes with parked leaf primitives
  ExtIn* in = s_in[warp];
  ExtOut* out = s_out[warp];
  uint8_t* list = s_list[warp];
  uint32_t idle = 0xffffffffu;  // warp-uniform: lanes without a ray in flight
  uint32_t slot = 0;
  uint32_t in_head = 0, in_count = 0, out_count = 0;  // warp-uniform
  uint32_t chunk_base = 0, list_pos = 0, list_len = 0;  // warp-uniform: the claimed chunk's ordered slot list
  bool exhausted = false;                              // warp-uniform: no more chunks to claim
  uint32_t n_rays = 0;                                 // warp-uniform
  Trav tv;
  uint2 stack[RTB_STACK];
  uint32_t nv = 0;
  TestCount nt{};
  // idle lanes are refilled when at least this many wait (or nobody runs): a swap costs the whole warp ~40 issue slots
  // however few lanes take part (C4 ext_ms: 1 -> 21.6, 4 -> 21.2, 8 -> 21.1, 16 -> 21.7; profiles/r2_ab.md §7)
  const uint32_t refill_min = 8u;
  auto flush = [&]() {  // executed by the whole warp
    __syncwarp();
    if (lane < out_count) {
      const ExtOut h = out[lane];
      float3 o = f3(0.f, 0.f, 0.f), d = o;
      if (sc.n_media) {
        o = xyz(pool.ray[2 * h.slot]);
        d = xyz(pool.ray[2 * h.slot + 1]);
      }
      finish_ray(sc, pool, prm, h.slot, o, d, Closest{h.t, h.t, h.ref});
      uint32_t redo = h.redo;
      if (redo == FIX_NOMINATED) redo = resolve_nominated(sc, h.ref, xyz(pool.ray[2 * h.slot]), xyz(pool.ray[2 * h.slot + 1]));
      if (redo) queue_fix(pool, h.slot, redo, h.lo, h.hi);
    }
    out_count = 0;
    __syncwarp();
  };

  for (;;) {
    // ---- idle lanes take prepared rays ----------------------------------------------------------------------------
    const uint32_t n_idle = __popc(idle);
    if (n_idle >= refill_min || idle == 0xffffffffu) {
      while (in_head == in_count && !(exhausted && list_pos == list_len)) {  // prepare the next 32 rays
        if (list_pos == list_len) {  // claim the next chunk and order its live slots by ray kind
          uint32_t ch = 0;
          if (lane == 0) ch = atomicAdd(&c->ext_cursor, 1u);
          ch = __shfl_sync(0xffffffffu, ch, 0);
          if (ch >= pool.n_chunks) {
            exhausted = true;
            break;
          }
          chunk_base = ch * RTB_CHUNK;
          list_len = build_extend_list(pool, ch, list, lane);
          list_pos = 0;
          n_rays += list_len;
          if (list_len == 0) continue;
        }
        const bool live = list_pos + lane < list_len;
        const uint32_t sl = chunk_base + (live ? list[list_pos + lane] : 0u);
        in_head = 0;
        in_count = min(32u, list_len - list_pos);
        list_pos += in_count;
        __syncwarp();
        if (live) {
          const float4 ro = pool.ray[2 * sl], rd = pool.ray[2 * sl + 1];
          // set-up runs here with the whole warp: 1/d, and the scene's global primitives (tested before the tree)
          Trav t0;
          trav_init(t0, xyz(ro), xyz(rd), ro.w);
          trav_globals<COUNT>(sc, t0, RTB_TMIN, nt);
          ExtIn& e = in[lane];
          e.o_time = ro;
          e.d_slot = make_float4(rd.x, rd.y, rd.z, __uint_as_float(sl));
          // (an ambiguity among the global primitives is handed over as "undecided from distance 0": bit 9)
          e.idir_oct = make_float4(t0.idx, t0.idy, t0.idz, __uint_as_float(t0.octinv | (t0.amb < INFINITY ? 0x200u : 0u)));
          e.best = make_float4(t0.best.t, __uint_as_float(t0.best.ref), __uint_as_float(t0.grp.y), t0.best.hi);
        }
        __syncwarp();
      }
      const uint32_t avail = in_count - in_head;
      if (avail) {
        const uint32_t rank = __popc(idle & lt_mask);
        const bool take = ((idle >> lane) & 1u) && rank < avail;
        if (take) {
          const ExtIn r = in[in_head + rank];
          tv.o = xyz(r.o_time); tv.time = r.o_time.w;
          tv.d = xyz(r.d_slot); slot = __float_as_uint(r.d_slot.w);
          tv.idx = r.idir_oct.x; tv.idy = r.idir_oct.y; tv.idz = r.idir_oct.z;
          tv.octinv = __float_as_uint(r.idir_oct.w) & (7u | RTB_TRAV_COARSE);
          tv.amb = (__float_as_uint(r.idir_oct.w) & 0x200u) ? 0.0f : INFINITY;
          tv.grp = make_uint2(0u, __float_as_uint(r.best.z));
          tv.sp = 0;
          tv.best = Closest{r.best.x, r.best.w, __float_as_uint(r.best.y)};
        }
        idle &= ~__ballot_sync(0xffffffffu, take);
        in_head += min(n_idle, avail);
      }
    }
    if (idle == 0xffffffffu) {  // nobody runs and nothing could be taken
      if (out_count) flush();
      if (exhausted && list_pos == list_len && in_head == in_count) break;
      continue;
    }
    // ---- one node visit (or pop) per running lane -------------------------------------------------------------------
    bool finished = false;
    {
      bool parked = (parked_mask >> lane) & 1u;
      if (!(((idle | parked_mask) >> lane) & 1u))
        finished = !trav_step_park<COUNT>(sc, snodes, sbase, n_snodes, tv, stack, RTB_TMIN, nv, park, parked);
      parked_mask = __ballot_sync(0xffffffffu, parked);
      // drain when enough lanes wait, or when nobody is left to visit nodes meanwhile
      if (parked_mask && ((uint32_t)__popc(parked_mask) >= park_min || (~(idle | parked_mask | __ballot_sync(0xffffffffu, finished))) == 0u)) {
        drain_parked<COUNT>(sc, tv, RTB_TMIN, park, parked, nt);
        parked_mask = 0;
      }
    }
    // ---- finished lanes push their result -------------------------------------------------------------------------
    const uint32_t done = __ballot_sync(0xffffffffu, finished);
    if (done) {
      if (out_count + __popc(done) > 32u) flush();
      if (finished) out[out_count + __popc(done & lt_mask)] = ExtOut{tv.best.t, tv.best.ref, slot, fix_kind_cheap(tv), slab_lo(tv), tv.best.hi, {0u, 0u}};
      out_count += __popc(done);
      idle |= done;
    }
  }
  if (lane == 0 && n_rays) atomicAdd(&c->iter_rays, n_rays);
  if (COUNT) report_counts(c, nv, nt, lane);
}

// ---- warp-queue extend (deep trees) ----------------------------------------------------------------------------------
// The per-line profile of the kernels above on trees outside the stage (profiles/r3g_lines.md): node visits run with
// 13-17 of 32 lanes (lanes whose ray waits for a refill or for its leaf tests) and the primitive tests with 3-4 of 32 (the
// few lanes whose node happened to have a leaf hit) — a third of all issued warp instructions at a tenth of the width.
// Here the WARP, not the lane, owns the rays: RTB_WQ_RAYS rays per warp live entirely in shared memory (ray, closest hit,
// traversal group AND stack), and any lane can advance any of them:
//   * a node step takes (up to) 32 READY rays — lane j the j-th of them — through one node visit each;
//   * a node visit that hits leaves does not test them: the ray goes to the queue of its leaf's primitive class (sphere /
//     quad / triangle) and waits; a queue is served by all lanes, 32 rays at a time, a bounded number of primitives per ray
//     and round (same per-ray order of tests as everywhere else, hence the same hits and counters);
//   * each loop iteration does whichever has more lanes' worth of work (node step / serving the fullest queue);
//   * finished rays are pushed to the per-warp result buffer and written out 32 at a time, free table entries take new rays
//     straight from the chunk list.
// All scheduling state (free / ready masks, queue heads) is warp-uniform registers.
#define RTB_WQ_RAYS 48u
#define RTB_WQ_STACK 12u  /* levels: configure_launch() uses this kernel only for trees of at most this depth */
struct WqWarp {
  float4 o_time[RTB_WQ_RAYS];
  float4 d_slot[RTB_WQ_RAYS];
  float4 idir_oct[RTB_WQ_RAYS];
  float4 best[RTB_WQ_RAYS];      // t, ref, upper bound of the exact t, ambiguity horizon
  uint4 trav[RTB_WQ_RAYS];       // current group (x, y), stack depth, flags (RTB_TRAV_COARSE)
  uint4 rec[RTB_WQ_RAYS];        // the leaf record of the last node visit (x = leaf mask | next primitive << 8) while the ray waits
  uint2 stack[RTB_WQ_STACK][RTB_WQ_RAYS];  // level-major: the lanes of a node step touch consecutive words
  ExtOut out[32];
  uint8_t list[RTB_CHUNK];
  uint8_t q[3][64];              // per class: ring of waiting rays (a ray waits in at most one queue: never overflows)
  uint8_t ready[64];             // the ready rays of the current node step, compacted
};

template <bool COUNT>
__global__ void __maxnreg__(RTB_EXTEND_MAXREG)
k_extend_wq(DevScene sc, DevPool pool, DevParams prm, uint32_t n_snodes) {
  extern __shared__ uint4 snodes[];
  DevCounters* c = pool.c;
  stage_nodes(sc, snodes, n_snodes);
  uint32_t sbase = (uint32_t)__cvta_generic_to_shared(snodes);
  asm volatile("mov.u32 %0, %0;" : "+r"(sbase));
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t lt_mask = (1u << lane) - 1u;
  WqWarp& W = reinterpret_cast<WqWarp*>(snodes + 5u * n_snodes)[warp];
  // warp-uniform scheduling state: rays 0-31 in the *_lo masks, 32-47 in *_hi
  uint32_t free_lo = 0xffffffffu, free_hi = (1u << (RTB_WQ_RAYS - 32u)) - 1u, rdy_lo = 0u, rdy_hi = 0u;
  uint32_t qh0 = 0, qh1 = 0, qh2 = 0, qn0 = 0, qn1 = 0, qn2 = 0;  // ring head / length per class
  uint32_t out_count = 0, flip = 0;
  uint32_t chunk_base = 0, list_pos = 0, list_len = 0;
  bool exhausted = false;
  uint32_t n_rays = 0;
  uint32_t nv = 0;
  TestCount nt{};
  const uint32_t refill_min = 8u;
  // a queue is served before a node step when it holds at least this many rays (or more rays than lanes could step)
  const uint32_t serve_min = max(1u, (prm.opt >> RTB_OPT_PARK_SHIFT) & RTB_OPT_PARK_MASK);
  const uint32_t serve_tests = max(1u, (prm.opt >> 16) & 15u);  // primitive tests per ray and serving round
  auto flush = [&]() {
    __syncwarp();
    if (lane < out_count) {
      const ExtOut h = W.out[lane];
      float3 o = f3(0.f, 0.f, 0.f), d = o;
      if (sc.n_media) {
        o = xyz(pool.ray[2 * h.slot]);
        d = xyz(pool.ray[2 * h.slot + 1]);
      }
      finish_ray(sc, pool, prm, h.slot, o, d, Closest{h.t, h.t, h.ref});
      uint32_t redo = h.redo;
      if (redo == FIX_NOMINATED) redo = resolve_nominated(sc, h.ref, xyz(pool.ray[2 * h.slot]), xyz(pool.ray[2 * h.slot + 1]));
      if (redo) queue_fix(pool, h.slot, redo, h.lo, h.hi);
    }
    out_count = 0;
    __syncwarp();
  };

  for (;;) {
    const uint32_t n_ready = __popc(rdy_lo) + __popc(rdy_hi);
    const uint32_t n_free = __popc(free_lo) + __popc(free_hi);
    const bool more_rays = !(exhausted && list_pos == list_len);
    const uint32_t q_max = max(qn0, max(qn1, qn2));
    // ---- free table entries take new rays ---------------------------------------------------------------------------
    if (more_rays && n_free && (n_free >= refill_min || (n_ready == 0u && q_max == 0u))) {
      uint32_t left = n_free;
      while (left) {
        if (list_pos == list_len) {
          uint32_t ch = 0;
          if (lane == 0) ch = atomicAdd(&c->ext_cursor, 1u);
          ch = __shfl_sync(0xffffffffu, ch, 0);
          if (ch >= pool.n_chunks) {
            exhausted = true;
            break;
          }
          __syncwarp();
          chunk_base = ch * RTB_CHUNK;
          prefetch_chunk_rays(pool, chunk_base, lane);
          list_len = build_extend_list(pool, ch, W.list, lane);
          list_pos = 0;
          n_rays += list_len;
          if (list_len == 0) continue;
        }
        const uint32_t n = min(left, list_len - list_pos);
        const uint32_t base_hi = __popc(free_lo);
#pragma unroll 1
        for (uint32_t w = 0; w < 2u; ++w) {  // lane l fills table entry l, then entry 32 + l
          const uint32_t fm = w ? free_hi : free_lo;
          const uint32_t rank = (w ? base_hi : 0u) + __popc(fm & lt_mask);
          const bool take = ((fm >> lane) & 1u) && rank < n;
          if (take) {
            const uint32_t sl = chunk_base + W.list[list_pos + rank];
            const float4 ro = pool.ray[2 * sl], rd = pool.ray[2 * sl + 1];
            Trav t0;
            trav_init(t0, xyz(ro), xyz(rd), ro.w);
            trav_globals<COUNT>(sc, t0, RTB_TMIN, nt);
            const uint32_t r = w * 32u + lane;
            W.o_time[r] = ro;
            W.d_slot[r] = make_float4(rd.x, rd.y, rd.z, __uint_as_float(sl));
            W.idir_oct[r] = make_float4(t0.idx, t0.idy, t0.idz, __uint_as_float(t0.octinv & 7u));
            W.best[r] = make_float4(t0.best.t, __uint_as_float(t0.best.ref), t0.best.hi, t0.amb);
            W.trav[r] = make_uint4(0u, t0.grp.y, 0u, t0.octinv & RTB_TRAV_COARSE);
          }
          const uint32_t took = __ballot_sync(0xffffffffu, take);
          if (w) { free_hi &= ~took; rdy_hi |= took; } else { free_lo &= ~took; rdy_lo |= took; }
        }
        list_pos += n;
        left -= n;
      }
      __syncwarp();
      continue;
    }
    if (n_ready == 0u && q_max == 0u) {  // nothing in flight and nothing left to take
      if (out_count) flush();
      break;
    }
    if (q_max >= serve_min || q_max > n_ready) {
      // ---- serve the fullest queue: lane j runs leaf tests of the j-th waiting ray ---------------------------------------
      const uint32_t cls = qn0 == q_max ? 0u : (qn1 == q_max ? 1u : 2u);
      const uint32_t head = cls == 0u ? qh0 : (cls == 1u ? qh1 : qh2);
      const uint32_t n = min(32u, q_max);
      uint32_t r = 64u;
      bool again = false;  // primitives left in the record: the ray goes back to the end of the queue
      if (lane < n) {
        r = W.q[cls][(head + lane) & 63u];
        RTB_CHECK(CHK_QUEUE, r < RTB_WQ_RAYS);
        const float4 ro = W.o_time[r], rd = W.d_slot[r], b = W.best[r];
        const uint4 rc = W.rec[r];
        Closest best{b.x, b.z, __float_as_uint(b.y)};
        float amb = b.w;
        uint32_t flags = W.trav[r].w;
        // at most `serve_tests` primitives per ray and round, so that the lanes of a round stay together (a ray that grazes a
        // row of leaves has 6+ primitives to test, most have 1-2)
        uint32_t leaf = rc.x & 0xFFu, k = rc.x >> 8;
        const uint32_t ptype = rc.y >> REF_TYPE_SHIFT, pbase = rc.y & REF_INDEX_MASK;
        for (uint32_t it = 0; it < serve_tests && leaf; ++it) {
          const uint32_t sl = __ffs(leaf) - 1;
          const uint32_t m = ((sl < 4 ? rc.z : rc.w) >> (8 * (sl & 3))) & 0xFFu;
          intersect_prim<COUNT>(sc, ptype, pbase + (m & 31u) + k, xyz(ro), xyz(rd), ro.w, RTB_TMIN, best, amb, flags, nt);
          if (++k >= (m >> 5)) { k = 0; leaf &= leaf - 1; }
        }
        W.best[r] = make_float4(best.t, __uint_as_float(best.ref), best.hi, amb);
        W.trav[r].w = flags;
        again = leaf != 0u;
        if (again) W.rec[r].x = leaf | (k << 8);
      }
      const uint32_t again_mask = __ballot_sync(0xffffffffu, again);
      rdy_lo |= __reduce_or_sync(0xffffffffu, !again && r < 32u ? 1u << r : 0u);
      rdy_hi |= __reduce_or_sync(0xffffffffu, !again && (r & 32u) ? 1u << (r & 31u) : 0u);
      __syncwarp();
      if (again) W.q[cls][(head + q_max + __popc(again_mask & lt_mask)) & 63u] = (uint8_t)r;  // (n <= 32 entries were read above)
      const uint32_t delta = __popc(again_mask) - n;
      if (cls == 0u) { qh0 += n; qn0 += delta; } else if (cls == 1u) { qh1 += n; qn1 += delta; } else { qh2 += n; qn2 += delta; }
      __syncwarp();
      continue;
    }
    // ---- one node visit (or pop) of up to 32 ready rays: lane j takes the j-th ------------------------------------------
    if ((rdy_lo >> lane) & 1u) W.ready[__popc(rdy_lo & lt_mask)] = (uint8_t)lane;
    if ((rdy_hi >> lane) & 1u) W.ready[__popc(rdy_lo) + __popc(rdy_hi & lt_mask)] = (uint8_t)(32u + lane);
    __syncwarp();
    flip ^= 1u;
    bool finished = false, leafed = false;
    uint32_t cls = 3u, r = 64u;
    if (lane < n_ready) {
      r = W.ready[lane + (flip && n_ready > 32u ? n_ready - 32u : 0u)];  // (more than 32 ready: alternate which end waits)
      Trav tv;
      const float4 ro = W.o_time[r], id = W.idir_oct[r];
      const uint4 tr = W.trav[r];
      tv.o = xyz(ro);
      tv.idx = id.x; tv.idy = id.y; tv.idz = id.z;
      tv.octinv = __float_as_uint(id.w);
      tv.grp = make_uint2(tr.x, tr.y);
      tv.sp = (int)tr.z;
      tv.best.hi = W.best[r].z;
      finished = !trav_step<COUNT, false, (int)RTB_WQ_RAYS>(sc, snodes, sbase, n_snodes, tv, &W.stack[0][r], RTB_TMIN, nv,
                                                            [&](uint32_t leaf, uint32_t w1y, uint32_t w1z, uint32_t w1w) {
                                                              W.rec[r] = make_uint4(leaf, w1y, w1z, w1w);
                                                              const uint32_t type = w1y >> REF_TYPE_SHIFT;
                                                              cls = type <= PT_MOVING ? 0u : type - 1u;
                                                              leafed = true;
                                                            });
      RTB_CHECK(CHK_STACK, tv.sp <= (int)RTB_WQ_STACK);
      if (!finished) {
        *reinterpret_cast<uint2*>(&W.trav[r]) = tv.grp;
        W.trav[r].z = (uint32_t)tv.sp;
      }
    }
    const uint32_t done = __ballot_sync(0xffffffffu, finished);
    const uint32_t leafs = __ballot_sync(0xffffffffu, leafed);
    if (done | leafs) {
      const uint32_t bit_lo = r < 32u ? 1u << r : 0u, bit_hi = (r & 32u) ? 1u << (r & 31u) : 0u;
      rdy_lo &= ~__reduce_or_sync(0xffffffffu, finished || leafed ? bit_lo : 0u);
      rdy_hi &= ~__reduce_or_sync(0xffffffffu, finished || leafed ? bit_hi : 0u);
      // ---- rays with leaf hits queue up by class ----------------------------------------------------------------------------
      if (leafs) {
        const uint32_t m0 = __ballot_sync(0xffffffffu, cls == 0u), m1 = __ballot_sync(0xffffffffu, cls == 1u), m2 = leafs & ~(m0 | m1);
        if (leafed) {
          const uint32_t mine = cls == 0u ? m0 : (cls == 1u ? m1 : m2);
          const uint32_t end = cls == 0u ? qh0 + qn0 : (cls == 1u ? qh1 + qn1 : qh2 + qn2);
          W.q[cls][(end + __popc(mine & lt_mask)) & 63u] = (uint8_t)r;
        }
        qn0 += __popc(m0); qn1 += __popc(m1); qn2 += __popc(m2);
      }
      // ---- finished rays push their result ------------------------------------------------------------------------------
      if (done) {
        free_lo |= __reduce_or_sync(0xffffffffu, finished ? bit_lo : 0u);
        free_hi |= __reduce_or_sync(0xffffffffu, finished ? bit_hi : 0u);
        if (out_count + __popc(done) > 32u) flush();
        if (finished) {
          const float4 b = W.best[r];
          Trav tv;
          tv.best = Closest{b.x, b.z, __float_as_uint(b.y)};
          tv.amb = b.w;
          tv.octinv = W.trav[r].w;
          W.out[out_count + __popc(done & lt_mask)] =
              ExtOut{tv.best.t, tv.best.ref, __float_as_uint(W.d_slot[r].w), fix_kind_cheap(tv), slab_lo(tv), tv.best.hi, {0u, 0u}};
        }
        out_count += __popc(done);
      }
    }
    __syncwarp();
  }
  if (lane == 0 && n_rays) atomicAdd(&c->iter_rays, n_rays);
  if (COUNT) report_counts(c, nv, nt, lane);
}

// One ray per thread to completion (small trees: all lanes start at the root together, so root-level work stays
// converged).  Slot-stable pool: a warp takes one chunk of RTB_CHUNK slots at a time, orders its live slots by ray kind
// (build_extend_list) and traces them 32 at a time; the next round's ray sectors are prefetched into L1 during the
// current traversal.  No queue, no atomics apart from one ray-count add per warp at the end.
// SORT: each chunk's rays are ordered by (ray kind, direction octant) instead of by kind alone (trees that do not fit the
// stage: C3 +6 %; fully staged trees lose 3 %, the dynamic kernel is indifferent — profiles/r3_ab.md §4).  Parking the
// leaf tests (as the dynamic kernel does) costs this kernel 13 %: with one ray per thread the lanes that wait for a drain
// are simply idle.  Both are compile-time choices so that each variant's loop carries only its own path.
// SPHSTAGE (fully staged trees whose sphere array fits RTB_SPHERE_STAGE_BYTES, configure_launch): the sphere records are
// staged in shared memory after the nodes and the leaf tests read them from there (trav_step_fast).
template <bool COUNT, bool ALL_STAGED, bool SORT, bool SPHSTAGE = false>
__global__ void __maxnreg__(RTB_EXTEND_MAXREG)
k_extend_static(DevScene sc, DevPool pool, DevParams prm, uint32_t n_snodes) {
  static_assert(!SPHSTAGE || (ALL_STAGED && !COUNT), "the sphere stage is built for the fully staged production kernel");
  extern __shared__ uint4 snodes[];
  __shared__ uint8_t s_list[RTB_EXTEND_WARPS][RTB_CHUNK];
  __shared__ uint32_t s_cnt[SORT ? RTB_EXTEND_WARPS : 1][64];
  DevCounters* c = pool.c;
  if constexpr (ALL_STAGED) octmap_fill();
  if constexpr (SPHSTAGE) {  // the sphere array right after the nodes (float4 records = 16-byte words), before stage_nodes()' barrier
    const uint4* sph = reinterpret_cast<const uint4*>(sc.geom[PT_SPHERE]);
    for (uint32_t i = threadIdx.x; i < sc.n_prims[PT_SPHERE]; i += blockDim.x) snodes[5u * n_snodes + i] = __ldg(sph + i);
  }
  stage_nodes(sc, snodes, n_snodes);
  uint32_t sbase = (uint32_t)__cvta_generic_to_shared(snodes);
  asm volatile("mov.u32 %0, %0;" : "+r"(sbase));  // opaque: keep it in a register instead of re-deriving it per node visit
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint8_t* list = s_list[warp];
  const uint32_t n_warps = gridDim.x * RTB_EXTEND_WARPS;
  uint32_t n_rays = 0, nv = 0;
  TestCount nt{};
  for (uint32_t chunk = blockIdx.x * RTB_EXTEND_WARPS + warp; chunk < pool.n_chunks; chunk += n_warps) {
    const uint32_t base = chunk * RTB_CHUNK;
    const uint32_t total = SORT ? build_extend_list_sorted(pool, chunk, list, s_cnt[SORT ? warp : 0], lane) : build_extend_list(pool, chunk, list, lane);
    n_rays += total;
    for (uint32_t r = 0; r < total; r += 32) {
      if (r + 32 + lane < total) prefetch_l1(pool.ray + 2 * (size_t)(base + list[r + 32 + lane]));
      if (r + lane < total) {
        const uint32_t slot = base + list[r + lane];
        const float4 ro = pool.ray[2 * slot];
        const float4 rd = pool.ray[2 * slot + 1];
        Closest best;
        float lo;
        // packed slab test and remap table in the fully staged production kernel (the counting build keeps the scalar
        // test: same decisions, and the packed one spills there)
        const uint32_t fix = traverse<COUNT, ALL_STAGED, ALL_STAGED && !COUNT, ALL_STAGED, SPHSTAGE>(
            sc, snodes, sbase, n_snodes, xyz(ro), xyz(rd), ro.w, RTB_TMIN, best, lo, nv, nt, sbase + n_snodes * 80u);
        finish_ray(sc, pool, prm, slot, xyz(ro), xyz(rd), best);
        if (fix) queue_fix(pool, slot, fix, lo, best.hi);
      }
    }
    __syncwarp();  // the list is rewritten for the next chunk
  }
  if (lane == 0 && n_rays) atomicAdd(&c->iter_rays, n_rays);
  if (COUNT) report_counts(c, nv, nt, lane);
}

// ---- surface reconstruction in the shade kernels -------------------------------------------------------------------
struct Surf {
  float3 p, n, outward;  // n = normal against the ray (set_face_normal, hittable.rs:41-48)
  bool front;
  uint32_t mat, ref;
  bool uv;               // ATTR kernels: (tu, tv) are the texture coordinates of a triangle's shading record
  float tu, tv;
};

// barycentrics (u, v) of the point p in the triangle (v0, v0 + e1, v0 + e2): the (u, v) a triangle reports
__device__ __forceinline__ void tri_bary(float3 v0, float3 e1, float3 e2, float3 p, float& u, float& v) {
  const float3 nn = cross(e1, e2), pl = p - v0;
  const float inv = 1.0f / dot(nn, nn);
  u = dot(nn, cross(pl, e2)) * inv;
  v = dot(nn, cross(e1, pl)) * inv;
}

// Shading record of a mesh triangle (info bit 31 in an ATTR kernel; include/rtb200.h rtb_scene_set_mesh_attributes):
// ns = normalize(b0 n0 + b1 n1 + b2 n2) turned to the side of the ray-facing geometric normal s.n, which it then replaces
// (front_face stays the geometric one: surface_at has decided it); (u, v) interpolated the same way.  A non-finite or
// near-zero interpolated normal keeps the geometric one.  No bending towards the geometric surface (DESIGN.md §9).
__device__ __forceinline__ void surface_attr(const DevScene& sc, uint32_t idx, Surf& s) {
  RTB_CHECK(CHK_ATTR, idx < sc.xtab->n_attr);
  const float4* rec = sc.xtab->attr + 4 * (size_t)idx;
  const float3 v0 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx)), e1 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx + 1)) - v0,
               e2 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx + 2)) - v0;
  float b1, b2;
  tri_bary(v0, e1, e2, s.p, b1, b2);
  const float b0 = 1.0f - b1 - b2;
  const float4 w0 = __ldg(rec), w1 = __ldg(rec + 1), w2 = __ldg(rec + 2), w3 = __ldg(rec + 3);
  const uint32_t flags = __float_as_uint(w3.w);
  if (flags & ATTR_NORMALS) {
    const float3 sum = fma3(b0, xyz(w0), fma3(b1, xyz(w1), b2 * xyz(w2)));
    const float len2 = dot(sum, sum);
    if (isfinite(len2) && len2 >= 1e-20f) {
      const float3 ns = rsqrtf(len2) * sum;
      s.n = dot(ns, s.n) < 0.0f ? -ns : ns;
    }
  }
  if (flags & ATTR_UVS) {
    s.uv = true;
    s.tu = fmaf(b0, w0.w, fmaf(b1, w1.w, b2 * w2.w));
    s.tv = fmaf(b0, w3.x, fmaf(b1, w3.y, b2 * w3.z));
  }
}

// ATTR: the scene has triangles with shading records (rtb_scene_set_mesh_attributes); the kernels of other scenes are
// compiled without that path
template <bool ATTR = false>
__device__ __forceinline__ Surf surface_at(const DevScene& sc, uint32_t ref, uint32_t minfo, float3 o, float3 d, float time, float t) {
  Surf s;
  s.ref = ref;
  s.p = fma3(t, d, o);
  const uint32_t type = ref >> REF_TYPE_SHIFT, idx = ref & REF_INDEX_MASK;
  if (type == PT_MEDIUM) {  // constant_medium.rs:65-67: arbitrary normal, front_face = true
    s.n = s.outward = f3(1.f, 0.f, 0.f);
    s.front = true;
    s.mat = RTB_MINFO_MAT(minfo);
    return s;
  }
  if (type == PT_SPHERE) {
    const float4 g = __ldg(sc.geom[PT_SPHERE] + idx);
    s.outward = rcp_fast(g.w) * (s.p - xyz(g));  // sphere.rs:59
  } else if (type == PT_MOVING) {
    const float4 a = __ldg(sc.geom[PT_MOVING] + 2 * idx), b = __ldg(sc.geom[PT_MOVING] + 2 * idx + 1);
    s.outward = rcp_fast(a.w) * (s.p - fma3(time, xyz(b), xyz(a)));  // moving_sphere.rs:57-58
  } else if (type == PT_QUAD) {
    s.outward = xyz(__ldg(sc.geom[PT_QUAD] + 3 * idx));
  } else {
    const float3 v0 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx));
    const float3 e1 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx + 1)) - v0, e2 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx + 2)) - v0;
    s.outward = unit(cross(e1, e2));
  }
  s.mat = RTB_MINFO_MAT(minfo);
  bool ff = dot(d, s.outward) < 0.0f;
  s.n = ff ? s.outward : -s.outward;
  // wrappers rewrite front_face (hittable.rs:82-83,173,199; flatten.cpp eval_face has the algebra)
  const uint32_t mode = RTB_MINFO_FACE(minfo), base = mode & 7u;
  if (mode >= FACE_Q) {  // under a RotateY: q = RotateY::hit's test of the OBJECT-space ray against the WORLD-space normal
    float sn, cs;  // the chain's rotation: in the exact record, for a triangle in the spare words of its vertices
    if (type == PT_TRI) {
      sn = __ldg(sc.geom[PT_TRI] + 3 * idx).w;
      cs = __ldg(sc.geom[PT_TRI] + 3 * idx + 1).w;
    } else {
      const double* ex = sc.xtab->exact[type] + (size_t)idx * RTB_EXACT_STRIDE;
      sn = (float)ex[4]; cs = (float)ex[5];
    }
    const bool q = dot(f3(cs * d.x - sn * d.z, d.y, sn * d.x + cs * d.z), s.n) < 0.0f;
    s.front = base == FACE_Q ? q : base == FACE_NOT_Q ? !q : base == FACE_NATURAL ? ff : base == FACE_FLIPPED ? !ff : base == FACE_TRUE;
    if ((mode & FACE_BARE) && !q) s.n = -s.n;  // no Translate outside the RotateY re-oriented the normal
  } else {
    s.front = base == FACE_NATURAL ? ff : base == FACE_FLIPPED ? !ff : base == FACE_TRUE;
  }
  if constexpr (ATTR) {
    s.uv = false;
    if (type == PT_TRI && (minfo >> 31)) surface_attr(sc, idx, s);
  }
  return s;
}

template <bool ATTR = false>
__device__ __forceinline__ void surface_uv(const DevScene& sc, const Surf& s, float& u, float& v) {
  if constexpr (ATTR) {
    if (s.uv) { u = s.tu; v = s.tv; return; }
  }
  const uint32_t type = s.ref >> REF_TYPE_SHIFT, idx = s.ref & REF_INDEX_MASK;
  u = v = 0.f;  // MovingSphere / ConstantMedium leave u,v stale in the reference; defined 0 (SURVEY App. A #17)
  if (type == PT_SPHERE) {  // sphere.rs:32-37, on the OBJECT-space outward normal: a sphere under RotateY gets its
    // world-space normal rotated back (hittable.rs:150-156 maps world -> object; the record keeps that sin / cos)
    const double* ex = sc.xtab->exact[PT_SPHERE] + (size_t)idx * RTB_EXACT_STRIDE;
    const float sn = (float)ex[4], cs = (float)ex[5];
    const float3 on = f3(cs * s.outward.x - sn * s.outward.z, s.outward.y, sn * s.outward.x + cs * s.outward.z);
    const float theta = acosf(fminf(fmaxf(-on.y, -1.f), 1.f));
    const float phi = atan2f(-on.z, on.x) + RTB_PI;
    u = phi / (2.0f * RTB_PI);
    v = theta / RTB_PI;
  } else if (type == PT_QUAD) {
    const float4 w1 = __ldg(sc.geom[PT_QUAD] + 3 * idx + 1), w2 = __ldg(sc.geom[PT_QUAD] + 3 * idx + 2);
    u = dot(xyz(w1), s.p) - w1.w;
    v = dot(xyz(w2), s.p) - w2.w;
  } else if (type == PT_TRI) {
    const float3 v0 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx)), e1 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx + 1)) - v0,
                 e2 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx + 2)) - v0;
    tri_bary(v0, e1, e2, s.p, u, v);
  }
}

// Perlin::noise with the reference's double Hermite smoothing (perlin.rs:26-52,67-85) and turb (perlin.rs:86-98)
__device__ float perlin_noise(const float4* __restrict__ vec, const uint8_t* __restrict__ perm, float3 p) {
  const float fx = floorf(p.x), fy = floorf(p.y), fz = floorf(p.z);
  float u = p.x - fx, v = p.y - fy, w = p.z - fz;
  u = u * u * (3.f - 2.f * u);
  v = v * v * (3.f - 2.f * v);
  w = w * w * (3.f - 2.f * w);
  const int i = (int)fx, j = (int)fy, k = (int)fz;
  const float uu = u * u * (3.f - 2.f * u), vv = v * v * (3.f - 2.f * v), ww = w * w * (3.f - 2.f * w);
  float accum = 0.f;
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b)
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const uint32_t h = perm[(i + a) & 255] ^ perm[256 + ((j + b) & 255)] ^ perm[512 + ((k + c) & 255)];
        const float4 g = __ldg(vec + h);
        const float wgt = (a ? uu : 1.f - uu) * (b ? vv : 1.f - vv) * (c ? ww : 1.f - ww);
        accum += wgt * (g.x * (u - a) + g.y * (v - b) + g.z * (w - c));
      }
  return accum;
}

__device__ float perlin_turb(const float4* __restrict__ vec, const uint8_t* __restrict__ perm, float3 p) {  // perlin.rs:86-98
  float accum = 0.f, weight = 1.f;
  float3 tp = p;
  for (int i = 0; i < 7; ++i) {
    accum += weight * perlin_noise(vec, perm, tp);
    weight *= 0.5f;
    tp = 2.0f * tp;
  }
  return fabsf(accum);
}

template <bool ATTR = false>
__device__ float3 tex_value_slow(const DevScene& sc, uint32_t tex, const Surf& s) {
  DevTexture t = sc.textures[tex];
  if (t.type == RTB_TEX_CHECKER) {  // texture.rs:60-69, on the world-space point
    // (children are Arc<dyn Texture>: a checker of checkers evaluates the same sign at every level; the host bounds the depth)
    const float sines = sinf(10.f * s.p.x) * sinf(10.f * s.p.y) * sinf(10.f * s.p.z);
    for (int level = 0; level < RTB_MAX_CHECKER_DEPTH && t.type == RTB_TEX_CHECKER; ++level) t = sc.textures[sines < 0.f ? t.odd : t.even];
  }
  if (t.type == RTB_TEX_NOISE) {  // texture.rs:90-96
    const float g = 0.5f * (1.0f + sinf(t.scale * s.p.z + 10.f * perlin_turb(sc.perlin_vec + 256u * t.table, sc.perlin_perm + 768u * t.table, s.p)));
    return f3(g, g, g);
  }
  if (t.type == RTB_TEX_IMAGE) {  // texture.rs:118-140: nearest texel, v flipped
    if (t.table >= sc.n_images) return f3(0.f, 1.f, 1.f);
    const DevImage im = sc.images[t.table];
    if (im.data == nullptr) return f3(0.f, 1.f, 1.f);
    float u, v;
    surface_uv<ATTR>(sc, s, u, v);
    u = fminf(fmaxf(u, 0.f), 1.f);
    v = 1.0f - fminf(fmaxf(v, 0.f), 1.f);
    uint32_t i = (uint32_t)(u * (float)im.w), j = (uint32_t)(v * (float)im.h);
    if (i >= im.w) i = im.w - 1;
    if (j >= im.h) j = im.h - 1;
    const uint8_t* px = im.data + ((size_t)j * im.w + i) * 3;
    const float k = 1.0f / 255.0f;
    return f3(k * px[0], k * px[1], k * px[2]);
  }
  return f3(t.r, t.g, t.b);
}

// material word 0 = (type, texture, param, texture type); word 1 = solid albedo (saves the texture fetch)
template <bool ATTR = false>
__device__ __forceinline__ float3 tex_value(const DevScene& sc, const float4 m0, uint32_t mat, const Surf& s) {
  if (__float_as_uint(m0.w) == RTB_TEX_SOLID) return xyz(__ldg(&sc.materials[2 * mat + 1]));
  return tex_value_slow<ATTR>(sc, __float_as_uint(m0.y), s);
}

struct Onb {  // onb.rs:19-42
  float3 u, v, w;
  __device__ __forceinline__ explicit Onb(float3 n) {
    w = unit(n);
    const float3 a = fabsf(w.x) > 0.9f ? f3(0.f, 1.f, 0.f) : f3(1.f, 0.f, 0.f);
    v = unit(cross(w, a));
    u = cross(w, v);
  }
  __device__ __forceinline__ float3 local(float3 a) const { return a.x * u + a.y * v + a.z * w; }
};

// HittableList::pdf_value over the light proxies (hittable_list.rs:73-80; aarect.rs:107-117; sphere.rs:75-84)
__device__ float lights_pdf(const DevScene& sc, float3 o, float3 v) {
  float sum = 0.f;
  const float weight = 1.0f / (float)sc.n_lights;
  for (uint32_t k = 0; k < sc.n_lights; ++k) {
    const DevLight& L = sc.lights[k];
    float pdf = 0.f;
    if (L.type == RTB_LIGHT_XZ_RECT) {
      const float t = (L.p[4] - o.y) * rcp_fast(v.y);
      if (t >= RTB_TMIN && t < INFINITY) {
        const float x = fmaf(t, v.x, o.x), z = fmaf(t, v.z, o.z);
        if (!(x < L.p[0] || x > L.p[1] || z < L.p[2] || z > L.p[3])) {
          const float area = (L.p[1] - L.p[0]) * (L.p[3] - L.p[2]);
          const float vv = dot(v, v);
          const float cosine = fabsf(v.y) * rsqrtf(vv);
          pdf = t * t * vv * rcp_fast(cosine * area);
        }
      }
    } else {
      const float3 c = f3(L.p[0], L.p[1], L.p[2]);
      float t;
      if (sphere_roots(o, v, c, L.p[3], RTB_TMIN, INFINITY, t)) {
        const float3 oc = c - o;
        const float q = L.p[3] * L.p[3] * rcp_fast(dot(oc, oc));
        const float cos_max = sqrt_fast(1.0f - q);
        pdf = (1.0f + cos_max) * rcp_fast(2.0f * RTB_PI * q);  // 1/(2 pi (1-cos)) with 1-cos = q/(1+cos)
      }
    }
    sum += weight * pdf;
  }
  return sum;
}

// HittableList::random (hittable_list.rs:81-84) -> XzRect::random (aarect.rs:118-125) | Sphere::random (sphere.rs:85-90)
__device__ float3 lights_random(const DevScene& sc, float3 o, float pick, float r1, float r2) {
  uint32_t k = (uint32_t)(pick * (float)sc.n_lights);
  if (k >= sc.n_lights) k = sc.n_lights - 1;
  const DevLight& L = sc.lights[k];
  if (L.type == RTB_LIGHT_XZ_RECT)
    return f3(fmaf(L.p[1] - L.p[0], r1, L.p[0]), L.p[4], fmaf(L.p[3] - L.p[2], r2, L.p[2])) - o;
  const float3 dir = f3(L.p[0], L.p[1], L.p[2]) - o;
  const float dist2 = dot(dir, dir);
  const float q = L.p[3] * L.p[3] * rcp_fast(dist2);
  const float cos_max = sqrt_fast(1.0f - q);
  const float z = 1.0f - r2 * (q * rcp_fast(1.0f + cos_max));  // pdf.rs:85: 1 + r2 (cos_max - 1)
  const float phi = 2.0f * RTB_PI * r1;
  const float s = sqrt_fast(fmaxf(0.f, 1.0f - z * z));
  float sn, cs;
  __sincosf(phi, &sn, &cs);
  return Onb(dir).local(f3(cs * s, sn * s, z));
}

__device__ __forceinline__ float3 reflect3(float3 v, float3 n) { return fma3(-2.0f * dot(v, n), n, v); }  // vec3.rs:115-117
__device__ __forceinline__ float3 refract3(float3 uv, float3 n, float ratio) {                               // vec3.rs:246-251
  const float cos_theta = fminf(-dot(uv, n), 1.0f);
  const float3 perp = ratio * fma3(cos_theta, n, uv);
  const float par = -sqrt_fast(fabsf(1.0f - dot(perp, perp)));
  return fma3(par, n, perp);
}

// ---- common shade prologue/epilogue --------------------------------------------------------------------------------
struct PathIO {
  uint32_t slot, pixel, sample, segs;
  float3 o, d, beta, L;
  float time, t;
  uint32_t ref, minfo;
};

__device__ __forceinline__ PathIO load_path(const DevPool& pool, uint32_t slot) {
  PathIO io;
  io.slot = slot;
  const float4 ro = pool.ray[2 * slot], rd = pool.ray[2 * slot + 1], b = pool.st[2 * slot], r = pool.st[2 * slot + 1];
  const float4 h = pool.hit[slot];
  io.o = xyz(ro); io.time = ro.w; io.d = xyz(rd);
  io.beta = xyz(b); io.pixel = __float_as_uint(b.w);
  io.L = xyz(r);
  const uint32_t st = __float_as_uint(r.w);
  io.sample = st >> 8;
  io.segs = (st & 0xFFu) + 1u;  // this hit closes segment number `segs`
  io.t = h.x; io.ref = __float_as_uint(h.y); io.minfo = __float_as_uint(h.z);
  return io;
}

// decide continuation (depth budget main.rs:71-73, Russian roulette), then write back or deposit.
// returns true if the path continues.
__device__ __forceinline__ bool finish_bounce(const DevPool& pool, const DevParams& prm, PathIO& io, bool scattered,
                                              float3 no, float3 nd, float ntime, float rr_xi) {
  bool alive = scattered && (int)io.segs < prm.max_depth;
  if (alive && prm.rr_start > 0 && io.segs >= prm.rr_start) {
    float qv = fmaxf(io.beta.x, fmaxf(io.beta.y, io.beta.z));
    qv = qv < 0.2f ? 0.2f : (qv > 1.0f ? 1.0f : qv);  // survival probability in [0.2, 1]: weights grow by <= 5x
    if (!(rr_xi < qv)) alive = false;
    else io.beta = rcp_fast(qv) * io.beta;
  }
  if (alive) {
    // the slot keeps its class; with octant ordering on, bits 3-5 carry the new ray's direction octant for extend
    if (prm.opt & RTB_OPT_OCTANT_SORT) pool.cls[io.slot] = (uint8_t)(RTB_MINFO_QUEUE(io.minfo) | ray_octant(nd) << 3);
    pool.ray[2 * io.slot] = make_float4(no.x, no.y, no.z, ntime);
    pool.ray[2 * io.slot + 1] = make_float4(nd.x, nd.y, nd.z, 0.f);
    pool.st[2 * io.slot] = make_float4(io.beta.x, io.beta.y, io.beta.z, __uint_as_float(io.pixel));
    pool.st[2 * io.slot + 1] = make_float4(io.L.x, io.L.y, io.L.z, __uint_as_float((io.sample << 8) | io.segs));
  } else {
    deposit(prm, pool.c, io.pixel, io.L);
  }
  return alive;
}

// ---- generate: camera.rs:60-70 get_ray + the jitter of main.rs:752-753 ---------------------------------------------
__device__ __forceinline__ void camera_ray(const DevCamera& cam, const DevParams& prm, uint32_t pixel, uint32_t sample,
                                           float3& o, float3& d, float& time) {
  const uint32_t row = pixel / prm.width, col = pixel - row * prm.width;
  const uint32_t j = prm.height - 1 - row;  // scanline j is stored at image row H-1-j, main.rs:733
  const float4 u0 = philox_u(pixel, sample, BLK_CAMERA0, 0, prm.seed);
  const float s = ((float)col + u0.x) * prm.inv_wm1;  // main.rs:752-753: (i + xi) / (W - 1), (j + xi) / (H - 1)
  const float t = ((float)j + u0.y) * prm.inv_hm1;
  o = ld3(cam.origin);
  d = fma3(s, ld3(cam.horizontal), fma3(t, ld3(cam.vertical), ld3(cam.lmo)));
  if (cam.lens_radius > 0.0f) {  // random_in_unit_disk (vec3.rs:101-113) in closed form; a pinhole's offset is exactly 0
    const float rr = cam.lens_radius * sqrt_fast(u0.z);
    float sn, cs;
    __sincosf(2.0f * RTB_PI * u0.w, &sn, &cs);
    const float3 off = (rr * cs) * ld3(cam.u) + (rr * sn) * ld3(cam.v);
    o = o + off;
    d = d - off;
  }
  time = cam.time0;
  if (cam.time1 != cam.time0)  // camera.rs:68; the second Philox block is only drawn when the shutter is open
    time = fmaf(cam.time1 - cam.time0, philox_u(pixel, sample, BLK_CAMERA1, 0, prm.seed).x, cam.time0);
}

// start camera path number `path` in `slot`.  Sample-major order: all pixels (8x4 tiles) of sample k, then k+1, so
// consecutive path numbers are neighbouring pixels.
__device__ __forceinline__ void start_path(const DevPool& pool, const DevParams& prm, const DevCamera& cam, uint32_t slot,
                                           unsigned long long path) {
  const uint32_t npix = prm.width * prm.height;
  // path / npix without a 64-bit integer division: double reciprocal + one correction step (exact below 2^52)
  uint32_t s_local = (uint32_t)((double)path * prm.inv_npix);
  if ((unsigned long long)s_local * npix > path) --s_local;
  else if ((unsigned long long)(s_local + 1u) * npix <= path) ++s_local;
  const uint32_t pixel = __ldg(prm.pix_order + (uint32_t)(path - (unsigned long long)s_local * npix));
  const uint32_t sample = prm.sample_offset + s_local;
  float3 o, d;
  float time;
  camera_ray(cam, prm, pixel, sample, o, d, time);
  if (prm.opt & RTB_OPT_OCTANT_SORT) pool.cls[slot] = (uint8_t)(CLS_NEW | ray_octant(d) << 3);
  pool.ray[2 * slot] = make_float4(o.x, o.y, o.z, time);
  pool.ray[2 * slot + 1] = make_float4(d.x, d.y, d.z, 0.f);
  pool.st[2 * slot] = make_float4(1.f, 1.f, 1.f, __uint_as_float(pixel));
  pool.st[2 * slot + 1] = make_float4(0.f, 0.f, 0.f, __uint_as_float(sample << 8));
}

// ---- the shade loop: warp-local compaction of one chunk of slots, shading, in-place restart ---------------------------
// One warp owns one chunk of RTB_CHUNK consecutive slots at a time.  Lane l reads the class bytes of slots 8l..8l+7 (one
// coalesced 256-byte read per warp), the slots of class QID are compacted into a per-warp shared-memory list with a
// warp scan, and the list is processed 32 entries at a time.  `body(slot)` shades one path and returns true if it
// continues (its next ray is in the pool).  A finished path's slot is restarted immediately with the chunk's next path
// number (fused regeneration); when the chunk's numbers are used up the slot is marked CLS_DEAD.
// (An L2 prefetch of the next path's state sectors was measured and removed: it doubled the request count of a
// request-bound kernel, profiles/r2_ab.md §2.)
#define RTB_SHADE_WARPS (RTB_SHADE_THREADS / 32)

template <uint32_t QID, uint32_t QID2 = QID, class Body>
__device__ __forceinline__ void shade_loop(const DevPool& pool, const DevParams& prm, const DevCamera& cam, Body&& body) {
  __shared__ uint8_t s_list[RTB_SHADE_WARPS][RTB_CHUNK];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t lt_mask = (1u << lane) - 1u;
  uint8_t* list = s_list[warp];
  const unsigned long long total_paths = pool.c->total_paths;
  const uint32_t n_warps = gridDim.x * RTB_SHADE_WARPS;
  for (uint32_t chunk = blockIdx.x * RTB_SHADE_WARPS + warp; chunk < pool.n_chunks; chunk += n_warps) {
    const uint32_t base = chunk * RTB_CHUNK;
    const uint2 cw = *reinterpret_cast<const uint2*>(pool.cls + base + 8u * lane);
    uint32_t total = append_class(cw, QID, list, 0u, lane);
    if (QID2 != QID) total = append_class(cw, QID2, list, total, lane);  // a second (small) class shares the kernel
    if (total == 0) continue;
    __syncwarp();
    unsigned long long m_cur = pool.cursor[chunk];
    const unsigned long long m_first = m_cur;
    for (uint32_t r = 0; r < total; r += 32) {
      const bool valid = r + lane < total;
      const uint32_t slot = base + (valid ? list[r + lane] : 0u);
      bool alive = false;
      if (valid) alive = body(slot);
      const bool dead = valid && !alive;
      const uint32_t dmask = __ballot_sync(0xffffffffu, dead);
      if (dead) {
        const unsigned long long path = chunk_path(m_cur + __popc(dmask & lt_mask), chunk, pool.n_chunks);
        if (path < total_paths) start_path(pool, prm, cam, slot, path);
        else pool.cls[slot] = (uint8_t)CLS_DEAD;
      }
      m_cur += __popc(dmask);
    }
    if (lane == 0 && m_cur != m_first) pool.cursor[chunk] = m_cur;
    __syncwarp();  // the list is rewritten for the next chunk
  }
}

// miss -> background (main.rs:74-76); DiffuseLight -> emitted iff front_face, no scatter (material.rs:184-190, main.rs:85-87)
template <bool ATTR>
__global__ void __launch_bounds__(RTB_SHADE_THREADS, RTB_SHADE_MIN_BLOCKS) k_shade_terminal(DevScene sc, DevPool pool, DevParams prm, DevCamera cam) {
  shade_loop<Q_TERMINAL>(pool, prm, cam, [&](uint32_t slot) {
    // a miss needs only the throughput/radiance sector; the ray is fetched for emitters alone
    const float4 h = pool.hit[slot], b = pool.st[2 * slot], r = pool.st[2 * slot + 1];
    float3 L = xyz(r);
    const float3 beta = xyz(b);
    const uint32_t ref = __float_as_uint(h.y);
    if (ref == REF_MISS) {
      L = L + beta * f3(prm.bg[0], prm.bg[1], prm.bg[2]);
    } else {
      const float4 ro = pool.ray[2 * slot], rd = pool.ray[2 * slot + 1];
      const Surf s = surface_at<ATTR>(sc, ref, __float_as_uint(h.z), xyz(ro), xyz(rd), ro.w, h.x);
      const float4 m = __ldg(&sc.materials[2 * s.mat]);
      if (__float_as_uint(m.x) == RTB_MAT_DIFFUSE_LIGHT && s.front) L = L + beta * tex_value<ATTR>(sc, m, s.mat, s);
    }
    deposit(prm, pool.c, __float_as_uint(b.w), L);
    return false;
  });
}
// (instantiated here: the ATTR = false kernels keep their place, and so their code, in the module)
template __global__ void k_shade_terminal<false>(DevScene, DevPool, DevParams, DevCamera);

// Lambertian (material.rs:48-71) / Isotropic (SURVEY §8a M6) through the mixture pdf of main.rs:94-138
template <bool ISO, bool ATTR>
__device__ __forceinline__ bool shade_diffuse(const DevScene& sc, const DevPool& pool, const DevParams& prm, uint32_t slot) {
  PathIO io = load_path(pool, slot);
  const Surf s = surface_at<ATTR>(sc, io.ref, io.minfo, io.o, io.d, io.time, io.t);
  const float4 m = __ldg(&sc.materials[2 * s.mat]);
  const float3 atten = tex_value<ATTR>(sc, m, s.mat, s);
  const float4 us = philox_u(io.pixel, io.sample, BLK_SCATTER, io.segs, prm.seed);
  const bool have_lights = sc.n_lights > 0;
  float3 dir;
  if (have_lights && us.x < 0.5f) {  // MixturePdf::generate, pdf.rs:73-79
    dir = lights_random(sc, s.p, us.y, us.z, us.w);
  } else if (ISO) {
    const float z = 1.0f - 2.0f * us.z, phi = 2.0f * RTB_PI * us.w;
    const float r = sqrt_fast(fmaxf(0.f, 1.0f - z * z));
    float sn, cs;
    __sincosf(phi, &sn, &cs);
    dir = f3(r * cs, r * sn, z);
  } else {  // random_cosine_direction vec3.rs:253-262 (r1 = us.z, r2 = us.w) in the ONB of the normal, pdf.rs:32-34
    const float phi = 2.0f * RTB_PI * us.z, sq = sqrt_fast(us.w);
    float sn, cs;
    __sincosf(phi, &sn, &cs);
    dir = Onb(s.n).local(f3(cs * sq, sn * sq, sqrt_fast(1.0f - us.w)));
  }
  float mat_pdf, spdf;
  if (ISO) {
    mat_pdf = spdf = 1.0f / (4.0f * RTB_PI);
  } else {
    const float cosine = dot(unit(dir), unit(s.n));  // CosinePdf::value pdf.rs:24-31 ; scattering_pdf material.rs:64-71
    mat_pdf = cosine <= 0.f ? 0.f : cosine * (1.0f / RTB_PI);
    spdf = mat_pdf;
  }
  const float pdf_val = have_lights ? 0.5f * lights_pdf(sc, s.p, dir) + 0.5f * mat_pdf : mat_pdf;  // pdf.rs:70-72
  const bool scattered = spdf > 0.f;  // zero-weight continuation culled (SURVEY App. A #10)
  // without lights the mixture is the material pdf itself: the weight is exactly 1 (white-furnace test relies on it)
  if (scattered) io.beta = have_lights ? io.beta * atten * (spdf * rcp_fast(pdf_val)) : io.beta * atten;
  float rr = 0.f;
  if (prm.rr_start > 0 && io.segs >= prm.rr_start) rr = u01(philox4(io.pixel, io.sample, BLK_AUX, io.segs, prm.seed).x);
  return finish_bounce(pool, prm, io, scattered, s.p, dir, io.time, rr);
}

template <bool ATTR>
__global__ void __launch_bounds__(RTB_SHADE_THREADS, RTB_SHADE_MIN_BLOCKS) k_shade_lambert(DevScene sc, DevPool pool, DevParams prm, DevCamera cam) {
  shade_loop<Q_LAMBERT>(pool, prm, cam, [&](uint32_t slot) { return shade_diffuse<false, ATTR>(sc, pool, prm, slot); });
}
template __global__ void k_shade_lambert<false>(DevScene, DevPool, DevParams, DevCamera);

template <bool ATTR>
__global__ void __launch_bounds__(RTB_SHADE_THREADS, RTB_SHADE_MIN_BLOCKS) k_shade_isotropic(DevScene sc, DevPool pool, DevParams prm, DevCamera cam) {
  shade_loop<Q_ISOTROPIC>(pool, prm, cam, [&](uint32_t slot) { return shade_diffuse<true, ATTR>(sc, pool, prm, slot); });
}
template __global__ void k_shade_isotropic<false>(DevScene, DevPool, DevParams, DevCamera);

// The two specular materials share one kernel (their classes are small: 10 % and 7 % of C1's hits; as separate kernels
// each paid a launch, a scan of the class bytes and a tail, profiles/r2e_ncu_summary.md).  A chunk's metal slots come
// first in the warp's list, then its glass slots, so only one round per chunk mixes the two branches.
//   Metal::scatter, material.rs:95-107: reflect(unit(d), n) + fuzz * (uniform ball); specular; ray time reset to 0
//   Dielectric::scatter, material.rs:123-155 (+ reflectance :118-122, refract vec3.rs:246-251)
template <bool ATTR>
__global__ void __launch_bounds__(RTB_SHADE_THREADS, RTB_SHADE_MIN_BLOCKS) k_shade_specular(DevScene sc, DevPool pool, DevParams prm, DevCamera cam) {
  shade_loop<Q_METAL, Q_DIELECTRIC>(pool, prm, cam, [&](uint32_t slot) {
      PathIO io = load_path(pool, slot);
      const Surf s = surface_at<ATTR>(sc, io.ref, io.minfo, io.o, io.d, io.time, io.t);
      const float4 m = __ldg(&sc.materials[2 * s.mat]);
      const float3 ud = unit(io.d);
      const float4 ua = philox_u(io.pixel, io.sample, BLK_AUX, io.segs, prm.seed);
      float3 dir;
      float ntime = io.time;
      if (__float_as_uint(m.x) == RTB_MAT_METAL) {
        const float fuzz = fminf(m.z, 1.0f);
        dir = reflect3(ud, s.n);
        if (fuzz > 0.f) {  // random_in_unit_sphere (vec3.rs:78-86) in closed form: uniform direction * cbrt(xi)
          const float z = 1.0f - 2.0f * ua.y, phi = 2.0f * RTB_PI * ua.z, rad = cbrtf(ua.w);
          const float r = sqrt_fast(fmaxf(0.f, 1.0f - z * z));
          float sn, cs;
          __sincosf(phi, &sn, &cs);
          dir = fma3(fuzz * rad, f3(r * cs, r * sn, z), dir);
        }
        io.beta = io.beta * tex_value<ATTR>(sc, m, s.mat, s);
        ntime = 0.0f;  // material.rs:101
      } else {
        const float ir = m.z;
        const float ratio = s.front ? rcp_fast(ir) : ir;
        const float cos_theta = fminf(-dot(ud, s.n), 1.0f);
        const float sin_theta = sqrt_fast(fmaxf(0.f, 1.0f - cos_theta * cos_theta));
        const bool cannot_refract = ratio * sin_theta > 1.0f;
        float r0 = (1.0f - ratio) * rcp_fast(1.0f + ratio);
        r0 *= r0;
        const float om = 1.0f - cos_theta;
        const float reflectance = r0 + (1.0f - r0) * (om * om) * (om * om) * om;
        dir = (cannot_refract || reflectance > ua.y) ? reflect3(ud, s.n) : refract3(ud, s.n, ratio);
      }
      return finish_bounce(pool, prm, io, true, s.p, dir, ntime, ua.x);
  });
}
template __global__ void k_shade_specular<false>(DevScene, DevPool, DevParams, DevCamera);

// ---- generate: initial fill — every chunk starts its first paths (afterwards slots are restarted inside shade_loop) ----
__global__ void __launch_bounds__(RTB_SHADE_THREADS) k_generate(DevPool pool, DevParams prm, DevCamera cam) {
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const unsigned long long total = pool.c->total_paths;
  const uint32_t n_warps = gridDim.x * RTB_SHADE_WARPS;
  for (uint32_t chunk = blockIdx.x * RTB_SHADE_WARPS + warp; chunk < pool.n_chunks; chunk += n_warps) {
    const uint32_t base = chunk * RTB_CHUNK;
    const uint32_t cnt = min(RTB_CHUNK, pool.n - base);
    for (uint32_t m = lane; m < cnt; m += 32) {
      const unsigned long long path = chunk_path(m, chunk, pool.n_chunks);
      if (path < total) {
        start_path(pool, prm, cam, base + m, path);
        if (!(prm.opt & RTB_OPT_OCTANT_SORT)) pool.cls[base + m] = (uint8_t)CLS_NEW;
      }
    }
    if (lane == 0) pool.cursor[chunk] = cnt;
  }
}

__global__ void k_init_pool(DevPool pool, unsigned long long total_paths) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < pool.n_chunks * RTB_CHUNK) pool.cls[i] = (uint8_t)CLS_DEAD;
  if (i < pool.n_chunks) pool.cursor[i] = 0ull;
  if (i == 0) {
    DevCounters* c = pool.c;
    c->iter_rays = c->last_rays = 0;
    c->iter = 0;
    c->ext_cursor = 0;
    c->redo_count[0] = c->redo_count[1] = 0;
    c->redo_sel = 0;
    c->iter_fixed = c->ext_ticket = 0;
    c->redone = c->refined = 0;
    c->total_paths = total_paths;
    c->segments = c->rejected = 0;
    c->nodes_visited = c->prims_tested = 0;
    for (uint32_t t = 0; t < PT_COUNT; ++t) c->prims_tested_type[t] = 0;
  }
}

// ---- the exact pass: runs right after every extend launch, before the shade kernels (and after the probes' single launch) ---
// Processes the queue that launch filled and empties it.  On its own stream position it overlaps the extend / shade kernels
// of the other wavefront lanes; what it costs is latency on this lane only (one queue entry = one thread).
#define RTB_FIXUP_THREADS 128
__global__ void __launch_bounds__(RTB_FIXUP_THREADS) k_fixup(DevScene sc, DevPool pool, DevParams prm) {
  DevCounters* c = pool.c;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warps = RTB_FIXUP_THREADS / 32u;
  uint2 done = fix_prologue(sc, pool, prm, blockIdx.x * warps + (threadIdx.x >> 5), gridDim.x * warps, lane);
  if (c->redo_count[0]) {  // (uniform) one pair of atomics per warp, not per entry
    done.x = __reduce_add_sync(0xffffffffu, done.x);
    done.y = __reduce_add_sync(0xffffffffu, done.y);
    if (lane == 0 && done.x) {
      atomicAdd(&c->redone, (unsigned long long)done.x);
      if (done.y) atomicAdd(&c->refined, (unsigned long long)done.y);
    }
  }
  __shared__ bool last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(&c->ext_ticket, 1u) == gridDim.x - 1u;
  }
  __syncthreads();
  if (last && threadIdx.x == 0) {  // the last CTA rotates the iteration counters (what a one-thread kernel did in round 1)
    c->segments += c->iter_rays;
    c->last_rays = c->iter_rays;
    c->iter_rays = 0;
    c->ext_cursor = 0;
    c->redo_count[0] = 0;
    c->ext_ticket = 0;
    c->iter += 1;
  }
}

// the very first "iteration" of a render has no extend launch yet: only the counters rotate
__global__ void k_rotate(DevPool pool) {
  DevCounters* c = pool.c;
  c->last_rays = 1;  // paths were just started
  c->iter += 1;
}

// ---- write_color, main.rs:141-169 ----------------------------------------------------------------------------------
__global__ void k_finalize(const float4* __restrict__ accum, uint8_t* __restrict__ rgb, uint32_t npix, float inv_spp) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  const float4 a = accum[i];
  float ch[3] = {a.x, a.y, a.z};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float v = ch[k];
    if (v != v) v = 0.f;
    v = sqrtf(inv_spp * v);
    v = v < 0.f ? 0.f : (v > 0.999f ? 0.999f : v);
    rgb[3 * (size_t)i + k] = (uint8_t)(256.0f * v);
  }
}

// ---- parity probes: the PRODUCTION kernels (extend + k_fixup) run over a pool filled with the caller's rays ---------
__global__ void k_probe_fill(DevPool pool, const float* __restrict__ org, const float* __restrict__ dir,
                             const float* __restrict__ time, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= pool.n_chunks * RTB_CHUNK) return;
  if (i < n) {
    pool.ray[2 * i] = make_float4(org[3 * i], org[3 * i + 1], org[3 * i + 2], time ? time[i] : 0.f);
    pool.ray[2 * i + 1] = make_float4(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2], 0.f);
    pool.st[2 * i] = make_float4(1.f, 1.f, 1.f, 0.f);
    pool.st[2 * i + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
    pool.cls[i] = (uint8_t)CLS_NEW;
  } else {
    pool.cls[i] = (uint8_t)CLS_DEAD;
  }
}
__global__ void k_probe_collect(DevScene sc, DevPool pool, uint32_t n, uint32_t* __restrict__ id_out, float* __restrict__ t_out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 h = pool.hit[i];
  const uint32_t ref = __float_as_uint(h.y);
  id_out[i] = ref == REF_MISS ? RTB_NONE : ref_gid(sc, ref);
  t_out[i] = h.x;
}

// ---- denoiser guide buffers (rtb_render_aov): the first segment of every render sample, traced by the production extend +
// k_fixup over a pool these two kernels fill and read ---------------------------------------------------------------------
// slot i holds path number first_path + i: start_path() is the render's own path start, so the ray is that sample's first ray
__global__ void k_aov_fill(DevPool pool, DevParams prm, DevCamera cam, unsigned long long first_path, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= pool.n_chunks * RTB_CHUNK) return;
  if (i < n) {
    start_path(pool, prm, cam, i, first_path + i);
    if (!(prm.opt & RTB_OPT_OCTANT_SORT)) pool.cls[i] = (uint8_t)CLS_NEW;
  } else {
    pool.cls[i] = (uint8_t)CLS_DEAD;
  }
}

// per-sample (albedo, coverage) and (shading normal, depth) of the hit record, summed into aov[2 pixel], aov[2 pixel + 1]
template <bool ATTR>
__global__ void __launch_bounds__(RTB_SHADE_THREADS) k_aov_collect(DevScene sc, DevPool pool, DevParams prm, float4* aov,
                                                                  uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 h = pool.hit[i];
  const uint32_t pixel = __float_as_uint(pool.st[2 * i].w), ref = __float_as_uint(h.y);
  float3 albedo = f3(prm.bg[0], prm.bg[1], prm.bg[2]), n3 = f3(0.f, 0.f, 0.f);
  float cover = 0.f, depth = 0.f;
  if (ref != REF_MISS) {
    const float4 ro = pool.ray[2 * i], rd = pool.ray[2 * i + 1];
    const Surf s = surface_at<ATTR>(sc, ref, __float_as_uint(h.z), xyz(ro), xyz(rd), ro.w, h.x);
    const float4 m = __ldg(&sc.materials[2 * s.mat]);
    const uint32_t type = __float_as_uint(m.x);
    if (type == RTB_MAT_DIELECTRIC) albedo = f3(1.f, 1.f, 1.f);
    else if (type == RTB_MAT_DIFFUSE_LIGHT && !s.front) albedo = f3(0.f, 0.f, 0.f);
    else albedo = tex_value<ATTR>(sc, m, s.mat, s);
    if ((ref >> REF_TYPE_SHIFT) != PT_MEDIUM) n3 = s.n;
    cover = 1.f;
    depth = h.x * sqrtf(dot(xyz(rd), xyz(rd)));
  }
  if (!(isfinite(albedo.x) && isfinite(albedo.y) && isfinite(albedo.z) && isfinite(n3.x) && isfinite(n3.y) &&
        isfinite(n3.z) && isfinite(depth))) {  // deposit()'s policy: a non-finite sample is dropped and counted
    atomicAdd(&pool.c->rejected, 1ull);
    return;
  }
  albedo = f3(__saturatef(albedo.x), __saturatef(albedo.y), __saturatef(albedo.z));
  red_add_v4(aov + 2 * (size_t)pixel, albedo.x, albedo.y, albedo.z, cover);
  red_add_v4(aov + 2 * (size_t)pixel + 1, n3.x, n3.y, n3.z, depth);
}
template __global__ void k_aov_collect<false>(DevScene, DevPool, DevParams, float4*, uint32_t);

// pixel-centre primary rays, generated in f64 like the reference's camera (camera.rs:60-70) and rounded once
__global__ void k_primary_rays(DevCameraF64 cam, uint32_t W, uint32_t H, float* __restrict__ org, float* __restrict__ dir,
                               float* __restrict__ time) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= W * H) return;
  const uint32_t row = i / W, col = i - row * W, j = H - 1 - row;
  const double s = ((double)col + 0.5) / (double)(W - 1), t = ((double)j + 0.5) / (double)(H - 1);
  for (int a = 0; a < 3; ++a) {
    org[3 * i + a] = (float)cam.origin[a];
    dir[3 * i + a] = (float)(cam.llc[a] + s * cam.horizontal[a] + t * cam.vertical[a] - cam.origin[a]);
  }
  time[i] = (float)cam.time0;
}

// ---- tier U2: the device functions themselves, evaluated on known-answer inputs (tests/test_gpu_kat.py) ---------------
// in / out are raw 32-bit words (floats by bit pattern, integers as they are); one thread per item.
__global__ void k_kat(DevScene sc, DevCamera cam, DevParams prm, uint32_t op, const uint32_t* __restrict__ in, uint32_t n,
                      uint32_t in_stride, uint32_t* __restrict__ out, uint32_t out_stride) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t* a = in + (size_t)i * in_stride;
  uint32_t* o = out + (size_t)i * out_stride;
  auto F = [&](uint32_t k) { return __uint_as_float(a[k]); };
  auto V = [&](uint32_t k) { return f3(__uint_as_float(a[k]), __uint_as_float(a[k + 1]), __uint_as_float(a[k + 2])); };
  auto put = [&](uint32_t k, float v) { o[k] = __float_as_uint(v); };
  auto put3 = [&](uint32_t k, float3 v) { put(k, v.x); put(k + 1, v.y); put(k + 2, v.z); };
  switch (op) {
    case RTB_KAT_PHILOX: {  // (pixel, sample, block, bounce, seed) -> 4 words
      const uint4 r = philox4(a[0], a[1], a[2], a[3], a[4]);
      o[0] = r.x; o[1] = r.y; o[2] = r.z; o[3] = r.w;
      break;
    }
    case RTB_KAT_SPHERE: {  // (c, r, o, d, tmin, tmax) -> (status, t, e): the f32 sphere test with its error bound
      float t = 0.f, e = 0.f;
      bool coarse = false;
      const int st = sphere_fast(V(4), V(7), V(0), F(3), F(10), F(11), t, e, coarse);
      o[0] = (uint32_t)st | (coarse ? 16u : 0u); put(1, t); put(2, e);
      break;
    }
    case RTB_KAT_SPHERE_F64: {  // same inputs -> (status, t): the Newton-refined f64 form used for "global" spheres
      float t = 0.f;
      const int st = sphere_roots_f64(V(4), V(7), V(0), F(3), F(10), t);
      o[0] = (uint32_t)st; put(1, t);
      break;
    }
    case RTB_KAT_LIGHTS_PDF: put(0, lights_pdf(sc, V(0), V(3))); break;                      // (o, v) -> pdf over sc.lights
    case RTB_KAT_LIGHTS_RANDOM: put3(0, lights_random(sc, V(0), F(3), F(4), F(5))); break;   // (o, pick, r1, r2) -> direction
    case RTB_KAT_PERLIN_NOISE: put(0, perlin_noise(sc.perlin_vec + 256u * a[0], sc.perlin_perm + 768u * a[0], V(1))); break;  // (table, p)
    case RTB_KAT_PERLIN_TURB: put(0, perlin_turb(sc.perlin_vec + 256u * a[0], sc.perlin_perm + 768u * a[0], V(1))); break;
    case RTB_KAT_Q2F: put(0, q2f(a[0], sc.prmt_magic, 0x7044u | ((a[1] & 3u) << 8))); break;  // (plane word, byte) -> 128 + q
    case RTB_KAT_ONB: { const Onb b(V(0)); put3(0, b.u); put3(3, b.v); put3(6, b.w); break; }
    case RTB_KAT_REFLECT: put3(0, reflect3(V(0), V(3))); break;
    case RTB_KAT_REFRACT: put3(0, refract3(V(0), V(3), F(6))); break;
    case RTB_KAT_CAMERA_RAY: {  // (pixel, sample) -> (o, d, time) of camera_ray(), drawn from the path's own Philox blocks
      float3 ro, rd;
      float tm;
      camera_ray(cam, prm, a[0], a[1], ro, rd, tm);
      put3(0, ro); put3(3, rd); put(6, tm);
      break;
    }
    case RTB_KAT_MEDIA: {  // (o, d, t_max) -> (hit, t, medium index) of intersect_media() at xi = 0.5
      Closest best{F(6), F(6), REF_MISS};
      intersect_media(sc, V(0), V(3), RTB_TMIN, best, 0, 0, 0, 0, false);
      o[0] = best.ref != REF_MISS ? 1u : 0u; put(1, best.t); o[2] = best.ref & REF_INDEX_MASK;
      break;
    }
    case RTB_KAT_TEXTURE: {  // (texture id, p, outward normal of a unit sphere at the origin) -> rgb of tex_value_slow()
      Surf s;
      s.p = V(1); s.outward = s.n = V(4); s.front = true; s.mat = 0; s.ref = ((uint32_t)PT_SPHERE << REF_TYPE_SHIFT) | a[7];
      put3(0, tex_value_slow(sc, a[0], s));
      break;
    }
    case RTB_KAT_EXACT: {  // (ref, o, d, time) -> exact_hit() as (hi word, lo word) of the f64 distance (-1: miss)
      const double t = exact_hit(sc.xtab, a[0], V(1), V(4), F(7));
      const unsigned long long b = (unsigned long long)__double_as_longlong(t);
      o[0] = (uint32_t)(b >> 32); o[1] = (uint32_t)b;
      break;
    }
    default: break;
  }
}

// ---- bandwidth microbenchmarks: the physical denominators of the roofline (bench.py, profiles/) ------------------------
// Read-only 128-bit loads (ld.global.nc, the instruction the node / primitive fetches use) streaming a buffer `reps` times:
// a 48 MB buffer stays in the 126 MB L2 (L2 read bandwidth), a 2 GB one does not (HBM read bandwidth).
__global__ void __launch_bounds__(256) k_bw_global(const uint4* __restrict__ p, size_t n_vec, uint32_t reps, uint4* __restrict__ sink) {
  uint4 acc = make_uint4(0u, 0u, 0u, 0u);
  const size_t stride = (size_t)gridDim.x * blockDim.x, tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  // every repetition an SM reads a DIFFERENT slice of the buffer (rotated by a fraction of it), so its 256 KB L1 cannot
  // serve the re-reads: with a fixed assignment each SM's 1/148 of a 48 MB buffer would partly live in L1
  const size_t rot = (n_vec / 37) | 1;
  for (uint32_t r = 0; r < reps; ++r) {
    size_t i = (tid + (size_t)r * rot) % n_vec;
    for (size_t k = tid; k < n_vec; k += stride) {
      const uint4 v = __ldg(p + i);
      acc.x ^= v.x; acc.y ^= v.y; acc.z ^= v.z; acc.w ^= v.w;
      i += stride;
      if (i >= n_vec) i -= n_vec;
    }
  }
  if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x12345679u) sink[0] = acc;  // keeps the loads alive; practically never true
}
// 128-bit shared-memory loads at conflict-free addresses (how the node stage is read): bytes = threads x reps x 16.
// (volatile asm: the addresses repeat, a plain load would be hoisted out of the loop)
__global__ void __launch_bounds__(256) k_bw_shared(uint32_t reps, uint4* __restrict__ sink) {
  extern __shared__ uint4 sm[];
  const uint32_t n = 2048;  // 32 KB
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) sm[i] = make_uint4(i, i * 3u, i * 5u, i * 7u);
  __syncthreads();
  uint4 acc = make_uint4(0u, 0u, 0u, 0u);
  const uint32_t base = (uint32_t)__cvta_generic_to_shared(sm);
  uint32_t k = threadIdx.x;
#pragma unroll 8
  for (uint32_t r = 0; r < reps; ++r) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(base + k * 16u));
    acc.x ^= v.x; acc.y ^= v.y; acc.z ^= v.z; acc.w ^= v.w;
    k = (k + 256u) & (n - 1u);
  }
  if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x12345679u) sink[0] = acc;
}

#ifdef RTB_CHECKED
int read_check_failures(unsigned int* out8) {
  return (int)cudaMemcpyFromSymbol(out8, g_rtb_check_fail, sizeof(unsigned int) * 8);
}
#else
int read_check_failures(unsigned int* out8) {
  for (int i = 0; i < 8; ++i) out8[i] = 0xFFFFFFFFu;  // not a checked build
  return 0;
}
#endif

// ================================================= launchers ========================================================
static inline uint32_t cdiv(uint32_t a, uint32_t b) { return (a + b - 1) / b; }

void launch_init_pool(const DevPool& pool, unsigned long long total_paths, cudaStream_t st) {
  k_init_pool<<<cdiv(pool.n_chunks * RTB_CHUNK, 256), 256, 0, st>>>(pool, total_paths);
}
void launch_generate(const LaunchCfg& lc, const DevPool& pool, const DevParams& prm, const DevCamera& cam, cudaStream_t st) {
  k_generate<<<lc.shade_grid, RTB_SHADE_THREADS, 0, st>>>(pool, prm, cam);
}
void launch_fixup(const LaunchCfg& lc, const DevScene& sc, const DevPool& pool, const DevParams& prm, cudaStream_t st) {
  k_fixup<<<lc.fixup_grid, RTB_FIXUP_THREADS, 0, st>>>(sc, pool, prm);
}
void launch_rotate(const DevPool& pool, cudaStream_t st) { k_rotate<<<1, 1, 0, st>>>(pool); }
void launch_extend(const LaunchCfg& lc, const DevScene& sc, const DevPool& pool, const DevParams& prm, bool count,
                   cudaStream_t st) {
  // one-ray-per-thread wins on small trees (all lanes start at the root together); dynamic fetch wins on deep trees
  // where the number of node visits per ray varies widely (measured: profiles/r1_ab_extend.md)
  if (lc.mode == EXTEND_WQ) {
    if (count) k_extend_wq<true><<<lc.extend_grid, RTB_EXTEND_THREADS, lc.extend_smem, st>>>(sc, pool, prm, lc.n_snodes);
    else k_extend_wq<false><<<lc.extend_grid, RTB_EXTEND_THREADS, lc.extend_smem, st>>>(sc, pool, prm, lc.n_snodes);
    return;
  }
  if (lc.mode == EXTEND_STATIC) {
    const bool sort = (prm.opt & RTB_OPT_OCTANT_SORT) != 0u;  // (the shade kernels write the octant bits under the same flag)
    if (count) {
      if (sort) k_extend_static<true, false, true><<<lc.extend_grid, RTB_EXTEND_THREADS, lc.extend_smem, st>>>(sc, pool, prm, lc.n_snodes);
      else k_extend_static<true, false, false><<<lc.extend_grid, RTB_EXTEND_THREADS, lc.extend_smem, st>>>(sc, pool, prm, lc.n_snodes);
    } else if (lc.all_staged && lc.sphere_smem) {
      const uint32_t smem = lc.extend_smem + lc.sphere_smem;
      if (sort) k_extend_static<false, true, true, true><<<lc.extend_grid, RTB_EXTEND_THREADS, smem, st>>>(sc, pool, prm, lc.n_snodes);
      else k_extend_static<false, true, false, true><<<lc.extend_grid, RTB_EXTEND_THREADS, smem, st>>>(sc, pool, prm, lc.n_snodes);
    } else if (lc.all_staged) {
      if (sort) k_extend_static<false, true, true><<<lc.extend_grid, RTB_EXTEND_THREADS, lc.extend_smem, st>>>(sc, pool, prm, lc.n_snodes);
      else k_extend_static<false, true, false><<<lc.extend_grid, RTB_EXTEND_THREADS, lc.extend_smem, st>>>(sc, pool, prm, lc.n_snodes);
    } else {
      if (sort) k_extend_static<false, false, true><<<lc.extend_grid, RTB_EXTEND_THREADS, lc.extend_smem, st>>>(sc, pool, prm, lc.n_snodes);
      else k_extend_static<false, false, false><<<lc.extend_grid, RTB_EXTEND_THREADS, lc.extend_smem, st>>>(sc, pool, prm, lc.n_snodes);
    }
    return;
  }
  if (count) k_extend<true><<<lc.extend_grid, RTB_EXTEND_THREADS, lc.extend_smem, st>>>(sc, pool, prm, lc.n_snodes);
  else k_extend<false><<<lc.extend_grid, RTB_EXTEND_THREADS, lc.extend_smem, st>>>(sc, pool, prm, lc.n_snodes);
}
// The per-material kernels of one iteration run back to back on the lane's stream; they touch disjoint slots (each
// slot has exactly one class per iteration) and each chunk's path cursor is updated by one warp per kernel.
template <bool ATTR>
static void launch_shade_kernels(const LaunchCfg& lc, const DevScene& sc, const DevPool& pool, const DevParams& prm,
                                 const DevCamera& cam, uint32_t present, cudaStream_t st) {
  k_shade_terminal<ATTR><<<lc.shade_grid, RTB_SHADE_THREADS, 0, st>>>(sc, pool, prm, cam);
  if (present & (1u << RTB_MAT_LAMBERTIAN)) k_shade_lambert<ATTR><<<lc.shade_grid, RTB_SHADE_THREADS, 0, st>>>(sc, pool, prm, cam);
  if (present & ((1u << RTB_MAT_METAL) | (1u << RTB_MAT_DIELECTRIC)))
    k_shade_specular<ATTR><<<lc.shade_grid, RTB_SHADE_THREADS, 0, st>>>(sc, pool, prm, cam);
  if (present & (1u << RTB_MAT_ISOTROPIC)) k_shade_isotropic<ATTR><<<lc.shade_grid, RTB_SHADE_THREADS, 0, st>>>(sc, pool, prm, cam);
}
void launch_shade(const LaunchCfg& lc, const DevScene& sc, const DevPool& pool, const DevParams& prm,
                  const DevCamera& cam, uint32_t present, cudaStream_t st) {
  if (lc.attr) launch_shade_kernels<true>(lc, sc, pool, prm, cam, present, st);
  else launch_shade_kernels<false>(lc, sc, pool, prm, cam, present, st);
}
void launch_finalize(const float4* accum, uint8_t* rgb, uint32_t npix, float inv_spp, cudaStream_t st) {
  k_finalize<<<cdiv(npix, 256), 256, 0, st>>>(accum, rgb, npix, inv_spp);
}
void launch_probe_fill(const DevPool& pool, const float* org, const float* dir, const float* time, uint32_t n, cudaStream_t st) {
  k_probe_fill<<<cdiv(pool.n_chunks * RTB_CHUNK, 256), 256, 0, st>>>(pool, org, dir, time, n);
}
void launch_probe_collect(const DevScene& sc, const DevPool& pool, uint32_t n, uint32_t* id_out, float* t_out, cudaStream_t st) {
  k_probe_collect<<<cdiv(n, 256), 256, 0, st>>>(sc, pool, n, id_out, t_out);
}
void launch_kat(const DevScene& sc, const DevCamera& cam, const DevParams& prm, uint32_t op, const uint32_t* in, uint32_t n,
                uint32_t in_stride, uint32_t* out, uint32_t out_stride, cudaStream_t st) {
  k_kat<<<cdiv(n, 128), 128, 0, st>>>(sc, cam, prm, op, in, n, in_stride, out, out_stride);
}
void launch_bw_global(const uint4* p, size_t n_vec, uint32_t reps, uint4* sink, uint32_t grid, cudaStream_t st) {
  k_bw_global<<<grid, 256, 0, st>>>(p, n_vec, reps, sink);
}
void launch_bw_shared(uint32_t reps, uint4* sink, uint32_t grid, cudaStream_t st) {
  k_bw_shared<<<grid, 256, 32768, st>>>(reps, sink);
}
void launch_aov_fill(const DevPool& pool, const DevParams& prm, const DevCamera& cam, unsigned long long first_path,
                     uint32_t n, cudaStream_t st) {
  k_aov_fill<<<cdiv(pool.n_chunks * RTB_CHUNK, 256), 256, 0, st>>>(pool, prm, cam, first_path, n);
}
void launch_aov_collect(const LaunchCfg& lc, const DevScene& sc, const DevPool& pool, const DevParams& prm, float4* aov,
                        uint32_t n, cudaStream_t st) {
  if (lc.attr) k_aov_collect<true><<<cdiv(n, RTB_SHADE_THREADS), RTB_SHADE_THREADS, 0, st>>>(sc, pool, prm, aov, n);
  else k_aov_collect<false><<<cdiv(n, RTB_SHADE_THREADS), RTB_SHADE_THREADS, 0, st>>>(sc, pool, prm, aov, n);
}
void launch_primary_rays(const DevCameraF64& cam, uint32_t W, uint32_t H, float* org, float* dir, float* time,
                         cudaStream_t st) {
  k_primary_rays<<<cdiv(W * H, 256), 256, 0, st>>>(cam, W, H, org, dir, time);
}

int configure_launch(LaunchCfg& lc, uint32_t n_nodes, uint32_t max_depth, uint32_t n_spheres, int sm_count) {
  // stage as much of the (breadth-first ordered) node array as fits the shared-memory budget
  // extend runs 2 CTAs per SM: 2 x (stage + 2 KB list [+ 20 KB of per-warp ray/result buffers, dynamic fetch]) must fit
  // the 227 KB of an SM beside one 3 KB shade CTA
  lc.dynamic_fetch = n_nodes > 4096;
  // 12 KB (153 nodes = the top two to three levels).  Larger stages do not speed extend up (deeper nodes hit L1 anyway:
  // one-lane ext_ms C3 66.3 at 12 KB vs 68.5 at 56 KB, C4 20.8 vs 21.1) and cost the multi-lane pipeline its overlap —
  // with <= ~62 KB per CTA a third extend CTA (of another lane) fits an SM: C4 2748 -> 3268 Mrays/s, C3 3585 -> 3694
  // (profiles/r2_ab.md §9).
  // Deep trees (dynamic fetch, four extend CTAs of four lanes per SM): 6 KB — the root and its children's children; what the
  // stage does not hold comes from an L1 that is 24 KB larger (C4 4075 -> 4108 Mrays/s).
  uint32_t budget = (getenv("RTB_STAGE_KB") ? (uint32_t)atoi(getenv("RTB_STAGE_KB")) : (lc.dynamic_fetch ? 6u : 12u)) * 1024u;
  budget = std::min(budget, (lc.dynamic_fetch ? 84u : 104u) * 1024u);
  uint32_t n_s = n_nodes;
  if ((size_t)n_s * 80 > budget) n_s = budget / 80;
  lc.n_snodes = n_s;
  lc.all_staged = n_s == n_nodes && !(getenv("RTB_ALL_STAGED") && atoi(getenv("RTB_ALL_STAGED")) == 0);
  lc.extend_smem = n_s * 80;
  // which scheduler: one ray per thread for small trees, the warp-queue kernel for trees outside the stage
  // (RTB_EXTEND_MODE = static | dynamic | wq overrides; profiles/r3_ab.md)
  const char* mode = getenv("RTB_EXTEND_MODE");
  lc.mode = lc.dynamic_fetch ? EXTEND_DYNAMIC : EXTEND_STATIC;
  if (mode) lc.mode = !strcmp(mode, "static") ? EXTEND_STATIC : (!strcmp(mode, "wq") ? EXTEND_WQ : EXTEND_DYNAMIC);
  if (lc.mode == EXTEND_WQ && (lc.all_staged || max_depth + 2u > RTB_WQ_STACK))  // (pushes <= internal levels on a path)
    lc.mode = lc.dynamic_fetch ? EXTEND_DYNAMIC : EXTEND_STATIC;
  // fully staged tree: the sphere records go to shared memory too (C1: 486 x 16 B); the leaf tests read them with LDS
  // (only the production kernel reads them: the counting build and the other kernels launch without these bytes)
  lc.sphere_smem = lc.mode == EXTEND_STATIC && lc.all_staged && n_spheres <= RTB_SPHERE_STAGE_BYTES / 16u ? n_spheres * 16u : 0u;
  cudaError_t e;
  const void* extend_fn = (const void*)k_extend<false>;
  if (lc.mode == EXTEND_WQ) {
    const uint32_t wq_bytes = RTB_EXTEND_WARPS * (uint32_t)sizeof(WqWarp);
    lc.extend_smem += wq_bytes;
    extend_fn = (const void*)k_extend_wq<false>;
    for (const void* fn : {(const void*)k_extend_wq<false>, (const void*)k_extend_wq<true>}) {
      e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(budget + wq_bytes));
      if (e != cudaSuccess) return (int)e;
    }
  }
  e = cudaFuncSetAttribute(k_extend<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(k_extend<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget);
  if (e != cudaSuccess) return (int)e;
  for (const void* fn : {(const void*)k_extend_static<true, false, false>, (const void*)k_extend_static<true, false, true>,
                         (const void*)k_extend_static<false, true, false>, (const void*)k_extend_static<false, true, true>,
                         (const void*)k_extend_static<false, false, false>, (const void*)k_extend_static<false, false, true>}) {
    e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget);
    if (e != cudaSuccess) return (int)e;
  }
  // (only for a scene that uses them: with the attribute set on these two kernels for every scene, C4 measured 3.4 % and
  //  C3 1.5 % slower on a B200 at 1000 W, although none of the kernels they run changed; profiles/r6_sphere_stage.md)
  if (lc.sphere_smem) {
    for (const void* fn : {(const void*)k_extend_static<false, true, false, true>, (const void*)k_extend_static<false, true, true, true>}) {
      e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(budget + RTB_SPHERE_STAGE_BYTES));
      if (e != cudaSuccess) return (int)e;
    }
  }
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, extend_fn, RTB_EXTEND_THREADS, lc.extend_smem + lc.sphere_smem);
  if (e != cudaSuccess) return (int)e;
  if (occ < 1) occ = 1;
  // two extend CTAs per SM (of the three that fit): leaves a third of the register file to the shade kernels of the
  // other wavefront lanes, which then really run beside extend (measured +8 % on C1, profiles/r1_ab_extend.md)
  // (512 resident extend threads per SM whatever the CTA size: RTB_EXTEND_THREADS is a build-time knob)
  occ = std::min(occ, getenv("RTB_EXTEND_OCC") ? std::max(1, atoi(getenv("RTB_EXTEND_OCC"))) : std::max(1, 512 / RTB_EXTEND_THREADS));
  lc.extend_grid = (uint32_t)(sm_count * occ);
  int occ2 = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, k_shade_lambert<false>, RTB_SHADE_THREADS, 0);
  if (e != cudaSuccess) return (int)e;
  if (occ2 < 1) occ2 = 1;
  if (getenv("RTB_SHADE_OCC")) occ2 = std::max(1, std::min(occ2, atoi(getenv("RTB_SHADE_OCC"))));
  lc.shade_grid = (uint32_t)(sm_count * occ2);
  lc.fixup_grid = (uint32_t)std::max(1, sm_count * 2);
  {  // smallest pool that gives every resident extend warp AND every resident shade warp a whole number of chunks
    uint32_t a = lc.extend_grid * RTB_EXTEND_WARPS, b = lc.shade_grid * RTB_SHADE_WARPS, x = a, y = b;
    while (y) { const uint32_t t = x % y; x = y; y = t; }
    const uint64_t lcm = (uint64_t)a / x * b;
    lc.pool_unit = lcm * RTB_CHUNK <= (1ull << 23) ? (uint32_t)(lcm * RTB_CHUNK) : b * RTB_CHUNK;
  }
  return 0;
}

}  // namespace rtb
