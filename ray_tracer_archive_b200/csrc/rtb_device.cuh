// rtb_device.cuh — device-side data layout, Philox streams, wide-BVH traversal and primitive tests (sm_100a).
// FP32 restatement of the reference's f64 arithmetic; every routine cites the reference lines it replaces.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <cstring>

#include "rtb_internal.hpp"

namespace rtb {

// RTB_CHECKED build (make -C csrc checked -> librtb200_checked.so): bounds assertions on every index the kernels form
// (traversal stack, node and primitive indices, pool slots, fix-up queue).  compute-sanitizer is closed on the GPU pool, so
// this build + tests/test_gpu_checked.py take its place; a failed assertion bumps a device counter by kind
// (rtb_debug_check_failures) instead of trapping, so one run reports everything.
#ifdef RTB_CHECKED
__device__ unsigned int g_rtb_check_fail[8];
enum CheckKind : int { CHK_STACK = 0, CHK_NODE = 1, CHK_PRIM = 2, CHK_SLOT = 3, CHK_QUEUE = 4, CHK_LIST = 5 };
#define RTB_CHECK(kind, cond)                          \
  do {                                                 \
    if (!(cond)) atomicAdd(&g_rtb_check_fail[kind], 1u); \
  } while (0)
#else
#define RTB_CHECK(kind, cond) ((void)0)
#endif

#define RTB_MAX_LIGHTS 8
#define RTB_MAX_MEDIA 8
#define RTB_MAX_CHECKER_DEPTH 8  /* checker textures nested in checker textures (texture.rs:41-45: Arc<dyn Texture> children) */
#define RTB_MAX_TABLES 4096  /* sanity cap on perlin / image ids (the tables live in device memory, not in DevScene) */
#define RTB_STACK 32
#define RTB_TMIN 0.001f  // main.rs:74
#define RTB_PI 3.14159265358979323846f

enum Queue : uint32_t { Q_TERMINAL = 0, Q_LAMBERT = 1, Q_METAL = 2, Q_DIELECTRIC = 3, Q_ISOTROPIC = 4, Q_COUNT = 5 };
// per-primitive info word y (device copy): material (24 bits) | face mode << 24 (4 bits, FaceMode) | shade queue << 28 (3 bits) | bit 31: quad with an exact plane.
// The queue is resolved from the material type on the host at commit, so `extend` classifies a hit without touching
// the material table (one dependent load less on its tail).
#define RTB_MINFO_MAT(m) ((m) & 0xFFFFFFu)
#define RTB_MINFO_FACE(m) (((m) >> 24) & 15u)
#define RTB_MINFO_QUEUE(m) (((m) >> 28) & 7u)

struct DevTexture {  // 32 bytes
  uint32_t type, even, odd, table;
  float r, g, b, scale;
};
struct DevLight { uint32_t type; float p[5]; float _pad[2]; };
struct DevMedium {
  uint32_t boundary_type, material, prim_id;
  float neg_inv_density;
  float p[6];
  float sin_t, cos_t;
  float off[3];
  uint32_t minfo;  // hit-record word of this medium: material | FACE_TRUE << 24 | queue << 28
};
struct DevImage { const uint8_t* data; uint32_t w, h; };

// Everything the (rare, out-of-line) exact path reads, in device memory: the out-of-line functions get ONE pointer, so the
// kernel's parameter block never has to be materialised in local memory to be passed by reference.
struct ExactTab {
  const float4* tri;              // triangle vertices (their f32 values are the exact record)
  const double* exact[3];         // sphere / moving sphere / quad records, RTB_EXACT_STRIDE doubles each
  const uint2* info[PT_COUNT];    // (primitive id, material word) per leaf entry
  uint32_t media_prim_id[RTB_MAX_MEDIA];
};

struct DevScene {  // passed by value as a kernel parameter (constant bank)
  const uint4* nodes;
  uint32_t n_nodes;
  uint32_t n_lights, n_media, n_materials;
  uint32_t prmt_magic;  // = 0x43000000, see q2f()
  uint32_t n_global;    // primitives tested for every ray before the traversal (kept out of the tree)
  uint32_t tree_empty;  // all primitives are global (tiny scene): skip the traversal
  uint32_t _reserved0;
  uint32_t global_ref[RTB_MAX_GLOBALS];
  uint32_t global_f64;  // bit k: global k is a sphere so large next to the rest of the scene (radius >= 16 scene
                        // extents) that the f32 test can never be trusted for a hit: go to the f64 form directly
  const float4* geom[PT_COUNT];
  const uint2* info[PT_COUNT];
  uint32_t n_prims[PT_COUNT];     // leaf entries per type (RTB_CHECKED bounds)
  const ExactTab* xtab;           // tables of the exact path (device memory)
  const DevScene* self;           // this struct in device memory: the out-of-line exact pass takes ONE pointer
  float coord_max;                // 2 x the largest |coordinate| of the scene box: scale of the plane-test rounding bound
  float eps_ab;                   // rounding bound of a quad's in-plane coordinates (alpha, beta), see intersect_prim
  const float4* materials;   // [2m] (type bits, texture bits, param, texture-type bits) ; [2m+1] solid albedo rgb, 0
  const DevTexture* textures;
  const float4* perlin_vec;   // n_perlin tables x 256 unit vectors
  const uint8_t* perlin_perm; // n_perlin tables x 3 x 256 permutation bytes
  const DevImage* images;     // n_images descriptors (data = nullptr: never set, renders cyan like texture.rs:119-121)
  uint32_t n_perlin, n_images;
  DevLight lights[RTB_MAX_LIGHTS];
  DevMedium media[RTB_MAX_MEDIA];
};

struct DevCamera {  // camera.rs:6-17, basis computed on the host in f64
  float origin[3], lmo[3] /* lower_left_corner - origin */, horizontal[3], vertical[3], u[3], v[3];
  float lens_radius, time0, time1;
};

struct DevCounters {
  uint32_t iter_rays;   // rays extended in the current iteration (one atomicAdd per extend warp at kernel end)
  uint32_t last_rays;   // ... in the previous iteration: 0 = the pool has drained (host check)
  uint32_t iter;
  uint32_t ext_cursor;  // next unclaimed slot batch (dynamic ray fetch)
  uint32_t redo_count[2];  // [0]: length of the fix-up queue this extend launch fills and k_fixup then empties
  uint32_t redo_sel, iter_fixed;  // (spare)
  uint32_t ext_ticket;  // CTAs of k_fixup that have finished (the last one rotates the counters)
  unsigned long long redone;  // total rays re-traced exactly
  unsigned long long refined; // total hits whose distance was recomputed in f64
  unsigned long long total_paths;
  unsigned long long segments, rejected;
  unsigned long long nodes_visited, prims_tested;
  unsigned long long prims_tested_type[PT_COUNT];  // ... per primitive type (the roofline weights each type's bytes / flops)
};

// Path pool of one wavefront instance ("lane").  SLOT-STABLE: a path lives in slot i until it terminates, and slot i is
// then restarted in place with a new camera path.  There are NO global work queues: `extend` walks the pool one
// RTB_CHUNK-slot chunk per warp, orders the chunk's live slots by the kind (and, for trees outside the stage, direction
// octant) of the ray they hold, traces them and writes the hit record and the slot's shade class (the few rays f32 cannot
// decide go to the small fix-up queue of k_fixup); every per-material shade kernel walks the
// class bytes in chunks of RTB_CHUNK slots per warp and compacts the matching slots warp-locally (ballot/scan into a
// shared-memory list).  Path numbers for restarted slots come from a per-chunk cursor over the chunk's own sequence of
// 32-path blocks, so no kernel issues a contended global atomic (the queue-compacting version spent 77 % of
// k_shade_terminal's stall samples on two same-address atomics per warp, profiles/r2_ab.md §3).
#define RTB_CHUNK 256u
// 0..4 = Queue of the slot's current hit.  Class byte: bits 0-2 class; bits 3-5 direction octant of the slot's ray (written
// by the shade kernels when octant ordering is on).
enum SlotClass : uint32_t { CLS_NEW = 6, CLS_DEAD = 7 };
struct DevPool {
  uint32_t n;         // slots
  uint32_t n_chunks;  // ceil(n / RTB_CHUNK)
  float4* ray;        // [2s] origin xyz, time ; [2s+1] direction xyz (un-normalised, ray.rs), 0   — one 32-byte sector
  float4* st;         // [2s] throughput rgb, pixel index bits ; [2s+1] radiance rgb, (sample << 8 | segments) bits
  float4* hit;        // t, ref bits, (material | face mode << 24 | shade queue << 28) bits, 0
  uint8_t* cls;       // [n_chunks * RTB_CHUNK] SlotClass / Queue per slot; padding slots are CLS_DEAD
  uint4* redo[2];     // [0]: [n] rays for the exact pass, (slot | RTB_REDO_REFINE, slab lower bound, upper bound, -)
  unsigned long long* cursor;  // [n_chunks] path numbers consumed so far from the chunk's sequence
  DevCounters* c;
};

// m-th path number of chunk `chunk`: the chunk owns the 32-path blocks chunk, chunk + n_chunks, chunk + 2 n_chunks, ...
// (consecutive numbers are neighbouring pixels of one 8x4 tile, so slots restarted together get coherent primary rays)
__device__ __forceinline__ unsigned long long chunk_path(unsigned long long m, uint32_t chunk, uint32_t n_chunks) {
  return (((m >> 5) * n_chunks + chunk) << 5) | (m & 31ull);
}

struct DevParams {
  uint32_t width, height, spp, sample_offset;
  int32_t max_depth;
  uint32_t rr_start, seed;
  float bg[3];
  const uint32_t* pix_order;  // tile-ordered pixel indices
  double inv_npix;
  float inv_wm1, inv_hm1;     // 1/(W-1), 1/(H-1)
  uint32_t opt;               // A/B switch bits for experiments (env RTB_OPT; 0 in production, currently unused)
  float4* accum;
};

// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
__device__ __forceinline__ float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ float3 operator*(float s, float3 a) { return f3(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ float3 operator*(float3 a, float s) { return f3(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ float dot(float3 a, float3 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, a.z * b.z)); }
__device__ __forceinline__ float3 cross(float3 a, float3 b) {  // vec3.rs:68-76
  return f3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ float3 fma3(float s, float3 a, float3 b) {
  return f3(fmaf(s, a.x, b.x), fmaf(s, a.y, b.y), fmaf(s, a.z, b.z));
}
__device__ __forceinline__ float3 unit(float3 a) { return rsqrtf(dot(a, a)) * a; }
__device__ __forceinline__ float3 xyz(float4 a) { return f3(a.x, a.y, a.z); }
__device__ __forceinline__ float3 ld3(const float* p) { return f3(p[0], p[1], p[2]); }

// One-instruction MUFU reciprocal / square root (<= 1-2 ulp) instead of the IEEE sequences `1.0f / x` and sqrtf()
// compile to (MUFU + Newton step + range check + slow-path call, ~10 instructions each).  Every use is covered by an
// explicit error bound: the slab test is widened (trav_step), the sphere test falls back to f64 when ill-conditioned.
// The host build (tests/emul) uses the exact operations.
__device__ __forceinline__ float rcp_fast(float x) {
#ifdef __CUDA_ARCH__
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
#else
  return 1.0f / x;
#endif
}
__device__ __forceinline__ float log_fast(float x) {
#ifdef __CUDA_ARCH__
  return __logf(x);
#else
  return logf(x);
#endif
}
__device__ __forceinline__ float sqrt_fast(float x) {
#ifdef __CUDA_ARCH__
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
#else
  return sqrtf(x);
#endif
}

// Packed FP32 pairs (sm_100 FFMA2 / FADD2 / FMUL2: two lanes of the FMA pipe in ONE issued instruction).  Each element is
// the scalar IEEE round-to-nearest operation (no .ftz: the library is built without fast-math), so a pair of results is
// bit for bit what two scalar instructions give.  Inline PTX keeps the compiler from contracting an add into a
// neighbouring multiply or splitting the pair; a float2 whose halves are equal (make_float2(s, s)) becomes a broadcast
// operand, no register copy.  The host build (tests/emul) uses the scalar operations.
#ifdef __CUDA_ARCH__
__device__ __forceinline__ unsigned long long pk2(float2 a) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y));
  return r;
}
__device__ __forceinline__ float2 upk2(unsigned long long r) {
  float2 a;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a.x), "=f"(a.y) : "l"(r));
  return a;
}
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {  // a * b + c, one rounding per element
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(b)), "l"(pk2(c)));
  return upk2(r);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  unsigned long long r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(b)));
  return upk2(r);
}
__device__ __forceinline__ float2 fsub2(float2 a, float2 b) {
  unsigned long long r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(b)));
  return upk2(r);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  unsigned long long r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(b)));
  return upk2(r);
}
#else
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) { return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)); }
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 fsub2(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) { return make_float2(a.x * b.x, a.y * b.y); }
#endif
__device__ __forceinline__ float2 f2s(float s) { return make_float2(s, s); }  // broadcast

// ---- Philox4x32-10: key = (pixel, sample), counter = (block, bounce, seed, 'RTB2').  Replaces rand::random
// (rt_weekend.rs:8-19); identical to oracle/rt_oracle.hpp so streams can be compared draw by draw.
enum RngBlock : uint32_t { BLK_CAMERA0 = 0, BLK_CAMERA1 = 1, BLK_SCATTER = 2, BLK_AUX = 3, BLK_MEDIUM0 = 8 };

__device__ __forceinline__ uint4 philox4(uint32_t pixel, uint32_t sample, uint32_t block, uint32_t bounce, uint32_t seed) {
  uint32_t c0 = block, c1 = bounce, c2 = seed, c3 = 0x52544232u;
  uint32_t k0 = pixel, k1 = sample;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }
__device__ __forceinline__ float4 philox_u(uint32_t pixel, uint32_t sample, uint32_t block, uint32_t bounce, uint32_t seed) {
  uint4 r = philox4(pixel, sample, block, bounce, seed);
  return make_float4(u01(r.x), u01(r.y), u01(r.z), u01(r.w));
}

// ---- closest-hit record -----------------------------------------------------------------------------------------
// Parity contract (BASELINE.json: primary-ray primitive ids bit-exact against the f64 reference): every f32 primitive
// test returns its hit distance WITH a bound e on |t_f32 - t_ref| and knows whether each of its own decisions (inside /
// outside, t against t_min) was certain under f32 rounding.  The hot kernels accept or reject a candidate in f32 only
// when that is certain.  Anything f32 leaves open — an edge-grazing hit, two surfaces meeting at the hit point (their
// intervals [t - e, t + e] overlap), an exact tie, an ill-conditioned sphere — lowers the ray's AMBIGUITY HORIZON
// `amb` = the smallest distance at which an undecided candidate may lie.  A later hit that is certainly closer makes
// the open question irrelevant; if at the end of the traversal amb <= the closest hit's upper bound, the ray is
// re-traced by traverse_exact(): the same BVH, every candidate evaluated with the reference's literal f64 arithmetic
// (sphere.rs:41-65, aarect.rs:31-48, hittable.rs:76-85,147-176; same operation order, no FMA contraction) on the
// constructor's own f64 arguments, equal t going to the larger primitive id (hittable_list.rs:44-47).  That happens
// for 0.01-0.2 % of the rays, in a small kernel of its own between extend and shade (k_fixup -> fix_one(), one queue entry
// per thread), so the hot loop contains no call and no f64.  On identical rays the device therefore returns the primitive id the reference's f64 linear scan returns.
struct Closest {
  float t;        // f32 distance of `ref` (closest_so_far, hittable_list.rs:42)
  float hi;       // upper bound of the exact distance of the closest hit (t + error bound): the traversal's t_max
  uint32_t ref;   // type << 29 | leaf index
};
#define RTB_U20 9.5367432e-7f   // 2^-20
#define RTB_U21 4.7683716e-7f
#define RTB_U22 2.3841858e-7f
#define RTB_U23 1.1920929e-7f
enum HitStatus : int { HIT_MISS = 0, HIT_CERTAIN = 1, HIT_AMBIGUOUS = 2 };
struct TestCount { uint32_t n[PT_COUNT]; };  // primitive tests per type (instrumented build only)

// primitive id of a hit reference (list order of the reference's scene graph).  Needed only for the "later primitive
// wins equal t" rule (hittable_list.rs:44-47) and by the parity probe, so it is fetched lazily: an accepted hit does
// not pay the dependent info load (1-5 % of extend's stall samples, profiles/r2e_ncu_summary.md).
__device__ __forceinline__ uint32_t ref_gid(const DevScene& sc, uint32_t ref) {
  const uint32_t type = ref >> REF_TYPE_SHIFT, idx = ref & REF_INDEX_MASK;
  return type == PT_MEDIUM ? sc.media[idx].prim_id : __ldg(&sc.info[type][idx].x);
}

__device__ __forceinline__ uint32_t tab_gid(const ExactTab* tab, uint32_t ref) {
  const uint32_t type = ref >> REF_TYPE_SHIFT, idx = ref & REF_INDEX_MASK;
  return type == PT_MEDIUM ? tab->media_prim_id[idx] : __ldg(&tab->info[type][idx].x);
}

__device__ __forceinline__ float abs1(float3 a) { return fabsf(a.x) + fabsf(a.y) + fabsf(a.z); }

// ---- the reference's f64 arithmetic, operation by operation (no contraction: Rust does not fuse) ------------------
#ifdef __CUDA_ARCH__
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ double dsqrt(double a) { return __dsqrt_rn(a); }
__device__ __forceinline__ uint32_t exact_bits(double v) { return (uint32_t)__double_as_longlong(v); }
#else  // host build (tests/emul), compiled with -ffp-contract=off
__host__ __device__ inline double dadd(double a, double b) { return a + b; }
__host__ __device__ inline double dsub(double a, double b) { return a - b; }
__host__ __device__ inline double dmul(double a, double b) { return a * b; }
__host__ __device__ inline double ddiv(double a, double b) { return a / b; }
__host__ __device__ inline double dsqrt(double a) { return sqrt(a); }
__host__ __device__ inline uint32_t exact_bits(double v) { unsigned long long u; memcpy(&u, &v, 8); return (uint32_t)u; }
#endif
struct D3 { double x, y, z; };
__device__ __forceinline__ D3 d3sub(D3 a, D3 b) { return D3{dsub(a.x, b.x), dsub(a.y, b.y), dsub(a.z, b.z)}; }
__device__ __forceinline__ double d3dot(D3 a, D3 b) {  // vec3.rs:64-66: a.x*b.x + a.y*b.y + a.z*b.z
  return dadd(dadd(dmul(a.x, b.x), dmul(a.y, b.y)), dmul(a.z, b.z));
}
__device__ __forceinline__ D3 d3cross(D3 u, D3 v) {    // vec3.rs:68-76
  return D3{dsub(dmul(u.y, v.z), dmul(u.z, v.y)), -dsub(dmul(u.x, v.z), dmul(u.z, v.x)), dsub(dmul(u.x, v.y), dmul(u.y, v.x))};
}
__device__ __forceinline__ D3 d3at(D3 o, double t, D3 d) {  // ray.rs: origin + t * direction
  return D3{dadd(o.x, dmul(t, d.x)), dadd(o.y, dmul(t, d.y)), dadd(o.z, dmul(t, d.z))};
}

// Sphere::hit root selection (sphere.rs:47-57) with t_max = +inf: the primitive's own first root >= t_min
#define RTB_EXACT_MISS (-1.0)
__device__ __forceinline__ double exact_sphere(D3 o, D3 d, D3 c, double r, double tmin) {
  const D3 oc = d3sub(o, c);
  const double a = d3dot(d, d), half_b = d3dot(oc, d);
  const double cc = dsub(d3dot(oc, oc), dmul(r, r));
  const double det = dsub(dmul(half_b, half_b), dmul(a, cc));
  if (det < 0.0) return RTB_EXACT_MISS;
  const double sqrtd = dsqrt(det);
  double root = ddiv(dsub(-half_b, sqrtd), a);
  if (root < tmin) {
    root = ddiv(dadd(-half_b, sqrtd), a);
    if (root < tmin) return RTB_EXACT_MISS;
  }
  return root < (double)INFINITY ? root : RTB_EXACT_MISS;
}

// The reference's own evaluation of primitive `ref` for the ray (o, d, time), t_min = 0.001 (main.rs:74), t_max = inf.
// Returns the hit distance, or RTB_EXACT_MISS.
static __device__ __noinline__ double exact_hit(const ExactTab* __restrict__ tab, uint32_t ref, float3 of, float3 df, float timef) {
  const uint32_t type = ref >> REF_TYPE_SHIFT, idx = ref & REF_INDEX_MASK;
  const double tmin = 0.001;
  D3 o{(double)of.x, (double)of.y, (double)of.z}, d{(double)df.x, (double)df.y, (double)df.z};
  if (type == PT_TRI) {  // Moller-Trumbore on the f32 vertices (SURVEY §8a N1; the oracle's Triangle::hit)
    const float4 a4 = __ldg(tab->tri + 3 * idx), b4 = __ldg(tab->tri + 3 * idx + 1), c4 = __ldg(tab->tri + 3 * idx + 2);
    const D3 v0{(double)a4.x, (double)a4.y, (double)a4.z};
    const D3 e1 = d3sub(D3{(double)b4.x, (double)b4.y, (double)b4.z}, v0), e2 = d3sub(D3{(double)c4.x, (double)c4.y, (double)c4.z}, v0);
    const D3 pv = d3cross(d, e2);
    const double det = d3dot(e1, pv);
    if (det == 0.0) return RTB_EXACT_MISS;
    const double inv = ddiv(1.0, det);
    const D3 tv = d3sub(o, v0);
    const double u = dmul(d3dot(tv, pv), inv);
    if (u < 0.0 || u > 1.0) return RTB_EXACT_MISS;
    const D3 qv = d3cross(tv, e1);
    const double v = dmul(d3dot(d, qv), inv);
    if (v < 0.0 || dadd(u, v) > 1.0) return RTB_EXACT_MISS;
    const double t = dmul(d3dot(e2, qv), inv);
    return (t >= tmin && t < (double)INFINITY) ? t : RTB_EXACT_MISS;
  }
  const double* e = tab->exact[type] + (size_t)idx * RTB_EXACT_STRIDE;
  const uint32_t bits = exact_bits(e[0]);
  if (bits & EX_TRANSLATE) o = d3sub(o, D3{e[1], e[2], e[3]});  // Translate::hit, hittable.rs:77
  if (bits & EX_ROTATE) {                                       // RotateY::hit, hittable.rs:150-156
    const double sn = e[4], cs = e[5];
    const double ox = dsub(dmul(cs, o.x), dmul(sn, o.z)), oz = dadd(dmul(sn, o.x), dmul(cs, o.z));
    const double dx = dsub(dmul(cs, d.x), dmul(sn, d.z)), dz = dadd(dmul(sn, d.x), dmul(cs, d.z));
    o.x = ox; o.z = oz; d.x = dx; d.z = dz;
  }
  if (type == PT_SPHERE) return exact_sphere(o, d, D3{e[6], e[7], e[8]}, e[9], tmin);
  if (type == PT_MOVING) {  // moving_sphere.rs:36-39: c0 + ((time - t0) / (t1 - t0)) * (c1 - c0)
    const double s = ddiv(dsub((double)timef, e[12]), dsub(e[13], e[12]));
    const D3 dc = d3sub(D3{e[9], e[10], e[11]}, D3{e[6], e[7], e[8]});
    const D3 c{dadd(e[6], dmul(s, dc.x)), dadd(e[7], dmul(s, dc.y)), dadd(e[8], dmul(s, dc.z))};
    return exact_sphere(o, d, c, e[14], tmin);
  }
  const uint32_t sub = (bits >> 8) & 0xFFu;
  if (sub < 3u) {  // XyRect / XzRect / YzRect::hit, aarect.rs:31-48,81-98,150-167
    // normal axis `sub`; in-plane axes (ia, ib) = (sub == 0 ? y : x, sub == 2 ? y : z), selected without local arrays
    const double on = sub == 0u ? o.x : (sub == 1u ? o.y : o.z), dn = sub == 0u ? d.x : (sub == 1u ? d.y : d.z);
    const double oia = sub == 0u ? o.y : o.x, dia = sub == 0u ? d.y : d.x;
    const double oib = sub == 2u ? o.y : o.z, dib = sub == 2u ? d.y : d.z;
    const double t = ddiv(dsub(e[6], on), dn);
    if (!(t >= tmin && t < (double)INFINITY)) return RTB_EXACT_MISS;
    const double a = dadd(oia, dmul(t, dia)), b = dadd(oib, dmul(t, dib));
    if (a < e[7] || a > e[8] || b < e[9] || b > e[10]) return RTB_EXACT_MISS;
    return t;
  }
  // general quad(Q, u, v) (SURVEY §8a N1; the oracle's Quad::hit)
  const D3 Q{e[6], e[7], e[8]}, u{e[9], e[10], e[11]}, v{e[12], e[13], e[14]};
  const D3 n = d3cross(u, v);
  const double nn = d3dot(n, n), denom = d3dot(n, d);
  if (denom == 0.0) return RTB_EXACT_MISS;
  const double t = ddiv(d3dot(n, d3sub(Q, o)), denom);
  if (!(t >= tmin && t < (double)INFINITY)) return RTB_EXACT_MISS;
  const D3 pl = d3sub(d3at(o, t, d), Q);
  const double alpha = ddiv(d3dot(n, d3cross(pl, v)), nn), beta = ddiv(d3dot(n, d3cross(u, pl)), nn);
  if (alpha < 0.0 || alpha > 1.0 || beta < 0.0 || beta > 1.0) return RTB_EXACT_MISS;
  return t;
}

// closest-hit update with a certain hit at t, |t - t_exact| <= e.  `coarse`: the decision is certain but t itself is only
// known to ~1e-5 (a grazing sphere hit): if this hit ends up the closest, its distance is recomputed in f64 afterwards
// (k_fixup, one exact_hit of that primitive — no re-traversal).  The mark lives in bit 8 of the ray's octant word.
#define RTB_TRAV_COARSE 0x100u
__device__ __forceinline__ void consider(Closest& best, float& amb, uint32_t& flags, float t, float e, uint32_t ref, bool coarse) {
  if (!(t < INFINITY)) return;  // degenerate rays (0/0, x/0) never produce a hit
  const float hi = t + e, lo = t - e;
  if (lo > best.hi) return;                     // certainly farther (best.hi = inf while nothing is hit)
  if (best.ref != REF_MISS) {
    const float blo = best.t - (best.hi - best.t);
    if (!(hi < blo)) amb = fminf(amb, fminf(lo, blo));  // the two intervals overlap: which is closer is open
  }
  if (t < best.t) {
    best.t = t; best.ref = ref;
    flags = coarse ? (flags | RTB_TRAV_COARSE) : (flags & ~RTB_TRAV_COARSE);
  }
  best.hi = fminf(best.hi, hi);                 // the closer of the two exact distances is <= both upper bounds
}
// a candidate that may or may not be a hit, at a distance >= lo
__device__ __forceinline__ void undecided(const Closest& best, float& amb, float lo) {
  if (!(lo > best.hi)) amb = fminf(amb, lo);
}

// t against t_min = 0.001 (main.rs:74): certain unless within the error bound AND within a quarter of t_min (the
// self-intersection of a bounce ray sits at |t| ~ 1e-5, far below the band; the band keeps the exact path off it)
__device__ __forceinline__ int tmin_status(float t, float e, float tmin) {
  const float band = fminf(e, 0.25f * tmin);
  return t > tmin + band ? HIT_CERTAIN : (t < tmin - band ? HIT_MISS : HIT_AMBIGUOUS);
}

// Sphere::hit, sphere.rs:41-65, in f64 with MUFU-seeded Newton sqrt / reciprocal (~1e-14 relative): used for the
// "global" sphere whose f32 test can never be trusted (book 1's r = 1000 ground sphere is hit at distances << r from
// points ~r from its centre).  Its own decisions are certain unless within 1e-12 of the threshold.
static __device__ __noinline__ int sphere_roots_f64(float3 o, float3 d, float3 c, float r, float tmin, float& t_out) {
  const double ox = (double)o.x - (double)c.x, oy = (double)o.y - (double)c.y, oz = (double)o.z - (double)c.z;
  const double dx = d.x, dy = d.y, dz = d.z;
  const double a = dx * dx + dy * dy + dz * dz;
  const double hb = ox * dx + oy * dy + oz * dz;
  const double oo = ox * ox + oy * oy + oz * oz, rr = (double)r * (double)r;
  const double cc = oo - rr;
  const double det = hb * hb - a * cc;
  if (fabs(det) <= 1e-12 * (hb * hb + a * (oo + rr))) return HIT_AMBIGUOUS;
  if (det < 0.0) return HIT_MISS;
#ifdef __CUDA_ARCH__
  // sqrt(det) and 1/a to ~1e-14 relative: f32 MUFU seed + one Newton step in f64 (the result is rounded to f32)
  const double y = (double)rsqrtf((float)det);
  double sq = det * y;
  sq = fma(0.5 * y, fma(-sq, sq, det), sq);
  double inv_a = (double)rcp_fast((float)a);
  inv_a = inv_a * fma(-a, inv_a, 2.0);
#else
  const double sq = sqrt(det);
  const double inv_a = 1.0 / a;
#endif
  const double band = 1e-12 * (fabs(hb) + sq) * inv_a + 1e-10;
  double root = (-hb - sq) * inv_a;
  if (fabs(root - (double)tmin) <= band) return HIT_AMBIGUOUS;
  if (root < (double)tmin) {
    root = (-hb + sq) * inv_a;
    if (fabs(root - (double)tmin) <= band) return HIT_AMBIGUOUS;
    if (root < (double)tmin) return HIT_MISS;
  }
  t_out = (float)root;
  return HIT_CERTAIN;
}

// Sphere::hit in f32, in the cancellation-free form  disc' = r^2 - |oc - (oc.d/a) d|^2  (= det/a): the reference's
// c = |oc|^2 - r^2 loses all bits in f32 for large spheres.  Error model (position space): every intermediate carries
// at most epos = 2^-21 (|oc|_1 + r) + 2^-23 (|c|_1 + r) (the second term: f32 rounding of the stored centre / radius
// against the f64 constructor arguments); half-chord h = sqrt(disc'); a root moves by <= epos/|d| (1 + 2r/h) — the 1/h
// term is the grazing amplification.  HIT_AMBIGUOUS (t_out = a lower bound of the possible hit distance) when a
// decision (disc' sign, root against t_min) is inside its bound.  `coarse` = the bound exceeds RTB_SPHERE_REL_MAX t
// (measured: the bound is 50-80x the worst actual error, and the reported t must hold 1e-5 relative): such a hit is
// certain, only its distance wants an f64 recomputation if it ends up the closest.  The same threshold marks the hits of
// rays nearly parallel to a quad's plane / edge-on to a triangle (found by the random scene-graph tests: n.d = 3e-4 |d|,
// bound 3e-3 t, actual error 5e-5 t).
#define RTB_SPHERE_REL_MAX 1.5e-4f  /* (2e-4 let a moving sphere 0.05 away slip to 1.2e-5: random-scene sweep, seed 281) */
// quads / triangles: their bounds are within 2-60x of the actual error, so anything that may exceed 1e-5 is nominated and
// the (cheap, once per ray) conditioning test of fix_kind() decides
#define RTB_FLAT_REL_MAX 1.0e-5f
// (a triangle's bound carries the distance to its vertices, not its size: far, well-conditioned hits sit at 1e-5 t with an
//  actual error of 1e-7 t, while an origin a hair from the plane gives >= 3e-4 t — nominating at 1e-5 sends a third of the
//  mesh hits through the conditioning test, 3 % of C4)
#define RTB_TRI_REL_MAX 1.0e-4f
__device__ __forceinline__ int sphere_fast(float3 o, float3 d, float3 c, float r, float tmin, float tmax_hi, float& t_out, float& e_out,
                                           bool& coarse) {
  const float3 oc = o - c;
  const float a = dot(d, d);
  const float hb = dot(oc, d);
  const float inv_a = rcp_fast(a);
  const float3 l = fma3(-hb * inv_a, d, oc);
  const float disc = fmaf(r, r, -dot(l, l));
  const float epos = fmaf(RTB_U21, abs1(oc) + fabsf(r), RTB_U23 * (abs1(c) + fabsf(r)));
  const float edisc = 4.0f * fabsf(r) * epos;
  if (disc < -edisc) return HIT_MISS;
#ifdef __CUDA_ARCH__
  const float inv_d = rsqrtf(a);
#else
  const float inv_d = 1.0f / sqrtf(a);
#endif
  if (disc <= edisc) {  // grazing: any hit lies within sqrt(2 edisc)/|d| of the closest approach -hb/a
    t_out = fmaf(-hb, inv_a, -(sqrt_fast(2.0f * edisc) * inv_d + RTB_U20 * fabsf(hb * inv_a)));
    return HIT_AMBIGUOUS;
  }
#ifdef __CUDA_ARCH__
  const float rh = rsqrtf(disc);
#else
  const float rh = 1.0f / sqrtf(disc);
#endif
  const float sq = (disc * rh) * (a * inv_d);  // sqrt(a disc')
  const float ebase = epos * inv_d * fmaf(2.0f * fabsf(r), rh, 1.0f);
  float root = (-hb - sq) * inv_a;
  float e = fmaf(RTB_U21, fabsf(root), ebase);
  int st = tmin_status(root, e, tmin);
  if (st == HIT_MISS) {
    root = (-hb + sq) * inv_a;
    e = fmaf(RTB_U21, fabsf(root), ebase);
    st = tmin_status(root, e, tmin);
    if (st == HIT_MISS) return HIT_MISS;
  }
  if (root - e > tmax_hi) return HIT_MISS;
  t_out = root; e_out = e;
  coarse = e > RTB_SPHERE_REL_MAX * root;
  if (st == HIT_AMBIGUOUS) {
    t_out = fmaxf(root - e, 0.0f);
    return HIT_AMBIGUOUS;
  }
  return HIT_CERTAIN;
}

// shade-side sphere root (light pdf, sphere.rs:75-84): f32, f64 only when ill-conditioned; no closest-hit decision hangs on it
__device__ __forceinline__ bool sphere_roots(float3 o, float3 d, float3 c, float r, float tmin, float tmax, float& t_out) {
  float t, e;
  bool coarse = false;
  int st = sphere_fast(o, d, c, r, tmin, tmax, t, e, coarse);
  if (st == HIT_AMBIGUOUS || (st == HIT_CERTAIN && coarse)) st = sphere_roots_f64(o, d, c, r, tmin, t);
  if (st != HIT_CERTAIN || t > tmax) return false;  // (within 1e-12 of tangency / t_min: measure zero for a pdf)
  t_out = t;
  return true;
}

// One f32 primitive test as a PURE function of (ray, primitive): HIT_MISS, HIT_CERTAIN (t, bound e on |t - t_exact|,
// `coarse`) or HIT_AMBIGUOUS (t = a lower bound of the distance at which the undecided candidate may lie).  `tmax_hi` is
// only an early-out (a candidate certainly beyond it is reported as a miss); apply_result() re-checks against the ray's
// current bound, so a stale (larger) tmax_hi changes nothing — which lets the warp-queue extend kernel run the tests of
// many rays side by side and merge afterwards.
template <bool COUNT>
__device__ __forceinline__ int prim_test(const DevScene& sc, uint32_t type, uint32_t idx, float3 o, float3 d, float time, float tmin,
                                         float tmax_hi, float& t, float& e, bool& coarse, TestCount& n_tests) {
  if (COUNT) ++n_tests.n[type];
  RTB_CHECK(CHK_PRIM, type < PT_COUNT && idx < sc.n_prims[type]);
  coarse = false;
  e = 0.0f;
  if (type == PT_SPHERE) {
    const float4 s = __ldg(sc.geom[PT_SPHERE] + idx);
    return sphere_fast(o, d, xyz(s), s.w, tmin, tmax_hi, t, e, coarse);
  } else if (type == PT_QUAD) {
    // aarect.rs:31-48 generalised: t = (n.Q - n.o)/(n.d); in-plane coordinates must lie in the CLOSED unit square.
    // Numerator error <= 2^-22 (|o|_1 + coord_max) (three FMAs on |n_i| <= 1, the stored n.Q); denominator error <=
    // 2^-22 |d|_1; alpha / beta inherit t's error through wa.d, wb.d plus eps_ab (rounding of p and of the plane words).
    const float4 w0 = __ldg(sc.geom[PT_QUAD] + 3 * idx);
    const float nd = dot(xyz(w0), d);
    const float inv = rcp_fast(nd);
    t = (w0.w - dot(xyz(w0), o)) * inv;
    e = fmaf(fabsf(inv), fmaf(RTB_U22 * abs1(d), fabsf(t), RTB_U22 * (abs1(o) + sc.coord_max)), RTB_U21 * fabsf(t));
    if (!(t - e <= tmax_hi)) return HIT_MISS;  // also rejects NaN
    const int st = tmin_status(t, e, tmin);
    if (st == HIT_MISS) return HIT_MISS;
    const float4 w1 = __ldg(sc.geom[PT_QUAD] + 3 * idx + 1);
    const float4 w2 = __ldg(sc.geom[PT_QUAD] + 3 * idx + 2);
    const float3 p = fma3(t, d, o);
    const float alpha = dot(xyz(w1), p) - w1.w;
    const float beta = dot(xyz(w2), p) - w2.w;
    const float ea = fmaf(e, fabsf(dot(xyz(w1), d)), fmaf(RTB_U20, fabsf(alpha), sc.eps_ab));
    const float eb = fmaf(e, fabsf(dot(xyz(w2), d)), fmaf(RTB_U20, fabsf(beta), sc.eps_ab));
    const float ma = fminf(alpha, 1.0f - alpha), mb = fminf(beta, 1.0f - beta);
    if (ma < -ea || mb < -eb) return HIT_MISS;
    if (st == HIT_AMBIGUOUS || !(ma > ea && mb > eb)) { t = fmaxf(t - e, 0.0f); return HIT_AMBIGUOUS; }
    return HIT_CERTAIN;
  } else if (type == PT_TRI) {
    // Triangle (SURVEY §8a N1; no reference counterpart): closed edges and closed t-range like aarect.rs:33,38.
    // Watertight edge functions (Woop, Benthin, Wald 2013): vertices are translated to the ray origin and sheared so
    // the ray runs along +z; the edge function of a shared edge is computed from the SAME two translated vertices by
    // both triangles (exact negatives, no FMA contraction), so f32 rounding can never open a crack in a mesh.
    // An edge function within its rounding bound of zero (the ray passes within ~1e-6 of an edge or vertex) leaves the
    // triangle undecided, so on a shared edge BOTH neighbours are decided — and tie-broken — by the exact pass.
    const float3 v0 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx));
    const float3 v1 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx + 1));
    const float3 v2 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx + 2));
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    const int kz = ax > ay ? (ax > az ? 0 : 2) : (ay > az ? 1 : 2);
    // (kx, ky, kz) cyclic; swapped when d[kz] < 0 to keep the winding
    float3 dp = kz == 0 ? f3(d.y, d.z, d.x) : (kz == 1 ? f3(d.z, d.x, d.y) : d);
    float3 A = v0 - o, B = v1 - o, C = v2 - o;
    const float amax = fmaxf(fmaxf(abs1(A), abs1(B)), abs1(C));
    A = kz == 0 ? f3(A.y, A.z, A.x) : (kz == 1 ? f3(A.z, A.x, A.y) : A);
    B = kz == 0 ? f3(B.y, B.z, B.x) : (kz == 1 ? f3(B.z, B.x, B.y) : B);
    C = kz == 0 ? f3(C.y, C.z, C.x) : (kz == 1 ? f3(C.z, C.x, C.y) : C);
    if (dp.z < 0.0f) {
      float s;
      s = dp.x; dp.x = dp.y; dp.y = s;
      s = A.x; A.x = A.y; A.y = s;
      s = B.x; B.x = B.y; B.y = s;
      s = C.x; C.x = C.y; C.y = s;
    }
    const float Sz = rcp_fast(dp.z), Sx = dp.x * Sz, Sy = dp.y * Sz;
    const float Ax = __fsub_rn(A.x, __fmul_rn(Sx, A.z)), Ay = __fsub_rn(A.y, __fmul_rn(Sy, A.z));
    const float Bx = __fsub_rn(B.x, __fmul_rn(Sx, B.z)), By = __fsub_rn(B.y, __fmul_rn(Sy, B.z));
    const float Cx = __fsub_rn(C.x, __fmul_rn(Sx, C.z)), Cy = __fsub_rn(C.y, __fmul_rn(Sy, C.z));
    const float U = __fsub_rn(__fmul_rn(Cx, By), __fmul_rn(Cy, Bx));
    const float V = __fsub_rn(__fmul_rn(Ax, Cy), __fmul_rn(Ay, Cx));
    const float W = __fsub_rn(__fmul_rn(Bx, Ay), __fmul_rn(By, Ax));
    // a sheared coordinate is off by <= 1.2 2^-22 |A|_1 (translate: 2^-24 |A.x|; shear S A.z with S = d_x (1/d_z): 2^-22 |A.z|;
    // the subtraction: 2^-24), so an edge function (two products of one exact and one perturbed factor pair) by <= m
    const float m = (1.25f * RTB_U22 * amax) * (fabsf(Ax) + fabsf(Ay) + fabsf(Bx) + fabsf(By) + fabsf(Cx) + fabsf(Cy));
    const float mn = fminf(fminf(U, V), W), mx = fmaxf(fmaxf(U, V), W);
    if (mn < -m && mx > m) return HIT_MISS;  // certainly outside
    const float det = U + V + W;
    const float idet = rcp_fast(det), za = Sz * A.z, zb = Sz * B.z, zc = Sz * C.z;
    const float zlo = fminf(fminf(za, zb), zc), zhi = fmaxf(fmaxf(za, zb), zc);
    if (!(mn > m || mx < -m)) {  // on an edge / vertex / edge-on: any hit lies within the triangle's depth range
      if (!(zhi >= tmin)) return HIT_MISS;
      t = fmaxf(zlo - RTB_U20 * fabsf(zlo), 0.0f);
      return HIT_AMBIGUOUS;
    }
    t = (U * za + V * zb + W * zc) * idet;
    // t is the (U, V, W)-weighted mean of the vertex depths: the weights' error m/|det| moves it by at most the depth
    // spread of the triangle (which also covers the rounding of the sum itself: for depths of mixed sign the spread is at
    // least their largest magnitude, for depths of one sign the sum rounds by 2^-22 t)
    e = fmaf(RTB_U20, fabsf(t), 4.0f * m * fabsf(idet) * (zhi - zlo));
    if (!(t - e <= tmax_hi)) return HIT_MISS;
    const int st = tmin_status(t, e, tmin);
    if (st == HIT_AMBIGUOUS) t = fmaxf(t - e, 0.0f);
    return st;
  } else {  // PT_MOVING: MovingSphere::hit, moving_sphere.rs:43-66, centre = A + time*B
    const float4 a = __ldg(sc.geom[PT_MOVING] + 2 * idx);
    const float4 b = __ldg(sc.geom[PT_MOVING] + 2 * idx + 1);
    const float3 c = fma3(time, xyz(b), xyz(a));
    return sphere_fast(o, d, c, a.w, tmin, tmax_hi, t, e, coarse);
  }
}
// the closest-hit update of one test result (hittable_list.rs:42-48 with the certainty bookkeeping)
__device__ __forceinline__ void apply_result(Closest& best, float& amb, uint32_t& flags, int st, float t, float e, uint32_t ref,
                                             bool coarse) {
  if (st == HIT_CERTAIN) consider(best, amb, flags, t, e, ref, coarse);
  else if (st == HIT_AMBIGUOUS) undecided(best, amb, t);
}
template <bool COUNT>
__device__ __forceinline__ void intersect_prim(const DevScene& sc, uint32_t type, uint32_t idx, float3 o, float3 d,
                                               float time, float tmin, Closest& best, float& amb, uint32_t& flags, TestCount& n_tests) {
  float t, e;
  bool coarse;
  const int st = prim_test<COUNT>(sc, type, idx, o, d, time, tmin, best.hi, t, e, coarse, n_tests);
  apply_result(best, amb, flags, st, t, e, (type << REF_TYPE_SHIFT) | idx, coarse);
}

__device__ __forceinline__ float q2f(uint32_t word, uint32_t magic, uint32_t sel) {
  // 7-bit plane byte `sel>>8 & 3` of `word` -> the float 128 + q, with ONE byte permute and no conversion:
  // bits = 0x43000000 | q << 16  (exponent 2^7, q in the top mantissa bits).  The 128 is folded into the node bias.
  // `magic` = 0x43000000 is kept in a REGISTER so that the selector can be the instruction's immediate operand
  // (otherwise ptxas materialises a selector register with an extra MOV before each of the 48 PRMTs of a node).
  return __uint_as_float(__byte_perm(word, magic, sel));
}

// Wide-BVH closest-hit traversal.  `snodes` = first `n_snodes` nodes staged in shared memory (uint4 x5 each);
// the rest are fetched with 128-bit read-only loads.  Semantics = HittableList::hit (hittable_list.rs:39-51)
// over all surface primitives; media are handled by the caller.
// The traversal is split into trav_init / trav_step (ONE node visit or one stack pop per call) so that the extend
// kernel can keep all 32 lanes of a warp busy by swapping finished rays for new ones between steps.
// Every step is exactly one node visit: lanes never spend an iteration on bookkeeping while others decode a node.
#if !defined(__CUDA_ARCH__) && defined(RTB_EMUL_STATS)
inline unsigned long long g_emul_stats[8];  // host build only (tools/emul_stats.py)
inline float g_emul_tmax0 = INFINITY;       // ... initial t_max of the next traversal ("what if the hit distance were known")
#endif
struct Trav {
  float3 o, d;
  float idx, idy, idz, time;
  uint32_t octinv;  // bits 0-2: 7 ^ (sign bits of d): children are visited in descending (slot ^ octinv); bit 8: RTB_TRAV_COARSE
  uint2 grp;        // current node group: x = first child node, y = hit-priority mask << 8 | internal mask
  int sp;
  Closest best;
  float amb;        // ambiguity horizon: smallest distance at which an undecided candidate may lie (inf = none)
};
// slot mask -> priority mask of a ray with octant word `octinv` (bit p of the result = bit p ^ octinv of `m`)
__device__ __forceinline__ uint32_t octant_remap(uint32_t m, uint32_t octinv) {
  if (octinv & 1u) m = ((m & 0x55u) << 1) | ((m & 0xAAu) >> 1);
  if (octinv & 2u) m = ((m & 0x33u) << 2) | ((m & 0xCCu) >> 2);
  if (octinv & 4u) m = ((m & 0x0Fu) << 4) | ((m & 0xF0u) >> 4);
  return m;
}
// octant_remap() of every (octinv, 8-bit mask) as a 2 KB table in shared memory, for the fully staged static kernels:
// one LDS.U8 per node visit (table base in a uniform register) instead of the three conditional swaps (~12 ALU-pipe
// instructions).  The kernel fills it (octmap_fill(), rtb_kernels.cu) before its first __syncthreads().
__shared__ uint8_t s_octmap[8 * 256];
// the ray must be re-traced exactly: something undecided may lie at or before the closest certain hit
__device__ __forceinline__ bool needs_exact(const Closest& best, float amb) { return amb < INFINITY && amb <= best.hi; }
// what k_fixup has to do for a finished ray: 0 nothing, 1 exact re-trace, 2 recompute the distance of its (certain) hit
enum FixKind : uint32_t { FIX_NONE = 0, FIX_RETRACE = 1, FIX_REFINE = 2 };
#define RTB_REDO_REFINE 0x80000000u  /* redo-queue entry: slot | this bit = FIX_REFINE */
// A quad / triangle hit whose error interval (the cheap, loose bound of prim_test(): for a quad it takes |o|_1 + coord_max as
// the magnitude of the plane equation's terms, which would send 2-4 % of the rays of a box-shaped scene to k_fixup — every
// origin within a unit or two of a wall) exceeds RTB_FLAT_REL_MAX t is only NOMINATED; the CONDITIONING of the hit decides: t =
// (n.Q - n.o) / (n.d) loses bits only by cancellation, about 3 x 2^-24 x (sum of the terms' magnitudes / |result|) — so
// 1e-5 needs a cancellation factor below ~64 in the numerator and in the denominator.  An axis-aligned plane whose constant
// is exactly a float (555, 0, 213 ...) has none: one exact product, and the difference of two nearby floats is exact.
__device__ __forceinline__ bool quad_distance_is_coarse(const DevScene& sc, uint32_t idx, float3 o, float3 d) {
  const float4 w0 = __ldg(sc.geom[PT_QUAD] + 3 * idx);
  if (__ldg(&sc.info[PT_QUAD][idx].y) >> 31) return false;  // axis-aligned, plane constant exactly a float (flatten.cpp pack_quad)
  const float mag_num = fabsf(w0.w) + fabsf(w0.x * o.x) + fabsf(w0.y * o.y) + fabsf(w0.z * o.z);
  const float mag_den = fabsf(w0.x * d.x) + fabsf(w0.y * d.y) + fabsf(w0.z * d.z);
  return 64.0f * fabsf(dot(xyz(w0), d)) < mag_den || 64.0f * fabsf(w0.w - dot(xyz(w0), o)) < mag_num;
}
__device__ __forceinline__ bool tri_distance_is_coarse(const DevScene& sc, uint32_t idx, float3 o, float3 d) {
  const float3 v0 = xyz(__ldg(sc.geom[PT_TRI] + 3 * idx));
  const float3 n = cross(xyz(__ldg(sc.geom[PT_TRI] + 3 * idx + 1)) - v0, xyz(__ldg(sc.geom[PT_TRI] + 3 * idx + 2)) - v0);
  const float3 r = v0 - o;  // (the test translates the vertices to the ray origin: magnitudes are local)
  const float mag_num = fabsf(n.x * r.x) + fabsf(n.y * r.y) + fabsf(n.z * r.z);
  const float mag_den = fabsf(n.x * d.x) + fabsf(n.y * d.y) + fabsf(n.z * d.z);
  return 64.0f * fabsf(dot(n, d)) < mag_den || 64.0f * fabsf(dot(n, r)) < mag_num;
}
// fix_kind_cheap(): what can be said without touching memory — FIX_NOMINATED = a quad / triangle hit whose error interval
// (hi - t; no per-test work) exceeds RTB_FLAT_REL_MAX t; resolve_nominated() then looks at the conditioning of that hit.
// The dynamic-fetch kernels resolve in their full-warp result flush, outside the traversal loop (inside it the extra code
// costs the 64-register kernel 4 %).
#define FIX_NOMINATED 3u
__device__ __forceinline__ uint32_t fix_kind_cheap(const Trav& tv) {
  if (needs_exact(tv.best, tv.amb)) return FIX_RETRACE;
  if (tv.best.ref == REF_MISS) return FIX_NONE;
  const uint32_t type = tv.best.ref >> REF_TYPE_SHIFT;
  if (type == PT_QUAD || type == PT_TRI)
    return tv.best.hi - tv.best.t > (type == PT_QUAD ? RTB_FLAT_REL_MAX : RTB_TRI_REL_MAX) * tv.best.t ? FIX_NOMINATED : FIX_NONE;
  return (tv.octinv & RTB_TRAV_COARSE) ? FIX_REFINE : FIX_NONE;
}
__device__ __forceinline__ uint32_t resolve_nominated(const DevScene& sc, uint32_t ref, float3 o, float3 d) {
  const uint32_t type = ref >> REF_TYPE_SHIFT, idx = ref & REF_INDEX_MASK;
  const bool coarse = type == PT_QUAD ? quad_distance_is_coarse(sc, idx, o, d) : tri_distance_is_coarse(sc, idx, o, d);
  return coarse ? FIX_REFINE : FIX_NONE;
}
__device__ __forceinline__ uint32_t fix_kind(const DevScene& sc, const Trav& tv) {
  const uint32_t k = fix_kind_cheap(tv);
  return k == FIX_NOMINATED ? resolve_nominated(sc, tv.best.ref, tv.o, tv.d) : k;
}
// The distance slab the exact pass has to search: every candidate f32 left open lies at or beyond `amb`, the closest
// certain hit within [2t - hi, hi], and whatever the traversal culled lies beyond hi.  Nothing closer than the slab can be
// a hit (a certain candidate entirely below amb would have pulled hi below amb, and the ray would not be here).
__device__ __forceinline__ float slab_lo(const Trav& tv) {
  return tv.best.ref == REF_MISS ? tv.amb : fminf(tv.amb, tv.best.t - (tv.best.hi - tv.best.t));
}

__device__ __forceinline__ void trav_init(Trav& tv, float3 o, float3 d, float time) {
  const float tiny = 1e-30f;
  tv.o = o; tv.d = d; tv.time = time;
  tv.idx = rcp_fast(fabsf(d.x) > tiny ? d.x : copysignf(tiny, d.x));  // <= 1 ulp: covered by the slab widening below
  tv.idy = rcp_fast(fabsf(d.y) > tiny ? d.y : copysignf(tiny, d.y));
  tv.idz = rcp_fast(fabsf(d.z) > tiny ? d.z : copysignf(tiny, d.z));
  tv.octinv = 7u ^ ((d.x < 0.0f ? 1u : 0u) | (d.y < 0.0f ? 2u : 0u) | (d.z < 0.0f ? 4u : 0u));
  tv.grp = make_uint2(0u, (1u << (tv.octinv + 8)) | 1u);  // virtual group whose slot 0 is the root node
  tv.sp = 0;
  tv.best = Closest{INFINITY, INFINITY, REF_MISS};
#if !defined(__CUDA_ARCH__) && defined(RTB_EMUL_STATS)
  tv.best.hi = g_emul_tmax0;
#endif
  tv.amb = INFINITY;
}

// 128-bit load from the shared-memory node stage.  On the device the stage is addressed through a 32-bit shared-space
// address computed ONCE per kernel (`sbase`): through the generic pointer ptxas re-derives the shared window base
// (S2R CgaCtaId, MOV, LEA) at every node visit.
__device__ __forceinline__ uint4 lds_node_word(const uint4* __restrict__ snodes, uint32_t sbase, uint32_t node, uint32_t w) {
#ifdef __CUDA_ARCH__
  uint4 r;
  asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(sbase + node * 80u + w * 16u));
  return r;
#else
  return snodes[5 * node + w];
#endif
}
// sphere record `idx` from the shared-memory copy of the sphere array (the fully staged production kernel stages it after
// the nodes; `ssph` = its 32-bit shared address, kept in a register like `sbase`).  The host build reads the scene's array.
__device__ __forceinline__ float4 lds_sphere(const DevScene& sc, uint32_t ssph, uint32_t idx) {
#ifdef __CUDA_ARCH__
  float4 r;
  asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(ssph + idx * 16u));
  return r;
#else
  return sc.geom[PT_SPHERE][idx];
#endif
}

// returns false when the traversal is complete.  ALL_STAGED: every node of the tree is in the shared-memory stage (small
// scenes), so the global-memory fetch path and its five predicated loads + register moves are compiled out.
// The leaf children a node visit found: `leaf` = slot mask, (w1y, w1z, w1w) = the node's primitive base word and the
// eight (count << 5 | offset) bytes.  expand_leaves() walks them in slot order, ONE primitive per loop iteration (a
// single call site: the lanes of a warp that expand together execute the primitive test together).
template <class Leaf>
__device__ __forceinline__ void expand_leaves(uint32_t leaf, uint32_t w1y, uint32_t w1z, uint32_t w1w, Leaf&& leaf_fn) {
  const uint32_t ptype = w1y >> REF_TYPE_SHIFT, pbase = w1y & REF_INDEX_MASK;
  uint32_t k = 0;
  while (leaf) {
    const uint32_t s = __ffs(leaf) - 1;
    const uint32_t m = ((s < 4 ? w1z : w1w) >> (8 * (s & 3))) & 0xFFu;
    leaf_fn(ptype, pbase + (m & 31u) + k);
    if (++k >= (m >> 5)) { k = 0; leaf &= leaf - 1; }
  }
}

// `leaves(leaf mask, w1y, w1z, w1w)` receives the hit leaf children of the visited node: the hot kernels test them at once
// (intersect_prim) or park them to test many lanes' primitives together; the exact pass runs exact_hit on them.
// STRIDE: distance (in entries) between consecutive levels of the ray's stack (1 = a private array; the warp-queue kernel
// keeps the stacks of a warp's rays interleaved in shared memory).
// PACKED: the child slab test on packed FP32 pairs (FFMA2 / FADD2); the same bits as the scalar form, fewer instructions.
// Used by the fully staged static kernels (C1 / C2); the others keep the scalar form, which measured as fast or faster
// there (the deep-tree kernels' register allocation: C4 -1 % packed).
// OCTMAP: the hit mask's octant remap through the shared-memory table (the kernel fills it, see octmap_fill()).
template <bool COUNT, bool ALL_STAGED, int STRIDE = 1, bool PACKED = false, bool OCTMAP = false, class Leaves>
__device__ __forceinline__ bool trav_step(const DevScene& sc, const uint4* __restrict__ snodes, uint32_t sbase, uint32_t n_snodes,
                                          Trav& tv, uint2* __restrict__ stack, float tmin,
                                          uint32_t& n_nodes_visited, Leaves&& leaves_fn) {
  if (!(tv.grp.y & 0xFF00u)) {  // group exhausted: pop (stack entries always have hits left) and visit in the same step
    if (tv.sp == 0) return false;
    tv.grp = stack[(--tv.sp) * STRIDE];
  }
  const uint32_t octinv = tv.octinv & 7u;
  uint32_t hits = tv.grp.y >> 8;
  const uint32_t prio = 31u - __clz(hits);
  hits &= ~(1u << prio);
  const uint32_t slot = prio ^ octinv;
  const uint32_t gmask = tv.grp.y & 0xFFu;
  const uint32_t node = tv.grp.x + __popc(gmask & ((1u << slot) - 1u));
  RTB_CHECK(CHK_STACK, !hits || tv.sp < RTB_STACK);
  RTB_CHECK(CHK_NODE, node < sc.n_nodes);
  if (hits) stack[(tv.sp++) * STRIDE] = make_uint2(tv.grp.x, (hits << 8) | gmask);
  if (COUNT) ++n_nodes_visited;
  uint4 w0, w1, w2, w3, w4;
  if (ALL_STAGED || node < n_snodes) {
    w0 = lds_node_word(snodes, sbase, node, 0); w1 = lds_node_word(snodes, sbase, node, 1);
    w2 = lds_node_word(snodes, sbase, node, 2); w3 = lds_node_word(snodes, sbase, node, 3);
    w4 = lds_node_word(snodes, sbase, node, 4);
  } else {
    const uint4* p = sc.nodes + 5 * (size_t)node;
    w0 = __ldg(p); w1 = __ldg(p + 1); w2 = __ldg(p + 2); w3 = __ldg(p + 3); w4 = __ldg(p + 4);
  }
  const uint32_t imask = w0.w >> 24;
  const bool nx = !(octinv & 1u), ny = !(octinv & 2u), nz = !(octinv & 4u);  // direction component negative
  // t = q * (step * idir) + (origin - o) * idir ; widened by the f32 rounding bound so that no true hit is culled
  const float ax = __uint_as_float((w0.w & 0xFFu) << 23) * tv.idx;
  const float ay = __uint_as_float(((w0.w >> 8) & 0xFFu) << 23) * tv.idy;
  const float az = __uint_as_float(((w0.w >> 16) & 0xFFu) << 23) * tv.idz;
  const float bx = (__uint_as_float(w0.x) - tv.o.x) * tv.idx;
  const float by = (__uint_as_float(w0.y) - tv.o.y) * tv.idy;
  const float bz = (__uint_as_float(w0.z) - tv.o.z) * tv.idz;
  const float eps = 5.0e-7f;  // bound on the f32 rounding of q a + b (|q a| <= 255 |a| incl. the folded 128) + 1 ulp of idir
  const float ex = eps * fmaf(256.0f, fabsf(ax), fabsf(bx));
  const float ey = eps * fmaf(256.0f, fabsf(ay), fabsf(by));
  const float ez = eps * fmaf(256.0f, fabsf(az), fabsf(bz));
  // planes decode as (128 + q): fold -128 a into the bias (error 128 ulp(a) << the quantisation step a)
  const float cx = fmaf(-128.0f, ax, bx), cy = fmaf(-128.0f, ay, by), cz = fmaf(-128.0f, az, bz);
  const float bnx = cx - ex, bfx = cx + ex, bny = cy - ey, bfy = cy + ey, bnz = cz - ez, bfz = cz + ez;
  // near/far plane words per axis (children 0-3 | 4-7)
  const uint32_t nx0 = nx ? w3.z : w2.x, nx1 = nx ? w3.w : w2.y, fx0 = nx ? w2.x : w3.z, fx1 = nx ? w2.y : w3.w;
  const uint32_t ny0 = ny ? w4.x : w2.z, ny1 = ny ? w4.y : w2.w, fy0 = ny ? w2.z : w4.x, fy1 = ny ? w2.w : w4.y;
  const uint32_t nz0 = nz ? w4.z : w3.x, nz1 = nz ? w4.w : w3.y, fz0 = nz ? w3.x : w4.z, fz1 = nz ? w3.y : w4.w;
  // child i is hit iff max(tn_xyz, tmin) <= min(tf_xyz, t_max)  <=>  tn3 <= tf3  and  tn3 <= t_max  and  tmin <= tf3
  // (tmin <= t_max always).  The three differences are on the FMA pipe; their sign bits are OR-ed with one LOP3 and
  // shifted into the mask with one funnel shift: 4 ALU-pipe instructions per child (2 FMNMX3, LOP3, SHF) instead of
  // 6.4 (2 FMNMX, 2 FMNMX3, FSETP, SEL, IADD3/3) — the node test is ALU-pipe bound (profiles/r1d_c1_ncu_summary.md).
  const uint32_t magic = sc.prmt_magic;  // 0x43000000, read from the constant bank (ptxas cannot fold it into the PRMT)
  const float tmax = tv.best.hi;  // upper bound of the closest hit's exact distance: a subtree is culled only if it
                                  // cannot hold a hit at or before it (equal t must still reach the id tie-break)
  uint32_t missmask;
  if constexpr (PACKED) {
    // Children i and i + 4 read their plane bytes from the same byte of the 0-3 / 4-7 words and share scale and bias:
    // each plane of the pair is one FFMA2 (the two PRMTs write an aligned register pair), and tf - tn one FADD2.  The
    // min / max (no packed form), the two differences against the ray's bounds and the sign-bit assembly stay per child
    // (packing those too costs the 80-register kernels spills).  Every element is the scalar operation, bit for bit.
    uint32_t mlo = 0, mhi = 0;  // miss bits of children 0-3 | 4-7
#pragma unroll
    for (int i = 3; i >= 0; --i) {
      const uint32_t sel = 0x7044u | ((uint32_t)i << 8);
      const float2 tnx = ffma2(make_float2(q2f(nx0, magic, sel), q2f(nx1, magic, sel)), f2s(ax), f2s(bnx));
      const float2 tny = ffma2(make_float2(q2f(ny0, magic, sel), q2f(ny1, magic, sel)), f2s(ay), f2s(bny));
      const float2 tnz = ffma2(make_float2(q2f(nz0, magic, sel), q2f(nz1, magic, sel)), f2s(az), f2s(bnz));
      const float2 tfx = ffma2(make_float2(q2f(fx0, magic, sel), q2f(fx1, magic, sel)), f2s(ax), f2s(bfx));
      const float2 tfy = ffma2(make_float2(q2f(fy0, magic, sel), q2f(fy1, magic, sel)), f2s(ay), f2s(bfy));
      const float2 tfz = ffma2(make_float2(q2f(fz0, magic, sel), q2f(fz1, magic, sel)), f2s(az), f2s(bfz));
      const float2 tn = make_float2(fmaxf(fmaxf(tnx.x, tny.x), tnz.x), fmaxf(fmaxf(tnx.y, tny.y), tnz.y));
      const float2 tf = make_float2(fminf(fminf(tfx.x, tfy.x), tfz.x), fminf(fminf(tfx.y, tfy.y), tfz.y));
      const float2 d = fsub2(tf, tn);
      // (m << 1) | sign bit: child i ends in bit i of its half
      mlo = __funnelshift_l(__float_as_uint(d.x) | __float_as_uint(tmax - tn.x) | __float_as_uint(tf.x - tmin), mlo, 1);
      mhi = __funnelshift_l(__float_as_uint(d.y) | __float_as_uint(tmax - tn.y) | __float_as_uint(tf.y - tmin), mhi, 1);
    }
    missmask = (mhi << 4) | mlo;
  } else {
    missmask = 0;
#pragma unroll
    for (int i = 7; i >= 0; --i) {
      const uint32_t sel = 0x7044u | ((uint32_t)(i & 3) << 8);
      const float tnx = fmaf(q2f(i < 4 ? nx0 : nx1, magic, sel), ax, bnx);
      const float tny = fmaf(q2f(i < 4 ? ny0 : ny1, magic, sel), ay, bny);
      const float tnz = fmaf(q2f(i < 4 ? nz0 : nz1, magic, sel), az, bnz);
      const float tfx = fmaf(q2f(i < 4 ? fx0 : fx1, magic, sel), ax, bfx);
      const float tfy = fmaf(q2f(i < 4 ? fy0 : fy1, magic, sel), ay, bfy);
      const float tfz = fmaf(q2f(i < 4 ? fz0 : fz1, magic, sel), az, bfz);
      const float tn = fmaxf(fmaxf(tnx, tny), tnz);
      const float tf = fminf(fminf(tfx, tfy), tfz);
      const uint32_t neg = __float_as_uint(tf - tn) | __float_as_uint(tmax - tn) | __float_as_uint(tf - tmin);
      missmask = __funnelshift_l(neg, missmask, 1);  // (missmask << 1) | sign bit; child 0 ends in bit 0
    }
  }
  const uint32_t hitmask = ~missmask & 0xFFu;
#if !defined(__CUDA_ARCH__) && defined(RTB_EMUL_STATS)
  ++g_emul_stats[0];                    // node visits
  if (!hitmask) ++g_emul_stats[1];      // ... that found no child to continue with (stale stack entries, loose boxes)
  g_emul_stats[2] += __builtin_popcount(hitmask & imask);   // internal children hit
  g_emul_stats[3] += __builtin_popcount(hitmask & ~imask);  // leaf children hit
  {  // visits whose hit leaves hold 1 / 2 / 3+ primitives (the trips of the leaf loop)
    uint32_t np = 0;
    for (uint32_t s = 0; s < 8; ++s)
      if ((hitmask & ~imask) >> s & 1u) np += (((s < 4 ? w1.z : w1.w) >> (8 * (s & 3))) & 0xFFu) >> 5;
    if (np) ++g_emul_stats[np == 1 ? 4 : (np == 2 ? 5 : 6)];
    g_emul_stats[7] += np;
  }
#endif
  // internal children: slot mask -> priority mask (bit p = slot ^ octinv)
  uint32_t ih = hitmask & imask;
  if constexpr (OCTMAP) ih = s_octmap[(octinv << 8) | ih];  // one shared-memory byte instead of three conditional swaps
  else ih = octant_remap(ih, octinv);
  tv.grp = make_uint2(w1.x, (ih << 8) | imask);
  // (measured and removed: prefetching the next step's node into L1 here, -4 % — and even switched off the dormant path
  //  cost the deep-tree kernels 2-3 %, profiles/r3_ab.md §3)
  // leaf children (all primitives of one node share a type)
  const uint32_t leaf = hitmask & ~imask;
  if (leaf) leaves_fn(leaf, w1.y, w1.z, w1.w);
  return true;
}

// the scene's "global" primitives (huge relative to the scene, kept out of the tree): tested first, which also
// establishes an early t_max for the traversal
template <bool COUNT>
__device__ __forceinline__ void trav_globals(const DevScene& sc, Trav& tv, float tmin, TestCount& n_tests) {
  for (uint32_t k = 0; k < sc.n_global; ++k) {
    const uint32_t ref = sc.global_ref[k];
    if ((sc.global_f64 >> k) & 1u) {  // the r = 1000 ground sphere of book 1: skip the f32 attempt (~100 instructions per ray)
      if (COUNT) ++n_tests.n[PT_SPHERE];
      const float4 s = __ldg(sc.geom[PT_SPHERE] + (ref & REF_INDEX_MASK));
      float t;
      const int st = sphere_roots_f64(tv.o, tv.d, xyz(s), s.w, tmin, t);
      if (st == HIT_CERTAIN) consider(tv.best, tv.amb, tv.octinv, t, RTB_U22 * t, ref, false);
      else if (st == HIT_AMBIGUOUS) tv.amb = 0.0f;  // within 1e-12 of tangency / t_min: exact pass
    } else {
      intersect_prim<COUNT>(sc, ref >> REF_TYPE_SHIFT, ref & REF_INDEX_MASK, tv.o, tv.d, tv.time, tmin, tv.best, tv.amb, tv.octinv, n_tests);
    }
  }
  if (sc.tree_empty) tv.grp.y = 0u;  // nothing left to traverse: the first trav_step returns false
}

// one hot-path step: the leaf primitives go through the f32 tests
// SPHSTAGE: sphere records come from the shared-memory copy at `ssph` (lds_sphere: one LDS.128 through a register address)
// instead of a read-only global load; the test itself is prim_test()'s sphere_fast(), so the results are the same bits.
template <bool COUNT, bool ALL_STAGED = false, bool PACKED = false, bool OCTMAP = false, bool SPHSTAGE = false>
__device__ __forceinline__ bool trav_step_fast(const DevScene& sc, const uint4* __restrict__ snodes, uint32_t sbase, uint32_t n_snodes,
                                               Trav& tv, uint2* __restrict__ stack, float tmin,
                                               uint32_t& n_nodes_visited, TestCount& n_tests, uint32_t ssph = 0u) {
  return trav_step<COUNT, ALL_STAGED, 1, PACKED, OCTMAP>(sc, snodes, sbase, n_snodes, tv, stack, tmin, n_nodes_visited,
                                      [&](uint32_t leaf, uint32_t w1y, uint32_t w1z, uint32_t w1w) {
                                        expand_leaves(leaf, w1y, w1z, w1w, [&](uint32_t type, uint32_t idx) {
                                          if (SPHSTAGE && type == PT_SPHERE) {
                                            if (COUNT) ++n_tests.n[PT_SPHERE];
                                            RTB_CHECK(CHK_PRIM, idx < sc.n_prims[PT_SPHERE]);
                                            float t, e = 0.0f;
                                            bool coarse = false;
                                            const float4 s = lds_sphere(sc, ssph, idx);
                                            const int st = sphere_fast(tv.o, tv.d, xyz(s), s.w, tmin, tv.best.hi, t, e, coarse);
                                            apply_result(tv.best, tv.amb, tv.octinv, st, t, e, ((uint32_t)PT_SPHERE << REF_TYPE_SHIFT) | idx, coarse);
                                          } else {
                                            intersect_prim<COUNT>(sc, type, idx, tv.o, tv.d, tv.time, tmin, tv.best, tv.amb, tv.octinv, n_tests);
                                          }
                                        });
                                      });
}

// Deferred leaf tests.  A node visit parks its hit leaves in the lane's shared-memory record instead of testing them; the
// lane then sits out the node phases (its t_max must see those tests before it descends further) until the warp
// drains: all parked lanes test their primitives TOGETHER, one primitive type at a time, one primitive per iteration.
// The per-ray order of node visits and primitive tests is unchanged, so results, counters and the exact-pass set are
// identical to the inline form; only how many lanes execute a primitive test at once changes (inline: the ~1/3 of the
// lanes whose node happened to have a leaf hit; drained: >= the threshold).  Used by the 64-register dynamic-fetch kernel,
// with the scalar slab test (the packed one spills there).
template <bool COUNT, bool ALL_STAGED = false>
__device__ __forceinline__ bool trav_step_park(const DevScene& sc, const uint4* __restrict__ snodes, uint32_t sbase, uint32_t n_snodes,
                                               Trav& tv, uint2* __restrict__ stack, float tmin, uint32_t& n_nodes_visited,
                                               uint4* __restrict__ park, bool& parked) {
  return trav_step<COUNT, ALL_STAGED, 1, false>(sc, snodes, sbase, n_snodes, tv, stack, tmin, n_nodes_visited,
                                      [&](uint32_t leaf, uint32_t w1y, uint32_t w1z, uint32_t w1w) {
                                        *park = make_uint4(leaf, w1y, w1z, w1w);
                                        parked = true;
                                      });
}
// executed by the whole warp; `parked` lanes test what they parked
template <bool COUNT>
__device__ __forceinline__ void drain_parked(const DevScene& sc, Trav& tv, float tmin, const uint4* __restrict__ park, bool parked,
                                             TestCount& n_tests) {
  uint4 pd = make_uint4(0u, 0u, 0u, 0u);
  if (parked) pd = *park;
  const uint32_t mytype = pd.y >> REF_TYPE_SHIFT;
#pragma unroll
  for (uint32_t t = 0; t < PT_COUNT; ++t) {  // one type at a time: the type switch inside intersect_prim folds away
    const bool mine = parked && mytype == t;
    if (!__any_sync(0xffffffffu, mine)) continue;
    if (mine)
      expand_leaves(pd.x, pd.y, pd.z, pd.w, [&](uint32_t, uint32_t idx) {
        intersect_prim<COUNT>(sc, t, idx, tv.o, tv.d, tv.time, tmin, tv.best, tv.amb, tv.octinv, n_tests);
      });
    __syncwarp();
  }
}

// returns the ray's FixKind
template <bool COUNT, bool ALL_STAGED = false, bool PACKED = false, bool OCTMAP = false, bool SPHSTAGE = false>
__device__ __forceinline__ uint32_t traverse(const DevScene& sc, const uint4* __restrict__ snodes, uint32_t sbase, uint32_t n_snodes,
                                         float3 o, float3 d, float time, float tmin, Closest& best, float& slab_lo_out,
                                         uint32_t& n_nodes_visited, TestCount& n_tests, uint32_t ssph = 0u) {
  Trav tv;
  uint2 stack[RTB_STACK];
  trav_init(tv, o, d, time);
  trav_globals<COUNT>(sc, tv, tmin, n_tests);
  while (trav_step_fast<COUNT, ALL_STAGED, PACKED, OCTMAP, SPHSTAGE>(sc, snodes, sbase, n_snodes, tv, stack, tmin, n_nodes_visited, n_tests, ssph)) {}
  best = tv.best;
  slab_lo_out = slab_lo(tv);
  return fix_kind(sc, tv);
}

// FIX_REFINE: the hit is certain, its distance is recomputed with the reference's arithmetic
__device__ __forceinline__ float refine_hit(const DevScene& sc, uint32_t ref, float3 o, float3 d, float time, float t) {
  if ((ref >> REF_TYPE_SHIFT) >= PT_COUNT) return t;  // a medium's sampled distance
  const double tc = exact_hit(sc.xtab, ref, o, d, time);
  return tc >= 0.0 ? (float)tc : t;
}

// The exact pass: the same BVH (its conservative boxes cull against the closest exact distance so far), every candidate
// evaluated by exact_hit(), min t with equal t going to the larger primitive id = HittableList::hit
// (hittable_list.rs:39-51) in f64.  Nodes come from global memory (n_snodes = 0).  [t_lo, t_hi] = the slab handed over by
// the hot kernel (0, inf = search everything): only the nodes the ray crosses inside it are visited.
__device__ __forceinline__ Closest traverse_exact(const DevScene& sc, float3 o, float3 d, float time, float t_lo = 0.0f, float t_hi = INFINITY) {
  Trav tv;
  uint2 stack[RTB_STACK];
  trav_init(tv, o, d, time);
  tv.best.hi = fmaf(t_hi, 4.0e-6f, t_hi) + 1.0e-6f;                       // slack: the bounds are f32 themselves
  const float tmin = fmaxf(fmaf(t_lo, -4.0e-6f, t_lo) - 1.0e-6f, 0.0f);  // (exact_hit applies the real t_min = 0.001)
  double bt = 0.0;
  const ExactTab* tab = sc.xtab;
  auto leaf = [&](uint32_t type, uint32_t idx) {
    const uint32_t ref = (type << REF_TYPE_SHIFT) | idx;
    {  // the f32 test first: a CERTAIN miss (most candidates of a long slab) needs no f64 evaluation
      Closest probe{INFINITY, tv.best.hi, REF_MISS};
      float probe_amb = INFINITY;
      uint32_t probe_flags = 0;
      TestCount none{};
      intersect_prim<false>(sc, type, idx, tv.o, tv.d, tv.time, RTB_TMIN, probe, probe_amb, probe_flags, none);
      if (probe.ref == REF_MISS && !(probe_amb < INFINITY)) return;
    }
    const double tc = exact_hit(tab, ref, tv.o, tv.d, tv.time);
    if (tc < 0.0) return;
    if (tv.best.ref == REF_MISS || tc < bt || (tc == bt && tab_gid(tab, ref) > tab_gid(tab, tv.best.ref))) {
      bt = tc;
      const float tf = (float)tc;
      tv.best.t = tf;
      tv.best.hi = tf * (1.0f + RTB_U22);
      tv.best.ref = ref;
    }
  };
  for (uint32_t k = 0; k < sc.n_global; ++k) leaf(sc.global_ref[k] >> REF_TYPE_SHIFT, sc.global_ref[k] & REF_INDEX_MASK);
  if (sc.tree_empty) tv.grp.y = 0u;
  uint32_t nv = 0;
  while (trav_step<false, false>(sc, nullptr, 0u, 0u, tv, stack, tmin, nv,
                                 [&](uint32_t lf, uint32_t w1y, uint32_t w1z, uint32_t w1w) { expand_leaves(lf, w1y, w1z, w1w, leaf); })) {}
  if (tv.best.ref == REF_MISS) tv.best.t = tv.best.hi = INFINITY;
  return tv.best;
}

// ConstantMedium::hit, constant_medium.rs:31-71, for the (few) media of the scene; the boundary interval is found
// analytically (sphere: both roots; box: slabs in the boundary's object space).  One uniform per (path, segment, medium).
__device__ __forceinline__ void intersect_media(const DevScene& sc, float3 o, float3 d, float tmin, Closest& best,
                                                uint32_t pixel, uint32_t sample, uint32_t bounce, uint32_t seed,
                                                bool have_rng) {
  for (uint32_t m = 0; m < sc.n_media; ++m) {
    const DevMedium& md = sc.media[m];
    float t1, t2;
    if (md.boundary_type == RTB_BOUNDARY_SPHERE) {
      float3 c = f3(md.p[0], md.p[1], md.p[2]);
      float3 oc = o - c;
      float a = dot(d, d), hb = dot(oc, d), inv_a = rcp_fast(a);
      float3 l = fma3(-hb * inv_a, d, oc);
      float disc = fmaf(md.p[3], md.p[3], -dot(l, l));
      if (disc < 0.0f) continue;
      float sq = sqrt_fast(a * disc);
      t1 = (-hb - sq) * inv_a;      // boundary.hit(r, -inf, inf): first root always in range
      t2 = (-hb + sq) * inv_a;      // boundary.hit(r, t1 + 0.0001, inf)
      if (t2 < t1 + 0.0001f) continue;
    } else {
      // object space of Translate(RotateY(Box)): hittable.rs:76,150-156
      float3 oo = o - f3(md.off[0], md.off[1], md.off[2]);
      float3 ro = f3(md.cos_t * oo.x - md.sin_t * oo.z, oo.y, md.sin_t * oo.x + md.cos_t * oo.z);
      float3 rd = f3(md.cos_t * d.x - md.sin_t * d.z, d.y, md.sin_t * d.x + md.cos_t * d.z);
      float lo = -INFINITY, hi = INFINITY;
      const float ro_[3] = {ro.x, ro.y, ro.z}, rd_[3] = {rd.x, rd.y, rd.z};
      bool miss = false;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        if (rd_[a] == 0.0f) {
          if (ro_[a] < md.p[a] || ro_[a] > md.p[3 + a]) miss = true;
          continue;
        }
        float inv = rcp_fast(rd_[a]);
        float ta = (md.p[a] - ro_[a]) * inv, tb = (md.p[3 + a] - ro_[a]) * inv;
        lo = fmaxf(lo, fminf(ta, tb));
        hi = fminf(hi, fmaxf(ta, tb));
      }
      if (miss || !(hi >= lo + 0.0001f)) continue;
      t1 = lo; t2 = hi;
    }
    if (t1 < tmin) t1 = tmin;
    if (t2 > best.t) t2 = best.t;
    if (t1 >= t2) continue;
    if (t1 < 0.0f) t1 = 0.0f;
    float len = sqrt_fast(dot(d, d));
    float inside = (t2 - t1) * len;
    float xi = have_rng ? u01(philox4(pixel, sample, BLK_MEDIUM0 + m, bounce, seed).x) : 0.5f;
    float hd = md.neg_inv_density * log_fast(xi);
    if (hd > inside) continue;
    float t = t1 + hd * rcp_fast(len);
    // a sampled (continuous) distance: accepted iff closer than the closest surface / earlier medium, no tie rule needed
    if (t < INFINITY && (best.ref == REF_MISS || t < best.t)) {
      best.t = t; best.hi = t; best.ref = ((uint32_t)PT_MEDIUM << REF_TYPE_SHIFT) | m;
    }
  }
}

}  // namespace rtb
