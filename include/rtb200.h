/*
 * rtb200.h — C ABI of librtb200.so: the B200-native (sm_100a) implementation of the
 * per-pixel Monte Carlo `ray_color` bounce loop of OrientalHorizon/Ray-Tracer-Archive.
 *
 * The reference (a Rust binary crate) has no FFI; the narrowest seam on its hot path is
 *     ray_color(&Ray, &Color3, &dyn Hittable, Arc<dyn Hittable>, i32) -> Color3   raytracer/src/main.rs:63-139
 * called once per sample by the pixel loop                                         raytracer/src/main.rs:731-784
 * A per-ray FFI is meaningless for a GPU, so the boundary sits one level up:
 * "render this scene (described with the reference's own constructors) into a float accumulation buffer".
 *
 * Two ways to hand a scene over, both plain C (pointers + sizes, no C++/torch types):
 *   1. GRAPH records (rtb_node[]): one record per reference constructor call
 *      (Sphere::construct, XzRect::construct, Box::construct, Translate::construct, ...).  The library's host
 *      C++ flattens the graph (instances -> world space, Box -> 6 quads, ids in list order) and builds the wide BVH.
 *      This is what the Rust shim's `flatten()` emits (see INTEGRATION.md).
 *   2. FLAT SoA arrays (rtb_scene_set_*): for callers that flatten themselves.
 *
 * Conventions (all from the reference):
 *   - primitive id  = depth-first leaf order of the scene graph (HittableList order, raytracer/src/hittable_list.rs:43-49;
 *                     Box expands to its 6 sides in raytracer/src/boxes.rs:19-68 order).  Equal-t ties are won by
 *                     the LATER primitive (larger id)        raytracer/src/hittable_list.rs:44-47, sphere.rs:52, aarect.rs:33
 *   - ray directions are NOT normalised; t is in units of the ray's own direction; t_min = 0.001   main.rs:74
 *   - image row 0 is the TOP row (reference stores scanline j at row H-1-j, main.rs:733); v = (j+xi)/(H-1), u = (i+xi)/(W-1)
 *
 * Error behaviour: every call returns 0 on success, a negative rtb_status otherwise; rtb_last_error() returns a
 * thread-local message.  (The reference panics via unwrap()/assert_eq!, main.rs:656,762,777,779.)
 * There is NO CPU fallback: without a CUDA device rtb_context_create fails with RTB_ERR_NO_DEVICE.
 *
 * Threading: a context is not re-entrant; serialise calls on one context (the reference's render loop is owned by
 * one thread, main.rs:731).  One context drives one GPU; multi-GPU = one process (context) per GPU, samples split
 * by `sample_offset`, accumulation buffers summed by the caller's NCCL reduce (see rtb_render_device).
 */
#ifndef RTB200_H
#define RTB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTB_ABI_VERSION 2u
#define RTB_NONE 0xFFFFFFFFu

typedef enum rtb_status {
  RTB_OK = 0,
  RTB_ERR_INVALID = -1,     /* bad argument / malformed graph            */
  RTB_ERR_NO_DEVICE = -2,   /* no usable CUDA device (no CPU fallback)   */
  RTB_ERR_CUDA = -3,        /* CUDA runtime error, see rtb_last_error()  */
  RTB_ERR_STATE = -4,       /* call order (e.g. render before commit)    */
  RTB_ERR_UNSUPPORTED = -5  /* e.g. light on a primitive that cannot be sampled */
} rtb_status;

/* ---- graph records: one per reference constructor ------------------------------------------------------ */
typedef enum rtb_node_type {
  RTB_NODE_SPHERE = 1,          /* Sphere::construct(center, radius, mat)          sphere.rs:19   p = cx cy cz r            */
  RTB_NODE_MOVING_SPHERE = 2,   /* MovingSphere::construct(c0,c1,t0,t1,r,mat)      moving_sphere.rs:18  p = c0[3] c1[3] t0 t1 r */
  RTB_NODE_XY_RECT = 3,         /* XyRect::construct(x0,x1,y0,y1,k,mat)            aarect.rs:19   p = a0 a1 b0 b1 k         */
  RTB_NODE_XZ_RECT = 4,         /* XzRect::construct(x0,x1,z0,z1,k,mat)            aarect.rs:69                              */
  RTB_NODE_YZ_RECT = 5,         /* YzRect::construct(y0,y1,z0,z1,k,mat)            aarect.rs:138                             */
  RTB_NODE_BOX = 6,             /* Box::construct(p0,p1,mat)                       boxes.rs:18    p = p0[3] p1[3]           */
  RTB_NODE_TRIANGLE = 7,        /* new (SURVEY §8a N1)                             p = v0[3] v1[3] v2[3]                    */
  RTB_NODE_QUAD = 8,            /* new, RTTNW quad(Q,u,v)                          p = Q[3] u[3] v[3]                       */
  RTB_NODE_MESH = 9,            /* new: triangle mesh set with rtb_scene_set_mesh; p[0] = mesh id                           */
  RTB_NODE_TRANSLATE = 16,      /* Translate::construct(child, offset)             hittable.rs:68  p = off[3]               */
  RTB_NODE_ROTATE_Y = 17,       /* RotateY::construct(child, angle_degrees)        hittable.rs:107 p = angle                */
  RTB_NODE_FLIP_FACE = 18,      /* FlipFace::construct(child)                      hittable.rs:187                           */
  RTB_NODE_CONSTANT_MEDIUM = 19,/* ConstantMedium::construct_color(boundary,d,c)   constant_medium.rs:23 p = density; material = Isotropic */
  RTB_NODE_LIST = 32,           /* HittableList                                    hittable_list.rs:14                       */
  RTB_NODE_BVH = 33             /* BVHNode::construct2(list,t0,t1): same closest-hit semantics as LIST (the reference's
                                   builder drops objects, bvh.rs:86,108 — not replicated)                                   */
} rtb_node_type;

typedef struct rtb_node {
  uint32_t type;        /* rtb_node_type */
  uint32_t material;    /* index into materials[], RTB_NONE for wrappers/lists */
  uint32_t first_child; /* index into child_index[] */
  uint32_t n_children;
  double p[12];         /* constructor arguments, f64 like the reference (vec3.rs:7) */
} rtb_node;

typedef enum rtb_material_type {
  RTB_MAT_LAMBERTIAN = 0,    /* material.rs:24-72    texture = albedo             */
  RTB_MAT_METAL = 1,         /* material.rs:74-108   texture = albedo (solid), param = fuzz (clamped to <=1) */
  RTB_MAT_DIELECTRIC = 2,    /* material.rs:110-156  param = index of refraction  */
  RTB_MAT_DIFFUSE_LIGHT = 3, /* material.rs:158-191  texture = emit               */
  RTB_MAT_ISOTROPIC = 4      /* material.rs:193-220 (commented in the reference; book-3 form, SURVEY §8a M6) */
} rtb_material_type;

typedef struct rtb_material {
  uint32_t type;
  uint32_t texture;
  double param;
} rtb_material;

typedef enum rtb_texture_type {
  RTB_TEX_SOLID = 0,   /* texture.rs:12-38   rgb                                    */
  RTB_TEX_CHECKER = 1, /* texture.rs:40-69   even/odd = texture indices             */
  RTB_TEX_NOISE = 2,   /* texture.rs:71-96   scale, table = perlin table id         */
  RTB_TEX_IMAGE = 3    /* texture.rs:98-141  table = image id (RTB_NONE => cyan)    */
} rtb_texture_type;

typedef struct rtb_texture {
  uint32_t type;
  uint32_t even, odd; /* checker children */
  uint32_t table;     /* perlin or image id */
  double rgb[3];
  double scale;
} rtb_texture;

/* ---- flat records ---------------------------------------------------------------------------------------- */
#define RTB_PRIM_FLIP_FACE   1u /* FlipFace: front_face toggled, normal untouched         hittable.rs:195-201 */
#define RTB_PRIM_FORCE_FRONT 2u /* wrapped by a Translate: front_face = true                 hittable.rs:82-83
                                   (the flat API has no rotation record: RotateY's object-ray / world-normal
                                   front_face, hittable.rs:173, is reproduced for scene-graph input only) */

typedef enum rtb_light_type { RTB_LIGHT_XZ_RECT = 0, RTB_LIGHT_SPHERE = 1 } rtb_light_type;
/* the only two Hittables with pdf_value/random (aarect.rs:107-125, sphere.rs:75-90) */
typedef struct rtb_light {
  uint32_t type;
  uint32_t _pad;
  double p[5]; /* XZ_RECT: x0 x1 z0 z1 k ; SPHERE: cx cy cz r */
} rtb_light;

typedef enum rtb_boundary_type { RTB_BOUNDARY_SPHERE = 0, RTB_BOUNDARY_BOX = 1 } rtb_boundary_type;
typedef struct rtb_medium { /* flat form of ConstantMedium (convex boundaries only, as in the reference) */
  uint32_t boundary_type;
  uint32_t material;  /* Isotropic */
  uint32_t prim_id;
  uint32_t _pad;
  double density;
  double p[6];        /* SPHERE: cx cy cz r ; BOX: object-space p0[3] p1[3] */
  double rot_y_deg;   /* BOX: object->world = translate(offset) * rotate_y(rot_y_deg) */
  double offset[3];
} rtb_medium;

/* ---- camera / params / stats ----------------------------------------------------------------------------- */
typedef struct rtb_camera { /* Camera::new arguments, camera.rs:21-28 */
  double lookfrom[3], lookat[3], vup[3];
  double vfov_deg, aspect_ratio, aperture, focus_dist;
  double time0, time1;
} rtb_camera;

typedef struct rtb_params {
  uint32_t width, height;
  uint32_t spp;            /* samples per pixel rendered by THIS call */
  uint32_t sample_offset;  /* global index of the first sample (multi-GPU: rank * spp); keys the Philox stream */
  uint32_t total_spp;      /* spp over all ranks (informational; finalize divides by it) */
  int32_t max_depth;       /* MAX_DEPTH, main.rs:663 */
  uint32_t rr_start_depth; /* Russian roulette after this many segments; 0 = off (reference behaviour) */
  uint32_t seed;
  float background[3];     /* main.rs:692 */
  uint32_t pool_paths;     /* path-pool slots, all wavefront lanes together; 0 = default (sized to the device) */
  uint32_t flags;          /* RTB_RENDER_* */
} rtb_params;
#define RTB_RENDER_ACCUMULATE 1u  /* add into the accumulation buffer instead of clearing it first */
#define RTB_RENDER_COUNT 2u       /* instrumented extend: fills stats->nodes_visited / prims_tested (slower) */
#define RTB_RENDER_TIME_EXTEND 4u /* CUDA events around every extend launch: fills stats->ms_extend */
#define RTB_RENDER_REDUCE 8u      /* rtb_render_device on a context with a communicator (rtb_context_comm_init): after the
                                     render, the library sums the ranks' accumulation buffers onto rank 0 with ONE
                                     ncclReduce(float32, 4 W H, sum, root 0) on `stream`; its time goes to stats->ms_nccl */

typedef struct rtb_stats {
  uint64_t paths;          /* camera paths started */
  uint64_t segments;       /* world.hit queries (main.rs:74) issued by the integrator */
  uint64_t rejected;       /* samples rejected because non-finite (per-sample NaN scrub, SURVEY App. A #10) */
  uint64_t iterations;     /* wavefront iterations */
  uint64_t launches;       /* kernels launched by this call */
  uint64_t extend_launches;
  double ms_total;         /* device time of the whole call (CUDA events) */
  double ms_extend;        /* summed device time of the extend launches (RTB_RENDER_TIME_EXTEND, else 0) */
  uint64_t nodes_visited;  /* BVH nodes fetched / primitives tested by extend (RTB_RENDER_COUNT or the probes, else 0) */
  uint64_t prims_tested;
  uint64_t exact_rays;     /* rays whose closest hit f32 rounding left open and that were re-traced with the reference's f64 arithmetic */
  uint64_t refined_rays;   /* certain hits (grazing spheres) whose distance was recomputed in f64 */
  double ms_nccl;          /* device time of the framebuffer reduce on this rank / on device 0 (0 on one GPU) */
  double ms_render;        /* multi-device context: slowest device's render time (ms_total = ms_render + ms_nccl) */
  uint32_t n_devices;      /* GPUs that took part in this call */
  uint32_t _pad;
  uint64_t prims_tested_type[4]; /* prims_tested per type: sphere, moving sphere, quad, triangle */
  double ms_nccl_wait;     /* one process per GPU: time this rank waited for the others to arrive at the reduce (render skew) */
} rtb_stats;

typedef struct rtb_context rtb_context;
typedef struct rtb_scene rtb_scene;

/* ---- context --------------------------------------------------------------------------------------------- */
uint32_t rtb_abi_version(void);
const char* rtb_last_error(void);
int rtb_context_create(int device_id, rtb_context** out);
void rtb_context_destroy(rtb_context* ctx);
int rtb_context_device_info(rtb_context* ctx, int* sm_count, int* l2_bytes, int* clock_khz, char* name, size_t name_cap);

/* ---- multi-GPU: the only parallelism of the reference is its per-pixel thread fan-out (main.rs:730-778); here the
 * samples of every pixel are split across the GPUs of one box and the float4 accumulation buffers are summed by the
 * LIBRARY with one NCCL reduce per frame (NVLink 5 / NVSwitch).  Philox streams are keyed by the GLOBAL sample index, so
 * the sample set does not depend on the number of GPUs.  NCCL (libnccl.so.2) is bound at run time: single-GPU callers
 * do not need it.
 *   (a) one process drives n GPUs: rtb_context_create_multi(ids, n) -> ncclCommInitAll.  The SAME calls then work on that
 *       context: scenes are uploaded to every device, rtb_render renders spp / n samples on each (remainder to the
 *       lowest ranks), reduces onto device ids[0] and returns that buffer; stats aggregate all devices.
 *   (b) one process per GPU (torchrun, MPI): rank 0 calls rtb_comm_unique_id and hands the 128 bytes to the others by
 *       any means; every rank calls rtb_context_comm_init; rtb_render_device(..., RTB_RENDER_REDUCE) then reduces. */
#define RTB_COMM_ID_BYTES 128
int rtb_context_create_multi(const int* device_ids, int n_devices, rtb_context** out);
int rtb_context_device_count(rtb_context* ctx);
int rtb_comm_unique_id(uint8_t* id_128_bytes);
int rtb_context_comm_init(rtb_context* ctx, const uint8_t* id_128_bytes, int rank, int n_ranks);

/* ---- scene: tables ---------------------------------------------------------------------------------------- */
/* ctx may be NULL: a host-only scene that can be flattened, built and exported but not committed/rendered */
int rtb_scene_create(rtb_context* ctx, rtb_scene** out);
void rtb_scene_destroy(rtb_scene* scene);
int rtb_scene_set_materials(rtb_scene* s, const rtb_material* mats, uint32_t n);
int rtb_scene_set_textures(rtb_scene* s, const rtb_texture* tex, uint32_t n);
int rtb_scene_set_image(rtb_scene* s, uint32_t image_id, const uint8_t* rgb, uint32_t width, uint32_t height);
int rtb_scene_set_perlin(rtb_scene* s, uint32_t table_id, const double* ranvec_256x3, const uint32_t* perm_x,
                         const uint32_t* perm_y, const uint32_t* perm_z);
int rtb_scene_set_mesh(rtb_scene* s, uint32_t mesh_id, const float* vertices_xyz, uint32_t n_vertices,
                       const uint32_t* indices, uint32_t n_triangles);
int rtb_scene_set_lights(rtb_scene* s, const rtb_light* lights, uint32_t n);
/* Limits (RTB_ERR_UNSUPPORTED beyond them): at most 8 entries in the light list and 8 ConstantMedium objects per scene (both
 * live in the kernels' constant bank: every shaded hit walks the light list, every ray tests every medium boundary; the
 * reference's scenes have <= 2 of each); a ConstantMedium's boundary is a Sphere or a Box, optionally under
 * Translate / RotateY; checker textures nest at most 8 deep.  Any number of image / perlin tables, textures, materials,
 * primitives (per type < 2^29) and wrapper levels (< 256). */

/* ---- scene: geometry, way 1 (graph records; replaces the reference's trait-object world, main.rs:668) ------ */
int rtb_scene_set_graph(rtb_scene* s, const rtb_node* nodes, uint32_t n_nodes, const uint32_t* child_index,
                        uint32_t n_child_index, uint32_t root);

/* ---- scene: geometry, way 2 (flat SoA; array order irrelevant, prim_id carries the list order) ------------- */
int rtb_scene_set_spheres(rtb_scene* s, const float* center_radius_4, const uint32_t* material, const uint32_t* flags,
                          const uint32_t* prim_id, uint32_t n);
int rtb_scene_set_moving_spheres(rtb_scene* s, const float* c0_radius_4, const float* c1_3, const float* time01_2,
                                 const uint32_t* material, const uint32_t* flags, const uint32_t* prim_id, uint32_t n);
int rtb_scene_set_quads(rtb_scene* s, const float* q_3, const float* u_3, const float* v_3, const uint32_t* material,
                        const uint32_t* flags, const uint32_t* prim_id, uint32_t n);
int rtb_scene_set_triangles(rtb_scene* s, const float* v0_3, const float* v1_3, const float* v2_3,
                            const uint32_t* material, const uint32_t* flags, const uint32_t* prim_id, uint32_t n);
int rtb_scene_set_media(rtb_scene* s, const rtb_medium* media, uint32_t n);

/* BVH builder quality knobs (README.md:150-152 of the reference asks for an accelerated mesh path; defaults = what the
 * benchmarks use).  Results never depend on them (closest-hit semantics stay those of the list scan), only speed. */
typedef struct rtb_build_options {
  uint32_t max_leaf_triangles;   /* triangles per leaf slot, 1..3 (default 2: halves the node count of large meshes) */
  uint32_t keep_huge_primitives_out; /* default 1: primitives whose box is >= 80 % of the scene box are tested first for
                                        every ray instead of coarsening the quantisation grid of the node that holds them */
  float open_min_extent;         /* default 0.125: the collapse to 8-wide nodes never opens a subtree smaller than this
                                    fraction of the node's extent (keeps the 7-bit child boxes tight) */
  uint32_t _reserved;
} rtb_build_options;
int rtb_scene_set_build_options(rtb_scene* s, const rtb_build_options* opt);
/* build the wide BVH (width 8, quantised child boxes) on the host; replaces BVHNode::construct2 (bvh.rs:74-130) */
int rtb_scene_build_bvh(rtb_scene* s);
/* build if needed, then upload everything to the device */
int rtb_scene_commit(rtb_scene* s);

/* ---- introspection (used by the test harness to drive the oracle over the SAME flattened scene / BVH) ------ */
typedef struct rtb_scene_info {
  uint32_t n_spheres, n_moving, n_quads, n_triangles, n_media, n_lights, n_materials, n_textures;
  uint32_t n_prims;      /* size of the primitive-id space */
  uint32_t n_bvh_nodes;  /* 80-byte nodes */
  uint32_t bvh_width;
  uint32_t bvh_max_depth;
  uint64_t bvh_bytes, prim_bytes;
  uint32_t global_f64_mask; /* bit k: global primitive k is a sphere so large next to the rest of the scene that it is tested in f64 */
  uint32_t _pad;
} rtb_scene_info;
int rtb_scene_get_info(rtb_scene* s, rtb_scene_info* out);
/* copies out the leaf-ordered device layout: geometry as float4 words + (prim_id, material|flags<<24) pairs */
int rtb_scene_export_bvh(rtb_scene* s, void* nodes_80B, size_t cap_bytes);
/* primitives kept out of the tree and tested first for every ray: refs = type << 29 | index into that type's arrays */
int rtb_scene_export_globals(rtb_scene* s, uint32_t* refs, uint32_t cap, uint32_t* n_out);
int rtb_scene_export_prims(rtb_scene* s, uint32_t type /*0 sphere 1 moving 2 quad 3 triangle*/, float* geom,
                           size_t geom_cap_bytes, uint32_t* info_pairs, size_t info_cap_bytes);
/* leaf-ordered reference-exact records (16 doubles per sphere / moving sphere / quad; none for triangles): the
 * constructor's f64 arguments + its Translate/RotateY chain, on which the device re-decides every closest-hit
 * comparison that f32 rounding leaves open (sphere.rs:41-65, aarect.rs:31-48, hittable.rs:76-85,147-176).  Also the
 * two rounding scales of the f32 quad test.  Any pointer may be NULL. */
int rtb_scene_export_exact(rtb_scene* s, uint32_t type, double* records, size_t cap_bytes, float* coord_max,
                           float* eps_ab);

/* ---- the hot path ------------------------------------------------------------------------------------------ */
/* Renders params->spp samples of every pixel into the context's float4 accumulation buffer
 * (sum R, sum G, sum B, sum Y^2 per pixel; row 0 = top).  Replaces main.rs:731-784 + ray_color.
 * rtb_render: host-facing; if accum_out != NULL copies W*H*4 floats back to the host buffer. */
int rtb_render(rtb_context* ctx, rtb_scene* scene, const rtb_camera* cam, const rtb_params* params, float* accum_out,
               rtb_stats* stats);
/* rtb_render_device: device-facing; d_accum is a DEVICE pointer to W*H*4 floats owned by the caller (e.g. a torch
 * tensor that is then reduced with NCCL), stream is a cudaStream_t (NULL = default stream).  Asynchronous w.r.t.
 * the host only up to the internal termination checks; on return the work is complete on `stream`. */
int rtb_render_device(rtb_context* ctx, rtb_scene* scene, const rtb_camera* cam, const rtb_params* params,
                      void* d_accum, void* stream, rtb_stats* stats);
/* ---- denoiser guide buffers (AOVs, "arbitrary output variables") ------------------------------------------------------
 * Albedo, normal and depth images of the same sample set a render with the same rtb_params draws: global sample indices
 * [sample_offset, sample_offset + spp) of every pixel.  Sample s of pixel p traces exactly the FIRST ray of that render
 * sample (the same jitter, thin-lens and shutter-time draws), and its closest hit comes from the render's own extend
 * kernels, including the exact f64 pass.  A ConstantMedium decides its scatter distance from the path's own stream at
 * segment 1, as in the render.  Denoisers (OIDN, the OptiX denoiser) take these as guides of a low-spp render.
 *
 * Output: 8 floats per pixel, (H, W, 8) float32, row 0 = top.  Each value is a SUM over samples, like the accumulation
 * buffer, so calls compose with sample_offset, RTB_RENDER_ACCUMULATE and a caller's own reduce across ranks:
 *   [0..2] albedo, each channel clamped to [0, 1]:
 *            Lambertian, Metal, Isotropic: the texture value at the hit (the attenuation the integrator applies);
 *            Dielectric: (1, 1, 1); DiffuseLight: the emitted colour on its front face, else 0; a miss: params->background
 *   [3]    coverage: 1 if the ray hit a surface or scattered in a medium, else 0
 *   [4..6] shading normal: world space, unit length, facing the ray (the normal the integrator scatters about, including
 *          RotateY's front_face rule, hittable.rs:173); (0, 0, 0) for a medium scatter or a miss
 *   [7]    depth: t * |d|, the distance from the ray origin (the lens point) to the hit or scatter point; 0 for a miss
 * Divide albedo, coverage and normal by spp and depth by the coverage sum.  A sample with a non-finite value is skipped
 * and counted in stats->rejected.  stats->paths = stats->segments = W * H * spp.
 * Arguments are checked as by rtb_render_device; the only accepted flag is RTB_RENDER_ACCUMULATE.  A multi-device context
 * returns RTB_ERR_UNSUPPORTED: split the samples over per-device contexts with sample_offset and sum the buffers.
 * rtb_render_aov_device: d_aov is a DEVICE pointer to W*H*8 floats, stream a cudaStream_t (NULL = default stream); on
 * return the work is complete on `stream`.
 * rtb_render_aov: into the context's own buffer; if aov_out != NULL copies W*H*8 floats back to the host. */
int rtb_render_aov_device(rtb_context* ctx, rtb_scene* scene, const rtb_camera* cam, const rtb_params* params, void* d_aov,
                          void* stream, rtb_stats* stats);
int rtb_render_aov(rtb_context* ctx, rtb_scene* scene, const rtb_camera* cam, const rtb_params* params, float* aov_out,
                   rtb_stats* stats);
/* write_color (main.rs:141-169): /total_spp, NaN->0, sqrt, clamp [0,0.999], *256 -> u8.  d_accum device, rgb8_out host. */
int rtb_finalize_rgb8(rtb_context* ctx, const void* d_accum, uint32_t width, uint32_t height, uint32_t total_spp,
                      uint8_t* rgb8_out);
/* parity probe: closest hit of the pixel-centre primary rays (jitter 0.5, lens centre, time = time0).
 * prim_id_out[j*W+i] = primitive id or RTB_NONE, t_out = hit distance in the (un-normalised) ray parametrisation. */
int rtb_primary_hits(rtb_context* ctx, rtb_scene* scene, const rtb_camera* cam, uint32_t width, uint32_t height,
                     uint32_t* prim_id_out, float* t_out, rtb_stats* stats);
/* closest hit of caller-supplied rays (origin xyz, direction xyz, time): unit-level probe of `extend`. */
int rtb_trace_rays(rtb_context* ctx, rtb_scene* scene, const float* origin_3, const float* direction_3,
                   const float* time, uint32_t n, uint32_t* prim_id_out, float* t_out, rtb_stats* stats);

/* the f32 rays rtb_primary_hits traces (generated in f64 like camera.rs:60-70, rounded once): lets a checker trace
 * exactly the same rays.  origin_3 / direction_3: W*H*3 floats, time: W*H floats (host). */
int rtb_primary_rays(rtb_context* ctx, const rtb_camera* cam, uint32_t width, uint32_t height, float* origin_3,
                     float* direction_3, float* time);

/* ---- tier-U2 test hook: evaluates ONE device function per item on caller-supplied inputs ----------------------- */
/* in / out are raw 32-bit words (floats by bit pattern).  scene may be NULL for ops that need no tables; cam / params may
 * be NULL except for RTB_KAT_CAMERA_RAY.  See rtb_kernels.cu:k_kat for each op's word layout. */
typedef enum rtb_kat_op {
  RTB_KAT_PHILOX = 0,        /* rt_weekend.rs:8-19 replacement: Philox4x32-10 words, bit-exact against the oracle      */
  RTB_KAT_SPHERE = 1,        /* sphere.rs:41-65 (f32 form + error bound)                                                */
  RTB_KAT_SPHERE_F64 = 2,    /* sphere.rs:41-65 (f64 form used for global spheres)                                      */
  RTB_KAT_LIGHTS_PDF = 3,    /* hittable_list.rs:73-80, aarect.rs:107-117, sphere.rs:75-84                              */
  RTB_KAT_LIGHTS_RANDOM = 4, /* hittable_list.rs:81-84, aarect.rs:118-125, sphere.rs:85-90, pdf.rs:82-91                */
  RTB_KAT_PERLIN_NOISE = 5,  /* perlin.rs:26-52,67-85                                                                   */
  RTB_KAT_PERLIN_TURB = 6,   /* perlin.rs:86-98                                                                         */
  RTB_KAT_Q2F = 7,           /* BVH plane-byte decode                                                                   */
  RTB_KAT_ONB = 8,           /* onb.rs:19-30                                                                            */
  RTB_KAT_REFLECT = 9,       /* vec3.rs:115-117                                                                         */
  RTB_KAT_REFRACT = 10,      /* vec3.rs:246-251                                                                         */
  RTB_KAT_CAMERA_RAY = 11,   /* camera.rs:60-70 + main.rs:752-753                                                       */
  RTB_KAT_MEDIA = 12,        /* constant_medium.rs:31-71                                                                */
  RTB_KAT_TEXTURE = 13,      /* texture.rs:61-68,91-95,118-140                                                          */
  RTB_KAT_EXACT = 14         /* the reference-exact f64 primitive test (exact_hit)                                      */
} rtb_kat_op;
int rtb_device_kat(rtb_context* ctx, rtb_scene* scene, const rtb_camera* cam, const rtb_params* params, uint32_t op,
                   const uint32_t* in_words, uint32_t n_items, uint32_t in_stride, uint32_t* out_words,
                   uint32_t out_stride);

/* RTB_CHECKED build of the library (make -C csrc checked): failed device-side bounds assertions by kind (traversal stack,
 * node index, primitive index, pool slot, fix-up queue, chunk list, 2 spare); every entry is 0xFFFFFFFF in a normal build. */
int rtb_debug_check_failures(rtb_context* ctx, uint32_t* out_8);

/* ---- measurement: the physical bandwidths the extend kernel's roofline is quoted against -------------------------- */
typedef enum rtb_bw_kind {
  RTB_BW_L2_READ = 0,     /* 128-bit ld.global.nc over a 48 MB (L2-resident) buffer, read-only */
  RTB_BW_HBM_READ = 1,    /* the same over a 2 GB buffer (streams from HBM)                    */
  RTB_BW_SHARED_READ = 2  /* 128-bit shared-memory loads, all SMs (where staged nodes come from) */
} rtb_bw_kind;
/* best of `repeats` timed launches, GB/s (1e9 bytes per second) */
int rtb_measure_bandwidth(rtb_context* ctx, uint32_t kind, uint32_t repeats, double* gb_per_s);

#ifdef __cplusplus
}
#endif
#endif /* RTB200_H */
