// rtb_internal.hpp — host-side data model of librtb200: the flattened scene (SoA primitives in primitive-id order),
// the wide BVH, and the device layout they are uploaded to.  No oracle code is reachable from here.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/rtb200.h"

namespace rtb {

enum PrimType : uint32_t { PT_SPHERE = 0, PT_MOVING = 1, PT_QUAD = 2, PT_TRI = 3, PT_MEDIUM = 4, PT_COUNT = 4 };
// hit reference written by `extend`: type << 29 | index into the leaf-ordered array of that type
static const uint32_t REF_TYPE_SHIFT = 29u;
static const uint32_t REF_INDEX_MASK = (1u << REF_TYPE_SHIFT) - 1u;
static const uint32_t REF_MISS = 0xFFFFFFFFu;
#define RTB_MAX_GLOBALS 16

// face-orientation modes: how Translate/RotateY/FlipFace wrappers rewrite front_face (hittable.rs:82-83,173,199)
// front_face of the hit record as the reference's wrapper chain leaves it (flatten.cpp: eval_face).  q = the value
// RotateY::hit computes by testing the OBJECT-space ray against the WORLD-space normal (hittable.rs:173);
// FACE_BARE: no Translate outside that RotateY re-oriented the normal, so the normal itself is q ? n : -n.
enum FaceMode : uint32_t { FACE_NATURAL = 0, FACE_FLIPPED = 1, FACE_TRUE = 2, FACE_FALSE = 3, FACE_Q = 4, FACE_NOT_Q = 5,
                           FACE_BARE = 8 };

struct Float3 { float x, y, z; };

struct HostPrim {      // one flattened primitive, any type
  uint32_t type;       // PrimType
  uint32_t prim_id;    // list-order id (hittable_list.rs:43-49)
  uint32_t material;
  uint32_t face_mode;  // FaceMode
  float g[12];         // device geometry words: sphere (c,r); moving (A,r)(B,0); quad plane form; triangle v0,v1,v2
  float lo[3], hi[3];  // bounds (padded)
  uint32_t exact;      // index into HostScene::exact (RTB_NONE for triangles: their f32 vertices ARE the exact record)
  uint32_t plane_exact;  // quad: axis-aligned and its plane constant is exactly a float (info word bit 31)
  uint32_t attr;         // triangle: index into HostScene::attrs (RTB_NONE: flat shading)
};

// Shading record of a mesh triangle with vertex normals and / or texture coordinates (rtb_scene_set_mesh_attributes),
// 16 floats: [0..2] n0 [3] u0 [4..6] n1 [7] u1 [8..10] n2 [11] u2 [12] v0 [13] v1 [14] v2 [15] flags (bits).  Normals are
// world-space unit vectors.  The device reads it as four float4 words (surface_at<ATTR>, rtb_kernels.cu).
#define RTB_ATTR_FLOATS 16
enum AttrFlags : uint32_t { ATTR_NORMALS = 1u, ATTR_UVS = 2u };
struct AttrRec { float f[RTB_ATTR_FLOATS]; };

// Reference-exact record of one sphere / moving sphere / quad: the constructor's own f64 arguments in OBJECT space plus
// the wrapper chain the reference evaluates per ray (Translate outside RotateY, hittable.rs:76-85,147-176).  The device
// falls back to the reference's literal f64 arithmetic on these whenever an f32 decision is within its rounding bound
// (exact_hit, rtb_device.cuh), so closest-hit ids equal the f64 linear scan's on identical rays.
// Layout (16 doubles): [0] bits: xform flags | subtype << 8 ; [1..3] Translate offset ; [4] sin ; [5] cos ;
//   sphere [6..8] c [9] r ; moving [6..8] c0 [9..11] c1 [12] t0 [13] t1 [14] r ;
//   rect (subtype = normal axis 0..2) [6] k [7] a0 [8] a1 [9] b0 [10] b1 ; general quad (subtype 3) [6..8] Q [9..11] u [12..14] v
#define RTB_EXACT_STRIDE 16
enum ExactFlags : uint32_t { EX_TRANSLATE = 1u, EX_ROTATE = 2u, EX_QUAD_GENERAL = 3u };
struct ExactRec { double v[RTB_EXACT_STRIDE]; };

struct HostMedium {
  uint32_t boundary_type, material, prim_id;
  float neg_inv_density;
  float p[6];          // sphere: c, r ; box: object-space p0,p1
  float sin_t, cos_t;  // box: object->world rotation about y
  float offset[3];
};

struct HostLight { uint32_t type; float p[5]; };

#pragma pack(push, 1)
struct Node8 {  // 80 bytes, five 16-byte words; see DESIGN.md "BVH8 node"
  float ox, oy, oz;
  uint8_t ex, ey, ez, imask;  // biased exponents of the per-axis quantisation step; bit i of imask: child i is internal
  uint32_t child_base;        // node index of the first internal child (internal children contiguous, slot order)
  uint32_t prim_base;         // type << 29 | index of the node's first leaf primitive (leaf-ordered array of that type)
  uint8_t meta[8];            // leaf child: count << 5 | offset from prim_base ; internal/empty: 0
  uint8_t qlo[3][8];
  uint8_t qhi[3][8];
};
#pragma pack(pop)
static_assert(sizeof(Node8) == 80, "Node8 must be 80 bytes");

struct HostBvh {
  std::vector<Node8> nodes;
  // leaf-ordered primitive arrays per type: geometry words and (prim_id, material | face_mode << 24)
  std::vector<float> geom[PT_COUNT];
  std::vector<uint32_t> info[PT_COUNT];
  uint32_t max_depth = 0;
  std::vector<uint32_t> global_refs;  // type << 29 | leaf index of the primitives tested before the traversal
  // leaf-ordered reference-exact records (RTB_EXACT_STRIDE doubles per sphere / moving sphere / quad) and the scene's
  // rounding scales of the f32 quad test (rtb_device.cuh: DevScene::coord_max, eps_ab)
  std::vector<double> exact[PT_COUNT];
  float coord_max = 0.f, eps_ab = 0.f;
  uint32_t global_f64 = 0;  // bit k: global k is a sphere tested in f64 directly (DevScene::global_f64)
  // leaf-ordered shading records of the triangles (RTB_ATTR_FLOATS per triangle); empty when no triangle has attributes
  std::vector<float> attr;
};

static inline uint32_t geom_words(uint32_t type) { return type == PT_SPHERE ? 4u : (type == PT_MOVING ? 8u : 12u); }

struct HostScene {
  std::vector<HostPrim> prims;
  std::vector<HostMedium> media;
  std::vector<HostLight> lights;
  std::vector<rtb_material> materials;
  std::vector<rtb_texture> textures;
  struct Image { std::vector<uint8_t> rgb; uint32_t w = 0, h = 0; };
  std::vector<Image> images;
  struct Perlin { std::vector<float> ranvec; std::vector<uint8_t> perm; bool set = false; };  // 256x4 floats, 3x256 bytes
  std::vector<Perlin> perlins;
  // normals: unit f32 vectors (normalised in f64) and their per-corner indices; uvs likewise (empty: no such stream)
  struct Mesh {
    std::vector<float> verts; std::vector<uint32_t> idx;
    std::vector<float> normals; std::vector<uint32_t> normal_idx;
    std::vector<float> uvs; std::vector<uint32_t> uv_idx;
  };
  std::vector<Mesh> meshes;
  std::vector<ExactRec> exact;
  std::vector<AttrRec> attrs;  // shading records of mesh triangles (HostPrim::attr)
  uint32_t n_prim_ids = 0;
  // BVH builder quality knobs (rtb_scene_set_build_options)
  uint32_t opt_max_leaf_tris = 2;   // triangles per leaf slot, 1..3
  uint32_t opt_globals = 1;         // keep scene-dominating primitives out of the tree
  float opt_open_min_rel = 0.125f;  // collapse: never open a subtree smaller than this fraction of the node's extent
};

// flatten.cpp
int flatten_graph(HostScene& hs, const rtb_node* nodes, uint32_t n_nodes, const uint32_t* child_index,
                  uint32_t n_child_index, uint32_t root, std::string& err);
// wrapper chain of a primitive as the reference evaluates it: [Translate(offset)] outside [RotateY(sin, cos)]
struct ExactXform { uint32_t flags = 0; double off[3] = {0, 0, 0}; double sin_t = 0, cos_t = 1; };
uint32_t add_exact(HostScene& hs, const ExactXform& x, uint32_t subtype, const double* params, int n_params);
void pack_sphere(HostPrim& p, const double c[3], double r);
void pack_moving(HostPrim& p, const double c0[3], const double c1[3], double t0, double t1, double r);
void pack_quad(HostPrim& p, const double Q[3], const double u[3], const double v[3], const double* outward_or_null);
void pack_tri(HostPrim& p, const double v0[3], const double v1[3], const double v2[3]);

// bvh_build.cpp
int build_bvh8(const HostScene& hs, HostBvh& out, std::string& err);

}  // namespace rtb
