// rtb200_scene.hpp — header-only C++ mirror of the reference's scene-construction API
// (raytracer/src/{sphere,moving_sphere,aarect,boxes,hittable,hittable_list,bvh,constant_medium,material,texture}.rs).
//
// The reference is Rust and no Rust toolchain exists in the build image, so the host side above the C ABI is C++:
// same type names, constructor names (`X::construct(...)`), argument order and meaning as the Rust code, so the
// reference's scene functions (main.rs:337-433 cornell_box, :171-242 random_scene, :521-649 final_scene) port line by
// line.  Instead of building trait objects, every constructor records one `rtb_node` / `rtb_material` / `rtb_texture`
// (include/rtb200.h); `SceneRecords::upload()` hands them to librtb200, whose host C++ flattens the graph and builds
// the BVH.  The Rust shim in INTEGRATION.md does exactly the same from Rust.
#pragma once
#include <array>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "rtb200.h"

namespace rtb200 {

using Vec3 = std::array<double, 3>;  // vec3.rs:7
using Point3 = Vec3;
using Color3 = Vec3;

// ------------------------------------------------------------------------------------------------ textures
struct Texture { virtual ~Texture() = default; };                       // texture.rs:7-9
struct SolidColor : Texture {                                           // texture.rs:12-38
  Color3 color_value;
  static std::shared_ptr<SolidColor> construct(const Color3& c) { auto t = std::make_shared<SolidColor>(); t->color_value = c; return t; }
};
struct CheckerTexture : Texture {                                       // texture.rs:40-69
  std::shared_ptr<Texture> even, odd;
  static std::shared_ptr<CheckerTexture> construct_color(const Color3& c1, const Color3& c2) {
    auto t = std::make_shared<CheckerTexture>(); t->even = SolidColor::construct(c1); t->odd = SolidColor::construct(c2); return t;
  }
};
struct NoiseTexture : Texture {                                         // texture.rs:71-96; tables from the caller's RNG
  double scale = 1.0;
  std::vector<double> ranvec;            // 256 x 3 unit vectors (perlin.rs:14-25)
  std::vector<uint32_t> perm_x, perm_y, perm_z;
};
struct ImageTexture : Texture {                                         // texture.rs:98-141, RGB8 row-major from the top
  std::vector<uint8_t> data; uint32_t width = 0, height = 0;
  static std::shared_ptr<ImageTexture> construct(const std::vector<uint8_t>& d, uint32_t w, uint32_t h) {
    auto t = std::make_shared<ImageTexture>(); t->data = d; t->width = w; t->height = h; return t;
  }
};

// ------------------------------------------------------------------------------------------------ materials
struct Material { virtual ~Material() = default; };                     // material.rs:11-21
struct Lambertian : Material {                                          // material.rs:24-72
  std::shared_ptr<Texture> albedo;
  static std::shared_ptr<Lambertian> construct(const Color3& a) { auto m = std::make_shared<Lambertian>(); m->albedo = SolidColor::construct(a); return m; }
  static std::shared_ptr<Lambertian> construct_texture(std::shared_ptr<Texture> a) { auto m = std::make_shared<Lambertian>(); m->albedo = std::move(a); return m; }
};
struct Metal : Material {                                               // material.rs:74-108 (fuzz clamped to 1)
  Color3 albedo; double fuzz;
  static std::shared_ptr<Metal> construct(const Color3& a, double f) { auto m = std::make_shared<Metal>(); m->albedo = a; m->fuzz = f < 1.0 ? f : 1.0; return m; }
};
struct Dielectric : Material {                                          // material.rs:110-156
  double ir;
  static std::shared_ptr<Dielectric> construct(double ir) { auto m = std::make_shared<Dielectric>(); m->ir = ir; return m; }
};
struct DiffuseLight : Material {                                        // material.rs:158-191
  std::shared_ptr<Texture> emit;
  static std::shared_ptr<DiffuseLight> construct_color(const Color3& c) { auto m = std::make_shared<DiffuseLight>(); m->emit = SolidColor::construct(c); return m; }
};
struct Isotropic : Material {                                           // material.rs:193-220 (commented in the reference)
  std::shared_ptr<Texture> albedo;
  static std::shared_ptr<Isotropic> construct_color(const Color3& c) { auto m = std::make_shared<Isotropic>(); m->albedo = SolidColor::construct(c); return m; }
};

// ------------------------------------------------------------------------------------------------ hittables
struct Hittable { virtual ~Hittable() = default; };                     // hittable.rs:51-60
using HittablePtr = std::shared_ptr<Hittable>;
using MaterialPtr = std::shared_ptr<Material>;

struct Sphere : Hittable {                                              // sphere.rs:19-25
  Point3 center; double radius; MaterialPtr mat_ptr;
  static std::shared_ptr<Sphere> construct(const Point3& c, double r, MaterialPtr m) { auto s = std::make_shared<Sphere>(); s->center = c; s->radius = r; s->mat_ptr = std::move(m); return s; }
};
struct MovingSphere : Hittable {                                        // moving_sphere.rs:18-34
  Point3 center0, center1; double time0, time1, radius; MaterialPtr mat_ptr;
  static std::shared_ptr<MovingSphere> construct(const Point3& c0, const Point3& c1, double t0, double t1, double r, MaterialPtr m) {
    auto s = std::make_shared<MovingSphere>(); s->center0 = c0; s->center1 = c1; s->time0 = t0; s->time1 = t1; s->radius = r; s->mat_ptr = std::move(m); return s;
  }
};
struct AARect : Hittable { uint32_t node_type; double a0, a1, b0, b1, k; MaterialPtr mp; };
#define RTB200_RECT(NAME, TYPE)                                                                                   \
  struct NAME : AARect {                                                                                          \
    static std::shared_ptr<NAME> construct(double a0, double a1, double b0, double b1, double k, MaterialPtr m) { \
      auto r = std::make_shared<NAME>(); r->node_type = TYPE; r->a0 = a0; r->a1 = a1; r->b0 = b0; r->b1 = b1;     \
      r->k = k; r->mp = std::move(m); return r;                                                                   \
    }                                                                                                             \
  };
RTB200_RECT(XyRect, RTB_NODE_XY_RECT)                                   // aarect.rs:19-29
RTB200_RECT(XzRect, RTB_NODE_XZ_RECT)                                   // aarect.rs:69-79
RTB200_RECT(YzRect, RTB_NODE_YZ_RECT)                                   // aarect.rs:138-148
#undef RTB200_RECT
struct Box : Hittable {                                                 // boxes.rs:18-76
  Point3 box_min, box_max; MaterialPtr ptr;
  static std::shared_ptr<Box> construct(const Point3& p0, const Point3& p1, MaterialPtr m) { auto b = std::make_shared<Box>(); b->box_min = p0; b->box_max = p1; b->ptr = std::move(m); return b; }
};
struct Translate : Hittable {                                           // hittable.rs:62-74
  HittablePtr ptr; Vec3 offset;
  static std::shared_ptr<Translate> construct(HittablePtr p, const Vec3& d) { auto t = std::make_shared<Translate>(); t->ptr = std::move(p); t->offset = d; return t; }
};
struct RotateY : Hittable {                                             // hittable.rs:99-144 (angle in degrees)
  HittablePtr ptr; double angle;
  static std::shared_ptr<RotateY> construct(HittablePtr p, double angle) { auto r = std::make_shared<RotateY>(); r->ptr = std::move(p); r->angle = angle; return r; }
};
struct FlipFace : Hittable {                                            // hittable.rs:183-193
  HittablePtr ptr;
  static std::shared_ptr<FlipFace> construct(HittablePtr p) { auto f = std::make_shared<FlipFace>(); f->ptr = std::move(p); return f; }
};
struct ConstantMedium : Hittable {                                      // constant_medium.rs:8-29
  HittablePtr boundary; double density; MaterialPtr phase_function;
  static std::shared_ptr<ConstantMedium> construct_color(HittablePtr b, double d, const Color3& c) {
    auto m = std::make_shared<ConstantMedium>(); m->boundary = std::move(b); m->density = d; m->phase_function = Isotropic::construct_color(c); return m;
  }
};
struct HittableList : Hittable {                                        // hittable_list.rs:14-37
  std::vector<HittablePtr> objects;
  static std::shared_ptr<HittableList> new_() { return std::make_shared<HittableList>(); }
  void add(HittablePtr o) { objects.push_back(std::move(o)); }
};
struct BVHNode : Hittable {                                             // bvh.rs:74-76; closest-hit semantics of the list
  std::shared_ptr<HittableList> src;
  static std::shared_ptr<BVHNode> construct2(std::shared_ptr<HittableList> l, double, double) { auto b = std::make_shared<BVHNode>(); b->src = std::move(l); return b; }
};
struct TriangleMesh : Hittable {                                        // new (SURVEY §8a N1): OBJ-style indexed mesh
  std::vector<float> vertices; std::vector<uint32_t> indices; MaterialPtr mat_ptr;
  // optional smooth shading / texture coordinates (rtb_scene_set_mesh_attributes): xyz per normal, uv per texture
  // coordinate, each with its own per-corner indices (empty: the position indices)
  std::vector<float> normals; std::vector<uint32_t> normal_indices;
  std::vector<float> uvs; std::vector<uint32_t> uv_indices;
};

// ------------------------------------------------------------------------------------------------ records
struct SceneRecords {
  std::vector<rtb_node> nodes;
  std::vector<uint32_t> child_index;
  std::vector<rtb_material> materials;
  std::vector<rtb_texture> textures;
  std::vector<rtb_light> lights;
  std::vector<const ImageTexture*> images;
  std::vector<const NoiseTexture*> perlins;
  std::vector<const TriangleMesh*> meshes;
  uint32_t root = 0;

  uint32_t tex(const std::shared_ptr<Texture>& t) {
    auto it = tex_ids_.find(t.get());
    if (it != tex_ids_.end()) return it->second;
    keep_.push_back(t);
    rtb_texture r{};
    r.even = r.odd = r.table = RTB_NONE;
    if (auto s = dynamic_cast<SolidColor*>(t.get())) { r.type = RTB_TEX_SOLID; for (int i = 0; i < 3; ++i) r.rgb[i] = s->color_value[i]; }
    else if (auto c = dynamic_cast<CheckerTexture*>(t.get())) { r.type = RTB_TEX_CHECKER; r.even = tex(c->even); r.odd = tex(c->odd); }
    else if (auto n = dynamic_cast<NoiseTexture*>(t.get())) { r.type = RTB_TEX_NOISE; r.scale = n->scale; r.table = (uint32_t)perlins.size(); perlins.push_back(n); }
    else if (auto im = dynamic_cast<ImageTexture*>(t.get())) { r.type = RTB_TEX_IMAGE; if (!im->data.empty()) { r.table = (uint32_t)images.size(); images.push_back(im); } }
    else throw std::invalid_argument("unknown texture");
    textures.push_back(r);
    return tex_ids_[t.get()] = (uint32_t)textures.size() - 1;
  }
  uint32_t mat(const MaterialPtr& m) {
    auto it = mat_ids_.find(m.get());
    if (it != mat_ids_.end()) return it->second;
    keep_m_.push_back(m);
    rtb_material r{};
    if (auto l = dynamic_cast<Lambertian*>(m.get())) { r.type = RTB_MAT_LAMBERTIAN; r.texture = tex(l->albedo); }
    else if (auto me = dynamic_cast<Metal*>(m.get())) { r.type = RTB_MAT_METAL; r.texture = tex(SolidColor::construct(me->albedo)); r.param = me->fuzz; }
    else if (auto d = dynamic_cast<Dielectric*>(m.get())) { r.type = RTB_MAT_DIELECTRIC; r.texture = RTB_NONE; r.param = d->ir; }
    else if (auto dl = dynamic_cast<DiffuseLight*>(m.get())) { r.type = RTB_MAT_DIFFUSE_LIGHT; r.texture = tex(dl->emit); }
    else if (auto is = dynamic_cast<Isotropic*>(m.get())) { r.type = RTB_MAT_ISOTROPIC; r.texture = tex(is->albedo); }
    else throw std::invalid_argument("unknown material");
    materials.push_back(r);
    return mat_ids_[m.get()] = (uint32_t)materials.size() - 1;
  }
  uint32_t node(const HittablePtr& h) {
    rtb_node n{};
    n.material = RTB_NONE;
    std::vector<uint32_t> kids;
    auto set = [&](std::initializer_list<double> v) { int i = 0; for (double x : v) n.p[i++] = x; };
    if (auto s = dynamic_cast<Sphere*>(h.get())) { n.type = RTB_NODE_SPHERE; n.material = mat(s->mat_ptr); set({s->center[0], s->center[1], s->center[2], s->radius}); }
    else if (auto ms = dynamic_cast<MovingSphere*>(h.get())) { n.type = RTB_NODE_MOVING_SPHERE; n.material = mat(ms->mat_ptr);
      set({ms->center0[0], ms->center0[1], ms->center0[2], ms->center1[0], ms->center1[1], ms->center1[2], ms->time0, ms->time1, ms->radius}); }
    else if (auto r = dynamic_cast<AARect*>(h.get())) { n.type = r->node_type; n.material = mat(r->mp); set({r->a0, r->a1, r->b0, r->b1, r->k}); }
    else if (auto b = dynamic_cast<Box*>(h.get())) { n.type = RTB_NODE_BOX; n.material = mat(b->ptr); set({b->box_min[0], b->box_min[1], b->box_min[2], b->box_max[0], b->box_max[1], b->box_max[2]}); }
    else if (auto t = dynamic_cast<Translate*>(h.get())) { n.type = RTB_NODE_TRANSLATE; set({t->offset[0], t->offset[1], t->offset[2]}); kids.push_back(node(t->ptr)); }
    else if (auto ry = dynamic_cast<RotateY*>(h.get())) { n.type = RTB_NODE_ROTATE_Y; set({ry->angle}); kids.push_back(node(ry->ptr)); }
    else if (auto f = dynamic_cast<FlipFace*>(h.get())) { n.type = RTB_NODE_FLIP_FACE; kids.push_back(node(f->ptr)); }
    else if (auto cm = dynamic_cast<ConstantMedium*>(h.get())) { n.type = RTB_NODE_CONSTANT_MEDIUM; n.material = mat(cm->phase_function); set({cm->density}); kids.push_back(node(cm->boundary)); }
    else if (auto l = dynamic_cast<HittableList*>(h.get())) { n.type = RTB_NODE_LIST; for (auto& o : l->objects) kids.push_back(node(o)); }
    else if (auto bv = dynamic_cast<BVHNode*>(h.get())) { n.type = RTB_NODE_BVH; for (auto& o : bv->src->objects) kids.push_back(node(o)); }
    else if (auto tm = dynamic_cast<TriangleMesh*>(h.get())) { n.type = RTB_NODE_MESH; n.material = mat(tm->mat_ptr); set({(double)meshes.size()}); meshes.push_back(tm); }
    else throw std::invalid_argument("unknown hittable");
    n.first_child = (uint32_t)child_index.size();
    n.n_children = (uint32_t)kids.size();
    child_index.insert(child_index.end(), kids.begin(), kids.end());
    nodes.push_back(n);
    return (uint32_t)nodes.size() - 1;
  }
  // world + the reference's separate light-proxy list (main.rs:669-686): only XzRect and Sphere can be sampled
  void set_world(const HittablePtr& world, const std::shared_ptr<HittableList>& light_list = nullptr) {
    root = node(world);
    lights.clear();
    if (light_list)
      for (auto& o : light_list->objects) {
        rtb_light l{};
        if (auto r = dynamic_cast<XzRect*>(o.get())) { l.type = RTB_LIGHT_XZ_RECT; l.p[0] = r->a0; l.p[1] = r->a1; l.p[2] = r->b0; l.p[3] = r->b1; l.p[4] = r->k; }
        else if (auto s = dynamic_cast<Sphere*>(o.get())) { l.type = RTB_LIGHT_SPHERE; l.p[0] = s->center[0]; l.p[1] = s->center[1]; l.p[2] = s->center[2]; l.p[3] = s->radius; }
        else throw std::invalid_argument("only XzRect and Sphere implement pdf_value/random (hittable.rs:54-59)");
        lights.push_back(l);
      }
  }
  // hand everything to librtb200 (throws with rtb_last_error() on failure, like the reference's unwrap())
  void upload(rtb_scene* s) const {
    auto ck = [](int rc) { if (rc != 0) throw std::runtime_error(std::string("rtb200: ") + rtb_last_error()); };
    ck(rtb_scene_set_materials(s, materials.data(), (uint32_t)materials.size()));
    ck(rtb_scene_set_textures(s, textures.data(), (uint32_t)textures.size()));
    for (size_t i = 0; i < images.size(); ++i) ck(rtb_scene_set_image(s, (uint32_t)i, images[i]->data.data(), images[i]->width, images[i]->height));
    for (size_t i = 0; i < perlins.size(); ++i)
      ck(rtb_scene_set_perlin(s, (uint32_t)i, perlins[i]->ranvec.data(), perlins[i]->perm_x.data(), perlins[i]->perm_y.data(), perlins[i]->perm_z.data()));
    for (size_t i = 0; i < meshes.size(); ++i)
      ck(rtb_scene_set_mesh(s, (uint32_t)i, meshes[i]->vertices.data(), (uint32_t)(meshes[i]->vertices.size() / 3), meshes[i]->indices.data(), (uint32_t)(meshes[i]->indices.size() / 3)));
    for (size_t i = 0; i < meshes.size(); ++i) {
      const TriangleMesh& m = *meshes[i];
      if (m.normals.empty() && m.uvs.empty()) continue;
      auto ptr = [](const auto& v) { return v.empty() ? nullptr : v.data(); };
      ck(rtb_scene_set_mesh_attributes(s, (uint32_t)i, ptr(m.normals), (uint32_t)(m.normals.size() / 3), ptr(m.normal_indices),
                                       ptr(m.uvs), (uint32_t)(m.uvs.size() / 2), ptr(m.uv_indices)));
    }
    ck(rtb_scene_set_lights(s, lights.empty() ? nullptr : lights.data(), (uint32_t)lights.size()));
    ck(rtb_scene_set_graph(s, nodes.data(), (uint32_t)nodes.size(), child_index.data(), (uint32_t)child_index.size(), root));
  }

 private:
  std::unordered_map<const Texture*, uint32_t> tex_ids_;
  std::unordered_map<const Material*, uint32_t> mat_ids_;
  std::vector<std::shared_ptr<Texture>> keep_;
  std::vector<MaterialPtr> keep_m_;
};

}  // namespace rtb200
