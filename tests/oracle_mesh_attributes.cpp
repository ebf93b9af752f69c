// oracle_mesh_attributes.cpp — TEST INFRASTRUCTURE ONLY.  The f64 reference of smooth-shaded, UV-mapped mesh triangles
// (rtb_scene_set_mesh_attributes).  Compiled in one translation unit with the CPU oracle (oracle/rt_oracle.cpp, through
// tests/oracle_aov.cpp), which stays as it is: its hit records, wrappers and front_face rules are used unchanged, and after
// world_hit an attribute triangle's normal and (u, v) are replaced in f64 from the record's barycentrics (rec.u, rec.v) and
// the world-space vertex normals, with the normal turned to the side of the geometric rec.normal (include/rtb200.h).
// ray_color / orc_render / orc_aov_rays are restated here with that one step added (tests/mesh_attr_oracle.py binds them).
#include "oracle_aov.cpp"

#include <map>
#include <mutex>

namespace {

struct MeshAttr {  // one mesh's streams as the caller gave them (normals normalised in f64, like the product's host)
  std::vector<double> normals, uvs;
  std::vector<uint32_t> normal_idx, uv_idx;
};
struct PrimAttr {
  uint32_t flags = 0;  // bit 0 normals, bit 1 uvs
  V3 n[3];
  double u[3] = {0, 0, 0}, v[3] = {0, 0, 0};
};
struct AttrScene {
  std::map<uint32_t, MeshAttr> meshes;
  std::vector<PrimAttr> by_prim;  // resolved against the built scene: primitive id -> shading record
  bool resolved = false;
};
std::mutex g_mu;
std::map<const orc_scene*, AttrScene> g_attr;

// primitive ids in build_node's order (list order, Box -> 6, mesh triangles in index order, a ConstantMedium before its
// boundary, no ids inside a boundary), with the RotateY angles above each mesh (outermost first)
void resolve_walk(const Scene& sc, AttrScene& as, uint32_t ni, bool in_boundary, std::vector<std::pair<double, double>>& rot,
                  uint32_t& next_id) {
  const rtb_node& n = sc.nodes[ni];
  auto id = [&]() { return in_boundary ? RTB_NONE : next_id++; };
  auto kid = [&](uint32_t k) { return sc.child_index[n.first_child + k]; };
  switch (n.type) {
    case RTB_NODE_SPHERE: case RTB_NODE_MOVING_SPHERE: case RTB_NODE_XY_RECT: case RTB_NODE_XZ_RECT:
    case RTB_NODE_YZ_RECT: case RTB_NODE_TRIANGLE: case RTB_NODE_QUAD:
      id();
      break;
    case RTB_NODE_BOX:
      for (int k = 0; k < 6; ++k) id();
      break;
    case RTB_NODE_MESH: {
      const uint32_t mid = (uint32_t)n.p[0];
      const size_t ntri = sc.meshes[mid].idx.size() / 3;
      auto it = as.meshes.find(mid);
      for (size_t t = 0; t < ntri; ++t) {
        const uint32_t pid = id();
        if (pid == RTB_NONE || it == as.meshes.end()) continue;
        const MeshAttr& m = it->second;
        PrimAttr a;
        for (int q = 0; q < 3; ++q) {
          if (!m.normals.empty()) {
            const double* f = &m.normals[3 * (size_t)m.normal_idx[3 * t + q]];
            V3 w(f[0], f[1], f[2]);
            for (size_t k = rot.size(); k-- > 0;) {  // innermost RotateY first (hittable.rs:168-171)
              const double s = rot[k].first, c = rot[k].second;
              w = V3(c * w.x + s * w.z, w.y, -s * w.x + c * w.z);
            }
            a.n[q] = w;
            a.flags |= 1u;
          }
          if (!m.uvs.empty()) {
            const double* f = &m.uvs[2 * (size_t)m.uv_idx[3 * t + q]];
            a.u[q] = f[0]; a.v[q] = f[1];
            a.flags |= 2u;
          }
        }
        if (as.by_prim.size() <= pid) as.by_prim.resize(pid + 1);
        as.by_prim[pid] = a;
      }
      break;
    }
    case RTB_NODE_TRANSLATE: case RTB_NODE_FLIP_FACE:
      resolve_walk(sc, as, kid(0), in_boundary, rot, next_id);
      break;
    case RTB_NODE_ROTATE_Y: {
      const double radians = n.p[0] * PI / 180.0;  // hittable.rs:107-111
      rot.emplace_back(std::sin(radians), std::cos(radians));
      resolve_walk(sc, as, kid(0), in_boundary, rot, next_id);
      rot.pop_back();
      break;
    }
    case RTB_NODE_CONSTANT_MEDIUM:
      id();
      resolve_walk(sc, as, kid(0), true, rot, next_id);
      break;
    default:  // LIST, BVH
      for (uint32_t k = 0; k < n.n_children; ++k) resolve_walk(sc, as, kid(k), in_boundary, rot, next_id);
  }
}

const std::vector<PrimAttr>* attrs_of(orc_scene* o) {
  if (!o->s.build()) return nullptr;
  std::lock_guard<std::mutex> lk(g_mu);
  AttrScene& as = g_attr[o];
  if (!as.resolved) {
    as.by_prim.clear();
    std::vector<std::pair<double, double>> rot;
    uint32_t next_id = 0;
    resolve_walk(o->s, as, o->s.root, false, rot, next_id);
    if (next_id != o->s.n_prims) return nullptr;  // the walk must number primitives exactly as build_node did
    as.resolved = true;
  }
  return &as.by_prim;
}

// the shading rule of include/rtb200.h, in f64, on a hit record world_hit returned
void shade_attrs(const std::vector<PrimAttr>& tab, HitRecord& rec) {
  if (rec.prim >= tab.size() || !tab[rec.prim].flags) return;
  const PrimAttr& a = tab[rec.prim];
  const double b1 = rec.u, b2 = rec.v, b0 = 1.0 - b1 - b2;
  if (a.flags & 1u) {
    const V3 s = b0 * a.n[0] + b1 * a.n[1] + b2 * a.n[2];
    const double l2 = dot(s, s);
    if (std::isfinite(l2) && l2 >= 1e-20) {
      const V3 ns = s / std::sqrt(l2);
      rec.normal = dot(ns, rec.normal) < 0.0 ? -ns : ns;
    }
  }
  if (a.flags & 2u) {
    rec.u = b0 * a.u[0] + b1 * a.u[1] + b2 * a.u[2];
    rec.v = b0 * a.v[0] + b1 * a.v[1] + b2 * a.v[2];
  }
}

// oracle/rt_oracle.cpp ray_color with shade_attrs() after the closest hit
SampleOut ray_color_attr(const Scene& sc, const std::vector<PrimAttr>& tab, Ray r, V3 background, int max_depth,
                         uint32_t rr_start, const PathRng& rng) {
  V3 L(0, 0, 0), beta(1, 1, 1);
  uint32_t segments = 0;
  const bool have_lights = !sc.lights->objects.empty();
  for (int depth = max_depth; depth > 0; --depth) {
    ++segments;
    const uint32_t bounce = segments;
    HitRecord rec;
    HitCtx cx; cx.rng = &rng; cx.bounce = bounce;
    if (!world_hit(sc, r, 0.001, INF, rec, cx)) {
      L = L + beta * background;
      break;
    }
    shade_attrs(tab, rec);
    const rtb_material& m = sc.mats[rec.mat];
    double us[4], ua[4];
    rng.block(BLK_SCATTER, bounce, us);
    rng.block(BLK_AUX, bounce, ua);
    if (m.type == RTB_MAT_DIFFUSE_LIGHT) {
      if (rec.front_face) L = L + beta * sc.tex_value(m.texture, rec.u, rec.v, rec.p);
      break;
    }
    if (m.type == RTB_MAT_METAL) {
      double fuzz = m.param < 1.0 ? m.param : 1.0;
      V3 reflected = reflect(unit(r.d), rec.normal);
      double z = 1.0 - 2.0 * ua[1], phi = 2.0 * PI * ua[2], rad = std::cbrt(ua[3]);
      double s = std::sqrt(std::fmax(0.0, 1.0 - z * z));
      V3 ball(rad * s * std::cos(phi), rad * s * std::sin(phi), rad * z);
      beta = beta * sc.tex_value(m.texture, rec.u, rec.v, rec.p);
      r = Ray{rec.p, reflected + fuzz * ball, 0.0};
    } else if (m.type == RTB_MAT_DIELECTRIC) {
      double ratio = rec.front_face ? 1.0 / m.param : m.param;
      V3 ud = unit(r.d);
      double cos_theta = std::fmin(dot(-ud, rec.normal), 1.0);
      double sin_theta = std::sqrt(1.0 - cos_theta * cos_theta);
      bool cannot_refract = ratio * sin_theta > 1.0;
      double r0 = (1.0 - ratio) / (1.0 + ratio);
      r0 *= r0;
      double reflectance = r0 + (1.0 - r0) * std::pow(1.0 - cos_theta, 5);
      V3 dir = (cannot_refract || reflectance > ua[1]) ? reflect(ud, rec.normal) : refract(ud, rec.normal, ratio);
      r = Ray{rec.p, dir, r.tm};
    } else {
      const bool iso = m.type == RTB_MAT_ISOTROPIC;
      V3 atten = sc.tex_value(m.texture, rec.u, rec.v, rec.p);
      V3 dir;
      bool pick_light = have_lights && us[0] < 0.5;
      if (pick_light) {
        size_t n = sc.lights->objects.size();
        size_t k = (size_t)(us[1] * (double)n);
        if (k >= n) k = n - 1;
        dir = sc.lights->objects[k]->random(rec.p, us[2], us[3]);
      } else if (iso) {
        double z = 1.0 - 2.0 * us[2], phi = 2.0 * PI * us[3];
        double s = std::sqrt(std::fmax(0.0, 1.0 - z * z));
        dir = V3(s * std::cos(phi), s * std::sin(phi), z);
      } else {
        double zz = std::sqrt(1.0 - us[3]);
        double phi = 2.0 * PI * us[2];
        V3 a(std::cos(phi) * std::sqrt(us[3]), std::sin(phi) * std::sqrt(us[3]), zz);
        dir = Onb(rec.normal).local(a);
      }
      double mat_pdf, spdf;
      if (iso) {
        mat_pdf = spdf = 1.0 / (4.0 * PI);
      } else {
        double cosine = dot(unit(dir), unit(rec.normal));
        mat_pdf = cosine <= 0.0 ? 0.0 : cosine / PI;
        double c2 = dot(rec.normal, unit(dir));
        spdf = c2 < 0.0 ? 0.0 : c2 / PI;
      }
      double pdf_val = have_lights ? 0.5 * sc.lights->pdf_value(rec.p, dir) + 0.5 * mat_pdf : mat_pdf;
      if (!(spdf > 0.0)) break;
      beta = beta * atten * (spdf / pdf_val);
      r = Ray{rec.p, dir, r.tm};
    }
    if (rr_start > 0 && segments >= rr_start) {
      double q = std::fmax(beta.x, std::fmax(beta.y, beta.z));
      q = q < 0.2 ? 0.2 : (q > 1.0 ? 1.0 : q);
      if (!(ua[0] < q)) break;
      beta = beta / q;
    }
  }
  return SampleOut{L, segments};
}

}  // namespace

extern "C" {

// rtb_scene_set_mesh_attributes' streams for mesh `id` (NULL index pointer: the mesh's position indices).  Returns -1 when
// the mesh was not set or an index is out of range; call orc_attr_reset first on a new handle.
int orc_scene_set_mesh_attributes(orc_scene* o, uint32_t id, const float* normals, uint32_t n_normals,
                                  const uint32_t* normal_idx, const float* uvs, uint32_t n_uvs, const uint32_t* uv_idx) {
  if (id >= o->s.meshes.size()) return -1;
  const Scene::Mesh& mesh = o->s.meshes[id];
  MeshAttr m;
  if (normals) {
    for (uint32_t i = 0; i < n_normals; ++i) {
      const double x = normals[3 * i], y = normals[3 * i + 1], z = normals[3 * i + 2];
      const double len = std::sqrt(x * x + y * y + z * z), k = len > 0.0 ? 1.0 / len : 0.0;
      m.normals.push_back(x * k); m.normals.push_back(y * k); m.normals.push_back(z * k);
    }
    m.normal_idx = normal_idx ? std::vector<uint32_t>(normal_idx, normal_idx + mesh.idx.size()) : mesh.idx;
    for (uint32_t i : m.normal_idx) if (i >= n_normals) return -1;
  }
  if (uvs) {
    m.uvs.assign(uvs, uvs + 2 * (size_t)n_uvs);
    m.uv_idx = uv_idx ? std::vector<uint32_t>(uv_idx, uv_idx + mesh.idx.size()) : mesh.idx;
    for (uint32_t i : m.uv_idx) if (i >= n_uvs) return -1;
  }
  std::lock_guard<std::mutex> lk(g_mu);
  AttrScene& as = g_attr[o];
  as.meshes[id] = std::move(m);
  as.resolved = false;
  return 0;
}

// forget every attribute stored for this handle (a new oracle scene may reuse a destroyed one's address)
void orc_attr_reset(orc_scene* o) {
  std::lock_guard<std::mutex> lk(g_mu);
  g_attr.erase(o);
}

// orc_render (oracle/rt_oracle.cpp) with the attribute shading
int orc_render_attr(orc_scene* o, const rtb_camera* cam, const rtb_params* p, double* accum, uint64_t* segments_out,
                    uint64_t* rejected_out, int threads) {
  const std::vector<PrimAttr>* tab = attrs_of(o);
  if (!tab) return -1;
  Camera c(*cam);
  const Scene& sc = o->s;
  const uint32_t W = p->width, H = p->height;
  std::atomic<uint64_t> segs(0), rej(0);
  V3 bg(p->background[0], p->background[1], p->background[2]);
  parallel_rows(H, threads, [&](uint32_t row) {
    uint32_t j = H - 1 - row;
    uint64_t local_segs = 0, local_rej = 0;
    for (uint32_t i = 0; i < W; ++i) {
      double acc[4] = {0, 0, 0, 0};
      uint32_t pixel = row * W + i;
      for (uint32_t s = 0; s < p->spp; ++s) {
        PathRng rng; rng.pixel = pixel; rng.sample = p->sample_offset + s; rng.seed = p->seed;
        double u0[4], u1[4];
        rng.block(BLK_CAMERA0, 0, u0);
        rng.block(BLK_CAMERA1, 0, u1);
        double u = ((double)i + u0[0]) / (double)(W - 1), v = ((double)j + u0[1]) / (double)(H - 1);
        double dx, dy;
        disk_sample(u0[2], u0[3], dx, dy);
        double time = c.time0 + (c.time1 - c.time0) * u1[0];
        Ray r = c.get_ray(u, v, dx, dy, time);
        SampleOut so = ray_color_attr(sc, *tab, r, bg, p->max_depth, p->rr_start_depth, rng);
        local_segs += so.segments;
        if (!(std::isfinite(so.L.x) && std::isfinite(so.L.y) && std::isfinite(so.L.z))) { ++local_rej; continue; }
        double Y = 0.2126 * so.L.x + 0.7152 * so.L.y + 0.0722 * so.L.z;
        acc[0] += so.L.x; acc[1] += so.L.y; acc[2] += so.L.z; acc[3] += Y * Y;
      }
      double* dst = accum + (size_t)pixel * 4;
      for (int k = 0; k < 4; ++k) dst[k] = acc[k];
    }
    segs += local_segs; rej += local_rej;
  });
  if (segments_out) *segments_out = segs.load();
  if (rejected_out) *rejected_out = rej.load();
  return 0;
}

// orc_aov_rays (tests/oracle_aov.cpp) with the attribute shading
int orc_aov_rays_attr(orc_scene* o, const double* org, const double* dir, const double* time, const uint32_t* pixel,
                      const uint32_t* sample, uint32_t seed, uint32_t n, uint32_t* ids_out, double* vals_out,
                      uint32_t* kinds_out) {
  const std::vector<PrimAttr>* tab = attrs_of(o);
  if (!tab) return -1;
  const Scene& sc = o->s;
  const uint32_t block = 4096;
  parallel_rows((n + block - 1) / block, n >= 8 * block ? 0 : 1, [&](uint32_t b) {
    const uint32_t end = std::min<uint64_t>(n, (uint64_t)(b + 1) * block);
    for (uint32_t i = b * block; i < end; ++i) {
      Ray r{V3(org[3 * i], org[3 * i + 1], org[3 * i + 2]), V3(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]), time[i]};
      PathRng rng;
      rng.pixel = pixel[i]; rng.sample = sample[i]; rng.seed = seed;
      HitCtx cx;
      cx.rng = &rng; cx.bounce = 1;
      HitRecord rec;
      double* v = vals_out + 8 * (size_t)i;
      for (int k = 0; k < 8; ++k) v[k] = 0.0;
      uint32_t kind = 0xFFu;
      if (!world_hit(sc, r, 0.001, INF, rec, cx)) {
        ids_out[i] = RTB_NONE;
      } else {
        shade_attrs(*tab, rec);
        ids_out[i] = rec.prim;
        const rtb_material& m = sc.mats[rec.mat];
        V3 a(0, 0, 0);
        if (m.type == RTB_MAT_DIELECTRIC) {
          a = V3(1, 1, 1);
        } else if (m.type != RTB_MAT_DIFFUSE_LIGHT || rec.front_face) {
          a = sc.tex_value(m.texture, rec.u, rec.v, rec.p);
          kind = sc.texs[m.texture].type;
        }
        const bool medium = rec.prim >= sc.prim_obj.size() || !sc.prim_obj[rec.prim];
        v[0] = clampd(a.x, 0.0, 1.0); v[1] = clampd(a.y, 0.0, 1.0); v[2] = clampd(a.z, 0.0, 1.0);
        v[3] = 1.0;
        if (!medium) { v[4] = rec.normal.x; v[5] = rec.normal.y; v[6] = rec.normal.z; }
        v[7] = rec.t * length(r.d);
      }
      if (kinds_out) kinds_out[i] = kind;
    }
  });
  return 0;
}

}  // extern "C"
