// flatten.cpp — host side of the drop-in boundary: turns the reference's scene graph (one rtb_node per constructor
// call) into world-space SoA primitives in primitive-id order.  What the reference evaluates lazily through
// trait-object wrappers at every ray (hittable.rs:76-85 Translate, :147-176 RotateY, :195-201 FlipFace,
// boxes.rs:19-68 Box, hittable_list.rs:43-49 list order) is resolved here once.
#include <cmath>
#include <cstring>
#include <thread>

#include "rtb_internal.hpp"

namespace rtb {

namespace {

const double kPi = 3.14159265358979323846;

struct Xform {           // world = Ry(angle) * p + t   (the reference only has Y rotations and translations)
  double c = 1, s = 0;   // cos / sin of the accumulated angle
  double t[3] = {0, 0, 0};
  double angle_deg = 0;
  bool identity_rot = true;
  void point(const double p[3], double out[3]) const {  // hit -> world direction of hittable.rs:162-166
    out[0] = c * p[0] + s * p[2] + t[0];
    out[1] = p[1] + t[1];
    out[2] = -s * p[0] + c * p[2] + t[2];
  }
  void vec(const double p[3], double out[3]) const {
    out[0] = c * p[0] + s * p[2];
    out[1] = p[1];
    out[2] = -s * p[0] + c * p[2];
  }
};

// front_face / normal rewriting by the wrappers between the root and a primitive, evaluated the way the reference
// does per hit, innermost first (`wr` is stored outermost first):
//   primitive        set_face_normal(ray, outward): normal n against the ray, front = natural
//   FlipFace         front = !front                                                     (hittable.rs:197-201)
//   Translate        set_face_normal(moved ray, normal): the normal is re-oriented against the ray,
//                    front = "the incoming normal already was"                           (hittable.rs:82-83)
//   RotateY          set_face_normal(OBJECT-space ray, WORLD-space normal): q = dot(R^T d, n) < 0;
//                    front = q (or !q if the incoming normal was mis-oriented), normal = q ? n : -n   (hittable.rs:173)
// One RotateY gives a closed form in q (FACE_Q / FACE_NOT_Q / FACE_BARE); with two the outer one's q depends on the inner
// one's and the chain falls back to "front = true" for transforms (what round 1 did for every chain).
enum : uint8_t { WR_TRANSLATE = 1, WR_ROTATE = 2, WR_FLIP = 3 };
uint32_t eval_face(const uint8_t* wr, int n) {
  enum { F0, NF0, T, F, Q, NQ } front = F0;
  bool sign_q = false;  // the normal is q ? n : -n instead of n
  int n_rot = 0;
  auto neg = [](decltype(front) f) { return f == F0 ? NF0 : f == NF0 ? F0 : f == T ? F : f == F ? T : f == Q ? NQ : Q; };
  for (int i = n - 1; i >= 0; --i) {
    if (wr[i] == WR_FLIP) {
      front = neg(front);
    } else if (wr[i] == WR_TRANSLATE || n_rot >= 1) {
      if (wr[i] == WR_ROTATE) ++n_rot;
      front = sign_q ? Q : T;
      sign_q = false;
    } else {  // the chain's first (innermost) RotateY
      ++n_rot;
      front = Q;  // (the incoming normal is correctly oriented: nothing before it can have flipped it)
      sign_q = true;
    }
  }
  const uint32_t base = front == F0 ? FACE_NATURAL : front == NF0 ? FACE_FLIPPED : front == T ? FACE_TRUE
                        : front == F ? FACE_FALSE : front == Q ? FACE_Q : FACE_NOT_Q;
  return base | (sign_q ? FACE_BARE : 0u);
}
void set_bounds(HostPrim& p, const double lo[3], const double hi[3]) {
  for (int a = 0; a < 3; ++a) {
    double m = std::fmax(std::fabs(lo[a]), std::fabs(hi[a]));
    double pad = 1e-4 + 2e-6 * m;  // reference pads rect boxes by 1e-4 (aarect.rs:52-53); plus f32 slack
    p.lo[a] = std::nextafterf((float)(lo[a] - pad), -INFINITY);
    p.hi[a] = std::nextafterf((float)(hi[a] + pad), INFINITY);
  }
}

// the wrapper chain in the form the reference evaluates it per ray; `canonical` = at most one Translate outside at most
// one RotateY (every reference scene: main.rs:398-422,507-516,630-641).  Other nestings are flattened to world space:
// still f64 on the exact path, but the reference's per-wrapper rounding sequence is not reproduced bit for bit.
struct Chain {
  ExactXform x;
  bool canonical = true;
  uint8_t wr[32];  // wrapper kinds from the root down to here (eval_face)
  int n_wr = 0;
  Chain with(uint8_t kind) const {
    Chain c = *this;
    if (c.n_wr < 32) c.wr[c.n_wr++] = kind;
    return c;
  }
};

struct Walker {
  HostScene& hs;
  const rtb_node* nodes;
  uint32_t n_nodes;
  const uint32_t* child_index;
  uint32_t n_child_index;
  std::string& err;
  uint32_t depth = 0;

  bool fail(const char* m) { err = m; return false; }

  HostPrim& emit(uint32_t type, uint32_t material, uint32_t face_mode) {
    hs.prims.emplace_back();
    HostPrim& p = hs.prims.back();
    std::memset(&p, 0, sizeof(p));
    p.type = type;
    p.prim_id = hs.n_prim_ids++;
    p.material = material;
    p.face_mode = face_mode;
    p.exact = RTB_NONE;
    p.attr = RTB_NONE;
    return p;
  }

  // header of a non-canonical chain: no per-ray transform (parameters are world-space), total rotation kept for uv
  static ExactXform world_header(const Xform& x) {
    ExactXform h;
    h.sin_t = x.s; h.cos_t = x.c;
    return h;
  }

  bool check_mat(uint32_t m) {
    if (m == RTB_NONE || m >= hs.materials.size()) return fail("primitive references a material that was not set");
    return true;
  }

  void rect(int axis, double a0, double a1, double b0, double b1, double k, uint32_t mat, const Xform& x, uint32_t fm,
            const Chain& ch) {
    // aarect.rs: XyRect axis 2 (a=x,b=y), XzRect axis 1 (a=x,b=z), YzRect axis 0 (a=y,b=z); outward normal = +axis
    int ia = axis == 0 ? 1 : 0, ib = axis == 2 ? 1 : 2;
    double Q[3], U[3] = {0, 0, 0}, V[3] = {0, 0, 0}, N[3] = {0, 0, 0};
    Q[axis] = k; Q[ia] = a0; Q[ib] = b0;
    U[ia] = a1 - a0;
    V[ib] = b1 - b0;
    N[axis] = 1.0;
    double Qw[3], Uw[3], Vw[3], Nw[3];
    x.point(Q, Qw); x.vec(U, Uw); x.vec(V, Vw); x.vec(N, Nw);
    HostPrim& p = emit(PT_QUAD, mat, fm);
    pack_quad(p, Qw, Uw, Vw, Nw);
    if (ch.canonical) {
      const double prm[5] = {k, a0, a1, b0, b1};
      p.exact = add_exact(hs, ch.x, (uint32_t)axis, prm, 5);
    } else {
      const double prm[9] = {Qw[0], Qw[1], Qw[2], Uw[0], Uw[1], Uw[2], Vw[0], Vw[1], Vw[2]};
      p.exact = add_exact(hs, world_header(x), EX_QUAD_GENERAL, prm, 9);
    }
  }

  bool walk(uint32_t ni, const Xform& x, uint32_t fm, const Chain& ch) {
    if (ni >= n_nodes) return fail("node index out of range");
    if (++depth > 256) return fail("scene graph too deep (cycle?)");
    const rtb_node& n = nodes[ni];
    const double* p = n.p;
    bool ok = true;
    auto child = [&](uint32_t k, uint32_t& out) -> bool {
      if (k >= n.n_children || (uint64_t)n.first_child + k >= n_child_index) return fail("node is missing a child");
      out = child_index[n.first_child + k];
      return true;
    };
    switch (n.type) {
      case RTB_NODE_SPHERE: {
        if (!check_mat(n.material)) { ok = false; break; }
        // uv are object-space (sphere.rs:32-37): the record keeps the rotation, surface_uv() rotates the normal back
        double c[3];
        x.point(p, c);
        HostPrim& pr = emit(PT_SPHERE, n.material, fm);
        pack_sphere(pr, c, p[3]);
        if (ch.canonical) {
          const double prm[4] = {p[0], p[1], p[2], p[3]};
          pr.exact = add_exact(hs, ch.x, 0, prm, 4);
        } else {
          const double prm[4] = {c[0], c[1], c[2], p[3]};
          pr.exact = add_exact(hs, world_header(x), 0, prm, 4);
        }
        break;
      }
      case RTB_NODE_MOVING_SPHERE: {
        if (!check_mat(n.material)) { ok = false; break; }
        double c0[3], c1[3];
        x.point(p, c0); x.point(p + 3, c1);
        HostPrim& pr = emit(PT_MOVING, n.material, fm);
        pack_moving(pr, c0, c1, p[6], p[7], p[8]);
        if (ch.canonical) {
          const double prm[9] = {p[0], p[1], p[2], p[3], p[4], p[5], p[6], p[7], p[8]};
          pr.exact = add_exact(hs, ch.x, 0, prm, 9);
        } else {
          const double prm[9] = {c0[0], c0[1], c0[2], c1[0], c1[1], c1[2], p[6], p[7], p[8]};
          pr.exact = add_exact(hs, world_header(x), 0, prm, 9);
        }
        break;
      }
      case RTB_NODE_XY_RECT: if (!check_mat(n.material)) { ok = false; break; } rect(2, p[0], p[1], p[2], p[3], p[4], n.material, x, fm, ch); break;
      case RTB_NODE_XZ_RECT: if (!check_mat(n.material)) { ok = false; break; } rect(1, p[0], p[1], p[2], p[3], p[4], n.material, x, fm, ch); break;
      case RTB_NODE_YZ_RECT: if (!check_mat(n.material)) { ok = false; break; } rect(0, p[0], p[1], p[2], p[3], p[4], n.material, x, fm, ch); break;
      case RTB_NODE_BOX: {  // boxes.rs:19-68: XY(z1) XY(z0) XZ(y1) XZ(y0) YZ(x1) YZ(x0)
        if (!check_mat(n.material)) { ok = false; break; }
        rect(2, p[0], p[3], p[1], p[4], p[5], n.material, x, fm, ch);
        rect(2, p[0], p[3], p[1], p[4], p[2], n.material, x, fm, ch);
        rect(1, p[0], p[3], p[2], p[5], p[4], n.material, x, fm, ch);
        rect(1, p[0], p[3], p[2], p[5], p[1], n.material, x, fm, ch);
        rect(0, p[1], p[4], p[2], p[5], p[3], n.material, x, fm, ch);
        rect(0, p[1], p[4], p[2], p[5], p[0], n.material, x, fm, ch);
        break;
      }
      case RTB_NODE_TRIANGLE: {
        if (!check_mat(n.material)) { ok = false; break; }
        // triangle vertices are single precision by contract (include/rtb200.h): rounded before the transform
        double pf[9], a[3], b[3], c[3];
        for (int q = 0; q < 9; ++q) pf[q] = (double)(float)p[q];
        x.point(pf, a); x.point(pf + 3, b); x.point(pf + 6, c);
        HostPrim& pr = emit(PT_TRI, n.material, fm);
        pack_tri(pr, a, b, c);
        pr.g[3] = (float)x.s; pr.g[7] = (float)x.c;  // the chain's rotation, for RotateY's front_face test (surface_at)
        break;
      }
      case RTB_NODE_QUAD: {
        if (!check_mat(n.material)) { ok = false; break; }
        double Q[3], U[3], V[3];
        x.point(p, Q); x.vec(p + 3, U); x.vec(p + 6, V);
        HostPrim& pr = emit(PT_QUAD, n.material, fm);
        pack_quad(pr, Q, U, V, nullptr);
        if (ch.canonical) {
          pr.exact = add_exact(hs, ch.x, EX_QUAD_GENERAL, p, 9);
        } else {
          const double prm[9] = {Q[0], Q[1], Q[2], U[0], U[1], U[2], V[0], V[1], V[2]};
          pr.exact = add_exact(hs, world_header(x), EX_QUAD_GENERAL, prm, 9);
        }
        break;
      }
      case RTB_NODE_MESH: {
        if (!check_mat(n.material)) { ok = false; break; }
        uint32_t mid = (uint32_t)p[0];
        if (mid >= hs.meshes.size() || hs.meshes[mid].idx.empty()) { ok = fail("mesh id was not set"); break; }
        const HostScene::Mesh& m = hs.meshes[mid];
        // triangles take consecutive primitive ids in index order; large meshes are packed by several threads
        const size_t ntri = m.idx.size() / 3, first = hs.prims.size();
        const uint32_t id0 = hs.n_prim_ids;
        hs.prims.resize(first + ntri);
        hs.n_prim_ids += (uint32_t)ntri;
        const uint32_t material = n.material;
        // shading records: one per triangle when the mesh has vertex normals or texture coordinates
        const bool has_n = !m.normals.empty(), has_uv = !m.uvs.empty();
        const size_t attr0 = hs.attrs.size();
        if (has_n || has_uv) hs.attrs.resize(attr0 + ntri);
        auto pack_range = [&](size_t t0, size_t t1) {
          for (size_t t = t0; t < t1; ++t) {
            double v[3][3];
            for (int q = 0; q < 3; ++q) {
              const float* f = &m.verts[3 * (size_t)m.idx[3 * t + q]];
              double d[3] = {f[0], f[1], f[2]};
              x.point(d, v[q]);
            }
            HostPrim& pr = hs.prims[first + t];
            std::memset(&pr, 0, sizeof(pr));
            pr.type = PT_TRI;
            pr.prim_id = id0 + (uint32_t)t;
            pr.material = material;
            pr.face_mode = fm;
            pr.exact = RTB_NONE;
            pr.attr = RTB_NONE;
            pack_tri(pr, v[0], v[1], v[2]);
            pr.g[3] = (float)x.s; pr.g[7] = (float)x.c;
            if (has_n || has_uv) {
              AttrRec& a = hs.attrs[attr0 + t];
              std::memset(&a, 0, sizeof(a));
              uint32_t flags = 0;
              if (has_n) {  // the vertices' RotateY turns the normals; a Translate leaves them alone
                for (int q = 0; q < 3; ++q) {
                  const float* f = &m.normals[3 * (size_t)m.normal_idx[3 * t + q]];
                  const double d[3] = {f[0], f[1], f[2]};
                  double w[3];
                  x.vec(d, w);
                  for (int c = 0; c < 3; ++c) a.f[4 * q + c] = (float)w[c];
                }
                flags |= ATTR_NORMALS;
              }
              if (has_uv) {
                for (int q = 0; q < 3; ++q) {
                  const float* f = &m.uvs[2 * (size_t)m.uv_idx[3 * t + q]];
                  a.f[4 * q + 3] = f[0];
                  a.f[12 + q] = f[1];
                }
                flags |= ATTR_UVS;
              }
              std::memcpy(&a.f[15], &flags, 4);
              pr.attr = (uint32_t)(attr0 + t);
            }
          }
        };
        unsigned n_thr = ntri >= 100000 ? std::max(1u, std::min(std::thread::hardware_concurrency(), 16u)) : 1u;
        if (n_thr <= 1) {
          pack_range(0, ntri);
        } else {
          std::vector<std::thread> pool;
          const size_t per = (ntri + n_thr - 1) / n_thr;
          for (unsigned t = 0; t < n_thr; ++t) {
            const size_t t0 = std::min(ntri, t * per), t1 = std::min(ntri, t0 + per);
            if (t0 < t1) pool.emplace_back(pack_range, t0, t1);
          }
          for (std::thread& th : pool) th.join();
        }
        break;
      }
      case RTB_NODE_TRANSLATE: {
        uint32_t c;
        if (!child(0, c)) { ok = false; break; }
        Xform y = x;
        double off[3];
        x.vec(p, off);
        for (int a = 0; a < 3; ++a) y.t[a] += off[a];
        Chain c2 = ch.with(WR_TRANSLATE);
        if (ch.canonical && ch.x.flags == 0) {
          c2.x.flags = EX_TRANSLATE;
          for (int a = 0; a < 3; ++a) c2.x.off[a] = p[a];
        } else {
          c2.canonical = false;  // Translate inside RotateY / inside another Translate
        }
        ok = walk(c, y, eval_face(c2.wr, c2.n_wr), c2);
        break;
      }
      case RTB_NODE_ROTATE_Y: {
        uint32_t c;
        if (!child(0, c)) { ok = false; break; }
        Xform y = x;
        y.angle_deg = x.angle_deg + p[0];
        double rad = y.angle_deg * kPi / 180.0;  // hittable.rs:108
        y.c = std::cos(rad); y.s = std::sin(rad);
        y.identity_rot = false;
        Chain c2 = ch.with(WR_ROTATE);
        if (ch.canonical && !(ch.x.flags & EX_ROTATE)) {
          const double r1 = p[0] * kPi / 180.0;  // hittable.rs:108
          c2.x.flags |= EX_ROTATE;
          c2.x.sin_t = std::sin(r1); c2.x.cos_t = std::cos(r1);
        } else {
          c2.canonical = false;
        }
        ok = walk(c, y, eval_face(c2.wr, c2.n_wr), c2);
        break;
      }
      case RTB_NODE_FLIP_FACE: {
        uint32_t c;
        if (!child(0, c)) { ok = false; break; }
        const Chain c2 = ch.with(WR_FLIP);
        ok = walk(c, x, eval_face(c2.wr, c2.n_wr), c2);
        break;
      }
      case RTB_NODE_CONSTANT_MEDIUM: {
        if (!check_mat(n.material)) { ok = false; break; }
        if (!(p[0] > 0.0) || !std::isfinite(p[0])) { ok = fail("ConstantMedium density must be positive and finite"); break; }
        uint32_t c;
        if (!child(0, c)) { ok = false; break; }
        // resolve the boundary: Sphere or Box under Translate/RotateY wrappers (convex, as the reference requires)
        Xform y = x;
        uint32_t guard = 0;
        while (ok) {
          if (c >= n_nodes || ++guard > 64) { ok = fail("bad medium boundary"); break; }
          const rtb_node& b = nodes[c];
          if (b.type == RTB_NODE_TRANSLATE) {
            double off[3];
            y.vec(b.p, off);
            for (int a = 0; a < 3; ++a) y.t[a] += off[a];
          } else if (b.type == RTB_NODE_ROTATE_Y) {
            y.angle_deg += b.p[0];
            double rad = y.angle_deg * kPi / 180.0;
            y.c = std::cos(rad); y.s = std::sin(rad);
            y.identity_rot = false;
          } else if (b.type == RTB_NODE_FLIP_FACE) {
          } else {
            break;
          }
          if (b.n_children < 1 || (uint64_t)b.first_child >= n_child_index) { ok = fail("bad medium boundary"); break; }
          c = child_index[b.first_child];
        }
        if (!ok) break;
        const rtb_node& b = nodes[c];
        HostMedium m;
        std::memset(&m, 0, sizeof(m));
        m.material = n.material;
        m.prim_id = hs.n_prim_ids++;
        m.neg_inv_density = (float)(-1.0 / p[0]);  // constant_medium.rs:26
        m.sin_t = (float)y.s; m.cos_t = (float)y.c;
        for (int a = 0; a < 3; ++a) m.offset[a] = (float)y.t[a];
        if (b.type == RTB_NODE_SPHERE) {
          double cw[3];
          y.point(b.p, cw);
          m.boundary_type = RTB_BOUNDARY_SPHERE;
          m.p[0] = (float)cw[0]; m.p[1] = (float)cw[1]; m.p[2] = (float)cw[2]; m.p[3] = (float)b.p[3];
        } else if (b.type == RTB_NODE_BOX) {
          m.boundary_type = RTB_BOUNDARY_BOX;
          for (int a = 0; a < 6; ++a) m.p[a] = (float)b.p[a];
        } else {
          ok = fail("ConstantMedium boundary must be a Sphere or a Box (optionally under Translate/RotateY)");
          break;
        }
        hs.media.push_back(m);
        break;
      }
      case RTB_NODE_LIST:
      case RTB_NODE_BVH: {
        for (uint32_t k = 0; k < n.n_children && ok; ++k) {
          uint32_t c;
          if (!child(k, c)) { ok = false; break; }
          ok = walk(c, x, fm, ch);
        }
        break;
      }
      default: ok = fail("unknown node type");
    }
    --depth;
    return ok;
  }
};

}  // namespace

uint32_t add_exact(HostScene& hs, const ExactXform& x, uint32_t subtype, const double* params, int n_params) {
  ExactRec r;
  std::memset(&r, 0, sizeof(r));
  const uint64_t bits = (uint64_t)x.flags | ((uint64_t)subtype << 8);
  std::memcpy(&r.v[0], &bits, 8);
  for (int a = 0; a < 3; ++a) r.v[1 + a] = x.off[a];
  r.v[4] = x.sin_t;
  r.v[5] = x.cos_t;
  for (int k = 0; k < n_params && 6 + k < RTB_EXACT_STRIDE; ++k) r.v[6 + k] = params[k];
  hs.exact.push_back(r);
  return (uint32_t)(hs.exact.size() - 1);
}

void pack_sphere(HostPrim& p, const double c[3], double r) {
  p.g[0] = (float)c[0]; p.g[1] = (float)c[1]; p.g[2] = (float)c[2]; p.g[3] = (float)r;
  double ar = std::fabs(r);
  double lo[3] = {c[0] - ar, c[1] - ar, c[2] - ar}, hi[3] = {c[0] + ar, c[1] + ar, c[2] + ar};
  set_bounds(p, lo, hi);
}

void pack_moving(HostPrim& p, const double c0[3], const double c1[3], double t0, double t1, double r) {
  // centre(time) = c0 + (time - t0)/(t1 - t0) * (c1 - c0) = A + time * B      moving_sphere.rs:36-39
  double inv = 1.0 / (t1 - t0);
  double lo[3], hi[3];
  double ta = std::fmin(t0, 0.0), tb = std::fmax(t1, 1.0);  // bounds cover shutter times in [min(t0,0), max(t1,1)]
  for (int a = 0; a < 3; ++a) {
    double B = (c1[a] - c0[a]) * inv, A = c0[a] - t0 * B;
    p.g[a] = (float)A;
    p.g[4 + a] = (float)B;
    double pa = A + ta * B, pb = A + tb * B;
    lo[a] = std::fmin(pa, pb) - std::fabs(r);
    hi[a] = std::fmax(pa, pb) + std::fabs(r);
  }
  p.g[3] = (float)r;
  p.g[7] = 0.f;
  set_bounds(p, lo, hi);
}

static void cross3(const double a[3], const double b[3], double o[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
static double dot3(const double a[3], const double b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

void pack_quad(HostPrim& p, const double Q[3], const double U[3], const double V[3], const double* outward) {
  // plane form: word0 = (n, n.Q), word1 = (wa, wa.Q), word2 = (wb, wb.Q) with
  //   t = (n.Q - n.o)/(n.d),  alpha = wa.P - wa.Q,  beta = wb.P - wb.Q,   wa = (V x n')/(n'.n'), wb = (n' x U)/(n'.n'), n' = U x V
  double n[3], wa[3], wb[3];
  cross3(U, V, n);
  double nn = dot3(n, n);
  cross3(V, n, wa);
  cross3(n, U, wb);
  double len = std::sqrt(nn);
  double nh[3];
  for (int a = 0; a < 3; ++a) { wa[a] /= nn; wb[a] /= nn; nh[a] = n[a] / len; }
  if (outward) {  // axis-aligned rects have outward normal = +axis regardless of the (a,b) handedness (aarect.rs:43,93,162)
    double ol = std::sqrt(dot3(outward, outward));
    for (int a = 0; a < 3; ++a) nh[a] = outward[a] / ol;
  }
  for (int a = 0; a < 3; ++a) { p.g[a] = (float)nh[a]; p.g[4 + a] = (float)wa[a]; p.g[8 + a] = (float)wb[a]; }
  p.g[3] = (float)dot3(nh, Q);
  {  // an axis-aligned plane whose constant is a float (555, 0, 213 ...): t = (k - o_a) / d_a carries no rounding but its own
    const double nq = dot3(nh, Q);
    const int zeros = (p.g[0] == 0.f) + (p.g[1] == 0.f) + (p.g[2] == 0.f);
    p.plane_exact = zeros == 2 && (double)p.g[3] == nq && std::fabs(p.g[0] + p.g[1] + p.g[2]) == 1.0f;
  }
  p.g[7] = (float)dot3(wa, Q);
  p.g[11] = (float)dot3(wb, Q);
  double lo[3], hi[3];
  for (int a = 0; a < 3; ++a) {
    double c0 = Q[a], c1 = Q[a] + U[a], c2 = Q[a] + V[a], c3 = Q[a] + U[a] + V[a];
    lo[a] = std::fmin(std::fmin(c0, c1), std::fmin(c2, c3));
    hi[a] = std::fmax(std::fmax(c0, c1), std::fmax(c2, c3));
  }
  set_bounds(p, lo, hi);
}

void pack_tri(HostPrim& p, const double v0[3], const double v1[3], const double v2[3]) {
  double lo[3], hi[3];
  for (int a = 0; a < 3; ++a) {
    p.g[a] = (float)v0[a];      // vertices, not edges: the watertight test needs the shared vertices bit-identical
    p.g[4 + a] = (float)v1[a];
    p.g[8 + a] = (float)v2[a];
    lo[a] = std::fmin(v0[a], std::fmin(v1[a], v2[a]));
    hi[a] = std::fmax(v0[a], std::fmax(v1[a], v2[a]));
  }
  p.g[3] = 0.f; p.g[7] = 1.f; p.g[11] = 0.f;  // (sin, cos) of the wrapper chain's rotation: identity unless the caller sets it
  set_bounds(p, lo, hi);
}

int flatten_graph(HostScene& hs, const rtb_node* nodes, uint32_t n_nodes, const uint32_t* child_index,
                  uint32_t n_child_index, uint32_t root, std::string& err) {
  hs.prims.clear();
  hs.media.clear();
  hs.exact.clear();
  hs.attrs.clear();
  hs.n_prim_ids = 0;
  Walker w{hs, nodes, n_nodes, child_index, n_child_index, err};
  Xform id;
  Chain ch;
  if (!w.walk(root, id, FACE_NATURAL, ch)) return RTB_ERR_INVALID;
  return RTB_OK;
}

}  // namespace rtb
