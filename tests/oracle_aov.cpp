// oracle_aov.cpp — TEST INFRASTRUCTURE ONLY.  The f64 reference of rtb_render_aov's per-sample guide values.  It is compiled
// in one translation unit with the CPU oracle (oracle/rt_oracle.cpp), so the oracle's scene handle, world_hit and
// Scene::tex_value are used exactly as its other entry points use them (tests/aov_oracle.py builds and binds it).
#include "../oracle/rt_oracle.cpp"

extern "C" {

// Closest hit of caller rays (origin, direction, time: n x 3, n x 3, n doubles) with the ConstantMedium draw taken from the
// path stream (pixel[i], sample[i], seed) at segment 1, as the render's first segment draws it.  Per ray: ids_out = primitive
// id or RTB_NONE; vals_out = 8 doubles (albedo rgb clamped to [0, 1], coverage, shading normal xyz, depth = t |d|), all 0 for
// a miss (the caller supplies the background); kinds_out (may be NULL) = texture type the albedo was read from, or 0xFF
// when it is not a texture value (Dielectric, the back of a DiffuseLight, a miss).
int orc_aov_rays(orc_scene* o, const double* org, const double* dir, const double* time, const uint32_t* pixel,
                 const uint32_t* sample, uint32_t seed, uint32_t n, uint32_t* ids_out, double* vals_out,
                 uint32_t* kinds_out) {
  if (!o->s.build()) return -1;
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
        ids_out[i] = rec.prim;
        const rtb_material& m = sc.mats[rec.mat];
        V3 a(0, 0, 0);
        if (m.type == RTB_MAT_DIELECTRIC) {
          a = V3(1, 1, 1);
        } else if (m.type != RTB_MAT_DIFFUSE_LIGHT || rec.front_face) {
          a = sc.tex_value(m.texture, rec.u, rec.v, rec.p);
          kind = sc.texs[m.texture].type;
        }
        // a ConstantMedium is the one hittable that registers no primitive of its own (rt_oracle.cpp build_node)
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
