"""GPU tier (-m gpu): smooth-shaded, UV-mapped mesh triangles (rtb_scene_set_mesh_attributes) against the f64 oracle
(tests/oracle_mesh_attributes.cpp) and against the flat path.

- Hits: primary-hit ids and t are bitwise the same with and without attributes (geometry is untouched).
- AOV parity on identical rays (the device's own f32 camera rays, traced by the oracle with the same stream): coverage
  equal on every pixel; shading normals within 1e-4 per component on >= 99.9 % of the covered pixels and within 1e-3 on
  all; solid albedo within 1e-5; image albedo within 1e-4 on >= 99.9 %.
- Identity: face normals given as vertex normals plus corner UVs (0,0), (1,0), (0,1) on their own index stream render
  like no attributes at all with the same seed: >= 99.9 % of the pixels within 0.2 %, segment counts equal to 5 digits.
- P2: converged images against the oracle (independent sample sets): mean luminance error <= 1 %, no pixel beyond 5 sigma.
- The bounds-checked build renders the smooth scenes with no failed check; attributes follow the mesh's call order.
Measured on a B200: shading normals within 8.7e-6 (smooth_meshes) and 2.6e-5 (smooth C4) of the oracle's on every covered
pixel; solid albedo 2.4e-8; image albedo over 1e-4 on 4.4e-4 of the textured pixels (texel flips); identity 99.99 % of the
pixels within 0.2 %, segments 0.9999969; P2 0.035 % / max z 3.91 (smooth_meshes 200x200x1024) and 0.029 % / 4.07 (smooth
C4 208x117x1024); no failed check in the bounds-checked build.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers as H
import mesh_attr_oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _flat(cs):
    """The same compiled scene without any mesh attributes."""
    return cs.__class__(**{**cs.__dict__, "mesh_attrs": []})


def _cfgs():
    from ray_tracer_archive_b200 import scenes
    return {"smooth_meshes": (scenes.config_smooth_meshes(), 200, 200),
            "smooth_c4": (scenes.config_mesh(nx=200, nz=100, smooth=True), 192, 108)}


@pytest.mark.parametrize("name", ["smooth_meshes", "smooth_c4"])
def test_hits_unchanged_by_attributes(rtb, ctx, name):
    cfg, W, Hh = _cfgs()[name]
    cs = rtb.compile_scene(cfg.world, cfg.lights)
    a, f = rtb.Scene(ctx, cs), rtb.Scene(ctx, _flat(cs))
    ia, ta, _ = a.primary_hits(cfg.camera, W, Hh)
    iff, tf, _ = f.primary_hits(cfg.camera, W, Hh)
    assert np.array_equal(ia, iff) and np.array_equal(ta.view(np.uint32), tf.view(np.uint32))
    assert (a.export_triangle_attributes()[:, 15].view(np.uint32) != 0).any()
    a.close(); f.close()


@pytest.mark.parametrize("name", ["smooth_meshes", "smooth_c4"])
def test_aov_parity_on_identical_rays(rtb, ctx, name):
    F = rtb._ffi
    cfg, W, Hh = _cfgs()[name]
    cs = rtb.compile_scene(cfg.world, cfg.lights)
    dev = rtb.Scene(ctx, cs)
    osc = mesh_attr_oracle.OracleScene(cs)
    osc.attach_bvh(dev)
    seed = 3
    for s0 in (0, 5):
        prm = rtb.make_params(W, Hh, 1, cfg.max_depth, cfg.background, seed=seed, sample_offset=s0)
        sums, st = dev.render_aov(cfg.camera, prm)
        assert st["paths"] == W * Hh and st["rejected"] == 0
        px = np.arange(W * Hh, dtype=np.uint32)
        words = ctx.kat(F.KAT_CAMERA_RAY, np.stack([px, np.full_like(px, s0)], 1), 7, cam=cfg.camera, params=prm)
        ray = words.view(np.float32).astype(np.float64)
        _, ref, kinds = osc.aov_rays(ray[:, 0:3], ray[:, 3:6], ray[:, 6], px, s0, seed, cfg.background)
        got = sums.reshape(-1, 8).astype(np.float64)
        assert np.array_equal(got[:, 3], ref[:, 3])
        cov = got[:, 3] == 1.0
        nerr = np.abs(got[:, 4:7] - ref[:, 4:7]).max(1)[cov]
        aerr = np.abs(got[:, 0:3] - ref[:, 0:3]).max(1)
        solid = (kinds == 0) | (kinds == 0xFF)
        img = cov & (kinds == 3)
        img_bad = float((aerr[img] > 1e-4).mean()) if img.any() else 0.0
        print(f"{name} sample {s0}: normal max {nerr.max():.2e}, share > 1e-4 {(nerr > 1e-4).mean():.2e}; "
              f"solid albedo {aerr[solid].max(initial=0):.2e}; image albedo over 1e-4 on {img_bad:.2e} of {int(img.sum())}")
        assert (nerr <= 1e-4).mean() >= 0.999 and nerr.max() <= 1e-3
        assert np.all(aerr[solid] <= 1e-5)
        assert img_bad <= 1e-3
    dev.close()


def _identity_pair(rtb):
    """A textured height field: no attributes, and face normals + corner UVs as attributes."""
    from ray_tracer_archive_b200 import scenes, scene as S
    cfg = scenes.config_mesh(nx=40, nz=20)
    verts, tris = scenes.heightfield_mesh(40, 20)
    img = scenes.synthetic_earth(64, 32)
    mat = S.Lambertian.construct_texture(S.ImageTexture.construct(img, 64, 32))
    walls = cfg.world.objects[:6]
    v = verts.astype(np.float64)
    fn = np.cross(v[tris[:, 1]] - v[tris[:, 0]], v[tris[:, 2]] - v[tris[:, 0]])
    m = len(tris)
    flat = S.TriangleMesh(verts, tris, mat)
    attr = S.TriangleMesh(verts, tris, mat, normals=fn.astype(np.float32),
                          normal_indices=np.repeat(np.arange(m, dtype=np.uint32)[:, None], 3, 1),
                          uvs=np.array([[0, 0], [1, 0], [0, 1]], np.float32),
                          uv_indices=np.tile(np.arange(3, dtype=np.uint32), (m, 1)))
    return cfg, S.HittableList(walls + [flat]), S.HittableList(walls + [attr])


def test_face_normals_and_corner_uvs_render_like_no_attributes(rtb, ctx):
    cfg, wf, wa = _identity_pair(rtb)
    W, Hh, spp = 192, 108, 64
    prm = rtb.make_params(W, Hh, spp, cfg.max_depth, cfg.background, seed=21)
    f = rtb.Scene(ctx, rtb.compile_scene(wf, cfg.lights))
    a = rtb.Scene(ctx, rtb.compile_scene(wa, cfg.lights))
    accf, stf = f.render(cfg.camera, prm)
    acca, sta = a.render(cfg.camera, prm)
    mf, _ = H.image_stats(accf, spp)
    ma, _ = H.image_stats(acca, spp)
    close = (np.abs(ma - mf) <= 2e-3 * (np.abs(mf) + 1e-3)).mean()
    seg = sta["segments"] / stf["segments"]
    print(f"identity: {100 * close:.3f} % of pixels within 0.2 %, segments attr / flat {seg:.7f}")
    assert close >= 0.999
    assert abs(seg - 1.0) < 1e-5
    f.close(); a.close()


def _p2(rtb, ctx, cfg, W, Hh, spp):
    cs = rtb.compile_scene(cfg.world, cfg.lights)
    dev = rtb.Scene(ctx, cs)
    osc = mesh_attr_oracle.OracleScene(cs)
    osc.attach_bvh(dev)
    acc, st = dev.render(cfg.camera, rtb.make_params(W, Hh, spp, cfg.max_depth, cfg.background, seed=3))
    oacc, oseg, orej = osc.render(cfg.camera, rtb.make_params(W, Hh, spp, cfg.max_depth, cfg.background, seed=1234))
    mean_rel, z, se_rel = H.compare_images(acc, oacc, spp, spp)
    print(f"{cfg.name}: {W}x{Hh}x{spp} mean-lum err {100 * mean_rel:.3f}% (MC s.e. {100 * se_rel:.3f}%)  max z {z.max():.2f}"
          f"  segments gpu/oracle {st['segments'] / oseg:.4f}")
    assert st["paths"] == W * Hh * spp
    assert se_rel < 0.004
    assert mean_rel <= 0.01
    assert z.max() <= 5.0
    assert abs(st["segments"] / oseg - 1) < 0.01
    dev.close()


def test_p2_smooth_meshes(rtb, ctx):
    from ray_tracer_archive_b200 import scenes
    _p2(rtb, ctx, scenes.config_smooth_meshes(), 200, 200, 1024)


def test_p2_smooth_c4(rtb, ctx):
    from ray_tracer_archive_b200 import scenes
    _p2(rtb, ctx, scenes.config_mesh(smooth=True), 208, 117, 1024)


def test_call_order(rtb, ctx):
    """set_mesh clears the attributes; attributes set after a commit take effect when the graph is set and committed again."""
    cfg, W, Hh = _cfgs()["smooth_c4"]
    cs = rtb.compile_scene(cfg.world, cfg.lights)
    prm = rtb.make_params(W, Hh, 1, cfg.max_depth, cfg.background, seed=5)
    ref_flat = rtb.Scene(ctx, _flat(cs)).render_aov(cfg.camera, prm)[0]
    ref_smooth = rtb.Scene(ctx, cs).render_aov(cfg.camera, prm)[0]
    assert not np.array_equal(ref_flat[..., 4:7], ref_smooth[..., 4:7])
    s = rtb.Scene(ctx, cs)
    v, idx = cs.meshes[0]
    rtb._ffi.check(s.lib.rtb_scene_set_mesh(s.h, 0, rtb._ffi.ptr(v), len(v), rtb._ffi.ptr(idx), len(idx)))
    rtb._ffi.check(s.lib.rtb_scene_set_graph(s.h, rtb._ffi.ptr(cs.nodes), len(cs.nodes), rtb._ffi.ptr(cs.child_index),
                                             len(cs.child_index), cs.root))
    s.commit()
    assert np.array_equal(s.render_aov(cfg.camera, prm)[0], ref_flat)
    s.set_mesh_attributes(0, *cs.mesh_attrs[0])
    rtb._ffi.check(s.lib.rtb_scene_set_graph(s.h, rtb._ffi.ptr(cs.nodes), len(cs.nodes), rtb._ffi.ptr(cs.child_index),
                                             len(cs.child_index), cs.root))
    s.commit()
    assert np.array_equal(s.render_aov(cfg.camera, prm)[0], ref_smooth)
    s.close()


CHILD = r'''
import os, sys
sys.path.insert(0, os.environ["RTB_ROOT"])
import numpy as np
import ray_tracer_archive_b200 as rtb
from ray_tracer_archive_b200 import scenes
ctx = rtb.Context(0)
assert (ctx.check_failures() == 0).all(), "not a checked build"
for cfg in (scenes.config_smooth_meshes(), scenes.config_mesh(nx=200, nz=100, smooth=True)):
    sc = rtb.Scene(ctx, rtb.compile_scene(cfg.world, cfg.lights))
    for pool in (0, 1025):
        acc, st = sc.render(cfg.camera, rtb.make_params(96, 54, 12, cfg.max_depth, cfg.background, pool_paths=pool))
        assert st["paths"] == 96 * 54 * 12 and np.isfinite(acc).all()
    aov, st = sc.render_aov(cfg.camera, rtb.make_params(96, 54, 4, cfg.max_depth, cfg.background))
    assert np.isfinite(aov).all()
    sc.close()
f = ctx.check_failures()
print("check failures", f.tolist())
assert (f == 0).all(), f
ctx.close()
print("checked ok")
'''


def test_checked_build_smooth_scenes():
    lib = os.path.join(ROOT, "ray_tracer_archive_b200", "librtb200_checked.so")
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "ray_tracer_archive_b200", "csrc"), "checked"])
    env = dict(os.environ, RTB200_LIB=lib, RTB_ROOT=ROOT)
    out = subprocess.run([sys.executable, "-c", CHILD], env=env, capture_output=True, text=True, timeout=600)
    print(out.stdout.strip().splitlines()[-2:] if out.stdout else "")
    assert out.returncode == 0 and "checked ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
