"""GPU tier (-m gpu): the denoiser guide buffers (rtb_render_aov) against the f64 oracle on identical rays, their
composition over sample ranges and pools, the render being left alone, the error paths and the bounds-checked build.

Parity on identical rays (one sample per pixel, sample_offset 0 and 5): the device's own f32 camera rays of those samples
(RTB_KAT_CAMERA_RAY) are traced by the oracle with the same (pixel, sample, seed) stream (tests/oracle_aov.cpp).
Bars: coverage equal on every pixel of media-free scenes and on all but 1e-4 of the pixels of media scenes.  Where both
sides hit:
- depth of a surface hit within 1e-5 relative (P1's bar on t);
- depth of a medium scatter point within 1e-5 relative + 1e-6 / density: the device draws -log(xi) with the fast log,
  whose absolute error (~2^-22) the distance 1/density * -log(xi) scales;
- surface normals within 1e-4 per component, (0, 0, 0) at a scatter point;
- albedo of solid colours (and of dielectrics, emitters, misses) within 1e-5;
- checker and image albedo within 1e-4 on >= 99.9 % of the pixels (a checker sign or a texel index flips where the f32
  and f64 hit points straddle a boundary); noise albedo within 1e-4 + 512 ulp(|p|) on >= 99.9 %: the f32 hit point's
  rounding goes through seven octaves of turbulence and a sine (the render's shade kernels evaluate the same f32 noise).
Measured on a B200 over the scenes below: coverage equal on every pixel (media scenes included); surface depth <= 1.3e-6
relative (C1); medium depth <= 2.2e-3 absolute at 1/density = 1e4 (C3's mist), i.e. 2.2e-7 / density; normals <= 6.5e-5
(C1, C3: (p - c) / r of an f32 hit point on large spheres; <= 1.1e-5 elsewhere); solid albedo <= 3e-8; checker <= 1.2e-5; image <= 7.5e-8 apart from
texel flips on <= 5e-4 of the textured pixels; noise <= 4.5e-5 at |p| <= 51 (two_perlin_spheres) and <= 3.4e-3 at
|p| ~ 360 (C3's marble sphere), at most 330 ulp(|p|).
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import aov_oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fuzz_cfg(rtb, scenes, S, seed):
    from test_gpu_fuzz import _random_scene
    dim, extended = seed % 24 >= 12, seed % 2 == 1  # the halves / odd seeds of test_gpu_fuzz
    world, lights = _random_scene(seed, S, scenes, dim, extended)
    cfg = scenes.config_cornell()
    cfg.world, cfg.lights, cfg.name = world, lights, f"random scene graph {seed}"
    cfg.background = (0.03, 0.04, 0.06) if dim else (0.55, 0.65, 0.85)
    cfg.camera = rtb.Camera.new((2.0, 7.0, 19.0), (0.0, 2.0, 0.0), (0, 1, 0), 40.0, 1.5, 0.3 if extended else 0.0, 19.0, 0.0, 1.0)
    return cfg


def _rotated_earth_cfg(rtb, scenes, S):
    img = scenes.earthmap()
    globe = S.Sphere.construct((0.0, 0.0, 0.0), 2.0, S.Lambertian.construct_texture(S.ImageTexture.construct(img, img.shape[1], img.shape[0])))
    world = S.HittableList([S.Translate.construct(S.RotateY.construct(globe, 75.0), (0.5, 0.2, -0.3)),
                            S.Translate.construct(S.RotateY.construct(S.Sphere.construct((4.5, 0.0, 0.0), 1.0, S.Lambertian.construct_texture(
                                S.ImageTexture.construct(scenes.synthetic_earth(64, 32), 64, 32))), -130.0), (0.0, 0.0, 0.0))])
    cfg = scenes.config_cornell()
    cfg.world, cfg.lights, cfg.name, cfg.background = world, None, "rotated earth", (0.7, 0.8, 1.0)
    cfg.camera = rtb.Camera.new((13, 2, 3), (0, 0, 0), (0, 1, 0), 24.0, 1.5, 0.0, 10.0)
    return cfg


_SIDE = ((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, 1.5, 0.0, 10.0)
_FUZZ_SEEDS = (0, 1, 5, 12, 13, 17)  # both halves of test_gpu_fuzz's seeds; the odd ones have a thin lens
# name -> image size of the parity run
_SIZES = {"C1": (400, 225), "C2": (200, 200), "C3": (200, 200), "cornell_smoke": (160, 160), "earth": (192, 128),
          "two_perlin_spheres": (192, 128), "rotated_earth": (240, 160), "mesh_cornell": (192, 108),
          **{f"fuzz{s}": (192, 128) for s in _FUZZ_SEEDS}}


def _make_cfg(rtb, name):
    from ray_tracer_archive_b200 import scenes, scene as S
    if name == "C1":
        return scenes.config_random_spheres()
    if name == "C2":
        return scenes.config_cornell()
    if name == "C3":  # media, noise, the earth image, moving spheres, an open shutter
        return scenes.config_final_scene()
    if name == "mesh_cornell":
        return scenes.config_mesh(nx=200, nz=100)
    if name == "rotated_earth":
        return _rotated_earth_cfg(rtb, scenes, S)
    if name.startswith("fuzz"):
        return _fuzz_cfg(rtb, scenes, S, int(name[4:]))
    cfg = scenes.config_cornell()
    cfg.name = name
    if name == "cornell_smoke":
        cfg.world, cfg.lights = scenes.cornell_smoke(), scenes.cornell_smoke_lights()
    else:
        cfg.world, cfg.lights, cfg.camera, cfg.background = getattr(scenes, name)(), None, rtb.Camera.new(*_SIDE), (0.7, 0.8, 1.0)
    return cfg


def _parity(rtb, ctx, cfg, W, Hh, seed=3):
    F = rtb._ffi
    cs = rtb.compile_scene(cfg.world, cfg.lights)
    dev = rtb.Scene(ctx, cs)
    osc = aov_oracle.OracleScene(cs)
    osc.attach_bvh(dev)  # candidate culling only: the per-primitive tests stay the oracle's
    media = dev.info()["n_media"] > 0
    inv_density = max([1.0 / n["p"][0] for n in cs.nodes if n["type"] == F.NODE_CONSTANT_MEDIUM], default=0.0)
    for s0 in (0, 5):
        prm = rtb.make_params(W, Hh, 1, cfg.max_depth, cfg.background, seed=seed, sample_offset=s0)
        sums, st = dev.render_aov(cfg.camera, prm)
        assert st["paths"] == W * Hh and st["segments"] == W * Hh and st["rejected"] == 0
        px = np.arange(W * Hh, dtype=np.uint32)
        words = ctx.kat(F.KAT_CAMERA_RAY, np.stack([px, np.full_like(px, s0)], 1), 7, cam=cfg.camera, params=prm)
        ray = words.view(np.float32).astype(np.float64)
        _, ref, kinds = osc.aov_rays(ray[:, 0:3], ray[:, 3:6], ray[:, 6], px, s0, seed, cfg.background)
        got = sums.reshape(-1, 8).astype(np.float64)
        cov_diff = got[:, 3] != ref[:, 3]
        both = (got[:, 3] == 1.0) & (ref[:, 3] == 1.0)
        medium = both & (np.abs(ref[:, 4:7]).sum(1) == 0)  # a scatter point has no normal
        surf = both & ~medium
        derr = np.abs(got[:, 7] - ref[:, 7])
        nerr = np.abs(got[:, 4:7] - ref[:, 4:7]).max(1)
        aerr = np.abs(got[:, 0:3] - ref[:, 0:3]).max(1)
        solid = ~cov_diff & ((kinds == 0) | (kinds == 0xFF))
        pmax = np.abs(ray[:, 0:3] + (ref[:, 7] / np.linalg.norm(ray[:, 3:6], axis=1))[:, None] * ray[:, 3:6]).max(1)
        tex_tol = np.where(kinds == 2, 1e-4 + 512.0 * np.spacing(pmax.astype(np.float32)), 1e-4)
        tex = both & (kinds != 0) & (kinds != 0xFF)
        tex_bad = float((aerr[tex] > tex_tol[tex]).mean()) if tex.any() else 0.0
        print(f"{cfg.name} sample {s0}: coverage differs on {int(cov_diff.sum())} of {len(px)}, "
              f"surface depth rel {(derr[surf] / ref[surf, 7]).max(initial=0):.2e}, "
              f"medium depth abs {derr[medium].max(initial=0):.2e} (1/density {inv_density:g}), "
              f"normal {nerr[surf].max(initial=0):.2e}, solid albedo {aerr[solid].max(initial=0):.2e}, "
              f"textured albedo over its bar on {tex_bad:.2e} of {int(tex.sum())}")
        if media:
            assert cov_diff.mean() <= 1e-4, np.argwhere(cov_diff).ravel()[:8]
        else:
            assert not cov_diff.any(), np.argwhere(cov_diff).ravel()[:8]
        assert np.all(derr[surf] <= 1e-5 * ref[surf, 7])
        assert np.all(derr[medium] <= 1e-5 * ref[medium, 7] + 1e-6 * inv_density)
        assert np.all(nerr[surf] <= 1e-4) and np.all(got[medium, 4:7] == 0.0)
        assert np.all(aerr[solid] <= 1e-5)
        assert tex_bad <= 1e-3
    dev.close()


@pytest.mark.parametrize("name", list(_SIZES))
def test_aov_parity_on_identical_rays(rtb, ctx, name):
    _parity(rtb, ctx, _make_cfg(rtb, name), *_SIZES[name])


def _close(a, b):
    np.testing.assert_allclose(a, b, rtol=1e-6, atol=1e-6)


def test_aov_sums_compose(rtb, ctx):
    """spp 8 in one call == spp 3 + spp 5 (ACCUMULATE) == eight spp 1 calls; pools of 1024, 1025 slots and the default
    give the same sums; the device entry on a non-default torch stream gives the host entry's sums."""
    import torch
    from ray_tracer_archive_b200 import scenes
    F = rtb._ffi
    cfg = scenes.config_cornell()
    cfg.world, cfg.lights = scenes.cornell_smoke(), scenes.cornell_smoke_lights()  # media draw from the sample's stream
    dev = rtb.Scene(ctx, rtb.compile_scene(cfg.world, cfg.lights))
    W, Hh, seed = 72, 56, 11
    prm = lambda spp, off=0, pool=0, flags=0: rtb.make_params(W, Hh, spp, cfg.max_depth, cfg.background, seed=seed,
                                                              sample_offset=off, pool_paths=pool, flags=flags)
    a8, st = dev.render_aov(cfg.camera, prm(8))
    assert st["paths"] == W * Hh * 8 and st["segments"] == W * Hh * 8 and st["extend_launches"] >= 1
    assert a8[..., 3].max() == 8.0 and a8[..., 3].min() >= 0.0
    dev.render_aov(cfg.camera, prm(3))
    b, st = dev.render_aov(cfg.camera, prm(5, 3, flags=F.RENDER_ACCUMULATE))
    assert st["paths"] == W * Hh * 5
    _close(b, a8)
    ones = sum(dev.render_aov(cfg.camera, prm(1, k))[0].astype(np.float64) for k in range(8))
    _close(ones, a8)
    for pool in (1024, 1025):
        p, st = dev.render_aov(cfg.camera, prm(8, pool=pool))
        assert st["paths"] == W * Hh * 8 and st["extend_launches"] >= W * Hh * 8 // pool
        _close(p, a8)
    t = torch.full((Hh, W, 8), float("nan"), device=f"cuda:{ctx.device_id}", dtype=torch.float32)
    s = torch.cuda.Stream(device=ctx.device_id)
    with torch.cuda.stream(s):
        st = dev.render_aov_device(cfg.camera, prm(8), t.data_ptr(), s.cuda_stream)
    s.synchronize()
    assert st["paths"] == W * Hh * 8
    _close(t.cpu().numpy(), a8)
    dev.close()


@pytest.mark.parametrize("pool", [0, 3000])
def test_render_unchanged_by_aov_pass(rtb, ctx, pool):
    """A seeded C2 render before and after an AOV pass on the same context: equal segments, buffers within 1e-6."""
    from ray_tracer_archive_b200 import scenes
    cfg = scenes.config_cornell()
    dev = rtb.Scene(ctx, rtb.compile_scene(cfg.world, cfg.lights))
    prm = rtb.make_params(96, 96, 16, cfg.max_depth, cfg.background, seed=9, pool_paths=pool)
    acc1, st1 = dev.render(cfg.camera, prm)
    _, ast = dev.render_aov(cfg.camera, prm)
    assert ast["paths"] == 96 * 96 * 16
    acc2, st2 = dev.render(cfg.camera, prm)
    assert st1["segments"] == st2["segments"] and st1["paths"] == st2["paths"]
    np.testing.assert_allclose(acc2, acc1, rtol=1e-6, atol=1e-6)
    dev.close()


def test_aov_errors(rtb, ctx):
    from ray_tracer_archive_b200 import scenes
    F = rtb._ffi
    lib = F.load()
    cfg = scenes.config_cornell()
    cs = rtb.compile_scene(cfg.world, cfg.lights)
    dev = rtb.Scene(ctx, cs)
    buf = np.zeros(8 * 16 * 16, np.float32)

    def rc(scene=dev, cam=cfg.camera, W=16, Hh=16, spp=1, off=0, flags=0, out=buf, device=False):
        p = rtb.make_params(W, Hh, spp, cfg.max_depth, cfg.background, sample_offset=off, flags=flags)
        cp = C.byref(cam) if cam is not None else None
        if device:
            return lib.rtb_render_aov_device(ctx.h, scene.h, cp, C.byref(p), None, None, None)
        return lib.rtb_render_aov(ctx.h, scene.h, cp, C.byref(p), F.ptr(out), None)

    assert rc() == 0
    loose = rtb.Scene(ctx)
    loose.set_compiled(cs)  # never committed
    assert rc(scene=loose) == -4
    assert rc(W=1) == -1 and rc(Hh=1) == -1
    assert rc(spp=0) == -1
    assert rc(off=(1 << 24)) == -1 and rc(off=(1 << 24) - 1) == 0
    same = rtb.Camera.new((1, 1, 1), (1, 1, 1), (0, 1, 0), 40.0, 1.0, 0.0, 10.0)
    assert rc(cam=same) == -1
    assert rc(cam=None) == -1
    assert rc(device=True) == -1  # NULL device buffer
    for flag in (F.RENDER_COUNT, F.RENDER_TIME_EXTEND, F.RENDER_REDUCE):
        assert rc(flags=flag) == -1
        assert b"RTB_RENDER_ACCUMULATE" in lib.rtb_last_error()
    assert rc(flags=F.RENDER_ACCUMULATE) == 0
    loose.close()
    dev.close()


def test_aov_multi_device_context_unsupported(rtb):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from ray_tracer_archive_b200 import scenes
    cfg = scenes.config_cornell()
    mctx = rtb.Context([0, 1])
    dev = rtb.Scene(mctx, rtb.compile_scene(cfg.world, cfg.lights))
    with pytest.raises(rtb.RtbError) as e:
        dev.render_aov(cfg.camera, rtb.make_params(16, 16, 2))
    assert e.value.code == -5
    dev.close()
    mctx.close()


CHILD = r'''
import os, sys
sys.path.insert(0, os.environ["RTB_ROOT"])
import numpy as np
import ray_tracer_archive_b200 as rtb
from ray_tracer_archive_b200 import scenes
ctx = rtb.Context(0)
assert (ctx.check_failures() == 0).all(), "not a checked build"
smoke = scenes.config_cornell(); smoke.world, smoke.lights, smoke.name = scenes.cornell_smoke(), scenes.cornell_smoke_lights(), "cornell_smoke"
cfgs = [scenes.config_cornell(), scenes.config_random_spheres(), scenes.config_final_scene(), scenes.config_mesh(nx=200, nz=100), smoke]
for cfg in cfgs:
    sc = rtb.Scene(ctx, rtb.compile_scene(cfg.world, cfg.lights))
    for pool in (0, 1025):
        aov, st = sc.render_aov(cfg.camera, rtb.make_params(96, 54, 6, cfg.max_depth, cfg.background, pool_paths=pool))
        assert st["paths"] == 96 * 54 * 6 and np.isfinite(aov).all()
    sc.close()
f = ctx.check_failures()
print("check failures", f.tolist())
assert (f == 0).all(), f
ctx.close()
print("checked ok")
'''


def test_aov_checked_build_finds_no_out_of_bounds_index():
    lib = os.path.join(ROOT, "ray_tracer_archive_b200", "librtb200_checked.so")
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "ray_tracer_archive_b200", "csrc"), "checked"])
    env = dict(os.environ, RTB200_LIB=lib, RTB_ROOT=ROOT)
    out = subprocess.run([sys.executable, "-c", CHILD], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "checked ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
