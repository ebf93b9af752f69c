"""The reference's scene functions (raytracer/src/main.rs) restated with the mirrored constructors, plus the synthetic
configurations BASELINE.json names.  All randomness comes from a seeded numpy Generator (the reference is OS-seeded,
rt_weekend.rs:8-15, so only the distributions can match).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np

from . import _ffi as F
from .scene import (BVHNode, Box, ConstantMedium, Dielectric, DiffuseLight, FlipFace, HittableList, ImageTexture,
                    Lambertian, Metal, MovingSphere, NoiseTexture, CheckerTexture, RotateY, Sphere, Translate,
                    TriangleMesh, XyRect, XzRect, YzRect, Hittable)


@dataclass
class Config:
    name: str
    world: Hittable
    lights: Optional[HittableList]
    camera: F.Camera
    width: int
    height: int
    spp: int
    max_depth: int
    background: Tuple[float, float, float]


def _cam(lookfrom, lookat, vfov, aspect, aperture, focus=10.0, t0=0.0, t1=1.0):
    return F.Camera.new(lookfrom, lookat, (0.0, 1.0, 0.0), vfov, aspect, aperture, focus, t0, t1)


# ---------------------------------------------------------------------------------------------- C2: live scene
def cornell_box() -> HittableList:
    """main.rs:337-433, verbatim order (primitive ids 0..12)."""
    objects = HittableList.new()
    red = Lambertian.construct((0.65, 0.05, 0.05))
    white = Lambertian.construct((0.73, 0.73, 0.73))
    green = Lambertian.construct((0.12, 0.45, 0.15))
    light = DiffuseLight.construct_color((15.0, 15.0, 15.0))
    objects.add(YzRect.construct(0.0, 555.0, 0.0, 555.0, 555.0, green))
    objects.add(YzRect.construct(0.0, 555.0, 0.0, 555.0, 0.0, red))
    objects.add(FlipFace.construct(XzRect.construct(213.0, 343.0, 227.0, 332.0, 554.0, light)))
    objects.add(XzRect.construct(0.0, 555.0, 0.0, 555.0, 0.0, white))
    objects.add(XzRect.construct(0.0, 555.0, 0.0, 555.0, 555.0, white))
    objects.add(XyRect.construct(0.0, 555.0, 0.0, 555.0, 555.0, white))
    box1 = Box.construct((0.0, 0.0, 0.0), (165.0, 330.0, 165.0), white)
    box1 = RotateY.construct(box1, 15.0)
    box1 = Translate.construct(box1, (265.0, 0.0, 295.0))
    objects.add(box1)
    glass = Dielectric.construct(1.5)
    objects.add(Sphere.construct((190.0, 90.0, 190.0), 90.0, glass))
    return objects


def cornell_lights() -> HittableList:
    """main.rs:669-686: untransformed proxies — the area light and the glass sphere."""
    lights = HittableList.new()
    lights.add(XzRect.construct(213.0, 343.0, 227.0, 332.0, 554.0, DiffuseLight.construct_color((15.0, 15.0, 15.0))))
    lights.add(Sphere.construct((190.0, 90.0, 190.0), 90.0, Dielectric.construct(1.5)))
    return lights


def config_cornell(width=600, height=600, spp=1000) -> Config:
    cam = _cam((278.0, 278.0, -800.0), (278.0, 278.0, 0.0), 40.0, width / height, 0.0)  # main.rs:688-718
    return Config("C2 book-3 Cornell box, mixture pdf", cornell_box(), cornell_lights(), cam, width, height, spp, 50,
                  (0.0, 0.0, 0.0))


# ---------------------------------------------------------------------------------------------- C1: book-1 final
def random_scene(seed=1) -> HittableList:
    """main.rs:171-242 with the Metal / glass branches restored from the book (SURVEY §8c) and static spheres."""
    rng = np.random.default_rng(seed)
    world = HittableList.new()
    world.add(Sphere.construct((0.0, -1000.0, 0.0), 1000.0, Lambertian.construct((0.5, 0.5, 0.5))))
    for a in range(-11, 11):
        for b in range(-11, 11):
            choose_mat = rng.random()
            center = (a + 0.9 * rng.random(), 0.2, b + 0.9 * rng.random())
            if np.linalg.norm(np.subtract(center, (4.0, 0.2, 0.0))) > 0.9:
                if choose_mat < 0.8:
                    albedo = rng.random(3) * rng.random(3)
                    mat = Lambertian.construct(tuple(albedo))
                elif choose_mat < 0.95:
                    mat = Metal.construct(tuple(rng.uniform(0.5, 1.0, 3)), float(rng.uniform(0.0, 0.5)))
                else:
                    mat = Dielectric.construct(1.5)
                world.add(Sphere.construct(center, 0.2, mat))
    world.add(Sphere.construct((0.0, 1.0, 0.0), 1.0, Dielectric.construct(1.5)))
    world.add(Sphere.construct((-4.0, 1.0, 0.0), 1.0, Lambertian.construct((0.4, 0.2, 0.1))))
    world.add(Sphere.construct((4.0, 1.0, 0.0), 1.0, Metal.construct((0.7, 0.6, 0.5), 0.0)))
    return world


def config_random_spheres(width=1200, height=675, spp=500, seed=1) -> Config:
    cam = _cam((13.0, 2.0, 3.0), (0.0, 0.0, 0.0), 20.0, width / height, 0.1)  # main.rs:706-709 defaults
    return Config("C1 book-1 final scene (random spheres)", random_scene(seed), None, cam, width, height, spp, 50,
                  (0.70, 0.80, 1.00))


# ---------------------------------------------------------------------------------------------- C3/C5: book-2 final
def earthmap() -> np.ndarray:
    """The reference's earthmap.jpg (main.rs:281,601) as raw RGB8 texels (512, 1024, 3): decoded once from
    /root/reference/earthmap.jpg by tests/golden/make_earthmap.py and committed as tests/golden/earthmap_rgb8.npz
    (RTB_EARTHMAP overrides the path).  Falls back to the seeded synthetic map only if that file is missing."""
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    path = os.environ.get("RTB_EARTHMAP", os.path.join(os.path.dirname(here), "tests", "golden", "earthmap_rgb8.npz"))
    if os.path.exists(path):
        return np.ascontiguousarray(np.load(path)["rgb"], dtype=np.uint8)
    return synthetic_earth()


def synthetic_earth(width=1024, height=512, seed=7) -> np.ndarray:
    """Seeded stand-in for an RGB8 map (used by tests that want a second image, and as earthmap()'s fallback)."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:height, 0:width]
    lon, lat = x / width * 2 * np.pi, (y / height - 0.5) * np.pi
    f = np.zeros((height, width))
    for k in range(1, 7):
        ph = rng.uniform(0, 2 * np.pi, 3)
        f += (np.sin(k * lon + ph[0]) * np.cos(k * lat * 1.3 + ph[1]) + 0.5 * np.sin(2 * k * lat + ph[2])) / k
    land = f > 0.25
    img = np.zeros((height, width, 3), dtype=np.uint8)
    img[..., 0] = np.where(land, 60 + 80 * np.clip(f, 0, 1), 10)
    img[..., 1] = np.where(land, 110 + 60 * np.clip(f, 0, 1), 40 + 30 * np.clip(-f, 0, 1))
    img[..., 2] = np.where(land, 40, 120 + 80 * np.clip(-f, 0, 1))
    return img


def final_scene(seed=1, boxes_per_side=20, n_small=1000, earth: Optional[np.ndarray] = None,
                flip_light=True) -> HittableList:
    """main.rs:521-649 (commented in the reference).  flip_light: the commented scene predates the front_face test in
    DiffuseLight::emitted (material.rs:184-190); with the live emitted() its un-flipped ceiling light would shine
    upward only, so it is wrapped in FlipFace exactly like the live cornell_box does (main.rs:360-362)."""
    rng = np.random.default_rng(seed)
    boxes1 = HittableList.new()
    ground = Lambertian.construct((0.48, 0.83, 0.53))
    for i in range(boxes_per_side):
        for j in range(boxes_per_side):
            w = 100.0
            x0, z0, y0 = -1000.0 + i * w, -1000.0 + j * w, 0.0
            x1, y1, z1 = x0 + w, float(rng.uniform(1.0, 101.0)), z0 + w
            boxes1.add(Box.construct((x0, y0, z0), (x1, y1, z1), ground))
    objects = HittableList.new()
    objects.add(BVHNode.construct2(boxes1, 0.0, 1.0))
    light = DiffuseLight.construct_color((7.0, 7.0, 7.0))
    lrect = XzRect.construct(123.0, 423.0, 147.0, 412.0, 554.0, light)
    objects.add(FlipFace.construct(lrect) if flip_light else lrect)
    center1 = (400.0, 400.0, 200.0)
    center2 = (430.0, 400.0, 200.0)
    objects.add(MovingSphere.construct(center1, center2, 0.0, 1.0, 50.0, Lambertian.construct((0.7, 0.3, 0.1))))
    objects.add(Sphere.construct((260.0, 150.0, 45.0), 50.0, Dielectric.construct(1.5)))
    objects.add(Sphere.construct((0.0, 150.0, 145.0), 50.0, Metal.construct((0.8, 0.8, 0.9), 1.0)))
    boundary = Sphere.construct((360.0, 150.0, 145.0), 70.0, Dielectric.construct(1.5))
    objects.add(boundary)
    objects.add(ConstantMedium.construct_color(boundary, 0.2, (0.2, 0.4, 0.9)))
    boundary2 = Sphere.construct((0.0, 0.0, 0.0), 5000.0, Dielectric.construct(1.5))
    objects.add(ConstantMedium.construct_color(boundary2, 0.0001, (1.0, 1.0, 1.0)))
    img = earth if earth is not None else earthmap()
    emat = Lambertian.construct_texture(ImageTexture.construct(img, img.shape[1], img.shape[0]))
    objects.add(Sphere.construct((400.0, 200.0, 400.0), 100.0, emat))
    pertext = NoiseTexture.construct(0.1, rng)
    objects.add(Sphere.construct((220.0, 280.0, 300.0), 80.0, Lambertian.construct_texture(pertext)))
    boxes2 = HittableList.new()
    white = Lambertian.construct((0.73, 0.73, 0.73))
    for _ in range(n_small):
        boxes2.add(Sphere.construct(tuple(rng.uniform(0.0, 165.0, 3)), 10.0, white))
    objects.add(Translate.construct(RotateY.construct(BVHNode.construct2(boxes2, 0.0, 1.0), 15.0),
                                    (-100.0, 270.0, 395.0)))
    return objects


def final_scene_lights() -> HittableList:
    lights = HittableList.new()
    lights.add(XzRect.construct(123.0, 423.0, 147.0, 412.0, 554.0, DiffuseLight.construct_color((7.0, 7.0, 7.0))))
    return lights


def config_final_scene(width=800, height=800, spp=10000, seed=1, **kw) -> Config:
    cam = _cam((478.0, 278.0, -600.0), (278.0, 278.0, 0.0), 40.0, width / height, 0.0)
    return Config("C3 book-2 final scene", final_scene(seed, **kw), final_scene_lights(), cam, width, height, spp, 50,
                  (0.0, 0.0, 0.0))


def config_scaling(width=3840, height=2160, spp=16384, seed=1) -> Config:
    c = config_final_scene(width, height, spp, seed)
    c.name = "C5 scaling sweep (book-2 final scene, 4K)"
    return c


# ---------------------------------------------------------------------------------------------- C4: mesh stress
def _value_noise(x, z, rng_table):
    xi, zi = np.floor(x).astype(np.int64), np.floor(z).astype(np.int64)
    fx, fz = x - xi, z - zi
    fx, fz = fx * fx * (3 - 2 * fx), fz * fz * (3 - 2 * fz)
    n = rng_table.shape[0]
    g = lambda a, b: rng_table[a % n, b % n]
    return (g(xi, zi) * (1 - fx) * (1 - fz) + g(xi + 1, zi) * fx * (1 - fz) + g(xi, zi + 1) * (1 - fx) * fz +
            g(xi + 1, zi + 1) * fx * fz)


def heightfield_mesh(nx=1000, nz=500, seed=1, x0=65.0, x1=490.0, z0=65.0, z1=490.0):
    """(nx x nz) cells = 2*nx*nz triangles, y = 150 + 80*fbm(x,z) (SURVEY §8d C4)."""
    rng = np.random.default_rng(seed)
    table = rng.uniform(-1.0, 1.0, size=(64, 64))
    xs = np.linspace(x0, x1, nx + 1)
    zs = np.linspace(z0, z1, nz + 1)
    X, Z = np.meshgrid(xs, zs, indexing="ij")
    f = np.zeros_like(X)
    amp, freq = 0.5, 1.0 / 60.0
    for _ in range(4):
        f += amp * _value_noise(X * freq, Z * freq, table)
        amp *= 0.5
        freq *= 2.0
    Y = 150.0 + 80.0 * f
    verts = np.stack([X, Y, Z], axis=-1).reshape(-1, 3).astype(np.float32)
    i, j = np.meshgrid(np.arange(nx), np.arange(nz), indexing="ij")
    v00 = (i * (nz + 1) + j).ravel()
    v10, v01, v11 = v00 + (nz + 1), v00 + 1, v00 + (nz + 1) + 1
    # counter-clockwise seen from above so the geometric normal points up
    tris = np.concatenate([np.stack([v00, v01, v11], 1), np.stack([v00, v11, v10], 1)], 0).astype(np.uint32)
    return verts, tris


def mesh_cornell(nx=1000, nz=500, seed=1, smooth=False) -> HittableList:
    objects = HittableList.new()
    red = Lambertian.construct((0.65, 0.05, 0.05))
    white = Lambertian.construct((0.73, 0.73, 0.73))
    green = Lambertian.construct((0.12, 0.45, 0.15))
    light = DiffuseLight.construct_color((15.0, 15.0, 15.0))
    objects.add(YzRect.construct(0.0, 555.0, 0.0, 555.0, 555.0, green))
    objects.add(YzRect.construct(0.0, 555.0, 0.0, 555.0, 0.0, red))
    objects.add(FlipFace.construct(XzRect.construct(213.0, 343.0, 227.0, 332.0, 554.0, light)))
    objects.add(XzRect.construct(0.0, 555.0, 0.0, 555.0, 0.0, white))
    objects.add(XzRect.construct(0.0, 555.0, 0.0, 555.0, 555.0, white))
    objects.add(XyRect.construct(0.0, 555.0, 0.0, 555.0, 555.0, white))
    verts, tris = heightfield_mesh(nx, nz, seed)
    from .io import vertex_normals
    objects.add(TriangleMesh(verts, tris, white, normals=vertex_normals(verts, tris) if smooth else None))
    return objects


def mesh_lights() -> HittableList:
    lights = HittableList.new()
    lights.add(XzRect.construct(213.0, 343.0, 227.0, 332.0, 554.0, DiffuseLight.construct_color((15.0, 15.0, 15.0))))
    return lights


def config_mesh(width=1920, height=1080, spp=1024, nx=1000, nz=500, seed=1, smooth=False) -> Config:
    """smooth=True: the height field carries area-weighted vertex normals (io.vertex_normals) and is shaded smooth."""
    cam = _cam((278.0, 278.0, -800.0), (278.0, 278.0, 0.0), 40.0, width / height, 0.0)
    return Config(f"C4 {2 * nx * nz}-triangle {'smooth ' if smooth else ''}mesh in a Cornell box",
                  mesh_cornell(nx, nz, seed, smooth), mesh_lights(), cam, width, height, spp, 50, (0.0, 0.0, 0.0))


def uv_sphere_mesh(center, radius, n_lon, n_lat, mat, uvs=True) -> TriangleMesh:
    """Latitude-longitude sphere: 2 poles + (n_lat - 1) rings of n_lon positions, shared along the seam, with unit
    vertex normals on the positions' own indices.  Texture coordinates (sphere.rs:32-37's u = phi / 2pi, v = theta / pi
    convention) live on their own index stream: the seam has u = 0 on one side and u = 1 on the other, and each pole
    triangle has its own pole texel column."""
    c = np.asarray(center, dtype=np.float64)
    theta = np.pi * np.arange(1, n_lat) / n_lat                  # polar angle from -y (v = theta / pi), rings only
    phi = 2.0 * np.pi * np.arange(n_lon) / n_lon                 # u = phi / 2pi
    T, P = np.meshgrid(theta, phi, indexing="ij")
    # sphere.rs:32-37: theta = acos(-y), phi = atan2(-z, x) + pi  ->  x = -cos(phi) sin(theta), z = sin(phi) sin(theta)
    ring = np.stack([-np.cos(P) * np.sin(T), -np.cos(T), np.sin(P) * np.sin(T)], -1).reshape(-1, 3)
    unit = np.concatenate([[[0.0, -1.0, 0.0]], ring, [[0.0, 1.0, 0.0]]])
    south, north = 0, len(unit) - 1
    pos = lambda i, j: 1 + i * n_lon + (j % n_lon)               # ring i, longitude j (the seam wraps to j = 0)
    # texture coordinates: (n_lat - 1) rings of n_lon + 1 (u = 1 duplicates the seam), then one pole texel per column
    uv_ring = np.stack(np.meshgrid(np.arange(n_lon + 1) / n_lon, theta / np.pi, indexing="xy"), -1).reshape(-1, 2)
    cols = (np.arange(n_lon) + 0.5) / n_lon
    uv = np.concatenate([uv_ring, np.stack([cols, np.zeros(n_lon)], 1), np.stack([cols, np.ones(n_lon)], 1)])
    tuv = lambda i, j: i * (n_lon + 1) + j
    s_uv, n_uv = (n_lat - 1) * (n_lon + 1), (n_lat - 1) * (n_lon + 1) + n_lon
    tri, tri_uv = [], []
    for j in range(n_lon):  # outward-facing winding: cross(e1, e2) points away from the centre
        tri.append([south, pos(0, j + 1), pos(0, j)]); tri_uv.append([s_uv + j, tuv(0, j + 1), tuv(0, j)])
        for i in range(n_lat - 2):
            tri.append([pos(i, j), pos(i, j + 1), pos(i + 1, j + 1)])
            tri_uv.append([tuv(i, j), tuv(i, j + 1), tuv(i + 1, j + 1)])
            tri.append([pos(i, j), pos(i + 1, j + 1), pos(i + 1, j)])
            tri_uv.append([tuv(i, j), tuv(i + 1, j + 1), tuv(i + 1, j)])
        tri.append([north, pos(n_lat - 2, j), pos(n_lat - 2, j + 1)])
        tri_uv.append([n_uv + j, tuv(n_lat - 2, j), tuv(n_lat - 2, j + 1)])
    verts = (c + radius * unit).astype(np.float32)
    return TriangleMesh(verts, np.asarray(tri, np.uint32), mat, normals=unit.astype(np.float32),
                        uvs=uv.astype(np.float32) if uvs else None,
                        uv_indices=np.asarray(tri_uv, np.uint32) if uvs else None)


def smooth_meshes(earth_img: Optional[np.ndarray] = None) -> HittableList:
    """The Cornell box of C4 (walls, light) holding three smooth-shaded meshes: an earthmap-textured UV sphere under
    RotateY + Translate, a mirror-metal sphere and a glass sphere, both coarse enough that flat facets would show."""
    objects = HittableList.new()
    for o in mesh_cornell(1, 1).objects[:6]:  # the walls and the light (the height field is left out)
        objects.add(o)
    img = earth_img if earth_img is not None else earthmap()
    earth_mat = Lambertian.construct_texture(ImageTexture.construct(img, img.shape[1], img.shape[0]))
    globe = uv_sphere_mesh((0.0, 0.0, 0.0), 110.0, 48, 24, earth_mat)
    objects.add(Translate.construct(RotateY.construct(globe, 40.0), (390.0, 110.0, 330.0)))
    objects.add(uv_sphere_mesh((150.0, 90.0, 160.0), 90.0, 16, 8, Metal.construct((0.8, 0.85, 0.88), 0.0), uvs=False))
    objects.add(uv_sphere_mesh((300.0, 330.0, 150.0), 70.0, 12, 6, Dielectric.construct(1.5), uvs=False))
    return objects


def config_smooth_meshes(width=400, height=400, spp=256) -> Config:
    cam = _cam((278.0, 278.0, -800.0), (278.0, 278.0, 0.0), 40.0, width / height, 0.0)
    return Config("smooth-shaded, UV-mapped meshes in a Cornell box", smooth_meshes(), mesh_lights(), cam, width,
                  height, spp, 50, (0.0, 0.0, 0.0))


# ---------------------------------------------------------------------------------------------- small regression scenes
def two_spheres() -> HittableList:  # main.rs:244-263
    objects = HittableList.new()
    checker = CheckerTexture.construct_color((0.2, 0.3, 0.1), (0.9, 0.9, 0.9))
    objects.add(Sphere.construct((0.0, -10.0, 0.0), 10.0, Lambertian.construct_texture(checker)))
    objects.add(Sphere.construct((0.0, 10.0, 0.0), 10.0, Lambertian.construct_texture(checker)))
    return objects


def two_perlin_spheres(seed=1) -> HittableList:  # main.rs:265-279
    objects = HittableList.new()
    pertext = NoiseTexture.construct(4.0, np.random.default_rng(seed))
    objects.add(Sphere.construct((0.0, -1000.0, 0.0), 1000.0, Lambertian.construct_texture(pertext)))
    objects.add(Sphere.construct((0.0, 2.0, 0.0), 2.0, Lambertian.construct_texture(pertext)))
    return objects


def earth(img: Optional[np.ndarray] = None) -> HittableList:  # main.rs:280-299
    img = img if img is not None else earthmap()
    surface = Lambertian.construct_texture(ImageTexture.construct(img, img.shape[1], img.shape[0]))
    return HittableList.construct(Sphere.construct((0.0, 0.0, 0.0), 2.0, surface))


def simple_light(seed=1) -> HittableList:  # main.rs:300-335
    objects = two_perlin_spheres(seed)
    difflight = DiffuseLight.construct_color((4.0, 4.0, 4.0))
    objects.add(XyRect.construct(3.0, 5.0, 1.0, 3.0, -2.0, difflight))
    objects.add(Sphere.construct((0.0, 7.0, 0.0), 2.0, difflight))
    return objects


def cornell_smoke(flip_light=True) -> HittableList:  # main.rs:435-519 (flip_light: see final_scene)
    objects = HittableList.new()
    red = Lambertian.construct((0.65, 0.05, 0.05))
    white = Lambertian.construct((0.73, 0.73, 0.73))
    green = Lambertian.construct((0.12, 0.45, 0.15))
    light = DiffuseLight.construct_color((7.0, 7.0, 7.0))
    objects.add(YzRect.construct(0.0, 555.0, 0.0, 555.0, 555.0, green))
    objects.add(YzRect.construct(0.0, 555.0, 0.0, 555.0, 0.0, red))
    lrect = XzRect.construct(113.0, 443.0, 127.0, 432.0, 554.0, light)
    objects.add(FlipFace.construct(lrect) if flip_light else lrect)
    objects.add(XzRect.construct(0.0, 555.0, 0.0, 555.0, 555.0, white))
    objects.add(XzRect.construct(0.0, 555.0, 0.0, 555.0, 0.0, white))
    objects.add(XyRect.construct(0.0, 555.0, 0.0, 555.0, 555.0, white))
    box1 = Translate.construct(RotateY.construct(Box.construct((0.0, 0.0, 0.0), (165.0, 330.0, 165.0), white), 15.0),
                               (265.0, 0.0, 295.0))
    box2 = Translate.construct(RotateY.construct(Box.construct((0.0, 0.0, 0.0), (165.0, 165.0, 165.0), white), -18.0),
                               (130.0, 0.0, 65.0))
    objects.add(ConstantMedium.construct_color(box1, 0.01, (0.0, 0.0, 0.0)))
    objects.add(ConstantMedium.construct_color(box2, 0.01, (1.0, 1.0, 1.0)))
    return objects


def cornell_smoke_lights() -> HittableList:
    lights = HittableList.new()
    lights.add(XzRect.construct(113.0, 443.0, 127.0, 432.0, 554.0, DiffuseLight.construct_color((7.0, 7.0, 7.0))))
    return lights
