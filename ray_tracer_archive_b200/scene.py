"""Host-side mirror of the reference's scene-construction API (raytracer/src/{sphere,moving_sphere,aarect,boxes,
hittable,hittable_list,bvh,constant_medium,material,texture,perlin}.rs).

Same names and argument meaning as the Rust constructors; instead of building trait objects each constructor records
one `rtb_node` (include/rtb200.h).  `compile()` serialises the graph into the arrays `rtb_scene_set_graph` consumes;
the flattening itself (instances -> world space, Box -> 6 quads, primitive ids in list order) is done by the
library's host C++ (csrc/flatten.cpp).  The test oracle consumes the very same records.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from . import _ffi as F


# ------------------------------------------------------------------------------------------------ textures
class Texture:
    pass


@dataclass(eq=False)
class SolidColor(Texture):  # texture.rs:12-38
    color: Sequence[float]


@dataclass(eq=False)
class CheckerTexture(Texture):  # texture.rs:40-69 (construct_color: two solid colours; construct: any two textures, :46-51)
    even: object  # colour triple or Texture
    odd: object

    @classmethod
    def construct_color(cls, c1, c2):
        return cls(c1, c2)

    @classmethod
    def construct(cls, ev: "Texture", od: "Texture"):
        return cls(ev, od)


@dataclass(eq=False)
class Perlin:  # perlin.rs:14-25,53-66: 256 unit vectors of U[-1,1]^3 + three Fisher-Yates permutations
    ranvec: np.ndarray
    perm_x: np.ndarray
    perm_y: np.ndarray
    perm_z: np.ndarray

    @classmethod
    def new(cls, rng: np.random.Generator):
        v = rng.uniform(-1.0, 1.0, size=(256, 3))
        v /= np.linalg.norm(v, axis=1, keepdims=True)

        def perm():
            p = np.arange(256, dtype=np.uint32)
            for i in range(255, 0, -1):  # perlin.rs:61-66, random_int(0, i) rt_weekend.rs:17-19
                target = int(math.floor(rng.random() * (i + 1)))
                p[i], p[target] = p[target], p[i]
            return p

        return cls(v, perm(), perm(), perm())


@dataclass(eq=False)
class NoiseTexture(Texture):  # texture.rs:71-96
    noise: Perlin
    scale: float

    @classmethod
    def construct(cls, scale, rng):
        return cls(Perlin.new(rng), scale)


@dataclass(eq=False)
class ImageTexture(Texture):  # texture.rs:98-141: RGB8, row-major from the top
    data: np.ndarray  # (h, w, 3) uint8, or empty
    width: int
    height: int

    @classmethod
    def construct(cls, data, width, height):
        return cls(np.ascontiguousarray(data, dtype=np.uint8).reshape(height, width, 3), width, height)


# ------------------------------------------------------------------------------------------------ materials
class Material:
    pass


def _tex(a) -> Texture:
    return a if isinstance(a, Texture) else SolidColor(tuple(float(x) for x in a))


@dataclass(eq=False)
class Lambertian(Material):  # material.rs:24-72
    albedo: Texture

    @classmethod
    def construct(cls, color):
        return cls(_tex(color))

    @classmethod
    def construct_texture(cls, tex):
        return cls(tex)


@dataclass(eq=False)
class Metal(Material):  # material.rs:74-108
    albedo: Texture
    fuzz: float

    @classmethod
    def construct(cls, albedo, fuzz):
        return cls(_tex(albedo), fuzz if fuzz < 1.0 else 1.0)


@dataclass(eq=False)
class Dielectric(Material):  # material.rs:110-156
    ir: float

    @classmethod
    def construct(cls, ir):
        return cls(ir)


@dataclass(eq=False)
class DiffuseLight(Material):  # material.rs:158-191
    emit: Texture

    @classmethod
    def construct_color(cls, c):
        return cls(_tex(c))


@dataclass(eq=False)
class Isotropic(Material):  # material.rs:193-220 (commented in the reference)
    albedo: Texture

    @classmethod
    def construct_color(cls, c):
        return cls(_tex(c))


# ------------------------------------------------------------------------------------------------ hittables
class Hittable:
    pass


@dataclass(eq=False)
class Sphere(Hittable):  # sphere.rs:19-25
    center: Sequence[float]
    radius: float
    mat: Material

    construct = classmethod(lambda cls, center, radius, mat: cls(center, radius, mat))


@dataclass(eq=False)
class MovingSphere(Hittable):  # moving_sphere.rs:18-34
    center0: Sequence[float]
    center1: Sequence[float]
    time0: float
    time1: float
    radius: float
    mat: Material

    construct = classmethod(lambda cls, c0, c1, t0, t1, r, m: cls(c0, c1, t0, t1, r, m))


@dataclass(eq=False)
class _AARect(Hittable):
    a0: float
    a1: float
    b0: float
    b1: float
    k: float
    mat: Material

    @classmethod
    def construct(cls, a0, a1, b0, b1, k, mat):
        return cls(a0, a1, b0, b1, k, mat)


class XyRect(_AARect):  # aarect.rs:19-29
    NODE = F.NODE_XY_RECT


class XzRect(_AARect):  # aarect.rs:69-79
    NODE = F.NODE_XZ_RECT


class YzRect(_AARect):  # aarect.rs:138-148
    NODE = F.NODE_YZ_RECT


@dataclass(eq=False)
class Box(Hittable):  # boxes.rs:18-76
    p0: Sequence[float]
    p1: Sequence[float]
    mat: Material

    construct = classmethod(lambda cls, p0, p1, mat: cls(p0, p1, mat))


@dataclass(eq=False)
class Triangle(Hittable):  # new (SURVEY §8a N1)
    v0: Sequence[float]
    v1: Sequence[float]
    v2: Sequence[float]
    mat: Material


@dataclass(eq=False)
class Quad(Hittable):  # new: RTTNW quad(Q, u, v)
    Q: Sequence[float]
    u: Sequence[float]
    v: Sequence[float]
    mat: Material


@dataclass(eq=False)
class TriangleMesh(Hittable):  # new: indexed mesh (OBJ-style), vertices f32
    """Optional shading attributes (rtb_scene_set_mesh_attributes): per-vertex `normals` (k, 3) for smooth shading and
    texture coordinates `uvs` (j, 2), each with its own (m, 3) index array as in OBJ; an index array of None reuses
    `indices` (the stream then has one entry per vertex)."""
    vertices: np.ndarray  # (n, 3) float32
    indices: np.ndarray   # (m, 3) uint32
    mat: Material
    normals: Optional[np.ndarray] = None
    uvs: Optional[np.ndarray] = None
    normal_indices: Optional[np.ndarray] = None
    uv_indices: Optional[np.ndarray] = None


@dataclass(eq=False)
class Translate(Hittable):  # hittable.rs:62-74
    ptr: Hittable
    offset: Sequence[float]

    construct = classmethod(lambda cls, p, displacement: cls(p, displacement))


@dataclass(eq=False)
class RotateY(Hittable):  # hittable.rs:99-144
    ptr: Hittable
    angle: float

    construct = classmethod(lambda cls, p, angle: cls(p, angle))


@dataclass(eq=False)
class FlipFace(Hittable):  # hittable.rs:183-193
    ptr: Hittable

    construct = classmethod(lambda cls, p: cls(p))


@dataclass(eq=False)
class ConstantMedium(Hittable):  # constant_medium.rs:8-29
    boundary: Hittable
    density: float
    color: Sequence[float]

    @classmethod
    def construct_color(cls, b, d, c):
        return cls(b, d, c)


@dataclass(eq=False)
class HittableList(Hittable):  # hittable_list.rs:14-37
    objects: List[Hittable] = field(default_factory=list)

    @classmethod
    def new(cls):
        return cls([])

    @classmethod
    def construct(cls, obj):
        return cls([obj])

    def add(self, obj):
        self.objects.append(obj)


@dataclass(eq=False)
class BVHNode(Hittable):  # bvh.rs:74-76 construct2(list, t0, t1): closest-hit semantics of the list
    src: HittableList
    time0: float = 0.0
    time1: float = 1.0

    @classmethod
    def construct2(cls, lst, t0, t1):
        return cls(lst, t0, t1)


# ------------------------------------------------------------------------------------------------ compile
@dataclass
class CompiledScene:
    nodes: np.ndarray        # NODE_DTYPE
    child_index: np.ndarray  # uint32
    root: int
    materials: np.ndarray    # MATERIAL_DTYPE
    textures: np.ndarray     # TEXTURE_DTYPE
    lights: np.ndarray       # LIGHT_DTYPE
    images: list             # [(h,w,3) uint8]
    perlins: list            # [Perlin]
    meshes: list             # [(verts f32 (n,3), idx u32 (m,3))]
    # per mesh: None, or (normals f32 (k,3) | None, normal idx u32 (m,3) | None, uvs f32 (j,2) | None, uv idx u32 (m,3) | None)
    mesh_attrs: list = field(default_factory=list)


class _Compiler:
    def __init__(self):
        self.nodes, self.children = [], []
        self.materials, self.textures = [], []
        self.images, self.perlins, self.meshes, self.mesh_attrs = [], [], [], []
        self._mat_ids, self._tex_ids = {}, {}
        self._keep = []  # keeps temporaries alive so id() keys stay unique

    def tex(self, t: Texture) -> int:
        if id(t) in self._tex_ids:
            return self._tex_ids[id(t)]
        self._keep.append(t)
        rec = dict(type=F.TEX_SOLID, even=F.RTB_NONE, odd=F.RTB_NONE, table=F.RTB_NONE, rgb=(0, 0, 0), scale=0.0)
        if isinstance(t, SolidColor):
            rec["rgb"] = tuple(t.color)
        elif isinstance(t, CheckerTexture):
            rec["type"] = F.TEX_CHECKER
            rec["even"] = self.tex(t.even if isinstance(t.even, Texture) else SolidColor(tuple(t.even)))
            rec["odd"] = self.tex(t.odd if isinstance(t.odd, Texture) else SolidColor(tuple(t.odd)))
        elif isinstance(t, NoiseTexture):
            rec["type"] = F.TEX_NOISE
            rec["scale"] = t.scale
            rec["table"] = len(self.perlins)
            self.perlins.append(t.noise)
        elif isinstance(t, ImageTexture):
            rec["type"] = F.TEX_IMAGE
            if t.data.size:
                rec["table"] = len(self.images)
                self.images.append(t.data)
        else:
            raise TypeError(f"unknown texture {t!r}")
        self.textures.append(rec)
        self._tex_ids[id(t)] = len(self.textures) - 1
        return len(self.textures) - 1

    def mat(self, m: Material) -> int:
        if id(m) in self._mat_ids:
            return self._mat_ids[id(m)]
        self._keep.append(m)
        if isinstance(m, Lambertian):
            rec = (F.MAT_LAMBERTIAN, self.tex(m.albedo), 0.0)
        elif isinstance(m, Metal):
            rec = (F.MAT_METAL, self.tex(m.albedo), m.fuzz)
        elif isinstance(m, Dielectric):
            rec = (F.MAT_DIELECTRIC, F.RTB_NONE, m.ir)
        elif isinstance(m, DiffuseLight):
            rec = (F.MAT_DIFFUSE_LIGHT, self.tex(m.emit), 0.0)
        elif isinstance(m, Isotropic):
            rec = (F.MAT_ISOTROPIC, self.tex(m.albedo), 0.0)
        else:
            raise TypeError(f"unknown material {m!r}")
        self.materials.append(rec)
        self._mat_ids[id(m)] = len(self.materials) - 1
        return len(self.materials) - 1

    def node(self, h: Hittable) -> int:
        p = [0.0] * 12
        kids: List[int] = []
        mat = F.RTB_NONE
        if isinstance(h, Sphere):
            ty, mat = F.NODE_SPHERE, self.mat(h.mat)
            p[0:4] = [*h.center, h.radius]
        elif isinstance(h, MovingSphere):
            ty, mat = F.NODE_MOVING_SPHERE, self.mat(h.mat)
            p[0:9] = [*h.center0, *h.center1, h.time0, h.time1, h.radius]
        elif isinstance(h, _AARect):
            ty, mat = h.NODE, self.mat(h.mat)
            p[0:5] = [h.a0, h.a1, h.b0, h.b1, h.k]
        elif isinstance(h, Box):
            ty, mat = F.NODE_BOX, self.mat(h.mat)
            p[0:6] = [*h.p0, *h.p1]
        elif isinstance(h, Triangle):
            ty, mat = F.NODE_TRIANGLE, self.mat(h.mat)
            p[0:9] = [*h.v0, *h.v1, *h.v2]
        elif isinstance(h, Quad):
            ty, mat = F.NODE_QUAD, self.mat(h.mat)
            p[0:9] = [*h.Q, *h.u, *h.v]
        elif isinstance(h, TriangleMesh):
            ty, mat = F.NODE_MESH, self.mat(h.mat)
            p[0] = float(len(self.meshes))
            self.meshes.append((np.ascontiguousarray(h.vertices, dtype=np.float32).reshape(-1, 3),
                                np.ascontiguousarray(h.indices, dtype=np.uint32).reshape(-1, 3)))
            a = lambda x, dt, k: None if x is None else np.ascontiguousarray(x, dtype=dt).reshape(-1, k)
            attrs = (a(h.normals, np.float32, 3), a(h.normal_indices, np.uint32, 3), a(h.uvs, np.float32, 2),
                     a(h.uv_indices, np.uint32, 3))
            self.mesh_attrs.append(None if attrs[0] is None and attrs[2] is None else attrs)
        elif isinstance(h, Translate):
            ty = F.NODE_TRANSLATE
            p[0:3] = list(h.offset)
            kids = [self.node(h.ptr)]
        elif isinstance(h, RotateY):
            ty = F.NODE_ROTATE_Y
            p[0] = h.angle
            kids = [self.node(h.ptr)]
        elif isinstance(h, FlipFace):
            ty = F.NODE_FLIP_FACE
            kids = [self.node(h.ptr)]
        elif isinstance(h, ConstantMedium):
            ty, mat = F.NODE_CONSTANT_MEDIUM, self.mat(Isotropic.construct_color(h.color))
            p[0] = h.density
            kids = [self.node(h.boundary)]
        elif isinstance(h, HittableList):
            ty = F.NODE_LIST
            kids = [self.node(o) for o in h.objects]
        elif isinstance(h, BVHNode):
            ty = F.NODE_BVH
            kids = [self.node(o) for o in h.src.objects]
        else:
            raise TypeError(f"unknown hittable {h!r}")
        first = len(self.children)
        self.children.extend(kids)
        self.nodes.append((ty, mat, first, len(kids), p))
        return len(self.nodes) - 1


def compile_scene(world: Hittable, lights: Optional[HittableList] = None) -> CompiledScene:
    """Serialise the graph.  `lights` is the reference's separate, untransformed proxy list (main.rs:669-686):
    only XzRect and Sphere implement pdf_value/random (aarect.rs:107-125, sphere.rs:75-90)."""
    c = _Compiler()
    root = c.node(world)
    nodes = np.zeros(len(c.nodes), dtype=F.NODE_DTYPE)
    for i, (ty, mat, first, n, p) in enumerate(c.nodes):
        nodes[i] = (ty, mat, first, n, p)
    mats = np.zeros(max(len(c.materials), 1), dtype=F.MATERIAL_DTYPE)[:len(c.materials)]
    for i, rec in enumerate(c.materials):
        mats[i] = rec
    texs = np.zeros(len(c.textures), dtype=F.TEXTURE_DTYPE)
    for i, r in enumerate(c.textures):
        texs[i] = (r["type"], r["even"], r["odd"], r["table"], r["rgb"], r["scale"])
    lrec = []
    for l in (lights.objects if lights is not None else []):
        if isinstance(l, XzRect):
            lrec.append((F.LIGHT_XZ_RECT, 0, [l.a0, l.a1, l.b0, l.b1, l.k]))
        elif isinstance(l, Sphere):
            lrec.append((F.LIGHT_SPHERE, 0, [*l.center, l.radius, 0.0]))
        else:
            raise TypeError("only XzRect and Sphere can be sampled as lights (hittable.rs:54-59 defaults)")
    larr = np.zeros(len(lrec), dtype=F.LIGHT_DTYPE)
    for i, r in enumerate(lrec):
        larr[i] = r
    return CompiledScene(nodes, np.asarray(c.children, dtype=np.uint32), root, mats, texs, larr, c.images, c.perlins,
                         c.meshes, c.mesh_attrs)
