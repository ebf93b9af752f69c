"""Small host-side I/O helpers around the hot path (SURVEY §8f "next" rows 2 and 3): an OBJ-style triangle-mesh loader
(the course hand-out asks for one, README.md:151-153 of the reference; the reference never implemented it) and an image
writer for the RGB8 output of `rtb_finalize_rgb8` (write_color, main.rs:141-169; the reference encodes a JPEG with the
`image` crate, main.rs:791-796 — here binary PPM, or PNG when PIL is importable)."""
from __future__ import annotations

import numpy as np

from .scene import Material, TriangleMesh


def load_obj(path_or_lines, mat: Material, scale: float = 1.0, offset=(0.0, 0.0, 0.0)) -> TriangleMesh:
    """Wavefront OBJ: `v x y z` and `f a b c ...` (1-based, negative = relative, `a/b/c` forms accepted; polygons are
    fan-triangulated).  Returns a TriangleMesh for the scene graph (-> rtb_scene_set_mesh)."""
    lines = open(path_or_lines).read().splitlines() if isinstance(path_or_lines, str) else list(path_or_lines)
    verts, tris = [], []
    for ln in lines:
        p = ln.split()
        if not p or p[0].startswith("#"):
            continue
        if p[0] == "v":
            verts.append([float(p[1]), float(p[2]), float(p[3])])
        elif p[0] == "f":
            idx = []
            for tok in p[1:]:
                i = int(tok.split("/")[0])
                idx.append(i - 1 if i > 0 else len(verts) + i)
            for k in range(1, len(idx) - 1):
                tris.append([idx[0], idx[k], idx[k + 1]])
    v = np.asarray(verts, dtype=np.float64) * scale + np.asarray(offset, dtype=np.float64)
    t = np.asarray(tris, dtype=np.uint32).reshape(-1, 3)
    if len(v) == 0 or len(t) == 0 or t.max() >= len(v):
        raise ValueError("OBJ has no triangles or references a missing vertex")
    return TriangleMesh(v.astype(np.float32), t, mat)


def save_image(path: str, rgb8: np.ndarray) -> None:
    """rgb8: (H, W, 3) uint8, row 0 = top (the layout rtb_finalize_rgb8 returns)."""
    a = np.ascontiguousarray(rgb8, dtype=np.uint8)
    if path.lower().endswith(".ppm"):
        with open(path, "wb") as f:
            f.write(b"P6\n%d %d\n255\n" % (a.shape[1], a.shape[0]))
            f.write(a.tobytes())
        return
    from PIL import Image  # PNG / JPEG (quality 100 like main.rs:720) when available
    Image.fromarray(a).save(path, quality=100)


# ---- denoiser guide images (rtb_render_aov) ----------------------------------------------------------------------------
def aov_images(sums: np.ndarray, spp: int) -> dict:
    """(H, W, 8) sums of rtb_render_aov over `spp` samples -> {"albedo" (H,W,3), "normal" (H,W,3), "depth" (H,W),
    "coverage" (H,W)} float32.  Albedo, normal and coverage are means over the samples; depth is the mean over the samples
    that hit something (0 where none did).  The normal is the mean of unit vectors, so it is shorter than 1 at edges."""
    a = np.asarray(sums, dtype=np.float32)
    if a.ndim != 3 or a.shape[2] != 8:
        raise ValueError("AOV sums must have shape (H, W, 8)")
    if spp <= 0:
        raise ValueError("spp must be > 0")
    inv = np.float32(1.0 / spp)
    cover = a[..., 3]
    depth = np.zeros_like(cover)
    np.divide(a[..., 7], cover, out=depth, where=cover > 0)
    return {"albedo": a[..., 0:3] * inv, "normal": a[..., 4:7] * inv, "depth": depth, "coverage": cover * inv}


def save_pfm(path: str, img: np.ndarray) -> None:
    """Portable float map: (H, W) -> "Pf", (H, W, 3) -> "PF"; row 0 = top as everywhere here.  Written little-endian
    (negative scale) with rows bottom-up, as the format stores them; OIDN's example tool reads it."""
    a = np.asarray(img, dtype=np.float32)
    if a.ndim == 3 and a.shape[2] == 1:
        a = a[..., 0]
    if not (a.ndim == 2 or (a.ndim == 3 and a.shape[2] == 3)):
        raise ValueError("PFM takes (H, W) or (H, W, 3) images")
    with open(path, "wb") as f:
        f.write(b"%s\n%d %d\n-1.0\n" % (b"Pf" if a.ndim == 2 else b"PF", a.shape[1], a.shape[0]))
        f.write(np.ascontiguousarray(a[::-1], dtype="<f4").tobytes())


# ---- checkpoint / resume of the accumulation buffer (SURVEY §8f row 3: "resume = add more spp") -----------------------
# The accumulation buffer holds SUMS over samples (main.rs:767-781) and samples are keyed by their global index, so a
# render can be continued later — or on another GPU — by loading the sums, passing sample_offset = samples already
# done and RTB_RENDER_ACCUMULATE to rtb_render_device.
def save_checkpoint(path: str, accum: np.ndarray, spp_done: int, seed: int, **meta) -> None:
    """accum: (H, W, 4) float32 sums (ΣR, ΣG, ΣB, ΣY²) as returned by rtb_render / read back from the device buffer."""
    a = np.ascontiguousarray(accum, dtype=np.float32)
    if a.ndim != 3 or a.shape[2] != 4:
        raise ValueError("accum must have shape (H, W, 4)")
    np.savez(path, accum=a, spp_done=np.int64(spp_done), seed=np.int64(seed),
             meta=np.array(repr(sorted(meta.items()))))


def load_checkpoint(path: str, width: int | None = None, height: int | None = None, seed: int | None = None):
    """-> (accum (H, W, 4) float32, spp_done).  Raises if the image size or seed does not match the render being resumed
    (a different seed is a different sample set: its sums must not be mixed with this one's sample indices)."""
    with np.load(path if path.endswith(".npz") else path + ".npz") as z:
        a, done, sd = z["accum"], int(z["spp_done"]), int(z["seed"])
    if a.ndim != 3 or a.shape[2] != 4:
        raise ValueError("not an rtb200 checkpoint")
    if (height is not None and a.shape[0] != height) or (width is not None and a.shape[1] != width):
        raise ValueError(f"checkpoint is {a.shape[1]}x{a.shape[0]}, render is {width}x{height}")
    if seed is not None and sd != seed:
        raise ValueError(f"checkpoint was rendered with seed {sd}, not {seed}")
    return np.ascontiguousarray(a, dtype=np.float32), done
