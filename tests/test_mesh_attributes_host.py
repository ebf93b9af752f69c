"""CPU tier: smooth-shaded, UV-mapped meshes on the host side — io.load_obj's vn / vt streams, io.vertex_normals, the
argument checks of rtb_scene_set_mesh_attributes, and the leaf-ordered shading records the BVH build exports
(rtb_scene_export_triangle_attributes).  No device calls."""
import math

import numpy as np
import pytest

from ray_tracer_archive_b200 import io, scene as S

MAT = S.Lambertian.construct((0.5, 0.5, 0.5))
OBJ = ["v 0 0 0", "v 1 0 0", "v 1 1 0", "v 0 1 0", "v 0.5 2 1",
       "vt 0 0", "vt 1 0", "vt 1 1", "vt 0 1", "vt 0.5 0.5",
       "vn 0 0 1", "vn 0 0 2", "vn 1 0 1", "vn 0 1 1",
       "f 1/1/1 2/2/2 3/3/3 4/4/4",      # quad: fan-triangulated in every stream
       "f -1/-1/-1 3/3/2 4/4/3"]         # negative (relative) indices


def test_load_obj_every_face_form_and_stream():
    m = io.load_obj(OBJ, MAT, normals="file", uvs=True)
    assert m.indices.tolist() == [[0, 1, 2], [0, 2, 3], [4, 2, 3]]
    assert m.normal_indices.tolist() == [[0, 1, 2], [0, 2, 3], [3, 1, 2]]
    assert m.uv_indices.tolist() == [[0, 1, 2], [0, 2, 3], [4, 2, 3]]
    np.testing.assert_array_equal(m.normals[1], [0, 0, 2])  # as in the file: the library normalises
    np.testing.assert_array_equal(m.uvs[4], [0.5, 0.5])
    forms = ["v 0 0 0", "v 1 0 0", "v 0 1 0", "vt 0 0", "vt 1 0", "vt 0 1", "vn 0 0 1"]
    for face, want_uv, want_n in [("f 1 2 3", False, False), ("f 1/1 2/2 3/3", True, False),
                                  ("f 1//1 2//1 3//1", False, True), ("f 1/1/1 2/2/1 3/3/1", True, True)]:
        base = io.load_obj(forms + [face], MAT)
        assert base.normals is None and base.uvs is None and base.indices.tolist() == [[0, 1, 2]]
        if want_uv:
            assert io.load_obj(forms + [face], MAT, uvs=True).uv_indices.tolist() == [[0, 1, 2]]
        else:
            with pytest.raises(ValueError):
                io.load_obj(forms + [face], MAT, uvs=True)
        if want_n:
            assert io.load_obj(forms + [face], MAT, normals="file").normal_indices.tolist() == [[0, 0, 0]]
        else:
            with pytest.raises(ValueError):
                io.load_obj(forms + [face], MAT, normals="file")


def test_load_obj_defaults_unchanged_and_partial_streams_refused():
    plain = io.load_obj([ln for ln in OBJ if not ln.startswith(("vt", "vn"))], MAT)
    full = io.load_obj(OBJ, MAT)  # vn / vt present in the file but not asked for: exactly the flat mesh
    np.testing.assert_array_equal(full.vertices, plain.vertices)
    np.testing.assert_array_equal(full.indices, plain.indices)
    assert full.normals is None and full.uvs is None and full.normal_indices is None and full.uv_indices is None
    mixed = OBJ[:-1] + ["f 5 3 4"]  # the second face has no vt / vn
    with pytest.raises(ValueError):
        io.load_obj(mixed, MAT, normals="file")
    with pytest.raises(ValueError):
        io.load_obj(mixed, MAT, uvs=True)
    with pytest.raises(ValueError):
        io.load_obj(OBJ[:-1] + ["f 1/1/9 2/2/2 3/3/3"], MAT, normals="file")  # missing normal
    with pytest.raises(ValueError):
        io.load_obj(OBJ, MAT, normals="flat")


def test_load_obj_negative_scale_negates_file_normals():
    a = io.load_obj(OBJ, MAT, normals="file")
    b = io.load_obj(OBJ, MAT, normals="file", scale=-2.0)
    np.testing.assert_array_equal(b.normals, -a.normals)
    np.testing.assert_allclose(b.vertices, -2.0 * a.vertices)


def test_vertex_normals_smooth():
    m = io.load_obj(OBJ, MAT, normals="smooth")
    np.testing.assert_array_equal(m.normals, io.vertex_normals(m.vertices, m.indices))
    assert m.normal_indices is None
    # area weighting by hand: position 2 is shared by all three faces
    v = m.vertices.astype(np.float64)
    fn = [np.cross(v[b] - v[a], v[c] - v[a]) for a, b, c in m.indices]
    s = fn[0] + fn[1] + fn[2]
    np.testing.assert_allclose(m.normals[2], s / np.linalg.norm(s), atol=1e-7)
    # a position whose faces cancel gets a zero normal
    z = io.vertex_normals(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32), np.array([[0, 1, 2], [0, 2, 1]]))
    assert (z == 0).all()


def _host_scene(rtb, world):
    cs = rtb.compile_scene(world)
    s = rtb.Scene(None)
    s.set_compiled(cs)
    return s, cs


def test_set_mesh_attributes_argument_checks(rtb):
    lib = rtb._ffi.load()
    p = rtb._ffi.ptr
    verts = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0]], np.float32)
    idx = np.array([[0, 1, 2], [1, 3, 2]], np.uint32)
    s, _ = _host_scene(rtb, S.HittableList([S.TriangleMesh(verts, idx, MAT)]))
    n4 = np.array([[0, 0, 1]] * 4, np.float32)
    uv4 = np.zeros((4, 2), np.float32)
    ok_idx = np.array([[0, 0, 0], [0, 0, 0]], np.uint32)
    call = lambda mid, n, nn, ni, uv, nu, ui: lib.rtb_scene_set_mesh_attributes(s.h, mid, p(n), nn, p(ni), p(uv), nu, p(ui))
    assert call(0, n4, 4, None, uv4, 4, None) == 0
    assert call(0, n4[:1], 1, ok_idx, None, 0, None) == 0                # own index stream, normals only
    assert call(0, None, 0, None, uv4[:1], 1, ok_idx) == 0               # uvs only
    assert call(0, np.zeros((4, 3), np.float32), 4, None, None, 0, None) == 0  # a zero normal is accepted
    assert call(1, n4, 4, None, None, 0, None) == -1                     # mesh id not set
    assert call(99, n4, 4, None, None, 0, None) == -1
    assert call(0, n4[:3], 3, None, None, 0, None) == -1                 # NULL indices: one per vertex
    assert call(0, None, 0, None, uv4[:3], 3, None) == -1
    assert call(0, n4[:1], 1, np.array([[0, 0, 0], [0, 1, 0]], np.uint32), None, 0, None) == -1  # index out of range
    assert call(0, None, 0, None, uv4[:2], 2, np.array([[0, 0, 0], [0, 2, 0]], np.uint32)) == -1
    bad = n4.copy(); bad[2, 1] = np.nan
    assert call(0, bad, 4, None, None, 0, None) == -1                    # non-finite
    badu = uv4.copy(); badu[1, 0] = np.inf
    assert call(0, None, 0, None, badu, 4, None) == -1
    assert lib.rtb_scene_set_mesh_attributes(None, 0, None, 0, None, None, 0, None) == -1
    out = np.zeros((2, 16), np.float32)
    assert lib.rtb_scene_export_triangle_attributes(s.h, p(out), out.nbytes) == -4  # not built yet
    s.build_bvh()
    assert lib.rtb_scene_export_triangle_attributes(s.h, p(out), out.nbytes - 1) == -1
    assert lib.rtb_scene_export_triangle_attributes(s.h, None, 0) == -1


def _ry(theta_deg):
    t = math.radians(theta_deg)
    c, s = math.cos(t), math.sin(t)
    return np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]])


def _attr_world(with_attrs, theta=35.0):
    rng = np.random.default_rng(4)
    verts = rng.uniform(-1, 1, (40, 3)).astype(np.float32)
    idx = rng.integers(0, 40, (60, 3)).astype(np.uint32)
    normals = rng.normal(size=(25, 3)).astype(np.float32)
    n_idx = rng.integers(0, 25, (60, 3)).astype(np.uint32)
    uvs = rng.uniform(0, 1, (30, 2)).astype(np.float32)
    uv_idx = rng.integers(0, 30, (60, 3)).astype(np.uint32)
    mesh = S.TriangleMesh(verts, idx, MAT)
    if with_attrs:
        mesh.normals, mesh.normal_indices, mesh.uvs, mesh.uv_indices = normals, n_idx, uvs, uv_idx
    world = S.HittableList([S.Sphere((0, 5, 0), 1.0, MAT),
                            S.Translate.construct(S.RotateY.construct(S.FlipFace.construct(mesh), theta), (3.0, -1.0, 2.0)),
                            S.TriangleMesh(verts + 5, idx[:7], MAT)])  # a second mesh without attributes
    return world, (normals, n_idx, uvs, uv_idx)


def test_exported_records_transform_order_and_geometry(rtb):
    theta = 35.0
    wa, (normals, n_idx, uvs, uv_idx) = _attr_world(True, theta)
    wf, _ = _attr_world(False, theta)
    for opts in ({}, {"max_leaf_triangles": 3}):
        sa, sf = rtb.Scene(None), rtb.Scene(None)
        for s, w in ((sa, wa), (sf, wf)):
            s.set_compiled(rtb.compile_scene(w))
            if opts:
                s.set_build_options(**opts)
            s.build_bvh()
        na, pa = sa.export_bvh()
        nf, pf = sf.export_bvh()
        # geometry, BVH and info words are the same with and without attributes, bit 31 of attribute triangles aside
        assert np.array_equal(na, nf)
        for t in range(4):
            assert np.array_equal(pa[t][0], pf[t][0])
        for t in range(3):
            assert np.array_equal(pa[t][1], pf[t][1])
        ia, iff = pa[3][1].reshape(-1, 2), pf[3][1].reshape(-1, 2)
        assert np.array_equal(ia[:, 0], iff[:, 0]) and np.array_equal(ia[:, 1] & 0x7FFFFFFF, iff[:, 1])
        assert not (iff[:, 1] >> 31).any()
        rec = sa.export_triangle_attributes()
        assert rec.shape == (len(ia), 16)
        assert not sf.export_triangle_attributes().any()
        R = _ry(theta)
        nunit = normals.astype(np.float64) / np.linalg.norm(normals.astype(np.float64), axis=1, keepdims=True)
        first_mesh_id = 1  # the sphere is primitive 0; the attribute mesh's triangles follow in index order
        for k, (pid, word) in enumerate(ia):
            t = int(pid) - first_mesh_id
            flags = rec[k, 15:16].view(np.uint32)[0]
            if 0 <= t < 60:
                assert word >> 31 == 1 and flags == 3
                for q in range(3):
                    want = R @ nunit[n_idx[t, q]]
                    np.testing.assert_allclose(rec[k, 4 * q:4 * q + 3], want, atol=1e-6)
                    assert rec[k, 4 * q + 3] == uvs[uv_idx[t, q], 0] and rec[k, 12 + q] == uvs[uv_idx[t, q], 1]
            else:
                assert word >> 31 == 0 and not rec[k].any()


def test_set_mesh_clears_attributes(rtb):
    world, (normals, n_idx, uvs, uv_idx) = _attr_world(True)
    cs = rtb.compile_scene(world)
    s = rtb.Scene(None)
    s.set_compiled(cs)
    s.build_bvh()
    assert s.export_triangle_attributes()[:, 15].view(np.uint32).max() == 3
    v, idx = cs.meshes[0]
    rtb._ffi.check(s.lib.rtb_scene_set_mesh(s.h, 0, rtb._ffi.ptr(v), len(v), rtb._ffi.ptr(idx), len(idx)))
    s.set_compiled(cs.__class__(**{**cs.__dict__, "mesh_attrs": []}))
    s.build_bvh()
    assert not s.export_triangle_attributes().any()
    s.set_mesh_attributes(0, uvs=uvs, uv_indices=uv_idx)  # uvs only: read when the graph is flattened again
    s.build_bvh()
    assert not s.export_triangle_attributes().any()
    rtb._ffi.check(s.lib.rtb_scene_set_graph(s.h, rtb._ffi.ptr(cs.nodes), len(cs.nodes), rtb._ffi.ptr(cs.child_index),
                                             len(cs.child_index), cs.root))
    s.build_bvh()
    assert set(s.export_triangle_attributes()[:, 15].view(np.uint32).tolist()) == {0, 2}


def test_smooth_scenes_compile(rtb):
    from ray_tracer_archive_b200 import scenes
    cfg = scenes.config_smooth_meshes()
    s = rtb.Scene(None, rtb.compile_scene(cfg.world, cfg.lights))
    rec = s.export_triangle_attributes()
    flags = rec[:, 15].view(np.uint32)
    assert (flags == 3).sum() == 48 * 24 * 2 - 2 * 48 and (flags == 1).sum() == (16 * 8 * 2 - 32) + (12 * 6 * 2 - 24)
    c4 = scenes.config_mesh(nx=30, nz=20, smooth=True)
    s4 = rtb.Scene(None, rtb.compile_scene(c4.world, c4.lights))
    assert (s4.export_triangle_attributes()[:, 15].view(np.uint32) == 1).sum() == 2 * 30 * 20
