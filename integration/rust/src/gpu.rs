// raytracer/src/gpu.rs — `extern "C"` declarations mirroring include/rtb200.h one to one (ABI version 2), the record
// builder the `flatten()` methods push into, and a small safe wrapper.  NOT compiled in the build image (no rustc/cargo
// there).  Layouts are checked on the C side by tests/test_abi.py (struct sizes / offsets of the same header) and the
// ctypes binding ray_tracer_archive_b200/_ffi.py binds the same symbols.
#![allow(dead_code)]
use std::collections::HashMap;
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};

pub const RTB_NONE: u32 = 0xFFFF_FFFF;
// rtb_node_type
pub const NODE_SPHERE: u32 = 1;
pub const NODE_MOVING_SPHERE: u32 = 2;
pub const NODE_XY_RECT: u32 = 3;
pub const NODE_XZ_RECT: u32 = 4;
pub const NODE_YZ_RECT: u32 = 5;
pub const NODE_BOX: u32 = 6;
pub const NODE_TRIANGLE: u32 = 7;
pub const NODE_QUAD: u32 = 8;
pub const NODE_MESH: u32 = 9;
pub const NODE_TRANSLATE: u32 = 16;
pub const NODE_ROTATE_Y: u32 = 17;
pub const NODE_FLIP_FACE: u32 = 18;
pub const NODE_CONSTANT_MEDIUM: u32 = 19;
pub const NODE_LIST: u32 = 32;
pub const NODE_BVH: u32 = 33;
// rtb_material_type / rtb_texture_type / rtb_light_type
pub const MAT_LAMBERTIAN: u32 = 0;
pub const MAT_METAL: u32 = 1;
pub const MAT_DIELECTRIC: u32 = 2;
pub const MAT_DIFFUSE_LIGHT: u32 = 3;
pub const MAT_ISOTROPIC: u32 = 4;
pub const TEX_SOLID: u32 = 0;
pub const TEX_CHECKER: u32 = 1;
pub const TEX_NOISE: u32 = 2;
pub const TEX_IMAGE: u32 = 3;
pub const LIGHT_XZ_RECT: u32 = 0;
pub const LIGHT_SPHERE: u32 = 1;
// rtb_params.flags
pub const RENDER_ACCUMULATE: u32 = 1;
pub const RENDER_REDUCE: u32 = 8;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtbNode {
    pub ty: u32,
    pub material: u32,
    pub first_child: u32,
    pub n_children: u32,
    pub p: [f64; 12],
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtbMaterial {
    pub ty: u32,
    pub texture: u32,
    pub param: f64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtbTexture {
    pub ty: u32,
    pub even: u32,
    pub odd: u32,
    pub table: u32,
    pub rgb: [f64; 3],
    pub scale: f64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtbLight {
    pub ty: u32,
    pub _pad: u32,
    pub p: [f64; 5],
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtbCamera {
    pub lookfrom: [f64; 3],
    pub lookat: [f64; 3],
    pub vup: [f64; 3],
    pub vfov_deg: f64,
    pub aspect_ratio: f64,
    pub aperture: f64,
    pub focus_dist: f64,
    pub time0: f64,
    pub time1: f64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtbParams {
    pub width: u32,
    pub height: u32,
    pub spp: u32,
    pub sample_offset: u32,
    pub total_spp: u32,
    pub max_depth: i32,
    pub rr_start_depth: u32,
    pub seed: u32,
    pub background: [f32; 3],
    pub pool_paths: u32,
    pub flags: u32,
}
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct RtbStats {
    pub paths: u64,
    pub segments: u64,
    pub rejected: u64,
    pub iterations: u64,
    pub launches: u64,
    pub extend_launches: u64,
    pub ms_total: f64,
    pub ms_extend: f64,
    pub nodes_visited: u64,
    pub prims_tested: u64,
    pub exact_rays: u64,
    pub refined_rays: u64,
    pub ms_nccl: f64,
    pub ms_render: f64,
    pub n_devices: u32,
    pub _pad: u32,
    pub prims_tested_type: [u64; 4],
    pub ms_nccl_wait: f64,
}
pub enum RtbContext {}
pub enum RtbScene {}

extern "C" {
    pub fn rtb_abi_version() -> u32;
    pub fn rtb_last_error() -> *const c_char;
    pub fn rtb_context_create(device_id: c_int, out: *mut *mut RtbContext) -> c_int;
    pub fn rtb_context_create_multi(device_ids: *const c_int, n: c_int, out: *mut *mut RtbContext) -> c_int;
    pub fn rtb_context_device_count(ctx: *mut RtbContext) -> c_int;
    pub fn rtb_comm_unique_id(id128: *mut u8) -> c_int;
    pub fn rtb_context_comm_init(ctx: *mut RtbContext, id128: *const u8, rank: c_int, n_ranks: c_int) -> c_int;
    pub fn rtb_context_destroy(ctx: *mut RtbContext);
    pub fn rtb_scene_create(ctx: *mut RtbContext, out: *mut *mut RtbScene) -> c_int;
    pub fn rtb_scene_destroy(s: *mut RtbScene);
    pub fn rtb_scene_set_materials(s: *mut RtbScene, m: *const RtbMaterial, n: u32) -> c_int;
    pub fn rtb_scene_set_textures(s: *mut RtbScene, t: *const RtbTexture, n: u32) -> c_int;
    pub fn rtb_scene_set_image(s: *mut RtbScene, id: u32, rgb: *const u8, w: u32, h: u32) -> c_int;
    pub fn rtb_scene_set_perlin(s: *mut RtbScene, id: u32, ranvec: *const f64, px: *const u32, py: *const u32, pz: *const u32) -> c_int;
    pub fn rtb_scene_set_mesh(s: *mut RtbScene, id: u32, verts: *const f32, nv: u32, idx: *const u32, nt: u32) -> c_int;
    pub fn rtb_scene_set_lights(s: *mut RtbScene, l: *const RtbLight, n: u32) -> c_int;
    pub fn rtb_scene_set_graph(s: *mut RtbScene, nodes: *const RtbNode, n: u32, child: *const u32, nc: u32, root: u32) -> c_int;
    pub fn rtb_scene_build_bvh(s: *mut RtbScene) -> c_int;
    pub fn rtb_scene_commit(s: *mut RtbScene) -> c_int;
    pub fn rtb_render(ctx: *mut RtbContext, s: *mut RtbScene, cam: *const RtbCamera, p: *const RtbParams, accum_out: *mut f32,
                      stats: *mut RtbStats) -> c_int;
    pub fn rtb_render_device(ctx: *mut RtbContext, s: *mut RtbScene, cam: *const RtbCamera, p: *const RtbParams,
                             d_accum: *mut c_void, stream: *mut c_void, stats: *mut RtbStats) -> c_int;
    // denoiser guide buffers (W*H*8 float sums: albedo rgb, coverage, normal xyz, depth; see rtb200.h).  Declared for
    // callers of the shim; this file is not compiled in the project's own build and test image.
    pub fn rtb_render_aov_device(ctx: *mut RtbContext, s: *mut RtbScene, cam: *const RtbCamera, p: *const RtbParams,
                                 d_aov: *mut c_void, stream: *mut c_void, stats: *mut RtbStats) -> c_int;
    pub fn rtb_render_aov(ctx: *mut RtbContext, s: *mut RtbScene, cam: *const RtbCamera, p: *const RtbParams,
                          aov_out: *mut f32, stats: *mut RtbStats) -> c_int;
    pub fn rtb_finalize_rgb8(ctx: *mut RtbContext, d_accum: *const c_void, w: u32, h: u32, total_spp: u32, out: *mut u8) -> c_int;
    pub fn rtb_primary_hits(ctx: *mut RtbContext, s: *mut RtbScene, cam: *const RtbCamera, w: u32, h: u32, prim_id: *mut u32,
                            t: *mut f32, stats: *mut RtbStats) -> c_int;
}

fn check(rc: c_int) {
    // the reference panics through unwrap()/expect()/assert_eq! (main.rs:656,762,777,779,792); so does the shim
    if rc != 0 {
        let msg = unsafe { CStr::from_ptr(rtb_last_error()) }.to_string_lossy().into_owned();
        panic!("rtb200 error {}: {}", rc, msg);
    }
}

/// Collects the records; ids of materials / textures are positions in these vectors.  Shared `Arc`s are recorded once
/// (keyed by their address), like the C++ mirror does, so both emit the same tables.
#[derive(Default)]
pub struct SceneBuilder {
    pub nodes: Vec<RtbNode>,
    pub children: Vec<u32>,
    pub materials: Vec<RtbMaterial>,
    pub textures: Vec<RtbTexture>,
    pub images: Vec<(Vec<u8>, u32, u32)>,
    pub perlins: Vec<(Vec<f64>, Vec<u32>, Vec<u32>, Vec<u32>)>,
    pub meshes: Vec<(Vec<f32>, Vec<u32>)>,
    pub material_ids: HashMap<usize, u32>,
    pub texture_ids: HashMap<usize, u32>,
}
impl SceneBuilder {
    fn pack(p: &[f64]) -> [f64; 12] {
        let mut q = [0.0; 12];
        q[..p.len()].copy_from_slice(p);
        q
    }
    /// a primitive: one record, no children
    pub fn leaf(&mut self, ty: u32, material: u32, p: &[f64]) -> u32 {
        self.nodes.push(RtbNode { ty, material, first_child: self.children.len() as u32, n_children: 0, p: Self::pack(p) });
        (self.nodes.len() - 1) as u32
    }
    /// a wrapper / list: its children were flattened BEFORE this call (post-order, like include/rtb200_scene.hpp)
    pub fn inner(&mut self, ty: u32, material: u32, p: &[f64], kids: &[u32]) -> u32 {
        let first = self.children.len() as u32;
        self.children.extend_from_slice(kids);
        self.nodes.push(RtbNode { ty, material, first_child: first, n_children: kids.len() as u32, p: Self::pack(p) });
        (self.nodes.len() - 1) as u32
    }
    pub fn push_material(&mut self, key: usize, ty: u32, texture: u32, param: f64) -> u32 {
        self.materials.push(RtbMaterial { ty, texture, param });
        let id = (self.materials.len() - 1) as u32;
        self.material_ids.insert(key, id);
        id
    }
    pub fn push_texture(&mut self, key: usize, t: RtbTexture) -> u32 {
        self.textures.push(t);
        let id = (self.textures.len() - 1) as u32;
        self.texture_ids.insert(key, id);
        id
    }
}

/// Owns a context (one GPU, or several driven by this process) and renders flattened scenes.
pub struct Gpu {
    ctx: *mut RtbContext,
}
impl Gpu {
    /// `devices`: one id = one GPU; several = rtb_context_create_multi (samples split across them, one NCCL reduce)
    pub fn new(devices: &[i32]) -> Self {
        assert_eq!(unsafe { rtb_abi_version() }, 2);
        let mut ctx = std::ptr::null_mut();
        if devices.len() == 1 {
            check(unsafe { rtb_context_create(devices[0], &mut ctx) });
        } else {
            check(unsafe { rtb_context_create_multi(devices.as_ptr(), devices.len() as c_int, &mut ctx) });
        }
        Self { ctx }
    }
    /// uploads the records, renders `params.spp` samples per pixel and returns (RGB8 rows from the top, stats)
    pub fn render(&self, b: &SceneBuilder, root: u32, lights: &[RtbLight], cam: &RtbCamera, params: &RtbParams) -> (Vec<u8>, RtbStats) {
        let mut sc = std::ptr::null_mut();
        let mut stats = RtbStats::default();
        let mut rgb = vec![0u8; (params.width * params.height * 3) as usize];
        unsafe {
            check(rtb_scene_create(self.ctx, &mut sc));
            check(rtb_scene_set_materials(sc, b.materials.as_ptr(), b.materials.len() as u32));
            check(rtb_scene_set_textures(sc, b.textures.as_ptr(), b.textures.len() as u32));
            for (i, (data, w, h)) in b.images.iter().enumerate() {
                check(rtb_scene_set_image(sc, i as u32, data.as_ptr(), *w, *h));
            }
            for (i, (rv, px, py, pz)) in b.perlins.iter().enumerate() {
                check(rtb_scene_set_perlin(sc, i as u32, rv.as_ptr(), px.as_ptr(), py.as_ptr(), pz.as_ptr()));
            }
            for (i, (v, idx)) in b.meshes.iter().enumerate() {
                check(rtb_scene_set_mesh(sc, i as u32, v.as_ptr(), (v.len() / 3) as u32, idx.as_ptr(), (idx.len() / 3) as u32));
            }
            check(rtb_scene_set_lights(sc, if lights.is_empty() { std::ptr::null() } else { lights.as_ptr() }, lights.len() as u32));
            check(rtb_scene_set_graph(sc, b.nodes.as_ptr(), b.nodes.len() as u32, b.children.as_ptr(), b.children.len() as u32, root));
            check(rtb_scene_commit(sc));
            check(rtb_render(self.ctx, sc, cam, params, std::ptr::null_mut(), &mut stats));
            check(rtb_finalize_rgb8(self.ctx, std::ptr::null(), params.width, params.height, params.total_spp, rgb.as_mut_ptr()));
            rtb_scene_destroy(sc);
        }
        (rgb, stats)
    }
}
impl Drop for Gpu {
    fn drop(&mut self) {
        unsafe { rtb_context_destroy(self.ctx) }
    }
}
