// rtb_api.cu — the extern "C" boundary declared in include/rtb200.h.  Host orchestration only: scene tables,
// flatten + BVH build (flatten.cpp, bvh_build.cpp), uploads, and the wavefront iteration loop that replaces the
// reference's pixel/sample loop (main.rs:731-784).  There is no CPU path: without a CUDA device every entry fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <atomic>
#include <memory>
#include <thread>

#include "rtb_device.cuh"
#include "rtb_launch.hpp"
#include "rtb_nccl.hpp"

using namespace rtb;

static thread_local std::string g_err;
static int set_err(int code, const std::string& m) { g_err = m; return code; }
#define CU(call)                                                                                              \
  do {                                                                                                        \
    cudaError_t e_ = (call);                                                                                  \
    if (e_ != cudaSuccess)                                                                                    \
      return set_err(RTB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                       \
  } while (0)

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  ~DevBuf() { release(); }
  void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
  cudaError_t resize(size_t count) {
    if (count <= n && p) return cudaSuccess;
    release();
    if (count == 0) count = 1;
    cudaError_t e = cudaMalloc((void**)&p, count * sizeof(T));
    if (e == cudaSuccess) n = count;
    return e;
  }
  cudaError_t upload(const T* src, size_t count, cudaStream_t st = 0) {
    cudaError_t e = resize(count);
    if (e != cudaSuccess || count == 0) return e;
    return cudaMemcpyAsync(p, src, count * sizeof(T), cudaMemcpyHostToDevice, st);
  }
};

// One wavefront instance: its own path pool, queues, counters and stream.  A render runs RTB_LANES of them
// concurrently on disjoint sample ranges: while one lane is in its ALU-bound extend kernel another is in its
// DRAM-latency-bound shade kernels, so the two kinds of work overlap on the SMs.
struct Lane {
  uint32_t pool_n = 0;
  DevBuf<float4> ray, st, hit;
  DevBuf<uint8_t> cls;                    // per-slot shade class
  DevBuf<uint4> redo[2];                  // rays queued for the exact pass (slot, distance slab), double-buffered
  DevBuf<unsigned long long> cursor;      // per-chunk path cursor
  DevBuf<DevCounters> counters;
  DevCounters* h_counters = nullptr;     // pinned; [0], [1]: the drain check of batch k is read while batch k + 1 runs
  cudaStream_t stream = nullptr;
  cudaEvent_t done = nullptr;
  cudaEvent_t batch_done[2] = {nullptr, nullptr};
};
#define RTB_MAX_LANES 8

struct rtb_context {
  int device = 0;
  cudaDeviceProp prop;
  Lane lanes[RTB_MAX_LANES];
  cudaEvent_t ev_fork = nullptr;
  DevBuf<DevCounters> counters;        // probes
  DevCounters* h_counters = nullptr;   // pinned
  // image-sized buffers
  DevBuf<float4> accum;
  DevBuf<float4> aov;  // rtb_render_aov's sums, 2 per pixel (kept apart from accum: either call may accumulate)
  DevBuf<uint32_t> pix_order;
  uint32_t pix_w = 0, pix_h = 0;
  DevBuf<uint8_t> rgb8;
  // probe scratch
  DevBuf<float> p_org, p_dir, p_time, p_t;
  DevBuf<uint32_t> p_id;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<cudaEvent_t> ext_events;  // pairs around every extend launch when RTB_RENDER_TIME_EXTEND is set
  // ---- multi-GPU (SURVEY §8b/§8e): the framebuffer reduce lives in the library --------------------------------
  // single process, n devices: `peers` are the contexts of device_ids[1..] (owned), every one with its communicator from
  // ncclCommInitAll; one process per device: `comm` comes from rtb_context_comm_init (ncclCommInitRank)
  std::vector<rtb_context*> peers;
  NcclComm comm = nullptr;
  int rank = 0, n_ranks = 1;
  cudaEvent_t ev_n0 = nullptr, ev_n1 = nullptr, ev_w0 = nullptr;
  DevBuf<float> comm_scratch;  // 1 float: the arrival barrier in front of the timed reduce
};

struct rtb_scene {
  rtb_context* ctx = nullptr;
  int device = -1;                   // ctx's device, kept here: the context may be destroyed before the scene
  std::vector<rtb_scene*> replicas;  // multi-device context: device copies on the peers (host data stays with this one)
  HostScene hs;
  HostBvh bvh;
  bool built = false;      // host BVH is current
  bool committed = false;  // device copies are current
  uint32_t present_materials = 0;  // bit per rtb_material_type that some primitive/medium uses
  // device copies
  DevBuf<uint4> d_nodes;
  DevBuf<float4> d_geom[PT_COUNT];
  DevBuf<uint2> d_info[PT_COUNT];
  DevBuf<double> d_exact[PT_COUNT];
  DevBuf<ExactTab> d_xtab;
  DevBuf<DevScene> d_self;
  DevBuf<float4> d_materials;
  DevBuf<DevTexture> d_textures;
  DevBuf<float4> d_perlin_vec;   // all perlin tables, 256 vectors each
  DevBuf<uint8_t> d_perlin_perm; // all perlin tables, 768 bytes each
  DevBuf<uint8_t> d_image_data;  // all images, packed
  DevBuf<DevImage> d_images;     // their descriptors
  DevScene dev;
  LaunchCfg lc;
};

extern "C" {

uint32_t rtb_abi_version(void) { return RTB_ABI_VERSION; }
const char* rtb_last_error(void) { return g_err.c_str(); }

static int context_init(rtb_context* c, int device_id) {
  CU(cudaSetDevice(device_id));
  c->device = device_id;
  CU(cudaGetDeviceProperties(&c->prop, device_id));
  if (c->prop.major < 10) return set_err(RTB_ERR_NO_DEVICE, "librtb200 is built for sm_100a only");
  CU(cudaMallocHost((void**)&c->h_counters, sizeof(DevCounters)));
  for (int k = 0; k < RTB_MAX_LANES; ++k) {
    Lane& L = c->lanes[k];
    CU(cudaMallocHost((void**)&L.h_counters, 2 * sizeof(DevCounters)));
    CU(cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&L.done, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&L.batch_done[0], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&L.batch_done[1], cudaEventDisableTiming));
    CU(L.counters.resize(1));
  }
  CU(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  CU(cudaEventCreate(&c->ev0));
  CU(cudaEventCreate(&c->ev1));
  CU(cudaEventCreate(&c->ev_n0));
  CU(cudaEventCreate(&c->ev_n1));
  CU(cudaEventCreate(&c->ev_w0));
  CU(c->comm_scratch.resize(1));
  CU(c->counters.resize(1));
  return RTB_OK;
}

int rtb_context_create(int device_id, rtb_context** out) {
  if (!out) return set_err(RTB_ERR_INVALID, "out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return set_err(RTB_ERR_NO_DEVICE, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count 0") +
                                          " (librtb200 has no CPU fallback)");
  if (device_id < 0 || device_id >= n) return set_err(RTB_ERR_INVALID, "device_id out of range");
  // a partly built context is torn down by its destructor path (streams, events, pinned buffers)
  std::unique_ptr<rtb_context, void (*)(rtb_context*)> c(new rtb_context(), rtb_context_destroy);
  const int rc = context_init(c.get(), device_id);
  if (rc != RTB_OK) return rc;
  *out = c.release();
  return RTB_OK;
}

void rtb_context_destroy(rtb_context* c) {
  if (!c) return;
  for (rtb_context* p : c->peers) rtb_context_destroy(p);
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  if (c->comm && nccl_api().ok) nccl_api().CommDestroy(c->comm);
  if (c->h_counters) cudaFreeHost(c->h_counters);
  for (int k = 0; k < RTB_MAX_LANES; ++k) {
    Lane& L = c->lanes[k];
    if (L.h_counters) cudaFreeHost(L.h_counters);
    if (L.stream) cudaStreamDestroy(L.stream);
    if (L.done) cudaEventDestroy(L.done);
    for (cudaEvent_t e : L.batch_done) if (e) cudaEventDestroy(e);
  }
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->ev_n0) cudaEventDestroy(c->ev_n0);
  if (c->ev_n1) cudaEventDestroy(c->ev_n1);
  if (c->ev_w0) cudaEventDestroy(c->ev_w0);
  for (cudaEvent_t e : c->ext_events) cudaEventDestroy(e);
  delete c;
}

// ---- multi-GPU: communicators ---------------------------------------------------------------------------------------
#define NCCLCHECK(call)                                                                                        \
  do {                                                                                                         \
    const int r_ = (call);                                                                                     \
    if (r_ != kNcclSuccess)                                                                                    \
      return set_err(RTB_ERR_CUDA, std::string(#call) + ": " + nccl_api().GetErrorString(r_));                  \
  } while (0)

int rtb_context_create_multi(const int* device_ids, int n_devices, rtb_context** out) {
  if (!out || !device_ids || n_devices < 1) return set_err(RTB_ERR_INVALID, "bad argument");
  *out = nullptr;
  for (int a = 0; a < n_devices; ++a)
    for (int b = a + 1; b < n_devices; ++b)
      if (device_ids[a] == device_ids[b]) return set_err(RTB_ERR_INVALID, "device ids must be distinct");
  rtb_context* root = nullptr;
  int rc = rtb_context_create(device_ids[0], &root);
  if (rc != RTB_OK) return rc;
  std::unique_ptr<rtb_context, void (*)(rtb_context*)> guard(root, rtb_context_destroy);
  root->n_ranks = n_devices;
  if (n_devices > 1) {
    const NcclApi& api = nccl_api();
    if (!api.ok) return set_err(RTB_ERR_UNSUPPORTED, "multi-GPU needs NCCL: " + api.error);
    for (int k = 1; k < n_devices; ++k) {
      rtb_context* p = nullptr;
      rc = rtb_context_create(device_ids[k], &p);
      if (rc != RTB_OK) return rc;
      p->rank = k;
      p->n_ranks = n_devices;
      root->peers.push_back(p);
    }
    std::vector<NcclComm> comms((size_t)n_devices, nullptr);
    NCCLCHECK(api.CommInitAll(comms.data(), n_devices, device_ids));  // one communicator per device, ranks = list order
    root->comm = comms[0];
    for (int k = 1; k < n_devices; ++k) root->peers[(size_t)k - 1]->comm = comms[(size_t)k];
    // one-float reduce now: NCCL sets its NVLink connections up on first use (~0.3 s), which must not land in a frame
    NCCLCHECK(api.GroupStart());
    for (int k = 0; k < n_devices; ++k) {
      rtb_context* ck = k == 0 ? root : root->peers[(size_t)k - 1];
      CU(cudaSetDevice(ck->device));
      NCCLCHECK(api.Reduce(ck->comm_scratch.p, ck->comm_scratch.p, 1, kNcclFloat32, kNcclSum, 0, ck->comm, (cudaStream_t)0));
    }
    NCCLCHECK(api.GroupEnd());
    for (int k = 0; k < n_devices; ++k) {
      rtb_context* ck = k == 0 ? root : root->peers[(size_t)k - 1];
      CU(cudaSetDevice(ck->device));
      CU(cudaStreamSynchronize(0));
    }
    CU(cudaSetDevice(root->device));
  }
  *out = guard.release();
  return RTB_OK;
}

int rtb_comm_unique_id(uint8_t* id128) {
  if (!id128) return set_err(RTB_ERR_INVALID, "id is NULL");
  const NcclApi& api = nccl_api();
  if (!api.ok) return set_err(RTB_ERR_UNSUPPORTED, "multi-GPU needs NCCL: " + api.error);
  NcclUniqueId id;
  NCCLCHECK(api.GetUniqueId(&id));
  std::memcpy(id128, id.internal, RTB_COMM_ID_BYTES);
  return RTB_OK;
}

int rtb_context_comm_init(rtb_context* c, const uint8_t* id128, int rank, int n_ranks) {
  if (!c || !id128 || n_ranks < 1 || rank < 0 || rank >= n_ranks) return set_err(RTB_ERR_INVALID, "bad argument");
  if (!c->peers.empty() || c->comm) return set_err(RTB_ERR_STATE, "context already has a communicator");
  const NcclApi& api = nccl_api();
  if (!api.ok) return set_err(RTB_ERR_UNSUPPORTED, "multi-GPU needs NCCL: " + api.error);
  CU(cudaSetDevice(c->device));
  NcclUniqueId id;
  std::memcpy(id.internal, id128, RTB_COMM_ID_BYTES);
  NCCLCHECK(api.CommInitRank(&c->comm, n_ranks, id, rank));
  c->rank = rank;
  c->n_ranks = n_ranks;
  // one-float reduce now (collective: every rank is here): connection set-up must not land in the first frame
  NCCLCHECK(api.Reduce(c->comm_scratch.p, c->comm_scratch.p, 1, kNcclFloat32, kNcclSum, 0, c->comm, (cudaStream_t)0));
  CU(cudaStreamSynchronize(0));
  return RTB_OK;
}

int rtb_context_device_count(rtb_context* c) { return c ? 1 + (int)c->peers.size() : 0; }

int rtb_context_device_info(rtb_context* c, int* sm_count, int* l2_bytes, int* clock_khz, char* name, size_t cap) {
  if (!c) return set_err(RTB_ERR_INVALID, "ctx is NULL");
  if (sm_count) *sm_count = c->prop.multiProcessorCount;
  if (l2_bytes) *l2_bytes = c->prop.l2CacheSize;
  if (clock_khz) {
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, c->device);
    *clock_khz = khz;
  }
  if (name && cap) { std::strncpy(name, c->prop.name, cap - 1); name[cap - 1] = 0; }
  return RTB_OK;
}

// ---- scene tables ---------------------------------------------------------------------------------------------
int rtb_scene_create(rtb_context* ctx, rtb_scene** out) {
  if (!out) return set_err(RTB_ERR_INVALID, "NULL argument");
  rtb_scene* s = new rtb_scene();  // ctx == NULL: host-only scene (flatten / BVH build / export; cannot be committed)
  s->ctx = ctx;
  s->device = ctx ? ctx->device : -1;
  if (ctx)
    for (rtb_context* p : ctx->peers) {  // device copies on the other GPUs of a multi-device context
      rtb_scene* r = new rtb_scene();
      r->ctx = p;
      r->device = p->device;
      s->replicas.push_back(r);
    }
  *out = s;
  return RTB_OK;
}
void rtb_scene_destroy(rtb_scene* s) {
  if (!s) return;
  for (rtb_scene* r : s->replicas) rtb_scene_destroy(r);
  if (s->device >= 0 && cudaSetDevice(s->device) == cudaSuccess) cudaDeviceSynchronize();  // (never touches s->ctx: it may be gone)
  delete s;
}

int rtb_scene_set_materials(rtb_scene* s, const rtb_material* mats, uint32_t n) {
  if (!s || (!mats && n)) return set_err(RTB_ERR_INVALID, "NULL argument");
  for (uint32_t i = 0; i < n; ++i)
    if (mats[i].type > RTB_MAT_ISOTROPIC) return set_err(RTB_ERR_INVALID, "unknown material type");
  s->hs.materials.assign(mats, mats + n);
  s->built = s->committed = false;
  return RTB_OK;
}
int rtb_scene_set_textures(rtb_scene* s, const rtb_texture* tex, uint32_t n) {
  if (!s || (!tex && n)) return set_err(RTB_ERR_INVALID, "NULL argument");
  for (uint32_t i = 0; i < n; ++i) {
    if (tex[i].type > RTB_TEX_IMAGE) return set_err(RTB_ERR_INVALID, "unknown texture type");
    if (tex[i].type == RTB_TEX_CHECKER && (tex[i].even >= n || tex[i].odd >= n))
      return set_err(RTB_ERR_INVALID, "checker child out of range");
    // the reference's Arc<dyn Texture> children can nest (texture.rs:41-45): followed on the device up to
    // RTB_MAX_CHECKER_DEPTH levels, so deeper chains (and cycles, which Arc cannot express) are refused here
    if (tex[i].type == RTB_TEX_CHECKER) {
      for (int side = 0; side < 2; ++side) {
        uint32_t c = side ? tex[i].odd : tex[i].even;
        int depth = 1;
        while (tex[c].type == RTB_TEX_CHECKER && depth <= RTB_MAX_CHECKER_DEPTH) {
          const uint32_t nx = side ? tex[c].odd : tex[c].even;
          if (nx >= n) return set_err(RTB_ERR_INVALID, "checker child out of range");
          c = nx;
          ++depth;
        }
        if (depth > RTB_MAX_CHECKER_DEPTH) return set_err(RTB_ERR_UNSUPPORTED, "checker textures nested deeper than 8 levels (or cyclic)");
      }
    }
    if (tex[i].type == RTB_TEX_NOISE && tex[i].table >= RTB_MAX_TABLES) return set_err(RTB_ERR_INVALID, "perlin table id too large");
  }
  s->hs.textures.assign(tex, tex + n);
  s->built = s->committed = false;
  return RTB_OK;
}
int rtb_scene_set_image(rtb_scene* s, uint32_t id, const uint8_t* rgb, uint32_t w, uint32_t h) {
  if (!s || id >= RTB_MAX_TABLES) return set_err(RTB_ERR_INVALID, "image id out of range");
  if ((!rgb && w && h) || ((size_t)w * h == 0 && rgb)) return set_err(RTB_ERR_INVALID, "image pointer / size mismatch");
  if (!rgb) w = h = 0;  // an empty image: the texture renders cyan (texture.rs:119-121)
  if (s->hs.images.size() <= id) s->hs.images.resize(id + 1);
  if (rgb) s->hs.images[id].rgb.assign(rgb, rgb + (size_t)w * h * 3);
  else s->hs.images[id].rgb.clear();
  s->hs.images[id].w = w;
  s->hs.images[id].h = h;
  s->built = s->committed = false;
  return RTB_OK;
}
int rtb_scene_set_perlin(rtb_scene* s, uint32_t id, const double* ranvec, const uint32_t* px, const uint32_t* py,
                         const uint32_t* pz) {
  if (!s || id >= RTB_MAX_TABLES || !ranvec || !px || !py || !pz) return set_err(RTB_ERR_INVALID, "bad perlin table");
  for (int i = 0; i < 256; ++i)  // validate before the stored table is touched
    if (px[i] > 255 || py[i] > 255 || pz[i] > 255) return set_err(RTB_ERR_INVALID, "perm entry > 255");
  if (s->hs.perlins.size() <= id) s->hs.perlins.resize(id + 1);
  HostScene::Perlin& p = s->hs.perlins[id];
  p.ranvec.resize(256 * 4);
  p.perm.resize(768);
  for (int i = 0; i < 256; ++i) {
    p.ranvec[4 * i] = (float)ranvec[3 * i];
    p.ranvec[4 * i + 1] = (float)ranvec[3 * i + 1];
    p.ranvec[4 * i + 2] = (float)ranvec[3 * i + 2];
    p.ranvec[4 * i + 3] = 0.f;
    p.perm[i] = (uint8_t)px[i];
    p.perm[256 + i] = (uint8_t)py[i];
    p.perm[512 + i] = (uint8_t)pz[i];
  }
  p.set = true;
  s->built = s->committed = false;
  return RTB_OK;
}
int rtb_scene_set_mesh(rtb_scene* s, uint32_t id, const float* verts, uint32_t nv, const uint32_t* idx, uint32_t nt) {
  if (!s || !verts || !idx) return set_err(RTB_ERR_INVALID, "NULL argument");
  if (id >= 64) return set_err(RTB_ERR_INVALID, "mesh id out of range");
  for (size_t i = 0; i < (size_t)nt * 3; ++i)
    if (idx[i] >= nv) return set_err(RTB_ERR_INVALID, "mesh index out of range");
  if (s->hs.meshes.size() <= id) s->hs.meshes.resize(id + 1);
  s->hs.meshes[id].verts.assign(verts, verts + (size_t)nv * 3);
  s->hs.meshes[id].idx.assign(idx, idx + (size_t)nt * 3);
  s->built = s->committed = false;
  return RTB_OK;
}
int rtb_scene_set_lights(rtb_scene* s, const rtb_light* lights, uint32_t n) {
  if (!s || (!lights && n)) return set_err(RTB_ERR_INVALID, "NULL argument");
  if (n > RTB_MAX_LIGHTS) return set_err(RTB_ERR_UNSUPPORTED, "too many lights");
  s->hs.lights.clear();
  for (uint32_t i = 0; i < n; ++i) {
    if (lights[i].type > RTB_LIGHT_SPHERE)
      return set_err(RTB_ERR_UNSUPPORTED, "only XzRect and Sphere implement pdf_value/random (aarect.rs:107, sphere.rs:75)");
    HostLight l;
    l.type = lights[i].type;
    for (int k = 0; k < 5; ++k) l.p[k] = (float)lights[i].p[k];
    s->hs.lights.push_back(l);
  }
  s->built = s->committed = false;
  return RTB_OK;
}

int rtb_scene_set_graph(rtb_scene* s, const rtb_node* nodes, uint32_t n_nodes, const uint32_t* child_index,
                        uint32_t n_child_index, uint32_t root) {
  if (!s || !nodes || (!child_index && n_child_index)) return set_err(RTB_ERR_INVALID, "NULL argument");
  std::string err;
  int rc = flatten_graph(s->hs, nodes, n_nodes, child_index, n_child_index, root, err);
  s->built = s->committed = false;
  if (rc != RTB_OK) return set_err(rc, err);
  return RTB_OK;
}

// ---- flat SoA setters ------------------------------------------------------------------------------------------
static void drop_type(HostScene& hs, uint32_t type) {
  hs.prims.erase(std::remove_if(hs.prims.begin(), hs.prims.end(), [&](const HostPrim& p) { return p.type == type; }),
                 hs.prims.end());
}
static uint32_t face_mode_of(uint32_t flags) {
  if (flags & RTB_PRIM_FORCE_FRONT) return (flags & RTB_PRIM_FLIP_FACE) ? FACE_FALSE : FACE_TRUE;
  return (flags & RTB_PRIM_FLIP_FACE) ? FACE_FLIPPED : FACE_NATURAL;
}
static HostPrim& add_flat(rtb_scene* s, uint32_t type, const uint32_t* mat, const uint32_t* flags, const uint32_t* id,
                          uint32_t i) {
  s->hs.prims.emplace_back();
  HostPrim& p = s->hs.prims.back();
  std::memset(&p, 0, sizeof(p));
  p.type = type;
  p.material = mat[i];
  p.face_mode = flags ? face_mode_of(flags[i]) : FACE_NATURAL;
  p.exact = RTB_NONE;
  p.prim_id = id ? id[i] : s->hs.n_prim_ids;
  s->hs.n_prim_ids = std::max(s->hs.n_prim_ids, p.prim_id + 1);
  return p;
}

int rtb_scene_set_spheres(rtb_scene* s, const float* cr, const uint32_t* mat, const uint32_t* flags, const uint32_t* id,
                          uint32_t n) {
  if (!s || (n && (!cr || !mat))) return set_err(RTB_ERR_INVALID, "NULL argument");
  drop_type(s->hs, PT_SPHERE);
  for (uint32_t i = 0; i < n; ++i) {
    HostPrim& p = add_flat(s, PT_SPHERE, mat, flags, id, i);
    double c[3] = {cr[4 * i], cr[4 * i + 1], cr[4 * i + 2]};
    pack_sphere(p, c, cr[4 * i + 3]);
    const double prm[4] = {c[0], c[1], c[2], cr[4 * i + 3]};
    const uint32_t ex = add_exact(s->hs, ExactXform(), 0, prm, 4);  // (may reallocate hs.exact, not hs.prims)
    s->hs.prims.back().exact = ex;
  }
  s->built = s->committed = false;
  return RTB_OK;
}
int rtb_scene_set_moving_spheres(rtb_scene* s, const float* c0r, const float* c1, const float* t01, const uint32_t* mat,
                                 const uint32_t* flags, const uint32_t* id, uint32_t n) {
  if (!s || (n && (!c0r || !c1 || !t01 || !mat))) return set_err(RTB_ERR_INVALID, "NULL argument");
  drop_type(s->hs, PT_MOVING);
  for (uint32_t i = 0; i < n; ++i) {
    HostPrim& p = add_flat(s, PT_MOVING, mat, flags, id, i);
    double a[3] = {c0r[4 * i], c0r[4 * i + 1], c0r[4 * i + 2]}, b[3] = {c1[3 * i], c1[3 * i + 1], c1[3 * i + 2]};
    pack_moving(p, a, b, t01[2 * i], t01[2 * i + 1], c0r[4 * i + 3]);
    const double prm[9] = {a[0], a[1], a[2], b[0], b[1], b[2], t01[2 * i], t01[2 * i + 1], c0r[4 * i + 3]};
    s->hs.prims.back().exact = add_exact(s->hs, ExactXform(), 0, prm, 9);
  }
  s->built = s->committed = false;
  return RTB_OK;
}
int rtb_scene_set_quads(rtb_scene* s, const float* q, const float* u, const float* v, const uint32_t* mat,
                        const uint32_t* flags, const uint32_t* id, uint32_t n) {
  if (!s || (n && (!q || !u || !v || !mat))) return set_err(RTB_ERR_INVALID, "NULL argument");
  drop_type(s->hs, PT_QUAD);
  for (uint32_t i = 0; i < n; ++i) {
    HostPrim& p = add_flat(s, PT_QUAD, mat, flags, id, i);
    double Q[3] = {q[3 * i], q[3 * i + 1], q[3 * i + 2]}, U[3] = {u[3 * i], u[3 * i + 1], u[3 * i + 2]},
           V[3] = {v[3 * i], v[3 * i + 1], v[3 * i + 2]};
    pack_quad(p, Q, U, V, nullptr);
    const double prm[9] = {Q[0], Q[1], Q[2], U[0], U[1], U[2], V[0], V[1], V[2]};
    s->hs.prims.back().exact = add_exact(s->hs, ExactXform(), EX_QUAD_GENERAL, prm, 9);
  }
  s->built = s->committed = false;
  return RTB_OK;
}
int rtb_scene_set_triangles(rtb_scene* s, const float* v0, const float* v1, const float* v2, const uint32_t* mat,
                            const uint32_t* flags, const uint32_t* id, uint32_t n) {
  if (!s || (n && (!v0 || !v1 || !v2 || !mat))) return set_err(RTB_ERR_INVALID, "NULL argument");
  drop_type(s->hs, PT_TRI);
  s->hs.prims.reserve(s->hs.prims.size() + n);
  for (uint32_t i = 0; i < n; ++i) {
    HostPrim& p = add_flat(s, PT_TRI, mat, flags, id, i);
    double a[3] = {v0[3 * i], v0[3 * i + 1], v0[3 * i + 2]}, b[3] = {v1[3 * i], v1[3 * i + 1], v1[3 * i + 2]},
           c[3] = {v2[3 * i], v2[3 * i + 1], v2[3 * i + 2]};
    pack_tri(p, a, b, c);
  }
  s->built = s->committed = false;
  return RTB_OK;
}
int rtb_scene_set_media(rtb_scene* s, const rtb_medium* media, uint32_t n) {
  if (!s || (n && !media)) return set_err(RTB_ERR_INVALID, "NULL argument");
  s->hs.media.clear();
  for (uint32_t i = 0; i < n; ++i) {
    const rtb_medium& m = media[i];
    if (m.boundary_type > RTB_BOUNDARY_BOX) return set_err(RTB_ERR_UNSUPPORTED, "medium boundary must be sphere or box");
    if (!(m.density > 0.0) || !std::isfinite(m.density)) return set_err(RTB_ERR_INVALID, "medium density must be positive and finite");
    HostMedium h;
    std::memset(&h, 0, sizeof(h));
    h.boundary_type = m.boundary_type;
    h.material = m.material;
    h.prim_id = m.prim_id;
    s->hs.n_prim_ids = std::max(s->hs.n_prim_ids, m.prim_id + 1);
    h.neg_inv_density = (float)(-1.0 / m.density);
    for (int k = 0; k < 6; ++k) h.p[k] = (float)m.p[k];
    double rad = m.rot_y_deg * 3.14159265358979323846 / 180.0;
    h.sin_t = (float)std::sin(rad);
    h.cos_t = (float)std::cos(rad);
    for (int k = 0; k < 3; ++k) h.offset[k] = (float)m.offset[k];
    s->hs.media.push_back(h);
  }
  s->built = s->committed = false;
  return RTB_OK;
}

int rtb_scene_set_build_options(rtb_scene* s, const rtb_build_options* o) {
  if (!s || !o) return set_err(RTB_ERR_INVALID, "NULL argument");
  if (o->max_leaf_triangles < 1 || o->max_leaf_triangles > 3) return set_err(RTB_ERR_INVALID, "max_leaf_triangles must be 1..3");
  if (!(o->open_min_extent >= 0.f && o->open_min_extent <= 1.f)) return set_err(RTB_ERR_INVALID, "open_min_extent must be in [0, 1]");
  s->hs.opt_max_leaf_tris = o->max_leaf_triangles;
  s->hs.opt_globals = o->keep_huge_primitives_out ? 1u : 0u;
  s->hs.opt_open_min_rel = o->open_min_extent;
  s->built = s->committed = false;
  return RTB_OK;
}

// ---- build (host) and commit (upload) ------------------------------------------------------------------------------
int rtb_scene_build_bvh(rtb_scene* s) {
  if (!s) return set_err(RTB_ERR_INVALID, "scene is NULL");
  HostScene& hs = s->hs;
  if (hs.media.size() > RTB_MAX_MEDIA) return set_err(RTB_ERR_UNSUPPORTED, "too many media");
  if (hs.materials.empty()) return set_err(RTB_ERR_STATE, "materials were not set");
  s->present_materials = 0;
  for (const HostPrim& p : hs.prims) {
    if (p.material >= hs.materials.size()) return set_err(RTB_ERR_INVALID, "primitive material out of range");
    s->present_materials |= 1u << hs.materials[p.material].type;
  }
  for (const HostMedium& m : hs.media) {
    if (m.material >= hs.materials.size()) return set_err(RTB_ERR_INVALID, "medium material out of range");
    s->present_materials |= 1u << hs.materials[m.material].type;
  }
  for (const rtb_material& m : hs.materials) {
    if (m.type != RTB_MAT_DIELECTRIC && m.texture >= hs.textures.size())
      return set_err(RTB_ERR_INVALID, "material texture out of range");
  }
  for (const rtb_texture& t : hs.textures) {
    if (t.type == RTB_TEX_NOISE && (t.table >= hs.perlins.size() || !hs.perlins[t.table].set))
      return set_err(RTB_ERR_STATE, "noise texture references a perlin table that was not set");
  }
  std::string err;
  int rc = build_bvh8(hs, s->bvh, err);
  if (rc != RTB_OK) return set_err(rc, err);
  {
    const uint32_t n_global = (uint32_t)s->bvh.global_refs.size();
    s->bvh.global_f64 = 0;
    // a global sphere whose radius is >= 16 extents of everything else can only be hit at distances < r/16 from
    // points ~r away from its centre — exactly where sphere_roots() rejects its f32 result — so it is tested in f64
    // directly.  Extent = diagonal of the union box of the primitives that are in the tree.
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    // global refs point at the END of their type's leaf-ordered arrays; recover radius / centre from the geometry words
    for (const HostPrim& p : hs.prims) {
      bool glob = false;
      for (uint32_t k = 0; k < n_global && !glob; ++k) {
        const uint32_t ref = s->bvh.global_refs[k], type = ref >> REF_TYPE_SHIFT, idx = ref & REF_INDEX_MASK;
        glob = type == p.type && s->bvh.info[type][2 * idx] == p.prim_id;
      }
      if (glob) continue;
      for (int a = 0; a < 3; ++a) { lo[a] = std::min(lo[a], p.lo[a]); hi[a] = std::max(hi[a], p.hi[a]); }
    }
    double diag2 = 0;
    for (int a = 0; a < 3; ++a) if (hi[a] > lo[a]) diag2 += (double)(hi[a] - lo[a]) * (hi[a] - lo[a]);
    const double extent = std::sqrt(diag2);
    for (uint32_t k = 0; k < n_global ; ++k) {
      const uint32_t ref = s->bvh.global_refs[k], type = ref >> REF_TYPE_SHIFT, idx = ref & REF_INDEX_MASK;
      if (type != PT_SPHERE || extent <= 0) continue;
      const float r = s->bvh.geom[PT_SPHERE][4 * idx + 3];
      if ((double)r >= 16.0 * extent) s->bvh.global_f64 |= 1u << k;
    }
  }
  {  // leaf-ordered exact records + the rounding scales of the f32 quad test
    HostBvh& bvh = s->bvh;
    std::vector<uint32_t> by_id(hs.n_prim_ids, RTB_NONE);
    for (size_t i = 0; i < hs.prims.size(); ++i)
      if (hs.prims[i].prim_id < by_id.size()) by_id[hs.prims[i].prim_id] = (uint32_t)i;
    double pmax = 0.0, wmax = 0.0;
    for (uint32_t t = 0; t < PT_COUNT; ++t) {
      bvh.exact[t].clear();
      if (t == PT_TRI) continue;
      const size_t n = bvh.info[t].size() / 2;
      bvh.exact[t].assign(n * RTB_EXACT_STRIDE, 0.0);
      for (size_t k = 0; k < n; ++k) {
        const uint32_t pid = bvh.info[t][2 * k];
        const uint32_t pi = pid < by_id.size() ? by_id[pid] : RTB_NONE;
        if (pi == RTB_NONE || hs.prims[pi].type != t || hs.prims[pi].exact >= hs.exact.size())
          return set_err(RTB_ERR_INVALID, "primitive ids must be unique (exact record lookup failed)");
        std::memcpy(&bvh.exact[t][k * RTB_EXACT_STRIDE], hs.exact[hs.prims[pi].exact].v, sizeof(ExactRec));
      }
    }
    for (const HostPrim& p : hs.prims) {
      if (p.type != PT_QUAD) continue;
      for (int a = 0; a < 3; ++a) pmax = std::max(pmax, (double)std::max(std::fabs(p.lo[a]), std::fabs(p.hi[a])));
      wmax = std::max(wmax, (double)(std::fabs(p.g[4]) + std::fabs(p.g[5]) + std::fabs(p.g[6]) + std::fabs(p.g[8]) +
                                     std::fabs(p.g[9]) + std::fabs(p.g[10])));
    }
    bvh.coord_max = (float)(2.0 * pmax);
    bvh.eps_ab = (float)(std::ldexp(1.0, -20) * wmax * pmax + 1e-7);
  }
  s->built = true;
  return RTB_OK;
}

// Material trait dispatch (material.rs:11-21) resolved on the host: which per-material shade kernel handles a hit
static uint32_t queue_of_material(const HostScene& hs, uint32_t m) {
  if (m >= hs.materials.size()) return Q_TERMINAL;
  switch (hs.materials[m].type) {
    case RTB_MAT_LAMBERTIAN: return Q_LAMBERT;
    case RTB_MAT_METAL: return Q_METAL;
    case RTB_MAT_DIELECTRIC: return Q_DIELECTRIC;
    case RTB_MAT_ISOTROPIC: return Q_ISOTROPIC;
    default: return Q_TERMINAL;  // DiffuseLight: emitted, no scatter (material.rs:184-190)
  }
}

// uploads the flattened scene + BVH of `host` to the device of `s` (s == host, or one of its replicas)
static int upload_scene(rtb_scene* s, const rtb_scene* host) {
  const HostScene& hs = host->hs;
  const HostBvh& bvh = host->bvh;
  CU(cudaSetDevice(s->ctx->device));
  s->present_materials = host->present_materials;

  DevScene& d = s->dev;
  std::memset(&d, 0, sizeof(d));
  CU(s->d_nodes.upload(reinterpret_cast<const uint4*>(bvh.nodes.data()), bvh.nodes.size() * 5));
  d.nodes = s->d_nodes.p;
  d.n_nodes = (uint32_t)bvh.nodes.size();
  d.prmt_magic = 0x43000000u;
  d.n_global = (uint32_t)bvh.global_refs.size();
  d.tree_empty = (d.n_global == (uint32_t)hs.prims.size()) ? 1u : 0u;
  for (uint32_t k = 0; k < d.n_global; ++k) d.global_ref[k] = bvh.global_refs[k];
  d.global_f64 = d.tree_empty ? 0u : bvh.global_f64;
  d._reserved0 = 0u;
  for (uint32_t t = 0; t < PT_COUNT; ++t) {
    CU(s->d_geom[t].upload(reinterpret_cast<const float4*>(bvh.geom[t].data()), bvh.geom[t].size() / 4));
    // device copy of the info words carries the shade queue of the primitive's material (RTB_MINFO_QUEUE)
    std::vector<uint32_t> info = bvh.info[t];
    for (size_t i = 1; i < info.size(); i += 2) info[i] |= queue_of_material(hs, info[i] & 0xFFFFFFu) << 28;
    CU(s->d_info[t].upload(reinterpret_cast<const uint2*>(info.data()), info.size() / 2));
    CU(cudaStreamSynchronize(0));  // `info` is a temporary
    d.geom[t] = s->d_geom[t].p;
    d.info[t] = s->d_info[t].p;
    d.n_prims[t] = (uint32_t)(bvh.info[t].size() / 2);
    CU(s->d_exact[t].upload(bvh.exact[t].data(), bvh.exact[t].size()));
  }
  d.coord_max = bvh.coord_max;
  d.eps_ab = bvh.eps_ab;
  std::vector<float4> mats(hs.materials.size() * 2);
  for (size_t i = 0; i < hs.materials.size(); ++i) {
    uint32_t ty = hs.materials[i].type, tx = hs.materials[i].texture, tt = 0xFFu;
    float4 rgb = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tx < hs.textures.size()) {
      tt = hs.textures[tx].type;
      if (tt == RTB_TEX_SOLID) rgb = make_float4((float)hs.textures[tx].rgb[0], (float)hs.textures[tx].rgb[1], (float)hs.textures[tx].rgb[2], 0.f);
    }
    float a, b, d;
    std::memcpy(&a, &ty, 4);
    std::memcpy(&b, &tx, 4);
    std::memcpy(&d, &tt, 4);
    mats[2 * i] = make_float4(a, b, (float)hs.materials[i].param, d);
    mats[2 * i + 1] = rgb;
  }
  CU(s->d_materials.upload(mats.data(), mats.size()));
  d.materials = s->d_materials.p;
  d.n_materials = (uint32_t)hs.materials.size();
  std::vector<DevTexture> texs(hs.textures.size());
  for (size_t i = 0; i < texs.size(); ++i) {
    const rtb_texture& t = hs.textures[i];
    texs[i] = DevTexture{t.type, t.even, t.odd, t.table, (float)t.rgb[0], (float)t.rgb[1], (float)t.rgb[2], (float)t.scale};
  }
  CU(s->d_textures.upload(texs.data(), texs.size()));
  d.textures = s->d_textures.p;
  {  // perlin tables and images: any number of them, packed into one buffer each (an unset perlin table stays zero)
    const size_t np = hs.perlins.size();
    std::vector<float> vec(np * 1024, 0.f);
    std::vector<uint8_t> perm(np * 768, 0);
    for (size_t i = 0; i < np; ++i) {
      if (!hs.perlins[i].set) continue;
      std::copy(hs.perlins[i].ranvec.begin(), hs.perlins[i].ranvec.end(), vec.begin() + i * 1024);
      std::copy(hs.perlins[i].perm.begin(), hs.perlins[i].perm.end(), perm.begin() + i * 768);
    }
    CU(s->d_perlin_vec.upload(reinterpret_cast<const float4*>(vec.data()), np * 256));
    CU(s->d_perlin_perm.upload(perm.data(), perm.size()));
    d.perlin_vec = s->d_perlin_vec.p;
    d.perlin_perm = s->d_perlin_perm.p;
    d.n_perlin = (uint32_t)np;
    const size_t ni = hs.images.size();
    size_t total = 0;
    for (size_t i = 0; i < ni; ++i) total += (hs.images[i].rgb.size() + 15) & ~(size_t)15;
    std::vector<uint8_t> data(total, 0);
    std::vector<DevImage> desc(ni);
    CU(s->d_image_data.resize(total));
    size_t off = 0;
    for (size_t i = 0; i < ni; ++i) {
      desc[i].data = hs.images[i].rgb.empty() ? nullptr : s->d_image_data.p + off;
      desc[i].w = hs.images[i].w;
      desc[i].h = hs.images[i].h;
      std::copy(hs.images[i].rgb.begin(), hs.images[i].rgb.end(), data.begin() + off);
      off += (hs.images[i].rgb.size() + 15) & ~(size_t)15;
    }
    CU(s->d_image_data.upload(data.data(), total));
    CU(s->d_images.upload(desc.data(), ni));
    CU(cudaStreamSynchronize(0));  // the staging vectors are temporaries
    d.images = s->d_images.p;
    d.n_images = (uint32_t)ni;
  }
  d.n_lights = (uint32_t)hs.lights.size();
  for (size_t i = 0; i < hs.lights.size(); ++i) {
    d.lights[i].type = hs.lights[i].type;
    for (int k = 0; k < 5; ++k) d.lights[i].p[k] = hs.lights[i].p[k];
  }
  d.n_media = (uint32_t)hs.media.size();
  for (size_t i = 0; i < hs.media.size(); ++i) {
    const HostMedium& m = hs.media[i];
    DevMedium& o = d.media[i];
    o.boundary_type = m.boundary_type; o.material = m.material; o.prim_id = m.prim_id;
    o.minfo = (m.material & 0xFFFFFFu) | (FACE_TRUE << 24) | (queue_of_material(hs, m.material) << 28);
    o.neg_inv_density = m.neg_inv_density;
    for (int k = 0; k < 6; ++k) o.p[k] = m.p[k];
    o.sin_t = m.sin_t; o.cos_t = m.cos_t;
    for (int k = 0; k < 3; ++k) o.off[k] = m.offset[k];
  }
  {
    ExactTab xt;
    std::memset(&xt, 0, sizeof(xt));
    xt.tri = s->d_geom[PT_TRI].p;
    for (int t = 0; t < 3; ++t) xt.exact[t] = s->d_exact[t].p;
    for (uint32_t t = 0; t < PT_COUNT; ++t) xt.info[t] = s->d_info[t].p;
    for (size_t i = 0; i < hs.media.size() && i < RTB_MAX_MEDIA; ++i) xt.media_prim_id[i] = hs.media[i].prim_id;
    CU(s->d_xtab.upload(&xt, 1));
    CU(cudaStreamSynchronize(0));  // `xt` is a temporary
    d.xtab = s->d_xtab.p;
  }
  CU(s->d_self.resize(1));
  d.self = s->d_self.p;
  CU(cudaMemcpy(s->d_self.p, &d, sizeof(DevScene), cudaMemcpyHostToDevice));  // (after every other field is final)
  int e = configure_launch(s->lc, d.n_nodes, s->bvh.max_depth, d.n_prims[PT_SPHERE], s->ctx->prop.multiProcessorCount);
  if (e != 0) return set_err(RTB_ERR_CUDA, std::string("configure_launch: ") + cudaGetErrorString((cudaError_t)e));
  CU(cudaStreamSynchronize(0));
  s->committed = true;
  return RTB_OK;
}

int rtb_scene_commit(rtb_scene* s) {
  if (!s) return set_err(RTB_ERR_INVALID, "scene is NULL");
  if (!s->ctx) return set_err(RTB_ERR_STATE, "host-only scene (created without a context) cannot be committed");
  if (!s->built) {
    int rc = rtb_scene_build_bvh(s);
    if (rc != RTB_OK) return rc;
  }
  int rc = upload_scene(s, s);
  for (size_t k = 0; k < s->replicas.size() && rc == RTB_OK; ++k) rc = upload_scene(s->replicas[k], s);  // same host data, every GPU
  return rc;
}


int rtb_scene_get_info(rtb_scene* s, rtb_scene_info* o) {
  if (!s || !o) return set_err(RTB_ERR_INVALID, "NULL argument");
  std::memset(o, 0, sizeof(*o));
  for (const HostPrim& p : s->hs.prims) {
    if (p.type == PT_SPHERE) o->n_spheres++;
    else if (p.type == PT_MOVING) o->n_moving++;
    else if (p.type == PT_QUAD) o->n_quads++;
    else o->n_triangles++;
  }
  o->n_media = (uint32_t)s->hs.media.size();
  o->n_lights = (uint32_t)s->hs.lights.size();
  o->n_materials = (uint32_t)s->hs.materials.size();
  o->n_textures = (uint32_t)s->hs.textures.size();
  o->n_prims = s->hs.n_prim_ids;
  o->n_bvh_nodes = (uint32_t)s->bvh.nodes.size();
  o->bvh_width = 8;
  o->bvh_max_depth = s->bvh.max_depth;
  o->bvh_bytes = (uint64_t)s->bvh.nodes.size() * sizeof(Node8);
  o->prim_bytes = 0;
  for (uint32_t t = 0; t < PT_COUNT; ++t) o->prim_bytes += s->bvh.geom[t].size() * 4 + s->bvh.info[t].size() * 4;
  o->global_f64_mask = (s->bvh.global_refs.size() == s->hs.prims.size()) ? 0u : s->bvh.global_f64;
  return RTB_OK;
}
int rtb_scene_export_bvh(rtb_scene* s, void* nodes, size_t cap) {
  if (!s || !nodes) return set_err(RTB_ERR_INVALID, "NULL argument");
  if (!s->built) return set_err(RTB_ERR_STATE, "BVH not built (call rtb_scene_build_bvh or rtb_scene_commit)");
  size_t bytes = s->bvh.nodes.size() * sizeof(Node8);
  if (cap < bytes) return set_err(RTB_ERR_INVALID, "buffer too small");
  std::memcpy(nodes, s->bvh.nodes.data(), bytes);
  return RTB_OK;
}
int rtb_scene_export_globals(rtb_scene* s, uint32_t* refs, uint32_t cap, uint32_t* n_out) {
  if (!s || !n_out) return set_err(RTB_ERR_INVALID, "bad argument");
  if (!s->built) return set_err(RTB_ERR_STATE, "BVH not built (call rtb_scene_build_bvh or rtb_scene_commit)");
  *n_out = (uint32_t)s->bvh.global_refs.size();
  if (refs) {
    if (cap < *n_out) return set_err(RTB_ERR_INVALID, "buffer too small");
    for (uint32_t k = 0; k < *n_out; ++k) refs[k] = s->bvh.global_refs[k];
  }
  return RTB_OK;
}
int rtb_scene_export_exact(rtb_scene* s, uint32_t type, double* out, size_t cap_bytes, float* coord_max, float* eps_ab) {
  if (!s || type >= PT_COUNT) return set_err(RTB_ERR_INVALID, "bad argument");
  if (!s->built) return set_err(RTB_ERR_STATE, "BVH not built (call rtb_scene_build_bvh or rtb_scene_commit)");
  const size_t bytes = s->bvh.exact[type].size() * sizeof(double);
  if (out && cap_bytes < bytes) return set_err(RTB_ERR_INVALID, "buffer too small");
  if (out && bytes) std::memcpy(out, s->bvh.exact[type].data(), bytes);
  if (coord_max) *coord_max = s->bvh.coord_max;
  if (eps_ab) *eps_ab = s->bvh.eps_ab;
  return RTB_OK;
}
int rtb_scene_export_prims(rtb_scene* s, uint32_t type, float* geom, size_t gcap, uint32_t* info, size_t icap) {
  if (!s || type >= PT_COUNT) return set_err(RTB_ERR_INVALID, "bad argument");
  if (!s->built) return set_err(RTB_ERR_STATE, "BVH not built (call rtb_scene_build_bvh or rtb_scene_commit)");
  size_t gb = s->bvh.geom[type].size() * 4, ib = s->bvh.info[type].size() * 4;
  if ((geom && gcap < gb) || (info && icap < ib)) return set_err(RTB_ERR_INVALID, "buffer too small");
  if (geom && gb) std::memcpy(geom, s->bvh.geom[type].data(), gb);
  if (info && ib) std::memcpy(info, s->bvh.info[type].data(), ib);
  return RTB_OK;
}

// ---- camera ------------------------------------------------------------------------------------------------------
static void camera_basis(const rtb_camera& c, DevCamera& f, DevCameraF64& g) {  // Camera::new, camera.rs:21-59
  const double PI = 3.14159265358979323846;
  double theta = c.vfov_deg * PI / 180.0;
  double h = std::tan(theta / 2.0);
  double vh = 2.0 * h, vw = c.aspect_ratio * vh;
  double w[3], u[3], v[3];
  double len = 0;
  for (int a = 0; a < 3; ++a) { w[a] = c.lookfrom[a] - c.lookat[a]; len += w[a] * w[a]; }
  len = std::sqrt(len);
  for (int a = 0; a < 3; ++a) w[a] /= len;
  u[0] = c.vup[1] * w[2] - c.vup[2] * w[1];
  u[1] = c.vup[2] * w[0] - c.vup[0] * w[2];
  u[2] = c.vup[0] * w[1] - c.vup[1] * w[0];
  len = std::sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
  for (int a = 0; a < 3; ++a) u[a] /= len;
  v[0] = w[1] * u[2] - w[2] * u[1];
  v[1] = w[2] * u[0] - w[0] * u[2];
  v[2] = w[0] * u[1] - w[1] * u[0];
  for (int a = 0; a < 3; ++a) {
    double hor = c.focus_dist * vw * u[a], ver = c.focus_dist * vh * v[a];
    double llc = c.lookfrom[a] - hor / 2.0 - ver / 2.0 - c.focus_dist * w[a];
    g.origin[a] = c.lookfrom[a]; g.llc[a] = llc; g.horizontal[a] = hor; g.vertical[a] = ver;
    f.origin[a] = (float)c.lookfrom[a];
    f.lmo[a] = (float)(llc - c.lookfrom[a]);
    f.horizontal[a] = (float)hor; f.vertical[a] = (float)ver;
    f.u[a] = (float)u[a]; f.v[a] = (float)v[a];
  }
  g.time0 = c.time0;
  f.lens_radius = (float)(c.aperture / 2.0);
  f.time0 = (float)c.time0; f.time1 = (float)c.time1;
}

// ---- render --------------------------------------------------------------------------------------------------------
static int ensure_pool(Lane& c, uint32_t n) {
  if (c.pool_n >= n) return RTB_OK;
  CU(c.ray.resize((size_t)n * 2)); CU(c.st.resize((size_t)n * 2)); CU(c.hit.resize(n));
  const size_t chunks = ((size_t)n + RTB_CHUNK - 1) / RTB_CHUNK;
  CU(c.cls.resize(chunks * RTB_CHUNK)); CU(c.cursor.resize(chunks));
  CU(c.redo[0].resize(n));
  c.pool_n = n;
  return RTB_OK;
}

static DevPool lane_pool(Lane& L, uint32_t n) {
  DevPool p;
  p.n = n;
  p.n_chunks = (n + RTB_CHUNK - 1) / RTB_CHUNK;
  p.ray = L.ray.p; p.st = L.st.p; p.hit = L.hit.p;
  p.cls = L.cls.p; p.redo[0] = L.redo[0].p; p.redo[1] = L.redo[1].p; p.cursor = L.cursor.p;
  p.c = L.counters.p;
  return p;
}

static int ensure_pix_order(rtb_context* c, uint32_t W, uint32_t H, cudaStream_t st) {
  if (c->pix_w == W && c->pix_h == H && c->pix_order.p) return RTB_OK;
  // 8x4-pixel tiles (one warp of neighbouring primary rays), tiles row-major
  std::vector<uint32_t> order;
  order.reserve((size_t)W * H);
  for (uint32_t ty = 0; ty < H; ty += 4)
    for (uint32_t tx = 0; tx < W; tx += 8)
      for (uint32_t y = ty; y < std::min(ty + 4, H); ++y)
        for (uint32_t x = tx; x < std::min(tx + 8, W); ++x) order.push_back(y * W + x);
  CU(c->pix_order.upload(order.data(), order.size(), st));
  CU(cudaStreamSynchronize(st));
  c->pix_w = W; c->pix_h = H;
  return RTB_OK;
}

#define RTB_DEFAULT_POOL (1u << 22)  // path-pool slots of all lanes together when rtb_params::pool_paths is 0

// the argument checks rtb_render_device and rtb_render_aov_device share
static int check_render_args(rtb_context* c, rtb_scene* s, const rtb_camera* cam, const rtb_params* p, const void* buf) {
  if (!c || !s || !cam || !p || !buf) return set_err(RTB_ERR_INVALID, "NULL argument");
  if (!s->committed) return set_err(RTB_ERR_STATE, "scene not committed (call rtb_scene_commit)");
  if (p->width < 2 || p->height < 2) return set_err(RTB_ERR_INVALID, "image must be at least 2x2 (u = (i+xi)/(W-1), main.rs:752)");
  if (p->max_depth < 1 || p->max_depth > 255) return set_err(RTB_ERR_INVALID, "max_depth must be in [1,255]");
  if (p->spp == 0) return set_err(RTB_ERR_INVALID, "spp must be > 0");
  if ((uint64_t)p->sample_offset + p->spp > (1u << 24)) return set_err(RTB_ERR_INVALID, "sample index exceeds 2^24");
  return RTB_OK;
}

// the f32 camera of the render's primary rays; refuses a camera whose basis is not finite
static int render_camera(const rtb_camera& cam, DevCamera& dcam) {
  DevCameraF64 dcam64;
  camera_basis(cam, dcam, dcam64);
  for (int a = 0; a < 3; ++a)  // lookfrom == lookat, vup parallel to the view direction, NaN / inf arguments
    if (!std::isfinite(dcam.origin[a]) || !std::isfinite(dcam.lmo[a]) || !std::isfinite(dcam.horizontal[a]) || !std::isfinite(dcam.vertical[a]) ||
        !std::isfinite(dcam.u[a]) || !std::isfinite(dcam.v[a]))
      return set_err(RTB_ERR_INVALID, "degenerate camera (non-finite basis: lookfrom == lookat, vup along the view direction, or non-finite arguments)");
  return RTB_OK;
}

// DevParams::opt of the scene's extend launches.  Per-scene scheduling of the extend kernel (profiles/r3_ab.md): deep trees
// (dynamic fetch) park their leaf tests, trees that do not fit the shared-memory stage order each chunk's rays by direction
// octant, small staged trees do neither.  RTB_OPT overrides (experiments).
static uint32_t extend_opt(const rtb_scene* s) {
  static const char* env_opt = getenv("RTB_OPT");
  return env_opt ? (uint32_t)atoi(env_opt)
         : s->lc.mode == EXTEND_WQ ? ((24u << RTB_OPT_PARK_SHIFT) | (2u << 16))  // serve queues of >= 24 rays, 2 tests per ray and round
         : s->lc.mode == EXTEND_DYNAMIC ? (14u << RTB_OPT_PARK_SHIFT)
                                        : (s->lc.all_staged ? 0u : 2u /* RTB_OPT_OCTANT_SORT */);
}

// lanes: concurrent wavefront instances on disjoint sample ranges
// 4 lanes: C1 7696 -> 7882, C3 +2.6 % against 3; the dynamic-fetch kernel at 64 registers co-schedules the extend CTAs of
// four lanes on an SM: C4 3915 (3 lanes) -> 4096 (4), 5 / 6 lanes add nothing (profiles/r3_ab.md §9)
static int default_lanes() {
  static const int env_lanes = getenv("RTB_LANES") ? atoi(getenv("RTB_LANES")) : 0;
  const int want_lanes = env_lanes > 0 ? env_lanes : 4;
  return std::max(1, std::min(want_lanes, RTB_MAX_LANES));
}

int rtb_render_device(rtb_context* c, rtb_scene* s, const rtb_camera* cam, const rtb_params* p, void* d_accum,
                      void* stream, rtb_stats* stats) {
  int rc = check_render_args(c, s, cam, p, d_accum);
  if (rc) return rc;
  CU(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  const uint64_t npix = (uint64_t)p->width * p->height;
  const bool count = (p->flags & RTB_RENDER_COUNT) != 0, time_ext = (p->flags & RTB_RENDER_TIME_EXTEND) != 0;
  // instrumented runs use one lane so that the per-launch timings / counters describe the kernel alone
  int n_lanes = (count || time_ext) ? 1 : default_lanes();
  if ((uint32_t)n_lanes > p->spp) n_lanes = (int)p->spp;
  uint32_t pool_total = p->pool_paths ? p->pool_paths : RTB_DEFAULT_POOL;  // all lanes together; 112 B per slot
  rc = ensure_pix_order(c, p->width, p->height, st);
  if (rc) return rc;
  DevCamera dcam;
  rc = render_camera(*cam, dcam);
  if (rc) return rc;

  struct LaneRun { DevPool pool; DevParams prm; unsigned long long total; bool active; uint64_t iters, iter_cap; };
  LaneRun run[RTB_MAX_LANES];
  uint32_t first_sample = 0;
  for (int k = 0; k < n_lanes; ++k) {
    Lane& L = c->lanes[k];
    const uint32_t cnt = p->spp / n_lanes + ((uint32_t)k < p->spp % n_lanes ? 1u : 0u);
    LaneRun& R = run[k];
    R.total = npix * cnt;
    // Pools are a whole number of "units" (one RTB_CHUNK-slot chunk per resident shade warp) so that every warp of a
    // shade kernel gets the same number of chunks; small renders get a pool no larger than their path count.
    uint32_t pool_n = std::max(1024u, pool_total / (uint32_t)n_lanes);
    const uint32_t unit = s->lc.pool_unit;
    if (!p->pool_paths && unit) pool_n = std::max(1u, (pool_n + unit / 2) / unit) * unit;
    if ((unsigned long long)pool_n > R.total) pool_n = (uint32_t)std::max<unsigned long long>(1024ull, R.total);
    rc = ensure_pool(L, pool_n);
    if (rc) return rc;
    R.pool = lane_pool(L, pool_n);
    DevParams& prm = R.prm;
    prm.width = p->width; prm.height = p->height; prm.spp = cnt; prm.sample_offset = p->sample_offset + first_sample;
    prm.max_depth = p->max_depth; prm.rr_start = p->rr_start_depth; prm.seed = p->seed;
    for (int a = 0; a < 3; ++a) prm.bg[a] = p->background[a];
    prm.pix_order = c->pix_order.p;
    prm.inv_npix = 1.0 / (double)npix;
    prm.opt = extend_opt(s);
    prm.inv_wm1 = (float)(1.0 / (double)(p->width - 1));
    prm.inv_hm1 = (float)(1.0 / (double)(p->height - 1));
    prm.accum = (float4*)d_accum;
    first_sample += cnt;
    R.active = true;
    R.iters = 0;
    R.iter_cap = 2 * (uint64_t)(R.total / pool_n + 2) * (uint64_t)(p->max_depth + 2) + 64;
  }

  uint64_t launches = 0, extend_launches = 0;
  CU(cudaEventRecord(c->ev0, st));
  if (!(p->flags & RTB_RENDER_ACCUMULATE)) CU(cudaMemsetAsync(d_accum, 0, npix * sizeof(float4), st));
  CU(cudaEventRecord(c->ev_fork, st));
  for (int k = 0; k < n_lanes; ++k) {
    cudaStream_t ls = c->lanes[k].stream;
    CU(cudaStreamWaitEvent(ls, c->ev_fork, 0));
    launch_init_pool(run[k].pool, run[k].total, ls);
    launch_generate(s->lc, run[k].pool, run[k].prm, dcam, ls);
    launch_rotate(run[k].pool, ls);
    launches += 3;
  }
  const uint32_t present = s->present_materials;
  const uint32_t n_shade = 1 + ((present >> RTB_MAT_LAMBERTIAN) & 1u) + ((present >> RTB_MAT_ISOTROPIC) & 1u) +
                           ((present & ((1u << RTB_MAT_METAL) | (1u << RTB_MAT_DIELECTRIC))) ? 1u : 0u);
  // The drain check is PIPELINED: batch b + 1 (8 iterations per lane) is queued before the host waits for the counters of
  // batch b, so the lanes never run dry while the host looks at a counter (a lane that turns out to have drained has
  // queued one more batch of iterations over an all-dead pool: a few microseconds each).  On any error every lane stream is
  // synchronised before returning: nothing may still be writing the caller's accumulation buffer.
  const uint32_t check_every = 8;
  size_t ev_used = 0;
  int n_active = n_lanes;
  auto sync_all = [&]() { for (int q = 0; q < n_lanes; ++q) cudaStreamSynchronize(c->lanes[q].stream); };
  auto enqueue_batch = [&](uint32_t b) -> cudaError_t {
    cudaError_t e = cudaSuccess;
    for (uint32_t it = 0; it < check_every; ++it) {
      for (int k = 0; k < n_lanes; ++k) {  // interleave the lanes' launches so that their phases stay staggered
        if (!run[k].active) continue;
        cudaStream_t ls = c->lanes[k].stream;
        if (time_ext) {
          if (c->ext_events.size() < ev_used + 2) {
            cudaEvent_t a2, b2;
            if ((e = cudaEventCreate(&a2)) != cudaSuccess) return e;
            if ((e = cudaEventCreate(&b2)) != cudaSuccess) return e;
            c->ext_events.push_back(a2);
            c->ext_events.push_back(b2);
          }
          if ((e = cudaEventRecord(c->ext_events[ev_used], ls)) != cudaSuccess) return e;
        }
        launch_extend(s->lc, s->dev, run[k].pool, run[k].prm, count, ls);
        if (time_ext) {
          if ((e = cudaEventRecord(c->ext_events[ev_used + 1], ls)) != cudaSuccess) return e;
          ev_used += 2;
        }
        launch_fixup(s->lc, s->dev, run[k].pool, run[k].prm, ls);  // exact pass over the rays this launch queued
        launch_shade(s->lc, s->dev, run[k].pool, run[k].prm, dcam, present, ls);
        launches += 2 + n_shade;
        extend_launches += 1;
      }
    }
    for (int k = 0; k < n_lanes; ++k) {
      if (!run[k].active) continue;
      Lane& L = c->lanes[k];
      if ((e = cudaMemcpyAsync(L.h_counters + (b & 1u), L.counters.p, sizeof(DevCounters), cudaMemcpyDeviceToHost, L.stream)) != cudaSuccess) return e;
      if ((e = cudaEventRecord(L.batch_done[b & 1u], L.stream)) != cudaSuccess) return e;
    }
    return cudaGetLastError();
  };
  auto fail_cuda = [&](cudaError_t e, const char* what) {
    sync_all();
    return set_err(RTB_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  };
  cudaError_t qe = enqueue_batch(0);
  if (qe != cudaSuccess) return fail_cuda(qe, "wavefront launch");
  for (uint32_t b = 0; n_active > 0; ++b) {
    // (instrumented runs keep the strict order: their per-launch timings must not contain idle iterations)
    const bool ahead = !(count || time_ext);
    if (ahead && (qe = enqueue_batch(b + 1)) != cudaSuccess) return fail_cuda(qe, "wavefront launch");
    for (int k = 0; k < n_lanes; ++k) {
      if (!run[k].active) continue;
      if ((qe = cudaEventSynchronize(c->lanes[k].batch_done[b & 1u])) != cudaSuccess) return fail_cuda(qe, "wavefront");
      run[k].iters += check_every;
      const DevCounters* h = c->lanes[k].h_counters + (b & 1u);
      if (h->last_rays == 0) {
        run[k].active = false;
        --n_active;
      } else if (run[k].iters > run[k].iter_cap) {
        sync_all();
        return set_err(RTB_ERR_CUDA, "wavefront did not drain (internal error)");
      }
    }
    if (!ahead && n_active > 0 && (qe = enqueue_batch(b + 1)) != cudaSuccess) return fail_cuda(qe, "wavefront launch");
  }
  for (int k = 0; k < n_lanes; ++k) {  // final counters (a drained lane may still have an idle batch in flight)
    Lane& L = c->lanes[k];
    if ((qe = cudaMemcpyAsync(L.h_counters, L.counters.p, sizeof(DevCounters), cudaMemcpyDeviceToHost, L.stream)) != cudaSuccess)
      return fail_cuda(qe, "counter read-back");
  }
  for (int k = 0; k < n_lanes; ++k) {
    CU(cudaEventRecord(c->lanes[k].done, c->lanes[k].stream));
    CU(cudaStreamWaitEvent(st, c->lanes[k].done, 0));
  }
  CU(cudaEventRecord(c->ev1, st));
  float ms_nccl = 0.f, ms_wait = 0.f;
  if ((p->flags & RTB_RENDER_REDUCE) && c->n_ranks > 1) {
    // one ncclReduce(float32, 4 W H, sum, root 0) per frame, in place, on the caller's stream (SURVEY §8e).  A one-float
    // reduce in front of it is the arrival barrier: ranks finish rendering a few ms apart, and that skew is waiting,
    // not collective time (ms_nccl_wait vs ms_nccl).
    if (!c->comm) return set_err(RTB_ERR_STATE, "RTB_RENDER_REDUCE needs a communicator (rtb_context_comm_init)");
    CU(cudaEventRecord(c->ev_w0, st));
    int r = nccl_api().Reduce(c->comm_scratch.p, c->comm_scratch.p, 1, kNcclFloat32, kNcclSum, 0, c->comm, st);
    CU(cudaEventRecord(c->ev_n0, st));
    if (r == kNcclSuccess) r = nccl_api().Reduce(d_accum, d_accum, npix * 4, kNcclFloat32, kNcclSum, 0, c->comm, st);
    if (r != kNcclSuccess) return set_err(RTB_ERR_CUDA, std::string("ncclReduce: ") + nccl_api().GetErrorString(r));
    CU(cudaEventRecord(c->ev_n1, st));
    CU(cudaEventSynchronize(c->ev_n1));
    cudaEventElapsedTime(&ms_nccl, c->ev_n0, c->ev_n1);
    cudaEventElapsedTime(&ms_wait, c->ev_w0, c->ev_n0);
  }
  CU(cudaEventSynchronize(c->ev1));
  CU(cudaGetLastError());
  if (stats) {
    std::memset(stats, 0, sizeof(*stats));
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    stats->ms_nccl = ms_nccl;
    stats->ms_nccl_wait = ms_wait;
    stats->ms_render = ms;
    stats->n_devices = 1;
    ms += ms_nccl + ms_wait;
    for (int k = 0; k < n_lanes; ++k) {
      const DevCounters* h = c->lanes[k].h_counters;
      stats->paths += run[k].total;  // a render always runs to completion: every path number was started exactly once
      stats->segments += h->segments;
      stats->rejected += h->rejected;
      stats->exact_rays += h->redone - h->refined;
      stats->refined_rays += h->refined;
      stats->iterations = std::max<uint64_t>(stats->iterations, h->iter);
      stats->nodes_visited += h->nodes_visited;
      stats->prims_tested += h->prims_tested;
      for (uint32_t t = 0; t < PT_COUNT; ++t) stats->prims_tested_type[t] += h->prims_tested_type[t];
    }
    stats->launches = launches;
    stats->extend_launches = extend_launches;
    stats->ms_total = ms;
    double ms_ext = 0;
    for (size_t k = 0; k + 1 < ev_used; k += 2) {
      float e = 0;
      cudaEventElapsedTime(&e, c->ext_events[k], c->ext_events[k + 1]);
      ms_ext += e;
    }
    stats->ms_extend = ms_ext;
  }
  return RTB_OK;
}

// One process, n GPUs: device k renders its share of the samples of EVERY pixel on its own thread, then all of them join one
// ncclReduce onto device 0 (replaces the reference's only parallelism, the per-pixel thread fan-out of main.rs:730-778).
static int render_multi(rtb_context* c, rtb_scene* s, const rtb_camera* cam, const rtb_params* p, rtb_stats* stats) {
  const int n = 1 + (int)c->peers.size();
  if ((int)s->replicas.size() != n - 1) return set_err(RTB_ERR_STATE, "scene was not created on this multi-device context");
  const size_t npix = (size_t)p->width * p->height;
  std::vector<rtb_context*> ctxs{c};
  std::vector<rtb_scene*> scs{s};
  for (int k = 1; k < n; ++k) { ctxs.push_back(c->peers[(size_t)k - 1]); scs.push_back(s->replicas[(size_t)k - 1]); }
  std::vector<int> rc((size_t)n, RTB_OK);
  std::vector<std::string> msg((size_t)n);
  std::vector<rtb_stats> st((size_t)n);
  std::vector<float> ms_nccl((size_t)n, 0.f);
  std::atomic<int> arrived{0};
  std::atomic<bool> failed{false};
  auto work = [&](int k) {
    rtb_context* ck = ctxs[(size_t)k];
    auto fail = [&](int code, const std::string& m) { rc[(size_t)k] = code; msg[(size_t)k] = m; failed = true; };
    std::memset(&st[(size_t)k], 0, sizeof(rtb_stats));
    const uint32_t base = p->spp / (uint32_t)n, rem = p->spp % (uint32_t)n;
    const uint32_t cnt = base + ((uint32_t)k < rem ? 1u : 0u), first = (uint32_t)k * base + std::min((uint32_t)k, rem);
    cudaError_t e = cudaSetDevice(ck->device);
    if (e == cudaSuccess) e = ck->accum.resize(npix);
    if (e != cudaSuccess) fail(RTB_ERR_CUDA, cudaGetErrorString(e));
    if (rc[(size_t)k] == RTB_OK) {
      if (cnt == 0) {
        e = (p->flags & RTB_RENDER_ACCUMULATE) ? cudaSuccess : cudaMemset(ck->accum.p, 0, npix * sizeof(float4));
        if (e != cudaSuccess) fail(RTB_ERR_CUDA, cudaGetErrorString(e));
      } else {
        rtb_params pk = *p;
        pk.spp = cnt;
        pk.sample_offset = p->sample_offset + first;
        pk.flags &= ~RTB_RENDER_REDUCE;
        if (pk.pool_paths) pk.pool_paths = std::max(1024u, pk.pool_paths);
        const int r = rtb_render_device(ck, scs[(size_t)k], cam, &pk, ck->accum.p, nullptr, &st[(size_t)k]);
        if (r != RTB_OK) fail(r, g_err);
      }
    }
    // every device finished rendering before the collective starts: ms_nccl is the reduce alone
    arrived.fetch_add(1);
    while (arrived.load() < n) std::this_thread::yield();
    if (failed.load()) return;  // no device enters the collective when one of them failed
    cudaEventRecord(ck->ev_n0, 0);
    const int r = nccl_api().Reduce(ck->accum.p, ck->accum.p, npix * 4, kNcclFloat32, kNcclSum, 0, ck->comm, (cudaStream_t)0);
    cudaEventRecord(ck->ev_n1, 0);
    e = cudaEventSynchronize(ck->ev_n1);
    if (r != kNcclSuccess) fail(RTB_ERR_CUDA, std::string("ncclReduce: ") + nccl_api().GetErrorString(r));
    else if (e != cudaSuccess) fail(RTB_ERR_CUDA, cudaGetErrorString(e));
    else cudaEventElapsedTime(&ms_nccl[(size_t)k], ck->ev_n0, ck->ev_n1);
  };
  std::vector<std::thread> pool;
  for (int k = 1; k < n; ++k) pool.emplace_back(work, k);
  work(0);
  for (std::thread& t : pool) t.join();
  for (int k = 0; k < n; ++k)
    if (rc[(size_t)k] != RTB_OK) return set_err(rc[(size_t)k], "device " + std::to_string(ctxs[(size_t)k]->device) + ": " + msg[(size_t)k]);
  CU(cudaSetDevice(c->device));
  if (stats) {
    std::memset(stats, 0, sizeof(*stats));
    for (int k = 0; k < n; ++k) {
      const rtb_stats& q = st[(size_t)k];
      stats->paths += q.paths; stats->segments += q.segments; stats->rejected += q.rejected;
      stats->launches += q.launches; stats->extend_launches += q.extend_launches;
      stats->nodes_visited += q.nodes_visited; stats->prims_tested += q.prims_tested;
      for (uint32_t t = 0; t < PT_COUNT; ++t) stats->prims_tested_type[t] += q.prims_tested_type[t];
      stats->exact_rays += q.exact_rays; stats->refined_rays += q.refined_rays;
      stats->iterations = std::max(stats->iterations, q.iterations);
      stats->ms_render = std::max(stats->ms_render, q.ms_total);
      stats->ms_extend = std::max(stats->ms_extend, q.ms_extend);
    }
    stats->ms_nccl = ms_nccl[0];
    stats->ms_total = stats->ms_render + stats->ms_nccl;
    stats->n_devices = (uint32_t)n;
  }
  return RTB_OK;
}

int rtb_render(rtb_context* c, rtb_scene* s, const rtb_camera* cam, const rtb_params* p, float* accum_out,
               rtb_stats* stats) {
  if (!c || !p) return set_err(RTB_ERR_INVALID, "NULL argument");
  CU(cudaSetDevice(c->device));
  const size_t npix = (size_t)p->width * p->height;
  if (!c->peers.empty()) {
    if (!s || !cam) return set_err(RTB_ERR_INVALID, "NULL argument");
    if (!s->committed) return set_err(RTB_ERR_STATE, "scene not committed (call rtb_scene_commit)");
    if (p->spp == 0) return set_err(RTB_ERR_INVALID, "spp must be > 0");
    int rc = render_multi(c, s, cam, p, stats);
    if (rc) return rc;
    if (accum_out) CU(cudaMemcpy(accum_out, c->accum.p, npix * sizeof(float4), cudaMemcpyDeviceToHost));
    return RTB_OK;
  }
  CU(c->accum.resize(npix));
  int rc = rtb_render_device(c, s, cam, p, c->accum.p, nullptr, stats);
  if (rc) return rc;
  if (accum_out) CU(cudaMemcpy(accum_out, c->accum.p, npix * sizeof(float4), cudaMemcpyDeviceToHost));
  return RTB_OK;
}

// ---- denoiser guide buffers ---------------------------------------------------------------------------------------------
// The first segment of every sample a render with the same params traces, through the production extend + k_fixup.  The
// W*H*spp paths are numbered as the render numbers them (start_path) and processed in batches of one lane pool each; batch
// b runs on lane b % n_lanes, so one lane's fill / collect overlaps another lane's extend.  A lane's pool is initialised
// once: k_fixup leaves the per-launch counters cleared, so the lane's totals (exact rays, rejected samples) add up over its
// batches.
int rtb_render_aov_device(rtb_context* c, rtb_scene* s, const rtb_camera* cam, const rtb_params* p, void* d_aov,
                          void* stream, rtb_stats* stats) {
  int rc = check_render_args(c, s, cam, p, d_aov);
  if (rc) return rc;
  if (p->flags & ~RTB_RENDER_ACCUMULATE) return set_err(RTB_ERR_INVALID, "rtb_render_aov accepts no flag but RTB_RENDER_ACCUMULATE");
  if (!c->peers.empty())
    return set_err(RTB_ERR_UNSUPPORTED, "rtb_render_aov runs on one device: split the samples with sample_offset and sum the buffers");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  const uint64_t npix = (uint64_t)p->width * p->height, total = npix * p->spp;
  rc = ensure_pix_order(c, p->width, p->height, st);
  if (rc) return rc;
  DevCamera dcam;
  rc = render_camera(*cam, dcam);
  if (rc) return rc;
  DevParams prm;
  std::memset(&prm, 0, sizeof(prm));
  prm.width = p->width; prm.height = p->height; prm.spp = p->spp; prm.sample_offset = p->sample_offset;
  prm.max_depth = p->max_depth; prm.rr_start = p->rr_start_depth; prm.seed = p->seed;
  for (int a = 0; a < 3; ++a) prm.bg[a] = p->background[a];
  prm.pix_order = c->pix_order.p;
  prm.inv_npix = 1.0 / (double)npix;
  prm.opt = extend_opt(s);
  prm.inv_wm1 = (float)(1.0 / (double)(p->width - 1));
  prm.inv_hm1 = (float)(1.0 / (double)(p->height - 1));

  // one round of batches = the pool of all lanes together (pool_paths, as for the render), split as evenly as it goes
  const uint64_t round = std::min<uint64_t>(p->pool_paths ? p->pool_paths : RTB_DEFAULT_POOL, total);
  const int n_lanes = (int)std::min<uint64_t>((uint64_t)default_lanes(), round);
  DevPool pool[RTB_MAX_LANES];
  for (int k = 0; k < n_lanes; ++k) {
    const uint32_t n = (uint32_t)(round / n_lanes + ((uint64_t)k < round % n_lanes ? 1u : 0u));
    rc = ensure_pool(c->lanes[k], n);
    if (rc) return rc;
    pool[k] = lane_pool(c->lanes[k], n);
  }
  float4* aov = (float4*)d_aov;
  uint64_t launches = 0, extend_launches = 0;
  CU(cudaEventRecord(c->ev0, st));
  if (!(p->flags & RTB_RENDER_ACCUMULATE)) CU(cudaMemsetAsync(d_aov, 0, npix * 2 * sizeof(float4), st));
  CU(cudaEventRecord(c->ev_fork, st));
  for (int k = 0; k < n_lanes; ++k) {
    CU(cudaStreamWaitEvent(c->lanes[k].stream, c->ev_fork, 0));
    launch_init_pool(pool[k], 0ull, c->lanes[k].stream);
    launches += 1;
  }
  for (uint64_t first = 0, b = 0; first < total; ++b) {
    const int k = (int)(b % (uint64_t)n_lanes);
    const cudaStream_t ls = c->lanes[k].stream;
    const uint32_t n = (uint32_t)std::min<uint64_t>(pool[k].n, total - first);
    launch_aov_fill(pool[k], prm, dcam, first, n, ls);
    launch_extend(s->lc, s->dev, pool[k], prm, false, ls);
    launch_fixup(s->lc, s->dev, pool[k], prm, ls);
    launch_aov_collect(s->dev, pool[k], prm, aov, n, ls);
    launches += 4;
    extend_launches += 1;
    first += n;
  }
  cudaError_t e = cudaGetLastError();
  for (int k = 0; k < n_lanes && e == cudaSuccess; ++k) {
    Lane& L = c->lanes[k];
    e = cudaMemcpyAsync(L.h_counters, L.counters.p, sizeof(DevCounters), cudaMemcpyDeviceToHost, L.stream);
    if (e == cudaSuccess) e = cudaEventRecord(L.done, L.stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(st, L.done, 0);
  }
  if (e != cudaSuccess) {  // nothing may still be writing the caller's buffer
    for (int k = 0; k < n_lanes; ++k) cudaStreamSynchronize(c->lanes[k].stream);
    return set_err(RTB_ERR_CUDA, std::string("aov pass: ") + cudaGetErrorString(e));
  }
  CU(cudaEventRecord(c->ev1, st));
  CU(cudaEventSynchronize(c->ev1));
  CU(cudaGetLastError());
  if (stats) {
    std::memset(stats, 0, sizeof(*stats));
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    stats->paths = total;
    stats->segments = total;
    for (int k = 0; k < n_lanes; ++k) {
      const DevCounters* h = c->lanes[k].h_counters;
      stats->rejected += h->rejected;
      stats->exact_rays += h->redone - h->refined;
      stats->refined_rays += h->refined;
    }
    stats->launches = launches;
    stats->extend_launches = extend_launches;
    stats->ms_total = ms;
    stats->ms_render = ms;
    stats->n_devices = 1;
  }
  return RTB_OK;
}

int rtb_render_aov(rtb_context* c, rtb_scene* s, const rtb_camera* cam, const rtb_params* p, float* aov_out,
                   rtb_stats* stats) {
  if (!c || !p) return set_err(RTB_ERR_INVALID, "NULL argument");
  if (!c->peers.empty())
    return set_err(RTB_ERR_UNSUPPORTED, "rtb_render_aov runs on one device: split the samples with sample_offset and sum the buffers");
  CU(cudaSetDevice(c->device));
  const size_t npix = (size_t)p->width * p->height;
  CU(c->aov.resize(npix * 2));
  int rc = rtb_render_aov_device(c, s, cam, p, c->aov.p, nullptr, stats);
  if (rc) return rc;
  if (aov_out) CU(cudaMemcpy(aov_out, c->aov.p, npix * 2 * sizeof(float4), cudaMemcpyDeviceToHost));
  return RTB_OK;
}

int rtb_finalize_rgb8(rtb_context* c, const void* d_accum, uint32_t W, uint32_t H, uint32_t total_spp, uint8_t* out) {
  if (!c || !out || !total_spp) return set_err(RTB_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  const size_t npix = (size_t)W * H;
  const float4* src = d_accum ? (const float4*)d_accum : c->accum.p;
  if (!src) return set_err(RTB_ERR_STATE, "nothing rendered yet");
  CU(c->rgb8.resize(npix * 3));
  launch_finalize(src, c->rgb8.p, (uint32_t)npix, 1.0f / (float)total_spp, 0);
  CU(cudaMemcpy(out, c->rgb8.p, npix * 3, cudaMemcpyDeviceToHost));
  return RTB_OK;
}

// The probes run the PRODUCTION kernels: the rays are written into a path pool, one extend launch (the variant the
// scene's renders use) + k_fixup trace them, and the hit records are read back.
static int run_probe(rtb_context* c, rtb_scene* s, uint32_t n, uint32_t* id_out, float* t_out, rtb_stats* stats) {
  CU(c->p_id.resize(n));
  CU(c->p_t.resize(n));
  Lane& L = c->lanes[0];
  int rc = ensure_pool(L, std::max(n, 1024u));
  if (rc) return rc;
  const DevPool pool = lane_pool(L, n);
  DevParams prm;
  std::memset(&prm, 0, sizeof(prm));
  prm.opt = RTB_OPT_PROBE;
  float ms = 0;
  for (int pass = 0; pass < (stats ? 2 : 1); ++pass) {  // pass 1: the instrumented variant, for the counters only
    launch_init_pool(pool, 0ull, 0);
    launch_probe_fill(pool, c->p_org.p, c->p_dir.p, c->p_time.p, n, 0);
    CU(cudaEventRecord(c->ev0, 0));
    launch_extend(s->lc, s->dev, pool, prm, pass == 1, 0);
    launch_fixup(s->lc, s->dev, pool, prm, 0);
    CU(cudaEventRecord(c->ev1, 0));
    if (pass == 0) {
      launch_probe_collect(s->dev, pool, n, c->p_id.p, c->p_t.p, 0);
      CU(cudaMemcpy(id_out, c->p_id.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
      CU(cudaMemcpy(t_out, c->p_t.p, n * sizeof(float), cudaMemcpyDeviceToHost));
      cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    }
  }
  CU(cudaMemcpy(c->h_counters, L.counters.p, sizeof(DevCounters), cudaMemcpyDeviceToHost));
  CU(cudaGetLastError());
  if (stats) {
    std::memset(stats, 0, sizeof(*stats));
    stats->paths = n;
    stats->segments = n;
    stats->launches = 2;
    stats->extend_launches = 1;
    stats->ms_total = ms;
    stats->ms_extend = ms;
    stats->nodes_visited = c->h_counters->nodes_visited;
    stats->prims_tested = c->h_counters->prims_tested;
    for (uint32_t t = 0; t < PT_COUNT; ++t) stats->prims_tested_type[t] = c->h_counters->prims_tested_type[t];
    stats->exact_rays = c->h_counters->redone - c->h_counters->refined;
    stats->refined_rays = c->h_counters->refined;
  }
  return RTB_OK;
}

int rtb_primary_hits(rtb_context* c, rtb_scene* s, const rtb_camera* cam, uint32_t W, uint32_t H, uint32_t* id_out,
                     float* t_out, rtb_stats* stats) {
  if (!c || !s || !cam || !id_out || !t_out) return set_err(RTB_ERR_INVALID, "NULL argument");
  if (!s->committed) return set_err(RTB_ERR_STATE, "scene not committed (call rtb_scene_commit)");
  if (W < 2 || H < 2) return set_err(RTB_ERR_INVALID, "image must be at least 2x2");
  CU(cudaSetDevice(c->device));
  const uint32_t n = W * H;
  CU(c->p_org.resize((size_t)n * 3)); CU(c->p_dir.resize((size_t)n * 3)); CU(c->p_time.resize(n));
  DevCamera f;
  DevCameraF64 g;
  camera_basis(*cam, f, g);
  launch_primary_rays(g, W, H, c->p_org.p, c->p_dir.p, c->p_time.p, 0);
  return run_probe(c, s, n, id_out, t_out, stats);
}

int rtb_primary_rays(rtb_context* c, const rtb_camera* cam, uint32_t W, uint32_t H, float* org, float* dir, float* time) {
  if (!c || !cam || !org || !dir) return set_err(RTB_ERR_INVALID, "NULL argument");
  if (W < 2 || H < 2) return set_err(RTB_ERR_INVALID, "image must be at least 2x2");
  CU(cudaSetDevice(c->device));
  const size_t n = (size_t)W * H;
  CU(c->p_org.resize(n * 3)); CU(c->p_dir.resize(n * 3)); CU(c->p_time.resize(n));
  DevCamera f;
  DevCameraF64 g;
  camera_basis(*cam, f, g);
  launch_primary_rays(g, W, H, c->p_org.p, c->p_dir.p, c->p_time.p, 0);
  CU(cudaMemcpy(org, c->p_org.p, n * 3 * sizeof(float), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(dir, c->p_dir.p, n * 3 * sizeof(float), cudaMemcpyDeviceToHost));
  if (time) CU(cudaMemcpy(time, c->p_time.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  return RTB_OK;
}

int rtb_device_kat(rtb_context* c, rtb_scene* s, const rtb_camera* cam, const rtb_params* p, uint32_t op,
                   const uint32_t* in, uint32_t n, uint32_t in_stride, uint32_t* out, uint32_t out_stride) {
  if (!c || !in || !out || !n || !in_stride || !out_stride) return set_err(RTB_ERR_INVALID, "bad argument");
  if (s && !s->committed) return set_err(RTB_ERR_STATE, "scene not committed (call rtb_scene_commit)");
  if (op == RTB_KAT_CAMERA_RAY && (!cam || !p || p->width < 2 || p->height < 2)) return set_err(RTB_ERR_INVALID, "camera op needs cam and params");
  if (!s && (op == RTB_KAT_LIGHTS_PDF || op == RTB_KAT_LIGHTS_RANDOM || op == RTB_KAT_PERLIN_NOISE || op == RTB_KAT_PERLIN_TURB ||
             op == RTB_KAT_MEDIA || op == RTB_KAT_TEXTURE || op == RTB_KAT_EXACT))
    return set_err(RTB_ERR_INVALID, "this op reads the scene's tables");
  CU(cudaSetDevice(c->device));
  DevBuf<uint32_t> d_in, d_out;
  CU(d_in.upload(in, (size_t)n * in_stride));
  CU(d_out.resize((size_t)n * out_stride));
  CU(cudaMemsetAsync(d_out.p, 0, (size_t)n * out_stride * 4, 0));
  DevScene dev;
  if (s) dev = s->dev;
  else { std::memset(&dev, 0, sizeof(dev)); dev.prmt_magic = 0x43000000u; }
  DevCamera dcam;
  DevCameraF64 dcam64;
  std::memset(&dcam, 0, sizeof(dcam));
  if (cam) camera_basis(*cam, dcam, dcam64);
  DevParams prm;
  std::memset(&prm, 0, sizeof(prm));
  if (p) {
    prm.width = p->width; prm.height = p->height; prm.seed = p->seed;
    if (p->width > 1) prm.inv_wm1 = (float)(1.0 / (double)(p->width - 1));
    if (p->height > 1) prm.inv_hm1 = (float)(1.0 / (double)(p->height - 1));
  }
  launch_kat(dev, dcam, prm, op, d_in.p, n, in_stride, d_out.p, out_stride, 0);
  CU(cudaMemcpy(out, d_out.p, (size_t)n * out_stride * 4, cudaMemcpyDeviceToHost));
  CU(cudaGetLastError());
  return RTB_OK;
}

int rtb_debug_check_failures(rtb_context* c, uint32_t* out8) {
  if (!c || !out8) return set_err(RTB_ERR_INVALID, "NULL argument");
  CU(cudaSetDevice(c->device));
  CU(cudaDeviceSynchronize());
  unsigned int v[8];
  const int e = read_check_failures(v);
  if (e != 0) return set_err(RTB_ERR_CUDA, cudaGetErrorString((cudaError_t)e));
  for (int i = 0; i < 8; ++i) out8[i] = v[i];
  return RTB_OK;
}

int rtb_measure_bandwidth(rtb_context* c, uint32_t kind, uint32_t repeats, double* gbs) {
  if (!c || !gbs || kind > RTB_BW_SHARED_READ) return set_err(RTB_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  if (repeats == 0) repeats = 5;
  const uint32_t grid = (uint32_t)c->prop.multiProcessorCount * 8u;
  DevBuf<uint4> sink, buf;
  CU(sink.resize(1));
  double bytes = 0.0;
  uint32_t reps = 1;
  size_t n_vec = 0;
  if (kind == RTB_BW_SHARED_READ) {
    reps = 1u << 16;
    bytes = (double)grid * 256.0 * reps * 16.0;
  } else {
    const size_t sz = kind == RTB_BW_L2_READ ? ((size_t)48 << 20) : ((size_t)2 << 30);
    n_vec = sz / 16;
    CU(buf.resize(n_vec));
    CU(cudaMemsetAsync(buf.p, 1, sz, 0));
    reps = kind == RTB_BW_L2_READ ? 64u : 2u;
    bytes = (double)sz * reps;
  }
  double best = 0.0;
  for (uint32_t r = 0; r < repeats + 1; ++r) {  // first launch = warm-up (fills L2)
    CU(cudaEventRecord(c->ev0, 0));
    if (kind == RTB_BW_SHARED_READ) launch_bw_shared(reps, sink.p, grid, 0);
    else launch_bw_global(buf.p, n_vec, reps, sink.p, grid, 0);
    CU(cudaEventRecord(c->ev1, 0));
    CU(cudaEventSynchronize(c->ev1));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    if (r > 0 && ms > 0.f) best = std::max(best, bytes / (ms * 1e-3) / 1e9);
  }
  CU(cudaGetLastError());
  *gbs = best;
  return RTB_OK;
}

int rtb_trace_rays(rtb_context* c, rtb_scene* s, const float* org, const float* dir, const float* time, uint32_t n,
                   uint32_t* id_out, float* t_out, rtb_stats* stats) {
  if (!c || !s || !org || !dir || !id_out || !t_out) return set_err(RTB_ERR_INVALID, "NULL argument");
  if (!s->committed) return set_err(RTB_ERR_STATE, "scene not committed (call rtb_scene_commit)");
  if (n == 0) return RTB_OK;
  CU(cudaSetDevice(c->device));
  CU(c->p_org.upload(org, (size_t)n * 3));
  CU(c->p_dir.upload(dir, (size_t)n * 3));
  CU(c->p_time.resize(n));
  if (time) CU(cudaMemcpyAsync(c->p_time.p, time, n * sizeof(float), cudaMemcpyHostToDevice, 0));
  else CU(cudaMemsetAsync(c->p_time.p, 0, n * sizeof(float), 0));
  return run_probe(c, s, n, id_out, t_out, stats);
}

}  // extern "C"
