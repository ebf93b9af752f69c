// rtb_launch.hpp — host-visible launch interface of rtb_kernels.cu
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#ifndef RTB_EXTEND_THREADS
#define RTB_EXTEND_THREADS 256
#endif
#define RTB_SHADE_THREADS 256
#define RTB_SPHERE_STAGE_BYTES (16u * 1024u)  /* shared-memory cap of the sphere records staged beside a fully staged tree */
#ifndef RTB_SHADE_MIN_BLOCKS
#define RTB_SHADE_MIN_BLOCKS 3
#endif

#define RTB_OPT_PROBE 1u  /* DevParams::opt bit: parity probe (media sampled at xi = 0.5 instead of the path's stream) */
/* DevParams::opt bits 8-13: leaf-test parking threshold of the extend kernels (lanes that must have parked primitives before
   the warp drains them together); 0 = test leaves inline at the node visit */
#define RTB_OPT_OCTANT_SORT 2u  /* DevParams::opt bit: extend orders each chunk's rays by (kind, direction octant) */
#define RTB_OPT_PARK_SHIFT 8
#define RTB_OPT_PARK_MASK 63u

namespace rtb {

struct DevScene;
struct DevPool;
struct DevParams;
struct DevCamera;
struct DevCounters;

struct DevCameraF64 {  // camera.rs:6-17 in f64, for the parity probe's primary rays
  double origin[3], llc[3], horizontal[3], vertical[3];
  double time0;
};

enum ExtendMode : uint32_t { EXTEND_STATIC = 0, EXTEND_DYNAMIC = 1, EXTEND_WQ = 2 };
struct LaunchCfg {
  uint32_t mode = EXTEND_STATIC;  // which extend scheduler (configure_launch)
  uint32_t extend_grid = 0, shade_grid = 0, fixup_grid = 0, extend_smem = 0, n_snodes = 0;
  bool dynamic_fetch = false;
  bool all_staged = false;  // every BVH node fits the shared-memory stage: the kernel without a global node path is used
  uint32_t sphere_smem = 0;  // > 0: ... and the sphere records (these bytes) are staged after the nodes by the production
                             // static kernel; added to extend_smem for that kernel's launch only
  // slots that give every resident shade warp exactly one chunk: pools are sized in multiples of this
  uint32_t pool_unit = 0;
};

// max_depth: levels of the tree (the warp-queue kernel keeps fixed-depth stacks in shared memory)
// n_spheres: records of the sphere array (RTB_SPHERE_STAGE_BYTES / 16 at most are staged with a fully staged tree)
int configure_launch(LaunchCfg& lc, uint32_t n_nodes, uint32_t max_depth, uint32_t n_spheres, int sm_count);
int read_check_failures(unsigned int* out8);  // RTB_CHECKED build: failed bounds assertions by kind; 0xFFFFFFFF otherwise
void launch_init_pool(const DevPool& pool, unsigned long long total_paths, cudaStream_t st);
void launch_generate(const LaunchCfg& lc, const DevPool& pool, const DevParams& prm, const DevCamera& cam, cudaStream_t st);
void launch_fixup(const LaunchCfg& lc, const DevScene& sc, const DevPool& pool, const DevParams& prm, cudaStream_t st);
void launch_rotate(const DevPool& pool, cudaStream_t st);
void launch_extend(const LaunchCfg& lc, const DevScene& sc, const DevPool& pool, const DevParams& prm, bool count,
                   cudaStream_t st);
void launch_shade(const LaunchCfg& lc, const DevScene& sc, const DevPool& pool, const DevParams& prm,
                  const DevCamera& cam, uint32_t present, cudaStream_t st);
void launch_finalize(const float4* accum, uint8_t* rgb, uint32_t npix, float inv_spp, cudaStream_t st);
void launch_probe_fill(const DevPool& pool, const float* org, const float* dir, const float* time, uint32_t n, cudaStream_t st);
void launch_probe_collect(const DevScene& sc, const DevPool& pool, uint32_t n, uint32_t* id_out, float* t_out, cudaStream_t st);
// denoiser guide buffers: slot i of `pool` starts path number first_path + i (i < n); the hit records of those slots are
// then summed as 8 floats per pixel into aov (2 float4 per pixel)
void launch_aov_fill(const DevPool& pool, const DevParams& prm, const DevCamera& cam, unsigned long long first_path,
                     uint32_t n, cudaStream_t st);
void launch_aov_collect(const DevScene& sc, const DevPool& pool, const DevParams& prm, float4* aov, uint32_t n,
                        cudaStream_t st);
void launch_primary_rays(const DevCameraF64& cam, uint32_t W, uint32_t H, float* org, float* dir, float* time,
                         cudaStream_t st);
void launch_bw_global(const uint4* p, size_t n_vec, uint32_t reps, uint4* sink, uint32_t grid, cudaStream_t st);
void launch_bw_shared(uint32_t reps, uint4* sink, uint32_t grid, cudaStream_t st);
void launch_kat(const DevScene& sc, const DevCamera& cam, const DevParams& prm, uint32_t op, const uint32_t* in, uint32_t n,
                uint32_t in_stride, uint32_t* out, uint32_t out_stride, cudaStream_t st);

}  // namespace rtb
