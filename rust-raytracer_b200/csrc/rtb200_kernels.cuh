// rtb200_kernels.cuh — parameter blocks and launch wrappers shared by the kernels and rtb200_api.cu
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rtb200.h"
#include "rtb200_device.cuh"

namespace rtk {

#ifndef RT_BLOCK
#define RT_BLOCK 256
#endif
constexpr int kBlock = RT_BLOCK;   // threads (= ray slots) per CTA of the trace kernel
#ifndef RT_LEAF_K
#define RT_LEAF_K 8
#endif
constexpr int kLeafK = RT_LEAF_K;  // sphere slots per BVH leaf            (= rtbvh::kLeafK)
constexpr int kNodeVec = 14;       // float4 per 8-wide BVH node (224 B)   (= rtbvh::kNodeFloats / 4)
// per-warp work lists of the closest-hit stage (entries: id << 5 | ray lane)
#ifndef RT_CAP_IN
#define RT_CAP_IN 192
#endif
#ifndef RT_CAP_LF
#define RT_CAP_LF 160
#endif
#ifndef RT_CAP_CD
#define RT_CAP_CD 96
#endif
constexpr int kCapIn = RT_CAP_IN;   // (ray, inner node) pairs: LIFO stack; 7*depth+8 entries are reserved for single-entry descents
constexpr int kCapLf = RT_CAP_LF;   // (ray, leaf) pairs
constexpr int kCapCd = RT_CAP_CD;   // (ray, sphere) pairs awaiting the exact f64 test

// 32-byte material record (device copy of the material half of rt_sphere)
struct DevMat { float r, g, b; uint32_t kind; double param; int32_t tex; int32_t pad; };
static_assert(sizeof(DevMat) == 32, "DevMat must be 32 bytes");

// One pending light test (raytracer.rs:99-114): the vertex it belongs to and the partial sum over the lights.
struct ShadowFrame {
    double px, py, pz;      // hit point = origin of the shadow rays and of the scattered ray
    double ndx, ndy, ndz;   // scattered direction (continuation of the main path)
    float ar, ag, ab;       // albedo of the vertex
    float sr, sg, sb;       // sum over lights of albedo * ray_color(light_ray, 2, 1)
    uint32_t li, code, is_light, pad;
};
static_assert(sizeof(ShadowFrame) == 88, "ShadowFrame layout");

enum TraceMode : uint32_t { MODE_TREE = 0, MODE_BRUTE = 1, MODE_EXACT = 2 };

struct TraceParams {
    // ---- scene, resident in HBM (built by rtbvh::build_records) ----
    const float4*   nodes;       // n_nodes * kNodeVec: lo_x[8] lo_y[8] lo_z[8] hi_x[8] hi_y[8] hi_z[8] child[8], f32 boxes rounded outwards
    const float4*   leaf_rec;    // n_leaves * kLeafK float4: kLeafK/2 pair-packed sphere records {cx0,cx1,cy0,cy1},{cz0,cz1,nk0,nk1}
    const uint32_t* leaf_id;     // n_leaves * kLeafK: slot -> ORIGINAL sphere index (0xffffffff = padding)
    const uint32_t* always;      // n_always sphere indices tested in f64 for every ray (not representable in the f32 frame)
    const float4*   filt;        // n_pairs * 2 float4: every sphere in list order, pair-packed (MODE_BRUTE)
    const double4*  geo;         // n: {cx,cy,cz,radius} exact f64
    const DevMat*   mat;         // n
    const rtd::DevTex* tex;      // n_tex
    uint32_t n, n_pairs, n_nodes, n_leaves, n_always, depth;
    uint32_t n_lights;
    uint32_t scene_in_smem;      // bit0: nodes + leaves (MODE_TREE) / flat records (MODE_BRUTE), bit1: geo, bit2: mat staged into shared memory
    double gx, gy, gz;           // recentring offset of the f32 frame
    float  er_coef;              // per-ray error coefficient of the sphere test (DESIGN.md "filter soundness")
    rt_camera cam;
    uint32_t width, height, spp, max_depth;
    uint32_t sky_mode;
    rtd::DevTex sky;
    uint32_t key0, key1;         // Philox key = seed
    // ---- work of this launch: samples [s0, s0+s_count) of every pixel of the shard ----
    uint32_t s0, s_count;
    uint32_t npix_local, rows_local;
    int32_t  rank, world;
    uint32_t band_rows;
    uint32_t total_work;         // npix_local * s_count
    unsigned int* work_counter;
    float4*  samplebuf;          // [s_count][npix_local] per-sample radiance (w = rays of the sample)
    uint32_t* stack;             // [max_depth][stack_stride] per-slot albedo codes (levels beyond the shared-memory part)
    uint32_t stack_stride;
    const uint32_t* lights;      // sphere indices of the Light spheres in list order (find_lights, raytracer.rs:220-229)
    ShadowFrame* frames;         // [max_shadow][stack_stride], only when n_lights > 0
    uint32_t max_shadow;         // nested light-test frames per path (a level nests with probability <= n_lights*0.1)
    float* lterm;                // [2 levels][3][stack_stride] light terms of the first two path levels
    unsigned long long* stat;    // per frame: [0]=rays [1]=f64 tests [2]=all-spheres fallbacks [3]=samples [4]=leaf visits [6]=node visits
                                 // [8..15] phase clocks (RT_PROFILE_PHASES)
    unsigned long long* err;     // per scene handle, accumulated over frames: [0]=shadow-frame-stack overflows [1]=traversal guard trips (must stay 0)
};

struct ResolveParams {
    const float4* samplebuf;
    float*   accum;        // [npix_local][3] running f32 sums in sample order
    uint32_t npix_local, s_count;
    uint32_t first, last;  // first batch zeroes accum, last batch writes outputs
    uint32_t spp;
    float*   out_linear;   // [npix_local][3] or null
    uint8_t* out_rgb8;     // [npix_local][3] or null
};

// On-device refit of a resident scene after a sphere edit (rtb200_scene_update, rtb200_refit.cu). The topology (child refs,
// leaf_id, always-list) and the recentring g are those of the upload; everything else is rebuilt from `sp`.
struct RefitParams {
    const rt_sphere* sp;         // n new spheres (device copy of the caller's array)
    uint32_t n, n_nodes, n_leaves;
    double gx, gy, gz;
    double4* geo;                // n
    DevMat*  mat;                // n
    float*   flat;               // n_pairs * 8, or null (only MODE_BRUTE handles hold flat records)
    float*   leaf_rec;           // n_leaves * kLeafK * 4
    const uint32_t* leaf_id;     // n_leaves * kLeafK
    float*   nodes;              // n_nodes * kNodeVec * 4: the boxes are rewritten, child[] is read
    uint32_t* slot_of;           // n: sphere -> leaf slot (0xffffffff: not in the hierarchy)
    uint32_t* parent;            // n_nodes: parent node (root: 0xffffffff)
    uint32_t* level;             // n_nodes: wide level, root = 1 (emit_wide's numbering)
    double*  box64;              // n_nodes * 8 * 6: exact f64 box of every child slot {lo xyz, hi xyz} before inflation
};

struct KernelInfo { int registers, max_threads, const_bytes, local_bytes; char name[96]; };

size_t wavefront_smem_bytes(const TraceParams& p, uint32_t mode, uint32_t smem_mask);
cudaError_t launch_wavefront(const TraceParams& p, uint32_t mode, int grid, size_t smem, int minb, cudaStream_t st);
int wavefront_max_ctas_per_sm(uint32_t mode, bool lights, size_t smem, int minb);
cudaError_t wavefront_info(uint32_t mode, bool lights, int minb, KernelInfo* out);
cudaError_t launch_resolve(const ResolveParams& p, cudaStream_t st);
// refit: maps once per handle (slot_of / parent / level), then per edit the sphere pass and one node pass per level, deepest first
cudaError_t launch_refit_maps(const RefitParams& p, cudaStream_t st);
cudaError_t launch_refit(const RefitParams& p, uint32_t depth, cudaStream_t st);

// single-thread probes of the device routines (known-answer tests)
cudaError_t probe_sphere_hit(const double* in /*12*/, double* out /*9*/, cudaStream_t st);
cudaError_t probe_refract(const double* in /*7*/, double* out /*3*/, cudaStream_t st);
cudaError_t probe_reflectance(const double* in /*2*/, double* out /*1*/, cudaStream_t st);
cudaError_t probe_sky(const double* in /*3*/, uint32_t mode, float* out /*3*/, cudaStream_t st);
cudaError_t probe_get_ray(const rt_camera* cam_dev, const double* in /*2*/, double* out /*6*/, cudaStream_t st);
cudaError_t probe_rng(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t kind, uint32_t n, double* out, cudaStream_t st);
cudaError_t probe_quantise(const float* in, uint32_t n, uint8_t* out, cudaStream_t st);
cudaError_t probe_sphere_uv(const double* in /*3n*/, uint32_t n, double* out /*2n*/, cudaStream_t st);

}  // namespace rtk
