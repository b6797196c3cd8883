/* rtb200.h — C ABI of the B200-native render path.
 *
 * This is the drop-in boundary for ONE hot path of dps/rust-raytracer: the timed
 * region of `pub fn render(filename, scene)` (reference raytracer/src/raytracer.rs:250-266,
 * precisely lines 259-263: the rayon `into_par_iter().for_each(render_line)` over row bands).
 * The reference has no FFI; the contract of that region is
 *     "given an immutable parsed scene, fill a caller-owned w*h*3 RGB8 row-major buffer, top row first".
 * A Rust maintainer binds these entry points with an `extern "C"` block and calls
 * rtb200_render_rgb8() in place of raytracer.rs:259-263 (see INTEGRATION.md).
 *
 * Conventions
 *   - every struct is POD, little-endian, caller-owned and read-only for the callee;
 *   - the callee copies what it needs before returning; no callee allocation escapes
 *     except opaque handles released with the matching *_release call;
 *   - every function returns 0 on success, a negative rt_status otherwise, and
 *     rtb200_last_error() then returns a thread-local message (the reference panics instead); no C++
 *     exception leaves the library (host out-of-memory while building the hierarchy is RT_ERR_OOM);
 *   - calls are blocking unless stated otherwise. Thread safety: every device has its own execution context guarded
 *     by a mutex, so two host threads may render on two DIFFERENT devices concurrently; calls that use the same
 *     device are serialised. A scene handle must not be used from two threads at once. The caller's current CUDA
 *     device is restored before every entry point returns;
 *   - there is NO CPU fallback: without a CUDA device / the sm_100a kernels every render call fails.
 */
#ifndef RTB200_H
#define RTB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTB200_ABI_VERSION 2   /* 2: rt_image.bytes, rt_stats.nodes/gpus_used, multi-GPU entry point, BVH diagnostics, RT_VARIANT_LANES retired */

/* ---- scene records (reference types flattened) --------------------------------------------- */

/* Point3D {x,y,z: f64} — raytracer/src/point3d.rs:10-15 */
typedef struct { double x, y, z; } rt_vec3;

/* The four computed fields of Camera that get_ray uses — raytracer/src/camera.rs:12-21,79-84.
 * Fill with rtb200_camera_from_params() (= Camera::new, camera.rs:45-77). */
typedef struct { rt_vec3 origin, lower_left_corner, horizontal, vertical; } rt_camera;

/* CameraParams — raytracer/src/camera.rs:29-36 (the JSON form of the camera) */
typedef struct { rt_vec3 look_from, look_at, vup; double vfov_deg, aspect; } rt_camera_params;

/* Material variants — raytracer/src/materials.rs:35-42 */
enum rt_material_kind {
    RT_LAMBERTIAN = 0, /* materials.rs:73-95   albedo                              */
    RT_METAL      = 1, /* materials.rs:99-129  albedo, param = fuzz                */
    RT_GLASS      = 2, /* materials.rs:132-199 param = index_of_refraction         */
    RT_TEXTURE    = 3, /* materials.rs:203-267 texture index, param = h_offset     */
    RT_LIGHT      = 4  /* materials.rs:57-69                                       */
};

/* Sphere {center, radius, material} — raytracer/src/sphere.rs:18-23. radius may be negative
 * (hollow glass shell, data/test_scene.json:137). List ORDER is semantic: hit_world keeps the
 * first sphere on equal t (raytracer.rs:52-56) and lights are visited in list order (raytracer.rs:103). */
typedef struct {
    rt_vec3  center;
    double   radius;
    uint32_t kind;        /* enum rt_material_kind */
    float    albedo[3];   /* Srgb<f32>; ignored for Glass/Light; ignored for Texture (materials.rs:264) */
    double   param;       /* fuzz | index_of_refraction | h_offset */
    int32_t  texture;     /* index into rt_scene.textures for RT_TEXTURE, else -1 */
    int32_t  reserved;
} rt_sphere;

/* Decoded RGB8 image, row-major, 3 B/texel. For Texture materials width/height are the values
 * written in the JSON, NOT the decoded file's (materials.rs:208-209 with loader result .0 only, :32). */
typedef struct {
    const uint8_t* rgb8;
    uint64_t width, height;
    uint64_t bytes;       /* size of the buffer rgb8 points to; the callee reads width*height*3 bytes and rejects bytes < that */
} rt_image;

/* Sky — raytracer/src/config.rs:22-28 and the miss branch raytracer.rs:134-163 */
enum rt_sky_mode { RT_SKY_NONE = 0 /* black */, RT_SKY_GRADIENT = 1, RT_SKY_TEXTURE = 2 };
typedef struct { uint32_t mode; uint32_t reserved; rt_image tex; } rt_sky;

/* Config — raytracer/src/config.rs:66-75, plus the seed (the reference draws from an OS-seeded
 * thread_rng and is not reproducible; see DESIGN.md "RNG contract"). */
typedef struct {
    uint32_t width, height, samples_per_pixel, max_depth;
    rt_camera camera;
    rt_sky    sky;
    const rt_sphere* spheres;  uint64_t n_spheres;
    const rt_image*  textures; uint64_t n_textures;
    uint64_t seed;
} rt_scene;

/* ---- execution options and results ---------------------------------------------------------- */

enum rt_trace_variant {
    RT_VARIANT_AUTO      = 0,
    RT_VARIANT_FILTERED  = 1, /* CTA-wavefront kernel: warp-cooperative traversal of an 8-wide BVH with conservative f32 tests + exact f64 confirmation (default) */
    RT_VARIANT_EXACT_F64 = 2, /* every sphere tested in f64 (validation of the conservative tests) */
    RT_VARIANT_RETIRED_LANES = 3, /* ABI 1's lane-autonomous kernel; retired: RT_ERR_UNSUPPORTED */
    RT_VARIANT_BRUTE_FORCE = 4 /* CTA-wavefront kernel scanning every sphere in list order (no hierarchy), like the reference's hit_world */
};

/* Which rows this call renders. Row-band b (band_rows consecutive rows) belongs to shard
 * (b mod world). world=1 renders everything. Output buffers of a shard call are COMPACT: the
 * shard's rows in increasing y, see rtb200_shard_rows(). */
typedef struct {
    int32_t  device;      /* CUDA ordinal; -1 = current device */
    int32_t  rank, world; /* shard of the image rendered by this call */
    uint32_t band_rows;   /* rows per interleaved band; 0 = default (1) */
    uint32_t variant;     /* enum rt_trace_variant */
    uint32_t flags;       /* reserved, must be 0 */
    uint64_t sample_buffer_bytes; /* cap for the per-sample radiance staging buffer; 0 = default */
} rt_options;

typedef struct {
    uint64_t rays;          /* hit_world invocations (primary + scattered + shadow), raytracer.rs:83 */
    uint64_t samples;       /* camera samples traced */
    uint64_t candidates;    /* f64-confirmed sphere tests (diagnostic) */
    double   device_ms;     /* CUDA-event time of all kernels of this call on the launching stream */
    double   trace_ms;      /* the trace kernel(s) alone */
    double   wall_ms;       /* host wall time of the call, copies included */
    uint32_t kernel_launches;
    uint32_t batches;
    uint64_t h2d_bytes, d2h_bytes;
    uint64_t clusters;      /* BVH leaves visited (diagnostic) */
    uint64_t frames;        /* frames covered by device_ms / trace_ms / kernel_launches (1 for the blocking calls) */
    uint64_t nodes;         /* BVH nodes visited (diagnostic) */
    int32_t  gpus_used;     /* devices that rendered this frame */
    int32_t  reserved;
} rt_stats;

/* The trace kernel a scene handle launches (cudaFuncGetAttributes + the launch geometry chosen at upload). */
typedef struct {
    int32_t  registers, local_bytes;       /* per thread */
    uint32_t smem_bytes, grid, block, ctas_per_sm;
    uint32_t smem_mask;                    /* bit0 hierarchy, bit1 exact geometry, bit2 materials staged into shared memory */
    uint32_t bvh_nodes, bvh_leaves, bvh_depth;
    uint32_t pool_slots;                   /* ray slots per CTA */
    char     name[96];
} rt_kernel_info;

enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID = -1,     /* bad argument / inconsistent scene */
    RT_ERR_NO_DEVICE = -2,   /* no CUDA device or not sm_100 */
    RT_ERR_CUDA = -3,        /* CUDA runtime failure (message has the detail) */
    RT_ERR_UNSUPPORTED = -4, /* scene needs a feature this build lacks */
    RT_ERR_OOM = -5
};

/* ---- entry points ---------------------------------------------------------------------------- */

int rtb200_abi_version(void);
const char* rtb200_last_error(void);

/* Camera::new — camera.rs:45-77 (host, f64, once per frame). */
int rtb200_camera_from_params(const rt_camera_params* p, rt_camera* out);

/* Number of rows of `height` that shard `rank` of `world` owns with the given band size. */
uint32_t rtb200_shard_rows(uint32_t height, int32_t rank, int32_t world, uint32_t band_rows);

/* Replaces raytracer.rs:259-263 (+ the Vec<u8> it fills, :254): host scene in, host RGB8 out.
 * Uploads the scene, renders on one GPU (opts==NULL) or the shard opts describes, copies back.
 * out_rgb8: width*height*3 bytes (or shard_rows*width*3 when opts->world > 1). */
int rtb200_render_rgb8(const rt_scene* scene, const rt_options* opts, uint8_t* out_rgb8, rt_stats* stats);

/* The same frame on n_gpus devices of this process (0 = all; devices opts->device.. when opts->device >= 0, else 0..):
 * the reference's row bands (raytracer.rs:254-262) are dealt round-robin to the devices (band b -> device b mod G), the
 * scene is replicated, every device renders its shard, the shards are copied peer-to-peer into the frame on the first
 * device and ONE device->host copy fills out_rgb8 (width*height*3 bytes). Bit-identical to rtb200_render_rgb8.
 * opts->rank/world must be 0/1 (or opts NULL). */
int rtb200_device_count(void);
int rtb200_render_rgb8_multi(const rt_scene* scene, const rt_options* opts, int32_t n_gpus, uint8_t* out_rgb8, rt_stats* stats);

/* Same path, but returns the per-pixel mean radiance BEFORE sqrt/quantisation (raytracer.rs:207-212
 * computes sqrt(scale*sum)); used by parity tests. out_rgb: width*height*3 floats (or the shard's). */
int rtb200_render_linear_f32(const rt_scene* scene, const rt_options* opts, float* out_rgb, rt_stats* stats);

/* Resident form (scene stays in HBM between frames; output stays on the device). */
typedef struct rtb200_scene_t* rtb200_scene_handle;
int rtb200_scene_upload(const rt_scene* scene, const rt_options* opts, rtb200_scene_handle* out);
/* dev_rgb8 / dev_linear_f32 are DEVICE pointers (either may be NULL); stream is a cudaStream_t, or NULL for the library's
 * own non-blocking stream (pass cudaStreamLegacy / cudaStreamPerThread explicitly to order against the default stream). */
int rtb200_render_device(rtb200_scene_handle h, void* dev_rgb8, void* dev_linear_f32, void* stream, rt_stats* stats);
/* Non-blocking form for frame loops: enqueue a frame on `stream` and return; rtb200_render_device_wait() blocks until the
 * frames enqueued so far are done and returns statistics. Successive frames alternate between two sets of work buffers, so a caller
 * that alternates two streams (and two output buffers) lets frame k+1 start while frame k drains its last paths; frames on the
 * same stream are ordered by it. One scene at a time may have asynchronous frames in flight on a device. */
int rtb200_render_device_async(rtb200_scene_handle h, void* dev_rgb8, void* dev_linear_f32, void* stream);
int rtb200_render_device_wait(rtb200_scene_handle h, rt_stats* stats);
int rtb200_scene_release(rtb200_scene_handle h);
int rtb200_scene_kernel_info(rtb200_scene_handle h, rt_kernel_info* out);

/* Per-frame edits of a resident scene (animation, interactive camera) without a new upload. NULL fields are kept.
 *   - camera and seed change host-side state only;
 *   - spheres: exactly the uploaded count, same order (order is semantic). Centre, radius, material kind, albedo, param and
 *     texture index may change. The host validates every new sphere with the rules of rtb200_scene_upload, copies the array
 *     to the device once (64 B per sphere), and the device rebuilds what the closest-hit stage reads: exact geometry and
 *     materials (every variant), the flat records (RT_VARIANT_BRUTE_FORCE) and, for the hierarchy, the leaf records and the
 *     node boxes. The hierarchy's topology and recentring are those of the upload; boxes are recomputed with the builder's
 *     own formulas (refit), so the frame is bit-identical to a fresh upload of the edited scene, but the tree gets looser as
 *     spheres drift (rt_stats.nodes / clusters grow). Re-upload to rebuild it (DESIGN.md §4.6).
 *   - refused, with the handle unchanged: a different count (RT_ERR_INVALID); a Light at a different set of indices
 *     (RT_ERR_UNSUPPORTED: the kernel variant, light list and launch geometry were chosen from it); a sphere of the hierarchy
 *     that leaves the upload's recentred f32 frame, i.e. non-finite or max|c-g|+|r| >= 1e15 (RT_ERR_UNSUPPORTED: re-upload);
 *     spheres the upload put on the always-list may take any valid value. Also refused while asynchronous frames of the
 *     handle are pending (RT_ERR_INVALID: call rtb200_render_device_wait first; they read the same scene arrays).
 *   - every render enqueued after the call returns, on any stream, sees the edited scene. */
typedef struct {
    const rt_camera* camera;     /* NULL: keep */
    const uint64_t*  seed;       /* NULL: keep */
    const rt_sphere* spheres;    /* NULL: keep; else n_spheres == the uploaded count, same order */
    uint64_t         n_spheres;
} rt_scene_edit;
int rtb200_scene_update(rtb200_scene_handle h, const rt_scene_edit* e);
/* What the handle's closest-hit stage reads NOW, copied back from the device: the arrays and info[] of rtb200_debug_bvh.
 * The flat records exist only on RT_VARIANT_BRUTE_FORCE handles (info[6] = 0 otherwise); RT_VARIANT_EXACT_F64 handles
 * hold no hierarchy (info[0] = info[1] = 0). */
int rtb200_scene_debug_bvh(rtb200_scene_handle h, double recentre[3], uint32_t info[8], float* nodes, uint64_t cap_nodes,
                           float* leaf_rec, uint64_t cap_leaf_rec, uint32_t* leaf_id, uint64_t cap_leaf_id,
                           uint32_t* always, uint64_t cap_always, float* flat, uint64_t cap_flat);

/* load_texture_image — materials.rs:213-219, config.rs:36-47: decode a baseline JPEG file to RGB8 (host-side scene staging
 * helper for hosts without their own decoder; the reference uses the jpeg-decoder crate). *out_rgb8 is released with rtb200_free(). */
int  rtb200_decode_jpeg_file(const char* path, uint8_t** out_rgb8, uint64_t* width, uint64_t* height);
void rtb200_free(void* p);

/* Diagnostic, host only (no GPU needed): what the closest-hit stage of hit_world (raytracer.rs:44-59) would read for `scene`:
 * recentring offset; the 8-wide BVH nodes (floats_per_node floats each: lo_x[8] lo_y[8] lo_z[8] hi_x[8] hi_y[8] hi_z[8]
 * child[8], child = 0xffffffff empty | 0x80000000+leaf | node); the leaves (leaf_size pair-packed sphere records
 * {cx0,cx1,cy0,cy1},{cz0,cz1,nk0,nk1} + slot -> sphere index, 0xffffffff = padding); the spheres tested for every ray; the
 * flat records of RT_VARIANT_BRUTE_FORCE. info = {n_nodes, n_leaves, depth, leaf_size, n_always, floats_per_node, flat_pairs, 0}.
 * Arrays are filled up to their capacities (elements). */
int rtb200_debug_bvh(const rt_scene* scene, double recentre[3], uint32_t info[8], float* nodes, uint64_t cap_nodes,
                     float* leaf_rec, uint64_t cap_leaf_rec, uint32_t* leaf_id, uint64_t cap_leaf_id,
                     uint32_t* always, uint64_t cap_always, float* flat, uint64_t cap_flat);

/* Device-function probes: run the kernel's own device routines on one thread and return the result,
 * so the reference's known-answer tests can be asserted against the GPU code itself.
 *   sphere.rs:81-88, materials.rs:157-174, raytracer.rs:167-189, camera.rs:105-122 */
int rtb200_probe_sphere_hit(const rt_vec3* center, double radius, const rt_vec3* origin, const rt_vec3* dir,
                            double t_min, double t_max, int32_t* hit, double* t, rt_vec3* point, rt_vec3* normal,
                            int32_t* front_face);
int rtb200_probe_refract(const rt_vec3* uv, const rt_vec3* n, double etai_over_etat, rt_vec3* out);
int rtb200_probe_reflectance(double cosine, double ref_idx, double* out);
int rtb200_probe_sky(const rt_vec3* dir, uint32_t sky_mode, float out_rgb[3]);
int rtb200_probe_get_ray(const rt_camera* cam, double u, double v, rt_vec3* origin, rt_vec3* dir);
/* n uniform draws of the per-(pixel,sample) stream: kind 0 = gen::<f64>() in [0,1), 1 = gen_range(-1.0..1.0) */
int rtb200_probe_rng(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t kind, uint32_t n, double* out);
/* u_v_from_sphere_hit_point (sphere.rs:35-43) of n vectors hp = hit point - centre (3 doubles each); out = n {u, v} pairs */
int rtb200_probe_sphere_uv(const double* hp_xyz, uint32_t n, double* out_uv);
/* u8 quantisation of raytracer.rs:207-213 for n linear means */
int rtb200_probe_quantise(const float* mean_linear, uint32_t n, uint8_t* out);

#ifdef __cplusplus
}
#endif
#endif /* RTB200_H */
