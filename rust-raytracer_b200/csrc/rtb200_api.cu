// rtb200_api.cu — the C ABI of include/rtb200.h: scene staging into HBM, batch scheduling of the trace /
// resolve kernels, single- and multi-GPU frames, device<->host copies and error reporting. No CPU render path exists here.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "rtb200_bvh.hpp"
#include "rtb200_kernels.cuh"

using namespace rtk;

static_assert(sizeof(rtbvh::Mat32) == sizeof(DevMat), "host and device material records must agree");
static_assert(rtbvh::kLeafK == kLeafK && rtbvh::kNodeFloats == kNodeVec * 4, "host and device BVH layouts must agree");
static_assert(kCapIn >= 32 + 7 * rtbvh::kMaxDepth + 8, "the node stack must hold 32 roots plus a single-entry descent of the deepest tree (LIFO reserve, DESIGN.md 4.1)");

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) { g_last_error = msg; return code; }
int fail_cuda(cudaError_t e, const char* what) {
    g_last_error = std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
    return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? RT_ERR_NO_DEVICE
           : (e == cudaErrorMemoryAllocation ? RT_ERR_OOM : RT_ERR_CUDA);
}
#define CU(call)                                              \
    do {                                                      \
        cudaError_t e__ = (call);                             \
        if (e__ != cudaSuccess) return fail_cuda(e__, #call); \
    } while (0)

struct GrowBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaError_t e = cudaFree(p); if (e != cudaSuccess) return e; p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { cudaGetLastError(); e = cudaMalloc(&p, bytes); want = bytes; }
        if (e != cudaSuccess) return e;
        cap = want;
        return cudaSuccess;
    }
};
struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        cudaError_t e = cudaHostAlloc(&p, bytes + bytes / 8, cudaHostAllocDefault);
        if (e != cudaSuccess) return e;
        cap = bytes + bytes / 8;
        return cudaSuccess;
    }
};

// Per-device execution context: one stream, grow-only work buffers. `mu` serialises the calls that use the context, so two
// host threads may render on two DIFFERENT devices concurrently; calls on the same device take turns.
struct DeviceCtx {
    std::recursive_mutex mu;
    bool init = false;
    int device = -1;
    int sm_count = 0;
    size_t max_smem = 0;
    cudaStream_t stream = nullptr;
    // Two sets of per-frame work buffers: a frame loop that alternates two streams lets frame k+1 start tracing while frame k
    // drains its last paths and resolves (rtb200_render_device_async); blocking calls use set 0 only.
    struct WorkSet { GrowBuf samplebuf, accum, stack, small, frames, lterm; } ws[2];
    GrowBuf out_rgb8, out_lin, probe, frame;
    // scene arenas of released handles, kept for the next upload (a per-frame upload costs no cudaMalloc / cudaFree)
    struct Arena { void* p; size_t cap; };
    std::vector<Arena> arena_cache;
    std::vector<cudaEvent_t> event_pool;  // timing events of released handles (creating four events per one-shot render costs more than the upload)
    struct OccKey { uint32_t mode; bool lights; int minb; size_t smem; int occ; };
    std::vector<OccKey> occ_cache;        // cudaOccupancyMaxActiveBlocksPerMultiprocessor answers
    PinnedBuf staging;                    // host image of the arena being uploaded
    cudaEvent_t staging_free = nullptr;   // the last H2D copy out of `staging` has finished
};
DeviceCtx g_ctx[64];
std::mutex g_ctx_mu;

int get_ctx(int device, DeviceCtx** out) {
    if (device < 0) {
        cudaError_t e = cudaGetDevice(&device);
        if (e != cudaSuccess) return fail_cuda(e, "cudaGetDevice");
    }
    if (device >= 64) return fail(RT_ERR_INVALID, "device ordinal out of range");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) return fail_cuda(e, "cudaGetDeviceCount");
    if (device >= count) return fail(RT_ERR_NO_DEVICE, "no such CUDA device");
    CU(cudaSetDevice(device));
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    DeviceCtx& c = g_ctx[device];
    if (!c.init) {
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10) {
            char buf[160];
            snprintf(buf, sizeof buf, "device %d is sm_%d%d; this library carries sm_100a code only", device, prop.major, prop.minor);
            return fail(RT_ERR_NO_DEVICE, buf);
        }
        c.device = device;
        c.sm_count = prop.multiProcessorCount;
        c.max_smem = prop.sharedMemPerBlockOptin;
        CU(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&c.staging_free, cudaEventDisableTiming));
        c.init = true;
    }
    *out = &c;
    return RT_OK;
}

// RAII: restores the caller's current device (the ABI must not leave cudaSetDevice changed behind the caller's back)
struct DeviceRestore {
    int prev = -1;
    DeviceRestore() { if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; } }
    ~DeviceRestore() { if (prev >= 0) cudaSetDevice(prev); }
};

struct V3 { double x, y, z; };
inline V3 v3(const rt_vec3& a) { return V3{a.x, a.y, a.z}; }
inline V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
inline V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 operator*(V3 a, double s) { return V3{a.x * s, a.y * s, a.z * s}; }
inline double vlen(V3 a) { return std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }
inline V3 vunit(V3 a) { double l = vlen(a); return V3{a.x / l, a.y / l, a.z / l}; }
inline V3 vcross(V3 a, V3 b) { return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline rt_vec3 rv(V3 a) { return rt_vec3{a.x, a.y, a.z}; }

// No C++ exception may unwind through the C boundary (std::bad_alloc while building the hierarchy of a huge scene, ...).
template <typename F>
int guarded(F&& f) {
    try { return f(); }
    catch (const std::bad_alloc&) { return fail(RT_ERR_OOM, "host memory allocation failed"); }
    catch (const std::exception& e) { return fail(RT_ERR_INVALID, std::string("internal error: ") + e.what()); }
    catch (...) { return fail(RT_ERR_INVALID, "internal error: unknown exception"); }
}

uint32_t mode_of(uint32_t variant) {
    return variant == RT_VARIANT_EXACT_F64 ? MODE_EXACT : (variant == RT_VARIANT_BRUTE_FORCE ? MODE_BRUTE : MODE_TREE);
}

bool image_ok(const rt_image& im) {
    if (!im.rgb8 || im.width == 0 || im.height == 0) return false;
    if (im.width > (1ull << 20) || im.height > (1ull << 20)) return false;
    return im.width * im.height * 3ull <= im.bytes;   // the callee reads width*height*3 bytes: the buffer must hold them
}

// The per-sphere rules of a scene (rtb200_scene_upload and rtb200_scene_update); tex_ok(t): texture t passes image_ok.
template <typename TexOk>
int validate_sphere(const rt_sphere& sp, uint64_t n_textures, TexOk tex_ok) {
    if (sp.kind > RT_LIGHT) return fail(RT_ERR_INVALID, "unknown material kind");
    if (sp.kind == RT_TEXTURE) {
        if (sp.texture < 0 || (uint64_t)sp.texture >= n_textures) return fail(RT_ERR_INVALID, "texture index out of range");
        if (!tex_ok(sp.texture)) return fail(RT_ERR_INVALID, "texture image is empty or smaller than width*height*3 bytes (rt_image.bytes)");
    }
    return RT_OK;
}

}  // namespace

struct rtb200_scene_t {
    int device = -1;
    DeviceCtx* ctx = nullptr;
    TraceParams tp{};
    rt_options opts{};
    uint32_t mode = MODE_TREE;
    uint32_t slots_per_cta = kBlock;     // ray slots per CTA (one per thread)
    int minb = 3;
    int grid = 0;
    int ctas_per_sm = 0;
    size_t smem = 0;
    uint32_t spp_batch = 0;
    void* arena = nullptr;               // ONE device allocation holding every scene array (returned to the context's cache on release)
    size_t arena_cap = 0;
    unsigned long long* err = nullptr;   // device: [0] shadow-frame-stack overflows, [1] traversal guard trips; accumulated over frames, cleared by wait
    struct Upload { const void* src; size_t bytes; void** field; };
    std::vector<Upload> uploads;         // pending scene arrays (commit_uploads)
    std::vector<cudaEvent_t> ev;         // event ring of the frames in flight (per handle)
    cudaStream_t last_stream = nullptr;  // stream, work set, batch and launch count of the most recently enqueued frame
    int last_set = 0;
    cudaStream_t streams[2] = {nullptr, nullptr};   // distinct streams used by the pending frames
    int n_streams = 0;
    uint32_t frame_counter = 0;
    uint32_t last_batches = 0, last_launches = 0;
    uint32_t pending_frames = 0;
    uint64_t h2d_bytes = 0;
    // what rtb200_scene_update checks edits against (fixed at upload)
    std::vector<uint32_t> light_ids;     // Light spheres, list order
    std::vector<uint32_t> always_ids;    // spheres outside the hierarchy (MODE_TREE), increasing
    std::vector<uint8_t> tex_ok;         // per texture: holds width*height*3 bytes
    // refit state, allocated by the first sphere edit: ONE device allocation (sphere copy, maps, f64 slot boxes)
    void* refit = nullptr;
    RefitParams rp{};
    cudaEvent_t written = nullptr;       // the last edit's device work; renders on other streams wait for it
};

extern "C" {

int rtb200_abi_version(void) { return RTB200_ABI_VERSION; }
const char* rtb200_last_error(void) { return g_last_error.c_str(); }

int rtb200_device_count(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); return 0; }
    return count;
}

// Camera::new — camera.rs:45-77. Host, once per frame, f64, same operation order as the reference.
// (Compiled with -ffp-contract=off: see the Makefile.)
int rtb200_camera_from_params(const rt_camera_params* p, rt_camera* out) {
    if (!p || !out) return fail(RT_ERR_INVALID, "null argument");
    const double PI = 3.14159265358979323846264338327950288;
    double theta = p->vfov_deg * (PI / 180.0);
    double half_height = std::tan(theta / 2.0);
    double half_width = p->aspect * half_height;
    V3 look_from = v3(p->look_from), look_at = v3(p->look_at), vup = v3(p->vup);
    V3 w = vunit(look_from - look_at);
    V3 u = vunit(vcross(vup, w));
    V3 v = vcross(w, u);
    V3 origin = look_from;
    V3 llc = origin - (u * half_width) - (v * half_height) - w;
    V3 horizontal = u * 2.0 * half_width;
    V3 vertical = v * 2.0 * half_height;
    out->origin = rv(origin); out->lower_left_corner = rv(llc); out->horizontal = rv(horizontal); out->vertical = rv(vertical);
    return RT_OK;
}

uint32_t rtb200_shard_rows(uint32_t height, int32_t rank, int32_t world, uint32_t band_rows) {
    if (world <= 1) return height;
    if (band_rows == 0) band_rows = 1;
    const uint64_t bands = ((uint64_t)height + band_rows - 1) / band_rows;   // last band may be partial
    if ((uint64_t)rank >= bands) return 0;
    const uint64_t mine = (bands - 1 - (uint64_t)rank) / (uint64_t)world + 1;   // bands rank, rank+world, ...
    uint64_t rows = mine * band_rows;
    const uint64_t last = bands - 1;
    if (last % (uint64_t)world == (uint64_t)rank) rows -= bands * band_rows - height;   // the partial band is ours
    return (uint32_t)rows;
}

static int render_collect(rtb200_scene_handle h, rt_stats* stats);

// Diagnostic (host only, no GPU needed): the hierarchy rtb200_scene_upload would stage for `scene`.
// info = {n_nodes, n_leaves, depth, leaf_size, n_always, floats_per_node, n_pairs_flat, 0}; arrays are filled up to their capacities (elements).
int rtb200_debug_bvh(const rt_scene* s, double recentre[3], uint32_t info[8], float* nodes, uint64_t cap_nodes, float* leaf_rec,
                     uint64_t cap_leaf_rec, uint32_t* leaf_id, uint64_t cap_leaf_id, uint32_t* always, uint64_t cap_always,
                     float* flat, uint64_t cap_flat) {
  return guarded([&]() -> int {
    if (!s || !info) return fail(RT_ERR_INVALID, "null argument");
    if (s->n_spheres >= (1ull << 26)) return fail(RT_ERR_UNSUPPORTED, "2^26 or more spheres (list entries carry 27-bit ids)");
    if (s->n_spheres && !s->spheres) return fail(RT_ERR_INVALID, "spheres is null");
    rtbvh::Records R;
    rtbvh::build_records(s, true, R);
    if (recentre) { recentre[0] = R.g[0]; recentre[1] = R.g[1]; recentre[2] = R.g[2]; }
    info[0] = R.n_nodes; info[1] = R.n_leaves; info[2] = R.depth; info[3] = (uint32_t)rtbvh::kLeafK; info[4] = (uint32_t)R.always.size();
    info[5] = (uint32_t)rtbvh::kNodeFloats; info[6] = R.n_pairs; info[7] = 0;
    if (nodes) memcpy(nodes, R.nodes.data(), std::min<uint64_t>(cap_nodes, R.nodes.size()) * 4);
    if (leaf_rec) memcpy(leaf_rec, R.leaf_rec.data(), std::min<uint64_t>(cap_leaf_rec, R.leaf_rec.size()) * 4);
    if (leaf_id) memcpy(leaf_id, R.leaf_id.data(), std::min<uint64_t>(cap_leaf_id, R.leaf_id.size()) * 4);
    if (always) memcpy(always, R.always.data(), std::min<uint64_t>(cap_always, R.always.size()) * 4);
    if (flat) memcpy(flat, R.flat.data(), std::min<uint64_t>(cap_flat, R.flat.size()) * 4);
    return RT_OK;
  });
}

int rtb200_scene_release(rtb200_scene_handle h) {
    if (!h) return RT_OK;
    DeviceRestore restore;
    if (h->ctx) {
        std::lock_guard<std::recursive_mutex> lk(h->ctx->mu);
        cudaSetDevice(h->device);
        if (h->pending_frames) render_collect(h, nullptr);   // frames still in flight read the scene arrays
        else if (h->ctx->stream) cudaStreamSynchronize(h->ctx->stream);
        for (cudaEvent_t e : h->ev) h->ctx->event_pool.push_back(e);
        if (h->arena) {
            auto& cache = h->ctx->arena_cache;
            if (h->arena_cap <= (64u << 20) && cache.size() < 4) cache.push_back(DeviceCtx::Arena{h->arena, h->arena_cap});
            else cudaFree(h->arena);
        }
        if (h->refit) cudaFree(h->refit);
        if (h->written) cudaEventDestroy(h->written);
    }
    delete h;
    return RT_OK;
}

// Scene arrays are collected first and then placed in ONE device arena filled by ONE host->device copy from pinned
// staging memory; arenas of released scenes are reused. `field` is patched with the device address.
static void upload_array(rtb200_scene_t* h, const void* src, size_t bytes, void** field) {
    *field = nullptr;
    if (bytes == 0) bytes = 16;
    h->uploads.push_back(rtb200_scene_t::Upload{src, bytes, field});
}

static int commit_uploads(rtb200_scene_t* h) {
    DeviceCtx* ctx = h->ctx;
    size_t total = 0;
    for (auto& u : h->uploads) total += (u.bytes + 255) & ~(size_t)255;
    if (total == 0) total = 256;
    // smallest cached arena that is large enough, else a new allocation
    int pick = -1;
    for (int i = 0; i < (int)ctx->arena_cache.size(); ++i)
        if (ctx->arena_cache[i].cap >= total && (pick < 0 || ctx->arena_cache[i].cap < ctx->arena_cache[pick].cap)) pick = i;
    if (pick >= 0) {
        h->arena = ctx->arena_cache[pick].p; h->arena_cap = ctx->arena_cache[pick].cap;
        ctx->arena_cache.erase(ctx->arena_cache.begin() + pick);
    } else {
        size_t want = total + total / 4;
        cudaError_t e = cudaMalloc(&h->arena, want);
        if (e != cudaSuccess) { cudaGetLastError(); want = total; CU(cudaMalloc(&h->arena, want)); }
        h->arena_cap = want;
    }
    char* base = (char*)h->arena;
    size_t off = 0;
    for (auto& u : h->uploads) { *u.field = base + off; off += (u.bytes + 255) & ~(size_t)255; }   // addresses first: tables may hold them
    CU(cudaEventSynchronize(ctx->staging_free));   // the previous upload's copy has left the staging buffer
    CU(ctx->staging.ensure(total));
    off = 0;
    for (auto& u : h->uploads) {
        if (u.src) { memcpy((char*)ctx->staging.p + off, u.src, u.bytes); h->h2d_bytes += u.bytes; }
        else memset((char*)ctx->staging.p + off, 0, u.bytes);
        off += (u.bytes + 255) & ~(size_t)255;
    }
    CU(cudaMemcpyAsync(base, ctx->staging.p, off, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaEventRecord(ctx->staging_free, ctx->stream));
    h->uploads.clear();
    return RT_OK;
}

static int validate_scene(const rt_scene* s, uint32_t* n_lights_out) {
    if (s->width < 2 || s->height < 2) return fail(RT_ERR_INVALID, "width and height must be >= 2 (u,v divide by w-1, h-1: raytracer.rs:199-200)");
    if (s->samples_per_pixel == 0) return fail(RT_ERR_INVALID, "samples_per_pixel must be > 0");
    if ((uint64_t)s->width * s->height >= (1ull << 31)) return fail(RT_ERR_INVALID, "image too large");
    if (s->n_spheres >= (1ull << 26)) return fail(RT_ERR_UNSUPPORTED, "2^26 or more spheres (list entries carry 27-bit ids)");
    if (s->n_spheres && !s->spheres) return fail(RT_ERR_INVALID, "spheres is null");
    if (s->n_textures && !s->textures) return fail(RT_ERR_INVALID, "textures is null");
    uint32_t n_lights = 0;
    for (uint64_t i = 0; i < s->n_spheres; ++i) {
        const rt_sphere& sp = s->spheres[i];
        int rc = validate_sphere(sp, s->n_textures, [&](int32_t t) { return image_ok(s->textures[t]); });
        if (rc != RT_OK) return rc;
        if (sp.kind == RT_LIGHT) ++n_lights;
    }
    if (n_lights >= 10) return fail(RT_ERR_UNSUPPORTED, "10 or more lights: the reference's light recursion (raytracer.rs:99-114) does not terminate when n_lights * 0.1 >= 1");
    if (s->sky.mode > RT_SKY_TEXTURE) return fail(RT_ERR_INVALID, "unknown sky mode");
    if (s->sky.mode == RT_SKY_TEXTURE && !image_ok(s->sky.tex)) return fail(RT_ERR_INVALID, "sky texture is empty or smaller than width*height*3 bytes (rt_image.bytes)");
    *n_lights_out = n_lights;
    return RT_OK;
}

static int normalise_options(const rt_options* opts_in, rt_options* o) {
    memset(o, 0, sizeof *o);
    o->device = -1; o->rank = 0; o->world = 1; o->band_rows = 1; o->variant = RT_VARIANT_AUTO;
    if (opts_in) *o = *opts_in;
    if (o->world <= 0) o->world = 1;
    if (o->band_rows == 0) o->band_rows = 1;
    if (o->rank < 0 || o->rank >= o->world) return fail(RT_ERR_INVALID, "rank outside [0, world)");
    if (o->flags != 0) return fail(RT_ERR_INVALID, "flags must be 0");
    if (o->variant == RT_VARIANT_RETIRED_LANES) return fail(RT_ERR_UNSUPPORTED, "RT_VARIANT_LANES was retired in ABI 2");
    if (o->variant > RT_VARIANT_BRUTE_FORCE) return fail(RT_ERR_INVALID, "unknown variant");
    return RT_OK;
}

// `R` holds the host-side records (built once; the multi-GPU entry point shares them between its devices).
static int scene_upload_records(const rt_scene* s, const rt_options& opts, uint32_t n_lights, const rtbvh::Records& R, rtb200_scene_handle* out) {
    *out = nullptr;
    DeviceCtx* ctx = nullptr;
    int rc = get_ctx(opts.device, &ctx);
    if (rc != RT_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    if (R.depth > (uint32_t)rtbvh::kMaxDepth) return fail(RT_ERR_UNSUPPORTED, "hierarchy deeper than the traversal stack reserve");

    rtb200_scene_t* h = new rtb200_scene_t();
    struct Guard { rtb200_scene_t* h; bool ok = false; ~Guard() { if (!ok) rtb200_scene_release(h); } } guard{h};
    h->device = ctx->device; h->ctx = ctx; h->opts = opts;
    h->mode = mode_of(opts.variant);
    const uint32_t n = (uint32_t)s->n_spheres;

    TraceParams& tp = h->tp;
    tp.n = n; tp.n_pairs = R.n_pairs; tp.n_nodes = R.n_nodes; tp.n_leaves = R.n_leaves; tp.n_always = (uint32_t)R.always.size();
    tp.depth = R.depth; tp.n_lights = n_lights;
    upload_array(h, R.nodes.data(), R.nodes.size() * 4, (void**)&tp.nodes);
    upload_array(h, R.leaf_rec.data(), R.leaf_rec.size() * 4, (void**)&tp.leaf_rec);
    upload_array(h, R.leaf_id.data(), R.leaf_id.size() * 4, (void**)&tp.leaf_id);
    upload_array(h, R.always.data(), R.always.size() * 4, (void**)&tp.always);
    if (h->mode == MODE_BRUTE) upload_array(h, R.flat.data(), R.flat.size() * 4, (void**)&tp.filt);
    upload_array(h, R.geo.data(), R.geo.size() * 8, (void**)&tp.geo);
    upload_array(h, R.mat.data(), R.mat.size() * sizeof(DevMat), (void**)&tp.mat);

    std::vector<rtd::DevTex> texs(std::max<uint64_t>(s->n_textures, 1));
    for (uint64_t t = 0; t < s->n_textures; ++t) {
        const rt_image& im = s->textures[t];
        texs[t].rgb8 = nullptr; texs[t].width = im.width; texs[t].height = im.height;
        if (im.rgb8 && im.width && im.height && im.width * im.height * 3ull <= im.bytes)
            upload_array(h, im.rgb8, im.width * im.height * 3, (void**)&texs[t].rgb8);
    }
    upload_array(h, texs.data(), texs.size() * sizeof(rtd::DevTex), (void**)&tp.tex);
    tp.sky_mode = s->sky.mode;
    tp.sky.rgb8 = nullptr; tp.sky.width = 0; tp.sky.height = 0;
    if (s->sky.mode == RT_SKY_TEXTURE) {
        upload_array(h, s->sky.tex.rgb8, s->sky.tex.width * s->sky.tex.height * 3, (void**)&tp.sky.rgb8);
        tp.sky.width = s->sky.tex.width; tp.sky.height = s->sky.tex.height;
    }
    std::vector<uint32_t> lights;
    for (uint32_t i = 0; i < n; ++i) if (s->spheres[i].kind == RT_LIGHT) lights.push_back(i);
    h->light_ids = lights;
    h->always_ids = R.always;
    h->tex_ok.resize(s->n_textures);
    for (uint64_t t = 0; t < s->n_textures; ++t) h->tex_ok[t] = image_ok(s->textures[t]);
    lights.push_back(0);
    upload_array(h, lights.data(), lights.size() * 4, (void**)&tp.lights);
    upload_array(h, nullptr, 16, (void**)&h->err);   // zero-filled error counters
    tp.err = nullptr;                                // patched after commit
    tp.gx = R.g[0]; tp.gy = R.g[1]; tp.gz = R.g[2];
    tp.er_coef = 1.0f - (float)(96.0 * rtbvh::kU);
    tp.cam = s->camera;
    tp.width = s->width; tp.height = s->height; tp.spp = s->samples_per_pixel; tp.max_depth = s->max_depth;
    tp.key0 = (uint32_t)s->seed; tp.key1 = (uint32_t)(s->seed >> 32);
    tp.rank = opts.rank; tp.world = opts.world; tp.band_rows = opts.band_rows;
    tp.rows_local = rtb200_shard_rows(s->height, opts.rank, opts.world, opts.band_rows);
    tp.npix_local = tp.rows_local * s->width;

    // ---- launch geometry: persistent grid = SMs x resident CTAs ----
    // RTB200_WF_SMEM=<mask> (bit0 hierarchy / flat records, bit1 geo, bit2 mat in shared memory) and RTB200_WF_MINB=<2|3|4>
    // pin the tuning knobs for experiments.
    const char* es = getenv("RTB200_WF_SMEM");
    {
        // What could be staged into shared memory next to the ray pool: the hierarchy, exact geometry, materials. Measured in
        // round 2 (DESIGN.md §4.5): for scenes this small a larger L1 beats the staging, so "nothing staged" is tried first.
        const char* eb = getenv("RTB200_WF_MINB");
        const uint32_t masks[] = {0u, 7u, 3u, 1u};   // measured (round 2): a larger L1 beats staging the small scenes' records
        bool found = false;
        for (int minb : {4, 3, 2}) {
            if (minb == 4 && !(eb && atoi(eb) == 4)) continue;   // the 64-register build: only on request
            if (eb && atoi(eb) != minb) continue;
            for (int need : {std::max(1, minb * 256 / kBlock), 1}) {   // CTAs per SM this register budget is built for
                for (uint32_t mask : masks) {
                    if (found) break;
                    if (es && (uint32_t)atoi(es) != mask) continue;
                    if (h->mode == MODE_EXACT && (mask & 1u)) continue;
                    size_t sm = wavefront_smem_bytes(tp, h->mode, mask);
                    if (sm > ctx->max_smem) continue;
                    int occ = -1;
                    for (auto& k : ctx->occ_cache) if (k.mode == h->mode && k.lights == (n_lights > 0) && k.minb == minb && k.smem == sm) occ = k.occ;
                    if (occ < 0) {
                        occ = wavefront_max_ctas_per_sm(h->mode, n_lights > 0, sm, minb);
                        ctx->occ_cache.push_back(DeviceCtx::OccKey{h->mode, n_lights > 0, minb, sm, occ});
                    }
                    if (occ < need || occ <= 0) continue;
                    h->minb = minb; h->smem = sm; tp.scene_in_smem = mask; h->ctas_per_sm = occ; h->grid = ctx->sm_count * occ;
                    found = true;
                }
                if (found || minb >= 3) break;   // the 80 / 64-register builds are only worth it at full residency
            }
            if (found) break;
        }
        if (!found) return fail(RT_ERR_UNSUPPORTED, "no launch configuration fits shared memory");
        h->slots_per_cta = kBlock;
    }

    // ---- per-sample staging: samples per batch bounded by the buffer cap ----
    uint64_t cap = opts.sample_buffer_bytes ? opts.sample_buffer_bytes : (1ull << 30);
    uint64_t per_spp = (uint64_t)std::max<uint32_t>(tp.npix_local, 1) * 16ull;
    uint64_t spb = std::max<uint64_t>(1, cap / per_spp);
    spb = std::min<uint64_t>(spb, s->samples_per_pixel);
    while (spb > 1 && spb * tp.npix_local >= (1ull << 31)) spb /= 2;
    h->spp_batch = (uint32_t)spb;

    if ((rc = commit_uploads(h)) != RT_OK) return rc;
    h->tp.err = h->err;
    guard.ok = true;
    *out = h;
    return RT_OK;
}

int rtb200_scene_upload(const rt_scene* s, const rt_options* opts_in, rtb200_scene_handle* out) {
  return guarded([&]() -> int {
    if (!s || !out) return fail(RT_ERR_INVALID, "null argument");
    *out = nullptr;
    rt_options opts;
    int rc = normalise_options(opts_in, &opts);
    if (rc != RT_OK) return rc;
    uint32_t n_lights = 0;
    if ((rc = validate_scene(s, &n_lights)) != RT_OK) return rc;
    DeviceRestore restore;
    rtbvh::Records R;
    rtbvh::build_records(s, mode_of(opts.variant) == MODE_TREE, R);
    return scene_upload_records(s, opts, n_lights, R, out);
  });
}

int rtb200_scene_kernel_info(rtb200_scene_handle h, rt_kernel_info* out) {
    if (!h || !out) return fail(RT_ERR_INVALID, "null argument");
    DeviceRestore restore;
    CU(cudaSetDevice(h->device));
    memset(out, 0, sizeof *out);
    KernelInfo ki{};
    CU(wavefront_info(h->mode, h->tp.n_lights > 0, h->minb, &ki));
    out->registers = ki.registers; out->local_bytes = ki.local_bytes; out->smem_bytes = (uint32_t)h->smem; out->grid = (uint32_t)h->grid;
    out->block = (uint32_t)kBlock; out->pool_slots = h->slots_per_cta;
    out->ctas_per_sm = (uint32_t)h->ctas_per_sm; out->smem_mask = h->tp.scene_in_smem;
    out->bvh_nodes = h->tp.n_nodes; out->bvh_leaves = h->tp.n_leaves; out->bvh_depth = h->tp.depth;
    snprintf(out->name, sizeof out->name, "%s", ki.name);
    return RT_OK;
}

// ---- resident scene edits ------------------------------------------------------------------------------
// Host side of rtb200_scene_update: O(n) validation, ONE host->device copy of the rt_sphere array, then the device rebuilds
// the records (rtb200_refit.cu). Nothing on the device is written before the whole edit has been validated.
static int validate_edit(const rtb200_scene_t* h, const rt_sphere* sp, uint64_t n) {
    if (n != h->tp.n) return fail(RT_ERR_INVALID, "rt_scene_edit.n_spheres must equal the uploaded sphere count");
    const double g[3] = {h->tp.gx, h->tp.gy, h->tp.gz};
    size_t li = 0, ai = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const rt_sphere& s = sp[i];
        int rc = validate_sphere(s, h->tex_ok.size(), [&](int32_t t) { return h->tex_ok[t] != 0; });
        if (rc != RT_OK) return rc;
        const bool was_light = li < h->light_ids.size() && h->light_ids[li] == i;
        li += was_light;
        if ((s.kind == RT_LIGHT) != was_light)
            return fail(RT_ERR_UNSUPPORTED, "the Light spheres must stay at the uploaded indices (kernel variant, light list and launch geometry were chosen from them): re-upload");
        if (h->mode != MODE_TREE) continue;
        const bool always = ai < h->always_ids.size() && h->always_ids[ai] == i;
        ai += always;
        if (!always && !rtbvh::in_f32_frame(s, g))
            return fail(RT_ERR_UNSUPPORTED, "sphere " + std::to_string(i) + " of the hierarchy leaves the upload's recentred f32 frame (non-finite, or max|c-g|+|r| >= 1e15): re-upload");
    }
    return RT_OK;
}

// First sphere edit of a handle: one allocation for the sphere copy and the maps of the refit, which are built on the device.
static int refit_init(rtb200_scene_t* h) {
    const TraceParams& tp = h->tp;
    const size_t n = tp.n, nn = tp.n_nodes;
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t b_sp = al(n * sizeof(rt_sphere)), b_slot = al(n * 4), b_node = al(nn * 4), b_box = al(nn * 8 * 6 * sizeof(double));
    CU(cudaMalloc(&h->refit, b_sp + b_slot + 2 * b_node + b_box + 256));
    char* b = (char*)h->refit;
    RefitParams& p = h->rp;
    p.sp = (const rt_sphere*)b;                     b += b_sp;
    p.slot_of = (uint32_t*)b;                       b += b_slot;
    p.parent = (uint32_t*)b;                        b += b_node;
    p.level = (uint32_t*)b;                         b += b_node;
    p.box64 = (double*)b;
    p.n = tp.n; p.n_nodes = tp.n_nodes; p.n_leaves = tp.n_leaves;
    p.gx = tp.gx; p.gy = tp.gy; p.gz = tp.gz;
    p.geo = (double4*)tp.geo; p.mat = (DevMat*)tp.mat;
    p.flat = h->mode == MODE_BRUTE ? (float*)tp.filt : nullptr;
    p.leaf_rec = (float*)tp.leaf_rec; p.leaf_id = tp.leaf_id; p.nodes = (float*)tp.nodes;
    cudaStream_t st = h->ctx->stream;
    CU(cudaMemsetAsync(p.slot_of, 0xff, n * 4, st));
    CU(cudaMemsetAsync(p.parent, 0xff, nn * 4, st));
    CU(launch_refit_maps(p, st));
    CU(cudaEventCreateWithFlags(&h->written, cudaEventDisableTiming));
    return RT_OK;
}

static int refit(rtb200_scene_t* h, const rt_sphere* sp) {
    DeviceCtx* ctx = h->ctx;
    CU(cudaSetDevice(h->device));
    if (!h->refit) {
        int rc = refit_init(h);
        if (rc != RT_OK) {
            if (h->refit) cudaFree(h->refit);
            if (h->written) cudaEventDestroy(h->written);
            h->refit = nullptr; h->written = nullptr;
            return rc;
        }
    }
    // through the context's pinned staging buffer (like an upload): the caller may reuse its array as soon as we return
    const size_t bytes = (size_t)h->tp.n * sizeof(rt_sphere);
    CU(cudaEventSynchronize(ctx->staging_free));
    CU(ctx->staging.ensure(bytes));
    memcpy(ctx->staging.p, sp, bytes);
    CU(cudaMemcpyAsync((void*)h->rp.sp, ctx->staging.p, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaEventRecord(ctx->staging_free, ctx->stream));
    CU(launch_refit(h->rp, h->tp.depth, ctx->stream));
    CU(cudaEventRecord(h->written, ctx->stream));
    return RT_OK;
}

int rtb200_scene_update(rtb200_scene_handle h, const rt_scene_edit* e) {
  return guarded([&]() -> int {
    if (!h || !e) return fail(RT_ERR_INVALID, "null argument");
    DeviceRestore restore;
    std::lock_guard<std::recursive_mutex> lk(h->ctx->mu);
    if (h->pending_frames) return fail(RT_ERR_INVALID, "asynchronous frames of this scene are in flight and read its arrays: call rtb200_render_device_wait first");
    if (e->spheres) {
        int rc = validate_edit(h, e->spheres, e->n_spheres);
        if (rc != RT_OK) return rc;
        if (h->tp.n && (rc = refit(h, e->spheres)) != RT_OK) return rc;
    }
    if (e->camera) h->tp.cam = *e->camera;
    if (e->seed) { h->tp.key0 = (uint32_t)*e->seed; h->tp.key1 = (uint32_t)(*e->seed >> 32); }
    return RT_OK;
  });
}

int rtb200_scene_debug_bvh(rtb200_scene_handle h, double recentre[3], uint32_t info[8], float* nodes, uint64_t cap_nodes,
                           float* leaf_rec, uint64_t cap_leaf_rec, uint32_t* leaf_id, uint64_t cap_leaf_id,
                           uint32_t* always, uint64_t cap_always, float* flat, uint64_t cap_flat) {
  return guarded([&]() -> int {
    if (!h || !info) return fail(RT_ERR_INVALID, "null argument");
    DeviceRestore restore;
    std::lock_guard<std::recursive_mutex> lk(h->ctx->mu);
    CU(cudaSetDevice(h->device));
    const TraceParams& tp = h->tp;
    const uint32_t n_pairs = h->mode == MODE_BRUTE ? tp.n_pairs : 0u;
    if (recentre) { recentre[0] = tp.gx; recentre[1] = tp.gy; recentre[2] = tp.gz; }
    info[0] = tp.n_nodes; info[1] = tp.n_leaves; info[2] = tp.depth; info[3] = (uint32_t)rtbvh::kLeafK; info[4] = tp.n_always;
    info[5] = (uint32_t)rtbvh::kNodeFloats; info[6] = n_pairs; info[7] = 0;
    cudaStream_t st = h->ctx->stream;   // after the handle's edits
    auto get = [&](void* dst, uint64_t cap, const void* src, uint64_t count) -> cudaError_t {
        const uint64_t k = std::min(cap, count);
        return dst && k ? cudaMemcpyAsync(dst, src, k * 4, cudaMemcpyDeviceToHost, st) : cudaSuccess;
    };
    CU(get(nodes, cap_nodes, tp.nodes, (uint64_t)tp.n_nodes * rtbvh::kNodeFloats));
    CU(get(leaf_rec, cap_leaf_rec, tp.leaf_rec, (uint64_t)tp.n_leaves * rtbvh::kLeafK * 4));
    CU(get(leaf_id, cap_leaf_id, tp.leaf_id, (uint64_t)tp.n_leaves * rtbvh::kLeafK));
    CU(get(always, cap_always, tp.always, tp.n_always));
    CU(get(flat, cap_flat, tp.filt, (uint64_t)n_pairs * 8));
    CU(cudaStreamSynchronize(st));
    return RT_OK;
  });
}

// Enqueue one frame on `stream_in` (or the context's stream) without waiting for it.
static int render_enqueue(rtb200_scene_handle h, void* dev_rgb8, void* dev_linear_f32, void* stream_in, int set) {
    if (!h) return fail(RT_ERR_INVALID, "null scene handle");
    DeviceCtx* ctx = h->ctx;
    DeviceCtx::WorkSet& W = ctx->ws[set & 1];
    CU(cudaSetDevice(h->device));
    cudaStream_t st = stream_in ? (cudaStream_t)stream_in : ctx->stream;
    if (st != ctx->stream) {   // the scene upload and edits ran on the context's stream
        CU(cudaStreamWaitEvent(st, ctx->staging_free, 0));
        if (h->written) CU(cudaStreamWaitEvent(st, h->written, 0));
    }
    TraceParams tp = h->tp;
    h->last_stream = st; h->last_set = set & 1; h->last_batches = 0; h->last_launches = 0;
    if (h->n_streams < 2 && (h->n_streams == 0 || h->streams[0] != st)) h->streams[h->n_streams++] = st;
    if (tp.npix_local == 0) return RT_OK;

    const uint32_t spp = tp.spp, spb = h->spp_batch;
    const uint32_t n_batches = (spp + spb - 1) / spb;
    const uint32_t threads_total = (uint32_t)h->grid * h->slots_per_cta;   // ray slots of the whole grid: columns of the per-slot global arrays

    CU(W.samplebuf.ensure((size_t)spb * tp.npix_local * 16));
    CU(W.accum.ensure((size_t)tp.npix_local * 12));
    CU(W.stack.ensure((size_t)std::max<uint32_t>(tp.max_depth, 1) * threads_total * 4));
    CU(W.small.ensure(256 + (size_t)n_batches * 4));
    if (tp.n_lights > 0) {
        // Nested light tests form a branching process: a vertex nests with probability 0.1 n and then spawns n shadow rays, so
        // depth d is reached with probability ~(0.1 n^2 P_hit)^d: harmless for 1-2 lights, near-critical for 3 (the reference
        // itself recurses hundreds of frames deep there) and super-critical beyond. Size the per-path frame stack accordingly;
        // an overflow is reported as an error, never rendered wrongly.
        tp.max_shadow = tp.n_lights == 1 ? 32u : tp.n_lights == 2 ? 96u : 384u;
        CU(W.frames.ensure((size_t)tp.max_shadow * threads_total * sizeof(ShadowFrame)));
        CU(W.lterm.ensure((size_t)6 * threads_total * 4));
    }
    tp.frames = (ShadowFrame*)W.frames.p;
    tp.lterm = (float*)W.lterm.p;
    // event ring: every pending frame owns 2 + 2*n_batches events (begin, end, and a pair around each trace launch)
    const uint32_t kRing = 64, per_frame = 2 + 2 * n_batches;
    if (h->pending_frames >= kRing) return fail(RT_ERR_INVALID, "more than 64 frames enqueued without rtb200_render_device_wait");
    while (h->ev.size() < (size_t)(h->pending_frames + 1) * per_frame) {
        cudaEvent_t e;
        if (!ctx->event_pool.empty()) { e = ctx->event_pool.back(); ctx->event_pool.pop_back(); }
        else CU(cudaEventCreate(&e));
        h->ev.push_back(e);
    }
    cudaEvent_t* fev = h->ev.data() + (size_t)h->pending_frames * per_frame;
    unsigned long long* stat = (unsigned long long*)W.small.p;
    unsigned int* counters = (unsigned int*)((char*)W.small.p + 256);
    CU(cudaMemsetAsync(W.small.p, 0, 256 + (size_t)n_batches * 4, st));
    CU(cudaMemsetAsync((char*)W.small.p + 64, 0xff, 16, st));   // stat[8], stat[9]: minima (kernel start / first dry-queue time, ns)

    tp.samplebuf = (float4*)W.samplebuf.p;
    tp.stack = (uint32_t*)W.stack.p;
    tp.stack_stride = threads_total;
    tp.stat = stat;

    CU(cudaEventRecord(fev[0], st));
    uint32_t launches = 0;
    for (uint32_t b = 0; b < n_batches; ++b) {
        tp.s0 = b * spb;
        tp.s_count = std::min(spb, spp - tp.s0);
        tp.total_work = tp.s_count * tp.npix_local;
        tp.work_counter = counters + b;
        CU(cudaEventRecord(fev[2 + 2 * b], st));
        if (tp.max_depth == 0) {
            CU(cudaMemsetAsync(tp.samplebuf, 0, (size_t)tp.total_work * 16, st));   // ray_color(depth 0) = black, no ray (raytracer.rs:80-82)
        } else {
            CU(launch_wavefront(tp, h->mode, h->grid, h->smem, h->minb, st));
        }
        CU(cudaEventRecord(fev[3 + 2 * b], st));
        ResolveParams q{};
        q.samplebuf = tp.samplebuf; q.accum = (float*)W.accum.p; q.npix_local = tp.npix_local; q.s_count = tp.s_count;
        q.first = b == 0; q.last = b + 1 == n_batches; q.spp = spp;
        q.out_linear = (float*)dev_linear_f32; q.out_rgb8 = (uint8_t*)dev_rgb8;
        CU(launch_resolve(q, st));
        launches += 2;
    }
    CU(cudaEventRecord(fev[1], st));
    h->last_batches = n_batches; h->last_launches = launches;
    ++h->pending_frames;
    return RT_OK;
}

// Wait for the frames of `h` enqueued so far and fetch statistics (counters: the last frame's; times: summed over the frames).
static int render_collect(rtb200_scene_handle h, rt_stats* stats) {
    if (!h) return fail(RT_ERR_INVALID, "null scene handle");
    DeviceCtx* ctx = h->ctx;
    CU(cudaSetDevice(h->device));
    if (stats) memset(stats, 0, sizeof *stats);
    if (h->tp.npix_local == 0 || h->last_batches == 0 || h->pending_frames == 0) { h->pending_frames = 0; h->n_streams = 0; return RT_OK; }
    cudaStream_t st = h->last_stream;
    DeviceCtx::WorkSet& W = ctx->ws[h->last_set];
    unsigned long long hstat[16] = {0}, herr[2] = {0, 0};
    for (int i = 0; i < h->n_streams; ++i) if (h->streams[i] != st) CU(cudaStreamSynchronize(h->streams[i]));
    h->n_streams = 0;
    // error counters accumulate over every frame since the last wait (each frame adds to them; nothing clears them in between)
    CU(cudaMemcpyAsync(hstat, W.small.p, sizeof hstat, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(herr, h->err, sizeof herr, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (herr[0] | herr[1]) CU(cudaMemset(h->err, 0, sizeof herr));
    const uint32_t frames = h->pending_frames;
    h->pending_frames = 0;
    if (herr[1] != 0) return fail(RT_ERR_CUDA, "internal error: the traversal guard tripped; the frame is not valid");
    if (herr[0] != 0) return fail(RT_ERR_UNSUPPORTED, "light-test recursion deeper than the shadow-frame stack occurred in one of the frames; it is not exact (the reference recursion is near-critical for this many lights)");
    if (stats) {
        float ms = 0.f;
        double dv = 0.0, tr = 0.0;
        const uint32_t per_frame = 2 + 2 * h->last_batches;
        for (uint32_t f = 0; f < frames; ++f) {
            cudaEvent_t* fev = h->ev.data() + (size_t)f * per_frame;
            CU(cudaEventElapsedTime(&ms, fev[0], fev[1])); dv += ms;
            for (uint32_t b = 0; b < h->last_batches; ++b) { CU(cudaEventElapsedTime(&ms, fev[2 + 2 * b], fev[3 + 2 * b])); tr += ms; }
        }
        stats->device_ms = dv; stats->trace_ms = tr; stats->frames = frames;
        stats->rays = hstat[0]; stats->candidates = hstat[1]; stats->samples = hstat[3]; stats->clusters = hstat[4]; stats->nodes = hstat[6];
        stats->gpus_used = 1;
        if (getenv("RTB200_PRINT_TAIL") && hstat[8] != ~0ull) {   // last batch of the last frame: when did the global queue run dry, when did the last CTA exit
            const double total = (double)(hstat[10] - hstat[8]) * 1e-6, tail = hstat[9] != ~0ull ? (double)(hstat[10] - hstat[9]) * 1e-6 : 0.0;
            fprintf(stderr, "[rtb200] trace kernel: first CTA start -> last CTA exit %.3f ms; queue dry -> last CTA exit (tail) %.3f ms; iterations after the queue ran dry: max %llu, mean %.1f per CTA\n",
                    total, tail, hstat[11], (double)hstat[12] / std::max(1, h->grid));
        }
        if (getenv("RTB200_PRINT_PHASES")) {
            fprintf(stderr, "[rtb200] fallbacks=%llu phases(warp-cycles): traverse=%llu exact=%llu waitA=%llu sort=%llu shade=%llu waitC=%llu warp_iters=%llu\n",
                    hstat[2], hstat[8], hstat[9], hstat[10], hstat[11], hstat[12], hstat[13], hstat[14]);
        }
        if (h->tp.max_depth == 0) stats->samples = (uint64_t)h->tp.npix_local * h->tp.spp;   // no kernel ran: every sample is black
        stats->kernel_launches = h->last_launches * frames; stats->batches = h->last_batches;
    }
    return RT_OK;
}

int rtb200_render_device(rtb200_scene_handle h, void* dev_rgb8, void* dev_linear_f32, void* stream_in, rt_stats* stats) {
    if (!h) return fail(RT_ERR_INVALID, "null scene handle");
    auto wall0 = std::chrono::steady_clock::now();
    DeviceRestore restore;
    std::lock_guard<std::recursive_mutex> lk(h->ctx->mu);
    if (h->pending_frames) { int rcw = render_collect(h, nullptr); if (rcw != RT_OK) return rcw; }   // drain frames enqueued earlier
    int rc = render_enqueue(h, dev_rgb8, dev_linear_f32, stream_in, 0);
    if (rc != RT_OK) return rc;
    rc = render_collect(h, stats);
    if (rc == RT_OK && stats) stats->wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
    return rc;
}

int rtb200_render_device_async(rtb200_scene_handle h, void* dev_rgb8, void* dev_linear_f32, void* stream_in) {
    if (!h) return fail(RT_ERR_INVALID, "null scene handle");
    DeviceRestore restore;
    std::lock_guard<std::recursive_mutex> lk(h->ctx->mu);
    return render_enqueue(h, dev_rgb8, dev_linear_f32, stream_in, (int)(h->frame_counter++ & 1u));
}

int rtb200_render_device_wait(rtb200_scene_handle h, rt_stats* stats) {
    if (!h) return fail(RT_ERR_INVALID, "null scene handle");
    DeviceRestore restore;
    std::lock_guard<std::recursive_mutex> lk(h->ctx->mu);
    return render_collect(h, stats);
}

static int render_host(const rt_scene* s, const rt_options* opts, uint8_t* out_rgb8, float* out_lin, rt_stats* stats) {
    auto wall0 = std::chrono::steady_clock::now();
    DeviceRestore restore;
    rtb200_scene_handle h = nullptr;
    int rc = rtb200_scene_upload(s, opts, &h);
    if (rc != RT_OK) return rc;
    DeviceCtx* ctx = h->ctx;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    cudaSetDevice(h->device);
    size_t npl = h->tp.npix_local;
    void *d8 = nullptr, *dl = nullptr;
    cudaError_t e = cudaSuccess;
    if (out_rgb8) { e = ctx->out_rgb8.ensure(npl * 3 + 16); d8 = ctx->out_rgb8.p; }
    if (e == cudaSuccess && out_lin) { e = ctx->out_lin.ensure(npl * 12 + 16); dl = ctx->out_lin.p; }
    if (e != cudaSuccess) { rtb200_scene_release(h); return fail_cuda(e, "output buffer allocation"); }
    rt_stats st{};
    rc = rtb200_render_device(h, d8, dl, nullptr, &st);
    if (rc == RT_OK && npl) {
        if (out_rgb8) e = cudaMemcpyAsync(out_rgb8, d8, npl * 3, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess && out_lin) e = cudaMemcpyAsync(out_lin, dl, npl * 12, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail_cuda(e, "device->host copy of the frame");
    }
    st.h2d_bytes = h->h2d_bytes;
    st.d2h_bytes = (out_rgb8 ? npl * 3 : 0) + (out_lin ? npl * 12 : 0) + 128 + 16;
    std::string keep = g_last_error;
    rtb200_scene_release(h);
    if (rc != RT_OK) g_last_error = keep;
    st.wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
    if (stats) *stats = st;
    return rc;
}

int rtb200_render_rgb8(const rt_scene* scene, const rt_options* opts, uint8_t* out_rgb8, rt_stats* stats) {
    if (!scene || !out_rgb8) return fail(RT_ERR_INVALID, "null argument");
    return guarded([&]() -> int { return render_host(scene, opts, out_rgb8, nullptr, stats); });
}
int rtb200_render_linear_f32(const rt_scene* scene, const rt_options* opts, float* out_rgb, rt_stats* stats) {
    if (!scene || !out_rgb) return fail(RT_ERR_INVALID, "null argument");
    return guarded([&]() -> int { return render_host(scene, opts, nullptr, out_rgb, stats); });
}

// One process, n_gpus devices: the reference's row bands (raytracer.rs:254-262) dealt round-robin to the devices (band b ->
// device b mod G, like the torchrun flavour in rtb200/dist.py). The hierarchy is built once; one host thread per device
// uploads the scene, enqueues trace + resolve, copies its compact shard peer-to-peer over NVLink straight into its interleaved
// rows of the frame on the first device and waits for its stream; then ONE device->host copy.
static std::mutex g_multi_mu;   // multi-GPU calls take turns (they share the frame buffer of the first device)

int rtb200_render_rgb8_multi(const rt_scene* s, const rt_options* opts_in, int32_t n_gpus, uint8_t* out_rgb8, rt_stats* stats) {
  return guarded([&]() -> int {
    if (!s || !out_rgb8) return fail(RT_ERR_INVALID, "null argument");
    auto wall0 = std::chrono::steady_clock::now();
    rt_options base;
    int rc = normalise_options(opts_in, &base);
    if (rc != RT_OK) return rc;
    if (base.world != 1 || base.rank != 0) return fail(RT_ERR_INVALID, "rtb200_render_rgb8_multi shards the frame itself: opts->rank/world must be 0/1");
    uint32_t n_lights = 0;
    if ((rc = validate_scene(s, &n_lights)) != RT_OK) return rc;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) return fail_cuda(e, "cudaGetDeviceCount");
    if (count <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device");
    const int first = base.device < 0 ? 0 : base.device;
    if (first >= count) return fail(RT_ERR_NO_DEVICE, "no such CUDA device");
    int G = n_gpus <= 0 ? count - first : std::min(n_gpus, count - first);
    G = std::min(G, 64 - first);   // device contexts exist for ordinals below 64
    const uint32_t bands = (s->height + base.band_rows - 1) / base.band_rows;
    G = (int)std::min<uint32_t>((uint32_t)G, bands);   // a device needs at least one band
    if (G <= 1) { base.device = first; int r = render_host(s, &base, out_rgb8, nullptr, stats); if (r == RT_OK && stats) stats->gpus_used = 1; return r; }

    DeviceRestore restore;
    std::lock_guard<std::mutex> multi_lock(g_multi_mu);
    rtbvh::Records R;
    rtbvh::build_records(s, mode_of(base.variant) == MODE_TREE, R);
    const size_t row_bytes = (size_t)s->width * 3;
    // the frame lives on the first device; peers get access both ways once per process (without it the copies stage through the host)
    DeviceCtx* c0 = nullptr;
    if ((rc = get_ctx(first, &c0)) != RT_OK) return rc;
    uint8_t* frame = nullptr;
    {
        std::lock_guard<std::recursive_mutex> lk(c0->mu);
        CU(c0->frame.ensure((size_t)s->height * row_bytes + 16));
        frame = (uint8_t*)c0->frame.p;
        static bool peered[64] = {false};
        for (int g = 1; g < G; ++g) {
            if (peered[first + g]) continue;
            cudaSetDevice(first); if (cudaDeviceEnablePeerAccess(first + g, 0) != cudaSuccess) cudaGetLastError();
            cudaSetDevice(first + g); if (cudaDeviceEnablePeerAccess(first, 0) != cudaSuccess) cudaGetLastError();
            peered[first + g] = true;
        }
    }
    struct Result { int rc = RT_OK; std::string err; rt_stats st{}; uint64_t h2d = 0; };
    std::vector<Result> res((size_t)G);
    auto worker = [&](int g) {
        Result& r = res[(size_t)g];
        auto body = [&]() -> int {
            rt_options o = base; o.device = first + g; o.rank = g; o.world = G;
            rtb200_scene_handle h = nullptr;
            int rcw = scene_upload_records(s, o, n_lights, R, &h);
            if (rcw != RT_OK) return rcw;
            struct Rel { rtb200_scene_handle h; ~Rel() { std::string keep = g_last_error; rtb200_scene_release(h); g_last_error = keep; } } rel{h};
            DeviceCtx* c = h->ctx;
            std::lock_guard<std::recursive_mutex> lk(c->mu);
            CU(cudaSetDevice(first + g));
            const size_t rows = h->tp.rows_local;
            CU(c->out_rgb8.ensure(rows * row_bytes + 16));
            if ((rcw = render_enqueue(h, c->out_rgb8.p, nullptr, nullptr, 0)) != RT_OK) return rcw;
            // shard -> frame: full bands as one strided 2-D copy (a "row" of the copy = one band), then the partial last band
            const size_t band_bytes = (size_t)base.band_rows * row_bytes;
            const size_t full = rows / base.band_rows, rem = rows - full * base.band_rows;
            if (full) CU(cudaMemcpy2DAsync(frame + (size_t)g * band_bytes, (size_t)G * band_bytes, c->out_rgb8.p, band_bytes, band_bytes, full, cudaMemcpyDefault, c->stream));
            if (rem) CU(cudaMemcpyAsync(frame + ((size_t)full * G + g) * band_bytes, (uint8_t*)c->out_rgb8.p + full * band_bytes, rem * row_bytes, cudaMemcpyDefault, c->stream));
            if ((rcw = render_collect(h, &r.st)) != RT_OK) return rcw;   // waits for the stream: the shard is in the frame
            r.h2d = h->h2d_bytes;
            return RT_OK;
        };
        r.rc = guarded(body);
        if (r.rc != RT_OK) r.err = g_last_error;
    };
    std::vector<std::thread> threads;
    threads.reserve((size_t)G);
    struct Joiner { std::vector<std::thread>& ts; ~Joiner() { for (auto& t : ts) if (t.joinable()) t.join(); } };
    {
        Joiner joiner{threads};   // also on the exceptional path (thread creation can throw): never destroy a joinable thread
        for (int g = 1; g < G; ++g) threads.emplace_back(worker, g);
        worker(0);
    }
    for (int g = 0; g < G; ++g) if (res[(size_t)g].rc != RT_OK) return fail(res[(size_t)g].rc, "device " + std::to_string(first + g) + ": " + res[(size_t)g].err);
    rt_stats total{};
    for (int g = 0; g < G; ++g) {
        const rt_stats& st = res[(size_t)g].st;
        total.rays += st.rays; total.samples += st.samples; total.candidates += st.candidates; total.clusters += st.clusters; total.nodes += st.nodes;
        total.device_ms = std::max(total.device_ms, st.device_ms); total.trace_ms = std::max(total.trace_ms, st.trace_ms);
        total.kernel_launches += st.kernel_launches; total.batches = std::max(total.batches, st.batches);
        total.h2d_bytes += res[(size_t)g].h2d;
    }
    {
        std::lock_guard<std::recursive_mutex> lk(c0->mu);
        CU(cudaSetDevice(first));
        CU(cudaMemcpyAsync(out_rgb8, frame, (size_t)s->height * row_bytes, cudaMemcpyDeviceToHost, c0->stream));
        CU(cudaStreamSynchronize(c0->stream));
    }
    total.frames = 1; total.gpus_used = G;
    total.d2h_bytes = (size_t)s->height * row_bytes + (size_t)G * (128 + 16);
    total.wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
    if (stats) *stats = total;
    return RT_OK;
  });
}

// ---- probes ------------------------------------------------------------------------------------------
static int probe_io(const void* in, size_t in_bytes, size_t out_bytes, DeviceCtx** pctx, void** din, void** dout) {
    int rc = get_ctx(-1, pctx);
    if (rc != RT_OK) return rc;
    DeviceCtx* c = *pctx;
    CU(c->probe.ensure(in_bytes + out_bytes + 512));
    *din = c->probe.p;
    *dout = (char*)c->probe.p + ((in_bytes + 255) / 256) * 256;
    CU(cudaMemsetAsync(*dout, 0, out_bytes, c->stream));
    if (in_bytes) CU(cudaMemcpyAsync(*din, in, in_bytes, cudaMemcpyHostToDevice, c->stream));
    return RT_OK;
}
static int probe_finish(DeviceCtx* c, void* host_out, const void* dout, size_t out_bytes) {
    CU(cudaMemcpyAsync(host_out, dout, out_bytes, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return RT_OK;
}

int rtb200_probe_sphere_hit(const rt_vec3* center, double radius, const rt_vec3* origin, const rt_vec3* dir, double t_min,
                            double t_max, int32_t* hit, double* t, rt_vec3* point, rt_vec3* normal, int32_t* front_face) {
    double in[12] = {center->x, center->y, center->z, radius, origin->x, origin->y, origin->z, dir->x, dir->y, dir->z, t_min, t_max};
    double out[9];
    DeviceCtx* c; void *din, *dout;
    int rc = probe_io(in, sizeof in, sizeof out, &c, &din, &dout);
    if (rc != RT_OK) return rc;
    CU(probe_sphere_hit((const double*)din, (double*)dout, c->stream));
    if ((rc = probe_finish(c, out, dout, sizeof out)) != RT_OK) return rc;
    *hit = out[0] != 0.0;
    if (*hit) {
        *t = out[1]; *point = rt_vec3{out[2], out[3], out[4]}; *normal = rt_vec3{out[5], out[6], out[7]};
        *front_face = out[8] != 0.0;
    }
    return RT_OK;
}
int rtb200_probe_refract(const rt_vec3* uv, const rt_vec3* n, double eta, rt_vec3* o) {
    double in[7] = {uv->x, uv->y, uv->z, n->x, n->y, n->z, eta}, out[3];
    DeviceCtx* c; void *din, *dout;
    int rc = probe_io(in, sizeof in, sizeof out, &c, &din, &dout);
    if (rc != RT_OK) return rc;
    CU(probe_refract((const double*)din, (double*)dout, c->stream));
    if ((rc = probe_finish(c, out, dout, sizeof out)) != RT_OK) return rc;
    *o = rt_vec3{out[0], out[1], out[2]};
    return RT_OK;
}
int rtb200_probe_reflectance(double cosine, double ref_idx, double* o) {
    double in[2] = {cosine, ref_idx};
    DeviceCtx* c; void *din, *dout;
    int rc = probe_io(in, sizeof in, 8, &c, &din, &dout);
    if (rc != RT_OK) return rc;
    CU(probe_reflectance((const double*)din, (double*)dout, c->stream));
    return probe_finish(c, o, dout, 8);
}
int rtb200_probe_sky(const rt_vec3* dir, uint32_t sky_mode, float out_rgb[3]) {
    if (sky_mode == RT_SKY_TEXTURE) return fail(RT_ERR_INVALID, "probe_sky supports none/gradient only");
    double in[3] = {dir->x, dir->y, dir->z};
    DeviceCtx* c; void *din, *dout;
    int rc = probe_io(in, sizeof in, 12, &c, &din, &dout);
    if (rc != RT_OK) return rc;
    CU(probe_sky((const double*)din, sky_mode, (float*)dout, c->stream));
    return probe_finish(c, out_rgb, dout, 12);
}
int rtb200_probe_get_ray(const rt_camera* cam, double u, double v, rt_vec3* origin, rt_vec3* dir) {
    struct { rt_camera cam; double uv[2]; } in;
    in.cam = *cam; in.uv[0] = u; in.uv[1] = v;
    double out[6];
    DeviceCtx* c; void *din, *dout;
    int rc = probe_io(&in, sizeof in, sizeof out, &c, &din, &dout);
    if (rc != RT_OK) return rc;
    CU(probe_get_ray((const rt_camera*)din, (const double*)((char*)din + sizeof(rt_camera)), (double*)dout, c->stream));
    if ((rc = probe_finish(c, out, dout, sizeof out)) != RT_OK) return rc;
    *origin = rt_vec3{out[0], out[1], out[2]}; *dir = rt_vec3{out[3], out[4], out[5]};
    return RT_OK;
}
int rtb200_probe_rng(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t kind, uint32_t n, double* o) {
    DeviceCtx* c; void *din, *dout;
    int rc = probe_io(nullptr, 0, (size_t)n * 8, &c, &din, &dout);
    if (rc != RT_OK) return rc;
    CU(probe_rng(seed, pixel, sample, kind, n, (double*)dout, c->stream));
    return probe_finish(c, o, dout, (size_t)n * 8);
}
int rtb200_probe_sphere_uv(const double* hp_xyz, uint32_t n, double* out_uv) {
    DeviceCtx* c; void *din, *dout;
    int rc = probe_io(hp_xyz, (size_t)n * 24, (size_t)n * 16, &c, &din, &dout);
    if (rc != RT_OK) return rc;
    CU(probe_sphere_uv((const double*)din, n, (double*)dout, c->stream));
    return probe_finish(c, out_uv, dout, (size_t)n * 16);
}
int rtb200_probe_quantise(const float* mean_linear, uint32_t n, uint8_t* o) {
    DeviceCtx* c; void *din, *dout;
    int rc = probe_io(mean_linear, (size_t)n * 4, n, &c, &din, &dout);
    if (rc != RT_OK) return rc;
    CU(probe_quantise((const float*)din, n, (uint8_t*)dout, c->stream));
    return probe_finish(c, o, dout, n);
}

}  // extern "C"
