// rtb200_refit.cu — on-device refit of a resident scene after a sphere edit (rtb200_scene_update).
//
// The hierarchy's topology (child refs, leaf_id, always-list) and the recentring g stay those of the upload; every record
// the closest-hit stage reads is rebuilt from the new spheres with the formulas of the host builder (rtb200_bvh.hpp), written
// with explicit round-to-nearest f64 intrinsics because the host side is compiled with -ffp-contract=off. Same topology, same
// spheres -> same bits as rtbvh::build_records, so the soundness argument of DESIGN.md §4.2 carries over unchanged (§4.6).
//
//   rt_refit_spheres_kernel  one thread per sphere: exact geometry, material, flat record (MODE_BRUTE), leaf slot record
//   rt_refit_nodes_kernel    one launch per wide level, deepest first, one thread per child slot of that level's nodes:
//                            exact f64 union of the member boxes c-g +- |r| (leaf slots) or of the child node's slot boxes
//                            (inner slots, from the previous launch), kept in box64, then inflated and rounded outwards to f32
#include "rtb200_kernels.cuh"

namespace rtk {

namespace {

constexpr uint32_t kEmpty = 0xffffffffu;
constexpr uint32_t kLeaf = 0x80000000u;
constexpr double kU = 5.9604644775390625e-8;   // 2^-24 (= rtbvh::kU)

// rtbvh::sphere_record: candidate iff b^2 + 2c.o + nk >= |o|^2 (1 - 96u), nk = -(|c|^2 - r^2) + Es rounded up
__device__ __forceinline__ void sphere_record(double x, double y, double z, double r2, float rec[4]) {
    const double c2 = __dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z));
    const double Es = __dadd_rn(__dadd_rn(__dmul_rn(96.0 * kU, c2), __dmul_rn(16.0 * kU, r2)), 1e-30);
    const double nkd = __dadd_rn(-__dsub_rn(c2, r2), Es);
    rec[0] = __double2float_rn(x); rec[1] = __double2float_rn(y); rec[2] = __double2float_rn(z);
    rec[3] = isfinite(nkd) ? __double2float_ru(nkd) : __int_as_float(0x7f800000);
    const bool ok = isfinite(rec[0]) && isfinite(rec[1]) && isfinite(rec[2]) && isfinite(nkd) && c2 < 1e30;
    if (!ok) { rec[0] = rec[1] = rec[2] = 0.f; rec[3] = __int_as_float(0x7f800000); }   // always a candidate
}

__global__ void __launch_bounds__(256) rt_refit_maps_kernel(const RefitParams p) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < p.n_leaves * (uint32_t)kLeafK) {
        const uint32_t id = p.leaf_id[t];
        if (id != kEmpty) p.slot_of[id] = t;
    }
    if (t < p.n_nodes * 8u) {
        const uint32_t ref = __float_as_uint(p.nodes[(size_t)(t >> 3) * (kNodeVec * 4) + 48 + (t & 7u)]);
        if (ref != kEmpty && !(ref & kLeaf)) p.parent[ref] = t >> 3;
    }
}

__global__ void __launch_bounds__(256) rt_refit_levels_kernel(const RefitParams p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_nodes) return;
    uint32_t l = 1, q = i;
    while (q != 0u && q != kEmpty && l < 64u) { q = p.parent[q]; ++l; }
    p.level[i] = l;
}

__global__ void __launch_bounds__(256) rt_refit_spheres_kernel(const RefitParams p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const rt_sphere sp = p.sp[i];
    p.geo[i] = make_double4(sp.center.x, sp.center.y, sp.center.z, sp.radius);
    DevMat m;
    m.kind = sp.kind; m.param = sp.param; m.tex = sp.texture; m.pad = 0;
    if (sp.kind == RT_LAMBERTIAN || sp.kind == RT_METAL) { m.r = sp.albedo[0]; m.g = sp.albedo[1]; m.b = sp.albedo[2]; }
    else { m.r = m.g = m.b = 1.0f; }   // Glass/Light attenuation is (1,1,1); Texture uses texels
    p.mat[i] = m;
    if (!p.flat && p.slot_of[i] == kEmpty) return;
    float rec[4];
    sphere_record(__dsub_rn(sp.center.x, p.gx), __dsub_rn(sp.center.y, p.gy), __dsub_rn(sp.center.z, p.gz), __dmul_rn(sp.radius, sp.radius), rec);
    if (p.flat) {
        float* A = p.flat + (size_t)(i >> 1) * 8;
        const uint32_t k = i & 1u;
        A[0 + k] = rec[0]; A[2 + k] = rec[1]; A[4 + k] = rec[2]; A[6 + k] = rec[3];
    }
    const uint32_t s = p.slot_of[i];
    if (s != kEmpty) {
        float* A = p.leaf_rec + (size_t)(s / kLeafK) * (kLeafK * 4) + (size_t)((s % kLeafK) >> 1) * 8;
        const uint32_t k = s & 1u;
        A[0 + k] = rec[0]; A[2 + k] = rec[1]; A[4 + k] = rec[2]; A[6 + k] = rec[3];
    }
}

__global__ void __launch_bounds__(256) rt_refit_nodes_kernel(const RefitParams p, uint32_t level) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.n_nodes * 8u) return;
    const uint32_t node = t >> 3, k = t & 7u;
    if (p.level[node] != level) return;
    float* N = p.nodes + (size_t)node * (kNodeVec * 4);
    const uint32_t ref = __float_as_uint(N[48 + k]);
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    double lo[3] = {inf, inf, inf}, hi[3] = {-inf, -inf, -inf};
    if (ref != kEmpty && (ref & kLeaf)) {
        const uint32_t* ids = p.leaf_id + (size_t)(ref & ~kLeaf) * kLeafK;
        for (int j = 0; j < kLeafK; ++j) {
            const uint32_t id = ids[j];
            if (id == kEmpty) continue;
            const rt_sphere& sp = p.sp[id];
            const double c[3] = {__dsub_rn(sp.center.x, p.gx), __dsub_rn(sp.center.y, p.gy), __dsub_rn(sp.center.z, p.gz)};
            const double r = fabs(sp.radius);
            for (int a = 0; a < 3; ++a) { lo[a] = fmin(lo[a], __dsub_rn(c[a], r)); hi[a] = fmax(hi[a], __dadd_rn(c[a], r)); }
        }
    } else if (ref != kEmpty) {   // inner child: its slots were refitted by the previous (deeper) launch
        const double* B = p.box64 + (size_t)ref * 48;
        for (int j = 0; j < 8; ++j)
            for (int a = 0; a < 3; ++a) { lo[a] = fmin(lo[a], B[j * 6 + a]); hi[a] = fmax(hi[a], B[j * 6 + 3 + a]); }
    }
    double* Bo = p.box64 + (size_t)t * 6;
    for (int a = 0; a < 3; ++a) { Bo[a] = lo[a]; Bo[3 + a] = hi[a]; }
    if (ref == kEmpty) return;   // empty slot: {+inf, -inf} as emitted, never hit
    // rtbvh::Builder::emit_wide: m = 32u * max|coordinate| + 1e-30 covers the f32 rounding of the slab test (DESIGN.md §4.2)
    double bmax = 0.0;
    for (int a = 0; a < 3; ++a) bmax = fmax(bmax, fmax(fabs(lo[a]), fabs(hi[a])));
    const double m = __dadd_rn(__dmul_rn(32.0 * kU, bmax), 1e-30);
    for (int a = 0; a < 3; ++a) {
        N[a * 8 + k] = __double2float_rd(__dsub_rn(lo[a], m));
        N[24 + a * 8 + k] = __double2float_ru(__dadd_rn(hi[a], m));
    }
}

inline int blocks_for(uint32_t n) { return (int)((n + 255u) / 256u); }

}  // namespace

cudaError_t launch_refit_maps(const RefitParams& p, cudaStream_t st) {
    const uint32_t work = max(p.n_leaves * (uint32_t)kLeafK, p.n_nodes * 8u);
    if (work == 0) return cudaSuccess;
    rt_refit_maps_kernel<<<blocks_for(work), 256, 0, st>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess || p.n_nodes == 0) return e;
    rt_refit_levels_kernel<<<blocks_for(p.n_nodes), 256, 0, st>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_refit(const RefitParams& p, uint32_t depth, cudaStream_t st) {
    if (p.n == 0) return cudaSuccess;
    rt_refit_spheres_kernel<<<blocks_for(p.n), 256, 0, st>>>(p);
    cudaError_t e = cudaGetLastError();
    for (uint32_t l = depth; l >= 1 && p.n_nodes > 0 && e == cudaSuccess; --l) {
        rt_refit_nodes_kernel<<<blocks_for(p.n_nodes * 8u), 256, 0, st>>>(p, l);
        e = cudaGetLastError();
    }
    return e;
}

}  // namespace rtk
