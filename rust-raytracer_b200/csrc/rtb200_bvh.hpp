// rtb200_bvh.hpp — host-side construction of everything the closest-hit stage reads (no CUDA calls).
//
// hit_world (reference raytracer/src/raytracer.rs:44-59) scans ALL spheres and keeps the closest root, first index on
// ties. That fold equals the lexicographic minimum of (first root beyond t_min, sphere index) over the spheres the
// exact f64 Sphere::hit (sphere.rs:46-78) accepts, so ANY conservative pre-selection that never drops an accepted
// sphere gives identical results. This file builds that pre-selection as a hierarchy:
//
//   * an 8-wide bounding-volume hierarchy over the spheres' axis-aligned boxes (binned-SAH binary build, collapsed to
//     8 children per node), node boxes stored in f32, rounded outwards and inflated by 32u*max|coordinate| so that the
//     kernel's f32 slab test can only err towards "hit" (soundness argument: DESIGN.md §4.2);
//   * leaves of kLeafK spheres as pair-packed f32 records of the 7-FMA conservative sphere test
//     ({cx0,cx1,cy0,cy1},{cz0,cz1,nk0,nk1}, nk = -(|c|^2-r^2) + Es rounded up), plus slot -> ORIGINAL sphere index;
//   * an "always" list: spheres that cannot live in the f32 frame (non-finite, |c| >= 1e15) are tested in f64 for
//     every ray;
//   * the flat pair-packed record array of all spheres (RT_VARIANT_BRUTE_FORCE scans it like hit_world scans the Vec);
//   * exact geometry {cx,cy,cz,radius} f64 and the material records.
//
// Everything is expressed in a frame recentred on the component-wise median of the centres (f32 keeps more bits there).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/rtb200.h"

namespace rtbvh {

#ifndef RT_LEAF_K
#define RT_LEAF_K 8
#endif
constexpr int kLeafK = RT_LEAF_K; // sphere slots per leaf (RT_LEAF_K/2 FFMA2 pairs); even
constexpr int kWide = 8;          // children per node
constexpr int kNodeFloats = 56;   // lo_x[8] lo_y[8] lo_z[8] hi_x[8] hi_y[8] hi_z[8] child[8]  (224 bytes)
constexpr uint32_t kEmptyChild = 0xffffffffu;
constexpr uint32_t kLeafBit = 0x80000000u;
constexpr int kMaxDepth = 21;     // wide levels the builder can produce; the kernel's node stack needs 32 + 7*depth + 8 entries (rtb200_api.cu asserts it)
constexpr int kAreaFirstLevels = 15;   // below this wide level children are expanded breadth-first (3 binary levels per wide level)
constexpr double kU = 5.9604644775390625e-8;   // 2^-24

struct Mat32 { float r, g, b; uint32_t kind; double param; int32_t tex; int32_t pad; };   // = rtk::DevMat

struct Records {
    double g[3] = {0, 0, 0};
    uint32_t n = 0;
    uint32_t n_nodes = 0, n_leaves = 0, depth = 0;
    std::vector<float> nodes;         // n_nodes * kNodeFloats
    std::vector<float> leaf_rec;      // n_leaves * kLeafK * 4
    std::vector<uint32_t> leaf_id;    // n_leaves * kLeafK, 0xffffffff = padding slot
    std::vector<uint32_t> always;     // spheres tested in f64 for every ray
    uint32_t n_pairs = 0;
    std::vector<float> flat;          // n_pairs * 8: every sphere, list order, pair-packed (padding never hits)
    std::vector<double> geo;          // max(n,1) * 4
    std::vector<Mat32> mat;           // max(n,1)
};

inline float f32_up(double x) {     // smallest float >= x
    float f = (float)x;
    if ((double)f < x) f = std::nextafterf(f, INFINITY);
    return f;
}
inline float f32_down(double x) {   // largest float <= x
    float f = (float)x;
    if ((double)f > x) f = std::nextafterf(f, -INFINITY);
    return f;
}

// Record of the conservative sphere test for a sphere at recentred (x,y,z) with squared radius r2.
// candidate iff  b^2 + 2c.o + nk >= |o|^2 (1 - 96u),  nk = -(|c|^2 - r^2) + Es rounded up,  Es = 96u|c|^2 + 16u r^2.
inline bool sphere_record(double x, double y, double z, double r2, float rec[4]) {
    const double c2 = x * x + y * y + z * z;
    const double Es = 96.0 * kU * c2 + 16.0 * kU * r2 + 1e-30;
    const double nkd = -(c2 - r2) + Es;
    rec[0] = (float)x; rec[1] = (float)y; rec[2] = (float)z;
    rec[3] = std::isfinite(nkd) ? f32_up(nkd) : INFINITY;
    return std::isfinite(rec[0]) && std::isfinite(rec[1]) && std::isfinite(rec[2]) && std::isfinite(nkd) && c2 < 1e30;
}

// Whether sphere `sp` lives in the hierarchy of the frame recentred on g (else it goes to the always-list): finite, and
// max|c-g| + |r| < 1e15. rtb200_scene_update applies the same test to edited spheres of the hierarchy.
inline bool in_f32_frame(const rt_sphere& sp, const double g[3]) {
    const double c[3] = {sp.center.x - g[0], sp.center.y - g[1], sp.center.z - g[2]};
    const double r = std::fabs(sp.radius);
    const bool fin = std::isfinite(c[0]) && std::isfinite(c[1]) && std::isfinite(c[2]) && std::isfinite(r);
    const double ext = fin ? std::max(std::max(std::fabs(c[0]), std::fabs(c[1])), std::fabs(c[2])) + r : INFINITY;
    return fin && ext < 1e15;
}

struct Box {
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    void grow(const Box& o) { for (int a = 0; a < 3; ++a) { lo[a] = std::min(lo[a], o.lo[a]); hi[a] = std::max(hi[a], o.hi[a]); } }
    void grow_pt(const double p[3]) { for (int a = 0; a < 3; ++a) { lo[a] = std::min(lo[a], p[a]); hi[a] = std::max(hi[a], p[a]); } }
    double area() const {
        const double dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        if (!(dx >= 0 && dy >= 0 && dz >= 0)) return 0.0;
        return 2.0 * (dx * dy + dy * dz + dz * dx);
    }
};

struct BinNode { Box box; int left = -1, right = -1; uint32_t first = 0, count = 0; };

class Builder {
public:
    Builder(const rt_scene* s, Records& R) : s_(s), R_(R) {}

    void run(bool want_tree) {
        const uint32_t n = (uint32_t)s_->n_spheres;
        R_.n = n;
        recentre();
        flat_and_exact();
        if (!want_tree) return;
        // primitives of the hierarchy: spheres that live in the f32 frame; the rest is tested for every ray
        for (uint32_t i = 0; i < n; ++i) {
            const rt_sphere& sp = s_->spheres[i];
            if (!in_f32_frame(sp, R_.g)) { R_.always.push_back(i); continue; }
            double c[3] = {sp.center.x - R_.g[0], sp.center.y - R_.g[1], sp.center.z - R_.g[2]};
            const double r = std::fabs(sp.radius);
            Box b;
            for (int a = 0; a < 3; ++a) { b.lo[a] = c[a] - r; b.hi[a] = c[a] + r; }
            prim_box_.push_back(b);
            prim_id_.push_back(i);
            prim_c_.push_back({c[0], c[1], c[2]});
        }
        if (prim_id_.empty()) return;
        order_.resize(prim_id_.size());
        for (uint32_t i = 0; i < order_.size(); ++i) order_[i] = i;
        bin_.reserve(2 * order_.size() / kLeafK + 8);
        // depth budget: SAH splits down to binary level sah_limit_, balanced median splits below, so that the binary (hence
        // the 8-wide) depth stays <= 30 < kMaxDepth whatever the input
        int lg = 0;
        while (((size_t)kLeafK << lg) < order_.size()) ++lg;
        sah_limit_ = std::max(4, 30 - lg - 1);
        if (const char* e = getenv("RTB200_BVH_AREA_LEVELS")) area_levels_ = std::max(1, atoi(e));   // test hook: exercise the breadth-first collapse
        const int root = build(0, (uint32_t)order_.size(), 0);
        R_.depth = 0;
        emit_wide(root, 1);
        R_.n_nodes = (uint32_t)(R_.nodes.size() / kNodeFloats);
        R_.n_leaves = (uint32_t)(R_.leaf_id.size() / kLeafK);
    }

private:
    struct P3 { double x, y, z; };
    const rt_scene* s_;
    Records& R_;
    std::vector<Box> prim_box_;
    std::vector<uint32_t> prim_id_;
    std::vector<P3> prim_c_;
    std::vector<uint32_t> order_;
    std::vector<BinNode> bin_;
    int sah_limit_ = 24;
    int area_levels_ = kAreaFirstLevels;

    void recentre() {
        const uint32_t n = R_.n;
        if (!n) return;
        std::vector<double> tmp(n);
        for (int c = 0; c < 3; ++c) {
            for (uint32_t i = 0; i < n; ++i) tmp[i] = c == 0 ? s_->spheres[i].center.x : (c == 1 ? s_->spheres[i].center.y : s_->spheres[i].center.z);
            std::nth_element(tmp.begin(), tmp.begin() + n / 2, tmp.end());
            R_.g[c] = std::isfinite(tmp[n / 2]) ? tmp[n / 2] : 0.0;
        }
    }

    void flat_and_exact() {
        const uint32_t n = R_.n;
        uint32_t n_pairs = ((n + 1) / 2 + 7) / 8 * 8;   // the scan loop consumes blocks of 4 pairs; padding records never hit
        if (n_pairs == 0) n_pairs = 8;
        R_.n_pairs = n_pairs;
        R_.flat.assign((size_t)n_pairs * 8, 0.f);
        R_.geo.assign((size_t)std::max<uint32_t>(n, 1) * 4, 0.0);
        R_.mat.resize(std::max<uint32_t>(n, 1));
        std::memset(R_.mat.data(), 0, R_.mat.size() * sizeof(Mat32));
        for (uint32_t pp = 0; pp < n_pairs; ++pp) {
            float* A = &R_.flat[(size_t)pp * 8];
            for (int k = 0; k < 2; ++k) {
                const uint32_t i = 2 * pp + k;
                float rec[4] = {0.f, 0.f, 0.f, -INFINITY};
                if (i < n) {
                    const rt_sphere& sp = s_->spheres[i];
                    if (!sphere_record(sp.center.x - R_.g[0], sp.center.y - R_.g[1], sp.center.z - R_.g[2], sp.radius * sp.radius, rec)) {
                        rec[0] = rec[1] = rec[2] = 0.f; rec[3] = INFINITY;   // always a candidate
                    }
                    double* G = &R_.geo[4 * (size_t)i];
                    G[0] = sp.center.x; G[1] = sp.center.y; G[2] = sp.center.z; G[3] = sp.radius;
                    Mat32& m = R_.mat[i];
                    m.kind = sp.kind; m.param = sp.param; m.tex = sp.texture; m.pad = 0;
                    if (sp.kind == RT_LAMBERTIAN || sp.kind == RT_METAL) { m.r = sp.albedo[0]; m.g = sp.albedo[1]; m.b = sp.albedo[2]; }
                    else { m.r = m.g = m.b = 1.0f; }   // Glass/Light attenuation is (1,1,1) (materials.rs:67,179); Texture uses texels
                }
                A[0 + k] = rec[0]; A[2 + k] = rec[1]; A[4 + k] = rec[2]; A[6 + k] = rec[3];
            }
        }
    }

    double coord(uint32_t prim, int a) const { return a == 0 ? prim_c_[prim].x : (a == 1 ? prim_c_[prim].y : prim_c_[prim].z); }

    // Binary build over order_[first, first+count): binned SAH on the centroids (16 bins x 3 axes); median split on the widest
    // centroid axis when the SAH degenerates or the tree gets deep (bounded depth); halves by index when all centroids coincide.
    int build(uint32_t first, uint32_t count, int depth) {
        const int me = (int)bin_.size();
        bin_.emplace_back();
        Box box, cbox;
        for (uint32_t t = first; t < first + count; ++t) {
            const uint32_t p = order_[t];
            box.grow(prim_box_[p]);
            const double c[3] = {prim_c_[p].x, prim_c_[p].y, prim_c_[p].z};
            cbox.grow_pt(c);
        }
        bin_[me].box = box; bin_[me].first = first; bin_[me].count = count;
        if (count <= (uint32_t)kLeafK) return me;
        constexpr int NB = 16;
        double best = INFINITY; int best_axis = -1, best_bin = -1;
        if (depth < sah_limit_) {
            // one pass over the primitives fills the bins of all three axes
            Box bb[3][NB]; uint32_t bc[3][NB] = {{0}};
            double lo3[3], scale3[3]; bool use[3];
            for (int a = 0; a < 3; ++a) {
                const double ext = cbox.hi[a] - cbox.lo[a];
                use[a] = ext > 0; lo3[a] = cbox.lo[a]; scale3[a] = use[a] ? ext : 1.0;
            }
            for (uint32_t t = first; t < first + count; ++t) {
                const uint32_t p = order_[t];
                const Box& pb = prim_box_[p];
                const double c[3] = {prim_c_[p].x, prim_c_[p].y, prim_c_[p].z};
                for (int a = 0; a < 3; ++a) {
                    if (!use[a]) continue;
                    int bi = (int)((c[a] - lo3[a]) / scale3[a] * NB);
                    bi = bi < 0 ? 0 : (bi >= NB ? NB - 1 : bi);
                    bb[a][bi].grow(pb); ++bc[a][bi];
                }
            }
            for (int a = 0; a < 3; ++a) {
                if (!use[a]) continue;
                double ra[NB]; uint32_t rc[NB];
                Box acc; uint32_t cnt = 0;
                for (int bi = NB - 1; bi > 0; --bi) { acc.grow(bb[a][bi]); cnt += bc[a][bi]; ra[bi] = acc.area(); rc[bi] = cnt; }
                acc = Box(); cnt = 0;
                for (int bi = 0; bi + 1 < NB; ++bi) {
                    acc.grow(bb[a][bi]); cnt += bc[a][bi];
                    if (cnt == 0 || rc[bi + 1] == 0) continue;
                    // leaves hold kLeafK slots: cost counts slot blocks, which favours full leaves
                    const double cost = acc.area() * std::ceil(cnt / (double)kLeafK) + ra[bi + 1] * std::ceil(rc[bi + 1] / (double)kLeafK);
                    if (cost < best) { best = cost; best_axis = a; best_bin = bi; }
                }
            }
        }
        uint32_t mid = first;
        if (best_axis >= 0) {
            const double lo = cbox.lo[best_axis], ext = cbox.hi[best_axis] - cbox.lo[best_axis];
            auto it = std::partition(order_.begin() + first, order_.begin() + first + count, [&](uint32_t p) {
                int b = (int)((coord(p, best_axis) - lo) / ext * NB);
                b = b < 0 ? 0 : (b >= NB ? NB - 1 : b);
                return b <= best_bin;
            });
            mid = (uint32_t)(it - order_.begin());
        }
        if (mid == first || mid == first + count) {   // degenerate: median on the widest centroid axis, ties by index
            int ax = 0;
            for (int a = 1; a < 3; ++a) if (cbox.hi[a] - cbox.lo[a] > cbox.hi[ax] - cbox.lo[ax]) ax = a;
            mid = first + count / 2;
            std::nth_element(order_.begin() + first, order_.begin() + mid, order_.begin() + first + count, [&](uint32_t x, uint32_t y) {
                const double cx = coord(x, ax), cy = coord(y, ax);
                return cx < cy || (cx == cy && x < y);
            });
        }
        const int l = build(first, mid - first, depth + 1);
        const int r = build(mid, first + count - mid, depth + 1);
        bin_[me].left = l; bin_[me].right = r;
        return me;
    }

    uint32_t emit_leaf(const BinNode& b) {
        const uint32_t leaf = (uint32_t)(R_.leaf_id.size() / kLeafK);
        R_.leaf_rec.resize(R_.leaf_rec.size() + (size_t)kLeafK * 4, 0.f);
        R_.leaf_id.resize(R_.leaf_id.size() + kLeafK, 0xffffffffu);
        float* rec = &R_.leaf_rec[(size_t)leaf * kLeafK * 4];
        uint32_t* ids = &R_.leaf_id[(size_t)leaf * kLeafK];
        // members in increasing ORIGINAL index (not required for correctness; keeps the layout deterministic)
        uint32_t mem[kLeafK];
        const int n_mem = (int)b.count;
        for (int t = 0; t < n_mem; ++t) mem[t] = prim_id_[order_[b.first + (uint32_t)t]];
        std::sort(mem, mem + n_mem);
        for (int j = 0; j < kLeafK; ++j) {
            float r4[4] = {0.f, 0.f, 0.f, -INFINITY};   // padding slot: never hit
            if (j < n_mem) {
                const rt_sphere& sp = s_->spheres[mem[j]];
                if (!sphere_record(sp.center.x - R_.g[0], sp.center.y - R_.g[1], sp.center.z - R_.g[2], sp.radius * sp.radius, r4)) {
                    r4[0] = r4[1] = r4[2] = 0.f; r4[3] = INFINITY;
                }
                ids[j] = mem[j];
            }
            float* A = rec + (size_t)(j / 2) * 8; const int kk = j & 1;
            A[0 + kk] = r4[0]; A[2 + kk] = r4[1]; A[4 + kk] = r4[2]; A[6 + kk] = r4[3];
        }
        return leaf;
    }

    // Collapse the binary tree under `b` into one 8-wide node (largest-area inner child expanded first) and recurse.
    uint32_t emit_wide(int b, uint32_t level) {
        R_.depth = std::max(R_.depth, level);
        const uint32_t me = (uint32_t)(R_.nodes.size() / kNodeFloats);
        R_.nodes.resize(R_.nodes.size() + kNodeFloats, 0.f);
        std::vector<int> kids;
        if (bin_[b].left < 0) kids.push_back(b);   // the whole tree is one leaf
        else { kids.push_back(bin_[b].left); kids.push_back(bin_[b].right); }
        // Largest-area-first expansion gives the tightest nodes but only guarantees ONE binary level per wide level on a path.
        // From wide level kAreaFirstLevels on, every inner child is expanded twice instead (2 -> 4 -> 8 children): three binary
        // levels per wide level on every path, so with a binary depth <= 30 the wide depth is <= 15 + ceil(16/3) = 21 = kMaxDepth
        // whatever the input (real scenes stay far below level 15: cover 3, 10 k spheres 4, 100 k spheres 6).
        if ((int)level >= area_levels_) {
            for (int round = 0; round < 2; ++round) {
                std::vector<int> next;
                for (int k : kids) {
                    if (bin_[k].left < 0) next.push_back(k);
                    else { next.push_back(bin_[k].left); next.push_back(bin_[k].right); }
                }
                kids.swap(next);
            }
        }
        while ((int)level < area_levels_ && (int)kids.size() < kWide) {
            int pick = -1; double pa = -1.0;
            for (int i = 0; i < (int)kids.size(); ++i) {
                const BinNode& c = bin_[kids[i]];
                if (c.left < 0) continue;
                const double a = c.box.area();
                if (a > pa) { pa = a; pick = i; }
            }
            if (pick < 0) break;
            const int c = kids[pick];
            kids[pick] = bin_[c].left;
            kids.push_back(bin_[c].right);
        }
        for (int i = 0; i < kWide; ++i) {
            float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};   // empty slot: never hit
            uint32_t ref = kEmptyChild;
            if (i < (int)kids.size()) {
                const BinNode& c = bin_[kids[i]];
                double bmax = 0.0;
                for (int a = 0; a < 3; ++a) bmax = std::max(bmax, std::max(std::fabs(c.box.lo[a]), std::fabs(c.box.hi[a])));
                const double m = 32.0 * kU * bmax + 1e-30;   // DESIGN.md §4.2: covers the f32 rounding of the slab test on the box's side
                for (int a = 0; a < 3; ++a) { lo[a] = f32_down(c.box.lo[a] - m); hi[a] = f32_up(c.box.hi[a] + m); }
                if (c.left < 0) ref = kLeafBit | emit_leaf(c);
                else ref = emit_wide(kids[i], level + 1);
            }
            float* N = &R_.nodes[(size_t)me * kNodeFloats];   // re-fetch: the vector may have grown
            for (int a = 0; a < 3; ++a) { N[a * 8 + i] = lo[a]; N[24 + a * 8 + i] = hi[a]; }
            std::memcpy(&N[48 + i], &ref, 4);
        }
        return me;
    }
};

// want_tree = false: only the flat records / exact geometry / materials (RT_VARIANT_EXACT_F64, RT_VARIANT_BRUTE_FORCE).
inline void build_records(const rt_scene* s, bool want_tree, Records& R) {
    Builder b(s, R);
    b.run(want_tree);
}

}  // namespace rtbvh
