// dev_traverse.cuh — device scene layout, ray/box/primitive tests and the three
// BVH traversals of the reference, restated as iterative stack traversals.
//
// HBM layout (all read-only during a frame, L2/L1 resident: ~0.6 MB for the bunny):
//   nodes  float4[2*n_nodes]   record i = {pMin.xyz, link} {pMax.xyz, pad}; sibling
//                              pairs adjacent and 64-byte aligned (one 2x LDG.128 per box)
//   geom   float4[3*n_prims]   triangle: {v0.xyz, radius=0} {E1.xyz, 1-alpha} {E2.xyz, flags}
//                              sphere:   {c.xyz,  radius  } {0,      1-alpha} {0,      flags}
//                              (E1 = v1-v0, E2 = v2-v0: the same subtractions Triangle.hpp:22-23 does)
// Primitive index == depth-first leaf rank, so BVH.hpp:157's "left subtree wins
// ties" is "smaller primitive index wins".
#pragma once
#include "dev_math.cuh"
#include "prune_rule.h"
#include "wide_bvh.h"
#include "shadow_assoc.h"
#include "../../../include/wrt_scene.h"

namespace wrt {

#define WRT_INLINE_LIGHTS 4

struct DevScene {
    const float4* nodes;      // reference-topology tree (host-built, BVH.hpp:49-125)
    const float4* fnodes;     // SAH tree over the same leaf boxes (fast_bvh.hpp), same record layout
    const float4* onodes;     // 8 copies of the SAH tree, one per ray-direction octant, whose records hold
                              // {near planes, link}{far planes, pad}: the reference's swap-on-negative-direction
                              // (BoundBox.hpp:68-70) is done once at upload instead of at every box
    const float4* ronodes;    // the same 8 octant copies of the reference-topology tree (axis-degenerate rays)
    const float4* wnodes;     // 4-wide view of each octant copy of the SAH tree (wide_bvh.h): node of pair c at float4 4*c
    const float4* dnodes;     // the SAH tree with every box dilated: conservative culling for the box-free
                              // directional-shadow loop (Renderer.hpp:381-400)
    const float4* geom;
    const float4* prim_box;   // per prim {pMin.xyz, 0} {pMax.xyz, 0}: the primitive's own (leaf) box, for the occluder cache
    const float4* tri_aux;    // per prim {unit plane normal, |E1|+|E2|} (w < 0: do not filter): ray-independent terms of the
                              // candidate-list pruning (shaft_cull.h wrt_triangle_aux)
    const WrtPathCode* path_codes;   // per prim: its root-to-leaf path in the REFERENCE tree (shadow_assoc.h); nullptr: tree deeper than 64
    const float4* attr;       // per prim 4x float4: {n0,uv0.x} {n1,uv0.y} {n2,uv1.x} {uv1.y,uv2.x,uv2.y,0}
    const int4*   ids;        // per prim {material, texture, normalmap, object}
    const int*    object_prim;
    const float4* materials;  // per material 3x float4: {Od.rgb, ka} {Os.rgb, kd} {ks, n, alpha, eta}
    const WrtLight* lights;
    WrtLight lights_c[WRT_INLINE_LIGHTS];   // the first lights again, in the kernel-parameter constant bank
    const WrtTexture* textures;
    const WrtTexture* normalmaps;
    const float* texels;
    int n_nodes, n_prims, n_lights, n_point_lights, n_dir_lights;
    int has_light_prims;      // any WRT_PRIM_LIGHT primitive in the scene
    int shadow_type, depth_cueing;
    float bkg[3], eta;
    float dc[3], amin, amax, distmin, distmax;
    float eye[3];
    float prune_slack;        // max over the triangles of how far outside its box an accepted hit can lie (prune_rule.h)
};

struct Ray {
    f3 o, d;
    f3 inv;                   // 1/d, BoundBox.hpp:55 (hoisted: same value at every node)
};

__device__ __forceinline__ Ray make_ray(f3 o, f3 d) {
    Ray r;
    r.o = o; r.d = d;
    r.inv = mk3(1 / d.x, 1 / d.y, 1 / d.z);
    return r;
}

// BoundBox::IntersectRay, BoundBox.hpp:53-85.  The swap-on-negative-direction is
// done by selecting which plane feeds tmin/tmax: identical values, no extra ops.
__device__ __forceinline__ bool slab(const float4 lo, const float4 hi, const Ray& r, float& t_enter) {
    float ax = (lo.x - r.o.x) * r.inv.x, bx = (hi.x - r.o.x) * r.inv.x;
    float ay = (lo.y - r.o.y) * r.inv.y, by = (hi.y - r.o.y) * r.inv.y;
    float az = (lo.z - r.o.z) * r.inv.z, bz = (hi.z - r.o.z) * r.inv.z;
    bool sx = r.d.x < 0, sy = r.d.y < 0, sz = r.d.z < 0;
    float tmin_x = sx ? bx : ax, tmax_x = sx ? ax : bx;
    float tmin_y = sy ? by : ay, tmax_y = sy ? ay : by;
    float tmin_z = sz ? bz : az, tmax_z = sz ? az : bz;
    t_enter = fmaxf(tmin_x, fmaxf(tmin_y, tmin_z));
    float t_exit = fminf(tmax_x, fminf(tmax_y, tmax_z));
    return (t_enter <= t_exit) && (t_exit >= 0);
}

// The same test on a record of the octant tree: `lo` holds the planes the ray enters through and
// `hi` the planes it leaves through, so tmin/tmax need no selection.  Identical values, identical
// result; 6 selects and 3 sign tests fewer per box.
__device__ __forceinline__ bool slab_presorted(const float4 nearp, const float4 farp, const Ray& r, float& t_enter) {
    float tmin_x = (nearp.x - r.o.x) * r.inv.x, tmax_x = (farp.x - r.o.x) * r.inv.x;
    float tmin_y = (nearp.y - r.o.y) * r.inv.y, tmax_y = (farp.y - r.o.y) * r.inv.y;
    float tmin_z = (nearp.z - r.o.z) * r.inv.z, tmax_z = (farp.z - r.o.z) * r.inv.z;
    t_enter = fmaxf(tmin_x, fmaxf(tmin_y, tmin_z));
    float t_exit = fminf(tmax_x, fminf(tmax_y, tmax_z));
    return (t_enter <= t_exit) && (t_exit >= 0);
}
__device__ __forceinline__ int ray_octant(f3 d) { return (d.x < 0 ? 1 : 0) | (d.y < 0 ? 2 : 0) | (d.z < 0 ? 4 : 0); }

struct PrimHit {
    float t, u, v;            // u,v = barycentric b1,b2 (triangles only)
};

// Triangle::intersect acceptance test, Triangle.hpp:22-41
__device__ __forceinline__ bool tri_test(const float4 A, const float4 B, const float4 C, const Ray& r, PrimHit& h) {
    f3 v0 = mk3(A), E1 = mk3(B), E2 = mk3(C);
    f3 S = r.o - v0;
    f3 S1 = cross(r.d, E2);
    f3 S2 = cross(S, E1);
    float rx = dot(S2, E2), ry = dot(S1, S), rz = dot(S2, r.d);
    float left = 1.0f / dot(S1, E1);
    float t = rx * left, u = ry * left, v = rz * left;
    const float EPS = 0.00001f;
    if (t + EPS > 0 && 1 - u - v + EPS > 0 && u + EPS > 0 && v + EPS > 0) {
        h.t = t; h.u = u; h.v = v;
        return true;
    }
    return false;
}

// Sphere::intersect root selection, Sphere.hpp:25-47,80-90 + solveQuadratic global.hpp:105-125.
// Out of line (spheres are rare next to triangle meshes) and by value, so that the
// caller's ray stays in registers.  Returns {hit ? 1 : 0, t}.
__device__ __noinline__ float2 sphere_test(float cx, float cy, float cz, float radius, float ox, float oy, float oz,
                                           float dx_, float dy_, float dz_) {
    float Aq = 1.f;
    float Bq = 2 * (dx_ * (ox - cx) + dy_ * (oy - cy) + dz_ * (oz - cz));
    double dx = (double)(ox - cx), dy = (double)(oy - cy), dz = (double)(oz - cz);
    float Cq = (float)(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)),
                                 -(double)(radius * radius)));
    float disc = Bq * Bq - 4 * Aq * Cq;
    float t1, t2;
    if (disc < 0) { t1 = FLT_MAX; t2 = FLT_MAX; }
    else if (disc == 0) { t1 = (-Bq + sqrtf(disc)) / 2 * Aq; t2 = t1; }
    else { t1 = (-Bq + sqrtf(disc)) / 2 * Aq; t2 = (-Bq - sqrtf(disc)) / 2 * Aq; }
    if (t1 > t2) { float s = t1; t1 = t2; t2 = s; }
    float t;
    if (float_equal(t1, FLT_MAX) && float_equal(t2, FLT_MAX)) return make_float2(0.f, 0.f);
    else if (float_equal(t1, t2)) {
        if (t1 < 0) return make_float2(0.f, 0.f);
        t = t1;
    } else {
        if (t1 > 0 && t2 > 0) t = t1;
        else if (t1 > 0 && t2 < 0) t = t1;
        else if (t1 < 0 && t2 > 0) t = t2;
        else return make_float2(0.f, 0.f);
    }
    return make_float2(1.f, t);
}

__device__ __forceinline__ bool prim_test(const DevScene& s, int p, const Ray& r, PrimHit& h, float& one_minus_alpha,
                                          unsigned& flags) {
    const float4* g = s.geom + 3 * (size_t)p;
    float4 A = ldg4(g), B = ldg4(g + 1), C = ldg4(g + 2);
    one_minus_alpha = B.w;
    flags = __float_as_uint(C.w);
    if ((flags & WRT_PRIM_KIND_MASK) == WRT_PRIM_SPHERE) {
        float2 sp = sphere_test(A.x, A.y, A.z, A.w, r.o.x, r.o.y, r.o.z, r.d.x, r.d.y, r.d.z);
        h.t = sp.y; h.u = 0.f; h.v = 0.f;
        return sp.x != 0.f;
    }
    return tri_test(A, B, C, r, h);
}

// Per-thread traversal stack in shared memory, column `tid` of a
// [rows][blockDim.x] array (rows = tree depth + 2): consecutive lanes hit consecutive banks.
// (A hybrid stack — the first 8 / 12 / 16 rows in shared memory, deeper ones in a per-thread local array, to give the 88 KB
// L1 the 168 KB carve-out leaves more room — measured slower: closest hit 3.79-3.85 ms against 3.67; profiles/NOTES.md.)
#ifdef WRT_DEBUG_BOUNDS
__device__ unsigned g_wrt_stack_overflow = 0;       // latched by Stack::push in the bounds-checking build
#endif
struct Stack {
    int* base;
    int stride;
    int sp;
#ifdef WRT_DEBUG_BOUNDS
    int rows;
    __device__ __forceinline__ void init(int* smem, int tid, int nthreads) {
        base = smem + tid; stride = nthreads; sp = 0;
        unsigned dyn;
        asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn));
        rows = (int)(dyn / (4u * (unsigned)nthreads));
    }
    __device__ __forceinline__ void push(int v) {
        if (sp >= rows) { atomicExch(&g_wrt_stack_overflow, (unsigned)sp + 1u); return; }
        base[sp * stride] = v; ++sp;
    }
    __device__ __forceinline__ int pop() { --sp; return base[sp * stride]; }
#else
    __device__ __forceinline__ void init(int* smem, int tid, int nthreads) { base = smem + tid; stride = nthreads; sp = 0; }
    __device__ __forceinline__ void push(int v) { base[sp * stride] = v; ++sp; }
    __device__ __forceinline__ int pop() { --sp; return base[sp * stride]; }
#endif
    __device__ __forceinline__ bool empty() const { return sp == 0; }
};

// A ray whose direction has a zero component takes the inf/NaN paths of
// BoundBox::IntersectRay (BoundBox.hpp:55-84), where box inclusion no longer implies
// slab-test inclusion; such rays walk the reference-topology tree exhaustively.
__device__ __forceinline__ bool degenerate_dir(f3 d) { return d.x == 0.f || d.y == 0.f || d.z == 0.f; }

// One traversal step: test the two children of pair `cur`, hand hit leaves to `leaf`,
// descend / push / pop.  Returns false when the walk is over.  `limit`: boxes entered
// beyond it are skipped (FLT_MAX or +inf = never).  NEAR_FIRST orders by entry distance.
template <bool NEAR_FIRST, bool PRESORTED = false, class LeafFn>
__device__ __forceinline__ bool traverse_step(const float4* __restrict__ nodes, const Ray& r, Stack& st, int& cur,
                                              const float& limit, LeafFn&& leaf) {
    const float4* n = nodes + 2 * cur;
    float4 l0, l1, r0, r1;
    ldg8(n, l0, l1);
    ldg8(n + 2, r0, r1);
    float tl, tr;
    bool hl = PRESORTED ? slab_presorted(l0, l1, r, tl) : slab(l0, l1, r, tl);
    bool hr = PRESORTED ? slab_presorted(r0, r1, r, tr) : slab(r0, r1, r, tr);
    hl = hl && !(tl > limit);
    int linkL = __float_as_int(l0.w), linkR = __float_as_int(r0.w);
    if (hl && linkL < 0) { leaf(~linkL); hl = false; }
    hr = hr && !(tr > limit);                      // `limit` may have tightened in leaf()
    if (hr && linkR < 0) { leaf(~linkR); hr = false; }
    if (hl && hr) {
        bool right_first = NEAR_FIRST && (tr < tl);
        int far_link = right_first ? linkL : linkR;
        st.push(far_link);
        cur = right_first ? linkR : linkL;
        return true;
    }
    if (hl) { cur = linkL; return true; }
    if (hr) { cur = linkR; return true; }
    if (st.empty()) return false;
    cur = st.pop();
    return true;
}

// One step over a 4-wide node (wide_bvh.h): the four grandchild records of pair `cur` in one 128-byte block, on a
// presorted octant copy, with DEFERRED leaves.  Testing every hit leaf of a node at once, a lane with two leaf hits runs
// the ~110-instruction intersection code twice while the warp's other lanes wait, and in a warp of ~24 walking lanes
// some lane has a second leaf in nearly every step — so the warp pays two or three rounds of leaf code per node step, the
// later ones with 2-3 lanes.  Here a lane tests at most ONE leaf per step, at one code site: of a node's hits, taken
// nearest first (NEAR_FIRST: the closest-hit walk) or in slot order (the hard-shadow walk), the first leaf goes to the
// lane's leaf slot, the first other hit becomes `cur` (an inner pair, or a leaf link: it is then tested by the next
// step), the rest is pushed far to near — leaf links (< 0) lie on the stack beside pair indices.  A step whose `cur` is
// a leaf link takes it into the leaf slot and visits the pair on top of the stack beside it.  Exactness: every tested
// primitive has had its own box hit by the ray, and the closest-hit result (min t, ties to the smaller primitive index)
// does not depend on the order of the tests; a deferred leaf is tested without its entry distance (a superset of what the
// pruning keeps).
#define WRT_NO_LINK (-2147483647 - 1)      // (also the link of a wide node's empty slot, which no ray reaches)
template <bool NEAR_FIRST, class LeafFn>
__device__ __forceinline__ bool traverse_step4_defer(const float4* __restrict__ wnodes, const Ray& r, Stack& st, int& cur,
                                                     const float& limit, LeafFn&& leaf) {
    const float inf = INFINITY;
    int pend = WRT_NO_LINK;
    float tp = -inf;
    if (cur < 0) {                                         // a deferred leaf
        pend = cur;
        cur = WRT_NO_LINK;
        if (!st.empty()) {
            const int nx = st.pop();
            if (nx >= 0) cur = nx; else ++st.sp;           // a pair: visit it in this step; another leaf: leave it there
        }
    }
    if (cur >= 0) {
        const float4* n = wnodes + WRT_WIDE_FLOAT4_PER_RECORD * (size_t)cur;
        float4 a0, a1, b0, b1, c0, c1, d0, d1;
        ldg8(n, a0, a1);
        ldg8(n + 2, b0, b1);
        ldg8(n + 4, c0, c1);
        ldg8(n + 6, d0, d1);
        float t0, t1, t2, t3;
        const bool h0 = slab_presorted(a0, a1, r, t0), h1 = slab_presorted(b0, b1, r, t1);
        const bool h2 = slab_presorted(c0, c1, r, t2), h3 = slab_presorted(d0, d1, r, t3);
        int l0 = __float_as_int(a0.w), l1 = __float_as_int(b0.w), l2 = __float_as_int(c0.w), l3 = __float_as_int(d0.w);
        float k0 = (h0 && !(t0 > limit)) ? t0 : inf, k1 = (h1 && !(t1 > limit)) ? t1 : inf;
        float k2 = (h2 && !(t2 > limit)) ? t2 : inf, k3 = (h3 && !(t3 > limit)) ? t3 : inf;
#define WRT_CSWAP(ka, la, kb, lb) { const bool sw = kb < ka; const float kt = sw ? ka : kb; ka = sw ? kb : ka; kb = kt; const int lt = sw ? la : lb; la = sw ? lb : la; lb = lt; }
        if (NEAR_FIRST) { WRT_CSWAP(k0, l0, k1, l1) WRT_CSWAP(k2, l2, k3, l3) WRT_CSWAP(k0, l0, k2, l2) WRT_CSWAP(k1, l1, k3, l3) WRT_CSWAP(k1, l1, k2, l2) }
#undef WRT_CSWAP
        if (NEAR_FIRST) {
            // sorted: the hits are k0 <= k1 <= ..., misses (+inf) last.  Only the NEAREST hit may go to the leaf slot; a leaf
            // further back becomes `cur` or waits on the stack like a pair (a third of the bookkeeping instructions of the
            // general rule below)
            const bool tk = (k0 < inf) && (l0 < 0) && (pend == WRT_NO_LINK);
            if (tk) { pend = l0; tp = k0; }
            const float kc = tk ? k1 : k0;
            const int lc = tk ? l1 : l0;
            cur = kc < inf ? lc : WRT_NO_LINK;
            if (k3 < inf) st.push(l3);
            if (k2 < inf) st.push(l2);
            if (!tk && k1 < inf) st.push(l1);
        } else {
            bool have_p = pend != WRT_NO_LINK, have_c = false;
            cur = WRT_NO_LINK;
            // in slot order: leaf slot, then `cur`, the others wait on the stack
#define WRT_TAKE(kj, lj, pushj)                                                                    \
            bool pushj = false;                                                                    \
            if (kj < inf) {                                                                        \
                if (lj < 0 && !have_p) { pend = lj; tp = kj; have_p = true; }                      \
                else if (!have_c) { cur = lj; have_c = true; }                                     \
                else pushj = true;                                                                 \
            }
            WRT_TAKE(k0, l0, p0) WRT_TAKE(k1, l1, p1) WRT_TAKE(k2, l2, p2) WRT_TAKE(k3, l3, p3)
#undef WRT_TAKE
            (void)p0;                                          // the first hit always finds a free place
            if (p3) st.push(l3);
            if (p2) st.push(l2);
            if (p1) st.push(l1);
        }
    }
    // (Taking the next node from the stack BEFORE the leaf test and prefetching its line to L1 meanwhile: closest hit 3.68 ->
    // 3.64 ms, hard shadows 3.86 -> 3.82 — with ~1000 lanes per SM each prefetching its own 128-byte line, 131 KB of lines
    // compete for the 88 KB of L1 the stacks leave.  Not kept.)
    if (pend != WRT_NO_LINK && !(tp > limit)) leaf(~pend);
    if (cur == WRT_NO_LINK) {
        if (st.empty()) return false;
        cur = st.pop();
    }
    return true;
}

struct Closest {
    float t; int prim; float u, v;
};

// ---- closest hit: getIntersection, BVH.hpp:137-159 ----
// Minimum t over every primitive whose own box and intersection test pass; ties go to the
// smaller reference DFS rank (the left subtree of BVH.hpp:157).  With prune_scale >= 0 a box
// entered beyond wrt_prune_limit(best_t, prune_scale) is skipped (prune_rule.h: why no primitive
// inside it can be accepted with a smaller t; prune_scale is the ray's own part of the margin).
// prune_scale < 0 visits every hit box like the reference does.
struct ClosestState {
    Closest best;
    float limit;
    float prune_scale;
    __device__ __forceinline__ void reset(float prune) {
        best.t = FLT_MAX; best.prim = -1; best.u = 0.f; best.v = 0.f;
        limit = FLT_MAX; prune_scale = prune;
    }
    // pruning on (prune_cfg >= 0): the margin of this ray; off: -1
    __device__ __forceinline__ void set_ray(const DevScene& s, const Ray& r, float prune_cfg) {
        const float o[3] = {r.o.x, r.o.y, r.o.z}, inv[3] = {r.inv.x, r.inv.y, r.inv.z};
        prune_scale = prune_cfg >= 0.f ? wrt_prune_ray_scale(o, inv, s.prune_slack) : -1.f;
    }
    __device__ __forceinline__ void leaf(const DevScene& s, const Ray& r, int p) {
        PrimHit h; float oma; unsigned fl;
        if (prim_test(s, p, r, h, oma, fl)) {
            if (h.t < best.t || (h.t == best.t && p < best.prim)) {
                best.t = h.t; best.prim = p; best.u = h.u; best.v = h.v;
                if (prune_scale >= 0.f) limit = wrt_prune_limit(h.t, prune_scale);
            }
        }
    }
    // returns true when a traversal starting at pair `cur` is needed
    __device__ __forceinline__ bool begin(const DevScene& s, const float4* nodes, int root, const Ray& r, int& cur) {
        float te;
        float4 lo = ldg4(nodes + 2 * root), hi = ldg4(nodes + 2 * root + 1);
        if (!slab(lo, hi, r, te)) return false;
        int link = __float_as_int(lo.w);
        if (link < 0) { leaf(s, r, ~link); return false; }
        cur = link;
        return true;
    }
};

// Whole closest-hit query in one call (batch kernels, literal hasIntersection path).
__device__ __forceinline__ Closest closest_hit(const DevScene& s, const float4* nodes, int root, const Ray& r, Stack& st,
                                               float prune_rel) {
    ClosestState cs;
    cs.reset(prune_rel);
    cs.set_ray(s, r, prune_rel);
    int cur = 0;
    st.sp = 0;
    if (cs.begin(s, nodes, root, r, cur)) {
        while (traverse_step<true>(nodes, r, st, cur, cs.limit, [&](int p) { cs.leaf(s, r, p); })) {}
    }
    return cs.best;
}

// Tree and pruning a ray uses: the SAH tree with pruning, unless the caller asked for the
// reference's literal exhaustive walk or the ray is axis-degenerate.
__device__ __forceinline__ const float4* pick_tree(const DevScene& s, f3 dir, float& prune_rel) {
    if (prune_rel < 0.f || degenerate_dir(dir)) { prune_rel = -1.f; return s.nodes; }
    return s.fnodes;
}

// ---- hard shadow: BVHStrategy::ShadowHelper, BVHStrategy.hpp:24-48 ----
// Product of (1-alpha) over every tested primitive hit with t < dis that is not a light avatar; the walk stops once
// the product is exactly 0 (0 * x == 0 for finite x).  The reference multiplies in the association of ITS tree (`l * r`), a
// stack walk in visit order: the same bits for up to two factors != 1, not beyond (shadow_assoc.h).  ShadowAcc therefore
// keeps the blocking primitives whose factor is not 1; a ray with three or more of them gets its product from
// wrt_tree_product — the reference's association, rebuilt from the primitives' path codes — so the coefficient is the
// reference's bit for bit.  (More than WRT_SHADOW_HITS such crossings on one ray, or a reference tree deeper than 64: the
// visit-order product, within a few ulp.)
struct ShadowAcc {
    float res;
    int n;                                 // blocking primitives with a factor != 1 so far
    int prim[WRT_SHADOW_HITS];
    float fac[WRT_SHADOW_HITS];
    WrtPathCode code[WRT_SHADOW_HITS];     // fetched when the hit is made: the load is long back when the walk ends
    __device__ __forceinline__ void reset() { res = 1.f; n = 0; }
    // (counting only on the first walk and walking rays with three or more translucent crossings a second time measured
    // 10 % slower than keeping every such hit: profiles/NOTES.md)
    __device__ __forceinline__ void add(int p, float f, const WrtPathCode* codes) {
        res = res * f;
        if (f != 1.f && f != 0.f) {            // (an opaque blocker ends the walk with an exact 0: nothing to associate)
            if (n < WRT_SHADOW_HITS) {
                prim[n] = p; fac[n] = f;
                if (codes) {
                    const int4 c4 = __ldg(reinterpret_cast<const int4*>(codes + p));
                    code[n].hi = (unsigned)c4.x; code[n].lo = (unsigned)c4.y; code[n].depth = c4.z; code[n].pad = 0;
                }
            }
            ++n;
        }
    }
    __device__ __forceinline__ bool needs_tree(const WrtPathCode* codes) const {
        return res != 0.f && n >= 3 && n <= WRT_SHADOW_HITS && codes != nullptr;
    }
};

// (out of line: one ray in ten of a glass-bunny frame, a few dozen instructions of sort + reduction on local arrays)
__device__ __noinline__ float shadow_tree_value(const int* prim, const float* fac, const WrtPathCode* code, int n) {
    int idx[WRT_SHADOW_HITS];
    float fs[WRT_SHADOW_HITS];
    for (int i = 0; i < n; i++) {          // insertion sort by primitive index = the reference tree's leaf order
        const int key = prim[i];
        int k = i;
        while (k > 0 && prim[idx[k - 1]] > key) { idx[k] = idx[k - 1]; --k; }
        idx[k] = i;
    }
    for (int i = 0; i < n; i++) fs[i] = fac[idx[i]];
    return wrt_tree_product(n, idx, fs, code);             // (codes are looked up as code[idx[i]]: the hits' own copies)
}

__device__ __forceinline__ float shadow_value(const DevScene& s, const ShadowAcc& acc) {
    return acc.needs_tree(s.path_codes) ? shadow_tree_value(acc.prim, acc.fac, acc.code, acc.n) : acc.res;
}

__device__ __forceinline__ void shadow_leaf(const DevScene& s, const Ray& r, float dis, int p, ShadowAcc& acc) {
    PrimHit h; float oma; unsigned fl;
    if (prim_test(s, p, r, h, oma, fl) && h.t < dis && !(fl & WRT_PRIM_LIGHT)) acc.add(p, oma, s.path_codes);
}

__device__ __forceinline__ float shadow_product(const DevScene& s, const float4* nodes, const Ray& r, float dis, Stack& st) {
    ShadowAcc acc;
    acc.reset();
    if (s.n_nodes == 0) return acc.res;
    float te;
    float4 lo = ldg4(nodes), hi = ldg4(nodes + 1);
    if (!slab(lo, hi, r, te)) return acc.res;
    int cur = __float_as_int(lo.w);
    if (cur < 0) { shadow_leaf(s, r, dis, ~cur, acc); return acc.res; }
    st.sp = 0;
    const float never = INFINITY;
    while (acc.res != 0.f && traverse_step<false>(nodes, r, st, cur, never, [&](int p) { shadow_leaf(s, r, dis, p, acc); })) {}
    return shadow_value(s, acc);
}

// ---- soft-shadow visibility: hasIntersection, BVH.hpp:162-186 ----
// No root-box test.  The reference takes the CLOSEST hit of each root child and calls the
// ray occluded when that hit has t < dis and is not a light avatar.  Without light-avatar
// primitives this is "some tested primitive is hit with t < dis" (the closest hit is < dis
// iff some hit is), an early-out any-hit walk; with light avatars the two per-child
// closest-hit queries are done literally on the reference tree.
__device__ __noinline__ bool occluded_literal(const DevScene& s, const Ray r, float dis, Stack& st) {
    int root_link = __float_as_int(ldg4(s.nodes).w);
    for (int k = 0; k < 2; k++) {
        Closest a = closest_hit(s, s.nodes, root_link + k, r, st, -1.f);
        if (a.prim >= 0 && a.t < dis && !(__float_as_uint(ldg4(s.geom + 3 * (size_t)a.prim + 2).w) & WRT_PRIM_LIGHT))
            return true;
    }
    return false;
}

// returns true when an any-hit walk from pair `cur` is needed; otherwise `occ` is final
__device__ __forceinline__ bool occluded_begin(const DevScene& s, const float4* nodes, const Ray& r, float dis, Stack& st,
                                               int& cur, bool& occ) {
    occ = false;
    if (s.n_nodes == 0) return false;
    int root_link = __float_as_int(ldg4(nodes).w);
    if (root_link < 0) {
        PrimHit h; float oma; unsigned fl;
        // (the reference dereferences a null obj here when the lone primitive is missed)
        if (prim_test(s, ~root_link, r, h, oma, fl) && !(fl & WRT_PRIM_LIGHT)) occ = h.t < dis;
        return false;
    }
    if (s.has_light_prims) { occ = occluded_literal(s, r, dis, st); return false; }
    cur = root_link;
    return true;
}

__device__ __forceinline__ void occluded_leaf(const DevScene& s, const Ray& r, float dis, int p, bool& occ) {
    PrimHit h; float oma; unsigned fl;
    if (prim_test(s, p, r, h, oma, fl) && h.t < dis) occ = true;
}

// Occluder cache: the primitive that blocked this lane's previous shadow ray is tried first.  The
// any-hit answer is an OR over primitives of (own box hit && intersection accepted && t < dis), so
// testing one of them early is only a reordering; the own-box test keeps the predicate exact.
__device__ __forceinline__ bool occluder_cache_hit(const DevScene& s, const Ray& r, float dis, int p) {
    float te;
    float4 blo, bhi;
    ldg8(s.prim_box + 2 * (size_t)p, blo, bhi);
    if (!slab(blo, bhi, r, te)) return false;
    PrimHit h; float oma; unsigned fl;
    return prim_test(s, p, r, h, oma, fl) && h.t < dis;
}

__device__ __forceinline__ bool occluded(const DevScene& s, const float4* nodes, const Ray& r, float dis, Stack& st) {
    bool occ;
    int cur = 0;
    st.sp = 0;
    if (occluded_begin(s, nodes, r, dis, st, cur, occ)) {
        const float never = INFINITY;
        while (!occ && traverse_step<true>(nodes, r, st, cur, never, [&](int p) { occluded_leaf(s, r, dis, p, occ); })) {}
    }
    return occ;
}

// Renderer::getShadowCoeffi(Intersection&, Vector4f&), Renderer.hpp:381-400: every
// object in objList order, skipping self and light avatars; no distance bound, NO boxes.
// Brute-force form, literally the reference's loop.
__device__ __forceinline__ float directional_product(const DevScene& s, const Ray& r, int self_prim) {
    float res = 1.f;
    for (int k = 0; k < s.n_prims; k++) {
        int p = __ldg(s.object_prim + k);
        if (p == self_prim) continue;
        PrimHit h; float oma; unsigned fl;
        const float4* g = s.geom + 3 * (size_t)p;
        if (__float_as_uint(ldg4(g + 2).w) & WRT_PRIM_LIGHT) continue;
        if (prim_test(s, p, r, h, oma, fl)) res = res * oma;
        if (res == 0.f) break;
    }
    return res;
}

// The same product through the dilated tree.  The reference tests every object, so culling must
// never drop a primitive its intersection routine would accept: leaf boxes are dilated on the host
// by 1e-3 of their size (100x the 1e-5 barycentric / distance slack of Triangle.hpp:41) plus an
// absolute pad, and -0 direction components are turned into +0 so a ray inside a slab is never
// culled by the inf/NaN paths.  Accepted hits are multiplied in objList order, like the loop:
// factors are collected (sorted by object index) and multiplied at the end; an exact 0 factor ends
// the walk at once (0 * finite == 0 in any order).  More than WRT_DIR_HITS translucent hits on one
// ray fall back to the literal loop.
#define WRT_DIR_HITS 8
__device__ __forceinline__ float directional_product_bvh(const DevScene& s, const Ray& r, int self_prim, Stack& st) {
    if (s.n_nodes == 0) return 1.f;
    Ray c = r;                                     // culling ray: +0 instead of -0 components
    c.d = mk3(r.d.x + 0.f, r.d.y + 0.f, r.d.z + 0.f);
    c.inv = mk3(1 / c.d.x, 1 / c.d.y, 1 / c.d.z);
    int objs[WRT_DIR_HITS] = {0};
    float facs[WRT_DIR_HITS] = {0.f};
    int nh = 0;
    bool zero = false, overflow = false;
    auto leaf = [&](int p) {
        if (p == self_prim) return;
        PrimHit h; float oma; unsigned fl;
        if (!prim_test(s, p, r, h, oma, fl) || (fl & WRT_PRIM_LIGHT)) return;
        if (oma == 0.f) { zero = true; return; }
        if (nh == WRT_DIR_HITS) { overflow = true; return; }
        int obj = __ldg(s.ids + p).w;
        int k = nh++;
        while (k > 0 && objs[k - 1] > obj) { objs[k] = objs[k - 1]; facs[k] = facs[k - 1]; --k; }
        objs[k] = obj; facs[k] = oma;
    };
    float te;
    float4 lo = ldg4(s.dnodes), hi = ldg4(s.dnodes + 1);
    if (slab(lo, hi, c, te)) {
        int cur = __float_as_int(lo.w);
        if (cur < 0) leaf(~cur);
        else {
            st.sp = 0;
            const float never = INFINITY;
            while (!(zero || overflow) && traverse_step<false>(s.dnodes, c, st, cur, never, leaf)) {}
        }
    }
    if (zero) return 0.f;
    if (overflow) return directional_product(s, r, self_prim);
    float res = 1.f;
    for (int k = 0; k < nh; k++) res = res * facs[k];
    return res;
}

// ---- persistent warps with per-lane refill ----
// A warp keeps pulling work items from a global counter; a lane that finishes its ray
// goes idle, and once `refill` lanes are idle the warp fetches that many new items in one
// atomic.  Deep ray-tree levels hold rays of wildly different traversal lengths (a
// reflection that escapes to the background next to a refraction bouncing inside the
// bunny); refilling keeps the SIMD lanes occupied where fixed 32-ray batches do not.
// Q provides: bool begin(item, cur, st)  — load + start; false = resolved without a walk
//             bool step(cur, st)         — one traversal step; false = finished
//             bool finish(cur, st)       — a walk ended: write results, or start the item's next
//                                          walk and return true
#define WRT_STEPS_PER_ROUND 4      // traversal steps between two looks at the warp's idle lanes (the deep closest-hit levels: 8)
#define WRT_CHUNK_MIN_PER 256

template <class Q, int STEPS = WRT_STEPS_PER_ROUND>
__device__ __forceinline__ void run_queue(Q& q, unsigned long long n, unsigned long long* work, Stack& st, int refill_cfg) {
    const int refill = refill_cfg & 0xff;
    const unsigned chunk_div = (unsigned)(refill_cfg >> 8);     // 0: one claim per refill; k: chunks of n / (warps * k)

    const unsigned lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    // Work is claimed from the global counter in chunks and handed out to idle lanes from the warp's
    // private range: one atomic per `chunk` items instead of one per refill.  (ncu, v5: 27 % of the
    // level-0 stall samples sat on the SHFL behind this atomic — 13 M single-address atomics per frame.)

    unsigned long long warps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    unsigned long long per = chunk_div ? n / (warps * (unsigned long long)chunk_div) : 0;
    // Short queues claim exactly what a refill needs (A/B on one rank's 1/8 share of the 4K frame:
    // 6.5 ms vs 7.1 ms with chunks — chunk tails dominate there); long ones claim 256 items at a time
    // (full frame: 45.1 ms vs 47.7 ms without chunks — the claim atomic was the limiter).
    const bool chunked = per >= (unsigned long long)WRT_CHUNK_MIN_PER;
    unsigned long long loc_next = 0, loc_end = 0;      // warp-uniform private range
    bool active = false, drained = false;
    int cur = 0;
    while (true) {
        const unsigned idle = __ballot_sync(0xffffffffu, !active);
        if (!drained && (idle == 0xffffffffu || __popc(idle) >= refill)) {
            {
                unsigned cnt = __popc(idle);
                unsigned long long avail = loc_end - loc_next;
                unsigned long long first = loc_next, second = 0;   // items [first, first+avail) then [second, ...)
                if (avail < cnt) {
                    unsigned long long base = 0;
                    const unsigned claim = chunked ? 256u : cnt - (unsigned)avail;
                    if (lane == 0) base = atomicAdd(work, (unsigned long long)claim);
                    base = __shfl_sync(0xffffffffu, base, 0);
                    second = base;
                    loc_next = base + (cnt - avail);
                    loc_end = base + claim;
                    if (base >= n) drained = true;           // nothing left behind this chunk either
                } else {
                    loc_next += cnt;
                }
                if (!active) {
                    unsigned k = __popc(idle & lt_mask);
                    unsigned long long item = k < avail ? first + k : second + (k - avail);
                    if (item < n) {
                        st.sp = 0;
                        active = q.begin(item, cur, st);
                        while (!active && q.finish(cur, st)) active = true;
                    }
                }
                if (loc_next >= n) drained = true;
            }
            if (!__any_sync(0xffffffffu, active)) {
                if (drained) break;
                continue;
            }
        } else if (idle == 0xffffffffu) {
            break;                                   // drained and nothing in flight
        }
#pragma unroll 1
        for (int k = 0; k < STEPS; k++) {
            if (active) {
                active = q.step(cur, st);
                if (!active) active = q.finish(cur, st);
            }
        }
    }
}

} // namespace wrt
