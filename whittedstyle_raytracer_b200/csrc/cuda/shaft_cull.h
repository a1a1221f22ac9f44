// shaft_cull.h — conservative "is this soft-shadow request trivially unoccluded?" test.
//
// A soft-shadow request is 50 rays from ONE origin to random points of ONE area light
// (Renderer.hpp:405-414; the sampled region is the parallelogram (1-u-v)*tv0 + u*tv1 + v*tv2,
// u, v in [0,1), Triangle.hpp:139-145).  A sample ray can only be blocked by a primitive whose own
// box it hits (DESIGN.md section 4: "tested <=> own box hit" for non-degenerate rays), so when NO
// leaf box can be hit by ANY ray of the shaft, all 50 samples are lit and the coefficient is
// exactly 50 * 1.0f — without generating a single sample.  In the metric frame 79 % of the
// primary-hit requests (floor and walls far from the bunny) are of that kind.
//
// Why the verdict is exact, not approximate:
//  1. Bounds.  Per axis, D_k = lightPos_k - o_k of every sample lies between the extremes over the
//     four parallelogram corners (linear in u, v), up to float rounding of the reference's
//     evaluation order (<= 1e-6 * M, M = largest |coordinate| involved).  The ranges are padded by
//     1e-5 * M.  An axis whose padded range excludes 0 is "definite": every sample direction has
//     the same non-zero sign there.  |D| lies in [dmin, dmax] (dmax: farthest corner, convexity;
//     dmin: the box lower bound sqrt(sum min|D_k|^2)), and inv_k = 1 / (D_k * (1/|D|)) = |D| / D_k
//     up to 4 roundings (< 5e-7), so on a definite axis inv_k is inside [dmin/hi_k, dmax/lo_k]
//     (signs handled), widened by 1e-5 relative.
//     An axis whose range touches 0 is DROPPED from the test (no constraint).  That stays exact even
//     for samples that are axis-degenerate there (d_k == 0: 1/0 = inf, 0*inf = NaN in
//     BoundBox.hpp:55-84): with fmaxf/fminf the exact t_enter is >= the maximum over the other axes
//     and t_exit <= their minimum (a NaN operand is ignored, +-inf only tightens), so a box that
//     fails on the remaining axes fails the exact test.  At least one axis must be definite.
//  2. Interval slab test.  All rays share the origin, so a = plane - o_k is the SAME float in
//     every ray's BoundBox::IntersectRay (BoundBox.hpp:53-85); t = a * inv_k is monotonic in inv_k
//     under round-to-nearest, hence t_near_k >= min(a*ilo_k, a*ihi_k) and t_far_k <= max(...)
//     hold for the rounded values.  If max_k(lower) > min_k(upper) or min_k(upper) < 0, the exact
//     test fails for every ray of the shaft.
//  3. Inner boxes are exact unions of their children and the interval bounds are monotonic under box
//     inclusion (a sub-box is entered later and left earlier; rounding is monotonic), so a failed
//     interval test at an inner node implies a failed one — hence a failed exact own-box test for
//     every ray — at every leaf below it.  A primitive is only ever tested after its own (leaf) box
//     passed, in the SAH tree and in the reference-topology tree that axis-degenerate rays walk.
// Any doubt (no definite axis, stack overflow, single-primitive scene whose root is tested
// without a box, BVH.hpp:166-172) answers "not empty" and the request is traced as before.
//
// The function is host/device so that tests/ can run the SAME source on the CPU against a
// brute-force check (tests/shaft_cull_check.cpp).
#ifndef WRT_SHAFT_CULL_H
#define WRT_SHAFT_CULL_H

#include <math.h>

#include "wide_bvh.h"

#ifdef __CUDACC__
#define WRT_SHAFT_HD __host__ __device__ __forceinline__
#else
#include <vector_types.h>
#define WRT_SHAFT_HD static inline
#endif

#if defined(__CUDA_ARCH__)
#define WRT_SHAFT_LD4(p) __ldg(p)
#define WRT_SHAFT_LD8(p, a, b) wrt::ldg8(p, a, b)       /* one 256-bit load per tree record (dev_math.cuh) */
#else
#define WRT_SHAFT_LD4(p) (*(p))
#define WRT_SHAFT_LD8(p, a, b) do { (a) = (p)[0]; (b) = (p)[1]; } while (0)
#endif

#define WRT_SHAFT_STACK 48
#define WRT_SHAFT_PAD_REL 1e-5f

struct WrtShaft {
    float o[3];
    float ilo[3], ihi[3];      // bounds of 1/d per definite axis (same sign, finite)
    int octant;                // bit k set: every sample direction is negative on axis k
    int use;                   // bit k set: axis k is definite and takes part in the test
};

// Builds the bounds of step 1.  tri = the light's tv0, tv1, tv2 (9 floats).  false = give up.
WRT_SHAFT_HD bool wrt_shaft_make(const float o[3], const float tri[9], WrtShaft* sh) {
    float c[4][3];
    float M = 0.f;
    for (int k = 0; k < 3; k++) {
        c[0][k] = tri[k]; c[1][k] = tri[3 + k]; c[2][k] = tri[6 + k];
        c[3][k] = tri[3 + k] + tri[6 + k] - tri[k];                       // u = v = 1 corner
        M = fmaxf(M, fabsf(o[k]));
        for (int j = 0; j < 4; j++) M = fmaxf(M, fabsf(c[j][k]));
    }
    if (!(M > 0.f) || !(M < 1e30f)) return false;
    const float pad = WRT_SHAFT_PAD_REL * M;
    float lo[3], hi[3], dmax = 0.f, mn2 = 0.f;
    for (int j = 0; j < 4; j++) {
        float dx = c[j][0] - o[0], dy = c[j][1] - o[1], dz = c[j][2] - o[2];
        dmax = fmaxf(dmax, sqrtf(dx * dx + dy * dy + dz * dz));
    }
    sh->octant = 0;
    sh->use = 0;
    for (int k = 0; k < 3; k++) {
        float l = c[0][k] - o[k], h = l;
        for (int j = 1; j < 4; j++) { float d = c[j][k] - o[k]; l = fminf(l, d); h = fmaxf(h, d); }
        l -= pad; h += pad;
        sh->o[k] = o[k];
        lo[k] = l; hi[k] = h;
        if (!(l == l) || !(h == h)) return false;                         // NaN
        if (!(l > 0.f) && !(h < 0.f)) continue;                           // sign not definite: axis dropped, |D_k| >= 0
        sh->use |= 1 << k;
        float m = fminf(fabsf(l), fabsf(h));
        mn2 += m * m;
        if (h < 0.f) sh->octant |= 1 << k;
    }
    if (sh->use == 0) return false;
    const float dmin = sqrtf(mn2) * (1.f - WRT_SHAFT_PAD_REL);
    dmax = dmax * (1.f + WRT_SHAFT_PAD_REL) + 4.f * pad;
    for (int k = 0; k < 3; k++) {
        sh->ilo[k] = 0.f; sh->ihi[k] = 0.f;
        if (!((sh->use >> k) & 1)) continue;
        float a, b;                                                       // inv = |D| / D_k
        if (lo[k] > 0.f) { a = dmin / hi[k]; b = dmax / lo[k]; }          // positive: smallest |D| over largest D_k ...
        else             { a = dmax / hi[k]; b = dmin / lo[k]; }          // negative: hi is the one closest to 0
        // widen outwards (a <= b, both of one sign)
        sh->ilo[k] = a > 0.f ? a * (1.f - WRT_SHAFT_PAD_REL) : a * (1.f + WRT_SHAFT_PAD_REL);
        sh->ihi[k] = b > 0.f ? b * (1.f + WRT_SHAFT_PAD_REL) : b * (1.f - WRT_SHAFT_PAD_REL);
        if (!(fabsf(sh->ilo[k]) < 1e30f) || !(fabsf(sh->ihi[k]) < 1e30f)) return false;
    }
    return true;
}

// Step 2 on a record of the octant tree: `nearp` = planes the rays enter through, `farp` = exit planes.
WRT_SHAFT_HD bool wrt_shaft_may_hit(const WrtShaft* sh, const float4 nearp, const float4 farp) {
    float ax = nearp.x - sh->o[0], ay = nearp.y - sh->o[1], az = nearp.z - sh->o[2];
    float bx = farp.x - sh->o[0], by = farp.y - sh->o[1], bz = farp.z - sh->o[2];
    float lx = fminf(ax * sh->ilo[0], ax * sh->ihi[0]), ux = fmaxf(bx * sh->ilo[0], bx * sh->ihi[0]);
    float ly = fminf(ay * sh->ilo[1], ay * sh->ihi[1]), uy = fmaxf(by * sh->ilo[1], by * sh->ihi[1]);
    float lz = fminf(az * sh->ilo[2], az * sh->ihi[2]), uz = fmaxf(bz * sh->ilo[2], bz * sh->ihi[2]);
    if (!(sh->use & 1)) { lx = -INFINITY; ux = INFINITY; }                // dropped axes do not constrain
    if (!(sh->use & 2)) { ly = -INFINITY; uy = INFINITY; }
    if (!(sh->use & 4)) { lz = -INFINITY; uz = INFINITY; }
    float lb = fmaxf(lx, fmaxf(ly, lz)), ub = fminf(ux, fminf(uy, uz));
    return lb <= ub && ub >= 0.f;
}

// The same test, also returning the lower bound of the entry distance (orders the candidate walk).
WRT_SHAFT_HD bool wrt_shaft_may_hit_lb(const WrtShaft* sh, const float4 nearp, const float4 farp, float* lb_out) {
    float ax = nearp.x - sh->o[0], ay = nearp.y - sh->o[1], az = nearp.z - sh->o[2];
    float bx = farp.x - sh->o[0], by = farp.y - sh->o[1], bz = farp.z - sh->o[2];
    float lx = fminf(ax * sh->ilo[0], ax * sh->ihi[0]), ux = fmaxf(bx * sh->ilo[0], bx * sh->ihi[0]);
    float ly = fminf(ay * sh->ilo[1], ay * sh->ihi[1]), uy = fmaxf(by * sh->ilo[1], by * sh->ihi[1]);
    float lz = fminf(az * sh->ilo[2], az * sh->ihi[2]), uz = fmaxf(bz * sh->ilo[2], bz * sh->ihi[2]);
    if (!(sh->use & 1)) { lx = -INFINITY; ux = INFINITY; }
    if (!(sh->use & 2)) { ly = -INFINITY; uy = INFINITY; }
    if (!(sh->use & 4)) { lz = -INFINITY; uz = INFINITY; }
    float lb = fmaxf(lx, fmaxf(ly, lz)), ub = fminf(ux, fminf(uy, uz));
    *lb_out = lb;
    return lb <= ub && ub >= 0.f;
}

// Candidate occluders of a shaft: every primitive whose leaf box may be hit by some ray of the shaft, written
// to out[0 .. n) nearest-first (by the entry lower bound).  A sample ray of the request that is not
// axis-degenerate tests exactly the primitives whose own box it hits (DESIGN.md section 4) and all of those are
// in the list, so "any list member blocks the ray" equals the any-hit traversal's answer.
// The walk is a resumable state machine (the list kernel interleaves the walks of a warp's lanes and refills lanes
// as they finish): wrt_shaft_walk_begin, then wrt_shaft_walk_step until it stops returning 1.
// stack[k * stack_stride], k < stack_cap, is the caller's traversal stack.
typedef struct WrtShaftWalk {
    const float4* nodes;   // the shaft's octant copy of the tree
    int cur, sp, n;        // node pair to visit next, stack fill, list length so far
} WrtShaftWalk;

// 1 = walk started; 0 = finished at once with an empty list (no tree); -1 = give up (trace the request ray by ray).
WRT_SHAFT_HD int wrt_shaft_walk_begin(const float4* onodes, int n_nodes, const WrtShaft* sh, WrtShaftWalk* w) {
    w->sp = 0; w->n = 0; w->cur = 0; w->nodes = onodes;
    if (n_nodes <= 0) return 0;
    w->nodes = onodes + (size_t)sh->octant * 2 * (size_t)n_nodes;
    union { float f; int i; } u;
    u.f = WRT_SHAFT_LD4(w->nodes).w;
    w->cur = u.i;
    return w->cur < 0 ? -1 : 1;                                           // lone primitive: tested without its box
}

// One node pair.  1 = call again; 0 = done, out[0 .. w->n) is the list; -1 = the list would exceed out_cap or the
// stack would overflow.
WRT_SHAFT_HD int wrt_shaft_walk_step(const WrtShaft* sh, WrtShaftWalk* w, int* stack, int stack_stride, int stack_cap,
                                     int* out, int out_cap) {
    const float4* nd = w->nodes + 2 * (size_t)w->cur;
    float4 l0, l1, r0, r1;
    WRT_SHAFT_LD8(nd, l0, l1);
    WRT_SHAFT_LD8(nd + 2, r0, r1);
    float tl, tr;
    bool hl = wrt_shaft_may_hit_lb(sh, l0, l1, &tl), hr = wrt_shaft_may_hit_lb(sh, r0, r1, &tr);
    union { float f; int i; } u;
    u.f = l0.w; const int linkL = u.i;
    u.f = r0.w; const int linkR = u.i;
    const bool right_first = hl && hr && tr < tl;
    int n = w->n;
    // leaves: into the list, nearer one first
    if (hl && linkL < 0 && hr && linkR < 0) {
        if (n + 2 > out_cap) return -1;
        out[n++] = right_first ? ~linkR : ~linkL;
        out[n++] = right_first ? ~linkL : ~linkR;
        hl = false; hr = false;
    } else {
        if (hl && linkL < 0) { if (n == out_cap) return -1; out[n++] = ~linkL; hl = false; }
        if (hr && linkR < 0) { if (n == out_cap) return -1; out[n++] = ~linkR; hr = false; }
    }
    w->n = n;
    if (hl && hr) {
        if (w->sp == stack_cap) return -1;
        stack[w->sp * stack_stride] = right_first ? linkL : linkR;
        ++w->sp;
        w->cur = right_first ? linkR : linkL;
    } else if (hl) w->cur = linkL;
    else if (hr) w->cur = linkR;
    else {
        if (w->sp == 0) return 0;
        --w->sp;
        w->cur = stack[w->sp * stack_stride];
    }
    return 1;
}

// The whole walk in one call.  Returns the list length, or -1 (see wrt_shaft_walk_step).
WRT_SHAFT_HD int wrt_shaft_candidates(const float4* onodes, int n_nodes, const WrtShaft* sh, int* stack, int stack_stride,
                                      int stack_cap, int* out, int out_cap) {
    WrtShaftWalk w;
    int rc = wrt_shaft_walk_begin(onodes, n_nodes, sh, &w);
    if (rc <= 0) return rc;
    while ((rc = wrt_shaft_walk_step(sh, &w, stack, stack_stride, stack_cap, out, out_cap)) == 1) {}
    return rc < 0 ? -1 : w.n;
}

// True when no leaf box of the tree can be hit by any ray of the shaft.
// onodes: the 8 octant copies of the SAH tree (2 float4 per record, n_nodes records per copy).
WRT_SHAFT_HD bool wrt_shaft_is_empty(const float4* onodes, int n_nodes, const float o[3], const float tri[9]) {
    if (n_nodes <= 0) return true;                                        // nothing to hit
    WrtShaft sh;
    if (!wrt_shaft_make(o, tri, &sh)) return false;
    const float4* nodes = onodes + (size_t)sh.octant * 2 * (size_t)n_nodes;
    union { float f; int i; } w;
    w.f = WRT_SHAFT_LD4(nodes).w;
    int cur = w.i;
    if (cur < 0) return false;                                            // lone primitive: tested without its box
    int stack[WRT_SHAFT_STACK];
    int sp = 0;
    while (true) {
        const float4* n = nodes + 2 * (size_t)cur;
        float4 l0, l1, r0, r1;
        WRT_SHAFT_LD8(n, l0, l1);
        WRT_SHAFT_LD8(n + 2, r0, r1);
        bool hl = wrt_shaft_may_hit(&sh, l0, l1), hr = wrt_shaft_may_hit(&sh, r0, r1);
        w.f = l0.w; const int linkL = w.i;
        w.f = r0.w; const int linkR = w.i;
        if ((hl && linkL < 0) || (hr && linkR < 0)) return false;         // a leaf box is inside the shaft
        if (hl && hr) {
            if (sp == WRT_SHAFT_STACK) return false;
            stack[sp++] = linkR;
            cur = linkL;
        } else if (hl) cur = linkL;
        else if (hr) cur = linkR;
        else {
            if (sp == 0) return true;
            cur = stack[--sp];
        }
    }
}

// ---- the same walks over the 4-wide view of the tree (wide_bvh.h): half the dependent node fetches ----
// wnodes: the 8 wide copies (WRT_WIDE_FLOAT4_PER_RECORD float4 per binary record); onodes: the binary octant copies
// (record 0 holds the root's link).  A wide node's slots are records of the octant copy, so the interval test is
// wrt_shaft_may_hit(_lb) unchanged; an empty slot fails it on every used axis.
WRT_SHAFT_HD int wrt_shaft_walk_begin4(const float4* onodes, const float4* wnodes, int n_nodes, const WrtShaft* sh, WrtShaftWalk* w) {
    w->sp = 0; w->n = 0; w->cur = 0; w->nodes = wnodes;
    if (n_nodes <= 0) return 0;
    union { float f; int i; } u;
    u.f = WRT_SHAFT_LD4(onodes + (size_t)sh->octant * 2 * (size_t)n_nodes).w;
    w->cur = u.i;
    w->nodes = wnodes + WRT_WIDE_FLOAT4_PER_RECORD * (size_t)sh->octant * (size_t)n_nodes;
    return w->cur < 0 ? -1 : 1;                                           // lone primitive: tested without its box
}

#define WRT_SHAFT_CSWAP(ka, la, kb, lb) { const bool sw_ = (kb) < (ka); const float kt_ = sw_ ? (ka) : (kb); (ka) = sw_ ? (kb) : (ka); (kb) = kt_; \
                                          const int lt_ = sw_ ? (la) : (lb); (la) = sw_ ? (lb) : (la); (lb) = lt_; }

// One wide node: up to four leaves into the list (nearest first), up to three inner children pushed (farthest first).
WRT_SHAFT_HD int wrt_shaft_walk_step4(const WrtShaft* sh, WrtShaftWalk* w, int* stack, int stack_stride, int stack_cap,
                                      int* out, int out_cap) {
    const float4* nd = w->nodes + WRT_WIDE_FLOAT4_PER_RECORD * (size_t)w->cur;
    float4 a0, a1, b0, b1, c0, c1, d0, d1;
    WRT_SHAFT_LD8(nd, a0, a1);
    WRT_SHAFT_LD8(nd + 2, b0, b1);
    WRT_SHAFT_LD8(nd + 4, c0, c1);
    WRT_SHAFT_LD8(nd + 6, d0, d1);
    float k0, k1, k2, k3;
    const bool h0 = wrt_shaft_may_hit_lb(sh, a0, a1, &k0), h1 = wrt_shaft_may_hit_lb(sh, b0, b1, &k1);
    const bool h2 = wrt_shaft_may_hit_lb(sh, c0, c1, &k2), h3 = wrt_shaft_may_hit_lb(sh, d0, d1, &k3);
    const float inf = INFINITY;
    if (!h0) k0 = inf;
    if (!h1) k1 = inf;
    if (!h2) k2 = inf;
    if (!h3) k3 = inf;
    union { float f; int i; } u;
    u.f = a0.w; int l0 = u.i;
    u.f = b0.w; int l1 = u.i;
    u.f = c0.w; int l2 = u.i;
    u.f = d0.w; int l3 = u.i;
    WRT_SHAFT_CSWAP(k0, l0, k1, l1) WRT_SHAFT_CSWAP(k2, l2, k3, l3) WRT_SHAFT_CSWAP(k0, l0, k2, l2)
    WRT_SHAFT_CSWAP(k1, l1, k3, l3) WRT_SHAFT_CSWAP(k1, l1, k2, l2)
    int n = w->n;
    // Straight-line form: the capacity checks once per step (a list / stack within 4 / 3 entries of its capacity gives up a
    // step early: the request is then traced ray by ray, an exact path too), the appends and pushes as predicated stores.
    // (ncu source view of a branching form, one capacity check per append / push: 36 % of k_soft_lists' warp instructions
    // sat in its eight conditionals, at 9-12 of 32 lanes.)
    if (n + 4 > out_cap || w->sp + 3 > stack_cap) return -1;
    const bool e0 = k0 < inf && l0 < 0, e1 = k1 < inf && l1 < 0, e2 = k2 < inf && l2 < 0, e3 = k3 < inf && l3 < 0;
    if (e0) out[n] = ~l0;
    n += e0 ? 1 : 0;
    if (e1) out[n] = ~l1;
    n += e1 ? 1 : 0;
    if (e2) out[n] = ~l2;
    n += e2 ? 1 : 0;
    if (e3) out[n] = ~l3;
    n += e3 ? 1 : 0;
    w->n = n;
    const bool i0 = k0 < inf && l0 >= 0, i1 = k1 < inf && l1 >= 0, i2 = k2 < inf && l2 >= 0, i3 = k3 < inf && l3 >= 0;
    const int nearest = i0 ? l0 : (i1 ? l1 : (i2 ? l2 : (i3 ? l3 : -1)));
    const bool p3 = i3 && (i0 || i1 || i2), p2 = i2 && (i0 || i1), p1 = i1 && i0;
    int sp = w->sp;
    if (p3) stack[sp * stack_stride] = l3;
    sp += p3 ? 1 : 0;
    if (p2) stack[sp * stack_stride] = l2;
    sp += p2 ? 1 : 0;
    if (p1) stack[sp * stack_stride] = l1;
    sp += p1 ? 1 : 0;
    w->sp = sp;
    if (nearest >= 0) { w->cur = nearest; return 1; }
    if (sp == 0) return 0;
    w->sp = sp - 1;
    w->cur = stack[(sp - 1) * stack_stride];
    return 1;
}

WRT_SHAFT_HD int wrt_shaft_candidates4(const float4* onodes, const float4* wnodes, int n_nodes, const WrtShaft* sh, int* stack,
                                       int stack_stride, int stack_cap, int* out, int out_cap) {
    WrtShaftWalk w;
    int rc = wrt_shaft_walk_begin4(onodes, wnodes, n_nodes, sh, &w);
    if (rc <= 0) return rc;
    while ((rc = wrt_shaft_walk_step4(sh, &w, stack, stack_stride, stack_cap, out, out_cap)) == 1) {}
    return rc < 0 ? -1 : w.n;
}

// wrt_shaft_is_empty over the wide copies
WRT_SHAFT_HD bool wrt_shaft_is_empty4(const float4* onodes, const float4* wnodes, int n_nodes, const float o[3], const float tri[9]) {
    if (n_nodes <= 0) return true;
    WrtShaft sh;
    if (!wrt_shaft_make(o, tri, &sh)) return false;
    union { float f; int i; } u;
    u.f = WRT_SHAFT_LD4(onodes + (size_t)sh.octant * 2 * (size_t)n_nodes).w;
    int cur = u.i;
    if (cur < 0) return false;                                            // lone primitive: tested without its box
    const float4* nodes = wnodes + WRT_WIDE_FLOAT4_PER_RECORD * (size_t)sh.octant * (size_t)n_nodes;
    int stack[WRT_SHAFT_STACK];
    int sp = 0;
    while (true) {
        const float4* nd = nodes + WRT_WIDE_FLOAT4_PER_RECORD * (size_t)cur;
        float4 a0, a1, b0, b1, c0, c1, d0, d1;
        WRT_SHAFT_LD8(nd, a0, a1);
        WRT_SHAFT_LD8(nd + 2, b0, b1);
        WRT_SHAFT_LD8(nd + 4, c0, c1);
        WRT_SHAFT_LD8(nd + 6, d0, d1);
        const bool h0 = wrt_shaft_may_hit(&sh, a0, a1), h1 = wrt_shaft_may_hit(&sh, b0, b1);
        const bool h2 = wrt_shaft_may_hit(&sh, c0, c1), h3 = wrt_shaft_may_hit(&sh, d0, d1);
        u.f = a0.w; const int l0 = u.i;
        u.f = b0.w; const int l1 = u.i;
        u.f = c0.w; const int l2 = u.i;
        u.f = d0.w; const int l3 = u.i;
        if ((h0 && l0 < 0) || (h1 && l1 < 0) || (h2 && l2 < 0) || (h3 && l3 < 0)) return false;   // a leaf box is inside the shaft
        int next = -1;
        if (h3) next = l3;
        if (h2) { if (next >= 0) { if (sp == WRT_SHAFT_STACK) return false; stack[sp++] = next; } next = l2; }
        if (h1) { if (next >= 0) { if (sp == WRT_SHAFT_STACK) return false; stack[sp++] = next; } next = l1; }
        if (h0) { if (next >= 0) { if (sp == WRT_SHAFT_STACK) return false; stack[sp++] = next; } next = l0; }
        if (next >= 0) { cur = next; continue; }
        if (sp == 0) return true;
        cur = stack[--sp];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Triangle-level pruning of a candidate list (k_soft_filter).  The list holds every primitive whose BOX some ray of the
// shaft may hit; most of those triangles cannot be hit themselves.  A candidate is removed when it provably blocks no
// sample: it is then never the reason a ray is occluded, so "OR over the list" keeps its value (a ray that tests it in
// the reference gets "no hit with t < dis" from it).  The rays of a request are the segments from the origin o to points
// of the light's parallelogram, i.e. they lie in the pyramid P = hull(o, 4 corners).  Three sufficient conditions, in exact
// geometry, each applied with a margin far above every rounding involved:
//   side planes   all three vertices of the triangle lie outside ONE of the pyramid's four side planes (planes through o
//                 and two adjacent corners): the triangle and the convex pyramid are disjoint;
//   own plane     o and all four corners lie strictly on the same side of the triangle's plane: no segment o -> corner hull
//                 crosses that plane, so every ray's plane parameter t is < 0 or > dis.
//   edge planes   all four corners lie outside ONE of the three planes through o and a triangle edge: together with the
//                 side planes these are all the separating planes two convex cones with apex o can have, so a triangle
//                 that survives can really be hit by some ray from o into the parallelogram (or is too close to call).
// Margins.  Triangle.hpp:41 accepts barycentrics and t down to -1e-5, i.e. points up to 1e-5 * (|E1| + |E2|) outside the
// triangle and 1e-5 behind the origin; the samples' float evaluation moves a target by <= 1e-6 * |coordinate|
// (shaft_cull.h header, step 1).  The tests demand 1e-4 relative (to the vertex / corner distance from o) plus 2e-5 * (|E1|
// + |E2|) plus 1e-5 absolute for the side planes, and 1e-3 * (|E1| + |E2|) + 2e-5 for the origin's height over the triangle's
// plane (the 5e-4 offset of BVHStrategy.hpp:15 over centimetre triangles passes; an origin ON a 40-unit triangle's plane
// does not, and is left to the box test).  A pyramid seen almost edge-on (a side-plane normal that does not separate the
// opposite corners by 1e-3 of their distance) disables the filter for the request.
// tests/shaft_cull_check.cpp runs this same source on the CPU and checks every removed candidate against every sample
// ray with Triangle::intersect's own arithmetic: 0 violations over > 1e7 (ray, candidate) pairs per run.
typedef struct WrtShaftPyramid {
    float o[3];
    float D[4][3];         /* corners - o, in order around the parallelogram */
    float Dlen[4];
    float N[4][3];         /* unit inward normals of the side planes (plane k holds o, corner k, corner k+1) */
    int ok;
} WrtShaftPyramid;
#define WRT_PYRAMID_FLOATS 32          /* words a WrtShaftPyramid occupies when staged in shared memory */

WRT_SHAFT_HD void wrt_pyramid_make(const float o[3], const float tri[9], WrtShaftPyramid* p) {
    for (int k = 0; k < 3; k++) {
        p->o[k] = o[k];
        p->D[0][k] = tri[k] - o[k];
        p->D[1][k] = tri[3 + k] - o[k];
        p->D[2][k] = (tri[3 + k] + tri[6 + k] - tri[k]) - o[k];
        p->D[3][k] = tri[6 + k] - o[k];
    }
    for (int j = 0; j < 4; j++) p->Dlen[j] = sqrtf(p->D[j][0] * p->D[j][0] + p->D[j][1] * p->D[j][1] + p->D[j][2] * p->D[j][2]);
    p->ok = 1;
    for (int k = 0; k < 4; k++) {
        const float* a = p->D[k];
        const float* b = p->D[(k + 1) & 3];
        float n[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
        const float l = sqrtf(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
        if (!(l > 0.f) || !(l < 1e30f)) { p->ok = 0; n[0] = n[1] = n[2] = 0.f; }
        const float il = p->ok ? 1.f / l : 0.f;
        n[0] *= il; n[1] *= il; n[2] *= il;
        const float* c = p->D[(k + 2) & 3];
        const float* d = p->D[(k + 3) & 3];
        float s2 = n[0] * c[0] + n[1] * c[1] + n[2] * c[2], s3 = n[0] * d[0] + n[1] * d[1] + n[2] * d[2];
        if (s2 < 0.f) { n[0] = -n[0]; n[1] = -n[1]; n[2] = -n[2]; s2 = -s2; s3 = -s3; }
        const float dm = fmaxf(p->Dlen[(k + 2) & 3], p->Dlen[(k + 3) & 3]);
        if (!(s2 > 1e-3f * dm) || !(s3 > 1e-3f * dm)) p->ok = 0;                  /* edge-on: no filtering */
        p->N[k][0] = n[0]; p->N[k][1] = n[1]; p->N[k][2] = n[2];
    }
}

/* Ray-independent terms of a triangle, computed once per primitive at upload: unit normal of its plane and
 * |E1| + |E2| (the scale of the acceptance slack).  aux = {n.x, n.y, n.z, esz}; esz < 0 marks "do not filter"
 * (degenerate triangle, non-finite data, or not a triangle). */
WRT_SHAFT_HD void wrt_triangle_aux(const float E1[3], const float E2[3], float aux[4]) {
    float n[3] = {E1[1] * E2[2] - E1[2] * E2[1], E1[2] * E2[0] - E1[0] * E2[2], E1[0] * E2[1] - E1[1] * E2[0]};
    const float l = sqrtf(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    const float esz = sqrtf(E1[0] * E1[0] + E1[1] * E1[1] + E1[2] * E1[2]) + sqrtf(E2[0] * E2[0] + E2[1] * E2[1] + E2[2] * E2[2]);
    if (!(l > 0.f) || !(l < 1e30f) || !(esz < 1e30f)) { aux[0] = aux[1] = aux[2] = 0.f; aux[3] = -1.f; return; }
    const float il = 1.f / l;
    aux[0] = n[0] * il; aux[1] = n[1] * il; aux[2] = n[2] * il; aux[3] = esz;
}

/* false = the triangle (v0, E1 = v1 - v0, E2 = v2 - v0; aux from wrt_triangle_aux) provably blocks no sample ray of
 * the request.  Distances from o enter the margins through the L1 norm (>= the Euclidean one: more margin, no sqrt). */
WRT_SHAFT_HD bool wrt_pyramid_triangle_may_block(const WrtShaftPyramid* p, const float v0[3], const float E1[3], const float E2[3],
                                                 const float aux[4]) {
    const float esz = aux[3];
    if (!p->ok || !(esz >= 0.f)) return true;
    float w[3][3], m[3];
    for (int k = 0; k < 3; k++) {
        w[0][k] = v0[k] - p->o[k];
        w[1][k] = (v0[k] + E1[k]) - p->o[k];
        w[2][k] = (v0[k] + E2[k]) - p->o[k];
    }
    for (int i = 0; i < 3; i++) m[i] = 1e-4f * (fabsf(w[i][0]) + fabsf(w[i][1]) + fabsf(w[i][2])) + 2e-5f * esz + 1e-5f;
    for (int k = 0; k < 4; k++) {                          /* side planes */
        bool out = true;
        for (int i = 0; i < 3; i++) {
            const float s = p->N[k][0] * w[i][0] + p->N[k][1] * w[i][1] + p->N[k][2] * w[i][2];
            out = out && (s < -m[i]);
        }
        if (out) return false;
    }
    const float ho = -(aux[0] * w[0][0] + aux[1] * w[0][1] + aux[2] * w[0][2]);      /* own plane: height of o over it */
    if (fabsf(ho) > 1e-3f * esz + 2e-5f) {
        bool same = true;
        for (int j = 0; j < 4; j++) {
            const float H = aux[0] * (p->D[j][0] - w[0][0]) + aux[1] * (p->D[j][1] - w[0][1]) + aux[2] * (p->D[j][2] - w[0][2]);
            same = same && (H * ho > 0.f) && (fabsf(H) > 1e-3f * esz + 1e-4f * p->Dlen[j]);
        }
        if (same) return false;
    }
    return true;
}

/* Second stage, for the candidates the first stage kept: false = provably blocks no sample ray.
 * edge planes: the plane through o and a triangle edge (a, b), oriented towards the third vertex c.  Seen from o, the
 * triangle and the light are two convex polygons on the sphere of directions; they are disjoint iff an edge of one of
 * them separates them — the four side planes of the first stage, or one of these three.  With unit normal n and all four
 * corner directions at least (m + 1e-4) * Dmax outside it, every sample direction d has n.d < -(m + 1e-4); the only part of
 * the slack-widened triangle outside the plane lies within `slack` of the edge's line, i.e. at least h - slack from o
 * (h = distance from o to that line), where the ray is already (h - slack) * m = slack outside.
 * (Costs about as much as the first stage: k_soft_filter runs it on short survivor lists only — the fully lit requests,
 * which it empties; a long list belongs to a request in shadow or penumbra and cannot become empty.) */
WRT_SHAFT_HD bool wrt_pyramid_triangle_may_block_edges(const WrtShaftPyramid* p, const float v0[3], const float E1[3], const float E2[3],
                                                       const float aux[4]) {
    const float esz = aux[3];
    if (!p->ok || !(esz >= 0.f)) return true;
    float w[3][3];
    for (int k = 0; k < 3; k++) {
        w[0][k] = v0[k] - p->o[k];
        w[1][k] = (v0[k] + E1[k]) - p->o[k];
        w[2][k] = (v0[k] + E2[k]) - p->o[k];
    }
    {
        const float slack = 2e-5f * esz + 1e-5f;
        const float dmax = fmaxf(fmaxf(p->Dlen[0], p->Dlen[1]), fmaxf(p->Dlen[2], p->Dlen[3]));
        for (int e = 0; e < 3; e++) {
            const float* a = w[e];
            const float* b = w[e == 2 ? 0 : e + 1];
            const float* c = w[e == 0 ? 2 : e - 1];
            const float n[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
            const float l = sqrtf(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
            const float ex = b[0] - a[0], ey = b[1] - a[1], ez = b[2] - a[2];
            const float el = sqrtf(ex * ex + ey * ey + ez * ez);
            if (!(l > 0.f) || !(el > 0.f) || !(l < 1e30f)) continue;
            const float h = l / el;
            if (!(h > 4.f * slack)) continue;
            const float sc = n[0] * c[0] + n[1] * c[1] + n[2] * c[2];          /* l * (distance of c from the plane) */
            if (!(fabsf(sc) > l * (1e-3f * esz + 1e-4f * (fabsf(c[0]) + fabsf(c[1]) + fabsf(c[2]))))) continue;   /* o (almost) in the triangle's plane */
            const float sgn = sc > 0.f ? 1.f : -1.f;
            const float need = l * ((slack / (h - slack) + 1e-4f) * dmax);
            bool out = true;
            for (int j = 0; j < 4; j++) {
                const float s = sgn * (n[0] * p->D[j][0] + n[1] * p->D[j][1] + n[2] * p->D[j][2]);
                out = out && (s < -need);
            }
            if (out) return false;
        }
    }
    return true;
}

#endif /* WRT_SHAFT_CULL_H */
