// kernels.cuh — the wavefront kernels (sm_100a, SIMT FP32; tensor cores unused:
// the path is divergent traversal, not a dense contraction).
//
// One frame (Renderer.hpp:57-137), 24 launches with hard shadows, 30 for a soft-shadow frame:
//   chain stream  for each ray-tree level d = 0..8 (Renderer.hpp:25 MAX_DEPTH 9)
//                   k_trace_closest   rays[d] -> hits (level 0: primary rays generated in registers, Renderer.hpp:104-125;
//                                     levels 1..8 walk the 4-wide view of the tree, wide_bvh.h, one leaf test per lane and
//                                     step: traverse_step4_defer, dev_traverse.cuh)
//                   k_surface_spawn   hits -> surface records, child rays[d+1], shadow requests into one of three queues:
//                                     queue 0 = level 0, queue 1 = levels 1..5, queue 2 = levels 6..8
//                 after level 8: the shadow kernels of queue 2
//   side stream   the shadow kernels of queue 0 + k_shade(level 0) beside the deep chain, then — once level 5's surface
//                 stage is done — the shadow kernels of queue 1 beside the chain of levels 6..8
//                 shadow kernels of a queue: k_shadow_hard, or k_soft_lists -> k_soft_filter -> k_soft_list_rays
//                 (+ k_shadow_directional)
//   chain stream  k_combine_resolve         shades the deep nodes, then colour = local + fr*R + (1-fr)(1-alpha)*T bottom-up in
//                                           the reference's own association (Renderer.hpp:259) and int(255*min(c,1))
//                                           (Renderer.hpp:128-130); one cooperative launch.
// (Fusing the surface stage into the closest-hit kernel — finished lanes keep their hit and the warp runs the surface code
// at its next refill — was built and measured: 21.0 vs 18.0 ms per frame.  The surface code wants ~100 registers; under
// the 64 the traversal needs for its occupancy, ptxas spills the ray's 1/d and the node pointer inside the hot loop
// (profiles/NOTES.md).)
// The only dependent chain is the 9 closest-hit launches; the shadow work of the deep levels — independent of the
// chain — is cut into two sets of launches, not eight with eight tails, and level 0's shadow work fills the SMs the
// short deep levels leave idle.
//
// Every queue length lives in device memory (Counters); kernels read it there, so
// the host enqueues the whole frame without synchronising.
#pragma once
#include <cooperative_groups.h>

#include "dev_shade.cuh"
#include "shaft_cull.h"
#include "../../../include/wrt_rng.h"
#include "../../../include/wrt_tiles.h"

// Traversal kernels: 128-thread CTAs; ptxas settles at 48-61 registers (8-9 CTAs per SM).  Forcing more
// CTAs per SM through a minimum-blocks bound spills and is slower (profiles/NOTES.md).
#define WRT_TRACE_BOUNDS __launch_bounds__(128)
#define WRT_TRACE_DEEP_STEPS 8
namespace wrt {

// ---- debug build (-DWRT_DEBUG_BOUNDS): every queue / pool / stack / node index is checked before the access; the first
// failing source line is latched into a device variable the host reads after the frame (wrt_cuda.cu: finish_frame).
#ifdef WRT_DEBUG_BOUNDS
__device__ unsigned g_wrt_bounds_line = 0;
__device__ __forceinline__ bool wrt_bounds_ok(bool ok, unsigned line) {
    if (!ok) atomicCAS(&g_wrt_bounds_line, 0u, line);
    return ok;
}
#define WRT_IN_BOUNDS(idx, cap) wrt_bounds_ok((unsigned long long)(idx) < (unsigned long long)(cap), (unsigned)__LINE__)
#else
#define WRT_IN_BOUNDS(idx, cap) true
#endif

enum CounterSlot {
    C_NRAYS = 0,                 // [WRT_MAX_DEPTH + 1] level d >= 1: reflection rays (first half of the level's arrays)
    C_NTRAYS = 112,              // [WRT_MAX_DEPTH + 1] level d >= 1: transmission rays (second half)
    C_NPREQ = 16,                // [WRT_QUEUES] point-light shadow requests per request queue (FrameBuffers::queue_of_level)
    C_NDREQ = 32,                // [WRT_QUEUES] directional-light shadow requests, same queues
    C_VALID0 = 48,               // valid (non-padding) primary rays
    C_OVERFLOW = 49,             // set when a queue append was dropped
    C_NEMPTY = 50,               // queued soft-shadow requests whose candidate list came out empty (= 50 lit samples)
    C_NCULL = 128,               // [9] soft-shadow requests answered by the shaft test (shaft_cull.h), never queued
    C_NSKIP = 144,               // [9] point-light requests whose light terms vanish (dev_shade.cuh), never queued
    C_NDSKIP = 160,              // [9] the same for directional lights
    C_POOL = 176,                // [WRT_QUEUES] fill level of the candidate-list pools (k_soft_lists)
    C_NWORK = 180,               // [WRT_QUEUES] requests that still need rays after k_soft_filter (SoftListBuffers::work)
    C_WORK = 192,                // [<= 32 x 2] work-distribution counters (64-bit), one per persistent launch
    C_TOTAL = 256
};

struct TileMap : WrtTileMap {     // include/wrt_tiles.h
    __host__ __device__ bool slot_to_pixel(long long slot, int rank_, int& px, int& py) const {
        return wrt_tilemap_slot_to_pixel(this, slot, rank_, &px, &py) != 0;
    }
};

#define WRT_QUEUES 3

// Everything a kernel needs to (re)generate the primary ray of a slot: level-0 rays never exist in memory.
struct PrimaryGen {
    WrtCamera cam;
    TileMap tm;
    long long slot0;             // first slot of the batch
};

// Per-frame buffers.  A ray-tree node is addressed by ONE global id: level 0 -> its slot in the batch,
// level d >= 1 -> cap0 + (d-1)*capd + slot.  Deep levels are sized capd (default a quarter of the batch: in the bunny
// frames <= 16 % of the pixels spawn children); an overflow is detected, the buffers grow and the batch is re-rendered.
struct FrameBuffers {
    float4* ray_o[2];            // deep levels, by level & 1: {o.xyz, pixel id}
    float4* ray_d[2];            //                            {d.xyz, path id}
    float4* hit;                 // unfused path only: {t, prim, b1, b2} by slot
    float4* surf;                // 4 per node: {pos, prim} {nDir, material} {Od, -} {ray origin, -}
    float4* node_a;              // per node {local.rgb -> colour.rgb, fr}
    float4* node_b;              // per node {kT, childR, childT, composite flag}  (children as node ids)
    // Shadow requests go to WRT_QUEUES queues by ray-tree level: queue 0 = level 0, queue 1 = levels 1..k, queue 2 = levels
    // k+1..8.  Each queue gets ONE set of shadow launches, started as soon as its last level's surface stage is done.
    float4* preq_o[WRT_QUEUES];  // point-light request: {shadow ray origin, node}
    uint4*  preq_k[WRT_QUEUES];  //                      {light, pixel, path, -}
    float4* dreq_o[WRT_QUEUES];  // directional request: {pos, node}
    uint4*  dreq_k[WRT_QUEUES];  //                      {light, self prim, -, -}
    unsigned char queue_of_level[WRT_MAX_DEPTH + 3];
    float*  coeff;               // [node * n_lights + light]
    unsigned* counters;
    unsigned cap0, capd;         // slots of level 0 (batch capacity) and of every deeper level
    unsigned preq_cap[WRT_QUEUES], dreq_cap[WRT_QUEUES];
    unsigned n_node_cap;         // cap0 + (WRT_MAX_DEPTH-1) * capd
};

__device__ __forceinline__ unsigned node_id(const FrameBuffers& fb, int level, unsigned slot) {
    return level == 0 ? slot : fb.cap0 + (unsigned)(level - 1) * fb.capd + slot;
}

// ---- warp-aggregated queue append: k in {0,1,2,...} slots per lane, one atomic per warp ----
__device__ __forceinline__ unsigned warp_alloc(unsigned* counter, int k, unsigned cap, unsigned* overflow) {
    unsigned lane = threadIdx.x & 31;
    int incl = k;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        int n = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= (unsigned)off) incl += n;
    }
    int total = __shfl_sync(0xffffffffu, incl, 31);
    unsigned base = 0;
    if (lane == 31 && total > 0) base = atomicAdd(counter, (unsigned)total);
    base = __shfl_sync(0xffffffffu, base, 31);
    unsigned mine = base + (unsigned)(incl - k);
    if (k > 0 && (mine > cap || (unsigned)k > cap - mine)) { *overflow = 1u; return 0xffffffffu; }
    return mine;
}

// Rays of a ray-tree level.  Level 0 is one segment [0, n).  Deeper levels keep reflection
// rays in the first half of the level's arrays and transmission rays in the second half:
// a warp then traces rays of one kind from neighbouring pixels, which stay on similar
// paths much longer than an interleaved reflect/refract mix does.
struct LevelSpan {
    unsigned nR, nT, half;
    __device__ __forceinline__ unsigned count() const { return nR + nT; }
    __device__ __forceinline__ unsigned slot(unsigned item) const { return item < nR ? item : half + (item - nR); }
};
__device__ __forceinline__ LevelSpan level_span(const FrameBuffers& fb, int level, unsigned n0) {
    LevelSpan sp;
    if (level == 0) {
        sp.half = fb.cap0; sp.nT = 0;
        sp.nR = n0 < fb.cap0 ? n0 : fb.cap0;
    } else {
        const unsigned* counters = fb.counters;
        sp.half = fb.capd / 2;
        sp.nR = counters[C_NRAYS + level] < sp.half ? counters[C_NRAYS + level] : sp.half;
        sp.nT = counters[C_NTRAYS + level] < fb.capd - sp.half ? counters[C_NTRAYS + level] : fb.capd - sp.half;
    }
    return sp;
}

__device__ __forceinline__ unsigned queue_len(const unsigned* counters, int slot, unsigned cap) {
    unsigned n = counters[slot];
    return n < cap ? n : cap;
}

// ---- primary ray of a slot, Renderer.hpp:104-125.  false = padding slot of a clipped border tile ----
__device__ __forceinline__ bool primary_ray(const PrimaryGen& pg, unsigned item, f3& org, f3& dir, unsigned& pixel) {
    const WrtCamera& cam = pg.cam;
    int x, y;
    if (!pg.tm.slot_to_pixel(pg.slot0 + item, pg.tm.rank, x, y)) {
        org = mk3(0.f, 0.f, 0.f); dir = mk3(0.f, 0.f, 1.f); pixel = 0xffffffffu;
        return false;
    }
    f3 ul = mk3(cam.ul[0], cam.ul[1], cam.ul[2]);
    f3 v_off = (float)y * mk3(cam.delta_v[0], cam.delta_v[1], cam.delta_v[2]);
    f3 h_off = (float)x * mk3(cam.delta_h[0], cam.delta_h[1], cam.delta_h[2]);
    f3 pixelPos = ul + h_off + v_off + mk3(cam.c_off_h[0], cam.c_off_h[1], cam.c_off_h[2]) +
                  mk3(cam.c_off_v[0], cam.c_off_v[1], cam.c_off_v[2]);
    f3 eye = mk3(cam.eye[0], cam.eye[1], cam.eye[2]);
    f3 nrm = mk3(cam.n[0], cam.n[1], cam.n[2]);
    if (!cam.parallel) { dir = normalized(pixelPos - eye); org = eye; }
    else { dir = nrm; org = pixelPos - cam.d * nrm; }
    pixel = (unsigned)(y * cam.width + x);
    return true;
}

// ---- hit -> surface, shadow requests, child rays (Renderer.hpp:170-257); called by a whole, converged warp ----
// `cull`: shadow requests that provably cannot change the image are answered here and never queued.
//   WRT_CULL_UNLIT  the light's diffuse AND specular factors at this point are exactly 0 (dev_shade.cuh,
//                   light_terms_vanish): whatever the coefficient, the light adds +-0;
//   WRT_CULL_SHAFT  (soft shadows) the whole shaft origin -> area light misses every leaf box: all 50
//                   samples are lit, coefficient = 50 (shaft_cull.h).
// The reference traces these rays; WrtStats keeps counting them and reports how many were answered this way.
// `live`: this lane carries a finished closest-hit query (prim: -1 miss, -2 padding slot, >= 0 hit).
#define WRT_CULL_UNLIT 1
#define WRT_CULL_SHAFT 2
__device__ __forceinline__ void surface_warp(const DevScene& s, const FrameBuffers& fb, int level, int cull, bool live,
                                             f3 org, f3 dir, unsigned pixel, unsigned path, float hit_t, int prim,
                                             float b1, float b2, unsigned slot) {
    const unsigned child_half = fb.capd / 2;
    const int q = fb.queue_of_level[level];
    float4* nray_o = fb.ray_o[(level + 1) & 1];
    float4* nray_d = fb.ray_d[(level + 1) & 1];
    unsigned* overflow = fb.counters + C_OVERFLOW;
    const unsigned g = node_id(fb, level, slot);
    bool shade = false;
    bool spawnT = false, spawnR = false;
    float4 na = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 nb = make_float4(0.f, __int_as_float(-1), __int_as_float(-1), 0.f);
    f3 pos = mk3(0.f, 0.f, 0.f), nDir = pos, N = pos;
    f3 refractDir = pos, reflectDir = pos, refRayOrig = pos, traRayOrig = pos;
    float shade_n = 0.f;                                   // Phong exponent of the shaded material
    unsigned lit_mask = 0, skip_mask = 0;                  // lights (< 32) answered without a request
    if (live) {
        if (prim == -1) {
            na = make_float4(s.bkg[0], s.bkg[1], s.bkg[2], 0.f);            // miss: bkgcolor, :170
        } else if (prim >= 0) {
            Surface sf = complete_hit(s, org, dir, hit_t, prim, b1, b2);
            Mtl m = load_material(s, sf.material);
            if (sf.flags & WRT_PRIM_LIGHT) {
                na = make_float4(m.diffuse.x, m.diffuse.y, m.diffuse.z, 0.f); // light avatar, :172
            } else {
                shade = true;
                shade_n = m.n;
                f3 Od = m.diffuse;
                if (!float_equal(-1.f, (float)sf.textureIndex) && !float_equal(-1.f, sf.u) && !float_equal(-1.f, sf.v))
                    Od = texture_at(s, s.textures + sf.textureIndex, sf.u, sf.v);      // :176-180
                if (sf.normalMapIndex != -1) sf.nDir = change_normal_dir(s, sf);        // :182-184
                pos = sf.pos; nDir = sf.nDir;
                if (WRT_IN_BOUNDS(g, fb.n_node_cap)) {
                    float4* sv = fb.surf + 4 * (size_t)g;
                    sv[0] = make_float4(pos.x, pos.y, pos.z, __int_as_float(prim));
                    sv[1] = make_float4(nDir.x, nDir.y, nDir.z, __int_as_float(sf.material));
                    sv[2] = make_float4(Od.x, Od.y, Od.z, 0.f);
                    sv[3] = make_float4(org.x, org.y, org.z, 0.f);          // p_eye_dir needs the ray origin, :267
                }
                // ---- reflection / transmission, :194-257 ----
                refRayOrig = pos; traRayOrig = pos;
                N = normalized(nDir);
                float fr, eta_i, eta_t;
                float cosN_Dir = dot(N, -dir);
                if (cosN_Dir > 0) { eta_i = s.eta; eta_t = m.eta; }
                else { eta_i = m.eta; eta_t = s.eta; }
                fr = fresnel(dir, N, eta_i, eta_t);
                refractDir = normalized(refraction_dir(dir, N, eta_i, eta_t));
                reflectDir = normalized(reflection_dir(dir, nDir));
                float cos_refle_N = dot(reflectDir, N);
                float cos_refra_N = dot(refractDir, N);
                const float EPSILON = 0.00005f;
                if (cos_refle_N < 0) refRayOrig = refRayOrig - EPSILON * N;
                else refRayOrig = refRayOrig + EPSILON * N;
                if (cos_refra_N < 0) traRayOrig = traRayOrig - EPSILON * N;
                else traRayOrig = traRayOrig + EPSILON * N;
                if (float_equal(0.f, norm(refractDir))) fr = 1.f;
                spawnT = !float_equal(1.f, m.alpha) && !float_equal(fr, 1.f);
                spawnR = m.ks != 0;
                if (level + 1 >= WRT_MAX_DEPTH) { spawnT = false; spawnR = false; }    // traceRay depth cut, :152
                na.w = fr;
                nb.x = (1 - fr) * (1 - m.alpha);
                nb.w = 1.f;                                                    // composite node
            }
        }
    }
    if (live && !shade && WRT_IN_BOUNDS(g, fb.n_node_cap)) fb.surf[4 * (size_t)g] = make_float4(0.f, 0.f, 0.f, __int_as_float(-1));
    // child rays: reflections into the first half of the next level, transmissions into the second
    unsigned rslot = warp_alloc(fb.counters + C_NRAYS + level + 1, spawnR ? 1 : 0, child_half, overflow);
    unsigned tslot = warp_alloc(fb.counters + C_NTRAYS + level + 1, spawnT ? 1 : 0, fb.capd - child_half, overflow);
    if (spawnR && rslot != 0xffffffffu && WRT_IN_BOUNDS(rslot, fb.capd)) {
        nray_o[rslot] = make_float4(refRayOrig.x, refRayOrig.y, refRayOrig.z, __uint_as_float(pixel));
        nray_d[rslot] = make_float4(reflectDir.x, reflectDir.y, reflectDir.z, __uint_as_float(path * 2u));
        nb.y = __int_as_float((int)node_id(fb, level + 1, rslot));
    }
    if (spawnT && tslot != 0xffffffffu && WRT_IN_BOUNDS(child_half + tslot, fb.capd)) {
        unsigned c = child_half + tslot;
        nray_o[c] = make_float4(traRayOrig.x, traRayOrig.y, traRayOrig.z, __uint_as_float(pixel));
        nray_d[c] = make_float4(refractDir.x, refractDir.y, refractDir.z, __uint_as_float(path * 2u + 1u));
        nb.z = __int_as_float((int)node_id(fb, level + 1, c));
    }
    // shadow requests: one per (shaded hit, light) — minus the ones that cannot change the image
    const f3 sorig = pos + 0.0005f * nDir;                             // BVHStrategy.hpp:15, Renderer.hpp:349
    int n_preq = shade ? s.n_point_lights : 0, n_dreq = shade ? s.n_dir_lights : 0;
    if (shade && cull) {
        const float so[3] = {sorig.x, sorig.y, sorig.z};
        const f3 p_eye_dir = normalized(org - pos);                    // as blinn_phong() will compute it
        for (int li = 0; li < s.n_lights && li < 32; li++) {
            const WrtLight* L = s.lights + li;
            const bool point = float_equal(L->pos[3], 1.f);
            if ((cull & WRT_CULL_UNLIT) && light_terms_vanish(L, p_eye_dir, pos, nDir, shade_n)) {
                skip_mask |= 1u << li;                                 // coefficient is multiplied by 0 twice
                if (point) --n_preq; else --n_dreq;
            } else if ((cull & WRT_CULL_SHAFT) && point) {
                float tri[9];
                for (int k = 0; k < 9; k++) tri[k] = L->tri[k];
                // (binary walk: most level-0 shafts miss the bunny's subtree after 2-3 nodes; the 4-wide walk measured 832 vs 768 us)
                if (wrt_shaft_is_empty(s.onodes, s.n_nodes, so, tri)) { lit_mask |= 1u << li; --n_preq; }
            }
        }
    }
    unsigned pslot = warp_alloc(fb.counters + C_NPREQ + q, n_preq, fb.preq_cap[q], overflow);
    unsigned dslot = 0xffffffffu;
    if (s.n_dir_lights > 0) dslot = warp_alloc(fb.counters + C_NDREQ + q, n_dreq, fb.dreq_cap[q], overflow);
    if (cull) {                                                        // statistics: the reference traces these rays
        unsigned n_lit = __reduce_add_sync(0xffffffffu, (unsigned)__popc(lit_mask));
        unsigned n_skip_p = __reduce_add_sync(0xffffffffu, (unsigned)((shade ? s.n_point_lights : 0) - n_preq - __popc(lit_mask)));
        unsigned n_skip_d = __reduce_add_sync(0xffffffffu, (unsigned)((shade ? s.n_dir_lights : 0) - n_dreq));
        if ((threadIdx.x & 31) == 0) {
            if (n_lit) atomicAdd(fb.counters + C_NCULL + level, n_lit);
            if (n_skip_p) atomicAdd(fb.counters + C_NSKIP + level, n_skip_p);
            if (n_skip_d) atomicAdd(fb.counters + C_NDSKIP + level, n_skip_d);
        }
    }
    if (shade) {
        for (int li = 0; li < s.n_lights; li++) {
            const bool lit = li < 32 && ((lit_mask >> li) & 1u), skip = li < 32 && ((skip_mask >> li) & 1u);
            if (WRT_IN_BOUNDS(g, fb.n_node_cap)) fb.coeff[(size_t)g * s.n_lights + li] = lit ? (float)WRT_SOFT_SAMPLES : 0.f;
            if (lit || skip) continue;
            bool point = float_equal(s.lights[li].pos[3], 1.f);
            if (point && pslot != 0xffffffffu) {
                if (WRT_IN_BOUNDS(pslot, fb.preq_cap[q])) {
                    fb.preq_o[q][pslot] = make_float4(sorig.x, sorig.y, sorig.z, __uint_as_float(g));
                    fb.preq_k[q][pslot] = make_uint4((unsigned)li, pixel, path, 0u);
                }
                ++pslot;
            } else if (!point && dslot != 0xffffffffu) {
                if (WRT_IN_BOUNDS(dslot, fb.dreq_cap[q])) {
                    fb.dreq_o[q][dslot] = make_float4(pos.x, pos.y, pos.z, __uint_as_float(g));
                    fb.dreq_k[q][dslot] = make_uint4((unsigned)li, (unsigned)prim, 0u, 0u);
                }
                ++dslot;
            }
        }
    }
    if (live && WRT_IN_BOUNDS(g, fb.n_node_cap)) {
        fb.node_a[g] = na;
        fb.node_b[g] = nb;
    }
}

// ---- K2: closest hit; persistent warps, per-lane refill (dev_traverse.cuh run_queue) ----
template <bool LEVEL0>
struct ClosestQuery {
    const DevScene& s;
    const FrameBuffers& fb;
    const PrimaryGen& pg;
    const float4* ray_o;
    const float4* ray_d;
    float prune_cfg;
    // per-lane state
    Ray r;
    ClosestState cs;
    const float4* nodes;
    bool wide;                 // this lane walks the 4-wide view of its octant copy (wide_bvh.h)
    unsigned idx;
    LevelSpan span;
    __device__ __forceinline__ ClosestQuery(const DevScene& s_, const FrameBuffers& fb_, const PrimaryGen& pg_, int level,
                                            unsigned n0, float prune)
        : s(s_), fb(fb_), pg(pg_), ray_o(fb_.ray_o[level & 1]), ray_d(fb_.ray_d[level & 1]), prune_cfg(prune),
          span(level_span(fb_, level, n0)) {}
    __device__ __forceinline__ bool begin(unsigned long long item, int& cur, Stack&) {
        idx = span.slot((unsigned)item);
        f3 o, d;
        cs.reset(prune_cfg);
        if (LEVEL0) {
            unsigned pixel;
            if (!primary_ray(pg, (unsigned)item, o, d, pixel)) { cs.best.prim = -2; return false; }     // padding slot
        } else {
            o = mk3(ray_o[idx]); d = mk3(ray_d[idx]);
        }
        if (s.n_nodes == 0) return false;
        r = make_ray(o, d);
        float prune = prune_cfg;
        const bool ref_tree = prune < 0.f || degenerate_dir(r.d);       // literal walk / axis-degenerate ray
        if (ref_tree) prune = -1.f;
        const size_t oct_off = (size_t)ray_octant(r.d) * 2 * (size_t)s.n_nodes;
        nodes = (ref_tree ? s.ronodes : s.onodes) + oct_off;
        cs.set_ray(s, r, prune);
        float te;
        float4 lo = ldg4(nodes), hi = ldg4(nodes + 1);
        if (!slab_presorted(lo, hi, r, te)) return false;
        cur = __float_as_int(lo.w);
        if (cur < 0) { cs.leaf(s, r, ~cur); return false; }
        // (level 0: coherent primary rays, two thirds of them end on a wall after a few steps — the 4-wide node costs
        // registers there and buys nothing: 378 vs 338 us)
        wide = !LEVEL0 && !ref_tree;
        // (One copy for all octants — octant 0's holds the plain {pMin}{pMax} records — with the select-based slab test, to
        // shrink the L1 footprint of the deep levels 8x: 3.73 against 3.70 ms, no gain; the fetches that stall are L2 hits
        // deep in the tree, not the shared top levels.)
        if (wide) nodes = s.wnodes + (WRT_WIDE_FLOAT4_PER_RECORD / 2) * oct_off;
        return true;
    }
    __device__ __forceinline__ bool step(int& cur, Stack& st) {
        if (!LEVEL0 && wide) return traverse_step4_defer<true>(nodes, r, st, cur, cs.limit, [&](int p) { cs.leaf(s, r, p); });
        return traverse_step<true, true>(nodes, r, st, cur, cs.limit, [&](int p) { cs.leaf(s, r, p); });
    }
    __device__ __forceinline__ bool finish(int&, Stack&) {
        if (WRT_IN_BOUNDS(idx, fb.cap0 > fb.capd ? fb.cap0 : fb.capd))
            fb.hit[idx] = make_float4(cs.best.t, __int_as_float(cs.best.prim), cs.best.u, cs.best.v);
        return false;
    }
};

template <bool LEVEL0>
__global__ void WRT_TRACE_BOUNDS k_trace_closest(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb,
                                                 const __grid_constant__ PrimaryGen pg, int level, unsigned n0, int work_slot,
                                                 float prune_rel, int refill) {
    extern __shared__ int smem[];
    Stack st;
    st.init(smem, threadIdx.x, blockDim.x);
    ClosestQuery<LEVEL0> q(s, fb, pg, level, n0, prune_rel);
    // (deep levels: a deferred-leaf step is short; 8 steps between two looks at the idle lanes measured 3.68 against 3.74 ms)
    run_queue<ClosestQuery<LEVEL0>, LEVEL0 ? WRT_STEPS_PER_ROUND : WRT_TRACE_DEEP_STEPS>(
        q, q.span.count(), reinterpret_cast<unsigned long long*>(fb.counters + work_slot), st, refill);
}

// ---- K3: hit -> surface, shadow requests, child rays: one streaming pass, whole warps call surface_warp() ----
// (launch bound: 64 registers = 4 CTAs of 256 per SM.  Unbounded the kernel takes 80 registers, 3 CTAs: 1.67 ms per 4K
// frame against 1.61 / hard-shadow frame 1.72 against 1.36; 5 CTAs (48 registers) spill too much: 1.97.)
#define WRT_SURFACE_MIN_BLOCKS 4
__global__ void __launch_bounds__(256, WRT_SURFACE_MIN_BLOCKS) k_surface_spawn(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb,
                                                       const __grid_constant__ PrimaryGen pg, int level, unsigned n0, int cull) {
    const LevelSpan span = level_span(fb, level, n0);
    const unsigned n = span.count();
    const unsigned n_round = (n + 31u) & ~31u;         // whole warps stay converged for the aggregated appends
    unsigned valid = 0;
    for (unsigned item = blockIdx.x * blockDim.x + threadIdx.x; item < n_round; item += gridDim.x * blockDim.x) {
        const bool live = item < n;
        const unsigned i = span.slot(live ? item : 0);
        f3 org = mk3(0.f, 0.f, 0.f), dir = org;
        unsigned pixel = 0, path = 0;
        float4 h = make_float4(0.f, __int_as_float(-2), 0.f, 0.f);
        if (live) {
            h = fb.hit[i];
            if (level == 0) {
                path = 1u;
                if (primary_ray(pg, item, org, dir, pixel)) ++valid;
            } else {
                float4 o4 = fb.ray_o[level & 1][i], d4 = fb.ray_d[level & 1][i];
                org = mk3(o4); dir = mk3(d4);
                pixel = __float_as_uint(o4.w); path = __float_as_uint(d4.w);
            }
        }
        surface_warp(s, fb, level, cull, live, org, dir, pixel, path, h.x, __float_as_int(h.y), h.z, h.w, i);
    }
    if (level == 0) {
        valid = __reduce_add_sync(0xffffffffu, valid);
        if ((threadIdx.x & 31) == 0 && valid) atomicAdd(fb.counters + C_VALID0, valid);
    }
}

// ---- K4a: hard shadows, BVHStrategy::getShadowCoeffi ----
struct HardShadowQuery {
    const DevScene& s;
    const FrameBuffers& fb;
    Ray r;
    const float4* nodes;
    float dis;
    ShadowAcc acc;
    size_t out;
    int q;
    bool wide;
    bool literal;              // WRT_TRAVERSAL_EXHAUSTIVE: walk the reference-topology tree (the product's association comes from ShadowAcc either way)
    __device__ __forceinline__ HardShadowQuery(const DevScene& s_, const FrameBuffers& fb_, int q_, bool literal_)
        : s(s_), fb(fb_), q(q_), literal(literal_) {}
    __device__ __forceinline__ bool begin(unsigned long long item, int& cur, Stack&) {
        float4 o4 = fb.preq_o[q][item];
        uint4 k = fb.preq_k[q][item];
        const WrtLight* L = s.lights + k.x;
        f3 orig = mk3(o4);
        f3 lightPos = mk3(L->pos[0], L->pos[1], L->pos[2]);
        f3 raydir = normalized(lightPos - orig);
        dis = norm(lightPos - orig);
        r = make_ray(orig, raydir);
        out = (size_t)__float_as_uint(o4.w) * (unsigned)s.n_lights + k.x;
        acc.reset();
        if (s.n_nodes == 0) return false;
        const bool ref_tree = literal || degenerate_dir(raydir);
        const size_t oct_off = (size_t)ray_octant(raydir) * 2 * (size_t)s.n_nodes;
        nodes = (ref_tree ? s.ronodes : s.onodes) + oct_off;
        float te;
        float4 lo = ldg4(nodes), hi = ldg4(nodes + 1);
        if (!slab_presorted(lo, hi, r, te)) return false;
        cur = __float_as_int(lo.w);
        if (cur < 0) { shadow_leaf(s, r, dis, ~cur, acc); return false; }
        wide = !ref_tree;
        if (wide) nodes = s.wnodes + (WRT_WIDE_FLOAT4_PER_RECORD / 2) * oct_off;
        return true;
    }
    __device__ __forceinline__ bool step(int& cur, Stack& st) {
        const float never = INFINITY;
        bool more;
        if (wide) more = traverse_step4_defer<false>(nodes, r, st, cur, never, [&](int p) { shadow_leaf(s, r, dis, p, acc); });
        else more = traverse_step<false, true>(nodes, r, st, cur, never, [&](int p) { shadow_leaf(s, r, dis, p, acc); });
        return more && acc.res != 0.f;
    }
    __device__ __forceinline__ bool finish(int&, Stack&) {
        // three or more translucent crossings: the product in the reference tree's association (shadow_assoc.h)
        const float v = shadow_value(s, acc);
        if (WRT_IN_BOUNDS(out, (size_t)fb.n_node_cap * s.n_lights)) fb.coeff[out] = v;
        return false;
    }
};

__global__ void WRT_TRACE_BOUNDS k_shadow_hard(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb, int q, int work_slot, int refill,
                                               int literal) {
    extern __shared__ int smem[];
    Stack st;
    st.init(smem, threadIdx.x, blockDim.x);
    const unsigned n = queue_len(fb.counters, C_NPREQ + q, fb.preq_cap[q]);
    HardShadowQuery hq(s, fb, q, literal != 0);
    run_queue(hq, n, reinterpret_cast<unsigned long long*>(fb.counters + work_slot), st, refill);
}

// ---- K4b: soft shadows: 50 area-light samples per request (Renderer.hpp:405-414) ----
// Work item = (request, sample): consecutive items share the shading point, so a warp's
// rays start at one or two origins and stay coherent.  Each lit sample adds 1.0f to the
// request's coefficient (float atomics on small integers are exact and order-free).
// (Tracing a sample pair per lane from one Philox block was tried: 16 % slower — register
// pressure and a less coherent second walk; profiles/NOTES.md.)
struct SoftShadowQuery {
    const DevScene& s;
    const FrameBuffers& fb;
    unsigned seed;
    Ray r;
    const float4* nodes;
    float dis;
    bool occ;
    size_t out;
    int q;
    int last_occ;              // occluder cache: primitive that blocked this lane's previous ray, or -1
    bool use_cache;
    __device__ __forceinline__ SoftShadowQuery(const DevScene& s_, const FrameBuffers& fb_, unsigned seed_, int q_, bool cache)
        : s(s_), fb(fb_), seed(seed_), q(q_), last_occ(-1), use_cache(cache && !s_.has_light_prims) {}
    __device__ __forceinline__ bool begin(unsigned long long item, int& cur, Stack& st) {
        unsigned req = (unsigned)(item / WRT_SOFT_SAMPLES);
        unsigned sample = (unsigned)(item - (unsigned long long)req * WRT_SOFT_SAMPLES);
        float4 o4 = fb.preq_o[q][req];
        uint4 k = fb.preq_k[q][req];
        f3 v0, v1, v2;
        if (k.x < WRT_INLINE_LIGHTS) {                 // kernel-parameter constant bank
            const WrtLight& L = s.lights_c[k.x];
            v0 = mk3(L.tri[0], L.tri[1], L.tri[2]); v1 = mk3(L.tri[3], L.tri[4], L.tri[5]); v2 = mk3(L.tri[6], L.tri[7], L.tri[8]);
        } else {
            const WrtLight* L = s.lights + k.x;
            v0 = mk3(L->tri[0], L->tri[1], L->tri[2]); v1 = mk3(L->tri[3], L->tri[4], L->tri[5]); v2 = mk3(L->tri[6], L->tri[7], L->tri[8]);
        }
        float u, v;
        wrt_light_sample_uv(seed, k.y, k.z, k.x, sample, &u, &v);
        // randomSampleTriangle, Triangle.hpp:139-145: (1-u-v)*v0 + u*v1 + v*v2
        f3 lightPos = (1 - u - v) * v0 + u * v1 + v * v2;
        f3 orig = mk3(o4);
        f3 raydir = normalized(lightPos - orig);
        dis = norm(lightPos - orig);
        r = make_ray(orig, raydir);
        out = (size_t)__float_as_uint(o4.w) * (unsigned)s.n_lights + k.x;
        const bool degenerate = degenerate_dir(raydir);
        // octant copy: ray_octant() uses `d < 0` exactly like the reference's swap, so +-0 components pick the
        // unswapped planes and the presorted slab test equals BoundBox::IntersectRay for every ray
        nodes = (degenerate ? s.ronodes : s.onodes) + (size_t)ray_octant(raydir) * 2 * (size_t)s.n_nodes;
        if (use_cache && last_occ >= 0 && !degenerate) {
            if (occluder_cache_hit(s, r, dis, last_occ)) { occ = true; return false; }
            last_occ = -1;                                   // stale: do not pay for it again
        }
        return occluded_begin(s, nodes, r, dis, st, cur, occ);
    }
    __device__ __forceinline__ bool step(int& cur, Stack& st) {
        const float never = INFINITY;
        auto leaf = [&](int p) {
            occluded_leaf(s, r, dis, p, occ);
            if (occ) last_occ = p;
        };
        bool more = traverse_step<true, true>(nodes, r, st, cur, never, leaf);
        return more && !occ;
    }
    __device__ __forceinline__ bool finish(int&, Stack&) {
        if (!occ && WRT_IN_BOUNDS(out, (size_t)fb.n_node_cap * s.n_lights)) atomicAdd(fb.coeff + out, 1.0f);
        return false;
    }
};

__global__ void WRT_TRACE_BOUNDS k_shadow_soft(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb, int q, int work_slot,
                                               unsigned seed, int refill, int occluder_cache) {
    extern __shared__ int smem[];
    Stack st;
    st.init(smem, threadIdx.x, blockDim.x);
    const unsigned nreq = queue_len(fb.counters, C_NPREQ + q, fb.preq_cap[q]);
    SoftShadowQuery sq(s, fb, seed, q, occluder_cache != 0);
    run_queue(sq, (unsigned long long)nreq * WRT_SOFT_SAMPLES, reinterpret_cast<unsigned long long*>(fb.counters + work_slot),
              st, refill);
}

// ---- K4b': soft shadows through per-request candidate lists ----
// The 50 rays of a request share their origin and aim at one small light, so they cross almost the same
// nodes; k_shadow_soft pays that walk (descend from the root to the neighbourhood of the origin, ~20-30 node
// steps on the bunny's surface) 50 times.  Instead:
//   k_soft_lists      one lane per request walks the SAH tree ONCE with the conservative shaft test (shaft_cull.h)
//                     and writes the primitives whose leaf box some ray of the shaft may hit, nearest first, to a
//                     pool (bump allocation, one atomic per warp); the request keeps {offset, count}, count < 0 =
//                     trace ray by ray.
//   k_soft_list_rays  the queue's nreq x 50 rays are cut into warp passes of 32 consecutive rays, handed out 8 passes
//                     at a time from a global counter (balanced to ~10 us).  A ray tests only its request's list:
//                     own-box test (exact BoundBox::IntersectRay) + intersection test, first blocker ends it.
// Exact: a non-degenerate ray tests precisely the primitives whose own box it hits (DESIGN.md section 4), and
// those are all in the list, so OR over the list == the any-hit walk.  Requests whose list would exceed
// WRT_LIST_CAP, shafts without a definite axis, and axis-degenerate rays are traced by the ordinary per-ray
// walk.  Not used for scenes with light-avatar primitives (literal hasIntersection path).
// Tried and dropped (profiles/NOTES.md): one fused kernel in which a warp owns 32 requests from the walk to the last
// of their 1600 rays (19.1 vs 18.3 ms: ~0.4 ms of dependent work per batch, ~1.7 batches per warp on a deep level,
// long under-filled tail); 32-byte list entries carrying `plane - o` so that the ray kernel needs no box fetch
// (-11 % instructions, but 4x the DRAM traffic of both kernels: 18.4 ms); list build with per-lane refill (19.5 ms).
#ifndef WRT_LIST_CAP
#define WRT_LIST_CAP 192
#endif
struct SoftListBuffers {
    int*  scratch;        // WRT_LIST_CAP ints per thread of the grid: a walk writes here, then copies into the pool
    float* shafts;        // WRT_LISTS_CHUNK x WRT_SHAFT_SLOT floats per warp of the grid: the warp's ring of prepared shafts
    int*  pool;           // the lists
    int2* ref;            // per request: {pool offset, count}
    unsigned* work;       // k_soft_filter: the requests that need rays (non-empty list, or count < 0), compacted
    unsigned pool_cap;
};
#define WRT_LIST_CHUNK_PASSES 8
#define WRT_LISTS_CHUNK 128
#define WRT_LISTS_REFILL 8
#define WRT_SHAFT_SLOT 12         // floats a staged shaft occupies: o, ilo, ihi, octant | use, -, request index

// One lane walks one request's shaft, but walk lengths differ a lot (3 ... 400 node pairs; ncu: 8.6 of 32 lanes
// active when every lane takes one request and the warp waits for the longest).  So a finished lane keeps its list in its
// scratch column and goes idle; whenever WRT_LISTS_REFILL lanes are idle the WHOLE warp flushes the finished lists into the
// pool (coalesced copies, 32 entries per step — a lane copying its own list alone stalls the other 31: measured, 27 %
// slower than no refill at all) and hands the idle lanes new requests from a small ring of PREPARED requests, a per-warp
// slot array (global scratch, L1-resident).  All lanes build the ring's shafts (wrt_shaft_make, ~200 instructions, fully
// converged — set-up code on a few lanes at a time is what made a refill through run_queue slower than no refill at
// all), 32 requests per claim from the global counter, whenever the idle lanes outnumber the prepared requests.  A lane
// keeps the index of its request in a register: its ring slot may be reused while it is still walking.  Pool space is
// taken per flush (>= WRT_LISTS_REFILL lists, one atomic); an exhausted pool means count = -1 (per-ray walk).
// (A chunked form — a warp owns up to 128 consecutive requests, walks them all, then claims the next chunk — ends every
// chunk with its longest walk: on a short queue (one GPU's share of an 8-GPU frame: 2-3 requests per lane) a chunk is one
// request per lane, almost every chunk holds a request in shadow whose walk is 5x the average, and the lanes wait for it:
// 695 us for 0.5 M requests where the work is ~150 us.)
// (launch bound, with the 4-wide walk: 8 CTAs per SM = 63 registers, no spills: 2.86 ms per 4K frame; 10 CTAs = 48 registers,
// 24 bytes of spills: 3.13 ms; unbounded 80 registers: 5 CTAs.)
// (A per-leaf "own plane" test inside the walk — three quarters of the leaves a fully lit request finds are its own
// neighbours, which k_soft_filter then removes — was built and measured: the walk runs one lane per request, the test
// costs two dependent loads and ~40 instructions at that width: 6.3 ms against 3.1.  The same test a candidate per lane
// while the warp copies a finished list into the pool: 3.7 ms against 2.6 — the flush is the serial part of this kernel.
// The filter kernel, which spreads (request, candidate) pairs over all lanes, is the right place.)
#define WRT_LISTS_MIN_BLOCKS 8
__global__ void __launch_bounds__(128, WRT_LISTS_MIN_BLOCKS) k_soft_lists(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb, int q,
                                                        int work_slot, int stack_rows, SoftListBuffers lb) {
    extern __shared__ int smem[];
    Stack st;
    st.init(smem, threadIdx.x, blockDim.x);
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const unsigned nreq = queue_len(fb.counters, C_NPREQ + q, fb.preq_cap[q]);
    const size_t gwarp = (size_t)blockIdx.x * (blockDim.x >> 5) + warp;
    int* warp_scratch = lb.scratch + gwarp * 32 * WRT_LIST_CAP;
    int* mine = warp_scratch + (size_t)lane * WRT_LIST_CAP;
    float* slots = lb.shafts + gwarp * (size_t)WRT_LISTS_CHUNK * WRT_SHAFT_SLOT;     // ring of WRT_LISTS_CHUNK prepared requests
    unsigned long long* work = reinterpret_cast<unsigned long long*>(fb.counters + work_slot);
    unsigned* pool_head = fb.counters + C_POOL + q;
    unsigned n_empty = 0;
    unsigned head = 0, tail = 0;                             // warp-uniform: ring entries [head, tail) are prepared, not yet handed out
    bool drained = false;                                    // warp-uniform: the global queue has nothing left
    bool active = false;
    int pend = -2;                                           // finished walk waiting for the flush: list length, -1 = give up; -2 = nothing
    unsigned req = 0;                                        // the request this lane is walking / has walked
    WrtShaft sh;
    WrtShaftWalk w;
    w.nodes = s.onodes; w.cur = 0; w.sp = 0; w.n = 0;
    while (true) {
        const unsigned idle = __ballot_sync(0xffffffffu, !active);
        const bool more = !drained || head != tail;
        if (idle == 0xffffffffu || (more && __popc(idle) >= WRT_LISTS_REFILL)) {
            // ---- flush: the finished lists -> pool, all lanes copying ----
            __syncwarp();                                    // the lists other lanes wrote to their scratch columns are visible
            const int cnt = pend > 0 ? pend : 0;
            int incl = cnt;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                int v = __shfl_up_sync(0xffffffffu, incl, off);
                if (lane >= (unsigned)off) incl += v;
            }
            const unsigned total = (unsigned)__shfl_sync(0xffffffffu, incl, 31);
            if (total > 0) {
                unsigned first = 0xffffffffu;
                if (lane == 0 && *(volatile unsigned*)pool_head < lb.pool_cap) first = atomicAdd(pool_head, total);
                first = __shfl_sync(0xffffffffu, first, 0);
                const bool fits = first < lb.pool_cap && total <= lb.pool_cap - first;   // a full pool: count = -1, ray by ray
                const unsigned dst = first + (unsigned)(incl - cnt);
                unsigned todo = __ballot_sync(0xffffffffu, cnt > 0);
                while (todo) {
                    const int src_lane = __ffs(todo) - 1;
                    todo &= todo - 1;
                    const int c = __shfl_sync(0xffffffffu, cnt, src_lane);
                    const unsigned d0 = __shfl_sync(0xffffffffu, dst, src_lane);
                    if (fits) {
                        const int* src = warp_scratch + (size_t)src_lane * WRT_LIST_CAP;
                        for (int i = (int)lane; i < c; i += 32)
                            if (WRT_IN_BOUNDS(d0 + i, lb.pool_cap)) lb.pool[d0 + i] = src[i];
                    }
                }
                if (cnt > 0 && WRT_IN_BOUNDS(req, fb.preq_cap[q])) lb.ref[req] = fits ? make_int2((int)dst, cnt) : make_int2(0, -1);
            }
            if (pend == 0 || pend == -1) {                   // empty list (= lit, no rays needed) / give up (= ray by ray)
                if (WRT_IN_BOUNDS(req, fb.preq_cap[q])) lb.ref[req] = make_int2(0, pend);
                if (pend == 0) ++n_empty;
            }
            pend = -2;
            __syncwarp();                                    // the scratch columns are free again
            // ---- top up the ring: 32 requests per claim, shafts built by all lanes ----
            const unsigned need = __popc(idle);
            while (!drained && tail - head < need) {
                unsigned long long claimed = 0;
                if (lane == 0) claimed = atomicAdd(work, 32ull);
                claimed = __shfl_sync(0xffffffffu, claimed, 0);
                if (claimed >= nreq) { drained = true; break; }
                const unsigned base = (unsigned)claimed;
                const unsigned n = nreq - base < 32u ? nreq - base : 32u;
                if (lane < n) {
                    const float4 o4 = fb.preq_o[q][base + lane];
                    const uint4 k = fb.preq_k[q][base + lane];
                    const WrtLight* L = s.lights + k.x;
                    float tri[9];
                    for (int i = 0; i < 9; i++) tri[i] = L->tri[i];
                    const float o[3] = {o4.x, o4.y, o4.z};
                    WrtShaft t;
                    const bool ok = wrt_shaft_make(o, tri, &t);
                    float* d = slots + (size_t)((tail + lane) % WRT_LISTS_CHUNK) * WRT_SHAFT_SLOT;
                    d[0] = t.o[0]; d[1] = t.o[1]; d[2] = t.o[2];
                    d[3] = t.ilo[0]; d[4] = t.ilo[1]; d[5] = t.ilo[2];
                    d[6] = t.ihi[0]; d[7] = t.ihi[1]; d[8] = t.ihi[2];
                    d[9] = __int_as_float(ok ? (t.octant | (t.use << 3)) : -1);
                    d[10] = 0.f;
                    d[11] = __uint_as_float(base + lane);
                }
                tail += n;
                __syncwarp();
            }
            // ---- hand the prepared requests to the idle lanes ----
            {
                const unsigned avail = tail - head;
                const unsigned rank = __popc(idle & lt_mask);
                if (!active && rank < avail) {
                    const float* d = slots + (size_t)((head + rank) % WRT_LISTS_CHUNK) * WRT_SHAFT_SLOT;
                    const int ou = __float_as_int(d[9]);
                    req = __float_as_uint(d[11]);
                    int rc = -1;
                    if (ou >= 0) {
                        sh.o[0] = d[0]; sh.o[1] = d[1]; sh.o[2] = d[2];
                        sh.ilo[0] = d[3]; sh.ilo[1] = d[4]; sh.ilo[2] = d[5];
                        sh.ihi[0] = d[6]; sh.ihi[1] = d[7]; sh.ihi[2] = d[8];
                        sh.octant = ou & 7; sh.use = ou >> 3;
                        rc = wrt_shaft_walk_begin4(s.onodes, s.wnodes, s.n_nodes, &sh, &w);
                    }
                    if (rc == 1) active = true;
                    else pend = rc;                          // answered without a walk; recorded by the next flush
                }
                head += need < avail ? need : avail;
                __syncwarp();                                // the slots just read may be rewritten by the next top-up
            }
            if (!__any_sync(0xffffffffu, active)) {
                if (drained && head == tail && !__any_sync(0xffffffffu, pend != -2)) break;
                continue;
            }
        }
#pragma unroll 1
        for (int it = 0; it < 4; it++) {
            if (active) {
                const int rc = wrt_shaft_walk_step4(&sh, &w, st.base, st.stride, stack_rows, mine, WRT_LIST_CAP);
                if (rc != 1) { active = false; pend = rc < 0 ? -1 : w.n; }
            }
        }
    }
    n_empty = __reduce_add_sync(0xffffffffu, n_empty);
    if (lane == 0 && n_empty) atomicAdd(fb.counters + C_NEMPTY, n_empty);
}

// ---- K4b'': triangle-level pruning of the candidate lists (shaft_cull.h, wrt_pyramid_*) ----
// The lists hold every primitive whose BOX a ray of the shaft may hit.  On the bunny's surface half of those triangles
// cannot be hit by any ray of the request (they lie outside the pyramid origin -> light, or the pyramid lies on one side of
// their plane); every one of them would cost each of the request's 50 rays an own-box test, often a triangle test.  One warp
// per request drops them (ballot compaction, in place, order kept).  A quarter of the fully lit deep requests end up
// with an empty list and need no rays at all.  Exact: a removed triangle blocks no sample ray (proof obligations and the
// brute-force check: shaft_cull.h, tests/shaft_cull_check.cpp).
#define WRT_FILTER_MIN 1          // every non-empty list: with the edge planes most 1- and 2-member lists of fully lit requests
                                  // come out empty and their 50 rays are never built (3 / 2 / 1: 14.19 / 13.64 / 13.57 ms per 4K frame)
// A warp takes 32 consecutive requests: (A) each lane builds its request's pyramid (4 cross products, 8 square roots, 4
// divisions — once per request, not once per candidate) into shared memory; (B) the 32 lists are treated as ONE sequence
// of (request, candidate) pairs, 32 pairs per step, one per lane: most lists of fully lit requests hold 1-4 candidates, and
// a warp that took the lists one after the other (round 2's first version: 18 of 32 lanes, lane-issue utilisation 0.23)
// idled on them.  A lane finds its pair's request by binary search over the lists' start offsets, loads geometry + the
// primitive's precomputed plane normal and edge scale (DevScene::tri_aux) and the request's pyramid (row stride 33 words:
// lanes on different requests hit different banks), runs the tests, and the survivors are compacted in place, order
// kept: rank = kept-so-far of the request (shared memory) + survivors of the same request on lower lanes
// (__match_any_sync).  A request's write cursor never passes its read cursor, and every step reads before it writes.
// (no minimum-blocks bound: the pyramid spills under one)
#define WRT_FILTER_EDGE_MAX 16    // survivor lists up to this length get the edge-plane stage
// One pass of k_soft_filter over the lists of a warp's 32 requests (lane r <-> request r): kept[r] entries of list r
// (request r takes part iff `take`), all lists as one sequence of pairs, 32 per step; survivors compacted in place.
template <int STAGE>
__device__ __forceinline__ void filter_pass(const DevScene& s, const SoftListBuffers& lb, const float (*py_rows)[WRT_PYRAMID_FLOATS + 1],
                                            int* start, const int* offs, int* kept, unsigned lane, bool take) {
    const unsigned lt_mask = (1u << lane) - 1u;
    const int cnt = take ? kept[lane] : 0;
    int incl = cnt;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= (unsigned)off) incl += v;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    if (total == 0) return;
    __syncwarp();
    start[lane] = incl - cnt;
    if (lane == 31) start[32] = total;
    if (take) kept[lane] = 0;
    __syncwarp();
    for (int g0 = 0; g0 < total; g0 += 32) {
        const int g = g0 + (int)lane;
        unsigned r = 0xffffffffu;
        int prim = -1, off = 0;
        bool keep = false;
        if (g < total) {
            int lo = 0, hi = 31;                       // last request whose start offset is <= g (empty lists share a start)
#pragma unroll
            for (int it = 0; it < 5; it++) {
                const int mid = (lo + hi + 1) >> 1;
                if (start[mid] <= g) lo = mid; else hi = mid - 1;
            }
            r = (unsigned)lo;
            off = offs[lo];
            prim = lb.pool[off + (g - start[lo])];
            WrtShaftPyramid py;
            const float* d = py_rows[lo];
            py.o[0] = d[0]; py.o[1] = d[1]; py.o[2] = d[2];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                py.D[j][0] = d[3 + 3 * j]; py.D[j][1] = d[4 + 3 * j]; py.D[j][2] = d[5 + 3 * j];
                py.Dlen[j] = d[15 + j];
                py.N[j][0] = d[19 + 3 * j]; py.N[j][1] = d[20 + 3 * j]; py.N[j][2] = d[21 + 3 * j];
            }
            py.ok = 1;
            const float4* gm = s.geom + 3 * (size_t)prim;
            const float4 A = ldg4(gm), B = ldg4(gm + 1), C = ldg4(gm + 2), X = ldg4(s.tri_aux + prim);
            const float v0[3] = {A.x, A.y, A.z}, E1[3] = {B.x, B.y, B.z}, E2[3] = {C.x, C.y, C.z};
            const float aux[4] = {X.x, X.y, X.z, X.w};
            keep = STAGE == 0 ? wrt_pyramid_triangle_may_block(&py, v0, E1, E2, aux) : wrt_pyramid_triangle_may_block_edges(&py, v0, E1, E2, aux);
        }
        const unsigned same = __match_any_sync(0xffffffffu, r);            // lanes working on the same request
        const unsigned kmask = __ballot_sync(0xffffffffu, keep) & same;
        const int kept0 = r != 0xffffffffu ? kept[r] : 0;
        __syncwarp();                                  // every lane has read its entry and its request's cursor
        if (keep && WRT_IN_BOUNDS((unsigned)off + kept0 + __popc(kmask & lt_mask), lb.pool_cap))
            lb.pool[off + kept0 + __popc(kmask & lt_mask)] = prim;
        if (r != 0xffffffffu && (same & lt_mask) == 0u) kept[r] = kept0 + __popc(kmask);
        __syncwarp();
    }
}

#define WRT_FILTER_MIN_BLOCKS 8   // 64 registers, no spills (unbounded: 70 registers, 7 CTAs per SM, 1.51 against 1.44 ms)
#define WRT_FILTER_BOUNDS __launch_bounds__(128, WRT_FILTER_MIN_BLOCKS)
// Work distribution: blocks of 32 requests are claimed from a global counter (the host sizes the grid to what is
// resident).  The static round-robin over 8 CTAs per SM it replaces ran in two waves — 7 CTAs of 72 registers fit —
// the second one with a single CTA per SM (ncu: 22-31 % achieved occupancy of 44 % possible).
__global__ void WRT_FILTER_BOUNDS k_soft_filter(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb, int q,
                                                     SoftListBuffers lb, int work_slot) {
    __shared__ float s_py[4][32][WRT_PYRAMID_FLOATS + 1];
    __shared__ int s_start[4][33], s_off[4][32], s_kept[4][32];
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const unsigned nreq = queue_len(fb.counters, C_NPREQ + q, fb.preq_cap[q]);
    const unsigned warps = gridDim.x * (blockDim.x >> 5);
    unsigned n_empty = 0;
    unsigned long long* work = reinterpret_cast<unsigned long long*>(fb.counters + work_slot);
    // requests per claim: 32 (one per lane) on a long queue; on a short one — a rank's share of a multi-GPU frame holds
    // less than a block per warp — 16 or 8, so that the launch does not end with the one warp that drew 32 long lists
    const unsigned per_claim = nreq >= warps * 64u ? 32u : (nreq >= warps * 16u ? 16u : 8u);
    while (true) {
        unsigned long long claimed = 0;
        if (lane == 0) claimed = atomicAdd(work, (unsigned long long)per_claim);
        claimed = __shfl_sync(0xffffffffu, claimed, 0);
        if (claimed >= nreq) break;
        const unsigned base = (unsigned)claimed;
        const unsigned lim = base + per_claim < nreq ? base + per_claim : nreq;    // this claim's requests end here
        // ---- A ----
        const unsigned req = base + lane;
        int2 ref = make_int2(0, 0);
        bool ok = false;
        size_t out = 0;
        if (req < lim) {
            ref = lb.ref[req];
            const float4 o4 = fb.preq_o[q][req];
            const uint4 k = fb.preq_k[q][req];
            out = (size_t)__float_as_uint(o4.w) * (unsigned)s.n_lights + k.x;
            if (ref.y >= WRT_FILTER_MIN) {
                const WrtLight* L = s.lights + k.x;
                float tri[9];
                for (int i = 0; i < 9; i++) tri[i] = L->tri[i];
                const float o[3] = {o4.x, o4.y, o4.z};
                WrtShaftPyramid py;
                wrt_pyramid_make(o, tri, &py);
                ok = py.ok != 0;
                float* d = s_py[warp][lane];
                d[0] = py.o[0]; d[1] = py.o[1]; d[2] = py.o[2];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    d[3 + 3 * j] = py.D[j][0]; d[4 + 3 * j] = py.D[j][1]; d[5 + 3 * j] = py.D[j][2];
                    d[15 + j] = py.Dlen[j];
                    d[19 + 3 * j] = py.N[j][0]; d[20 + 3 * j] = py.N[j][1]; d[21 + 3 * j] = py.N[j][2];
                }
            }
        }
        s_off[warp][lane] = ref.x;
        s_kept[warp][lane] = ok ? ref.y : 0;
        __syncwarp();
        // ---- B: first stage (side planes, own plane) on every list; second stage (edge planes) on the short survivor
        // lists only — those of fully lit requests, which it empties ----
        filter_pass<0>(s, lb, s_py[warp], s_start[warp], s_off[warp], s_kept[warp], lane, ok);
        filter_pass<1>(s, lb, s_py[warp], s_start[warp], s_off[warp], s_kept[warp], lane, ok && s_kept[warp][lane] <= WRT_FILTER_EDGE_MAX);
        int final_cnt = ref.y;                             // 0: empty already; < 0: ray by ray; else a list this kernel left alone
        if (ok) {
            final_cnt = s_kept[warp][lane];
            lb.ref[req] = make_int2(ref.x, final_cnt);
            if (final_cnt == 0) ++n_empty;                 // lit, and no ray needs to be built (statistics)
        }
        // ---- C: an empty list answers the request (all samples lit: the coefficient's start value 0 + 50, what the ray
        // kernel's atomics would add up to); the others go, compacted, to the ray kernel's work list ----
        const bool live = req < lim;
        if (live && final_cnt == 0 && WRT_IN_BOUNDS(out, (size_t)fb.n_node_cap * s.n_lights)) fb.coeff[out] = (float)WRT_SOFT_SAMPLES;
        const unsigned need = __ballot_sync(0xffffffffu, live && final_cnt != 0);
        if (need) {
            unsigned w0 = 0;
            if (lane == 0) w0 = atomicAdd(fb.counters + C_NWORK + q, (unsigned)__popc(need));
            w0 = __shfl_sync(0xffffffffu, w0, 0);
            if (((need >> lane) & 1u) && WRT_IN_BOUNDS(w0 + __popc(need & lt_mask), fb.preq_cap[q])) lb.work[w0 + __popc(need & lt_mask)] = req;
        }
        __syncwarp();                                      // the pyramids are rebuilt by the next block of requests
    }
    n_empty = __reduce_add_sync(0xffffffffu, n_empty);
    if (lane == 0 && n_empty) atomicAdd(fb.counters + C_NEMPTY, n_empty);
}

// use_work != 0: k_soft_filter ran on this queue — it answered the requests whose list is empty and left the ids of the
// others in lb.work; the passes then run over those only (9 of 10 queued deep requests of the metric frame end up empty).
__global__ void WRT_TRACE_BOUNDS k_soft_list_rays(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb, int q,
                                                  int work_slot, unsigned seed, SoftListBuffers lb, int use_work) {
    extern __shared__ int smem[];
    Stack st;
    st.init(smem, threadIdx.x, blockDim.x);
    const unsigned lane = threadIdx.x & 31;
    const unsigned nreq = use_work ? queue_len(fb.counters, C_NWORK + q, fb.preq_cap[q])
                                   : queue_len(fb.counters, C_NPREQ + q, fb.preq_cap[q]);   // host guarantees nreq * 50 < 2^32
    const unsigned n_rays = nreq * WRT_SOFT_SAMPLES, n_pass = (n_rays + 31u) / 32u;
    unsigned long long* work = reinterpret_cast<unsigned long long*>(fb.counters + work_slot);
    // passes per claim: WRT_LIST_CHUNK_PASSES on a long queue, fewer when the launch holds less than four such claims per warp
    // (a rank's share of a multi-GPU frame: the launch then ends with its last claim, not with the warp that drew two)
    const unsigned warps_total = gridDim.x * (blockDim.x >> 5);
    const unsigned chunk_passes = n_pass >= warps_total * 4u * WRT_LIST_CHUNK_PASSES ? (unsigned)WRT_LIST_CHUNK_PASSES
                                  : (n_pass >= warps_total * 8u ? 2u : 1u);
    while (true) {
        unsigned long long claimed = 0;
        if (lane == 0) claimed = atomicAdd(work, (unsigned long long)chunk_passes);
        claimed = __shfl_sync(0xffffffffu, claimed, 0);
        if (claimed >= n_pass) break;
        const unsigned p0 = (unsigned)claimed, p1 = p0 + chunk_passes < n_pass ? p0 + chunk_passes : n_pass;
#pragma unroll 1
        for (unsigned pass = p0; pass < p1; pass++) {
            const unsigned j = pass * 32u + lane;
            const unsigned w = j / WRT_SOFT_SAMPLES, sample = j - w * WRT_SOFT_SAMPLES;      // w: position in the work sequence
            const unsigned req = w < nreq ? (use_work ? lb.work[w] : w) : 0u;
            bool lit = false;
            size_t out = 0;
            const int2 ref = w < nreq ? lb.ref[req] : make_int2(0, 0);
            if (w < nreq && ref.y == 0) {
                // empty list = no leaf box can be hit by any sample of this request (shaft_cull.h, axis-degenerate
                // samples included): lit, and the ray itself is never needed
                out = (size_t)__float_as_uint(fb.preq_o[q][req].w) * (unsigned)s.n_lights + fb.preq_k[q][req].x;
                lit = true;
            } else if (w < nreq) {
                float4 o4 = fb.preq_o[q][req];
                uint4 k = fb.preq_k[q][req];
                f3 v0, v1, v2;
                if (k.x < WRT_INLINE_LIGHTS) {
                    const WrtLight& L = s.lights_c[k.x];
                    v0 = mk3(L.tri[0], L.tri[1], L.tri[2]); v1 = mk3(L.tri[3], L.tri[4], L.tri[5]); v2 = mk3(L.tri[6], L.tri[7], L.tri[8]);
                } else {
                    const WrtLight* L = s.lights + k.x;
                    v0 = mk3(L->tri[0], L->tri[1], L->tri[2]); v1 = mk3(L->tri[3], L->tri[4], L->tri[5]); v2 = mk3(L->tri[6], L->tri[7], L->tri[8]);
                }
                float u, v;
                wrt_light_sample_uv(seed, k.y, k.z, k.x, sample, &u, &v);
                f3 lightPos = (1 - u - v) * v0 + u * v1 + v * v2;                 // Triangle.hpp:139-145
                f3 orig = mk3(o4);
                f3 raydir = normalized(lightPos - orig);
                const float dis = norm(lightPos - orig);
                const Ray r = make_ray(orig, raydir);
                out = (size_t)__float_as_uint(o4.w) * (unsigned)s.n_lights + k.x;
                bool occ = false;
                if (ref.y < 0 || degenerate_dir(raydir)) {
                    occ = occluded(s, degenerate_dir(raydir) ? s.nodes : s.fnodes, r, dis, st);
                } else {
                    const int* list = lb.pool + ref.x;
                    // occ = OR over the list of (own box hit && intersection accepted && t < dis): the same conjunction with
                    // the intersection test first.  k_soft_filter leaves candidates that can really block, so 7 of 10 box
                    // tests pass and the warp runs the intersection code in every iteration anyway; the box test (two
                    // fetches, 25 instructions) is then only needed to confirm a blocker.
                    for (int c = 0; c < ref.y && !occ; c++) {
                        const int p = list[c];
                        PrimHit h; float oma; unsigned fl;
                        if (prim_test(s, p, r, h, oma, fl) && h.t < dis) {
                            float te;
                            float4 blo, bhi;
                            ldg8(s.prim_box + 2 * (size_t)p, blo, bhi);
                            occ = slab(blo, bhi, r, te);
                        }
                    }
                }
                lit = !occ;
            }
            // one float atomic per request segment of the pass (small integer sums are exact and order-free)
            const unsigned lit_mask = __ballot_sync(0xffffffffu, lit);
            const unsigned rq0 = (pass * 32u) / WRT_SOFT_SAMPLES;
            const unsigned first = __ballot_sync(0xffffffffu, w == rq0);         // lanes of the pass's first request
            const unsigned mine = w == rq0 ? first : ~first;
            const unsigned n_lit = __popc(lit_mask & mine);
            if (n_lit && lane == (unsigned)(__ffs(mine) - 1) && WRT_IN_BOUNDS(out, (size_t)fb.n_node_cap * s.n_lights))
                atomicAdd(fb.coeff + out, (float)n_lit);
        }
    }
}

// ---- K4c: directional-light shadows, Renderer.hpp:381-400 (dilated-tree culling, dev_traverse.cuh) ----
// literal != 0 (WRT_TRAVERSAL_EXHAUSTIVE): the reference's own O(N) loop over objList.
// (The same walk on persistent warps with per-lane refill was built and measured: 12.7 instead of 9.4 lanes, but 3.04 ms
// against 2.63 for the directional requests of f4_directional_4k — the sorted hit buffer and the query state go to local memory.)
__global__ void __launch_bounds__(128) k_shadow_directional(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb,
                                                            int q, int literal) {
    extern __shared__ int smem[];
    Stack st;
    st.init(smem, threadIdx.x, blockDim.x);
    const unsigned n = queue_len(fb.counters, C_NDREQ + q, fb.dreq_cap[q]);
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 o4 = fb.dreq_o[q][i];
        uint4 k = fb.dreq_k[q][i];
        const WrtLight* L = s.lights + k.x;
        f3 negDir = mk3(-L->pos[0], -L->pos[1], -L->pos[2]);
        Ray r = make_ray(mk3(o4), normalized(negDir));
        const size_t out = (size_t)__float_as_uint(o4.w) * s.n_lights + k.x;
        const float c = literal ? directional_product(s, r, (int)k.y) : directional_product_bvh(s, r, (int)k.y, st);
        if (WRT_IN_BOUNDS(out, (size_t)fb.n_node_cap * s.n_lights)) fb.coeff[out] = c;
    }
}

// ---- K5: local shading, Renderer::blinnPhongShader ----
__device__ __forceinline__ void shade_node(const DevScene& s, const FrameBuffers& fb, unsigned g) {
    const float4* sv = fb.surf + 4 * (size_t)g;
    float4 s0 = sv[0];
    if (__float_as_int(s0.w) < 0) return;
    float4 s1 = sv[1], s2 = sv[2], s3 = sv[3];
    Mtl m = load_material(s, __float_as_int(s1.w));
    m.diffuse = mk3(s2);
    f3 local = blinn_phong(s, mk3(s3), mk3(s0), mk3(s1), m, fb.coeff + (size_t)g * s.n_lights);
    float4 na = fb.node_a[g];
    na.x = local.x; na.y = local.y; na.z = local.z;
    fb.node_a[g] = na;
}

// Shades the nodes of levels [level_lo, level_hi] in one sweep (the levels' spans concatenated).
__device__ __forceinline__ void shade_levels(const DevScene& s, const FrameBuffers& fb, unsigned n0, int level_lo, int level_hi) {
    for (int level = level_lo; level <= level_hi; level++) {
        const LevelSpan span = level_span(fb, level, n0);
        const unsigned n = span.count();
        for (unsigned item = blockIdx.x * blockDim.x + threadIdx.x; item < n; item += gridDim.x * blockDim.x)
            shade_node(s, fb, node_id(fb, level, span.slot(item)));
    }
}

__global__ void __launch_bounds__(256) k_shade(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb, unsigned n0,
                                               int level_lo, int level_hi) {
    shade_levels(s, fb, n0, level_lo, level_hi);
}

// ---- K6 + K7: bottom-up combine (Renderer.hpp:259) and 8-bit resolve (Renderer.hpp:128-130) ----
// One cooperative launch: shade the levels no k_shade launch has covered (shade_from .. 8), then walk the levels
// 8 -> 0 with a grid-wide barrier between them (each level reads the finished colours of the level below), then
// quantise level 0.
__device__ __forceinline__ void combine_level(const FrameBuffers& fb, int level, unsigned n0) {
    const LevelSpan span = level_span(fb, level, n0);
    const unsigned n = span.count();
    for (unsigned item = blockIdx.x * blockDim.x + threadIdx.x; item < n; item += gridDim.x * blockDim.x) {
        const unsigned g = node_id(fb, level, span.slot(item));
        float4 nb = fb.node_b[g];
        if (nb.w == 0.f) continue;                       // miss / light avatar: returned as is
        float4 na = fb.node_a[g];
        int cR = __float_as_int(nb.y), cT = __float_as_int(nb.z);
        f3 R = mk3(0.f, 0.f, 0.f), T = R;
        if (cR >= 0) R = mk3(fb.node_a[cR]);
        if (cT >= 0) T = mk3(fb.node_a[cT]);
        f3 c = mk3(na) + na.w * R + nb.x * T;            // blinnPhongRes + fr * R_lambda + (1-fr)(1-alpha) * T_lambda
        fb.node_a[g] = make_float4(c.x, c.y, c.z, na.w);
    }
}

__device__ __forceinline__ unsigned char quantize(float c) {   // int(255 * std::min(c, 1.f)), truncating
    float m = (1.f < c) ? 1.f : c;
    int q = (int)(255 * m);
    return (unsigned char)(q < 0 ? 0 : (q > 255 ? 255 : q));
}

// image != nullptr: row-major image (may live on a peer GPU: multi-GPU contexts store straight into device 0's
// frame over NVLink); packed != nullptr: tile-order buffer (NCCL gather)
__global__ void __launch_bounds__(256) k_combine_resolve(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb,
                                                         const __grid_constant__ TileMap tm, long long slot0, unsigned n, int shade_from,
                                                         unsigned char* image, unsigned char* packed) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    if (shade_from < WRT_MAX_DEPTH) {
        shade_levels(s, fb, n, shade_from, WRT_MAX_DEPTH - 1);
        grid.sync();
    }
    for (int level = WRT_MAX_DEPTH - 1; level >= 0; level--) {
        // (a level without rays has nothing to combine and nothing below it either, but every CTA must take
        // part in the same number of barriers)
        combine_level(fb, level, n);
        if (level > 0) grid.sync();
    }
    // level 0: every thread quantises the nodes it has just combined (same grid-stride mapping), no barrier needed
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 c = fb.node_a[i];
        unsigned char r = quantize(c.x), g = quantize(c.y), b = quantize(c.z);
        if (packed) {
            unsigned char* p = packed + 3 * (size_t)(slot0 + i);
            p[0] = r; p[1] = g; p[2] = b;
        }
        int x, y;
        if (image && tm.slot_to_pixel(slot0 + i, tm.rank, x, y)) {
            unsigned char* p = image + 3 * ((size_t)y * tm.width + x);
            p[0] = r; p[1] = g; p[2] = b;
        }
    }
}

// ---- rank-0 de-interleave after the NCCL gather ----
__global__ void __launch_bounds__(256) k_scatter_tiles(const unsigned char* gathered, long long stride_bytes, TileMap tm,
                                                       int world, long long slots_per_rank, unsigned char* image) {
    long long total = slots_per_rank * world;
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
        int r = (int)(g / slots_per_rank);
        long long slot = g - (long long)r * slots_per_rank;
        int x, y;
        if (tm.slot_to_pixel(slot, r, x, y)) {
            const unsigned char* p = gathered + (size_t)r * stride_bytes + 3 * (size_t)slot;
            unsigned char* q = image + 3 * ((size_t)y * tm.width + x);
            q[0] = p[0]; q[1] = p[1]; q[2] = p[2];
        }
    }
}

// ======================= batch forms of the strategy queries =======================

// Intersection record of a finished closest-hit query (what UpdateInter leaves in the reference's Intersection)
__device__ __forceinline__ WrtHit hit_record(const DevScene& s, f3 o, f3 d, const Closest& c) {
    WrtHit h;
    h.hit = 0; h.object = -1; h.t = FLT_MAX; h.pos[0] = h.pos[1] = h.pos[2] = 0.f;
    h.ndir[0] = h.ndir[1] = h.ndir[2] = 0.f; h.uv[0] = h.uv[1] = -1.f;
    h.texture = -1; h.normalmap = -1; h.material = -1; h.prim = -1;
    if (c.prim >= 0) {
        Surface sf = complete_hit(s, o, d, c.t, c.prim, c.u, c.v);
        h.hit = 1; h.prim = c.prim; h.object = __ldg(s.ids + c.prim).w; h.t = c.t;
        h.pos[0] = sf.pos.x; h.pos[1] = sf.pos.y; h.pos[2] = sf.pos.z;
        h.ndir[0] = sf.nDir.x; h.ndir[1] = sf.nDir.y; h.ndir[2] = sf.nDir.z;
        h.uv[0] = sf.u; h.uv[1] = sf.v; h.texture = sf.textureIndex; h.normalmap = sf.normalMapIndex;
        h.material = sf.material;
    }
    return h;
}

__global__ void __launch_bounds__(128) k_batch_closest(DevScene s, const float* orig, const float* dir, long long n,
                                                       WrtHit* out, float prune_rel) {
    extern __shared__ int smem[];
    Stack st;
    st.init(smem, threadIdx.x, blockDim.x);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        f3 o = mk3(orig[3 * i], orig[3 * i + 1], orig[3 * i + 2]);
        f3 d = mk3(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
        Closest c;
        c.t = FLT_MAX; c.prim = -1; c.u = 0.f; c.v = 0.f;
        if (s.n_nodes > 0) {
            Ray r = make_ray(o, d);
            float prune = prune_rel;
            const float4* nodes = pick_tree(s, d, prune);
            c = closest_hit(s, nodes, 0, r, st, prune);
        }
        out[i] = hit_record(s, o, d, c);
    }
}

// ---- the same query answered by the FRAME's deep-level kernel (wrt_trace_closest_wavefront: the parity tests put
// their ray batches through k_trace_closest<false> itself — octant copies, 4-wide nodes, deferred leaves, lane refill) ----
__global__ void __launch_bounds__(256) k_pack_rays(const float* orig, const float* dir, unsigned n, float4* ray_o, float4* ray_d,
                                                   unsigned* counters, int level) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        ray_o[i] = make_float4(orig[3 * (size_t)i], orig[3 * (size_t)i + 1], orig[3 * (size_t)i + 2], __uint_as_float(i));
        ray_d[i] = make_float4(dir[3 * (size_t)i], dir[3 * (size_t)i + 1], dir[3 * (size_t)i + 2], __uint_as_float(1u));
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) counters[C_NRAYS + level] = n;     // all in the level's first (reflection) half
}

__global__ void __launch_bounds__(256) k_unpack_hits(const __grid_constant__ DevScene s, const float* orig, const float* dir, unsigned n,
                                                     const float4* hit, WrtHit* out) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const f3 o = mk3(orig[3 * (size_t)i], orig[3 * (size_t)i + 1], orig[3 * (size_t)i + 2]);
        const f3 d = mk3(dir[3 * (size_t)i], dir[3 * (size_t)i + 1], dir[3 * (size_t)i + 2]);
        const float4 h = hit[i];
        Closest c;
        c.t = h.x; c.prim = __float_as_int(h.y); c.u = h.z; c.v = h.w;
        out[i] = hit_record(s, o, d, c);
    }
}

// ---- per-pixel surface planes of level 0 (wrt_render_gbuffer, wrt_render_gbuffer_device) ----
// Two output modes.  row_major == 0: slot i of the batch goes to element i of one batch's slot-ordered staging (the host
// form scatters it to pixels).  row_major != 0: it goes to its pixel y * W + x of the caller's row-major W x H plane
// (PrimaryGen::tm, slot0: the batch's tile map); padding slots have no pixel and are skipped.
// k_gbuffer_hit runs right after level 0's k_surface_spawn: level 1's k_trace_closest overwrites fb.hit.  The record is
// the one k_unpack_hits builds, from the eye ray regenerated as k_trace_closest<true> generated it (a padding slot gets a
// miss record in slot order; it has no pixel).
__global__ void __launch_bounds__(256) k_gbuffer_hit(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb,
                                                     const __grid_constant__ PrimaryGen pg, unsigned n, int row_major, WrtHit* out) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        f3 o, d;
        unsigned pixel;
        const bool live = primary_ray(pg, i, o, d, pixel);
        if (row_major && !live) continue;
        const float4 h = fb.hit[i];
        Closest c;
        c.t = h.x; c.prim = __float_as_int(h.y); c.u = h.z; c.v = h.w;
        const WrtHit rec = hit_record(s, o, d, c);
        if (!row_major) out[i] = rec;
        else if (WRT_IN_BOUNDS(pixel, (size_t)pg.cam.width * pg.cam.height)) out[pixel] = rec;
    }
}

// k_gbuffer_surface runs after k_combine_resolve (level 0's shadow kernels have finished; nothing after surface_warp
// rewrites a level-0 surface record or coefficient).  A shaded node (surf[4g].w holds a primitive >= 0) exports what
// surface_warp stored: the shading normal after changeNormalDir, Od, and per light the coefficient blinn_phong
// multiplies (soft point lights: lit samples / 50, as blinn_phong divides).  A light < 32 whose terms vanish was never
// given a coefficient when level 0 ran with WRT_CULL_UNLIT: light_terms_vanish on surface_warp's inputs finds it again,
// and it reads -1.  Unshaded nodes (miss, light avatar, padding): normal and albedo 0, every coefficient -1.
// rgb_f (row-major mode only): the combined level-0 colour k_combine_resolve quantised, fb.node_a[g].xyz.
// NULL planes are skipped.
__global__ void __launch_bounds__(256) k_gbuffer_surface(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb,
                                                         const __grid_constant__ TileMap tm, long long slot0, unsigned n, int cull,
                                                         int row_major, float* normal, float* albedo, float* shadow, float* rgb_f) {
    for (unsigned g = blockIdx.x * blockDim.x + threadIdx.x; g < n; g += gridDim.x * blockDim.x) {
        size_t p = g;                                  // the output element of this node
        if (row_major) {
            int x, y;
            if (!tm.slot_to_pixel(slot0 + g, tm.rank, x, y)) continue;
            p = (size_t)y * tm.width + x;
            if (!WRT_IN_BOUNDS(p, (size_t)tm.width * tm.height)) continue;
        }
        if (rgb_f) {
            const float4 c = fb.node_a[g];
            rgb_f[3 * p] = c.x; rgb_f[3 * p + 1] = c.y; rgb_f[3 * p + 2] = c.z;
        }
        const float4* sv = fb.surf + 4 * (size_t)g;
        const float4 s0 = sv[0];
        const bool shaded = __float_as_int(s0.w) >= 0;
        const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 s1 = shaded ? sv[1] : zero, s2 = shaded ? sv[2] : zero;
        if (normal) { normal[3 * p] = s1.x; normal[3 * p + 1] = s1.y; normal[3 * p + 2] = s1.z; }
        if (albedo) { albedo[3 * p] = s2.x; albedo[3 * p + 1] = s2.y; albedo[3 * p + 2] = s2.z; }
        if (!shadow) continue;
        const f3 pos = mk3(s0), nDir = mk3(s1);
        const bool unlit_cull = shaded && (cull & WRT_CULL_UNLIT);
        f3 p_eye_dir = mk3(0.f, 0.f, 0.f);
        float shade_n = 0.f;
        if (unlit_cull) {
            p_eye_dir = normalized(mk3(sv[3]) - pos);
            shade_n = load_material(s, __float_as_int(s1.w)).n;
        }
        for (int li = 0; li < s.n_lights; li++) {
            const WrtLight* L = s.lights + li;
            float v = -1.f;
            if (shaded && !(unlit_cull && li < 32 && light_terms_vanish(L, p_eye_dir, pos, nDir, shade_n))) {
                v = fb.coeff[(size_t)g * s.n_lights + li];
                if (float_equal(L->pos[3], 1.f) && s.shadow_type != 0) v = v / (float)WRT_SOFT_SAMPLES;
            }
            shadow[p * s.n_lights + li] = v;
        }
    }
}

// ---- shadow requests answered by the FRAME's shadow kernels (wrt_shadow_requests_wavefront: the tests put their
// requests through k_shadow_hard, the candidate-list kernels, k_shadow_soft and k_shadow_directional themselves) ----
struct ShadowRequestIn {
    float pos[3], ndir[3];
    int light;                 // scene light index
    unsigned pixel, path;      // soft-shadow RNG key (point lights)
    int self_object;           // directional lights: the object the point lies on
    int slot;                  // position in its request queue (host-assigned, input order); -1: answered by the shaft test
    int pad;
};

// kind[i]: 0 directional light, 1 point light, 2 soft point-light request answered by the spawn-time shaft test of
// surface_warp (WRT_CULL_SHAFT, only with shaft_cull != 0): its whole shaft to the area light misses every leaf box.
__global__ void __launch_bounds__(128) k_classify_shadow_requests(const __grid_constant__ DevScene s, const ShadowRequestIn* in,
                                                                 long long n, int shaft_cull, unsigned char* kind) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const ShadowRequestIn r = in[i];
        const WrtLight* L = s.lights + r.light;
        unsigned char k = 0;
        if (float_equal(L->pos[3], 1.f)) {
            k = 1;
            if (shaft_cull && s.shadow_type != 0) {
                const f3 sorig = mk3(r.pos[0], r.pos[1], r.pos[2]) + 0.0005f * mk3(r.ndir[0], r.ndir[1], r.ndir[2]);
                const float so[3] = {sorig.x, sorig.y, sorig.z};
                float tri[9];
                for (int j = 0; j < 9; j++) tri[j] = L->tri[j];
                if (wrt_shaft_is_empty(s.onodes, s.n_nodes, so, tri)) k = 2;
            }
        }
        kind[i] = k;
    }
}

// Queues requests [0, n) of `in` into request queue q exactly as surface_warp writes them: node id = index, shadow-ray
// origin pos + 0.0005 * nDir, coefficient slot 0 (50 for a request the shaft test answered); then sets the queue lengths.
__global__ void __launch_bounds__(256) k_pack_shadow_requests(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb,
                                                              int q, const ShadowRequestIn* in, unsigned n, unsigned n_point,
                                                              unsigned n_dir) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const ShadowRequestIn r = in[i];
        const unsigned li = (unsigned)r.light;
        const f3 pos = mk3(r.pos[0], r.pos[1], r.pos[2]), nDir = mk3(r.ndir[0], r.ndir[1], r.ndir[2]);
        const f3 sorig = pos + 0.0005f * nDir;                         // BVHStrategy.hpp:15, Renderer.hpp:349
        if (WRT_IN_BOUNDS((size_t)i * s.n_lights + li, (size_t)fb.n_node_cap * s.n_lights))
            fb.coeff[(size_t)i * s.n_lights + li] = r.slot < 0 ? (float)WRT_SOFT_SAMPLES : 0.f;
        if (r.slot < 0) continue;
        const unsigned slot = (unsigned)r.slot;
        if (float_equal(s.lights[li].pos[3], 1.f)) {
            if (WRT_IN_BOUNDS(slot, fb.preq_cap[q])) {
                fb.preq_o[q][slot] = make_float4(sorig.x, sorig.y, sorig.z, __uint_as_float(i));
                fb.preq_k[q][slot] = make_uint4(li, r.pixel, r.path, 0u);
            }
        } else {
            const int prim = (r.self_object >= 0 && r.self_object < s.n_prims) ? __ldg(s.object_prim + r.self_object) : -1;
            if (WRT_IN_BOUNDS(slot, fb.dreq_cap[q])) {
                fb.dreq_o[q][slot] = make_float4(pos.x, pos.y, pos.z, __uint_as_float(i));
                fb.dreq_k[q][slot] = make_uint4(li, (unsigned)prim, 0u, 0u);
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        fb.counters[C_NPREQ + q] = n_point;
        fb.counters[C_NDREQ + q] = n_dir;
    }
}

__global__ void __launch_bounds__(256) k_unpack_shadow_requests(const __grid_constant__ DevScene s, const __grid_constant__ FrameBuffers fb,
                                                                const ShadowRequestIn* in, unsigned n, float* out) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        out[i] = fb.coeff[(size_t)i * s.n_lights + (unsigned)in[i].light];
}

// mode 0: BVHStrategy::getShadowCoeffi (hard); mode 1: Renderer::getShadowCoeffi(Vector3f&) (soft sample)
__global__ void __launch_bounds__(128) k_batch_shadow(DevScene s, const float* pos, const float* ndir, const float* lightpos,
                                                      long long n, float* out, int mode, float prune_rel) {
    extern __shared__ int smem[];
    Stack st;
    st.init(smem, threadIdx.x, blockDim.x);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        f3 p = mk3(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]);
        f3 nd = mk3(ndir[3 * i], ndir[3 * i + 1], ndir[3 * i + 2]);
        f3 lightPos = mk3(lightpos[3 * i], lightpos[3 * i + 1], lightpos[3 * i + 2]);
        f3 orig = p + 0.0005f * nd;
        f3 raydir = normalized(lightPos - orig);
        float distance = norm(lightPos - orig);
        Ray r = make_ray(orig, raydir);
        const float4* nodes = (prune_rel < 0.f || degenerate_dir(raydir)) ? s.nodes : s.fnodes;
        if (mode == 0) out[i] = shadow_product(s, nodes, r, distance, st);
        else out[i] = occluded(s, nodes, r, distance, st) ? 0.f : 1.f;
    }
}

__global__ void __launch_bounds__(128) k_batch_shadow_directional(const __grid_constant__ DevScene s, const float* pos,
                                                                  const int* self_object, const float* lightdir4,
                                                                  long long n, float* out, int literal) {
    extern __shared__ int smem[];
    Stack st;
    st.init(smem, threadIdx.x, blockDim.x);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        f3 p = mk3(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]);
        f3 negDir = mk3(-lightdir4[4 * i], -lightdir4[4 * i + 1], -lightdir4[4 * i + 2]);
        int so = self_object[i];
        int self_prim = (so >= 0 && so < s.n_prims) ? __ldg(s.object_prim + so) : -1;
        Ray r = make_ray(p, normalized(negDir));
        out[i] = literal ? directional_product(s, r, self_prim) : directional_product_bvh(s, r, self_prim, st);
    }
}

// ---- FP32 issue-rate microbenchmark (the roofline denominator SURVEY.md section 8d asks for) ----
// mode 0: 8 independent FFMA chains per thread (2 flops per instruction);
// mode 1: the same chains as separate FMUL + FADD (what -fmad=false code issues).
__global__ void __launch_bounds__(256) k_fp32_peak(float* out, int iters, int mode) {
    float a[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = 1.0f + 1e-3f * (float)((threadIdx.x + k) & 31);
    const float m = 0.999999f, c = 1e-7f;
    if (mode == 0) {
        for (int i = 0; i < iters; i++) {
#pragma unroll
            for (int k = 0; k < 8; k++) a[k] = __fmaf_rn(a[k], m, c);
        }
    } else {
        for (int i = 0; i < iters; i++) {
#pragma unroll
            for (int k = 0; k < 8; k++) a[k] = __fadd_rn(__fmul_rn(a[k], m), c);
        }
    }
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 8; k++) sum += a[k];
    if (sum == 12345.678f) out[0] = sum;       // never true; keeps the chains alive
}

} // namespace wrt
