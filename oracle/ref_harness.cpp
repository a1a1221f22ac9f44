// ref_harness.cpp — TEST INFRASTRUCTURE.  Thin C ABI around the UNMODIFIED
// reference headers, compiled from where they lie (-I$(REF)/include, REF = the
// reference's source tree, oracle/Makefile)
// into oracle/_ref/libwhitted_ref.so by oracle/Makefile.  No reference source is
// copied into this repository; this file only *calls* the reference:
//   PPMGenerator(path) + main()'s bunny load     src/main.cpp:20-56
//   Renderer(&g) -> BVHStrategy, initializeBVH   include/Renderer.hpp:38-49
//   IIntersectStrategy::UpdateInter              include/IIntersectStrategy.h:10-11
//   IIntersectStrategy::getShadowCoeffi          include/IIntersectStrategy.h:14
//   hasIntersection                              include/BVH.hpp:162-186
//   Renderer::getShadowCoeffi(Vector4f)          include/Renderer.hpp:381-400
//   Renderer::traceRay / render                  include/Renderer.hpp:57-260
// It is used (a) to validate oracle/whitted_oracle.c and the host front-end in
// this container, (b) to generate tests/golden/*, and (c) as the CPU baseline
// ("kind": "reference") in bench.py.  It is never linked into the product.
#include <algorithm>
#include <cassert>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <fstream>
#include <iostream>
#include <map>
#include <memory>
#include <random>
#include <regex>
#include <sstream>
#include <stack>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>
#include <unistd.h>

#define private public
#define protected public
#include "PPMGenerator.hpp"
#include "Sphere.hpp"
#include "Scene.hpp"
#include "Object.hpp"
#include "Renderer.hpp"
#include "OBJ_Loader.h"
#undef private
#undef protected

#include "../include/wrt_scene.h"

namespace {

// Delegating strategy that counts queries; installed in place of the
// Renderer's BVHStrategy so ray counts follow SURVEY.md section 3.3.
struct CountingStrategy : public IIntersectStrategy {
    IIntersectStrategy* inner;
    int64_t closest = 0, hard_shadow = 0, shaded_hits = 0;
    explicit CountingStrategy(IIntersectStrategy* i) : inner(i) {}
    void UpdateInter(Intersection& inter, Scene& sce, const Vector3f& o, const Vector3f& d) override {
        inner->UpdateInter(inter, sce, o, d);
        ++closest;
        if (inter.intersected && !inter.obj->isLight) ++shaded_hits;
    }
    float getShadowCoeffi(Scene& sce, Intersection& p, Vector3f& lightpos) override {
        ++hard_shadow;
        return inner->getShadowCoeffi(sce, p, lightpos);
    }
};

struct RefScene {
    PPMGenerator* g = nullptr;
    Renderer* r = nullptr;
    CountingStrategy* counter = nullptr;
    std::unordered_map<const Object*, int> index;
};

void dfs_leaves(BVHNode* n, RefScene* s, std::vector<int>& out, int depth, int& maxdepth) {
    if (!n) return;
    maxdepth = std::max(maxdepth, depth);
    if (!n->left && !n->right) {
        if (n->obj) out.push_back(s->index.at(n->obj));
        return;
    }
    dfs_leaves(n->left, s, out, depth + 1, maxdepth);
    dfs_leaves(n->right, s, out, depth + 1, maxdepth);
}

void fill_hit(RefScene* s, const Intersection& in, WrtHit* h) {
    memset(h, 0, sizeof *h);
    h->hit = in.intersected ? 1 : 0;
    h->object = in.obj ? s->index.at(in.obj) : -1;
    h->prim = -1;
    h->t = in.t;
    h->pos[0] = in.pos.x; h->pos[1] = in.pos.y; h->pos[2] = in.pos.z;
    h->ndir[0] = in.nDir.x; h->ndir[1] = in.nDir.y; h->ndir[2] = in.nDir.z;
    h->uv[0] = in.textPos.x; h->uv[1] = in.textPos.y;
    h->texture = in.textureIndex;
    h->normalmap = in.normalMapIndex;
    h->material = -1;
}

} // namespace

extern "C" {

// Mirrors main(): cwd must hold the textures the config names.  `obj_path`
// NULL/"" skips the mesh (as when bunny.obj is absent from the cwd).
void* ref_scene_load(const char* config_path, const char* obj_path, int glass_variant) {
    RefScene* s = new RefScene();
    s->g = new PPMGenerator(config_path);
    Material floor_mtl;
    floor_mtl.diffuse = { 0.529, 0.807, 0.921 };
    floor_mtl.specular = { 0.33, 0.66, 0.99 };
    floor_mtl.ka = 0.05;
    floor_mtl.kd = 0.1;
    floor_mtl.ks = glass_variant ? 0.2 : 0.1;
    floor_mtl.n = 64;
    floor_mtl.alpha = 0.2;
    floor_mtl.eta = glass_variant ? 1.33 : 1.52;
    if (obj_path && *obj_path) {
        objl::Loader mesh;
        if (mesh.LoadFile(obj_path)) {
            for (auto& i : mesh.LoadedMeshes)
                for (auto& j : i.Vertices) {
                    j.Position = j.Position * 20;
                    j.Position.Y -= 3;
                    j.Position.Z -= 3;
                }
            s->g->loadObj(mesh, floor_mtl, -1, -1);
        }
    }
    s->r = new Renderer(s->g);
    s->counter = new CountingStrategy(s->r->interStrategy);
    s->r->interStrategy = s->counter;
    int k = 0;
    for (auto& o : s->g->scene.objList) s->index[o.get()] = k++;
    PRINT = false;
    return s;
}

int ref_num_objects(void* h) { return (int)((RefScene*)h)->g->scene.objList.size(); }
int ref_width(void* h) { return ((RefScene*)h)->g->width; }
int ref_height(void* h) { return ((RefScene*)h)->g->height; }
void ref_set_imsize(void* h, int w, int ht) {
    RefScene* s = (RefScene*)h;
    s->g->width = w; s->g->height = ht;
    s->g->rgb.assign((size_t)w * ht, Vector3i());
}
void ref_set_shadow_type(void* h, int soft) { ((RefScene*)h)->g->shadowType = soft ? 1 : 0; }

// Objects in left-to-right leaf order of the reference's own tree.
int ref_bvh_leaf_order(void* h, int* out, int cap, int* depth) {
    RefScene* s = (RefScene*)h;
    std::vector<int> v;
    int md = 0;
    if (!s->g->scene.objList.empty()) dfs_leaves(s->g->scene.BVHaccelerator->getNode(), s, v, 0, md);
    for (size_t i = 0; i < v.size() && (int)i < cap; i++) out[i] = v[i];
    if (depth) *depth = md;
    return (int)v.size();
}

void ref_trace_closest(void* h, const float* orig, const float* dir, int64_t n, WrtHit* out) {
    RefScene* s = (RefScene*)h;
    for (int64_t i = 0; i < n; i++) {
        Intersection inter;
        Vector3f o(orig[3 * i], orig[3 * i + 1], orig[3 * i + 2]);
        Vector3f d(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
        s->r->interStrategy->UpdateInter(inter, s->g->scene, o, d);
        fill_hit(s, inter, &out[i]);
    }
}

void ref_shadow_hard(void* h, const float* pos, const float* ndir, const float* lightpos, int64_t n, float* out) {
    RefScene* s = (RefScene*)h;
    for (int64_t i = 0; i < n; i++) {
        Intersection p;
        p.pos = Vector3f(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]);
        p.nDir = Vector3f(ndir[3 * i], ndir[3 * i + 1], ndir[3 * i + 2]);
        Vector3f lp(lightpos[3 * i], lightpos[3 * i + 1], lightpos[3 * i + 2]);
        out[i] = s->r->interStrategy->getShadowCoeffi(s->g->scene, p, lp);
    }
}

// Soft-shadow visibility query of Renderer::getShadowCoeffi(Intersection&, Vector3f&)
// with EXPEDITE: 0 when hasIntersection(), else 1.
void ref_shadow_soft(void* h, const float* pos, const float* ndir, const float* lightpos, int64_t n, float* out) {
    RefScene* s = (RefScene*)h;
    for (int64_t i = 0; i < n; i++) {
        Intersection p;
        p.pos = Vector3f(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]);
        p.nDir = Vector3f(ndir[3 * i], ndir[3 * i + 1], ndir[3 * i + 2]);
        Vector3f lp(lightpos[3 * i], lightpos[3 * i + 1], lightpos[3 * i + 2]);
        out[i] = s->r->getShadowCoeffi(p, lp);
    }
}

void ref_shadow_directional(void* h, const float* pos, const int* self_object, const float* lightdir4,
                            int64_t n, float* out) {
    RefScene* s = (RefScene*)h;
    for (int64_t i = 0; i < n; i++) {
        Intersection p;
        p.pos = Vector3f(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]);
        p.obj = self_object[i] >= 0 ? s->g->scene.objList[self_object[i]].get() : nullptr;
        Vector4f ld(lightdir4[4 * i], lightdir4[4 * i + 1], lightdir4[4 * i + 2], lightdir4[4 * i + 3]);
        out[i] = s->r->getShadowCoeffi(p, ld);
    }
}

// Float colour of Renderer::traceRay for arbitrary rays (deterministic for hard shadows).
void ref_trace_ray(void* h, const float* orig, const float* dir, const int* depth, int64_t n, float* rgb) {
    RefScene* s = (RefScene*)h;
    for (int64_t i = 0; i < n; i++) {
        Vector3f o(orig[3 * i], orig[3 * i + 1], orig[3 * i + 2]);
        Vector3f d(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
        Vector3f c = s->r->traceRay(o, d, depth ? depth[i] : 0);
        rgb[3 * i] = c.x; rgb[3 * i + 1] = c.y; rgb[3 * i + 2] = c.z;
    }
}

// Full Renderer::render(); returns seconds spent inside render() only.
double ref_render(void* h, int32_t* rgb_out) {
    RefScene* s = (RefScene*)h;
    std::streambuf* old = std::cout.rdbuf(nullptr);      // silence the progress bar
    auto t0 = std::chrono::steady_clock::now();
    s->r->render();
    auto t1 = std::chrono::steady_clock::now();
    std::cout.rdbuf(old);
    size_t n = (size_t)s->g->width * s->g->height;
    for (size_t i = 0; i < n; i++) {
        rgb_out[3 * i] = s->g->rgb[i].x; rgb_out[3 * i + 1] = s->g->rgb[i].y; rgb_out[3 * i + 2] = s->g->rgb[i].z;
    }
    return std::chrono::duration<double>(t1 - t0).count();
}

void ref_counters_reset(void* h) {
    RefScene* s = (RefScene*)h;
    s->counter->closest = s->counter->hard_shadow = s->counter->shaded_hits = 0;
}

// closest-hit rays, shadow rays (SURVEY.md section 3.3 definition).  Soft and
// directional shadow queries bypass the strategy interface, so they are derived
// from the number of shaded hits: 50 per point light (soft), 1 per directional light.
void ref_counters_get(void* h, int64_t* closest, int64_t* shadow) {
    RefScene* s = (RefScene*)h;
    int64_t npoint = 0, ndir = 0;
    for (auto& l : s->g->scene.lightList) (FLOAT_EQUAL(l->pos.w, 1.f) ? npoint : ndir)++;
    int64_t sh = s->counter->shaded_hits * ndir;
    if (s->g->shadowType == 0) sh += s->counter->hard_shadow;
    else sh += s->counter->shaded_hits * npoint * 50;
    *closest = s->counter->closest;
    *shadow = sh;
}

// Traces the reference's own traceRay through every (sx,sy)-th pixel of the
// configured image: a bounded sample of the frame with the frame's own ray mix.
// pixel_pos/dir are produced by the caller (host camera), so this file does not
// restate the camera.  Returns seconds.
double ref_trace_pixels(void* h, const float* orig, const float* dir, int64_t n, int32_t* rgb_out) {
    RefScene* s = (RefScene*)h;
    auto t0 = std::chrono::steady_clock::now();
    for (int64_t i = 0; i < n; i++) {
        Vector3f o(orig[3 * i], orig[3 * i + 1], orig[3 * i + 2]);
        Vector3f d(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
        Vector3f res = s->r->traceRay(o, d, 0);
        if (rgb_out) {
            rgb_out[3 * i] = 255 * std::min(res.x, 1.f);
            rgb_out[3 * i + 1] = 255 * std::min(res.y, 1.f);
            rgb_out[3 * i + 2] = 255 * std::min(res.z, 1.f);
        }
    }
    auto t1 = std::chrono::steady_clock::now();
    return std::chrono::duration<double>(t1 - t0).count();
}

} // extern "C"
