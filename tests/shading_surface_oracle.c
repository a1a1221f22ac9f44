/* shading_surface_oracle.c — TEST INFRASTRUCTURE: the surface the oracle's traceRay shades at a hit record, for the
 * frame's per-pixel surface planes (wrt_render_gbuffer, tests/test_gpu_gbuffer.py).
 *
 * Compiled by tests/test_oracle_shading_surface.py into a temporary library together with the oracle itself (the
 * #include below), with the oracle's own flags, once as is and once with -DORC_DEVICE_MATH.  It calls the oracle's
 * static functions (mtl_of, is_light, texture_at, change_normal_dir) under the conditions and in the order trace_ray
 * calls them (whitted_oracle.c, Renderer.hpp:172-184); every operation on a value is one of those functions. */
#include "../oracle/whitted_oracle.c"

/* ndir[3i..]: the shading normal after changeNormalDir; od[3i..]: Od, the material's diffuse colour or the texel.
 * 0 for a miss or a light avatar, which are not shaded.  hits[i] is a record as orc_trace_closest returns it. */
void orc_shading_surface(const WrtSceneDesc* s, const WrtHit* hits, int64_t n, float* ndir, float* od) {
#pragma omp parallel for schedule(dynamic, 256)
    for (int64_t i = 0; i < n; i++) {
        const WrtHit* h = &hits[i];
        v3 nd = V(0, 0, 0), d = V(0, 0, 0);
        if (h->hit && !is_light(s, h->prim)) {                      /* Renderer.hpp:172 */
            Inter inter = inter_default();
            inter.intersected = 1; inter.t = h->t; inter.pos = ld3(h->pos); inter.nDir = ld3(h->ndir);
            inter.u = h->uv[0]; inter.v = h->uv[1];
            inter.textureIndex = h->texture; inter.normalMapIndex = h->normalmap; inter.prim = h->prim;
            d = ld3(mtl_of(s, inter.prim)->diffuse);
            if (!float_equal(-1.f, (float)inter.textureIndex) && !float_equal(-1.f, inter.u) && !float_equal(-1.f, inter.v))
                d = texture_at(s, &s->textures[inter.textureIndex], inter.u, inter.v);      /* :176-180 */
            if (inter.normalMapIndex != -1) change_normal_dir(s, &inter);                    /* :182-184 */
            nd = inter.nDir;
        }
        ndir[3 * i] = nd.x; ndir[3 * i + 1] = nd.y; ndir[3 * i + 2] = nd.z;
        od[3 * i] = d.x; od[3 * i + 1] = d.y; od[3 * i + 2] = d.z;
    }
}
