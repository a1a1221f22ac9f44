// TEST INFRASTRUCTURE: runs the device BVH build's per-item steps (csrc/cuda/ploc_bvh.h, the same source the kernels
// compile) on the CPU, passes emulated by loops in the order the kernel's barriers impose, and checks the tree:
//   every primitive in exactly one leaf, leaf boxes == the reference's per-primitive boxes, every inner box the exact
//   union of its children (and likewise the dilated boxes), sibling pairs adjacent with the parent's link pointing at
//   them, record count 2n, depth as reported, surface-area cost close to the host's binned-SAH build.
// Also prints the depths of the host's binned-SAH tree and of the scene's own (reference) tree: the traversal stack is
// sized from all three (wrt_upload_scene).
// usage: ploc_check <config> <obj|""> <asset_dir>      prints one JSON line
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <vector>

#include "../include/wrt_host.h"
#include "../whittedstyle_raytracer_b200/csrc/cuda/fast_bvh.hpp"
#include "../whittedstyle_raytracer_b200/csrc/cuda/ploc_bvh.h"



int main(int argc, char** argv) {
    if (argc < 4) return 2;
    WrtScene* h = nullptr;
    if (wrt_scene_load(argv[1], argv[2][0] ? argv[2] : nullptr, argv[3], 0, &h)) { printf("{\"error\": \"%s\"}\n", wrt_host_last_error()); return 1; }
    const WrtSceneDesc* s = wrt_scene_desc(h);
    const int n = s->n_prims;
    std::vector<float4> lo(2 * n), hi(2 * n), dlo(2 * n), dhi(2 * n);
    std::vector<int> parent(2 * n, -1), cnt(2 * n, 0);
    PlocTree t{lo.data(), hi.data(), dlo.data(), dhi.data(), parent.data(), cnt.data()};
    // pass 0: leaves + Morton keys (k_bvh_leaves)
    std::vector<std::pair<uint64_t, int>> keys(n);
    float bmin[3] = {3.4e38f, 3.4e38f, 3.4e38f}, bmax[3] = {-3.4e38f, -3.4e38f, -3.4e38f};      // centroid bounds (k_bvh_leaves)
    for (int i = 0; i < s->n_nodes; i++) {
        const WrtNode& nd = s->nodes[i];
        if (nd.link >= 0 || i == 1) continue;
        for (int k = 0; k < 3; k++) { float c = 0.5f * nd.pmin[k] + 0.5f * nd.pmax[k]; bmin[k] = std::min(bmin[k], c); bmax[k] = std::max(bmax[k], c); }
    }
    std::vector<int> seen(n, 0);
    for (int i = 0; i < s->n_nodes; i++) {
        const WrtNode& nd = s->nodes[i];
        if (nd.link >= 0 || i == 1) continue;
        const int p = ~nd.link;
        ploc_init_leaf(t, p, nd.pmin, nd.pmax, 1e-3f, 1e-4f);
        float c[3];
        for (int k = 0; k < 3; k++) c[k] = 0.5f * nd.pmin[k] + 0.5f * nd.pmax[k];
        keys[p] = {ploc_morton(c, bmin, bmax), p};
        seen[p]++;
    }
    for (int p = 0; p < n; p++) if (seen[p] != 1) { printf("{\"error\": \"leaf records do not cover primitive %d once\"}\n", p); return 1; }
    std::stable_sort(keys.begin(), keys.end(), [](auto& a, auto& b) { return a.first < b.first; });   // radix sort is stable
    std::vector<int> cur(n), nxt(n), nn(n);
    for (int i = 0; i < n; i++) cur[i] = keys[i].second;
    int m = n, alloc = n, passes = 0;
    while (m > 1) {
        ++passes;
        for (int i = 0; i < m; i++) nn[i] = ploc_nearest(t, cur.data(), m, i, WRT_PLOC_RADIUS);      // barrier
        int out = 0;
        for (int i = 0; i < m; i++) {                                                                 // ordered compaction
            const int fate = ploc_fate(nn.data(), i);
            if (fate == 2) { ploc_make_node(t, alloc, cur[i], cur[nn[i]]); nxt[out++] = alloc++; }
            else if (fate == 1) nxt[out++] = cur[i];
        }
        if (out >= m) { printf("{\"error\": \"no progress in pass %d\"}\n", passes); return 1; }
        cur.swap(nxt);
        m = out;
    }
    if (n > 0 && alloc != 2 * n - 1) { printf("{\"error\": \"node count %d != 2n-1\"}\n", alloc); return 1; }
    // layout (k_bvh_layout)
    std::vector<WrtNode> rec(2 * std::max(n, 1)), drec(2 * std::max(n, 1));
    memset(rec.data(), 0, rec.size() * sizeof(WrtNode));
    std::vector<int> written(rec.size(), 0);
    int max_depth = 0;
    for (int v = 0; v < 2 * n - 1; v++) {
        int link, depth;
        const int r = ploc_record_of(t, n, v, &link, &depth);
        if (r < 0 || r >= (int)rec.size() || r == 1) { printf("{\"error\": \"record %d out of range\"}\n", r); return 1; }
        written[r]++;
        rec[r].pmin[0] = lo[v].x; rec[r].pmin[1] = lo[v].y; rec[r].pmin[2] = lo[v].z; rec[r].link = link;
        rec[r].pmax[0] = hi[v].x; rec[r].pmax[1] = hi[v].y; rec[r].pmax[2] = hi[v].z;
        drec[r].pmin[0] = dlo[v].x; drec[r].pmin[1] = dlo[v].y; drec[r].pmin[2] = dlo[v].z; drec[r].link = link;
        drec[r].pmax[0] = dhi[v].x; drec[r].pmax[1] = dhi[v].y; drec[r].pmax[2] = dhi[v].z;
        if (v < n) max_depth = std::max(max_depth, depth);
    }
    for (size_t r = 0; r < rec.size(); r++)
        if (written[r] != (r == 1 ? 0 : 1)) { printf("{\"error\": \"record %zu written %d times\"}\n", r, written[r]); return 1; }
    // checks on the flattened tree
    std::vector<int> leaf_of(n, 0);
    long long bad_union = 0, bad_leaf = 0, bad_dil = 0;
    int depth_seen = 0;
    std::vector<std::pair<int, int>> st{{0, 0}};
    auto area = [](const WrtNode& b) { float dx = b.pmax[0] - b.pmin[0], dy = b.pmax[1] - b.pmin[1], dz = b.pmax[2] - b.pmin[2]; return (double)(dx * dy + dy * dz + dz * dx); };
    double cost = 0;
    const double root_area = area(rec[0]);
    std::vector<const WrtNode*> ref_leaf(n, nullptr);
    for (int i = 0; i < s->n_nodes; i++) if (s->nodes[i].link < 0 && i != 1) ref_leaf[~s->nodes[i].link] = &s->nodes[i];
    while (!st.empty()) {
        auto [r, d] = st.back();
        st.pop_back();
        depth_seen = std::max(depth_seen, d);
        cost += area(rec[r]) / root_area;
        if (rec[r].link < 0) {
            const int p = ~rec[r].link;
            if (p < 0 || p >= n) { printf("{\"error\": \"bad leaf link\"}\n"); return 1; }
            leaf_of[p]++;
            if (memcmp(rec[r].pmin, ref_leaf[p]->pmin, 12) || memcmp(rec[r].pmax, ref_leaf[p]->pmax, 12)) ++bad_leaf;
            continue;
        }
        const int c = rec[r].link;
        if (c < 2 || c + 1 >= (int)rec.size() || (c & 1)) { printf("{\"error\": \"bad pair link %d\"}\n", c); return 1; }
        for (int k = 0; k < 3; k++) {
            if (rec[r].pmin[k] != std::min(rec[c].pmin[k], rec[c + 1].pmin[k]) || rec[r].pmax[k] != std::max(rec[c].pmax[k], rec[c + 1].pmax[k])) ++bad_union;
            if (drec[r].pmin[k] != std::min(drec[c].pmin[k], drec[c + 1].pmin[k]) || drec[r].pmax[k] != std::max(drec[c].pmax[k], drec[c + 1].pmax[k])) ++bad_dil;
        }
        st.push_back({c, d + 1});
        st.push_back({c + 1, d + 1});
    }
    long long missing = 0;
    for (int p = 0; p < n; p++) if (leaf_of[p] != 1) ++missing;
    wrt::FastBvhBuilder fb;
    fb.build(s);
    double host_cost = 0;
    for (size_t i = 0; i < fb.nodes.size(); i++) if (i != 1) host_cost += area(fb.nodes[i]) / area(fb.nodes[0]);
    // the host's dilated leaves must equal the device formula's
    long long dil_leaf_diff = 0;
    {
        std::vector<WrtNode> hd = fb.dilated(1e-3f, 1e-4f);
        std::vector<const WrtNode*> hl(n, nullptr);
        for (size_t i = 0; i < hd.size(); i++) if (hd[i].link < 0 && i != 1) hl[~hd[i].link] = &hd[i];
        for (size_t r = 0; r < drec.size(); r++) {
            if (r == 1 || drec[r].link >= 0) continue;
            const int p = ~drec[r].link;
            if (memcmp(drec[r].pmin, hl[p]->pmin, 12) || memcmp(drec[r].pmax, hl[p]->pmax, 12)) ++dil_leaf_diff;
        }
    }
    printf("{\"n\": %d, \"passes\": %d, \"records\": %zu, \"depth\": %d, \"depth_seen\": %d, \"missing\": %lld, \"bad_union\": %lld, "
           "\"bad_leaf_box\": %lld, \"bad_dilated_union\": %lld, \"dilated_leaf_diff\": %lld, \"cost\": %.4f, \"host_sah_cost\": %.4f, "
           "\"host_depth\": %d, \"ref_depth\": %d, \"ref_nodes\": %d}\n",
           n, passes, rec.size(), max_depth, depth_seen, missing, bad_union, bad_leaf, bad_dil, dil_leaf_diff, cost, host_cost,
           fb.max_depth, wrt_scene_bvh_depth(h), s->n_nodes);
    return 0;
}
