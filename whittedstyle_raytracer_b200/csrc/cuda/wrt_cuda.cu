// wrt_cuda.cu — host side of libwrt_cuda.so: context, scene upload, frame
// scheduling and the C ABI of include/wrt_cuda.h.  Compiled for sm_100a only,
// with -fmad=false (see dev_math.cuh).  No CPU fallback exists in this library.
#include <algorithm>
#include <cstdio>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "../../../include/wrt_cuda.h"
#include "fast_bvh.hpp"
#include "kernels.cuh"
#include "bvh_build.cuh"

namespace {

thread_local std::string g_err;

int fail(const std::string& msg) {
    g_err = msg;
    return 1;
}

#define CK(call)                                                                                      \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess) {                                                                      \
            return fail(std::string(#call) + ": " + cudaGetErrorString(e_) + " (" + __FILE__ + ":" + \
                        std::to_string(__LINE__) + ")");                                              \
        }                                                                                             \
    } while (0)

enum Family { F_RAYGEN, F_TRACE, F_SURFACE, F_SHADOW_HARD, F_SHADOW_SOFT, F_SHADOW_DIR, F_SHADE, F_COMBINE, F_RESOLVE, F_SOFT_LISTS, F_SOFT_FILTER };

struct TimedLaunch {
    int family;
    cudaEvent_t e0, e1;
    bool on_chain;
};

} // namespace

struct WrtContext {
    int device = 0;
    int num_sms = 0;
    // All frame work runs on two internal streams: `chain` (high priority: the dependent closest-hit chain, the deep
    // levels' shadow kernels, combine + resolve) and `side` (level 0's shadow + shade kernels).  A caller-provided stream
    // (wrt_render_device) is joined to them by two events, nothing else runs on it.
    cudaStream_t chain = nullptr, side = nullptr;
    cudaEvent_t ev_in = nullptr, ev_lvl0 = nullptr, ev_mid = nullptr, ev_side = nullptr, ev_out = nullptr;
    bool overlap = true;

    // scene
    wrt::DevScene ds{};
    std::vector<void*> scene_allocs;
    std::vector<size_t> scene_alloc_bytes;
    size_t scene_slot = 0;
    bool has_scene = false;
    bool textures_complete = true;
    int bvh_depth = 0;
    int stack_rows = 2;
    std::vector<WrtPathCode> path_codes;   // host copy staged by wrt_upload_scene

    // camera / tiling / options
    WrtCamera cam{};
    bool has_cam = false;
    int tile_w = 8, tile_h = 4, rank = 0, world = 1;   // one warp-sized 8x4 block per tile: finest interleave
    int traversal = WRT_TRAVERSAL_PRUNED;
    uint32_t seed = WRT_DEFAULT_SEED;
    float queue_factor = 0.f;          // > 0: caller-fixed deep-level capacity (multiple of the batch); 0: automatic
    float deep_factor = 0.25f;         // automatic mode: current deep-level capacity factor (grows on overflow)
    float prune_rel = 1e-3f;
    bool kernel_timing = false;
    int refill = 16;                   // idle lanes that trigger a refill on deep ray-tree levels
    int refill_soft = 24;
    bool shaft_cull = true;            // soft shadows: answer requests whose light shaft is empty without tracing (shaft_cull.h)
    bool soft_lists = true;            // soft shadows: per-request candidate lists (k_soft_lists + k_soft_list_rays) instead of per-ray walks
    long long list_pool_cap_override = 0;
    int shaft_cull_max_level = 0;      // deepest ray-tree level whose surface stage runs the shaft test (when lists are on)
    wrt::SoftListBuffers list_bufs[WRT_QUEUES] = {};
    wrt::FastBvhBuilder fbvh;          // WRT_HOST_BVH=1 only: the host's binned-SAH build (development A/B)
    bool host_bvh = false;
    uint8_t* h_stage = nullptr;        // pinned staging of the scene description: one H2D per upload
    size_t h_stage_bytes = 0;
    int ploc_coop_grid = 1;            // co-resident CTAs of k_bvh_ploc
    int fast_depth = 0, build_passes = 0;
    bool unlit_cull = true;            // drop shadow requests of lights whose shading terms are exactly 0 at the point
    int cache_from_level = 0;          // per-ray soft-shadow kernel: occluder cache (99 = off)
    int chunk_div = 16;                // work claiming: 0 = one atomic per refill, k = chunks of n/(warps*k) items
    int refill0 = 32;                  // level 0 (coherent primary rays and their shadow rays)
    int trace_blocks_per_sm = 10;      // persistent shadow / unfused closest-hit kernels
    bool shade0_separate = true;       // level 0 is shaded by its own launch on the side stream (else inside combine)
    int soft_filter = 2;               // 0: off, 1: prune the deep queues' candidate lists (k_soft_filter), 2: level 0's as well
    int deep_split = 5;                // request queues: level 0 | levels 1..deep_split | deeper.  The shadow kernels of levels
                                       // 1..5 run beside the closest-hit chain of levels 6..8 (4K soft frame: 14.55 ms with one
                                       // deep queue, 14.34 / 14.14 / 14.40 with a split at 4 / 5 / 3; 1/8 share 2.56 -> 2.46 ms)
    int side_blocks_per_sm = 6;        // persistent shadow kernels on the side stream: CTAs per SM (0 = trace_blocks_per_sm).  6 leave
                                       // register file for two CTAs of the chain's kernel on every SM, so the chain keeps moving
                                       // beside a long shadow kernel: 4K soft frame 12.73 -> 12.50 ms (5: 12.40, 7: 12.65, 8: 12.70);
                                       // hard-shadow, 8K and sphere frames within +-0.5 %
    int fb_split = -1;
    bool small_batch_full_levels = true; // automatic sizing: batches under 1 M slots get full-size deep levels
    long long max_batch = 1ll << 25;   // primary slots per batch (8K = 33.2 M slots fits)
    long long learned_batch = 1ll << 40; // a batch size that overflowed with the deep levels at their largest: later frames of
                                       // the same scene / image size start with the halved batches right away
    long long learned_key[4] = {0, 0, 0, 0};

    // frame buffers
    wrt::FrameBuffers fb{};
    std::vector<void*> frame_allocs;
    unsigned batch_slots = 0;          // primary slots the buffers were sized for
    unsigned deep_slots = 0;           // slots of each deeper level
    int fb_lights = -1, fb_point = -1, fb_dir = -1;
    unsigned* h_counters = nullptr;    // pinned
    uint8_t* d_image = nullptr;        // full image, row-major (wrt_render)
    size_t d_image_bytes = 0;
    uint8_t* h_image = nullptr;        // pinned staging
    size_t h_image_bytes = 0;
    float4* h_float = nullptr;         // pinned, slot order: level-0 {colour, fr} of every local slot (wrt_render_float)
    size_t h_float_bytes = 0;
    bool copy_float = false;           // set for the duration of wrt_render_float: each batch copies its level 0 to h_float

    // batch-query scratch
    void* d_scratch[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t scratch_bytes[5] = {0, 0, 0, 0, 0};

    // bookkeeping
    int64_t launches = 0;
    int work_seq = 0;
    int coop_grid = 0;                 // co-resident CTAs of k_combine_resolve (cooperative launch)
    int filter_grid = 0;               // resident CTAs of k_soft_filter
    WrtStats stats{};
    std::vector<TimedLaunch> timed;
    std::vector<cudaEvent_t> event_pool;
    size_t event_next = 0;
    float family_ms[WRT_KERNEL_FAMILIES] = {0};
    int family_launches[WRT_KERNEL_FAMILIES] = {0};
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    cudaStream_t user_stream = nullptr;
    bool user_stream_joined = false;
    uint8_t* last_image = nullptr;     // targets of the frame in flight (needed again if an overflowed batch is redone)
    uint8_t* last_packed = nullptr;
    bool frame_pending = false;
    bool has_frame = false;

    wrt::TileMap tilemap() const {
        wrt::TileMap tm;
        static_cast<WrtTileMap&>(tm) = wrt_tilemap_make(cam.width, cam.height, tile_w, tile_h, rank, world);
        return tm;
    }
    long long local_slots(int r, int w) const {
        WrtTileMap tm = wrt_tilemap_make(cam.width, cam.height, tile_w, tile_h, r, w);
        return wrt_tilemap_slots(&tm, r, w);
    }
};

namespace {

using wrt::FrameBuffers;

// Scene arrays keep their device allocation across uploads when the new array fits
// (re-uploading a scene of the same size costs copies and kernels only, no cudaMalloc/cudaFree).
int dev_alloc(WrtContext* c, size_t bytes, void** out) {
    *out = nullptr;
    bytes = std::max<size_t>(bytes, 256);
    size_t slot = c->scene_slot++;
    if (slot >= c->scene_allocs.size()) { c->scene_allocs.push_back(nullptr); c->scene_alloc_bytes.push_back(0); }
    if (c->scene_alloc_bytes[slot] < bytes) {
        if (c->scene_allocs[slot]) {
            CK(cudaDeviceSynchronize());               // a frame in flight may still read the old array
            cudaFree(c->scene_allocs[slot]);
        }
        c->scene_allocs[slot] = nullptr; c->scene_alloc_bytes[slot] = 0;
        CK(cudaMalloc(&c->scene_allocs[slot], bytes));
        c->scene_alloc_bytes[slot] = bytes;
    }
    *out = c->scene_allocs[slot];
    return 0;
}

void free_scene(WrtContext* c) {
    for (void* p : c->scene_allocs) if (p) cudaFree(p);
    c->scene_allocs.clear();
    c->scene_alloc_bytes.clear();
    c->has_scene = false;
}

void free_frame(WrtContext* c) {
    for (void* p : c->frame_allocs) cudaFree(p);
    c->frame_allocs.clear();
    c->batch_slots = 0;
    c->deep_slots = 0;
    memset(&c->fb, 0, sizeof c->fb);
}

int tree_depth(const WrtSceneDesc* s) {
    if (s->n_nodes == 0) return 0;
    int maxd = 0;
    std::vector<std::pair<int, int>> st;
    st.push_back({0, 0});
    while (!st.empty()) {
        auto [n, d] = st.back();
        st.pop_back();
        maxd = std::max(maxd, d);
        int link = s->nodes[n].link;
        if (link >= 0) { st.push_back({link, d + 1}); st.push_back({link + 1, d + 1}); }
    }
    return maxd;
}

template <class T>
int frame_alloc(WrtContext* c, T** p, size_t count) {
    void* q = nullptr;
    CK(cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T)));
    c->frame_allocs.push_back(q);
    *p = (T*)q;
    return 0;
}

// Slots of each deeper level for a batch of `slots` primary slots.  Caller-fixed factor: factor x slots.  Automatic:
// small batches get a full-size level (memory is no object there), large ones `deep_factor` of the batch — in the bunny
// frames <= 16 % of the pixels spawn secondary rays (SURVEY.md section 3.3); the factor doubles when a level overflows.
unsigned deep_slots_for(const WrtContext* c, unsigned slots) {
    double want;
    if (c->queue_factor > 0.f) want = (double)slots * c->queue_factor;
    else want = std::max((double)slots * c->deep_factor, c->small_batch_full_levels ? std::min((double)slots, 1048576.0) : 0.0);
    want = std::min(want, 2.0e9);
    return ((unsigned)std::max(want, 64.0) + 63u) & ~63u;
}

int ensure_frame_buffers(WrtContext* c, unsigned slots) {
    const wrt::DevScene& ds = c->ds;
    const unsigned capd = deep_slots_for(c, slots);
    if (c->batch_slots >= slots && c->deep_slots >= capd && c->fb_lights == ds.n_lights && c->fb_point == ds.n_point_lights &&
        c->fb_dir == ds.n_dir_lights && c->fb_split == c->deep_split)
        return 0;
    CK(cudaDeviceSynchronize());
    free_frame(c);
    FrameBuffers& fb = c->fb;
    const unsigned cap0 = slots + 64;
    const unsigned long long nodes64 = (unsigned long long)cap0 + (unsigned long long)(WRT_MAX_DEPTH - 1) * capd;
    if (nodes64 > 0x7fffff00ull) return fail("frame batch too large for 32-bit node indices");
    if (nodes64 * std::max(1, ds.n_lights) > 0xffffffffffull) return fail("too many (node, light) pairs");
    fb.cap0 = cap0; fb.capd = capd; fb.n_node_cap = (unsigned)nodes64;
    const unsigned long long deep_nodes = (unsigned long long)(WRT_MAX_DEPTH - 1) * capd;
    auto req_cap = [](unsigned long long nodes, int lights) {
        return (unsigned)std::min<unsigned long long>(nodes * (unsigned long long)std::max(1, lights), 0xffffff00ull);
    };
    (void)deep_nodes;
    const int split = std::max(1, std::min(WRT_MAX_DEPTH - 1, c->deep_split));
    const unsigned long long q_nodes[WRT_QUEUES] = {cap0, (unsigned long long)split * capd, (unsigned long long)(WRT_MAX_DEPTH - 1 - split) * capd};
    for (int q = 0; q < WRT_QUEUES; q++) {
        fb.preq_cap[q] = req_cap(std::max(q_nodes[q], 1ull), ds.n_point_lights);
        fb.dreq_cap[q] = req_cap(std::max(q_nodes[q], 1ull), ds.n_dir_lights);
    }
    for (int d = 0; d < WRT_MAX_DEPTH; d++) fb.queue_of_level[d] = (unsigned char)(d == 0 ? 0 : (d <= split ? 1 : 2));
    for (int k = 0; k < 2; k++) {
        if (frame_alloc(c, &fb.ray_o[k], capd)) return 1;
        if (frame_alloc(c, &fb.ray_d[k], capd)) return 1;
    }
    if (frame_alloc(c, &fb.hit, std::max(cap0, capd))) return 1;
    if (frame_alloc(c, &fb.surf, 4 * (size_t)nodes64)) return 1;
    if (frame_alloc(c, &fb.node_a, (size_t)nodes64)) return 1;
    if (frame_alloc(c, &fb.node_b, (size_t)nodes64)) return 1;
    if (frame_alloc(c, &fb.coeff, (size_t)nodes64 * std::max(1, ds.n_lights))) return 1;
    for (int q = 0; q < WRT_QUEUES; q++) {
        if (frame_alloc(c, &fb.preq_o[q], ds.n_point_lights ? fb.preq_cap[q] : 1)) return 1;
        if (frame_alloc(c, &fb.preq_k[q], ds.n_point_lights ? fb.preq_cap[q] : 1)) return 1;
        if (frame_alloc(c, &fb.dreq_o[q], ds.n_dir_lights ? fb.dreq_cap[q] : 1)) return 1;
        if (frame_alloc(c, &fb.dreq_k[q], ds.n_dir_lights ? fb.dreq_cap[q] : 1)) return 1;
    }
    if (frame_alloc(c, &fb.counters, wrt::C_TOTAL)) return 1;
    // candidate lists of the soft-shadow path (kernels.cuh, K4b'), one set per request queue (their launches overlap):
    // walk scratch per thread, list pool, per-request {offset, count}.  A full pool only means per-ray walks for the
    // remaining requests.  Level-0 requests that survive the shaft test at spawn time have 1-2 candidates; deep-level
    // ones (origins on the bunny) ~30.
    for (int q = 0; q < WRT_QUEUES; q++) {
        wrt::SoftListBuffers& lb = c->list_bufs[q];
        // Level-0 requests that survive the shaft test at spawn time have 1-2 candidates, deep-level ones (origins on
        // the bunny) ~30.  A warp reserves region_per_request entries per request of its chunk; the pool holds that for
        // half of the queue's capacity (queues run far below capacity; a full pool only means per-ray walks).
        lb.region_per_request = q == 0 ? 4u : 32u;
        const unsigned long long per_req = q == 0 ? 4ull : 16ull;
        lb.pool_cap = (unsigned)std::min<unsigned long long>(std::max<unsigned long long>(8ull << 20, per_req * fb.preq_cap[q]), 1ull << 30);
        if (!ds.n_point_lights || ds.shadow_type == 0) lb.pool_cap = 64;
        if (c->list_pool_cap_override > 0) lb.pool_cap = (unsigned)c->list_pool_cap_override;     // tests: force the pool-full path
        const bool lists_possible = ds.n_point_lights && ds.shadow_type != 0;
        if (frame_alloc(c, &lb.scratch, lists_possible ? (size_t)c->num_sms * c->trace_blocks_per_sm * 128 * WRT_LIST_CAP : 1)) return 1;
        if (frame_alloc(c, &lb.shafts, lists_possible ? (size_t)c->num_sms * c->trace_blocks_per_sm * 4 * WRT_LISTS_CHUNK * WRT_SHAFT_SLOT : 1)) return 1;
        if (frame_alloc(c, &lb.pool, lb.pool_cap)) return 1;
        if (frame_alloc(c, &lb.ref, lists_possible ? fb.preq_cap[q] : 1)) return 1;
        if (frame_alloc(c, &lb.work, lists_possible ? fb.preq_cap[q] : 1)) return 1;
    }
    c->batch_slots = slots;
    c->deep_slots = capd;
    c->fb_lights = ds.n_lights; c->fb_point = ds.n_point_lights; c->fb_dir = ds.n_dir_lights;
    c->fb_split = c->deep_split;
    return 0;
}

int ensure_scratch(WrtContext* c, int k, size_t bytes) {
    if (c->scratch_bytes[k] >= bytes) return 0;
    if (c->d_scratch[k]) cudaFree(c->d_scratch[k]);
    c->d_scratch[k] = nullptr;
    c->scratch_bytes[k] = 0;
    CK(cudaMalloc(&c->d_scratch[k], bytes));
    c->scratch_bytes[k] = bytes;
    return 0;
}

cudaEvent_t next_event(WrtContext* c) {
    if (c->event_next == c->event_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        c->event_pool.push_back(e);
    }
    return c->event_pool[c->event_next++];
}

struct LaunchScope {                      // counts the launch; optionally brackets it with events
    WrtContext* c;
    cudaStream_t st;
    TimedLaunch tl{};
    bool timed;
    LaunchScope(WrtContext* ctx, cudaStream_t s, int family) : c(ctx), st(s), timed(ctx->kernel_timing) {
        ++c->launches;
        if (timed) {
            tl.family = family;
            tl.on_chain = s == ctx->chain;
            tl.e0 = next_event(c);
            tl.e1 = next_event(c);
            cudaEventRecord(tl.e0, st);
        }
    }
    ~LaunchScope() {
        if (timed) {
            cudaEventRecord(tl.e1, st);
            c->timed.push_back(tl);
        }
    }
};

int grid_for(WrtContext* c, int blocks_per_sm) { return c->num_sms * blocks_per_sm; }

size_t stack_bytes(WrtContext* c, int threads) { return (size_t)c->stack_rows * threads * sizeof(int); }

float prune_value(const WrtContext* c) { return c->traversal == WRT_TRAVERSAL_PRUNED ? c->prune_rel : -1.f; }

// The shadow kernels of request queue q (0: level 0, 1: levels 1..8 together) on stream `st`.
int enqueue_shadows(WrtContext* c, cudaStream_t st, int q, int& work_seq) {
    using namespace wrt;
    FrameBuffers& fb = c->fb;
    const DevScene& ds = c->ds;
    const int TB = 128;
    const bool on_side = st == c->side && c->side_blocks_per_sm > 0;
    const int trace_grid = grid_for(c, on_side ? std::min(c->side_blocks_per_sm, c->trace_blocks_per_sm) : c->trace_blocks_per_sm), wide_grid = grid_for(c, 8);
    const size_t sb = stack_bytes(c, TB);
    auto work_slot = [&]() { int s = C_WORK + 2 * work_seq; ++work_seq; return s; };
    const int refill = (q == 0 ? c->refill0 : c->refill) | (c->chunk_div << 8);
    if (ds.n_point_lights > 0) {
        if (ds.shadow_type == 0) {
            LaunchScope ls(c, st, F_SHADOW_HARD);
            k_shadow_hard<<<trace_grid, TB, sb, st>>>(ds, fb, q, work_slot(), refill, c->traversal == WRT_TRAVERSAL_EXHAUSTIVE ? 1 : 0);
        } else {
            // per-request candidate lists (kernels.cuh, K4b'); scenes with light avatars keep the per-ray kernel,
            // whose literal hasIntersection path they need, and so does WRT_TRAVERSAL_EXHAUSTIVE
            const bool lists = c->soft_lists && !ds.has_light_prims && ds.n_nodes > 0 && c->traversal == WRT_TRAVERSAL_PRUNED &&
                               (unsigned long long)fb.preq_cap[q] * WRT_SOFT_SAMPLES < (1ull << 32);
            if (lists) {
                const SoftListBuffers& lb = c->list_bufs[q];
                {
                    LaunchScope ls(c, st, F_SOFT_LISTS);
                    k_soft_lists<<<trace_grid, TB, sb, st>>>(ds, fb, q, work_slot(), c->stack_rows, lb);
                }
                const bool filtered = c->soft_filter >= (q == 0 ? 2 : 1);
                if (filtered) {                                     // triangle-level pruning of the lists
                    LaunchScope ls(c, st, F_SOFT_FILTER);
                    k_soft_filter<<<WRT_FILTER_DYNAMIC ? c->filter_grid : wide_grid, TB, 0, st>>>(ds, fb, q, lb, WRT_FILTER_DYNAMIC ? work_slot() : 0);
                }
                LaunchScope ls(c, st, F_SHADOW_SOFT);
                k_soft_list_rays<<<trace_grid, TB, sb, st>>>(ds, fb, q, work_slot(), c->seed, lb, filtered ? 1 : 0);
            } else {
                LaunchScope ls(c, st, F_SHADOW_SOFT);
                k_shadow_soft<<<trace_grid, TB, sb, st>>>(ds, fb, q, work_slot(), c->seed, c->refill_soft | (c->chunk_div << 8),
                                                          c->cache_from_level <= (q == 0 ? 0 : 1) ? 1 : 0);
            }
        }
    }
    if (ds.n_dir_lights > 0) {
        LaunchScope ls(c, st, F_SHADOW_DIR);
        k_shadow_directional<<<wide_grid, TB, sb, st>>>(ds, fb, q, c->traversal == WRT_TRAVERSAL_EXHAUSTIVE ? 1 : 0);
    }
    return 0;
}

// Enqueues one batch of primary slots [slot0, slot0+n): closest-hit chain + deep shadows on `chain`, level 0's shadow
// work on `side`.
int enqueue_batch(WrtContext* c, long long slot0, unsigned n, uint8_t* d_image, uint8_t* d_packed) {
    using namespace wrt;
    FrameBuffers& fb = c->fb;
    const DevScene& ds = c->ds;
    cudaStream_t st = c->chain;
    // (kernel timing serialises the frame: every launch on the chain stream.  WRT_TIMING_OVERLAP=1 keeps the two streams and
    // turns the event pairs into a timeline of the frame as it really runs: WRT_TIMING_DUMP prints start and end of every launch)
    const bool overlap = c->overlap && (!c->kernel_timing || getenv("WRT_TIMING_OVERLAP") != nullptr);
    cudaStream_t ss = overlap ? c->side : st;
    PrimaryGen pg;
    pg.cam = c->cam; pg.tm = c->tilemap(); pg.slot0 = slot0;
    CK(cudaMemsetAsync(fb.counters, 0, C_TOTAL * sizeof(unsigned), st));
    int work_seq = 0;
    auto work_slot = [&]() { int s = C_WORK + 2 * work_seq; ++work_seq; return s; };
    const int TB = 128;
    const int trace_grid = grid_for(c, c->trace_blocks_per_sm), wide_grid = grid_for(c, 8);
    const size_t sb = stack_bytes(c, TB);
    const float prune = prune_value(c);
    auto cull_for = [&](int d) {
        // request culling belongs to the pruned mode; WRT_TRAVERSAL_EXHAUSTIVE traces every ray the reference traces
        int cull = 0;
        if (c->traversal == WRT_TRAVERSAL_PRUNED) {
            if (c->unlit_cull) cull |= WRT_CULL_UNLIT;
            // The shaft test at spawn time pays where most shafts are empty (primary hits: 79 % in the metric frame); on
            // deeper levels (~8 %) k_soft_lists finds the empty ones anyway (an empty list), off the critical
            // closest-hit chain.  Without the list kernels the test runs on every level.
            const bool lists_on = c->soft_lists && !ds.has_light_prims;
            if (c->shaft_cull && ds.shadow_type != 0 && (d <= c->shaft_cull_max_level || !lists_on)) cull |= WRT_CULL_SHAFT;
        }
        return cull;
    };
    auto level_kernels = [&](int d) {
        const int refill = (d == 0 ? c->refill0 : c->refill) | (c->chunk_div << 8);
        {
            LaunchScope ls(c, st, F_TRACE);
            if (d == 0) k_trace_closest<true><<<trace_grid, TB, sb, st>>>(ds, fb, pg, d, n, work_slot(), prune, refill);
            else k_trace_closest<false><<<trace_grid, TB, sb, st>>>(ds, fb, pg, d, n, work_slot(), prune, refill);
        }
        LaunchScope ls(c, st, F_SURFACE);
        k_surface_spawn<<<wide_grid, 256, 0, st>>>(ds, fb, pg, d, n, cull_for(d));
    };
    level_kernels(0);
    if (overlap) {
        CK(cudaEventRecord(c->ev_lvl0, st));
        CK(cudaStreamWaitEvent(ss, c->ev_lvl0, 0));
    }
    // Level 0's shadow + shade kernels run beside the deep chain on the side stream, then the shadow kernels of levels
    // 1..split (queue 1) as soon as those levels' surface stages are done; the chain goes on with the deeper levels and
    // ends with their shadow kernels (queue 2).  A deep level holds few, long, incoherent rays and leaves most of the SMs
    // idle, and a persistent traversal kernel ends with its longest ray: the shadow work fills those gaps.
    if (enqueue_shadows(c, ss, 0, work_seq)) return 1;
    if (c->shade0_separate) {
        LaunchScope ls(c, ss, F_SHADE);
        k_shade<<<wide_grid, 256, 0, ss>>>(ds, fb, n, 0, 0);
    }
    const int split = std::max(1, std::min(WRT_MAX_DEPTH - 1, c->deep_split));
    for (int d = 1; d <= split; d++) level_kernels(d);
    if (overlap) {
        CK(cudaEventRecord(c->ev_mid, st));
        CK(cudaStreamWaitEvent(ss, c->ev_mid, 0));
    }
    if (enqueue_shadows(c, ss, 1, work_seq)) return 1;
    if (overlap) CK(cudaEventRecord(c->ev_side, ss));
    for (int d = split + 1; d < WRT_MAX_DEPTH; d++) level_kernels(d);
    if (split < WRT_MAX_DEPTH - 1 && enqueue_shadows(c, st, 2, work_seq)) return 1;
    if (overlap) CK(cudaStreamWaitEvent(st, c->ev_side, 0));
    {
        LaunchScope ls(c, st, F_COMBINE);
        int shade_from = c->shade0_separate ? 1 : 0;
        TileMap tm = pg.tm;
        void* args[] = {(void*)&ds, (void*)&fb, (void*)&tm, (void*)&slot0, (void*)&n, (void*)&shade_from, (void*)&d_image, (void*)&d_packed};
        CK(cudaLaunchCooperativeKernel((const void*)k_combine_resolve, dim3(c->coop_grid), dim3(256), args, 0, st));
    }
    if (c->copy_float)                                 // the combined level-0 colours this batch quantised, in slot order
        CK(cudaMemcpyAsync(c->h_float + slot0, fb.node_a, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, st));
    CK(cudaGetLastError());
    if (C_WORK + 2 * work_seq > C_TOTAL) return fail("internal: work counters exceed the counter block");
    return 0;
}

void add_batch_stats(WrtContext* c, const unsigned* cnt) {
    WrtStats& s = c->stats;
    const wrt::DevScene& ds = c->ds;
    s.rays_per_depth[0] += cnt[wrt::C_VALID0];
    s.closest_rays += cnt[wrt::C_VALID0];
    for (int d = 1; d < WRT_MAX_DEPTH; d++) {
        s.rays_per_depth[d] += cnt[wrt::C_NRAYS + d] + cnt[wrt::C_NTRAYS + d];
        s.closest_rays += cnt[wrt::C_NRAYS + d] + cnt[wrt::C_NTRAYS + d];
    }
    // requests answered without tracing count like the reference counts them (it traces them)
    int64_t culled = 0, skip_p = 0, skip_d = 0;
    for (int d = 0; d < WRT_MAX_DEPTH; d++) { culled += cnt[wrt::C_NCULL + d]; skip_p += cnt[wrt::C_NSKIP + d]; skip_d += cnt[wrt::C_NDSKIP + d]; }
    int64_t queued_p = 0, queued_d = 0;
    for (int q = 0; q < WRT_QUEUES; q++) { queued_p += cnt[wrt::C_NPREQ + q]; queued_d += cnt[wrt::C_NDREQ + q]; }
    const int64_t empty = cnt[wrt::C_NEMPTY];          // queued, but their candidate list came out empty: no rays built
    const int64_t p = queued_p + culled + skip_p, q = queued_d + skip_d;
    const int64_t per = ds.shadow_type ? WRT_SOFT_SAMPLES : 1;
    s.shadow_requests += p + q;
    s.shadow_rays += p * per + q;
    s.shaft_culled_requests += culled + empty;
    s.unlit_skipped_requests += skip_p + skip_d;
    s.shadow_rays_traced += (queued_p - empty) * per + queued_d;
}

#ifdef WRT_DEBUG_BOUNDS
int check_debug_bounds() {
    unsigned line = 0, stack = 0;
    CK(cudaMemcpyFromSymbol(&line, wrt::g_wrt_bounds_line, sizeof line));
    CK(cudaMemcpyFromSymbol(&stack, wrt::g_wrt_stack_overflow, sizeof stack));
    if (line || stack) {                                // report once, then re-arm
        const unsigned zero = 0;
        cudaMemcpyToSymbol(wrt::g_wrt_bounds_line, &zero, sizeof zero);
        cudaMemcpyToSymbol(wrt::g_wrt_stack_overflow, &zero, sizeof zero);
    }
    if (line) return fail("WRT_DEBUG_BOUNDS: index out of bounds at kernels.cuh:" + std::to_string(line));
    if (stack) return fail("WRT_DEBUG_BOUNDS: traversal stack overflow (sp " + std::to_string(stack - 1) + ")");
    return 0;
}
#else
int check_debug_bounds() { return 0; }
#endif

// A batch overflowed a deep-level queue.  Automatic sizing: double the deep-level capacity (kept for the following
// frames) while it is below 2x the batch; otherwise (or with a caller-fixed factor) the batch is split in halves.
// Returns true when the buffers grew and the same batch should simply be rendered again.
bool grow_after_overflow(WrtContext* c) {
    const float effective = (float)c->deep_slots / (float)std::max(1u, c->batch_slots);
    const float limit = 4.f;                           // (per-level capacity in primary-batch units; beyond it: smaller batches)
    if (c->queue_factor > 0.f || effective >= limit) return false;
    const float old = c->deep_factor;
    c->deep_factor = std::min(limit, std::max(old, effective) * 2.f);
    if (ensure_frame_buffers(c, c->batch_slots) == 0) return true;
    c->deep_factor = old;                              // out of memory: fall back to halving
    cudaGetLastError();
    return false;
}

// Renders the spans on `todo` (popped from the back) synchronously, re-rendering what overflows.
int render_spans_sync(WrtContext* c, std::vector<std::pair<long long, long long>>& todo, uint8_t* d_image, uint8_t* d_packed) {
    cudaStream_t st = c->chain;
    while (!todo.empty()) {
        auto [s0, n] = todo.back();
        todo.pop_back();
        if (n <= 0) continue;
        if (enqueue_batch(c, s0, (unsigned)n, d_image, d_packed)) return 1;
        CK(cudaMemcpyAsync(c->h_counters, c->fb.counters, wrt::C_TOTAL * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (c->h_counters[wrt::C_OVERFLOW]) {
            ++c->stats.overflow_retries;
            if (grow_after_overflow(c)) { todo.push_back({s0, n}); continue; }
            if (n <= 64) return fail("ray queue overflow on a 64-slot batch: raise queue_factor");
            long long half = ((n / 2 + 31) / 32) * 32;
            if (c->queue_factor <= 0.f) c->learned_batch = std::min(c->learned_batch, half);
            todo.push_back({s0 + half, n - half});
            todo.push_back({s0, half});
            continue;
        }
        add_batch_stats(c, c->h_counters);
    }
    return 0;
}

// Renders all local slots.  A single-batch frame (the common case) is enqueued without any host synchronisation;
// overflow is checked — and the frame redone — in finish_frame.
int render_all(WrtContext* c, cudaStream_t user, bool join_user, uint8_t* d_image, uint8_t* d_packed) {
    if (!c->has_scene) return fail("wrt_render: no scene uploaded");
    if (!c->has_cam) return fail("wrt_render: no camera set");
    if (c->cam.width <= 0 || c->cam.height <= 0) return fail("wrt_render: empty image");
    if (!c->textures_complete) return fail("wrt_render: a primitive references a texture / normal map that was not uploaded");
    const long long total = c->local_slots(c->rank, c->world);
    {
        const long long key[4] = {c->cam.width, c->cam.height, ((long long)c->ds.n_prims << 8) | (c->ds.n_lights << 1) | (c->ds.shadow_type & 1),
                                  ((long long)c->world << 32) | (unsigned)c->traversal};
        if (memcmp(key, c->learned_key, sizeof key)) { memcpy(c->learned_key, key, sizeof key); c->learned_batch = 1ll << 40; }
    }
    const long long max_batch = std::min(c->max_batch, c->learned_batch);
    memset(&c->stats, 0, sizeof c->stats);
    c->timed.clear();
    c->event_next = 0;
    c->user_stream = user;
    c->user_stream_joined = join_user;
    c->last_image = d_image; c->last_packed = d_packed;
    c->has_frame = true;
    cudaStream_t st = c->chain;
    if (total > 0) {
        unsigned want = (unsigned)std::min(total, max_batch);
        if (ensure_frame_buffers(c, want)) return 1;
    }
    if (join_user) {                                    // everything the caller enqueued before is visible to the frame
        CK(cudaEventRecord(c->ev_in, user));
        CK(cudaStreamWaitEvent(st, c->ev_in, 0));
    }
    CK(cudaEventRecord(c->ev_begin, st));
    std::vector<std::pair<long long, long long>> todo;
    for (long long s0 = total; s0 > 0;) {              // push in reverse so spans pop in order
        long long b = (s0 - 1) / max_batch * max_batch;
        todo.push_back({b, s0 - b});
        s0 = b;
    }
    if (todo.size() == 1) {                            // stay asynchronous, check in finish
        if (enqueue_batch(c, todo[0].first, (unsigned)todo[0].second, d_image, d_packed)) return 1;
        CK(cudaMemcpyAsync(c->h_counters, c->fb.counters, wrt::C_TOTAL * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
        c->frame_pending = true;
    } else if (render_spans_sync(c, todo, d_image, d_packed)) return 1;
    CK(cudaEventRecord(c->ev_end, st));
    if (join_user) {
        CK(cudaEventRecord(c->ev_out, st));
        CK(cudaStreamWaitEvent(user, c->ev_out, 0));
    }
    return 0;
}

void tally_kernel_times(WrtContext* c);

int finish_frame(WrtContext* c) {
    cudaStream_t st = c->chain;
    CK(cudaStreamSynchronize(st));
    if (c->frame_pending) {
        c->frame_pending = false;
        if (c->h_counters[wrt::C_OVERFLOW]) {
            // the single-batch frame overflowed a queue: redo it synchronously (larger deep levels, or in halves)
            const long long total = c->local_slots(c->rank, c->world);
            memset(&c->stats, 0, sizeof c->stats);
            c->stats.overflow_retries = 1;
            std::vector<std::pair<long long, long long>> todo;
            if (grow_after_overflow(c)) todo.push_back({0, total});
            else {
                if (total <= 64) return fail("ray queue overflow on a 64-slot batch: raise queue_factor");
                long long half = ((total / 2 + 31) / 32) * 32;
                if (c->queue_factor <= 0.f) c->learned_batch = std::min(c->learned_batch, half);
                todo.push_back({half, total - half});
                todo.push_back({0, half});
            }
            if (render_spans_sync(c, todo, c->last_image, c->last_packed)) return 1;
            CK(cudaEventRecord(c->ev_end, st));
            CK(cudaStreamSynchronize(st));
        } else {
            add_batch_stats(c, c->h_counters);
        }
    }
    if (check_debug_bounds()) return 1;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev_begin, c->ev_end) == cudaSuccess) c->stats.gpu_ms = ms;
    tally_kernel_times(c);
    return 0;
}

// Per-family times and launch counts of the timed launches since c->timed was cleared (ev_begin: their common start).
void tally_kernel_times(WrtContext* c) {
    for (float& f : c->family_ms) f = 0.f;
    for (int& n : c->family_launches) n = 0;
    const bool dump = getenv("WRT_TIMING_DUMP") != nullptr;      // development: every timed launch, in enqueue order
    for (const TimedLaunch& tl : c->timed) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, tl.e0, tl.e1) == cudaSuccess) { c->family_ms[tl.family] += t; ++c->family_launches[tl.family]; }
        if (dump) {
            float t0 = 0.f, t1 = 0.f;
            cudaEventElapsedTime(&t0, c->ev_begin, tl.e0);
            cudaEventElapsedTime(&t1, c->ev_begin, tl.e1);
            fprintf(stderr, "[wrt] launch family %d: %.1f us  (%s stream, %.1f -> %.1f us after the frame's start)\n", tl.family, t * 1e3f,
                    tl.on_chain ? "chain" : "side", t0 * 1e3f, t1 * 1e3f);
        }
    }
}

} // namespace

extern "C" {

const char* wrt_last_error(void) { return g_err.c_str(); }

int wrt_create(int device, WrtContext** out) {
    if (!out) return fail("wrt_create: null out pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(std::string("wrt_create: no CUDA device (") + cudaGetErrorString(e) +
                    "); this library has no CPU fallback");
    if (device < 0 || device >= n) return fail("wrt_create: device index out of range");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(std::string("wrt_create: ") + prop.name + " is sm_" + std::to_string(prop.major) +
                    std::to_string(prop.minor) + "; this library is built for sm_100a only");
    WrtContext* c = new WrtContext();
    c->device = device;
    c->num_sms = prop.multiProcessorCount;
    int prio_least = 0, prio_greatest = 0;
    cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    bool ev_ok = cudaStreamCreateWithPriority(&c->chain, cudaStreamNonBlocking, prio_greatest) == cudaSuccess &&
                 cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, prio_least) == cudaSuccess;
    for (cudaEvent_t* e : {&c->ev_in, &c->ev_lvl0, &c->ev_mid, &c->ev_side, &c->ev_out})
        ev_ok = ev_ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
    if (!ev_ok ||
        cudaEventCreate(&c->ev_begin) != cudaSuccess || cudaEventCreate(&c->ev_end) != cudaSuccess ||
        cudaMallocHost((void**)&c->h_counters, (wrt::C_TOTAL + 64) * sizeof(unsigned)) != cudaSuccess) {
        delete c;
        return fail("wrt_create: stream/event/pinned allocation failed");
    }
    memset(c->h_counters, 0, wrt::C_TOTAL * sizeof(unsigned));
    {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wrt::k_combine_resolve, 256, 0) != cudaSuccess || per_sm < 1) {
            wrt_destroy(c);
            return fail("wrt_create: cooperative launch of k_combine_resolve is not possible on this device");
        }
        c->coop_grid = c->num_sms * std::min(per_sm, 4);
        per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wrt::k_bvh_ploc, WRT_PLOC_THREADS, 0) != cudaSuccess || per_sm < 1) {
            wrt_destroy(c);
            return fail("wrt_create: cooperative launch of k_bvh_ploc is not possible on this device");
        }
        c->ploc_coop_grid = c->num_sms * std::min(per_sm, 2);
        per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wrt::k_soft_filter, 128, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
        c->filter_grid = c->num_sms * per_sm;           // one wave: the kernel claims its work dynamically
    }
    // tuning overrides (development only; defaults are what bench.py measures)
    if (const char* e = getenv("WRT_REFILL")) c->refill = std::max(1, std::min(32, atoi(e)));
    if (const char* e = getenv("WRT_REFILL_SOFT")) c->refill_soft = std::max(1, std::min(32, atoi(e)));
    if (const char* e = getenv("WRT_TRACE_BLOCKS")) c->trace_blocks_per_sm = std::max(1, std::min(32, atoi(e)));
    if (const char* e = getenv("WRT_OVERLAP")) c->overlap = atoi(e) != 0;
    if (const char* e = getenv("WRT_CACHE_FROM")) c->cache_from_level = atoi(e);
    if (const char* e = getenv("WRT_SHAFT_CULL")) c->shaft_cull = atoi(e) != 0;
    if (const char* e = getenv("WRT_UNLIT_CULL")) c->unlit_cull = atoi(e) != 0;
    if (const char* e = getenv("WRT_SOFT_LISTS")) c->soft_lists = atoi(e) != 0;
    if (const char* e = getenv("WRT_LIST_POOL_CAP")) c->list_pool_cap_override = atoll(e);
    if (const char* e = getenv("WRT_SHAFT_LEVELS")) c->shaft_cull_max_level = atoi(e);
    if (const char* e = getenv("WRT_CHUNK_DIV")) c->chunk_div = std::max(0, std::min(255, atoi(e)));
    if (const char* e = getenv("WRT_REFILL0")) c->refill0 = std::max(1, std::min(32, atoi(e)));
    if (const char* e = getenv("WRT_HOST_BVH")) c->host_bvh = atoi(e) != 0;
    if (const char* e = getenv("WRT_SHADE0_SEPARATE")) c->shade0_separate = atoi(e) != 0;
    if (const char* e = getenv("WRT_SOFT_FILTER")) c->soft_filter = atoi(e);
    if (const char* e = getenv("WRT_SIDE_BLOCKS")) c->side_blocks_per_sm = std::max(0, std::min(32, atoi(e)));
    if (const char* e = getenv("WRT_DEEP_SPLIT")) c->deep_split = std::max(1, std::min(WRT_MAX_DEPTH - 1, atoi(e)));
    if (const char* e = getenv("WRT_DEEP_FACTOR")) { c->deep_factor = std::max(0.001f, std::min(2.f, (float)atof(e))); c->small_batch_full_levels = false; }
    if (const char* e = getenv("WRT_MAX_BATCH")) c->max_batch = std::max(64ll, (atoll(e) + 31) / 32 * 32);   // tests: force multi-batch frames
    *out = c;
    return 0;
}

void wrt_destroy(WrtContext* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    free_scene(c);
    free_frame(c);
    for (int k = 0; k < 5; k++) if (c->d_scratch[k]) cudaFree(c->d_scratch[k]);
    if (c->d_image) cudaFree(c->d_image);
    if (c->h_image) cudaFreeHost(c->h_image);
    if (c->h_float) cudaFreeHost(c->h_float);
    if (c->h_counters) cudaFreeHost(c->h_counters);
    if (c->h_stage) cudaFreeHost(c->h_stage);
    for (cudaEvent_t e : c->event_pool) cudaEventDestroy(e);
    if (c->ev_begin) cudaEventDestroy(c->ev_begin);
    if (c->ev_end) cudaEventDestroy(c->ev_end);
    for (cudaEvent_t e : {c->ev_in, c->ev_lvl0, c->ev_mid, c->ev_side, c->ev_out}) if (e) cudaEventDestroy(e);
    if (c->side) cudaStreamDestroy(c->side);
    if (c->chain) cudaStreamDestroy(c->chain);
    delete c;
}

// Scene upload.  The host only STAGES bytes: every array of the description is copied into one pinned staging
// buffer and crosses PCIe in a single cudaMemcpyAsync; everything derived — per-primitive boxes, the SAH-quality tree
// the kernels walk (PLOC build, bvh_build.cuh), its dilated copy, the 8 octant copies of both trees, the float4
// geometry / attribute / id / material layouts — is produced by kernels on the device.  One small read-back (tree
// depth, flags) ends the call.
int wrt_upload_scene(WrtContext* c, const WrtSceneDesc* s) {
    if (!c || !s) return fail("wrt_upload_scene: null argument");
    CK(cudaSetDevice(c->device));
    if (s->n_nodes < 0 || s->n_prims < 0 || s->n_materials < 0 || s->n_lights < 0 || s->n_textures < 0 || s->n_normalmaps < 0 || s->n_texels < 0)
        return fail("wrt_upload_scene: negative count in the scene description");
    if (s->n_prims > 0 && s->n_nodes != 2 * s->n_prims)
        return fail("wrt_upload_scene: a tree over n one-primitive leaves has 2n records (root, padding, n-1 sibling pairs)");
    if (s->n_prims > 0 && s->n_materials == 0) return fail("wrt_upload_scene: primitives without materials");
    // indices a kernel follows without a device-side check are validated here (the rest — material, texture, leaf
    // links — by the kernels that unpack them)
    for (int i = 0; i < s->n_textures + s->n_normalmaps; i++) {
        const WrtTexture& t = i < s->n_textures ? s->textures[i] : s->normalmaps[i - s->n_textures];
        if (t.offset < 0 || t.count < 0 || t.offset + t.count > s->n_texels) return fail("wrt_upload_scene: texture texel range outside texels[]");
    }
    for (int i = 0; i < s->n_nodes; i++) {             // child links of the caller's tree stay inside it
        const int link = s->nodes[i].link;
        if (i != 1 && link >= 0 && (link < 2 || link + 1 >= s->n_nodes)) return fail("wrt_upload_scene: tree child link out of range");
    }
    cudaStream_t st = c->chain;                         // ordered behind any frame still in flight: it may read the old scene
    c->has_scene = false;
    c->scene_slot = 0;
    wrt::DevScene& ds = c->ds;
    memset(&ds, 0, sizeof ds);
    c->textures_complete = true;
    const int np = s->n_prims, nn = s->n_nodes;
    static_assert(sizeof(WrtNode) == 32, "WrtNode must be 32 bytes");
    static_assert(sizeof(WrtMaterial) == 48, "WrtMaterial must be 12 floats");

    c->bvh_depth = tree_depth(s);

    // ---- 1. stage + one H2D ----
    struct Part { const void* src; size_t bytes; size_t off; };
    Part parts[] = {
        {s->nodes, (size_t)nn * sizeof(WrtNode), 0},                 // 0
        {s->prim_geom, (size_t)np * 48, 0},                          // 1
        {s->prim_flags, (size_t)np * 4, 0},                          // 2
        {s->prim_material, (size_t)np * 4, 0},                       // 3
        {s->prim_texture, (size_t)np * 4, 0},                        // 4
        {s->prim_normalmap, (size_t)np * 4, 0},                      // 5
        {s->prim_object, (size_t)np * 4, 0},                         // 6
        {s->object_prim, (size_t)np * 4, 0},                         // 7
        {s->prim_normals, (size_t)np * 36, 0},                       // 8
        {s->prim_uv, (size_t)np * 24, 0},                            // 9
        {s->materials, (size_t)s->n_materials * sizeof(WrtMaterial), 0},   // 10
        {s->lights, (size_t)s->n_lights * sizeof(WrtLight), 0},      // 11
        {s->textures, (size_t)s->n_textures * sizeof(WrtTexture), 0},      // 12
        {s->normalmaps, (size_t)s->n_normalmaps * sizeof(WrtTexture), 0},  // 13
        {s->texels, (size_t)s->n_texels * 12, 0},                    // 14
        {nullptr, 0, 0},                                             // 15: path codes of the primitives (below)
    };
    // Root-to-leaf paths of the primitives in the scene's (= the reference's) tree: what the hard-shadow product needs to
    // multiply in that tree's association (shadow_assoc.h).  A tree deeper than 64 gets none (visit-order product).
    if (wrt_make_path_codes(s->nodes, nn, np, c->path_codes)) {
        parts[15].src = c->path_codes.data();
        parts[15].bytes = c->path_codes.size() * sizeof(WrtPathCode);
    }
    size_t total = 0;
    for (Part& p : parts) {
        if (p.bytes && !p.src) return fail("wrt_upload_scene: null array with a non-zero count");
        p.off = total;
        total += (p.bytes + 255) & ~(size_t)255;
    }
    total = std::max<size_t>(total, 256);
    if (c->h_stage_bytes < total) {
        if (c->h_stage) cudaFreeHost(c->h_stage);
        c->h_stage = nullptr; c->h_stage_bytes = 0;
        CK(cudaMallocHost((void**)&c->h_stage, total + total / 4));
        c->h_stage_bytes = total + total / 4;
    }
    for (const Part& p : parts) if (p.bytes) memcpy(c->h_stage + p.off, p.src, p.bytes);
    uint8_t* d_stage = nullptr;
    if (dev_alloc(c, total, (void**)&d_stage)) return 1;
    CK(cudaMemcpyAsync(d_stage, c->h_stage, total, cudaMemcpyHostToDevice, st));
    auto dptr = [&](int k) { return d_stage + parts[k].off; };
    ds.nodes = (const float4*)dptr(0);
    ds.object_prim = (const int*)dptr(7);
    ds.lights = (const WrtLight*)dptr(11);
    ds.textures = (const WrtTexture*)dptr(12);
    ds.normalmaps = (const WrtTexture*)dptr(13);
    ds.texels = (const float*)dptr(14);
    ds.path_codes = parts[15].bytes ? (const WrtPathCode*)dptr(15) : nullptr;

    // ---- 2. device-side layouts ----
    float4 *geom = nullptr, *attr = nullptr, *mats = nullptr, *pbox = nullptr, *taux = nullptr, *fnodes = nullptr, *dnodes = nullptr, *onodes = nullptr, *ronodes = nullptr, *wnodes = nullptr;
    int4* ids = nullptr;
    int* d_flags = nullptr;
    if (dev_alloc(c, (size_t)np * 48, (void**)&geom) || dev_alloc(c, (size_t)np * 64, (void**)&attr) || dev_alloc(c, (size_t)np * 16, (void**)&ids) ||
        dev_alloc(c, (size_t)s->n_materials * 48, (void**)&mats) || dev_alloc(c, (size_t)np * 32, (void**)&pbox) ||
        dev_alloc(c, (size_t)np * 16, (void**)&taux) ||
        dev_alloc(c, (size_t)nn * 32, (void**)&fnodes) || dev_alloc(c, (size_t)nn * 32, (void**)&dnodes) ||
        dev_alloc(c, (size_t)nn * 32 * 8, (void**)&onodes) || dev_alloc(c, (size_t)nn * 32 * 8, (void**)&ronodes) ||
        dev_alloc(c, (size_t)nn * 64 * 8, (void**)&wnodes) ||
        dev_alloc(c, (wrt::BS_TOTAL + 16) * sizeof(int), (void**)&d_flags))
        return 1;
    int* d_state = d_flags + 8;
    float* d_bounds = (float*)(d_flags + 8 + wrt::BS_TOTAL);           // centroid bounds of the leaf boxes (min xyz, max xyz)
    CK(cudaMemsetAsync(d_flags, 0, (wrt::BS_TOTAL + 8) * sizeof(int), st));
    {
        const float init[8] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX, 0.f, 0.f};
        memcpy(c->h_counters + wrt::C_TOTAL + 32, init, sizeof init);   // (pinned; the copy below reads it asynchronously)
        CK(cudaMemcpyAsync(d_bounds, c->h_counters + wrt::C_TOTAL + 32, sizeof init, cudaMemcpyHostToDevice, st));
    }
    const int wide = c->num_sms * 4;
    if (np > 0) {
        ++c->launches;
        wrt::k_pack_prims<<<std::min(wide, (np + 255) / 256), 256, 0, st>>>(
            np, (const float*)dptr(1), (const unsigned*)dptr(2), (const int*)dptr(3), (const int*)dptr(4), (const int*)dptr(5),
            (const int*)dptr(6), (const float*)dptr(8), (const float*)dptr(9), (const float*)dptr(10), s->n_materials, s->n_textures,
            s->n_normalmaps, geom, attr, ids, taux, d_flags);
    }
    if (s->n_materials > 0) {
        ++c->launches;
        wrt::k_pack_materials<<<std::min(wide, (s->n_materials + 255) / 256), 256, 0, st>>>((const float*)dptr(10), s->n_materials, mats);
    }
    ds.geom = geom; ds.attr = attr; ds.ids = ids; ds.materials = mats; ds.prim_box = pbox; ds.tri_aux = taux;
    ds.fnodes = fnodes; ds.dnodes = dnodes; ds.onodes = onodes; ds.ronodes = ronodes; ds.wnodes = wnodes;

    // ---- 3. trees ----
    int fast_depth = 0;
    bool host_build = c->host_bvh;
    // the host's binned-SAH build of fast_bvh.hpp into fnodes / dnodes / prim_box (synchronous)
    auto build_on_host = [&]() -> int {
        wrt::FastBvhBuilder& fbvh = c->fbvh;
        fbvh.build(s);
        if (fbvh.nodes.size() != (size_t)nn) return fail("wrt_upload_scene: fast BVH build failed");
        std::vector<WrtNode> dil = fbvh.dilated(1e-3f, 1e-4f);
        std::vector<float4> hb(2 * (size_t)np, make_float4(0.f, 0.f, 0.f, 0.f));
        for (int i = 0; i < nn; i++) {
            const WrtNode& nd = s->nodes[i];
            if (nd.link >= 0 || i == 1) continue;
            int p = ~nd.link;
            if (p < 0 || p >= np) return fail("wrt_upload_scene: leaf link out of range");
            hb[2 * (size_t)p] = make_float4(nd.pmin[0], nd.pmin[1], nd.pmin[2], 0.f);
            hb[2 * (size_t)p + 1] = make_float4(nd.pmax[0], nd.pmax[1], nd.pmax[2], 0.f);
        }
        CK(cudaMemcpyAsync(fnodes, fbvh.nodes.data(), (size_t)nn * 32, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(dnodes, dil.data(), (size_t)nn * 32, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(pbox, hb.data(), hb.size() * 16, cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));                  // the host vectors above go out of scope
        fast_depth = fbvh.max_depth;
        return 0;
    };
    // the per-octant and 4-wide copies of the walked tree, and the octant copies of the reference's tree
    auto copy_walked_tree = [&](bool with_reference) {
        const int g = (int)std::min<long long>(wide, (8ll * nn + 255) / 256);
        c->launches += with_reference ? 3 : 2;
        wrt::k_octant_copies<<<g, 256, 0, st>>>(fnodes, nn, onodes);
        if (with_reference) wrt::k_octant_copies<<<g, 256, 0, st>>>(ds.nodes, nn, ronodes);
        wrt::k_wide4_copies<<<(int)std::min<long long>(wide, (4ll * nn + 255) / 256), 256, 0, st>>>(onodes, nn, wnodes);
    };
    auto t_b0 = std::chrono::steady_clock::now();
    if (np > 0 && !host_build) {
        wrt::BuildBuffers bb{};
        const size_t n2 = 2 * (size_t)np;
        size_t cub_bytes = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                        (const int*)nullptr, (int*)nullptr, np, 0, 63, st);
        const int ploc_grid = std::max(1, std::min(c->ploc_coop_grid, (np + 2 * WRT_PLOC_THREADS - 1) / (2 * WRT_PLOC_THREADS)));
        if (dev_alloc(c, n2 * 16, (void**)&bb.tree.lo) || dev_alloc(c, n2 * 16, (void**)&bb.tree.hi) || dev_alloc(c, n2 * 16, (void**)&bb.tree.dlo) ||
            dev_alloc(c, n2 * 16, (void**)&bb.tree.dhi) || dev_alloc(c, n2 * 4, (void**)&bb.tree.parent) || dev_alloc(c, n2 * 4, (void**)&bb.tree.cnt) ||
            dev_alloc(c, (size_t)np * 8, (void**)&bb.keys[0]) || dev_alloc(c, (size_t)np * 8, (void**)&bb.keys[1]) ||
            dev_alloc(c, (size_t)np * 4, (void**)&bb.vals[0]) || dev_alloc(c, (size_t)np * 4, (void**)&bb.vals[1]) ||
            dev_alloc(c, (size_t)np * 4, (void**)&bb.cl[0]) || dev_alloc(c, (size_t)np * 4, (void**)&bb.cl[1]) ||
            dev_alloc(c, (size_t)np * 4, (void**)&bb.nn) || dev_alloc(c, (size_t)ploc_grid * 4, (void**)&bb.blk) ||
            dev_alloc(c, cub_bytes, &bb.cub_temp))
            return 1;
        bb.state = d_state;
        bb.cub_temp_bytes = cub_bytes;
        c->launches += 5;
        CK(cudaMemsetAsync(bb.tree.cnt, 0, (size_t)np * 4, st));
        wrt::k_bvh_leaves<<<std::min(wide, (nn + 255) / 256), 256, 0, st>>>(ds.nodes, nn, np, bb, pbox, d_bounds, 1e-3f, 1e-4f);
        wrt::k_bvh_keys<<<std::min(wide, (np + 255) / 256), 256, 0, st>>>(np, bb, d_bounds);
        CK(cub::DeviceRadixSort::SortPairs(bb.cub_temp, cub_bytes, bb.keys[0], bb.keys[1], bb.vals[0], bb.vals[1], np, 0, 63, st));
        {
            const int* sorted = bb.vals[1];
            int n_arg = np, radius = WRT_PLOC_RADIUS;
            void* args[] = {(void*)&bb, (void*)&sorted, (void*)&n_arg, (void*)&radius};
            CK(cudaLaunchCooperativeKernel((const void*)wrt::k_bvh_ploc, dim3(ploc_grid), dim3(WRT_PLOC_THREADS), args, 0, st));
        }
        wrt::k_bvh_layout<<<std::min(wide, (int)((n2 + 255) / 256)), 256, 0, st>>>(bb, np, fnodes, dnodes);
    } else if (np > 0) {
        // WRT_HOST_BVH=1 (development A/B)
        if (build_on_host()) return 1;
    }
    if (nn > 0) copy_walked_tree(true);
    CK(cudaGetLastError());
    unsigned* h_rb = c->h_counters + wrt::C_TOTAL;     // (the first C_TOTAL words belong to a frame that may still be in flight)
    CK(cudaMemcpyAsync(h_rb, d_flags, (wrt::BS_TOTAL + 8) * sizeof(int), cudaMemcpyDeviceToHost, st));

    // ---- 4. host-side scalars (while the device builds) ----
    for (int i = 0; i < s->n_lights && i < WRT_INLINE_LIGHTS; i++) ds.lights_c[i] = s->lights[i];
    ds.n_nodes = nn; ds.n_prims = np; ds.n_lights = s->n_lights;
    ds.n_point_lights = ds.n_dir_lights = 0;
    for (int i = 0; i < s->n_lights; i++) {
        if (fabsf(s->lights[i].pos[3] - 1.f) < 0.00001f) ++ds.n_point_lights;      // FLOAT_EQUAL(w, 1), Renderer.hpp:275
        else ++ds.n_dir_lights;
    }
    ds.shadow_type = s->shadow_type; ds.depth_cueing = s->depth_cueing;
    for (int k = 0; k < 3; k++) { ds.bkg[k] = s->bkgcolor[k]; ds.dc[k] = s->dc[k]; ds.eye[k] = s->eye[k]; }
    ds.eta = s->eta;
    ds.amin = s->amin; ds.amax = s->amax; ds.distmin = s->distmin; ds.distmax = s->distmax;
    CK(cudaStreamSynchronize(st));
    auto t_b1 = std::chrono::steady_clock::now();
    const int* rb = (const int*)h_rb;
    const int flags = rb[0];
    const int* state = rb + 8;
    if (state[wrt::BS_ERROR] == 1) return fail("wrt_upload_scene: leaf link out of range in the scene's tree (every primitive needs exactly one leaf record)");
    if (state[wrt::BS_ERROR]) return fail("wrt_upload_scene: device BVH build made no progress (non-finite boxes?)");
    if (flags & 4) return fail("wrt_upload_scene: primitive material index out of range");
    if (np > 0 && !host_build) {
        fast_depth = state[wrt::BS_DEPTH];
        if (state[wrt::BS_ALLOC] != 2 * np - 1) return fail("wrt_upload_scene: device BVH build is incomplete (a primitive without a leaf record?)");
    }
    ds.has_light_prims = (flags & 1) ? 1 : 0;
    memcpy(&ds.prune_slack, rb + 1, sizeof(float));     // k_pack_prims: scene maximum of wrt_prune_triangle_slack
    // the strategy queries never read texels; a frame render needs every referenced map present
    c->textures_complete = !(flags & 2);
    // binary walks push at most one entry per level; the 4-wide walks (wide_bvh.h) descend two levels per node and push up
    // to three.  90 rows x 128 threads x 4 B = 45 KB of dynamic shared memory per CTA: the reference's tree may be 88
    // levels deep, the walked tree 58.
    const int max_rows = 90;
    auto rows_for = [&](int walked) { return std::max(std::max(c->bvh_depth, walked), 3 * ((walked + 1) / 2)) + 2; };
    const int ploc_depth = host_build ? -1 : fast_depth;
    if (np > 0 && !host_build && rows_for(fast_depth) > max_rows) {
        // PLOC builds very deep trees over fans of triangles sharing a vertex and over boxes of very mixed sizes; the
        // host's binned SAH stays shallow on them.  Results do not depend on the walked tree's shape (DESIGN.md section 4).
        host_build = true;
        if (build_on_host()) return 1;
        copy_walked_tree(false);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(st));
        t_b1 = std::chrono::steady_clock::now();
    }
    c->stack_rows = rows_for(fast_depth);
#ifdef WRT_DEBUG_BOUNDS
    if (const char* e = getenv("WRT_DEBUG_STACK_ROWS")) c->stack_rows = std::max(1, atoi(e));   // provoke the stack check (tests)
#endif
    if (c->stack_rows > max_rows)
        return fail("wrt_upload_scene: acceleration tree too deep for the 90-row traversal stack (reference tree depth " +
                    std::to_string(c->bvh_depth) + ", at most 88; walked tree depth " + std::to_string(fast_depth) +
                    ", at most 58)");
    c->fast_depth = fast_depth;
    c->build_passes = state[wrt::BS_PASSES];
    c->has_scene = true;
    if (getenv("WRT_VERBOSE")) {
        char builder[96];
        if (!host_build) snprintf(builder, sizeof builder, "device PLOC, %d passes", c->build_passes);
        else if (c->host_bvh) snprintf(builder, sizeof builder, "host SAH");
        else snprintf(builder, sizeof builder, "host SAH: the %d-pass PLOC tree was %d levels deep", c->build_passes, ploc_depth);
        fprintf(stderr, "[wrt] upload: %d prims, %zu bytes staged, reference tree depth %d, walked tree depth %d (%s), %d stack rows, %.3f ms\n",
                np, total, c->bvh_depth, fast_depth, builder, c->stack_rows, std::chrono::duration<double, std::milli>(t_b1 - t_b0).count());
    }
    return 0;
}

int wrt_set_camera(WrtContext* c, const WrtCamera* cam) {
    if (!c || !cam) return fail("wrt_set_camera: null argument");
    if (cam->width < 0 || cam->height < 0) return fail("wrt_set_camera: negative image size");
    c->cam = *cam;
    c->has_cam = true;
    return 0;
}

int wrt_set_tiles(WrtContext* c, int tile_w, int tile_h, int rank, int world) {
    if (!c) return fail("wrt_set_tiles: null context");
    if (tile_w <= 0 || tile_h <= 0 || tile_w % 8 || tile_h % 4) return fail("wrt_set_tiles: tile must be a multiple of 8 x 4");
    if (world < 1 || rank < 0 || rank >= world) return fail("wrt_set_tiles: bad rank/world");
    c->tile_w = tile_w; c->tile_h = tile_h; c->rank = rank; c->world = world;
    return 0;
}

int wrt_set_options(WrtContext* c, int traversal, uint32_t seed, float queue_factor) {
    if (!c) return fail("wrt_set_options: null context");
    if (traversal != WRT_TRAVERSAL_EXHAUSTIVE && traversal != WRT_TRAVERSAL_PRUNED) return fail("wrt_set_options: bad traversal mode");
    c->traversal = traversal;
    c->seed = seed;
    if (queue_factor > 0 && queue_factor != c->queue_factor) {
        c->queue_factor = queue_factor;                // caller-fixed deep-level capacity: no automatic growth
        cudaSetDevice(c->device);
        cudaDeviceSynchronize();
        free_frame(c);
    }
    return 0;
}

int wrt_enable_kernel_timing(WrtContext* c, int on) {
    if (!c) return fail("wrt_enable_kernel_timing: null context");
    c->kernel_timing = on != 0;
    return 0;
}

// ---------------- batch queries ----------------

static int batch_common(WrtContext* c, int64_t n) {
    if (!c) return fail("null context");
    if (!c->has_scene) return fail("no scene uploaded");
    if (n < 0) return fail("negative count");
    CK(cudaSetDevice(c->device));
    return 0;
}

int wrt_trace_closest(WrtContext* c, const float* orig, const float* dir, int64_t n, WrtHit* hits) {
    if (batch_common(c, n)) return 1;
    if (n == 0) return 0;
    cudaStream_t st = c->chain;
    size_t vb = (size_t)n * 3 * sizeof(float);
    if (ensure_scratch(c, 0, vb) || ensure_scratch(c, 1, vb) || ensure_scratch(c, 2, (size_t)n * sizeof(WrtHit))) return 1;
    CK(cudaMemcpyAsync(c->d_scratch[0], orig, vb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_scratch[1], dir, vb, cudaMemcpyHostToDevice, st));
    int grid = (int)std::min<int64_t>((n + 127) / 128, grid_for(c, 8));
    ++c->launches;
    wrt::k_batch_closest<<<grid, 128, stack_bytes(c, 128), st>>>(c->ds, (const float*)c->d_scratch[0],
                                                                  (const float*)c->d_scratch[1], n,
                                                                  (WrtHit*)c->d_scratch[2], prune_value(c));
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(hits, c->d_scratch[2], (size_t)n * sizeof(WrtHit), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// The same query through the frame's own deep-level closest-hit kernel: the rays are written into ray-tree level 1's arrays
// (all in its first half) and traced by k_trace_closest<false> exactly as a frame traces its secondary rays.
int wrt_trace_closest_wavefront(WrtContext* c, const float* orig, const float* dir, int64_t n, WrtHit* hits) {
    if (batch_common(c, n)) return 1;
    if (n == 0) return 0;
    if (c->frame_pending && finish_frame(c)) return 1;
    cudaStream_t st = c->chain;
    if (ensure_frame_buffers(c, std::max(c->batch_slots, 1u << 20))) return 1;
    wrt::FrameBuffers& fb = c->fb;
    const int64_t chunk = fb.capd / 2;
    size_t vb = (size_t)n * 3 * sizeof(float);
    if (ensure_scratch(c, 0, vb) || ensure_scratch(c, 1, vb) || ensure_scratch(c, 2, (size_t)n * sizeof(WrtHit))) return 1;
    CK(cudaMemcpyAsync(c->d_scratch[0], orig, vb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_scratch[1], dir, vb, cudaMemcpyHostToDevice, st));
    wrt::PrimaryGen pg;
    memset(&pg, 0, sizeof pg);
    const int level = 1;
    for (int64_t off = 0; off < n; off += chunk) {
        const unsigned m = (unsigned)std::min<int64_t>(chunk, n - off);
        const float* o = (const float*)c->d_scratch[0] + 3 * off;
        const float* d = (const float*)c->d_scratch[1] + 3 * off;
        CK(cudaMemsetAsync(fb.counters, 0, wrt::C_TOTAL * sizeof(unsigned), st));
        c->launches += 3;
        wrt::k_pack_rays<<<grid_for(c, 4), 256, 0, st>>>(o, d, m, fb.ray_o[level & 1], fb.ray_d[level & 1], fb.counters, level);
        wrt::k_trace_closest<false><<<grid_for(c, c->trace_blocks_per_sm), 128, stack_bytes(c, 128), st>>>(
            c->ds, fb, pg, level, 0u, wrt::C_WORK, prune_value(c), c->refill | (c->chunk_div << 8));
        wrt::k_unpack_hits<<<grid_for(c, 4), 256, 0, st>>>(c->ds, o, d, m, fb.hit, (WrtHit*)c->d_scratch[2] + off);
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(hits, c->d_scratch[2], (size_t)n * sizeof(WrtHit), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

static int batch_shadow(WrtContext* c, const float* pos, const float* ndir, const float* lightpos, int64_t n,
                        float* coeff, int mode) {
    if (batch_common(c, n)) return 1;
    if (n == 0) return 0;
    cudaStream_t st = c->chain;
    size_t vb = (size_t)n * 3 * sizeof(float);
    for (int k = 0; k < 3; k++) if (ensure_scratch(c, k, std::max(vb, c->scratch_bytes[k]))) return 1;
    if (ensure_scratch(c, 3, (size_t)n * sizeof(float))) return 1;
    CK(cudaMemcpyAsync(c->d_scratch[0], pos, vb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_scratch[1], ndir, vb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_scratch[2], lightpos, vb, cudaMemcpyHostToDevice, st));
    int grid = (int)std::min<int64_t>((n + 127) / 128, grid_for(c, 8));
    ++c->launches;
    wrt::k_batch_shadow<<<grid, 128, stack_bytes(c, 128), st>>>(c->ds, (const float*)c->d_scratch[0],
                                                                 (const float*)c->d_scratch[1],
                                                                 (const float*)c->d_scratch[2], n,
                                                                 (float*)c->d_scratch[3], mode, prune_value(c));
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(coeff, c->d_scratch[3], (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

int wrt_shadow_hard(WrtContext* c, const float* pos, const float* ndir, const float* lightpos, int64_t n, float* coeff) {
    return batch_shadow(c, pos, ndir, lightpos, n, coeff, 0);
}

int wrt_shadow_soft(WrtContext* c, const float* pos, const float* ndir, const float* lightpos, int64_t n, float* coeff) {
    return batch_shadow(c, pos, ndir, lightpos, n, coeff, 1);
}

int wrt_shadow_directional(WrtContext* c, const float* pos, const int32_t* self_object, const float* lightdir4,
                           int64_t n, float* coeff) {
    if (batch_common(c, n)) return 1;
    if (n == 0) return 0;
    cudaStream_t st = c->chain;
    if (ensure_scratch(c, 0, (size_t)n * 12) || ensure_scratch(c, 1, (size_t)n * 4) ||
        ensure_scratch(c, 2, (size_t)n * 16) || ensure_scratch(c, 3, (size_t)n * 4))
        return 1;
    CK(cudaMemcpyAsync(c->d_scratch[0], pos, (size_t)n * 12, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_scratch[1], self_object, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->d_scratch[2], lightdir4, (size_t)n * 16, cudaMemcpyHostToDevice, st));
    int grid = (int)std::min<int64_t>((n + 127) / 128, grid_for(c, 8));
    ++c->launches;
    wrt::k_batch_shadow_directional<<<grid, 128, stack_bytes(c, 128), st>>>(
        c->ds, (const float*)c->d_scratch[0], (const int*)c->d_scratch[1], (const float*)c->d_scratch[2], n,
        (float*)c->d_scratch[3], c->traversal == WRT_TRAVERSAL_EXHAUSTIVE ? 1 : 0);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(coeff, c->d_scratch[3], (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// Shadow requests answered by the frame's own shadow kernels: queued into request queue `queue` in input order, exactly as
// k_surface_spawn queues them (one ray-tree node per request), and run by enqueue_shadows on the stream and grid a frame
// uses for that queue.  The result is what the frame stores for the (node, light) pair.
int wrt_shadow_requests_wavefront(WrtContext* c, int queue, int flags, const float* pos, const float* ndir, const int32_t* light,
                                  const uint32_t* pixel, const uint32_t* path, const int32_t* self_object, int64_t n, float* coeff) {
    if (batch_common(c, n)) return 1;
    if (queue < 0 || queue >= WRT_QUEUES) return fail("wrt_shadow_requests_wavefront: queue out of range");
    if (n == 0) return 0;
    if (!pos || !ndir || !light || !pixel || !path || !self_object || !coeff) return fail("wrt_shadow_requests_wavefront: null argument");
    std::vector<wrt::ShadowRequestIn> req((size_t)n);
    for (int64_t i = 0; i < n; i++) {
        if (light[i] < 0 || light[i] >= c->ds.n_lights) return fail("wrt_shadow_requests_wavefront: light index out of range");
        wrt::ShadowRequestIn& r = req[i];
        for (int k = 0; k < 3; k++) { r.pos[k] = pos[3 * i + k]; r.ndir[k] = ndir[3 * i + k]; }
        r.light = light[i]; r.pixel = pixel[i]; r.path = path[i]; r.self_object = self_object[i];
        r.slot = -1; r.pad = 0;
    }
    if (c->frame_pending && finish_frame(c)) return 1;
    if (ensure_frame_buffers(c, std::max(c->batch_slots, 1u << 20))) return 1;
    wrt::FrameBuffers& fb = c->fb;
    // the frame's streams: queues 0 and 1 on the side stream (when the frame overlaps them), queue 2 on the chain
    const bool overlap = c->overlap && (!c->kernel_timing || getenv("WRT_TIMING_OVERLAP") != nullptr);
    cudaStream_t st = queue < 2 && overlap ? c->side : c->chain;
    const size_t in_bytes = (size_t)n * sizeof(wrt::ShadowRequestIn);
    if (ensure_scratch(c, 0, in_bytes) || ensure_scratch(c, 1, (size_t)n) || ensure_scratch(c, 2, (size_t)n * sizeof(float))) return 1;
    wrt::ShadowRequestIn* d_in = (wrt::ShadowRequestIn*)c->d_scratch[0];
    unsigned char* d_kind = (unsigned char*)c->d_scratch[1];
    float* d_out = (float*)c->d_scratch[2];
    if (c->kernel_timing) {
        c->timed.clear();
        c->event_next = 0;
        CK(cudaEventRecord(c->ev_begin, st));
    }
    // point or directional light, and the spawn-time shaft test; the host then assigns the queue slots in input order
    CK(cudaMemcpyAsync(d_in, req.data(), in_bytes, cudaMemcpyHostToDevice, st));
    ++c->launches;
    wrt::k_classify_shadow_requests<<<(int)std::min<int64_t>((n + 127) / 128, grid_for(c, 8)), 128, 0, st>>>(
        c->ds, d_in, n, (flags & WRT_REQ_SHAFT_CULL) ? 1 : 0, d_kind);
    CK(cudaGetLastError());
    std::vector<unsigned char> kind((size_t)n);
    CK(cudaMemcpyAsync(kind.data(), d_kind, (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    // one node per request: a chunk fits the queue, the nodes, and the list kernels' 32-bit ray index (nreq * 50 < 2^32)
    const int64_t chunk = (int64_t)std::min<unsigned long long>(
        {(unsigned long long)fb.preq_cap[queue], (unsigned long long)fb.dreq_cap[queue], (unsigned long long)fb.n_node_cap,
         ((1ull << 32) - 1) / WRT_SOFT_SAMPLES});
    std::vector<std::pair<unsigned, unsigned>> counts;
    for (int64_t off = 0; off < n; off += chunk) {
        unsigned np = 0, nd = 0;
        for (int64_t i = off; i < std::min(n, off + chunk); i++)
            req[i].slot = kind[i] == 0 ? (int)nd++ : (kind[i] == 1 ? (int)np++ : -1);
        counts.push_back({np, nd});
    }
    CK(cudaMemcpyAsync(d_in, req.data(), in_bytes, cudaMemcpyHostToDevice, st));
    for (int64_t off = 0, k = 0; off < n; off += chunk, k++) {
        const unsigned m = (unsigned)std::min<int64_t>(chunk, n - off);
        CK(cudaMemsetAsync(fb.counters, 0, wrt::C_TOTAL * sizeof(unsigned), st));
        ++c->launches;
        wrt::k_pack_shadow_requests<<<grid_for(c, 4), 256, 0, st>>>(c->ds, fb, queue, d_in + off, m, counts[k].first, counts[k].second);
        int work_seq = 0;
        if (enqueue_shadows(c, st, queue, work_seq)) return 1;
        ++c->launches;
        wrt::k_unpack_shadow_requests<<<grid_for(c, 4), 256, 0, st>>>(c->ds, fb, d_in + off, m, d_out + off);
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(coeff, d_out, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (c->kernel_timing) tally_kernel_times(c);
    return check_debug_bounds();
}

// ---------------- frame ----------------

int wrt_render(WrtContext* c, uint8_t* rgb_host, WrtStats* stats) {
    if (!c || !rgb_host) return fail("wrt_render: null argument");
    CK(cudaSetDevice(c->device));
    if (!c->has_cam) return fail("wrt_render: no camera set");
    size_t bytes = (size_t)c->cam.width * c->cam.height * 3;
    if (bytes == 0) return fail("wrt_render: empty image");
    if (c->d_image_bytes < bytes) {
        if (c->d_image) cudaFree(c->d_image);
        c->d_image = nullptr; c->d_image_bytes = 0;
        CK(cudaMalloc((void**)&c->d_image, bytes));
        c->d_image_bytes = bytes;
    }
    if (c->h_image_bytes < bytes) {
        if (c->h_image) cudaFreeHost(c->h_image);
        c->h_image = nullptr; c->h_image_bytes = 0;
        CK(cudaMallocHost((void**)&c->h_image, bytes));
        c->h_image_bytes = bytes;
    }
    cudaStream_t st = c->chain;
    if (c->world > 1) CK(cudaMemsetAsync(c->d_image, 0, bytes, st));
    if (render_all(c, nullptr, false, c->d_image, nullptr)) return 1;
    if (finish_frame(c)) return 1;
    cudaPointerAttributes attr;
    bool user_pinned = c->world == 1 && cudaPointerGetAttributes(&attr, rgb_host) == cudaSuccess &&
                       attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    if (user_pinned) {                                 // caller's buffer is page-locked: no staging copy
        CK(cudaMemcpyAsync(rgb_host, c->d_image, bytes, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (stats) *stats = c->stats;
        return 0;
    }
    CK(cudaMemcpyAsync(c->h_image, c->d_image, bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (c->world == 1) memcpy(rgb_host, c->h_image, bytes);
    else {
        // only this rank's pixels are defined; copy them, leave the rest of the caller's buffer alone
        wrt::TileMap tm = c->tilemap();
        long long slots = c->local_slots(c->rank, c->world);
        for (long long s = 0; s < slots; s++) {
            int x, y;
            if (tm.slot_to_pixel(s, c->rank, x, y)) {
                size_t o = 3 * ((size_t)y * tm.width + x);
                rgb_host[o] = c->h_image[o]; rgb_host[o + 1] = c->h_image[o + 1]; rgb_host[o + 2] = c->h_image[o + 2];
            }
        }
    }
    if (stats) *stats = c->stats;
    return 0;
}

int wrt_render_float(WrtContext* c, float* rgb_f_host, uint8_t* rgb_host, WrtStats* stats) {
    if (!c || !rgb_f_host || !rgb_host) return fail("wrt_render_float: null argument");
    CK(cudaSetDevice(c->device));
    if (!c->has_cam) return fail("wrt_render_float: no camera set");
    const long long slots = c->local_slots(c->rank, c->world);
    const size_t bytes = (size_t)std::max(slots, 1ll) * sizeof(float4);
    if (c->h_float_bytes < bytes) {
        if (c->h_float) cudaFreeHost(c->h_float);
        c->h_float = nullptr; c->h_float_bytes = 0;
        CK(cudaMallocHost((void**)&c->h_float, bytes));
        c->h_float_bytes = bytes;
    }
    c->copy_float = true;
    const int rc = wrt_render(c, rgb_host, stats);     // synchronous: every batch's copy has landed when it returns
    c->copy_float = false;
    if (rc) return rc;
    wrt::TileMap tm = c->tilemap();
    for (long long s = 0; s < slots; s++) {
        int x, y;
        if (tm.slot_to_pixel(s, c->rank, x, y)) {
            float* p = rgb_f_host + 3 * ((size_t)y * tm.width + x);
            p[0] = c->h_float[s].x; p[1] = c->h_float[s].y; p[2] = c->h_float[s].z;
        }
    }
    return 0;
}

int wrt_render_device(WrtContext* c, void* d_rgb_tiles, void* cuda_stream) {
    if (!c || !d_rgb_tiles) return fail("wrt_render_device: null argument");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;        // NULL = the legacy default stream, as in CUDA
    return render_all(c, st, true, nullptr, (uint8_t*)d_rgb_tiles);
}

int wrt_finish_device(WrtContext* c, WrtStats* stats) {
    if (!c) return fail("wrt_finish_device: null context");
    CK(cudaSetDevice(c->device));
    if (!c->has_frame) return fail("wrt_finish_device: no frame in flight");
    // A frame that overflowed a queue is re-rendered here (synchronously, into the same device buffer): when
    // stats->overflow_retries != 0 the caller must repeat whatever it had already enqueued behind the frame on
    // its own stream (parallel.py: the gather).
    if (finish_frame(c)) return 1;
    if (stats) *stats = c->stats;
    return 0;
}

int wrt_get_stats(WrtContext* c, WrtStats* stats) {
    if (!c || !stats) return fail("wrt_get_stats: null argument");
    *stats = c->stats;
    return 0;
}

int64_t wrt_tile_pixel_count(WrtContext* c, int rank, int world) {
    if (!c || !c->has_cam || world < 1 || rank < 0 || rank >= world) return -1;
    return c->local_slots(rank, world);
}

int wrt_scatter_tiles(WrtContext* c, const void* d_gathered, int world, int64_t stride_bytes, void* d_rgb_image,
                      void* cuda_stream) {
    if (!c || !d_gathered || !d_rgb_image) return fail("wrt_scatter_tiles: null argument");
    if (!c->has_cam) return fail("wrt_scatter_tiles: no camera set");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;        // NULL = the legacy default stream, as in CUDA
    wrt::TileMap tm = c->tilemap();
    tm.world = world;
    long long slots_per_rank = c->local_slots(0, world);   // rank 0 owns the most tiles
    if (stride_bytes < slots_per_rank * 3) return fail("wrt_scatter_tiles: stride smaller than rank 0's tile buffer");
    ++c->launches;
    wrt::k_scatter_tiles<<<grid_for(c, 8), 256, 0, st>>>((const unsigned char*)d_gathered, stride_bytes, tm, world,
                                                         slots_per_rank, (unsigned char*)d_rgb_image);
    CK(cudaGetLastError());
    return 0;
}

int64_t wrt_kernel_launch_count(WrtContext* c) { return c ? c->launches : 0; }

int wrt_measure_fp32_peak(WrtContext* c, float* tflops_fma, float* tflops_mul_add) {
    if (!c || !tflops_fma || !tflops_mul_add) return fail("wrt_measure_fp32_peak: null argument");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = c->chain;
    if (ensure_scratch(c, 4, 256)) return 1;
    const int iters = 1 << 15, blocks = c->num_sms * 8, threads = 256;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    float best[2] = {0.f, 0.f};
    for (int mode = 0; mode < 2; mode++) {
        for (int rep = 0; rep < 4; rep++) {
            CK(cudaEventRecord(e0, st));
            wrt::k_fp32_peak<<<blocks, threads, 0, st>>>((float*)c->d_scratch[4], iters, mode);
            CK(cudaEventRecord(e1, st));
            CK(cudaStreamSynchronize(st));
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, e0, e1));
            double flops = (double)blocks * threads * (double)iters * 8.0 * 2.0;
            float tf = (float)(flops / (ms * 1e-3) / 1e12);
            if (rep > 0 && tf > best[mode]) best[mode] = tf;
        }
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tflops_fma = best[0];
    *tflops_mul_add = best[1];
    return 0;
}

int wrt_get_kernel_times(WrtContext* c, float* ms, int capacity) {
    if (!c || !ms) return 0;
    int n = std::min(capacity, (int)WRT_KERNEL_FAMILIES);
    for (int i = 0; i < n; i++) ms[i] = c->family_ms[i];
    return n;
}

int wrt_get_kernel_launches(WrtContext* c, int32_t* launches, int capacity) {
    if (!c || !launches) return 0;
    int n = std::min(capacity, (int)WRT_KERNEL_FAMILIES);
    for (int i = 0; i < n; i++) launches[i] = c->family_launches[i];
    return n;
}


// ======================= multi-GPU in one process (SURVEY.md section 8b / 5.8) =======================
// wrt_multi_*: the scene replicated on n GPUs, the image sharded as interleaved tiles (include/wrt_tiles.h), one host
// thread per GPU driving an ordinary WrtContext.  There is no gather step: with peer access every GPU's resolve kernel
// stores its 8-bit pixels straight into device 0's row-major frame over NVLink (k_combine_resolve's `image` pointer is a
// peer pointer), so the exchange overlaps the last kernel of each GPU and rank 0 only copies the finished frame to the
// host.  Without peer access (never the case on an NVSwitch box) the ranks' tile buffers are copied to device 0 and
// de-interleaved there by k_scatter_tiles.

} // extern "C"

struct WrtMulti {
    std::vector<WrtContext*> ctx;
    std::vector<int> devices;
    bool peer_stores = true;
    uint8_t* d_gathered = nullptr;       // fallback path only (on device 0)
    size_t gathered_bytes = 0;
    std::vector<uint8_t*> d_packed;      // fallback path only (per device)
    std::vector<size_t> packed_bytes;
    std::vector<std::string> errors;
    // one persistent host thread per GPU 1..n-1 (GPU 0 is driven by the caller's thread): a frame is a few milliseconds,
    // thread creation per call would show
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_go, cv_done;
    std::function<int(int)> job;
    std::vector<int> rc;
    uint64_t generation = 0;
    int pending = 0;
    bool quit = false;
};

namespace {

void multi_worker(WrtMulti* m, int r) {
    uint64_t seen = 0;
    while (true) {
        std::function<int(int)> job;
        {
            std::unique_lock<std::mutex> lk(m->mu);
            m->cv_go.wait(lk, [&] { return m->quit || m->generation != seen; });
            if (m->quit) return;
            seen = m->generation;
            job = m->job;
        }
        const int rc = job(r);
        {
            std::lock_guard<std::mutex> lk(m->mu);
            m->rc[r] = rc;
            if (rc) m->errors[r] = g_err;               // g_err is thread_local
            if (--m->pending == 0) m->cv_done.notify_one();
        }
    }
}

// Runs fn(rank) for every GPU (rank 0 on the caller's thread) and collects the error strings.
int multi_run(WrtMulti* m, std::function<int(int)> fn) {
    const int n = (int)m->ctx.size();
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->rc.assign(n, 0);
        m->errors.assign(n, std::string());
        m->job = fn;
        m->pending = n - 1;
        ++m->generation;
    }
    m->cv_go.notify_all();
    const int rc0 = fn(0);
    {
        std::unique_lock<std::mutex> lk(m->mu);
        m->cv_done.wait(lk, [&] { return m->pending == 0; });
        m->rc[0] = rc0;
        if (rc0) m->errors[0] = g_err;
    }
    for (int r = 0; r < n; r++)
        if (m->rc[r]) return fail("GPU " + std::to_string(m->devices[r]) + ": " + m->errors[r]);
    return 0;
}

} // namespace

extern "C" {

int wrt_multi_create(const int* devices, int n, WrtMulti** out) {
    if (!out) return fail("wrt_multi_create: null out pointer");
    *out = nullptr;
    if (!devices || n < 1) return fail("wrt_multi_create: need at least one device");
    for (int i = 0; i < n; i++)
        for (int j = 0; j < i; j++)
            if (devices[i] == devices[j]) return fail("wrt_multi_create: device listed twice");
    WrtMulti* m = new WrtMulti();
    m->devices.assign(devices, devices + n);
    m->ctx.assign(n, nullptr);
    m->d_packed.assign(n, nullptr);
    m->packed_bytes.assign(n, 0);
    for (int r = 0; r < n; r++) {
        if (wrt_create(devices[r], &m->ctx[r]) != 0) { wrt_multi_destroy(m); return 1; }
    }
    // every GPU must be able to store into device 0's frame
    for (int r = 1; r < n && m->peer_stores; r++) {
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, devices[r], devices[0]) != cudaSuccess || !can) { m->peer_stores = false; break; }
        cudaSetDevice(devices[r]);
        cudaError_t e = cudaDeviceEnablePeerAccess(devices[0], 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) m->peer_stores = false;
        cudaGetLastError();
    }
    if (getenv("WRT_MULTI_NO_PEER")) m->peer_stores = false;          // tests: force the copy + scatter path
    for (int r = 1; r < n; r++) m->workers.emplace_back(multi_worker, m, r);
    *out = m;
    return 0;
}

void wrt_multi_destroy(WrtMulti* m) {
    if (!m) return;
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->quit = true;
    }
    m->cv_go.notify_all();
    for (std::thread& t : m->workers) t.join();
    for (size_t r = 0; r < m->ctx.size(); r++) {
        if (m->d_packed[r]) { cudaSetDevice(m->devices[r]); cudaFree(m->d_packed[r]); }
        if (m->ctx[r]) wrt_destroy(m->ctx[r]);
    }
    if (m->d_gathered) { cudaSetDevice(m->devices[0]); cudaFree(m->d_gathered); }
    delete m;
}

int wrt_multi_device_count(WrtMulti* m) { return m ? (int)m->ctx.size() : 0; }
WrtContext* wrt_multi_context(WrtMulti* m, int rank) { return (m && rank >= 0 && rank < (int)m->ctx.size()) ? m->ctx[rank] : nullptr; }
int wrt_multi_uses_peer_stores(WrtMulti* m) { return m && m->peer_stores ? 1 : 0; }

int wrt_multi_upload_scene(WrtMulti* m, const WrtSceneDesc* s) {
    if (!m || !s) return fail("wrt_multi_upload_scene: null argument");
    return multi_run(m, [&](int r) { return wrt_upload_scene(m->ctx[r], s); });
}

int wrt_multi_set_camera(WrtMulti* m, const WrtCamera* cam) {
    if (!m || !cam) return fail("wrt_multi_set_camera: null argument");
    for (WrtContext* c : m->ctx) if (wrt_set_camera(c, cam)) return 1;
    return 0;
}

int wrt_multi_set_options(WrtMulti* m, int traversal, uint32_t seed, float queue_factor) {
    if (!m) return fail("wrt_multi_set_options: null argument");
    for (WrtContext* c : m->ctx) if (wrt_set_options(c, traversal, seed, queue_factor)) return 1;
    return 0;
}

int wrt_multi_render(WrtMulti* m, uint8_t* rgb_host, WrtStats* stats) {
    if (!m || !rgb_host) return fail("wrt_multi_render: null argument");
    const int n = (int)m->ctx.size();
    WrtContext* c0 = m->ctx[0];
    if (!c0->has_cam) return fail("wrt_multi_render: no camera set");
    const size_t bytes = (size_t)c0->cam.width * c0->cam.height * 3;
    if (bytes == 0) return fail("wrt_multi_render: empty image");
    CK(cudaSetDevice(c0->device));
    if (c0->d_image_bytes < bytes) {
        CK(cudaDeviceSynchronize());
        if (c0->d_image) cudaFree(c0->d_image);
        c0->d_image = nullptr; c0->d_image_bytes = 0;
        CK(cudaMalloc((void**)&c0->d_image, bytes));
        c0->d_image_bytes = bytes;
    }
    const int tw = c0->tile_w, thh = c0->tile_h;
    for (int r = 0; r < n; r++) if (wrt_set_tiles(m->ctx[r], tw, thh, r, n)) return 1;
    const long long stride = c0->local_slots(0, n) * 3;               // rank 0 owns the most tiles
    if (!m->peer_stores) {
        if (m->gathered_bytes < (size_t)stride * n) {
            if (m->d_gathered) cudaFree(m->d_gathered);
            m->d_gathered = nullptr; m->gathered_bytes = 0;
            CK(cudaMalloc((void**)&m->d_gathered, (size_t)stride * n));
            m->gathered_bytes = (size_t)stride * n;
        }
    }
    uint8_t* d_image0 = c0->d_image;
    int rc = multi_run(m, [&](int r) -> int {
        WrtContext* c = m->ctx[r];
        CK(cudaSetDevice(c->device));
        if (m->peer_stores) {
            if (render_all(c, nullptr, false, d_image0, nullptr)) return 1;      // stores cross NVLink from the resolve kernel
            return finish_frame(c);
        }
        if (m->packed_bytes[r] < (size_t)stride) {
            if (m->d_packed[r]) cudaFree(m->d_packed[r]);
            m->d_packed[r] = nullptr; m->packed_bytes[r] = 0;
            CK(cudaMalloc((void**)&m->d_packed[r], (size_t)stride));
            m->packed_bytes[r] = (size_t)stride;
        }
        if (render_all(c, nullptr, false, nullptr, m->d_packed[r])) return 1;
        if (finish_frame(c)) return 1;
        CK(cudaMemcpyPeerAsync(m->d_gathered + (size_t)r * stride, m->devices[0], m->d_packed[r], c->device, (size_t)stride, c->chain));
        CK(cudaStreamSynchronize(c->chain));
        return 0;
    });
    for (int r = 0; r < n; r++) wrt_set_tiles(m->ctx[r], tw, thh, 0, 1);         // the contexts stay usable on their own
    if (rc) return 1;
    CK(cudaSetDevice(c0->device));
    cudaStream_t st = c0->chain;
    if (!m->peer_stores) {
        wrt_set_tiles(c0, tw, thh, 0, n);
        int src = wrt_scatter_tiles(c0, m->d_gathered, n, stride, c0->d_image, (void*)st);
        wrt_set_tiles(c0, tw, thh, 0, 1);
        if (src) return 1;
    }
    cudaPointerAttributes attr;
    const bool user_pinned = cudaPointerGetAttributes(&attr, rgb_host) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    if (user_pinned) {
        CK(cudaMemcpyAsync(rgb_host, c0->d_image, bytes, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    } else {
        if (c0->h_image_bytes < bytes) {
            if (c0->h_image) cudaFreeHost(c0->h_image);
            c0->h_image = nullptr; c0->h_image_bytes = 0;
            CK(cudaMallocHost((void**)&c0->h_image, bytes));
            c0->h_image_bytes = bytes;
        }
        CK(cudaMemcpyAsync(c0->h_image, c0->d_image, bytes, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        memcpy(rgb_host, c0->h_image, bytes);
    }
    if (stats) {
        WrtStats t{};
        for (int r = 0; r < n; r++) {
            const WrtStats& a = m->ctx[r]->stats;
            t.closest_rays += a.closest_rays; t.shadow_rays += a.shadow_rays; t.shadow_requests += a.shadow_requests;
            for (int d = 0; d < WRT_MAX_DEPTH; d++) t.rays_per_depth[d] += a.rays_per_depth[d];
            t.overflow_retries += a.overflow_retries;
            t.gpu_ms = std::max(t.gpu_ms, a.gpu_ms);                   // the frame takes as long as its slowest GPU
            t.shaft_culled_requests += a.shaft_culled_requests; t.unlit_skipped_requests += a.unlit_skipped_requests;
            t.shadow_rays_traced += a.shadow_rays_traced;
        }
        *stats = t;
    }
    return 0;
}

} // extern "C"
