/* wrt_cuda.h — C ABI of the sm_100a render core (libwrt_cuda.so).
 *
 * Drop-in boundary for the reference's render hot path.  Each entry point
 * names the reference interface it replaces (paths relative to /root/reference):
 *
 *   wrt_trace_closest      <- IIntersectStrategy::UpdateInter         include/IIntersectStrategy.h:10-11
 *                             (BVHStrategy::UpdateInter -> getIntersection, include/BVHStrategy.hpp:8-11, include/BVH.hpp:137-159)
 *   wrt_shadow_hard        <- IIntersectStrategy::getShadowCoeffi     include/IIntersectStrategy.h:14
 *                             (BVHStrategy::getShadowCoeffi/ShadowHelper, include/BVHStrategy.hpp:13-48)
 *   wrt_shadow_soft        <- Renderer::getShadowCoeffi(Intersection&, Vector3f&) with EXPEDITE
 *                             (include/Renderer.hpp:347-376 -> hasIntersection, include/BVH.hpp:162-186);
 *                             this query bypasses the strategy interface in the reference
 *   wrt_shadow_directional <- Renderer::getShadowCoeffi(Intersection&, Vector4f&)   include/Renderer.hpp:381-400
 *   wrt_render*            <- Renderer::render()                      include/Renderer.hpp:57-137
 *                             (traceRay :151-260, blinnPhongShader :265-341, getAreaLightShadowCoeffi :405-414,
 *                              changeNormalDir :417-474), output = PPMGenerator::rgb as 8-bit
 *   wrt_upload_scene       <- the Scene& / PPMGenerator* the Renderer reads (include/Renderer.hpp:38-49)
 *   wrt_set_camera         <- camera locals of Renderer::render       include/Renderer.hpp:65-100
 *
 * Conventions: plain C, opaque handle, every call returns 0 on success and a
 * non-zero code on failure with wrt_last_error() describing it.  Host buffers
 * stay owned by the caller; the library copies during upload.  There is no CPU
 * fallback: without a CUDA device wrt_create() fails.
 * Not thread-safe per context; use one context per GPU / per host thread.
 */
#ifndef WRT_CUDA_H
#define WRT_CUDA_H

#include "wrt_scene.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct WrtContext WrtContext;

#define WRT_TRAVERSAL_EXHAUSTIVE 0  /* visit every node whose box is hit, like BVH.hpp:137-159; every shadow ray the
                                     * reference traces is traced */
#define WRT_TRAVERSAL_PRUNED     1  /* near-first order, skip boxes entered beyond the best hit; shadow requests that
                                     * provably cannot change the image are answered without tracing and soft-shadow
                                     * rays test per-request candidate lists (DESIGN.md section 4b).  Same result. */

/* Development switches read from the environment by wrt_create() (all default to "on"; results are identical
 * either way, the GPU tests compare them): WRT_UNLIT_CULL=0 (queue shadow requests of lights whose Blinn-Phong
 * factors are exactly 0), WRT_SHAFT_CULL=0 (trace soft-shadow requests whose shaft to the light is empty),
 * WRT_SOFT_LISTS=0 (per-ray soft-shadow kernel instead of the candidate-list kernels).
 * Test hooks: WRT_MAX_BATCH=n (primary slots per batch: forces multi-batch frames), WRT_DEEP_FACTOR=f (initial
 * automatic deep-level capacity), WRT_LIST_POOL_CAP=n (candidate-list pool entries). */

int  wrt_create(int device, WrtContext** out);
void wrt_destroy(WrtContext* ctx);
const char* wrt_last_error(void);

/* Uploads the scene and builds the walked tree on the device (PLOC).  The traversal stack holds 90 rows:
 * max(reference tree depth, walked depth, 3 * ceil(walked depth / 2)) + 2 <= 90, i.e. the caller's (reference) tree
 * may be 88 levels deep and the walked tree 58.  When PLOC's tree is deeper (fans of triangles sharing a vertex,
 * slivers, boxes of very mixed sizes), the walked tree is rebuilt with the host's binned SAH instead; the scene is
 * refused only if that tree or the reference's does not fit either.  Results do not depend on which tree is walked.
 * Hard-shadow coefficients are the reference's bit for bit up to 12 translucent blockers on one ray; beyond, the
 * product is taken in visit order (within a few ulp: the tests allow k ulp for k blockers).  WRT_VERBOSE=1 prints
 * the builder used and the stack rows. */
int wrt_upload_scene(WrtContext* ctx, const WrtSceneDesc* scene);
int wrt_set_camera(WrtContext* ctx, const WrtCamera* cam);

/* Image sharding: the image is cut into tile_w x tile_h tiles (multiples of 8 x 4),
 * tiles are dealt to the ranks through the permuted interleave of wrt_tiles.h.
 * Default: 8 x 4 (one warp-sized pixel block per tile: ray counts balance within 1 %
 * over 8 ranks on the bunny scenes), rank 0 of 1. */
int wrt_set_tiles(WrtContext* ctx, int tile_w, int tile_h, int rank, int world);

/* traversal: WRT_TRAVERSAL_*; seed: soft-shadow RNG seed (include/wrt_rng.h);
 * queue_factor: capacity of each secondary-ray level as a multiple of the primary
 * level.  <= 0 keeps the automatic sizing: a quarter of the primary level (a full
 * level for frames under 1 M pixels), doubled — and kept — whenever a level
 * overflows.  > 0 fixes it; an overflowing batch is then re-rendered in halves.
 * Either way overflow is detected and the batch redone, never dropped. */
int wrt_set_options(WrtContext* ctx, int traversal, uint32_t seed, float queue_factor);

/* Brackets every kernel launch of wrt_render* with CUDA events on the launching
 * stream so that wrt_get_kernel_times() can report per-family device time. */
int wrt_enable_kernel_timing(WrtContext* ctx, int on);

/* ---- batch forms of the strategy queries (host pointers, synchronous) ---- */
int wrt_trace_closest(WrtContext* ctx, const float* orig, const float* dir, int64_t n, WrtHit* hits);
/* The same query (same arguments, same results bit for bit) answered by the kernel a frame traces its secondary rays with:
 * the rays are written into ray-tree level 1 and traced by the wavefront closest-hit kernel (octant copies, 4-wide nodes,
 * deferred leaves, per-lane refill).  wrt_trace_closest walks the plain binary tree one ray per thread; this entry exists
 * so that the parity tests can hold the frame kernel itself to the oracle on arbitrary ray batches
 * (IIntersectStrategy::UpdateInter, include/IIntersectStrategy.h:10-11). */
int wrt_trace_closest_wavefront(WrtContext* ctx, const float* orig, const float* dir, int64_t n, WrtHit* hits);
/* Shadow requests answered by the kernels a frame answers its own with (k_shadow_hard; k_soft_lists -> k_soft_filter ->
 * k_soft_list_rays, or k_shadow_soft; k_shadow_directional), for the parity tests.  Request i is the shading point pos[i]
 * with normal ndir[i] and scene light light[i]; pixel[i] and path[i] (a ray-tree path id >= 1) key the soft-shadow RNG,
 * self_object[i] is the object a directional-light request's point lies on.  The requests are queued in input order into
 * request queue `queue` (0: level 0, 1: levels 1..5, 2: deeper) exactly as the frame's surface stage queues them and run on
 * that queue's stream and grid.  With WRT_REQ_SHAFT_CULL, soft requests whose shaft to the light is empty are answered by
 * the surface stage's shaft test instead, as on level 0.  coeff[i] is what the frame stores: the hard-shadow or
 * directional product, or the number of lit samples of 50 (as a float).  Kernel timing, when on, covers these launches. */
#define WRT_REQ_SHAFT_CULL 1
int wrt_shadow_requests_wavefront(WrtContext* ctx, int queue, int flags, const float* pos, const float* ndir, const int32_t* light,
                                  const uint32_t* pixel, const uint32_t* path, const int32_t* self_object, int64_t n, float* coeff);
/* BVHStrategy::getShadowCoeffi / ShadowHelper (include/BVHStrategy.hpp:13-48): the product of (1 - alpha) over the blocking
 * leaves, multiplied in the association of the caller's tree (`l * r` at every inner node) — the reference's float bit
 * for bit, whichever tree the kernel walks (csrc/cuda/shadow_assoc.h; beyond 12 translucent crossings on one ray or a
 * tree deeper than 64 levels: the same factors in visit order).  The frame's kernel is held to the same bar, request by
 * request, through wrt_shadow_requests_wavefront (tests/test_gpu_shadow_requests.py). */
int wrt_shadow_hard(WrtContext* ctx, const float* pos, const float* ndir, const float* lightpos, int64_t n, float* coeff);
int wrt_shadow_soft(WrtContext* ctx, const float* pos, const float* ndir, const float* lightpos, int64_t n, float* coeff);
int wrt_shadow_directional(WrtContext* ctx, const float* pos, const int32_t* self_object, const float* lightdir4,
                           int64_t n, float* coeff);

/* ---- frame ---- */
/* Renders this rank's tiles and copies the 8-bit image (width*height*3, row-major,
 * pixels of other ranks' tiles left untouched) to host memory.  Synchronous. */
int wrt_render(WrtContext* ctx, uint8_t* rgb_host, WrtStats* stats);

/* The frame wrt_render renders, and also its unquantised colour: rgb_f_host (width*height*3 float, row-major) receives
 * the level-0 colour k_combine_resolve quantises (Renderer.hpp:259, before `255 * min(c, 1)`); pixels of other ranks'
 * tiles are left untouched in both buffers.  After each batch's combine one device-to-host copy of the batch's level-0
 * nodes is queued on the frame's stream (a batch re-rendered after a queue overflow copies again, over its first
 * attempt); wrt_render and wrt_render_device queue no such copy.  Synchronous. */
int wrt_render_float(WrtContext* ctx, float* rgb_f_host, uint8_t* rgb_host, WrtStats* stats);

/* Asynchronous form on caller-provided device memory and stream (cudaStream_t as void*;
 * NULL is CUDA's legacy default stream, e.g. torch's default current stream).  d_rgb_tiles receives this rank's pixels in tile
 * order: wrt_tile_pixel_count(ctx, rank, world) * 3 bytes.  Call wrt_finish_device()
 * before reading statistics. */
int wrt_render_device(WrtContext* ctx, void* d_rgb_tiles, void* cuda_stream);
/* Waits for the frame.  A frame that overflowed a ray queue is re-rendered inside this call
 * (synchronously, into the same d_rgb_tiles); stats->overflow_retries != 0 then tells the caller
 * to repeat whatever it had already enqueued behind the frame on its stream (e.g. the gather). */
int wrt_finish_device(WrtContext* ctx, WrtStats* stats);
int wrt_get_stats(WrtContext* ctx, WrtStats* stats);

/* Pixel slots (tile area, including clipped padding) rank `rank` of `world` owns. */
int64_t wrt_tile_pixel_count(WrtContext* ctx, int rank, int world);

/* Rank-0 side of the NCCL gather: d_gathered holds `world` buffers of `stride_bytes`
 * each (rank r's tile-order pixels at r*stride_bytes); writes the row-major
 * width*height*3 image to d_rgb_image. */
int wrt_scatter_tiles(WrtContext* ctx, const void* d_gathered, int world, int64_t stride_bytes,
                      void* d_rgb_image, void* cuda_stream);

/* Kernels launched by this context since creation (bench.py's gpu_launches). */
int64_t wrt_kernel_launch_count(WrtContext* ctx);

/* FP32 SIMT issue-rate microbenchmark on this GPU: TFLOP/s of dependent-chain FFMA
 * (2 flops/instruction) and of the separate FMUL+FADD form this library's
 * -fmad=false kernels issue (1 flop/instruction).  Roofline denominators. */
int wrt_measure_fp32_peak(WrtContext* ctx, float* tflops_fma, float* tflops_mul_add);

/* Per-kernel-family device milliseconds of the last wrt_render* call (CUDA events
 * on the launching stream).  Order: raygen, trace_closest, surface, shadow_hard,
 * shadow_soft (the soft-shadow ray kernels), shadow_directional, shade, combine, resolve,
 * soft_lists (candidate-list build of the soft-shadow path), soft_filter (triangle-level pruning of
 * those lists).  Returns the number of entries written. */
#define WRT_KERNEL_FAMILIES 11
int wrt_get_kernel_times(WrtContext* ctx, float* ms, int capacity);
/* Launches per family behind those times (same order). */
int wrt_get_kernel_launches(WrtContext* ctx, int32_t* launches, int capacity);

/* ---- multi-GPU in one process: `Renderer::render()` over n GPUs (what `wrt --gpus n` uses) ----
 * The scene is replicated, the image is sharded as interleaved tiles (wrt_tiles.h), one host thread drives each GPU.
 * With peer access (NVLink / NVSwitch) there is no gather step: every GPU's resolve kernel stores its 8-bit pixels
 * straight into device devices[0]'s frame, which is then copied to rgb_host.  The image is identical to the 1-GPU
 * image (every pixel is independent; the soft-shadow RNG is keyed on the global pixel). */
typedef struct WrtMulti WrtMulti;
int  wrt_multi_create(const int* devices, int n, WrtMulti** out);
void wrt_multi_destroy(WrtMulti* m);
int  wrt_multi_device_count(WrtMulti* m);
WrtContext* wrt_multi_context(WrtMulti* m, int rank);      /* rank's own context (options, timing, batch queries) */
int  wrt_multi_uses_peer_stores(WrtMulti* m);              /* 1: pixels cross NVLink from the resolve kernels; 0: copy + scatter */
int  wrt_multi_upload_scene(WrtMulti* m, const WrtSceneDesc* scene);
int  wrt_multi_set_camera(WrtMulti* m, const WrtCamera* cam);
int  wrt_multi_set_options(WrtMulti* m, int traversal, uint32_t seed, float queue_factor);
int  wrt_multi_render(WrtMulti* m, uint8_t* rgb_host, WrtStats* stats);   /* stats: sums over the GPUs, gpu_ms = slowest GPU */

#ifdef __cplusplus
}
#endif
#endif /* WRT_CUDA_H */
