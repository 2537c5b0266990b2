/* crt.h — C-ABI of the B200-native path tracer (libcrt.so).
 *
 * The reference (guomc9/CudaRayTracing) has no FFI; its de-facto surface is three C++ classes
 * called from src/main.cu. Each entry point below replaces one of those call sites (cited as
 * file:line relative to the reference checkout). Conventions:
 *   - every function returns 0 (CRT_OK) or a negative crt_status; the message of the last error on
 *     the calling thread is available from crt_last_error();
 *   - handles own all host and device memory; inputs are copied at the call, outputs are written
 *     into caller-allocated buffers; nothing throws, nothing calls exit();
 *   - a handle is not thread-safe; distinct handles are independent;
 *   - there is no CPU fallback: a call that needs the GPU fails with CRT_ERR_CUDA when there is none.
 */
#ifndef CRT_H_
#define CRT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRT_ABI_VERSION 2

typedef enum crt_status {
    CRT_OK = 0,
    CRT_ERR_INVALID = -1,   /* bad argument or handle state */
    CRT_ERR_IO = -2,        /* file missing / unreadable / malformed */
    CRT_ERR_CUDA = -3,      /* CUDA runtime error (message has the cudaError string) */
    CRT_ERR_NOMEM = -4,
    CRT_ERR_STATE = -5      /* call order violated (e.g. render before build_bvh) */
} crt_status;

typedef struct crt_scene crt_scene;     /* Scene (include/Scene.h:16-101) + BVH + device copies */
typedef struct crt_render crt_render;   /* Render (include/Render.cuh:357-557) */

/* Material as the MTL states it (include/OBJLoader.h:159-200). ks is kept for the `mis`
 * estimator; the `compat` estimator ignores it like the reference does (include/Loader.h:45-47). */
typedef struct crt_material {
    float kd[3];
    float ks[3];
    float ke[3];
    float ns;
} crt_material;

/* config.json (src/main.cu:40-90, scenes/<name>/config.json). Extra optional keys: "seed", "estimator". */
#define CRT_MAX_OBJ_PATHS 16
#define CRT_PATH_LEN 1024
typedef struct crt_config {
    uint32_t n_obj;
    char obj_path[CRT_MAX_OBJ_PATHS][CRT_PATH_LEN];
    char mtl_dir[CRT_MAX_OBJ_PATHS][CRT_PATH_LEN];
    float eye_pos[3], lookat[3], up[3];
    float fov_y;             /* degrees, as in the file */
    uint32_t width, height;
    uint32_t bvh_thresh_n;
    float p_rr;
    uint32_t spp;
    uint32_t light_sample_n;
    uint32_t seed;           /* optional key, default 0 */
    uint32_t estimator;      /* optional key "estimator": "compat" (0, default) | "mis" (1) */
} crt_config;

typedef enum crt_estimator { CRT_ESTIMATOR_COMPAT = 0, CRT_ESTIMATOR_MIS = 1 } crt_estimator;
/* CRT_BUILDER_LBVH: Morton-sorted binary radix tree emitted as 64-byte child-pair nodes (crt_bvh_node).
 * CRT_BUILDER_LBVH8: the same radix tree collapsed into 80-byte 8-wide nodes with 8-bit quantised child
 * boxes (crt_bvh8_node); bvh_thresh_n is clamped to 15. Hits and images do not depend on the builder. */
/* Bit 1 selects the tree topology: CRT_BUILDER_PLOC / CRT_BUILDER_PLOC8 agglomerate the Morton-ordered triangles
 * bottom-up by union-box area (parallel locally-ordered clustering, search radius 8) instead of splitting by key
 * prefix; the tree costs a few more build kernels and needs about a third fewer node visits per ray
 * (DESIGN.md "BVH build"). Node layouts, leaf rule and exports are those of LBVH / LBVH8. */
typedef enum crt_builder { CRT_BUILDER_LBVH = 0, CRT_BUILDER_LBVH8 = 1, CRT_BUILDER_PLOC = 2, CRT_BUILDER_PLOC8 = 3 } crt_builder;
typedef enum crt_ray_mode { CRT_RAY_CLOSEST = 0, CRT_RAY_ANY = 1 } crt_ray_mode;
/* Flag to OR into a ray mode: trace the batch (each chunk of a host-buffer batch) in the order of (Morton code of the origin's cell
 * on a 128^3 grid over the scene, direction octant) - "warp-coherent ray sorting" - and write the hits back in the caller's order. The
 * results are the same; on this hardware the order buys less than the sort costs (profiles/r02_late_levers.md), so it is off unless asked for. */
#define CRT_RAY_SORTED 0x100

/* 64-byte BVH node as exported by crt_scene_export_bvh (DESIGN.md "Layout"). */
typedef struct crt_bvh_node {
    float c0lox, c0hix, c0loy, c0hiy;
    float c1lox, c1hix, c1loy, c1hiy;
    float c0loz, c0hiz, c1loz, c1hiz;
    int32_t c0, c1;          /* >= 0 node index, < 0 leaf = ~first_slot, 0x7fffffff = absent */
    int32_t n0, n1;          /* triangles below each child */
} crt_bvh_node;

/* 80-byte 8-wide node as exported by crt_scene_export_bvh8 (DESIGN.md "Wide nodes"). Child k's box is
 * origin + q * 2^(exp - 127) per axis; the internal child in slot s is node child_base + popcount(imask
 * below s); a leaf child (meta 1..127) starts at triangle slot tri_base + meta - 1. */
typedef struct crt_bvh8_node {
    float origin[3];
    uint8_t exp[3];          /* exponent field of the per-axis cell size */
    uint8_t imask;           /* bit s set: slot s holds an internal node */
    uint32_t child_base, tri_base;
    uint8_t meta[8];         /* 0 empty, 0x80 internal node, else 1 + triangle offset of a leaf */
    uint8_t qlo_x[8], qlo_y[8], qlo_z[8], qhi_x[8], qhi_y[8], qhi_z[8];
} crt_bvh8_node;

typedef struct crt_render_stats {
    uint64_t samples;
    uint64_t extend_rays, shadow_rays, probe_rays;
    uint64_t iterations;     /* wavefront iterations of the last run_view */
    uint64_t kernel_launches;/* kernels launched by the last run_view */
    float ms_total;          /* CUDA-event time of the last run_view, first launch to accumulation final */
    float ms_extend, ms_shade, ms_shadow, ms_generate;   /* per-stage totals when stage timing is on */
    float ms_tail;           /* k_tail (paths finished in place at the end of the frame) */
} crt_render_stats;

const char* crt_last_error(void);
int crt_abi_version(void);
/* number of CUDA devices visible, 0 when there is none (never an error) */
int crt_device_count(void);

/* ---- config / camera ------------------------------------------------------------------- */
/* config_task(), src/main.cu:67-90. Paths are returned as written in the file. */
int crt_config_load(const char* json_path, crt_config* out);
/* get_inverse_view_matrix(), include/Camera.h:9-36. out9 is row-major with columns [r u f]. */
int crt_inverse_view_matrix(const float eye[3], const float lookat[3], const float up[3], float out9[9]);

/* ---- scene ----------------------------------------------------------------------------- */
/* Coordinate range: for vertex coordinates and ray origins within +-2^72 no term of the traversal's box tests can
 * overflow, whatever the ray direction (derivation: csrc/crt_device.cuh kParallelDir), so the hits equal a brute-force
 * test of every triangle. Ingest refuses only non-finite coordinates; beyond 2^72 a box test can lose hits. The triangle
 * test itself multiplies three lengths, so triangles and distances beyond ~2^42 overflow in it. */
/* Scene::Scene, include/Scene.h:28 (width/height live on the render handle here). */
int crt_scene_create(crt_scene** out);
/* Loader::read_OBJ + the load_object / add_normal_obj / add_light_obj loop, src/main.cu:122-145,
 * include/Loader.h:30-124, include/OBJLoader.h:61-203. May be called once per OBJ_paths entry.
 * The text is parsed in newline-aligned chunks on all host threads (environment CRT_INGEST_THREADS overrides the count);
 * the scene, the first error and its line number do not depend on the thread count. Besides the reference's "v" and
 * "v/vt/vn" corners, "v//vn", "v/vt", a leading '+' and negative (relative) indices are read. */
int crt_scene_add_obj(crt_scene* s, const char* obj_path, const char* mtl_dir);
/* Same, from memory: verts n_tris*9 (v1 v2 v3), mat_id / obj_id per triangle (obj = usemtl group,
 * numbered from 0 in first-use order), mats[n_mats]. */
int crt_scene_add_triangles(crt_scene* s, const float* verts, const uint32_t* mat_id, const uint32_t* obj_id,
                            uint64_t n_tris, const crt_material* mats, uint32_t n_mats);
/* Scene::set_BVH, include/Scene.h:50-54 / BVH::BVH, include/BVH.h:30-84 — but built on the GPU
 * `device`, followed by the uploads of DeviceBVH::DeviceBVH (include/DeviceBVH.cuh:52-80) and
 * DeviceLights::DeviceLights (include/DeviceLights.cuh:63-87). build_ms (optional) receives the
 * CUDA-event time of the build kernels. */
int crt_scene_build_bvh(crt_scene* s, uint32_t thresh_n, int builder, int device, float* build_ms);
int crt_scene_counts(crt_scene* s, uint64_t* n_tris, uint32_t* n_mats, uint32_t* n_lights, uint64_t* n_nodes);
/* Host-side triangle table in scene order (face id = index); any pointer may be NULL.
 * verts n*9, normal n*3, area n, area_of_obj n, mat n, obj n. (include/Triangle.h:23-41, Object.h:12-26) */
int crt_scene_export_tris(crt_scene* s, float* verts, float* normal, float* area, float* area_of_obj,
                          int32_t* mat, int32_t* obj);
/* mats n*9: kd(3) ke(3) ns has_emit mode (include/Material.h:33-40, Loader.h:107) */
int crt_scene_export_mats(crt_scene* s, float* out);
/* light object li: n (in/out: capacity/size) face ids and the object's area (include/Object.h:15-23) */
int crt_scene_export_light(crt_scene* s, uint32_t li, int32_t* faces, uint32_t* n, float* area);
/* The GPU-built BVH, copied back: nodes[n_nodes], tri_order[n_tris] (slot -> face id),
 * last[n_tris] (leaf terminators), bounds lo(3) hi(3). Any pointer may be NULL. */
int crt_scene_export_bvh(crt_scene* s, crt_bvh_node* nodes, int32_t* tri_order, uint8_t* last, float bounds[6]);
/* Same for a scene built with CRT_BUILDER_LBVH8 (CRT_ERR_STATE otherwise; crt_scene_export_bvh likewise
 * refuses a wide scene). crt_scene_bvh_kind reports the crt_builder the scene was built with. */
int crt_scene_export_bvh8(crt_scene* s, crt_bvh8_node* nodes, int32_t* tri_order, uint8_t* last, float bounds[6]);
int crt_scene_bvh_kind(crt_scene* s, int* builder);
/* Scene::free, include/Scene.h:56-59 */
int crt_scene_destroy(crt_scene* s);

/* ---- ray batches (hit-id KAT, incoherent-ray microbenchmark) ---------------------------- */
/* DeviceBVH::intersect (include/DeviceBVH.cuh:128-170) / blocked (include/Render.cuh:19-27) for a
 * batch. rays: n*8 floats {o.xyz, tmax, d.xyz, 0}; d must be normalised by the caller.
 * mode CLOSEST: t > 1e-5, smallest t, ties -> lower face id; face -1 and t = FLT_MAX on a miss.
 * mode ANY: reports a blocker with t > 1e-5 and tmax - t > 1e-5 (face >= 0) or -1.
 * Host-buffer variant copies in and out; kernel_ms (optional) is the CUDA-event kernel time. */
int crt_trace_rays(crt_scene* s, const float* rays, uint64_t n, int mode, float* t_out, int32_t* face_out,
                   float* kernel_ms);
/* Device-buffer variant: pointers are device memory on the scene's device; stream may be NULL. */
int crt_trace_rays_device(crt_scene* s, const void* d_rays, uint64_t n, int mode, void* d_t_out, void* d_face_out,
                          void* stream, float* kernel_ms);

/* Incoherent-ray microbenchmark input (BASELINE config C5), generated on the device: ray i (i = start .. start+n-1)
 * has its origin uniform in the scene's bounding box and its direction uniform on the sphere, from
 * Philox4x32-10 with key (key, 0) and counters (i, 0) / (i, 1); any_hit != 0 draws tmax uniform in
 * (0, box diagonal], else tmax = FLT_MAX. d_rays: n * 8 floats of device memory. */
int crt_random_rays_device(crt_scene* s, void* d_rays, uint64_t n, uint64_t start, uint32_t key, int any_hit, void* stream);

/* ---- render ---------------------------------------------------------------------------- */
/* Render::Render, include/Render.cuh:379-433. The scene must outlive the render handle. */
int crt_render_create(crt_scene* s, uint32_t width, uint32_t height, crt_render** out);
/* Render::set_spp / set_P_RR / set_light_sample_n, include/Render.cuh:543-556 */
int crt_render_set_spp(crt_render* r, uint32_t spp);
int crt_render_set_p_rr(crt_render* r, float p_rr);
int crt_render_set_light_sample_n(crt_render* r, uint32_t light_sample_n);
int crt_render_set_seed(crt_render* r, uint32_t seed);
int crt_render_set_estimator(crt_render* r, int estimator);
/* Multi-GPU sharding: this handle renders sample indices [begin, end) of the spp set above
 * (default [0, spp)). The accumulation buffer of every shard sums to the full image exactly. */
int crt_render_set_sample_range(crt_render* r, uint32_t begin, uint32_t end);
/* Finer sharding for spp < number of GPUs: work items [begin, end) of the sample-major index space
 * w = sample * (width*height) + pixel, 0 <= w < width*height*spp. Ranges past the end are clipped. */
int crt_render_set_work_range(crt_render* r, uint64_t begin, uint64_t end);
/* Back to the default (all samples). */
int crt_render_clear_range(crt_render* r);
/* Optional: run on this CUDA stream (cudaStream_t) instead of the handle's own. */
int crt_render_set_stream(crt_render* r, void* cuda_stream);
/* Render::run_view, include/Render.cuh:435-475 (without the GL PBO). Blocking. Clears the
 * accumulation buffer, renders the sample range, leaves the fixed-point buffer on the device. */
int crt_render_run_view(crt_render* r, const float eye[3], const float inv_view[9], float fovy_rad);
/* Progressive rendering (SURVEY.md section 8(f) rank 2; the reference has no accumulation buffer, Render.cuh:342-350):
 * on != 0 makes run_view ADD its work range to the accumulation buffer instead of clearing it first, so a frame can
 * be rendered in chunks of the sample-major work index space (crt_render_set_sample_range / set_work_range). The
 * buffer is integer, so any chunking gives the bit-identical image. crt_render_clear_accum zeroes the buffer. */
int crt_render_set_accumulate(crt_render* r, int on);
int crt_render_clear_accum(crt_render* r);
/* Checkpoint / resume of a progressive render. save: writes the render settings, the camera of the last run_view,
 * `work_done` (the caller's count of finished work items, w in [0, work_done)) and the int64 accumulation buffer to
 * `path` (written to path.tmp, then renamed). load: the file's width, height, spp, seed, estimator, P_RR and
 * light_sample_n must equal the handle's current settings (CRT_ERR_STATE otherwise; CRT_ERR_IO for a truncated or
 * corrupt file - the payload carries an FNV-1a checksum); fills the accumulation buffer, turns accumulate on and
 * returns work_done and the camera (any out pointer may be NULL). With AOVs on (crt_render_set_aov) the file also holds the AOV
 * buffer; load requires the file's AOV flag to equal the handle's setting (CRT_ERR_STATE otherwise). A later run_view with a different camera fails with
 * CRT_ERR_STATE until crt_render_clear_accum is called. */
int crt_render_save_checkpoint(crt_render* r, const char* path, uint64_t work_done);
int crt_render_load_checkpoint(crt_render* r, const char* path, uint64_t* work_done, float eye[3], float inv_view[9],
                               float* fovy_rad);
/* Device pointer of the accumulation buffer: int64[width*height*3], radiance * 2^32 summed over
 * samples. Callers reduce it across GPUs (NCCL sum of int64) before resolving. */
int crt_render_device_accum(crt_render* r, void** d_accum);
/* Copies of the accumulation buffer: raw fixed point, or linear float mean over `spp`. */
int crt_render_get_accum_i64(crt_render* r, int64_t* out);
int crt_render_get_accum(crt_render* r, float* rgb);
/* Render::get_frame_buffer, include/Render.cuh:495 — tone-mapped RGB8, top row first
 * (include/Render.cuh:350: 255 * pow(clamp(c,0,1), 0.6), truncated). */
int crt_render_get_rgb8(crt_render* r, uint8_t* out);
/* The display path of Render::run_view(..., cudaGraphicsResource*), include/Render.cuh:446-469 (kernel -> device_frame_buffer ->
 * cudaMemcpy device to device into the mapped pixel buffer object), for a viewer that owns the GL side: the tone-mapped RGB8 frame
 * is written straight into d_rgb8, a DEVICE buffer of width*height*3 bytes on the render's device (e.g. the pointer
 * cudaGraphicsResourceGetMappedPointer returns for the viewer's PBO). Returns when the frame is in the buffer. */
int crt_render_get_rgb8_device(crt_render* r, void* d_rgb8);
/* Render::save_frame_buffer, include/Render.cuh:489-493 */
int crt_render_save_png(crt_render* r, const char* path);
/* AOV buffers for denoisers (DESIGN.md "AOV buffers"): with on != 0 (default 0), every run_view also traces the camera ray of
 * each of its work items - the ray the colour's path starts with, same jitter - closest-hit, and adds to aov[8 * pixel + k] the
 * fixed-point (value * 2^32) albedo (k 0-2: Kd of the hit face's material, columns 0-2 of crt_scene_export_mats), face normal
 * (3-5, as crt_scene_export_tris returns it, not flipped toward the camera), depth (6: min(t / depth_unit, 1)) and coverage
 * (7: 1); a miss adds nothing. depth_unit is the smallest power of two >= the largest distance from the eye to a corner of the
 * scene bounds (1 if that is 0). The buffer is cleared with the accumulation buffer and, like it, bit-identical for any chunking
 * of the work range and any GPU count. The pass runs after the wavefront, inside ms_total and kernel_launches; with AOVs off
 * nothing is launched or allocated (the buffer takes 64 bytes per pixel).
 * set_aov: CRT_ERR_STATE while accumulate is on and the accumulation buffer holds work since the last clear.
 * get_aov: albedo and normal n*3, depth and coverage n floats (n = width*height, top row first, any pointer may be NULL);
 * albedo, normal, coverage are the sums / 2^32 / spp, depth the mean over the samples that hit (in scene units), +inf where none did.
 * get_aov_i64: the raw int64[n*8] buffer and depth_unit. device_aov: its device pointer (for a caller-side int64 sum across GPUs,
 * as crt_render_device_accum). Every get returns CRT_ERR_STATE until a run_view with AOVs on (or a checkpoint with AOVs) has
 * filled the buffer for the current accumulation. */
int crt_render_set_aov(crt_render* r, int on);
int crt_render_get_aov(crt_render* r, float* albedo, float* normal, float* depth, float* coverage);
int crt_render_get_aov_i64(crt_render* r, int64_t* out, float* depth_unit);
int crt_render_device_aov(crt_render* r, void** d_aov, float* depth_unit);
int crt_render_get_stats(crt_render* r, crt_render_stats* out);
/* 1: time every wavefront stage with CUDA events (slower; for profiles). Default 0. */
int crt_render_set_stage_timing(crt_render* r, int on);
/* Render::free, include/Render.cuh:477-487 */
int crt_render_destroy(crt_render* r);

/* ---- several GPUs of one box behind one handle ------------------------------------------- */
/* The reference renders on device 0 only (src/main.cu:99-100). A crt_group is Render::Render + run_view for N GPUs driven
 * by the calling thread (SURVEY.md section 8(b)/(e)): the scene `s` must be built on devices[0]; every other device gets a
 * device-to-device replica of the built scene (no second parse or build), GPU g renders a contiguous share of the sample-major
 * work index space (whole samples when spp >= N, pixel ranges of a sample otherwise) on its own stream, the int64
 * accumulation buffers are summed onto devices[0] with one ncclReduce (the NCCL library is loaded when a group of more than
 * one GPU is created: libnccl.so.2, or the file CRT_NCCL_LIB names) and resolved there. The buffer, and therefore the frame,
 * is bit-identical for every N. Not thread-safe; the scene must outlive the group. */
typedef struct crt_group crt_group;
int crt_group_create(crt_scene* s, uint32_t width, uint32_t height, const int* devices, uint32_t n_devices, crt_group** out);
/* Render::set_spp / set_P_RR / set_light_sample_n (include/Render.cuh:543-556) + seed and estimator, for every GPU of the group */
int crt_group_set_params(crt_group* g, uint32_t spp, float p_rr, uint32_t light_sample_n, uint32_t seed, int estimator);
/* Render::run_view (include/Render.cuh:435-475). Blocking; the reduced buffer is left on devices[0]. */
int crt_group_run_view(crt_group* g, const float eye[3], const float inv_view[9], float fovy_rad);
int crt_group_get_accum_i64(crt_group* g, int64_t* out);
int crt_group_get_rgb8(crt_group* g, uint8_t* out);
int crt_group_save_png(crt_group* g, const char* path);
/* AOVs for the group (see crt_render_set_aov): each GPU runs the AOV pass over its share, one more ncclReduce sums the int64 AOV
 * buffers onto devices[0]; raw and resolved AOVs are bit-identical to a single GPU's. */
int crt_group_set_aov(crt_group* g, int on);
int crt_group_get_aov(crt_group* g, float* albedo, float* normal, float* depth, float* coverage);
int crt_group_get_aov_i64(crt_group* g, int64_t* out, float* depth_unit);
/* Statistics of GPU `index` (0 .. n_devices-1) for the last run_view; reduce_ms (optional) = CUDA-event time of the ncclReduce. */
int crt_group_get_stats(crt_group* g, uint32_t index, crt_render_stats* out, float* reduce_ms);
int crt_group_destroy(crt_group* g);

/* PNG writer used by save_png, exposed for the host tools: rgb8 is width*height*3, top row first. 8-bit RGB, filter 0,
 * scanline bands of about 1 MB deflated on all host threads; the file depends on the image only. */
int crt_write_png(const char* path, const uint8_t* rgb8, uint32_t width, uint32_t height);

#ifdef __cplusplus
}
#endif
#endif /* CRT_H_ */
