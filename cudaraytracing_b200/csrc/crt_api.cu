// crt_api.cu — the C-ABI of include/crt.h. Thin glue: argument checks, handle state, error slot.
#include <cmath>
#include <cstring>
#include <cstdio>
#include <new>
#include <string>
#include <vector>

#include "crt_gpu.h"

using namespace crt;

struct crt_scene {
    HostScene host;
    DeviceScene dev;
    RayBatcherPtr batcher;
    uint32_t scene_hash = 0;            // identity of the built scene (checkpoints), 0 = not built
    bool built = false;
    uint32_t thresh_n = 0;
};

struct crt_render {
    crt_scene* scene = nullptr;
    WavefrontPtr wf;
    RenderSettings rs;
    Stream own_stream;                  // the render's own stream, until crt_render_set_stream replaces it
    cudaStream_t stream = nullptr;
    bool rendered = false;
    DevBuf<float> d_linear;
    DevBuf<uint8_t> d_rgb8;
    crt_render_stats stats{};
    // camera of the last run_view (or of the loaded checkpoint): what the accumulation buffer belongs to
    bool cam_set = false;
    float cam_eye[3] = {0, 0, 0}, cam_M[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, cam_fovy = 0;
};

// Checkpoint file: this header, then width*height*3 int64 (little endian).
struct CheckpointHeader {
    char magic[8];
    uint32_t width, height, spp, seed, estimator, light_sample_n;
    float p_rr;
    uint32_t scene_hash;          // crt_scene::scene_hash of the scene the buffer was rendered from (0 in files written before round 2)
    uint64_t work_done;
    float eye[3], M[9], fovy;
    uint32_t pad;
    uint64_t payload_bytes, payload_fnv1a;
};
static const char kCkptMagic[8] = {'C', 'R', 'T', 'C', 'K', 'P', 'T', '1'};
static uint64_t fnv1a64(const void* data, size_t n) {
    // 8 bytes at a time (word-wise FNV-1a variant; n is a multiple of 8 here)
    const uint64_t* p = (const uint64_t*)data;
    uint64_t h = 1469598103934665603ull;
    for (size_t i = 0; i < n / 8; ++i) { h ^= p[i]; h *= 1099511628211ull; }
    return h;
}
static bool same_camera(const crt_render* r, const float eye[3], const float M[9], float fovy) {
    return memcmp(r->cam_eye, eye, sizeof(r->cam_eye)) == 0 && memcmp(r->cam_M, M, sizeof(r->cam_M)) == 0 &&
           memcmp(&r->cam_fovy, &fovy, sizeof(float)) == 0;
}

namespace crt {
int cuda_fail(cudaError_t e, const char* what) {
    set_error(std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what);
    cudaGetLastError();   // clear sticky-free errors
    return CRT_ERR_CUDA;
}
}  // namespace crt

// No C++ exception crosses the C ABI: allocation failures (std::vector / std::string in the loaders, the checkpoint
// code, the PNG reader) and anything else thrown below an entry point become a status + message.
template <typename F>
static int guarded(const char* fn, F&& f) noexcept {
    try {
        return f();
    } catch (const std::bad_alloc&) {
        try { set_error(std::string(fn) + ": out of memory"); } catch (...) {}
        return CRT_ERR_NOMEM;
    } catch (const std::exception& e) {
        try { set_error(std::string(fn) + ": " + e.what()); } catch (...) {}
        return CRT_ERR_INVALID;
    } catch (...) {
        try { set_error(std::string(fn) + ": unknown exception"); } catch (...) {}
        return CRT_ERR_INVALID;
    }
}

#define CHECK_ARG(cond, msg)                         \
    do {                                             \
        if (!(cond)) { set_error(msg); return CRT_ERR_INVALID; } \
    } while (0)

extern "C" {

const char* crt_last_error(void) { return get_error(); }
int crt_abi_version(void) { return CRT_ABI_VERSION; }
int crt_device_count(void) {
    return guarded("crt_device_count", [&]() -> int {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
    });
}

int crt_config_load(const char* json_path, crt_config* out) {
    return guarded("crt_config_load", [&]() -> int {
    CHECK_ARG(json_path && out, "crt_config_load: null argument");
    return load_config(json_path, out);
    });
}

int crt_inverse_view_matrix(const float eye[3], const float lookat[3], const float up[3], float out9[9]) {
    return guarded("crt_inverse_view_matrix", [&]() -> int {
    CHECK_ARG(eye && lookat && up && out9, "crt_inverse_view_matrix: null argument");
    inverse_view_matrix(eye, lookat, up, out9);
    return CRT_OK;
    });
}

int crt_write_png(const char* path, const uint8_t* rgb8, uint32_t width, uint32_t height) {
    return guarded("crt_write_png", [&]() -> int {
    return write_png(path, rgb8, width, height);
    });
}

// ---- scene -------------------------------------------------------------------------------
int crt_scene_create(crt_scene** out) {
    return guarded("crt_scene_create", [&]() -> int {
    CHECK_ARG(out, "crt_scene_create: null argument");
    *out = new (std::nothrow) crt_scene();
    if (!*out) { set_error("out of memory"); return CRT_ERR_NOMEM; }
    return CRT_OK;
    });
}

int crt_scene_add_obj(crt_scene* s, const char* obj_path, const char* mtl_dir) {
    return guarded("crt_scene_add_obj", [&]() -> int {
    CHECK_ARG(s && obj_path && mtl_dir, "crt_scene_add_obj: null argument");
    if (s->built) { set_error("crt_scene_add_obj: BVH already built"); return CRT_ERR_STATE; }
    return load_obj(s->host, obj_path, mtl_dir);
    });
}

int crt_scene_add_triangles(crt_scene* s, const float* verts, const uint32_t* mat_id, const uint32_t* obj_id, uint64_t n_tris,
                            const crt_material* mats, uint32_t n_mats) {
    return guarded("crt_scene_add_triangles", [&]() -> int {
    CHECK_ARG(s && (n_tris == 0 || (verts && mat_id && obj_id)) && (n_mats == 0 || mats), "crt_scene_add_triangles: null argument");
    if (s->built) { set_error("crt_scene_add_triangles: BVH already built"); return CRT_ERR_STATE; }
    HostScene& h = s->host;
    const int mat0 = (int)h.mats.size(), obj0 = h.n_objects;
    // object ids number the usemtl groups of this call: at most one per triangle
    uint32_t max_obj = 0;
    for (uint64_t t = 0; t < n_tris; ++t) {
        CHECK_ARG(mat_id[t] < n_mats, "crt_scene_add_triangles: mat_id out of range");
        CHECK_ARG((uint64_t)obj_id[t] < n_tris, "crt_scene_add_triangles: obj_id out of range (ids number the groups of this call: < n_tris)");
        if (obj_id[t] > max_obj) max_obj = obj_id[t];
    }
    CHECK_ARG(n_tris <= 0x7fffffffull / 4 && (uint64_t)obj0 + max_obj + 1 <= 0x7fffffffull, "crt_scene_add_triangles: scene too large");
    if (!append_triangles(h, verts, mat_id, obj_id, (size_t)n_tris, mat0, obj0)) {      // leaves the scene unchanged when it fails
        set_error("crt_scene_add_triangles: non-finite vertex coordinate");
        return CRT_ERR_INVALID;
    }
    try {
        for (uint32_t m = 0; m < n_mats; ++m) {
            HostMaterial hm;
            memcpy(hm.kd, mats[m].kd, sizeof(hm.kd));
            memcpy(hm.ks, mats[m].ks, sizeof(hm.ks));
            memcpy(hm.ke, mats[m].ke, sizeof(hm.ke));
            hm.ns = mats[m].ns;
            finish_material(hm);
            h.mats.push_back(hm);
        }
        if (n_tris) h.n_objects = obj0 + (int)max_obj + 1;
        finish_objects(h);
    } catch (...) {                                        // allocation failure: back to the scene as it was
        const size_t t0 = h.n_tris() - (size_t)n_tris;
        h.verts.resize(9 * t0); h.normal.resize(3 * t0); h.area.resize(t0); h.area_of_obj.resize(t0); h.mat.resize(t0); h.obj.resize(t0);
        h.mats.resize(mat0);
        h.n_objects = obj0;
        throw;
    }
    return CRT_OK;
    });
}

int crt_scene_build_bvh(crt_scene* s, uint32_t thresh_n, int builder, int device, float* build_ms) {
    return guarded("crt_scene_build_bvh", [&]() -> int {
    CHECK_ARG(s, "crt_scene_build_bvh: null scene");
    CHECK_ARG(builder >= CRT_BUILDER_LBVH && builder <= CRT_BUILDER_PLOC8, "crt_scene_build_bvh: unknown builder");
    int n = crt_device_count();
    if (n <= 0) { set_error("crt_scene_build_bvh: no CUDA device (there is no CPU fallback)"); return CRT_ERR_CUDA; }
    CHECK_ARG(device >= 0 && device < n, "crt_scene_build_bvh: device out of range");
    s->batcher.reset();                                                              // its buffers belong to the previous build's device
    int rc = upload_scene(s->host, thresh_n, builder, device, s->dev, build_ms);
    s->built = rc == CRT_OK;
    s->thresh_n = thresh_n;
    if (rc != CRT_OK) { s->dev = DeviceScene(); return rc; }                         // nothing half-uploaded stays behind
    // identity of the scene for checkpoints: triangle count, leaf rule and an FNV-1a of the vertex and material tables
    {
        uint64_t h = fnv1a64(s->host.verts.data(), s->host.verts.size() * sizeof(float) / 8 * 8);
        for (const HostMaterial& m : s->host.mats) {
            uint32_t w[10];
            memcpy(w, m.kd, 12); memcpy(w + 3, m.ks, 12); memcpy(w + 6, m.ke, 12); memcpy(w + 9, &m.ns, 4);
            for (uint32_t x : w) { h ^= x; h *= 1099511628211ull; }
        }
        h ^= (uint64_t)s->host.n_tris() * 0x9E3779B97F4A7C15ull;
        s->scene_hash = (uint32_t)(h ^ (h >> 32));
        if (s->scene_hash == 0) s->scene_hash = 1;
    }
    return rc;
    });
}

int crt_scene_counts(crt_scene* s, uint64_t* n_tris, uint32_t* n_mats, uint32_t* n_lights, uint64_t* n_nodes) {
    return guarded("crt_scene_counts", [&]() -> int {
    CHECK_ARG(s, "crt_scene_counts: null scene");
    if (n_tris) *n_tris = s->host.n_tris();
    if (n_mats) *n_mats = (uint32_t)s->host.mats.size();
    if (n_lights) *n_lights = (uint32_t)s->host.lights.size();
    if (n_nodes) *n_nodes = s->built ? s->dev.n_nodes : 0;
    return CRT_OK;
    });
}

int crt_scene_export_tris(crt_scene* s, float* verts, float* normal, float* area, float* area_of_obj, int32_t* mat, int32_t* obj) {
    return guarded("crt_scene_export_tris", [&]() -> int {
    CHECK_ARG(s, "crt_scene_export_tris: null scene");
    const HostScene& h = s->host;
    const size_t n = h.n_tris();
    if (verts) memcpy(verts, h.verts.data(), sizeof(float) * 9 * n);
    if (normal) memcpy(normal, h.normal.data(), sizeof(float) * 3 * n);
    if (area) memcpy(area, h.area.data(), sizeof(float) * n);
    if (area_of_obj) memcpy(area_of_obj, h.area_of_obj.data(), sizeof(float) * n);
    if (mat) memcpy(mat, h.mat.data(), sizeof(int32_t) * n);
    if (obj) memcpy(obj, h.obj.data(), sizeof(int32_t) * n);
    return CRT_OK;
    });
}

int crt_scene_export_mats(crt_scene* s, float* out) {
    return guarded("crt_scene_export_mats", [&]() -> int {
    CHECK_ARG(s && out, "crt_scene_export_mats: null argument");
    for (size_t m = 0; m < s->host.mats.size(); ++m) {
        const HostMaterial& hm = s->host.mats[m];
        float* o = out + 9 * m;
        o[0] = hm.kd[0]; o[1] = hm.kd[1]; o[2] = hm.kd[2]; o[3] = hm.ke[0]; o[4] = hm.ke[1]; o[5] = hm.ke[2];
        o[6] = hm.ns; o[7] = (float)hm.has_emit; o[8] = (float)hm.mode;
    }
    return CRT_OK;
    });
}

int crt_scene_export_light(crt_scene* s, uint32_t li, int32_t* faces, uint32_t* n, float* area) {
    return guarded("crt_scene_export_light", [&]() -> int {
    CHECK_ARG(s && n, "crt_scene_export_light: null argument");
    CHECK_ARG(li < s->host.lights.size(), "crt_scene_export_light: light index out of range");
    const HostLight& L = s->host.lights[li];
    if (faces) {
        CHECK_ARG(*n >= L.faces.size(), "crt_scene_export_light: buffer too small");
        memcpy(faces, L.faces.data(), sizeof(int32_t) * L.faces.size());
    }
    *n = (uint32_t)L.faces.size();
    if (area) *area = L.area;
    return CRT_OK;
    });
}

int crt_scene_export_bvh(crt_scene* s, crt_bvh_node* nodes, int32_t* tri_order, uint8_t* last, float bounds[6]) {
    return guarded("crt_scene_export_bvh", [&]() -> int {
    CHECK_ARG(s, "crt_scene_export_bvh: null scene");
    if (!s->built) { set_error("crt_scene_export_bvh: BVH not built"); return CRT_ERR_STATE; }
    if (s->dev.wide) { set_error("crt_scene_export_bvh: the scene has 8-wide nodes (use crt_scene_export_bvh8)"); return CRT_ERR_STATE; }
    CRT_CUDA(cudaSetDevice(s->dev.device));
    if (nodes && s->dev.n_nodes) CRT_CUDA(cudaMemcpy(nodes, s->dev.nodes.get(), sizeof(crt_bvh_node) * s->dev.n_nodes, cudaMemcpyDeviceToHost));
    if (tri_order && s->dev.n_tris) CRT_CUDA(cudaMemcpy(tri_order, s->dev.order.get(), sizeof(int32_t) * s->dev.n_tris, cudaMemcpyDeviceToHost));
    if (last && s->dev.n_tris) CRT_CUDA(cudaMemcpy(last, s->dev.last.get(), s->dev.n_tris, cudaMemcpyDeviceToHost));
    if (bounds) memcpy(bounds, s->dev.bounds, sizeof(float) * 6);
    return CRT_OK;
    });
}

int crt_scene_export_bvh8(crt_scene* s, crt_bvh8_node* nodes, int32_t* tri_order, uint8_t* last, float bounds[6]) {
    return guarded("crt_scene_export_bvh8", [&]() -> int {
    static_assert(sizeof(crt_bvh8_node) == 80, "crt_bvh8_node must be 80 bytes");
    CHECK_ARG(s, "crt_scene_export_bvh8: null scene");
    if (!s->built) { set_error("crt_scene_export_bvh8: BVH not built"); return CRT_ERR_STATE; }
    if (!s->dev.wide) { set_error("crt_scene_export_bvh8: the scene has child-pair nodes (use crt_scene_export_bvh)"); return CRT_ERR_STATE; }
    CRT_CUDA(cudaSetDevice(s->dev.device));
    if (nodes && s->dev.n_nodes) CRT_CUDA(cudaMemcpy(nodes, s->dev.nodes.get(), sizeof(crt_bvh8_node) * s->dev.n_nodes, cudaMemcpyDeviceToHost));
    if (tri_order && s->dev.n_tris) CRT_CUDA(cudaMemcpy(tri_order, s->dev.order.get(), sizeof(int32_t) * s->dev.n_tris, cudaMemcpyDeviceToHost));
    if (last && s->dev.n_tris) CRT_CUDA(cudaMemcpy(last, s->dev.last.get(), s->dev.n_tris, cudaMemcpyDeviceToHost));
    if (bounds) memcpy(bounds, s->dev.bounds, sizeof(float) * 6);
    return CRT_OK;
    });
}

int crt_scene_bvh_kind(crt_scene* s, int* builder) {
    return guarded("crt_scene_bvh_kind", [&]() -> int {
    CHECK_ARG(s && builder, "crt_scene_bvh_kind: null argument");
    if (!s->built) { set_error("crt_scene_bvh_kind: BVH not built"); return CRT_ERR_STATE; }
    *builder = s->dev.builder;
    return CRT_OK;
    });
}

int crt_scene_destroy(crt_scene* s) {
    return guarded("crt_scene_destroy", [&]() -> int {
    if (!s) return CRT_OK;
    if (s->built) cudaSetDevice(s->dev.device);
    delete s;
    return CRT_OK;
    });
}

// ---- ray batches ---------------------------------------------------------------------------
static int scene_batcher(crt_scene* s) {
    if (s->batcher) return CRT_OK;
    return ray_batcher_create(s->dev, s->batcher);
}

int crt_trace_rays_device(crt_scene* s, const void* d_rays, uint64_t n, int mode, void* d_t_out, void* d_face_out, void* stream,
                          float* kernel_ms) {
    return guarded("crt_trace_rays_device", [&]() -> int {
    CHECK_ARG(s && (n == 0 || d_rays), "crt_trace_rays_device: null argument");
    CHECK_ARG((mode & ~CRT_RAY_SORTED) == CRT_RAY_CLOSEST || (mode & ~CRT_RAY_SORTED) == CRT_RAY_ANY, "crt_trace_rays_device: unknown mode");
    if (!s->built) { set_error("crt_trace_rays: BVH not built"); return CRT_ERR_STATE; }
    CRT_CUDA(cudaSetDevice(s->dev.device));
    if (n == 0) { if (kernel_ms) *kernel_ms = 0; return CRT_OK; }
    int rc = scene_batcher(s);
    if (rc != CRT_OK) return rc;
    return trace_rays_device(s->batcher.get(), s->dev, (const float4*)d_rays, n, mode, (float*)d_t_out, (int*)d_face_out, (cudaStream_t)stream, kernel_ms);
    });
}

int crt_trace_rays(crt_scene* s, const float* rays, uint64_t n, int mode, float* t_out, int32_t* face_out, float* kernel_ms) {
    return guarded("crt_trace_rays", [&]() -> int {
    CHECK_ARG(s && (n == 0 || rays), "crt_trace_rays: null argument");
    CHECK_ARG((mode & ~CRT_RAY_SORTED) == CRT_RAY_CLOSEST || (mode & ~CRT_RAY_SORTED) == CRT_RAY_ANY, "crt_trace_rays: unknown mode");
    if (!s->built) { set_error("crt_trace_rays: BVH not built"); return CRT_ERR_STATE; }
    CRT_CUDA(cudaSetDevice(s->dev.device));
    if (n == 0) { if (kernel_ms) *kernel_ms = 0; return CRT_OK; }
    int rc = scene_batcher(s);
    if (rc != CRT_OK) return rc;
    return trace_rays_host(s->batcher.get(), s->dev, rays, n, mode, t_out, face_out, kernel_ms);
    });
}

int crt_random_rays_device(crt_scene* s, void* d_rays, uint64_t n, uint64_t start, uint32_t key, int any_hit, void* stream) {
    return guarded("crt_random_rays_device", [&]() -> int {
    CHECK_ARG(s && (n == 0 || d_rays), "crt_random_rays_device: null argument");
    if (!s->built) { set_error("crt_random_rays_device: BVH not built"); return CRT_ERR_STATE; }
    CRT_CUDA(cudaSetDevice(s->dev.device));
    return random_rays_device(s->dev, (float4*)d_rays, n, start, key, any_hit, (cudaStream_t)stream);
    });
}

// ---- render ----------------------------------------------------------------------------------
int crt_render_create(crt_scene* s, uint32_t width, uint32_t height, crt_render** out) {
    return guarded("crt_render_create", [&]() -> int {
    CHECK_ARG(s && out, "crt_render_create: null argument");
    CHECK_ARG(width > 0 && height > 0 && (uint64_t)width * height <= (1ull << 28), "crt_render_create: bad image size");
    if (!s->built) { set_error("crt_render_create: build the BVH first (crt_scene_build_bvh)"); return CRT_ERR_STATE; }
    CRT_CUDA(cudaSetDevice(s->dev.device));
    std::unique_ptr<crt_render> r(new (std::nothrow) crt_render());      // released on failure, with the scene's device current
    if (!r) { set_error("out of memory"); return CRT_ERR_NOMEM; }
    r->scene = s;
    r->rs.width = width; r->rs.height = height;
    int rc = wavefront_create(s->dev, width, height, r->wf);
    if (rc != CRT_OK) return rc;
    CRT_CUDA(create(r->own_stream));
    r->stream = r->own_stream.get();
    CRT_CUDA(r->d_linear.alloc(3 * (size_t)width * height));
    CRT_CUDA(r->d_rgb8.alloc(3 * (size_t)width * height));
    *out = r.release();
    return CRT_OK;
    });
}

int crt_render_set_spp(crt_render* r, uint32_t spp) {
    return guarded("crt_render_set_spp", [&]() -> int {
    CHECK_ARG(r && spp > 0, "crt_render_set_spp: invalid argument");
    r->rs.spp = spp;
    return CRT_OK;
    });
}
int crt_render_set_p_rr(crt_render* r, float p_rr) {
    return guarded("crt_render_set_p_rr", [&]() -> int {
    CHECK_ARG(r && p_rr >= 0.0f && p_rr <= 1.0f, "crt_render_set_p_rr: P_RR must be in [0,1]");
    r->rs.p_rr = p_rr;
    return CRT_OK;
    });
}
int crt_render_set_light_sample_n(crt_render* r, uint32_t n) {
    return guarded("crt_render_set_light_sample_n", [&]() -> int {
    CHECK_ARG(r && n > 0 && n <= 4096, "crt_render_set_light_sample_n: invalid argument");
    r->rs.light_sample_n = n;
    return CRT_OK;
    });
}
int crt_render_set_seed(crt_render* r, uint32_t seed) {
    return guarded("crt_render_set_seed", [&]() -> int {
    CHECK_ARG(r, "crt_render_set_seed: null handle");
    r->rs.seed = seed;
    return CRT_OK;
    });
}
int crt_render_set_estimator(crt_render* r, int estimator) {
    return guarded("crt_render_set_estimator", [&]() -> int {
    CHECK_ARG(r && (estimator == CRT_ESTIMATOR_COMPAT || estimator == CRT_ESTIMATOR_MIS), "crt_render_set_estimator: unknown estimator");
    r->rs.estimator = estimator;
    return CRT_OK;
    });
}
int crt_render_set_sample_range(crt_render* r, uint32_t begin, uint32_t end) {
    return guarded("crt_render_set_sample_range", [&]() -> int {
    CHECK_ARG(r && begin <= end, "crt_render_set_sample_range: invalid range");
    const unsigned long long npix = (unsigned long long)r->rs.width * r->rs.height;
    r->rs.work_begin = npix * begin; r->rs.work_end = npix * end; r->rs.range_set = true;
    return CRT_OK;
    });
}
int crt_render_set_work_range(crt_render* r, uint64_t begin, uint64_t end) {
    return guarded("crt_render_set_work_range", [&]() -> int {
    CHECK_ARG(r && begin <= end, "crt_render_set_work_range: invalid range");
    r->rs.work_begin = begin; r->rs.work_end = end; r->rs.range_set = true;
    return CRT_OK;
    });
}
int crt_render_clear_range(crt_render* r) {
    return guarded("crt_render_clear_range", [&]() -> int {
    CHECK_ARG(r, "crt_render_clear_range: null handle");
    r->rs.range_set = false;
    return CRT_OK;
    });
}
int crt_render_set_stream(crt_render* r, void* cuda_stream) {
    return guarded("crt_render_set_stream", [&]() -> int {
    CHECK_ARG(r, "crt_render_set_stream: null handle");
    r->own_stream.reset();
    r->stream = (cudaStream_t)cuda_stream;
    return CRT_OK;
    });
}
int crt_render_set_stage_timing(crt_render* r, int on) {
    return guarded("crt_render_set_stage_timing", [&]() -> int {
    CHECK_ARG(r, "crt_render_set_stage_timing: null handle");
    r->rs.stage_timing = on != 0;
    return CRT_OK;
    });
}

int crt_render_run_view(crt_render* r, const float eye[3], const float inv_view[9], float fovy_rad) {
    return guarded("crt_render_run_view", [&]() -> int {
    CHECK_ARG(r && eye && inv_view, "crt_render_run_view: null argument");
    CRT_CUDA(cudaSetDevice(r->scene->dev.device));
    if (r->rs.accumulate && r->cam_set && !same_camera(r, eye, inv_view, fovy_rad)) {
        set_error("crt_render_run_view: accumulate is on and the camera differs from the one the accumulation buffer belongs to "
                  "(crt_render_clear_accum first)");
        return CRT_ERR_STATE;
    }
    memcpy(r->cam_eye, eye, sizeof(r->cam_eye)); memcpy(r->cam_M, inv_view, sizeof(r->cam_M)); r->cam_fovy = fovy_rad;
    r->cam_set = true;
    float tan_half = tanf(fovy_rad / 2);                          // Render.cuh:338, evaluated on the host
    int rc = wavefront_render(r->wf.get(), r->scene->dev, r->rs, eye, inv_view, tan_half, r->stream, &r->stats);
    r->rendered = rc == CRT_OK;
    return rc;
    });
}

int crt_render_set_accumulate(crt_render* r, int on) {
    return guarded("crt_render_set_accumulate", [&]() -> int {
    CHECK_ARG(r, "crt_render_set_accumulate: null handle");
    r->rs.accumulate = on != 0;
    return CRT_OK;
    });
}
int crt_render_clear_accum(crt_render* r) {
    return guarded("crt_render_clear_accum", [&]() -> int {
    CHECK_ARG(r, "crt_render_clear_accum: null handle");
    CRT_CUDA(cudaSetDevice(r->scene->dev.device));
    CRT_CUDA(cudaMemsetAsync(wavefront_accum(r->wf.get()), 0, sizeof(int64_t) * 3 * (size_t)r->rs.width * r->rs.height, r->stream));
    CRT_CUDA(cudaStreamSynchronize(r->stream));
    r->cam_set = false;
    return CRT_OK;
    });
}

int crt_render_save_checkpoint(crt_render* r, const char* path, uint64_t work_done) {
    return guarded("crt_render_save_checkpoint", [&]() -> int {
    CHECK_ARG(r && path, "crt_render_save_checkpoint: null argument");
    CHECK_ARG(work_done <= (uint64_t)r->rs.width * r->rs.height * r->rs.spp, "crt_render_save_checkpoint: work_done exceeds width * height * spp");
    if (!r->cam_set) { set_error("crt_render_save_checkpoint: nothing rendered yet"); return CRT_ERR_STATE; }
    CRT_CUDA(cudaSetDevice(r->scene->dev.device));
    const size_t n = 3 * (size_t)r->rs.width * r->rs.height;
    std::vector<int64_t> buf(n);
    CRT_CUDA(cudaMemcpy(buf.data(), wavefront_accum(r->wf.get()), sizeof(int64_t) * n, cudaMemcpyDeviceToHost));
    CheckpointHeader h;
    memset(&h, 0, sizeof(h));
    memcpy(h.magic, kCkptMagic, 8);
    h.width = r->rs.width; h.height = r->rs.height; h.spp = r->rs.spp; h.seed = r->rs.seed; h.estimator = (uint32_t)r->rs.estimator;
    h.light_sample_n = r->rs.light_sample_n; h.p_rr = r->rs.p_rr; h.work_done = work_done;
    h.scene_hash = r->scene->scene_hash;
    memcpy(h.eye, r->cam_eye, sizeof(h.eye)); memcpy(h.M, r->cam_M, sizeof(h.M)); h.fovy = r->cam_fovy;
    h.payload_bytes = sizeof(int64_t) * n;
    h.payload_fnv1a = fnv1a64(buf.data(), h.payload_bytes);
    const std::string tmp = std::string(path) + ".tmp";
    FILE* f = fopen(tmp.c_str(), "wb");
    if (!f) { set_error(std::string("crt_render_save_checkpoint: cannot open ") + tmp); return CRT_ERR_IO; }
    bool ok = fwrite(&h, sizeof(h), 1, f) == 1 && fwrite(buf.data(), sizeof(int64_t), n, f) == n;
    ok = (fclose(f) == 0) && ok;
    if (!ok || rename(tmp.c_str(), path) != 0) { remove(tmp.c_str()); set_error(std::string("crt_render_save_checkpoint: write failed: ") + path); return CRT_ERR_IO; }
    return CRT_OK;
    });
}

int crt_render_load_checkpoint(crt_render* r, const char* path, uint64_t* work_done, float eye[3], float inv_view[9], float* fovy_rad) {
    return guarded("crt_render_load_checkpoint", [&]() -> int {
    CHECK_ARG(r && path, "crt_render_load_checkpoint: null argument");
    FILE* f = fopen(path, "rb");
    if (!f) { set_error(std::string("crt_render_load_checkpoint: cannot open ") + path); return CRT_ERR_IO; }
    CheckpointHeader h;
    const size_t n = 3 * (size_t)r->rs.width * r->rs.height;
    std::vector<int64_t> buf;
    int rc = CRT_OK;
    if (fread(&h, sizeof(h), 1, f) != 1 || memcmp(h.magic, kCkptMagic, 8) != 0) {
        set_error(std::string("crt_render_load_checkpoint: not a checkpoint file: ") + path); rc = CRT_ERR_IO;
    } else if (h.width != r->rs.width || h.height != r->rs.height || h.spp != r->rs.spp || h.seed != r->rs.seed ||
               h.estimator != (uint32_t)r->rs.estimator || h.light_sample_n != r->rs.light_sample_n ||
               memcmp(&h.p_rr, &r->rs.p_rr, sizeof(float)) != 0) {
        set_error("crt_render_load_checkpoint: the checkpoint was written with different render settings "
                  "(width, height, spp, seed, estimator, P_RR, light_sample_n must match)");
        rc = CRT_ERR_STATE;
    } else if (h.scene_hash != 0 && h.scene_hash != r->scene->scene_hash) {
        set_error("crt_render_load_checkpoint: the checkpoint was rendered from a different scene");
        rc = CRT_ERR_STATE;
    } else if (h.work_done > (uint64_t)r->rs.width * r->rs.height * r->rs.spp) {
        set_error("crt_render_load_checkpoint: work_done exceeds width * height * spp"); rc = CRT_ERR_IO;
    } else if (h.payload_bytes != sizeof(int64_t) * n) {
        set_error("crt_render_load_checkpoint: payload size does not match the image size"); rc = CRT_ERR_IO;
    } else {
        buf.resize(n);
        char extra;
        if (fread(buf.data(), sizeof(int64_t), n, f) != n || fread(&extra, 1, 1, f) != 0 || fnv1a64(buf.data(), h.payload_bytes) != h.payload_fnv1a) {
            set_error(std::string("crt_render_load_checkpoint: truncated or corrupt checkpoint: ") + path); rc = CRT_ERR_IO;
        }
    }
    fclose(f);
    if (rc != CRT_OK) return rc;
    CRT_CUDA(cudaSetDevice(r->scene->dev.device));
    CRT_CUDA(cudaMemcpy(wavefront_accum(r->wf.get()), buf.data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice));
    memcpy(r->cam_eye, h.eye, sizeof(h.eye)); memcpy(r->cam_M, h.M, sizeof(h.M)); r->cam_fovy = h.fovy;
    r->cam_set = true;
    r->rs.accumulate = true;
    r->rendered = true;
    if (work_done) *work_done = h.work_done;
    if (eye) memcpy(eye, h.eye, sizeof(h.eye));
    if (inv_view) memcpy(inv_view, h.M, sizeof(h.M));
    if (fovy_rad) *fovy_rad = h.fovy;
    return CRT_OK;
    });
}

int crt_render_device_accum(crt_render* r, void** d_accum) {
    return guarded("crt_render_device_accum", [&]() -> int {
    CHECK_ARG(r && d_accum, "crt_render_device_accum: null argument");
    *d_accum = wavefront_accum(r->wf.get());
    return CRT_OK;
    });
}

int crt_render_get_accum_i64(crt_render* r, int64_t* out) {
    return guarded("crt_render_get_accum_i64", [&]() -> int {
    CHECK_ARG(r && out, "crt_render_get_accum_i64: null argument");
    CRT_CUDA(cudaSetDevice(r->scene->dev.device));
    CRT_CUDA(cudaMemcpy(out, wavefront_accum(r->wf.get()), sizeof(int64_t) * 3 * (size_t)r->rs.width * r->rs.height, cudaMemcpyDeviceToHost));
    return CRT_OK;
    });
}

static int resolve_to(crt_render* r, float* lin_host, uint8_t* rgb_host) {
    CRT_CUDA(cudaSetDevice(r->scene->dev.device));
    const uint32_t npix = r->rs.width * r->rs.height;
    int rc = resolve_device(wavefront_accum(r->wf.get()), npix, r->rs.spp, r->d_linear.get(), r->d_rgb8.get(), r->stream);
    if (rc != CRT_OK) return rc;
    if (lin_host) CRT_CUDA(cudaMemcpyAsync(lin_host, r->d_linear.get(), sizeof(float) * 3 * (size_t)npix, cudaMemcpyDeviceToHost, r->stream));
    if (rgb_host) CRT_CUDA(cudaMemcpyAsync(rgb_host, r->d_rgb8.get(), 3 * (size_t)npix, cudaMemcpyDeviceToHost, r->stream));
    CRT_CUDA(cudaStreamSynchronize(r->stream));
    return CRT_OK;
}

int crt_render_get_accum(crt_render* r, float* rgb) {
    return guarded("crt_render_get_accum", [&]() -> int {
    CHECK_ARG(r && rgb, "crt_render_get_accum: null argument");
    return resolve_to(r, rgb, nullptr);
    });
}
int crt_render_get_rgb8(crt_render* r, uint8_t* out) {
    return guarded("crt_render_get_rgb8", [&]() -> int {
    CHECK_ARG(r && out, "crt_render_get_rgb8: null argument");
    return resolve_to(r, nullptr, out);
    });
}
int crt_render_get_rgb8_device(crt_render* r, void* d_rgb8) {
    return guarded("crt_render_get_rgb8_device", [&]() -> int {
    CHECK_ARG(r && d_rgb8, "crt_render_get_rgb8_device: null argument");
    CRT_CUDA(cudaSetDevice(r->scene->dev.device));
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, d_rgb8) != cudaSuccess || (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) ||
        (at.type == cudaMemoryTypeDevice && at.device != r->scene->dev.device)) {
        cudaGetLastError();
        set_error("crt_render_get_rgb8_device: d_rgb8 is not device memory of the render's device " + std::to_string(r->scene->dev.device));
        return CRT_ERR_INVALID;
    }
    int rc = resolve_device(wavefront_accum(r->wf.get()), r->rs.width * r->rs.height, r->rs.spp, r->d_linear.get(), (uint8_t*)d_rgb8, r->stream);
    if (rc != CRT_OK) return rc;
    CRT_CUDA(cudaStreamSynchronize(r->stream));
    return CRT_OK;
    });
}
int crt_render_save_png(crt_render* r, const char* path) {
    return guarded("crt_render_save_png", [&]() -> int {
    CHECK_ARG(r && path, "crt_render_save_png: null argument");
    std::vector<uint8_t> rgb(3 * (size_t)r->rs.width * r->rs.height);
    int rc = resolve_to(r, nullptr, rgb.data());
    if (rc != CRT_OK) return rc;
    return write_png(path, rgb.data(), r->rs.width, r->rs.height);
    });
}
int crt_render_get_stats(crt_render* r, crt_render_stats* out) {
    return guarded("crt_render_get_stats", [&]() -> int {
    CHECK_ARG(r && out, "crt_render_get_stats: null argument");
    *out = r->stats;
    return CRT_OK;
    });
}

int crt_render_destroy(crt_render* r) {
    return guarded("crt_render_destroy", [&]() -> int {
    if (!r) return CRT_OK;
    if (r->scene) cudaSetDevice(r->scene->dev.device);
    delete r;
    return CRT_OK;
    });
}

// ---- group: N GPUs, one host thread --------------------------------------------------------------
}  // extern "C"

#include <dlfcn.h>
#include <nccl.h>       // types and enums only: the library is loaded with dlopen when a group of more than one GPU is created
#include <chrono>
#include <thread>

namespace {
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi g_nccl;
int load_nccl() {
    if (g_nccl.lib) return CRT_OK;
    const char* name = getenv("CRT_NCCL_LIB");
    void* h = dlopen(name && *name ? name : "libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { set_error(std::string("crt_group: cannot load NCCL: ") + dlerror()); return CRT_ERR_STATE; }
    NcclApi a;
    a.lib = h;
    a.CommInitAll = (decltype(a.CommInitAll))dlsym(h, "ncclCommInitAll");
    a.CommDestroy = (decltype(a.CommDestroy))dlsym(h, "ncclCommDestroy");
    a.Reduce = (decltype(a.Reduce))dlsym(h, "ncclReduce");
    a.GroupStart = (decltype(a.GroupStart))dlsym(h, "ncclGroupStart");
    a.GroupEnd = (decltype(a.GroupEnd))dlsym(h, "ncclGroupEnd");
    a.GetErrorString = (decltype(a.GetErrorString))dlsym(h, "ncclGetErrorString");
    if (!a.CommInitAll || !a.CommDestroy || !a.Reduce || !a.GroupStart || !a.GroupEnd || !a.GetErrorString) {
        set_error("crt_group: the NCCL library lacks a symbol");
        return CRT_ERR_STATE;
    }
    g_nccl = a;
    return CRT_OK;
}
int nccl_fail(ncclResult_t r, const char* what) {
    set_error(std::string("NCCL error: ") + g_nccl.GetErrorString(r) + " in " + what);
    return CRT_ERR_CUDA;
}
#define CRT_NCCL(x)                                              \
    do {                                                         \
        ncclResult_t r__ = (x);                                  \
        if (r__ != ncclSuccess) return nccl_fail(r__, #x);       \
    } while (0)
}  // namespace

static constexpr int kGroupBands = 8;
struct crt_group {
    crt_scene* scene = nullptr;
    uint32_t width = 0, height = 0;
    std::vector<int> devices;
    std::vector<DeviceScene> replicas;          // [0] unused: GPU 0 renders the scene handle's own tables
    std::vector<WavefrontPtr> wf;
    std::vector<Stream> streams;
    std::vector<ncclComm_t> comms;
    std::vector<crt_render_stats> stats;
    RenderSettings rs;
    // on devices[0]:
    Event ev_r0, ev_r1;
    Event ev_band[kGroupBands];
    Stream st_resolve;                          // resolves band c while band c + 1 is being reduced
    bool resolved = false;                      // d_linear / d_rgb8 hold the resolved frame of the last run_view
    float reduce_ms = 0;
    DevBuf<float> d_linear;
    DevBuf<uint8_t> d_rgb8;
    bool rendered = false;
    const DeviceScene& scene_of(size_t g) const { return g == 0 ? scene->dev : replicas[g]; }
};

extern "C" {

int crt_group_destroy(crt_group* g) {
    if (!g) return CRT_OK;
    for (size_t k = 0; k < g->devices.size(); ++k) {
        cudaSetDevice(g->devices[k]);
        if (k < g->wf.size()) g->wf[k].reset();
        if (k < g->streams.size()) g->streams[k].reset();
        if (k < g->comms.size() && g->comms[k]) g_nccl.CommDestroy(g->comms[k]);
        if (k > 0 && k < g->replicas.size()) g->replicas[k] = DeviceScene();
    }
    if (!g->devices.empty()) cudaSetDevice(g->devices[0]);
    delete g;                                   // what is left lives on devices[0]
    return CRT_OK;
}

int crt_group_create(crt_scene* s, uint32_t width, uint32_t height, const int* devices, uint32_t n_devices, crt_group** out) {
    return guarded("crt_group_create", [&]() -> int {
    CHECK_ARG(s && out && devices && n_devices > 0 && n_devices <= 64, "crt_group_create: invalid argument");
    CHECK_ARG(width > 0 && height > 0 && (uint64_t)width * height <= (1ull << 28), "crt_group_create: bad image size");
    if (!s->built) { set_error("crt_group_create: build the BVH first (crt_scene_build_bvh)"); return CRT_ERR_STATE; }
    const int n_dev = crt_device_count();
    for (uint32_t k = 0; k < n_devices; ++k) {
        CHECK_ARG(devices[k] >= 0 && devices[k] < n_dev, "crt_group_create: device out of range");
        for (uint32_t j = 0; j < k; ++j) CHECK_ARG(devices[j] != devices[k], "crt_group_create: a device is listed twice");
    }
    CHECK_ARG(devices[0] == s->dev.device, "crt_group_create: the scene must be built on devices[0]");
    if (n_devices > 1) { int rc = load_nccl(); if (rc != CRT_OK) return rc; }
    crt_group* g = new crt_group();
    g->scene = s; g->width = width; g->height = height;
    g->devices.assign(devices, devices + n_devices);
    g->replicas.resize(n_devices);
    g->wf.resize(n_devices);
    g->streams.resize(n_devices);
    g->comms.assign(n_devices, nullptr);
    g->stats.resize(n_devices);
    g->rs.width = width; g->rs.height = height;
    auto build = [&]() -> int {
        for (uint32_t k = 0; k < n_devices; ++k) {
            if (k > 0) { int rc = clone_scene(s->dev, devices[k], g->replicas[k]); if (rc != CRT_OK) return rc; }
            CRT_CUDA(cudaSetDevice(devices[k]));
            int rc = wavefront_create(g->scene_of(k), width, height, g->wf[k]);
            if (rc != CRT_OK) return rc;
            CRT_CUDA(create(g->streams[k]));
            // the first launch of a kernel on a device loads its code (CUDA loads modules lazily; a cold process spent ~0.2 s of
            // its first 4K frame on the second GPU doing that while the first one waited for the shared host thread): one work
            // item through the whole pipeline now, on every device, so that the first run_view starts warm
            RenderSettings warm = g->rs;
            warm.width = width; warm.height = height; warm.spp = 1; warm.light_sample_n = 1;
            warm.range_set = true; warm.work_begin = 0; warm.work_end = 1;
            const float eye0[3] = {0, 0, 0}, M0[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
            crt_render_stats ws;
            rc = wavefront_render(g->wf[k].get(), g->scene_of(k), warm, eye0, M0, 1.0f, g->streams[k].get(), &ws);
            if (rc != CRT_OK) return rc;
        }
        CRT_CUDA(cudaSetDevice(devices[0]));
        CRT_CUDA(g->d_linear.alloc(3 * (size_t)width * height));
        CRT_CUDA(g->d_rgb8.alloc(3 * (size_t)width * height));
        CRT_CUDA(create(g->ev_r0));
        CRT_CUDA(create(g->ev_r1));
        for (Event& e : g->ev_band) CRT_CUDA(create(e, cudaEventDisableTiming));
        CRT_CUDA(create(g->st_resolve));
        if (n_devices > 1) {
            CRT_NCCL(g_nccl.CommInitAll(g->comms.data(), (int)n_devices, devices));
            // the first collective of a communicator sets up its connections (~0.2 s): spent here on the 24 bytes of pixel 0,
            // not inside the first frame (the buffers are cleared at the start of every run_view)
            for (uint32_t k = 0; k < n_devices; ++k) {
                CRT_CUDA(cudaSetDevice(devices[k]));
                CRT_CUDA(cudaMemsetAsync(wavefront_accum(g->wf[k].get()), 0, 3 * sizeof(long long), g->streams[k].get()));
            }
            CRT_NCCL(g_nccl.GroupStart());
            for (uint32_t k = 0; k < n_devices; ++k) {
                long long* acc = wavefront_accum(g->wf[k].get());
                CRT_NCCL(g_nccl.Reduce(acc, acc, 3, ncclInt64, ncclSum, 0, g->comms[k], g->streams[k].get()));
            }
            CRT_NCCL(g_nccl.GroupEnd());
            for (uint32_t k = 0; k < n_devices; ++k) {
                CRT_CUDA(cudaSetDevice(devices[k]));
                CRT_CUDA(cudaStreamSynchronize(g->streams[k].get()));
            }
            CRT_CUDA(cudaSetDevice(devices[0]));
        }
        return CRT_OK;
    };
    int rc = build();
    if (rc != CRT_OK) { crt_group_destroy(g); return rc; }
    *out = g;
    return CRT_OK;
    });
}

int crt_group_set_params(crt_group* g, uint32_t spp, float p_rr, uint32_t light_sample_n, uint32_t seed, int estimator) {
    CHECK_ARG(g && spp > 0 && p_rr >= 0.0f && p_rr <= 1.0f && light_sample_n > 0 && light_sample_n <= 4096, "crt_group_set_params: invalid argument");
    CHECK_ARG(estimator == CRT_ESTIMATOR_COMPAT || estimator == CRT_ESTIMATOR_MIS, "crt_group_set_params: unknown estimator");
    g->rs.spp = spp; g->rs.p_rr = p_rr; g->rs.light_sample_n = light_sample_n; g->rs.seed = seed; g->rs.estimator = estimator;
    return CRT_OK;
}

int crt_group_run_view(crt_group* g, const float eye[3], const float inv_view[9], float fovy_rad) {
    return guarded("crt_group_run_view", [&]() -> int {
    CHECK_ARG(g && eye && inv_view, "crt_group_run_view: null argument");
    const size_t G = g->devices.size();
    const unsigned long long npix = (unsigned long long)g->width * g->height, total = npix * g->rs.spp;
    const float tan_half = tanf(fovy_rad / 2);
    g->rendered = false;
    // shares of the sample-major work index space: whole samples when spp >= G (every GPU renders whole frames), else pixel ranges
    for (size_t k = 0; k < G; ++k) {
        RenderSettings rs = g->rs;
        rs.range_set = true;
        if (g->rs.spp >= G) { rs.work_begin = (k * g->rs.spp / G) * npix; rs.work_end = ((k + 1) * g->rs.spp / G) * npix; }
        else { rs.work_begin = k * total / G; rs.work_end = (k + 1) * total / G; }
        CRT_CUDA(cudaSetDevice(g->devices[k]));
        int rc = wavefront_begin(g->wf[k].get(), g->scene_of(k), rs, eye, inv_view, tan_half, g->streams[k].get());
        if (rc != CRT_OK) return rc;
    }
    // one host thread feeds every GPU: a step enqueues one wavefront iteration where the GPU is ready for it
    std::vector<char> done(G, 0);
    for (size_t left = G; left > 0;) {
        bool any = false;
        for (size_t k = 0; k < G; ++k) {
            if (done[k]) continue;
            CRT_CUDA(cudaSetDevice(g->devices[k]));
            bool d = false, progressed = false;
            int rc = wavefront_step(g->wf[k].get(), false, &d, &progressed);
            if (rc != CRT_OK) return rc;
            any = any || progressed;
            if (d) { done[k] = 1; --left; }
        }
        if (!any) std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
    for (size_t k = 0; k < G; ++k) {
        CRT_CUDA(cudaSetDevice(g->devices[k]));
        int rc = wavefront_finish(g->wf[k].get(), &g->stats[k]);
        if (rc != CRT_OK) return rc;
    }
    // The collective: sum of the int64 buffers onto devices[0] (integer addition: the same buffer for every G), issued in bands
    // of pixel rows so that the resolve of band c (fixed point -> linear -> tone map, on a second stream of devices[0]) runs
    // beside the reduce of band c + 1 (SURVEY.md 8(f)2: chunked, overlapped reduce; the reference has no accumulation buffer).
    g->reduce_ms = 0;
    g->resolved = false;
    if (G > 1) {
        // a band is at least 2^20 pixels (25 MB): a collective costs ~20 us before it moves a byte, the 800x600 frames go in one piece
        const unsigned long long band_px = std::max<unsigned long long>((npix + kGroupBands - 1) / kGroupBands, 1ull << 20);
        CRT_CUDA(cudaSetDevice(g->devices[0]));
        CRT_CUDA(cudaEventRecord(g->ev_r0.get(), g->streams[0].get()));
        int band = 0;
        for (unsigned long long px0 = 0; px0 < npix; px0 += band_px, ++band) {
            const unsigned long long cnt_px = std::min(band_px, npix - px0);
            CRT_NCCL(g_nccl.GroupStart());
            for (size_t k = 0; k < G; ++k) {
                long long* acc = wavefront_accum(g->wf[k].get()) + 3 * px0;
                CRT_NCCL(g_nccl.Reduce(acc, acc, (size_t)(3 * cnt_px), ncclInt64, ncclSum, 0, g->comms[k], g->streams[k].get()));
            }
            CRT_NCCL(g_nccl.GroupEnd());
            CRT_CUDA(cudaSetDevice(g->devices[0]));
            CRT_CUDA(cudaEventRecord(g->ev_band[band % kGroupBands].get(), g->streams[0].get()));
            CRT_CUDA(cudaStreamWaitEvent(g->st_resolve.get(), g->ev_band[band % kGroupBands].get(), 0));
            int rc = resolve_device(wavefront_accum(g->wf[0].get()) + 3 * px0, (uint32_t)cnt_px, g->rs.spp, g->d_linear.get() + 3 * px0, g->d_rgb8.get() + 3 * px0,
                                    g->st_resolve.get());
            if (rc != CRT_OK) return rc;
        }
        CRT_CUDA(cudaEventRecord(g->ev_r1.get(), g->streams[0].get()));
        for (size_t k = 0; k < G; ++k) {
            CRT_CUDA(cudaSetDevice(g->devices[k]));
            CRT_CUDA(cudaStreamSynchronize(g->streams[k].get()));
        }
        CRT_CUDA(cudaSetDevice(g->devices[0]));
        CRT_CUDA(cudaStreamSynchronize(g->st_resolve.get()));
        CRT_CUDA(cudaEventElapsedTime(&g->reduce_ms, g->ev_r0.get(), g->ev_r1.get()));
        g->resolved = true;
    }
    g->rendered = true;
    return CRT_OK;
    });
}

int crt_group_get_accum_i64(crt_group* g, int64_t* out) {
    CHECK_ARG(g && out, "crt_group_get_accum_i64: null argument");
    CRT_CUDA(cudaSetDevice(g->devices[0]));
    CRT_CUDA(cudaMemcpy(out, wavefront_accum(g->wf[0].get()), sizeof(int64_t) * 3 * (size_t)g->width * g->height, cudaMemcpyDeviceToHost));
    return CRT_OK;
}

int crt_group_get_rgb8(crt_group* g, uint8_t* out) {
    CHECK_ARG(g && out, "crt_group_get_rgb8: null argument");
    CRT_CUDA(cudaSetDevice(g->devices[0]));
    const uint32_t npix = g->width * g->height;
    if (!g->resolved) {                          // one GPU: no collective, resolved here
        int rc = resolve_device(wavefront_accum(g->wf[0].get()), npix, g->rs.spp, g->d_linear.get(), g->d_rgb8.get(), g->streams[0].get());
        if (rc != CRT_OK) return rc;
    }
    CRT_CUDA(cudaMemcpyAsync(out, g->d_rgb8.get(), 3 * (size_t)npix, cudaMemcpyDeviceToHost, g->streams[0].get()));
    CRT_CUDA(cudaStreamSynchronize(g->streams[0].get()));
    return CRT_OK;
}

int crt_group_save_png(crt_group* g, const char* path) {
    return guarded("crt_group_save_png", [&]() -> int {
    CHECK_ARG(g && path, "crt_group_save_png: null argument");
    std::vector<uint8_t> rgb(3 * (size_t)g->width * g->height);
    int rc = crt_group_get_rgb8(g, rgb.data());
    if (rc != CRT_OK) return rc;
    return write_png(path, rgb.data(), g->width, g->height);
    });
}

int crt_group_get_stats(crt_group* g, uint32_t index, crt_render_stats* out, float* reduce_ms) {
    CHECK_ARG(g && out && index < g->devices.size(), "crt_group_get_stats: invalid argument");
    *out = g->stats[index];
    if (reduce_ms) *reduce_ms = g->reduce_ms;
    return CRT_OK;
}

}  // extern "C"
