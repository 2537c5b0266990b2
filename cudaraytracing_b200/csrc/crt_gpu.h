// crt_gpu.h — device-side scene and the host entry points of the CUDA translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <memory>
#include <type_traits>

#include "crt_device.cuh"
#include "crt_host.h"

namespace crt {

// records cudaGetErrorString + context in the thread's error slot, returns CRT_ERR_CUDA
int cuda_fail(cudaError_t e, const char* what);

#define CRT_CUDA(x)                                          \
    do {                                                     \
        cudaError_t e__ = (x);                               \
        if (e__ != cudaSuccess) return cuda_fail(e__, #x);   \
    } while (0)

// ---- owners of CUDA resources: each frees what it holds when it is destroyed, reset or assigned over ----------------------------
// Device memory: n elements of T.
template <typename T>
class DevBuf {
  public:
    DevBuf() = default;
    DevBuf(DevBuf&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) { reset(); p_ = o.p_; n_ = o.n_; o.p_ = nullptr; o.n_ = 0; }
        return *this;
    }
    ~DevBuf() { reset(); }
    cudaError_t alloc(size_t n) {
        reset();
        const cudaError_t e = cudaMalloc((void**)&p_, sizeof(T) * n);
        if (e != cudaSuccess) p_ = nullptr;
        else n_ = n;
        return e;
    }
    T* get() const { return p_; }
    size_t size() const { return n_; }
    void reset() {
        if (p_) cudaFree(p_);
        p_ = nullptr;
        n_ = 0;
    }
  private:
    T* p_ = nullptr;
    size_t n_ = 0;
};
struct PinnedFree { void operator()(void* p) const { cudaFreeHost(p); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
template <typename T> using Pinned = std::unique_ptr<T, PinnedFree>;         // page-locked host memory (cudaHostAlloc)
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;
template <typename T>
inline cudaError_t pinned_alloc(Pinned<T>& p, size_t n, unsigned flags = cudaHostAllocDefault) {
    void* h = nullptr;
    const cudaError_t e = cudaHostAlloc(&h, sizeof(T) * n, flags);
    p.reset(e == cudaSuccess ? (T*)h : nullptr);
    return e;
}
inline cudaError_t create(Event& ev, unsigned flags = cudaEventDefault) {
    cudaEvent_t e = nullptr;
    const cudaError_t r = cudaEventCreateWithFlags(&e, flags);
    ev.reset(r == cudaSuccess ? e : nullptr);
    return r;
}
inline cudaError_t create(Stream& st) {
    cudaStream_t s = nullptr;
    const cudaError_t r = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
    st.reset(r == cudaSuccess ? s : nullptr);
    return r;
}

// Everything the kernels read, resident in HBM for the life of the scene handle
// (replaces DeviceBVH / DeviceTriangle / DeviceLights / DeviceMaterial uploads,
//  reference DeviceBVH.cuh:52-80, DeviceLights.cuh:12-31,63-87).
struct SceneInfo {                  // what a scene is besides its tables
    int device = 0;
    uint32_t n_tris = 0, n_nodes = 0, n_mats = 0, n_lights = 0, n_light_tris = 0;
    int builder = 0;                // crt_builder the scene was built with
    bool wide = false;              // nodes are 80-byte 8-wide compressed nodes (5 x 16 B) instead of 64-byte pairs
    float bounds[6] = {0, 0, 0, 0, 0, 0};
    bool has_specular = false;
};
struct DeviceScene : SceneInfo {
    DevBuf<float4> nodes;           // n_nodes * 4 (pairs) or n_nodes * 5 (wide)
    DevBuf<float4> tri_geom;        // n_tris * 3, BVH slot order
    DevBuf<float4> tri_shade;       // n_tris, BVH slot order
    DevBuf<uint32_t> order;         // slot -> face id
    DevBuf<uint8_t> last;           // slot -> leaf terminator
    DevBuf<float4> mats;            // n_mats * 5
    DevBuf<float4> light_tris;      // n_light_tris * 4
    DevBuf<int4> lights;            // n_lights
    DevBuf<float> light_cdf;        // n_light_tris (mis estimator)
    // f(&DeviceScene::table) for every table
    template <typename F>
    static void for_each_table(F&& f) {
        f(&DeviceScene::nodes); f(&DeviceScene::tri_geom); f(&DeviceScene::tri_shade); f(&DeviceScene::order); f(&DeviceScene::last);
        f(&DeviceScene::mats); f(&DeviceScene::light_tris); f(&DeviceScene::lights); f(&DeviceScene::light_cdf);
    }
    SceneView view() const {
        SceneView v;
        v.nodes = nodes.get(); v.tri_geom = tri_geom.get(); v.tri_shade = tri_shade.get(); v.mats = mats.get();
        v.light_tris = light_tris.get(); v.lights = lights.get(); v.n_nodes = (int)n_nodes; v.n_lights = (int)n_lights;
        v.light_cdf = light_cdf.get(); v.n_light_tris = (int)n_light_tris;
        return v;
    }
};

// GPU BVH build; d_verts: n*9 floats (face order), d_face_shade: n float4 (normal, mat bits).
int build_bvh_device(DeviceScene& ds, const float* d_verts, const float4* d_face_shade, uint32_t n, uint32_t thresh_n,
                     int builder, cudaStream_t st, float* build_ms);

// The builder's stable LSD radix sort of (uint64 key, uint32 value) pairs, 8 bits per pass, on the low 8 * passes bits; k1 / v1 are
// the ping-pong buffers, ghist / scratch hold radix_sort_hist_words(n) / radix_sort_scratch_words(n) uint32. The sorted arrays are
// *k_sorted / *v_sorted (one of the two buffers each).
size_t radix_sort_hist_words(uint32_t n);
size_t radix_sort_scratch_words(uint32_t n);
cudaError_t radix_sort_pairs(uint64_t* k0, uint64_t* k1, uint32_t* v0, uint32_t* v1, uint32_t n, int passes, uint32_t* ghist,
                             uint32_t* scratch, cudaStream_t st, uint64_t** k_sorted, uint32_t** v_sorted);

// Uploads materials and lights, builds the BVH. Leaves the device selected.
int upload_scene(const HostScene& hs, uint32_t thresh_n, int builder, int device, DeviceScene& ds, float* build_ms);

// Ray batches. rays: n * 2 float4 {o,tmax}{d,0}. A RayBatcher holds what a batch call needs besides the scene - queue
// counters, events, two streams and, for host buffers, chunk-sized device buffers and pinned staging - for the life of
// the scene handle (round 1 paid a cudaMalloc / cudaFree / event create per call).
// mode: CRT_RAY_CLOSEST / CRT_RAY_ANY, optionally | CRT_RAY_SORTED (the batch, or each chunk of it, is traced in the order of
// (Morton code of the origin's cell on a 128^3 grid over the scene, direction octant) and the hits are written back in the caller's order).
struct RayBatcher;
struct Wavefront;   // opaque pipeline state (crt_render.cu)
struct StateDelete { void operator()(RayBatcher* b) const; void operator()(Wavefront* w) const; };
using RayBatcherPtr = std::unique_ptr<RayBatcher, StateDelete>;
using WavefrontPtr = std::unique_ptr<Wavefront, StateDelete>;
int ray_batcher_create(const DeviceScene& ds, RayBatcherPtr& out);
// Device pointers on the scene's device.
int trace_rays_device(RayBatcher* b, const DeviceScene& ds, const float4* d_rays, uint64_t n, int mode, float* d_t, int* d_face,
                      cudaStream_t st, float* kernel_ms);
// Host buffers: chunks of the batch go host -> device, through the kernel and back on two streams, so copy-in, trace and
// copy-out of neighbouring chunks overlap. Page-locked caller buffers are used in place; pageable ones are staged through
// pinned memory by host threads.
int trace_rays_host(RayBatcher* b, const DeviceScene& ds, const float* rays, uint64_t n, int mode, float* t_out, int32_t* face_out,
                    float* kernel_ms);

int random_rays_device(const DeviceScene& ds, float4* d_rays, uint64_t n, uint64_t start, uint32_t key, int any_hit, cudaStream_t st);

struct RenderSettings {
    uint32_t width = 0, height = 0;
    uint32_t spp = 16;               // Render.cuh:379 defaults
    float p_rr = 0.8f;
    uint32_t light_sample_n = 1;
    uint32_t seed = 0;
    int estimator = 0;
    // work items [work_begin, work_end) of the width*height*spp (sample-major) index space;
    // range_set == false -> everything
    unsigned long long work_begin = 0, work_end = 0;
    bool range_set = false;
    bool stage_timing = false;
    bool accumulate = false;         // run_view adds to the accumulation buffer instead of clearing it (progressive rendering)
    bool aov = false;                // run_view also adds the first-hit AOVs of its work range to the AOV buffer
};

int wavefront_create(const DeviceScene& ds, uint32_t width, uint32_t height, WavefrontPtr& out);
int wavefront_render(Wavefront* w, const DeviceScene& ds, const RenderSettings& rs, const float eye[3], const float M[9],
                     float tan_half, cudaStream_t st, crt_render_stats* stats);
// The same run_view as a state machine, for one host thread driving several GPUs (crt_group): begin resets the frame,
// step does the host side of one wavefront iteration (block == false: returns with *progressed == false instead of
// waiting for the GPU), finish drains the stream and fills the statistics. The caller selects the device.
int wavefront_begin(Wavefront* w, const DeviceScene& ds, const RenderSettings& rs, const float eye[3], const float M[9],
                    float tan_half, cudaStream_t st);
int wavefront_step(Wavefront* w, bool block, bool* done, bool* progressed);
int wavefront_finish(Wavefront* w, crt_render_stats* stats);
long long* wavefront_accum(Wavefront* w);
// AOV buffer: int64[8 * width * height] (albedo 3, normal 3, depth, coverage; fixed point summed over samples), nullptr until a run
// with AOVs on, or wavefront_ensure_aov, has allocated it (zeroed, on stream st).
long long* wavefront_aov(Wavefront* w);
int wavefront_ensure_aov(Wavefront* w, bool wide, cudaStream_t st);
// Depth unit of the AOV buffer: the smallest power of two >= the largest distance from the eye to a corner of the scene
// bounds (in double), 1 when that distance is 0.
float aov_depth_unit(const float bounds[6], const float eye[3]);
// Device-to-device replica of a built scene (cudaMemcpyPeer of every table): what the other GPUs of a crt_group get
// instead of a second parse + build. Leaves `device` selected.
int clone_scene(const DeviceScene& src, int device, DeviceScene& dst);
// fixed point -> linear float mean and tone-mapped RGB8 (reference Render.cuh:348,350), on the device
int resolve_device(const long long* d_accum, uint32_t n_pixels, uint32_t spp, float* d_linear, uint8_t* d_rgb8, cudaStream_t st);
// AOV buffer -> d_out: albedo[3n], normal[3n], depth[n], coverage[n] (n = n_pixels), on the device
int resolve_aov_device(const long long* d_aov, uint32_t n_pixels, uint32_t spp, float depth_unit, float* d_out, cudaStream_t st);

}  // namespace crt
