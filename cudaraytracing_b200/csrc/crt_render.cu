// crt_render.cu — ray-batch kernels and the wavefront path tracer.
//
// Replaces the reference's single per-pixel megakernel (include/Render.cuh:330-354 view_render_kernel
// + cast_ray_v2 :199-328 + per-pixel global-memory stacks, DeviceStack.cuh) by a wavefront:
//     prepare -> generate -> extend -> [probe] -> shade -> shadow        (one iteration)
// over a fixed pool of in-flight paths that is refilled with new camera paths every iteration
// (path regeneration), with double-buffered compacted queues (warp-aggregated atomics), persistent
// warps that fetch 32 rays at a time, counter-based Philox draws keyed by (pixel, sample, bounce,
// dimension), and an order-independent fixed-point accumulation buffer.
// The estimator arithmetic mirrors oracle/orc_render.cpp operation by operation (-fmad=false).
#include "crt_gpu.h"
#include "crt_wide.cuh"

// __launch_bounds__ min blocks/SM of the traversal kernels. 8 caps the wide-node kernels at 64 registers (no spills; the
// compiler's own choice is 77-79 = 6 blocks): cornell-box +3 %, C5 (HBM-latency bound) 4793 -> 5394 Mrays/s (r01_s27).
#ifndef CRT_MINB
#define CRT_MINB 8
#endif

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <type_traits>
#include <vector>

namespace crt {

// =============================================================================================
// scene upload
// =============================================================================================
int clone_scene(const DeviceScene& src, int device, DeviceScene& dst) {
    CRT_CUDA(cudaSetDevice(device));
    dst = DeviceScene();
    static_cast<SceneInfo&>(dst) = src;                         // counts, flags, bounds
    dst.device = device;
    cudaError_t e = cudaSuccess;
    DeviceScene::for_each_table([&](auto table) {
        const auto& s = src.*table;
        auto& d = dst.*table;
        if (e != cudaSuccess || s.size() == 0) return;
        e = d.alloc(s.size());
        if (e == cudaSuccess) e = cudaMemcpyPeer(d.get(), device, s.get(), src.device, sizeof(*s.get()) * s.size());
    });
    CRT_CUDA(e);
    CRT_CUDA(cudaDeviceSynchronize());
    return CRT_OK;
}

static inline float bits_f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static uint32_t env_u32(const char* name, uint32_t dflt) {
    const char* v = getenv(name);
    if (!v || !*v) return dflt;
    return (uint32_t)strtoul(v, nullptr, 0);
}

int upload_scene(const HostScene& hs, uint32_t thresh_n, int builder, int device, DeviceScene& ds, float* build_ms) {
    CRT_CUDA(cudaSetDevice(device));
    ds = DeviceScene();
    ds.device = device;
    const size_t n = hs.n_tris();
    if (n > 0x7fffffffu / 4) { set_error("scene too large (more than 2^29 triangles)"); return CRT_ERR_INVALID; }
    // materials: (kd, ns) (ke, flags) (probe_dtheta, probe_dphi, probe_shin, 0) (ks, mis light-sampling density per area) (kd / pi, 0)
    std::vector<float4> mats(hs.mats.size() * 5);
    ds.has_specular = false;
    for (size_t m = 0; m < hs.mats.size(); ++m) {
        const HostMaterial& hm = hs.mats[m];
        uint32_t flags = (hm.has_emit ? 1u : 0u) | (hm.mode == 1 ? 2u : 0u);
        if (hm.mode == 1 && !hm.has_emit) ds.has_specular = true;
        const float kPiF = 3.14159265358979323846f;
        mats[5 * m + 0] = make_float4(hm.kd[0], hm.kd[1], hm.kd[2], hm.ns);
        mats[5 * m + 1] = make_float4(hm.ke[0], hm.ke[1], hm.ke[2], bits_f(flags));
        mats[5 * m + 2] = make_float4(hm.probe_dtheta, hm.probe_dphi, hm.probe_shin, 0.0f);
        mats[5 * m + 3] = make_float4(hm.ks[0], hm.ks[1], hm.ks[2], hm.pdf_area);
        mats[5 * m + 4] = make_float4(hm.kd[0] / kPiF, hm.kd[1] / kPiF, hm.kd[2] / kPiF, 0.0f);     // kd / pi (Render.cuh:259), one IEEE division each
    }
    // lights (DeviceLights.cuh:63-87): object table + flat triangle table
    std::vector<int4> lights;
    std::vector<float4> ltris;
    for (const HostLight& L : hs.lights) {
        int4 rec;
        rec.x = (int)(ltris.size() / 4);
        rec.y = (int)L.faces.size();
        uint32_t ab; memcpy(&ab, &L.area, 4);
        rec.z = (int)ab;
        rec.w = 0;
        lights.push_back(rec);
        for (int32_t f : L.faces) {
            const float* v = &hs.verts[9 * (size_t)f];
            const float* nn = &hs.normal[3 * (size_t)f];
            const HostMaterial& hm = hs.mats[hs.mat[f]];
            ltris.push_back(make_float4(v[0], v[1], v[2], hm.ke[0]));
            ltris.push_back(make_float4(v[3], v[4], v[5], hm.ke[1]));
            ltris.push_back(make_float4(v[6], v[7], v[8], hm.ke[2]));
            ltris.push_back(make_float4(nn[0], nn[1], nn[2], hm.pdf_area));
        }
    }
    ds.n_mats = (uint32_t)hs.mats.size();
    ds.n_lights = (uint32_t)lights.size();
    ds.n_light_tris = (uint32_t)(ltris.size() / 4);
    if (!mats.empty()) {
        CRT_CUDA(ds.mats.alloc(mats.size()));
        CRT_CUDA(cudaMemcpy(ds.mats.get(), mats.data(), sizeof(float4) * mats.size(), cudaMemcpyHostToDevice));
    }
    if (!lights.empty()) {
        CRT_CUDA(ds.lights.alloc(lights.size()));
        CRT_CUDA(cudaMemcpy(ds.lights.get(), lights.data(), sizeof(int4) * lights.size(), cudaMemcpyHostToDevice));
        CRT_CUDA(ds.light_tris.alloc(ltris.size()));
        CRT_CUDA(cudaMemcpy(ds.light_tris.get(), ltris.data(), sizeof(float4) * ltris.size(), cudaMemcpyHostToDevice));
        if (hs.light_cdf.size() != ltris.size() / 4) { set_error("light table out of date (finish_objects not called)"); return CRT_ERR_STATE; }
        CRT_CUDA(ds.light_cdf.alloc(hs.light_cdf.size()));
        CRT_CUDA(cudaMemcpy(ds.light_cdf.get(), hs.light_cdf.data(), sizeof(float) * hs.light_cdf.size(), cudaMemcpyHostToDevice));
    }
    // geometry in face order for the builder
    DevBuf<float> d_verts;
    DevBuf<float4> d_shade;
    if (n > 0) {
        std::vector<float4> shade(n);
        for (size_t t = 0; t < n; ++t)
            shade[t] = make_float4(hs.normal[3 * t], hs.normal[3 * t + 1], hs.normal[3 * t + 2], bits_f((uint32_t)hs.mat[t]));
        CRT_CUDA(d_verts.alloc(9 * n));
        CRT_CUDA(d_shade.alloc(n));
        cudaMemcpy(d_verts.get(), hs.verts.data(), sizeof(float) * 9 * n, cudaMemcpyHostToDevice);
        cudaMemcpy(d_shade.get(), shade.data(), sizeof(float4) * n, cudaMemcpyHostToDevice);
    }
    return build_bvh_device(ds, d_verts.get(), d_shade.get(), (uint32_t)n, thresh_n, builder, 0, build_ms);
}

// =============================================================================================
// node-layout dispatch: WIDE = false: 64-byte child-pair nodes, true: 80-byte 8-wide compressed nodes
// =============================================================================================
// GATED: the 8-wide walker takes its second step of a turn only with enough lanes (WideWalkerGated, crt_wide.cuh)
template <int MODE, bool WIDE, bool GATED = false, typename Load, typename Done>
CRT_DEV void trace_queue(const SceneView& sc, uint32_t n, uint32_t* fetch, Load load, Done done) {
    if (WIDE && GATED) trace_persistent_queue<MODE, WideWalkerGated>(sc, n, fetch, load, done);
    else if (WIDE) trace_persistent_queue<MODE, WideWalker>(sc, n, fetch, load, done);
    else trace_persistent_queue<MODE, PairWalker>(sc, n, fetch, load, done);
}
// with_layout(wide, f): f(std::true_type()) or f(std::false_type()), so that f can pass WIDE to a kernel as W.value
template <typename F>
static auto with_layout(bool wide, F&& f) { return wide ? f(std::true_type()) : f(std::false_type()); }
template <int MODE, bool WIDE>
CRT_DEV HitRec trace_one(const SceneView& sc, V3 o, V3 d, float tmax) {
    if (WIDE) return traverse_wide<MODE>(sc, o, d, tmax);
    return traverse<MODE>(sc, o, d, tmax);
}

// =============================================================================================
// ray batches
// =============================================================================================
template <int MODE, bool WIDE>
__global__ void __launch_bounds__(128, CRT_MINB) k_trace_batch(SceneView sc, const float4* __restrict__ rays, uint32_t n,
                                                     float* __restrict__ t_out, int* __restrict__ face_out,
                                                     uint32_t* __restrict__ fetch) {
    trace_queue<MODE, WIDE, MODE == 1>(
        sc, n, fetch,
        [&](uint32_t i, V3& o, V3& d, float& tmax) {
            const float4 ro = __ldg(rays + 2 * (size_t)i), rd = __ldg(rays + 2 * (size_t)i + 1);
            o = mk3(ro); d = mk3(rd); tmax = ro.w;
            return true;
        },
        [&](uint32_t i, const HitRec& h) {
            if (t_out) t_out[i] = h.t;
            if (face_out) face_out[i] = h.face;
        });
}

static int g_num_sms = 0;
static int num_sms() {
    if (g_num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (g_num_sms <= 0) g_num_sms = 148;
    }
    return g_num_sms;
}

// ---- batch context ------------------------------------------------------------------------------
struct RayBatcher {
    int device = 0;
    int blocks = 0;
    DevBuf<uint32_t> fetch;                     // two queue counters, 128 bytes apart (one per pipeline slot)
    bool chunk_from_env = false;
    Event ev_a[2], ev_b[2], ev_done[2];
    Stream st[2];
    // host-buffer path, allocated on first use
    uint64_t chunk = 0;                         // rays per chunk
    DevBuf<float4> d_rays[2];
    DevBuf<float> d_t[2];
    DevBuf<int> d_face[2];
    Pinned<float4> h_rays[2];                   // pinned staging for pageable callers
    Pinned<float> h_t[2];
    Pinned<int> h_face[2];
    // CRT_RAY_SORTED, allocated on first use and grown: keys / permutation (ping-pong), the ordered copy of the rays and of the hits
    struct SortBufs {
        uint64_t cap = 0;
        DevBuf<uint64_t> k0, k1;
        DevBuf<uint32_t> v0, v1, ghist, scratch;
        DevBuf<float4> rays;
        DevBuf<float> t;
        DevBuf<int> face;
    } sort[2];
};
void StateDelete::operator()(RayBatcher* b) const { delete b; }

int ray_batcher_create(const DeviceScene& ds, RayBatcherPtr& out) {
    RayBatcherPtr b(new RayBatcher());
    b->device = ds.device;
    CRT_CUDA(b->fetch.alloc(64));
    for (int k = 0; k < 2; ++k) {
        CRT_CUDA(create(b->ev_a[k]));
        CRT_CUDA(create(b->ev_b[k]));
        CRT_CUDA(create(b->ev_done[k], cudaEventDisableTiming));
        CRT_CUDA(create(b->st[k]));
    }
    int occ = 0;
    CRT_CUDA(with_layout(ds.wide, [&](auto W) { return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_trace_batch<0, W.value>, 128, 0); }));
    b->blocks = num_sms() * std::max(occ, 1);
    out = std::move(b);
    return CRT_OK;
}

// ---- CRT_RAY_SORTED: "warp-coherent ray sorting" as an option of the batch calls --------------------------------------------------
// Key of a ray: Morton code of its origin's cell on a 128^3 grid over the scene's bounds, then the direction octant (24 bits, three
// passes of the builder's radix sort); the rays are gathered in that order, traced, and the hits scattered back to the caller's order.
// Off by default because it does not pay here: a PERFECT order, for free, makes the trace of C5 6-8 % faster (the kernels wait on
// instruction issue, not on memory coherence), and the sort costs more than that (profiles/r02_late_levers.md).
static constexpr int kRaySortCellBits = 7;
CRT_DEV uint32_t spread3(uint32_t x) {                   // 0b abcdefg -> 0b a00b00c00d00e00f00g
    x &= 0x3ffu;
    x = (x | (x << 16)) & 0x030000ffu;
    x = (x | (x << 8)) & 0x0300f00fu;
    x = (x | (x << 4)) & 0x030c30c3u;
    x = (x | (x << 2)) & 0x09249249u;
    return x;
}
__global__ void k_ray_keys(const float4* __restrict__ rays, uint32_t n, float lox, float loy, float loz, float sx, float sy, float sz,
                           uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 o = __ldg(rays + 2 * (size_t)i), d = __ldg(rays + 2 * (size_t)i + 1);
    const int hi = (1 << kRaySortCellBits) - 1;
    const int cx = min(max((int)((o.x - lox) * sx), 0), hi), cy = min(max((int)((o.y - loy) * sy), 0), hi),
              cz = min(max((int)((o.z - loz) * sz), 0), hi);
    const uint32_t cell = spread3((uint32_t)cx) | (spread3((uint32_t)cy) << 1) | (spread3((uint32_t)cz) << 2);
    const uint32_t oct = (d.x < 0.0f ? 1u : 0u) | (d.y < 0.0f ? 2u : 0u) | (d.z < 0.0f ? 4u : 0u);
    keys[i] = ((uint64_t)cell << 3) | oct;
    vals[i] = i;
}
__global__ void k_gather_rays(const float4* __restrict__ rays, const uint32_t* __restrict__ perm, uint32_t n, float4* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t j = perm[i];
    out[2 * (size_t)i] = __ldg(rays + 2 * (size_t)j);
    out[2 * (size_t)i + 1] = __ldg(rays + 2 * (size_t)j + 1);
}
__global__ void k_scatter_hits(const uint32_t* __restrict__ perm, uint32_t n, const float* __restrict__ t_in, const int* __restrict__ f_in,
                               float* __restrict__ t_out, int* __restrict__ f_out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t j = perm[i];
    if (t_out) t_out[j] = t_in[i];
    if (f_out) f_out[j] = f_in[i];
}
static int ensure_sort_bufs(RayBatcher::SortBufs& sb, uint64_t cnt) {
    if (sb.cap >= cnt) return CRT_OK;
    sb = RayBatcher::SortBufs();
    const uint32_t n = (uint32_t)cnt;
    CRT_CUDA(sb.k0.alloc(cnt));
    CRT_CUDA(sb.k1.alloc(cnt));
    CRT_CUDA(sb.v0.alloc(cnt));
    CRT_CUDA(sb.v1.alloc(cnt));
    CRT_CUDA(sb.ghist.alloc(radix_sort_hist_words(n)));
    CRT_CUDA(sb.scratch.alloc(radix_sort_scratch_words(n)));
    CRT_CUDA(sb.rays.alloc(2 * cnt));
    CRT_CUDA(sb.t.alloc(cnt));
    CRT_CUDA(sb.face.alloc(cnt));
    sb.cap = cnt;
    return CRT_OK;
}

static void launch_trace_kernel(const RayBatcher* b, const DeviceScene& ds, const float4* d_rays, uint32_t cnt, int mode, float* t_o, int* f_o,
                                uint32_t* fetch, cudaStream_t st) {
    cudaMemsetAsync(fetch, 0, sizeof(uint32_t), st);
    with_layout(ds.wide, [&](auto W) {
        if (mode == CRT_RAY_CLOSEST) k_trace_batch<0, W.value><<<b->blocks, 128, 0, st>>>(ds.view(), d_rays, cnt, t_o, f_o, fetch);
        else k_trace_batch<1, W.value><<<b->blocks, 128, 0, st>>>(ds.view(), d_rays, cnt, t_o, f_o, fetch);
    });
}

// slot: which of the batcher's two sets of ordering buffers (one per pipeline stream)
static int launch_trace_batch(RayBatcher* b, const DeviceScene& ds, const float4* d_rays, uint32_t cnt, int mode, float* t_o, int* f_o,
                              uint32_t* fetch, cudaStream_t st, int slot = 0) {
    const int kind = mode & ~CRT_RAY_SORTED;
    if (!(mode & CRT_RAY_SORTED) || cnt == 0) {
        launch_trace_kernel(b, ds, d_rays, cnt, kind, t_o, f_o, fetch, st);
        return CRT_OK;
    }
    RayBatcher::SortBufs& sb = b->sort[slot];
    int rc = ensure_sort_bufs(sb, cnt);
    if (rc != CRT_OK) return rc;
    const float cells = (float)(1 << kRaySortCellBits);
    float sc[3];
    for (int a = 0; a < 3; ++a) {
        const float ext = ds.bounds[3 + a] - ds.bounds[a];
        sc[a] = ext > 0.0f ? cells / ext : 0.0f;
    }
    const uint32_t nb = (cnt + 255) / 256;
    k_ray_keys<<<nb, 256, 0, st>>>(d_rays, cnt, ds.bounds[0], ds.bounds[1], ds.bounds[2], sc[0], sc[1], sc[2], sb.k0.get(), sb.v0.get());
    uint64_t* ks = nullptr;
    uint32_t* perm = nullptr;
    CRT_CUDA(radix_sort_pairs(sb.k0.get(), sb.k1.get(), sb.v0.get(), sb.v1.get(), cnt, (3 * kRaySortCellBits + 3 + 7) / 8, sb.ghist.get(),
                              sb.scratch.get(), st, &ks, &perm));
    k_gather_rays<<<nb, 256, 0, st>>>(d_rays, perm, cnt, sb.rays.get());
    launch_trace_kernel(b, ds, sb.rays.get(), cnt, kind, sb.t.get(), sb.face.get(), fetch, st);
    k_scatter_hits<<<nb, 256, 0, st>>>(perm, cnt, sb.t.get(), sb.face.get(), t_o, f_o);
    return CRT_OK;
}

int trace_rays_device(RayBatcher* b, const DeviceScene& ds, const float4* d_rays, uint64_t n, int mode, float* d_t, int* d_face,
                      cudaStream_t st, float* kernel_ms) {
    const uint64_t chunk = (mode & CRT_RAY_SORTED) ? 1ull << 27 : 1ull << 30;   // queue indices are 32-bit; ordering buffers are ~65 B per ray
    float ms_total = 0;
    for (uint64_t off = 0; off < n; off += chunk) {
        const uint32_t cnt = (uint32_t)std::min<uint64_t>(chunk, n - off);
        CRT_CUDA(cudaEventRecord(b->ev_a[0].get(), st));
        int rc = launch_trace_batch(b, ds, d_rays + 2 * off, cnt, mode, d_t ? d_t + off : nullptr, d_face ? d_face + off : nullptr, b->fetch.get(), st);
        if (rc != CRT_OK) return rc;
        CRT_CUDA(cudaGetLastError());
        CRT_CUDA(cudaEventRecord(b->ev_b[0].get(), st));
        CRT_CUDA(cudaStreamSynchronize(st));
        float ms = 0;
        CRT_CUDA(cudaEventElapsedTime(&ms, b->ev_a[0].get(), b->ev_b[0].get()));
        ms_total += ms;
    }
    if (kernel_ms) *kernel_ms = ms_total;
    return CRT_OK;
}

static bool is_page_locked(const void* p) {
    if (!p) return true;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// memcpy on all host threads (a pageable 128 MB chunk at one thread's ~10 GB/s would be slower than the PCIe link)
static void parallel_memcpy(void* dst, const void* src, size_t bytes) {
    unsigned T = std::thread::hardware_concurrency();
    T = std::max(1u, std::min(T, 16u));
    if (bytes < (8u << 20) || T == 1) { memcpy(dst, src, bytes); return; }
    std::vector<std::thread> th;
    const size_t per = ((bytes / T) + 4095) & ~(size_t)4095;
    for (unsigned k = 1; k < T; ++k) {
        const size_t o = per * k;
        if (o >= bytes) break;
        th.emplace_back([=] { memcpy((char*)dst + o, (const char*)src + o, std::min(per, bytes - o)); });
    }
    memcpy(dst, src, std::min(per, bytes));
    for (auto& t : th) t.join();
}

int trace_rays_host(RayBatcher* b, const DeviceScene& ds, const float* rays, uint64_t n, int mode, float* t_out, int32_t* face_out,
                    float* kernel_ms) {
    if (b->chunk == 0) {
        // 4 Mi rays (128 MB in, 32 MB out per chunk) suit the staged path (host threads copy a chunk while the previous one is on
        // the link: 721 Mrays/s pageable, 674 at 2 Mi); page-locked caller buffers go in halves of that - nothing is staged, and
        // the end of the pipeline (trace + results of the last chunk, not overlapped) is shorter: 1,616 vs 1,547 Mrays/s for 20 M
        // rays, 1,676 vs 1,659 for 100 M (profiles/r02_s33_e2e_chunks.log). CRT_BATCH_CHUNK sets one size for both.
        b->chunk_from_env = getenv("CRT_BATCH_CHUNK") != nullptr;
        uint64_t chunk = env_u32("CRT_BATCH_CHUNK", 4u << 20);
        chunk = std::max<uint64_t>(1024, std::min<uint64_t>(chunk, 1ull << 28));
        for (int k = 0; k < 2; ++k) {
            CRT_CUDA(b->d_rays[k].alloc(2 * chunk));
            CRT_CUDA(b->d_t[k].alloc(chunk));
            CRT_CUDA(b->d_face[k].alloc(chunk));
        }
        b->chunk = chunk;
    }
    const bool in_place_in = is_page_locked(rays), in_place_t = is_page_locked(t_out), in_place_f = is_page_locked(face_out);
    const uint64_t C = in_place_in && !b->chunk_from_env ? b->chunk / 2 : b->chunk;
    for (int k = 0; k < 2; ++k) {
        if (!in_place_in && !b->h_rays[k]) CRT_CUDA(pinned_alloc(b->h_rays[k], 2 * b->chunk));
        if (t_out && !in_place_t && !b->h_t[k]) CRT_CUDA(pinned_alloc(b->h_t[k], b->chunk));
        if (face_out && !in_place_f && !b->h_face[k]) CRT_CUDA(pinned_alloc(b->h_face[k], b->chunk));
    }
    const uint64_t n_chunks = (n + C - 1) / C;
    float ms_total = 0;
    auto retire = [&](uint64_t k) -> int {                // chunk k has left the GPU: kernel time, staged results to the caller
        const int s = (int)(k & 1);
        const uint64_t off = k * C, cnt = std::min<uint64_t>(C, n - off);
        CRT_CUDA(cudaEventSynchronize(b->ev_done[s].get()));
        float ms = 0;
        CRT_CUDA(cudaEventElapsedTime(&ms, b->ev_a[s].get(), b->ev_b[s].get()));
        ms_total += ms;
        if (t_out && !in_place_t) parallel_memcpy(t_out + off, b->h_t[s].get(), sizeof(float) * cnt);
        if (face_out && !in_place_f) parallel_memcpy(face_out + off, b->h_face[s].get(), sizeof(int) * cnt);
        return CRT_OK;
    };
    for (uint64_t k = 0; k < n_chunks; ++k) {
        const int s = (int)(k & 1);
        const uint64_t off = k * C, cnt = std::min<uint64_t>(C, n - off);
        cudaStream_t sk = b->st[s].get();
        float* d_t = b->d_t[s].get();
        int* d_face = b->d_face[s].get();
        if (k >= 2) { int rc = retire(k - 2); if (rc != CRT_OK) return rc; }      // the slot's buffers are free again
        const float* src = rays + 8 * off;
        if (!in_place_in) { parallel_memcpy(b->h_rays[s].get(), src, sizeof(float) * 8 * cnt); src = (const float*)b->h_rays[s].get(); }
        CRT_CUDA(cudaMemcpyAsync(b->d_rays[s].get(), src, sizeof(float) * 8 * cnt, cudaMemcpyHostToDevice, sk));
        CRT_CUDA(cudaEventRecord(b->ev_a[s].get(), sk));
        { int rc = launch_trace_batch(b, ds, b->d_rays[s].get(), (uint32_t)cnt, mode, d_t, d_face, b->fetch.get() + 32 * s, sk, s); if (rc != CRT_OK) return rc; }
        CRT_CUDA(cudaGetLastError());
        CRT_CUDA(cudaEventRecord(b->ev_b[s].get(), sk));
        if (t_out) CRT_CUDA(cudaMemcpyAsync(in_place_t ? t_out + off : b->h_t[s].get(), d_t, sizeof(float) * cnt, cudaMemcpyDeviceToHost, sk));
        if (face_out) CRT_CUDA(cudaMemcpyAsync(in_place_f ? face_out + off : b->h_face[s].get(), d_face, sizeof(int) * cnt, cudaMemcpyDeviceToHost, sk));
        CRT_CUDA(cudaEventRecord(b->ev_done[s].get(), sk));
    }
    for (uint64_t k = n_chunks >= 2 ? n_chunks - 2 : 0; k < n_chunks; ++k) { int rc = retire(k); if (rc != CRT_OK) return rc; }
    if (kernel_ms) *kernel_ms = ms_total;
    return CRT_OK;
}

// C5 input: see crt_random_rays_device in include/crt.h (numpy statement: tools/synthetic.py:random_rays)
__global__ void k_random_rays(float4* __restrict__ rays, unsigned long long n, unsigned long long start, float lox, float loy,
                              float loz, float hix, float hiy, float hiz, float diag, uint32_t key, int any_hit) {
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long idx = start + i;
        const uint32_t c0 = (uint32_t)idx, c1 = (uint32_t)(idx >> 32);
        const uint4 a = philox4x32_10(make_uint4(c0, c1, 0u, 0u), key, 0u);
        const uint4 b = philox4x32_10(make_uint4(c0, c1, 1u, 0u), key, 0u);
        const float ox = lox + (hix - lox) * u01(a.x), oy = loy + (hiy - loy) * u01(a.y), oz = loz + (hiz - loz) * u01(a.z);
        const float z = 1.0f - 2.0f * u01(a.w);
        const float rad = sqrtf(fmaxf(0.0f, 1.0f - z * z));
        float sn, cs;
        sincos_2pi(u01(b.x), &sn, &cs);
        rays[2 * i] = make_float4(ox, oy, oz, any_hit ? u01(b.y) * diag : FLT_MAX);
        rays[2 * i + 1] = make_float4(rad * cs, rad * sn, z, 0.0f);
    }
}

int random_rays_device(const DeviceScene& ds, float4* d_rays, uint64_t n, uint64_t start, uint32_t key, int any_hit, cudaStream_t st) {
    if (n == 0) return CRT_OK;
    const float* b = ds.bounds;
    double d2 = 0;
    for (int k = 0; k < 3; ++k) { double e = (double)(b[3 + k] - b[k]); d2 += e * e; }
    k_random_rays<<<num_sms() * 8, 256, 0, st>>>(d_rays, n, start, b[0], b[1], b[2], b[3], b[4], b[5], (float)sqrt(d2), key, any_hit);
    CRT_CUDA(cudaGetLastError());
    return CRT_OK;
}

// =============================================================================================
// wavefront state
// =============================================================================================
static constexpr int kShadowRegions = 8;
struct Counters {
    unsigned long long work_next, work_end, gen_work0;
    unsigned long long stat_extend, stat_shadow, stat_probe;
    uint32_t n_cur, n_probe_cur, n_probe_next;
    uint32_t gen_base, gen_count;
    uint32_t gen_tile, gen_jj0;        // tile order: tile and offset inside it of the first work item k_generate starts (k_prepare)
    uint32_t iterations;
    uint32_t tail_n, fetch_tail;       // paths handed to k_tail by the last k_prepare (0: none)
    uint32_t fetch_probe;
    // the words every warp of a kernel adds to, each alone in a 128-byte line: same-address atomics serialise in one L2 slice
    // (with n_next and n_shadow in one 32-byte sector the shade stage took 24.7 - 34.1 ms for the same work depending on the
    // box, profiles/r01_s35.md).
    alignas(128) uint32_t n_next;
    // The shadow queue is cut into kShadowRegions regions with a counter each (a warp of k_shade appends to region
    // global-warp-id % kShadowRegions): two appends per vertex and warp on ONE counter were ~1 atomic per ns, the rate one
    // address takes - once the vertex arithmetic had lost a third of its instructions, k_shade waited on exactly that
    // (24.7 % of its stall samples, box-dependent 19 - 30 ms per 1080p spp-128 frame, profiles/r02_s20.md).
    // [parity][region]: k_shadow of iteration k overlaps k_prepare .. k_extend of k + 1.
    struct alignas(128) Line { uint32_t v; };
    Line n_shadow[2][kShadowRegions];
    alignas(128) uint32_t fetch_extend;
    alignas(128) uint32_t fetch_shadow[2];
    alignas(128) uint32_t pad_;
};
struct HostStatus { volatile uint32_t done; volatile uint32_t n_cur; volatile unsigned long long work_next; };

struct RenderParamsDev {
    float eye[3];
    float M[9];
    float tan_half;
    uint32_t width, height;
    unsigned long long n_pixels;
    uint32_t s_begin;
    float two_pi_over_p_rr;                     // 2 pi / P_RR, divided once on the host (Render.cuh:288-293)
    // Order in which the work items of this run_view are started (any order gives the same buffer). tile_px > 0: the
    // range is whole samples [tile_s0, tile_s0 + tile_S) and is walked tile by tile - all its samples of pixels
    // [0, tile_px), then of the next tile_px pixels ... - so that the part of the accumulation buffer the paths in flight
    // add to (24 B per pixel) stays L2-resident on frames whose whole buffer is not (4K: 199 MB against 126 MB of L2).
    uint32_t tile_px, tile_s0, tile_S;
    uint32_t tile_fast;                         // per_tile = tile_px * tile_S fits 31 bits and is >= the pool: k_generate's 32-bit path
    unsigned long long w_begin;
    float p_rr;
    int light_sample_n;
    uint32_t seed;
    int max_vertices;
};

static constexpr uint32_t kFlagProbe = 0x100u;
static constexpr uint32_t kTailDefault = 1u << 19;   // paths alive when k_tail takes over (CRT_TAIL overrides, 0 = never)

struct WfRun {                      // the run_view in flight on a Wavefront (wavefront_begin / step / finish)
    bool active = false;
    const DeviceScene* ds = nullptr;
    RenderSettings rs;
    RenderParamsDev p;
    SceneView sv;
    cudaStream_t st = nullptr;
    bool wide = false, mis = false, overlap = false, timeline = false;
    uint32_t tail_max = 0, it = 0;
    uint64_t launches = 0;
    unsigned long long w_begin = 0, per_tile32 = 0;       // per_tile32: work items per tile when k_generate takes its 32-bit path, else 0
    float ms_stage[5] = {0, 0, 0, 0, 0};
    Event se[6];
    std::vector<std::pair<const char*, Event>> tl;            // CRT_TIMELINE
    void mark(const char* what, cudaStream_t s) {
        if (!timeline) return;
        Event e;
        create(e);
        cudaEventRecord(e.get(), s);
        tl.emplace_back(what, std::move(e));
    }
};

// The path queue of one iteration parity: o (origin, pixel), d (direction, sample), T (throughput, meta), pdf (mis: density of
// the BSDF sample that produced the ray) and, in scenes with SPECULAR materials, the pending probe rays (o, d, weight) and the
// list of the paths that have one. The kernels take these as separate __restrict__ pointer parameters: a pointer in a struct
// parameter, __restrict__ or not, loses the read-only loads (LDG.E.128.CONSTANT) of k_extend, k_shade, k_shadow and k_tail.
struct PathQueue {
    DevBuf<float4> o, d, T;
    DevBuf<float> pdf;
    DevBuf<float4> pr_o, pr_d, pr_w;
    DevBuf<uint32_t> pr_list;
};
// shadow rays: kShadowRegions regions of region_cap rays; o (origin, tmax), d (direction, pixel), c (contribution)
struct ShadowQueue {
    DevBuf<float4> o, d, c;
    uint32_t region_cap = 0;
};
struct PathPool {                  // everything sized by the number of paths in flight
    uint32_t pool = 0;             // path slots per queue
    uint32_t shadow_cap = 0;
    PathQueue q[2];
    DevBuf<float> hit_t;
    DevBuf<int> hit_slot, pr_hit;
    ShadowQueue sh;
};

struct Wavefront {
    WfRun run;
    uint32_t width = 0, height = 0;
    bool has_probe = false;
    PathPool paths;
    DevBuf<long long> accum;
    DevBuf<Counters> counters;
    Pinned<HostStatus> status_host;
    HostStatus* status_dev = nullptr;
    Event ev[4];
    Event ev_begin, ev_end;
    Stream st_shadow;                                     // k_shadow of iteration k runs here, beside k_prepare .. k_extend of k + 1
    Event ev_shaded, ev_shadowed;
    int grid_trace = 0, grid_shade = 0, grid_tail = 0;
};
void StateDelete::operator()(Wavefront* w) const { delete w; }

// =============================================================================================
// kernels
// =============================================================================================
__global__ void k_prepare(Counters* c, uint32_t pool, uint32_t tail_max, HostStatus* status, int par, unsigned long long per_tile,
                          unsigned long long w_begin) {
    for (int r = 0; r < kShadowRegions; ++r) {    // the shadow rays of iteration k - 2, traced long ago
        c->stat_shadow += c->n_shadow[par][r].v;
        c->n_shadow[par][r].v = 0;
    }
    uint32_t n_cur = c->n_next;
    uint32_t n_probe = c->n_probe_next;
    c->n_next = 0;
    c->n_probe_next = 0;
    unsigned long long remaining = c->work_end - c->work_next;
    uint32_t room = pool - n_cur;
    uint32_t n_new = remaining < (unsigned long long)room ? (uint32_t)remaining : room;
    c->gen_base = n_cur;
    c->gen_count = n_new;
    c->gen_work0 = c->work_next;
    if (per_tile) {                    // the one 64-bit division of the tile order, here instead of three per generated path
        const unsigned long long j = c->work_next - w_begin;
        c->gen_tile = (uint32_t)(j / per_tile);
        c->gen_jj0 = (uint32_t)(j - (unsigned long long)c->gen_tile * per_tile);
    }
    n_cur += n_new;
    c->work_next += n_new;
    c->fetch_extend = c->fetch_shadow[par] = c->fetch_probe = c->fetch_tail = 0;
    c->iterations += n_cur ? 1u : 0u;
    // tail: every camera path has been started and few paths are alive -> k_tail finishes them
    const bool tail = remaining == 0 && n_cur > 0 && n_cur <= tail_max;
    c->tail_n = tail ? n_cur : 0u;
    if (tail) n_cur = 0, n_probe = 0;
    c->n_cur = n_cur;
    c->n_probe_cur = n_probe;
    c->stat_extend += n_cur;
    status->n_cur = n_cur;
    status->work_next = c->work_next;
    if (n_cur == 0) status->done = 1;          // read by the host after this iteration's kernels have finished
    __threadfence_system();
}

// Primary rays: reference Render.cuh:338-347 + Ray.cuh:12-15. Work item w -> (sample, pixel) with
// consecutive items on consecutive pixels of one sample index (coherent warps, distinct pixels).
__global__ void __launch_bounds__(256) k_generate(const Counters* __restrict__ c, RenderParamsDev p, float4* __restrict__ q_o,
                                                  float4* __restrict__ q_d, float4* __restrict__ q_T, float* __restrict__ q_pdf) {
    const uint32_t count = c->gen_count, base = c->gen_base;
    const unsigned long long w0 = c->gen_work0;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < count; k += gridDim.x * blockDim.x) {
        unsigned long long w = w0 + k;
        // (an 8x4-tile order of the pixels inside a sample, alone or in blocks of 4-16 tiles, changes nothing measurable:
        //  profiles/r01_s21.md - the camera rays are a third of the extend rays and the cheapest ones)
        uint32_t pixel, sample;
        if (p.tile_fast) {
            // 32-bit arithmetic: k_prepare has located the first work item; a launch spans at most two tiles (per_tile >= pool)
            const uint32_t per_tile = p.tile_px * p.tile_S;
            uint32_t t = c->gen_tile, jj = c->gen_jj0 + k;
            if (jj >= per_tile) { jj -= per_tile; ++t; }
            const uint32_t first = t * p.tile_px;
            const uint32_t px = (uint32_t)min((unsigned long long)p.tile_px, p.n_pixels - first);
            sample = p.tile_s0 + jj / px;
            pixel = first + jj % px;
        } else if (p.tile_px) {
            const unsigned long long j = w - p.w_begin, per_tile = (unsigned long long)p.tile_px * p.tile_S;
            const uint32_t t = (uint32_t)(j / per_tile);
            const unsigned long long jj = j - (unsigned long long)t * per_tile;
            const uint32_t first = t * p.tile_px;
            const uint32_t px = (uint32_t)min((unsigned long long)p.tile_px, p.n_pixels - first);
            sample = p.tile_s0 + (uint32_t)(jj / px);
            pixel = first + (uint32_t)(jj % px);
        } else {
            pixel = (uint32_t)(w % p.n_pixels);
            sample = p.s_begin + (uint32_t)(w / p.n_pixels);
        }
        uint32_t i = pixel % p.width, j = pixel / p.width;
        uint4 r = draw(pixel, sample, kCameraBounce, 0, p.seed);
        float u1 = u01(r.x), u2 = u01(r.y);
        float ar = (float)p.width / (float)p.height;
        float x = (2.0f * ((float)i + u1) / (float)p.width - 1.0f) * p.tan_half * ar;
        float y = (1.0f - 2.0f * ((float)j + u2) / (float)p.height) * p.tan_half;
        V3 dc = normalize(mk3(-x, y, 1.0f));
        V3 d = mk3(dot(mk3(p.M[0], p.M[1], p.M[2]), dc), dot(mk3(p.M[3], p.M[4], p.M[5]), dc), dot(mk3(p.M[6], p.M[7], p.M[8]), dc));
        d = normalize(d);
        q_o[base + k] = make_float4(p.eye[0], p.eye[1], p.eye[2], __uint_as_float(pixel));
        q_d[base + k] = make_float4(d.x, d.y, d.z, __uint_as_float(sample));
        q_T[base + k] = make_float4(1.0f, 1.0f, 1.0f, __uint_as_float(0u));
        if (q_pdf) q_pdf[base + k] = 0.0f;
    }
}

template <bool WIDE>
__global__ void __launch_bounds__(128, CRT_MINB) k_extend(SceneView sc, Counters* c, const float4* __restrict__ q_o,
                                                const float4* __restrict__ q_d, float* __restrict__ hit_t,
                                                int* __restrict__ hit_slot) {
    trace_queue<0, WIDE>(
        sc, c->n_cur, &c->fetch_extend,
        [&](uint32_t i, V3& o, V3& d, float& tmax) { o = mk3(q_o[i]); d = mk3(q_d[i]); tmax = FLT_MAX; return true; },
        [&](uint32_t i, const HitRec& h) { hit_t[i] = h.t; hit_slot[i] = h.slot; });
}

// SPECULAR probe rays (reference Render.cuh:303): traced only when the continuation ray hit.
template <bool WIDE>
__global__ void __launch_bounds__(128, CRT_MINB) k_probe(SceneView sc, Counters* c, const uint32_t* __restrict__ list,
                                               const float4* __restrict__ pr_o, const float4* __restrict__ pr_d,
                                               const int* __restrict__ hit_slot, int* __restrict__ pr_hit) {
    unsigned long long traced = 0;
    trace_queue<0, WIDE>(
        sc, c->n_probe_cur, &c->fetch_probe,
        [&](uint32_t k, V3& o, V3& d, float& tmax) {
            const uint32_t i = list[k];
            if (hit_slot[i] < 0) return false;            // continuation missed: the probe is not traced
            o = mk3(pr_o[i]); d = mk3(pr_d[i]); tmax = FLT_MAX; traced++;
            return true;
        },
        [&](uint32_t k, const HitRec& h) { pr_hit[list[k]] = h.slot; });
    const int lane = threadIdx.x & 31;
    for (int o = 16; o > 0; o >>= 1) traced += __shfl_down_sync(0xffffffffu, traced, o);
    if (lane == 0 && traced) atomicAdd(&c->stat_probe, traced);
}

// Global.h:35-50
CRT_DEV V3 to_world(V3 a, V3 N) {
    V3 C;
    if (fabsf(N.x) > fabsf(N.y)) {
        float inv = 1.0f / sqrtf(fmaf(N.z, N.z, N.x * N.x));
        C = mk3(N.z * inv, 0.0f, -N.x * inv);
    } else {
        float inv = 1.0f / sqrtf(fmaf(N.z, N.z, N.y * N.y));
        C = mk3(0.0f, N.z * inv, -N.y * inv);
    }
    V3 B = cross(C, N);
    return (a.x * B + a.y * C) + a.z * N;
}
// Global.h:57-66
CRT_DEV V3 sample_hemisphere(V3 N, float u1, float u2) {
    float z = fabsf(1.0f - 2.0f * u1);
    float r = sqrtf(1.0f - z * z);
    float sn, cs;
    sincos_2pi(u2, &sn, &cs);
    return to_world(mk3(r * cs, r * sn, z), N);
}
// Global.h:68-94 by angle addition
CRT_DEV V3 sample_probe_lobe(V3 out, float dtheta, float dphi, float u1, float u2) {
    float eta1 = 2.0f * u1 - 1.0f, eta2 = 2.0f * u2 - 1.0f;
    float r = length(out);
    float ct0 = out.z / r;
    ct0 = fminf(1.0f, fmaxf(-1.0f, ct0));
    float st0 = sqrtf(fmaxf(0.0f, 1.0f - ct0 * ct0));
    float cp0, sp0;
    if (fabsf(out.x) < 1e-5f) {
        cp0 = 0.0f;
        sp0 = out.y > 0.0f ? 1.0f : -1.0f;
    } else {
        float rho = sqrtf(fmaf(out.y, out.y, out.x * out.x));
        cp0 = out.x / rho;
        sp0 = out.y / rho;
    }
    float sa, ca, sb, cb;
    sincos_rad(eta1 * dtheta, &sa, &ca);
    sincos_rad(eta2 * dphi, &sb, &cb);
    float st = fmaf(st0, ca, ct0 * sa), ct = fmaf(ct0, ca, -(st0 * sa));
    float sp = fmaf(sp0, cb, cp0 * sb), cp = fmaf(cp0, cb, -(sp0 * sb));
    return mk3(st * cp, st * sp, ct);
}

// compat estimator, one path vertex: the forward form of cast_ray_v2 (reference Render.cuh:199-328);
// statement shared with oracle/orc_render.cpp path_compat. Used by the wavefront shade kernel (shadow
// rays and the continuation go to queues) and by the tail kernel (traced in place).
//   shadow(needs_trace, pos, t_to_light, dir, contrib): called for every light sample by every lane that
//   reached this vertex; when needs_trace it must trace the any-hit ray and add contrib if unblocked.
// Returns true when the path continues; then nx / npr hold the next path state (npr only if
// nx.meta has kFlagProbe).
struct PathState { V3 o, d, T; uint32_t pixel, sample, meta; float pdf; };   // pdf: mis only (density of the last BSDF sample)
struct ProbeState { V3 o, d, w; };

template <typename ShadowFn>
CRT_DEV bool shade_vertex_compat(const SceneView& sc, const RenderParamsDev& p, const PathState& ps, float t, int slot,
                                 long long* __restrict__ accum, ShadowFn&& shadow, PathState& nx, ProbeState& npr) {
    const uint32_t pixel = ps.pixel, sample = ps.sample, bounce = ps.meta & 0xffu;
    const float lsn_f = (float)p.light_sample_n;
    const float4 sh = __ldg(sc.tri_shade + slot);
    const uint32_t mat = __float_as_uint(sh.w);
    const float4 m0 = __ldg(sc.mats + 5 * mat + 0), m1 = __ldg(sc.mats + 5 * mat + 1);
    const uint32_t mflags = __float_as_uint(m1.w);
    if (mflags & 1u) {                                          // emissive vertex, :210,249-255
        if (bounce == 0) accum_add(accum, pixel, mk3(m1));
        return false;
    }
    const V3 o = ps.o, d = ps.d, T = ps.T;
    const V3 pos = o + t * d;                                   // DeviceTriangle.cuh:50
    const V3 nrm = mk3(sh);
    const V3 f_r = mk3(__ldg(sc.mats + 5 * mat + 4));           // kd / pi, :259 (divided once per material on the host)
    const V3 Tf = cmul(T, f_r);
    // next-event estimation, :262-286
    for (int li = 0; li < sc.n_lights; ++li) {
        const int4 L = __ldg(sc.lights + li);
        const float area = __int_as_float(L.z);
        for (int sj = 0; sj < p.light_sample_n; ++sj) {
            uint4 q = draw(pixel, sample, bounce, 2u + (uint32_t)(li * p.light_sample_n + sj), p.seed);
            const float4* lt = sc.light_tris + 4 * (size_t)(L.x + (int)(q.x % (uint32_t)L.y));   // DeviceLights.cuh:35
            const float4 a = __ldg(lt), b = __ldg(lt + 1), cc = __ldg(lt + 2), ln = __ldg(lt + 3);
            float alpha = u01(q.y);                             // DeviceTriangle.cuh:69-72
            float beta = u01(q.z) * (1.0f - alpha);
            float gamma = (1.0f - alpha) - beta;
            V3 lp = (alpha * mk3(a) + beta * mk3(b)) + gamma * mk3(cc);
            V3 dist = lp - pos;
            V3 dir = normalize(dist);                           // the reference's operation sequence: its shadow test is rounding-dependent
            float d1 = length(dist);
            float d2 = d1 * d1;
            float cos1 = fmaxf(0.0f, dot(dir, nrm));
            float cos2 = fmaxf(0.0f, -dot(dir, mk3(ln)));
            const float geom = (cos1 * cos2) * area;            // zero for every sample on a surface that faces away: no slow division
            const float fac = d2 > 0.0f ? div_by_pos(div_by_pos(geom, d2), lsn_f) : geom / d2 / lsn_f;
            V3 contrib = cmul(mk3(a.w, b.w, cc.w), Tf) * fac;   // :274-283
            bool live = !(contrib.x == 0.0f && contrib.y == 0.0f && contrib.z == 0.0f);
            float t_to_light = dist.x / dir.x;                  // :272
            bool needs_trace = live && (t_to_light == t_to_light);
            if (live && !needs_trace) accum_add(accum, pixel, contrib);   // NaN: never blocked, :19-27
            shadow(needs_trace, pos, t_to_light, normalize(dir), contrib);     // Ray ctor normalises again
        }
    }
    if (bounce == (uint32_t)(p.max_vertices - 1)) return false;  // bounce stack full, :210
    const uint4 q = draw(pixel, sample, bounce, 0, p.seed);
    if (u01(q.x) > p.p_rr) return false;                         // :216-221
    V3 wdir = normalize_rcp(normalize_rcp(sample_hemisphere(nrm, u01(q.y), u01(q.z))));   // :225-227 + Ray ctor
    uint32_t nmeta = bounce + 1u;
    if (mflags & 2u) {                                          // SPECULAR probe, :294-303
        const float4 m2 = __ldg(sc.mats + 5 * mat + 2);
        V3 in = normalize_rcp(d);
        V3 out = in - (2.0f * dot(in, nrm)) * nrm;
        uint4 e = draw(pixel, sample, bounce, 1, p.seed);
        V3 pd = normalize_rcp(normalize_rcp(sample_probe_lobe(out, m2.x, m2.y, u01(e.x), u01(e.y))));
        float pc = fmaxf(0.0f, dot(pd, nrm));
        npr.o = pos;
        npr.d = pd;
        npr.w = cmul(T, mk3(m0)) * m2.z * pc * (kTwoPi / 8.0f);  // :306-312
        nmeta |= kFlagProbe;
    }
    float cosn = fmaxf(0.0f, dot(wdir, nrm));
    nx.o = pos;
    nx.d = wdir;
    nx.T = Tf * (cosn * p.two_pi_over_p_rr);                    // :288-293
    nx.pixel = pixel; nx.sample = sample; nx.meta = nmeta;
    return true;
}

// mis estimator, one path vertex (statement: oracle/orc_render.cpp path_mis; DESIGN.md "mis"): two-sided
// modified-Phong surfaces, one-sided emitters, light triangles picked ~ area * luminance(Ke), power
// heuristic between light_sample_n light samples and the BSDF sample, Russian roulette at P_RR.
CRT_DEV int pick_light(const float* __restrict__ cdf, int n, float u) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(cdf + mid) >= u) hi = mid; else lo = mid + 1;
    }
    return lo;
}
CRT_DEV void phong_eval(V3 fd /* kd / pi */, V3 ks, float ns, float pd, bool has_spec, float cos_s, float ca, V3* f, float* pdf) {
    const float pdf_d = cos_s / kPi;
    if (has_spec) {
        const float pw = det_pow(ca, ns);
        *f = fd + ks * ((ns + 2.0f) / kTwoPi * pw);
        const float pdf_s = (ns + 1.0f) / kTwoPi * pw;
        *pdf = fmaf(pd, pdf_d, (1.0f - pd) * pdf_s);
    } else {
        *f = fd;
        *pdf = pdf_d;
    }
}

template <typename ShadowFn>
CRT_DEV bool shade_vertex_mis(const SceneView& sc, const RenderParamsDev& p, const PathState& ps, float t, int slot,
                              long long* __restrict__ accum, ShadowFn&& shadow, PathState& nx) {
    const uint32_t pixel = ps.pixel, sample = ps.sample, bounce = ps.meta & 0xffu;
    const float lsn_f = (float)p.light_sample_n;
    const float4 sh = __ldg(sc.tri_shade + slot);
    const uint32_t mat = __float_as_uint(sh.w);
    const float4 m0 = __ldg(sc.mats + 5 * mat + 0), m1 = __ldg(sc.mats + 5 * mat + 1), m3 = __ldg(sc.mats + 5 * mat + 3);
    const V3 n = mk3(sh), d = ps.d, T = ps.T;
    const float dn = dot(n, d);
    if (__float_as_uint(m1.w) & 1u) {                            // emitter: seen from its front side only
        if (dn < 0.0f) {
            if (bounce == 0) accum_add(accum, pixel, mk3(m1));
            else {
                const float pl = m3.w * (t * t) / (-dn);
                const float pls = lsn_f * pl;
                const float w = (ps.pdf * ps.pdf) / fmaf(ps.pdf, ps.pdf, pls * pls);
                accum_add(accum, pixel, cmul(T, mk3(m1)) * w);
            }
        }
        return false;
    }
    const V3 ns = dn > 0.0f ? mk3(-n.x, -n.y, -n.z) : n;
    const V3 wo = mk3(-d.x, -d.y, -d.z);
    const V3 pos = ps.o + t * d;
    const float off = 1.0e-4f * (1.0f + fmaxf(fmaxf(fabsf(pos.x), fabsf(pos.y)), fabsf(pos.z)));
    const V3 org = pos + off * ns;
    const float cos_o = dot(ns, wo);
    const V3 refl = normalize_rcp((2.0f * cos_o) * ns - wo);
    const V3 kd = mk3(m0), ks = mk3(m3), kd_pi = mk3(__ldg(sc.mats + 5 * mat + 4));
    const float mns = m0.w;
    const float lkd = lumf(kd), lks = lumf(ks);
    const float lsum = lkd + lks;
    if (!(lsum > 0.0f)) return false;
    const float pd = lkd / lsum;
    const bool has_spec = lks > 0.0f;
    for (int sj = 0; sj < p.light_sample_n && sc.n_light_tris > 0; ++sj) {
        const uint4 q = draw(pixel, sample, bounce, 2u + (uint32_t)sj, p.seed);
        const int k = pick_light(sc.light_cdf, sc.n_light_tris, u01(q.x));
        const float4* lt = sc.light_tris + 4 * (size_t)k;
        const float4 a = __ldg(lt), b = __ldg(lt + 1), cc = __ldg(lt + 2), ln = __ldg(lt + 3);
        const float su = sqrtf(u01(q.y));
        const float b0 = 1.0f - su, b1 = u01(q.z) * su;
        const float b2 = (1.0f - b0) - b1;
        const V3 lp = (b0 * mk3(a) + b1 * mk3(b)) + b2 * mk3(cc);
        const V3 dist = lp - org;
        const float d2 = dot(dist, dist);
        const float d1 = sqrtf(d2);
        const V3 wi = dist * (1.0f / d1);
        const float cos_s = dot(ns, wi);
        const float cos_l = -dot(mk3(ln), wi);
        bool needs_trace = cos_s > 0.0f && cos_l > 0.0f;
        V3 contrib = mk3(0.0f, 0.0f, 0.0f);
        if (needs_trace) {
            const float ca = fmaxf(0.0f, dot(refl, wi));
            V3 f;
            float pb;
            phong_eval(kd_pi, ks, mns, pd, has_spec, cos_s, ca, &f, &pb);
            const float pl = ln.w * d2 / cos_l;
            const float pls = lsn_f * pl;
            const float w = (pls * pls) / fmaf(pls, pls, pb * pb);
            contrib = cmul(cmul(T, f), mk3(a.w, b.w, cc.w)) * (cos_s * w / pls);
            needs_trace = !(contrib.x == 0.0f && contrib.y == 0.0f && contrib.z == 0.0f);
        }
        shadow(needs_trace, org, d1 * 0.999f, wi, contrib);
    }
    if (bounce == (uint32_t)(p.max_vertices - 1)) return false;
    const uint4 q = draw(pixel, sample, bounce, 0, p.seed);
    if (u01(q.x) > p.p_rr) return false;
    const float u1 = u01(q.z), u2 = u01(q.w);
    float sn, cs;
    sincos_2pi(u2, &sn, &cs);
    V3 wi;
    if (u01(q.y) <= pd) {
        const float rr = sqrtf(u1);
        const float z = sqrtf(1.0f - u1);
        wi = to_world(mk3(rr * cs, rr * sn, z), ns);
    } else {
        const float ca0 = det_pow(u1, 1.0f / (mns + 1.0f));
        const float sa0 = sqrtf(fmaxf(0.0f, 1.0f - ca0 * ca0));
        wi = to_world(mk3(sa0 * cs, sa0 * sn, ca0), refl);
    }
    wi = normalize_rcp(wi);
    const float cos_s = dot(ns, wi);
    if (!(cos_s > 0.0f)) return false;
    const float ca = fmaxf(0.0f, dot(refl, wi));
    V3 f;
    float pb;
    phong_eval(kd_pi, ks, mns, pd, has_spec, cos_s, ca, &f, &pb);
    if (!(pb > 0.0f)) return false;
    nx.o = org;
    nx.d = wi;
    nx.T = cmul(T, f) * (cos_s / pb / p.p_rr);
    nx.pixel = pixel; nx.sample = sample; nx.meta = bounce + 1u;
    nx.pdf = pb;
    return true;
}

// SPECULAR probe of the previous vertex (reference Render.cuh:304-313): the probe hit an emitter.
CRT_DEV void probe_resolve(const SceneView& sc, int probe_slot, V3 w, uint32_t pixel, long long* __restrict__ accum) {
    if (probe_slot < 0) return;
    const uint32_t pm = __float_as_uint(__ldg(sc.tri_shade + probe_slot).w);
    const float4 m1 = __ldg(sc.mats + 5 * pm + 1);
    if (__float_as_uint(m1.w) & 1u) accum_add(accum, pixel, cmul(w, mk3(m1)));
}

// EST: CRT_ESTIMATOR_COMPAT (0) or CRT_ESTIMATOR_MIS (1)
// Resident blocks per SM asked of the compiler. The compat vertex is a long dependent chain of IEEE divisions and square
// roots behind three levels of dependent loads (queue -> triangle -> material / light): at 108 registers only 16 warps
// per SM hide it (warps active 24 %, profiles/r01_s17.md). Capping registers at 64 (a few spilled words) takes the
// stage from 14.7 to 10.3 ms on veach-mis and from 4.70 to 4.14 ms on cornell-box (1080p spp 16, r01_s18.md); the
// mis vertex (fewer live values, one light sample) gets slower under the same cap and keeps the compiler's choice.
#ifndef CRT_SHADE_MINB
#define CRT_SHADE_MINB 8
#endif
#ifndef CRT_SHADE_MINB_MIS
#define CRT_SHADE_MINB_MIS 1
#endif
template <int EST>
__global__ void __launch_bounds__(128, EST == CRT_ESTIMATOR_COMPAT ? CRT_SHADE_MINB : CRT_SHADE_MINB_MIS) k_shade(SceneView sc, Counters* c, RenderParamsDev p,
                                                      const float4* __restrict__ q_o, const float4* __restrict__ q_d,
                                                      const float4* __restrict__ q_T, const float* __restrict__ q_pdf,
                                                      float* __restrict__ n_pdf, const float* __restrict__ hit_t,
                                                      const int* __restrict__ hit_slot, const float4* __restrict__ pr_w_cur,
                                                      const int* __restrict__ pr_hit, float4* __restrict__ n_o,
                                                      float4* __restrict__ n_d, float4* __restrict__ n_T,
                                                      float4* __restrict__ pr_o_next, float4* __restrict__ pr_d_next,
                                                      float4* __restrict__ pr_w_next, uint32_t* __restrict__ pr_list_next,
                                                      float4* __restrict__ sh_o, float4* __restrict__ sh_d,
                                                      float4* __restrict__ sh_c, long long* __restrict__ accum, int par, uint32_t region_cap) {
    const uint32_t n = c->n_cur;
    const uint32_t region = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) % (uint32_t)kShadowRegions;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 qo = q_o[i], qd = q_d[i], qT = q_T[i];
        PathState ps;
        ps.o = mk3(qo); ps.d = mk3(qd); ps.T = mk3(qT);
        ps.pixel = __float_as_uint(qo.w); ps.sample = __float_as_uint(qd.w); ps.meta = __float_as_uint(qT.w);
        ps.pdf = EST == CRT_ESTIMATOR_MIS ? q_pdf[i] : 0.0f;
        const int slot = hit_slot[i];
        if (slot < 0) continue;                                     // miss, :210 (a pending probe is dropped, :294)
        if (EST == CRT_ESTIMATOR_COMPAT && (ps.meta & kFlagProbe)) probe_resolve(sc, pr_hit[i], mk3(pr_w_cur[i]), ps.pixel, accum);
        PathState nx;
        ProbeState npr;
        const uint32_t pixel = ps.pixel;
        auto shadow = [&](bool needs_trace, V3 pos, float tmax, V3 dir, V3 contrib) {
            int k = warp_append(&c->n_shadow[par][region].v, needs_trace);
            if (k >= 0) {
                k += (int)(region * region_cap);
                sh_o[k] = make_float4(pos.x, pos.y, pos.z, tmax);
                sh_d[k] = make_float4(dir.x, dir.y, dir.z, __uint_as_float(pixel));
                sh_c[k] = make_float4(contrib.x, contrib.y, contrib.z, 0.0f);
            }
        };
        bool alive;
        if (EST == CRT_ESTIMATOR_MIS) alive = shade_vertex_mis(sc, p, ps, hit_t[i], slot, accum, shadow, nx);
        else alive = shade_vertex_compat(sc, p, ps, hit_t[i], slot, accum, shadow, nx, npr);
        int k = warp_append(&c->n_next, alive);
        if (k < 0) continue;
        if (EST == CRT_ESTIMATOR_MIS) n_pdf[k] = nx.pdf;
        if (EST == CRT_ESTIMATOR_COMPAT && (nx.meta & kFlagProbe)) {
            pr_o_next[k] = make_float4(npr.o.x, npr.o.y, npr.o.z, 0.0f);
            pr_d_next[k] = make_float4(npr.d.x, npr.d.y, npr.d.z, 0.0f);
            pr_w_next[k] = make_float4(npr.w.x, npr.w.y, npr.w.z, 0.0f);
            int pk = warp_append(&c->n_probe_next, true);
            pr_list_next[pk] = (uint32_t)k;
        }
        n_o[k] = make_float4(nx.o.x, nx.o.y, nx.o.z, __uint_as_float(nx.pixel));
        n_d[k] = make_float4(nx.d.x, nx.d.y, nx.d.z, __uint_as_float(nx.sample));
        n_T[k] = make_float4(nx.T.x, nx.T.y, nx.T.z, __uint_as_float(nx.meta));
    }
}

// Tail of a frame: once no new camera paths remain and at most tail_max paths are alive, ONE persistent kernel runs
// them to their ends, instead of five launches per bounce for ever smaller wavefronts (a launch with 2-3 rays per lane
// lasts as long as its longest ray: the second and third bounce of an 800x600 frame cost more than the first,
// profiles/r02_s08.md). It is the leaf-queue traversal of trace_persistent_queue with three kinds of rays in flight in one
// warp - the extend ray of a path, shadow rays, SPECULAR probe rays - and a source of rays in front of the global path
// queue: a lane whose extend ray hit shades the vertex (same per-vertex statement, same Philox keys, same
// order-independent accumulation as k_shade, so the image does not depend on where the switch happens), pushes the
// shadow / probe rays onto the warp's stash in shared memory and parks the continuation; idle lanes take stash entries
// first (every lane, when the stash runs high), then their parked continuation, then a new path. Shadow rays are thereby
// off a path's critical chain, and a lane is never without work while the warp has any.
#ifndef CRT_TERM_HIGH
#define CRT_TERM_HIGH 16
#endif
#ifndef CRT_TAIL_MINB
#define CRT_TAIL_MINB 4
#endif
static constexpr int kTermCap = 80;                  // shadow / probe rays waiting per warp; beyond it a ray is traced in place
static constexpr int kTermHigh = CRT_TERM_HIGH;                 // at this many, parked continuations wait and every idle lane takes from the stash
#ifndef CRT_SHADE_BATCH
#define CRT_SHADE_BATCH 8                            // lanes with a vertex to shade that make the warp shade now (else after kShadeWait turns)
#endif
static constexpr int kShadeBatch = CRT_SHADE_BATCH;
static constexpr int kShadeWait = 2;
struct TermStash {
    float4 a[kTermCap];                              // origin, tmax
    float4 b[kTermCap];                              // direction, kind (1 shadow, 2 probe)
    float4 c[kTermCap];                              // contribution (shadow) / weight (probe), pixel
    int count;
};
enum { kPayT = 0, kPayPixel = 3, kPaySample = 4, kPayMeta = 5, kPayPdf = 6, kPayPd = 7, kPayPw = 10, kPayO = 13, kPayD = 16, kPayWords = 19 };

template <int EST, bool WIDE>
__global__ void __launch_bounds__(128, CRT_TAIL_MINB) k_tail(SceneView sc, Counters* c, RenderParamsDev p, const float4* __restrict__ q_o,
                                                 const float4* __restrict__ q_d, const float4* __restrict__ q_T,
                                                 const float* __restrict__ q_pdf, const float4* __restrict__ pr_d,
                                                 const float4* __restrict__ pr_w, long long* __restrict__ accum) {
    const uint32_t n = c->tail_n;
    if (n == 0) return;
    typedef typename std::conditional<WIDE, WideWalker, PairWalker>::type Walker;
    typedef WarpLeafQueue<Walker::kCap> Queue;
    __shared__ Queue s_wq[4];
    __shared__ TermStash s_ts[4];
    __shared__ float s_pay[kPayWords][128];           // the lane's path: throughput, pixel, sample, meta, pdf, pending probe, parked ray
    __shared__ float4 s_term[128];                    // the terminal ray the lane traces: contribution / weight, pixel
    Queue& q = s_wq[threadIdx.x >> 5];
    TermStash& ts = s_ts[threadIdx.x >> 5];
    const unsigned kFull = 0xffffffffu;
    const int lane = threadIdx.x & 31, tid = threadIdx.x;
    const unsigned lt_mask = (1u << lane) - 1u;
    typename Walker::Entry stack[Walker::kLocal];
    Walker wk;
    wk.init();
    V3 o = mk3(0, 0, 0), inv = mk3(0, 0, 0);
    float tlimit = 0.0f, sh_t = 0.0f;
    int pending = 0, kind = 0, sh_slot = -1, shade_wait = 0;
    bool have = false, zray = false, parked = false, needs_shade = false;
    unsigned long long n_ext = 0, n_sh = 0, n_pr = 0;
    RayFetch rf;
    rf.init(n);
    if (lane == 0) { q.count = 0; ts.count = 0; }
    __syncwarp();
    auto arm = [&](V3 ro, V3 rd, float tmax, int k) {          // this lane starts tracing a ray of kind k
        o = ro;
        inv = box_inv3(rd);
        zray = has_parallel_axis(inv);
        kind = k;
        tlimit = k == 1 ? tmax : FLT_MAX;
        q.ox[lane] = ro.x; q.oy[lane] = ro.y; q.oz[lane] = ro.z;
        q.dx[lane] = rd.x; q.dy[lane] = rd.y; q.dz[lane] = rd.z;
        q.tmax[lane] = tmax;
        q.any[lane] = k == 1;
        q.best[lane] = kNoHitKey;
        q.best_slot[lane] = -1;
        pending = 0;
        wk.start(sc.n_nodes != 0, inv);
        have = true;
    };
    // room for every push is reserved before a lane shades (C2), so the stash cannot overflow
    auto push_term = [&](V3 ro, float tmax, V3 rd, int k, V3 w, uint32_t pixel) {
        const int pos = atomicAdd(&ts.count, 1);
        ts.a[pos] = make_float4(ro.x, ro.y, ro.z, tmax);
        ts.b[pos] = make_float4(rd.x, rd.y, rd.z, __int_as_float(k));
        ts.c[pos] = make_float4(w.x, w.y, w.z, __uint_as_float(pixel));
    };
    const int per_vertex = sc.n_lights * p.light_sample_n + 1;       // shadow rays + the probe a vertex can push (EST mis: light_sample_n + 0)
    for (;;) {
        // A. node steps; leaves go to the queue
        wk.steps(sc, q, stack, o, inv, tlimit * 1.0001f, zray, lane, lt_mask, pending);
        // B. flush the leaf queue
        const unsigned walking = __ballot_sync(kFull, wk.walking());
        __syncwarp();
        const int q_count = wk.queued(q);
        if (q_count >= Walker::kFlush || (walking == 0 && q_count > 0)) {
            flush_leaf_queue<2>(sc, q, q_count, lane);
            wk.reset_queue(q, lane);
            pending = 0;
            if (have) {
                const unsigned long long b = q.best[lane];
                if (kind != 1) tlimit = __uint_as_float((uint32_t)(b >> 32));
                else if (b != kNoHitKey) wk.stop();
            }
            __syncwarp();
        }
        // C. finished rays
        if (have && !wk.walking() && pending == 0) {
            const unsigned long long b = q.best[lane];
            const bool hit = b != kNoHitKey;
            have = false;
            if (kind == 1) {
                n_sh++;
                if (!hit) { const float4 cc = s_term[tid]; accum_add(accum, __float_as_uint(cc.w), mk3(cc)); }
            } else if (kind == 2) {
                n_pr++;
                const float4 cc = s_term[tid];
                probe_resolve(sc, hit ? q.best_slot[lane] : -1, mk3(cc), __float_as_uint(cc.w), accum);
            } else {
                n_ext++;
                if (hit) {                                        // the ray is kept for the shading turn: the lane may trace stash entries meanwhile
                    needs_shade = true; sh_t = __uint_as_float((uint32_t)(b >> 32)); sh_slot = q.best_slot[lane];
                    s_pay[kPayO][tid] = q.ox[lane]; s_pay[kPayO + 1][tid] = q.oy[lane]; s_pay[kPayO + 2][tid] = q.oz[lane];
                    s_pay[kPayD][tid] = q.dx[lane]; s_pay[kPayD + 1][tid] = q.dy[lane]; s_pay[kPayD + 2][tid] = q.dz[lane];
                }
            }
        }
        // C2. vertices: shaded when enough lanes have one (the statement is long: a lane or two at a time would cost the
        // warp as many instructions as a full one), or when they have waited kShadeWait turns
        {
            const unsigned ns = __ballot_sync(kFull, needs_shade && !have);
            if (ns) {
                // ... or when a quarter of the paths this warp still has are waiting (late in the frame a warp holds a handful)
                const int live = __popc(__ballot_sync(kFull, needs_shade || parked || (have && kind == 0)));
                // as many lanes shade as the stash has room for all they can push; the others wait (and trace stash entries meanwhile)
                const int allowed = (kTermCap - ts.count) / per_vertex;
                if (allowed > 0 && (__popc(ns) >= kShadeBatch || 4 * __popc(ns) >= live || shade_wait >= kShadeWait)) {
                    shade_wait = 0;
                    if (needs_shade && !have && __popc(ns & lt_mask) < allowed) {
                        needs_shade = false;
                        PathState ps;
                        ps.o = mk3(s_pay[kPayO][tid], s_pay[kPayO + 1][tid], s_pay[kPayO + 2][tid]);
                        ps.d = mk3(s_pay[kPayD][tid], s_pay[kPayD + 1][tid], s_pay[kPayD + 2][tid]);
                        ps.T = mk3(s_pay[kPayT][tid], s_pay[kPayT + 1][tid], s_pay[kPayT + 2][tid]);
                        ps.pixel = __float_as_uint(s_pay[kPayPixel][tid]);
                        ps.sample = __float_as_uint(s_pay[kPaySample][tid]);
                        ps.meta = __float_as_uint(s_pay[kPayMeta][tid]);
                        ps.pdf = s_pay[kPayPdf][tid];
                        const uint32_t pixel = ps.pixel;
                        if (EST == CRT_ESTIMATOR_COMPAT && (ps.meta & kFlagProbe))     // the pending probe of the previous vertex, Render.cuh:303
                            push_term(ps.o, FLT_MAX, mk3(s_pay[kPayPd][tid], s_pay[kPayPd + 1][tid], s_pay[kPayPd + 2][tid]), 2,
                                      mk3(s_pay[kPayPw][tid], s_pay[kPayPw + 1][tid], s_pay[kPayPw + 2][tid]), pixel);
                        auto shadow = [&](bool needs_trace, V3 pos, float tmax, V3 dir, V3 contrib) {
                            if (needs_trace) push_term(pos, tmax, dir, 1, contrib, pixel);
                        };
                        PathState nx;
                        ProbeState npr;
                        bool alive;
                        if (EST == CRT_ESTIMATOR_MIS) alive = shade_vertex_mis(sc, p, ps, sh_t, sh_slot, accum, shadow, nx);
                        else alive = shade_vertex_compat(sc, p, ps, sh_t, sh_slot, accum, shadow, nx, npr);
                        if (alive) {
                            s_pay[kPayT][tid] = nx.T.x; s_pay[kPayT + 1][tid] = nx.T.y; s_pay[kPayT + 2][tid] = nx.T.z;
                            s_pay[kPayMeta][tid] = __uint_as_float(nx.meta);
                            if (EST == CRT_ESTIMATOR_MIS) s_pay[kPayPdf][tid] = nx.pdf;
                            if (EST == CRT_ESTIMATOR_COMPAT && (nx.meta & kFlagProbe)) {
                                s_pay[kPayPd][tid] = npr.d.x; s_pay[kPayPd + 1][tid] = npr.d.y; s_pay[kPayPd + 2][tid] = npr.d.z;
                                s_pay[kPayPw][tid] = npr.w.x; s_pay[kPayPw + 1][tid] = npr.w.y; s_pay[kPayPw + 2][tid] = npr.w.z;
                            }
                            s_pay[kPayO][tid] = nx.o.x; s_pay[kPayO + 1][tid] = nx.o.y; s_pay[kPayO + 2][tid] = nx.o.z;
                            s_pay[kPayD][tid] = nx.d.x; s_pay[kPayD + 1][tid] = nx.d.y; s_pay[kPayD + 2][tid] = nx.d.z;
                            parked = true;
                        }
                    }
                } else {
                    ++shade_wait;
                }
            }
        }
        // D. idle lanes: a stash entry, else the parked continuation, else a new path
        __syncwarp();
        const int t_cnt = ts.count;
        const bool idle_me = !have && !needs_shade;
        const unsigned idle = __ballot_sync(kFull, !have);
        if (idle) {
            bool got = false;
            const bool want_t = !have && (needs_shade || !parked || t_cnt >= kTermHigh);
            const unsigned wt = __ballot_sync(kFull, want_t);
            const int take_t = min(__popc(wt), t_cnt);
            if (want_t && __popc(wt & lt_mask) < take_t) {
                const int e = t_cnt - 1 - __popc(wt & lt_mask);
                const float4 a = ts.a[e], b = ts.b[e];
                s_term[tid] = ts.c[e];
                arm(mk3(a), mk3(b), a.w, __float_as_int(b.w));
                got = true;
            }
            __syncwarp();
            if (lane == 0 && take_t) ts.count = t_cnt - take_t;
            if (idle_me && !got && parked) {
                parked = false;
                arm(mk3(s_pay[kPayO][tid], s_pay[kPayO + 1][tid], s_pay[kPayO + 2][tid]),
                    mk3(s_pay[kPayD][tid], s_pay[kPayD + 1][tid], s_pay[kPayD + 2][tid]), FLT_MAX, 0);
                got = true;
            }
            const bool fresh_me = idle_me && !got;
            const unsigned fresh = __ballot_sync(kFull, fresh_me);
            if (fresh && !rf.drained()) {
                uint32_t first = 0;
                const uint32_t got_n = rf.take(&c->fetch_tail, n, lane, (uint32_t)__popc(fresh), first);
                const uint32_t rank = (uint32_t)__popc(fresh & lt_mask);
                if (fresh_me && rank < got_n) {
                    const uint32_t i = first + rank;
                    const float4 qo = q_o[i], qd = q_d[i], qT = q_T[i];
                    s_pay[kPayT][tid] = qT.x; s_pay[kPayT + 1][tid] = qT.y; s_pay[kPayT + 2][tid] = qT.z;
                    s_pay[kPayPixel][tid] = qo.w; s_pay[kPaySample][tid] = qd.w; s_pay[kPayMeta][tid] = qT.w;
                    s_pay[kPayPdf][tid] = EST == CRT_ESTIMATOR_MIS ? q_pdf[i] : 0.0f;
                    if (EST == CRT_ESTIMATOR_COMPAT && (__float_as_uint(qT.w) & kFlagProbe)) {
                        const float4 pd = pr_d[i], pw = pr_w[i];
                        s_pay[kPayPd][tid] = pd.x; s_pay[kPayPd + 1][tid] = pd.y; s_pay[kPayPd + 2][tid] = pd.z;
                        s_pay[kPayPw][tid] = pw.x; s_pay[kPayPw + 1][tid] = pw.y; s_pay[kPayPw + 2][tid] = pw.z;
                    }
                    arm(mk3(qo), mk3(qd), FLT_MAX, 0);
                }
            }
            __syncwarp();
            // nothing in flight, nothing parked or waiting to be shaded, nothing stashed, no path left in the queue
            if (!__any_sync(kFull, have || parked || needs_shade) && ts.count == 0 && rf.drained()) break;
        }
    }
    for (int off = 16; off > 0; off >>= 1) {
        n_ext += __shfl_down_sync(kFull, n_ext, off);
        n_sh += __shfl_down_sync(kFull, n_sh, off);
        n_pr += __shfl_down_sync(kFull, n_pr, off);
    }
    if (lane == 0) {
        if (n_ext) atomicAdd(&c->stat_extend, n_ext);
        if (n_sh) atomicAdd(&c->stat_shadow, n_sh);
        if (n_pr) atomicAdd(&c->stat_probe, n_pr);
    }
}

// Shadow rays: the decision of blocked() (reference Render.cuh:19-27) with an any-hit traversal.
template <bool WIDE>
__global__ void __launch_bounds__(128, CRT_MINB) k_shadow(SceneView sc, Counters* c, const float4* __restrict__ sh_o,
                                                const float4* __restrict__ sh_d, const float4* __restrict__ sh_c,
                                                long long* __restrict__ accum, int par, uint32_t region_cap) {
    // the contribution and pixel of the ray a lane owns wait in shared memory (loaded with the ray, one DRAM round trip
    // instead of a second one when the ray finishes: 3.7 % of this kernel's stall samples, profiles/r01_s20.md)
    __shared__ float4 s_contrib[128];
    // The regions are read interleaved in runs of 32: indices 32 b .. 32 b + 31 are entries 32 (b / 8) .. of region b % 8, so
    // that a warp's refill reads consecutive records of one region and the queue is still walked roughly in the order the
    // paths were shaded in. The regions hold nearly the same number of rays (each takes an eighth of the warps); an index past
    // the end of its region is a slot without a ray.
    __shared__ uint32_t s_cnt[kShadowRegions];
    __shared__ uint32_t s_n;
    if (threadIdx.x == 0) {
        uint32_t mx = 0;
        for (int r = 0; r < kShadowRegions; ++r) { s_cnt[r] = c->n_shadow[par][r].v; mx = max(mx, s_cnt[r]); }
        s_n = ((mx + 31u) & ~31u) * (uint32_t)kShadowRegions;
    }
    __syncthreads();
    trace_queue<1, WIDE>(
        sc, s_n, &c->fetch_shadow[par],
        [&](uint32_t i, V3& o, V3& d, float& tmax) {
            const uint32_t blk = i >> 5, r = blk % (uint32_t)kShadowRegions, e = ((blk / (uint32_t)kShadowRegions) << 5) | (i & 31u);
            if (e >= s_cnt[r]) {                                        // no ray here: nothing to trace, nothing to add
                o = mk3(0.0f, 0.0f, 0.0f); d = mk3(0.0f, 0.0f, 1.0f); tmax = 0.0f;
                s_contrib[threadIdx.x] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                return false;
            }
            const size_t k = (size_t)r * region_cap + e;
            const float4 a = sh_o[k], b = sh_d[k], cc = sh_c[k];
            o = mk3(a); tmax = a.w; d = mk3(b);
            s_contrib[threadIdx.x] = make_float4(cc.x, cc.y, cc.z, b.w);
            return true;
        },
        [&](uint32_t i, const HitRec& h) {
            if (h.slot < 0) { const float4 cc = s_contrib[threadIdx.x]; accum_add(accum, __float_as_uint(cc.w), mk3(cc)); }
        });
}

// E11 (reference Render.cuh:348,350): mean over spp, clamp, pow 0.6, *255, truncate.
__global__ void k_resolve(const long long* __restrict__ accum, uint32_t n_values, uint32_t spp, float* __restrict__ linear,
                          uint8_t* __restrict__ rgb8) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_values) return;
    float v = (float)((double)accum[k] / 4294967296.0 / (double)spp);
    if (linear) linear[k] = v;
    if (rgb8) {
        float cl = fmaxf(0.0f, fminf(1.0f, v));
        rgb8[k] = (uint8_t)(255.0f * powf(cl, 0.6f));
    }
}

int resolve_device(const long long* d_accum, uint32_t n_pixels, uint32_t spp, float* d_linear, uint8_t* d_rgb8, cudaStream_t st) {
    uint32_t nv = n_pixels * 3;
    k_resolve<<<(nv + 255) / 256, 256, 0, st>>>(d_accum, nv, spp ? spp : 1, d_linear, d_rgb8);
    CRT_CUDA(cudaGetLastError());
    return CRT_OK;
}

// =============================================================================================
// host driver
// =============================================================================================
// with_estimator(mis, f): f(integral_constant<int, CRT_ESTIMATOR_MIS or _COMPAT>), for a kernel's EST as E.value
template <typename F>
static auto with_estimator(bool mis, F&& f) {
    return mis ? f(std::integral_constant<int, CRT_ESTIMATOR_MIS>()) : f(std::integral_constant<int, CRT_ESTIMATOR_COMPAT>());
}

int wavefront_create(const DeviceScene& ds, uint32_t width, uint32_t height, WavefrontPtr& out) {
    WavefrontPtr w(new Wavefront());
    w->width = width; w->height = height;
    w->has_probe = ds.has_specular;
    const size_t npix = (size_t)width * height;
    CRT_CUDA(w->accum.alloc(3 * npix));
    CRT_CUDA(w->counters.alloc(1));
    CRT_CUDA(pinned_alloc(w->status_host, 1, cudaHostAllocMapped));
    CRT_CUDA(cudaHostGetDevicePointer((void**)&w->status_dev, (void*)w->status_host.get(), 0));
    for (int k = 0; k < 4; ++k) CRT_CUDA(create(w->ev[k], cudaEventDisableTiming));
    CRT_CUDA(create(w->ev_begin));
    CRT_CUDA(create(w->ev_end));
    int occ = 0;
    CRT_CUDA(with_layout(ds.wide, [&](auto W) { return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_extend<W.value>, 128, 0); }));
    w->grid_trace = num_sms() * std::max(occ, 1);
    w->grid_shade = num_sms() * 8;
    CRT_CUDA(with_layout(ds.wide, [&](auto W) {
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_tail<CRT_ESTIMATOR_MIS, W.value>, 128, 0);
    }));
    w->grid_tail = num_sms() * std::max(occ, 1);
    out = std::move(w);
    return CRT_OK;
}

// Pool = paths in flight. Measured on B200 (cornell-box 1920x1080 spp 16, tools/pool_sweep.py): 2^20 paths
// 916 Msamples/s, 2^22 1227, 2^23 1294, 2^24 1331 - every persistent lane gets more rays per launch, so the
// drain at the end of each launch and the per-iteration launches weigh less. HBM holds it easily
// (2^24 paths: 1.6 GB of path queues + 48 B per shadow ray).
static int ensure_pool(Wavefront* w, const DeviceScene& ds, const RenderSettings& rs, unsigned long long work_items) {
    uint32_t pool = env_u32("CRT_POOL", 0);
    if (pool == 0) {
        pool = 1u << 20;
        while (pool < (1u << 25) && pool < work_items) pool <<= 1;       // 2^25: +2 % over 2^24 at steady state (r01_s35), 7 GB
    }
    uint64_t per_vertex = (uint64_t)std::max<uint32_t>(ds.n_lights, 1) * std::max<uint32_t>(rs.light_sample_n, 1);
    const uint64_t shadow_budget = 1ull << 26;        // 64 Mi shadow rays in flight at most (3 GiB)
    while (pool > 4096 && (uint64_t)pool * per_vertex > shadow_budget) pool >>= 1;
    // a region takes the shadow rays of the warps with global id % kShadowRegions == r: at most this many paths each
    const uint64_t warps = (uint64_t)w->grid_shade * 4;
    const uint64_t region_paths = ((uint64_t)pool + warps * 32 - 1) / (warps * 32) * 32 * ((warps + kShadowRegions - 1) / kShadowRegions);
    const uint64_t region_cap = std::min<uint64_t>(region_paths, pool) * per_vertex;
    uint64_t shadow_cap = region_cap * kShadowRegions;
    if (shadow_cap > 0xffffffffull) { set_error("light_sample_n x lights too large"); return CRT_ERR_INVALID; }
    if (w->paths.pool == pool && w->paths.shadow_cap >= shadow_cap) return CRT_OK;
    w->paths = PathPool();                           // pool 0: nothing is valid until every allocation below has succeeded
    PathPool np;
    for (PathQueue& q : np.q) {
        CRT_CUDA(q.o.alloc(pool));
        CRT_CUDA(q.d.alloc(pool));
        CRT_CUDA(q.T.alloc(pool));
        CRT_CUDA(q.pdf.alloc(pool));
        if (w->has_probe) {
            CRT_CUDA(q.pr_o.alloc(pool));
            CRT_CUDA(q.pr_d.alloc(pool));
            CRT_CUDA(q.pr_w.alloc(pool));
            CRT_CUDA(q.pr_list.alloc(pool));
        }
    }
    CRT_CUDA(np.hit_t.alloc(pool));
    CRT_CUDA(np.hit_slot.alloc(pool));
    if (w->has_probe) CRT_CUDA(np.pr_hit.alloc(pool));
    CRT_CUDA(np.sh.o.alloc(shadow_cap));
    CRT_CUDA(np.sh.d.alloc(shadow_cap));
    CRT_CUDA(np.sh.c.alloc(shadow_cap));
    np.sh.region_cap = (uint32_t)region_cap;
    np.pool = pool;
    np.shadow_cap = (uint32_t)shadow_cap;
    w->paths = std::move(np);
    return CRT_OK;
}

long long* wavefront_accum(Wavefront* w) { return w->accum.get(); }

// A run_view is a small state machine - begin (reset + first settings), step (the host side of ONE wavefront iteration,
// optionally without blocking), finish (drain + statistics) - so that one host thread can drive the renders of several
// GPUs at once (crt_group, crt_api.cu); wavefront_render below is the blocking single-GPU composition.
int wavefront_begin(Wavefront* w, const DeviceScene& ds, const RenderSettings& rs, const float eye[3], const float M[9],
                    float tan_half, cudaStream_t st) {
    WfRun& r = w->run;
    if (r.active) { set_error("run_view: a render is already in flight on this handle"); return CRT_ERR_STATE; }
    if (rs.estimator != CRT_ESTIMATOR_COMPAT && rs.estimator != CRT_ESTIMATOR_MIS) { set_error("unknown estimator"); return CRT_ERR_INVALID; }
    const bool mis = rs.estimator == CRT_ESTIMATOR_MIS;
    const size_t npix = (size_t)w->width * w->height;
    const unsigned long long work_all = (unsigned long long)npix * rs.spp;
    const unsigned long long w_begin = rs.range_set ? std::min(rs.work_begin, work_all) : 0;
    const unsigned long long w_end = rs.range_set ? std::min(rs.work_end, work_all) : work_all;
    int rc = ensure_pool(w, ds, rs, w_end > w_begin ? w_end - w_begin : 0);
    if (rc != CRT_OK) return rc;
    RenderParamsDev& p = r.p;
    memcpy(p.eye, eye, sizeof(p.eye));
    memcpy(p.M, M, sizeof(p.M));
    p.tan_half = tan_half;
    p.width = w->width; p.height = w->height; p.n_pixels = npix;
    p.two_pi_over_p_rr = kTwoPi / rs.p_rr;
    p.s_begin = 0; p.p_rr = rs.p_rr; p.light_sample_n = (int)rs.light_sample_n; p.seed = rs.seed;
    p.max_vertices = 64;                                           // BOUNCE_STACK_SIZE, Global.h:18
    p.w_begin = w_begin;
    p.tile_px = p.tile_s0 = p.tile_S = p.tile_fast = 0;
    {
        const uint32_t tile_px = env_u32("CRT_TILE_PX", 1u << 20);    // 24 MB of accumulation buffer per tile (4K: 2^22 2465, 2^21 2658, 2^20 2724, 2^19 2743 Msamples/s, r02_s08)
        if (tile_px && npix > tile_px && w_end > w_begin && w_begin % npix == 0 && w_end % npix == 0) {
            p.tile_px = tile_px;
            p.tile_s0 = (uint32_t)(w_begin / npix);
            p.tile_S = (uint32_t)((w_end - w_begin) / npix);
        }
    }
    {
        const unsigned long long per_tile = (unsigned long long)p.tile_px * p.tile_S;
        p.tile_fast = (per_tile >= w->paths.pool && per_tile < (1ull << 31)) ? 1u : 0u;
        r.per_tile32 = p.tile_fast ? per_tile : 0ull;
    }
    Counters h;
    memset(&h, 0, sizeof(h));
    h.work_next = w_begin;
    h.work_end = std::max(w_end, w_begin);
    w->status_host->done = 0;
    w->status_host->n_cur = 0;
    CRT_CUDA(cudaEventRecord(w->ev_begin.get(), st));
    if (!rs.accumulate) CRT_CUDA(cudaMemsetAsync(w->accum.get(), 0, sizeof(long long) * 3 * npix, st));
    CRT_CUDA(cudaMemcpyAsync(w->counters.get(), &h, sizeof(h), cudaMemcpyHostToDevice, st));
    r.ds = &ds; r.rs = rs; r.st = st; r.mis = mis; r.w_begin = w_begin;
    r.sv = ds.view();
    r.wide = ds.wide;
    r.launches = 0;
    for (float& m : r.ms_stage) m = 0;
    r.tail_max = rs.stage_timing ? 0u : env_u32("CRT_TAIL", kTailDefault);
    // the tail path tracer reserves stash room for every ray a vertex can push; a scene whose vertices push more than half the
    // stash (lights x light_sample_n + 1) finishes with wavefront iterations instead
    if ((uint64_t)std::max<uint32_t>(ds.n_lights, 1) * rs.light_sample_n + 1 > (uint64_t)kTermCap / 2) r.tail_max = 0;
    if (rs.stage_timing) for (Event& e : r.se) create(e);
    // CRT_OVERLAP (default on): k_shadow of iteration k runs on a second stream beside k_prepare, k_generate and k_extend
    // of iteration k + 1 (it only adds to the accumulation buffer; its counters are indexed by iteration parity), so the
    // drain of one persistent kernel is filled by the start of the next. k_shade(k + 1) waits for it (one shadow queue).
    r.overlap = !rs.stage_timing && env_u32("CRT_OVERLAP", 1) != 0 && env_u32("CRT_TIMELINE", 0) == 0;
    if (r.overlap && !w->st_shadow) {
        CRT_CUDA(create(w->st_shadow));
        CRT_CUDA(create(w->ev_shaded, cudaEventDisableTiming));
        CRT_CUDA(create(w->ev_shadowed, cudaEventDisableTiming));
    }
    // CRT_TIMELINE=1 (profiling aid): an event behind every launch of the frame, printed to stderr at the end - the
    // real schedule (tail kernel and host polling included), one stream
    r.timeline = env_u32("CRT_TIMELINE", 0) != 0 && !rs.stage_timing;
    r.tl.clear();
    r.mark("begin", st);
    r.it = 0;
    r.active = true;
    return CRT_OK;
}

// The host keeps two iterations in flight: iteration `it` is enqueued once iteration it - 2 has finished and did not report
// the end of the frame. block == false: returns with *progressed == false instead of waiting for that event.
int wavefront_step(Wavefront* w, bool block, bool* done, bool* progressed) {
    WfRun& r = w->run;
    const DeviceScene& ds = *r.ds;
    const RenderSettings& rs = r.rs;
    const RenderParamsDev& p = r.p;
    const SceneView& sv = r.sv;
    cudaStream_t st = r.st;
    const bool wide = r.wide, mis = r.mis, overlap = r.overlap;
    const uint32_t tail_max = r.tail_max, it = r.it;
    uint64_t& launches = r.launches;
    float* ms_stage = r.ms_stage;
    const Event* se = r.se;
    auto mark = [&](const char* what, cudaStream_t s) { r.mark(what, s); };
    (void)ds;
    *done = false;
    if (progressed) *progressed = false;
    {
        if (it >= 2) {
            if (block) CRT_CUDA(cudaEventSynchronize(w->ev[(it - 2) & 3].get()));
            else {
                cudaError_t q = cudaEventQuery(w->ev[(it - 2) & 3].get());
                if (q == cudaErrorNotReady) return CRT_OK;
                if (q != cudaSuccess) return cuda_fail(q, "cudaEventQuery");
            }
            if (w->status_host->done) { *done = true; if (progressed) *progressed = true; return CRT_OK; }
        }
        const int cur = it & 1, nxt = cur ^ 1;
        Counters* const counters = w->counters.get();
        long long* const accum = w->accum.get();
        const PathPool& pp = w->paths;
        const PathQueue &qc = pp.q[cur], &qn = pp.q[nxt];
        const ShadowQueue& sh = pp.sh;
        k_prepare<<<1, 1, 0, st>>>(counters, pp.pool, tail_max, w->status_dev, cur, r.per_tile32, r.w_begin);
        mark("prepare", st);
        // The tail path tracer goes first: when k_prepare hands the remaining paths to it, the other kernels of this iteration are
        // empty, and it needs nothing from k_shadow of the previous iteration (still running on the second stream), which k_shade
        // below has to wait for. On the shipped frames that shadow launch is 0.2 ms the tail now runs beside.
        with_estimator(mis, [&](auto E) {
            with_layout(wide, [&](auto W) {
                k_tail<E.value, W.value><<<w->grid_tail, 128, 0, st>>>(sv, counters, p, qc.o.get(), qc.d.get(), qc.T.get(), qc.pdf.get(),
                                                                       qc.pr_d.get(), qc.pr_w.get(), accum);
            });
        });
        mark("tail", st);
        if (rs.stage_timing) cudaEventRecord(se[0].get(), st);
        k_generate<<<w->grid_shade, 256, 0, st>>>(counters, p, qc.o.get(), qc.d.get(), qc.T.get(), mis ? qc.pdf.get() : nullptr);
        mark("generate", st);
        if (rs.stage_timing) cudaEventRecord(se[1].get(), st);
        with_layout(wide, [&](auto W) {
            k_extend<W.value><<<w->grid_trace, 128, 0, st>>>(sv, counters, qc.o.get(), qc.d.get(), pp.hit_t.get(), pp.hit_slot.get());
        });
        launches += 3;
        if (w->has_probe && !mis) {
            with_layout(wide, [&](auto W) {
                k_probe<W.value><<<w->grid_trace, 128, 0, st>>>(sv, counters, qc.pr_list.get(), qc.pr_o.get(), qc.pr_d.get(), pp.hit_slot.get(),
                                                                pp.pr_hit.get());
            });
            launches++;
        }
        mark("extend", st);
        if (rs.stage_timing) cudaEventRecord(se[2].get(), st);
        if (overlap && it > 0) CRT_CUDA(cudaStreamWaitEvent(st, w->ev_shadowed.get(), 0));      // k_shadow(it - 1) still reads the shadow queue
        with_estimator(mis, [&](auto E) {
            k_shade<E.value><<<w->grid_shade, 128, 0, st>>>(sv, counters, p, qc.o.get(), qc.d.get(), qc.T.get(), qc.pdf.get(), qn.pdf.get(),
                                                            pp.hit_t.get(), pp.hit_slot.get(), qc.pr_w.get(), pp.pr_hit.get(), qn.o.get(),
                                                            qn.d.get(), qn.T.get(), qn.pr_o.get(), qn.pr_d.get(), qn.pr_w.get(), qn.pr_list.get(),
                                                            sh.o.get(), sh.d.get(), sh.c.get(), accum, cur, sh.region_cap);
        });
        mark("shade", st);
        if (rs.stage_timing) cudaEventRecord(se[3].get(), st);
        cudaStream_t ss = st;
        if (overlap) {
            CRT_CUDA(cudaEventRecord(w->ev_shaded.get(), st));
            CRT_CUDA(cudaStreamWaitEvent(w->st_shadow.get(), w->ev_shaded.get(), 0));
            ss = w->st_shadow.get();
        }
        with_layout(wide, [&](auto W) {
            k_shadow<W.value><<<w->grid_trace, 128, 0, ss>>>(sv, counters, sh.o.get(), sh.d.get(), sh.c.get(), accum, cur, sh.region_cap);
        });
        if (overlap) CRT_CUDA(cudaEventRecord(w->ev_shadowed.get(), ss));
        mark("shadow", st);
        if (rs.stage_timing) cudaEventRecord(se[4].get(), st);
        launches += 3;
        if (rs.stage_timing) {
            cudaEventRecord(se[5].get(), st);
            cudaEventSynchronize(se[5].get());
            for (int k = 0; k < 5; ++k) { float ms = 0; cudaEventElapsedTime(&ms, se[k].get(), se[k + 1].get()); ms_stage[k] += ms; }
        }
        CRT_CUDA(cudaEventRecord(w->ev[it & 3].get(), st));
        CRT_CUDA(cudaGetLastError());
    }
    r.it = it + 1;
    if (progressed) *progressed = true;
    return CRT_OK;
}

int wavefront_finish(Wavefront* w, crt_render_stats* stats) {
    WfRun& r = w->run;
    cudaStream_t st = r.st;
    const bool overlap = r.overlap, timeline = r.timeline;
    const uint32_t it = r.it;
    const unsigned long long w_begin = r.w_begin;
    const uint64_t launches = r.launches;
    float* ms_stage = r.ms_stage;
    auto& tl = r.tl;
    Counters h;
    r.active = false;
    if (overlap && it > 0) CRT_CUDA(cudaStreamWaitEvent(st, w->ev_shadowed.get(), 0));
    CRT_CUDA(cudaEventRecord(w->ev_end.get(), st));
    CRT_CUDA(cudaStreamSynchronize(st));
    for (Event& e : r.se) e.reset();
    if (timeline) {
        float t0 = 0;
        for (size_t k = 1; k < tl.size(); ++k) {
            float ms = 0, at = 0;
            cudaEventElapsedTime(&ms, tl[k - 1].second.get(), tl[k].second.get());
            cudaEventElapsedTime(&at, tl[0].second.get(), tl[k].second.get());
            fprintf(stderr, "timeline %8.1f us  +%7.1f us  %s\n", at * 1e3f, ms * 1e3f, tl[k].first);
        }
        tl.clear();
    }
    if (stats) {
        CRT_CUDA(cudaMemcpy(&h, w->counters.get(), sizeof(h), cudaMemcpyDeviceToHost));
        memset(stats, 0, sizeof(*stats));
        stats->samples = h.work_end - w_begin;
        stats->extend_rays = h.stat_extend;
        stats->shadow_rays = h.stat_shadow;
        for (int par = 0; par < 2; ++par)
            for (int r = 0; r < kShadowRegions; ++r) stats->shadow_rays += h.n_shadow[par][r].v;
        stats->probe_rays = h.stat_probe;
        stats->iterations = h.iterations;
        stats->kernel_launches = launches;
        CRT_CUDA(cudaEventElapsedTime(&stats->ms_total, w->ev_begin.get(), w->ev_end.get()));
        stats->ms_generate = ms_stage[0]; stats->ms_extend = ms_stage[1]; stats->ms_shade = ms_stage[2]; stats->ms_shadow = ms_stage[3];
        stats->ms_tail = ms_stage[4];
    }
    return CRT_OK;
}

int wavefront_render(Wavefront* w, const DeviceScene& ds, const RenderSettings& rs, const float eye[3], const float M[9],
                     float tan_half, cudaStream_t st, crt_render_stats* stats) {
    int rc = wavefront_begin(w, ds, rs, eye, M, tan_half, st);
    if (rc != CRT_OK) return rc;
    for (bool done = false; !done;) {
        rc = wavefront_step(w, true, &done, nullptr);
        if (rc != CRT_OK) { w->run.active = false; return rc; }
    }
    return wavefront_finish(w, stats);
}

}  // namespace crt
