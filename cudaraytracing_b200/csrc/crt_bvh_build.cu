// crt_bvh_build.cu — GPU BVH construction (replaces the host builder, reference include/BVH.h:37-84).
//
// Algorithm (DESIGN.md "BVH build"; the CPU statement of the same algorithm is oracle/orc_bvh.cpp
// build_new_bvh, and tests demand byte equality of nodes / order / leaf terminators):
//   1. per-triangle boxes, scene box by exact min/max reduction;
//   2. 63-bit Morton key of the box centre (21 bits/axis);
//   3. stable LSD radix sort of (key, face id), 8 passes x 8 bits;
//   4. Karras binary radix tree over the sorted keys (duplicates disambiguated by index);
//   5. bottom-up box refit with one atomic flag per internal node;
//   6. subtrees with <= thresh_n triangles become leaves (the reference's rule, BVH.h:57);
//      kept nodes are numbered by the rank of their radix index (exclusive scan of the keep flags);
//   7. emit 64-byte child-pair nodes and the per-slot triangle records.
// Every float operation is exact (min/max) or a single rounding shared with the CPU statement
// (this file is compiled with -fmad=false), so the result does not depend on thread scheduling.
#include "crt_gpu.h"
#include "crt_wide.cuh"

#include <algorithm>
#include <cstdio>
#include <vector>

namespace crt {

// ------------------------------------------------------------------------------------------
// small utilities
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void atomic_min_float(float* addr, float v) {
    if (v >= 0.0f) atomicMin((int*)addr, __float_as_int(v));
    else atomicMax((unsigned int*)addr, __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_float(float* addr, float v) {
    if (v >= 0.0f) atomicMax((int*)addr, __float_as_int(v));
    else atomicMin((unsigned int*)addr, __float_as_uint(v));
}

// exclusive scan of uint32, three phases; block = 256 threads x 4 items
static constexpr int kScanTile = 1024;

__global__ void k_scan_reduce(const uint32_t* __restrict__ in, uint32_t* __restrict__ block_sums, uint32_t n) {
    __shared__ uint32_t warp_sums[8];
    uint32_t base = blockIdx.x * kScanTile;
    uint32_t s = 0;
    for (int k = 0; k < 4; ++k) {
        uint32_t i = base + k * 256 + threadIdx.x;
        if (i < n) s += in[i];
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < 8; ++w) t += warp_sums[w];
        block_sums[blockIdx.x] = t;
    }
}

// single block: exclusive scan of block_sums in place, total written to *total (optional)
__global__ void k_scan_sums(uint32_t* __restrict__ sums, uint32_t n_blocks, uint32_t* __restrict__ total) {
    __shared__ uint32_t buf[1024];
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_blocks; base += 1024) {
        uint32_t i = base + threadIdx.x;
        uint32_t v = i < n_blocks ? sums[i] : 0;
        buf[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {          // Hillis-Steele inclusive
            uint32_t add = threadIdx.x >= (unsigned)o ? buf[threadIdx.x - o] : 0;
            __syncthreads();
            buf[threadIdx.x] += add;
            __syncthreads();
        }
        uint32_t incl = buf[threadIdx.x];
        uint32_t c = carry;
        if (i < n_blocks) sums[i] = c + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = c + incl;
        __syncthreads();
    }
    if (total && threadIdx.x == 0) *total = carry;
}

__global__ void k_scan_apply(const uint32_t* __restrict__ in, uint32_t* __restrict__ out,
                             const uint32_t* __restrict__ block_offsets, uint32_t n) {
    __shared__ uint32_t tsum[256];
    uint32_t base = blockIdx.x * kScanTile;
    // blocked arrangement: thread t owns items 4t..4t+3 of the tile
    uint32_t v[4];
    uint32_t s = 0;
    for (int k = 0; k < 4; ++k) {
        uint32_t i = base + threadIdx.x * 4 + k;
        v[k] = i < n ? in[i] : 0;
        s += v[k];
    }
    tsum[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
        uint32_t add = threadIdx.x >= (unsigned)o ? tsum[threadIdx.x - o] : 0;
        __syncthreads();
        tsum[threadIdx.x] += add;
        __syncthreads();
    }
    uint32_t run = block_offsets[blockIdx.x] + tsum[threadIdx.x] - s;
    for (int k = 0; k < 4; ++k) {
        uint32_t i = base + threadIdx.x * 4 + k;
        if (i < n) out[i] = run;
        run += v[k];
    }
}

// out may alias in. scratch must hold ceil(n/1024) uint32. total (device pointer) optional.
static cudaError_t exclusive_scan_u32(const uint32_t* in, uint32_t* out, uint32_t n, uint32_t* scratch, uint32_t* total,
                                      cudaStream_t st) {
    if (n == 0) {
        if (total) return cudaMemsetAsync(total, 0, sizeof(uint32_t), st);
        return cudaSuccess;
    }
    uint32_t nb = (n + kScanTile - 1) / kScanTile;
    k_scan_reduce<<<nb, 256, 0, st>>>(in, scratch, n);
    k_scan_sums<<<1, 1024, 0, st>>>(scratch, nb, total);
    k_scan_apply<<<nb, 256, 0, st>>>(in, out, scratch, n);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// stable LSD radix sort of (uint64 key, uint32 value), 8 bits per pass
// ------------------------------------------------------------------------------------------
static constexpr int kSortTile = 1024;   // 256 threads x 4 keys, striped: item r*256 + tid

__global__ void k_sort_hist(const uint64_t* __restrict__ keys, uint32_t n, int shift, uint32_t* __restrict__ ghist,
                            uint32_t n_tiles) {
    __shared__ uint32_t hist[256];
    hist[threadIdx.x] = 0;
    __syncthreads();
    uint32_t base = blockIdx.x * kSortTile;
    for (int r = 0; r < 4; ++r) {
        uint32_t i = base + r * 256 + threadIdx.x;
        if (i < n) atomicAdd(&hist[(uint32_t)(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    ghist[(size_t)threadIdx.x * n_tiles + blockIdx.x] = hist[threadIdx.x];   // digit-major
}

__global__ void k_sort_scatter(const uint64_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                               uint64_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, uint32_t n, int shift,
                               const uint32_t* __restrict__ ghist_scanned, uint32_t n_tiles) {
    __shared__ uint32_t cnt[4][8][256];      // [round][warp][digit] -> count, then start offset
    for (int k = threadIdx.x; k < 4 * 8 * 256; k += 256) ((uint32_t*)cnt)[k] = 0;
    __syncthreads();
    const uint32_t base = blockIdx.x * kSortTile;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t key[4];
    uint32_t val[4], rank[4], digit[4];
    bool valid[4];
    for (int r = 0; r < 4; ++r) {
        uint32_t i = base + r * 256 + threadIdx.x;
        valid[r] = i < n;
        key[r] = valid[r] ? keys_in[i] : 0;
        val[r] = valid[r] ? vals_in[i] : 0;
        digit[r] = (uint32_t)(key[r] >> shift) & 255u;
        // lanes with the same digit; invalid lanes get a private pseudo-digit
        unsigned m = __match_any_sync(0xffffffffu, valid[r] ? digit[r] : 256u + lane);
        rank[r] = __popc(m & ((1u << lane) - 1));
        if (valid[r] && rank[r] == 0) cnt[r][warp][digit[r]] = __popc(m);
    }
    __syncthreads();
    {   // thread d: running offset of digit d over (round, warp) in order
        const int d = threadIdx.x;
        uint32_t run = ghist_scanned[(size_t)d * n_tiles + blockIdx.x];
        for (int r = 0; r < 4; ++r)
            for (int w = 0; w < 8; ++w) {
                uint32_t c = cnt[r][w][d];
                cnt[r][w][d] = run;
                run += c;
            }
    }
    __syncthreads();
    for (int r = 0; r < 4; ++r) {
        if (!valid[r]) continue;
        uint32_t pos = cnt[r][warp][digit[r]] + rank[r];
        keys_out[pos] = key[r];
        vals_out[pos] = val[r];
    }
}

// The same sort for other callers (ordered ray batches, crt_render.cu): the low 8 * passes bits of the keys.
size_t radix_sort_hist_words(uint32_t n) { return 256 * (size_t)((n + kSortTile - 1) / kSortTile); }
size_t radix_sort_scratch_words(uint32_t n) { return (radix_sort_hist_words(n) + kScanTile - 1) / kScanTile + 1; }
cudaError_t radix_sort_pairs(uint64_t* k0, uint64_t* k1, uint32_t* v0, uint32_t* v1, uint32_t n, int passes, uint32_t* ghist,
                             uint32_t* scratch, cudaStream_t st, uint64_t** k_sorted, uint32_t** v_sorted) {
    const uint32_t n_tiles = (n + kSortTile - 1) / kSortTile;
    uint64_t *kin = k0, *kout = k1;
    uint32_t *vin = v0, *vout = v1;
    for (int pass = 0; pass < passes && n > 0; ++pass) {
        const int shift = pass * 8;
        k_sort_hist<<<n_tiles, 256, 0, st>>>(kin, n, shift, ghist, n_tiles);
        cudaError_t e = exclusive_scan_u32(ghist, ghist, 256 * n_tiles, scratch, nullptr, st);
        if (e != cudaSuccess) return e;
        k_sort_scatter<<<n_tiles, 256, 0, st>>>(kin, vin, kout, vout, n, shift, ghist, n_tiles);
        std::swap(kin, kout);
        std::swap(vin, vout);
    }
    *k_sorted = kin;
    *v_sorted = vin;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// build kernels
// ------------------------------------------------------------------------------------------
__global__ void k_tri_bounds(const float* __restrict__ verts, uint32_t n, float4* __restrict__ tlo, float4* __restrict__ thi,
                             float* __restrict__ scene_bounds /* lo[3], hi[3] */) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    if (i < n) {
        const float* v = verts + 9 * (size_t)i;
        for (int a = 0; a < 3; ++a) {
            lo[a] = fminf(fminf(v[a], v[3 + a]), v[6 + a]);
            hi[a] = fmaxf(fmaxf(v[a], v[3 + a]), v[6 + a]);
        }
        tlo[i] = make_float4(lo[0], lo[1], lo[2], 0.0f);
        thi[i] = make_float4(hi[0], hi[1], hi[2], 0.0f);
    }
    for (int a = 0; a < 3; ++a) {
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_down_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_down_sync(0xffffffffu, hi[a], o));
        }
    }
    if ((threadIdx.x & 31) == 0) {
        for (int a = 0; a < 3; ++a) {
            atomic_min_float(scene_bounds + a, lo[a]);
            atomic_max_float(scene_bounds + 3 + a, hi[a]);
        }
    }
}

__device__ __forceinline__ uint64_t expand21(uint64_t x) {
    x &= 0x1fffffull;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}
__device__ __forceinline__ uint64_t quant21(float c, float lo, float scale) {
    float f = (c - lo) * scale;
    int q = (int)f;
    if (q > 0x1fffff) q = 0x1fffff;
    if (q < 0) q = 0;
    return (uint64_t)q;
}

__global__ void k_morton(const float4* __restrict__ tlo, const float4* __restrict__ thi, uint32_t n,
                         const float* __restrict__ scene_bounds, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float slo[3] = {scene_bounds[0], scene_bounds[1], scene_bounds[2]};
    float scale[3];
    for (int a = 0; a < 3; ++a) {
        float ext = scene_bounds[3 + a] - slo[a];
        scale[a] = ext > 0.0f ? 2097152.0f / ext : 0.0f;
    }
    float4 lo = tlo[i], hi = thi[i];
    float cx = (lo.x + hi.x) * 0.5f, cy = (lo.y + hi.y) * 0.5f, cz = (lo.z + hi.z) * 0.5f;
    uint64_t qx = quant21(cx, slo[0], scale[0]), qy = quant21(cy, slo[1], scale[1]), qz = quant21(cz, slo[2], scale[2]);
    keys[i] = (expand21(qx) << 2) | (expand21(qy) << 1) | expand21(qz);
    vals[i] = i;
}

__device__ __forceinline__ int delta_fn(const uint64_t* __restrict__ key, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    uint64_t a = key[i], b = key[j];
    if (a == b) return 64 + __clz(i ^ j);
    return __clzll((long long)(a ^ b));
}

// Karras 2012, one thread per internal node i in [0, n-2]
__global__ void k_radix_tree(const uint64_t* __restrict__ key, int n, int* __restrict__ left, int* __restrict__ right,
                             int* __restrict__ first, int* __restrict__ last, int* __restrict__ parent_of_node,
                             int* __restrict__ parent_of_leaf) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int d = (delta_fn(key, n, i, i + 1) - delta_fn(key, n, i, i - 1)) >= 0 ? 1 : -1;
    int dmin = delta_fn(key, n, i, i - d);
    int lmax = 2;
    while (delta_fn(key, n, i, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (delta_fn(key, n, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta_fn(key, n, i, j);
    int s = 0, t = l;
    do {
        t = (t + 1) >> 1;
        if (delta_fn(key, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    int gamma = i + s * d + min(d, 0);
    int lo_i = min(i, j), hi_i = max(i, j);
    first[i] = lo_i;
    last[i] = hi_i;
    if (lo_i == gamma) { left[i] = ~gamma; parent_of_leaf[gamma] = i; }
    else { left[i] = gamma; parent_of_node[gamma] = i; }
    if (hi_i == gamma + 1) { right[i] = ~(gamma + 1); parent_of_leaf[gamma + 1] = i; }
    else { right[i] = gamma + 1; parent_of_node[gamma + 1] = i; }
    if (i == 0) parent_of_node[0] = -1;
}

// bottom-up refit: one thread per sorted slot; the second arrival at a node computes its box
__global__ void k_refit(int n, const uint32_t* __restrict__ order, const float4* __restrict__ tlo, const float4* __restrict__ thi,
                        const int* __restrict__ left, const int* __restrict__ right, const int* __restrict__ parent_of_node,
                        const int* __restrict__ parent_of_leaf, float4* __restrict__ blo, float4* __restrict__ bhi,
                        uint32_t* __restrict__ flags) {
    int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n) return;
    int node = parent_of_leaf[slot];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&flags[node], 1u) == 0) return;       // first arrival: the sibling finishes the job
        __threadfence();
        // child boxes were written by other threads of this launch: read and write them through
        // L2 (ld.cg / st.cg) so that no stale L1 line is used
        float4 llo, lhi, rlo, rhi;
        int l = left[node], r = right[node];
        if (l < 0) { uint32_t f = order[~l]; llo = tlo[f]; lhi = thi[f]; }
        else { llo = __ldcg(blo + l); lhi = __ldcg(bhi + l); }
        if (r < 0) { uint32_t f = order[~r]; rlo = tlo[f]; rhi = thi[f]; }
        else { rlo = __ldcg(blo + r); rhi = __ldcg(bhi + r); }
        __stcg(blo + node, make_float4(fminf(llo.x, rlo.x), fminf(llo.y, rlo.y), fminf(llo.z, rlo.z), 0.0f));
        __stcg(bhi + node, make_float4(fmaxf(lhi.x, rhi.x), fmaxf(lhi.y, rhi.y), fmaxf(lhi.z, rhi.z), 0.0f));
        node = parent_of_node[node];
    }
}

// ------------------------------------------------------------------------------------------
// PLOC topology (builders CRT_BUILDER_PLOC / PLOC8): bottom-up agglomeration over the Morton order instead of
// the Karras tree. Specification and CPU statement: oracle/orc_bvh.cpp build_ploc_tree (every array must come
// out bit-identical). One round = k_ploc_nn -> k_ploc_lower + scan -> k_ploc_merge; the host reads the number
// of clusters left after each round. k_ploc_finalize then walks the rounds in reverse (parents before
// children) to hand every node its slot range and writes the same arrays the Karras path produces
// (left/right/first/last/blo/bhi + the depth-first triangle order), so the leaf rule, the pair-node emitter
// and the 8-wide collapse run unchanged on either topology.
// A cluster is two float4: (box lo, ref bits) (box hi, triangle count); ref < 0: ~Morton position of a single
// triangle, else the creation index of the merge that made it.
// ------------------------------------------------------------------------------------------
static constexpr int kPlocRadius = 8;

__global__ void k_ploc_init(uint32_t n, const uint32_t* __restrict__ morton, const float4* __restrict__ tlo,
                            const float4* __restrict__ thi, float4* __restrict__ clo, float4* __restrict__ chi) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t f = morton[i];
    float4 lo = tlo[f], hi = thi[f];
    lo.w = __int_as_float(~(int)i);
    hi.w = __int_as_float(1);
    clo[i] = lo; chi[i] = hi;
}

// nearest neighbour by union-box area inside the window [k-R, k+R]; buddy k^1 first, then ascending j, strictly smaller wins
__global__ void __launch_bounds__(256) k_ploc_nn(int m, const float4* __restrict__ clo, const float4* __restrict__ chi,
                                                 int* __restrict__ nn) {
    __shared__ float4 slo[256 + 2 * kPlocRadius], shi[256 + 2 * kPlocRadius];
    const int base = (int)(blockIdx.x * 256) - kPlocRadius;
    for (int t = threadIdx.x; t < 256 + 2 * kPlocRadius; t += 256) {
        const int g = base + t;
        if (g >= 0 && g < m) { slo[t] = clo[g]; shi[t] = chi[g]; }
    }
    __syncthreads();
    const int k = (int)(blockIdx.x * 256 + threadIdx.x);
    if (k >= m) return;
    const float4 alo = slo[threadIdx.x + kPlocRadius], ahi = shi[threadIdx.x + kPlocRadius];
    auto area = [&](int dl) {
        const float4 b0 = slo[threadIdx.x + kPlocRadius + dl], b1 = shi[threadIdx.x + kPlocRadius + dl];
        const float ex = fmaxf(ahi.x, b1.x) - fminf(alo.x, b0.x);
        const float ey = fmaxf(ahi.y, b1.y) - fminf(alo.y, b0.y);
        const float ez = fmaxf(ahi.z, b1.z) - fminf(alo.z, b0.z);
        return (ex * ey + ey * ez) + ez * ex;
    };
    float best = FLT_MAX;
    int bj = -1;
    const int buddy = k ^ 1;                             // examined first: wins ties (oracle build_ploc_tree)
    if (buddy < m) { best = area(buddy - k); bj = buddy; }
#pragma unroll
    for (int dl = -kPlocRadius; dl <= kPlocRadius; ++dl) {
        const int j = k + dl;
        if (dl == 0 || j == buddy || j < 0 || j >= m) continue;
        const float a = area(dl);
        if (bj < 0 || a < best) { best = a; bj = j; }
    }
    nn[k] = bj;
}

// 1 for the lower member of every mutual pair (it becomes the merged cluster)
__global__ void k_ploc_lower(int m, const int* __restrict__ nn, uint32_t* __restrict__ lower) {
    const int k = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (k >= m) return;
    const int j = nn[k];
    lower[k] = (k < j && nn[j] == k) ? 1u : 0u;
}

__global__ void k_ploc_merge(int m, uint32_t created_base, const float4* __restrict__ clo, const float4* __restrict__ chi,
                             const int* __restrict__ nn, const uint32_t* __restrict__ lower_rank, float4* __restrict__ out_lo,
                             float4* __restrict__ out_hi, int* __restrict__ cl, int* __restrict__ cr, float4* __restrict__ nlo,
                             float4* __restrict__ nhi) {
    const int k = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (k >= m) return;
    const int j = nn[k];
    const bool mutual = nn[j] == k;
    if (mutual && k > j) return;                         // the upper member's place is dropped
    // places dropped before k = upper members before k = lower members before k - pairs still open at k
    int open = 0;
    for (int l = max(0, k - kPlocRadius); l < k; ++l) {
        const int jl = nn[l];
        if (jl >= k && nn[jl] == l) ++open;
    }
    const uint32_t lr = lower_rank[k];
    const int pos = k - ((int)lr - open);
    float4 lo = clo[k], hi = chi[k];
    if (mutual) {
        const float4 lo2 = clo[j], hi2 = chi[j];
        const int id = (int)(created_base + lr);
        const int cnt = __float_as_int(hi.w) + __float_as_int(hi2.w);
        cl[id] = __float_as_int(lo.w);
        cr[id] = __float_as_int(lo2.w);
        lo = make_float4(fminf(lo.x, lo2.x), fminf(lo.y, lo2.y), fminf(lo.z, lo2.z), __int_as_float(id));
        hi = make_float4(fmaxf(hi.x, hi2.x), fmaxf(hi.y, hi2.y), fmaxf(hi.z, hi2.z), __int_as_float(cnt));
        nlo[id] = lo; nhi[id] = hi;
    }
    out_lo[pos] = lo; out_hi[pos] = hi;
}

// merges [c_begin, c_end) of one round; node id = ni - 1 - creation index; the slot range of a node was written
// by its parent in an earlier launch (later round), the root's by k_ploc_root
__global__ void k_ploc_root(int n, int* __restrict__ first, int* __restrict__ last) { first[0] = 0; last[0] = n - 1; }
__global__ void k_ploc_finalize(uint32_t c_begin, uint32_t c_end, int ni, const int* __restrict__ cl, const int* __restrict__ cr,
                                const float4* __restrict__ nlo, const float4* __restrict__ nhi, const uint32_t* __restrict__ morton,
                                int* __restrict__ left, int* __restrict__ right, int* __restrict__ first, int* __restrict__ last,
                                float4* __restrict__ blo, float4* __restrict__ bhi, uint32_t* __restrict__ order) {
    const uint32_t c = c_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= c_end) return;
    const int nd = ni - 1 - (int)c;
    const int f = first[nd], l = last[nd];
    float4 lo = nlo[c], hi = nhi[c];
    lo.w = 0.0f; hi.w = 0.0f;
    blo[nd] = lo; bhi[nd] = hi;
    const int a = cl[c], b = cr[c];
    const int lcount = a < 0 ? 1 : __float_as_int(nhi[a].w);
    if (a < 0) { left[nd] = ~f; order[f] = morton[~a]; }
    else { const int ch = ni - 1 - a; left[nd] = ch; first[ch] = f; last[ch] = f + lcount - 1; }
    const int g = f + lcount;
    if (b < 0) { right[nd] = ~g; order[g] = morton[~b]; }
    else { const int ch = ni - 1 - b; right[nd] = ch; first[ch] = g; last[ch] = l; }
}

__global__ void k_keep_flags(int n_internal, const int* __restrict__ first, const int* __restrict__ last, uint32_t thresh,
                             uint32_t* __restrict__ keep) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_internal) return;
    keep[i] = (uint32_t)(last[i] - first[i] + 1) > thresh ? 1u : 0u;
}

__global__ void k_emit_nodes(int n_internal, const uint32_t* __restrict__ keep, const uint32_t* __restrict__ rank,
                             const int* __restrict__ left, const int* __restrict__ right, const int* __restrict__ first,
                             const int* __restrict__ last, const uint32_t* __restrict__ order, const float4* __restrict__ tlo,
                             const float4* __restrict__ thi, const float4* __restrict__ blo, const float4* __restrict__ bhi,
                             float4* __restrict__ nodes, uint8_t* __restrict__ last_flag) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_internal || !keep[i]) return;
    float4 lo[2], hi[2];
    int ref[2], cnt[2];
    for (int w = 0; w < 2; ++w) {
        int c = w == 0 ? left[i] : right[i];
        if (c < 0) {                       // single triangle
            uint32_t f = order[~c];
            lo[w] = tlo[f]; hi[w] = thi[f];
            ref[w] = c; cnt[w] = 1;
            last_flag[~c] = 1;
        } else {
            lo[w] = blo[c]; hi[w] = bhi[c];
            cnt[w] = last[c] - first[c] + 1;
            if (keep[c]) ref[w] = (int)rank[c];
            else { ref[w] = ~first[c]; last_flag[last[c]] = 1; }
        }
    }
    float4* o = nodes + 4 * (size_t)rank[i];
    o[0] = make_float4(lo[0].x, hi[0].x, lo[0].y, hi[0].y);
    o[1] = make_float4(lo[1].x, hi[1].x, lo[1].y, hi[1].y);
    o[2] = make_float4(lo[0].z, hi[0].z, lo[1].z, hi[1].z);
    o[3] = make_float4(__int_as_float(ref[0]), __int_as_float(ref[1]), __int_as_float(cnt[0]), __int_as_float(cnt[1]));
}

// the whole scene is one leaf: one node, child 1 absent with an inverted box
__global__ void k_emit_single_leaf(int n, const float* __restrict__ scene_bounds, float4* __restrict__ nodes,
                                   uint8_t* __restrict__ last_flag) {
    nodes[0] = make_float4(scene_bounds[0], scene_bounds[3], scene_bounds[1], scene_bounds[4]);
    nodes[1] = make_float4(FLT_MAX, -FLT_MAX, FLT_MAX, -FLT_MAX);
    nodes[2] = make_float4(scene_bounds[2], scene_bounds[5], FLT_MAX, -FLT_MAX);
    nodes[3] = make_float4(__int_as_float(~0), __int_as_float(kEmptyChild), __int_as_float(n), __int_as_float(0));
    last_flag[n - 1] = 1;
}

// per-slot triangle records (DeviceTriangle::DeviceTriangle, reference DeviceTriangle.cuh:22-33)
__global__ void k_emit_tris(uint32_t n, const uint32_t* __restrict__ order, const uint8_t* __restrict__ last_flag,
                            const float* __restrict__ verts, const float4* __restrict__ face_shade,
                            float4* __restrict__ tri_geom, float4* __restrict__ tri_shade) {
    uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n) return;
    uint32_t f = order[slot];
    const float* v = verts + 9 * (size_t)f;
    float4 sh = face_shade[f];
    uint32_t fw = f | (last_flag[slot] ? kLastBit : 0u);
    tri_geom[3 * (size_t)slot + 0] = make_float4(v[0], v[1], v[2], __uint_as_float(fw));
    tri_geom[3 * (size_t)slot + 1] = make_float4(v[3] - v[0], v[4] - v[1], v[5] - v[2], sh.w);
    tri_geom[3 * (size_t)slot + 2] = make_float4(v[6] - v[0], v[7] - v[1], v[8] - v[2], 0.0f);
    tri_shade[slot] = sh;
}

// ------------------------------------------------------------------------------------------
// 8-wide compressed nodes (builder CRT_BUILDER_LBVH8): collapse of the radix tree, one wide-tree level
// per pass. CPU statement: oracle/orc_bvh.cpp build_wide8_bvh (byte-identical output required).
//   k_wide_collapse  one thread per wide node of the level: greedy collapse (largest-area expandable
//                    child first) and greedy slot assignment by octant; counts its internal children
//                    and leaf triangles
//   (two exclusive scans: where the children / leaf triangles of every node of the level start)
//   k_wide_emit      quantises the child boxes outwards in double arithmetic, writes the 80-byte node,
//                    the next level's work list and the leaf triangles' slots
// ------------------------------------------------------------------------------------------
static constexpr int kWideEmpty = 0x7fffffff;
static constexpr int kWideWholeScene = 0x7ffffffe;     // the only child of the root when n <= thresh

struct WideBuildView {
    const int *left, *right, *first, *last;
    const float4 *blo, *bhi, *tlo, *thi;
    const uint32_t* order;                 // Morton-sorted slot -> face id
    const float* scene_bounds;
    int n_tris;
    uint32_t thresh;
};

__device__ __forceinline__ float wide_area(float4 lo, float4 hi) {
    float ex = hi.x - lo.x, ey = hi.y - lo.y, ez = hi.z - lo.z;
    return (ex * ey + ey * ez) + ez * ex;
}
__device__ __forceinline__ void wide_child_box(const WideBuildView& v, int ref, float4& lo, float4& hi) {
    if (ref == kWideWholeScene) {
        lo = make_float4(v.scene_bounds[0], v.scene_bounds[1], v.scene_bounds[2], 0.0f);
        hi = make_float4(v.scene_bounds[3], v.scene_bounds[4], v.scene_bounds[5], 0.0f);
    } else if (ref < 0) {
        const uint32_t f = v.order[~ref];
        lo = v.tlo[f]; hi = v.thi[f];
    } else {
        lo = v.blo[ref]; hi = v.bhi[ref];
    }
}
__device__ __forceinline__ void wide_make_child(const WideBuildView& v, int c, int& ref, int& cnt, float& sa) {
    ref = c;
    sa = 0.0f;
    if (c < 0) { cnt = 1; return; }
    const int m = v.last[c] - v.first[c] + 1;
    if ((uint32_t)m > v.thresh) { cnt = 0; sa = wide_area(v.blo[c], v.bhi[c]); }     // expandable
    else cnt = m;
}

__global__ void k_wide_collapse(WideBuildView v, uint32_t n_level, const int* __restrict__ work, int* __restrict__ tmp_ref,
                                int* __restrict__ tmp_cnt, uint32_t* __restrict__ cnt_int, uint32_t* __restrict__ cnt_tri) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_level) return;
    const int r = work[i];
    int ref[8], cnt[8];
    float sa[8];
    int k = 0;
    float4 nlo, nhi;
    if (r < 0) {
        ref[0] = kWideWholeScene; cnt[0] = v.n_tris; sa[0] = 0.0f;
        k = 1;
        wide_child_box(v, kWideWholeScene, nlo, nhi);
    } else {
        wide_make_child(v, v.left[r], ref[0], cnt[0], sa[0]);
        wide_make_child(v, v.right[r], ref[1], cnt[1], sa[1]);
        k = 2;
        nlo = v.blo[r]; nhi = v.bhi[r];
        while (k < 8) {
            int best = -1;
            float best_area = 0.0f;
            for (int j = 0; j < k; ++j) {
                if (cnt[j] != 0) continue;
                if (best < 0 || sa[j] > best_area) { best = j; best_area = sa[j]; }
            }
            if (best < 0) break;
            const int c = ref[best];
            for (int j = k; j > best + 1; --j) { ref[j] = ref[j - 1]; cnt[j] = cnt[j - 1]; sa[j] = sa[j - 1]; }
            wide_make_child(v, v.left[c], ref[best], cnt[best], sa[best]);
            wide_make_child(v, v.right[c], ref[best + 1], cnt[best + 1], sa[best + 1]);
            ++k;
        }
    }
    // greedy slot assignment: largest +-(child centre - node centre) sum first
    const float cx = (nlo.x + nhi.x) * 0.5f, cy = (nlo.y + nhi.y) * 0.5f, cz = (nlo.z + nhi.z) * 0.5f;
    float dx[8], dy[8], dz[8];
    for (int j = 0; j < k; ++j) {
        float4 lo, hi;
        wide_child_box(v, ref[j], lo, hi);
        dx[j] = (lo.x + hi.x) * 0.5f - cx;
        dy[j] = (lo.y + hi.y) * 0.5f - cy;
        dz[j] = (lo.z + hi.z) * 0.5f - cz;
    }
    int slot_of[8], child_in[8];
    for (int j = 0; j < 8; ++j) { slot_of[j] = -1; child_in[j] = -1; }
    for (int it = 0; it < k; ++it) {
        int bj = -1, bs = -1;
        float bc = 0.0f;
        for (int j = 0; j < k; ++j) {
            if (slot_of[j] >= 0) continue;
            for (int sl = 0; sl < 8; ++sl) {
                if (child_in[sl] >= 0) continue;
                const float tx = (sl & 1) ? dx[j] : -dx[j], ty = (sl & 2) ? dy[j] : -dy[j], tz = (sl & 4) ? dz[j] : -dz[j];
                const float c = (tx + ty) + tz;
                if (bj < 0 || c > bc) { bj = j; bs = sl; bc = c; }
            }
        }
        slot_of[bj] = bs;
        child_in[bs] = bj;
    }
    uint32_t ni = 0, nt = 0;
    for (int sl = 0; sl < 8; ++sl) {
        const int j = child_in[sl];
        tmp_ref[8 * (size_t)i + sl] = j < 0 ? kWideEmpty : ref[j];
        tmp_cnt[8 * (size_t)i + sl] = j < 0 ? 0 : cnt[j];
        if (j >= 0) { if (cnt[j] == 0) ++ni; else nt += (uint32_t)cnt[j]; }
    }
    cnt_int[i] = ni;
    cnt_tri[i] = nt;
}

__device__ __forceinline__ int exp_of_double(double x) {        // floor(log2 x), x a positive normal double
    return (int)((__double_as_longlong(x) >> 52) & 0x7ff) - 1023;
}

__global__ void k_wide_emit(WideBuildView v, uint32_t n_level, uint32_t level_start, uint32_t next_start, uint32_t tri_cursor,
                            const int* __restrict__ work, const int* __restrict__ tmp_ref, const int* __restrict__ tmp_cnt,
                            const uint32_t* __restrict__ off_int, const uint32_t* __restrict__ off_tri, uint4* __restrict__ nodes,
                            int* __restrict__ work_next, uint32_t* __restrict__ order8, uint8_t* __restrict__ last8) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_level) return;
    const int r = work[i];
    float4 nlo, nhi;
    if (r < 0) wide_child_box(v, kWideWholeScene, nlo, nhi);
    else { nlo = v.blo[r]; nhi = v.bhi[r]; }
    const float plo[3] = {nlo.x, nlo.y, nlo.z}, phi[3] = {nhi.x, nhi.y, nhi.z};
    uint32_t eb[3];
    double cell[3];
    for (int a = 0; a < 3; ++a) {
        const double ext = (double)phi[a] - (double)plo[a];
        if (!(ext > 0.0)) { eb[a] = 0; cell[a] = 0.0; continue; }
        int e = exp_of_double(ext / 255.0);
        if (ldexp(255.0, e) < ext) e += 1;
        int b = e + 127;
        if (b < 1) b = 1;
        if (b > 254) b = 254;
        eb[a] = (uint32_t)b;
        cell[a] = ldexp(1.0, b - 127);
    }
    const uint32_t child_base = next_start + off_int[i];
    const uint32_t tri_base = tri_cursor + off_tri[i];
    uint32_t meta[2] = {0, 0}, q[6][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}, {0, 0}, {0, 0}};
    uint32_t imask = 0, n_internal = 0, tri_off = 0;
    for (int sl = 0; sl < 8; ++sl) {
        const int ref = tmp_ref[8 * (size_t)i + sl];
        const int cnt = tmp_cnt[8 * (size_t)i + sl];
        const int sh = 8 * (sl & 3), w = sl >> 2;
        if (ref == kWideEmpty) {
            for (int a = 0; a < 3; ++a) q[a][w] |= 255u << sh;              // inverted box: lo 255, hi 0
            continue;
        }
        float4 lo, hi;
        wide_child_box(v, ref, lo, hi);
        const float clo[3] = {lo.x, lo.y, lo.z}, chi[3] = {hi.x, hi.y, hi.z};
        for (int a = 0; a < 3; ++a) {
            int ql = 0, qh = 0;
            if (cell[a] > 0.0) {
                const double fl = floor(((double)clo[a] - (double)plo[a]) / cell[a]);
                const double fh = ceil(((double)chi[a] - (double)plo[a]) / cell[a]);
                ql = fl < 0.0 ? 0 : (fl > 255.0 ? 255 : (int)fl);
                qh = fh < 0.0 ? 0 : (fh > 255.0 ? 255 : (int)fh);
            }
            q[a][w] |= (uint32_t)ql << sh;
            q[3 + a][w] |= (uint32_t)qh << sh;
        }
        if (cnt == 0) {
            meta[w] |= 0x80u << sh;
            imask |= 1u << sl;
            work_next[off_int[i] + n_internal] = ref;
            ++n_internal;
        } else {
            meta[w] |= (1u + tri_off) << sh;
            const int first = ref == kWideWholeScene ? 0 : (ref < 0 ? ~ref : v.first[ref]);
            for (int t = 0; t < cnt; ++t) order8[tri_base + tri_off + t] = v.order[first + t];
            last8[tri_base + tri_off + cnt - 1] = 1;
            tri_off += (uint32_t)cnt;
        }
    }
    uint4* o = nodes + 5 * (size_t)(level_start + i);
    o[0] = make_uint4(__float_as_uint(plo[0]), __float_as_uint(plo[1]), __float_as_uint(plo[2]),
                      eb[0] | (eb[1] << 8) | (eb[2] << 16) | (imask << 24));
    o[1] = make_uint4(child_base, tri_base, meta[0], meta[1]);
    o[2] = make_uint4(q[0][0], q[0][1], q[1][0], q[1][1]);
    o[3] = make_uint4(q[2][0], q[2][1], q[3][0], q[3][1]);
    o[4] = make_uint4(q[4][0], q[4][1], q[5][0], q[5][1]);
}

// ------------------------------------------------------------------------------------------
// host driver
// ------------------------------------------------------------------------------------------
int build_bvh_device(DeviceScene& ds, const float* d_verts, const float4* d_face_shade, uint32_t n, uint32_t thresh_n,
                     int builder, cudaStream_t st, float* build_ms) {
    const bool wide = (builder & 1) != 0;               // bit 0: 8-wide node layout, bit 1: PLOC topology
    const bool ploc = (builder & 2) != 0;
    if (thresh_n < 1) thresh_n = 1;
    if (wide && thresh_n > 15) thresh_n = 15;            // 7-bit leaf offsets inside a wide node
    const uint32_t n_tiles = (n + kSortTile - 1) / kSortTile;
    const int nb = (int)((n + 255) / 256);
    uint32_t n_kept = 0;
    const float init_bounds[6] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX};

    ds.n_tris = n;
    ds.n_nodes = 0;
    ds.wide = wide;
    ds.builder = builder;
    if (n == 0) { if (build_ms) *build_ms = 0; return CRT_OK; }

    // every temporary lives until the build has finished
    Event ev0, ev1;
    DevBuf<float4> tlo, thi, blo, bhi, pc_lo[2], pc_hi[2], pn_lo, pn_hi;
    DevBuf<float> bounds;
    DevBuf<uint64_t> keys0, keys1;
    DevBuf<uint32_t> vals0, vals1, ghist, scratch, flags, keep, rank, d_total, p_lower, p_rank, p_order;
    DevBuf<int> left, right, first, last, pnode, pleaf, p_nn, p_cl, p_cr;
    DevBuf<uint4> wnodes;
    DevBuf<int> work0, work1, tmp_ref, tmp_cnt;
    DevBuf<uint32_t> cnt_int, cnt_tri, off_int, off_tri, order8, d_tot2;
    DevBuf<uint8_t> last8;
    CRT_CUDA(create(ev0));
    CRT_CUDA(create(ev1));
    CRT_CUDA(tlo.alloc(n));
    CRT_CUDA(thi.alloc(n));
    CRT_CUDA(bounds.alloc(6));
    CRT_CUDA(keys0.alloc(n));
    CRT_CUDA(keys1.alloc(n));
    CRT_CUDA(vals0.alloc(n));
    CRT_CUDA(vals1.alloc(n));
    CRT_CUDA(ghist.alloc(256 * (size_t)n_tiles));
    CRT_CUDA(scratch.alloc(std::max((256 * (size_t)n_tiles + kScanTile - 1) / kScanTile, ((size_t)n + kScanTile - 1) / kScanTile) + 1));
    CRT_CUDA(d_total.alloc(1));
    CRT_CUDA(ds.order.alloc(n));
    CRT_CUDA(ds.last.alloc(n));
    CRT_CUDA(ds.tri_geom.alloc(3 * (size_t)n));
    CRT_CUDA(ds.tri_shade.alloc(n));
    CRT_CUDA(cudaMemsetAsync(ds.last.get(), 0, n, st));
    CRT_CUDA(cudaMemcpyAsync(bounds.get(), init_bounds, sizeof(init_bounds), cudaMemcpyHostToDevice, st));

    CRT_CUDA(cudaEventRecord(ev0.get(), st));
    k_tri_bounds<<<nb, 256, 0, st>>>(d_verts, n, tlo.get(), thi.get(), bounds.get());
    k_morton<<<nb, 256, 0, st>>>(tlo.get(), thi.get(), n, bounds.get(), keys0.get(), vals0.get());
    {
        uint64_t* sorted_keys = nullptr;                 // 8 passes: keys0 / vals0 again
        uint32_t* sorted_vals = nullptr;
        CRT_CUDA(radix_sort_pairs(keys0.get(), keys1.get(), vals0.get(), vals1.get(), n, 8, ghist.get(), scratch.get(), st, &sorted_keys,
                                  &sorted_vals));
        CRT_CUDA(cudaMemcpyAsync(ds.order.get(), sorted_vals, sizeof(uint32_t) * n, cudaMemcpyDeviceToDevice, st));
    }
    CRT_CUDA(cudaGetLastError());

    if (n <= thresh_n) {
        n_kept = 1;
        if (!wide) {
            CRT_CUDA(ds.nodes.alloc(4));
            k_emit_single_leaf<<<1, 1, 0, st>>>((int)n, bounds.get(), ds.nodes.get(), ds.last.get());
        }
    } else {
        const uint32_t ni = n - 1;
        const int nbi = (int)((ni + 255) / 256);
        CRT_CUDA(left.alloc(ni));
        CRT_CUDA(right.alloc(ni));
        CRT_CUDA(first.alloc(ni));
        CRT_CUDA(last.alloc(ni));
        CRT_CUDA(pnode.alloc(ni));
        CRT_CUDA(pleaf.alloc(n));
        CRT_CUDA(blo.alloc(ni));
        CRT_CUDA(bhi.alloc(ni));
        CRT_CUDA(flags.alloc(ni));
        CRT_CUDA(keep.alloc(ni));
        CRT_CUDA(rank.alloc(ni));
        if (!ploc) {
            CRT_CUDA(cudaMemsetAsync(flags.get(), 0, sizeof(uint32_t) * ni, st));
            k_radix_tree<<<nbi, 256, 0, st>>>(keys0.get(), (int)n, left.get(), right.get(), first.get(), last.get(), pnode.get(), pleaf.get());
            k_refit<<<nb, 256, 0, st>>>((int)n, ds.order.get(), tlo.get(), thi.get(), left.get(), right.get(), pnode.get(), pleaf.get(), blo.get(),
                                        bhi.get(), flags.get());
        } else {
            for (int b = 0; b < 2; ++b) {
                CRT_CUDA(pc_lo[b].alloc(n));
                CRT_CUDA(pc_hi[b].alloc(n));
            }
            CRT_CUDA(pn_lo.alloc(ni));
            CRT_CUDA(pn_hi.alloc(ni));
            CRT_CUDA(p_nn.alloc(n));
            CRT_CUDA(p_cl.alloc(ni));
            CRT_CUDA(p_cr.alloc(ni));
            CRT_CUDA(p_lower.alloc(n));
            CRT_CUDA(p_rank.alloc(n));
            CRT_CUDA(p_order.alloc(n));
            k_ploc_init<<<nb, 256, 0, st>>>(n, ds.order.get(), tlo.get(), thi.get(), pc_lo[0].get(), pc_hi[0].get());
            std::vector<uint32_t> round_start;            // creation index at which every round begins
            uint32_t m = n, created = 0;
            int cur = 0;
            while (m > 1) {
                const int nbm = (int)((m + 255) / 256);
                k_ploc_nn<<<nbm, 256, 0, st>>>((int)m, pc_lo[cur].get(), pc_hi[cur].get(), p_nn.get());
                k_ploc_lower<<<nbm, 256, 0, st>>>((int)m, p_nn.get(), p_lower.get());
                CRT_CUDA(exclusive_scan_u32(p_lower.get(), p_rank.get(), m, scratch.get(), d_total.get(), st));
                k_ploc_merge<<<nbm, 256, 0, st>>>((int)m, created, pc_lo[cur].get(), pc_hi[cur].get(), p_nn.get(), p_rank.get(), pc_lo[cur ^ 1].get(),
                                                  pc_hi[cur ^ 1].get(), p_cl.get(), p_cr.get(), pn_lo.get(), pn_hi.get());
                uint32_t merged = 0;
                CRT_CUDA(cudaMemcpyAsync(&merged, d_total.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
                CRT_CUDA(cudaStreamSynchronize(st));
                if (merged == 0 || merged > m / 2) { set_error("PLOC: a round merged nothing"); return CRT_ERR_STATE; }
                round_start.push_back(created);
                // Every round adds at most one level, so the number of rounds bounds the depth of the tree. The pair-node
                // traversal pushes onto a stack of kStackSize entries without a bounds check (a Karras tree cannot be deeper
                // than 63 Morton bits + duplicate levels; PLOC has no such bound: boxes that grow geometrically merge one
                // pair per round, a chain of depth ~n), and every round costs a host synchronisation.
                if (round_start.size() >= (size_t)(wide ? 1024 : kStackSize - 1)) {
                    set_error("PLOC: the agglomeration needs more rounds than the traversal stack is deep (" + std::to_string(round_start.size()) +
                              "); build this scene with CRT_BUILDER_LBVH / CRT_BUILDER_LBVH8");
                    return CRT_ERR_STATE;
                }
                created += merged;
                m -= merged;
                cur ^= 1;
            }
            if (created != ni) { set_error("PLOC: merge count mismatch"); return CRT_ERR_STATE; }
            round_start.push_back(created);
            k_ploc_root<<<1, 1, 0, st>>>((int)n, first.get(), last.get());
            for (size_t r = round_start.size() - 1; r-- > 0;) {
                const uint32_t c0 = round_start[r], c1 = round_start[r + 1];
                k_ploc_finalize<<<(int)((c1 - c0 + 255) / 256), 256, 0, st>>>(c0, c1, (int)ni, p_cl.get(), p_cr.get(), pn_lo.get(), pn_hi.get(),
                                                                               ds.order.get(), left.get(), right.get(), first.get(), last.get(),
                                                                               blo.get(), bhi.get(), p_order.get());
            }
            std::swap(ds.order, p_order);                 // depth-first order replaces the Morton order
        }
        k_keep_flags<<<nbi, 256, 0, st>>>((int)ni, first.get(), last.get(), thresh_n, keep.get());
        CRT_CUDA(exclusive_scan_u32(keep.get(), rank.get(), ni, scratch.get(), d_total.get(), st));
        CRT_CUDA(cudaMemcpyAsync(&n_kept, d_total.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        CRT_CUDA(cudaStreamSynchronize(st));
        if (!wide) {
            CRT_CUDA(ds.nodes.alloc(4 * (size_t)n_kept));
            k_emit_nodes<<<nbi, 256, 0, st>>>((int)ni, keep.get(), rank.get(), left.get(), right.get(), first.get(), last.get(), ds.order.get(),
                                              tlo.get(), thi.get(), blo.get(), bhi.get(), ds.nodes.get(), ds.last.get());
        }
    }
    if (wide) {
        // breadth-first collapse into 80-byte nodes; at most one wide node per expandable radix node
        const size_t cap = std::max<uint32_t>(n_kept, 1);
        CRT_CUDA(wnodes.alloc(5 * cap));
        CRT_CUDA(work0.alloc(cap));
        CRT_CUDA(work1.alloc(cap));
        CRT_CUDA(tmp_ref.alloc(8 * cap));
        CRT_CUDA(tmp_cnt.alloc(8 * cap));
        CRT_CUDA(cnt_int.alloc(cap));
        CRT_CUDA(cnt_tri.alloc(cap));
        CRT_CUDA(off_int.alloc(cap));
        CRT_CUDA(off_tri.alloc(cap));
        CRT_CUDA(d_tot2.alloc(2));
        CRT_CUDA(order8.alloc(n));
        CRT_CUDA(last8.alloc(n));
        CRT_CUDA(cudaMemsetAsync(last8.get(), 0, n, st));
        WideBuildView v;
        v.left = left.get(); v.right = right.get(); v.first = first.get(); v.last = last.get(); v.blo = blo.get(); v.bhi = bhi.get();
        v.tlo = tlo.get(); v.thi = thi.get(); v.order = ds.order.get(); v.scene_bounds = bounds.get(); v.n_tris = (int)n; v.thresh = thresh_n;
        const int root = n <= thresh_n ? -1 : 0;
        CRT_CUDA(cudaMemcpyAsync(work0.get(), &root, sizeof(int), cudaMemcpyHostToDevice, st));
        uint32_t level_start = 0, n_level = 1, tri_cursor = 0, levels = 0;
        int *wcur = work0.get(), *wnext = work1.get();
        while (n_level > 0) {
            // the traversal stack holds one entry per level (crt_wide.cuh kWideStack)
            if (++levels > (uint32_t)kWideStack) { set_error("wide BVH: tree deeper than the traversal stack"); return CRT_ERR_STATE; }
            if ((size_t)level_start + n_level > cap) { set_error("wide BVH: node bound exceeded"); return CRT_ERR_STATE; }
            const int nbl = (int)((n_level + 127) / 128);
            k_wide_collapse<<<nbl, 128, 0, st>>>(v, n_level, wcur, tmp_ref.get(), tmp_cnt.get(), cnt_int.get(), cnt_tri.get());
            CRT_CUDA(exclusive_scan_u32(cnt_int.get(), off_int.get(), n_level, scratch.get(), d_tot2.get(), st));
            CRT_CUDA(exclusive_scan_u32(cnt_tri.get(), off_tri.get(), n_level, scratch.get(), d_tot2.get() + 1, st));
            uint32_t tot[2] = {0, 0};
            CRT_CUDA(cudaMemcpyAsync(tot, d_tot2.get(), sizeof(tot), cudaMemcpyDeviceToHost, st));
            CRT_CUDA(cudaStreamSynchronize(st));
            k_wide_emit<<<nbl, 128, 0, st>>>(v, n_level, level_start, level_start + n_level, tri_cursor, wcur, tmp_ref.get(), tmp_cnt.get(),
                                             off_int.get(), off_tri.get(), wnodes.get(), wnext, order8.get(), last8.get());
            CRT_CUDA(cudaGetLastError());
            level_start += n_level;
            n_level = tot[0];
            tri_cursor += tot[1];
            std::swap(wcur, wnext);
        }
        if (tri_cursor != n) { set_error("wide BVH: triangle count mismatch"); return CRT_ERR_STATE; }
        n_kept = level_start;
        CRT_CUDA(ds.nodes.alloc(5 * (size_t)n_kept));
        CRT_CUDA(cudaMemcpyAsync(ds.nodes.get(), wnodes.get(), sizeof(uint4) * 5 * (size_t)n_kept, cudaMemcpyDeviceToDevice, st));
        std::swap(ds.order, order8);
        std::swap(ds.last, last8);
    }
    k_emit_tris<<<nb, 256, 0, st>>>(n, ds.order.get(), ds.last.get(), d_verts, d_face_shade, ds.tri_geom.get(), ds.tri_shade.get());
    CRT_CUDA(cudaGetLastError());
    CRT_CUDA(cudaEventRecord(ev1.get(), st));
    CRT_CUDA(cudaStreamSynchronize(st));
    CRT_CUDA(cudaMemcpy(ds.bounds, bounds.get(), sizeof(float) * 6, cudaMemcpyDeviceToHost));
    ds.n_nodes = n_kept;
    if (build_ms) CRT_CUDA(cudaEventElapsedTime(build_ms, ev0.get(), ev1.get()));
    return CRT_OK;
}

}  // namespace crt
