// crt_wide.cuh — traversal of the 8-wide compressed BVH (builder CRT_BUILDER_LBVH8).
//
// Node layout (80 bytes = five 16-byte words; built by crt_bvh_build.cu, stated on the CPU by
// oracle/orc_bvh.cpp build_wide8_bvh, byte-identical):
//   w0: origin p (3 floats), {ex, ey, ez, imask} bytes      scale_k = float with exponent field e_k
//   w1: child_base, tri_base, meta[0..3], meta[4..7]        meta: 0 empty, 0x80 node, 1 + offset leaf
//   w2: qlo_x[0..7], qlo_y[0..7]   w3: qlo_z[0..7], qhi_x[0..7]   w4: qhi_y[0..7], qhi_z[0..7]
// child box k = p + q * scale per axis; the internal child in slot s is node
// child_base + popcount(imask below s); a leaf child starts at triangle slot tri_base + offset and
// runs to the terminator bit of tri_geom.
//
// Per-ray rule = oracle/orc_bvh.cpp wide8_intersect (same visits in the same order, so the oracle's
// node/triangle counts are the algorithmic ones): conservative quantised slabs, children visited
// front to back by slot ^ octant (descending), the leaf children of a node tested before descending,
// one stack entry per node with hit children left. The (t, face) result equals the pair-node BVH's
// and brute force's: conservative boxes make the closest hit independent of the tree.
#pragma once
#include "crt_device.cuh"

namespace crt {

static constexpr int kWideStack = 48;      // one entry per wide-tree level at most; the builder refuses deeper trees

// byte k of w as the float 32768 + byte, exactly: PRMT puts the byte into mantissa bits 8..15 under the exponent of 2^15.
// The bias is folded into the per-axis addend of the plane distances (a - 32768 b, one FFMA per axis and node), so a plane
// costs one PRMT and one FFMA. (I2F.U8 is a quarter-rate XU instruction; PRMT under 2^23 needed an FADD per plane to
// remove the bias: 48 per node step, profiles/r02_s01.md.)
// (the constant lives in a register and the selector is the immediate: with the constant as the immediate the compiler
//  spends a move per PRMT on the selector.)
CRT_DEV uint32_t wide_bias_bits(uint32_t ni) { return 0x47000000u | (ni >> 31); }      // ni < 2^31: the compiler cannot fold it
CRT_DEV float wide_biased(uint32_t w, int k, uint32_t kb = 0x47000000u) { return __uint_as_float(__byte_perm(w, kb, 0x7504u | ((uint32_t)k << 4))); }
static constexpr float kWideBias = 32768.0f;
// byte k of w as a float (slow path only)
CRT_DEV float wide_byte(uint32_t w, int k) { return wide_biased(w, k) - kWideBias; }

// 4-bit mask of the non-zero bytes of w (bit k = byte k != 0)
CRT_DEV uint32_t wide_nonzero_bytes(uint32_t w) {
    const uint32_t t = (w | ((w & 0x7f7f7f7fu) + 0x7f7f7f7fu)) & 0x80808080u;      // bit 7 of every non-zero byte
    return (((t >> 7) * 0x01020408u) >> 24) & 0xfu;                                // bits 0, 8, 16, 24 -> bits 24..27
}

struct WideStep {
    uint32_t node_hits, leaf_hits;     // priority space: bit (slot ^ octant), visited in descending order
    uint32_t child_base, tri_base, meta_lo, meta_hi, imask;
};

// Rays with a parallel axis (direction component below kParallelDir, NaN inverse - box_inv; rare): the children that passed the slab test
// are tested on those axes by parallel_ok. Out of line, so that the common path carries no branch per child.
// The node is read again here (L1) rather than handed over in sixteen registers that would stay live across the child tests.
static __device__ __noinline__ uint32_t wide_parallel_filter(const uint4* __restrict__ p, V3 o, V3 inv, float lim, uint32_t hits) {
    const uint4 w0 = __ldg(p), w2 = __ldg(p + 2), w3 = __ldg(p + 3), w4 = __ldg(p + 4);
    const uint32_t ew = w0.w;
    const float px = __uint_as_float(w0.x), py = __uint_as_float(w0.y), pz = __uint_as_float(w0.z);
    const float sx = __uint_as_float((ew & 0xffu) << 23), sy = __uint_as_float(((ew >> 8) & 0xffu) << 23),
                sz = __uint_as_float(((ew >> 16) & 0xffu) << 23);
    const float ax = (px - o.x) * inv.x, ay = (py - o.y) * inv.y, az = (pz - o.z) * inv.z;
    const float bx = sx * inv.x, by = sy * inv.y, bz = sz * inv.z;
    float ex = fabsf(bx) * 0.0078125f, ey = fabsf(by) * 0.0078125f, ez = fabsf(bz) * 0.0078125f;
    if (!(ex <= FLT_MAX)) ex = 0.0f;
    if (!(ey <= FLT_MAX)) ey = 0.0f;
    if (!(ez <= FLT_MAX)) ez = 0.0f;
    const float a2x = fmaf(-kWideBias, bx, ax) + ex, a2y = fmaf(-kWideBias, by, ay) + ey, a2z = fmaf(-kWideBias, bz, az) + ez;     // far planes
    const uint32_t lox[2] = {w2.x, w2.y}, loy[2] = {w2.z, w2.w}, loz[2] = {w3.x, w3.y};
    const uint32_t hix[2] = {w3.z, w3.w}, hiy[2] = {w4.x, w4.y}, hiz[2] = {w4.z, w4.w};
    uint32_t keep = 0;
    for (int c = 0; c < 8; ++c) {
        if (!((hits >> c) & 1u)) continue;
        const int w = c >> 2, k = c & 3;
        // the exit distance of the slab test: the far planes of the axes with a finite inverse (NaN drops out of fminf)
        const float fx = inv.x < 0.0f ? wide_biased(lox[w], k) : wide_biased(hix[w], k);
        const float fy = inv.y < 0.0f ? wide_biased(loy[w], k) : wide_biased(hiy[w], k);
        const float fz = inv.z < 0.0f ? wide_biased(loz[w], k) : wide_biased(hiz[w], k);
        const float tmax = fminf(fminf(fmaf(fx, bx, a2x), fmaf(fy, by, a2y)), fminf(fmaf(fz, bz, a2z), lim));
        const float qlx = wide_byte(lox[w], k), qhx = wide_byte(hix[w], k), qly = wide_byte(loy[w], k), qhy = wide_byte(hiy[w], k),
                    qlz = wide_byte(loz[w], k), qhz = wide_byte(hiz[w], k);
        const float ext = (fabsf(qhx - qlx) * sx + fabsf(qhy - qly) * sy) + fabsf(qhz - qlz) * sz;
        bool hit = true;
        if (inv.x != inv.x) hit = parallel_ok(fmaf(qlx, sx, px), fmaf(qhx, sx, px), o.x, tmax, ext);
        if (hit && inv.y != inv.y) hit = parallel_ok(fmaf(qly, sy, py), fmaf(qhy, sy, py), o.y, tmax, ext);
        if (hit && inv.z != inv.z) hit = parallel_ok(fmaf(qlz, sz, pz), fmaf(qhz, sz, pz), o.z, tmax, ext);
        if (hit) keep |= 1u << c;
    }
    return keep;
}

// Box tests of the 8 children of node ni against the ray (o, inv); lim = 1.0001 * current t limit.
// Plane distance t = (p + q s - o) / d = q b + a with a = (p - o) inv, b = s inv, evaluated as fma(32768 + q, b, a - 32768 b -+ e).
CRT_DEV WideStep wide_node_test(const uint4* __restrict__ nodes, uint32_t ni, V3 o, V3 inv, uint32_t oinv, float lim, bool zray) {
    const uint4* p = nodes + 5 * (size_t)ni;
    const uint4 w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2), w3 = __ldg(p + 3), w4 = __ldg(p + 4);
    const uint32_t ew = w0.w;
    const float sx = __uint_as_float((ew & 0xffu) << 23), sy = __uint_as_float(((ew >> 8) & 0xffu) << 23),
                sz = __uint_as_float(((ew >> 16) & 0xffu) << 23);
    const float ax = (__uint_as_float(w0.x) - o.x) * inv.x, ay = (__uint_as_float(w0.y) - o.y) * inv.y,
                az = (__uint_as_float(w0.z) - o.z) * inv.z;
    const float bx = sx * inv.x, by = sy * inv.y, bz = sz * inv.z;
    float fax = fabsf(ax), fay = fabsf(ay), faz = fabsf(az);
    if (!(fax <= FLT_MAX)) fax = 0.0f;
    if (!(fay <= FLT_MAX)) fay = 0.0f;
    if (!(faz <= FLT_MAX)) faz = 0.0f;
    const float pad = fmaxf(fmaxf(fax, fay), faz) * 4.76837158203125e-07f;        // 2^-21
    // the folded bias costs one more rounding, 2^-9 |b| on the plane distances of ITS axis: near planes are taken
    // e = 2^-7 |b| earlier, far planes later. (One pad for all axes, 2^-7 max|b|, let a ray with one small direction
    // component - a cell is many units of t wide on that axis - into every box: C5 dropped from 5.4 to 1.8 Grays/s, r02_s13.)
    float ex = fabsf(bx) * 0.0078125f, ey = fabsf(by) * 0.0078125f, ez = fabsf(bz) * 0.0078125f;
    if (!(ex <= FLT_MAX)) ex = 0.0f;
    if (!(ey <= FLT_MAX)) ey = 0.0f;
    if (!(ez <= FLT_MAX)) ez = 0.0f;
    const float a2x = fmaf(-kWideBias, bx, ax), a2y = fmaf(-kWideBias, by, ay), a2z = fmaf(-kWideBias, bz, az);
    const float anx = a2x - ex, any_ = a2y - ey, anz = a2z - ez, afx = a2x + ex, afy = a2y + ey, afz = a2z + ez;
    // near planes: the low ones when the direction component is non-negative
    const bool px = oinv & 1u, py = oinv & 2u, pz = oinv & 4u;
    const uint32_t nx[2] = {px ? w2.x : w3.z, px ? w2.y : w3.w}, fx[2] = {px ? w3.z : w2.x, px ? w3.w : w2.y};
    const uint32_t ny[2] = {py ? w2.z : w4.x, py ? w2.w : w4.y}, fy[2] = {py ? w4.x : w2.z, py ? w4.y : w2.w};
    const uint32_t nz[2] = {pz ? w3.x : w4.z, pz ? w3.y : w4.w}, fz[2] = {pz ? w4.z : w3.x, pz ? w4.w : w3.y};
    WideStep r;
    r.child_base = w1.x; r.tri_base = w1.y; r.meta_lo = w1.z; r.meta_hi = w1.w; r.imask = ew >> 24;
    uint32_t hits = 0;                                     // slot space: bit c = the box of child c is hit
    const uint32_t kb = wide_bias_bits(ni);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const int w = c >> 2, k = c & 3;
        const float tnx = fmaf(wide_biased(nx[w], k, kb), bx, anx), tfx = fmaf(wide_biased(fx[w], k, kb), bx, afx);
        const float tny = fmaf(wide_biased(ny[w], k, kb), by, any_), tfy = fmaf(wide_biased(fy[w], k, kb), by, afy);
        const float tnz = fmaf(wide_biased(nz[w], k, kb), bz, anz), tfz = fmaf(wide_biased(fz[w], k, kb), bz, afz);
        const float tmin = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, 0.0f));
        const float tmax = fminf(fminf(tfx, tfy), fminf(tfz, lim));
        hits |= tmin <= fmaf(tmax, kSlabSlack, pad) ? 1u << c : 0u;
    }
    // children that exist (meta byte != 0), 4 bits per meta word
    hits &= wide_nonzero_bytes(w1.z) | (wide_nonzero_bytes(w1.w) << 4);
    if (zray && hits) hits = wide_parallel_filter(p, o, inv, lim, hits);
    // slot space -> priority space (bit i -> bit i ^ oinv) for both masks at once: node hits in bits 0-7, leaf hits in 8-15
    uint32_t both = (hits & r.imask) | ((hits & ~r.imask) << 8);
    if (oinv & 1u) both = ((both & 0x5555u) << 1) | ((both >> 1) & 0x5555u);
    if (oinv & 2u) both = ((both & 0x3333u) << 2) | ((both >> 2) & 0x3333u);
    if (oinv & 4u) both = ((both & 0x0f0fu) << 4) | ((both >> 4) & 0x0f0fu);
    r.node_hits = both & 0xffu;
    r.leaf_hits = both >> 8;
    return r;
}

CRT_DEV uint32_t wide_octant(V3 inv) { return (inv.x < 0.0f ? 0u : 1u) | (inv.y < 0.0f ? 0u : 2u) | (inv.z < 0.0f ? 0u : 4u); }
// first triangle slot of the leaf child with priority bit lp
CRT_DEV int wide_leaf_slot(const WideStep& s, int lp, uint32_t oinv) {
    const uint32_t c = (uint32_t)lp ^ oinv;
    const uint32_t m = ((c & 4u ? s.meta_hi : s.meta_lo) >> (8u * (c & 3u))) & 0xffu;
    return (int)(s.tri_base + m - 1u);
}

// Sequential rule, one ray per call (tail kernel; statement: oracle wide8_intersect).
template <int MODE>
CRT_DEV HitRec traverse_wide(const SceneView& sc, V3 o, V3 d, float tmax) {
    HitRec best;
    best.t = FLT_MAX; best.slot = -1; best.face = -1;
    if (sc.n_nodes == 0) return best;
    const uint4* nodes = (const uint4*)sc.nodes;
    const V3 inv = box_inv3(d);
    const uint32_t oinv = wide_octant(inv);
    const bool zray = has_parallel_axis(inv);
    float tlimit = MODE == 0 ? FLT_MAX : tmax;
    uint2 stack[kWideStack];
    int sp = 0;
    uint32_t g_base = 0, g_bits = (1u << 8) | (1u << oinv);      // imask << 8 | hit mask; the root as slot 0 of a virtual parent
    for (;;) {
        if ((g_bits & 0xffu) == 0u) {
            if (sp == 0) break;
            const uint2 e = stack[--sp];
            g_base = e.x; g_bits = e.y;
        }
        const int pr = 31 - __clz((int)(g_bits & 0xffu));
        g_bits &= ~(1u << pr);
        const uint32_t sl = (uint32_t)pr ^ oinv;
        const uint32_t ni = g_base + (uint32_t)__popc((g_bits >> 8) & ((1u << sl) - 1u));
        WideStep s = wide_node_test(nodes, ni, o, inv, oinv, tlimit * 1.0001f, zray);
        while (s.leaf_hits) {
            const int lp = 31 - __clz((int)s.leaf_hits);
            s.leaf_hits &= ~(1u << lp);
            int slot = wide_leaf_slot(s, lp, oinv);
            for (;; ++slot) {
                V3 tv1, te1, te2;
                const uint32_t fw = load_tri(sc.tri_geom, slot, tv1, te1, te2);
                const int face = (int)(fw & ~kLastBit);
                float t;
                if (tri_test(tv1, te1, te2, o, d, &t) && t > kEps) {
                    if (MODE == 0) {
                        if (t < best.t || (t == best.t && face < best.face)) {
                            best.t = t; best.slot = slot; best.face = face;
                            tlimit = t;
                        }
                    } else if (tmax - t > kEps) {
                        best.t = t; best.slot = slot; best.face = face;
                        return best;
                    }
                }
                if (fw & kLastBit) break;
            }
        }
        if (s.node_hits) {
            if (g_bits & 0xffu) stack[sp++] = make_uint2(g_base, g_bits);
            g_base = s.child_base;
            g_bits = (s.imask << 8) | s.node_hits;
        }
    }
    return best;
}

// ---- Walker for the 8-wide nodes (trace_persistent_queue, crt_device.cuh): same visits in the same order as
// traverse_wide. The leaf children hit by a node step are appended to the warp's queue (one shared atomicAdd per lane
// and step: ballot-positioned slots were measured slower here, -1 %, profiles/r01_s18.md) and the lane goes on with
// its next node. Measured and removed: prefetch.global.L1 of a leaf's triangles when it is queued, -5 % (r01_s21.md).
#ifndef CRT_WQFLUSH
#define CRT_WQFLUSH 12
#endif
#ifndef CRT_WQSTEPS
#define CRT_WQSTEPS 2
#endif
#ifndef CRT_WSSTACK
#define CRT_WSSTACK 4
#endif
// MINLANES (template parameter of the walker): a second node step in a turn only while at least that many lanes still have a
// node in hand; the others keep theirs for the next turn, when the refilled lanes step with them. Used by the any-hit batch
// kernel only (C5 any-hit +6.5 %). Everywhere else it was measured and left out (profiles/r02_late_levers.md, r02_s37 / s38 / s40):
// k_shadow +-0, closest-hit batches -1.5 %, the tail path tracer's small frames -5...9 %, and k_extend gains on cornell-box
// (42.1 -> 41.0 ms per 4K spp-48 frame) what it loses on the 10 M-triangle scene (C4 -1.3 %) and on veach-mis (-2 %).
#ifndef CRT_WQ_MINLANES
#define CRT_WQ_MINLANES 20
#endif
template <int MINLANES>
struct WideWalkerT {
    static constexpr int kFlush = CRT_WQFLUSH;
    static constexpr int kSteps = CRT_WQSTEPS;
    static constexpr int kCap = kFlush + 32 * 8 * kSteps;
    static constexpr int kShared = CRT_WSSTACK;
    // first kShared entries of every lane's stack in shared memory, [entry][thread]: a push / pop is one conflict-free
    // wavefront and a short-scoreboard wait instead of a local-memory round trip
    static constexpr int kLocal = kWideStack - kShared;
    typedef uint2 Entry;
    int sp;
    uint32_t g_base, g_bits, oinv;
    int min_lanes;
    CRT_DEV void init() { sp = 0; g_base = 0; g_bits = 0; oinv = 0; min_lanes = 0; }
    // queues of fewer than 2^22 rays (the shipped 800x600 frames) are bound by the latency of their rays, not by issue slots: no gate
    CRT_DEV void configure(uint32_t n_rays) { min_lanes = MINLANES > 0 && n_rays >= (1u << 22) ? MINLANES : 0; }
    CRT_DEV void start(bool live, V3 inv) {
        oinv = wide_octant(inv);
        sp = 0;
        g_base = 0;
        g_bits = live ? ((1u << 8) | (1u << oinv)) : 0u;     // the root as slot 0 of a virtual parent
    }
    CRT_DEV bool walking() const { return (g_bits & 0xffu) != 0u || sp > 0; }
    CRT_DEV void stop() { g_bits = 0; sp = 0; }
    template <typename Q> CRT_DEV int queued(const Q& q) const { return q.count; }
    template <typename Q> CRT_DEV void reset_queue(Q& q, int lane) { if (lane == 0) q.count = 0; }
    template <typename Q>
    CRT_DEV void steps(const SceneView& sc, Q& q, uint2* stack, V3 o, V3 inv, float lim, bool zray, int lane, unsigned, int& pending) {
        __shared__ uint2 s_wstack[kShared > 0 ? kShared : 1][128];
        const uint4* nodes = (const uint4*)sc.nodes;
#pragma unroll
        for (int r = 0; r < kSteps; ++r) {
            if (MINLANES > 0 && r > 0 && min_lanes > 0 && __popc(__ballot_sync(0xffffffffu, (g_bits & 0xffu) != 0u || sp > 0)) < min_lanes) break;
            if ((g_bits & 0xffu) == 0u && sp > 0) {
                --sp;
                const uint2 e = (kShared > 0 && sp < kShared) ? s_wstack[sp][threadIdx.x] : stack[sp - kShared];
                g_base = e.x; g_bits = e.y;
            }
            if (g_bits & 0xffu) {
                const int pr = 31 - __clz((int)(g_bits & 0xffu));
                g_bits &= ~(1u << pr);
                const uint32_t sl = (uint32_t)pr ^ oinv;
                const uint32_t ni = g_base + (uint32_t)__popc((g_bits >> 8) & ((1u << sl) - 1u));
                WideStep s = wide_node_test(nodes, ni, o, inv, oinv, lim, zray);
                if (s.leaf_hits) {
                    const int cnt = __popc(s.leaf_hits);
                    int pos = atomicAdd(&q.count, cnt);
                    pending += cnt;
                    while (s.leaf_hits) {
                        const int lp = 31 - __clz((int)s.leaf_hits);
                        s.leaf_hits &= ~(1u << lp);
                        q.q_slot[pos] = wide_leaf_slot(s, lp, oinv);
                        q.q_lane[pos] = (unsigned char)lane;
                        ++pos;
                    }
                }
                if (s.node_hits) {
                    if (g_bits & 0xffu) {
                        if (kShared > 0 && sp < kShared) s_wstack[sp][threadIdx.x] = make_uint2(g_base, g_bits);
                        else stack[sp - kShared] = make_uint2(g_base, g_bits);
                        ++sp;
                    }
                    g_base = s.child_base;
                    g_bits = (s.imask << 8) | s.node_hits;
                }
            }
        }
    }
};
typedef WideWalkerT<0> WideWalker;                       // every lane steps kSteps times per turn
typedef WideWalkerT<CRT_WQ_MINLANES> WideWalkerGated;

}  // namespace crt
