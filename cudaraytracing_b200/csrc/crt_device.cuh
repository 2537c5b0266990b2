// crt_device.cuh — device-side arithmetic, RNG and BVH traversal shared by all kernels.
//
// Arithmetic contract (DESIGN.md "Arithmetic"): this translation unit is compiled with
// -fmad=false, so every float operation below is a single IEEE-754 round-to-nearest operation and
// a fused multiply-add happens only where fmaf() is written. Division and sqrt are the IEEE ones
// (nvcc defaults -prec-div=true -prec-sqrt=true, -ftz=false). sin/cos are the fixed polynomials
// below. The CPU oracle states the same operations, so hit ids and the fixed-point accumulation
// buffer can be compared for exact equality.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>

namespace crt {

#define CRT_DEV __device__ __forceinline__

// Slack of the box tests: a child is entered iff tmin <= tmax * kSlabSlack, kSlabSlack = 1 + 2^-17 (64 ulp). The
// slab distances carry ~3 roundings each, but the margin has to cover the *triangle test's* error too: Moeller-
// Trumbore accepts points a few 1e-6 (relative to the distance) outside a small, far triangle, so a ray through a
// box corner (a light sample AT a vertex, veach-mis) was accepted by the triangle test and rejected by a 4-ulp box
// test - found as a one-pixel difference between the pair-node and the 8-wide render (profiles/r01_s15.md).
static constexpr float kSlabSlack = 1.00000762939453125f;
static constexpr float kEps = 0.00001f;                 // EPSILON, reference Global.h:11
static constexpr float kPi = 3.14159265358979323846f;
static constexpr float kTwoPi = 6.2831853071795864769f; // get_cuda_sphere_sample_inv_pdf(), Global.h:96-99
static constexpr int kEmptyChild = 0x7fffffff;
static constexpr uint32_t kLastBit = 0x80000000u;
static constexpr int kStackSize = 96;                   // 63 Morton bits + duplicate-key levels

struct V3 { float x, y, z; };
CRT_DEV V3 mk3(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
CRT_DEV V3 mk3(float4 v) { return mk3(v.x, v.y, v.z); }
CRT_DEV V3 operator+(V3 a, V3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
CRT_DEV V3 operator-(V3 a, V3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
CRT_DEV V3 operator*(V3 a, float s) { return mk3(a.x * s, a.y * s, a.z * s); }
CRT_DEV V3 operator*(float s, V3 a) { return mk3(a.x * s, a.y * s, a.z * s); }
CRT_DEV V3 operator/(V3 a, float s) { return mk3(a.x / s, a.y / s, a.z / s); }
CRT_DEV V3 cmul(V3 a, V3 b) { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
CRT_DEV float dot(V3 a, V3 b) { return fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)); }
CRT_DEV V3 cross(V3 a, V3 b) {
    return mk3(fmaf(a.y, b.z, -(a.z * b.y)), fmaf(a.z, b.x, -(a.x * b.z)), fmaf(a.x, b.y, -(a.y * b.x)));
}
// a / b for b > 0 (or b = +inf) where a is often exactly zero - a clamped cosine, a coordinate in the plane of the light. The
// compiler's IEEE division rejects a zero numerator in its fast path (FCHK) and calls a 31-instruction subroutine for the whole
// warp; in k_shade that was 17 % of the instructions (profiles/r02_div_zero.md). The quotient is a itself (the zero keeps its sign),
// so the division is given a harmless numerator and the result selected: same value, no call.
CRT_DEV float div_by_pos(float a, float b) {
#ifdef CRT_NO_DIV_GUARD                            // the plain division, for A/B measurements (tools/sessions/log/r02_s24.sh, r02_s35.sh)
    return a / b;
#endif
    const bool z = a == 0.0f;
    float n = z ? 1.0f : a;
    asm("" : "+f"(n));          // or the compiler folds the two selects back into a / b
    const float q = n / b;
    return z ? a : q;
}
// Eigen normalized(): v / sqrt(v.v) when v.v > 0 (reference include/Eigen/src/Core/Dot.h:121-131)
CRT_DEV V3 normalize(V3 a) {
    float n = dot(a, a);
    if (n > 0.0f) {
        const float s = sqrtf(n);
        return mk3(div_by_pos(a.x, s), div_by_pos(a.y, s), div_by_pos(a.z, s));
    }
    return a;
}
CRT_DEV float length(V3 a) { return sqrtf(dot(a, a)); }
// Shading only: one IEEE division and three products instead of three divisions (a division is ~9 instructions; the compat
// vertex had 38 of them, a third of k_shade's instructions, profiles/r02_s15.md). Statement: oracle/orc_math.h normalize_rcp.
CRT_DEV V3 normalize_rcp(V3 a) {
    float n = dot(a, a);
    if (n > 0.0f) return a * (1.0f / sqrtf(n));
    return a;
}

// ---- Philox4x32-10 (Salmon et al., SC'11). Replaces curand XORWOW + clock() seed
// (reference Global.h:52-55,106-109; Render.cuh:340-341).
CRT_DEV uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}
static constexpr uint32_t kPhiloxKey1 = 0x43525431u;    // "CRT1"
static constexpr uint32_t kCameraBounce = 0xFFFFFFFFu;
CRT_DEV uint4 draw(uint32_t pixel, uint32_t sample, uint32_t bounce, uint32_t dim, uint32_t seed) {
    return philox4x32_10(make_uint4(pixel, sample, bounce, dim), seed, kPhiloxKey1);
}
// (0,1], like curand_uniform (reference Global.h:52-55)
CRT_DEV float u01(uint32_t x) { return (float)((x >> 8) + 1u) * 5.9604644775390625e-08f; }

// ---- deterministic sin/cos
CRT_DEV void sincos_poly(float x, float* s, float* c) {
    float x2 = x * x;
    float ps = fmaf(x2, 2.7557319e-06f, -1.9841270e-04f);
    ps = fmaf(ps, x2, 8.3333333e-03f);
    ps = fmaf(ps, x2, -1.6666667e-01f);
    *s = fmaf(x * x2, ps, x);
    float pc = fmaf(x2, -2.7557319e-07f, 2.4801587e-05f);
    pc = fmaf(pc, x2, -1.3888889e-03f);
    pc = fmaf(pc, x2, 4.1666667e-02f);
    pc = fmaf(pc, x2, -0.5f);
    *c = fmaf(pc, x2, 1.0f);
}
CRT_DEV void quadrant(int q, float ss, float cc, float* s, float* c) {
    switch (q & 3) {
        case 0: *s = ss; *c = cc; break;
        case 1: *s = cc; *c = -ss; break;
        case 2: *s = -ss; *c = -cc; break;
        default: *s = -cc; *c = ss; break;
    }
}
CRT_DEV void sincos_2pi(float u, float* s, float* c) {
    int q = (int)fmaf(u, 4.0f, 0.5f);
    float r = u - (float)q * 0.25f;
    float ss, cc;
    sincos_poly(r * 6.2831855f, &ss, &cc);
    quadrant(q, ss, cc, s, c);
}
CRT_DEV void sincos_rad(float x, float* s, float* c) {
    if (!(fabsf(x) <= 1.0e6f)) x = 0.0f;
    float n = rintf(x * 0.63661975f);
    float r = fmaf(-n, 1.5707963705062866f, x);
    r = fmaf(-n, -4.371138828673793e-08f, r);
    float ss, cc;
    sincos_poly(r, &ss, &cc);
    quadrant((int)n, ss, cc, s, c);
}

// ---- deterministic log2 / exp2 / pow and luminance (mis estimator; statement: oracle/orc_math.h)
CRT_DEV float det_log2(float x) {
    const uint32_t b = __float_as_uint(x);
    int e = (int)(b >> 23) - 127;
    float m = __uint_as_float((b & 0x7fffffu) | 0x3f800000u);
    if (m > 1.41421354f) { m = m * 0.5f; e += 1; }
    const float f = m - 1.0f;
    const float sq = f / (2.0f + f);
    const float s2 = sq * sq;
    float p = fmaf(s2, 0.11111111f, 0.14285715f);
    p = fmaf(p, s2, 0.2f);
    p = fmaf(p, s2, 0.33333334f);
    const float r = fmaf(sq * s2, p, sq);
    return fmaf(r, 2.8853900f, (float)e);
}
CRT_DEV float det_exp2(float y) {
    if (!(y >= -126.0f)) return 0.0f;
    if (y > 127.0f) y = 127.0f;
    const float n = rintf(y);
    const float r = y - n;
    float p = fmaf(r, 1.5403530e-4f, 1.3333558e-3f);
    p = fmaf(p, r, 9.6181291e-3f);
    p = fmaf(p, r, 5.5504109e-2f);
    p = fmaf(p, r, 2.4022651e-1f);
    p = fmaf(p, r, 6.9314718e-1f);
    p = fmaf(p, r, 1.0f);
    return p * __uint_as_float((uint32_t)((int)n + 127) << 23);
}
CRT_DEV float det_pow(float x, float y) { return det_exp2(y * det_log2(x)); }
CRT_DEV float lumf(V3 c) { return fmaf(0.0722f, c.z, fmaf(0.7152f, c.y, 0.2126f * c.x)); }

// ---- scene view passed to kernels by value
struct SceneView {
    const float4* __restrict__ nodes;       // 4 x 16 B per node (crt_bvh_node)
    const float4* __restrict__ tri_geom;    // 3 x 16 B per slot: (v1, face|last) (e1, mat) (e2, 0)
    const float4* __restrict__ tri_shade;   // 1 x 16 B per slot: (normal, mat)
    const float4* __restrict__ mats;        // 5 x 16 B per material: (kd, ns) (ke, flags) (probe lobe) (ks, pdf) (kd / pi)
    const float4* __restrict__ light_tris;  // 4 x 16 B per light triangle: (v1,ke.r) (v2,ke.g) (v3,ke.b) (n, 0)
    const int4* __restrict__ lights;        // per light object: (first light tri, count, area bits, 0)
    const float* __restrict__ light_cdf;    // mis estimator: CDF over light_tris, P ~ area * luminance(Ke)
    int n_nodes;
    int n_lights;
    int n_light_tris;
};

// Canonical triangle test: Moeller-Trumbore of reference DeviceTriangle.cuh:39-65 (strict inside).
CRT_DEV bool tri_test(V3 v1, V3 e1, V3 e2, V3 o, V3 d, float* t_out) {
    V3 sv = o - v1;
    V3 s1 = cross(d, e2);
    V3 s2 = cross(sv, e1);
    float rcp = 1.0f / dot(s1, e1);
    float beta = dot(s1, sv) * rcp;
    float gamma = dot(s2, d) * rcp;
    float t = dot(s2, e2) * rcp;
    float alpha = (1.0f - beta) - gamma;
    *t_out = t;
    return 0.0f < alpha && alpha < 1.0f && 0.0f < beta && beta < 1.0f && 0.0f < gamma && gamma < 1.0f;
}

// Direction components below kParallelDir = 2^-40 in magnitude count as parallel in the box tests (box_inv gives them a
// NaN inverse); the triangle test keeps the true direction. The threshold is set by overflow alone:
//  * below 2^-128, 1/d overflows to inf, and a ray starting in a box plane got 0 * inf = NaN on one plane and +-inf on the
//    other, an empty slab; in the wide node step (crt_wide.cuh) b = s / d made the folded bias fma(-32768, b, a) overflow
//    to -inf once |d| < ~s * 2^-113 (s: the node's cell size), which culled every child of the node;
//  * above 2^-40, |1/d| <= 2^40: for coordinates and origins within +-2^72 (the range crt.h states) a node spans at most
//    2^73, its cell size is s <= 2^66, the folded bias 32768 * s / d <= 2^121, a = (p - o) / d <= 2^113 and the pair
//    slab's plane distances likewise <= 2^113 - below FLT_MAX ~ 2^128;
//  * treating a component below 2^-40 as parallel stays conservative: up to the exit distance texit the ray moves at most
//    2^-40 * texit along the axis, less than one rounding (2^-24 relative) of parallel_ok's margin, which holds
//    2^-17 * texit. Exact zeros therefore keep the margin they had.
static constexpr float kParallelDir = 9.094947017729282379e-13f;      // 2^-40

// Conservative slab test (DESIGN.md "Traversal rule"). NaN plane distances drop out of fminf / fmaxf.
// Axis the ray is parallel to (direction component below kParallelDir, inverse = NaN - box_inv below): its plane distances
// drop out of the min/max of the slab test, and the axis is tested here instead: o must lie in [lo, hi] widened by
// 2^-17 * (|o| + exit distance + summed box extent). Statement and rationale: oracle/orc_bvh.cpp parallel_ok.
CRT_DEV bool parallel_ok(float lo, float hi, float o, float texit, float ext) {
    const float dlt = ((fabsf(o) + texit) + ext) * 7.62939453125e-06f;
    return lo - o <= dlt && o - hi <= dlt;
}
CRT_DEV bool has_parallel_axis(V3 inv) { return inv.x != inv.x || inv.y != inv.y || inv.z != inv.z; }

// zray: the ray has a parallel axis (rare; hoisted so that the common path pays one predicate)
CRT_DEV bool slab(float lox, float hix, float loy, float hiy, float loz, float hiz, V3 o, V3 inv, float limit,
                  float* enter, bool zray) {
    float tx0 = (lox - o.x) * inv.x, tx1 = (hix - o.x) * inv.x;
    float ty0 = (loy - o.y) * inv.y, ty1 = (hiy - o.y) * inv.y;
    float tz0 = (loz - o.z) * inv.z, tz1 = (hiz - o.z) * inv.z;
    float tmin = fmaxf(fmaxf(fminf(tx0, tx1), fminf(ty0, ty1)), fmaxf(fminf(tz0, tz1), 0.0f));
    float tmax = fminf(fminf(fmaxf(tx0, tx1), fmaxf(ty0, ty1)), fminf(fmaxf(tz0, tz1), limit));
    *enter = tmin;
    // absolute slack: 2^-21 * the largest plane distance, as in the wide node step (statement: oracle/orc_bvh.cpp slab).
    // Without it a ray leaving a box plane (o.y == hi.y, d.y > 0) exits that slab at t = 0 exactly, the relative slack is 0,
    // and the hits the triangle test accepts just past the box's edge in that plane were lost, for any size of d.y.
    const float pad = fmaxf(fmaxf(fmaxf(fabsf(tx0), fabsf(tx1)), fmaxf(fabsf(ty0), fabsf(ty1))),
                            fmaxf(fabsf(tz0), fabsf(tz1))) * 4.76837158203125e-07f;
    bool hit = tmin <= fmaf(tmax, kSlabSlack, pad);
    if (zray && hit) {
        const float ext = ((hix - lox) + (hiy - loy)) + (hiz - loz);
        if (inv.x != inv.x) hit = parallel_ok(lox, hix, o.x, tmax, ext);
        if (hit && inv.y != inv.y) hit = parallel_ok(loy, hiy, o.y, tmax, ext);
        if (hit && inv.z != inv.z) hit = parallel_ok(loz, hiz, o.z, tmax, ext);
    }
    return hit;
}

// Inverse direction for the box tests: 1/d, and NaN for a component below kParallelDir in magnitude (zero included), so
// that this axis never culls (every plane distance on it is NaN and drops out of fminf / fmaxf) and parallel_ok tests it
// instead. With 1/0 = inf a ray lying IN a box plane (o.x == plane) gave 0 * inf = NaN on that plane and +-inf on the
// other, min(NaN, +inf) = +inf emptied the slab, and the traversal dropped boxes whose triangles the Moeller-Trumbore
// test accepts; the same happens when the origin (a computed hit point) sits one ulp outside a box whose triangle still
// passes the test. Exact zeros are not rare: sincos_2pi is exact at the quadrants. Found by the wide-node render
// (profiles/r01_s12_wide_vs_pair.md); tiny non-zero components: kParallelDir above. Statement: oracle/orc_math.h box_inv.
CRT_DEV float box_inv(float x) { return fabsf(x) < kParallelDir ? __int_as_float(0x7fc00000) : 1.0f / x; }
CRT_DEV V3 box_inv3(V3 d) { return mk3(box_inv(d.x), box_inv(d.y), box_inv(d.z)); }

struct HitRec { float t; int slot; int face; };


// One 64-byte pair node. CRT_LD256 = 1: two 256-bit loads (LDG.E.256, sm_100+) instead of four 128-bit ones -
// the traversal kernels are bound by L1 data-pipe wavefronts (profiles/r01_s11.md), which are paid per load
// instruction and distinct line.
#ifndef CRT_LD256
#define CRT_LD256 1
#endif
CRT_DEV void load_node(const float4* __restrict__ nodes, int cur, float4& n0, float4& n1, float4& n2, float4& n3) {
    const float4* p = nodes + 4 * (size_t)cur;
#if CRT_LD256
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(n0.x), "=f"(n0.y), "=f"(n0.z), "=f"(n0.w), "=f"(n1.x), "=f"(n1.y), "=f"(n1.z), "=f"(n1.w) : "l"(p));
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(n2.x), "=f"(n2.y), "=f"(n2.z), "=f"(n2.w), "=f"(n3.x), "=f"(n3.y), "=f"(n3.z), "=f"(n3.w) : "l"(p + 2));
#else
    n0 = __ldg(p); n1 = __ldg(p + 1); n2 = __ldg(p + 2); n3 = __ldg(p + 3);
#endif
}

// One triangle record: (v1, face|last) (e1, mat) (e2, 0). Reading only the 40 bytes the test needs (a re-laid-out record,
// LDG.128 + LDG.128 + LDG.64) and only 56 of a node's 64 bytes was measured: -1.5 % and 0 (profiles/r01_s18.md) - the L1
// data pipe is paid per load instruction and distinct line, not per byte.
CRT_DEV uint32_t load_tri(const float4* __restrict__ tri_geom, int slot, V3& v1, V3& e1, V3& e2) {
    const float4* p = tri_geom + 3 * (size_t)slot;
    const float4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
    v1 = mk3(a); e1 = mk3(b); e2 = mk3(c);
    return __float_as_uint(a.w);
}

// MODE 0: closest hit, t > 1e-5, ties -> lower face id (reference DeviceBVH.cuh:128-170 semantics
//         made BVH-independent). MODE 1: any hit with t > 1e-5 && tmax - t > 1e-5 (the decision of
//         reference Render.cuh:19-27, with early exit).
template <int MODE>
CRT_DEV HitRec traverse(const SceneView& sc, V3 o, V3 d, float tmax) {
    HitRec best;
    best.t = FLT_MAX; best.slot = -1; best.face = -1;
    if (sc.n_nodes == 0) return best;
    const V3 inv = box_inv3(d);
    const bool zray = has_parallel_axis(inv);
    float tlimit = MODE == 0 ? FLT_MAX : tmax;
    int stack[kStackSize];
    int sp = 0;
    int cur = 0;
    for (;;) {
        if (cur >= 0) {
            if (cur == kEmptyChild) { if (sp == 0) break; cur = stack[--sp]; continue; }
            float4 n0, n1, n2, n3;
            load_node(sc.nodes, cur, n0, n1, n2, n3);
            const float lim = tlimit * 1.0001f;
            float e0, e1;
            const bool h0 = slab(n0.x, n0.y, n0.z, n0.w, n2.x, n2.y, o, inv, lim, &e0, zray);
            const bool h1 = slab(n1.x, n1.y, n1.z, n1.w, n2.z, n2.w, o, inv, lim, &e1, zray);
            const int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
            if (h0 && h1) {
                int nearc = c0, farc = c1;
                if (e1 < e0) { nearc = c1; farc = c0; }
                stack[sp++] = farc;
                cur = nearc;
            } else if (h0) cur = c0;
            else if (h1) cur = c1;
            else { if (sp == 0) break; cur = stack[--sp]; }
        } else {
            int slot = ~cur;
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
            if (sp == 0) break;
            cur = stack[--sp];
        }
    }
    return best;
}

// ---- persistent-lane traversal with a per-warp leaf queue ------------------------------------------
// The per-ray rule is traverse<MODE> above (pair nodes) / traverse_wide<MODE> (crt_wide.cuh); what changes is how a
// warp's lanes are kept busy (measured alternatives - fixed 32-ray batches, while-while, if-if - in DESIGN.md 7.1):
//   * every lane owns one ray at a time and takes the next ray of the queue when it finishes (RayFetch below), as
//     soon as kRefillLanes lanes are idle, instead of waiting for the slowest ray of a fixed group of 32;
//   * node steps and triangle tests are decoupled: a lane that reaches a leaf does not test it, it appends
//     (lane, first slot) to a queue in shared memory and goes on with its next node, so every live lane does a node
//     step in every iteration (in a while-while loop ~10 of 32 lanes were active in the node phase, profiles/r01_c3.md);
//   * when enough leaves are queued (or no lane has a node left) the whole warp tests them, one queue entry per
//     lane, against the owners' rays (mirrored in shared memory); the owners' best hits are combined with a 64-bit
//     shared-memory atomicMin on (t bits, face id), which is exactly the "smaller t, ties -> lower face id" rule;
//   * the price is speculation: a lane keeps walking with the t-limit of the last flush, so it visits somewhat more
//     nodes than the sequential rule (the oracle's counts are the algorithmic minimum).
// One template for both node layouts: the Walker policy (PairWalker below, WideWalker in crt_wide.cuh) owns the
// per-lane traversal state and does the node steps; this function owns the queue flush, the finished rays and the refill.
// load(i, o, d, tmax) reads ray i (false: report a miss without tracing); done(i, hit) consumes the result.
#ifndef CRT_REFILL_LANES
#define CRT_REFILL_LANES 12
#endif
static constexpr int kRefillLanes = CRT_REFILL_LANES;
// How a warp takes ray indices from the queue counter `fetch`: one global atomicAdd of the idle-lane count per refill.
// Measured against it and removed (profiles/r02_fetch.md): per-warp reservations of 64-256 indices, with and without a
// reservation of lookahead (ptxas wraps its own vote + shuffle aggregation around an atomic in `if (lane == 0)`, inline PTX
// included, so the round trip is waited for on the spot anyway), and a static round-robin deal of 128-ray chunks with a
// dynamic tail and L2 prefetch of the next chunk: k_extend 15 % slower, k_shadow 9 % slower at 1080p. The returned value of
// this atomic is the largest single stall of k_shadow only when the accumulation buffer misses L2 (4K frames: its RED
// traffic to DRAM queues in front of it); the tile order of k_generate removes that. Also measured and removed (r02_s27,
// profiles/r02_late_levers.md): a reservation of 32 indices issued under elect.sync (which ptxas leaves un-aggregated) just
// before the leaf flush and read just after it, so that the flush covers the round trip - k_extend 8 % slower, C5 7 % slower:
// the register the value waits in and the bookkeeping of two open reservations cost more than the hidden latency returns.
struct RayFetch {
    bool exhausted = false;
    CRT_DEV void init(uint32_t n) { exhausted = n == 0; }
    CRT_DEV bool drained() const { return exhausted; }
    // Called by the whole warp with `want` idle lanes: returns how many indices [first, first + take) it may hand out.
    CRT_DEV uint32_t take(uint32_t* fetch, uint32_t n, int lane, uint32_t want, uint32_t& first) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(fetch, want);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base + want >= n) exhausted = true;
        first = base;
        return base < n ? min(want, n - base) : 0u;
    }
};

template <int CAP>
struct WarpLeafQueue {
    float ox[32], oy[32], oz[32], dx[32], dy[32], dz[32], tmax[32];     // the rays the lanes own
    unsigned long long best[32];                                         // (t bits, face id) of the owner's best hit
    int best_slot[32];
    int q_slot[CAP];                                                     // queued leaves: first triangle slot ...
    unsigned char q_lane[CAP];                                           // ... and the lane that owns the ray
    unsigned char any[32];                                               // flush_leaf_queue<2>: the owner's ray is an any-hit ray
    int count;
};
static constexpr unsigned long long kNoHitKey = ((unsigned long long)0x7f7fffffu << 32) | 0x7fffffffull;   // t = FLT_MAX

// The whole warp tests the queued leaves, one queue entry per lane, against the owners' rays (mirrored in the queue
// struct) and combines the owners' best hits. MODE 0: closest hit; 1: any hit with t > 1e-5 && tmax - t > 1e-5;
// 2: per ray, q.any[owner] says which (the tail path tracer mixes extend, probe and shadow rays in one warp).
template <int MODE, typename Q>
CRT_DEV void flush_leaf_queue(const SceneView& sc, Q& q, int q_count, int lane) {
    for (int base = 0; base < q_count; base += 32) {
        const int k = base + lane;
        unsigned long long mykey = kNoHitKey;
        int myslot = -1, owner = 0;
        if (k < q_count) {
            owner = q.q_lane[k];
            int slot = q.q_slot[k];
            const V3 ro = mk3(q.ox[owner], q.oy[owner], q.oz[owner]), rd = mk3(q.dx[owner], q.dy[owner], q.dz[owner]);
            const float rtmax = q.tmax[owner];
            const bool any = MODE == 1 || (MODE == 2 && q.any[owner]);
            // (Loading the first two triangles of a leaf together, to save the dependent second round trip of a two-triangle
            //  leaf, was measured: cornell-box 93.2 -> 96.3 ms per 1080p spp-128 frame, C5 6.10 -> 5.42 Grays/s, r02_s18.)
            for (;; ++slot) {
                V3 tv1, te1, te2;
                const uint32_t fw = load_tri(sc.tri_geom, slot, tv1, te1, te2);
                float t;
                if (tri_test(tv1, te1, te2, ro, rd, &t) && t > kEps && (!any || rtmax - t > kEps)) {
                    const unsigned long long key = ((unsigned long long)__float_as_uint(t) << 32) | (fw & ~kLastBit);
                    if (key < mykey) { mykey = key; myslot = slot; }
                }
                if (fw & kLastBit) break;
            }
            if (myslot >= 0) {
                if (MODE != 1) atomicMin(&q.best[owner], mykey);
                else q.best[owner] = mykey;                 // any blocker will do: one of the writers wins (64-bit store)
            }
        }
        __syncwarp();
        if (myslot >= 0 && q.best[owner] == mykey) q.best_slot[owner] = myslot;
        __syncwarp();
    }
}

template <int MODE, typename Walker, typename Load, typename Done>
CRT_DEV void trace_persistent_queue(const SceneView& sc, uint32_t n, uint32_t* fetch, Load load, Done done) {
    typedef WarpLeafQueue<Walker::kCap> Queue;
    __shared__ Queue s_wq[4];                              // launched with 128 threads per block
    Queue& q = s_wq[threadIdx.x >> 5];
    const unsigned kFull = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    // the deep part of the traversal stack is a plain local array next to the walker, not a member of it: a struct with
    // a dynamically indexed array stays in local memory as a whole, scalars and all (r02_s03: pair-node kernels 1.6x slower)
    typename Walker::Entry stack[Walker::kLocal];
    Walker wk;
    wk.init();
    wk.configure(n);
    uint32_t idx = 0;
    V3 o = mk3(0, 0, 0), inv = mk3(0, 0, 0);
    float tlimit = 0.0f;
    int pending = 0;                                       // leaves of this lane's ray waiting in the queue
    bool have = false, zray = false;
    RayFetch rf;
    rf.init(n);
    if (lane == 0) q.count = 0;
    __syncwarp();
    for (;;) {
        // A. node steps; leaves go to the queue
        wk.steps(sc, q, stack, o, inv, tlimit * 1.0001f, zray, lane, lt_mask, pending);
        // B. flush the leaf queue when it is full enough, or when no lane has a node in hand
        const unsigned walking = __ballot_sync(kFull, wk.walking());
        __syncwarp();
        const int q_count = wk.queued(q);
        if (q_count >= Walker::kFlush || (walking == 0 && q_count > 0)) {
            flush_leaf_queue<MODE>(sc, q, q_count, lane);
            wk.reset_queue(q, lane);
            pending = 0;
            if (have) {
                const unsigned long long b = q.best[lane];
                if (MODE == 0) tlimit = __uint_as_float((uint32_t)(b >> 32));
                else if (b != kNoHitKey) wk.stop();                  // blocked: nothing left to learn
            }
            __syncwarp();
        }
        // C. finished rays
        if (have && !wk.walking() && pending == 0) {
            const unsigned long long b = q.best[lane];
            HitRec h;
            h.t = __uint_as_float((uint32_t)(b >> 32));
            h.face = b == kNoHitKey ? -1 : (int)(uint32_t)b;
            h.slot = b == kNoHitKey ? -1 : q.best_slot[lane];
            done(idx, h);
            have = false;
        }
        // D. refill idle lanes from the ray queue
        const unsigned idle = __ballot_sync(kFull, !have);
        if (idle) {
            const int n_idle = __popc(idle);
            if (!rf.drained() && (n_idle >= kRefillLanes || n_idle == 32)) {
                uint32_t first = 0;
                const uint32_t got = rf.take(fetch, n, lane, (uint32_t)n_idle, first);
                const uint32_t rank = (uint32_t)__popc(idle & lt_mask);
                if (!have && rank < got) {
                    idx = first + rank;
                    V3 d;
                    float tmax;
                    const bool live = load(idx, o, d, tmax);
                    inv = box_inv3(d);
                    zray = has_parallel_axis(inv);
                    tlimit = MODE == 0 ? FLT_MAX : tmax;
                    q.ox[lane] = o.x; q.oy[lane] = o.y; q.oz[lane] = o.z;
                    q.dx[lane] = d.x; q.dy[lane] = d.y; q.dz[lane] = d.z;
                    q.tmax[lane] = tmax;
                    q.best[lane] = kNoHitKey;
                    q.best_slot[lane] = -1;
                    pending = 0;
                    wk.start(live && sc.n_nodes, inv);
                    have = true;
                }
                __syncwarp();
            }
            if (idle == kFull && rf.drained() && !__any_sync(kFull, have)) break;
        }
    }
}

// ---- Walker for the 64-byte child-pair nodes: same visits in the same order as traverse<MODE>.
#ifndef CRT_QFLUSH
#define CRT_QFLUSH 16
#endif
#ifndef CRT_QSTEPS
#define CRT_QSTEPS 6
#endif
// CRT_SSTACK = N > 0: the first N entries of every lane's traversal stack live in shared memory, laid out
// [entry][thread] so that a push / pop is one conflict-free wavefront whatever the lanes' depths are; a
// local-memory stack costs one L1 wavefront per distinct depth in the warp, and the pair-node kernels are
// bound by L1 wavefronts (profiles/r01_s11.md). Deeper entries spill to the local array.
#ifndef CRT_SSTACK
#define CRT_SSTACK 8       // with 256-bit node loads and ballot queue slots: +7 % on cornell-box, +3 % on veach-mis (profiles/r01_s18.md)
#endif
static constexpr int kDone = 0x7ffffffe;               // no node in hand and the stack is empty
struct PairWalker {
    static constexpr int kFlush = CRT_QFLUSH;          // queued leaves that trigger a flush
    static constexpr int kSteps = CRT_QSTEPS;          // node steps between two looks at the queue
    static constexpr int kCap = kFlush + 32 * kSteps;
    static constexpr int kShared = CRT_SSTACK;
    static constexpr int kLocal = kStackSize - kShared;
    typedef int Entry;
    int sp, cur, qn;                                   // qn: queued leaves, the same value in every lane
    CRT_DEV void init() { sp = 0; cur = kDone; qn = 0; }
    CRT_DEV void configure(uint32_t) {}
    CRT_DEV void start(bool live, V3) { sp = 0; cur = live ? 0 : kDone; }
    CRT_DEV bool walking() const { return cur != kDone; }
    CRT_DEV void stop() { cur = kDone; sp = 0; }
    template <typename Q> CRT_DEV int queued(const Q&) const { return qn; }
    template <typename Q> CRT_DEV void reset_queue(Q&, int) { qn = 0; }
    template <typename Q>
    CRT_DEV void steps(const SceneView& sc, Q& q, int* stack, V3 o, V3 inv, float lim, bool zray, int lane, unsigned lt_mask, int& pending) {
        __shared__ int s_stack[kShared > 0 ? kShared : 1][128];
        auto push = [&](int v) {
            if (kShared > 0 && sp < kShared) s_stack[sp][threadIdx.x] = v;
            else stack[sp - kShared] = v;
            ++sp;
        };
        auto pop = [&]() -> int {
            --sp;
            if (kShared > 0 && sp < kShared) return s_stack[sp][threadIdx.x];
            return stack[sp - kShared];
        };
#pragma unroll
        for (int r = 0; r < kSteps; ++r) {
            {   // a leaf in hand goes to the queue and the lane takes the next entry of its stack. The queue belongs to this
                // warp and every lane is here: positions from a ballot, no shared atomic (+2 %, profiles/r01_s18.md)
                const bool leaf = cur < 0;
                const unsigned lm = __ballot_sync(0xffffffffu, leaf);
                if (leaf) {
                    const int pos = qn + __popc(lm & lt_mask);
                    q.q_slot[pos] = ~cur;
                    q.q_lane[pos] = (unsigned char)lane;
                    pending++;
                    cur = sp ? pop() : kDone;
                }
                qn += __popc(lm);
            }
            if (cur >= 0 && cur != kDone) {
                if (cur == kEmptyChild) {                  // absent child of a one-leaf scene
                    cur = sp ? pop() : kDone;
                } else {
                    float4 n0, n1, n2, n3;
                    load_node(sc.nodes, cur, n0, n1, n2, n3);
                    float e0, e1;
                    const bool h0 = slab(n0.x, n0.y, n0.z, n0.w, n2.x, n2.y, o, inv, lim, &e0, zray);
                    const bool h1 = slab(n1.x, n1.y, n1.z, n1.w, n2.z, n2.w, o, inv, lim, &e1, zray);
                    const int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
                    if (h0 && h1) {
                        int nearc = c0, farc = c1;
                        if (e1 < e0) { nearc = c1; farc = c0; }
                        push(farc);
                        cur = nearc;
                    } else if (h0) cur = c0;
                    else if (h1) cur = c1;
                    else cur = sp ? pop() : kDone;
                }
            }
        }
    }
};

// ---- fixed-point accumulation (DESIGN.md "Accumulation"): radiance * 2^32 summed in int64, which
// makes the image independent of atomic ordering, wavefront scheduling and GPU count.
CRT_DEV long long quantize(float c) {
    if (!(fabsf(c) < 1073741824.0f)) return 0;
    return __double2ll_rn((double)c * 4294967296.0);
}
CRT_DEV void accum_add(long long* accum, uint32_t pixel, V3 c) {
    unsigned long long* p = (unsigned long long*)(accum + 3 * (size_t)pixel);
    long long qx = quantize(c.x), qy = quantize(c.y), qz = quantize(c.z);
    if (qx) atomicAdd(p + 0, (unsigned long long)qx);
    if (qy) atomicAdd(p + 1, (unsigned long long)qy);
    if (qz) atomicAdd(p + 2, (unsigned long long)qz);
}

// ---- warp-aggregated append: one atomicAdd per warp, returns this lane's slot (or -1)
CRT_DEV int warp_append(uint32_t* counter, bool want) {
    const unsigned mask = __ballot_sync(__activemask(), want);
    if (!want) return -1;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(mask));
    base = __shfl_sync(mask, base, leader);
    return (int)(base + __popc(mask & ((1u << lane) - 1)));
}

}  // namespace crt
