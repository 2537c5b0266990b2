// ORACLE — TEST INFRASTRUCTURE ONLY. Nothing under oracle/ is linked, imported or executed by
// the product (cudaraytracing_b200/). Only tests/, __graft_entry__.smoke() and bench.py's
// cpu_baseline / --impl reference legs may use it, and only as the checker.
//
// orc_math.h — scalar float arithmetic used by every oracle routine.
//
// Arithmetic contract (shared, by specification, with the CUDA kernels; DESIGN.md §"Arithmetic"):
//   * every operation is a single IEEE-754 binary32 operation, round-to-nearest-even;
//   * no contraction: this file is compiled with -ffp-contract=off; a fused multiply-add
//     happens only where fmaf() is written (CUDA side: -fmad=false and explicit fmaf());
//   * division and sqrt are the correctly rounded ones;
//   * sin/cos come from the fixed polynomials below, never from libm.
// Under that contract the CPU oracle and the GPU kernels produce bit-identical floats, which is
// what lets tests/ demand exact equality of hit ids and of the fixed-point accumulation buffer.
#pragma once
#include <limits>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <cfloat>

namespace orc {

struct V3 { float x, y, z; };

static inline V3 v3(float x, float y, float z) { return V3{x, y, z}; }
static inline V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
static inline V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
static inline V3 operator*(V3 a, float s) { return V3{a.x * s, a.y * s, a.z * s}; }
static inline V3 operator*(float s, V3 a) { return V3{a.x * s, a.y * s, a.z * s}; }
static inline V3 operator/(V3 a, float s) { return V3{a.x / s, a.y / s, a.z / s}; }
static inline V3 cmul(V3 a, V3 b) { return V3{a.x * b.x, a.y * b.y, a.z * b.z}; }
static inline V3 neg(V3 a) { return V3{-a.x, -a.y, -a.z}; }

// dot = fma(az,bz, fma(ay,by, ax*bx))   — the one place products are fused, by contract.
static inline float dot(V3 a, V3 b) { return fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)); }
// cross component = fma(p,q, -(r*s))
static inline V3 cross(V3 a, V3 b) {
    return V3{fmaf(a.y, b.z, -(a.z * b.y)), fmaf(a.z, b.x, -(a.x * b.z)), fmaf(a.x, b.y, -(a.y * b.x))};
}
// Eigen's normalized(): v / sqrt(v.v) when v.v > 0 (reference include/Eigen/src/Core/Dot.h:121-131)
static inline V3 normalize(V3 a) {
    float n = dot(a, a);
    if (n > 0.0f) return a / sqrtf(n);
    return a;
}
static inline float length(V3 a) { return sqrtf(dot(a, a)); }
// Shading only (crt_device.cuh normalize_rcp): one division and three products instead of three divisions. The camera rays
// and everything pinned against the reference's host code keep normalize().
static inline V3 normalize_rcp(V3 a) {
    float n = dot(a, a);
    if (n > 0.0f) return a * (1.0f / sqrtf(n));
    return a;
}
// Inverse direction for the box tests of the new traversal rules: 1/d, NaN for a component whose magnitude is below
// kParallelDir (zero included), so that this axis never culls (NaN plane distances drop out of fminf / fmaxf) and is
// tested by parallel_ok (orc_bvh.cpp) instead. With 1/0 = inf a ray lying in a box plane made the pair-node slab empty
// (min(0 * inf, +inf) = +inf) and boxes were dropped whose triangles pass the triangle test; small non-zero components
// lost hits too (1/d overflowing, the wide node step's folded bias overflowing). Choice of the threshold and its bounds:
// crt_device.cuh kParallelDir. The triangle test keeps the true direction. The reference rule (ref_intersect) keeps the
// reference's plain 1/d (Ray.cuh:14).
static const float kParallelDir = 9.094947017729282379e-13f;      // 2^-40
static inline float box_inv(float x) { return fabsf(x) < kParallelDir ? std::numeric_limits<float>::quiet_NaN() : 1.0f / x; }
static inline V3 vmin(V3 a, V3 b) { return V3{fminf(a.x, b.x), fminf(a.y, b.y), fminf(a.z, b.z)}; }
static inline V3 vmax(V3 a, V3 b) { return V3{fmaxf(a.x, b.x), fmaxf(a.y, b.y), fmaxf(a.z, b.z)}; }

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3",
// SC'11; Random123 v1.14).  Replaces the reference's clock()-seeded XORWOW (Global.h:52-55,
// Render.cuh:340-341).  Known-answer vectors from Random123's kat_vectors are in tests/.
// ---------------------------------------------------------------------------------------------
struct U4 { uint32_t x, y, z, w; };

static inline U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c.x;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c.z;
        U4 n;
        n.x = (uint32_t)(p1 >> 32) ^ c.y ^ k0;
        n.y = (uint32_t)p1;
        n.z = (uint32_t)(p0 >> 32) ^ c.w ^ k1;
        n.w = (uint32_t)p0;
        c = n;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}

// (0,1] like curand_uniform (reference Global.h:52-55): (top 24 bits + 1) * 2^-24
static inline float u01(uint32_t x) { return (float)((x >> 8) + 1u) * 5.9604644775390625e-08f; }

// ---------------------------------------------------------------------------------------------
// Deterministic sin/cos.  Taylor polynomials on |x| <= pi/4, Horner with fmaf.
// ---------------------------------------------------------------------------------------------
static inline void sincos_poly(float x, float* s, float* c) {
    float x2 = x * x;
    float ps = fmaf(x2, 2.7557319e-06f, -1.9841270e-04f);   // 1/9!, -1/7!
    ps = fmaf(ps, x2, 8.3333333e-03f);                      // 1/5!
    ps = fmaf(ps, x2, -1.6666667e-01f);                     // -1/3!
    *s = fmaf(x * x2, ps, x);
    float pc = fmaf(x2, -2.7557319e-07f, 2.4801587e-05f);   // -1/10!, 1/8!
    pc = fmaf(pc, x2, -1.3888889e-03f);                     // -1/6!
    pc = fmaf(pc, x2, 4.1666667e-02f);                      // 1/4!
    pc = fmaf(pc, x2, -0.5f);
    *c = fmaf(pc, x2, 1.0f);
}

// sin,cos of 2*pi*u for u in (0,1]; quadrant reduction is exact in u.
static inline void sincos_2pi(float u, float* s, float* c) {
    int q = (int)fmaf(u, 4.0f, 0.5f);            // nearest quarter turn, 0..4
    float r = u - (float)q * 0.25f;              // exact, |r| <= 1/8
    float ss, cc;
    sincos_poly(r * 6.2831855f, &ss, &cc);
    switch (q & 3) {
        case 0: *s = ss;  *c = cc;  break;
        case 1: *s = cc;  *c = -ss; break;
        case 2: *s = -ss; *c = -cc; break;
        default: *s = -cc; *c = ss; break;
    }
}

// sin,cos of an arbitrary angle (radians): two-term Cody-Waite reduction by pi/2.
// |x| > 1e6 (or NaN) is outside the reduction's range and is mapped to 0 so that CPU and GPU
// agree; it only occurs for the reference's degenerate 1 < Ns < ~1.6 lobes.
static inline void sincos_rad(float x, float* s, float* c) {
    if (!(fabsf(x) <= 1.0e6f)) x = 0.0f;
    float n = rintf(x * 0.63661975f);            // x * 2/pi, ties-to-even
    float r = fmaf(-n, 1.5707963705062866f, x);  // pi/2 high part (float)
    r = fmaf(-n, -4.371138828673793e-08f, r);    // pi/2 - high
    int q = (int)n;
    float ss, cc;
    sincos_poly(r, &ss, &cc);
    switch (q & 3) {
        case 0: *s = ss;  *c = cc;  break;
        case 1: *s = cc;  *c = -ss; break;
        case 2: *s = -ss; *c = -cc; break;
        default: *s = -cc; *c = ss; break;
    }
}

static inline uint32_t f2u(float f);
static inline float u2f(uint32_t u);

// ---------------------------------------------------------------------------------------------
// Deterministic log2 / exp2 / pow for the Phong lobe of the `mis` estimator (never libm).
//   log2: x = m * 2^e with m in [sqrt(1/2), sqrt(2)); log2(m) = 2/ln2 * atanh(s), s = (m-1)/(m+1),
//         odd series up to s^9 (|s| <= 0.1716: truncation < 4e-10);
//   exp2: y = n + r, |r| <= 1/2, 2^r by the degree-6 Taylor polynomial of exp(r ln2), scaled by 2^n
//         through the exponent field; y < -126 gives 0.
// ---------------------------------------------------------------------------------------------
static inline float det_log2(float x) {
    uint32_t b;
    memcpy(&b, &x, 4);
    int e = (int)(b >> 23) - 127;
    uint32_t mb = (b & 0x7fffffu) | 0x3f800000u;
    float m;
    memcpy(&m, &mb, 4);
    if (m > 1.41421354f) { m = m * 0.5f; e += 1; }
    float f = m - 1.0f;
    float sq = f / (2.0f + f);
    float s2 = sq * sq;
    float p = fmaf(s2, 0.11111111f, 0.14285715f);
    p = fmaf(p, s2, 0.2f);
    p = fmaf(p, s2, 0.33333334f);
    float r = fmaf(sq * s2, p, sq);
    return fmaf(r, 2.8853900f, (float)e);
}
static inline float det_exp2(float y) {
    if (!(y >= -126.0f)) return 0.0f;
    if (y > 127.0f) y = 127.0f;
    float n = rintf(y);
    float r = y - n;
    float p = fmaf(r, 1.5403530e-4f, 1.3333558e-3f);
    p = fmaf(p, r, 9.6181291e-3f);
    p = fmaf(p, r, 5.5504109e-2f);
    p = fmaf(p, r, 2.4022651e-1f);
    p = fmaf(p, r, 6.9314718e-1f);
    p = fmaf(p, r, 1.0f);
    uint32_t sb = (uint32_t)((int)n + 127) << 23;
    float sc;
    memcpy(&sc, &sb, 4);
    return p * sc;
}
static inline float det_pow(float x, float y) { return det_exp2(y * det_log2(x)); }
// Rec. 709 luminance, used only to choose between lobes and between light triangles
static inline float lumf(V3 c) { return fmaf(0.0722f, c.z, fmaf(0.7152f, c.y, 0.2126f * c.x)); }

static inline uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static inline float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }

}  // namespace orc
