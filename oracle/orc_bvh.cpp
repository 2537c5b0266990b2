// ORACLE — TEST INFRASTRUCTURE ONLY (see orc_math.h). Never linked into the product.
#include "orc_bvh.h"
#include <algorithm>
#include <numeric>

namespace orc {

// =============================================================================================
// Reference host BVH — BVH.h:37-84. Sorting an index array with std::sort and the same
// comparison outcomes yields the same permutation as the reference's std::sort of Triangle
// objects (introsort's moves depend only on comparison results), given the same libstdc++.
// =============================================================================================
namespace {
struct RefBuilder {
    const Scene& s;
    unsigned thresh;
    RefBVH& out;
    int build(int l, int r) {
        if (l >= r) return -1;
        RefNode node;
        node.lc = -1; node.rc = -1; node.it = -1; node.n = 0;
        for (int k = 0; k < 3; ++k) { node.AA[k] = FLT_MAX; node.BB[k] = -FLT_MAX; }
        for (int i = l; i < r; ++i) {                       // BVH.h:43-52
            const Tri& t = s.tris[out.order[i]];
            node.AA[0] = std::min(t.lo.x, node.AA[0]);
            node.AA[1] = std::min(t.lo.y, node.AA[1]);
            node.AA[2] = std::min(t.lo.z, node.AA[2]);
            node.BB[0] = std::max(t.hi.x, node.BB[0]);
            node.BB[1] = std::max(t.hi.y, node.BB[1]);
            node.BB[2] = std::max(t.hi.z, node.BB[2]);
        }
        node.it = l;
        node.n = (unsigned)(r - l);
        if (node.n <= thresh) {                             // BVH.h:57-61
            out.nodes.push_back(node);
            return (int)out.nodes.size() - 1;
        }
        float dx = node.BB[0] - node.AA[0], dy = node.BB[1] - node.AA[1], dz = node.BB[2] - node.AA[2];
        const Scene& sc = s;                                // BVH.h:64-76
        auto b = out.order.begin();
        if (dx >= dy && dx >= dz)
            std::sort(b + l, b + r, [&sc](int a, int c) { return sc.tris[a].center.x < sc.tris[c].center.x; });
        else if (dy >= dx && dy >= dz)
            std::sort(b + l, b + r, [&sc](int a, int c) { return sc.tris[a].center.y < sc.tris[c].center.y; });
        else if (dz >= dx && dz >= dy)
            std::sort(b + l, b + r, [&sc](int a, int c) { return sc.tris[a].center.z < sc.tris[c].center.z; });
        int mid = (l + r) / 2;                              // BVH.h:79-83
        node.lc = build(l, mid);
        node.rc = build(mid, r);
        out.nodes.push_back(node);
        return (int)out.nodes.size() - 1;
    }
};
}  // namespace

void build_ref_bvh(const Scene& s, unsigned thresh_n, RefBVH& out) {
    out.nodes.clear();
    out.order.resize(s.tris.size());
    std::iota(out.order.begin(), out.order.end(), 0);
    RefBuilder rb{s, thresh_n, out};
    out.root = rb.build(0, (int)s.tris.size());
}

// =============================================================================================
// Canonical triangle test — the arithmetic of DeviceTriangle.cuh:39-65 under the contract of
// orc_math.h (dot/cross with explicit fmaf).
// =============================================================================================
bool tri_test(const Tri& tr, V3 o, V3 d, float* t_out) {
    V3 e1 = tr.v2 - tr.v1, e2 = tr.v3 - tr.v1;              // DeviceTriangle.cuh:27-28
    V3 sv = o - tr.v1;
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

static const float kEps = 0.00001f;     // Global.h:11
// Slack of the new box tests: tmin <= tmax * (1 + 2^-17). It has to cover the triangle test's error, not only the
// slab arithmetic: Moeller-Trumbore accepts points a few 1e-6 (relative to the distance) outside a small, far
// triangle, so a shadow ray aimed AT a light-triangle vertex (veach-mis) passed the triangle test and failed a
// 4-ulp box test of the pair-node tree, while the looser quantised boxes of the 8-wide tree let it through.
static const float kSlabSlack = 1.00000762939453125f;

// DeviceBVH.cuh:87-126, literally (including the NaN behaviour of the ?: min/max).
static inline bool ref_hit_aabb(const RefNode& n, V3 o, V3 d, V3 inv) {
    float tminx = (n.AA[0] - o.x) * inv.x, tminy = (n.AA[1] - o.y) * inv.y, tminz = (n.AA[2] - o.z) * inv.z;
    float tmaxx = (n.BB[0] - o.x) * inv.x, tmaxy = (n.BB[1] - o.y) * inv.y, tmaxz = (n.BB[2] - o.z) * inv.z;
    if (d.x < 0) std::swap(tminx, tmaxx);
    if (d.y < 0) std::swap(tminy, tmaxy);
    if (d.z < 0) std::swap(tminz, tmaxz);
    auto mx = [](float x, float y) { return x > y ? x : y; };
    auto mn = [](float x, float y) { return x < y ? x : y; };
    float t_enter = mx(mx(tminx, tminy), tminz);
    float t_exit = mn(mn(tmaxx, tmaxy), tmaxz);
    return t_enter <= t_exit + kEps && t_exit >= 0;
}

Hit ref_intersect(const Scene& s, const RefBVH& b, V3 o, V3 d, bool canonical, TraceStats* st) {
    Hit best{FLT_MAX, -1};
    if (b.root < 0) return best;
    V3 inv{1.0f / d.x, 1.0f / d.y, 1.0f / d.z};            // Ray.cuh:14
    std::vector<int> stack;
    stack.reserve(64);
    stack.push_back(b.root);
    uint64_t max_stack = 1;
    while (!stack.empty()) {
        int cur = stack.back();
        stack.pop_back();
        if (cur < 0) continue;
        const RefNode& node = b.nodes[cur];
        if (st) st->inner++;
        if (node.lc < 0 && node.rc < 0) {                   // DeviceBVH.cuh:141-148, :31-43
            Hit leaf{FLT_MAX, -1};
            for (int i = node.it; i < (int)(node.it + node.n); ++i) {
                float t;
                int face = b.order[i];
                if (st) st->tris++;
                if (!tri_test(s.tris[face], o, d, &t)) continue;
                if (t > kEps && (t < leaf.t || (canonical && t == leaf.t && face < leaf.face))) leaf = Hit{t, face};
            }
            if (leaf.t < best.t || (canonical && leaf.face >= 0 && leaf.t == best.t && leaf.face < best.face)) best = leaf;
        } else {                                            // DeviceBVH.cuh:149-167
            bool hl = node.lc >= 0 && ref_hit_aabb(b.nodes[node.lc], o, d, inv);
            bool hr = node.rc >= 0 && ref_hit_aabb(b.nodes[node.rc], o, d, inv);
            if (st) st->boxes += 2;
            if (hl && hr) { stack.push_back(node.lc); stack.push_back(node.rc); }
            else if (hl) stack.push_back(node.lc);
            else if (hr) stack.push_back(node.rc);
            max_stack = std::max<uint64_t>(max_stack, stack.size());
        }
    }
    if (st) { st->rays++; st->max_stack = std::max(st->max_stack, max_stack); }
    return best;
}

// =============================================================================================
// New builder, CPU statement.  DESIGN.md §"BVH build" is the specification; the CUDA builder
// must reproduce nodes/order/last byte for byte.
//   1. triangle boxes (exact min/max), scene box = union of triangle boxes;
//   2. key = 63-bit Morton code of the box centre, 21 bits per axis,
//        q = clamp(int((c - lo) * (2^21 / extent)), 0, 2^21 - 1), extent == 0 -> q = 0;
//      x in the most significant interleave position;
//   3. stable sort by key (ties keep face-id order);
//   4. Karras 2012 binary radix tree over the sorted keys, duplicate keys disambiguated by index;
//   5. a subtree with <= thresh_n triangles is a leaf (the reference's rule, BVH.h:57);
//   6. kept nodes are numbered by the rank of their radix-tree index; node 0 is the root.
// =============================================================================================
static inline uint64_t expand21(uint64_t x) {
    x &= 0x1fffffull;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

static inline int quant21(float c, float lo, float scale) {
    float f = (c - lo) * scale;
    int q = (int)f;                 // f >= 0 always; NaN cannot occur (scale = 0 when extent == 0)
    if (q > 0x1fffff) q = 0x1fffff;
    if (q < 0) q = 0;
    return q;
}

namespace {
struct Radix {
    const std::vector<uint64_t>& key;
    int n;
    int delta(int i, int j) const {
        if (j < 0 || j >= n) return -1;
        uint64_t a = key[i], b = key[j];
        if (a == b) return 64 + __builtin_clz((unsigned)(i ^ j));
        return __builtin_clzll(a ^ b);
    }
};
}  // namespace

// Steps 1-4 above plus the boxes of the radix nodes: shared by the 64-byte pair-node emitter below
// and by the 8-wide collapse.
struct RadixTree {
    int n = 0;
    V3 lo, hi;                               // scene bounds
    std::vector<int> order;                  // sorted slot -> face id
    std::vector<int> left, right;            // per internal node: >= 0 internal node, < 0 ~slot (single triangle)
    std::vector<int> first, last;            // slot range of each internal node
    std::vector<V3> blo, bhi;                // boxes of the internal nodes
};

// Steps 1-3: scene box, Morton keys, stable sort. Returns the sorted keys (empty when n == 0).
static std::vector<uint64_t> morton_sort(const Scene& s, RadixTree& rt) {
    const int n = (int)s.tris.size();
    rt.n = n;
    rt.lo = V3{FLT_MAX, FLT_MAX, FLT_MAX};
    rt.hi = V3{-FLT_MAX, -FLT_MAX, -FLT_MAX};
    rt.order.clear(); rt.left.clear(); rt.right.clear(); rt.first.clear(); rt.last.clear(); rt.blo.clear(); rt.bhi.clear();
    if (n == 0) return {};
    for (const Tri& t : s.tris) { rt.lo = vmin(rt.lo, t.lo); rt.hi = vmax(rt.hi, t.hi); }
    V3 ext = rt.hi - rt.lo;
    V3 scale{ext.x > 0 ? 2097152.0f / ext.x : 0.0f, ext.y > 0 ? 2097152.0f / ext.y : 0.0f,
             ext.z > 0 ? 2097152.0f / ext.z : 0.0f};
    std::vector<uint64_t> key(n);
    for (int i = 0; i < n; ++i) {
        const Tri& t = s.tris[i];
        V3 c = (t.lo + t.hi) * 0.5f;
        uint64_t qx = quant21(c.x, rt.lo.x, scale.x), qy = quant21(c.y, rt.lo.y, scale.y),
                 qz = quant21(c.z, rt.lo.z, scale.z);
        key[i] = (expand21(qx) << 2) | (expand21(qy) << 1) | expand21(qz);
    }
    rt.order.resize(n);
    std::iota(rt.order.begin(), rt.order.end(), 0);
    std::stable_sort(rt.order.begin(), rt.order.end(), [&](int a, int b) { return key[a] < key[b]; });
    std::vector<uint64_t> skey(n);
    for (int i = 0; i < n; ++i) skey[i] = key[rt.order[i]];
    return skey;
}

static void build_radix_tree(const Scene& s, RadixTree& rt) {
    std::vector<uint64_t> skey = morton_sort(s, rt);
    const int n = rt.n;
    if (n < 2) return;
    // Karras radix tree: internal nodes 0..n-2
    Radix rx{skey, n};
    rt.left.resize(n - 1); rt.right.resize(n - 1); rt.first.resize(n - 1); rt.last.resize(n - 1);
    for (int i = 0; i < n - 1; ++i) {
        int d = (rx.delta(i, i + 1) - rx.delta(i, i - 1)) >= 0 ? 1 : -1;
        int dmin = rx.delta(i, i - d);
        int lmax = 2;
        while (rx.delta(i, i + lmax * d) > dmin) lmax *= 2;
        int l = 0;
        for (int t = lmax / 2; t >= 1; t /= 2)
            if (rx.delta(i, i + (l + t) * d) > dmin) l += t;
        int j = i + l * d;
        int dnode = rx.delta(i, j);
        int sp = 0;
        int t = l;
        do {
            t = (t + 1) >> 1;
            if (rx.delta(i, i + (sp + t) * d) > dnode) sp += t;
        } while (t > 1);
        int gamma = i + sp * d + std::min(d, 0);
        int lo_i = std::min(i, j), hi_i = std::max(i, j);
        rt.first[i] = lo_i; rt.last[i] = hi_i;
        rt.left[i] = (lo_i == gamma) ? ~gamma : gamma;            // ~slot = single-triangle leaf
        rt.right[i] = (hi_i == gamma + 1) ? ~(gamma + 1) : gamma + 1;
    }
    // boxes of radix nodes, bottom-up by recursion on an explicit stack (post-order)
    rt.blo.resize(n - 1); rt.bhi.resize(n - 1);
    auto tri_box = [&](int slot, V3& lo, V3& hi) { lo = s.tris[rt.order[slot]].lo; hi = s.tris[rt.order[slot]].hi; };
    std::vector<std::pair<int, int>> st;   // (node, state)
    st.emplace_back(0, 0);
    while (!st.empty()) {
        auto [nd, state] = st.back();
        if (state == 0) {
            st.back().second = 1;
            if (rt.left[nd] >= 0) st.emplace_back(rt.left[nd], 0);
            if (rt.right[nd] >= 0) st.emplace_back(rt.right[nd], 0);
        } else {
            st.pop_back();
            V3 llo, lhi, rlo, rhi;
            if (rt.left[nd] >= 0) { llo = rt.blo[rt.left[nd]]; lhi = rt.bhi[rt.left[nd]]; } else tri_box(~rt.left[nd], llo, lhi);
            if (rt.right[nd] >= 0) { rlo = rt.blo[rt.right[nd]]; rhi = rt.bhi[rt.right[nd]]; } else tri_box(~rt.right[nd], rlo, rhi);
            rt.blo[nd] = vmin(llo, rlo);
            rt.bhi[nd] = vmax(lhi, rhi);
        }
    }
}

// =============================================================================================
// PLOC topology (builders BUILDER_PLOC / PLOC8) - parallel locally-ordered clustering (Meister & Bittner
// 2018), stated sequentially. It replaces step 4 (the Karras tree) by bottom-up agglomeration, which looks
// at box areas instead of key prefixes and so copes with the large wall triangles next to dense meshes that
// a Morton split handles badly. Specification (the CUDA builder reproduces every array bit for bit):
//   * clusters start as the single triangles in Morton order (steps 1-3 unchanged);
//   * one round: every cluster k finds nn(k) = the cluster j in [k-R, k+R], j != k, that minimises
//     A(k, j) = half area of the union box, (ex*ey + ey*ez) + ez*ex with one rounding per operation;
//     the "buddy" k ^ 1 is examined first, then the window by ascending j, and only a strictly smaller
//     area replaces the choice - so among equal areas the buddy wins, and runs of identical or regularly
//     tessellated triangles pair up (k, k ^ 1) instead of forming one long chain with a single mutual pair
//     per round (257 copies of one triangle: 9 rounds instead of 256);
//     k and j = nn(k) merge iff nn(j) == k; the new cluster takes the place of min(k, j), the other
//     place is dropped, order otherwise kept; rounds repeat until one cluster is left;
//   * merges are numbered in creation order (round by round, by position inside a round); node id =
//     (n - 2) - creation index, so the root is node 0 and every child id is larger than its parent's;
//     left child = the cluster that stood at the lower position;
//   * triangle slots are the depth-first order of the finished tree (left before right), so every node
//     again owns a contiguous slot range [first, last] - what the leaf rule and the wide collapse need.
// =============================================================================================
static const int kPlocRadius = 8;

static void build_ploc_tree(const Scene& s, RadixTree& rt) {
    morton_sort(s, rt);
    const int n = rt.n;
    if (n < 2) return;
    const std::vector<int> morton = rt.order;            // Morton position -> face id
    struct Cl { int ref; int count; V3 lo, hi; };         // ref < 0: ~Morton position of a triangle; else creation index
    std::vector<Cl> cur(n), nxt;
    for (int i = 0; i < n; ++i) cur[i] = Cl{~i, 1, s.tris[morton[i]].lo, s.tris[morton[i]].hi};
    std::vector<int> cl(n - 1), cr(n - 1), ccount(n - 1);  // by creation index
    std::vector<V3> clo(n - 1), chi(n - 1);
    int created = 0, rounds = 0;
    std::vector<int> nn;
    while (cur.size() > 1) {
        const int m = (int)cur.size();
        nn.assign(m, -1);
        for (int k = 0; k < m; ++k) {
            auto area = [&](int j) {
                V3 lo = vmin(cur[k].lo, cur[j].lo), hi = vmax(cur[k].hi, cur[j].hi);
                float ex = hi.x - lo.x, ey = hi.y - lo.y, ez = hi.z - lo.z;
                return (ex * ey + ey * ez) + ez * ex;
            };
            float best = FLT_MAX;
            int bj = -1;
            const int buddy = k ^ 1;
            if (buddy < m) { best = area(buddy); bj = buddy; }
            for (int j = std::max(0, k - kPlocRadius); j <= std::min(m - 1, k + kPlocRadius); ++j) {
                if (j == k || j == buddy) continue;
                float a = area(j);
                if (bj < 0 || a < best) { best = a; bj = j; }
            }
            nn[k] = bj;
        }
        nxt.clear();
        for (int k = 0; k < m; ++k) {
            const int j = nn[k];
            if (nn[j] == k) {
                if (k < j) {
                    const int id = created++;
                    cl[id] = cur[k].ref; cr[id] = cur[j].ref;
                    ccount[id] = cur[k].count + cur[j].count;
                    clo[id] = vmin(cur[k].lo, cur[j].lo); chi[id] = vmax(cur[k].hi, cur[j].hi);
                    nxt.push_back(Cl{id, ccount[id], clo[id], chi[id]});
                }                                       // k > j: dropped
            } else nxt.push_back(cur[k]);
        }
        cur.swap(nxt);
        ++rounds;
    }
    if (getenv("ORC_PLOC_DEBUG")) fprintf(stderr, "ploc: n=%d rounds=%d\n", n, rounds);
    // node ids, slot ranges (top-down: a parent's id is smaller than its children's), final order
    const int ni = n - 1;
    rt.left.resize(ni); rt.right.resize(ni); rt.first.resize(ni); rt.last.resize(ni); rt.blo.resize(ni); rt.bhi.resize(ni);
    auto node_of = [&](int creation) { return ni - 1 - creation; };
    rt.first[0] = 0; rt.last[0] = n - 1;
    std::vector<int> order(n);
    for (int nd = 0; nd < ni; ++nd) {
        const int c = ni - 1 - nd;
        rt.blo[nd] = clo[c]; rt.bhi[nd] = chi[c];
        const int f = rt.first[nd];
        const int lcount = cl[c] < 0 ? 1 : ccount[cl[c]];
        if (cl[c] < 0) { rt.left[nd] = ~f; order[f] = morton[~cl[c]]; }
        else { const int ch = node_of(cl[c]); rt.left[nd] = ch; rt.first[ch] = f; rt.last[ch] = f + lcount - 1; }
        const int g = f + lcount;
        if (cr[c] < 0) { rt.right[nd] = ~g; order[g] = morton[~cr[c]]; }
        else { const int ch = node_of(cr[c]); rt.right[nd] = ch; rt.first[ch] = g; rt.last[ch] = rt.last[nd]; }
    }
    rt.order = order;
}

// Topology stage of a builder id (bit 0 of the product's crt_builder is the node layout, bit 1 the topology).
// A scene of at most thresh_n triangles is ONE leaf: no topology is needed and its slots keep the Morton order,
// whatever the builder (the GPU builder skips the PLOC rounds in that case, crt_bvh_build.cu build_bvh_device).
static void build_tree(const Scene& s, int builder, unsigned thresh_n, RadixTree& rt) {
    if ((builder & 2) && s.tris.size() > (size_t)thresh_n) build_ploc_tree(s, rt);
    else build_radix_tree(s, rt);
}

void build_new_bvh(const Scene& s, unsigned thresh_n, int builder, NewBVH& out) {
    const int n = (int)s.tris.size();
    out.nodes.clear(); out.order.clear(); out.last.clear();
    out.builder = builder;
    if (thresh_n < 1) thresh_n = 1;
    RadixTree rt;
    build_tree(s, builder, thresh_n, rt);
    out.lo = rt.lo; out.hi = rt.hi;
    if (n == 0) return;
    out.order = rt.order;
    out.last.assign(n, 0);
    const std::vector<int>&left = rt.left, &right = rt.right, &first = rt.first, &lastl = rt.last;
    const std::vector<V3>&blo = rt.blo, &bhi = rt.bhi;

    auto tri_box = [&](int slot, V3& lo, V3& hi) { lo = s.tris[out.order[slot]].lo; hi = s.tris[out.order[slot]].hi; };
    auto set_child = [&](PairNode& pn, int which, int ref, int cnt, V3 lo, V3 hi) {
        if (which == 0) { pn.c0 = ref; pn.n0 = cnt; pn.c0lox = lo.x; pn.c0hix = hi.x; pn.c0loy = lo.y; pn.c0hiy = hi.y; pn.c0loz = lo.z; pn.c0hiz = hi.z; }
        else { pn.c1 = ref; pn.n1 = cnt; pn.c1lox = lo.x; pn.c1hix = hi.x; pn.c1loy = lo.y; pn.c1hiy = hi.y; pn.c1loz = lo.z; pn.c1hiz = hi.z; }
    };
    if ((unsigned)n <= thresh_n) {                         // whole scene is one leaf
        PairNode pn{};
        set_child(pn, 0, ~0, n, out.lo, out.hi);
        set_child(pn, 1, kEmptyChild, 0, V3{FLT_MAX, FLT_MAX, FLT_MAX}, V3{-FLT_MAX, -FLT_MAX, -FLT_MAX});
        out.nodes.push_back(pn);
        out.last[n - 1] = 1;
        return;
    }
    // kept nodes: more than thresh_n triangles; rank by radix index
    std::vector<int> rank(n - 1, -1);
    int n_kept = 0;
    for (int i = 0; i < n - 1; ++i)
        if ((unsigned)(lastl[i] - first[i] + 1) > thresh_n) rank[i] = n_kept++;
    out.nodes.resize(n_kept);
    for (int i = 0; i < n - 1; ++i) {
        if (rank[i] < 0) continue;
        PairNode pn{};
        for (int w = 0; w < 2; ++w) {
            int c = w == 0 ? left[i] : right[i];
            V3 lo, hi;
            if (c < 0) {                                     // single triangle
                tri_box(~c, lo, hi);
                set_child(pn, w, ~(~c), 1, lo, hi);
                out.last[~c] = 1;
            } else {
                int cnt = lastl[c] - first[c] + 1;
                lo = blo[c]; hi = bhi[c];
                if (rank[c] >= 0) set_child(pn, w, rank[c], cnt, lo, hi);
                else { set_child(pn, w, ~first[c], cnt, lo, hi); out.last[lastl[c]] = 1; }
            }
        }
        out.nodes[rank[i]] = pn;
    }
}

// =============================================================================================
// New traversal rule (DESIGN.md §"Traversal rule"): conservative slabs, near child first,
// far child pushed, leaves postponed on the stack; t-culling against 1.0001 * current limit.
// =============================================================================================
// A direction component below kParallelDir (2^-40, zero included) has a NaN inverse (orc_math.h box_inv), so its plane
// distances drop out of the min/max above; the axis is tested here instead: the ray stays at o on it (to within
// 2^-40 * exit distance, less than one rounding of dlt), so o must lie inside [lo, hi],
// widened by 2^-17 * (|o| + exit distance + box extent summed over the axes) - the same relative slack as kSlabSlack,
// applied sideways: o is a computed hit point (a few ulp off its surface) and the triangle test's acceptance band scales
// with the distance AND with the triangle's size (a ray 3e-5 outside the 556-unit ceiling triangle of cornell-box is
// accepted; tests/golden/axis_planar_rays.npz). The extent is monotone up the tree, so an ancestor never culls what a
// descendant accepts.
// Without this test an axis-parallel ray (a hemisphere sample exactly along the normal of a wall, a few per frame)
// is culled on one axis only and walks most of the tree: 35 ms for ONE ray of a 1.8 ms launch (profiles/r01_s15.md).
static inline bool parallel_ok(float lo, float hi, float o, float texit, float ext) {
    const float dlt = ((fabsf(o) + texit) + ext) * 7.62939453125e-06f;
    return lo - o <= dlt && o - hi <= dlt;
}

static inline bool slab(float lox, float hix, float loy, float hiy, float loz, float hiz, V3 o, V3 inv,
                        float limit, float* enter) {
    float tx0 = (lox - o.x) * inv.x, tx1 = (hix - o.x) * inv.x;
    float ty0 = (loy - o.y) * inv.y, ty1 = (hiy - o.y) * inv.y;
    float tz0 = (loz - o.z) * inv.z, tz1 = (hiz - o.z) * inv.z;
    float tmin = fmaxf(fmaxf(fminf(tx0, tx1), fminf(ty0, ty1)), fmaxf(fminf(tz0, tz1), 0.0f));
    float tmax = fminf(fminf(fmaxf(tx0, tx1), fmaxf(ty0, ty1)), fminf(fmaxf(tz0, tz1), limit));
    *enter = tmin;
    // Absolute slack pad = 2^-21 * the largest plane distance, as in the wide node step (wide8_intersect). The relative
    // slack is 0 when tmax is: a ray leaving a box plane (o.y == hi.y, d.y > 0) exits that slab at t = 0 exactly, but the
    // triangle test accepts hits a little past the edge that lies in that plane (a ray from the ceiling hitting a wall
    // 2e-5 away). The pad is 2^-21 * |plane - o| / |d| on the axis that gives the largest distance: in position along
    // that axis, a band of at least 2^-22 of the box's extent.
    const float pad = fmaxf(fmaxf(fmaxf(fabsf(tx0), fabsf(tx1)), fmaxf(fabsf(ty0), fabsf(ty1))),
                            fmaxf(fabsf(tz0), fabsf(tz1))) * 4.76837158203125e-07f;
    if (!(tmin <= fmaf(tmax, kSlabSlack, pad))) return false;
    // axes the ray is parallel to (inverse = NaN, see box_inv): the origin coordinate must lie in the box's interval
    if (inv.x != inv.x || inv.y != inv.y || inv.z != inv.z) {
        const float ext = ((hix - lox) + (hiy - loy)) + (hiz - loz);
        if (inv.x != inv.x && !parallel_ok(lox, hix, o.x, tmax, ext)) return false;
        if (inv.y != inv.y && !parallel_ok(loy, hiy, o.y, tmax, ext)) return false;
        if (inv.z != inv.z && !parallel_ok(loz, hiz, o.z, tmax, ext)) return false;
    }
    return true;
}

Hit new_intersect(const Scene& s, const NewBVH& b, const Ray& r, int mode, TraceStats* st) {
    Hit best{FLT_MAX, -1};
    if (st) st->rays++;
    if (b.nodes.empty()) return best;
    V3 o = r.o, d = r.d;
    V3 inv{box_inv(d.x), box_inv(d.y), box_inv(d.z)};
    float tlimit = mode == 0 ? FLT_MAX : r.tmax;
    int stack[128];
    int sp = 0;
    int cur = 0;
    uint64_t max_sp = 0;
    for (;;) {
        if (cur >= 0) {
            if (cur == kEmptyChild) { if (sp == 0) break; cur = stack[--sp]; continue; }
            const PairNode& n = b.nodes[cur];
            if (st) { st->inner++; st->boxes += 2; }
            float lim = tlimit * 1.0001f;
            float e0, e1;
            bool h0 = slab(n.c0lox, n.c0hix, n.c0loy, n.c0hiy, n.c0loz, n.c0hiz, o, inv, lim, &e0);
            bool h1 = slab(n.c1lox, n.c1hix, n.c1loy, n.c1hiy, n.c1loz, n.c1hiz, o, inv, lim, &e1);
            if (h0 && h1) {
                int nearc = n.c0, farc = n.c1;
                if (e1 < e0) { nearc = n.c1; farc = n.c0; }
                stack[sp++] = farc;
                if ((uint64_t)sp > max_sp) max_sp = sp;
                cur = nearc;
            } else if (h0) cur = n.c0;
            else if (h1) cur = n.c1;
            else { if (sp == 0) break; cur = stack[--sp]; }
        } else {
            int slot = ~cur;
            for (;; ++slot) {
                int face = b.order[slot];
                float t;
                if (st) st->tris++;
                if (tri_test(s.tris[face], o, d, &t) && t > kEps) {
                    if (mode == 0) {
                        if (t < best.t || (t == best.t && face < best.face)) { best = Hit{t, face}; tlimit = t; }
                    } else if (r.tmax - t > kEps) {
                        if (st) st->max_stack = std::max(st->max_stack, max_sp);
                        return Hit{t, face};
                    }
                }
                if (b.last[slot]) break;
            }
            if (sp == 0) break;
            cur = stack[--sp];
        }
    }
    if (st) st->max_stack = std::max(st->max_stack, max_sp);
    return best;
}

// =============================================================================================
// 8-wide compressed BVH: collapse of the radix tree, CPU statement (the CUDA builder must
// reproduce nodes / order / last byte for byte; DESIGN.md "Wide nodes" is the specification).
//   * a radix node with more than thresh triangles is "expandable"; anything else is a leaf
//     (single triangle, or a radix node with <= thresh triangles);
//   * the children of a wide node start as the two children of its radix node; the expandable child
//     with the largest box area (first one on ties) is replaced in place by its own two children
//     until there are 8 children or nothing is expandable;
//   * children go to the 8 slots greedily by the largest sum of +-(child centre - node centre)
//     components, sign + where the slot's bit is set (bit 0 x, 1 y, 2 z); a ray then visits
//     slot ^ (its direction octant) in descending order, which is front to back;
//   * boxes are quantised to 8 bits per plane against the node box with power-of-two cell sizes,
//     rounded outwards in exact (double) arithmetic;
//   * nodes are numbered breadth first; the leaf triangles of one node are contiguous, slot order.
// =============================================================================================
namespace {
struct WideChild { int ref; int first, count; V3 lo, hi; bool expandable; };
static inline float box_area(V3 lo, V3 hi) {
    float ex = hi.x - lo.x, ey = hi.y - lo.y, ez = hi.z - lo.z;
    return (ex * ey + ey * ez) + ez * ex;
}
static inline int exp_of_double(double v) {          // floor(log2 v) for a positive normal double
    uint64_t b;
    memcpy(&b, &v, 8);
    return (int)((b >> 52) & 0x7ff) - 1023;
}
}  // namespace

void build_wide8_bvh(const Scene& s, unsigned thresh_n, Wide8BVH& out, int builder) {
    const int n = (int)s.tris.size();
    out.nodes.clear(); out.order.clear(); out.last.clear();
    if (thresh_n < 1) thresh_n = 1;
    if (thresh_n > kWideMaxLeaf) thresh_n = kWideMaxLeaf;
    RadixTree rt;
    build_tree(s, builder, thresh_n, rt);
    out.lo = rt.lo; out.hi = rt.hi;
    if (n == 0) return;
    out.order.assign(n, -1);
    out.last.assign(n, 0);
    auto make_child = [&](int c) {
        WideChild w;
        if (c < 0) {
            const Tri& t = s.tris[rt.order[~c]];
            w = WideChild{c, ~c, 1, t.lo, t.hi, false};
        } else {
            int cnt = rt.last[c] - rt.first[c] + 1;
            w = WideChild{c, rt.first[c], cnt, rt.blo[c], rt.bhi[c], (unsigned)cnt > thresh_n};
        }
        return w;
    };
    struct Pending { int radix; };             // radix < 0: the whole scene as one leaf
    std::vector<Pending> level, next;
    level.push_back(Pending{(unsigned)n <= thresh_n ? -1 : 0});
    int tri_cursor = 0;
    while (!level.empty()) {
        const int level_start = (int)out.nodes.size();
        const int next_start = level_start + (int)level.size();
        next.clear();
        for (const Pending& pn : level) {
            WideChild ch[8];
            int k = 0;
            V3 nlo, nhi;
            if (pn.radix < 0) {
                ch[k++] = WideChild{0, 0, n, rt.lo, rt.hi, false};
                nlo = rt.lo; nhi = rt.hi;
            } else {
                ch[k++] = make_child(rt.left[pn.radix]);
                ch[k++] = make_child(rt.right[pn.radix]);
                nlo = rt.blo[pn.radix]; nhi = rt.bhi[pn.radix];
                while (k < 8) {
                    int best = -1;
                    float best_area = 0.0f;
                    for (int j = 0; j < k; ++j) {
                        if (!ch[j].expandable) continue;
                        float a = box_area(ch[j].lo, ch[j].hi);
                        if (best < 0 || a > best_area) { best = j; best_area = a; }
                    }
                    if (best < 0) break;
                    int c = ch[best].ref;
                    for (int j = k; j > best + 1; --j) ch[j] = ch[j - 1];
                    ch[best] = make_child(rt.left[c]);
                    ch[best + 1] = make_child(rt.right[c]);
                    ++k;
                }
            }
            // slot assignment
            V3 cen = (nlo + nhi) * 0.5f;
            V3 dv[8];
            for (int j = 0; j < k; ++j) dv[j] = (ch[j].lo + ch[j].hi) * 0.5f - cen;
            int slot_of[8], child_in[8];
            for (int j = 0; j < 8; ++j) { slot_of[j] = -1; child_in[j] = -1; }
            for (int it = 0; it < k; ++it) {
                int bj = -1, bs = -1;
                float bc = 0.0f;
                for (int j = 0; j < k; ++j) {
                    if (slot_of[j] >= 0) continue;
                    for (int sl = 0; sl < 8; ++sl) {
                        if (child_in[sl] >= 0) continue;
                        float tx = (sl & 1) ? dv[j].x : -dv[j].x, ty = (sl & 2) ? dv[j].y : -dv[j].y,
                              tz = (sl & 4) ? dv[j].z : -dv[j].z;
                        float c = (tx + ty) + tz;
                        if (bj < 0 || c > bc) { bj = j; bs = sl; bc = c; }
                    }
                }
                slot_of[bj] = bs;
                child_in[bs] = bj;
            }
            // quantisation frame
            uint32_t eb[3];
            double cell[3];
            const float plo[3] = {nlo.x, nlo.y, nlo.z}, phi[3] = {nhi.x, nhi.y, nhi.z};
            for (int a = 0; a < 3; ++a) {
                double ext = (double)phi[a] - (double)plo[a];
                if (!(ext > 0.0)) { eb[a] = 0; cell[a] = 0.0; continue; }
                int e = exp_of_double(ext / 255.0);
                if (ldexp(255.0, e) < ext) e += 1;
                int b = e + 127;
                if (b < 1) b = 1;
                if (b > 254) b = 254;
                eb[a] = (uint32_t)b;
                cell[a] = ldexp(1.0, b - 127);
            }
            Wide8Node node;
            memset(&node, 0, sizeof(node));
            uint8_t meta[8], q[6][8];
            uint32_t imask = 0;
            int n_internal = 0, tri_off = 0;
            for (int sl = 0; sl < 8; ++sl) {
                meta[sl] = 0;
                for (int a = 0; a < 3; ++a) { q[a][sl] = 255; q[3 + a][sl] = 0; }
                int j = child_in[sl];
                if (j < 0) continue;
                const float clo[3] = {ch[j].lo.x, ch[j].lo.y, ch[j].lo.z}, chi[3] = {ch[j].hi.x, ch[j].hi.y, ch[j].hi.z};
                for (int a = 0; a < 3; ++a) {
                    int ql = 0, qh = 0;
                    if (cell[a] > 0.0) {
                        double fl = floor(((double)clo[a] - (double)plo[a]) / cell[a]);
                        double fh = ceil(((double)chi[a] - (double)plo[a]) / cell[a]);
                        ql = fl < 0.0 ? 0 : (fl > 255.0 ? 255 : (int)fl);
                        qh = fh < 0.0 ? 0 : (fh > 255.0 ? 255 : (int)fh);
                    }
                    q[a][sl] = (uint8_t)ql;
                    q[3 + a][sl] = (uint8_t)qh;
                }
                if (ch[j].expandable) {
                    meta[sl] = 0x80;
                    imask |= 1u << sl;
                    next.push_back(Pending{ch[j].ref});
                    ++n_internal;
                } else {
                    meta[sl] = (uint8_t)(1 + tri_off);
                    for (int t = 0; t < ch[j].count; ++t) out.order[tri_cursor + tri_off + t] = rt.order[ch[j].first + t];
                    out.last[tri_cursor + tri_off + ch[j].count - 1] = 1;
                    tri_off += ch[j].count;
                }
            }
            node.w[0] = f2u(plo[0]); node.w[1] = f2u(plo[1]); node.w[2] = f2u(plo[2]);
            node.w[3] = eb[0] | (eb[1] << 8) | (eb[2] << 16) | (imask << 24);
            node.w[4] = (uint32_t)(next_start + (int)next.size() - n_internal);
            node.w[5] = (uint32_t)tri_cursor;
            auto pack4 = [](const uint8_t* b) { return (uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24); };
            node.w[6] = pack4(meta); node.w[7] = pack4(meta + 4);
            for (int a = 0; a < 6; ++a) { node.w[8 + 2 * a] = pack4(q[a]); node.w[9 + 2 * a] = pack4(q[a] + 4); }
            out.nodes.push_back(node);
            tri_cursor += tri_off;
        }
        level.swap(next);
    }
}

// Traversal of the wide BVH, sequential rule (what the tail kernel runs per lane and what the visit counts
// of the roofline refer to): conservative quantised slabs, children visited front to back by slot ^ octant,
// leaf children of a node tested before descending, one stack entry per node with hits left.
Hit wide8_intersect(const Scene& s, const Wide8BVH& b, const Ray& r, int mode, TraceStats* st) {
    Hit best{FLT_MAX, -1};
    if (st) st->rays++;
    if (b.nodes.empty()) return best;
    const V3 o = r.o, d = r.d;
    const V3 inv{box_inv(d.x), box_inv(d.y), box_inv(d.z)};
    const bool negx = inv.x < 0.0f, negy = inv.y < 0.0f, negz = inv.z < 0.0f;
    const uint32_t oinv = (negx ? 0u : 1u) | (negy ? 0u : 2u) | (negz ? 0u : 4u);
    float tlimit = mode == 0 ? FLT_MAX : r.tmax;
    uint32_t stack_base[64], stack_bits[64];
    int sp = 0;
    uint64_t max_sp = 0;
    uint32_t g_base = 0, g_imask = 1, g_mask = 1u << oinv;     // the root as slot 0 of a virtual parent
    for (;;) {
        if (g_mask == 0) {
            if (sp == 0) break;
            --sp;
            g_base = stack_base[sp]; g_imask = stack_bits[sp] >> 8; g_mask = stack_bits[sp] & 0xffu;
        }
        const int pr = 31 - __builtin_clz(g_mask);
        g_mask &= ~(1u << pr);
        const uint32_t sl = (uint32_t)pr ^ oinv;
        const Wide8Node& nd = b.nodes[g_base + (uint32_t)__builtin_popcount(g_imask & ((1u << sl) - 1u))];
        if (st) { st->inner++; st->boxes += 8; }
        const uint32_t ew = nd.w[3];
        const float px = u2f(nd.w[0]), py = u2f(nd.w[1]), pz = u2f(nd.w[2]);
        const float sx = u2f((ew & 0xffu) << 23), sy = u2f(((ew >> 8) & 0xffu) << 23), sz = u2f(((ew >> 16) & 0xffu) << 23);
        const float ax = (px - o.x) * inv.x, ay = (py - o.y) * inv.y, az = (pz - o.z) * inv.z;
        const float bx = sx * inv.x, by = sy * inv.y, bz = sz * inv.z;
        float fax = fabsf(ax), fay = fabsf(ay), faz = fabsf(az);
        if (!(fax <= FLT_MAX)) fax = 0.0f;
        if (!(fay <= FLT_MAX)) fay = 0.0f;
        if (!(faz <= FLT_MAX)) faz = 0.0f;
        // plane distance t = q b + a evaluated as fma(32768 + q, b, a - 32768 b): the GPU gets 32768 + q from one PRMT
        // (crt_wide.cuh wide_biased). The folded bias costs one more rounding, 2^-9 |b| on the distances of ITS axis:
        // near planes are taken e = 2^-7 |b| earlier, far planes later; pad = 2^-21 max|a| as before.
        const float pad = fmaxf(fmaxf(fax, fay), faz) * 4.76837158203125e-07f;     // 2^-21
        float ex = fabsf(bx) * 0.0078125f, ey = fabsf(by) * 0.0078125f, ez = fabsf(bz) * 0.0078125f;
        if (!(ex <= FLT_MAX)) ex = 0.0f;
        if (!(ey <= FLT_MAX)) ey = 0.0f;
        if (!(ez <= FLT_MAX)) ez = 0.0f;
        const float a2x = fmaf(-32768.0f, bx, ax), a2y = fmaf(-32768.0f, by, ay), a2z = fmaf(-32768.0f, bz, az);
        const float anx = a2x - ex, any_ = a2y - ey, anz = a2z - ez, afx = a2x + ex, afy = a2y + ey, afz = a2z + ez;
        const float lim = tlimit * 1.0001f;
        const uint8_t* bytes = (const uint8_t*)nd.w;
        const uint8_t* meta = bytes + 24;
        const uint8_t* qnx = bytes + 32 + (negx ? 24 : 0);      // near planes: hi when the direction is negative
        const uint8_t* qfx = bytes + 32 + (negx ? 0 : 24);
        const uint8_t* qny = bytes + 40 + (negy ? 24 : 0);
        const uint8_t* qfy = bytes + 40 + (negy ? 0 : 24);
        const uint8_t* qnz = bytes + 48 + (negz ? 24 : 0);
        const uint8_t* qfz = bytes + 48 + (negz ? 0 : 24);
        uint32_t node_hits = 0, leaf_hits = 0;                  // priority space
        for (uint32_t c = 0; c < 8; ++c) {
            if (meta[c] == 0) continue;
            const float tnx = fmaf(32768.0f + (float)qnx[c], bx, anx), tfx = fmaf(32768.0f + (float)qfx[c], bx, afx);
            const float tny = fmaf(32768.0f + (float)qny[c], by, any_), tfy = fmaf(32768.0f + (float)qfy[c], by, afy);
            const float tnz = fmaf(32768.0f + (float)qnz[c], bz, anz), tfz = fmaf(32768.0f + (float)qfz[c], bz, afz);
            const float tmin = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, 0.0f));
            const float tmax = fminf(fminf(tfx, tfy), fminf(tfz, lim));
            if (tmin <= fmaf(tmax, kSlabSlack, pad)) {
                // parallel axes (NaN inverse: near = lo, far = hi bytes), same rule as the pair nodes
                if (inv.x != inv.x || inv.y != inv.y || inv.z != inv.z) {
                    const float ext = (fabsf((float)qfx[c] - (float)qnx[c]) * sx + fabsf((float)qfy[c] - (float)qny[c]) * sy) +
                                      fabsf((float)qfz[c] - (float)qnz[c]) * sz;
                    if (inv.x != inv.x && !parallel_ok(fmaf((float)qnx[c], sx, px), fmaf((float)qfx[c], sx, px), o.x, tmax, ext)) continue;
                    if (inv.y != inv.y && !parallel_ok(fmaf((float)qny[c], sy, py), fmaf((float)qfy[c], sy, py), o.y, tmax, ext)) continue;
                    if (inv.z != inv.z && !parallel_ok(fmaf((float)qnz[c], sz, pz), fmaf((float)qfz[c], sz, pz), o.z, tmax, ext)) continue;
                }
                if (meta[c] & 0x80) node_hits |= 1u << (c ^ oinv); else leaf_hits |= 1u << (c ^ oinv);
            }
        }
        while (leaf_hits) {
            const int lp = 31 - __builtin_clz(leaf_hits);
            leaf_hits &= ~(1u << lp);
            int slot = (int)(nd.w[5] + (uint32_t)(meta[(uint32_t)lp ^ oinv] - 1));
            for (;; ++slot) {
                const int face = b.order[slot];
                float t;
                if (st) st->tris++;
                if (tri_test(s.tris[face], o, d, &t) && t > kEps) {
                    if (mode == 0) {
                        if (t < best.t || (t == best.t && face < best.face)) { best = Hit{t, face}; tlimit = t; }
                    } else if (r.tmax - t > kEps) {
                        if (st) st->max_stack = std::max(st->max_stack, max_sp);
                        return Hit{t, face};
                    }
                }
                if (b.last[slot]) break;
            }
        }
        if (node_hits) {
            if (g_mask) {
                stack_base[sp] = g_base; stack_bits[sp] = (g_imask << 8) | g_mask;
                ++sp;
                if ((uint64_t)sp > max_sp) max_sp = sp;
            }
            g_base = nd.w[4]; g_imask = ew >> 24; g_mask = node_hits;
        }
    }
    if (st) st->max_stack = std::max(st->max_stack, max_sp);
    return best;
}

Hit brute_intersect(const Scene& s, const Ray& r, int mode) {
    Hit best{FLT_MAX, -1};
    for (int f = 0; f < (int)s.tris.size(); ++f) {
        float t;
        if (!tri_test(s.tris[f], r.o, r.d, &t) || !(t > kEps)) continue;
        if (mode == 0) { if (t < best.t) best = Hit{t, f}; }     // ascending f: ties keep the lower id
        else if (r.tmax - t > kEps) return Hit{t, f};
    }
    return best;
}

}  // namespace orc
