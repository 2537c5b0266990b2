"""Every traversal against brute force, at the ray directions and scene scales where box tests overflow.

The parity tests elsewhere compare the GPU with the oracle's traversal of the same tree, bit for bit; both state the
same box rule, so a flaw in that rule passes them. Here the references share neither the tree nor its rule:

* brute force (oracle `trace(which=3)`): every triangle, the product's float32 Moeller-Trumbore. The exact reference
  for the closest hit (face id and t bits) and, with mode 1, for "blocked or not";
* a float64 Moeller-Trumbore written below. Where its closest hit is unambiguous it fixes the face and t to 1e-5,
  which guards the float32 triangle test that brute force shares with the product.

Rays: origins uniform in the scene's box, on surfaces (primary hit points) or at triangle vertices moved by up to 1e-5
of the scene size with one coordinate left on the vertex (in a box plane, near its edges); directions random, with one
or two components log-uniform in [1e-45, 1e-3] (denormals included), exactly axis-aligned with signed zeros, or with
one component in [2^-12, 0.1]. Scenes: a box with a triangle soup inside and a free soup, each at scale 1e-4, 1 and 1e5,
offset by 3e5, and at scale 1e-3 offset by 1e3; and cornell-box as shipped. What these rays used to lose: 1 / d
overflowed below 2^-128 (pair and wide nodes); the wide node step's folded bias overflowed to -inf for tiny components
(every child culled); and a ray leaving a box plane, whatever its direction, exited that slab at t = 0 while the
triangle test accepted hits just past the box's edge (pair nodes, which had only a relative slack). box_inv now treats
|d| < 2^-40 as parallel, and the pair slab has the absolute pad of the wide node step (DESIGN.md 4.1)."""
import types

import numpy as np
import pytest

from conftest import BOX_CAMERA, box_scene, soup
from test_oracle import _surface_rays_with_zero_components

FLT_MAX = np.finfo(np.float32).max
EPS = np.float32(0.00001)
KINDS = ("random", "one_small", "two_small", "axis", "near_edge")
RAYS_PER_KIND = 2048                   # half from uniform origins, half from surface points
RAYS_PER_KIND_CORNELL = 512            # 103k triangles: brute force costs 50x more per ray
F64_PAIRS = 1 << 21                    # ray-triangle pairs per kind for the float64 reference (a sample of the rays)

SCENES = [(shape, scale, off) for shape in ("box", "soup")
          for scale, off in ((1e-4, 0.0), (1.0, 0.0), (1e5, 0.0), (1.0, 3e5), (1e-3, 1e3))] + [("cornell-box", None, None)]
SCENE_IDS = ["%s-s%g-o%g" % s if s[1] is not None else s[0] for s in SCENES]
MAT = [[.5, .5, .5, 0, 0, 0, 1]]


def _camera(eye, lookat, fovy):
    return types.SimpleNamespace(eye_pos=np.asarray(eye, np.float32), lookat=np.asarray(lookat, np.float32),
                                 up=np.array([0, 1, 0], np.float32), fovy_rad=np.float32(fovy))


def _directions(rng, kind, n):
    d = rng.normal(size=(n, 3))
    rows = np.arange(n)
    k = rng.integers(0, 3, n)
    k2 = (k + rng.integers(1, 3, n)) % 3
    if kind in ("one_small", "two_small"):
        d[rows, k] = np.copysign(10.0 ** rng.uniform(-45, -3, n), d[rows, k])
        if kind == "two_small":
            d[rows, k2] = np.copysign(10.0 ** rng.uniform(-45, -3, n), d[rows, k2])
    elif kind == "axis":                                          # one zero (in a coordinate plane) or two (along an axis)
        two = rng.random(n) < 0.5
        d[rows, k] = 0.0
        d[rows[two], k2[two]] = 0.0
    d /= np.linalg.norm(d, axis=1, keepdims=True)                 # renormalised in float64, rounded once to float32
    d = d.astype(np.float32)
    if kind == "axis":
        zero = d == 0.0
        d[zero] = np.where(rng.random(int(zero.sum())) < 0.5, np.float32(-0.0), np.float32(0.0))
    return d


def _near_edge_rays(rng, verts, n, size):
    """Origins at points of triangle edges moved by up to 1e-5 of the scene size, with one coordinate left exactly on the
    edge's - where the edge lies in an axis plane (a wall's top edge), that plane: the origin lies in a box plane, next to
    the edge a ray leaving the plane can hit just past. Half of the origins come from such axis-aligned edges when the
    scene has them. Ordinary directions; in half of them the component along that axis is in [2^-12, 0.1], so the ray
    stays near the plane for a while."""
    rows = np.arange(n)
    v = verts.astype(np.float64).reshape(-1, 3, 3)
    p = np.concatenate([v[:, 0], v[:, 1], v[:, 2]])
    q = np.concatenate([v[:, 1], v[:, 2], v[:, 0]])
    flat = np.flatnonzero((p == q).any(axis=1))
    e = rng.integers(0, len(p), n)
    if len(flat):
        e[: n // 2] = flat[rng.integers(0, len(flat), n // 2)]
    pe, qe = p[e], q[e]
    x = pe + rng.uniform(0, 1, (n, 1)) * (qe - pe)
    axis = np.argmax((pe == qe) + rng.uniform(0, 0.5, (n, 3)), axis=1)     # one of the edge's constant coordinates, if any
    o = x + rng.uniform(-1e-5, 1e-5, (n, 3)) * size
    o[rows, axis] = x[rows, axis]
    d = rng.normal(size=(n, 3))
    h = rows[: n // 2]
    d[h, axis[h]] = np.copysign(2.0 ** rng.uniform(-12, np.log2(0.1), len(h)), d[h, axis[h]])
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return o.astype(np.float32), d.astype(np.float32)


def _rays(rng, kind, n, lo, hi, surface, any_hit, verts):
    r = np.zeros((n, 8), np.float32)
    h = n // 2
    size = float(np.linalg.norm(hi - lo))
    if kind == "near_edge":
        r[:, 0:3], r[:, 4:7] = _near_edge_rays(rng, verts, n, size)
    else:
        r[:h, 0:3] = rng.uniform(lo, hi, (h, 3))
        r[h:, 0:3] = surface[rng.integers(0, len(surface), n - h)]
        r[:, 4:7] = _directions(rng, kind, n)
    r[:, 3] = rng.uniform(0, size, n) if any_hit else FLT_MAX
    return r


def _reference_f64(verts, rays):
    """float64 Moeller-Trumbore over all triangles. Returns (face, t, status): status 1 = unambiguous hit, 2 = unambiguous
    miss, 0 = ambiguous. m = 1e-6 + a first-order bound of the float32 test's rounding error in the barycentrics (8 ulp
    of the magnitudes of the products over |det|), terr the same bound for t. A triangle is a possible hit when its
    barycentrics are above -m and t + terr > 1e-5; a sure hit when they are above +m, t - terr > 1e-5 and terr < 5e-6 t
    (well-conditioned: a grazing hit is not). A hit is unambiguous when the nearest possible hit is sure and every other
    possible hit is more than 1e-4 (relative) farther; a miss when no triangle is a possible hit."""
    v = verts.astype(np.float64).reshape(-1, 9)
    v1 = [v[:, 0], v[:, 1], v[:, 2]]
    e1 = [v[:, 3] - v[:, 0], v[:, 4] - v[:, 1], v[:, 5] - v[:, 2]]
    e2 = [v[:, 6] - v[:, 0], v[:, 7] - v[:, 1], v[:, 8] - v[:, 2]]
    le1 = np.sqrt(e1[0] ** 2 + e1[1] ** 2 + e1[2] ** 2)
    le2 = np.sqrt(e2[0] ** 2 + e2[1] ** 2 + e2[2] ** 2)
    n = len(rays)
    face = np.full(n, -1, np.int64)
    t_out = np.full(n, np.inf)
    status = np.zeros(n, np.int8)
    ulp = 2.0 ** -24
    step = max(1, (1 << 20) // len(v))
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for b in range(0, n, step):
            r = rays[b:b + step].astype(np.float64)
            o = [r[:, k, None] for k in range(3)]
            d = [r[:, 4 + k, None] for k in range(3)]
            sv = [o[k] - v1[k] for k in range(3)]
            s1 = [d[1] * e2[2] - d[2] * e2[1], d[2] * e2[0] - d[0] * e2[2], d[0] * e2[1] - d[1] * e2[0]]
            s2 = [sv[1] * e1[2] - sv[2] * e1[1], sv[2] * e1[0] - sv[0] * e1[2], sv[0] * e1[1] - sv[1] * e1[0]]
            det = s1[0] * e1[0] + s1[1] * e1[1] + s1[2] * e1[2]
            beta = (s1[0] * sv[0] + s1[1] * sv[1] + s1[2] * sv[2]) / det
            gamma = (s2[0] * d[0] + s2[1] * d[1] + s2[2] * d[2]) / det
            t = (s2[0] * e2[0] + s2[1] * e2[1] + s2[2] * e2[2]) / det
            alpha = 1.0 - beta - gamma
            lsv = np.sqrt(sv[0] ** 2 + sv[1] ** 2 + sv[2] ** 2)
            adet = np.abs(det)
            m = 1e-6 + 8 * ulp * (le1 + le2) * (lsv + le1 + le2) / adet
            terr = 8 * ulp * le1 * le2 * (lsv + np.abs(t)) / adet + 2 * ulp * np.abs(t)
            ok = np.isfinite(beta) & np.isfinite(gamma) & np.isfinite(t) & np.isfinite(m)
            maybe = ok & (alpha > -m) & (beta > -m) & (gamma > -m) & (t + terr > float(EPS))
            sure = ok & (alpha > m) & (beta > m) & (gamma > m) & (t - terr > float(EPS)) & (terr < 5e-6 * t)
            tm = np.where(maybe, t, np.inf)
            j = np.argmin(tm, axis=1)
            rows = np.arange(len(r))
            t1 = tm[rows, j]
            tm[rows, j] = np.inf
            t2 = tm.min(axis=1)
            hit = sure[rows, j] & (t2 > t1 * (1 + 1e-4))
            miss = ~maybe.any(axis=1)
            face[b:b + step] = np.where(hit, j, -1)
            t_out[b:b + step] = t1
            status[b:b + step] = np.where(hit, 1, np.where(miss, 2, 0))
    return face, t_out, status


def _check_f64(ref, rays, t, f, what):
    """The closest hits of rays[:len(ref face)] against the float64 reference where it is unambiguous."""
    rf, rt, st = ref
    n = len(rf)
    t, f = t[:n], f[:n]
    hit, miss = st == 1, st == 2
    bad_face = hit & (f != rf)
    bad_t = hit & (f == rf) & ~(np.abs(t.astype(np.float64) - rt) <= 1e-5 * rt)
    bad_miss = miss & (f != -1)
    assert not (bad_face.any() or bad_t.any() or bad_miss.any()), \
        "%s: against float64: %d faces differ, %d t off by more than 1e-5 relative, %d hits where no triangle is near " \
        "(of %d unambiguous hits, %d unambiguous misses)" % (what, bad_face.sum(), bad_t.sum(), bad_miss.sum(), hit.sum(), miss.sum())


class Case:
    """One scene: oracle scene, rays per direction kind, brute-force and float64 references (computed once)."""

    def __init__(self, orc, crt, scene_files, spec, seed):
        shape, scale, off = spec
        rng = np.random.default_rng(seed)
        self.obj = None
        if shape == "cornell-box":
            f = scene_files[shape]
            cfg = crt.load_config(f["cfg_path"])
            self.obj = (f["obj"], f["dir"])
            self.S = orc.Scene().add_obj(*self.obj)
            self.thresh = cfg.bvh_thresh_n
            cam = cfg
            self.verts = self.S.tris()["verts"]
            n = RAYS_PER_KIND_CORNELL
        else:
            if shape == "box":
                verts, mat, obj, mats = box_scene(np.random.default_rng(0), 2000)
                cam = (BOX_CAMERA["eye"], BOX_CAMERA["lookat"], BOX_CAMERA["fovy"])
            else:
                verts = soup(np.random.default_rng(1), 2000)
                mat = obj = np.zeros(len(verts), np.int32)
                mats = MAT
                cam = ([0.0, 0.0, -30.0], [0.0, 0.0, 0.0], np.radians(40.0))
            self.verts = (verts.astype(np.float64) * scale + off).astype(np.float32)
            self.arrays = (self.verts, mat, obj, mats)
            self.S = orc.Scene().add_arrays(*self.arrays)
            self.thresh = 2
            cam = _camera(np.asarray(cam[0]) * scale + off, np.asarray(cam[1]) * scale + off, cam[2])
            n = RAYS_PER_KIND
        lo, hi = self.verts.reshape(-1, 3).min(0), self.verts.reshape(-1, 3).max(0)
        self.S.build_new_bvh(self.thresh)
        surface = _surface_rays_with_zero_components(orc, self.S, cam, rng)[:, 0:3]
        assert len(surface) > 100
        self.rays = {(kind, mode): _rays(rng, kind, n, lo, hi, surface, mode == 1, self.verts) for kind in KINDS for mode in (0, 1)}
        self.brute = {key: self.S.trace(r, which=3, mode=key[1]) for key, r in self.rays.items()}
        n64 = max(64, min(n, F64_PAIRS // len(self.verts)))
        self.f64 = {kind: _reference_f64(self.verts, self.rays[(kind, 0)][:n64]) for kind in KINDS}
        for kind in KINDS:                             # the references do test something
            hits = (self.brute[(kind, 0)][1] >= 0).mean()
            f64_hits = (self.f64[kind][2] == 1).mean()
            assert hits > 0.3 and (f64_hits > 0.15 or kind == "near_edge"), (spec, kind, hits, f64_hits)   # near edges: ambiguous by design


_CASES = {}


@pytest.fixture(scope="module")
def case(orc, crt, scene_files):
    def get(spec):
        if spec not in _CASES:
            _CASES[spec] = Case(orc, crt, scene_files, spec, seed=SCENES.index(spec) + 100)
        return _CASES[spec]
    yield get
    _CASES.clear()


def _check_closest(tb, fb, t, f, what):
    bad = (f != fb) | (t.view(np.uint32) != tb.view(np.uint32))
    assert not bad.any(), "%s: %d of %d closest hits differ from brute force (%d lost, %d extra, %d other face or t)" % (
        what, bad.sum(), len(f), (bad & (fb >= 0) & (f < 0)).sum(), (bad & (fb < 0) & (f >= 0)).sum(),
        (bad & (fb >= 0) & (f >= 0)).sum())


def _check_blocked(fb, f, what):
    bad = (f >= 0) != (fb >= 0)
    assert not bad.any(), "%s: 'blocked' differs from brute force for %d of %d rays (%d blockers lost, %d invented)" % (
        what, bad.sum(), len(f), (bad & (fb >= 0)).sum(), (bad & (fb < 0)).sum())


@pytest.mark.parametrize("spec", SCENES, ids=SCENE_IDS)
def test_oracle_traversals_equal_brute_force(case, spec):
    """The oracle's pair-node (which=0) and 8-wide (which=4) traversals, on the LBVH and the PLOC topology."""
    c = case(spec)
    S = c.S
    for kind in KINDS:
        tb, fb = c.brute[(kind, 0)]
        _check_f64(c.f64[kind], c.rays[(kind, 0)], tb, fb, "brute force, %s" % kind)
    for topo, pair_builder, wide_builder in (("lbvh", 0, 1), ("ploc", 2, 3)):
        S.build_new_bvh(c.thresh, pair_builder)
        S.build_wide8(c.thresh, wide_builder)
        for which, layout in ((0, "pair"), (4, "wide")):
            for (kind, mode), rays in c.rays.items():
                t, f = S.trace(rays, which=which, mode=mode)
                what = "%s %s, %s, %s" % (topo, layout, kind, "closest" if mode == 0 else "any")
                if mode == 0:
                    _check_closest(*c.brute[(kind, mode)], t, f, what)
                else:
                    _check_blocked(c.brute[(kind, mode)][1], f, what)


def test_small_components_on_both_sides_of_the_parallel_threshold(orc):
    """d = (1, 0, small) from inside box_scene to the right wall at x = 10, for small on both sides of 2^-40, down to the
    smallest denormal and -0: every traversal finds the wall at t = 5. And rays that leave the ceiling plane y = 10 (the
    top of the root box and of the walls' boxes): the triangle test accepts their wall hits just above the wall's top
    edge, and the pair nodes lost them because the slab test placed their exit from those boxes at t = 0 - for d.y of
    2e-12 .. 1e-9 and, starting 2e-5 beside the wall, for d.y of 0.001 .. 0.1."""
    verts, mat, obj, mats = box_scene(np.random.default_rng(0), 2000)
    S = orc.Scene().add_arrays(verts, mat, obj, mats)
    small = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-38, -1e-36, 2.0 ** -128, 2.0 ** -41, -2.0 ** -40, 2.0 ** -39, 1e-9,
                      1e-6, -2.0 ** -12, 1e-3], np.float32)
    n = len(small)
    side = np.zeros((n, 8), np.float32)
    side[:, 0:3] = [5.0, 2.0, 5.0]
    side[:, 3] = FLT_MAX
    side[:, 4] = 1.0
    side[:, 6] = small
    ceiling = np.array([
        [0.49787330627441406, 10.0, 4.356451034545898, FLT_MAX, -0.816028356552124, 1.0711779241390218e-09, 0.5780118107795715, 0.0],
        [1.9664883613586426, 10.0, 6.342540740966797, FLT_MAX, -0.015656515955924988, 1.8027978198817407e-12, 0.9998774528503418, 0.0],
        [8.546551704406738, 10.0, 7.713382720947266, FLT_MAX, 0.9857819676399231, 9.26690321700896e-12, -0.16802962124347687, 0.0],
        [8.109487533569336, 10.0, 7.351604461669922, FLT_MAX, 0.9818652868270874, 1.387894937865397e-10, 0.18957990407943726, 0.0],
    ], np.float32)
    m = 96                                                   # in the ceiling plane, 2e-5 from the wall x = 10
    edge = np.zeros((m, 8), np.float32)
    edge[:, 0] = np.float32(10.0) - np.float32(2e-5)
    edge[:, 1] = 10.0
    edge[:, 2] = np.linspace(0.5, 9.5, m)
    edge[:, 3] = FLT_MAX
    d = np.stack([np.ones(m), np.resize([0.001, 0.003, 0.01, 0.03, 0.1], m), np.resize([0.2, -0.3, 0.1, -0.05], m)], axis=1)
    edge[:, 4:7] = d / np.linalg.norm(d, axis=1, keepdims=True)   # far above 2^-40: ordinary directions
    rays = np.concatenate([side, ceiling, edge])
    tb, fb = S.trace(rays, which=3, mode=0)
    assert np.allclose(tb[:n], 5.0, rtol=1e-6) and np.all(fb[:n + 4] >= 0) and (fb[n + 4:] >= 0).sum() >= 10
    for builders in ((0, 1), (2, 3)):
        S.build_new_bvh(2, builders[0])
        S.build_wide8(2, builders[1])
        for which in (0, 4):
            t, f = S.trace(rays, which=which, mode=0)
            assert np.array_equal(f, fb) and np.array_equal(t, tb), (builders, which, np.flatnonzero(f != fb))


# ---- GPU --------------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def gpu(crt):
    if crt.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback and these tests need the B200")
    return crt


BUILDERS = ["lbvh", "lbvh8", "ploc", "ploc8"]


@pytest.mark.gpu
@pytest.mark.parametrize("builder", BUILDERS)
@pytest.mark.parametrize("spec", SCENES, ids=SCENE_IDS)
def test_gpu_traversal_equals_brute_force(gpu, case, spec, builder):
    """crt_trace_rays and crt_trace_rays_device, each with and without CRT_RAY_SORTED: closest hits equal brute force
    bit for bit and agree with float64; 'blocked' equals brute force, and a reported blocker passes the triangle test
    with t > 1e-5 and tmax - t > 1e-5 (its t bit for bit)."""
    import torch
    c = case(spec)
    a = gpu.Scene()
    if c.obj is not None:
        a.add_obj(*c.obj)
    else:
        v, mat, obj, mats = c.arrays
        a.add_triangles(v, mat.astype(np.uint32), obj.astype(np.uint32), mats)
    a.set_BVH(c.thresh, builder=BUILDERS.index(builder))
    for (kind, mode), rays in c.rays.items():
        n = len(rays)
        tb, fb = c.brute[(kind, mode)]
        d_rays = torch.from_numpy(rays).cuda()
        d_t = torch.empty(n, dtype=torch.float32, device="cuda")
        d_f = torch.empty(n, dtype=torch.int32, device="cuda")
        for sorted_ in (0, gpu.RAY_SORTED):
            for entry in ("host", "device"):
                what = "%s, %s, %s, %s%s" % (builder, kind, "closest" if mode == 0 else "any", entry, " sorted" if sorted_ else "")
                if entry == "host":
                    t, f, _ = a.trace_rays(rays, mode | sorted_)
                else:
                    a.trace_rays_device(d_rays.data_ptr(), n, mode | sorted_, d_t.data_ptr(), d_f.data_ptr())
                    torch.cuda.synchronize()
                    t, f = d_t.cpu().numpy(), d_f.cpu().numpy()
                if mode == 0:
                    _check_closest(tb, fb, t, f, what)
                    _check_f64(c.f64[kind], rays, t, f, what)
                    continue
                _check_blocked(fb, f, what)
                miss, hit = f < 0, f >= 0
                assert np.all(t[miss] == FLT_MAX), what
                tt, inside = c.S.tri_test(rays[hit], f[hit])
                th = t[hit]
                assert np.all(inside) and np.array_equal(tt.view(np.uint32), th.view(np.uint32)), what
                assert np.all(th > EPS) and np.all(rays[hit, 3] - th > EPS), what


def _range_scene(rng):
    """box_scene with two far triangles near -2^72 and +2^72 (crt.h's stated coordinate range): the root node's cell size
    is then 2^66, and with 1 / d up to 2^40 the wide node step's folded bias reaches 2^121. Rays from inside the box, one
    component just above and below 2^-40, half of the rest with one component in [2^-40, 0.1]."""
    verts, mat, obj, mats = box_scene(np.random.default_rng(0), 200)
    far = np.float32(2.0 ** 72)
    h = np.float32(2.0 ** 62)
    extra = np.array([[-far, 0, 0, -far + h, 0, 0, -far, h, 0], [far, 0, 0, far - h, 0, 0, far, h, 0]], np.float32)
    arrays = (np.concatenate([verts, extra]), np.concatenate([mat, [0, 0]]), np.concatenate([obj, [obj.max() + 1] * 2]), mats)
    n = 4000
    rays = np.zeros((n, 8), np.float32)
    rays[:, 0:3] = rng.uniform(0.5, 9.5, (n, 3))
    rays[:, 3] = FLT_MAX
    d = rng.normal(size=(n, 3))
    rows = np.arange(n)
    small = np.where(rows % 2 == 0, 2.0 ** -40 * rng.uniform(0.5, 4.0, n), 2.0 ** rng.uniform(-40, np.log2(0.1), n))
    d[rows, rng.integers(0, 3, n)] = np.copysign(small, rng.normal(size=n))
    rays[:, 4:7] = d / np.linalg.norm(d, axis=1, keepdims=True)
    return arrays, rays


def test_scene_spanning_the_stated_coordinate_range(orc):
    """The oracle's pair and wide traversals on both topologies equal brute force on _range_scene."""
    arrays, rays = _range_scene(np.random.default_rng(9))
    S = orc.Scene().add_arrays(*arrays)
    tb, fb = S.trace(rays, which=3, mode=0)
    assert (fb >= 0).mean() > 0.5
    for pair_builder, wide_builder in ((0, 1), (2, 3)):
        S.build_new_bvh(2, pair_builder)
        S.build_wide8(2, wide_builder)
        for which in (0, 4):
            t, f = S.trace(rays, which=which, mode=0)
            _check_closest(tb, fb, t, f, "builders %d/%d, which %d" % (pair_builder, wide_builder, which))


@pytest.mark.gpu
@pytest.mark.parametrize("builder", BUILDERS)
def test_gpu_scene_spanning_the_stated_coordinate_range(gpu, orc, builder):
    """The GPU's node steps (the wide one holds the folded bias) on _range_scene equal brute force, for every builder."""
    arrays, rays = _range_scene(np.random.default_rng(9))
    S = orc.Scene().add_arrays(*arrays)
    tb, fb = S.trace(rays, which=3, mode=0)
    v, mat, obj, mats = arrays
    a = gpu.Scene().add_triangles(v, mat.astype(np.uint32), obj.astype(np.uint32), mats)
    a.set_BVH(2, builder=BUILDERS.index(builder))
    t, f, _ = a.trace_rays(rays, gpu.RAY_CLOSEST)
    _check_closest(tb, fb, t, f, builder)
