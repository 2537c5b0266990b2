"""Host-side mirror of the reference's interface over the C-ABI (include/crt.h).

Reference call sites (file:line in guomc9/CudaRayTracing):
  Scene            include/Scene.h:16-101        -> class Scene
  Render           include/Render.cuh:357-557    -> class Render
  config_task      src/main.cu:67-90             -> load_config / Config
  get_inverse_view_matrix  include/Camera.h:9-36 -> inverse_view_matrix
"""
import ctypes as C
import math
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

ESTIMATOR_COMPAT, ESTIMATOR_MIS = 0, 1
RAY_CLOSEST, RAY_ANY = 0, 1
RAY_SORTED = 0x100                      # flag: trace in (origin cell, direction octant) order, hits back in the caller's order
BUILDER_LBVH, BUILDER_LBVH8, BUILDER_PLOC, BUILDER_PLOC8 = 0, 1, 2, 3     # bit 0: 8-wide nodes, bit 1: PLOC topology
MAX_OBJ_PATHS, PATH_LEN = 16, 1024


class CrtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("crt error %d: %s" % (code, msg))
        self.code = code


class _Material(C.Structure):
    _fields_ = [("kd", C.c_float * 3), ("ks", C.c_float * 3), ("ke", C.c_float * 3), ("ns", C.c_float)]


class _Config(C.Structure):
    _fields_ = [("n_obj", C.c_uint32), ("obj_path", (C.c_char * PATH_LEN) * MAX_OBJ_PATHS),
                ("mtl_dir", (C.c_char * PATH_LEN) * MAX_OBJ_PATHS), ("eye_pos", C.c_float * 3), ("lookat", C.c_float * 3),
                ("up", C.c_float * 3), ("fov_y", C.c_float), ("width", C.c_uint32), ("height", C.c_uint32),
                ("bvh_thresh_n", C.c_uint32), ("p_rr", C.c_float), ("spp", C.c_uint32), ("light_sample_n", C.c_uint32),
                ("seed", C.c_uint32), ("estimator", C.c_uint32)]


class _Stats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("extend_rays", C.c_uint64), ("shadow_rays", C.c_uint64), ("probe_rays", C.c_uint64),
                ("iterations", C.c_uint64), ("kernel_launches", C.c_uint64), ("ms_total", C.c_float), ("ms_extend", C.c_float),
                ("ms_shade", C.c_float), ("ms_shadow", C.c_float), ("ms_generate", C.c_float), ("ms_tail", C.c_float)]


BVH_NODE = np.dtype([("c0lox", "<f4"), ("c0hix", "<f4"), ("c0loy", "<f4"), ("c0hiy", "<f4"),
                     ("c1lox", "<f4"), ("c1hix", "<f4"), ("c1loy", "<f4"), ("c1hiy", "<f4"),
                     ("c0loz", "<f4"), ("c0hiz", "<f4"), ("c1loz", "<f4"), ("c1hiz", "<f4"),
                     ("c0", "<i4"), ("c1", "<i4"), ("n0", "<i4"), ("n1", "<i4")])
# crt_bvh8_node (include/crt.h): 80 bytes
BVH8_NODE = np.dtype([("origin", "<f4", 3), ("exp", "u1", 3), ("imask", "u1"), ("child_base", "<u4"), ("tri_base", "<u4"),
                      ("meta", "u1", 8), ("qlo_x", "u1", 8), ("qlo_y", "u1", 8), ("qlo_z", "u1", 8),
                      ("qhi_x", "u1", 8), ("qhi_y", "u1", 8), ("qhi_z", "u1", 8)])
assert BVH8_NODE.itemsize == 80


def lib_path():
    # CRT_LIB: development override (tools/build_variant.sh) to compare kernel variants in one GPU session
    return os.environ.get("CRT_LIB") or os.path.join(_HERE, "libcrt.so")


def load_library():
    """Loads libcrt.so. Raises (never falls back) when it has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    p = lib_path()
    if not os.path.exists(p):
        raise CrtError(-2, "native library %s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "or `make -C cudaraytracing_b200` (there is no CPU fallback)" % p)
    L = C.CDLL(p)
    vp, u32, u64, f32, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_float, C.c_int
    pp = C.POINTER(C.c_void_p)
    L.crt_last_error.restype = C.c_char_p
    sig = {
        "crt_config_load": [C.c_char_p, C.POINTER(_Config)],
        "crt_inverse_view_matrix": [vp, vp, vp, vp],
        "crt_write_png": [C.c_char_p, vp, u32, u32],
        "crt_scene_create": [pp],
        "crt_scene_add_obj": [vp, C.c_char_p, C.c_char_p],
        "crt_scene_add_triangles": [vp, vp, vp, vp, u64, vp, u32],
        "crt_scene_build_bvh": [vp, u32, i32, i32, C.POINTER(f32)],
        "crt_scene_counts": [vp, C.POINTER(u64), C.POINTER(u32), C.POINTER(u32), C.POINTER(u64)],
        "crt_scene_export_tris": [vp, vp, vp, vp, vp, vp, vp],
        "crt_scene_export_mats": [vp, vp],
        "crt_scene_export_light": [vp, u32, vp, C.POINTER(u32), C.POINTER(f32)],
        "crt_scene_export_bvh": [vp, vp, vp, vp, vp],
        "crt_scene_export_bvh8": [vp, vp, vp, vp, vp],
        "crt_scene_bvh_kind": [vp, C.POINTER(i32)],
        "crt_scene_destroy": [vp],
        "crt_trace_rays": [vp, vp, u64, i32, vp, vp, C.POINTER(f32)],
        "crt_trace_rays_device": [vp, vp, u64, i32, vp, vp, vp, C.POINTER(f32)],
        "crt_random_rays_device": [vp, vp, u64, u64, u32, i32, vp],
        "crt_render_create": [vp, u32, u32, pp],
        "crt_render_set_spp": [vp, u32],
        "crt_render_set_p_rr": [vp, f32],
        "crt_render_set_light_sample_n": [vp, u32],
        "crt_render_set_seed": [vp, u32],
        "crt_render_set_estimator": [vp, i32],
        "crt_render_set_sample_range": [vp, u32, u32],
        "crt_render_set_work_range": [vp, u64, u64],
        "crt_render_clear_range": [vp],
        "crt_render_set_stream": [vp, vp],
        "crt_render_set_stage_timing": [vp, i32],
        "crt_render_run_view": [vp, vp, vp, f32],
        "crt_render_set_accumulate": [vp, i32],
        "crt_render_clear_accum": [vp],
        "crt_render_save_checkpoint": [vp, C.c_char_p, u64],
        "crt_render_load_checkpoint": [vp, C.c_char_p, C.POINTER(u64), vp, vp, C.POINTER(f32)],
        "crt_render_device_accum": [vp, pp],
        "crt_render_get_accum_i64": [vp, vp],
        "crt_render_get_accum": [vp, vp],
        "crt_render_get_rgb8": [vp, vp],
        "crt_render_get_rgb8_device": [vp, vp],
        "crt_render_save_png": [vp, C.c_char_p],
        "crt_render_get_stats": [vp, C.POINTER(_Stats)],
        "crt_render_set_aov": [vp, i32],
        "crt_render_get_aov": [vp, vp, vp, vp, vp],
        "crt_render_get_aov_i64": [vp, vp, C.POINTER(f32)],
        "crt_render_device_aov": [vp, pp, C.POINTER(f32)],
        "crt_group_set_aov": [vp, i32],
        "crt_group_get_aov": [vp, vp, vp, vp, vp],
        "crt_group_get_aov_i64": [vp, vp, C.POINTER(f32)],
        "crt_render_destroy": [vp],
        "crt_group_create": [vp, u32, u32, vp, u32, pp],
        "crt_group_set_params": [vp, u32, f32, u32, u32, i32],
        "crt_group_run_view": [vp, vp, vp, f32],
        "crt_group_get_accum_i64": [vp, vp],
        "crt_group_get_rgb8": [vp, vp],
        "crt_group_save_png": [vp, C.c_char_p],
        "crt_group_get_stats": [vp, u32, C.POINTER(_Stats), C.POINTER(f32)],
        "crt_group_destroy": [vp],
    }
    for name, argtypes in sig.items():
        fn = getattr(L, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    _LIB = L
    return L


def _check(rc):
    if rc != 0:
        raise CrtError(rc, load_library().crt_last_error().decode(errors="replace"))


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def device_count():
    return load_library().crt_device_count()


def inverse_view_matrix(eye, lookat, up):
    """get_inverse_view_matrix, include/Camera.h:9-36 (row-major 3x3, columns [r u f])."""
    e, l, u = (np.ascontiguousarray(x, np.float32) for x in (eye, lookat, up))
    out = np.zeros(9, np.float32)
    _check(load_library().crt_inverse_view_matrix(_p(e), _p(l), _p(u), _p(out)))
    return out


def write_png(path, rgb8):
    rgb8 = np.ascontiguousarray(rgb8, np.uint8)
    h, w = rgb8.shape[0], rgb8.shape[1]
    _check(load_library().crt_write_png(path.encode(), _p(rgb8), w, h))


class Config:
    """struct Task, src/main.cu:40-56."""

    def __init__(self, c):
        self.OBJ_paths = [(c.obj_path[k].value.decode(), c.mtl_dir[k].value.decode()) for k in range(c.n_obj)]
        self.eye_pos = np.array(c.eye_pos[:], np.float32)
        self.lookat = np.array(c.lookat[:], np.float32)
        self.up = np.array(c.up[:], np.float32)
        self.fov_y = c.fov_y
        self.width, self.height = c.width, c.height
        self.bvh_thresh_n = c.bvh_thresh_n
        self.P_RR = c.p_rr
        self.spp = c.spp
        self.light_sample_n = c.light_sample_n
        self.seed = c.seed
        self.estimator = c.estimator

    @property
    def fovy_rad(self):
        return np.float32(np.float32(self.fov_y) * np.float32(math.pi) / np.float32(180.0))


def load_config(path):
    """config_task(), src/main.cu:67-90."""
    c = _Config()
    _check(load_library().crt_config_load(path.encode(), C.byref(c)))
    return Config(c)


class Scene:
    """Scene (include/Scene.h:16-101) + BVH (include/BVH.h) + the device uploads."""

    def __init__(self):
        self.L = load_library()
        h = C.c_void_p()
        _check(self.L.crt_scene_create(C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.crt_scene_destroy(self.h)
            self.h = None

    __del__ = close

    def add_obj(self, obj_path, mtl_dir):
        """Loader::read_OBJ + load_object loop (src/main.cu:122-145)."""
        _check(self.L.crt_scene_add_obj(self.h, obj_path.encode(), mtl_dir.encode()))
        return self

    def add_triangles(self, verts, mat_id, obj_id, mats):
        """mats: rows of (kd[3], ke[3], ns) or (kd[3], ks[3], ke[3], ns)."""
        verts = np.ascontiguousarray(verts, np.float32).reshape(-1, 9)
        mat_id = np.ascontiguousarray(mat_id, np.uint32)
        obj_id = np.ascontiguousarray(obj_id, np.uint32)
        if not (len(mat_id) == len(obj_id) == verts.shape[0]):
            raise ValueError("mat_id and obj_id need one entry per triangle (%d triangles, %d / %d ids)" % (verts.shape[0], len(mat_id), len(obj_id)))
        mats = np.asarray(mats, np.float32)
        if mats.ndim != 2 or mats.shape[1] not in (7, 10):
            raise ValueError("mats must be n x 7 (kd,ke,ns) or n x 10 (kd,ks,ke,ns)")
        arr = (_Material * len(mats))()
        for k, m in enumerate(mats):
            if len(m) == 7:
                arr[k].kd[:] = m[0:3]; arr[k].ks[:] = [0, 0, 0]; arr[k].ke[:] = m[3:6]; arr[k].ns = m[6]
            else:
                arr[k].kd[:] = m[0:3]; arr[k].ks[:] = m[3:6]; arr[k].ke[:] = m[6:9]; arr[k].ns = m[9]
        _check(self.L.crt_scene_add_triangles(self.h, _p(verts), _p(mat_id), _p(obj_id), verts.shape[0],
                                              C.cast(arr, C.c_void_p), len(mats)))
        return self

    def set_BVH(self, thresh_n, builder=0, device=0):
        """Scene::set_BVH (include/Scene.h:50-54), built on the GPU. Returns the build time in ms."""
        ms = C.c_float()
        _check(self.L.crt_scene_build_bvh(self.h, thresh_n, builder, device, C.byref(ms)))
        return ms.value

    def counts(self):
        nt, nm, nl, nn = C.c_uint64(), C.c_uint32(), C.c_uint32(), C.c_uint64()
        _check(self.L.crt_scene_counts(self.h, C.byref(nt), C.byref(nm), C.byref(nl), C.byref(nn)))
        return dict(n_tris=nt.value, n_mats=nm.value, n_lights=nl.value, n_nodes=nn.value)

    def tris(self):
        n = self.counts()["n_tris"]
        d = dict(verts=np.zeros((n, 9), np.float32), normal=np.zeros((n, 3), np.float32), area=np.zeros(n, np.float32),
                 area_of_obj=np.zeros(n, np.float32), mat=np.zeros(n, np.int32), obj=np.zeros(n, np.int32))
        _check(self.L.crt_scene_export_tris(self.h, *[_p(d[k]) for k in ("verts", "normal", "area", "area_of_obj", "mat", "obj")]))
        return d

    def mats(self):
        out = np.zeros((self.counts()["n_mats"], 9), np.float32)
        _check(self.L.crt_scene_export_mats(self.h, _p(out)))
        return out

    def lights(self):
        res = []
        for li in range(self.counts()["n_lights"]):
            n, area = C.c_uint32(0), C.c_float()
            _check(self.L.crt_scene_export_light(self.h, li, None, C.byref(n), C.byref(area)))
            faces = np.zeros(n.value, np.int32)
            _check(self.L.crt_scene_export_light(self.h, li, _p(faces), C.byref(n), C.byref(area)))
            res.append((faces, area.value))
        return res

    def bvh_kind(self):
        k = C.c_int()
        _check(self.L.crt_scene_bvh_kind(self.h, C.byref(k)))
        return k.value

    def export_bvh(self):
        """nodes (BVH_NODE, or BVH8_NODE for a scene built with BUILDER_LBVH8), order, last, bounds."""
        c = self.counts()
        wide = bool(self.bvh_kind() & 1)
        nodes = np.zeros(c["n_nodes"], BVH8_NODE if wide else BVH_NODE)
        order = np.zeros(c["n_tris"], np.int32)
        last = np.zeros(c["n_tris"], np.uint8)
        bounds = np.zeros(6, np.float32)
        fn = self.L.crt_scene_export_bvh8 if wide else self.L.crt_scene_export_bvh
        _check(fn(self.h, _p(nodes), _p(order), _p(last), _p(bounds)))
        return nodes, order, last, bounds

    def trace_rays(self, rays, mode=RAY_CLOSEST, out=None):
        """rays: n x 8 float32 {o, tmax, d, 0}. Returns (t, face, kernel_ms). out = (t, face): caller-owned result arrays
        (float32 / int32, n each), e.g. page-locked ones, which the library then fills by DMA without staging."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8)
        n = rays.shape[0]
        if out is not None:
            t, face = out
            if t.dtype != np.float32 or face.dtype != np.int32 or t.size < n or face.size < n or not (t.flags.c_contiguous and face.flags.c_contiguous):
                raise ValueError("trace_rays: out must be contiguous (float32[n], int32[n])")
        else:
            t = np.zeros(n, np.float32)
            face = np.zeros(n, np.int32)
        ms = C.c_float()
        _check(self.L.crt_trace_rays(self.h, _p(rays), n, mode, _p(t), _p(face), C.byref(ms)))
        return t, face, ms.value

    def trace_rays_device(self, d_rays_ptr, n, mode, d_t_ptr, d_face_ptr, stream=None):
        ms = C.c_float()
        _check(self.L.crt_trace_rays_device(self.h, d_rays_ptr, n, mode, d_t_ptr, d_face_ptr, stream, C.byref(ms)))
        return ms.value


    def random_rays_device(self, d_rays_ptr, n, start=0, key=0xC5, any_hit=False, stream=None):
        _check(self.L.crt_random_rays_device(self.h, d_rays_ptr, n, start, key, 1 if any_hit else 0, stream))


class Render:
    """Render (include/Render.cuh:357-557): ctor :379, run_view :435, setters :543-556, save :489."""

    def __init__(self, scene, width, height, spp=16, P_RR=0.8, light_sample_n=1):
        self.L = load_library()
        self.scene = scene
        self.width, self.height = width, height
        h = C.c_void_p()
        _check(self.L.crt_render_create(scene.h, width, height, C.byref(h)))
        self.h = h
        self.set_spp(spp)
        self.set_P_RR(P_RR)
        self.set_light_sample_n(light_sample_n)

    def close(self):
        if getattr(self, "h", None):
            self.L.crt_render_destroy(self.h)
            self.h = None

    __del__ = close

    def set_spp(self, spp):
        self.spp = spp
        _check(self.L.crt_render_set_spp(self.h, spp))

    def set_P_RR(self, p_rr):
        _check(self.L.crt_render_set_p_rr(self.h, p_rr))

    def set_light_sample_n(self, n):
        _check(self.L.crt_render_set_light_sample_n(self.h, n))

    def set_seed(self, seed):
        _check(self.L.crt_render_set_seed(self.h, seed))

    def set_estimator(self, estimator):
        _check(self.L.crt_render_set_estimator(self.h, estimator))

    def set_sample_range(self, begin, end):
        _check(self.L.crt_render_set_sample_range(self.h, begin, end))

    def set_work_range(self, begin, end):
        _check(self.L.crt_render_set_work_range(self.h, begin, end))

    def clear_range(self):
        _check(self.L.crt_render_clear_range(self.h))

    def set_stream(self, cuda_stream):
        _check(self.L.crt_render_set_stream(self.h, cuda_stream))

    def set_stage_timing(self, on):
        _check(self.L.crt_render_set_stage_timing(self.h, 1 if on else 0))

    def run_view(self, eye_pos, inv_view_mat, fovY):
        """Render::run_view (include/Render.cuh:435-475); fovY in radians like the reference."""
        e = np.ascontiguousarray(eye_pos, np.float32)
        m = np.ascontiguousarray(inv_view_mat, np.float32).reshape(9)
        _check(self.L.crt_render_run_view(self.h, _p(e), _p(m), float(fovY)))

    def set_accumulate(self, on):
        """Progressive rendering: run_view adds its work range to the accumulation buffer instead of clearing it."""
        _check(self.L.crt_render_set_accumulate(self.h, 1 if on else 0))

    def clear_accum(self):
        _check(self.L.crt_render_clear_accum(self.h))

    def save_checkpoint(self, path, work_done):
        _check(self.L.crt_render_save_checkpoint(self.h, str(path).encode(), int(work_done)))

    def load_checkpoint(self, path):
        """Returns (work_done, eye, inv_view 3x3, fovy_rad) of the checkpoint; the handle continues to accumulate."""
        wd, fov = C.c_uint64(), C.c_float()
        eye, M = np.zeros(3, np.float32), np.zeros(9, np.float32)
        _check(self.L.crt_render_load_checkpoint(self.h, str(path).encode(), C.byref(wd), _p(eye), _p(M), C.byref(fov)))
        return wd.value, eye, M.reshape(3, 3), np.float32(fov.value)

    def device_accum_ptr(self):
        p = C.c_void_p()
        _check(self.L.crt_render_device_accum(self.h, C.byref(p)))
        return p.value

    def get_accum_i64(self):
        out = np.zeros(self.width * self.height * 3, np.int64)
        _check(self.L.crt_render_get_accum_i64(self.h, _p(out)))
        return out

    def get_accum(self):
        out = np.zeros((self.height, self.width, 3), np.float32)
        _check(self.L.crt_render_get_accum(self.h, _p(out)))
        return out

    def get_frame_buffer(self, out=None):
        """Render::get_frame_buffer (include/Render.cuh:495): RGB8, top row first."""
        if out is None:
            out = np.zeros((self.height, self.width, 3), np.uint8)
        _check(self.L.crt_render_get_rgb8(self.h, _p(out)))
        return out

    def frame_to_device(self, device_ptr):
        """The display path of Render::run_view(..., cuda_pbo_resource) (include/Render.cuh:446-469): the RGB8 frame written
        into a device buffer of width*height*3 bytes the caller owns (a mapped GL pixel buffer object, a torch tensor ...)."""
        _check(self.L.crt_render_get_rgb8_device(self.h, C.c_void_p(device_ptr)))

    def save_frame_buffer(self, path):
        _check(self.L.crt_render_save_png(self.h, path.encode()))

    def set_aov(self, on):
        """AOV buffers for denoisers (include/crt.h crt_render_set_aov): run_view also accumulates first-hit albedo, normal,
        depth and coverage over the same samples as the colour."""
        _check(self.L.crt_render_set_aov(self.h, 1 if on else 0))

    def get_aov(self):
        """dict of albedo (H,W,3), normal (H,W,3), depth (H,W; +inf where no sample hit), coverage (H,W), top row first."""
        return _aov_images(self.L.crt_render_get_aov, self.h, self.width, self.height)

    def get_aov_i64(self):
        """(raw int64[W*H*8] fixed-point AOV buffer, depth_unit)"""
        return _aov_i64(self.L.crt_render_get_aov_i64, self.h, self.width, self.height)

    def device_aov_ptr(self):
        p = C.c_void_p()
        _check(self.L.crt_render_device_aov(self.h, C.byref(p), None))
        return p.value

    def stats(self):
        s = _Stats()
        _check(self.L.crt_render_get_stats(self.h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in _Stats._fields_}


def _aov_images(fn, h, width, height):
    d = dict(albedo=np.zeros((height, width, 3), np.float32), normal=np.zeros((height, width, 3), np.float32),
             depth=np.zeros((height, width), np.float32), coverage=np.zeros((height, width), np.float32))
    _check(fn(h, _p(d["albedo"]), _p(d["normal"]), _p(d["depth"]), _p(d["coverage"])))
    return d


def _aov_i64(fn, h, width, height):
    out = np.zeros(width * height * 8, np.int64)
    unit = C.c_float()
    _check(fn(h, _p(out), C.byref(unit)))
    return out, unit.value


def _prefer_bundled_nccl():
    """The library loads NCCL by name (`libnccl.so.2`, or CRT_NCCL_LIB) when a group of several GPUs is created. In a Python process
    that also imports torch, both must map the SAME file: torch's CUDA library is linked against the NCCL wheel next to it, and a
    different libnccl.so.2 loaded first (the system one) makes `import torch` fail on a missing symbol. So, unless the caller chose
    a file, name the wheel's library when there is one."""
    if os.environ.get("CRT_NCCL_LIB"):
        return
    import importlib.util
    try:
        spec = importlib.util.find_spec("nvidia.nccl")
    except (ImportError, ValueError):
        spec = None
    for base in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
        cand = os.path.join(base, "lib", "libnccl.so.2")
        if os.path.exists(cand):
            os.environ["CRT_NCCL_LIB"] = cand
            return


class RenderGroup:
    """Render for several GPUs of one box driven by the calling thread (crt_group, include/crt.h): the built scene is copied
    device to device, GPU g renders its share of the samples, one NCCL reduce sums the int64 buffers onto devices[0].
    The reduced buffer and the frame are bit-identical to the single-GPU Render's."""

    def __init__(self, scene, width, height, devices, spp=16, P_RR=0.8, light_sample_n=1, seed=0, estimator=ESTIMATOR_COMPAT):
        self.L = load_library()
        self.scene = scene
        self.width, self.height = int(width), int(height)
        self.devices = [int(d) for d in devices]
        self.h = C.c_void_p()
        arr = (C.c_int * len(self.devices))(*self.devices)
        _prefer_bundled_nccl()
        _check(self.L.crt_group_create(scene.h, self.width, self.height, C.cast(arr, C.c_void_p), len(self.devices), C.byref(self.h)))
        self.set_params(spp, P_RR, light_sample_n, seed, estimator)

    def set_params(self, spp, P_RR, light_sample_n, seed=0, estimator=ESTIMATOR_COMPAT):
        self.spp = int(spp)
        _check(self.L.crt_group_set_params(self.h, int(spp), float(P_RR), int(light_sample_n), int(seed), int(estimator)))

    def run_view(self, eye_pos, inv_view_mat, fovY):
        eye = np.ascontiguousarray(eye_pos, np.float32)
        M = np.ascontiguousarray(inv_view_mat, np.float32).reshape(9)
        _check(self.L.crt_group_run_view(self.h, _p(eye), _p(M), float(fovY)))

    def get_accum_i64(self):
        out = np.zeros(self.width * self.height * 3, np.int64)
        _check(self.L.crt_group_get_accum_i64(self.h, _p(out)))
        return out

    def get_frame_buffer(self):
        out = np.zeros((self.height, self.width, 3), np.uint8)
        _check(self.L.crt_group_get_rgb8(self.h, _p(out)))
        return out

    def save_frame_buffer(self, path):
        _check(self.L.crt_group_save_png(self.h, os.fsencode(path)))

    def set_aov(self, on):
        _check(self.L.crt_group_set_aov(self.h, 1 if on else 0))

    def get_aov(self):
        return _aov_images(self.L.crt_group_get_aov, self.h, self.width, self.height)

    def get_aov_i64(self):
        return _aov_i64(self.L.crt_group_get_aov_i64, self.h, self.width, self.height)

    def stats(self, index=0):
        st, ms = _Stats(), C.c_float()
        _check(self.L.crt_group_get_stats(self.h, int(index), C.byref(st), C.byref(ms)))
        d = {k: getattr(st, k) for k, _ in _Stats._fields_}
        d["reduce_ms"] = ms.value
        return d

    def close(self):
        if self.h:
            self.L.crt_group_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
