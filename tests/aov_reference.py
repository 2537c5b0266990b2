"""CPU statement of the AOV buffer (DESIGN.md "AOV buffers"), independent of the product.

The camera ray of every work item comes from the oracle's primary_ray and Philox draw (tests/aov_camera_rays.cpp, compiled
here against oracle/liborc.so); the oracle's closest-hit traversal (pair nodes or 8-wide nodes) traces it; a hit on face f
adds quantize() of Kd of f's material, f's normal, min(t / depth_unit, 1) and 1 to aov[8 * pixel + 0..7]."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB = None


def _lib(orc):
    global _LIB
    if _LIB is None:
        orc.lib()                                                       # builds / loads oracle/liborc.so
        oracle = os.path.join(ROOT, "oracle")
        out = tempfile.mkdtemp(prefix="crt_aov_ref_")
        so = os.path.join(out, "libaov_camera_rays.so")
        cxx = shutil.which("/usr/bin/g++") or "g++"
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-mfma", "-shared", "-o", so,
                               os.path.join(ROOT, "tests", "aov_camera_rays.cpp"), "-L" + oracle, "-l:liborc.so",
                               "-Wl,-rpath," + oracle])
        L = C.CDLL(so)
        L.aov_camera_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_uint32,
                                      C.c_void_p, C.c_void_p]
        L.aov_camera_rays.restype = None
        _LIB = L
    return _LIB


def camera_rays(orc, eye, M, fovy_rad, width, height, w_begin, w_end, seed):
    """(rays n x 8 float32, pixel n int32) of work items [w_begin, w_end)."""
    n = int(w_end) - int(w_begin)
    rays = np.zeros((n, 8), np.float32)
    pixel = np.zeros(n, np.int32)
    e = np.ascontiguousarray(eye, np.float32)
    m = np.ascontiguousarray(M, np.float32).reshape(9)
    _lib(orc).aov_camera_rays(e.ctypes.data, m.ctypes.data, float(fovy_rad), width, height, int(w_begin), int(w_end), seed,
                              rays.ctypes.data, pixel.ctypes.data)
    return rays, pixel


def quantize(v):
    """value * 2^32 rounded to nearest even, as int64; non-finite or |v| >= 2^30 gives 0 (crt_device.cuh quantize)."""
    v = np.asarray(v, np.float32)
    ok = np.abs(v) < np.float32(1073741824.0)
    q = np.rint(np.where(ok, v, 0).astype(np.float64) * 4294967296.0).astype(np.int64)
    return np.where(ok, q, 0)


def aov(orc, oscene, eye, M, fovy_rad, width, height, w_begin, w_end, seed, depth_unit, wide=False, out=None):
    """int64[W*H*8] AOV buffer of work items [w_begin, w_end), added to `out` when given. oscene: an oracle Scene with the
    pair BVH built (and the 8-wide one for wide=True)."""
    if out is None:
        out = np.zeros(width * height * 8, np.int64)
    rays, pixel = camera_rays(orc, eye, M, fovy_rad, width, height, w_begin, w_end, seed)
    t, face = oscene.trace(rays, which=4 if wide else 0, mode=0)
    hit = face >= 0
    f, t, px = face[hit], t[hit], pixel[hit]
    tris, mats = oscene.tris(), oscene.mats()
    v = np.zeros((len(f), 8), np.float32)
    v[:, 0:3] = mats[tris["mat"][f], 0:3]
    v[:, 3:6] = tris["normal"][f]
    v[:, 6] = np.minimum(t / np.float32(depth_unit), np.float32(1.0))
    v[:, 7] = 1.0
    np.add.at(out.reshape(-1, 8), px, quantize(v))
    return out
