"""Every handle releases what it creates: device memory, pinned host memory, events and streams.

A small interposer, preloaded into a subprocess, wraps the CUDA runtime calls that create and destroy those resources (it
forwards every call unchanged) and keeps the set of live handles. The subprocess drives every kind of handle through the
public API - scenes from all four builders, a rebuild, ray batches of every kind, renders with stage timing and the launch
timeline, a one-GPU render group, the argument-error paths - destroys them all, and reports what is still alive. It does
not import torch, whose caching allocator keeps blocks of its own."""
import json
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

INTERPOSER = r"""
#include <dlfcn.h>
#include <pthread.h>
#include <set>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>

typedef int cudaError_t;
typedef struct CUevent_st* cudaEvent_t;
typedef struct CUstream_st* cudaStream_t;

static pthread_mutex_t g_mu = PTHREAD_MUTEX_INITIALIZER;
static std::set<void*>* g_live[4];            // device memory, pinned memory, events, streams
static long long g_bad_frees, g_created;

// The real function. libcudart is loaded by the library that calls us, without RTLD_GLOBAL (ctypes), so RTLD_NEXT would not
// see it: look it up in the loaded libcudart itself.
template <typename F> static F next(const char* name) {
    void* rt = dlopen("libcudart.so.12", RTLD_LAZY | RTLD_NOLOAD);
    void* f = rt ? dlsym(rt, name) : nullptr;
    if (!f) { fprintf(stderr, "lifecycle interposer: no %s in a loaded libcudart.so.12\n", name); abort(); }
    return (F)f;
}
static void track(int kind, void* p) {
    if (!p) return;
    pthread_mutex_lock(&g_mu);
    if (!g_live[kind]) g_live[kind] = new std::set<void*>();
    g_live[kind]->insert(p);
    ++g_created;
    pthread_mutex_unlock(&g_mu);
}
static void untrack(int kind, void* p) {
    if (!p) return;
    pthread_mutex_lock(&g_mu);
    if (!g_live[kind] || g_live[kind]->erase(p) == 0) ++g_bad_frees;
    pthread_mutex_unlock(&g_mu);
}

extern "C" {
cudaError_t cudaMalloc(void** p, size_t n) {
    cudaError_t e = next<cudaError_t (*)(void**, size_t)>("cudaMalloc")(p, n);
    if (e == 0) track(0, *p);
    return e;
}
cudaError_t cudaFree(void* p) {
    untrack(0, p);
    return next<cudaError_t (*)(void*)>("cudaFree")(p);
}
cudaError_t cudaHostAlloc(void** p, size_t n, unsigned flags) {
    cudaError_t e = next<cudaError_t (*)(void**, size_t, unsigned)>("cudaHostAlloc")(p, n, flags);
    if (e == 0) track(1, *p);
    return e;
}
cudaError_t cudaFreeHost(void* p) {
    untrack(1, p);
    return next<cudaError_t (*)(void*)>("cudaFreeHost")(p);
}
cudaError_t cudaEventCreate(cudaEvent_t* ev) {
    cudaError_t e = next<cudaError_t (*)(cudaEvent_t*)>("cudaEventCreate")(ev);
    if (e == 0) track(2, *ev);
    return e;
}
cudaError_t cudaEventCreateWithFlags(cudaEvent_t* ev, unsigned flags) {
    cudaError_t e = next<cudaError_t (*)(cudaEvent_t*, unsigned)>("cudaEventCreateWithFlags")(ev, flags);
    if (e == 0) track(2, *ev);
    return e;
}
cudaError_t cudaEventDestroy(cudaEvent_t ev) {
    untrack(2, ev);
    return next<cudaError_t (*)(cudaEvent_t)>("cudaEventDestroy")(ev);
}
cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned flags) {
    cudaError_t e = next<cudaError_t (*)(cudaStream_t*, unsigned)>("cudaStreamCreateWithFlags")(s, flags);
    if (e == 0) track(3, *s);
    return e;
}
cudaError_t cudaStreamDestroy(cudaStream_t s) {
    untrack(3, s);
    return next<cudaError_t (*)(cudaStream_t)>("cudaStreamDestroy")(s);
}
// live device blocks, pinned blocks, events, streams, bad frees, handles created in all
void lifecycle_counts(long long* out) {
    pthread_mutex_lock(&g_mu);
    for (int k = 0; k < 4; ++k) out[k] = g_live[k] ? (long long)g_live[k]->size() : 0;
    out[4] = g_bad_frees;
    out[5] = g_created;
    pthread_mutex_unlock(&g_mu);
}
}
"""

SCRIPT = textwrap.dedent(r"""
    import ctypes as C, json, os, sys
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import BOX_CAMERA, box_scene, random_rays
    import cudaraytracing_b200.api as crt

    rng = np.random.default_rng(7)
    verts, mat, obj, mats = box_scene(rng, n_soup=300)
    scenes = []
    for builder in (crt.BUILDER_LBVH, crt.BUILDER_LBVH8, crt.BUILDER_PLOC, crt.BUILDER_PLOC8):
        s = crt.Scene().add_triangles(verts, mat, obj, mats)
        s.set_BVH(2, builder=builder)
        scenes.append(s)
    scenes[0].set_BVH(2, builder=crt.BUILDER_PLOC8)          # rebuilt in place

    cudart = C.CDLL("libcudart.so.12")
    n = 5000
    rays = random_rays(rng, [0.5] * 3, [9.5] * 3, n, tmax_any=True)
    d_rays, d_t, d_face = C.c_void_p(), C.c_void_p(), C.c_void_p()
    for p, size in ((d_rays, rays.nbytes), (d_t, 4 * n), (d_face, 4 * n)):
        assert cudart.cudaMalloc(C.byref(p), C.c_size_t(size)) == 0
    assert cudart.cudaMemcpy(d_rays, rays.ctypes.data_as(C.c_void_p), C.c_size_t(rays.nbytes), 1) == 0
    for s in scenes:
        for mode in (crt.RAY_CLOSEST, crt.RAY_ANY, crt.RAY_CLOSEST | crt.RAY_SORTED, crt.RAY_ANY | crt.RAY_SORTED):
            s.trace_rays(rays, mode)
            s.trace_rays_device(d_rays, n, mode, d_t, d_face)
            assert cudart.cudaDeviceSynchronize() == 0
    for p in (d_rays, d_t, d_face):
        assert cudart.cudaFree(p) == 0

    cam = BOX_CAMERA
    M = crt.inverse_view_matrix(cam["eye"], cam["lookat"], cam["up"])
    for s in scenes[:2]:
        R = crt.Render(s, 64, 48, spp=2)
        R.set_stage_timing(1)
        R.run_view(cam["eye"], M, cam["fovy"])
        R.set_stage_timing(0)
        os.environ["CRT_TIMELINE"] = "1"
        R.run_view(cam["eye"], M, cam["fovy"])
        del os.environ["CRT_TIMELINE"]
        R.get_frame_buffer()
        R.close()

    G = crt.RenderGroup(scenes[1], 64, 48, [0], spp=2)
    G.run_view(cam["eye"], M, cam["fovy"])
    G.get_frame_buffer()
    G.close()

    # the argument-error paths of test_error_paths_on_gpu
    s = crt.Scene().add_triangles([[0, 0, 0, 1, 0, 0, 0, 1, 0]], [0], [0], [[.5, .5, .5, 0, 0, 0, 1]])
    for f in (lambda: crt.Render(s, 8, 8), lambda: s.set_BVH(2, device=99)):
        try:
            f()
            raise AssertionError("expected an error")
        except crt.CrtError:
            pass
    s.set_BVH(2)
    R = crt.Render(s, 8, 8)
    for f in (lambda: R.set_P_RR(1.5), lambda: R.set_estimator(7)):
        try:
            f()
            raise AssertionError("expected an error")
        except crt.CrtError:
            pass
    R.run_view([0.2, 0.2, -1], np.eye(3, dtype=np.float32).reshape(9), 0.5)
    e0 = crt.Scene()
    e0.set_BVH(2)
    R0 = crt.Render(e0, 4, 4)
    R0.run_view([0, 0, 0], np.eye(3, dtype=np.float32).reshape(9), 0.5)
    for h in (R0, e0, R, s, *scenes):
        h.close()

    out = (C.c_longlong * 6)()
    C.CDLL(None).lifecycle_counts(out)
    print("COUNTS " + json.dumps(dict(zip(["device", "pinned", "events", "streams", "bad_frees", "created"], list(out)))))
""")


@pytest.mark.gpu
def test_handles_release_everything_they_create(crt, tmp_path):
    so = str(tmp_path / "liblifecycle.so")
    src = tmp_path / "lifecycle.cpp"
    src.write_text(INTERPOSER)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", "-o", so, str(src), "-ldl", "-lpthread"])
    env = dict(os.environ, LD_PRELOAD=so, PYTHONPATH=ROOT, CRT_LIB=crt.lib_path())
    env.pop("CRT_TIMELINE", None)
    r = subprocess.run([sys.executable, "-c", "ROOT = %r\n" % ROOT + SCRIPT], env=env, cwd=str(tmp_path), capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("COUNTS ")]
    assert line, r.stdout[-4000:]
    counts = json.loads(line[-1][len("COUNTS "):])
    assert counts.pop("created") > 100, "the interposer saw none of the library's calls"
    assert counts == dict(device=0, pinned=0, events=0, streams=0, bad_frees=0), counts
