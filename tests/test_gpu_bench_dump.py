"""bench.py --dump-outputs on the GPU: the files hold what the timed path returned in its last step (checked against the same
computation through the public API), at the seeded sample's indices, and two runs with the same arguments write the same arrays."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _bench(tmp, tag, args, env=None):
    out = os.path.join(tmp, tag)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "1", "--warmup", "1", "--dump-outputs", out] + args
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=tmp, env=env, timeout=1200)
    assert r.returncode == 0, r.stderr[-3000:]
    files = sorted(os.listdir(out))
    assert sum(os.path.getsize(os.path.join(out, f)) for f in files) <= 64 * 10 ** 6
    d = {f[:-4]: np.load(os.path.join(out, f)) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    return d


def test_render_dump_is_the_last_step(crt, tmp_path, monkeypatch):
    """C3 (8.3 M pixels: a sampled dump) without the sub-measurements."""
    monkeypatch.delenv("CRT_BUILDER", raising=False)
    a = _bench(str(tmp_path), "a", ["--workload", "c3", "--no-sub"])
    b = _bench(str(tmp_path), "b", ["--workload", "c3", "--no-sub"])
    assert sorted(a) == ["accum", "frame", "pixel_index"]
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    w = bench.Workload("c3")
    npix = w.width * w.height
    idx = a["pixel_index"].astype(np.int64)
    assert np.array_equal(idx, bench.dump_sample_index(npix, 3 * 8 + 3 * 4 + 8)) and len(idx) < npix
    S, _ = w.build_scene(crt, 0)
    R = crt.Render(S, w.width, w.height, w.spp, w.P_RR, w.light_sample_n)
    R.set_seed(0)
    R.set_estimator(0)
    R.run_view(w.eye, crt.inverse_view_matrix(w.eye, w.lookat, w.up), w.fovy_rad)
    assert np.array_equal(a["accum"], R.get_accum_i64().reshape(npix, 3)[idx].astype(np.float64))
    assert np.array_equal(a["frame"], R.get_frame_buffer().reshape(npix, 3)[idx].astype(np.float32))


def test_ray_dump_is_the_last_step(crt, tmp_path, monkeypatch):
    """C5 on a small grid with 4 M rays (a sampled dump): closest hits exactly, any-hit as hit / miss (which blocker an
    any-hit ray reports depends on scheduling)."""
    import torch
    monkeypatch.delenv("CRT_BUILDER", raising=False)
    monkeypatch.setenv("CRT_C4_GRID", "257")
    monkeypatch.setenv("CRT_C5_RAYS", "4000000")
    monkeypatch.setenv("CRT_C5_E2E_RAYS", "100000")
    a = _bench(str(tmp_path), "a", ["--workload", "c5"], env=dict(os.environ))
    b = _bench(str(tmp_path), "b", ["--workload", "c5"], env=dict(os.environ))
    assert sorted(a) == ["any_face", "any_t", "closest_face", "closest_t", "ray_index"]
    for k in ("ray_index", "closest_t", "closest_face"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["any_face"] >= 0, b["any_face"] >= 0)
    n = 4000000
    idx = a["ray_index"].astype(np.int64)
    assert np.array_equal(idx, bench.dump_sample_index(n, 2 * (4 + 8) + 8)) and len(idx) < n
    w = bench.Workload("c5")
    S, _ = w.build_scene(crt, 0)
    dev = torch.device("cuda", 0)
    rays = torch.empty((n, 8), dtype=torch.float32, device=dev)
    t = torch.empty(n, dtype=torch.float32, device=dev)
    f = torch.empty(n, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    for mode, name in ((crt.RAY_CLOSEST, "closest"), (crt.RAY_ANY, "any")):
        S.random_rays_device(rays.data_ptr(), n, start=0, key=0xC5, any_hit=(mode == crt.RAY_ANY), stream=stream)
        S.trace_rays_device(rays.data_ptr(), n, mode, t.data_ptr(), f.data_ptr(), stream)
        torch.cuda.synchronize()
        tt, ff = t.cpu().numpy()[idx], f.cpu().numpy()[idx]
        if name == "closest":
            assert np.array_equal(a["closest_t"], tt) and np.array_equal(a["closest_face"], ff.astype(np.float64))
        else:
            assert np.array_equal(a["any_face"] >= 0, ff >= 0)
