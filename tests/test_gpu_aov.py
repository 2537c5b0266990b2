"""AOV buffers for denoisers (include/crt.h crt_render_set_aov, DESIGN.md "AOV buffers").

For every work item, the camera ray k_generate makes (same Philox jitter, same float arithmetic) is traced closest-hit and adds
fixed-point albedo, face normal, depth / depth_unit and coverage to an int64 buffer of 8 values per pixel. The raw buffer must
equal the CPU statement of that rule (tests/aov_reference.py: the oracle's camera ray and traversal) exactly, for every builder and estimator and for any chunking of the work range or
number of GPUs; turning AOVs on must leave the colour bit-identical."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

import aov_reference
from conftest import ROOT

pytestmark = pytest.mark.gpu

STATE = -5
W, H = 200, 150


@pytest.fixture(scope="module")
def gpu(crt):
    if crt.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback and these tests need the B200")
    return crt


def _scene(gpu, files, builder=3):
    cfg = gpu.load_config(files["cfg_path"])
    S = gpu.Scene().add_obj(files["obj"], files["dir"])
    S.set_BVH(cfg.bvh_thresh_n, builder=builder, device=0)
    return cfg, S, gpu.inverse_view_matrix(cfg.eye_pos, cfg.lookat, cfg.up)


def _render(gpu, cfg, S, spp, est=0, seed=0, aov=True, w=W, h=H):
    R = gpu.Render(S, w, h, spp, cfg.P_RR, cfg.light_sample_n)
    R.set_estimator(est)
    R.set_seed(seed)
    R.set_aov(aov)
    return R


def depth_unit(bounds, eye):
    """Smallest power of two >= the largest eye-to-corner distance of the bounds (float64 from float32 inputs), 1 for 0."""
    b = np.asarray(bounds, np.float32).astype(np.float64)
    e = np.asarray(eye, np.float32).astype(np.float64)
    corners = np.array([[b[3 * ((c >> a) & 1) + a] for a in range(3)] for c in range(8)])
    d = corners - e
    far = np.sqrt(((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]).max())
    if far == 0:
        return 1.0
    m, ex = np.frexp(far)
    return float(np.ldexp(1.0, int(ex) - 1 if m == 0.5 else int(ex)))


def resolve(raw, spp, unit, w=W, h=H):
    """numpy statement of the resolve rule; images top row first."""
    a = raw.reshape(h, w, 8)
    mean = lambda x: (x.astype(np.float64) / 4294967296.0 / float(spp)).astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        depth = (a[..., 6].astype(np.float64) / a[..., 7].astype(np.float64) * float(unit)).astype(np.float32)
    depth[a[..., 7] == 0] = np.inf
    return dict(albedo=mean(a[..., 0:3]), normal=mean(a[..., 3:6]), depth=depth, coverage=mean(a[..., 7]))


def _same_aov(x, y):
    for k in ("albedo", "normal", "depth", "coverage"):
        assert np.array_equal(x[k], y[k]), k


_ORC = {}


def _oracle(orc, files, name, thresh, builder):
    key = (name, builder)
    if key not in _ORC:
        o = orc.Scene().add_obj(files["obj"], files["dir"])
        o.build_new_bvh(thresh, builder & 2)
        if builder & 1:
            o.build_wide8(thresh, builder)
        _ORC[key] = o
    return _ORC[key]


@pytest.mark.parametrize("builder", [0, 1, 2, 3])
@pytest.mark.parametrize("seed", [0, 7])
@pytest.mark.parametrize("name", ["cornell-box", "veach-mis"])
def test_aov_equals_the_oracle(gpu, orc, scene_files, name, seed, builder):
    spp = 3
    cfg, S, M = _scene(gpu, scene_files[name], builder)
    bounds = S.export_bvh()[3]
    want_unit = depth_unit(bounds, cfg.eye_pos)
    o = _oracle(orc, scene_files[name], name, cfg.bvh_thresh_n, builder)
    want = aov_reference.aov(orc, o, cfg.eye_pos, M, cfg.fovy_rad, W, H, 0, W * H * spp, seed, want_unit, wide=bool(builder & 1))
    assert (want.reshape(-1, 8)[:, 7] > 0).any()
    for est in (0, 1):
        R = _render(gpu, cfg, S, spp, est, seed)
        R.run_view(cfg.eye_pos, M, cfg.fovy_rad)
        raw, unit = R.get_aov_i64()
        assert unit == want_unit
        assert np.array_equal(raw, want), "%d of %d values differ" % (int((raw != want).sum()), raw.size)


@pytest.mark.parametrize("est", [0, 1])
def test_aov_leaves_the_colour_untouched(gpu, scene_files, est):
    cfg, S, M = _scene(gpu, scene_files["veach-mis"])
    out = {}
    for aov in (False, True):
        R = _render(gpu, cfg, S, 4, est, aov=aov)
        R.run_view(cfg.eye_pos, M, cfg.fovy_rad)
        out[aov] = (R.get_accum_i64(), R.get_frame_buffer(), R.stats())
    assert np.array_equal(out[False][0], out[True][0])
    assert np.array_equal(out[False][1], out[True][1])
    for k in ("samples", "extend_rays", "shadow_rays", "probe_rays"):
        assert out[False][2][k] == out[True][2][k], k
    # one AOV launch (below 2^31 work items) on top of whole wavefront iterations of 6 launches (7 with SPECULAR probes); how many
    # iterations the host enqueues after the last one depends on when it notices the end of the frame
    off, on = out[False][2]["kernel_launches"], out[True][2]["kernel_launches"]
    assert any(off % k == 0 and on % k == 1 for k in (6, 7)), (off, on)


def test_aov_work_ranges_sum_to_the_one_shot_buffer(gpu, scene_files):
    spp = 3
    cfg, S, M = _scene(gpu, scene_files["cornell-box"])
    total = W * H * spp
    R = _render(gpu, cfg, S, spp)
    R.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    one, unit = R.get_aov_i64()
    # progressive chunks, two of them ending inside a sample
    P = _render(gpu, cfg, S, spp)
    P.set_accumulate(True)
    P.clear_accum()
    cuts = [0, 17000, 45111, W * H * 2, total]
    for a, b in zip(cuts, cuts[1:]):
        P.set_work_range(a, b)
        P.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    assert np.array_equal(P.get_aov_i64()[0], one)
    assert np.array_equal(P.get_accum_i64(), R.get_accum_i64())
    # while the accumulation holds work, AOVs cannot be switched; after a clear they can
    for on in (False, True):
        with pytest.raises(gpu.CrtError) as e:
            P.set_aov(on)
        assert e.value.code == STATE
    P.clear_accum()
    P.set_aov(False)
    # sample-range shards
    acc = np.zeros_like(one)
    for s0, s1 in ((0, 1), (1, 3)):
        Q = _render(gpu, cfg, S, spp)
        Q.set_sample_range(s0, s1)
        Q.run_view(cfg.eye_pos, M, cfg.fovy_rad)
        acc += Q.get_aov_i64()[0]
    assert np.array_equal(acc, one)


def test_aov_get_before_a_run_is_a_state_error(gpu, scene_files):
    cfg, S, M = _scene(gpu, scene_files["cornell-box"])
    R = _render(gpu, cfg, S, 1, aov=False)
    R.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    for fn in (R.get_aov, R.get_aov_i64, R.device_aov_ptr):
        with pytest.raises(gpu.CrtError) as e:
            fn()
        assert e.value.code == STATE
    R.set_aov(True)
    with pytest.raises(gpu.CrtError) as e:
        R.get_aov()
    assert e.value.code == STATE
    R.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    R.get_aov()
    R.set_aov(False)
    R.run_view(cfg.eye_pos, M, cfg.fovy_rad)                          # the colour now has samples the AOV buffer lacks
    with pytest.raises(gpu.CrtError) as e:
        R.get_aov_i64()
    assert e.value.code == STATE


@pytest.mark.parametrize("name", ["cornell-box", "veach-mis"])
def test_aov_resolve(gpu, scene_files, name):
    spp = 5
    cfg, S, M = _scene(gpu, scene_files[name])
    R = _render(gpu, cfg, S, spp)
    R.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    raw, unit = R.get_aov_i64()
    got = R.get_aov()
    _same_aov(got, resolve(raw, spp, unit))
    cov = got["coverage"]
    assert cov.min() >= 0 and cov.max() <= 1
    assert np.all(np.isinf(got["depth"][cov == 0])) and np.all(np.isfinite(got["depth"][cov > 0]))
    if name == "cornell-box":
        # fully covered pixels whose samples all hit faces of one orientation (the walls): unit-length normals
        normals = np.unique(np.round(S.tris()["normal"], 6), axis=0)
        n = got["normal"][cov == 1]
        on_wall = (np.abs(n[:, None, :] - normals[None, :, :]).max(axis=2) < 1e-5).any(axis=1)
        assert on_wall.mean() > 0.5
        assert np.allclose(np.linalg.norm(n[on_wall], axis=1), 1.0, atol=1e-5)


@pytest.mark.parametrize("n_gpus", [1, 2, 4, 8])
def test_group_aov_equals_the_single_gpu_aov(gpu, scene_files, n_gpus):
    if gpu.device_count() < n_gpus:
        pytest.skip("needs %d GPUs" % n_gpus)
    cfg, S, M = _scene(gpu, scene_files["veach-mis"])
    for spp in (5, 3):
        R = _render(gpu, cfg, S, spp)
        R.run_view(cfg.eye_pos, M, cfg.fovy_rad)
        want, want_unit = R.get_aov_i64()
        G = gpu.RenderGroup(S, W, H, list(range(n_gpus)), spp, cfg.P_RR, cfg.light_sample_n, 0, 0)
        with pytest.raises(gpu.CrtError) as e:
            G.get_aov()
        assert e.value.code == STATE
        G.set_aov(True)
        for _ in range(2):
            G.run_view(cfg.eye_pos, M, cfg.fovy_rad)
            raw, unit = G.get_aov_i64()
            assert unit == want_unit and np.array_equal(raw, want)
            _same_aov(G.get_aov(), R.get_aov())
            assert np.array_equal(G.get_accum_i64(), R.get_accum_i64())
        G.close()


def test_aov_checkpoints(gpu, scene_files, tmp_path):
    spp = 4
    cfg, S, M = _scene(gpu, scene_files["veach-mis"])
    total = W * H * spp
    R = _render(gpu, cfg, S, spp)
    R.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    one, accum = R.get_aov_i64()[0], R.get_accum_i64()

    A = _render(gpu, cfg, S, spp)
    A.set_accumulate(True)
    A.clear_accum()
    A.set_work_range(0, 50000)
    A.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    on_file = str(tmp_path / "on.ckpt")
    A.save_checkpoint(on_file, 50000)
    B = _render(gpu, cfg, S, spp)
    done, eye, MM, fov = B.load_checkpoint(on_file)
    assert done == 50000
    B.set_work_range(done, total)
    B.run_view(eye, MM, fov)
    assert np.array_equal(B.get_aov_i64()[0], one)
    assert np.array_equal(B.get_accum_i64(), accum)

    off = _render(gpu, cfg, S, spp, aov=False)
    with pytest.raises(gpu.CrtError) as e:
        off.load_checkpoint(on_file)
    assert e.value.code == STATE

    C = _render(gpu, cfg, S, spp, aov=False)
    C.set_accumulate(True)
    C.clear_accum()
    C.set_work_range(0, 50000)
    C.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    off_file = str(tmp_path / "off.ckpt")
    C.save_checkpoint(off_file, 50000)
    header = 120                                                      # sizeof(CheckpointHeader), unchanged by AOVs
    assert os.path.getsize(off_file) == header + W * H * 24
    assert os.path.getsize(on_file) == header + W * H * (24 + 64)
    with open(off_file, "rb") as f:
        assert struct.unpack_from("<I", f.read(header), 100)[0] == 0  # the AOV flag (pad word)
    D = _render(gpu, cfg, S, spp, aov=True)
    with pytest.raises(gpu.CrtError) as e:
        D.load_checkpoint(off_file)
    assert e.value.code == STATE


def _read_pfm(path):
    with open(path, "rb") as f:
        kind = f.readline().strip()
        w, h = map(int, f.readline().split())
        scale = float(f.readline())
        assert scale < 0                                               # little endian
        ch = 3 if kind == b"PF" else 1
        assert kind in (b"PF", b"Pf")
        data = np.frombuffer(f.read(), "<f4")
    assert data.size == w * h * ch
    img = data.reshape((h, w, ch) if ch == 3 else (h, w))
    return img[::-1]                                                   # PFM rows go bottom first


def test_cli_writes_the_aov_pfms(gpu, scene_files, tmp_path):
    exe = os.path.join(ROOT, "cudaraytracing_b200", "crt")
    files = scene_files["cornell-box"]
    w, h, spp = 160, 120, 4
    base = [exe, "--config", files["cfg_path"], "--width", str(w), "--height", str(h), "--spp", str(spp)]
    r = subprocess.run(base + ["--out", str(tmp_path / "a.png"), "--aov", str(tmp_path / "a")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    cfg, S, M = _scene(gpu, files, builder=3)                        # the CLI's default builder (ploc8)
    R = gpu.Render(S, w, h, spp, cfg.P_RR, cfg.light_sample_n)
    R.set_seed(cfg.seed)
    R.set_estimator(cfg.estimator)
    R.set_aov(True)
    R.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    want = R.get_aov()
    for k in ("albedo", "normal", "depth"):
        assert np.array_equal(_read_pfm(str(tmp_path / ("a_%s.pfm" % k))), want[k]), k
    # progressive with a checkpoint: the same files
    ck = str(tmp_path / "c.ckpt")
    r = subprocess.run(base + ["--out", str(tmp_path / "c.png"), "--aov", str(tmp_path / "c"), "--checkpoint", ck, "--chunk-spp", "1"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    for k in ("albedo", "normal", "depth"):
        assert open(str(tmp_path / ("a_%s.pfm" % k)), "rb").read() == open(str(tmp_path / ("c_%s.pfm" % k)), "rb").read(), k
    if gpu.device_count() >= 2:
        r = subprocess.run(base + ["--out", str(tmp_path / "g.png"), "--aov", str(tmp_path / "g"), "--gpus", "2"], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert json.loads(r.stdout.strip().splitlines()[-1])["gpus"] == 2
        for k in ("albedo", "normal", "depth"):
            assert open(str(tmp_path / ("a_%s.pfm" % k)), "rb").read() == open(str(tmp_path / ("g_%s.pfm" % k)), "rb").read(), k


def test_device_aov_pointer_and_caller_side_sum(gpu, scene_files):
    import torch

    from cudaraytracing_b200 import distributed
    spp = 3
    cfg, S, M = _scene(gpu, scene_files["cornell-box"])
    R = _render(gpu, cfg, S, spp)
    R.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    raw, _ = R.get_aov_i64()
    t = distributed.aov_as_tensor(R, "cuda:0")
    assert t.dtype == torch.int64 and t.numel() == W * H * 8
    assert np.array_equal(t.cpu().numpy(), raw)
    # two shards summed by the caller into the first one's buffer: its get_aov resolves the sum
    A, B = _render(gpu, cfg, S, spp), _render(gpu, cfg, S, spp)
    A.set_sample_range(0, 2)
    B.set_sample_range(2, 3)
    A.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    B.run_view(cfg.eye_pos, M, cfg.fovy_rad)
    ta = distributed.aov_as_tensor(A, "cuda:0")
    ta += distributed.aov_as_tensor(B, "cuda:0")
    torch.cuda.synchronize()
    _same_aov(A.get_aov(), R.get_aov())
