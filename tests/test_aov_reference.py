"""The CPU statement of the AOV buffer (tests/aov_reference.py, DESIGN.md "AOV buffers"), checked on its own: integer sums,
so any split of the work range adds up to the whole; the pair and 8-wide traversals give the same buffer; the camera rays are
the oracle's primary_ray with the render's Philox jitter; every hit adds coverage 2^32 and a depth in (0, 2^32], a pixel no
sample hits stays zero."""
import math

import numpy as np

import aov_reference


def test_aov_reference_chunks_layouts_and_rays(orc, scene_files):
    files = scene_files["cornell-box"]
    o = orc.Scene().add_obj(files["obj"], files["dir"])
    o.build_new_bvh(2)
    o.build_wide8(2, 1)
    eye = np.array([278, 273, -800], np.float32)
    M = orc.inverse_view_matrix(eye, np.array([278, 273, -799], np.float32), np.array([0, 1, 0], np.float32))
    fovy = np.float32(math.radians(39.3077))
    w, h, spp, unit, seed = 40, 30, 3, 2048.0, 5
    total = w * h * spp
    one = aov_reference.aov(orc, o, eye, M, fovy, w, h, 0, total, seed, unit)
    assert np.array_equal(aov_reference.aov(orc, o, eye, M, fovy, w, h, 0, total, seed, unit, wide=True), one)
    acc = np.zeros_like(one)
    for a, b in ((0, 777), (777, 2500), (2500, total)):
        aov_reference.aov(orc, o, eye, M, fovy, w, h, a, b, seed, unit, out=acc)
    assert np.array_equal(acc, one)
    px = one.reshape(-1, 8)
    assert px[:, 7].max() == spp * 2 ** 32 and (px[:, 7] % 2 ** 32 == 0).all()
    assert (px[:, 6] <= px[:, 7]).all() and (px[px[:, 7] > 0, 6] > 0).all()
    assert (px[px[:, 7] == 0] == 0).all()
    # the rays start at the eye, are unit length, and differ from the pixel-centre rays only by the jitter
    rays, pixel = aov_reference.camera_rays(orc, eye, M, fovy, w, h, 0, w * h, seed)
    assert np.array_equal(pixel, np.arange(w * h))
    assert np.all(rays[:, 0:3] == eye) and np.allclose(np.linalg.norm(rays[:, 4:7], axis=1), 1.0, atol=1e-6)
    centre = orc.primary_rays(eye, M, fovy, w, h).reshape(-1, 8)
    assert not np.array_equal(rays[:, 4:7], centre[:, 4:7])
    assert np.abs(rays[:, 4:7] - centre[:, 4:7]).max() < 2 * math.tan(fovy / 2) / h
    # quantize rounds to nearest even and drops what the device drops
    q = aov_reference.quantize(np.array([0.5, -1.0, 2.0 ** -33, 3.0 * 2.0 ** -33, np.inf, np.nan, 2.0 ** 30], np.float32))
    assert q.tolist() == [2 ** 31, -2 ** 32, 0, 2, 0, 0, 0]
