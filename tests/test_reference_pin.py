"""Pins the oracle's restatement against the REAL reference code (oracle/_ref/libref.so = the reference's
own headers compiled in place). The tests marked `reference` need the reference's checkout and run only where it is present;
the others compare the product and the oracle with stored values of the same quantities: tests/golden/golden.json (digests
and scene settings taken from the reference's own code and files, tools/make_golden.py) and tests/golden/host_record.json
(the oracle's values of what golden.json does not hold, tools/make_host_record.py)."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, REFERENCE


@pytest.fixture(scope="module")
def ref():
    so = os.path.join(ROOT, "oracle", "_ref", "libref.so")
    if not os.path.exists(so):
        import subprocess
        subprocess.check_call(["bash", os.path.join(ROOT, "oracle", "ref_harness", "build.sh")])
    R = C.CDLL(so)
    R.ref_host_load.restype = C.c_void_p
    R.ref_host_load.argtypes = [C.c_char_p, C.c_char_p, C.c_uint, C.c_uint, C.c_uint]
    for f in ("ref_n_tris", "ref_n_nodes", "ref_root", "ref_n_lights"):
        getattr(R, f).argtypes = [C.c_void_p]
    R.ref_get_tris.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    R.ref_get_nodes.argtypes = [C.c_void_p, C.c_void_p]
    R.ref_get_light.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    R.ref_inverse_view.argtypes = [C.c_void_p] * 4
    return R


@pytest.mark.reference
@pytest.mark.parametrize("name,thresh", [("veach-mis", 2), ("veach-mis", 5), ("cornell-box", 2)])
def test_oracle_equals_real_reference_host_path(ref, orc, crt, name, thresh):
    d = "%s/scenes/%s/" % (REFERENCE, name)
    h = ref.ref_host_load((d + name + ".obj").encode(), d.encode(), 800, 600, thresh)
    n, nn = ref.ref_n_tris(h), ref.ref_n_nodes(h)
    t0 = np.zeros((n, 23), np.float32); ref.ref_get_tris(h, 0, t0.ctypes.data_as(C.c_void_p))
    t1 = np.zeros((n, 23), np.float32); ref.ref_get_tris(h, 1, t1.ctypes.data_as(C.c_void_p))
    nodes = np.zeros(nn, orc.REF_NODE); ref.ref_get_nodes(h, nodes.ctypes.data_as(C.c_void_p))
    for S in (orc.Scene().add_obj(d + name + ".obj", d), crt.Scene().add_obj(d + name + ".obj", d)):
        tr, mats = S.tris(), S.mats()
        bits = lambda a: np.ascontiguousarray(a).view(np.uint32)
        assert np.array_equal(bits(tr["verts"]), bits(t0[:, 0:9]))
        assert np.array_equal(bits(tr["normal"]), bits(t0[:, 9:12]))
        assert np.array_equal(bits(tr["area"]), bits(t0[:, 12]))
        assert np.array_equal(bits(tr["area_of_obj"]), bits(t0[:, 13]))
        m = mats[tr["mat"]]
        assert np.array_equal(m[:, 0:3], t0[:, 14:17]) and np.array_equal(m[:, 3:6], t0[:, 17:20])
        assert np.array_equal(m[:, 6], t0[:, 20]) and np.array_equal(m[:, 7], t0[:, 21]) and np.array_equal(m[:, 8], t0[:, 22])
        for li, (faces, area) in enumerate(S.lights()):
            nt, ar = C.c_int(), C.c_float()
            ref.ref_get_light(h, li, C.byref(nt), C.byref(ar))
            assert nt.value == len(faces) and np.float32(ar.value) == np.float32(area)
    S = orc.Scene().add_obj(d + name + ".obj", d)
    mynodes, order, root = S.build_ref_bvh(thresh)
    assert root == ref.ref_root(h) and mynodes.tobytes() == nodes.tobytes()          # BVH.h:37-84, byte for byte
    assert np.array_equal(S.tris()["verts"][order].view(np.uint32), np.ascontiguousarray(t1[:, 0:9]).view(np.uint32))


@pytest.mark.reference
def test_camera_matrix_equals_reference(ref, orc, crt):
    for eye, look, up in ([[278, 273, -800], [278, 273, -799], [0, 1, 0]], [[28.2792, 5.2, 1.23612e-06], [0, 2.8, 0], [0, 1, 0]]):
        e, l, u = (np.asarray(x, np.float32) for x in (eye, look, up))
        out = np.zeros(9, np.float32)
        ref.ref_inverse_view(*(a.ctypes.data_as(C.c_void_p) for a in (e, l, u, out)))
        assert np.array_equal(out, orc.inverse_view_matrix(eye, look, up))
        assert np.array_equal(out, crt.inverse_view_matrix(eye, look, up))


@pytest.mark.reference
def test_fixture_equals_reference_scene_files(crt, scene_files):
    for name in ("cornell-box", "veach-mis"):
        d = "%s/scenes/%s/" % (REFERENCE, name)
        a = crt.Scene().add_obj(d + name + ".obj", d)
        b = crt.Scene().add_obj(scene_files[name]["obj"], scene_files[name]["dir"])
        ta, tb = a.tris(), b.tris()
        for k in ta:
            assert np.array_equal(ta[k].view(np.uint32), tb[k].view(np.uint32)), k
        assert np.array_equal(a.mats(), b.mats())
        ca, cb = crt.load_config(d + "config.json"), crt.load_config(scene_files[name]["cfg_path"])
        for k in ("fov_y", "width", "height", "bvh_thresh_n", "P_RR", "spp", "light_sample_n"):
            assert getattr(ca, k) == getattr(cb, k)
        assert np.array_equal(ca.eye_pos, cb.eye_pos) and np.array_equal(ca.lookat, cb.lookat)


def _stored(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("name,thresh", [("veach-mis", 2), ("veach-mis", 5), ("cornell-box", 2)])
def test_host_path_equals_stored_values(orc, crt, scene_files, name, thresh):
    """What test_oracle_equals_real_reference_host_path compares, for the oracle and the product, on the stored fixtures."""
    g, r = _stored("golden.json")[name], _stored("host_record.json")[name]
    f = scene_files[name]
    for S in (orc.Scene().add_obj(f["obj"], f["dir"]), crt.Scene().add_obj(f["obj"], f["dir"])):
        tr, mats = S.tris(), S.mats()
        assert len(tr["verts"]) == g["n_tris"]
        assert _sha(tr["verts"]) == g["ref_verts_sha256"] and _sha(tr["normal"]) == g["ref_normal_sha256"]
        assert _sha(tr["area"]) == g["ref_area_sha256"] and _sha(tr["area_of_obj"]) == r["area_of_obj_sha256"]
        assert _sha(mats[tr["mat"]].astype(np.float32)) == r["tri_mats_sha256"]
        lights = S.lights()
        assert [len(faces) for faces, _ in lights] == g["light_sizes"] == r["light_tris"]
        assert [float(np.float32(area)) for _, area in lights] == g["light_areas"]
    S = orc.Scene().add_obj(f["obj"], f["dir"])
    nodes, order, root = S.build_ref_bvh(thresh)
    b = r["ref_bvh"][str(thresh)]
    assert len(nodes) == b["n_nodes"] and root == b["root"] and _sha(nodes) == b["nodes_sha256"]
    assert _sha(S.tris()["verts"][order]) == b["sorted_verts_sha256"]
    if thresh == g["thresh_n"]:
        assert _sha(nodes) == g["ref_nodes_sha256"] and root == g["ref_root"] and len(nodes) == g["ref_n_nodes"]
        assert _sha(S.tris()["verts"][order]) == g["ref_sorted_verts_sha256"]


def test_camera_matrix_equals_stored_values(orc, crt):
    """The cameras of test_camera_matrix_equals_reference, bit for bit."""
    for c in _stored("host_record.json")["cameras"]:
        want = np.array(c["inverse_view_f32_bits"], np.uint32)
        assert np.array_equal(orc.inverse_view_matrix(c["eye"], c["lookat"], c["up"]).view(np.uint32), want)
        assert np.array_equal(crt.inverse_view_matrix(c["eye"], c["lookat"], c["up"]).view(np.uint32), want)


def test_fixture_equals_stored_reference_values(crt, scene_files):
    """The stored fixtures against the reference scene files' values kept in golden.json: triangles (digests of the reference
    loader's output) and the config.json settings."""
    g = _stored("golden.json")
    for name in ("cornell-box", "veach-mis"):
        tr = crt.Scene().add_obj(scene_files[name]["obj"], scene_files[name]["dir"]).tris()
        assert _sha(tr["verts"]) == g[name]["ref_verts_sha256"] and _sha(tr["normal"]) == g[name]["ref_normal_sha256"]
        c, cam = crt.load_config(scene_files[name]["cfg_path"]), g[name]["camera"]
        for k, v in (("eye_pos", "eye"), ("lookat", "lookat"), ("up", "up")):
            assert np.array_equal(getattr(c, k), np.asarray(cam[v], np.float32)), k
        assert np.float32(c.fov_y) == np.float32(cam["fov_y"]) and np.float32(c.P_RR) == np.float32(cam["P_RR"])
        assert (c.spp, c.light_sample_n, c.bvh_thresh_n) == (cam["spp"], cam["light_sample_n"], g[name]["thresh_n"])
