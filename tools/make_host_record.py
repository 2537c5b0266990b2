"""Writes tests/golden/host_record.json: digests of the host-path quantities that tests/test_reference_pin.py compares with the
reference's own code and that golden.json does not hold (area_of_obj, the per-triangle material columns, the BVH at
bvh_thresh_n 5, the inverse view matrices). They are computed by the oracle (oracle/liborc.so) on the stored scene fixtures:
the oracle is the restatement that test_reference_pin pins byte for byte against the reference where its checkout is
present, and the record keeps the product and the oracle at those values where it is not.
Run:  python tools/make_host_record.py
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import orc  # noqa: E402
from tools import scene_fixture as sf  # noqa: E402

CAMERAS = ([[278, 273, -800], [278, 273, -799], [0, 1, 0]], [[28.2792, 5.2, 1.23612e-06], [0, 2.8, 0], [0, 1, 0]])
THRESH = {"cornell-box": (2,), "veach-mis": (2, 5)}


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def record():
    out = {"cameras": [{"eye": e, "lookat": l, "up": u, "inverse_view_f32_bits": [int(x) for x in orc.inverse_view_matrix(e, l, u).view(np.uint32)]}
                       for e, l, u in CAMERAS]}
    for name, threshes in THRESH.items():
        tmp = tempfile.mkdtemp(prefix="crt_record_")
        sf.unpack(sf.fixture(name), tmp)
        S = orc.Scene().add_obj(os.path.join(tmp, name + ".obj"), tmp)
        tr, mats = S.tris(), S.mats()
        g = {"area_of_obj_sha256": sha(tr["area_of_obj"]), "tri_mats_sha256": sha(mats[tr["mat"]].astype(np.float32)),
             "light_tris": [len(f) for f, _ in S.lights()], "ref_bvh": {}}
        for thresh in threshes:
            nodes, order, root = S.build_ref_bvh(thresh)
            g["ref_bvh"][str(thresh)] = {"n_nodes": int(len(nodes)), "root": int(root), "nodes_sha256": sha(nodes),
                                         "sorted_verts_sha256": sha(tr["verts"][order])}
        out[name] = g
    return out


if __name__ == "__main__":
    with open(os.path.join(ROOT, "tests", "golden", "host_record.json"), "w") as f:
        json.dump(record(), f, indent=1)
