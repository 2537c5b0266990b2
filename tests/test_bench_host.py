"""Host-side pieces of bench.py that run without a GPU: the workload table, the builder enum, and the cpu_baseline leg
(the oracle on a bounded sample, which also yields the per-ray visit counts the roofline is computed from)."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT

sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_builder_names_match_the_c_abi(crt):
    assert bench.BUILDERS == {"lbvh": crt.BUILDER_LBVH, "lbvh8": crt.BUILDER_LBVH8, "ploc": crt.BUILDER_PLOC, "ploc8": crt.BUILDER_PLOC8}
    hdr = open(os.path.join(ROOT, "include", "crt.h")).read()
    for name, val in bench.BUILDERS.items():
        assert "CRT_BUILDER_%s = %d" % (name.upper(), val) in hdr


@pytest.mark.parametrize("name,size,spp", [("c1", (800, 600), 2), ("c2", (800, 600), 4), ("c3", (3840, 2160), 1024)])
def test_workloads_follow_baseline_json(name, size, spp, monkeypatch):
    monkeypatch.delenv("CRT_BUILDER", raising=False)
    w = bench.Workload(name)
    assert (w.width, w.height, w.spp) == (size[0], size[1], spp)
    assert w.bvh_thresh_n == 2 and abs(float(w.P_RR) - 0.6) < 1e-6
    assert w.light_sample_n == (1 if name == "c2" else 2)
    assert w.builder == bench.BUILDERS["ploc8"]                 # the default the bench line names in config.builder
    assert os.path.exists(w.obj)


@pytest.mark.parametrize("builder", ["lbvh", "ploc", "ploc8"])
def test_cpu_baseline_leg_counts_visits_on_the_same_tree(builder, monkeypatch):
    monkeypatch.setenv("CRT_BUILDER", builder)
    w = bench.Workload("c2")
    base, per_ray = bench.cpu_baseline_leg(w, budget_samples=3.0e4)
    assert base["kind"] == "port" and base["unit"] == "Msamples/s" and base["value"] > 0 and base["cores"] >= 1
    assert "oracle" in base["sample"]
    assert per_ray["rays_per_sample"] > 1.0
    for k in ("closest_inner", "closest_tris", "any_inner", "any_tris"):
        assert per_ray[k] > 0
    if builder == "ploc8":                                       # 8-wide nodes: far fewer node steps than pair nodes
        w2 = bench.Workload("c2")
        w2.builder = bench.BUILDERS["ploc"]
        _, pr2 = bench.cpu_baseline_leg(w2, budget_samples=3.0e4)
        assert per_ray["closest_inner"] < 0.6 * pr2["closest_inner"]


def test_dump_sample_is_seeded_and_bounded(tmp_path):
    small = bench.dump_sample_index(1000, 44)
    assert np.array_equal(small, np.arange(1000))                # fits: every item
    npix = 3840 * 2160
    a, b = bench.dump_sample_index(npix, 44), bench.dump_sample_index(npix, 44)
    assert np.array_equal(a, b) and len(a) * 44 <= bench.DUMP_BYTES and len(a) > npix // 8
    assert np.all(np.diff(a) > 0) and a[0] >= 0 and a[-1] < npix
    full = {"pixel_index": a.astype(np.float64), "accum": np.zeros((len(a), 3)), "frame": np.zeros((len(a), 3), np.float32)}
    bench.dump_outputs(str(tmp_path / "full"), full)            # the C3 dump, headers included, within the budget
    assert sum(os.path.getsize(tmp_path / "full" / (k + ".npy")) for k in full) <= 64 * 10 ** 6
    bench.dump_outputs(str(tmp_path / "d"), {"x": np.ones(7, np.float32), "i": a[:5].astype(np.float64)})
    assert np.array_equal(np.load(tmp_path / "d" / "x.npy"), np.ones(7, np.float32))
    assert np.array_equal(np.load(tmp_path / "d" / "i.npy"), a[:5])
    with pytest.raises(AssertionError):
        bench.dump_outputs(str(tmp_path / "e"), {"x": np.ones(7, np.int64)})


def test_reference_arm_runs_on_rank_zero_only(monkeypatch, capsys):
    import argparse
    monkeypatch.setenv("RANK", "1")
    monkeypatch.setenv("WORLD_SIZE", "2")
    monkeypatch.setenv("LOCAL_RANK", "1")
    bench.reference(argparse.Namespace(workload="c1", ref_spp=1, steps=1, warmup=0))
    assert capsys.readouterr().out == ""                          # other ranks exit without work or output
