#!/usr/bin/env python
"""bench.py — headline benchmark: Msamples/s of the path-tracing hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c1|c2|c3] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one run_view of the whole frame (all spp). With N > 1 the samples are sharded over the
ranks (strong scaling: total work fixed), each rank renders its shard against its own scene replica,
and the int64 accumulation buffers are summed onto rank 0 with one NCCL reduce, then resolved.
Prints ONE JSON line on rank 0. See DESIGN.md "Measurement" for the definition of every key.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (source, width, height, spp, description)   None -> value from the shipped config
    "c1": ("cornell-box", None, None, None, "C1 cornell-box 800x600 spp=2 light_sample_n=2 bvh_thresh_n=2 P_RR=0.6 (shipped config.json)"),
    "c2": ("veach-mis", None, None, None, "C2 veach-mis 800x600 spp=4 light_sample_n=1 (shipped config.json)"),
    "c3": ("cornell-box", 3840, 2160, 1024, "C3 cornell-box 3840x2160 spp=1024, samples sharded across the GPUs"),
    "c4": ("synthetic", 1920, 1080, 64, "C4 synthetic 10M-triangle heightfield scene 1920x1080 spp=64 (GPU BVH build + deep traversal)"),
    "c5": ("synthetic", 0, 0, 0, "C5 incoherent rays: 100M random rays vs the 10M-triangle BVH, closest-hit and any-hit"),
}


BUILDERS = {"lbvh": 0, "lbvh8": 1, "ploc": 2, "ploc8": 3}     # include/crt.h crt_builder


def parse_config_json(path):
    """config.json (reference src/main.cu:67-90) read with Python's json: used by the reference arm, which must not map
    the product's library (the ours arm goes through the product's own loader, crt_config_load)."""
    import types
    import numpy as np
    with open(path) as f:
        j = json.load(f)
    c = types.SimpleNamespace()
    c.OBJ_paths = [(e["OBJ_path"], e["MTL_dir"]) for e in j["OBJ_paths"]]
    c.eye_pos, c.lookat, c.up = (np.asarray([j[k]["x"], j[k]["y"], j[k]["z"]], np.float32) for k in ("eye_pos", "lookat", "up"))
    c.fov_y = float(j["fov_y"])
    c.width, c.height, c.spp = int(j["width"]), int(j["height"]), int(j["spp"])
    c.light_sample_n, c.P_RR, c.bvh_thresh_n = int(j["light_sample_n"]), float(j["P_RR"]), int(j["bvh_thresh_n"])
    return c


class Workload:
    """Camera + render settings + how to build the scene (product and oracle side)."""

    def __init__(self, name, small=False, use_product_loader=True):
        import numpy as np
        self.name = name
        self.builder = BUILDERS[os.environ.get("CRT_BUILDER", "ploc8")]
        source, W, H, spp, self.desc = WORKLOADS[name]
        self.source = source
        self.tmp = tempfile.mkdtemp(prefix="crt_bench_")
        if source == "synthetic":
            from tools import synthetic as sy
            c = sy.C4_CAMERA
            self.eye, self.lookat, self.up = (np.asarray(c[k], np.float32) for k in ("eye", "lookat", "up"))
            self.fov_y = c["fov_y"]
            self.width, self.height, self.spp = W or c["width"], H or c["height"], spp or c["spp"]
            self.light_sample_n, self.P_RR, self.bvh_thresh_n = c["light_sample_n"], c["P_RR"], c["bvh_thresh_n"]
            self.grid_n = int(os.environ.get("CRT_C4_GRID", "257" if small else str(sy.C4_FULL_N)))
            self.obj = None
        else:
            from tools import scene_fixture as sf
            cfg_path = sf.unpack(sf.fixture(source), self.tmp)
            if use_product_loader:
                import cudaraytracing_b200 as crt
                cfg = crt.load_config(cfg_path)
            else:
                cfg = parse_config_json(cfg_path)
            self.eye, self.lookat, self.up, self.fov_y = cfg.eye_pos, cfg.lookat, cfg.up, cfg.fov_y
            self.width, self.height, self.spp = W or cfg.width, H or cfg.height, spp or cfg.spp
            self.light_sample_n, self.P_RR, self.bvh_thresh_n = cfg.light_sample_n, cfg.P_RR, cfg.bvh_thresh_n
            self.obj = os.path.join(self.tmp, cfg.OBJ_paths[0][0])
        self.fovy_rad = np.float32(np.float32(self.fov_y) * np.float32(math.pi) / np.float32(180.0))
        self._arrays = None

    def arrays(self):
        if self._arrays is None:
            from tools import synthetic as sy
            self._arrays = sy.c4_scene(self.grid_n)
        return self._arrays

    def build_scene(self, crt, device):
        if self.obj:
            scene = crt.Scene().add_obj(self.obj, self.tmp)
        else:
            scene = crt.Scene().add_triangles(*self.arrays())
        return scene, scene.set_BVH(self.bvh_thresh_n, builder=self.builder, device=device)

    def build_oracle(self, orc):
        import numpy as np
        if self.obj:
            S = orc.Scene().add_obj(self.obj, self.tmp)
        else:
            v, m, o, mats = self.arrays()
            S = orc.Scene().add_arrays(v, m.astype(np.int32), o.astype(np.int32), mats)
        S.build_new_bvh(self.bvh_thresh_n, self.builder & 2)          # same topology as the product
        if self.builder & 1:
            S.build_wide8(self.bvh_thresh_n, self.builder)
        return S


DATA_NOTE = {
    "fixture": "synthetic camera paths (Philox seed 0) over the reference's cornell-box / veach-mis geometry "
               "(tests/golden/scenes fixtures, regenerated to OBJ/MTL at run time)",
    "synthetic": "procedural scene generated from a seed at run time (tools/synthetic.py), Philox seed 0",
}

S_NODE, S_NODE_WIDE, S_TRI, S_RAY_IO_CLOSEST, S_RAY_IO_ANY = 64, 80, 48, 32 + 8, 48 + 0   # bytes, DESIGN.md "Algorithmic bytes"
F_BOX, F_TRI = 20, 50                                                                     # flop per child slab test / triangle test, SURVEY.md section 8(d)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); smax.append(float(p[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if p[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------------------
# CPU baseline (oracle port) — bounded sample of the same workload; also yields the per-ray
# node / triangle visit counts the roofline uses (counted by the oracle on the same BVH and rule).
# ------------------------------------------------------------------------------------------------
def cpu_baseline_leg(cfg, budget_samples=float(os.environ.get("CRT_CPU_BUDGET", "4.0e7")), estimator=0, oracle_scene=None):
    from oracle import orc
    import numpy as np
    S = oracle_scene or cfg.build_oracle(orc)
    M = orc.inverse_view_matrix(cfg.eye, cfg.lookat, cfg.up)
    # bounded sample: the full frame at reduced resolution (same camera, same per-ray statistics), 1..spp samples
    scale = 1
    while (cfg.width // scale) * (cfg.height // scale) > budget_samples:
        scale *= 2
    w, h = cfg.width // scale, cfg.height // scale
    spp = max(1, min(cfg.spp, int(budget_samples // (w * h))))
    threads = os.cpu_count() or orc.max_threads()          # torchrun exports OMP_NUM_THREADS=1; use every host core
    t0 = time.time()
    _, st = S.render(cfg.eye, M, float(cfg.fovy_rad), w, h, 0, spp, cfg.P_RR, cfg.light_sample_n, threads=threads,
                      wide=bool(cfg.builder & 1), estimator=estimator)
    dt = time.time() - t0
    per_ray = {
        "closest_inner": st["closest_inner"] / max(st["closest_rays"], 1), "closest_tris": st["closest_tris"] / max(st["closest_rays"], 1),
        "any_inner": st["any_inner"] / max(st["any_rays"], 1), "any_tris": st["any_tris"] / max(st["any_rays"], 1),
        "rays_per_sample": (st["extend_rays"] + st["shadow_rays"] + st["probe_rays"]) / st["samples"],
    }
    base = {"value": round(w * h * spp / dt / 1e6, 4), "unit": "Msamples/s", "cores": threads, "kind": "port",
            "sample": "%dx%d spp=%d of the workload's camera (oracle/liborc.so, OpenMP), %.1f s" % (w, h, spp, dt)}
    return base, per_ray


def fp32_peak_tflops(peaks):
    """SMs x 128 lanes x 2 flop x max SM clock (BASELINE.md section 2): 74.5 TFLOP/s at 148 SMs and 1965 MHz."""
    return 148 * 128 * 2 * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6 / 1e12


def ncu_facts(workload, kernel):
    """Counters of one steady-state launch of `kernel` from the committed ncu capture of the final binary
    (profiles/ncu_final.json, written by tools/summarize_profile.py): never measured under this run."""
    tp = os.path.join(ROOT, "profiles", "ncu_final.json")
    if not os.path.exists(tp):
        return None
    with open(tp) as f:
        return json.load(f).get(workload, {}).get(kernel)


class Ctx:
    """One process per GPU: rank / world / device, the launching stream, barrier and max-over-ranks."""

    def __init__(self, args):
        import torch
        self.torch = torch
        self.rank, self.world, self.local = dist_env()
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus %d must be launched with torch.distributed.run --nproc-per-node %d" % (args.gpus, args.gpus))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            torch.distributed.init_process_group("nccl", device_id=self.dev)
        self.stream = torch.cuda.current_stream()
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)      # > 126 MB L2

    def barrier(self):
        if self.world > 1:
            self.torch.distributed.barrier()
        self.torch.cuda.synchronize()

    def allmax(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.torch.distributed.all_reduce(t, op=self.torch.distributed.ReduceOp.MAX)
        return [float(x) for x in t]

    def timed(self, fn, steps):
        """K steps between barrier + synchronize, CUDA events on the launching stream, max over ranks."""
        torch = self.torch
        self.flush.zero_()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        e1.record(self.stream)
        self.barrier()
        wall = (time.time() - t0) * 1e3
        ms, wall = self.allmax([e0.elapsed_time(e1), wall])
        return ms, wall

    def close(self):
        if self.world > 1:
            self.torch.distributed.destroy_process_group()


DUMP_BYTES = 64 * 10 ** 6     # --dump-outputs: at most this many bytes of .npy files per run
DUMP_SEED = 0


def dump_sample_index(n, bytes_per_item):
    """Sorted indices of a fixed, seeded sample of n items that fits DUMP_BYTES with room for the .npy headers (all of
    them when they fit): the same arguments give the same indices on every run and every build."""
    import numpy as np
    k = min(n, (DUMP_BYTES - 4096) // bytes_per_item)
    if k == n:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=k, replace=False))


def dump_outputs(out_dir, arrays):
    """Writes {name: array} as out_dir/<name>.npy (float32 / float64 only, DUMP_BYTES in all)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a)
        total += os.path.getsize(path)
    assert total <= DUMP_BYTES, total


def render_workload(ctx, name, steps, warmup, estimator=0, headline=False, clocks=False, prebuilt=None, dump=None):
    """One render workload (C1-C4) at ctx.world GPUs: device-timed value, e2e through the public API with host buffers,
    hashes of the reduced buffer and of the frame, per-kernel roofline (rank 0). dump: directory that receives what the
    last timed step returned to the caller (rank 0): the reduced accumulation buffer (int64 fixed point, 2^32 per unit,
    as float64) and the RGB8 frame (as float32), each (pixels, 3), for a seeded sample of pixels (pixel_index.npy)."""
    import hashlib
    import numpy as np
    import cudaraytracing_b200 as crt
    from cudaraytracing_b200 import distributed as cd
    torch = ctx.torch
    if prebuilt:                                              # (Workload, scene, build_ms): the C4 frame reuses the scene C5 has built
        cfg, scene, build_ms = prebuilt[:3]
    else:
        cfg = Workload(name)
        scene, build_ms = cfg.build_scene(crt, ctx.local)
    npix = cfg.width * cfg.height
    M = crt.inverse_view_matrix(cfg.eye, cfg.lookat, cfg.up)
    render = crt.Render(scene, cfg.width, cfg.height, cfg.spp, cfg.P_RR, cfg.light_sample_n)
    render.set_seed(0)
    render.set_estimator(estimator)
    render.set_stream(ctx.stream.cuda_stream)
    w0, w1 = cd.shard_work(npix, cfg.spp, ctx.rank, ctx.world)
    render.set_work_range(w0, w1)
    accum_t = cd.accum_as_tensor(render, ctx.dev)
    frame_host = torch.empty((cfg.height, cfg.width, 3), dtype=torch.uint8).pin_memory()
    frame_np = frame_host.numpy()
    launches = [0]

    def step_device():
        render.run_view(cfg.eye, M, cfg.fovy_rad)
        launches[0] += render.stats()["kernel_launches"]
        cd.reduce_accum(accum_t, 0)

    def step_e2e():
        # host buffers in, host buffer out: camera (13 floats) goes in with the call, the RGB8 frame comes back
        render.run_view(cfg.eye, M, cfg.fovy_rad)
        cd.reduce_accum(accum_t, 0)
        if ctx.rank == 0:
            render.get_frame_buffer(frame_np)

    for _ in range(warmup):
        step_device()
    sampler = ClockSampler(ctx.local) if (clocks and ctx.rank == 0) else None
    if sampler:
        sampler.start()
    launches[0] = 0
    ms_dev, _ = ctx.timed(step_device, steps)
    n_launches = launches[0]
    clk = sampler.stop() if sampler else None
    step_e2e()
    ms_e2e, wall_e2e = ctx.timed(step_e2e, steps)
    total_samples = npix * cfg.spp
    out = None
    if ctx.rank == 0:
        # identity of the result: the reduced fixed-point buffer and the tone-mapped frame do not depend on the number of
        # GPUs, the pool size or the scheduling (DESIGN.md section 6) - these two hashes must be equal at N = 1, 2, 4, 8
        acc = render.get_accum_i64()
        if dump:
            idx = dump_sample_index(npix, 3 * 8 + 3 * 4 + 8)
            dump_outputs(dump, {"pixel_index": idx.astype(np.float64),
                                "accum": acc.reshape(npix, 3)[idx].astype(np.float64),
                                "frame": frame_np.reshape(npix, 3)[idx].astype(np.float32)})
        out = {
            "value": round(total_samples * steps / (ms_dev * 1e3), 2), "unit": "Msamples/s", "ms_per_step": round(ms_dev / steps, 4),
            "e2e": {"value": round(total_samples * steps / (max(ms_e2e, wall_e2e) * 1e3), 2), "unit": "Msamples/s", "h2d_bytes_per_step": 13 * 4,
                    "d2h_bytes_per_step": npix * 3, "ms_per_step": round(max(ms_e2e, wall_e2e) / steps, 4)},
            "gpu_launches": int(n_launches),
            "accum_sha256": hashlib.sha256(acc.tobytes()).hexdigest(), "frame_sha256": hashlib.sha256(frame_np.tobytes()).hexdigest(),
            "config": {"workload": cfg.desc, "width": cfg.width, "height": cfg.height, "spp": cfg.spp, "light_sample_n": cfg.light_sample_n,
                       "P_RR": round(float(cfg.P_RR), 4), "bvh_thresh_n": cfg.bvh_thresh_n, "estimator": "mis" if estimator else "compat",
                       "builder": [k for k, v in BUILDERS.items() if v == cfg.builder][0],
                       "parallelism": ("samples" if cfg.spp >= ctx.world else "pixel rows of a sample") + " sharded over %d GPU(s), one int64 NCCL reduce" % ctx.world,
                       "l2": "256 MiB buffer written before each timed region (L2 flush)" + ("; per-step path/shadow queues exceed L2" if headline else "")},
            "bvh_build_gpu_ms": round(build_ms, 3), "triangles": scene.counts()["n_tris"], "nodes": scene.counts()["n_nodes"],
        }
        if estimator:
            out["config"]["pin"] = "the reference has no MIS estimator: this number has no reference counterpart and no external pin " \
                                   "(bit-exact against its own CPU statement only)"
        if clk:
            out["clocks"] = clk
        # per-kernel roofline pass (stage timing on, bounded spp): CUDA events around every stage of this workload
        peaks, peak_kind = load_peaks()
        cpu_base, per_ray = cpu_baseline_leg(cfg, estimator=estimator, oracle_scene=prebuilt[3] if prebuilt and len(prebuilt) > 3 else None) if headline \
            else cpu_baseline_leg(cfg, budget_samples=2.0e6, estimator=estimator, oracle_scene=prebuilt[3] if prebuilt and len(prebuilt) > 3 else None)
        render.clear_range()
        spp_probe = min(cfg.spp, 16)
        render.set_spp(spp_probe)
        render.set_stage_timing(True)
        render.run_view(cfg.eye, M, cfg.fovy_rad)
        st = render.stats()
        render.set_stage_timing(False)
        render.set_spp(cfg.spp)
        wide = bool(cfg.builder & 1)
        s_node, kids = (S_NODE_WIDE, 8) if wide else (S_NODE, 2)
        kernels = {
            "k_extend": {"ms": st["ms_extend"], "rays": st["extend_rays"] + st["probe_rays"],
                         "bytes_per_ray": per_ray["closest_inner"] * s_node + per_ray["closest_tris"] * S_TRI + S_RAY_IO_CLOSEST,
                         "flop_per_ray": per_ray["closest_inner"] * kids * F_BOX + per_ray["closest_tris"] * F_TRI},
            "k_shadow": {"ms": st["ms_shadow"], "rays": st["shadow_rays"],
                         "bytes_per_ray": per_ray["any_inner"] * s_node + per_ray["any_tris"] * S_TRI + S_RAY_IO_ANY,
                         "flop_per_ray": per_ray["any_inner"] * kids * F_BOX + per_ray["any_tris"] * F_TRI},
        }
        for k in kernels.values():
            k["achieved_gbs"] = k["rays"] * k["bytes_per_ray"] / (k["ms"] * 1e6) if k["ms"] > 0 else 0.0
            k["mrays_s"] = k["rays"] / (k["ms"] * 1e3) if k["ms"] > 0 else 0.0
            k["tflops"] = k["rays"] * k["flop_per_ray"] / (k["ms"] * 1e9) if k["ms"] > 0 else 0.0
        dom = max(kernels, key=lambda n: kernels[n]["ms"])
        resident = cfg.source != "synthetic"
        facts = ncu_facts(name, dom) or {}
        bvh_mb = (scene.counts()["n_nodes"] * s_node + scene.counts()["n_tris"] * 64) / 1e6
        out["roofline"] = {
            # what ncu says bounds the kernel (profiles/): with the BVH L1/L2-resident the traversal kernels wait on L1 / L2
            # latency and issue slots, DRAM is < 10 % busy; on the 10M-triangle scene node and triangle fetches are HBM sectors
            "bound": "l1/issue" if resident else "hbm", "kernel": dom, "achieved": round(kernels[dom]["achieved_gbs"], 1), "peak": peaks["hbm_gbs"],
            "unit": "GB/s", "frac": round(kernels[dom]["achieved_gbs"] / peaks["hbm_gbs"], 4), "traffic": facts.get("dram_bytes"),
            "peak_kind": peak_kind,
            "fp32_frac": round(kernels[dom]["tflops"] / fp32_peak_tflops(peaks), 4), "fp32_tflops": round(kernels[dom]["tflops"], 2),
            "fp32_peak_tflops": round(fp32_peak_tflops(peaks), 1),
            "issue_frac": facts.get("issue_frac"), "l2_gbs": facts.get("l2_gbs"), "lane_efficiency": facts.get("lane_efficiency"),
            "ncu": {"source": facts.get("source"), "what": "issue_frac, l2_gbs (lts__t_bytes / duration), lane_efficiency (threads per warp "
                    "instruction / 32) and traffic (dram__bytes_read + write) are ncu counters of ONE steady-state launch of this kernel in the "
                    "committed capture of this binary, not measured in this run"} if facts else None,
            "note": "achieved = algorithmic bytes (oracle-counted node (%d B) and triangle (48 B) visits + ray I/O per ray) x rays / stage time; " % s_node +
                    ("the BVH and triangles (%.0f MB) exceed the 126 MB L2: node and triangle fetches are HBM sector traffic" % bvh_mb if not resident else
                     "the BVH (%.1f MB) is L1/L2-resident, so frac compares L1-bound work with the HBM copy peak; fp32_frac is the same rays x "
                     "algorithmic flops (20 per child box, 50 per triangle) against SMs x 128 x 2 x clock" % bvh_mb),
            "launches": int(st["iterations"]), "avg_launch_ms": round(kernels[dom]["ms"] / max(st["iterations"], 1), 4),
            "stage_ms": {"generate": round(st["ms_generate"], 3), "extend": round(st["ms_extend"], 3), "shade": round(st["ms_shade"], 3),
                         "shadow": round(st["ms_shadow"], 3), "tail": round(st["ms_tail"], 3), "spp": spp_probe},
            "kernels": {n: {"mrays_s": round(k["mrays_s"], 1), "achieved_gbs": round(k["achieved_gbs"], 1), "bytes_per_ray": round(k["bytes_per_ray"], 1),
                            "fp32_tflops": round(k["tflops"], 2)} for n, k in kernels.items()},
            "per_ray": {k: round(v, 3) for k, v in per_ray.items()}}
        out["cpu_baseline"] = cpu_base
    del render, scene
    return out


def ours(args):
    ctx = Ctx(args)
    main = render_workload(ctx, args.workload, args.steps, args.warmup, estimator=args.estimator, headline=True, clocks=True,
                           dump=args.dump_outputs)
    subs = {}
    if args.workload == "c3" and not args.no_sub:
        # the other BASELINE configs at the same number of GPUs and the same number of timed steps
        subs["c1"] = render_workload(ctx, "c1", args.steps, 3)
        subs["c2"] = render_workload(ctx, "c2", args.steps, 3)
        subs["c2_mis"] = render_workload(ctx, "c2", args.steps, 3, estimator=1)
        subs["c5"], subs["c4"] = c5_workload(ctx, args.steps, 3, with_c4=True)
    if ctx.rank == 0:
        out = {"metric": "Msamples/s", "value": main["value"], "unit": "Msamples/s", "n_gpus": ctx.world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
               "data": DATA_NOTE["synthetic" if main["triangles"] > 5000000 else "fixture"]}
        for key in ("config", "e2e", "gpu_launches", "clocks", "frame_sha256", "accum_sha256", "roofline", "cpu_baseline", "bvh_build_gpu_ms",
                    "triangles", "nodes"):
            out[key] = main.get(key)
        if subs:
            out["workloads"] = subs
        print(json.dumps(out), flush=True)
    ctx.close()


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own code (oracle/_ref/libref.so = its headers compiled headless for
# sm_100a): host OBJ load + BVH build on the CPU, then its view_render_kernel on one B200.
# ------------------------------------------------------------------------------------------------
class RefLib:
    """oracle/_ref/libref.so: the reference's own headers compiled headless for sm_100a (oracle/ref_harness)."""

    def __init__(self):
        import ctypes as C
        self.C = C
        so = os.path.join(ROOT, "oracle", "_ref", "libref.so")
        if not os.path.exists(so):
            raise FileNotFoundError("oracle/_ref/libref.so not built (needs /root/reference at build time)")
        R = self.R = C.CDLL(so)
        R.ref_host_load.restype = C.c_void_p
        R.ref_host_load.argtypes = [C.c_char_p, C.c_char_p, C.c_uint, C.c_uint, C.c_uint]
        R.ref_host_from_arrays.restype = C.c_void_p
        R.ref_host_from_arrays.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_uint, C.c_uint]
        R.ref_build_bvh.restype = C.c_double
        R.ref_build_bvh.argtypes = [C.c_void_p, C.c_uint]
        R.ref_host_times.argtypes = [C.c_void_p, C.c_void_p]
        R.ref_device_init.argtypes = [C.c_void_p]
        R.ref_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_uint, C.c_float, C.c_int, C.c_void_p,
                                 C.POINTER(C.c_float), C.POINTER(C.c_double)]
        R.ref_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.POINTER(C.c_float)]
        R.ref_inverse_view.argtypes = [C.c_void_p] * 4
        R.ref_free.argtypes = [C.c_void_p]
        R.ref_n_tris.argtypes = [C.c_void_p]
        R.ref_n_nodes.argtypes = [C.c_void_p]

    class quiet:
        """The reference printf()s from its loaders and Object constructor."""

        def __enter__(self):
            sys.stdout.flush()
            self.devnull = os.open(os.devnull, os.O_WRONLY)
            self.saved = os.dup(1)
            os.dup2(self.devnull, 1)

        def __exit__(self, *a):
            os.dup2(self.saved, 1)
            os.close(self.devnull)
            os.close(self.saved)


def ref_render_workload(ref, name, steps, warmup, spp_list):
    """view_render_kernel (Render.cuh:330) of the reference on ONE GPU for a shipped scene: host load + BVH build timed on
    the CPU (one thread: the reference has none), then the frame at every spp of spp_list (the kernel is a serial loop
    over spp per pixel: the rates show how linear its cost is). Returns the dict of the LAST spp as the headline."""
    import numpy as np
    C, R = ref.C, ref.R
    cfg = Workload(name, use_product_loader=False)
    with ref.quiet():
        h = R.ref_host_load(cfg.obj.encode(), (cfg.tmp + "/").encode(), cfg.width, cfg.height, cfg.bvh_thresh_n)
        host_ms = np.zeros(3)
        R.ref_host_times(h, host_ms.ctypes.data_as(C.c_void_p))
        rc = R.ref_device_init(h)
    if rc != 0:
        return {"unavailable": "reference device init failed rc=%d (per-pixel stacks need %.1f GB)" % (rc, 8712.0 * cfg.width * cfg.height / 1e9)}
    eye = np.asarray(cfg.eye, np.float32)
    M = np.zeros(9, np.float32)
    R.ref_inverse_view(eye.ctypes.data_as(C.c_void_p), np.asarray(cfg.lookat, np.float32).ctypes.data_as(C.c_void_p),
                       np.asarray(cfg.up, np.float32).ctypes.data_as(C.c_void_p), M.ctypes.data_as(C.c_void_p))
    frame = np.zeros(cfg.width * cfg.height * 3, np.uint8)
    kms, wms = C.c_float(), C.c_double()
    rates = {}
    for spp in spp_list:
        spp = min(spp, cfg.spp)

        def step():
            r = R.ref_render(h, eye.ctypes.data_as(C.c_void_p), M.ctypes.data_as(C.c_void_p), float(cfg.fovy_rad), spp, float(cfg.P_RR),
                             int(cfg.light_sample_n), frame.ctypes.data_as(C.c_void_p), C.byref(kms), C.byref(wms))
            if r != 0:
                raise RuntimeError("reference render failed")
            return kms.value, wms.value

        for _ in range(warmup):
            step()
        ks, ws = zip(*[step() for _ in range(steps)])
        samples = cfg.width * cfg.height * spp
        rates[spp] = {"value": round(samples * len(ws) / (sum(ws) * 1e3), 3), "kernel_only": round(samples * len(ks) / (sum(ks) * 1e3), 3),
                      "ms_per_step": round(sum(ws) / len(ws), 3)}
    with ref.quiet():
        R.ref_free(h)
    last = min(spp_list[-1], cfg.spp)
    return {"value": rates[last]["value"], "unit": "Msamples/s", "ms_per_step": rates[last]["ms_per_step"],
            "kernel_only_msamples_s": rates[last]["kernel_only"], "spp_timed": last,
            "by_spp": {str(k): v for k, v in rates.items()},
            "config": {"workload": cfg.desc, "width": cfg.width, "height": cfg.height, "spp": cfg.spp, "light_sample_n": cfg.light_sample_n,
                       "P_RR": round(float(cfg.P_RR), 4), "bvh_thresh_n": cfg.bvh_thresh_n,
                       "what": "view_render_kernel (Render.cuh:330) rebuilt headless for sm_100a, 16x16 blocks, timed like main.cu:370-376 "
                               "(kernel + sync + D2H of the RGB8 frame); single GPU (the reference has no multi-GPU path)"},
            "sample": "full frame %dx%d at spp=%s of %d (the kernel loops over spp per pixel; by_spp shows the rate at each)" %
                      (cfg.width, cfg.height, "/".join(str(min(x, cfg.spp)) for x in spp_list), cfg.spp),
            "host_ms": {"obj_parse": round(host_ms[0], 1), "load_object": round(host_ms[1], 1), "bvh_build": round(host_ms[2], 1), "threads": 1,
                        "cpu": cpu_model()}}


def ref_synthetic_child(grid_n, n_rays, spp, out_path, steps=3, warmup=1):
    """Runs in a child process (the parent enforces the time limit): the reference's host BVH build over the synthetic scene,
    its DeviceBVH::intersect on C5 rays (ref_trace; best kernel time of `steps` timed calls) and its render kernel on the C4
    camera (mean of `steps` timed calls); `warmup` untimed calls before each."""
    import numpy as np
    from tools import synthetic as sy
    ref = RefLib()
    C, R = ref.C, ref.R
    res = {"grid_n": grid_n}

    def save():
        with open(out_path, "w") as f:
            json.dump(res, f)

    v, m, o, mats = sy.c4_scene(grid_n)
    v = np.ascontiguousarray(v, np.float32); m = np.ascontiguousarray(m, np.int32); o = np.ascontiguousarray(o, np.int32)
    mats = np.ascontiguousarray(mats, np.float32)
    cam = sy.C4_CAMERA
    W, H = cam["width"], cam["height"]
    res["triangles"] = int(len(v))
    with ref.quiet():
        t0 = time.time()
        h = R.ref_host_from_arrays(v.ctypes.data, m.ctypes.data, o.ctypes.data, len(v), mats.ctypes.data, len(mats), W, H)
        res["host_load_ms"] = round((time.time() - t0) * 1e3, 1)
    save()
    with ref.quiet():
        res["host_bvh_build_ms"] = round(R.ref_build_bvh(h, cam["bvh_thresh_n"]), 1)
    res["nodes"] = int(R.ref_n_nodes(h))
    save()
    with ref.quiet():
        rc = R.ref_device_init(h)
    if rc != 0:
        res["device"] = "reference device init failed rc=%d" % rc
        save()
        return
    lo, hi = v.reshape(-1, 3).min(axis=0), v.reshape(-1, 3).max(axis=0)
    rays = sy.random_rays(lo, hi, n_rays, key=0xC5, any_hit=False)
    t = np.zeros(n_rays, np.float32)
    kms = C.c_float()
    best = 1e30
    for k in range(warmup + steps):
        if R.ref_trace(h, rays.ctypes.data, n_rays, t.ctypes.data, C.byref(kms)) != 0:
            res["c5"] = "ref_trace failed"
            save()
            return
        if k >= warmup:
            best = min(best, kms.value)
    res["c5"] = {"value": round(n_rays / best / 1e3, 2), "unit": "Mrays/s", "rays": n_rays, "kernel_ms": round(best, 3),
                 "hit_frac": round(float((t < 1e30).mean()), 4),
                 "what": "DeviceBVH::intersect (DeviceBVH.cuh:128-170), one thread per ray, closest hit; the reference has no any-hit traversal "
                         "(blocked(), Render.cuh:19-27, is a full closest-hit traversal)"}
    save()
    eye = np.asarray(cam["eye"], np.float32)
    M = np.zeros(9, np.float32)
    R.ref_inverse_view(eye.ctypes.data, np.asarray(cam["lookat"], np.float32).ctypes.data, np.asarray(cam["up"], np.float32).ctypes.data, M.ctypes.data)
    fovy = np.float32(np.float32(cam["fov_y"]) * np.float32(math.pi) / np.float32(180.0))
    frame = np.zeros(W * H * 3, np.uint8)
    wms = C.c_double()
    ws = []
    for k in range(warmup + steps):
        if R.ref_render(h, eye.ctypes.data, M.ctypes.data, float(fovy), spp, float(cam["P_RR"]), int(cam["light_sample_n"]), frame.ctypes.data,
                        C.byref(kms), C.byref(wms)) != 0:
            res["c4"] = "ref_render failed"
            save()
            return
        if k >= warmup:
            ws.append(wms.value)
    res["c4"] = {"value": round(W * H * spp * len(ws) / (sum(ws) * 1e3), 3), "unit": "Msamples/s", "spp_timed": spp, "ms_per_step": round(sum(ws) / len(ws), 2)}
    save()


def ref_synthetic_workload(limit_s, steps=3, warmup=1):
    """C4 / C5 reference numbers (BASELINE.md section 3): the full 10M-triangle scene under a time limit ("DNF > T" if its host
    build does not finish), and when it does not, the largest grid of the ladder that does."""
    import subprocess
    from tools import synthetic as sy
    out = {}
    for grid_n in (sy.C4_FULL_N, 1001, 513):
        path = os.path.join(tempfile.mkdtemp(prefix="crt_ref_"), "res.json")
        code = "import bench; bench.ref_synthetic_child(%d, %d, %d, %r, %d, %d)" % (grid_n, 2000000, 4, path, steps, warmup)
        t0 = time.time()
        try:
            subprocess.run([sys.executable, "-c", code], cwd=ROOT, timeout=limit_s, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            timed_out = False
        except subprocess.TimeoutExpired:
            timed_out = True
        r = {}
        if os.path.exists(path):
            with open(path) as f:
                r = json.load(f)
        r["wall_s"] = round(time.time() - t0, 1)
        if timed_out:
            r["dnf"] = "DNF > %d s" % limit_s
        out["grid_%d" % grid_n] = r
        if "c5" in r and not timed_out:
            break
    return out


def reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return
    os.environ.setdefault("CUDA_VISIBLE_DEVICES", str(local))
    try:
        ref = RefLib()
    except FileNotFoundError as e:
        print(json.dumps({"impl": "reference", "unavailable": str(e)}))
        return
    if WORKLOADS[args.workload][0] == "synthetic":
        r = ref_synthetic_workload(args.ref_limit, args.steps, args.warmup)
        done = [v for v in r.values() if "c5" in v and isinstance(v["c5"], dict)]
        key = "c5" if args.workload == "c5" else "c4"
        if not done or not isinstance(done[-1].get(key), dict):
            print(json.dumps({"impl": "reference", "unavailable": "reference did not finish the synthetic scene within the limit", "detail": r}))
            return
        d = done[-1]
        print(json.dumps({"impl": "reference", "metric": "Mrays/s (closest-hit)" if key == "c5" else "Msamples/s", "value": d[key]["value"],
                          "unit": d[key]["unit"], "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": d[key].get("kernel_ms", d[key].get("ms_per_step")),
                          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": DATA_NOTE["synthetic"],
                          "config": {"workload": WORKLOADS[args.workload][4], "triangles": d["triangles"], "grid_n": d["grid_n"]},
                          "e2e": {"value": d[key]["value"], "unit": d[key]["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "cpu_baseline": {"value": d[key]["value"], "unit": d[key]["unit"], "cores": 1, "kind": "reference",
                                           "sample": "grid %d (%d triangles); host BVH build %.1f s on one thread" %
                                                     (d["grid_n"], d["triangles"], d["host_bvh_build_ms"] / 1e3)},
                          "detail": r}), flush=True)
        return
    spp_list = [args.ref_spp, args.ref_spp * 8] if args.ref_spp > 0 else [WORKLOADS[args.workload][3] or 1 << 30]
    sampler = ClockSampler(local)
    sampler.start()
    main = ref_render_workload(ref, args.workload, args.steps, args.warmup, spp_list[:1] if args.workload != "c3" else spp_list)
    clocks = sampler.stop()
    if "unavailable" in main:
        print(json.dumps({"impl": "reference", "unavailable": main["unavailable"]}))
        return
    subs = {}
    if args.workload == "c3" and not args.no_sub:
        subs["c1"] = ref_render_workload(ref, "c1", args.steps, 3, [1 << 30])
        subs["c2"] = ref_render_workload(ref, "c2", args.steps, 3, [1 << 30])
        syn = ref_synthetic_workload(args.ref_limit, args.steps, args.warmup)
        done = [v for v in syn.values() if isinstance(v.get("c5"), dict)]
        subs["c5"] = dict(done[-1]["c5"], triangles=done[-1]["triangles"], grid_n=done[-1]["grid_n"],
                          host_bvh_build_ms=done[-1]["host_bvh_build_ms"]) if done else {"unavailable": "see synthetic"}
        subs["synthetic"] = syn
    out = {"impl": "reference", "metric": "Msamples/s", "value": main["value"], "unit": "Msamples/s", "n_gpus": 1, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "same fixtures as the ours arm, written back to OBJ/MTL and read by the reference's own loader",
           "config": main["config"], "e2e": {"value": main["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "kernel_only_msamples_s": main["kernel_only_msamples_s"], "by_spp": main["by_spp"],
           "cpu_baseline": {"value": main["value"], "unit": "Msamples/s", "cores": 1, "kind": "reference", "sample": main["sample"],
                            "host_ms": main["host_ms"]},
           "clocks": clocks}
    if subs:
        out["workloads"] = subs
    print(json.dumps(out), flush=True)


def c5_workload(ctx, steps, warmup, n_total=None, with_c4=False, dump=None):
    """C5: 100M incoherent rays against the 10M-triangle BVH; closest-hit and any-hit Mrays/s with the rays resident in HBM, and
    the same through crt_trace_rays with HOST buffers (rays H2D, hits D2H inside the timed call). Rays are independent: they
    are sharded over the ranks, no collective. dump: directory that receives, for a seeded sample of rank 0's rays
    (ray_index.npy), the hit distance (float32) and face id (float64, -1 on a miss) of the last timed closest-hit and
    any-hit steps. An any-hit ray reports one of its blockers, and which one depends on scheduling: compare any_face >= 0."""
    import hashlib
    import numpy as np
    import cudaraytracing_b200 as crt
    torch = ctx.torch
    cfg = Workload("c5")
    scene, build_ms = cfg.build_scene(crt, ctx.local)
    n_total = int(n_total or os.environ.get("CRT_C5_RAYS", "100000000"))
    n0, n1 = ctx.rank * n_total // ctx.world, (ctx.rank + 1) * n_total // ctx.world
    n = n1 - n0
    rays = torch.empty((n, 8), dtype=torch.float32, device=ctx.dev)
    t_out = torch.empty(n, dtype=torch.float32, device=ctx.dev)
    f_out = torch.empty(n, dtype=torch.int32, device=ctx.dev)
    res = {}
    dumped = {}
    if dump and ctx.rank == 0:
        idx = dump_sample_index(n, 2 * (4 + 8) + 8)
        dumped["ray_index"] = (idx + n0).astype(np.float64)
        idx_dev = torch.from_numpy(idx).to(ctx.dev)
    for mode, name in ((crt.RAY_CLOSEST, "closest"), (crt.RAY_ANY, "any")):
        scene.random_rays_device(rays.data_ptr(), n, start=n0, key=0xC5, any_hit=(mode == crt.RAY_ANY), stream=ctx.stream.cuda_stream)
        for _ in range(warmup):
            scene.trace_rays_device(rays.data_ptr(), n, mode, t_out.data_ptr(), f_out.data_ptr(), ctx.stream.cuda_stream)
        ctx.flush.zero_()
        ctx.barrier()
        kms = 0.0
        for _ in range(steps):
            kms += scene.trace_rays_device(rays.data_ptr(), n, mode, t_out.data_ptr(), f_out.data_ptr(), ctx.stream.cuda_stream)
        ctx.barrier()
        kms = ctx.allmax([kms])[0]
        hits = ctx.allmax([float((f_out >= 0).sum())])[0] if ctx.world == 1 else float((f_out >= 0).float().mean()) * n
        # identity of the result: hash of (t bits, face) of this rank's first million rays (rank 0 = rays 0 .. 10^6 - 1 for every N)
        head = min(n, 1000000)
        digest = hashlib.sha256(t_out[:head].cpu().numpy().tobytes() + f_out[:head].cpu().numpy().tobytes()).hexdigest()
        res[name] = dict(ms=kms / steps, mrays=n_total * steps / (kms * 1e3), hit_frac=hits / n, sha=digest)
        if dumped:
            dumped[name + "_t"] = t_out[idx_dev].cpu().numpy().astype(np.float32)
            dumped[name + "_face"] = f_out[idx_dev].cpu().numpy().astype(np.float64)
    if dumped:
        dump_outputs(dump, dumped)
    # e2e: host buffers through crt_trace_rays (pinned staging, chunks on two streams inside the library)
    nb = min(n, int(os.environ.get("CRT_C5_E2E_RAYS", "20000000")))
    scene.random_rays_device(rays.data_ptr(), nb, start=n0, key=0xC5, any_hit=False, stream=ctx.stream.cuda_stream)
    # the caller's buffers are page-locked host memory (the contract's "inputs from pinned host memory"): the library streams them
    # by DMA in chunks; a second measurement with pageable numpy arrays goes through its pinned staging + host-thread copies
    pin_rays = torch.empty((nb, 8), dtype=torch.float32).pin_memory()
    pin_rays.copy_(rays[:nb])
    pin_t, pin_f = torch.empty(nb, dtype=torch.float32).pin_memory(), torch.empty(nb, dtype=torch.int32).pin_memory()
    host_rays = pin_rays.numpy()
    for _ in range(max(1, min(warmup, 2))):               # warm-up at full size: chunk buffers, first touch of the result pages
        scene.trace_rays(host_rays, crt.RAY_CLOSEST, out=(pin_t.numpy(), pin_f.numpy()))
    ctx.barrier()
    e2e_calls = steps
    t0 = time.time()
    for _ in range(e2e_calls):
        ht, hf, _ = scene.trace_rays(host_rays, crt.RAY_CLOSEST, out=(pin_t.numpy(), pin_f.numpy()))
    e2e_s = ctx.allmax([(time.time() - t0) / e2e_calls])[0]
    pageable = np.array(host_rays[: min(nb, 8000000)])
    page_t, page_f = np.zeros(len(pageable), np.float32), np.zeros(len(pageable), np.int32)
    scene.trace_rays(pageable, crt.RAY_CLOSEST, out=(page_t, page_f))
    t0 = time.time()
    for _ in range(steps):
        scene.trace_rays(pageable, crt.RAY_CLOSEST, out=(page_t, page_f))
    pageable_s = ctx.allmax([(time.time() - t0) / steps])[0]
    out = None
    if ctx.rank == 0:
        peaks, peak_kind = load_peaks()
        from oracle import orc
        O = cfg.build_oracle(orc)
        sample = host_rays[:200000]
        which = 4 if cfg.builder & 1 else 0
        wide = bool(cfg.builder & 1)
        s_node, kids = (S_NODE_WIDE, 8) if wide else (S_NODE, 2)
        ot, of, st = O.trace(sample, which=which, mode=0, want_stats=True, threads=os.cpu_count())
        t0 = time.time()
        O.trace(sample, which=which, mode=0, threads=os.cpu_count())
        cpu_dt = time.time() - t0
        parity = bool(np.array_equal(of, hf[:len(sample)]) and np.array_equal(ot.view(np.uint32), ht[:len(sample)].view(np.uint32)))
        bpr = st["inner"] / st["rays"] * s_node + st["tris"] / st["rays"] * S_TRI + S_RAY_IO_CLOSEST
        fpr = st["inner"] / st["rays"] * kids * F_BOX + st["tris"] / st["rays"] * F_TRI
        per_gpu_rate = res["closest"]["mrays"] * 1e6 / ctx.world                  # the roofline is one GPU's: rays per second and GPU
        ach = per_gpu_rate * bpr / 1e9
        facts = ncu_facts("c5", "k_trace_batch") or {}
        pcie_gbs = float(os.environ.get("CRT_PCIE_GBS", "55.0"))
        e2e_rate = nb * ctx.world / e2e_s / 1e6
        out = {
            "value": round(res["closest"]["mrays"], 1), "unit": "Mrays/s", "metric": "Mrays/s (closest-hit)", "ms_per_step": round(res["closest"]["ms"], 3),
            "any_hit": {"mrays_s": round(res["any"]["mrays"], 1), "ms_per_step": round(res["any"]["ms"], 3), "blocked_frac": round(res["any"]["hit_frac"], 4),
                        "hits_sha256": res["any"]["sha"]},
            "closest_hit_frac": round(res["closest"]["hit_frac"], 4), "hits_sha256": res["closest"]["sha"],
            "e2e": {"value": round(e2e_rate, 1), "unit": "Mrays/s", "h2d_bytes_per_step": nb * 32, "d2h_bytes_per_step": nb * 8,
                    "pcie_frac": round(e2e_rate * 1e6 * 32 / 1e9 / ctx.world / pcie_gbs, 3),
                    "pageable_mrays_s": round(len(pageable) * ctx.world / pageable_s / 1e6, 1),
                    "calls": e2e_calls,
                    "note": "crt_trace_rays with page-locked host buffers, %d rays per GPU, mean of the timed calls after a full-size warm-up call; "
                            "pcie_frac = 32 B per ray host-to-device (the 8 B per ray of "
                            "results go the other way at the same time) against %.0f GB/s per direction of one PCIe gen5 x16 link (CRT_PCIE_GBS); "
                            "pageable_mrays_s: the same call with pageable numpy arrays (pinned staging + host-thread copies inside the library)" % (nb, pcie_gbs),
                    "parity": "first %d hits == oracle: %s" % (len(sample), parity)},
            "gpu_launches": 2 * steps,
            "config": {"workload": cfg.desc, "rays": n_total, "triangles": scene.counts()["n_tris"], "nodes": scene.counts()["n_nodes"],
                       "builder": [k for k, v in BUILDERS.items() if v == cfg.builder][0],
                       "l2": "BVH + triangles (%.0f MB) and the ray buffers exceed L2; 256 MiB flush before the timed region" %
                             ((scene.counts()["n_nodes"] * s_node + scene.counts()["n_tris"] * 64) / 1e6)},
            "roofline": {"bound": "hbm", "kernel": "k_trace_batch<closest>", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": round(ach / peaks["hbm_gbs"], 4), "traffic": facts.get("dram_bytes"), "peak_kind": peak_kind,
                         "fp32_frac": round(per_gpu_rate * fpr / 1e12 / fp32_peak_tflops(peaks), 4), "issue_frac": facts.get("issue_frac"),
                         "l2_gbs": facts.get("l2_gbs"), "lane_efficiency": facts.get("lane_efficiency"),
                         "note": "per GPU: aggregate rate / %d GPU(s) x algorithmic bytes per ray against one GPU's HBM copy peak" % ctx.world,
                         "per_ray": {"inner": round(st["inner"] / st["rays"], 2), "tris": round(st["tris"] / st["rays"], 2), "bytes": round(bpr, 1),
                                     "flop": round(fpr, 1)}},
            "cpu_baseline": {"value": round(len(sample) / cpu_dt / 1e6, 3), "unit": "Mrays/s", "cores": os.cpu_count(), "kind": "port",
                             "sample": "%d of the same rays, oracle traversal, %.1f s" % (len(sample), cpu_dt)},
            "bvh_build_gpu_ms": round(build_ms, 3)}
    del rays, t_out, f_out
    c4 = None
    if with_c4:
        # C4: the 1920x1080 spp 64 frame of the same 10M-triangle scene (no second build of scene or oracle tree)
        c4cfg = Workload("c4")
        c4cfg._arrays = cfg._arrays
        c4 = render_workload(ctx, "c4", steps, 2, prebuilt=(c4cfg, scene, build_ms) + ((O,) if ctx.rank == 0 else ()))
    del scene
    return (out, c4) if with_c4 else out


def ours_c5(args):
    ctx = Ctx(args)
    sampler = ClockSampler(ctx.local) if ctx.rank == 0 else None
    if sampler:
        sampler.start()
    r = c5_workload(ctx, args.steps, args.warmup, dump=args.dump_outputs)
    if ctx.rank == 0:
        out = {"metric": r.pop("metric"), "value": r.pop("value"), "unit": r.pop("unit"), "n_gpus": ctx.world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": r.pop("ms_per_step"), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
               "data": DATA_NOTE["synthetic"], "clocks": sampler.stop()}
        out.update(r)
        print(json.dumps(out), flush=True)
    ctx.close()


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip() + " x%d" % os.cpu_count()
    except OSError:
        pass
    return "unknown x%d" % (os.cpu_count() or 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3, help="timed steps of every measurement")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--builder", default=None, choices=sorted(BUILDERS), help="BVH topology + node layout (default: CRT_BUILDER or ploc8)")
    ap.add_argument("--ref-spp", type=int, default=4, help="reference arm: samples per pixel of the bounded sample (<=0: full)")
    ap.add_argument("--ref-limit", type=int, default=240, help="reference arm, synthetic scene: seconds before its host build is DNF")
    ap.add_argument("--estimator", type=int, default=0, choices=[0, 1], help="0 compat (the reference's estimator), 1 mis")
    ap.add_argument("--no-sub", action="store_true", help="default C3 run: skip the short C1 / C2 / C5 sub-measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the headline workload's last step returned as DIR/<name>.npy "
                         "(float32 / float64, at most 64 MB, a seeded sample of larger outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the ours arm's outputs")
    if args.builder:
        os.environ["CRT_BUILDER"] = args.builder
    if args.impl == "reference":
        reference(args)
    elif args.workload == "c5":
        ours_c5(args)
    else:
        ours(args)


if __name__ == "__main__":
    main()
