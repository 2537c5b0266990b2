"""Multi-GPU plumbing: one process per GPU, samples sharded, one sum-reduce of the accumulation buffer.

The reference is single-GPU (src/main.cu:99-100). Here rank g of G renders a contiguous slice of the
sample-major work index space  w = sample * (W*H) + pixel  against its own replica of the scene; the
fixed-point accumulation buffers (int64) are summed onto rank 0 with ONE collective (NCCL over
NVLink on GPUs, gloo in the CPU tests). Integer addition is associative, so the reduced buffer is
bit-identical for every G and every reduction order.
"""
import numpy as np


def shard_work(n_pixels, spp, rank, world):
    """Contiguous slice [begin, end) of the n_pixels*spp work items owned by `rank`.

    Slices are cut on sample boundaries whenever spp >= world (every rank renders whole frames, which
    keeps primary rays coherent); otherwise on pixel boundaries inside a sample (spp < world, e.g. the
    shipped cornell-box config with spp=2 on 4 or 8 GPUs)."""
    total = n_pixels * spp
    if spp >= world:
        return (rank * spp // world) * n_pixels, ((rank + 1) * spp // world) * n_pixels
    return rank * total // world, (rank + 1) * total // world


class DevicePointer:
    """Exposes a raw device pointer to torch through __cuda_array_interface__ (no copy)."""

    def __init__(self, ptr, n, typestr="<i8"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def accum_as_tensor(render, device):
    import torch
    n = render.width * render.height * 3
    return torch.as_tensor(DevicePointer(render.device_accum_ptr(), n), device=device)


def aov_as_tensor(render, device):
    """The render's int64 AOV buffer (W*H*8) as a tensor without a copy; after reduce_accum on it, rank 0's get_aov() resolves the sum."""
    import torch
    n = render.width * render.height * 8
    return torch.as_tensor(DevicePointer(render.device_aov_ptr(), n), device=device)


def reduce_accum(tensor, dst=0):
    """Sum of the int64 accumulation buffers onto `dst` (one collective)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.reduce(tensor, dst=dst, op=dist.ReduceOp.SUM)
    return tensor


def resolve_numpy(accum, spp):
    """Host-side E11 (reference Render.cuh:348,350) for reduced buffers that live on the CPU (tests)."""
    v = (accum.astype(np.float64) / 4294967296.0 / float(spp)).astype(np.float32)
    cl = np.clip(v, 0.0, 1.0)
    return v, (np.float32(255.0) * np.power(cl, np.float32(0.6), dtype=np.float32)).astype(np.uint8)
