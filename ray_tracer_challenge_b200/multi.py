"""Host plumbing for one frame rendered by several processes (one per GPU, `torchrun`): a canvas in POSIX shared
memory that every rank writes its bands into — the "simple host gather" of SURVEY.md §8e, with no copy and no
collective on the data path (render_samples_shared for an anti-aliased frame) — the same for the frame's PPM text
(SharedText, render_ppm_shared), plus the two scalar reductions the benchmark needs (torch.distributed is plumbing here,
not the product)."""
from __future__ import annotations

from multiprocessing import shared_memory

import numpy as np


def _shared_memory(name: str, size: int, create: bool) -> shared_memory.SharedMemory:
    """A POSIX shared memory segment: created afresh (create=True, the owning rank) or attached."""
    if create:
        try:
            shared_memory.SharedMemory(name=name).unlink()
        except FileNotFoundError:
            pass
        return shared_memory.SharedMemory(name=name, create=True, size=size)
    shm = shared_memory.SharedMemory(name=name)
    # Python < 3.13 registers attached segments with the resource tracker, which then tries to unlink them a second time at
    # exit; only the creating rank owns the segment
    try:
        from multiprocessing import resource_tracker

        resource_tracker.unregister(shm._name, "shared_memory")
    except Exception:
        pass
    return shm


class SharedCanvas:
    """width x height f32 RGB plane followed by the 8-bit plane, shared by all ranks of one node."""

    def __init__(self, name: str, width: int, height: int, create: bool):
        self.width, self.height = width, height
        size = width * height * 15
        self.shm, self.owner = _shared_memory(name, size, create), create
        self.buf = np.ndarray((size,), np.uint8, buffer=self.shm.buf)
        self.rgb = self.buf[: width * height * 12].view(np.float32).reshape(height, width, 3)
        self.u8 = self.buf[width * height * 12:].reshape(height, width, 3)

    @property
    def address(self) -> int:
        return self.buf.ctypes.data

    @property
    def nbytes(self) -> int:
        return self.buf.nbytes

    def close(self):
        self.rgb = self.u8 = self.buf = None
        self.shm.close()
        if self.owner:
            self.shm.unlink()


def open_shared_canvas(dist, rank: int, name: str, width: int, height: int) -> SharedCanvas:
    """Rank 0 creates the canvas, everybody else attaches after a barrier."""
    canvas = SharedCanvas(name, width, height, create=True) if rank == 0 else None
    dist.barrier()
    if rank != 0:
        canvas = SharedCanvas(name, width, height, create=False)
    return canvas


class SharedText:
    """The PPM text of one frame shared by all ranks of one node (render_ppm_shared): `height` uint64 row lengths, which
    every rank fills in for its own rows, followed by rtc_ppm_bound(width, height) bytes of text, into which every rank
    writes its own bands."""

    def __init__(self, name: str, width: int, height: int, create: bool):
        self.width, self.height = width, height
        self.bound = _ppm_bound(width, height)
        size = height * 8 + self.bound
        self.shm, self.owner = _shared_memory(name, size, create), create
        self.raw = np.ndarray((size,), np.uint8, buffer=self.shm.buf)
        self.row_bytes = self.raw[: height * 8].view(np.uint64)
        self.buf = self.raw[height * 8:]

    @property
    def address(self) -> int:
        return self.raw.ctypes.data

    @property
    def nbytes(self) -> int:
        return self.raw.nbytes

    def text(self, length: int) -> str:
        return self.buf[:length].tobytes().decode("ascii")

    def close(self):
        self.row_bytes = self.buf = self.raw = None
        self.shm.close()
        if self.owner:
            self.shm.unlink()


def _ppm_bound(width: int, height: int) -> int:
    import ctypes as C

    from . import device_library

    lib = device_library()
    lib.rtc_ppm_bound.restype = C.c_size_t
    lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    return int(lib.rtc_ppm_bound(width, height))


def open_shared_text(dist, rank: int, name: str, width: int, height: int) -> SharedText:
    """Rank 0 creates the text, everybody else attaches after a barrier."""
    text = SharedText(name, width, height, create=True) if rank == 0 else None
    dist.barrier()
    if rank != 0:
        text = SharedText(name, width, height, create=False)
    return text


def render_samples_shared(dist, rank: int, world_size: int, prepared, canvas: SharedCanvas, samples: int, depth: int = 5):
    """One anti-aliased frame (samples x samples samples per pixel) rendered by world_size ranks of one node into `canvas`,
    rank r writing the bands of shard r of `prepared` (a PreparedScene committed on one device) into both planes, then a
    barrier: canvas.rgb / canvas.u8 then hold render_samples(samples)'s frame."""
    prepared.render_samples(samples, depth, out_rgb=canvas.rgb, out_u8=canvas.u8, shard=rank, n_shards=world_size)
    dist.barrier()


def render_ppm_shared(dist, rank: int, world_size: int, prepared, text: SharedText, depth: int = 5, samples: int = 0) -> int:
    """One frame's `Canvas::to_ppm` text written by world_size ranks of one node, rank r rendering shard r of `prepared`
    (a PreparedScene committed on one device): phase 1 into text.row_bytes, a barrier (every row's length is then in
    place), phase 2 into text.buf, a barrier.  Returns the text's length on every rank: text.text(length) is the frame's
    text.  The exchange is shared memory; torch.distributed only provides the barriers.  samples >= 1: the anti-aliased
    frame's text, render_samples_ppm(samples)'s."""
    prepared.render_shard_ppm_rows(rank, world_size, text.row_bytes, depth, samples=samples)
    dist.barrier()
    length = prepared.write_shard_ppm(rank, world_size, text.row_bytes, text.buf)
    dist.barrier()
    return length


def reduce_scalar(dist, value: float, op: str, device="cpu") -> float:
    import torch

    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return float(t.item())
