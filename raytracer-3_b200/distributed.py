"""Frame-end gather for the row-tile partition (one process per GPU, torch.distributed plumbing).

Rendering needs no collective: tiles of ``tile_rows`` rows are dealt round-robin to the ranks
(the reference's own hook for this is the unused BlockInfo{x,y,w,h} uniform,
src/lib/shaders/raytracer/raytracer_v4.glsl:70-79) and every rank renders its tiles from a
replicated scene. Only the packed uint32 pixels travel, once per frame: each rank packs its
rows into a compact slab (padded to the largest slab so a plain gather works), rank 0 gathers
over NCCL (gloo in the CPU tests) and de-interleaves.

``SharedFrame`` removes that gather on a node with NVLink: rank 0's frame is mapped into every
other rank (CUDA IPC, include/rt3cuda.h rt3_frame_*), each rank's render kernels store their
rows straight into it (frames use full-frame indexing), and the frame end is one stream-ordered
barrier.
"""
import numpy as np
import torch


def owned_rows(height, tile_rows, part_index, part_count):
    """Global row indices rank ``part_index`` renders, top to bottom (== rt3_partition_rows ordering)."""
    rows = np.arange(height)
    return rows[(rows // max(tile_rows, 1)) % max(part_count, 1) == part_index]


def max_owned_rows(height, tile_rows, part_count):
    return max(len(owned_rows(height, tile_rows, r, part_count)) for r in range(part_count))


def pack_rows(frame, width, height, tile_rows, part_index, part_count, out=None):
    """Host/torch restatement of rt3_pack_partition: frame [H*W] -> slab [max_rows*W] (zero padded)."""
    rows = torch.as_tensor(owned_rows(height, tile_rows, part_index, part_count), device=frame.device)
    n = max_owned_rows(height, tile_rows, part_count) * width
    slab = out if out is not None else torch.zeros(n, dtype=frame.dtype, device=frame.device)
    slab[: len(rows) * width] = frame.view(height, width)[rows].reshape(-1)
    return slab


def unpack_rows(slab, frame, width, height, tile_rows, part_index, part_count):
    """Host/torch restatement of rt3_unpack_partition: slab -> the owner's rows of frame."""
    rows = torch.as_tensor(owned_rows(height, tile_rows, part_index, part_count), device=frame.device)
    frame.view(height, width)[rows] = slab[: len(rows) * width].view(len(rows), width)
    return frame


def gather_slabs(dist, slab, rank, world, dst=0):
    """Gathers every rank's (equal-sized) slab onto ``dst``; returns the list there, None elsewhere."""
    if world == 1:
        return [slab]
    bucket = [torch.empty_like(slab) for _ in range(world)] if rank == dst else None
    dist.gather(slab, bucket, dst=dst)
    return bucket


class _DevicePointer:
    """Lets torch view memory the render core allocated (``__cuda_array_interface__``, int32 words)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False), "version": 2}


class SharedFrame:
    """One frame in rank ``owner``'s HBM that every rank of the node renders into.

    ``ptr`` is what each rank passes to ``Context.render_device`` as the frame (the owner's own
    allocation there, the IPC mapping elsewhere); ``tensor`` is the owner's torch view of it
    (None on the other ranks). ``finish()`` is the frame-end barrier: an all-reduce of one
    element on the current stream, after which the owner's stream has every rank's pixels.
    Construction and ``close()`` are collective. If any rank cannot map the frame (no peer access
    between two GPUs, IPC unavailable), ``ok`` is False on every rank and ``error`` says why: the
    caller then closes it and gathers with NCCL instead.

    ``n_pixels`` counts 32-bit words, so the same class shares the stage of a frame denoised in parts:
    ``SharedFrame(ctx, dist, abi.denoise_stage_words(w, h), rank, world, device)``. Each rank then calls
    ``ctx.denoise_stage(w, h, shared.ptr, tag)`` and ``ctx.stats()`` (which waits for its stores), all ranks meet in a
    barrier that holds the host (``dist.barrier()``; ``finish()`` only orders torch's stream, not the library's), and the
    owner calls ``ctx.denoise_staged(w, h, shared.ptr, tag)``, or ``ctx.denoise_staged_temporal(w, h, shared.ptr, tag)`` to
    accumulate the frames of a sequence in the owner's history (the other ranks stage exactly as before and keep none; every
    rank uploads a new scene when the owner does).
    """

    def __init__(self, ctx, dist, n_pixels, rank, world, device, owner=0):
        self.ctx, self.dist, self.rank, self.world, self.owner = ctx, dist, rank, world, owner
        self.ptr, self.tensor, self._mapped, self.error = None, None, False, None
        handle = [None]
        if rank == owner:
            try:
                self.ptr = ctx.frame_alloc(n_pixels)
                self.tensor = torch.as_tensor(_DevicePointer(self.ptr, n_pixels), device=device)
                handle[0] = ctx.frame_export(self.ptr) if world > 1 else None
            except Exception as e:  # reported below, after the collectives every rank takes part in
                self.error = e
        if world > 1:
            dist.broadcast_object_list(handle, src=owner)
            if rank != owner:
                try:
                    if handle[0] is None:
                        raise RuntimeError(f"rank {owner} could not export its frame")
                    self.ptr = ctx.frame_import(handle[0])
                    self._mapped = True
                except Exception as e:
                    self.error = e
            self._token = torch.zeros(1, dtype=torch.int32, device=device)
            # all ranks agree on whether the mapping exists everywhere
            bad = torch.tensor([1 if self.error is not None else 0], dtype=torch.int32, device=device)
            dist.all_reduce(bad)
            if int(bad.item()) and self.error is None:
                self.error = RuntimeError("another rank could not map the shared frame")
        self.ok = self.error is None

    def finish(self):
        if self.world > 1:
            self.dist.all_reduce(self._token)

    def close(self):
        """Unmaps on the importing ranks, then frees on the owner (collective: every rank calls it)."""
        if self._mapped:
            self.ctx.frame_release(self.ptr)
            self._mapped = False
            self.ptr = None
        if self.world > 1:
            self.dist.barrier()
        if self.rank == self.owner and self.ptr is not None:
            self.tensor = None
            self.ctx.frame_free(self.ptr)
        self.ptr = None
