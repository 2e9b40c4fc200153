"""Ensemble sharding over the GPUs of one box (new relative to the reference, which has no
ensemble or multi-device code: SURVEY section 0.2, 8e).

Members are independent, so the solver loop needs no exchange step: member b goes to rank
b mod G (interleaved, so any smooth dependence of step count on the initial value spreads
evenly), every rank runs its persistent kernel on its shard, and ONE all-gather over
NCCL/NVLink collects checkpoint means, standard deviations and step statistics.

One collective, no copy passes: a rank's result tensors (u | u_std | n_accepted | n_rejected |
status) are VIEWS into one packed byte buffer that the smoothing kernel writes directly
(`PackedResults.local`), `all_gather_into_tensor` moves that buffer once, and the gathered results
are exposed as strided views `[i][rank]` of the gathered buffer -- flattening the first two axes of
such a view is member order b = i * G + rank, so nothing is padded, concatenated or permuted.
"""

import numpy as np

_FIELDS = (  # name, dtype name, trailing shape as a function of (K, d)
    ("u", "float64", lambda K, d: (K, d)),
    ("u_std", "float64", lambda K, d: (K, d)),
    ("n_accepted", "int64", lambda K, d: (K,)),
    ("n_rejected", "int64", lambda K, d: ()),
    ("status", "int32", lambda K, d: ()),
)


def shard_indices(B, rank, world_size):
    """Interleaved member assignment: rank r owns members r, r+G, r+2G, ..."""
    return np.arange(rank, B, world_size)


def shard_grid(save_at, rank, world_size):
    """This rank's checkpoint grid: a grid shared by all members ([K]) as it is, and of a per-member grid ([B, K],
    numpy or torch) the rows that go with the rank's members: rows r, r+G, r+2G, ..."""
    return save_at if save_at.ndim == 1 else save_at[rank::world_size]


def shard_sizes(B, world_size):
    return [(B - r + world_size - 1) // world_size for r in range(world_size)]


def unshard_order(B, world_size):
    """Permutation that maps rank-major concatenated shards back to member order."""
    order = np.concatenate([shard_indices(B, r, world_size) for r in range(world_size)])
    inv = np.empty(B, dtype=np.int64)
    inv[order] = np.arange(B)
    return inv


class PackedResults:
    """The result buffers of one rank's shard as views into ONE byte buffer.

    `capacity` = members the buffer has room for = the largest shard, identical on every rank, so
    that the gathered buffer is a regular [G][capacity] array; a rank whose shard is one member
    short simply leaves its last row unused."""

    def __init__(self, B_total, K, d, world_size, device):
        import torch

        self.B_total, self.K, self.d, self.world = int(B_total), int(K), int(d), int(world_size)
        self.capacity = max(shard_sizes(self.B_total, self.world)) if self.B_total else 0
        self.layout = []  # (name, dtype, shape, byte offset, byte length)
        off = 0
        for name, dt, shp in _FIELDS:
            dtype = getattr(torch, dt)
            shape = (self.capacity,) + tuple(shp(self.K, self.d))
            nbytes = int(np.prod(shape, dtype=np.int64)) * torch.empty((), dtype=dtype).element_size()
            self.layout.append((name, dtype, shape, off, nbytes))
            off += (nbytes + 255) // 256 * 256  # keep every field 256-byte aligned
        self.nbytes = off
        self.device = device
        self.buffer = torch.zeros(self.nbytes, dtype=torch.uint8, device=device)
        self._gathered = None

    def _views(self, buf, lead):
        out = {}
        for name, dtype, shape, off, nbytes in self.layout:
            flat = buf[..., off : off + nbytes].view(dtype)
            out[name] = flat.reshape(tuple(lead) + shape)
        return out

    def local(self, n_local=None):
        """Tensors for `_cabi.solve_device(..., out=...)`: the first n_local rows of every field."""
        views = self._views(self.buffer, ())
        if n_local is not None and n_local != self.capacity:
            views = {k: v[:n_local] for k, v in views.items()}
        return views

    def all_gather(self, group=None):
        """ONE all_gather_into_tensor of the packed buffer; returns member-ordered strided views.

        out[name][i, r] is member b = i * G + r (valid while b < B_total); `member_order(out[name])`
        gives the flat [B_total, ...] tensor when a contiguous copy is wanted."""
        import torch
        import torch.distributed as dist

        if self._gathered is None:
            self._gathered = torch.empty((self.world, self.nbytes), dtype=torch.uint8, device=self.device)
        dist.all_gather_into_tensor(self._gathered.view(-1), self.buffer, group=group)
        per_rank = self._views(self._gathered, (self.world,))  # [G][capacity][...]
        return {k: v.transpose(0, 1) for k, v in per_rank.items()}  # [capacity][G][...] views, no copy

    def member_order(self, view):
        """Flatten a gathered [capacity][G][...] view to [B_total, ...] (this one does copy)."""
        return view.reshape((self.capacity * self.world,) + tuple(view.shape[2:]))[: self.B_total]


def all_gather_results(local, B, group=None):
    """All-gather a dict of per-member tensors (leading axis = this rank's members r, r+G, ...) and
    return them in member order.  Convenience wrapper over `PackedResults` for results that were not
    produced in a packed buffer: one packing copy, ONE collective.  Works with NCCL (CUDA tensors) and
    gloo (CPU tensors)."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    cap = max(shard_sizes(B, world)) if B else 0
    any_x = next(iter(local.values()))
    layout, off = [], 0
    for key, x in local.items():
        per = int(np.prod(x.shape[1:], dtype=np.int64)) * x.element_size()
        layout.append((key, x.dtype, tuple(x.shape[1:]), off, cap * per))
        off += (cap * per + 255) // 256 * 256
    buf = torch.zeros(off, dtype=torch.uint8, device=any_x.device)
    for (key, dtype, shp, o, nb), x in zip(layout, local.values()):
        dst = buf[o : o + nb].view(dtype).reshape((cap,) + shp)
        dst[: x.shape[0]].copy_(x)
    gathered = torch.empty((world, off), dtype=torch.uint8, device=any_x.device)
    dist.all_gather_into_tensor(gathered.view(-1), buf, group=group)
    out = {}
    for key, dtype, shp, o, nb in layout:
        per_rank = gathered[:, o : o + nb].view(dtype).reshape((world, cap) + shp)
        out[key] = per_rank.transpose(0, 1).reshape((cap * world,) + shp)[:B]
    return out
