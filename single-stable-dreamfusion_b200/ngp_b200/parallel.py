"""Data-parallel plumbing for the -O train step: one process per GPU, views sharded across ranks,
ONE all-reduce per step over a flat fp32 gradient bucket (hash-grid table + both MLPs = 1.8 M
floats, 7.3 MB at the cfg3 sizes), NCCL over NVLink/NVSwitch on GPUs, gloo on CPU for the tests.

The reference has no working multi-GPU path (a dormant DDP wrap, nerf/utils.py:200-202); DDP would
all-reduce exactly these parameters.  Parameter .grad tensors are views into the bucket, so autograd
accumulates straight into it and no flatten / unflatten copies are needed.
"""
import torch
import torch.distributed as dist


class FlatGradBucket:
    def __init__(self, params, device=None, extra=0):
        self.params = [p for p in params if p.requires_grad]
        n = sum(p.numel() for p in self.params)
        device = device if device is not None else self.params[0].device
        # `extra` trailing floats ride along in the same collective (e.g. an inf/nan flag, a sample count)
        self.flat = torch.zeros(n + extra, dtype=torch.float32, device=device)
        self.extra = self.flat[n:]
        off = 0
        for p in self.params:
            p.grad = self.flat[off:off + p.numel()].view_as(p)
            off += p.numel()
        self.numel = n

    def zero(self):
        self.flat.zero_()

    def attach(self):
        """Re-point .grad at the bucket (needed after optimizer.zero_grad(set_to_none=True))."""
        off = 0
        for p in self.params:
            if p.grad is None or p.grad.data_ptr() != self.flat[off:].data_ptr():
                p.grad = self.flat[off:off + p.numel()].view_as(p)
            off += p.numel()

    def all_reduce(self, average=True, async_op=False):
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return None
        work = dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, async_op=async_op)
        if average and not async_op:
            self.flat[:self.numel].div_(dist.get_world_size())
        return work


def shard_views(n_views, rank, world_size):
    """Contiguous, balanced split of `n_views` camera views; returns (first, count) for `rank`."""
    base, rem = divmod(n_views, world_size)
    count = base + (1 if rank < rem else 0)
    first = rank * base + min(rank, rem)
    return first, count


def shard_rows(n_rows, rank, world_size):
    """Row-interleaved split of an image: rank r renders rows r, r + world, ... of EVERY view, so each rank sees the
    same mix of dense and empty image regions (camera views differ 4x in marched samples; whole-view sharding would
    leave the step waiting for the rank that drew the densest view).  Returns the row indices of `rank`."""
    return list(range(rank, n_rows, world_size))


def shard_pixels(H, W, rank, world_size, tile=8):
    """Pixel indices (row-major ids, as a list) of `rank`'s share of an H x W view, in the order the rays are rendered:
    the image is cut into tile x tile blocks, block (ty, tx) belongs to rank (ty + tx) % world (one block per block-row
    and block-column for every rank: the same mix of object and background as the whole image), and the rays of a
    block are contiguous, so neighbouring rays - which touch the same coarse grid cells - are processed together.
    Falls back to interleaved rows when the tiling does not divide evenly."""
    ty_n, tx_n = H // tile, W // tile
    if H % tile or W % tile or (ty_n * tx_n) % world_size or tx_n % world_size:
        return [r * W + c for r in shard_rows(H, rank, world_size) for c in range(W)]
    out = []
    for ty in range(ty_n):
        for tx in range(tx_n):
            if (ty + tx) % world_size == rank:
                for y in range(tile):
                    base = (ty * tile + y) * W + tx * tile
                    out.extend(range(base, base + tile))
    return out


def owner_slice(numel, rank, world_size):
    """[lo, hi) element range of the flat optimizer buffers that `rank` owns in the fused data-parallel step: the
    partition csrc/adam.cu uses (float4 granularity, ceil(n4 / world) float4s per rank, the tail ranks may own less)."""
    n4 = numel // 4
    per = (n4 + world_size - 1) // world_size
    lo = min(per * rank, n4)
    hi = min(lo + per, n4)
    return 4 * lo, 4 * hi


def gather_owner_slices(flat, group=None):
    """Every rank holds the valid values of `flat` only inside its owner_slice (sharded Adam moments); returns the fully
    valid buffer on every rank (one all_gather of equal, padded chunks).  Works on any backend / device."""
    if not (dist.is_available() and dist.is_initialized()):
        return flat.clone()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if world == 1:
        return flat.clone()
    numel = flat.numel()
    per = 4 * ((numel // 4 + world - 1) // world)
    lo, hi = owner_slice(numel, rank, world)
    mine = torch.zeros(per, dtype=flat.dtype, device=flat.device)
    mine[:hi - lo] = flat[lo:hi]
    out = torch.empty(per * world, dtype=flat.dtype, device=flat.device)
    dist.all_gather_into_tensor(out, mine, group=group)
    return out[:numel].clone()


class PeerMemory:
    """Device memory that every rank of the group can address directly (loads / stores / atomics over NVLink).

    alloc(nbytes) -> (local uint8 tensor, [device address of that allocation on every rank, in rank order],
                      NVLS multicast address of the allocation or 0).
    The plumbing is PyTorch's symmetric memory (torch.distributed._symmetric_memory: cuMem allocations whose handles
    are exchanged through the group's store and mapped into every rank); kernels only ever see raw addresses
    (csrc/adam.cu).  Raises RuntimeError when the box cannot do it; callers then fall back to an NCCL all-reduce.
    """

    def __init__(self, device, group=None):
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("PeerMemory needs an initialised process group")
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        self.device = torch.device(device)
        self._keep = []
        self.used = None

    def alloc(self, nbytes):
        nbytes = (int(nbytes) + 255) // 256 * 256
        try:
            out, err = self._alloc_symm(nbytes), None
        except Exception as e:  # noqa: BLE001 - any failure means "not available on this box"
            out, err = None, repr(e)
        ok = torch.tensor([0.0 if out is None else 1.0], device=self.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)  # every rank takes the same path
        if ok.item() > 0:
            self.used = "symm"
            return out
        raise RuntimeError("no peer-addressable memory on this box: %s" % (err or "another rank failed"))

    def _alloc_symm(self, nbytes):
        import torch.distributed._symmetric_memory as symm
        t = symm.empty(nbytes, dtype=torch.uint8, device=self.device)
        hdl = symm.rendezvous(t, self.group)
        bases = [int(p) for p in hdl.buffer_ptrs]
        if len(bases) != self.world or bases[self.rank] != t.data_ptr():
            raise RuntimeError("unexpected symmetric-memory handle layout")
        self._keep.append((t, hdl))
        mc = 0
        try:
            mc = int(getattr(hdl, "multicast_ptr", 0) or 0)
        except Exception:  # noqa: BLE001 - no multicast on this box / torch build
            mc = 0
        return t, bases, mc

    def barrier(self):
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)
