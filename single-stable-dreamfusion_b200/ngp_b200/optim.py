"""Adam + GradScaler over ONE flat parameter buffer, two launches per step (csrc/adam.cu, SURVEY.md 8f-1).

The reference's optimisation step is ``scaler.step(optimizer); scaler.update()`` on ``torch.optim.Adam(
model.get_params(lr), betas=(0.9, 0.99), eps=1e-15)`` with a ``LambdaLR(0.1 ** min(iter / iters, 1))`` schedule
(main.py:128-131, nerf/utils.py:708-713) - per parameter tensor an unscale kernel, an inf check, the Adam update and,
on the next forward, a fresh fp32 -> fp16 cast of the table (gridencoder/grid.py:38-39).  Here the parameters, their
gradients, both Adam moments and an fp16 shadow copy live in five flat buffers with the same layout:

    ngp_check_finite(grads)            -> state[found_inf]
    ngp_adam_step(params, grads, ...)  -> unscale, Adam, LambdaLR, GradScaler.update, fp16 shadow, zero the grads

``param.data`` / ``param.grad`` become views into the flat buffers, so autograd accumulates straight into the bucket
that the data-parallel all-reduce sends (parallel.py) and ``state_dict()`` keeps the reference's names and shapes.
All state (loss scale, growth tracker, step count) stays on the device: the step is CUDA-graph capturable.
"""
import ctypes
import math
import os

import torch

from . import _cabi, field

_ALIGN = 8  # elements: every tensor starts 16-byte aligned in the fp16 shadow (32 bytes in fp32)


class FusedAdamScaler:
    def __init__(self, param_groups, betas=(0.9, 0.99), eps=1e-15, init_scale=65536.0, growth_factor=2.0,
                 backoff_factor=0.5, growth_interval=2000, lr_decay=None, grad_div=1.0, peer_memory=None):
        """param_groups: [{'params': iterable, 'lr': float}, ...] as NeRFNetwork.get_params returns.
        lr_decay: None or (factor, iters) for lr * factor ** min(step / iters, 1).
        peer_memory: a parallel.PeerMemory (data parallel): the gradient bucket, the parameters and their fp16 shadow
        are then placed in memory that every rank of the group can address, and step() all-reduces the
        gradients itself over NVLink (csrc/adam.cu)."""
        groups = []
        for g in param_groups:
            ps = [p for p in g["params"] if p.requires_grad]
            if ps:
                groups.append((ps, float(g["lr"])))
        if not groups or len(groups) > 8:
            raise RuntimeError("1..8 non-empty parameter groups expected")
        self.params = [p for ps, _ in groups for p in ps]
        device = self.params[0].device
        _cabi.require_cuda(*self.params)
        self.device = device
        # layout: groups back to back, each tensor aligned
        self.offsets, seg_end, off = [], [], 0
        for ps, _ in groups:
            for p in ps:
                if p.dtype != torch.float32:
                    raise RuntimeError("fp32 master parameters expected")
                self.offsets.append(off)
                off += (p.numel() + _ALIGN - 1) // _ALIGN * _ALIGN
            seg_end.append(off)
        self.numel = off
        self.seg_end = (ctypes.c_uint64 * len(groups))(*seg_end)
        self.base_lrs = [lr for _, lr in groups]
        self.seg_lr = (ctypes.c_float * len(groups))(*self.base_lrs)
        self.n_seg = len(groups)
        f = lambda dt=torch.float32: torch.zeros(off, device=device, dtype=dt)  # noqa: E731
        self.exp_avg, self.exp_avg_sq = f(), f()
        self.peer = peer_memory
        self.peer_ptrs = None
        self.multicast = None
        # measured (profiles/dp_check_*): the switch-side reduction wins from 8 ranks on (64 vs 67 us per step), plain P2P
        # at 2 ranks (52 vs 64 us) - the multimem instructions cost latency and only pay once the fan-out is large
        env = os.environ.get("NGP_DP_MULTICAST", "auto")
        self.use_multicast = (peer_memory is not None and peer_memory.world > 4) if env == "auto" else env != "0"
        if os.environ.get("NGP_DP_BLOCKS"):
            _cabi.check(_cabi.load().ngp_dp_set_option(1, int(os.environ["NGP_DP_BLOCKS"])), "ngp_dp_set_option")
        if os.environ.get("NGP_DP_TIMEOUT_MS"):
            _cabi.check(_cabi.load().ngp_dp_set_option(0, int(os.environ["NGP_DP_TIMEOUT_MS"])), "ngp_dp_set_option")
        if peer_memory is None:
            self.flat_params, self.flat_grads, self.flat_half = f(), f(), f(torch.half)
        else:
            # one peer-addressable allocation: [grads f32 | params f32 | shadow f16 | barrier flags], 256-byte aligned parts
            lib = _cabi.load()
            al = lambda b: (b + 255) // 256 * 256  # noqa: E731
            o_g, o_p, o_h = 0, al(4 * off), al(4 * off) * 2
            o_f = o_h + al(2 * off)
            total = o_f + int(lib.ngp_dp_flags_bytes())
            raw, bases, mc_base = peer_memory.alloc(total)
            raw.zero_()
            self._peer_raw = raw
            self.flat_grads = raw[o_g:o_g + 4 * off].view(torch.float32)
            self.flat_params = raw[o_p:o_p + 4 * off].view(torch.float32)
            self.flat_half = raw[o_h:o_h + 2 * off].view(torch.half)
            mk = lambda o: (ctypes.c_uint64 * len(bases))(*[b + o for b in bases])  # noqa: E731
            self.peer_ptrs = (mk(o_g), mk(o_p), mk(o_h), mk(o_f))
            # NVLS multicast view of the same allocation (0 when the box has none): switch-side reduction / broadcast
            self.multicast = (ctypes.c_uint64 * 3)(mc_base + o_g, mc_base + o_p, mc_base + o_h) if mc_base else None
            peer_memory.barrier()  # every rank has zeroed its flags before anybody signals
        with torch.no_grad():
            for p, o in zip(self.params, self.offsets):
                view = self.flat_params[o:o + p.numel()].view_as(p)
                view.copy_(p)
                p.data = view
        self.attach_grads()
        self.flat_half.copy_(self.flat_params)
        for p, o in zip(self.params, self.offsets):
            field.register_half_shadow(p, self.flat_half[o:o + p.numel()].view_as(p))
        self._seen_versions = [p._version for p in self.params]
        self.betas, self.eps = betas, eps
        self.growth_factor, self.backoff_factor, self.growth_interval = growth_factor, backoff_factor, growth_interval
        self.grad_div = float(grad_div)
        self.set_lr_decay(lr_decay)
        # [scale, growth tracker, steps, found_inf, skipped, cross-GPU wait timed out, -, -]
        self.state = torch.tensor([init_scale, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0], device=device, dtype=torch.float32)
        self._blocks_done = torch.zeros(1, device=device, dtype=torch.int32)
        self._sync = torch.zeros(2, device=device, dtype=torch.int32)  # ngp_adam_step_dp: [block election, barrier epoch]

    # -- layout helpers ------------------------------------------------------------------------------------------
    def attach_grads(self):
        """(Re-)point every .grad at its slice of the flat gradient buffer."""
        for p, o in zip(self.params, self.offsets):
            if p.grad is None or p.grad.data_ptr() != self.flat_grads[o:].data_ptr():
                p.grad = self.flat_grads[o:o + p.numel()].view_as(p)

    def set_lr(self, lrs):
        self.base_lrs = [float(x) for x in lrs]
        self.seg_lr = (ctypes.c_float * self.n_seg)(*self.base_lrs)

    def set_lr_decay(self, lr_decay):
        if lr_decay is None:
            self.lr_decay_ln, self.lr_decay_steps = 0.0, 0.0
        else:
            factor, iters = lr_decay
            self.lr_decay_ln, self.lr_decay_steps = math.log(factor) / float(iters), float(iters)

    # -- GradScaler surface ----------------------------------------------------------------------------------------
    @property
    def scale_tensor(self):
        return self.state[0]

    def scale(self, loss):
        return loss * self.state[0]

    def get_scale(self):
        return float(self.state[0].item())

    @property
    def steps_taken(self):
        return int(self.state[2].item())

    def zero_grad(self):
        self.flat_grads.zero_()

    def step(self, zero_grads=True, deferred=False, fold=None):
        """scaler.step(optimizer) + scaler.update() (+ optimizer.zero_grad()): two plain launches, no host sync.
        ngp_check_finite sets found_inf, then ngp_adam_step applies the update - or, with peer memory, ngp_adam_step_dp
        all-reduces the gradients itself over NVLink on the way (reduce-scatter by P2P loads, Adam on this rank's slice,
        new parameters written to every replica; it always zero-fills the gradients).
        deferred: the launch only arms (state[6] = 1) when nothing is pending yet - see TrainStep(pipelined=True).
        fold: optional (grad_table view, odd-frame twin) of the split table scatter, added into the bucket inside the
        finite check."""
        dev = self.device
        if fold is not None:
            _cabi.call("ngp_check_finite_fold", dev, _cabi.ptr(self.flat_grads), self.numel, _cabi.ptr(fold[0]),
                       _cabi.ptr(fold[1]), fold[0].numel(), self.state[3:].data_ptr())
        else:
            _cabi.call("ngp_check_finite", dev, _cabi.ptr(self.flat_grads), self.numel, self.state[3:].data_ptr())
        args = (_cabi.ptr(self.flat_params), _cabi.ptr(self.flat_grads), _cabi.ptr(self.exp_avg), _cabi.ptr(self.exp_avg_sq),
                _cabi.ptr(self.flat_half), self.numel, self.n_seg, self.seg_end, self.seg_lr, float(self.betas[0]),
                float(self.betas[1]), float(self.eps), self.grad_div, self.lr_decay_ln, self.lr_decay_steps,
                float(self.growth_factor), float(self.backoff_factor), int(self.growth_interval))
        if self.peer is None or self.peer.world == 1:
            _cabi.call("ngp_adam_step", dev, *args, int(bool(zero_grads)) | (2 if deferred else 0), _cabi.ptr(self.state),
                       _cabi.ptr(self._blocks_done))
        else:
            mc = self.multicast if self.use_multicast else None
            _cabi.call("ngp_adam_step_dp", dev, *args, int(bool(deferred)), _cabi.ptr(self.state), _cabi.ptr(self._sync),
                       self.peer.rank, self.peer.world, *self.peer_ptrs, mc)

    def sync_shadow_if_changed(self):
        """Refresh the fp16 shadow if a parameter was edited through torch (load_state_dict, manual init) since the
        last look: such in-place edits land in the flat fp32 buffer and bump ``param._version``; the kernels read the
        shadow.  Host-side version compare, one copy kernel only when something changed."""
        versions = [p._version for p in self.params]
        if versions != self._seen_versions:
            with torch.no_grad():
                self.flat_half.copy_(self.flat_params)
            self._seen_versions = versions
            for p in self.params:       # keep field.cached_half's bookkeeping in step (same shadow tensors)
                s = field._shadows.get(id(p))
                if s is not None:
                    s[2][0] = p._version

    def grad_view(self, p):
        """The slice of the flat gradient bucket that backs `p.grad` (same shape as p)."""
        o = self.offsets[self._index(p)]
        return self.flat_grads[o:o + p.numel()].view_as(p)

    def half_view(self, p):
        """The maintained fp16 shadow of parameter `p`."""
        o = self.offsets[self._index(p)]
        return self.flat_half[o:o + p.numel()].view_as(p)

    def _index(self, p):
        for i, q in enumerate(self.params):
            if q is p:
                return i
        raise KeyError("parameter is not managed by this optimizer")

    @property
    def comm_error(self):
        """True if a cross-GPU wait inside step() ever timed out (one device->host read)."""
        return bool(self.state[5].item() != 0)

    # -- checkpointing (nerf/utils.py:847-968 saves optimizer / scaler state next to the model) ----------------------
    def state_dict(self):
        """Collective when the moments are sharded (fused data-parallel step): every rank must call it."""
        if self.peer_ptrs is not None:
            from .parallel import gather_owner_slices
            m, v = gather_owner_slices(self.exp_avg, self.peer.group), gather_owner_slices(self.exp_avg_sq, self.peer.group)
        else:
            m, v = self.exp_avg.clone(), self.exp_avg_sq.clone()
        return {"exp_avg": m, "exp_avg_sq": v, "state": self.state.clone(), "base_lrs": list(self.base_lrs),
                "offsets": list(self.offsets), "numel": self.numel}

    def load_state_dict(self, sd):
        if sd["numel"] != self.numel or list(sd["offsets"]) != list(self.offsets):
            raise RuntimeError("optimizer state does not match this parameter layout")
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        self.state.copy_(sd["state"])
        self.set_lr(sd["base_lrs"])
