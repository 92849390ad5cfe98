"""Sync-free training render: march -> fused field -> composite as ONE autograd Function over fixed-capacity
buffers, so a whole train step has static shapes, no device->host read and can be captured in a CUDA graph.

The reference's training branch of ``run_cuda`` (nerf/renderer.py:468-482) zero-fills N*max_steps rows, reads
the sample count back to the host to slice (raymarching.py:224) and flushes the allocator every step.  Here
the sample buffers are allocated once at their worst-case capacity (N * max_steps rows - a B200 has the HBM for
it), every kernel takes the device-side count written by the marcher, and nothing is sliced: rows past the
count are simply never touched.  Outputs (weights_sum, depth, image) and gradients are the same numbers the
modular path produces (same kernels).
"""
import numpy as np
import torch
from torch.autograd import Function

from . import _cabi
from .field import cached_half

_BYTES_PER_ROW = 12 + 8 + 4 + 12 + 64 + 128 + 128 + 4 + 12 + 64  # xyzs deltas sigma rgb enc h1 h2 d_sigma d_rgb d_enc
# Shaded steps of the hand-scheduled train step (trainer.py) also keep the 7 stencil rows of every sample (centre + six
# shifted points, csrc/shading.cu) and the per-sample ray direction (orientation regulariser):
#   extra bytes = 7 * cap * _STENCIL_BYTES_PER_ROW + 12 * cap,   cap = round_up(n_rays * max_steps, 128)
# e.g. one 64x64 view (4096 rays) at max_steps 1024: cap = 4 194 304 rows -> 12.6 GB of stencil rows (+ 50 MB of directions)
# on top of cap * _BYTES_PER_ROW = 1.8 GB of per-sample rows; 8 views: about 100 GB.
_STENCIL_BYTES_PER_ROW = 12 + 4 + 12 + 64 + 128 + 128 + 4 + 12 + 64  # xyzs sigma rgb enc h1 h2 d_sigma d_rgb d_enc


class StencilRows:
    """The field batch of a shaded step: 7 rows per sample (ngp_stencil_points), with the field's saved activations and
    gradients; counter[0] = 7 x the chain's sample count, written on the device by ngp_stencil_points."""

    def __init__(self, cap, device):
        rows = 7 * cap
        f32, f16 = torch.float32, torch.half
        e = lambda *shape, dtype=f32: torch.empty(*shape, device=device, dtype=dtype)  # noqa: E731
        self.cap = rows
        self.xyzs, self.sigma, self.rgb = e(rows, 3), e(rows), e(rows, 3)
        self.enc, self.h1, self.h2 = e(rows, 32, dtype=f16), e(rows, 64, dtype=f16), e(rows, 64, dtype=f16)
        self.d_sigma, self.d_rgb, self.d_enc = e(rows), e(rows, 3), e(rows, 32, dtype=f16)
        self.counter = torch.zeros(2, device=device, dtype=torch.int32)


class TrainWorkspace:
    """Static per-(N, max_steps) buffers of the training render."""

    def __init__(self, n_rays, max_steps, device, counter=None, shaded=False):
        # always the worst case (every ray emits max_steps samples): the marcher can then never overflow, so no ray is
        # ever dropped and rows >= counter[0] are never read
        cap = n_rays * max_steps
        cap = (cap + 127) // 128 * 128  # the field kernels save / restore whole 128-sample tiles
        self.n_rays, self.max_steps, self.cap = n_rays, max_steps, cap
        f32, f16 = torch.float32, torch.half
        e = lambda *shape, dtype=f32: torch.empty(*shape, device=device, dtype=dtype)  # noqa: E731
        self.xyzs, self.deltas = e(cap, 3), e(cap, 2)
        self.sigma, self.rgb = e(cap), e(cap, 3)
        self.enc, self.h1, self.h2 = e(cap, 32, dtype=f16), e(cap, 64, dtype=f16), e(cap, 64, dtype=f16)
        self.d_sigma, self.d_rgb, self.d_enc = e(cap), e(cap, 3), e(cap, 32, dtype=f16)
        self.rays = torch.empty(n_rays, 3, device=device, dtype=torch.int32)
        self._device = device
        self._march_ws = None
        self.counter = torch.zeros(2, device=device, dtype=torch.int32) if counter is None else counter
        # shaded steps: per-sample ray directions (written by the marcher) and the stencil rows
        self.dirs = e(cap, 3) if shaded else None
        self.stencil = StencilRows(cap, device) if shaded else None

    @property
    def march_ws(self):
        """Scratch of the ray-ordered marcher (per-ray slabs, 20 bytes x n_rays x max_steps): allocated on first use - the
        packed marcher of the hand-scheduled step (ngp_march_rays_train_packed) needs none."""
        if self._march_ws is None:
            lib = _cabi.load()
            self._march_ws = torch.empty(int(lib.ngp_march_rays_train_workspace(self.n_rays, int(self.max_steps))),
                                         device=self._device, dtype=torch.uint8)
            self._march_ws[:256].zero_()   # block-election word: zero once, every call leaves it zero (include/ngp_b200.h)
        return self._march_ws

    @property
    def nbytes(self):
        extra = 0 if self.stencil is None else 7 * self.cap * _STENCIL_BYTES_PER_ROW + 12 * self.cap
        return self.cap * _BYTES_PER_ROW + extra


class _RenderTrain(Function):
    @staticmethod
    def forward(ctx, rays_o, rays_d, nears, fars, noises, embeddings, w1, b1, w2, b2, w3, b3, ws, cfg):
        dev = rays_o.device
        N = rays_o.shape[0]
        enc = cfg["encoder"]
        L = enc.offsets.shape[0] - 1
        S = float(np.log2(enc.per_level_scale))
        table = cached_half(embeddings)
        hw = [cached_half(t) for t in (w1, b1, w2, b2, w3, b3)]
        ws.counter.zero_()
        # march: count -> ray-ordered exclusive scan -> write (device-side total in ws.counter[0])
        _cabi.call("ngp_march_rays_train", dev, _cabi.ptr(rays_o), _cabi.ptr(rays_d), _cabi.ptr(cfg["bitfield"]),
                   float(cfg["bound"]), float(cfg["dt_gamma"]), int(cfg["max_steps"]), N, int(cfg["cascade"]),
                   int(cfg["grid_size"]), ws.cap, _cabi.ptr(nears), _cabi.ptr(fars), _cabi.ptr(ws.xyzs), None,
                   _cabi.ptr(ws.deltas), _cabi.ptr(ws.rays), _cabi.ptr(ws.counter), _cabi.ptr(noises), _cabi.ptr(ws.march_ws),
                   ws.march_ws.numel())
        _cabi.call("ngp_field_forward", dev, _cabi.ptr(ws.xyzs), ws.cap, _cabi.ptr(ws.counter), _cabi.ptr(table),
                   _cabi.ptr(enc.offsets), L, 2, S, int(enc.base_resolution), int(enc.gridtype_id), int(bool(enc.align_corners)),
                   float(cfg["bound"]), *[_cabi.ptr(t) for t in hw], 64, 4, _cabi.ptr(ws.sigma), _cabi.ptr(ws.rgb),
                   _cabi.ptr(ws.enc), _cabi.ptr(ws.h1), _cabi.ptr(ws.h2))
        weights_sum = torch.empty(N, device=dev, dtype=torch.float32)
        depth = torch.empty(N, device=dev, dtype=torch.float32)
        image = torch.empty(N, 3, device=dev, dtype=torch.float32)
        _cabi.call("ngp_composite_rays_train_forward", dev, _cabi.ptr(ws.sigma), _cabi.ptr(ws.rgb), _cabi.ptr(ws.deltas),
                   _cabi.ptr(ws.rays), ws.cap, N, float(cfg["T_thresh"]), _cabi.ptr(weights_sum), _cabi.ptr(depth),
                   _cabi.ptr(image))
        ctx.save_for_backward(weights_sum, image, hw[0], hw[2], hw[4])
        ctx.ws, ctx.cfg, ctx.meta = ws, cfg, (N, L, S, embeddings.shape, embeddings.dtype)
        ctx.mark_non_differentiable(depth)  # the reference does not propagate grad_depth either (raymarching.py:275)
        return weights_sum, depth, image

    @staticmethod
    def backward(ctx, g_ws, g_depth, g_image):
        weights_sum, image, w1h, w2h, w3h = ctx.saved_tensors
        ws, cfg = ctx.ws, ctx.cfg
        N, L, S, emb_shape, emb_dtype = ctx.meta
        enc = cfg["encoder"]
        dev = weights_sum.device
        g_ws = torch.zeros_like(weights_sum) if g_ws is None else g_ws.contiguous().float()
        g_image = torch.zeros_like(image) if g_image is None else g_image.contiguous().float()
        _cabi.call("ngp_composite_rays_train_backward", dev, _cabi.ptr(g_ws), _cabi.ptr(g_image), _cabi.ptr(ws.sigma),
                   _cabi.ptr(ws.rgb), _cabi.ptr(ws.deltas), _cabi.ptr(ws.rays), _cabi.ptr(weights_sum), _cabi.ptr(image),
                   ws.cap, N, float(cfg["T_thresh"]), _cabi.ptr(ws.d_sigma), _cabi.ptr(ws.d_rgb))
        sizes = [64 * 32, 64, 64 * 64, 64, 4 * 64, 4]
        flat = torch.zeros(sum(sizes), device=dev, dtype=torch.float32)
        gw1, gb1, gw2, gb2, gw3, gb3 = torch.split(flat, sizes)
        _cabi.call("ngp_field_backward", dev, ws.cap, _cabi.ptr(ws.counter), _cabi.ptr(w1h), _cabi.ptr(w2h), _cabi.ptr(w3h),
                   64, 4, _cabi.ptr(ws.d_sigma), _cabi.ptr(ws.d_rgb), _cabi.ptr(ws.sigma), _cabi.ptr(ws.rgb), _cabi.ptr(ws.enc),
                   _cabi.ptr(ws.h1), _cabi.ptr(ws.h2), _cabi.ptr(ws.d_enc), _cabi.ptr(gw1), _cabi.ptr(gb1), _cabi.ptr(gw2),
                   _cabi.ptr(gb2), _cabi.ptr(gw3), _cabi.ptr(gb3))
        grad_table = torch.zeros(emb_shape, device=dev, dtype=torch.float32)
        _cabi.call("ngp_grid_scatter_samples", dev, _cabi.ptr(ws.d_enc), _cabi.ptr(ws.xyzs), float(cfg["bound"]),
                   _cabi.ptr(ws.counter), ws.cap, _cabi.ptr(enc.offsets), L, 2, S, int(enc.base_resolution),
                   int(enc.gridtype_id), int(bool(enc.align_corners)), _cabi.ptr(grad_table))
        if grad_table.dtype != emb_dtype:
            grad_table = grad_table.to(emb_dtype)
        return (None, None, None, None, None, grad_table, gw1.view(64, 32), gb1, gw2.view(64, 64), gb2, gw3.view(4, 64), gb3,
                None, None)


def render_train(model, rays_o, rays_d, nears, fars, noises, dt_gamma, max_steps, T_thresh):
    """weights_sum [N], depth [N], image [N,3] (before the background blend) for the training branch of run_cuda,
    albedo shading.  Leaves the sample count of this call in model._train_ws.counter[0] (device)."""
    N = rays_o.shape[0]
    ws = getattr(model, "_train_ws", None)
    if ws is None or ws.n_rays != N or ws.max_steps != max_steps or ws.xyzs.device != rays_o.device:
        ws = TrainWorkspace(N, max_steps, rays_o.device)
        model._train_ws = ws
    cfg = dict(encoder=model.encoder, bitfield=model.density_bitfield, bound=model.bound, dt_gamma=dt_gamma,
               max_steps=max_steps, cascade=model.cascade, grid_size=model.grid_size, T_thresh=T_thresh)
    l0, l1, l2 = model.sigma_net.net
    return _RenderTrain.apply(rays_o, rays_d, nears, fars, noises, model.encoder.embeddings, l0.weight, l0.bias, l1.weight,
                              l1.bias, l2.weight, l2.bias, ws, cfg)
