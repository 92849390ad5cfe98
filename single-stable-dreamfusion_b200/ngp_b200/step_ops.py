"""One-launch versions of the small ops either side of the render (csrc/train_step.cu), as autograd Functions.

``blend_background`` is the tail of ``run_cuda`` (nerf/renderer.py:535-557: background blend, depth normalisation,
hit mask); ``entropy_loss`` is the opacity regulariser of ``Trainer.train_step`` (nerf/utils.py:389-394).  The
reference evaluates each as a chain of ~10 eager elementwise kernels forward and as many backward; at sub-millisecond
step times those launches are a visible share of the step, so each direction is a single kernel here.
"""
import torch
from torch.autograd import Function

from . import _cabi
from .field import cached_half


class _BlendBackground(Function):
    @staticmethod
    def forward(ctx, image, weights_sum, depth, bg, nears, fars):
        dev = image.device
        N = image.shape[0]
        per_ray = bg.dim() == 2
        image_out = torch.empty_like(image)
        depth_out = torch.empty_like(depth)
        mask = torch.empty(N, device=dev, dtype=torch.bool)
        _cabi.call("ngp_blend_background_forward", dev, _cabi.ptr(image), _cabi.ptr(weights_sum), _cabi.ptr(depth),
                   _cabi.ptr(bg), int(per_ray), _cabi.ptr(nears), _cabi.ptr(fars), N, _cabi.ptr(image_out),
                   _cabi.ptr(depth_out), _cabi.ptr(mask))
        ctx.save_for_backward(weights_sum, bg)
        ctx.per_ray = per_ray
        # composite_rays_train does not propagate grad_depth (raymarching.py:275), so depth carries no gradient
        ctx.mark_non_differentiable(depth_out, mask)
        return image_out, depth_out, mask

    @staticmethod
    def backward(ctx, g_image, _g_depth, _g_mask):
        weights_sum, bg = ctx.saved_tensors
        dev = weights_sum.device
        N = weights_sum.shape[0]
        g_image = g_image.contiguous().float()
        d_ws = torch.empty_like(weights_sum)
        d_bg = torch.empty(N, 3, device=dev, dtype=torch.float32) if (ctx.per_ray and ctx.needs_input_grad[3]) else None
        _cabi.call("ngp_blend_background_backward", dev, _cabi.ptr(g_image), _cabi.ptr(weights_sum), _cabi.ptr(bg),
                   int(ctx.per_ray), N, _cabi.ptr(d_ws), _cabi.ptr(d_bg))
        return g_image, d_ws, None, d_bg, None, None


def blend_background(image, weights_sum, depth, bg_color, nears, fars):
    """image [N,3], weights_sum [N], depth [N] (fp32, CUDA); bg_color: [N,3] tensor, [3] tensor or python scalar.
    Returns (image + (1 - weights_sum) * bg, clamp(depth - nears, 0) / (fars - nears), nears < fars)."""
    dev = image.device
    if not torch.is_tensor(bg_color):
        bg = torch.full((3,), float(bg_color), device=dev, dtype=torch.float32)
    else:
        bg = bg_color.to(device=dev, dtype=torch.float32)
        if bg.dim() == 0:
            bg = bg.expand(3)
        elif bg.dim() >= 2:
            bg = bg.reshape(-1, 3)
            if bg.shape[0] == 1:
                bg = bg[0]
            elif bg.shape[0] != image.shape[0]:
                raise RuntimeError("bg_color must be a colour or one colour per ray")
        bg = bg.contiguous()
    return _BlendBackground.apply(image.contiguous(), weights_sum.contiguous(), depth.contiguous(), bg, nears, fars)


class _EntropyLoss(Function):
    @staticmethod
    def forward(ctx, weights_sum, lam):
        ws = weights_sum.contiguous().view(-1)
        loss = torch.empty((), device=ws.device, dtype=torch.float32)
        _cabi.call("ngp_entropy_loss_forward", ws.device, _cabi.ptr(ws), ws.numel(), float(lam), _cabi.ptr(loss))
        ctx.save_for_backward(ws)
        ctx.lam, ctx.shape = float(lam), weights_sum.shape
        return loss

    @staticmethod
    def backward(ctx, g):
        (ws,) = ctx.saved_tensors
        d_ws = torch.empty_like(ws)
        g = g.contiguous().float()
        _cabi.call("ngp_entropy_loss_backward", ws.device, _cabi.ptr(ws), ws.numel(), ctx.lam, _cabi.ptr(g), _cabi.ptr(d_ws), 0)
        return d_ws.view(ctx.shape), None


def entropy_loss(weights_sum, lam=1e-4):
    """lam * mean binary entropy (base 2) of clamp(weights_sum, 1e-5, 1 - 1e-5)."""
    _cabi.require_cuda(weights_sum)
    return _EntropyLoss.apply(weights_sum.float(), lam)


class _BackgroundNet(Function):
    """FreqEncoder(6) -> Linear(39,64)+ReLU -> Linear(64,3) -> sigmoid under fp16 autocast, one launch each way."""

    @staticmethod
    def forward(ctx, dirs, w1, b1, w2, b2):
        dev = dirs.device
        N = dirs.shape[0]
        hw = [cached_half(t) for t in (w1, b1, w2, b2)]
        out = torch.empty(N, 3, device=dev, dtype=torch.half)
        _cabi.call("ngp_bg_forward", dev, _cabi.ptr(dirs), N, *[_cabi.ptr(t) for t in hw], 6, 64, _cabi.ptr(out))
        ctx.save_for_backward(dirs, *hw)
        return out

    @staticmethod
    def backward(ctx, g):
        dirs, w1h, b1h, w2h, b2h = ctx.saved_tensors
        dev = dirs.device
        g = g.contiguous().float()
        sizes = [64 * 39, 64, 3 * 64, 3]
        flat = torch.zeros(sum(sizes), device=dev, dtype=torch.float32)
        gw1, gb1, gw2, gb2 = torch.split(flat, sizes)
        _cabi.call("ngp_bg_backward", dev, _cabi.ptr(dirs), _cabi.ptr(g), dirs.shape[0], _cabi.ptr(w1h), _cabi.ptr(b1h),
                   _cabi.ptr(w2h), _cabi.ptr(b2h), 6, 64, _cabi.ptr(gw1), _cabi.ptr(gb1), _cabi.ptr(gw2), _cabi.ptr(gb2))
        return None, gw1.view(64, 39), gb1, gw2.view(3, 64), gb2


def can_fuse_background(d, encoder_bg, bg_net):
    try:
        return (d.is_cuda and d.dim() == 2 and d.shape[-1] == 3 and not d.requires_grad
                and torch.is_autocast_enabled('cuda') and torch.get_autocast_dtype('cuda') == torch.float16
                and encoder_bg.input_dim == 3 and encoder_bg.degree == 6 and bg_net.num_layers == 2
                and bg_net.dim_hidden == 64 and bg_net.dim_out == 3 and bg_net.net[0].bias is not None
                and bg_net.net[0].weight.dtype == torch.float32)
    except AttributeError:
        return False


def background_net(d, bg_net):
    """sigmoid(bg_net(freq_encode(d))) as a half tensor [N,3] (what NeRFNetwork.background returns under autocast)."""
    l0, l1 = bg_net.net
    return _BackgroundNet.apply(d.contiguous().float(), l0.weight, l0.bias, l1.weight, l1.bias)


# ---------------------------------------------------------------------------------------------------------------------
# Shading stencil (csrc/shading.cu; nerf/network_grid.py:90-144): the K stencil points of a sample are K consecutive rows
# of one field batch; these ops build the points and turn the K densities into normal / colour, forward and backward.
# ---------------------------------------------------------------------------------------------------------------------
SHADING_MODES = {"lambertian": 0, "textureless": 1, "normal": 2}


def stencil_points(x, eps, bound, with_centre=True):
    """x [M,3] -> [M*K, 3] rows (K = 7: x, x+eps e_x, x-eps e_x, x+eps e_y, ...; K = 6 without the centre), every shifted
    point clamped to [-bound, bound] as network_grid.py:93-98 does.  No gradient flows to x (the reference's xyzs carry none)."""
    _cabi.require_cuda(x)
    x = x.detach().contiguous().float()
    M = x.shape[0]
    K = 7 if with_centre else 6
    out = torch.empty(M * K, 3, device=x.device, dtype=torch.float32)
    _cabi.call("ngp_stencil_points", x.device, _cabi.ptr(x), M, None, float(eps), float(bound), int(with_centre), _cabi.ptr(out),
               None)
    return out


class _Shade(Function):
    @staticmethod
    def forward(ctx, sigma_all, rgb_all, K, light, ratio, mode):
        dev = sigma_all.device
        sigma_all = sigma_all.contiguous().float()
        M = sigma_all.shape[0] // K
        want_color = mode is not None
        rgb_c = rgb_all.contiguous().float() if (want_color and rgb_all is not None) else None
        light_c = light.detach().contiguous().float() if light is not None else None
        normal = torch.empty(M, 3, device=dev, dtype=torch.float32)
        color = torch.empty(M, 3, device=dev, dtype=torch.float32) if want_color else None
        _cabi.call("ngp_shade_forward", dev, _cabi.ptr(sigma_all), _cabi.ptr(rgb_c), M, K, _cabi.ptr(light_c), float(ratio),
                   int(mode or 0), _cabi.ptr(normal), _cabi.ptr(color))
        ctx.save_for_backward(sigma_all, rgb_c, light_c)
        ctx.meta = (M, K, float(ratio), mode, bool(ctx.needs_input_grad[1]))
        if want_color:
            return normal, color
        return normal

    @staticmethod
    def backward(ctx, d_normal, d_color=None):
        sigma_all, rgb_c, light_c = ctx.saved_tensors
        M, K, ratio, mode, need_rgb = ctx.meta
        dev = sigma_all.device
        d_normal = d_normal.contiguous().float() if d_normal is not None else None
        d_color = d_color.contiguous().float() if (d_color is not None and mode is not None) else None
        d_sigma = torch.empty(M * K, device=dev, dtype=torch.float32)
        d_rgb = torch.empty(M * K, 3, device=dev, dtype=torch.float32) if (need_rgb and mode == 0 and d_color is not None) else None
        _cabi.call("ngp_shade_backward", dev, _cabi.ptr(sigma_all), _cabi.ptr(rgb_c), M, K, _cabi.ptr(light_c), ratio, int(mode or 0),
                   _cabi.ptr(d_normal), _cabi.ptr(d_color), _cabi.ptr(d_sigma), _cabi.ptr(d_rgb))
        return d_sigma, d_rgb, None, None, None, None


def shade(sigma_all, rgb_all, light, ratio, shading):
    """sigma_all [7M] / rgb_all [7M,3] of stencil_points(x, with_centre=True) -> (normal [M,3] fp32, color [M,3] fp32 holding
    the reference's half values) for shading in {'lambertian', 'textureless', 'normal'} (network_grid.py:126-140)."""
    return _Shade.apply(sigma_all, rgb_all, 7, light, ratio, SHADING_MODES[shading])


def stencil_normal(sigma6):
    """sigma6 [6M] of stencil_points(x, with_centre=False) -> NeRFNetwork.normal(x) [M,3] (network_grid.py:108-114)."""
    return _Shade.apply(sigma6, None, 6, None, 1.0, None)
