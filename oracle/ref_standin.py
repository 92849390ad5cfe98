"""TEST INFRASTRUCTURE: the C oracle behind the calling convention of the reference's CUDA extensions.

``load()`` returns a namespace with ``.grid``, ``.march`` and ``.freq`` whose functions take the same arguments as the
reference's pybind entry points (gridencoder.h:12-13, raymarching.h:7-17, freqencoder.h:7,10): device tensors in, results
written into the caller's output tensors.  Each call copies its inputs to the host, runs ``oracle.py`` and copies the
results back, except for the two whose device intrinsics a host cannot reproduce: the frequency encoder's forward
(oracle/ref_freq.cu, fast-math sinf) and the inference composite (oracle/ref_raymarching.cu, __expf) run on the device.
Tests use it in place of ``ref_ext.load()`` when the reference's extensions are not built.  tests/test_golden.py pins the
host oracle and ref_freq.cu to stored outputs of those extensions; no stored output of the reference's inference composite
exists, so ref_raymarching.cu is a transcription checked only against the host oracle (within the expf / __expf
difference), and bit-equality with it does not prove bit-equality with the reference.

Where the reference is nondeterministic the oracle takes one of its admissible outcomes: ``march_rays_train`` writes its
rows in ray order (the reference in completion order), and the table gradient is accumulated in the table's dtype in sample
order (the reference adds with atomics in arbitrary order).
"""
import ctypes
import os
import types

import numpy as np
import torch

from . import build as _build
from . import oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "ref_golden.npz")
_scales = {}
_dev_lib = None


def _np(t):
    return t.detach().cpu().numpy()


def _put(dst, a):
    dst.copy_(torch.from_numpy(np.ascontiguousarray(a)).reshape(dst.shape))


def _level_scales(L, S, H):
    """The reference's per-level scales fma(exp2f(level * S), H, -1) as its device computes them (MUFU.EX2, up to 2 ulp
    from libm): the stored reference values when (L, S, H) is the configuration they were recorded for."""
    key = (L, np.float32(S).item(), H)
    if key not in _scales:
        want = np.load(GOLDEN)["grid_scales"]
        libm, _ = O.grid_level_params(L, np.float32(S), H)
        ulps = np.abs(want.view(np.int32).astype(np.int64) - libm.view(np.int32).astype(np.int64)) if want.shape == libm.shape else None
        if ulps is None or ulps.max() > 4:
            raise RuntimeError("no stored reference level scales for L=%d S=%r H=%d" % key)
        _scales[key] = want
    return _scales[key]


def _grid_encode_forward(inputs, embeddings, offsets, outputs, B, D, C, L, S, H, dy_dx, gridtype, align_corners):
    out, dydx = O.grid_encode_forward(_np(inputs), _np(embeddings), _np(offsets), np.float32(S), H, calc_dydx=dy_dx is not None,
                                      gridtype=gridtype, align_corners=align_corners, out_layout=O.LBC,
                                      scale_override=_level_scales(L, S, H))
    _put(outputs, out)
    if dy_dx is not None:
        _put(dy_dx, dydx)


def _grid_encode_backward(grad, inputs, embeddings, offsets, grad_embeddings, B, D, C, L, S, H, dy_dx, grad_inputs, gridtype,
                          align_corners):
    g = _np(grad)
    table = O.grid_encode_backward(g, _np(inputs), _np(offsets), embeddings.shape[0], C, np.float32(S), H, gridtype=gridtype,
                                   align_corners=align_corners, grad_layout=O.LBC, round_addend_to_half=g.dtype == np.float16,
                                   scale_override=_level_scales(L, S, H),
                                   accumulate="f16" if embeddings.dtype == torch.float16 else "f32")
    grad_embeddings.copy_(torch.from_numpy(table).to(grad_embeddings.dtype))
    if dy_dx is not None and grad_inputs is not None:
        _put(grad_inputs, O.grid_input_backward(g, _np(dy_dx), B, D, C, L, grad_layout=O.LBC))


def _near_far_from_aabb(rays_o, rays_d, aabb, N, min_near, nears, fars):
    n, f = O.near_far_from_aabb(_np(rays_o), _np(rays_d), _np(aabb), min_near)
    _put(nears, n)
    _put(fars, f)


def _sph_from_ray(rays_o, rays_d, radius, N, coords):
    _put(coords, O.sph_from_ray(_np(rays_o), _np(rays_d), radius))


def _morton3D(coords, N, indices):
    _put(indices, O.morton3D(_np(coords)))


def _packbits(grid, N, density_thresh, bitfield):
    _put(bitfield, O.packbits(_np(grid), density_thresh))


def _march_rays_train(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, M, nears, fars, xyzs, dirs, deltas, rays,
                      counter, noises):
    x, d, dl, r, cnt = O.march_rays_train(_np(rays_o), _np(rays_d), bound, _np(grid), C, H, _np(nears), _np(fars), _np(noises),
                                          dt_gamma, max_steps, M=M, counter=_np(counter))
    for dst, a in ((xyzs, x), (dirs, d), (deltas, dl), (rays, r), (counter, cnt)):
        _put(dst, a)


def _composite_rays_train_forward(sigmas, rgbs, deltas, rays, M, N, T_thresh, weights_sum, depth, image):
    ws, dp, im = O.composite_rays_train_forward(_np(sigmas), _np(rgbs), _np(deltas), _np(rays), T_thresh)
    for dst, a in ((weights_sum, ws), (depth, dp), (image, im)):
        _put(dst, a)


def _composite_rays_train_backward(grad_weights_sum, grad_image, sigmas, rgbs, deltas, rays, weights_sum, image, M, N, T_thresh,
                                   grad_sigmas, grad_rgbs):
    gs, gc = O.composite_rays_train_backward(_np(grad_weights_sum), _np(grad_image), _np(sigmas), _np(rgbs), _np(deltas),
                                             _np(rays), _np(weights_sum), _np(image), T_thresh)
    _put(grad_sigmas, gs)
    _put(grad_rgbs, gc)


def _march_rays(n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, bound, dt_gamma, max_steps, C, H, grid, nears, fars, xyzs,
                dirs, deltas, noises):
    x, d, dl = O.march_rays(n_alive, n_step, _np(rays_alive), _np(rays_t), _np(rays_o), _np(rays_d), bound, _np(grid), C, H,
                            _np(nears), _np(fars), _np(noises), dt_gamma, max_steps)
    m = x.shape[0]
    for dst, a in ((xyzs, x), (dirs, d), (deltas, dl)):
        _put(dst[:m], a)


def _device_lib():
    global _dev_lib
    if _dev_lib is None:
        lib = ctypes.CDLL(_build.build_cuda())
        u32, f32, vp = ctypes.c_uint32, ctypes.c_float, ctypes.c_void_p
        lib.oracle_freq_encode_forward_cuda.argtypes = [vp, u32, u32, u32, vp, vp]
        lib.oracle_composite_rays_cuda.argtypes = [u32, u32, f32] + [vp] * 9
        _dev_lib = lib
    return _dev_lib


def _device_call(name, device, *args):
    with torch.cuda.device(device):
        rc = getattr(_device_lib(), name)(*args, torch.cuda.current_stream().cuda_stream)
    if rc != 0:
        raise RuntimeError("%s: CUDA error %d" % (name, rc))


def _composite_rays(n_alive, n_step, T_thresh, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image):
    """On the device (oracle/ref_raymarching.cu): alpha takes the reference's __expf."""
    ins = [t.float().contiguous() for t in (sigmas, rgbs, deltas)]
    outs = (rays_alive, rays_t, weights_sum, depth, image)
    assert all(t.is_cuda and t.is_contiguous() for t in ins + list(outs))
    _device_call("oracle_composite_rays_cuda", sigmas.device, n_alive, n_step, T_thresh, rays_alive.data_ptr(),
                 rays_t.data_ptr(), *[t.data_ptr() for t in ins], weights_sum.data_ptr(), depth.data_ptr(), image.data_ptr())


def _freq_encode_forward(inputs, B, D, deg, C, outputs):
    """On the device (oracle/ref_freq.cu): the reference's fast-math sinf is the device's sin.approx."""
    assert inputs.is_cuda and outputs.is_cuda and outputs.is_contiguous() and outputs.dtype == torch.float32
    inputs = inputs.float().contiguous()
    _device_call("oracle_freq_encode_forward_cuda", inputs.device, inputs.data_ptr(), B, D, C, outputs.data_ptr())


def _freq_encode_backward(grad, outputs, B, D, deg, C, grad_inputs):
    _put(grad_inputs, O.freq_encode_backward(_np(grad), _np(outputs), D, deg))


def load():
    return types.SimpleNamespace(
        grid=types.SimpleNamespace(grid_encode_forward=_grid_encode_forward, grid_encode_backward=_grid_encode_backward),
        march=types.SimpleNamespace(near_far_from_aabb=_near_far_from_aabb, sph_from_ray=_sph_from_ray, morton3D=_morton3D,
                                    packbits=_packbits, march_rays_train=_march_rays_train,
                                    composite_rays_train_forward=_composite_rays_train_forward,
                                    composite_rays_train_backward=_composite_rays_train_backward, march_rays=_march_rays,
                                    composite_rays=_composite_rays),
        freq=types.SimpleNamespace(freq_encode_forward=_freq_encode_forward, freq_encode_backward=_freq_encode_backward))
