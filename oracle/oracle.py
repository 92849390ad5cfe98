"""TEST INFRASTRUCTURE: numpy front-end of the C oracle (``ngp_oracle.c``).

Each function mirrors one native entry point of the reference (same argument meaning as the
pybind functions in gridencoder/src/gridencoder.h:12-13, raymarching/src/raymarching.h:7-17,
freqencoder/src/freqencoder.h:7-10) but takes / returns numpy arrays on the host and allocates
its own outputs.  Half tensors are numpy float16.
"""
import ctypes as C

import numpy as np

from . import build as _build

_lib = None

F32, F16 = 0, 1
LBC, BLC = 0, 1


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(_build.build())
        _lib.oracle_compact_alive.restype = C.c_uint32
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _dt(emb):
    if emb.dtype == np.float16:
        return F16
    if emb.dtype == np.float32:
        return F32
    raise TypeError("embeddings must be float32 or float16")


# ------------------------------------------------------------------ gridencoder
def grid_level_params(L, S, H):
    scales = np.empty(L, np.float32)
    res = np.empty(L, np.uint32)
    lib().oracle_grid_level_params(C.c_uint32(L), C.c_float(S), C.c_uint32(H), _p(scales), _p(res))
    return scales, res


def grid_encode_forward(inputs, embeddings, offsets, S, H, calc_dydx=False, gridtype=0, align_corners=False,
                        out_layout=BLC, scale_override=None):
    """kernel_grid (gridencoder.cu:76-223). Returns (outputs, dy_dx|None).
    outputs: [B, L*C] for BLC, [L, B, C] for LBC, in the embeddings' dtype."""
    inputs = _c(inputs, np.float32)
    offsets = _c(offsets, np.int32)
    embeddings = np.ascontiguousarray(embeddings)
    dt = _dt(embeddings)
    B, D = inputs.shape
    Cc = embeddings.shape[1]
    L = offsets.shape[0] - 1
    out = np.empty((B, L * Cc) if out_layout == BLC else (L, B, Cc), embeddings.dtype)
    dydx = np.empty((B, L * D * Cc), embeddings.dtype) if calc_dydx else None
    so = None if scale_override is None else _c(scale_override, np.float32)
    rc = lib().oracle_grid_encode_forward(_p(inputs), _p(embeddings), _p(offsets), _p(out), C.c_uint32(B), C.c_uint32(D),
                                          C.c_uint32(Cc), C.c_uint32(L), C.c_float(S), C.c_uint32(H), _p(dydx),
                                          C.c_uint32(gridtype), C.c_int(int(align_corners)), C.c_int(dt),
                                          C.c_int(out_layout), _p(so))
    if rc != 0:
        raise RuntimeError("oracle_grid_encode_forward rc=%d" % rc)
    return out, dydx


def grid_encode_backward(grad, inputs, offsets, n_rows, Cc, S, H, gridtype=0, align_corners=False, grad_layout=BLC,
                         round_addend_to_half=False, scale_override=None, accumulate="exact"):
    """kernel_grid_backward (gridencoder.cu:227-313) with exact (float64) accumulation, or with the running sum rounded
    to float32 / float16 after every add in sample order (accumulate "f32" / "f16", like the reference's atomics).
    Returns grad_embeddings float64 [n_rows, C]."""
    inputs = _c(inputs, np.float32)
    offsets = _c(offsets, np.int32)
    grad = np.ascontiguousarray(grad)
    dt = _dt(grad)
    B, D = inputs.shape
    L = offsets.shape[0] - 1
    table = np.zeros((n_rows, Cc), np.float64)
    so = None if scale_override is None else _c(scale_override, np.float32)
    rc = lib().oracle_grid_encode_backward(_p(grad), _p(inputs), _p(offsets), _p(table), C.c_uint32(B), C.c_uint32(D),
                                           C.c_uint32(Cc), C.c_uint32(L), C.c_float(S), C.c_uint32(H),
                                           C.c_uint32(gridtype), C.c_int(int(align_corners)), C.c_int(dt),
                                           C.c_int(grad_layout), C.c_int(int(round_addend_to_half)),
                                           C.c_int(("exact", "f32", "f16").index(accumulate)), _p(so))
    if rc != 0:
        raise RuntimeError("oracle_grid_encode_backward rc=%d" % rc)
    return table


def grid_input_backward(grad, dy_dx, B, D, Cc, L, grad_layout=BLC):
    grad = np.ascontiguousarray(grad)
    dy_dx = np.ascontiguousarray(dy_dx)
    dt = _dt(grad)
    out = np.empty((B, D), grad.dtype)
    lib().oracle_grid_input_backward(_p(grad), _p(dy_dx), _p(out), C.c_uint32(B), C.c_uint32(D), C.c_uint32(Cc),
                                     C.c_uint32(L), C.c_int(dt), C.c_int(grad_layout))
    return out


# ------------------------------------------------------------------ raymarching
def near_far_from_aabb(rays_o, rays_d, aabb, min_near=0.2):
    rays_o = _c(rays_o, np.float32).reshape(-1, 3)
    rays_d = _c(rays_d, np.float32).reshape(-1, 3)
    aabb = _c(aabb, np.float32)
    N = rays_o.shape[0]
    nears = np.empty(N, np.float32)
    fars = np.empty(N, np.float32)
    lib().oracle_near_far_from_aabb(_p(rays_o), _p(rays_d), _p(aabb), C.c_uint32(N), C.c_float(min_near), _p(nears),
                                    _p(fars))
    return nears, fars


def sph_from_ray(rays_o, rays_d, radius):
    rays_o = _c(rays_o, np.float32).reshape(-1, 3)
    rays_d = _c(rays_d, np.float32).reshape(-1, 3)
    N = rays_o.shape[0]
    coords = np.empty((N, 2), np.float32)
    lib().oracle_sph_from_ray(_p(rays_o), _p(rays_d), C.c_float(radius), C.c_uint32(N), _p(coords))
    return coords


def morton3D(coords):
    coords = _c(coords, np.int32)
    N = coords.shape[0]
    out = np.empty(N, np.int32)
    lib().oracle_morton3D(_p(coords), C.c_uint32(N), _p(out))
    return out


def morton3D_invert(indices):
    indices = _c(indices, np.int32)
    N = indices.shape[0]
    out = np.empty((N, 3), np.int32)
    lib().oracle_morton3D_invert(_p(indices), C.c_uint32(N), _p(out))
    return out


def packbits(grid, thresh):
    grid = _c(grid, np.float32)
    N = grid.size // 8
    out = np.empty(N, np.uint8)
    lib().oracle_packbits(_p(grid), C.c_uint32(N), C.c_float(thresh), _p(out))
    return out


def march_rays_train(rays_o, rays_d, bound, bitfield, Ccas, H, nears, fars, noises, dt_gamma=0.0, max_steps=1024,
                     M=None, counter=None):
    """kernel_march_rays_train (raymarching.cu:312-480), rows in ray order.
    Returns xyzs[M,3], dirs[M,3], deltas[M,2], rays[N,3], counter[2]; buffers zero-filled like raymarching.py:205-207."""
    rays_o = _c(rays_o, np.float32).reshape(-1, 3)
    rays_d = _c(rays_d, np.float32).reshape(-1, 3)
    bitfield = _c(bitfield, np.uint8)
    nears = _c(nears, np.float32)
    fars = _c(fars, np.float32)
    noises = _c(noises, np.float32)
    N = rays_o.shape[0]
    if M is None:
        M = N * max_steps
    xyzs = np.zeros((M, 3), np.float32)
    dirs = np.zeros((M, 3), np.float32)
    deltas = np.zeros((M, 2), np.float32)
    rays = np.empty((N, 3), np.int32)
    counter = np.zeros(2, np.int32) if counter is None else _c(counter, np.int32).copy()
    lib().oracle_march_rays_train(_p(rays_o), _p(rays_d), _p(bitfield), C.c_float(bound), C.c_float(dt_gamma),
                                  C.c_uint32(max_steps), C.c_uint32(N), C.c_uint32(Ccas), C.c_uint32(H), C.c_uint32(M),
                                  _p(nears), _p(fars), _p(xyzs), _p(dirs), _p(deltas), _p(rays), _p(counter), _p(noises))
    return xyzs, dirs, deltas, rays, counter


def composite_rays_train_forward(sigmas, rgbs, deltas, rays, T_thresh=1e-4):
    sigmas = _c(sigmas, np.float32)
    rgbs = _c(rgbs, np.float32)
    deltas = _c(deltas, np.float32)
    rays = _c(rays, np.int32)
    M, N = sigmas.shape[0], rays.shape[0]
    ws = np.empty(N, np.float32)
    depth = np.empty(N, np.float32)
    image = np.empty((N, 3), np.float32)
    lib().oracle_composite_rays_train_forward(_p(sigmas), _p(rgbs), _p(deltas), _p(rays), C.c_uint32(M), C.c_uint32(N),
                                              C.c_float(T_thresh), _p(ws), _p(depth), _p(image))
    return ws, depth, image


def composite_rays_train_backward(grad_ws, grad_image, sigmas, rgbs, deltas, rays, weights_sum, image, T_thresh=1e-4):
    sigmas = _c(sigmas, np.float32)
    rgbs = _c(rgbs, np.float32)
    deltas = _c(deltas, np.float32)
    rays = _c(rays, np.int32)
    grad_ws = _c(grad_ws, np.float32)
    grad_image = _c(grad_image, np.float32)
    weights_sum = _c(weights_sum, np.float32)
    image = _c(image, np.float32)
    M, N = sigmas.shape[0], rays.shape[0]
    gs = np.zeros(M, np.float32)
    gc = np.zeros((M, 3), np.float32)
    lib().oracle_composite_rays_train_backward(_p(grad_ws), _p(grad_image), _p(sigmas), _p(rgbs), _p(deltas), _p(rays),
                                               _p(weights_sum), _p(image), C.c_uint32(M), C.c_uint32(N),
                                               C.c_float(T_thresh), _p(gs), _p(gc))
    return gs, gc


def march_rays(n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, bound, bitfield, Ccas, H, nears, fars, noises,
               dt_gamma=0.0, max_steps=1024, align=-1):
    rays_o = _c(rays_o, np.float32).reshape(-1, 3)
    rays_d = _c(rays_d, np.float32).reshape(-1, 3)
    rays_alive = _c(rays_alive, np.int32)
    rays_t = _c(rays_t, np.float32)
    bitfield = _c(bitfield, np.uint8)
    nears = _c(nears, np.float32)
    fars = _c(fars, np.float32)
    noises = _c(noises, np.float32)
    M = n_alive * n_step
    if align > 0:
        M += align - (M % align)
    xyzs = np.zeros((M, 3), np.float32)
    dirs = np.zeros((M, 3), np.float32)
    deltas = np.zeros((M, 2), np.float32)
    lib().oracle_march_rays(C.c_uint32(n_alive), C.c_uint32(n_step), _p(rays_alive), _p(rays_t), _p(rays_o), _p(rays_d),
                            C.c_float(bound), C.c_float(dt_gamma), C.c_uint32(max_steps), C.c_uint32(Ccas), C.c_uint32(H),
                            _p(bitfield), _p(nears), _p(fars), _p(xyzs), _p(dirs), _p(deltas), _p(noises))
    return xyzs, dirs, deltas


def composite_rays(n_alive, n_step, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image, T_thresh=1e-2):
    """In place on copies; returns (rays_alive, rays_t, weights_sum, depth, image)."""
    rays_alive = _c(rays_alive, np.int32).copy()
    rays_t = _c(rays_t, np.float32).copy()
    weights_sum = _c(weights_sum, np.float32).copy()
    depth = _c(depth, np.float32).copy()
    image = _c(image, np.float32).copy()
    sigmas = _c(sigmas, np.float32)
    rgbs = _c(rgbs, np.float32)
    deltas = _c(deltas, np.float32)
    lib().oracle_composite_rays(C.c_uint32(n_alive), C.c_uint32(n_step), C.c_float(T_thresh), _p(rays_alive), _p(rays_t),
                                _p(sigmas), _p(rgbs), _p(deltas), _p(weights_sum), _p(depth), _p(image))
    return rays_alive, rays_t, weights_sum, depth, image


def compact_alive(rays_alive):
    rays_alive = _c(rays_alive, np.int32)
    out = np.empty_like(rays_alive)
    k = lib().oracle_compact_alive(_p(rays_alive), C.c_uint32(rays_alive.shape[0]), _p(out))
    return out[:k].copy()


# ------------------------------------------------------------------ freqencoder
def freq_encode_forward(inputs, degree):
    inputs = _c(inputs, np.float32)
    B, D = inputs.shape
    Cc = D + D * 2 * degree
    out = np.empty((B, Cc), np.float32)
    lib().oracle_freq_encode_forward(_p(inputs), C.c_uint32(B), C.c_uint32(D), C.c_uint32(degree), C.c_uint32(Cc), _p(out))
    return out


def freq_encode_backward(grad, outputs, D, degree):
    grad = _c(grad, np.float32)
    outputs = _c(outputs, np.float32)
    B, Cc = grad.shape
    out = np.empty((B, D), np.float32)
    lib().oracle_freq_encode_backward(_p(grad), _p(outputs), C.c_uint32(B), C.c_uint32(D), C.c_uint32(degree),
                                      C.c_uint32(Cc), _p(out))
    return out


# ------------------------------------------------------------------ occupancy grid
def occupancy_cell_points(H, cascade_bound, noise):
    noise = _c(noise, np.float32)
    hgs = cascade_bound / H
    xyzs = np.empty((H ** 3, 3), np.float32)
    lib().oracle_occupancy_cell_points(C.c_uint32(H), C.c_float(np.float32(cascade_bound - hgs)),
                                       C.c_float(np.float32(hgs)), _p(noise), _p(xyzs))
    return xyzs


def update_density_grid(grid, tmp_grid, decay=0.95, density_thresh=10.0):
    """Returns (new_grid, mean, bitfield)."""
    grid = _c(grid, np.float32).copy()
    tmp_grid = _c(tmp_grid, np.float32)
    n = grid.size
    mean = np.empty(1, np.float32)
    bits = np.empty(n // 8, np.uint8)
    lib().oracle_update_density_grid(_p(grid), _p(tmp_grid), C.c_uint32(n), C.c_float(decay), C.c_float(density_thresh),
                                     _p(mean), _p(bits))
    return grid, float(mean[0]), bits


def f2h(x):
    x = _c(x, np.float32)
    out = np.empty(x.shape, np.uint16)
    lib().oracle_f2h(_p(x), _p(out), C.c_uint64(x.size))
    return out.view(np.float16)


def train_ray_loss(sigmas, rgbs, deltas, rays, bg, grad_pred_nchw, pixels_per_view, lambda_entropy, scale, T_thresh=1e-4):
    """TEST INFRASTRUCTURE - restatement of what the reference's train_step does between "the field has been evaluated"
    and "the gradients of sigma / rgb are known" for rays in ray order (row n <-> ray n), fp32:

      composite_rays_train forward (raymarching.cu:501-588)                    -> weights_sum, depth, image
      image + (1 - weights_sum) * bg  (nerf/renderer.py:541-545)               -> the blended prediction
      d(pred) = G (nerf/sd.py:115, unscaled), loss = lambda * mean(H2(clamp(ws, 1e-5, 1 - 1e-5))) (nerf/utils.py:389-394)
      back-propagated with the GradScaler scale on the entropy term only (nerf/utils.py:708)
      composite_rays_train backward (raymarching.cu:602-693)                   -> grad_sigmas, grad_rgbs

    bg: [N,3] fp32 (already rounded to half if it came from the bg net); grad_pred_nchw: [B,3,pixels_per_view].
    Returns dict(weights_sum, depth, image, loss, grad_ws, grad_bg, grad_sigmas, grad_rgbs)."""
    rays = _c(rays, np.int32)
    N = rays.shape[0]
    bg = _c(bg, np.float32).reshape(N, 3)
    G = _c(grad_pred_nchw, np.float32)
    Bv = N // pixels_per_view
    g_ray = np.ascontiguousarray(G.reshape(Bv, 3, pixels_per_view).transpose(0, 2, 1).reshape(N, 3))
    ws, depth, image = composite_rays_train_forward(sigmas, rgbs, deltas, rays, T_thresh)
    f32 = np.float32
    # blend backward
    grad_ws = -(g_ray[:, 0] * bg[:, 0] + g_ray[:, 1] * bg[:, 1] + g_ray[:, 2] * bg[:, 2]).astype(f32)
    grad_bg = ((f32(1) - ws)[:, None] * g_ray).astype(f32)
    # entropy of the clamped opacity and its (sub)gradient
    lo, hi = f32(1e-5), f32(1) - f32(1e-5)
    a = np.clip(ws, lo, hi)
    ent = (-a * np.log2(a) - (f32(1) - a) * np.log2(f32(1) - a)).astype(f32)
    loss = f32(lambda_entropy) * f32(ent.astype(np.float64).mean())
    inside = (ws >= lo) & (ws <= hi)
    with np.errstate(divide="ignore", invalid="ignore"):
        dent = (np.log2(f32(1) - ws) - np.log2(ws)).astype(f32)
    grad_ws = grad_ws + np.where(inside, f32(scale) * (f32(lambda_entropy) / f32(N)) * dent, f32(0)).astype(f32)
    # rays in ray order: id == row, so the per-ray gradients index directly
    gs, gc = composite_rays_train_backward(grad_ws, g_ray, sigmas, rgbs, deltas, rays, ws, image, T_thresh)
    return dict(weights_sum=ws, depth=depth, image=image, loss=loss, grad_ws=grad_ws, grad_bg=grad_bg, grad_sigmas=gs,
                grad_rgbs=gc)


# ------------------------------------------------------------------ the field network (nerf/network_grid.py)
def _h16(a):
    """Round to fp16 and come back as float64 (what a half tensor holds)."""
    return np.asarray(a, np.float64).astype(np.float16).astype(np.float64)


def field_forward(xyzs, table, offsets, S, H, weights, biases, bound=1.0, gridtype=1, align_corners=False,
                  scale_override=None, round_hidden=True):
    """TEST INFRASTRUCTURE - fp64 restatement of ``NeRFNetwork.common_forward`` under fp16 autocast
    (nerf/network_grid.py:76-87: GridEncoder -> Linear/ReLU x2 -> Linear -> trunc_exp(h0 + blob), sigmoid(h1..3);
    blob = 5 exp(-|x|^2 / (2 * 0.2^2)), :66-74; trunc_exp = exp in fp32, activation.py:8).

    table / weights / biases are quantised to fp16 first (autocast feeds half operands to the encoder and to cuBLAS);
    the encoding is the bit-exact C restatement of the half kernel; everything after it is float64.
    round_hidden=True additionally rounds every Linear output to fp16 (a half GEMM returns half) - the arithmetic the
    reference and the fused kernel both implement; False gives the un-rounded fp64 value of the same network.
    Returns dict(enc [M,32] f16, h1, h2 (post-ReLU), out [M,4] (pre-activation), sigma [M], albedo [M,3]) in float64."""
    xyzs = _c(xyzs, np.float32)
    x01 = ((xyzs + np.float32(bound)) * (np.float32(1.0) / np.float32(2 * bound))).astype(np.float32)   # grid.py:142
    enc, _ = grid_encode_forward(x01, np.asarray(table).astype(np.float16), offsets, S, H, gridtype=gridtype,
                                 align_corners=align_corners, scale_override=scale_override)
    W = [_h16(w) for w in weights]
    b = [_h16(v) for v in biases]
    rnd = _h16 if round_hidden else (lambda a: a)
    e = enc.astype(np.float64)
    h1 = np.maximum(rnd(e @ W[0].T + b[0]), 0.0)
    h2 = np.maximum(rnd(h1 @ W[1].T + b[1]), 0.0)
    out = rnd(h2 @ W[2].T + b[2])
    x64 = xyzs.astype(np.float64)
    blob = 5.0 * np.exp(-(x64 ** 2).sum(-1) / (2 * 0.2 ** 2))
    sigma = np.exp(out[:, 0] + blob)
    albedo = 1.0 / (1.0 + np.exp(-out[:, 1:]))
    return dict(enc=enc, x01=x01, h1=h1, h2=h2, out=out, sigma=sigma, albedo=albedo, W=W, b=b)


def field_backward(fwd, d_sigma, d_albedo, offsets, n_rows, S, H, gridtype=1, align_corners=False, scale_override=None):
    """TEST INFRASTRUCTURE - exact (float64, no intermediate rounding) gradients of ``field_forward``'s outputs wrt the
    table and the MLP parameters, by the chain rule of nerf/network_grid.py:76-87 with trunc_exp's backward
    g * exp(clamp(x, -15, 15)) (activation.py:13-15).  `fwd` is field_forward's dict (either rounding mode: the ReLU masks
    and activations are taken from it).  Returns dict(table [n_rows,2], w1, b1, w2, b2, w3, b3, d_enc [M,32])."""
    d_sigma = np.asarray(d_sigma, np.float64)
    d_albedo = np.asarray(d_albedo, np.float64)
    W = fwd["W"]
    arg = np.log(fwd["sigma"])                                        # h0 + blob
    dout = np.empty_like(fwd["out"])
    dout[:, 0] = d_sigma * np.exp(np.clip(arg, -15.0, 15.0))
    dout[:, 1:] = d_albedo * fwd["albedo"] * (1.0 - fwd["albedo"])
    h2, h1, e = fwd["h2"], fwd["h1"], fwd["enc"].astype(np.float64)
    g = {}
    g["w3"], g["b3"] = dout.T @ h2, dout.sum(0)
    dh2 = (dout @ W[2]) * (h2 > 0)
    g["w2"], g["b2"] = dh2.T @ h1, dh2.sum(0)
    dh1 = (dh2 @ W[1]) * (h1 > 0)
    g["w1"], g["b1"] = dh1.T @ e, dh1.sum(0)
    d_enc = dh1 @ W[0]
    g["d_enc"] = d_enc
    # the encoder's backward with exact accumulation; gradients handed over in fp32 (nothing is rounded to half here)
    g["table"] = grid_encode_backward(d_enc.astype(np.float32), fwd["x01"], offsets, n_rows, 2, S, H, gridtype=gridtype,
                                      align_corners=align_corners, scale_override=scale_override)
    return g


def bg_forward(dirs, weights, biases, degree=6):
    """TEST INFRASTRUCTURE - fp64 restatement of ``NeRFNetwork.background`` under fp16 autocast (nerf/network_grid.py:
    158-167: FreqEncoder(degree 6) -> Linear(39,64)+ReLU -> Linear(64,3) -> sigmoid), fp16-quantised parameters, Linear
    outputs rounded to fp16 as a half GEMM returns them, encoder input rounded to half as autocast feeds it."""
    enc = freq_encode_forward(_c(dirs, np.float32), degree)            # fp32, bit-exact restatement of kernel_freq
    e = _h16(enc)                                                      # autocast casts the Linear's input to half
    W = [_h16(w) for w in weights]
    b = [_h16(v) for v in biases]
    h = np.maximum(_h16(e @ W[0].T + b[0]), 0.0)
    out = _h16(h @ W[1].T + b[1])
    rgb = _h16(1.0 / (1.0 + np.exp(-out)))
    return dict(e=e, h=h, out=out, rgb=rgb, W=W)


def bg_backward(fwd, d_rgb):
    """Exact float64 parameter gradients of bg_forward's rgb (chain rule, no intermediate rounding)."""
    d_rgb = np.asarray(d_rgb, np.float64)
    y = 1.0 / (1.0 + np.exp(-fwd["out"]))
    dout = d_rgb * y * (1.0 - y)
    g = {"w2": dout.T @ fwd["h"], "b2": dout.sum(0)}
    dh = (dout @ fwd["W"][1]) * (fwd["h"] > 0)
    g["w1"], g["b1"] = dh.T @ fwd["e"], dh.sum(0)
    return g


def adam_scaler_step(p, g, m, v, state, seg_end, seg_lr, betas=(0.9, 0.99), eps=1e-15, grad_div=1.0, lr_decay_ln=0.0,
                     lr_decay_steps=0.0, growth=2.0, backoff=0.5, growth_interval=2000):
    """TEST INFRASTRUCTURE - float64 restatement of ONE ``ngp_adam_step`` launch after its finite check (optim.py
    FusedAdamScaler.step; csrc/adam.cu adam_step_kernel), i.e. ``scaler.step(optimizer); scaler.update();
    optimizer.zero_grad()`` on torch.optim.Adam + LambdaLR + GradScaler over one flat buffer:

      found_inf = state[3] or any non-finite g  ->  p, m, v untouched; scale *= backoff, tracker = 0, skipped += 1
      else  g / (scale * grad_div) -> m.lerp_(g, 1 - b1), v = b2 v + (1 - b2) g^2,
            p -= lr_seg * exp(lr_decay_ln * min(step, lr_decay_steps)) / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)
            with t = step + 1; step = t; tracker += 1, scale *= growth (if finite) once tracker reaches growth_interval
      the gradients come back zeroed either way.

    p, g, m, v: flat float arrays of one length; state: [scale, growth tracker, steps, found_inf, skipped, ...] (optim.py
    FusedAdamScaler.state); seg_end: exclusive end of each lr group; seg_lr: its lr.  The scalar arguments are narrowed to
    float32 first, as the launch receives them.  Returns (p, g, m, v, state) as new float64 arrays."""
    f32 = lambda x: float(np.float32(x))  # noqa: E731
    b1, b2, eps = f32(betas[0]), f32(betas[1]), f32(eps)
    p = np.array(p, np.float64)
    m = np.array(m, np.float64)
    v = np.array(v, np.float64)
    g = np.asarray(g)
    st = np.array(state, np.float64)
    scale, tracker, steps = st[0], st[1], st[2]
    skip = st[3] != 0 or not np.isfinite(g).all()
    if skip:
        st[0], st[1], st[4] = scale * f32(backoff), 0.0, st[4] + 1
    else:
        t = steps + 1
        bc1, bc2_sqrt = 1.0 - b1 ** t, np.sqrt(1.0 - b2 ** t)
        lr_mult = np.exp(f32(lr_decay_ln) * min(steps, f32(lr_decay_steps))) if lr_decay_ln != 0 else 1.0
        lr = np.empty_like(p)
        start = 0
        for end, seg in zip(seg_end, seg_lr):
            lr[start:int(end)] = f32(seg)
            start = int(end)
        if start != p.size:
            raise ValueError("seg_end must end at the buffer's length")
        gr = np.asarray(g, np.float64) / (scale * f32(grad_div))
        m += (1.0 - b1) * (gr - m)
        v *= b2
        v += (1.0 - b2) * gr * gr
        denom = np.sqrt(v) / bc2_sqrt + eps
        p -= lr * (lr_mult / bc1) * m / denom
        tracker += 1
        if tracker >= growth_interval:
            grown = scale * f32(growth)
            if np.isfinite(np.float32(grown)):
                scale = grown
            tracker = 0.0
        st[0], st[1], st[2] = scale, tracker, t
    st[3] = 0.0
    return p, np.zeros(g.shape, np.float64), m, v, st


def get_rays(poses, intrinsics, H, W):
    """TEST INFRASTRUCTURE - numpy restatement of nerf/utils.py:43-106 get_rays for the full image (N = -1): pixel centres
    at +0.5 (:60-61), directions ((i - cx) / fx, (j - cy) / fy, 1) (:93-96) normalised by safe_normalize (:33-36, clamp of
    the squared norm at 1e-20), rays_d = directions @ R^T (:98), rays_o = translation (:100-101).  fp32 like torch.
    poses [B,4,4]; intrinsics [4] or [B,4].  Returns rays_o, rays_d [B, H*W, 3]."""
    poses = _c(poses, np.float32)
    K = np.broadcast_to(_c(intrinsics, np.float32).reshape(-1, 4), (poses.shape[0], 4))
    f32 = np.float32
    j, i = np.meshgrid(np.arange(H, dtype=f32), np.arange(W, dtype=f32), indexing="ij")   # i: column, j: row
    i = i.reshape(1, H * W) + f32(0.5)
    j = j.reshape(1, H * W) + f32(0.5)
    xs = ((i - K[:, 2:3]) / K[:, 0:1]).astype(f32)
    ys = ((j - K[:, 3:4]) / K[:, 1:2]).astype(f32)
    d = np.stack([xs, ys, np.ones_like(xs)], -1)
    d = (d / np.sqrt(np.maximum((d * d).sum(-1, keepdims=True), f32(1e-20)))).astype(f32)
    rays_d = np.einsum("bnc,bkc->bnk", d, poses[:, :3, :3]).astype(f32)
    rays_o = np.broadcast_to(poses[:, None, :3, 3], rays_d.shape).astype(f32).copy()
    return rays_o, rays_d
