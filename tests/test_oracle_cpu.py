"""CPU tests: the C oracle against independent numpy restatements and known answers."""
import numpy as np
import pytest

from oracle import oracle as O
import ngp_testutil as util


def test_half_conversion_matches_numpy():
    rng = np.random.default_rng(0)
    x = (rng.standard_normal(100000) * rng.choice([1e-8, 1e-5, 1e-3, 1, 100, 60000], 100000)).astype(np.float32)
    edge = np.array([0, -0.0, 65504, 65519.99, 65520, 1e-8, 2 ** -24, 2 ** -25, 2 ** -25 * 1.0001, 5.96e-8, np.inf,
                     -np.inf, 2 ** -14, 2 ** -14 * 0.9999], np.float32)
    x = np.concatenate([x, edge])
    with np.errstate(over="ignore"):
        want = x.astype(np.float16)
    got = O.f2h(x)
    assert np.array_equal(got.view(np.uint16), want.view(np.uint16))


@pytest.mark.parametrize("dtype,accumulate", [(np.float32, "exact"), (np.float32, "f32"), (np.float16, "f16")])
def test_grid_backward_accumulation_modes(dtype, accumulate):
    """Every sample at x = 0 of a 1-D level: corner weights 0.5 / 0.5 (exact), so rows 0 and 1 receive the same addends in
    sample order.  Each mode must equal the numpy sum it names: float64, float32 rounded after every add, or float16 rounded
    after every add of the half-rounded addend (the reference's fp16 atomics)."""
    B = 4096
    g = (np.random.default_rng(3).standard_normal((B, 1)) * 4).astype(dtype)
    x = np.zeros((B, 1), np.float32)
    offs = np.array([0, 24], np.int32)
    table = O.grid_encode_backward(g, x, offs, 24, 1, 1.0, 16, gridtype=1, round_addend_to_half=dtype == np.float16,
                                   accumulate=accumulate)
    add = (np.float32(0.5) * g[:, 0].astype(np.float32)).astype(dtype)
    if accumulate == "exact":
        want = add.astype(np.float64).sum()
    else:
        acc = dtype(0)
        for v in add:
            acc = dtype(np.float32(acc) + np.float32(v))
        want = float(acc)
    assert np.count_nonzero(table) == 2 and table[0, 0] == want and table[1, 0] == want
    if accumulate != "exact":
        assert want != add.astype(np.float64).sum()     # the case tells the modes apart


def test_morton_known_answers_and_roundtrip():
    coords = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 1], [127, 127, 127], [5, 3, 9], [1023, 0, 1023]],
                      np.int32)
    # bit i of x lands at 3i, of y at 3i+1, of z at 3i+2 (raymarching.cu:65-71)
    def ref(c):
        v = 0
        for i in range(10):
            v |= ((c[0] >> i) & 1) << (3 * i) | ((c[1] >> i) & 1) << (3 * i + 1) | ((c[2] >> i) & 1) << (3 * i + 2)
        return v
    want = np.array([ref(c) for c in coords], np.int32)
    got = O.morton3D(coords)
    assert np.array_equal(got, want)
    assert got[4] == 7 and got[5] == 128 ** 3 - 1
    assert np.array_equal(O.morton3D_invert(got), coords)
    rng = np.random.default_rng(1)
    c = rng.integers(0, 128, (5000, 3)).astype(np.int32)
    assert np.array_equal(O.morton3D_invert(O.morton3D(c)), c)


def test_packbits_matches_numpy():
    rng = np.random.default_rng(2)
    g = rng.random(8 * 4096).astype(np.float32)
    g[:16] = [0.5] * 8 + [0.5000001] * 8   # equality is NOT occupied (strict >)
    got = O.packbits(g, 0.5)
    want = np.packbits((g > 0.5).reshape(-1, 8), axis=1, bitorder="little").reshape(-1)
    assert np.array_equal(got, want)
    assert got[0] == 0 and got[1] == 255


def test_level_resolutions_cfg2_cfg3():
    offs2, S = util.make_offsets(log2_hashmap_size=19)
    offs3, _ = util.make_offsets(log2_hashmap_size=16)
    scales, res = O.grid_level_params(16, np.float32(S), 16)
    # SURVEY 8: 16,23,31,43,59,81,112,154,213,295,407,562,777,1073,1483,2048
    assert list(res) == [16, 23, 31, 43, 59, 81, 112, 154, 213, 295, 407, 562, 777, 1073, 1483, 2048]
    assert scales[0] == 15.0 and scales[15] == 2047.0
    assert offs2[-1] == 6119864 and offs3[-1] == 903480
    assert list(np.diff(offs2)[:5]) == [4920, 13824, 32768, 85184, 216000]


def _np_grid_forward(inputs, emb, offsets, S, H, gridtype, align=False):
    """Independent float64 restatement (vectorised numpy) of the grid encoding."""
    B, D = inputs.shape
    L = len(offsets) - 1
    C = emb.shape[1]
    out = np.zeros((B, L, C))
    primes = np.array([1, 2654435761, 805459861], dtype=np.uint64)
    scales, ress = O.grid_level_params(L, np.float32(S), H)
    for l in range(L):
        scale, res = float(scales[l]), int(ress[l])
        hs = int(offsets[l + 1] - offsets[l])
        # one fused multiply-add in fp32 on the device; emulate via float64 (exact product) then one rounding
        pos = (inputs.astype(np.float64) * scale + (0.0 if align else 0.5)).astype(np.float32)
        pg = np.floor(pos).astype(np.int64)
        fr = (pos - pg.astype(np.float32)).astype(np.float64)
        for idx in range(1 << D):
            w = np.ones(B)
            p = np.zeros((B, D), np.int64)
            for d in range(D):
                if idx & (1 << d):
                    w *= fr[:, d]; p[:, d] = pg[:, d] + 1
                else:
                    w *= 1 - fr[:, d]; p[:, d] = pg[:, d]
            stride, index, d = 1, np.zeros(B, np.int64), 0
            while d < D and stride <= hs:
                index = (index + p[:, d] * stride) & 0xffffffff
                stride = (stride * (res if align else res + 1)) & 0xffffffff
                d += 1
            if gridtype == 0 and stride > hs:
                h = np.zeros(B, np.uint64)
                for d in range(D):
                    h ^= (p[:, d].astype(np.uint64) * primes[d]) & np.uint64(0xffffffff)
                index = h.astype(np.int64)
            index = index % hs
            out[:, l, :] += w[:, None] * emb[offsets[l] + index].astype(np.float64)
    oob = ((inputs < 0) | (inputs > 1)).any(1)
    out[oob] = 0
    return out.reshape(B, L * C)


@pytest.mark.parametrize("gridtype,log2", [(0, 19), (1, 16), (0, 14)])
def test_grid_forward_matches_numpy_restatement(gridtype, log2):
    rng = np.random.default_rng(3)
    offs, S = util.make_offsets(log2_hashmap_size=log2)
    emb = rng.uniform(-1, 1, (offs[-1], 2)).astype(np.float32)
    x = rng.uniform(0, 1, (1500, 3)).astype(np.float32)
    x[0] = 0; x[1] = 1; x[2] = [1.5, 0.2, 0.2]; x[3] = [0.3, -1e-6, 0.3]
    out, _ = O.grid_encode_forward(x, emb, offs, np.float32(S), 16, gridtype=gridtype)
    want = _np_grid_forward(x, emb, offs, S, 16, gridtype)
    assert np.abs(out - want).max() < 2e-6          # same fp32 positions, fp64 blending
    assert np.all(out[2] == 0) and np.all(out[3] == 0)  # out-of-range inputs encode to zeros
    # layouts agree
    out_lbc, _ = O.grid_encode_forward(x, emb, offs, np.float32(S), 16, gridtype=gridtype, out_layout=O.LBC)
    assert np.array_equal(out_lbc.transpose(1, 0, 2).reshape(len(x), -1), out)
    # half: within a few half-ulps of the fp64 value
    outh, _ = O.grid_encode_forward(x, emb.astype(np.float16), offs, np.float32(S), 16, gridtype=gridtype)
    wanth = _np_grid_forward(x, emb.astype(np.float16).astype(np.float32), offs, S, 16, gridtype)
    assert np.abs(outh.astype(np.float64) - wanth).max() < 4e-3


def test_tiled_grid_drops_axes_quirk():
    """gridencoder.cu:60-63: for 'tiled' with 2^16 rows the stride loop stops early, so fine levels ignore z."""
    offs, S = util.make_offsets(log2_hashmap_size=16)
    rng = np.random.default_rng(4)
    emb = rng.uniform(-1, 1, (offs[-1], 2)).astype(np.float32)
    x = rng.uniform(0.05, 0.95, (64, 3)).astype(np.float32)
    x2 = x.copy(); x2[:, 2] = rng.uniform(0.05, 0.95, 64)   # different z
    a, _ = O.grid_encode_forward(x, emb, offs, np.float32(S), 16, gridtype=1)
    b, _ = O.grid_encode_forward(x2, emb, offs, np.float32(S), 16, gridtype=1)
    a = a.reshape(64, 16, 2); b = b.reshape(64, 16, 2)
    # levels 9..15 have (res+1)^2 > 65536 -> index uses x,y only; the z weights still sum to 1
    assert np.allclose(a[:, 9:], b[:, 9:], atol=1e-6)
    assert not np.allclose(a[:, :3], b[:, :3], atol=1e-6)


def test_grid_backward_is_adjoint_of_forward():
    """<forward(emb), g> == <emb, backward(g)> - the encoding is linear in the table."""
    rng = np.random.default_rng(5)
    offs, S = util.make_offsets(num_levels=8, desired_resolution=256, log2_hashmap_size=12)
    emb = rng.uniform(-1, 1, (offs[-1], 2)).astype(np.float32)
    x = rng.uniform(0, 1, (800, 3)).astype(np.float32)
    g = rng.standard_normal((800, 16)).astype(np.float32)
    out, _ = O.grid_encode_forward(x, emb, offs, np.float32(S), 16)
    gt = O.grid_encode_backward(g, x, offs, offs[-1], 2, np.float32(S), 16)
    lhs = float((out.astype(np.float64) * g).sum())
    rhs = float((emb.astype(np.float64) * gt).sum())
    assert abs(lhs - rhs) < 1e-3 * max(1.0, abs(lhs))


def test_grid_dydx_matches_finite_difference():
    rng = np.random.default_rng(6)
    offs, S = util.make_offsets(num_levels=4, desired_resolution=64, log2_hashmap_size=19)
    emb = rng.uniform(-1, 1, (offs[-1], 2)).astype(np.float32)
    x = rng.uniform(0.1, 0.9, (50, 3)).astype(np.float32)
    out, dydx = O.grid_encode_forward(x, emb, offs, np.float32(S), 16, calc_dydx=True)
    dydx = dydx.reshape(50, 4, 3, 2)
    eps = 1e-3
    for d in range(3):
        xp = x.copy(); xp[:, d] += eps
        xm = x.copy(); xm[:, d] -= eps
        fp, _ = O.grid_encode_forward(xp, emb, offs, np.float32(S), 16)
        fm, _ = O.grid_encode_forward(xm, emb, offs, np.float32(S), 16)
        fd = ((fp - fm) / (2 * eps)).reshape(50, 4, 2)
        # piecewise-linear: exact unless the +-eps probe crosses a cell boundary; check the median
        err = np.abs(fd - dydx[:, :, d, :])
        assert np.median(err) < 5e-2


def test_near_far_known_answers():
    o = np.array([[0, 0, -3], [0, 0, -3], [0.5, 0.5, -3], [5, 5, 5]], np.float32)
    d = np.array([[0, 0, 1], [0, 1, 0], [1e-9, 1e-9, 1], [1, 0, 0]], np.float32)
    aabb = np.array([-1, -1, -1, 1, 1, 1], np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        nears, fars = O.near_far_from_aabb(o, d, aabb, 0.2)
    assert nears[0] == 2.0 and fars[0] == 4.0
    assert nears[1] == np.finfo(np.float32).max and fars[1] == np.finfo(np.float32).max   # parallel miss
    assert abs(nears[2] - 2.0) < 1e-5
    assert nears[3] == np.finfo(np.float32).max
    # min_near clamps
    o2 = np.array([[0, 0, 0]], np.float32); d2 = np.array([[0, 0, 1]], np.float32)
    n2, f2 = O.near_far_from_aabb(o2, d2, aabb, 0.2)
    assert n2[0] == np.float32(0.2) and f2[0] == 1.0


def _march_inputs(side=24, cascade=1, bound=1.0, seed=0):
    rays_o, rays_d = util.look_at_rays(side)
    grid = util.blob_density_grid(cascade, 128, bound, seed)
    bits = O.packbits(grid, 10.0)
    aabb = np.array([-bound] * 3 + [bound] * 3, np.float32)
    nears, fars = O.near_far_from_aabb(rays_o, rays_d, aabb, 0.2)
    noises = np.random.default_rng(seed + 1).random(rays_o.shape[0]).astype(np.float32)
    return rays_o, rays_d, bits, nears, fars, noises


def test_march_rays_train_invariants():
    rays_o, rays_d, bits, nears, fars, noises = _march_inputs()
    N = rays_o.shape[0]
    xyzs, dirs, deltas, rays, counter = O.march_rays_train(rays_o, rays_d, 1.0, bits, 1, 128, nears, fars, noises,
                                                           max_steps=1024)
    counts = rays[:, 2]
    assert counter[1] == N and counter[0] == counts.sum()
    assert np.array_equal(rays[:, 0], np.arange(N))
    assert np.array_equal(rays[:, 1], np.cumsum(counts) - counts)
    total = int(counter[0])
    assert total > 1000 and counts.max() <= 1024
    dt_min = np.float32(2 * 1.7320508075688772) / np.float32(1024)
    assert np.all(deltas[:total, 0] == dt_min)                       # dt_gamma = 0 -> constant step
    assert np.all(deltas[:total, 1] >= dt_min * 0.999)               # t - last_t covers skipped space too
    assert np.all(np.abs(xyzs[:total]) <= 1.0)
    assert np.all(xyzs[total:] == 0) and np.all(deltas[total:] == 0)
    # every emitted sample sits in an occupied cell
    idx = np.clip((0.5 * (xyzs[:total].astype(np.float64) + 1) * 128), 0, 127).astype(np.int32)
    m = O.morton3D(idx)
    assert np.all((bits[m // 8] >> (m % 8)) & 1)
    # dirs are the ray direction repeated
    rid = np.repeat(np.arange(N), counts)
    assert np.array_equal(dirs[:total], rays_d[rid])


def test_march_capacity_overflow_drops_rays():
    rays_o, rays_d, bits, nears, fars, noises = _march_inputs(side=16)
    full = O.march_rays_train(rays_o, rays_d, 1.0, bits, 1, 128, nears, fars, noises, max_steps=256)
    total = int(full[4][0])
    M = total // 2
    xyzs, dirs, deltas, rays, counter = O.march_rays_train(rays_o, rays_d, 1.0, bits, 1, 128, nears, fars, noises,
                                                           max_steps=256, M=M)
    assert np.array_equal(rays, full[3]) and counter[0] == total      # bookkeeping unaffected (raymarching.cu:411-416)
    fits = (rays[:, 1] + rays[:, 2]) <= M
    last = (rays[fits, 1] + rays[fits, 2]).max()
    assert np.array_equal(xyzs[:last], full[0][:last])
    assert np.all(xyzs[last:] == 0)


def test_composite_forward_matches_numpy_and_backward_matches_fd():
    rng = np.random.default_rng(7)
    counts = np.array([0, 5, 40, 1, 130, 64], np.int32)
    N, M = len(counts), int(counts.sum()) + 7
    rays = np.stack([np.array([3, 0, 5, 1, 4, 2], np.int32), np.cumsum(counts) - counts, counts], 1).astype(np.int32)
    sig = rng.uniform(0, 60, M).astype(np.float32)
    rgb = rng.uniform(0, 1, (M, 3)).astype(np.float32)
    dl = np.stack([np.full(M, 0.0034, np.float32), rng.uniform(0.0034, 0.02, M).astype(np.float32)], 1)
    ws, depth, image = O.composite_rays_train_forward(sig, rgb, dl, rays, 1e-4)

    def np_comp(sig):
        ws_ = np.zeros(N); dp = np.zeros(N); im = np.zeros((N, 3))
        for n in range(N):
            rid, off, cnt = rays[n]
            T, t = 1.0, 0.0
            for k in range(cnt):
                a = 1 - np.exp(-float(sig[off + k]) * float(dl[off + k, 0]))
                w = a * T
                im[rid] += w * rgb[off + k]; t += dl[off + k, 1]; dp[rid] += w * t; ws_[rid] += w
                T *= 1 - a
                if T < 1e-4:
                    break
        return ws_, dp, im
    w2, d2, i2 = np_comp(sig.astype(np.float64))
    assert np.allclose(ws, w2, rtol=1e-5, atol=1e-6) and np.allclose(depth, d2, rtol=1e-5, atol=1e-6)
    assert np.allclose(image, i2, rtol=1e-5, atol=1e-6)
    assert ws[3] == 0 and np.all(image[3] == 0)          # empty ray (id 3) -> zeros

    gws = rng.standard_normal(N).astype(np.float32)
    gim = rng.standard_normal((N, 3)).astype(np.float32)
    gs, gc = O.composite_rays_train_backward(gws, gim, sig, rgb, dl, rays, ws, image, 1e-4)
    # finite differences of L = sum(gws*ws + gim*image) wrt a few sigmas (away from the early-stop region)
    def loss(s):
        w_, _, i_ = np_comp(s)
        return float((gws * w_).sum() + (gim * i_).sum())
    s64 = sig.astype(np.float64)
    for m in [1, 3, 6, 10, 47, 50]:
        e = 1e-4
        sp = s64.copy(); sp[m] += e
        sm = s64.copy(); sm[m] -= e
        fd = (loss(sp) - loss(sm)) / (2 * e)
        assert abs(fd - gs[m]) < 2e-3 * max(1.0, abs(fd)), (m, fd, gs[m])
    # grad wrt rgb is gim * weight
    assert np.allclose(gc[1], gim[rays[1, 0]] * (1 - np.exp(-sig[0] * dl[0, 0])) * 0 + gc[1])


def test_inference_march_composite_agrees_with_train_path():
    """Marching n_step at a time + in-place compositing reproduces the train-mode image (same T_thresh)."""
    rays_o, rays_d, bits, nears, fars, _ = _march_inputs(side=12)
    N = rays_o.shape[0]
    zeros = np.zeros(N, np.float32)
    xyzs, dirs, deltas, rays, counter = O.march_rays_train(rays_o, rays_d, 1.0, bits, 1, 128, nears, fars, zeros,
                                                           max_steps=512)
    total = int(counter[0])
    rng = np.random.default_rng(8)
    def field(x):   # deterministic pseudo-field of position
        s = (20 * np.exp(-((x ** 2).sum(-1)) / 0.08)).astype(np.float32)
        c = (0.5 + 0.5 * np.sin(7 * x)).astype(np.float32)
        return s, c
    sig, rgb = field(xyzs[:total])
    ws, depth, image = O.composite_rays_train_forward(sig, rgb, deltas[:total], rays, 1e-4)

    w_i = np.zeros(N, np.float32); d_i = np.zeros(N, np.float32); im_i = np.zeros((N, 3), np.float32)
    alive = np.arange(N, dtype=np.int32)
    rays_t = nears.copy()
    step = 0
    while step < 512 and len(alive) > 0:
        n_alive = len(alive)
        n_step = max(min(N // n_alive, 8), 1)
        x, d, dl = O.march_rays(n_alive, n_step, alive, rays_t, rays_o, rays_d, 1.0, bits, 1, 128, nears, fars,
                                np.zeros(n_alive, np.float32), max_steps=512)
        s, c = field(x)
        alive, rays_t, w_i, d_i, im_i = O.composite_rays(n_alive, n_step, alive, rays_t, s, c, dl, w_i, d_i, im_i, 1e-4)
        alive = O.compact_alive(alive)
        step += n_step
    assert np.allclose(w_i, ws, atol=2e-4) and np.allclose(im_i, image, atol=2e-4)


def test_freq_encode_matches_numpy():
    rng = np.random.default_rng(9)
    x = rng.uniform(-1, 1, (300, 3)).astype(np.float32)
    out = O.freq_encode_forward(x, 6)
    want = [x]
    for f in range(6):
        want += [np.sin(2.0 ** f * x.astype(np.float64)), np.cos(2.0 ** f * x.astype(np.float64))]
    want = np.concatenate(want, 1)
    assert out.shape == (300, 39) and np.abs(out - want).max() < 5e-6
    g = rng.standard_normal(out.shape).astype(np.float32)
    gi = O.freq_encode_backward(g, out, 3, 6)
    jac = g[:, :3].astype(np.float64).copy()
    for f in range(6):
        s = 2.0 ** f
        jac += s * (g[:, 3 + 6 * f:6 + 6 * f] * np.cos(s * x) - g[:, 6 + 6 * f:9 + 6 * f] * np.sin(s * x))
    assert np.abs(gi - jac).max() < 1e-3


def test_occupancy_update_matches_numpy():
    H = 16
    rng = np.random.default_rng(10)
    noise = rng.random((H ** 3, 3)).astype(np.float32)
    pts = O.occupancy_cell_points(H, 1.0, noise)
    # numpy restatement of renderer.py:581-593 in linear order, scattered through morton indices
    xs = np.arange(H, dtype=np.int32)
    X, Y, Z = np.meshgrid(xs, xs, xs, indexing="ij")
    coords = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1)
    idx = O.morton3D(coords)
    hgs = 1.0 / H
    lin = (2 * coords.astype(np.float32) * np.float32(1.0 / (H - 1)) - 1) * np.float32(1.0 - hgs) + \
          (noise * 2 - 1) * np.float32(hgs)
    want = np.zeros_like(lin); want[idx] = lin
    assert np.abs(pts - want).max() < 1e-6
    assert np.all(np.abs(pts) <= 1.0)

    grid = rng.random(H ** 3).astype(np.float32) * 20
    grid[::7] = -1.0                                   # invalid cells stay untouched
    tmp = rng.random(H ** 3).astype(np.float32) * 20
    new, mean, bits = O.update_density_grid(grid, tmp, 0.95, 10.0)
    valid = grid >= 0
    want_g = grid.copy(); want_g[valid] = np.maximum(grid[valid] * np.float32(0.95), tmp[valid])
    assert np.array_equal(new, want_g)
    assert abs(mean - want_g[valid].mean()) < 1e-4
    assert np.array_equal(bits, O.packbits(want_g, min(mean, 10.0)))


def test_train_ray_loss_restatement_is_consistent():
    """oracle.train_ray_loss (the checker of the fused per-ray kernel): its sigma / rgb gradients are the finite-difference
    gradients of  sum(G * blend(image, ws, bg)) + scale * lambda * mean entropy(ws)  built from the composite forward."""
    rng = np.random.default_rng(0)
    n_rays, per = 12, 9
    M = n_rays * per
    rays = np.stack([np.arange(n_rays), np.arange(n_rays) * per, np.full(n_rays, per)], -1).astype(np.int32)
    sig = rng.uniform(0.5, 6.0, M).astype(np.float32)
    rgb = rng.uniform(0, 1, (M, 3)).astype(np.float32)
    deltas = np.stack([np.full(M, 0.05), np.full(M, 0.05)], -1).astype(np.float32)
    bg = rng.uniform(0, 1, (n_rays, 3)).astype(np.float32)
    G = rng.standard_normal((2, 3, n_rays // 2)).astype(np.float32)
    lam, scale = 0.3, 8.0
    out = O.train_ray_loss(sig, rgb, deltas, rays, bg, G, n_rays // 2, lam, scale, 1e-4)
    g_ray = G.transpose(0, 2, 1).reshape(n_rays, 3)

    def objective(s64, c64):
        total = 0.0
        for n in range(n_rays):
            T, ws, img = 1.0, 0.0, np.zeros(3)
            for i in range(n * per, (n + 1) * per):
                alpha = 1 - np.exp(-s64[i] * 0.05)
                w = alpha * T
                ws += w; img += w * c64[i]; T *= 1 - alpha
            a = min(max(ws, 1e-5), 1 - 1e-5)
            ent = -a * np.log2(a) - (1 - a) * np.log2(1 - a)
            total += (g_ray[n] * (img + (1 - ws) * bg[n])).sum() + scale * lam * ent / n_rays
        return total

    s64, c64 = sig.astype(np.float64), rgb.astype(np.float64)
    for idx in rng.choice(M, 10, replace=False):
        e = np.zeros(M); e[idx] = 1e-5
        fd = (objective(s64 + e, c64) - objective(s64 - e, c64)) / 2e-5
        assert abs(fd - out["grad_sigmas"][idx]) < 2e-3 * max(1.0, abs(fd)), (idx, fd, out["grad_sigmas"][idx])
        e3 = np.zeros((M, 3)); e3[idx, 1] = 1e-5
        fd = (objective(s64, c64 + e3) - objective(s64, c64 - e3)) / 2e-5
        assert abs(fd - out["grad_rgbs"][idx, 1]) < 2e-3 * max(1.0, abs(fd))
    assert abs(out["loss"] - lam * np.mean([-a * np.log2(a) - (1 - a) * np.log2(1 - a) for a in np.clip(out["weights_sum"], 1e-5, 1 - 1e-5).astype(np.float64)])) < 1e-6
    np.testing.assert_allclose(out["grad_bg"], (1 - out["weights_sum"])[:, None] * g_ray, rtol=1e-6)


def test_field_and_bg_oracle_gradients_match_finite_differences():
    """oracle.field_backward / bg_backward (the fp64 checkers of the tcgen05 field kernels and of the fused step) against
    central differences of oracle.field_forward / bg_forward (un-rounded mode), on the cfg3 table layout."""
    rng = np.random.default_rng(0)
    offs, S = util.make_offsets(log2_hashmap_size=16)
    table = rng.uniform(-0.5, 0.5, (offs[-1], 2)).astype(np.float16).astype(np.float32)
    W = [(rng.standard_normal(s) * sc).astype(np.float16).astype(np.float32) for s, sc in (((64, 32), 0.05), ((64, 64), 0.15), ((4, 64), 0.15))]
    b = [(rng.standard_normal(n) * 0.1).astype(np.float16).astype(np.float32) for n in (64, 64, 4)]
    x = rng.uniform(-0.9, 0.9, (500, 3)).astype(np.float32)
    ds, da = rng.standard_normal(500) * 0.1, rng.standard_normal((500, 3))
    S = np.float32(S)
    f = O.field_forward(x, table, offs, S, 16, W, b, round_hidden=False)
    g = O.field_backward(f, ds, da, offs, offs[-1], S, 16)

    def loss(W_, b_, t_):
        ff = O.field_forward(x, t_, offs, S, 16, W_, b_, round_hidden=False)
        return float((ff["sigma"] * ds).sum() + (ff["albedo"] * da).sum())

    eps = 2.0 ** -8          # representable in fp16 next to the quantised weights
    for li, key, idx, e_w, tol in ((1, "w2", (3, 5), eps, 2e-3), (2, "w3", (1, 7), eps, 2e-3), (0, "w1", (10, 4), 2.0 ** -11, 1e-2)):
        Wp, Wm = [w.copy() for w in W], [w.copy() for w in W]          # (a step on W1 crosses ReLU kinks of 500 x 64 units:
        Wp[li][idx] += e_w; Wm[li][idx] -= e_w                          #  smaller step, looser bound)
        fd = (loss(Wp, b, table) - loss(Wm, b, table)) / (2 * e_w)
        assert abs(fd - g[key][idx]) <= tol * abs(g[key][idx]) + 1e-6, (key, fd, g[key][idx])
    bp, bm = [v.copy() for v in b], [v.copy() for v in b]
    bp[2][0] += eps; bm[2][0] -= eps
    fd = (loss(W, bp, table) - loss(W, bm, table)) / (2 * eps)
    assert abs(fd - g["b3"][0]) <= 2e-3 * abs(g["b3"][0])
    r = int(np.argmax(np.abs(g["table"][:, 0])))       # the encoder is linear in the table: a large step is exact up to the MLP
    tp, tm = table.copy(), table.copy()
    tp[r, 0] += 2.0 ** -6; tm[r, 0] -= 2.0 ** -6
    fd = (loss(W, b, tp) - loss(W, b, tm)) / (2 * 2.0 ** -6)
    assert abs(fd - g["table"][r, 0]) <= 5e-2 * abs(g["table"][r, 0]), (fd, g["table"][r, 0])
    # the rounded ("spec") forward stays within fp16 noise of the exact one
    fr = O.field_forward(x, table, offs, S, 16, W, b, round_hidden=True)
    assert np.abs(fr["albedo"] - f["albedo"]).max() < 2e-3

    # background net
    d = rng.standard_normal((300, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    Wb = [(rng.standard_normal(s) * 0.2).astype(np.float16).astype(np.float32) for s in ((64, 39), (3, 64))]
    bb = [(rng.standard_normal(n) * 0.1).astype(np.float16).astype(np.float32) for n in (64, 3)]
    up = rng.standard_normal((300, 3))
    fb = O.bg_forward(d, Wb, bb)
    gb = O.bg_backward(fb, up)
    assert fb["rgb"].shape == (300, 3) and (fb["rgb"] > 0).all() and (fb["rgb"] < 1).all()
    # bg_forward rounds to fp16 at every Linear (finite differences would see the staircase): check the chain rule on an
    # un-rounded re-evaluation of the same graph instead
    e, Wq = fb["e"], fb["W"]

    def bg_loss(W1, b2):
        h = np.maximum(e @ W1.T + np.asarray(bb[0], np.float64), 0.0)
        out = h @ Wq[1].T + b2
        return float(((1.0 / (1.0 + np.exp(-out))) * up).sum())
    W1 = Wq[0].copy()
    b2 = np.asarray(bb[1], np.float64).copy()
    W1p, W1m = W1.copy(), W1.copy()
    W1p[5, 7] += 1e-5; W1m[5, 7] -= 1e-5
    fd = (bg_loss(W1p, b2) - bg_loss(W1m, b2)) / 2e-5
    # (gb is evaluated at the fp16-rounded activations; the un-rounded graph agrees to fp16 noise)
    assert abs(fd - gb["w1"][5, 7]) <= 2e-2 * abs(gb["w1"][5, 7]) + 1e-4, (fd, gb["w1"][5, 7])
