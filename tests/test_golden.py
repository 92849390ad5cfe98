"""Golden-vector tests.  tests/golden/ref_golden.npz holds OUTPUTS of the reference's own CUDA extensions
(built unmodified from /root/reference, run on a B200 by oracle/make_golden.py) for the seeded cases in
ngp_testutil.  CPU: the C oracle must reproduce them (this is what pins the oracle).  GPU: so must the
CUDA path, through the C ABI."""
import os

import numpy as np
import pytest

import ngp_testutil as util
from oracle import oracle as O

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_golden.npz"))


def _ulps(a, b):
    a = np.ascontiguousarray(a, np.float32).view(np.int32).astype(np.int64)
    b = np.ascontiguousarray(b, np.float32).view(np.int32).astype(np.int64)
    return np.abs(a - b)


@pytest.mark.parametrize("dt", ["f32", "f16"])
@pytest.mark.parametrize("gridtype", [0, 1])
def test_oracle_grid_vs_reference_golden(gridtype, dt):
    c = util.golden_grid_case(gridtype, dt)
    key = "grid_g%d_%s_" % (gridtype, dt)
    want = GOLD[key + "out"]
    wj = GOLD[key + "dydx"]
    # 1) with the device's own per-level scales (exp2f on the GPU is MUFU.EX2, up to 2 ulp from libm) the oracle is
    #    BIT-EXACT with the reference kernel, fp32 and fp16, outputs and dy_dx
    out, dydx = O.grid_encode_forward(c["x"], c["emb"], c["offs"], c["S"], c["H"], calc_dydx=True, gridtype=gridtype,
                                      scale_override=GOLD["grid_scales"])
    assert np.array_equal(out, want)
    assert np.array_equal(dydx, wj)
    # 2) with libm's exp2f only the levels whose scale moved by an ulp differ, and only slightly
    out2, _ = O.grid_encode_forward(c["x"], c["emb"], c["offs"], c["S"], c["H"], gridtype=gridtype)
    assert np.abs(out2.astype(np.float32) - want.astype(np.float32)).max() <= (1e-3 if dt == "f32" else 4e-3)
    assert np.mean(out2 == want) > 0.3
    gt = O.grid_encode_backward(c["grad"], c["x"], c["offs"], c["offs"][-1], 2, c["S"], c["H"], gridtype=gridtype,
                                round_addend_to_half=(dt == "f16"), scale_override=GOLD["grid_scales"])
    rows = np.random.default_rng(5).integers(0, gt.shape[0], 4096)
    tol = 1e-5 if dt == "f32" else 3e-3      # the reference accumulates fp16 atomics under autocast
    assert util.rel_l2(gt[rows], GOLD[key + "gemb_rows"]) < tol
    assert abs(np.abs(gt).sum() - GOLD[key + "gemb_l1"][0]) < (1e-4 if dt == "f32" else 5e-3) * GOLD[key + "gemb_l1"][0]
    gi = O.grid_input_backward(c["grad"], dydx, c["x"].shape[0], 3, 2, 16)
    assert np.array_equal(gi, GOLD[key + "ginp"].astype(gi.dtype))


MARCH = (("m1", {}), ("m2", dict(cascade=2, bound=2.0, dt_gamma=1.0 / 128, max_steps=128, seed=21)))


@pytest.mark.parametrize("name,kw", MARCH)
def test_oracle_march_composite_vs_reference_golden(name, kw):
    c = util.golden_march_case(**kw)
    bits = O.packbits(c["grid"], c["thresh"])
    assert int(bits.astype(np.int64).sum()) == int(GOLD[name + "_bits_sum"][0])
    assert np.array_equal(bits[:4096], GOLD[name + "_bits_head"])
    nears, fars = O.near_far_from_aabb(c["rays_o"], c["rays_d"], c["aabb"], 0.2)
    assert np.array_equal(nears, GOLD[name + "_nears"]) and np.array_equal(fars, GOLD[name + "_fars"])
    xyzs, dirs, deltas, rays, counter = O.march_rays_train(c["rays_o"], c["rays_d"], c["bound"], bits, c["cascade"], 128,
                                                           nears, fars, c["noises"], c["dt_gamma"], c["max_steps"])
    # integer outputs and sample positions: BIT-EXACT with the reference kernel
    assert np.array_equal(counter, GOLD[name + "_counter"])
    assert np.array_equal(rays[:, 2], GOLD[name + "_counts"])
    total = int(counter[0])
    assert np.array_equal(xyzs[:total].view(np.uint32), GOLD[name + "_xyzs"].view(np.uint32))
    assert np.array_equal(deltas[:total].view(np.uint32), GOLD[name + "_deltas"].view(np.uint32))

    sig, rgb = util.pseudo_field(xyzs[:total])
    ws, depth, image = O.composite_rays_train_forward(sig, rgb, deltas[:total], rays, 1e-4)
    np.testing.assert_allclose(ws, GOLD[name + "_ws"], rtol=1e-5, atol=1e-6)      # expf vs ex2.approx
    np.testing.assert_allclose(depth, GOLD[name + "_depth"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(image, GOLD[name + "_image"], rtol=1e-5, atol=1e-6)
    rng = np.random.default_rng(33)
    N = rays.shape[0]
    gws = rng.standard_normal(N).astype(np.float32)
    gim = rng.standard_normal((N, 3)).astype(np.float32)
    gs, gc = O.composite_rays_train_backward(gws, gim, sig, rgb, deltas[:total], rays, GOLD[name + "_ws"],
                                             GOLD[name + "_image"], 1e-4)
    scale = np.abs(GOLD[name + "_gsig"]).max()
    assert np.abs(gs - GOLD[name + "_gsig"]).max() < 1e-4 * scale
    np.testing.assert_allclose(gc, GOLD[name + "_grgb"], rtol=1e-5, atol=1e-6)

    alive = np.arange(N, dtype=np.int32)
    ix, _, il = O.march_rays(N, 4, alive, nears.copy(), c["rays_o"], c["rays_d"], c["bound"], bits, c["cascade"], 128, nears,
                             fars, np.zeros(N, np.float32), c["dt_gamma"], c["max_steps"], align=128)
    assert np.array_equal(ix.view(np.uint32), GOLD[name + "_inf_xyzs"].view(np.uint32))
    assert np.array_equal(il.view(np.uint32), GOLD[name + "_inf_deltas"].view(np.uint32))


def test_oracle_morton_freq_vs_reference_golden():
    coords = np.random.default_rng(41).integers(0, 128, (512, 3)).astype(np.int32)
    assert np.array_equal(O.morton3D(coords), GOLD["morton"])
    fx = np.random.default_rng(42).uniform(-1, 1, (128, 3)).astype(np.float32)
    out = O.freq_encode_forward(fx, 6)
    assert np.abs(out - GOLD["freq_out"]).max() < 5e-6      # sinf vs sin.approx
    fg = np.random.default_rng(43).standard_normal((128, 39)).astype(np.float32)
    gi = O.freq_encode_backward(fg, GOLD["freq_out"], 3, 6)
    assert np.abs(gi - GOLD["freq_gin"]).max() < 1e-4 * np.abs(GOLD["freq_gin"]).max()


@pytest.mark.parametrize("dt", ["f32", "f16"])
@pytest.mark.parametrize("gridtype", [0, 1])
def test_reference_standin_grid_vs_reference_golden(gridtype, dt):
    """The stand-in the GPU tests use when the reference's extensions are not built, through the reference's calling
    convention: forward bit-exact, table gradient accumulated in the table's dtype within the reference's own spread."""
    import torch
    from oracle import ref_ext as R
    from oracle import ref_standin
    ns = ref_standin.load()
    c = util.golden_grid_case(gridtype, dt)
    key = "grid_g%d_%s_" % (gridtype, dt)
    T = torch.from_numpy
    out, dydx, _ = R.grid_encode_forward(ns, T(c["x"]), T(c["emb"]), T(c["offs"]), float(c["S"]), c["H"], True, gridtype, False)
    assert np.array_equal(out.numpy(), GOLD[key + "out"]) and np.array_equal(dydx.numpy(), GOLD[key + "dydx"])
    ge, gi = R.grid_encode_backward(ns, T(c["grad"]), T(c["x"]), T(c["emb"]), T(c["offs"]), float(c["S"]), c["H"], dydx, gridtype,
                                    False)
    assert ge.dtype == T(c["emb"]).dtype
    rows = np.random.default_rng(5).integers(0, ge.shape[0], 4096)
    assert util.rel_l2(ge.double().numpy()[rows], GOLD[key + "gemb_rows"]) < (1e-5 if dt == "f32" else 3e-3)
    assert np.array_equal(gi.numpy(), GOLD[key + "ginp"].astype(gi.numpy().dtype))


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_reference_standin_freq_kernel_vs_reference_golden():
    """oracle/ref_freq.cu, the stand-in's fast-math frequency encoder, is bit-exact with the reference's stored output."""
    import torch
    from oracle import ref_standin
    fx = np.random.default_rng(42).uniform(-1, 1, (128, 3)).astype(np.float32)
    out = torch.empty(128, 39, device="cuda:0")
    ref_standin.load().freq.freq_encode_forward(torch.from_numpy(fx).to("cuda:0"), 128, 3, 6, 39, out)
    assert np.array_equal(out.cpu().numpy(), GOLD["freq_out"])


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ["f32", "f16"])
@pytest.mark.parametrize("gridtype", [0, 1])
def test_cuda_grid_vs_reference_golden(gridtype, dt):
    import torch
    from test_gpu_parity import T, N_, my_grid_forward, my_grid_backward
    c = util.golden_grid_case(gridtype, dt)
    key = "grid_g%d_%s_" % (gridtype, dt)
    x, emb, offs = T(c["x"]), T(c["emb"]), T(c["offs"])
    out, j = my_grid_forward(x, emb, offs, c["S"], c["H"], gridtype, dydx=True)
    assert np.array_equal(N_(out), GOLD[key + "out"])             # bit-exact, fp32 and fp16
    assert np.array_equal(N_(j), GOLD[key + "dydx"])
    g = T(c["grad"])
    ge, gi = my_grid_backward(g, x, offs, emb.shape[0], 2, c["S"], c["H"], gridtype, torch.float32, dydx=j)
    rows = np.random.default_rng(5).integers(0, emb.shape[0], 4096)
    assert util.rel_l2(N_(ge)[rows], GOLD[key + "gemb_rows"]) < (1e-5 if dt == "f32" else 1e-3)
    assert np.array_equal(N_(gi).astype(np.float32), GOLD[key + "ginp"])


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw", MARCH)
def test_cuda_march_composite_vs_reference_golden(name, kw):
    import torch
    import raymarching
    from test_gpu_parity import T, N_
    c = util.golden_march_case(**kw)
    bits = raymarching.packbits(T(c["grid"]), c["thresh"])
    assert int(bits.long().sum().item()) == int(GOLD[name + "_bits_sum"][0])
    ro, rd = T(c["rays_o"]), T(c["rays_d"])
    nears, fars = raymarching.near_far_from_aabb(ro, rd, T(c["aabb"]), 0.2)
    assert np.array_equal(N_(nears), GOLD[name + "_nears"]) and np.array_equal(N_(fars), GOLD[name + "_fars"])
    # inject the golden noises through the C ABI (the python wrapper draws its own)
    from ngp_b200 import _cabi as cb
    N = ro.shape[0]
    M = N * c["max_steps"]
    xyzs = torch.zeros(M, 3, device=ro.device); dirs = torch.zeros(M, 3, device=ro.device)
    deltas = torch.zeros(M, 2, device=ro.device)
    rays = torch.empty(N, 3, dtype=torch.int32, device=ro.device)
    counter = torch.zeros(2, dtype=torch.int32, device=ro.device)
    nz = T(c["noises"])
    ws_ = torch.empty(int(cb.load().ngp_march_rays_train_workspace(N, c["max_steps"])), dtype=torch.uint8, device=ro.device)
    ws_[:256].zero_()   # a new workspace's head must be zero (include/ngp_b200.h)
    cb.call("ngp_march_rays_train", ro.device, cb.ptr(ro), cb.ptr(rd), cb.ptr(bits), float(c["bound"]), float(c["dt_gamma"]),
            c["max_steps"], N, c["cascade"], 128, M, cb.ptr(nears), cb.ptr(fars), cb.ptr(xyzs), cb.ptr(dirs), cb.ptr(deltas),
            cb.ptr(rays), cb.ptr(counter), cb.ptr(nz), cb.ptr(ws_), ws_.numel())
    assert np.array_equal(N_(counter), GOLD[name + "_counter"])
    assert np.array_equal(N_(rays[:, 2]), GOLD[name + "_counts"])
    total = int(counter[0].item())
    assert np.array_equal(N_(xyzs[:total]), GOLD[name + "_xyzs"]) and np.array_equal(N_(deltas[:total]), GOLD[name + "_deltas"])
    sig, rgb = util.pseudo_field(N_(xyzs[:total]))
    s_t, c_t = T(sig).requires_grad_(True), T(rgb).requires_grad_(True)
    ws, depth, image = raymarching.composite_rays_train(s_t, c_t, deltas[:total].contiguous(), rays, 1e-4)
    np.testing.assert_allclose(N_(ws), GOLD[name + "_ws"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(N_(depth), GOLD[name + "_depth"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(N_(image), GOLD[name + "_image"], rtol=1e-5, atol=1e-6)
    rng = np.random.default_rng(33)
    gws = rng.standard_normal(N).astype(np.float32)
    gim = rng.standard_normal((N, 3)).astype(np.float32)
    ((ws * T(gws)).sum() + (image * T(gim)).sum()).backward()
    scale = np.abs(GOLD[name + "_gsig"]).max()
    assert np.abs(N_(s_t.grad) - GOLD[name + "_gsig"]).max() < 1e-4 * scale
    np.testing.assert_allclose(N_(c_t.grad), GOLD[name + "_grgb"], rtol=1e-5, atol=1e-6)
