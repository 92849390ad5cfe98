"""GPU tests of the hand-scheduled shaded train step (shading 'lambertian' / 'textureless' / 'normal'; csrc/shading.cu
ngp_stencil_points / ngp_shade_forward_step / ngp_shade_backward_step, csrc/raymarch.cu ngp_train_light, trainer.py
_manual_compute): the same step as the autograd route (nerf/utils.py:345-356,396-398, nerf/renderer.py:461-464,485-486),
its kernels against a float64 restatement, graph capture and replay, the device-side light draw, guard bands and routing."""
import numpy as np
import pytest
import torch

from test_gpu_guards import Guards, _model as _guard_model
from test_gpu_train_step import _bench_like_model, _ray_noise_np

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MODES = {"lambertian": 0, "textureless": 1, "normal": 2}


def _param_grads(step, g):
    out = {}
    for name, p in step.model.named_parameters():
        o = step.opt.offsets[step.opt._index(p)]
        out[name] = g[o:o + p.numel()].view_as(p)
    return out


# -- 1. the hand-scheduled shaded step vs the autograd shaded step -------------------------------------------------------
@pytest.mark.parametrize("shading", list(MODES))
@pytest.mark.parametrize("views,n_chunks", [(1, 1), (1, 2), (2, 2)])
def test_hand_scheduled_shaded_step_matches_autograd_step(shading, views, n_chunks):
    """Both steps evaluate the same 7-row stencil batches with the same kernels, with the same jitter and light (mirror_rng);
    only the sample order (completion-order vs ray-order marcher) and the order of fp32 atomics differ."""
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(views, 64, 64, seed=3, pin=False)
    ro, rd = ro.to(DEV), rd.to(DEV)
    G = torch.randn(views, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1)) * 1e-2
    got = {}
    for manual in (True, False):
        m = _bench_like_model()
        step = TrainStep(m, 64, 64, lr=1e-3, graph=False, manual=manual, n_chunks=n_chunks, shading=shading)
        assert step.manual == manual
        step.mirror_rng = True   # same torch RNG consumption as run_cuda: same ray noise, same light
        grads = []

        def capture(*a, _s=step, _g=grads, **k):
            if _s.manual:
                _s.fold_table_grads()
            _g.append(_s.opt.flat_grads.clone())
            _s.opt.flat_grads.zero_()
        step.opt.step = capture
        torch.manual_seed(5)
        loss = step(ro, rd, G)
        torch.cuda.synchronize()
        got[manual] = dict(loss=loss.item(), g=_param_grads(step, grads[0]), counter=m.step_counter.clone(),
                           samples=step.samples.item(), local_step=m.local_step)
    a, b = got[True], got[False]
    assert a["samples"] == b["samples"] > 0
    assert torch.equal(a["counter"], b["counter"]) and a["local_step"] == b["local_step"] == 1
    # entropy + orientation.  The orientation mean sums ~0.5 M (1 view) to ~1 M (2 views) positive fp32 terms: torch's tree
    # reduction on one side, per-block partial sums added into the loss with fp32 atomics on the other.  Measured on a B200:
    # 1.2e-5 to 1.3e-5 relative at 2 views over four runs, 4e-6 to 6e-6 at 1 view (the entropy-only albedo step stays
    # within 1e-5), so the ceiling is 3e-5.
    assert abs(a["loss"] - b["loss"]) <= 3e-5 * abs(b["loss"]), (a["loss"], b["loss"])
    # Gradient ceiling 3e-3 (the albedo step's test: 1e-3).  Every row gets the same values on both sides, but the rows sit in
    # different 128-row tiles (completion-order vs ray-order marcher), and the field backward sums the weight / bias gradients
    # per tile in the tensor cores' fp32 accumulators before its atomics.  The six stencil rows of a sample carry +-50 dg
    # (central difference, eps = 1e-2), and the pairs 2 eps apart mostly cancel in those sums, so the summation differences
    # are large relative to the result.  Measured on a B200, the same in four runs: worst 2.1e-4 at 1 view, 1.23e-3 at
    # 2 views (sigma_net.net.0.bias, textureless), 5.3e-4 lambertian, 3.4e-4 normal.
    worst = 0.0
    for name, gb in b["g"].items():
        ga = a["g"][name]
        assert gb.abs().max() > 0 and ga.abs().max() > 0, name
        rel = ((ga - gb).norm() / gb.norm()).item()
        worst = max(worst, rel)
        assert rel < 3e-3, (name, rel)
    print("shaded vs autograd (%s, %d views, %d chains): loss rel %.3g, worst gradient rel-L2 %.3g"
          % (shading, views, n_chunks, abs(a["loss"] - b["loss"]) / abs(b["loss"]), worst))
    if shading != "lambertian":      # the albedo outputs take no gradient: rows 1..3 of the last layer stay exactly zero
        for g in (a["g"], b["g"]):
            assert g["sigma_net.net.2.weight"][1:].abs().max() == 0 and g["sigma_net.net.2.bias"][1:].abs().max() == 0


# -- 2. the step's shade kernels against a float64 restatement -----------------------------------------------------------
def _h16(x):
    return np.asarray(x, np.float64).astype(np.float16).astype(np.float64)


def _shade_ref(sig7, alb, dirs, light, ratio, mode, d_sigma, d_rgb, lam_o, scale, total):
    """float64 numpy restatement of network_grid.py:90-140 (under autocast's half roundings), renderer.py:485-486 and their
    gradients, per sample."""
    sp, sm = sig7[:, 1::2], sig7[:, 2::2]
    g = -(0.5 * (sp - sm) * 100.0)
    nn = (g * g).sum(1, keepdims=True)
    den = np.sqrt(np.where(np.isnan(nn), nn, np.maximum(nn, 1e-20)))
    with np.errstate(invalid="ignore"):
        n = g / den
    nan = np.isnan(n)
    n = np.where(nan, 0.0, n)
    clamped = ~(nn[:, 0] >= 1e-20)
    dot = _h16((_h16(n) * _h16(light[None])).sum(1))
    lam = _h16(ratio + _h16((1 - ratio) * np.maximum(dot, 0)))
    if mode == 2:
        color = (n + 1) * 0.5
    elif mode == 1:
        color = np.repeat(lam[:, None], 3, 1)
    else:
        color = _h16(alb * lam[:, None])
    # backward
    w = 1 - np.exp(-sig7[:, 0])
    nd = np.maximum((n * dirs).sum(1), 0)
    orient = w * nd * nd
    dn = (scale * lam_o / total * w * 2 * nd)[:, None] * dirs
    d_alb = np.zeros_like(alb)
    if mode == 2:
        dn = dn + 0.5 * d_rgb
    else:
        d_lam = d_rgb.sum(1) if mode == 1 else (d_rgb * alb).sum(1)
        if mode == 0:
            d_alb = d_rgb * lam[:, None]
        dn = dn + np.where(dot >= 0, d_lam * (1 - ratio), 0.0)[:, None] * light[None]
    dnm = np.where(nan, 0.0, dn)
    inv = 1 / np.sqrt(np.maximum(np.nan_to_num(nn, nan=0.0), 1e-20))
    proj = (n * dnm).sum(1, keepdims=True)
    dg = np.where(clamped[:, None], dnm * inv, (dnm - n * proj) * inv)
    ds = np.nan_to_num(-0.5 * 100.0 * dg, nan=0.0)
    d_sig7 = np.zeros_like(sig7)
    d_sig7[:, 0] = d_sigma
    d_sig7[:, 1::2], d_sig7[:, 2::2] = ds, -ds
    d_rgb7 = np.zeros((sig7.shape[0], 7, 3))
    d_rgb7[:, 0] = d_alb
    return color, d_sig7, d_rgb7, lam_o * orient.sum() / total


@pytest.mark.parametrize("shading", list(MODES))
def test_shade_step_kernels_match_float64(shading):
    from ngp_b200 import _cabi, step_ops
    P, dev = _cabi.ptr, torch.device(DEV)
    mode, ratio, lam_o = MODES[shading], 0.1, 1e-2
    cap, M, M_other = 1000, 777, 300          # the step's samples: this chain's 777 + another chain's 300
    rng = np.random.default_rng(4)
    sig7 = rng.uniform(0.0, 20.0, (cap, 7)).astype(np.float32)
    sig7[5, 1:] = 3.0                                                            # |g|^2 = 0 < 1e-20: the clamp
    sig7[6, 1:] = (rng.uniform(1, 2, 6) * 1e-12).astype(np.float32)              # 0 < |g|^2 < 1e-20: the clamp, n != 0
    sig7[7, 1:] = np.inf                                                         # inf - inf: NaN normal -> 0
    alb = _h16(rng.uniform(0, 1, (cap, 7, 3))).astype(np.float32)
    dirs = rng.normal(size=(cap, 3))
    dirs = (dirs / np.linalg.norm(dirs, axis=1, keepdims=True)).astype(np.float32)
    light = np.array([0.3, -0.5, 0.81], np.float32)
    light /= np.linalg.norm(light)
    d_sigma = rng.normal(size=cap).astype(np.float32)
    d_rgb = rng.normal(size=(cap, 3)).astype(np.float32)
    scale = 1024.0
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)   # noqa: E731
    sig_d, alb_d, dirs_d, l_d, ds_d, dr_d = T(sig7), T(alb), T(dirs), T(light), T(d_sigma), T(d_rgb)
    counters = torch.tensor([[M, 0], [M_other, 0]], dtype=torch.int32, device=DEV)
    state = torch.tensor([scale], device=DEV)
    nanf = lambda *s: torch.full(s, float("nan"), device=DEV)   # noqa: E731
    sigma, rgb, d_sig_all, d_rgb_all = nanf(cap), nanf(cap, 3), nanf(7 * cap), nanf(7 * cap, 3)
    loss = torch.zeros((), device=DEV)
    _cabi.call("ngp_shade_forward_step", dev, P(sig_d), P(alb_d), cap, P(counters[0]), P(l_d), ratio, mode, P(sigma), P(rgb))
    _cabi.call("ngp_shade_backward_step", dev, P(sig_d), P(alb_d), cap, P(counters[0]), P(counters), 2, P(dirs_d), P(l_d), ratio,
               mode, P(ds_d), P(dr_d), lam_o, P(state), P(d_sig_all), P(d_rgb_all), P(loss))
    torch.cuda.synchronize()
    with np.errstate(invalid="ignore"):
        color, d_sig7, d_rgb7, loss_ref = _shade_ref(sig7[:M].astype(np.float64), alb[:M, 0].astype(np.float64), dirs[:M].astype(np.float64),
                                                     light.astype(np.float64), ratio, mode, d_sigma[:M],
                                                     d_rgb[:M].astype(np.float64), lam_o, scale, M + M_other)
    sigma, rgb = sigma.cpu().numpy(), rgb.cpu().numpy()
    d_sig_all, d_rgb_all = d_sig_all.cpu().numpy().reshape(cap, 7), d_rgb_all.cpu().numpy().reshape(cap, 7, 3)
    # rows past the device count keep the sentinel
    assert np.isnan(sigma[M:]).all() and np.isnan(rgb[M:]).all() and np.isnan(d_sig_all[M:]).all() and np.isnan(d_rgb_all[M:]).all()
    assert np.array_equal(sigma[:M], sig7[:M, 0])
    # (half-rounding boundaries: one half ulp at most)
    np.testing.assert_allclose(rgb[:M], color, rtol=0, atol=1e-3)
    assert np.isfinite(d_sig_all[:M]).all() and np.isfinite(d_rgb_all[:M]).all()
    assert np.array_equal(d_sig_all[:M, 0], d_sigma[:M])
    assert (d_sig_all[7, 1:] == 0).all() and (rgb[7] == color[7]).all()
    # sample 6 (0 < |g|^2 < 1e-20: gradients scaled by 1e10) on its own, the rest together
    rest = np.arange(M) != 6
    for got, ref in ((d_sig_all[:M], d_sig7), (d_rgb_all[:M], d_rgb7)):
        np.testing.assert_allclose(got[6], ref[6], rtol=1e-4, atol=0)
        got, ref = got[rest], ref[rest]
        if not ref.any():                       # d(albedo) of textureless / normal shading: exactly zero
            assert not got.any()
            continue
        rel = np.linalg.norm(got - ref) / np.linalg.norm(ref)
        assert rel < 1e-5, rel
        np.testing.assert_allclose(got, ref, rtol=1e-3, atol=1e-4 * np.abs(ref).max())
    assert abs(loss.item() - loss_ref) <= 1e-5 * abs(loss_ref), (loss.item(), loss_ref)
    # the stencil with a device count: 7 M rows (written as the count) equal the host-count version; the rest untouched
    x = torch.from_numpy(rng.uniform(-1, 1, (cap, 3)).astype(np.float32)).to(DEV)
    out, cnt = nanf(7 * cap, 3), torch.zeros(2, dtype=torch.int32, device=DEV)
    _cabi.call("ngp_stencil_points", dev, P(x), cap, P(counters[0]), 1e-2, 1.0, 1, P(out), P(cnt))
    torch.cuda.synchronize()
    assert cnt[0].item() == 7 * M
    assert torch.equal(out[:7 * M], step_ops.stencil_points(x[:M], 1e-2, 1.0, True)) and torch.isnan(out[7 * M:]).all()


# -- 3. graphs ---------------------------------------------------------------------------------------------------------
def test_shaded_graph_capture_leaves_no_training_side_effects():
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(1, 64, 64, seed=4, pin=False)
    ro, rd = ro.to(DEV), rd.to(DEV)
    G = torch.randn(1, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)) * 1e-2
    for pipelined in (False, True):
        m = _bench_like_model()
        step = TrainStep(m, 64, 64, lr=1e-3, graph=True, pipelined=pipelined, shading="lambertian")
        assert step.manual and step._shade_mode == 0
        with torch.autocast("cuda", torch.float16):
            m.update_extra_state()
        o = step.opt
        before = [t.clone() for t in (o.flat_params, o.flat_half, o.exp_avg, o.exp_avg_sq, o.state, m.step_counter, step.samples,
                                      step._rng)]
        step._capture(ro, rd, G)
        torch.cuda.synchronize()
        after = (o.flat_params, o.flat_half, o.exp_avg, o.exp_avg_sq, o.state, m.step_counter, step.samples, step._rng)
        for a, b in zip(before, after):
            assert torch.equal(a, b)
        assert o.flat_grads.abs().sum().item() == 0 and m.local_step == 0 and o.steps_taken == 0
        assert step._g_table_odd is None or step._g_table_odd.abs().sum().item() == 0, pipelined


@pytest.mark.parametrize("shading", ["lambertian", "textureless"])
def test_graphed_shaded_steps_follow_eager_steps(shading):
    """Six graphed steps vs six eager steps, noise and light pinned: the same samples; losses and parameter updates equal up
    to the fp32 atomics order of the scatter and the per-block loss sums, which Adam carries from step to step."""
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(6, 64, 64, seed=4, pin=False)
    ro, rd = ro.view(6, 1, 4096, 3).to(DEV), rd.view(6, 1, 4096, 3).to(DEV)
    G = torch.randn(6, 1, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)) * 1e-2
    gen = torch.Generator(device=DEV).manual_seed(9)
    noises = torch.rand(6, 4096, device=DEV, generator=gen)
    lights = torch.nn.functional.normalize(torch.randn(6, 3, device=DEV, generator=gen), dim=-1)
    runs = []
    for graph in (False, True):
        m = _bench_like_model()
        step = TrainStep(m, 64, 64, lr=1e-3, graph=graph, n_chunks=2, shading=shading)
        assert step.manual
        step.fixed_noises, step.fixed_light = torch.empty(4096, device=DEV), torch.empty(3, device=DEV)
        p0 = step.opt.flat_params.clone()
        torch.manual_seed(7)
        losses = []
        for i in range(6):
            step.fixed_noises.copy_(noises[i])
            step.fixed_light.copy_(lights[i])
            losses.append(step(ro[i], rd[i], G[i]).item())
        torch.cuda.synchronize()
        assert step.opt.steps_taken == 6
        runs.append(dict(losses=np.array(losses), samples=step.samples.item(), counter=m.step_counter.clone(),
                         delta=step.opt.flat_params - p0))
    e, g = runs
    assert e["samples"] == g["samples"] > 0 and torch.equal(e["counter"], g["counter"])
    loss_rel = float(np.abs(g["losses"] - e["losses"]).max() / np.abs(e["losses"]).max())
    upd_rel = ((g["delta"] - e["delta"]).norm() / e["delta"].norm()).item()
    print("graphed vs eager (%s): loss rel %.3g, update rel-L2 %.3g" % (shading, loss_rel, upd_rel))
    assert loss_rel < 8e-6, loss_rel      # measured on a B200: 3.8e-6 (lambertian and textureless)
    assert upd_rel < 2.5e-2, upd_rel      # measured: 1.08e-2 (lambertian), 1.20e-2 (textureless)


# -- 4. the device-side light draw ---------------------------------------------------------------------------------------
def _light_np(seed, ctr, ro0):
    u = np.array([_ray_noise_np_at(seed, ctr, 0xFFFFFFFF - j) for j in range(4)], np.float64)
    r0, r1 = np.sqrt(-2 * np.log(1 - u[0])), np.sqrt(-2 * np.log(1 - u[2]))
    z = np.array([r0 * np.cos(2 * np.pi * u[1]), r0 * np.sin(2 * np.pi * u[1]), r1 * np.cos(2 * np.pi * u[3])])
    x = ro0 + z
    return x / np.sqrt(max((x * x).sum(), 1e-20)), z


def _ray_noise_np_at(seed, ctr, n):
    from test_gpu_train_step import _mix32
    with np.errstate(over="ignore"):
        x = _mix32(np.array([n], np.uint32) ^ np.uint32(seed & 0xffffffff))
        x = _mix32((x + np.uint32((ctr * 0x9E3779B9) & 0xffffffff) + np.uint32((ctr >> 32) & 0xffffffff)).astype(np.uint32))
        x = _mix32(x ^ np.uint32((seed >> 32) & 0xffffffff))
    return float((x >> np.uint32(8)).astype(np.float32)[0] * np.float32(1.0 / 16777216.0))


def test_device_light_draw():
    from ngp_b200 import _cabi
    P, dev = _cabi.ptr, torch.device(DEV)
    assert np.isclose(_ray_noise_np_at(5, 3, 17), _ray_noise_np(5, 3, 18)[17])
    seed, n = 0x2545F4914F6CDD1D, 3000
    ro = torch.tensor([[0.2, -1.1, 2.5]], device=DEV)
    rng = torch.tensor([seed, 7, 0], dtype=torch.int64, device=DEV)
    out = torch.empty(n, 6, device=DEV)
    for i in range(n):
        _cabi.call("ngp_train_light", dev, P(ro), P(rng), 1, P(out[i]))
    torch.cuda.synchronize()
    assert rng.tolist() == [seed, 7 + n, 0]
    out = out.cpu().numpy().astype(np.float64)
    light, z = out[:, :3], out[:, 3:]
    np.testing.assert_allclose(np.linalg.norm(light, axis=1), 1.0, atol=1e-6)
    zz = z.reshape(-1)
    assert abs(zz.mean()) < 0.05 and abs(zz.var() - 1) < 0.06, (zz.mean(), zz.var())
    assert len(np.unique(out, axis=0)) == n      # a fresh draw every step
    for k in (0, 1, 2, 1234):                    # reproducible from (seed, step counter), on the keys documented
        l_ref, z_ref = _light_np(seed, 7 + k, ro[0].cpu().numpy().astype(np.float64))
        np.testing.assert_allclose(z[k], z_ref, rtol=0, atol=2e-5)
        np.testing.assert_allclose(light[k], l_ref, rtol=0, atol=2e-5)
    # advance = 0 (after a prologue that advanced the counter): the previous counter, generator left alone
    rng = torch.tensor([seed, 8, 0], dtype=torch.int64, device=DEV)
    again = torch.empty(6, device=DEV)
    _cabi.call("ngp_train_light", dev, P(ro), P(rng), 0, P(again))
    torch.cuda.synchronize()
    assert rng.tolist() == [seed, 8, 0] and np.array_equal(again.cpu().numpy(), out[0].astype(np.float32))


def test_graphed_shaded_step_draws_a_fresh_light_every_replay():
    from ngp_b200 import _cabi, provider
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(1, 64, 64, seed=4, pin=False)
    ro, rd = ro.to(DEV), rd.to(DEV)
    G = torch.randn(1, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)) * 1e-2
    m = _bench_like_model()
    step = TrainStep(m, 64, 64, lr=1e-5, graph=True, n_chunks=2, shading="textureless")
    assert step.manual and step.device_noise
    seen = []
    for k in range(3):
        step(ro, rd, G)
        torch.cuda.synchronize()
        assert step._rng[1].item() == k + 1
        seen.append(step._mws["light"].clone())
        # the one light of the step (every chain reads this buffer) is the draw of (seed, step k) at rays_o[0]
        ref = torch.empty(6, device=DEV)
        rng = step._rng.clone()
        _cabi.call("ngp_train_light", torch.device(DEV), _cabi.ptr(ro.reshape(-1, 3)), _cabi.ptr(rng), 0, _cabi.ptr(ref))
        torch.cuda.synchronize()
        assert torch.equal(ref, seen[-1])
        assert abs(seen[-1][:3].norm().item() - 1) < 1e-6
    assert len(step._mws["chunks"]) == 2
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])


# -- 5. guard bands ------------------------------------------------------------------------------------------------------
def test_shaded_step_writes_nothing_outside_its_buffers():
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    g = Guards()
    side = 27                                   # 729 rays: not a multiple of 32 or 128
    with g.active():
        model = _guard_model()
        poses, intr = provider.make_training_poses(1, side, side, seed=1)
        G = torch.randn(1, 3, side, side, device=DEV) * 1e-2
        for graph in (False, True):
            step = TrainStep(model, side, side, lr=1e-4, max_steps=200, graph=graph, manual=True, n_chunks=2,
                             device_rays=(side, 0, 1), shading="lambertian")
            assert step._shade_mode == 0
            for _ in range(3):
                step(poses.to(DEV), intr.to(DEV), G)
            step.flush()
        n, bad = g.check()
    assert n > 30, n
    assert bad == 0, "%d of %d guarded buffers were written outside their bounds" % (bad, n)


# -- 6. routing ----------------------------------------------------------------------------------------------------------
def test_shaded_step_routing():
    from ngp_b200.trainer import TrainStep
    m = _bench_like_model()
    for shading in MODES:
        step = TrainStep(m, 64, 64, shading=shading)
        assert step.manual and step._shade_mode == MODES[shading]
        assert not TrainStep(m, 64, 64, shading=shading, manual=False).manual
    assert TrainStep(m, 64, 64).manual and TrainStep(m, 64, 64)._shade_mode is None          # albedo: unchanged
    for kw, name in ((dict(lambda_smooth=0.1), "lambda_smooth"), (dict(world_size=2, peer_allreduce=False), "world_size"),
                     (dict(overlap=True), "overlap")):
        step = TrainStep(m, 64, 64, shading="lambertian", **kw)
        assert not step.manual and step._shade_mode is None, kw
        with pytest.raises(RuntimeError, match=name):
            TrainStep(m, 64, 64, shading="lambertian", manual=True, **kw)
