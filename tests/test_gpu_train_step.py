"""GPU tests of the one-launch train-step pieces (csrc/train_step.cu, csrc/adam.cu) against the torch ops the reference uses:
Adam + GradScaler (main.py:128-131, nerf/utils.py:708-713), the run_cuda tail (nerf/renderer.py:535-557) and the
entropy regulariser (nerf/utils.py:389-394)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _two_models():
    torch.manual_seed(3)
    shapes = [(1001, 2), (64, 32), (64,), (4, 64), (3,)]
    a = [torch.nn.Parameter(torch.randn(s, device=DEV) * 0.1) for s in shapes]
    b = [torch.nn.Parameter(p.detach().clone()) for p in a]
    return a, b


@pytest.mark.parametrize("layout", ["padded", "unpadded"])
def test_fused_adam_scaler_matches_torch_adam_and_gradscaler(layout):
    """padded: FusedAdamScaler.step, whose flat buffers pad every tensor to 8 elements.  unpadded: ngp_check_finite +
    ngp_adam_step called directly on the same parameters packed back to back - 4373 elements, so the last float4 is
    partial and the second lr group starts inside a float4 (element 2002)."""
    import ctypes
    import math
    from ngp_b200 import _cabi, field
    from ngp_b200.optim import FusedAdamScaler
    a, b = _two_models()
    lr = 1e-3
    groups = lambda ps: [{"params": ps[:1], "lr": lr * 10}, {"params": ps[1:], "lr": lr}]  # noqa: E731
    if layout == "padded":
        mine = FusedAdamScaler(groups(a), betas=(0.9, 0.99), eps=1e-15, growth_interval=3, lr_decay=(0.1, 10), grad_div=2.0)
        state, step, half = mine.state, mine.step, field.cached_half
    else:
        flat_p = torch.cat([p.detach().reshape(-1) for p in a])
        n = flat_p.numel()
        assert n % 4 == 1 and a[0].numel() % 4 == 2
        flat_g, m, v, flat_h = torch.zeros_like(flat_p), torch.zeros_like(flat_p), torch.zeros_like(flat_p), flat_p.half()
        state = torch.tensor([65536.0] + [0.0] * 7, device=DEV)
        done = torch.zeros(1, dtype=torch.int32, device=DEV)
        seg_end, seg_lr = (ctypes.c_uint64 * 2)(a[0].numel(), n), (ctypes.c_float * 2)(lr * 10, lr)
        halves, o = {}, 0
        for p in a:     # parameters and gradients become views of the flat buffers, as FusedAdamScaler makes them
            p.data, p.grad = flat_p[o:o + p.numel()].view_as(p), flat_g[o:o + p.numel()].view_as(p)
            halves[id(p)] = flat_h[o:o + p.numel()].view_as(p)
            o += p.numel()
        P = _cabi.ptr

        def step():
            _cabi.call("ngp_check_finite", DEV, P(flat_g), n, state[3:].data_ptr())
            _cabi.call("ngp_adam_step", DEV, P(flat_p), P(flat_g), P(m), P(v), P(flat_h), n, 2, seg_end, seg_lr, 0.9, 0.99,
                       1e-15, 2.0, math.log(0.1) / 10, 10.0, 2.0, 0.5, 3, 1, P(state), P(done))
        half = lambda p: halves[id(p)]  # noqa: E731
    opt = torch.optim.Adam(groups(b), betas=(0.9, 0.99), eps=1e-15)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda it: 0.1 ** min(it / 10, 1))
    scaler = torch.amp.GradScaler("cuda", growth_interval=3)
    scaler.scale(torch.zeros(1, device=DEV))        # GradScaler creates its device-side scale lazily
    g = torch.Generator(device=DEV).manual_seed(0)
    for it in range(12):
        raw = [torch.randn(p.shape, device=DEV, generator=g) * (10.0 ** (it % 5 - 3)) for p in a]
        if it == 5:
            raw[2][7] = float("inf")            # one overflow step: skipped, scale backs off
        if it == 8:
            raw[0][3, 1] = float("nan")
        s_mine, s_ref = state[0].item(), scaler.get_scale()
        assert s_mine == s_ref, (it, s_mine, s_ref)
        for p, q, r in zip(a, b, raw):
            p.grad.copy_(r * s_mine * 2.0)      # "all-reduced sum over 2 ranks" of scaled grads
            q.grad = r * s_ref
        step()
        scaler.step(opt)
        scaler.update()
        if it not in (5, 8):
            sched.step()                        # the Trainer steps the scheduler once per (successful) iteration
        for p, q in zip(a, b):
            assert torch.isfinite(p).all()
            np.testing.assert_allclose(p.detach().cpu().numpy(), q.detach().cpu().numpy(), rtol=2e-5, atol=1e-7)
            assert torch.equal(half(p), p.detach().half())                  # fp16 shadow follows the parameter
            assert p.grad.abs().sum().item() == 0                           # zero_grad folded in
    assert state[2].item() == 10 and state[4].item() == 2


def test_fused_adam_params_are_views_and_state_dict_keeps_names():
    import argparse
    from ngp_b200.network_grid import NeRFNetwork
    from ngp_b200.optim import FusedAdamScaler
    opt = argparse.Namespace(bound=1, cuda_ray=True, min_near=0.1, density_thresh=10, bg_radius=1.4)
    m = NeRFNetwork(opt).to(DEV)
    before = {k: v.clone() for k, v in m.state_dict().items()}
    o = FusedAdamScaler(m.get_params(1e-3))
    after = m.state_dict()
    assert list(before) == list(after)
    for k in before:
        assert torch.equal(before[k], after[k]), k
    assert o.numel >= sum(p.numel() for p in m.parameters())
    assert m.encoder.embeddings.data_ptr() == o.flat_params.data_ptr()
    m.load_state_dict(before)                   # in-place copies land in the flat buffer
    assert torch.equal(o.flat_params[:10], m.encoder.embeddings.detach().view(-1)[:10])


def test_blend_background_matches_torch_ops():
    from ngp_b200.step_ops import blend_background
    g = torch.Generator(device=DEV).manual_seed(1)
    N = 5000
    image = torch.rand(N, 3, device=DEV, generator=g).requires_grad_()
    ws = torch.rand(N, device=DEV, generator=g).requires_grad_()
    depth = torch.rand(N, device=DEV, generator=g) * 3
    nears = torch.rand(N, device=DEV, generator=g) + 0.2
    fars = nears + torch.rand(N, device=DEV, generator=g)
    fars[::17] = nears[::17] = 3.4028234663852886e38        # box misses
    up = torch.randn(N, 3, device=DEV, generator=g)
    for bg in (torch.rand(N, 3, device=DEV, generator=g).half().requires_grad_(), torch.ones(3, device=DEV), 1):
        img, dep, mask = blend_background(image, ws, depth, bg, nears, fars)
        want = image + (1 - ws).unsqueeze(-1) * bg
        want_d = torch.clamp(depth - nears, min=0) / (fars - nears)
        assert torch.allclose(img, want.float(), rtol=1e-6, atol=1e-6)
        assert torch.equal(torch.isnan(dep), torch.isnan(want_d)) and torch.allclose(dep[mask], want_d[mask], rtol=1e-6)
        assert torch.equal(mask, nears < fars)
        leaves = [image, ws] + ([bg] if torch.is_tensor(bg) and bg.requires_grad else [])
        got = torch.autograd.grad(img, leaves, up)
        ref = torch.autograd.grad(want, leaves, up)
        for x, y in zip(got, ref):
            assert torch.allclose(x.float(), y.float(), rtol=1e-3 if y.dtype == torch.half else 1e-5, atol=1e-5)


def test_entropy_loss_matches_torch_ops():
    from ngp_b200.step_ops import entropy_loss
    from ngp_b200.trainer import entropy_loss as torch_entropy
    g = torch.Generator(device=DEV).manual_seed(2)
    ws = torch.rand(2, 1, 64, 64, device=DEV, generator=g)
    ws.view(-1)[:100] = 0.0
    ws.view(-1)[100:200] = 1.0
    ws.view(-1)[200:300] = 1e-7
    ws.requires_grad_()
    scale = torch.tensor(65536.0, device=DEV)
    a = entropy_loss(ws, 1e-4)
    b = torch_entropy(ws, 1e-4)
    assert abs(a.item() - b.item()) < 1e-6 * abs(b.item()) + 1e-12
    ga, = torch.autograd.grad(a * scale, ws)
    gb, = torch.autograd.grad(b * scale, ws)
    assert torch.allclose(ga, gb, rtol=1e-4, atol=1e-7)


def test_train_step_fused_optimizer_tracks_torch_optimizer(ref_ext):
    """Whole TrainStep: fused Adam/scaler/blend/entropy path vs the torch.optim path, same seeds, a few steps."""
    import argparse
    from ngp_b200 import provider
    from ngp_b200.network_grid import NeRFNetwork
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(4, 64, 64, seed=3, pin=False)
    ro = ro.view(4, 1, 4096, 3).to(DEV); rd = rd.view(4, 1, 4096, 3).to(DEV)
    G = torch.randn(4, 1, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1)) * 1e-2
    finals = []
    for fused in (True, False):
        opt = argparse.Namespace(bound=1, cuda_ray=True, min_near=0.1, density_thresh=10, bg_radius=1.4)
        torch.manual_seed(0)
        m = NeRFNetwork(opt).to(DEV).train()
        step = TrainStep(m, 64, 64, lr=1e-3, graph=False, fused_optimizer=fused, manual=False)
        torch.manual_seed(5)
        losses = [step(ro[i], rd[i], G[i]).item() for i in range(4)]
        finals.append((losses, {n: p.detach().clone() for n, p in m.named_parameters()}))
    # identical first step (same parameters, same noise); afterwards Adam with eps=1e-15 moves every touched weight by
    # ~lr * sign(g), so last-bit gradient differences (atomics order, fused vs chained rounding) flip noise-level
    # entries and the two runs drift apart slowly - they must stay close, not equal
    assert abs(finals[0][0][0] - finals[1][0][0]) < 1e-4 * abs(finals[1][0][0])
    np.testing.assert_allclose(finals[0][0], finals[1][0], rtol=5e-2)
    for n in finals[0][1]:
        a, b = finals[0][1][n], finals[1][1][n]
        assert torch.isfinite(a).all()
        assert ((a - b).norm() / (b.norm() + 1e-12)).item() < 0.5, n


def test_fused_background_net_matches_torch_modules():
    """FreqEncoder + bg_net + sigmoid as one kernel each way vs the module chain under autocast (cuBLAS half GEMMs)."""
    import argparse
    from ngp_b200.network_grid import NeRFNetwork
    opt = argparse.Namespace(bound=1, cuda_ray=True, min_near=0.1, density_thresh=10, bg_radius=1.4)
    torch.manual_seed(0)
    m = NeRFNetwork(opt).to(DEV).train()
    g = torch.Generator(device=DEV).manual_seed(4)
    for N in (1, 100, 4096 + 37):
        d = torch.nn.functional.normalize(torch.randn(N, 3, device=DEV, generator=g), dim=-1)
        up = torch.randn(N, 3, device=DEV, generator=g) * 1e-2
        res = []
        for fused in (True, False):
            m.fused = fused
            m.zero_grad(set_to_none=True)
            with torch.autocast("cuda", torch.float16):
                y = m.background(d)
            assert y.dtype == torch.half and y.shape == (N, 3)
            y.float().backward(up)
            res.append((y.detach().float(), {n: p.grad.clone() for n, p in m.bg_net.named_parameters()}))
        assert torch.allclose(res[0][0], res[1][0], atol=2e-3), (res[0][0] - res[1][0]).abs().max().item()
        for n in res[0][1]:
            a, b = res[0][1][n].float(), res[1][1][n].float()
            rel = ((a - b).norm() / b.norm().clamp_min(1e-12)).item()
            assert rel < 2e-2, (N, n, rel)       # the torch path rounds weight gradients (and their split-K partials) to fp16


def _bench_like_model():
    import argparse
    from ngp_b200.network_grid import NeRFNetwork
    opt = argparse.Namespace(bound=1, cuda_ray=True, min_near=0.1, density_thresh=10, bg_radius=1.4)
    torch.manual_seed(0)
    return NeRFNetwork(opt).to(DEV).train()


@pytest.mark.parametrize("views,n_chunks", [(1, 1), (1, 2), (2, 1), (2, 3)])
def test_hand_scheduled_step_matches_autograd_step(views, n_chunks):
    """TrainStep(manual=True) - 13 launches, no autograd - must produce the gradients, loss and bookkeeping of the
    autograd version of the same step (which tests/test_gpu_pipeline.py pins to the reference pipeline)."""
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(views, 64, 64, seed=3, pin=False)
    ro, rd = ro.to(DEV), rd.to(DEV)
    G = torch.randn(views, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1)) * 1e-2
    got = {}
    for manual in (True, False):
        m = _bench_like_model()
        step = TrainStep(m, 64, 64, lr=1e-3, graph=False, manual=manual, n_chunks=n_chunks)   # chunks: parallel ray chains
        assert step.manual == manual
        step.mirror_rng = True   # same torch RNG consumption as run_cuda, so both draw the same ray noise
        grads = []

        def capture(*a, _s=step, _g=grads, **k):
            if _s.manual:
                _s.fold_table_grads()     # (the step folds the split scatter's twin inside the optimizer's finite check)
            _g.append(_s.opt.flat_grads.clone())
            _s.opt.flat_grads.zero_()
        step.opt.step = capture
        torch.manual_seed(5)
        loss = step(ro, rd, G)
        torch.cuda.synchronize()
        got[manual] = dict(loss=loss.item(), g=grads[0], opt=step.opt, counter=m.step_counter.clone(), samples=step.samples.item(),
                           local_step=m.local_step, model=m)
    a, b = got[True], got[False]
    assert a["samples"] == b["samples"] > 0
    assert torch.equal(a["counter"], b["counter"]) and a["local_step"] == b["local_step"] == 1
    assert abs(a["loss"] - b["loss"]) <= 1e-5 * abs(b["loss"])   # (per-block atomics: summation order differs)
    for (name, p), (_, q) in zip(a["model"].named_parameters(), b["model"].named_parameters()):
        oa, ob = a["opt"].offsets[a["opt"]._index(p)], b["opt"].offsets[b["opt"]._index(q)]
        ga, gb = a["g"][oa:oa + p.numel()], b["g"][ob:ob + q.numel()]
        assert gb.abs().max() > 0, name
        rel = ((ga - gb).norm() / gb.norm()).item()
        assert rel < 1e-3, (name, rel)   # fp32 atomics order is the only difference


def test_hand_scheduled_step_graph_replay_and_packed_inputs():
    """Graph replays of the hand-scheduled step (optimizer launches + side-stream branch inside the graph)
    follow the eager step; packed inputs reach the static buffers with one copy."""
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(6, 64, 64, seed=4, pin=False)
    ro, rd = ro.view(6, 1, 4096, 3).to(DEV), rd.view(6, 1, 4096, 3).to(DEV)
    G = torch.randn(6, 1, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)) * 1e-2
    out = []
    for graph in (False, True):
        m = _bench_like_model()
        step = TrainStep(m, 64, 64, lr=1e-4, graph=graph, manual=True)
        torch.manual_seed(7)
        losses = []
        for i in range(6):
            if graph and i % 2 == 1:
                losses.append(step(step.pack_inputs(ro[i], rd[i], G[i])).item())
            else:
                losses.append(step(ro[i], rd[i], G[i]).item())
        torch.cuda.synchronize()
        assert not step.opt.comm_error
        assert step.opt.steps_taken == 6   # the capture's warm-up steps are rolled back (trainer._capture)
        out.append((losses, step.samples.item(), m.step_counter.clone(), m.local_step))
    (la, sa, ca, lsa), (lb, sb, cb, lsb) = out
    assert lsa == lsb == 6 and sa > 0 and sb > 0
    # different noise draws in the graphed run (its warm-up consumed torch RNG): the loss stays in the same range
    np.testing.assert_allclose(la, lb, rtol=0.2)
    assert (ca[:6, 1] == 4096).all() and (cb[:6, 1] == 4096).all()
    assert abs(sa - sb) < 0.2 * sa


def test_graph_capture_leaves_no_training_side_effects():
    """The three warm-up steps before capture are REAL steps; parameters, fp16 shadow, Adam moments, step count, loss
    scale, step_counter and the sample total must be exactly what they were before the capture."""
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(1, 64, 64, seed=4, pin=False)
    ro, rd = ro.to(DEV), rd.to(DEV)
    G = torch.randn(1, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)) * 1e-2
    for manual, pipelined in ((True, False), (True, True), (False, False)):
        m = _bench_like_model()
        step = TrainStep(m, 64, 64, lr=1e-3, graph=True, manual=manual, pipelined=pipelined)
        with torch.autocast("cuda", torch.float16):
            m.update_extra_state()
        o = step.opt
        before = [t.clone() for t in (o.flat_params, o.flat_half, o.exp_avg, o.exp_avg_sq, o.state, m.step_counter, step.samples)]
        step._capture(ro, rd, G)
        torch.cuda.synchronize()
        after = (o.flat_params, o.flat_half, o.exp_avg, o.exp_avg_sq, o.state, m.step_counter, step.samples)
        for a, b in zip(before, after):
            assert torch.equal(a, b)
        assert o.flat_grads.abs().sum().item() == 0 and m.local_step == 0 and o.steps_taken == 0
        # the odd-row twin of the table gradient too (pipelined: the last warm-up update, which folds it, is still pending)
        assert step._g_table_odd is None or step._g_table_odd.abs().sum().item() == 0, pipelined


def test_pixel_sharded_ranks_sum_to_the_one_gpu_step():
    """Data parallel = the same step: two virtual ranks, each rendering its interleaved rows of every view (bench.py's
    sharding), must produce gradient buckets whose SUM is the bucket of one GPU rendering all rays - guidance summed per
    pixel, entropy averaged over ALL rays of the job (nerf/sd.py:115, nerf/utils.py:389-394)."""
    from ngp_b200 import provider
    from ngp_b200.parallel import shard_rows
    from ngp_b200.trainer import TrainStep
    views, Hh, Ww, world = 2, 64, 64, 2
    ro, rd = provider.make_training_views(views, Hh, Ww, seed=3, pin=False)
    ro, rd = ro.to(DEV), rd.to(DEV)
    G = torch.randn(views, 3, Hh, Ww, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1)) * 1e-2
    noises = torch.rand(views * Hh * Ww, device=DEV, generator=torch.Generator(device=DEV).manual_seed(9))

    def one(rows, world_size):
        m = _bench_like_model()
        Hl = len(rows)
        step = TrainStep(m, Hl, Ww, lr=1e-3, graph=False, manual=True, world_size=world_size, peer_allreduce=False, lambda_entropy=1e-2)
        idx = torch.tensor(rows, device=DEV)
        sel = lambda t: t.view(views, Hh, Ww, 3)[:, idx].reshape(views, Hl * Ww, 3).contiguous()  # noqa: E731
        step.fixed_noises = noises.view(views, Hh, Ww)[:, idx].reshape(-1).contiguous()
        grads = []
        step._apply_update = lambda deferred=False, _s=step, _g=grads: (_s.fold_table_grads(), _g.append(_s.opt.flat_grads.clone()),
                                                                        _s.opt.flat_grads.zero_())
        loss = step(sel(ro), sel(rd), G[:, :, idx].contiguous())
        torch.cuda.synchronize()
        return grads[0], loss.item(), step.opt.get_scale(), int(step.samples.item())

    g_full, l_full, scale, n_full = one(list(range(Hh)), 1)
    parts = [one(shard_rows(Hh, r, world), world) for r in range(world)]
    assert sum(p[3] for p in parts) == n_full            # the same samples, split
    g_sum = sum(p[0] for p in parts)
    assert abs(sum(p[1] for p in parts) - l_full) <= 1e-5 * abs(l_full)
    rel = ((g_sum - g_full).norm() / g_full.norm()).item()
    assert rel < 1e-3, rel
    # and the entropy term really is in there at a visible weight: dropping the 1/world would be caught
    assert l_full > 0 and scale == 65536.0


def test_pipelined_optimizer_applies_the_same_updates_one_step_later():
    """pipelined=True defers step k's optimizer launch to the start of step k+1 (beside the ray marching); after
    flush() the same number of updates has been applied and the parameters agree with the un-pipelined run."""
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(5, 64, 64, seed=4, pin=False)
    ro, rd = ro.view(5, 1, 4096, 3).to(DEV), rd.view(5, 1, 4096, 3).to(DEV)
    G = torch.randn(5, 1, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)) * 1e-2
    finals = []
    for pipelined in (False, True):
        m = _bench_like_model()
        step = TrainStep(m, 64, 64, lr=1e-4, graph=False, manual=True, pipelined=pipelined)
        torch.manual_seed(7)
        losses = [step(ro[i], rd[i], G[i]).item() for i in range(5)]
        if pipelined:
            assert step.opt.steps_taken == 4            # the fifth update is still pending
            step.flush()
            step.flush()                                # idempotent
        assert step.opt.steps_taken == 5 and step.opt.state[4].item() == 0
        assert step.opt.flat_grads.abs().sum().item() == 0
        finals.append((losses, {n: p.detach().clone() for n, p in m.named_parameters()}))
    # step 1 sees identical parameters in both runs; afterwards only the atomics' summation order differs
    assert abs(finals[0][0][0] - finals[1][0][0]) <= 1e-6 * abs(finals[0][0][0])
    np.testing.assert_allclose(finals[0][0], finals[1][0], rtol=2e-2)
    for n in finals[0][1]:
        a, b = finals[0][1][n], finals[1][1][n]
        assert ((a - b).norm() / (b.norm() + 1e-12)).item() < 0.05, n


@pytest.mark.parametrize("split", [1, 2])
def test_train_ray_loss_kernel_vs_oracle(split):
    """ngp_train_ray_loss (composite fwd + blend + loss gradients + composite bwd, one launch) through the C ABI against
    the oracle restatement (oracle.train_ray_loss: C composite kernels + numpy blend / entropy), on marched samples of a
    blob scene; split = 2 runs it as two ray chunks (ray_base / n_rays_total), as the two-chain train step does."""
    import ngp_testutil as util
    from ngp_b200 import _cabi
    from oracle import oracle as O
    side, views = 16, 2
    rays_o, rays_d = [], []
    for v in range(views):
        ro, rd = util.look_at_rays(side, phi_deg=30.0 + 100.0 * v)
        rays_o.append(ro); rays_d.append(rd)
    rays_o, rays_d = np.concatenate(rays_o), np.concatenate(rays_d)
    N, hw = rays_o.shape[0], side * side
    grid = util.blob_density_grid(1, 128, 1.0, 0)
    bits = O.packbits(grid, 10.0)
    nears, fars = O.near_far_from_aabb(rays_o, rays_d, np.array([-1, -1, -1, 1, 1, 1], np.float32), 0.2)
    noises = np.random.default_rng(1).random(N).astype(np.float32)
    ox, _, ol, orays, ocnt = O.march_rays_train(rays_o, rays_d, 1.0, bits, 1, 128, nears, fars, noises, 0.0, 256)
    total = int(ocnt[0])
    assert total > 1000 and np.array_equal(orays[:, 0], np.arange(N))
    sig, rgb = util.pseudo_field(ox[:total])
    rng = np.random.default_rng(2)
    bg = rng.uniform(0, 1, (N, 3)).astype(np.float16)
    G = (rng.standard_normal((views, 3, hw)) * 1e-2).astype(np.float32)
    lam, scale = 1e-4, 65536.0
    want = O.train_ray_loss(sig, rgb, ol[:total], orays, bg.astype(np.float32), G, hw, lam, scale, 1e-4)

    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    sig_t, rgb_t, dl_t, bg_t, G_t = T(sig), T(rgb), T(ol[:total]), T(bg), T(G)
    scale_t = torch.tensor([scale], device=DEV)
    ws = torch.full((N,), -1.0, device=DEV); depth = torch.empty(N, device=DEV); image = torch.empty(N, 3, device=DEV)
    d_bg = torch.empty(N, 3, device=DEV)
    gs = torch.full((total,), 7.0, device=DEV); gc = torch.full((total, 3), 7.0, device=DEV)
    loss = torch.zeros((), device=DEV)
    samples = torch.zeros(1, dtype=torch.int64, device=DEV)
    step_counter = torch.zeros(16, 2, dtype=torch.int32, device=DEV)
    cur_row = torch.full((1,), 3, dtype=torch.int32, device=DEV)
    P = _cabi.ptr
    bounds = [0, N] if split == 1 else [0, N // 2 + 5, N]
    for lo, hi in zip(bounds, bounds[1:]):
        rays_c = orays[lo:hi].copy()
        rays_c[:, 0] -= lo                       # ray ids are local to the chunk; offsets stay global rows of the buffers
        cnt = torch.tensor([int(rays_c[:, 2].sum()), hi - lo], dtype=torch.int32, device=DEV)
        rays_t = T(rays_c)
        _cabi.call("ngp_train_ray_loss", torch.device(DEV), P(sig_t), P(rgb_t), P(dl_t), P(rays_t), total, hi - lo, 1e-4,
                   P(bg_t[lo:hi]), 1.0, P(G_t), hw, lo, N, lam, P(scale_t), P(ws[lo:hi]), P(depth[lo:hi]), P(image[lo:hi]),
                   P(d_bg[lo:hi]), P(gs), P(gc), P(loss), P(cnt), P(samples), P(step_counter), P(cur_row))
    torch.cuda.synchronize()
    N_ = lambda t: t.detach().cpu().numpy()  # noqa: E731
    for got, name in ((ws, "weights_sum"), (depth, "depth"), (image, "image"), (d_bg, "grad_bg")):
        np.testing.assert_allclose(N_(got), want[name], rtol=1e-5, atol=1e-6, err_msg=name)
    assert abs(loss.item() - want["loss"]) <= 1e-5 * abs(want["loss"])
    sc = max(np.abs(want["grad_sigmas"]).max(), 1e-6)
    assert np.abs(N_(gs) - want["grad_sigmas"]).max() < 1e-4 * sc + 1e-6
    np.testing.assert_allclose(N_(gc), want["grad_rgbs"], rtol=1e-5, atol=1e-7)
    assert samples.item() == total
    assert step_counter[3].tolist() == [total, N] and step_counter.sum().item() == total + N


def test_device_get_rays_matches_the_reference_golden():
    """ngp_get_rays (nerf/utils.py:43-106 on the device) against rays the REAL reference generated
    (tests/golden/rays_golden.npz, oracle/make_golden_host.py), full images and a rank's interleaved rows."""
    import os
    from ngp_b200 import provider
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rays_golden.npz"))
    H, W = int(gold["H"]), int(gold["W"])
    poses = torch.from_numpy(gold["poses"]).to(DEV)
    for tag in ("a", "b"):
        intr = torch.from_numpy(gold["intrinsics_" + tag]).to(DEV)
        ro, rd = provider.get_rays_device(poses, intr, H, W)
        assert np.array_equal(ro.cpu().numpy(), gold["rays_o_" + tag])
        np.testing.assert_allclose(rd.cpu().numpy(), gold["rays_d_" + tag], rtol=0, atol=2e-7)
        # per-view intrinsics + row sharding: rank 1 of 3 renders rows 1, 4, 7, ...
        rows = list(range(1, H, 3))
        ro_s, rd_s = provider.get_rays_device(poses, intr[None].repeat(poses.shape[0], 1).contiguous(), H, W, row0=1, row_stride=3)
        want = rd.view(-1, H, W, 3)[:, rows].reshape(poses.shape[0], -1, 3)
        assert torch.equal(rd_s, want) and ro_s.shape == want.shape


def test_device_rays_step_equals_the_host_rays_step():
    """TrainStep(device_rays=...): poses + intrinsics in, rays generated by the prologue kernel - the same step as feeding
    the (identical) rays from outside: bit-equal sample counts, gradients equal up to atomics order."""
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    views = 2
    poses, intr = provider.make_training_poses(views, 64, 64, seed=3)
    poses, intr = poses.to(DEV), intr.to(DEV)
    ro, rd = provider.get_rays_device(poses, intr, 64, 64)
    G = torch.randn(views, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1)) * 1e-2
    noises = torch.rand(views * 4096, device=DEV, generator=torch.Generator(device=DEV).manual_seed(9))
    got = []
    for device_rays, graph in ((None, False), ((64, 0, 1), False), ((64, 0, 1), True)):
        m = _bench_like_model()
        step = TrainStep(m, 64, 64, lr=0.0, graph=graph, manual=True, device_rays=device_rays)
        step.fixed_noises, step.keep_grads = noises, True
        if device_rays is None:
            loss = step(ro, rd, G)
        elif graph:
            loss = step(step.pack_pose_inputs(poses, intr, G))
        else:
            loss = step(poses, intr, G)
        torch.cuda.synchronize()
        got.append((loss.item(), step.grad_snapshot.clone(), int(step.samples.item()), m.step_counter[0].clone()))
    for other in got[1:]:
        assert other[2] == got[0][2] > 0 and torch.equal(other[3], got[0][3])
        assert abs(other[0] - got[0][0]) <= 1e-5 * abs(got[0][0])   # (fp32 atomic sum over the rays: the order varies)
        rel = ((other[1] - got[0][1]).norm() / got[0][1].norm()).item()
        assert rel < 1e-4, rel


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("device_rays", [False, True])
def test_overlapped_steps_match_sequential_steps(device_rays, fused, monkeypatch):
    """overlap=True runs the marching half of step k+1 beside the compute half of step k - as the two branches of ONE graph
    per call (fused, the default) or as two graphs on two streams tied by events; two workspace sets either way.  Parameter
    updates, sample counts and run_cuda's bookkeeping must be those of the sequential graphed step - across an occupancy
    refresh too (22 steps, update_interval 16)."""
    monkeypatch.setenv("NGP_OVERLAP_FUSED", "1" if fused else "0")
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    n_steps, views = 22, 2
    poses, intr = provider.make_training_poses(n_steps * views, 64, 64, seed=5)
    poses, intr = poses.view(n_steps, views, 4, 4).to(DEV), intr.view(n_steps, views, 4).to(DEV)
    G = torch.randn(n_steps, views, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)) * 1e-2
    noises = torch.rand(views * 4096, device=DEV, generator=torch.Generator(device=DEV).manual_seed(9))
    out = []
    for overlap in (False, True):
        m = _bench_like_model()
        step = TrainStep(m, 64, 64, lr=1e-4, graph=True, manual=True, overlap=overlap, device_rays=(64, 0, 1) if device_rays else None)
        step.fixed_noises = noises
        torch.manual_seed(3)       # the occupancy refresh draws its jitter from torch's generator
        losses = []
        for i in range(n_steps):
            if device_rays:
                batch = step.pack_pose_inputs(poses[i], intr[i], G[i])
            else:
                ro, rd = provider.get_rays_device(poses[i], intr[i], 64, 64)
                batch = step.pack_inputs(ro, rd, G[i])
            losses.append(float(step(batch).item()))
        step.flush()
        torch.cuda.synchronize()
        assert step.opt.steps_taken == n_steps and step.n_updates == 2 and not step.opt.comm_error
        out.append(dict(params={n: p.detach().clone() for n, p in m.named_parameters()}, samples=int(step.samples.item()),
                        counter=m.step_counter.clone(), local_step=m.local_step, losses=losses, bits=m.density_bitfield.clone()))
    a, b = out
    assert a["samples"] == b["samples"] > 0 and a["local_step"] == b["local_step"]
    assert torch.equal(a["counter"], b["counter"]) and torch.equal(a["bits"], b["bits"])
    # the overlapped run reports losses late: loss[k] of the sequential run == returned[k + lag]
    lag = 3 if fused else 2
    np.testing.assert_allclose(b["losses"][lag:], a["losses"][:-lag], rtol=1e-4)
    for n in a["params"]:
        rel = ((a["params"][n] - b["params"][n]).norm() / a["params"][n].norm()).item()
        assert rel < 1e-3, (n, rel)         # same updates in the same order; fp32 atomics order is the only difference


def test_read_loss_async_returns_the_lagged_loss_without_a_sync():
    """TrainStep.read_loss_async: every call copies the step's loss to a pinned ring and hands back the loss of `lag`
    calls ago - the values loss.item() would have returned, two calls later."""
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    views, n_steps = 1, 7
    poses, intr = provider.make_training_poses(n_steps * views, 64, 64, seed=8)
    poses, intr = poses.view(n_steps, views, 4, 4).to(DEV), intr.view(n_steps, views, 4).to(DEV)
    G = torch.randn(n_steps, views, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(4)) * 1e-2
    m = _bench_like_model()
    step = TrainStep(m, 64, 64, lr=1e-3, graph=True, manual=True, device_rays=(64, 0, 1))
    sync, lagged = [], []
    for i in range(n_steps):
        loss = step(step.pack_pose_inputs(poses[i], intr[i], G[i]))
        lagged.append(step.read_loss_async(lag=2))
        sync.append(float(loss.item()))
    assert lagged[:2] == [None, None]
    np.testing.assert_allclose(lagged[2:], sync[:-2], rtol=0, atol=0)
    assert len(set(sync)) > 1 and all(np.isfinite(sync))


def _mix32(x):
    x = x.astype(np.uint32)
    x ^= x >> np.uint32(16); x = (x * np.uint32(0x7feb352d)).astype(np.uint32)
    x ^= x >> np.uint32(15); x = (x * np.uint32(0x846ca68b)).astype(np.uint32)
    x ^= x >> np.uint32(16)
    return x


def _ray_noise_np(seed, ctr, n):
    """numpy restatement of csrc/raymarch.cu ray_noise (counter-based per-ray jitter of the hand-scheduled step)."""
    n = np.arange(n, dtype=np.uint32)
    with np.errstate(over="ignore"):
        x = _mix32(n ^ np.uint32(seed & 0xffffffff))
        x = _mix32((x + np.uint32((ctr * 0x9E3779B9) & 0xffffffff) + np.uint32((ctr >> 32) & 0xffffffff)).astype(np.uint32))
        x = _mix32(x ^ np.uint32((seed >> 32) & 0xffffffff))
    return (x >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)


def test_device_side_ray_noise():
    """The prologue kernel draws the per-ray march jitter itself (the reference: torch.rand(N), raymarching.py:213-216):
    values in [0, 1), reproducible from (seed, step counter, ray), a fresh draw every launch, counter advanced by exactly one."""
    from ngp_b200 import _cabi
    N = 5000
    g = torch.Generator(device=DEV).manual_seed(0)
    ro = torch.randn(N, 3, device=DEV, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 3.0], device=DEV)
    rd = torch.nn.functional.normalize(torch.randn(N, 3, device=DEV, generator=g) * 0.2 - torch.tensor([0.0, 0.0, 1.0], device=DEV), dim=-1)
    aabb = torch.tensor([-1.0, -1, -1, 1, 1, 1], device=DEV)
    nears, fars, noises = (torch.empty(N, device=DEV) for _ in range(3))
    seed = 0x123456789ABCDEF
    rng = torch.tensor([seed, 7, 0], dtype=torch.int64, device=DEV)
    P = _cabi.ptr
    draws = []
    for k in range(3):
        _cabi.call("ngp_train_prologue", torch.device(DEV), P(ro), P(rd), P(aabb), N, 0.2, P(nears), P(fars), None, 0, None, None,
                   None, None, P(noises), P(rng))
        torch.cuda.synchronize()
        assert rng.tolist() == [seed, 8 + k, 0]
        draws.append(noises.cpu().numpy().copy())
        assert np.array_equal(draws[-1], _ray_noise_np(seed, 7 + k, N))
    u = np.concatenate(draws)
    assert u.min() >= 0.0 and u.max() < 1.0 and abs(u.mean() - 0.5) < 0.01 and abs(u.var() - 1 / 12) < 0.005
    assert not np.array_equal(draws[0], draws[1])
    assert abs(np.corrcoef(draws[0], draws[1])[0, 1]) < 0.05 and abs(np.corrcoef(draws[0][:-1], draws[0][1:])[0, 1]) < 0.05
    # without a noise buffer the launch leaves the generator alone
    _cabi.call("ngp_train_prologue", torch.device(DEV), P(ro), P(rd), P(aabb), N, 0.2, P(nears), P(fars), None, 0, None, None,
               None, None, None, None)
    torch.cuda.synchronize()
    assert rng.tolist() == [seed, 10, 0]


def test_graphed_step_draws_fresh_noise_every_replay():
    """Graph replays of the hand-scheduled step advance the device-side generator (no torch generator inside the graph)."""
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(1, 64, 64, seed=4, pin=False)
    ro, rd = ro.to(DEV), rd.to(DEV)
    G = torch.randn(1, 3, 64, 64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)) * 1e-2
    m = _bench_like_model()
    step = TrainStep(m, 64, 64, lr=1e-5, graph=True, manual=True)
    assert step.device_noise
    seen = []
    for k in range(3):
        step(ro, rd, G)
        torch.cuda.synchronize()
        assert step._rng[1].item() == k + 1 and step._rng[2].item() == 0
        seen.append(step._mws["noises"].clone())
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])
    assert np.array_equal(seen[2].cpu().numpy(), _ray_noise_np(int(step._rng[0].item()), 2, 4096))
