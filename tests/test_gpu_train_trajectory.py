"""The hand-scheduled train step that bench.py times, run for 20 steps at a learning rate that moves the scene, and
checked step by step against independent references (teacher forcing: every check starts from the implementation's
own state right before the step, so nothing drifts and the tolerances stay tight):

  (a) gradients: the bucket the optimizer consumed (odd-row twin of the table gradient folded in) against the fp64 step
      oracle and the reference pipeline at the parameters, rays, noise and loss scale of that step;
  (b) optimizer: parameters, Adam moments, fp16 shadow and GradScaler state after every update against the float64
      Adam + GradScaler + LambdaLR restatement (oracle.adam_scaler_step) - including one skipped (inf) step;
  (c) carried state: zeroed gradient bucket and twin, the quad table rebuilt from the shadow the forward read, the
      step_counter ring, the sample total and the device-side noise counter;
  (d) occupancy refresh (steps 0 and 16): cell points, grid and bitfield bit-exact against the C oracle, densities
      against the fp64 field at the parameters of the completed previous update.

Every number goes to trajectory_parity.json, next to step_parity.json (test_gpu_step_parity._report).
"""
import hashlib
import time

import numpy as np
import pytest
import torch

from test_gpu_step_parity import _closer_or_equal, _enc_consts, _field_params, _np, _ref_step, _report, _step_truth
from test_gpu_train_step import _bench_like_model, _ray_noise_np

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
REPORT = {}
_REF_CACHE = {}

N_STEPS, SKIP_STEP, HW = 20, 9, 64
LR, GROWTH_INTERVAL = 1e-3, 4
CONFIGS = {
    # bench.py's one-GPU step
    "graph": dict(kw=dict(graph=True, device_rays=(HW, 0, 1)), env={}, grad_steps=(0, 1, 2, 7, 15, 16, 19)),
    # the schedule of the multi-GPU default: step k's update runs at the start of step k + 1
    "graph_pipelined": dict(kw=dict(graph=True, device_rays=(HW, 0, 1), pipelined=True), env={}, grad_steps=(0, 16, 19)),
    # bench.py's one-GPU step with a LambdaLR decay that saturates at step 10
    "graph_lr_decay": dict(kw=dict(graph=True, device_rays=(HW, 0, 1), lr_decay=(0.1, 10)), env={}, grad_steps=(0, 16, 19)),
    # eager, host rays, the fallback kernels: per-level gathers, one-buffer scatter, ray-ordered marcher
    "eager_fallbacks": dict(kw=dict(graph=False), env={"NGP_QUAD_TABLE": "0", "NGP_SPLIT_SCATTER": "0", "NGP_PACKED_MARCH": "0"},
                            grad_steps=(0, 16, 19)),
}

# rel-L2 of the consumed gradient to the fp64 step oracle, per tensor: ceilings at 2x the worst value measured over the
# checked steps of all four configurations (NVIDIA B200, 1000 W power limit); the worst value in the comment.  They are
# largest at step 0 (default init: tiny table, fp16 weight rounding dominates) and shrink as the scene forms.
GRAD_CEILING = {"encoder.embeddings": 0.04,         # 0.0195 (step 1)
                "sigma_net.net.0.weight": 0.023,    # 0.0111 (step 0)
                "sigma_net.net.0.bias": 0.014,      # 0.0066 (step 0)
                "sigma_net.net.1.weight": 0.0046,   # 0.0023 (step 0)
                "sigma_net.net.1.bias": 0.0046,     # 0.0023 (step 0)
                "sigma_net.net.2.weight": 5e-4,     # 0.00023 (step 0)
                "sigma_net.net.2.bias": 5e-4,       # 0.00023 (step 0)
                "bg_net.net.0.weight": 0.0083,      # 0.0040 (step 2; the reference: 0.0041)
                "bg_net.net.0.bias": 0.0083,        # 0.0041 (step 2; the reference: 0.0042)
                "bg_net.net.1.weight": 0.001,       # 0.00046
                "bg_net.net.1.bias": 0.0017}        # 0.00083
# refresh densities against the fp64 field at the parameters of the completed previous update, max relative error over
# 2^16 cells: measured 1.2e-4 at step 16, 7.7e-6 at step 0 (NVIDIA B200, 1000 W power limit)
SIGMA_REL = 5e-4


class _Recorder:
    """Wraps TrainStep._apply_update (and flush): every optimizer launch first copies the gradient bucket and the odd-row
    twin it is about to consume into buffers allocated up front, and copies them again once the launch has run.  Copies
    are capturable, so this works inside the replayed graph too; a flush() (eager, never captured) copies into a second
    set, so that the arm-only launch of the step after a flush does not overwrite what the flush consumed."""

    def __init__(self, step):
        self.step, self.opt = step, step.opt
        step._manual_consts()                       # allocates the twin and the quad table (the first call would)
        odd = step._g_table_odd
        z = lambda t: None if t is None else torch.zeros_like(t)  # noqa: E731
        self.sets = {k: dict(g=z(self.opt.flat_grads), odd=z(odd), g_after=z(self.opt.flat_grads), odd_after=z(odd))
                     for k in ("step", "flush")}
        self.in_flush = False
        orig_apply, orig_flush = step._apply_update, step.flush

        def apply_update(deferred):
            s = self.sets["flush" if self.in_flush else "step"]
            s["g"].copy_(self.opt.flat_grads)
            if odd is not None:
                s["odd"].copy_(odd)
            orig_apply(deferred=deferred)
            s["g_after"].copy_(self.opt.flat_grads)
            if odd is not None:
                s["odd_after"].copy_(odd)

        def flush():
            self.in_flush = True
            try:
                orig_flush()
            finally:
                self.in_flush = False

        step._apply_update, step.flush = apply_update, flush

    def take(self, which):
        return {k: (None if v is None else v.clone()) for k, v in self.sets[which].items()}


def _snapshot(step, model):
    torch.cuda.synchronize()
    o = step.opt
    c = lambda t: None if t is None else t.clone()  # noqa: E731
    return dict(p=o.flat_params.clone(), m=o.exp_avg.clone(), v=o.exp_avg_sq.clone(), h=o.flat_half.clone(), state=o.state.clone(),
                quads=c(step._quads), counter=model.step_counter.clone(), samples=int(step.samples.item()),
                rng=step._rng.clone(), local_step=model.local_step, grid=model.density_grid.clone(),
                bits=model.density_bitfield.clone())


def _folded(step, cap):
    """The bucket as the optimizer saw it: the twin added into the table rows in fp32 (what the fold kernels do)."""
    g = _np(cap["g"]).copy()
    if cap["odd"] is not None:
        o = step.opt.offsets[step.opt._index(step.model.encoder.embeddings)]
        odd = _np(cap["odd"])
        g[o:o + odd.size] = (g[o:o + odd.size] + odd).astype(np.float32)
    return g


def _load_flat(named, step, flat):
    """Copy the optimizer-layout parameter vector `flat` into (name, parameter) pairs named like the trained model's."""
    mine = dict(step.model.named_parameters())
    with torch.no_grad():
        for n, p in named:
            q = mine[n]
            o = step.opt.offsets[step.opt._index(q)]
            p.copy_(flat[o:o + q.numel()].view_as(q))


def _ulp32(x):
    return np.spacing(np.abs(x).astype(np.float32)).astype(np.float64)


def _lr_segments(step):
    """End and lr of each parameter group, from the model's own groups and the parameter offsets - not from the launch
    arguments under test.  (A group's end before the alignment padding: padding stays zero under any lr.)"""
    ends, lrs = [], []
    for grp in step.model.get_params(LR):
        ps = [p for p in grp["params"] if p.requires_grad]
        if ps:
            ends.append(max(step.opt.offsets[step.opt._index(p)] + p.numel() for p in ps))
            lrs.append(grp["lr"])
    ends[-1] = step.opt.numel
    return ends, lrs


def _check_update(k, step, pre, post, g, fails):
    """(b): one optimizer update against oracle.adam_scaler_step from the pre-update state and the consumed gradient."""
    from oracle import oracle as O
    o = step.opt
    seg_end, seg_lr = _lr_segments(step)
    ref_p, _, ref_m, ref_v, ref_st = O.adam_scaler_step(
        _np(pre["p"]), g, _np(pre["m"]), _np(pre["v"]), _np(pre["state"]), seg_end, seg_lr, o.betas, o.eps,
        o.grad_div, o.lr_decay_ln, o.lr_decay_steps, o.growth_factor, o.backoff_factor, o.growth_interval)
    row = dict(step=k, scale=float(pre["state"][0]))
    lims = {}
    for name, ref, before in (("m", ref_m, pre["m"]), ("v", ref_v, pre["v"]), ("p", ref_p, pre["p"])):
        got = _np(post[name]).astype(np.float64)
        d = np.abs(got - ref)
        # fp32 rounding: 2 ulp of the value + 1e-5 of this update's change of it
        lim = 2 * _ulp32(ref) + 1e-5 * np.abs(ref - _np(before))
        if name == "p":
            # ... + what m's own rounding allowance moves p by (update / m * lim_m): where the new m is a near-cancellation
            # of the old one and the gradient (a sign flip), m's few-ulp error is a large fraction of the small update
            dp = np.abs(ref - _np(before))
            with np.errstate(divide="ignore", invalid="ignore"):
                lim = lim + np.where(ref_m != 0, dp / np.abs(ref_m), 0.0) * lims["m"]
        lims[name] = lim
        row[name + "_max_over_limit"] = float((d / np.maximum(lim, 1e-45)).max())
        row[name + "_max_abs"] = float(d.max())
        if not (d <= lim).all():
            i = int(np.argmax(d - lim))
            fails.append("step %d: %s[%d] = %r, want %r (limit %.3g)" % (k, name, i, got[i], ref[i], lim[i]))
    want_state = ref_st[:5].astype(np.float32)
    got_state = _np(post["state"])[:5]
    row["state"] = got_state.tolist()
    if not np.array_equal(got_state, want_state):
        fails.append("step %d: state %s, want %s" % (k, got_state.tolist(), want_state.tolist()))
    if not torch.equal(post["h"], post["p"].half()):
        fails.append("step %d: fp16 shadow is not half(params)" % k)
    if k == SKIP_STEP:
        sp, sq = _np(pre["state"]), got_state
        ok = (all(torch.equal(post[n], pre[n]) for n in ("p", "m", "v", "h")) and sq[0] == sp[0] / 2 and sq[1] == 0
              and sq[4] == sp[4] + 1 and sq[2] == sp[2])
        row["skipped"] = bool(ok)
        if not ok:
            fails.append("step %d (inf in G): not a clean skipped step: state %s -> %s" % (k, sp[:5].tolist(), sq.tolist()))
    return row


def _check_grads(k, step, model, twin, ref, pre, g, ro, rd, G, noises, bits, fails):
    """(a): the consumed bucket against the fp64 step oracle and the reference pipeline at this step's state."""
    from unittest import mock
    scale = float(pre["state"][0])
    _load_flat(twin.named_parameters(), step, pre["p"])
    _load_flat(_ref_named(ref), step, pre["p"])
    ref.density_bitfield.copy_(bits)
    ref.local_step = 0
    # configurations that reach a step with identical inputs (all of them at step 0) share its references
    h = hashlib.sha1()
    for t in (pre["p"], ro, rd, G, noises, bits):
        h.update(t.contiguous().cpu().numpy().tobytes())
    key = (h.hexdigest(), scale)
    t0 = time.time()
    if key not in _REF_CACHE:
        truth = _step_truth(twin, ro.view(1, -1, 3), rd.view(1, -1, 3), G, noises, bits.cpu().numpy(), scale=scale)
        t1 = time.time()
        with mock.patch.object(torch, "rand", lambda *a, **kw: noises.clone()):   # the reference marcher draws torch.rand(N)
            _, _, rgrads = _ref_step(ref, ro.view(1, -1, 3), rd.view(1, -1, 3), G, 0, scale=scale)
        _REF_CACHE[key] = (truth, {n: _np(t).astype(np.float64) for n, t in rgrads.items()})
    else:
        t1 = t0
    truth, rgrads = _REF_CACHE[key]
    t2 = time.time()
    rows = []
    for n, p in model.named_parameters():
        o = step.opt.offsets[step.opt._index(p)]
        ours = g[o:o + p.numel()].astype(np.float64).reshape(tuple(p.shape))
        r = _closer_or_equal(n, ours, rgrads[n], truth["grads"][n])
        r["ceiling"] = GRAD_CEILING[n]
        r["ok"] = bool(r["ok"] and r["ours_vs_fp64"] <= GRAD_CEILING[n])
        rows.append(r)
        if not r["ok"]:
            fails.append("step %d: gradient %s: %s" % (k, n, r))
    return dict(step=k, scale=scale, samples=truth["total"], grads=rows, oracle_s=t1 - t0, reference_s=t2 - t1), truth["total"]


def _ref_named(r):
    """RefGridNeRF's parameters under NeRFNetwork's names."""
    yield "encoder.embeddings", r.embeddings
    for pre, net in (("sigma_net", r.sigma_net), ("bg_net", r.bg_net)):
        for i, l in enumerate(net):
            yield "%s.net.%d.weight" % (pre, i), l.weight
            yield "%s.net.%d.bias" % (pre, i), l.bias


def _quad_table(step, h):
    """A fresh ngp_grid_quad_table of the fp16 shadow `h` (flat, optimizer layout)."""
    from ngp_b200 import _cabi
    enc = step.model.encoder
    o = step.opt.offsets[step.opt._index(enc.embeddings)]
    table_h = h[o:o + enc.embeddings.numel()].view_as(enc.embeddings)
    out = torch.zeros_like(step._quads)
    L, S = enc.offsets.shape[0] - 1, float(np.log2(enc.per_level_scale))
    P = _cabi.ptr
    _cabi.call("ngp_grid_quad_table", torch.device(DEV), P(table_h), P(enc.offsets), L, table_h.shape[0], S,
               int(enc.base_resolution), int(enc.gridtype_id), int(bool(enc.align_corners)), P(out))
    torch.cuda.synchronize()
    return out


def _check_refresh(k, model, twin, step, old_grid, occ, params, fails):
    """(d): the occupancy refresh of step k against the C oracle, and its densities against the fp64 field evaluated at
    `params` (the parameters of the completed previous update)."""
    from oracle import oracle as O
    H = model.grid_size
    row = dict(step=k)
    pts = O.occupancy_cell_points(H, 1.0, _np(occ["u"]))
    row["cell_points_exact"] = bool(np.array_equal(pts, _np(occ["xyzs"])))
    sigma = _np(occ["sigma"])
    new_grid, mean, bits = O.update_density_grid(_np(old_grid).reshape(-1), sigma, 0.95, float(model.density_thresh))
    dev_mean = float(occ["mean"][0])
    row.update(grid_exact=bool(np.array_equal(new_grid, _np(occ["grid"]).reshape(-1))), mean=(dev_mean, mean),
               bits_exact=bool(np.array_equal(O.packbits(new_grid, min(dev_mean, float(model.density_thresh))),
                                               occ["bits"].cpu().numpy())))
    mean_ok = abs(dev_mean - mean) <= 1e-5 * abs(mean)
    # the densities themselves, on a seeded subsample of the cells
    _load_flat(twin.named_parameters(), step, params)
    idx = np.random.default_rng(100 + k).choice(H ** 3, 1 << 16, replace=False)
    S, sc, offs = _enc_consts(twin)
    W, b = _field_params(twin)
    want = O.field_forward(pts[idx], _np(twin.encoder.embeddings), offs, S, 16, W, b, scale_override=sc, round_hidden=True)["sigma"]
    rel = np.abs(sigma[idx].astype(np.float64) - want) / want
    row.update(sigma_max_rel=float(rel.max()), sigma_rel_l2=float(np.linalg.norm(sigma[idx] - want) / np.linalg.norm(want)))
    if not (row["cell_points_exact"] and row["grid_exact"] and row["bits_exact"] and mean_ok and row["sigma_max_rel"] <= SIGMA_REL):
        fails.append("step %d: occupancy refresh: %s" % (k, row))
    return row


@pytest.mark.parametrize("config", list(CONFIGS))
def test_graphed_train_step_trajectory_vs_fp64_and_float64_adam(ref_ext, config, monkeypatch):
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    from oracle.ref_pipeline import RefGridNeRF
    cfg = CONFIGS[config]
    for k, v in cfg["env"].items():
        monkeypatch.setenv(k, v)
    t_start = time.time()
    model = _bench_like_model()
    step = TrainStep(model, HW, HW, lr=LR, manual=True, **cfg["kw"])
    assert step.manual and step.update_interval == 16
    step.opt.growth_interval = GROWTH_INTERVAL          # a launch argument: frozen into the graph at capture
    pipelined, device_rays = step.pipelined, step.device_rays is not None
    assert pipelined == ("pipelined" in config)
    rec = _Recorder(step)
    twin = _bench_like_model()
    ref = RefGridNeRF(ref_ext).to(DEV).train()
    assert torch.equal(ref.offsets, model.encoder.offsets)

    poses, intr = provider.make_training_poses(N_STEPS, HW, HW, seed=5)
    poses, intr = poses.to(DEV), intr.to(DEV)
    G = torch.randn(N_STEPS, 1, 3, HW, HW, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)) * 1e-2
    G[SKIP_STEP, 0, 1, 17, 40] = float("inf")           # one overflow: the replayed graph takes one skipped step

    snaps = [_snapshot(step, model)]                    # snaps[k + 1]: after call k
    caps = {}                                           # update k -> what it consumed / left behind
    step_in = []                                        # per call: rays, noises, the refresh's scratch
    for k in range(N_STEPS):
        if device_rays:
            step(poses[k:k + 1], intr[k:k + 1], G[k])
        else:
            ro, rd = provider.get_rays_device(poses[k:k + 1], intr[k:k + 1], HW, HW)
            step(ro.contiguous(), rd.contiguous(), G[k])
        snaps.append(_snapshot(step, model))
        m = step._mws
        d = dict(ro=(m["ro"] if device_rays else m["ro_flat"]).clone(), rd=(m["rd"] if device_rays else m["rd_flat"]).clone(),
                 noises=m["noises"].clone())
        if k % 16 == 0:
            occ = model._occ_ws
            d["occ"] = dict(u=occ["u"].clone(), xyzs=occ["xyzs"].clone(), sigma=occ["sigma"].clone(), mean=occ["mean"].clone(),
                            grid=model.density_grid.clone(), bits=model.density_bitfield.clone())
        step_in.append(d)
        if not pipelined:
            caps[k] = rec.take("step")
        else:
            if k % 16 == 0 and k > 0:
                caps[k - 1] = rec.take("flush")         # the refresh's flush applied update k - 1
            elif k > 0:
                caps[k - 1] = rec.take("step")
    step.flush()
    torch.cuda.synchronize()
    if pipelined:
        caps[N_STEPS - 1] = rec.take("flush")
        snaps.append(_snapshot(step, model))
    t_run = time.time() - t_start

    def pre_post(k):   # the state right before / after update k
        return (snaps[k + 1], snaps[k + 2]) if pipelined else (snaps[k], snaps[k + 1])

    fails, rep = [], dict(updates=[], grads=[], carried=[], refresh=[])
    assert step.opt.steps_taken == N_STEPS - 1 and int(step.opt.state[4].item()) == 1 and step.n_updates == 2
    scales = [float(pre_post(k)[0]["state"][0]) for k in range(N_STEPS)]
    rep["scales"] = scales
    assert max(scales) > scales[0] and scales[SKIP_STEP + 1] == scales[SKIP_STEP] / 2 and scales[-1] > scales[SKIP_STEP + 1], scales
    for k in range(N_STEPS):
        pre, post = pre_post(k)
        cap = caps[k]
        g = _folded(step, cap)
        # (b) the update
        rep["updates"].append(_check_update(k, step, pre, post, g, fails))
        # (c) carried state
        before, after = snaps[k], snaps[k + 1]             # around call k
        c = dict(step=k, samples=after["samples"] - before["samples"])
        zero = cap["g_after"].count_nonzero().item() == 0 and (cap["odd_after"] is None or cap["odd_after"].count_nonzero().item() == 0)
        c["bucket_and_twin_zeroed"] = bool(zero)
        if not zero:
            fails.append("step %d: the update left the gradient bucket or the twin non-zero" % k)
        if step._quads is not None:
            # the table this step's forward read: built from the shadow of the update before it (pre-state of update k)
            c["quads_fresh"] = bool(torch.equal(after["quads"], _quad_table(step, pre["h"])))
            if not c["quads_fresh"]:
                fails.append("step %d: the quad table is not the one of the shadow the forward read" % k)
        row = before["local_step"] % 16 if k % 16 else 0
        got_row = after["counter"][row].tolist()
        c["counter_row"] = (row, got_row)
        if got_row != [c["samples"], HW * HW] or after["local_step"] != row + 1:
            fails.append("step %d: step_counter[%d] = %s, want [%d, %d]" % (k, row, got_row, c["samples"], HW * HW))
        r0, r1 = before["rng"].tolist(), after["rng"].tolist()
        seed, ctr = r0[0], r0[1]
        if r1 != [seed, ctr + 1, r0[2]] or not np.array_equal(_np(step_in[k]["noises"]), _ray_noise_np(seed, ctr, HW * HW)):
            fails.append("step %d: device noise counter %s -> %s or its draw is off" % (k, r0, r1))
        rep["carried"].append(c)
        # (a) gradients
        if k in cfg["grad_steps"]:
            d = step_in[k]
            row_a, total = _check_grads(k, step, model, twin, ref, pre, g, d["ro"], d["rd"], G[k], d["noises"], after["bits"], fails)
            if total != c["samples"]:
                fails.append("step %d: %d samples marched, the oracle marcher finds %d" % (k, c["samples"], total))
            rep["grads"].append(row_a)
        # (d) refresh
        if k % 16 == 0:
            old_grid = snaps[k]["grid"]
            params = snaps[0]["p"] if k == 0 else pre_post(k - 1)[1]["p"]
            rep["refresh"].append(_check_refresh(k, model, twin, step, old_grid, step_in[k]["occ"], params, fails))
    rep.update(run_s=t_run, total_s=time.time() - t_start, fails=fails[:20])
    worst = {}
    for r in rep["grads"]:
        for gr in r["grads"]:
            worst[gr["name"]] = max(worst.get(gr["name"], 0.0), gr["ours_vs_fp64"])
    rep["worst_grad_vs_fp64"] = worst
    _report(config, rep, REPORT, "trajectory_parity.json")
    assert not fails, fails[:10]
