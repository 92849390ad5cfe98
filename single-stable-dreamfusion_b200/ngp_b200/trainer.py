"""The `-O` train step around ``NeRFRenderer.render`` - eager, or captured once into a CUDA graph.

``TrainStep`` restates the reference Trainer's per-step call pattern (nerf/utils.py:337-403 train_step,
:696-713 train_one_epoch) for a synthetic guidance gradient: occupancy refresh every 16 steps, render under
fp16 autocast, the guidance's manual ``pred_rgb.backward(gradient=G, retain_graph=True)`` (nerf/sd.py:115),
the entropy regulariser through ``GradScaler``, Adam (betas 0.9/0.99, eps 1e-15, 10x lr for the encoder:
main.py:128, network_grid.py:170-181).  Data parallel: views are sharded across ranks and ONE all-reduce of
the flat gradient bucket precedes the optimizer step (parallel.py).

With ``graph=True`` everything between "inputs are in the static buffers" and "parameters are updated" is
one ``cudaGraphLaunch``: the training render has static shapes and no host sync (render_train.py), the
optimizer is torch's fused capturable Adam driven by the scaler's device-side found_inf, and NCCL
all-reduce is graph-capturable.  The occupancy refresh stays outside the graph (it runs every 16th step).
"""
import os
import numpy as np
import torch
import torch.distributed as dist

from . import _cabi, _nvtx
from .optim import FusedAdamScaler
from .parallel import FlatGradBucket, PeerMemory
from .step_ops import entropy_loss as fused_entropy_loss


def entropy_loss(weights_sum, lam=1e-4):
    """lambda_entropy * binary entropy of the per-ray opacity (nerf/utils.py:389-394), as the reference's chain of
    torch ops (the one-launch version is step_ops.entropy_loss)."""
    alphas = weights_sum.clamp(1e-5, 1 - 1e-5)
    return lam * (-alphas * torch.log2(alphas) - (1 - alphas) * torch.log2(1 - alphas)).mean()


class TrainStep:
    def __init__(self, model, H, W, lr=1e-3, max_steps=1024, lambda_entropy=1e-4, update_interval=16, graph=False,
                 world_size=1, fused_optimizer=True, lr_decay=None, manual=None, peer_allreduce=None, pipelined=None,
                 n_chunks=None, device_rays=None, shading="albedo", ambient_ratio=None, lambda_orient=1e-2, lambda_smooth=0.0,
                 overlap=False):
        """device_rays: None, or (H_full, row0, row_stride): the step's inputs are then camera POSES [B,4,4] and intrinsics
        [B,4] (fx, fy, cx, cy) instead of rays - the prologue kernel generates the rays of image rows row0, row0 + stride, ...
        (this TrainStep's H of them) of every view on the device (nerf/utils.py:43-106 get_rays; hand-scheduled step only).
        manual: run the step as the hand-scheduled kernel sequence of _body_manual (no autograd, 13 launches) instead
        of the autograd graph of _body (~58 launches); None = whenever the model has the reference's field shape.
        shading: 'albedo' (default), or 'lambertian' / 'textureless' / 'normal' for every step of this TrainStep (the
        reference draws these after albedo_iters with ambient_ratio 0.1 and adds lambda_orient * loss_orient,
        nerf/utils.py:345-356,396-398).  Shaded steps run hand-scheduled too - stencil, field forward over 7 rows per sample,
        shade, per-ray loss, shade backward with the orientation term, field backward, scatter (_manual_compute) - when
        world_size == 1, overlap is off and lambda_smooth == 0; otherwise (and with manual=False) through the autograd
        step.  manual=True with one of those settings raises.
        peer_allreduce: world_size > 1 only - fuse the gradient all-reduce into the optimizer kernel over NVLink peer
        memory (csrc/adam.cu) instead of calling NCCL; None = if peer-addressable memory is available.
        pipelined (hand-scheduled step only): apply step k's optimizer update (and gradient all-reduce) at the START of
        step k+1, on the side stream, overlapped with that step's ray marching (which reads no parameters).  Same
        arithmetic in the same order; the parameters lag one update behind until flush() - called automatically before
        every occupancy refresh, and by the user before reading the parameters.  None = on for world_size > 1 with the fused
        peer all-reduce (measured at 8 GPUs: 0.385 vs 0.432 ms per step - the cross-GPU exchange and its wait for the slowest
        rank hide behind the marcher), off on one GPU (the update is 1.6 % of the step and the marcher is issue-bound)."""
        self.model, self.H, self.W = model, H, W
        # shading != 'albedo' (after albedo_iters the reference draws 'textureless' / 'lambertian' with ambient_ratio 0.1,
        # nerf/utils.py:345-356, and adds lambda_orient * loss_orient [+ lambda_smooth * loss_smooth], :396-402): the
        # hand-scheduled step over the 7-point stencil kernels of csrc/shading.cu; the settings it does not cover take the
        # autograd step (the same kernels under run_cuda)
        from .step_ops import SHADING_MODES
        self.shading = shading
        self.ambient_ratio = (1.0 if shading == "albedo" else 0.1) if ambient_ratio is None else float(ambient_ratio)
        self.lambda_orient, self.lambda_smooth = float(lambda_orient), float(lambda_smooth)
        self._shade_mode = None     # hand-scheduled shaded step: csrc/shading.cu mode (0 lambertian, 1 textureless, 2 normal)
        if shading != "albedo":
            unsupported = [name for name, bad in (("shading=%r" % (shading,), shading not in SHADING_MODES),
                                                  ("lambda_smooth > 0", self.lambda_smooth > 0),
                                                  ("world_size > 1", world_size > 1), ("overlap=True", bool(overlap))) if bad]
            if unsupported:
                if manual:
                    raise RuntimeError("the hand-scheduled shaded step does not support %s; use manual=False"
                                       % ", ".join(unsupported))
                manual = False
            elif manual is None or manual:
                self._shade_mode = SHADING_MODES[shading]
        # overlap (hand-scheduled, graphed step only): the ray-marching half of step k+1 (prologue + march: it reads rays and
        # the occupancy bitfield, no parameters) runs on its own stream WHILE the field / loss / backward / optimizer half of
        # step k runs - two CUDA graphs per step and two alternating workspace sets, ordered by ordinary stream events.
        # Arithmetic and update order are those of the sequential step; results arrive with a lag (see __call__).
        self.overlap = bool(overlap)
        self._pipelined_request = pipelined
        self.pipelined = bool(pipelined)
        self.device_rays = None if device_rays is None else tuple(int(v) for v in device_rays)
        self._pending = False
        self.n_chunks = n_chunks            # ray chunks run as parallel chains; None = 2 (measured: -6 % step time at 32768
        #                                     rays, -2.5 % at 4096; 3 chains are slower than 2)
        self._chain = []
        self._chain_march = []
        self.max_steps, self.lam, self.update_interval = max_steps, lambda_entropy, update_interval
        self.world = world_size
        # Data parallel = the SAME step as one GPU rendering all rays: the guidance term is a per-pixel SUM (nerf/sd.py:115
        # `latents.backward(gradient=grad)`, un-normalised), so rank gradients are reduced with SUM and never divided; the
        # entropy term is a MEAN over all rays of the job, so each rank's local mean is weighted 1 / world.
        self.lam_local = float(lambda_entropy) / float(world_size)
        self.fixed_noises = None  # tests: per-ray perturbation noise [N] used instead of a fresh torch.rand draw
        self.fixed_light = None   # tests: light direction [3] of a shaded hand-scheduled step instead of a fresh draw
        # table-gradient scatter into two buffers (even / odd row pairs both as 16-byte reds); NGP_SPLIT_SCATTER=0: one buffer
        self.split_scatter = os.environ.get("NGP_SPLIT_SCATTER", "1") not in ("", "0")
        self._g_table_odd = None
        # overlap mode: ONE graph per call (march(k) || compute(k-1), forked and joined inside the graph) instead of two
        # graphs on two streams tied by events; NGP_OVERLAP_FUSED=0 keeps the two-graph form
        self.overlap_fused = os.environ.get("NGP_OVERLAP_FUSED", "1") not in ("", "0")
        self.keep_grads = False   # tests: copy the gradient bucket to self.grad_snapshot right before the optimizer
        self.grad_snapshot = None  # (a device-to-device copy inside the step, so it also works in a graph replay)
        self.use_graph = graph
        self.single_backward = True  # one engine pass for both roots (see _body); False = the reference's two passes
        device = next(model.parameters()).device
        self.device = device
        self.fused_optimizer = fused_optimizer
        self.manual = bool(fused_optimizer and self._manual_supported()) if manual is None else bool(manual)
        if not self.manual:
            self._shade_mode = None
        if self.manual and not (fused_optimizer and self._manual_supported()):
            raise RuntimeError("the hand-scheduled step needs the fused optimizer and the reference's field / bg-net shapes")
        if self.device_rays is not None and not self.manual:
            raise RuntimeError("device-side ray generation is part of the hand-scheduled step (manual=True)")
        self.peer = None
        self.peer_error = None
        if fused_optimizer and self.manual and world_size > 1 and peer_allreduce is not False:
            try:
                self.peer = PeerMemory(device)
            except RuntimeError as e:
                self.peer_error = repr(e)
        if fused_optimizer:
            # one flat buffer each for params / grads / moments / fp16 shadow; unscale + Adam + scaler.update + shadow
            # refresh + zero_grad in two launches (optim.py); gradients are SUMMED over ranks
            try:
                self.opt = FusedAdamScaler(model.get_params(lr), betas=(0.9, 0.99), eps=1e-15, grad_div=1.0,
                                           lr_decay=lr_decay, peer_memory=self.peer)
            except RuntimeError as e:
                if self.peer is None or peer_allreduce:
                    raise
                self.peer, self.peer_error = None, repr(e)  # no peer-addressable memory here: NCCL all-reduce instead
                self.opt = FusedAdamScaler(model.get_params(lr), betas=(0.9, 0.99), eps=1e-15, grad_div=1.0,
                                           lr_decay=lr_decay)
            self.scaler = self.opt
            self.bucket = None
            self.flat_grads = self.opt.flat_grads
        else:
            self.opt = torch.optim.Adam(model.get_params(lr), betas=(0.9, 0.99), eps=1e-15, fused=True, capturable=graph)
            self.scaler = torch.amp.GradScaler("cuda")
            self.bucket = FlatGradBucket(list(model.parameters()), device)
            self.flat_grads = self.bucket.flat
        if self._pipelined_request is None:
            self.pipelined = bool(self.manual and fused_optimizer and world_size > 1 and self.opt.peer_ptrs is not None
                                  and not self.overlap)
        if world_size > 1 and dist.is_available() and dist.is_initialized() and not hasattr(model, "dp_shard"):
            model.dp_shard = (dist.get_rank(), world_size)  # occupancy refresh: 1/world of the cells per rank + all-gather
        self.global_step = 0
        self.n_updates = 0
        self.samples = torch.zeros(1, dtype=torch.int64, device=device)  # running count of marched samples
        self._local_step_dev = torch.zeros(1, dtype=torch.int32, device=device)  # device mirror of model.local_step
        # background-net branch of the step (default priority: it fills the gaps of the main chain, measured faster than
        # a high-priority branch that takes SM slots away from the field kernels)
        self._side = torch.cuda.Stream(device=device) if self.manual else None
        # the background net's FORWARD is tiny (one CTA per 128 rays) and the per-ray loss kernels wait for it: on a
        # default-priority stream it queued behind the field forward's 592 CTAs whenever both became runnable together
        # (pipelined optimizer: both wait for the update) and delayed the loss kernels by ~25 us - high priority
        self._side_fwd = torch.cuda.Stream(device=device, priority=-1) if self.manual else None
        # pipelined optimizer launch: its own HIGH-priority stream, so that its CTAs are placed ahead of the thousands of
        # ray-marching CTAs it runs beside (otherwise it only starts when the marcher's last wave does)
        self._side_opt = torch.cuda.Stream(device=device, priority=-1) if (self.manual and self.pipelined) else None
        # draw the randn(3) run_cuda spends on light_d (and drop it under albedo shading), to keep torch's RNG stream aligned;
        # shaded steps then take their light from it as run_cuda does.  Otherwise a shaded step draws its light on the
        # device (ngp_train_light: same generator as the march jitter below).
        self.mirror_rng = False
        # Per-ray march jitter of the hand-scheduled step: drawn by the prologue kernel from a counter-based generator
        # (csrc/raymarch.cu ray_noise; [seed, step counter, scratch]) instead of a torch.rand launch - in graph mode torch
        # also enqueues two seed / offset fill kernels before every replay of a graph that holds one of its generators.
        # The seed follows torch.manual_seed (+ the rank, so ranks jitter differently); mirror_rng / fixed_noises /
        # NGP_DEVICE_NOISE=0 keep torch.rand.
        # ray marching of the hand-scheduled step as ONE launch without scratch (ngp_march_rays_train_packed: rays land in
        # completion order, like the reference's); NGP_PACKED_MARCH=0: ray-ordered walk -> scan -> packed copy
        self.packed_march = os.environ.get("NGP_PACKED_MARCH", "1") not in ("", "0")
        # field forward through a quad table of the fp16 embeddings (csrc/field_mlp.cu encode_level_quads: one or two 16-byte
        # gathers per level instead of four to eight 4-byte ones), rebuilt every step beside the ray marching (13 us on a
        # side stream).  Measured: forward 0.488 -> 0.417 ms at 3.3 M samples; 1-2 % of the step at 4096 rays per GPU too
        # (2 and 8 GPUs, bench.py --dp-sweep).  NGP_QUAD_TABLE=0 turns it off.
        self.quad_table = os.environ.get("NGP_QUAD_TABLE", "1") not in ("", "0")
        self._quads = None
        self.device_noise = bool(self.manual) and os.environ.get("NGP_DEVICE_NOISE", "1") not in ("", "0")
        rank = dist.get_rank() if (world_size > 1 and dist.is_available() and dist.is_initialized()) else 0
        seed = (int(torch.initial_seed()) + 0x9E3779B97F4A7C15 * rank) & 0x7FFFFFFFFFFFFFFF
        self._rng = torch.tensor([seed, 0, 0], dtype=torch.int64, device=device)
        self._mws = None
        self._mws_sets = [None, None]      # overlap mode: the two alternating workspace sets
        self._ls_mirror = 0
        self._static_packed = None
        self._graph = None
        self._graph_exec = 0
        self._graph_launches = 0
        self._static = None
        self.loss = None

    # -- one step's device work, shape-static when the fused training render is active ---------------------------
    def _step_body(self, rays_o, rays_d, G):
        return self._body_manual(rays_o, rays_d, G) if self.manual else self._body(rays_o, rays_d, G)

    def _body(self, rays_o, rays_d, G):
        model = self.model
        B = rays_o.shape[0]
        if not self.fused_optimizer:
            self.bucket.zero()  # (the fused optimizer kernel leaves the gradient buffer zeroed)
        with torch.autocast("cuda", torch.float16):
            out = model.render(rays_o, rays_d, staged=False, perturb=True, bg_color=None, ambient_ratio=self.ambient_ratio,
                               shading=self.shading, force_all_rays=True, max_steps=self.max_steps, dt_gamma=0)
            pred_rgb = out["image"].reshape(B, self.H, self.W, 3).permute(0, 3, 1, 2).contiguous()
            ws = out["weights_sum"].reshape(B, 1, self.H, self.W)
            loss = fused_entropy_loss(ws, self.lam_local) if self.fused_optimizer else entropy_loss(ws, self.lam_local)
            if self.lambda_orient > 0 and "loss_orient" in out:       # nerf/utils.py:396-398
                loss = loss + (self.lambda_orient / self.world) * out["loss_orient"]
            if self.lambda_smooth > 0 and "loss_smooth" in out:       # :400-402
                loss = loss + (self.lambda_smooth / self.world) * out["loss_smooth"]
        # The reference runs TWO backward passes over the render graph per step: the guidance's manual
        # `pred_rgb.backward(gradient=G, retain_graph=True)` (nerf/sd.py:115) and `scaler.scale(loss).backward()`
        # (nerf/utils.py:708).  Back-propagation is linear in the upstream gradient, so both roots are handed to the
        # engine at once: it sums d(image), d(weights_sum) at the render node and walks the heavy part (composite,
        # MLP, grid scatter) once.  Same accumulated .grad up to fp32 summation order (tests/test_gpu_pipeline.py).
        if self.single_backward:
            torch.autograd.backward([pred_rgb, self.scaler.scale(loss)], [G, None])
        else:
            pred_rgb.backward(gradient=G, retain_graph=True)
            self.scaler.scale(loss).backward()
        if self.world > 1:
            dist.all_reduce(self.flat_grads, op=dist.ReduceOp.SUM)
        if self.fused_optimizer:
            self.opt.step(zero_grads=True)
        else:
            self.scaler.step(self.opt)
            self.scaler.update()
        return loss

    # -- the same step without autograd: a fixed sequence of our kernels ----------------------------------------------
    def _manual_supported(self):
        from . import field as _field
        m = self.model
        enc, net = getattr(m, "encoder", None), getattr(m, "sigma_net", None)
        if enc is None or net is None or not getattr(m, "fused", False) or not getattr(m, "cuda_ray", False):
            return False
        try:
            ok = (enc.num_levels == 16 and enc.level_dim == 2 and enc.input_dim == 3 and net.num_layers == 3
                  and net.dim_hidden == 64 and net.dim_in == 32 and net.dim_out == 4 and net.net[0].bias is not None
                  and enc.embeddings.dtype == torch.float32 and enc.embeddings.is_cuda)
            if m.bg_radius > 0:
                bg = m.bg_net
                ok = ok and (m.encoder_bg.input_dim == 3 and m.encoder_bg.degree == 6 and bg.num_layers == 2
                             and bg.dim_hidden == 64 and bg.dim_out == 3 and bg.net[0].bias is not None)
            return bool(ok)
        except AttributeError:
            return False

    def _manual_workspace(self, N, which=None):
        """Per-ray buffers of the whole step plus one sample workspace per ray chunk (render_train.TrainWorkspace).
        which: None = the step's single set; 0 / 1 = one of the two alternating sets of overlap mode."""
        from .render_train import TrainWorkspace
        dev = self.device
        m = self._mws if which is None else self._mws_sets[which]
        if m is not None and m["N"] == N:
            return m
        n_chunks = self.n_chunks if self.n_chunks else 2
        n_chunks = max(1, min(int(n_chunks), N // 128 if N >= 256 else 1))
        e = lambda *shape, dtype=torch.float32: torch.empty(*shape, device=dev, dtype=dtype)  # noqa: E731
        shaded = self._shade_mode is not None
        m = dict(N=N, nears=e(N), fars=e(N), noises=e(N), weights_sum=e(N), depth=e(N), image=e(N, 3),
                 bg=e(N, 3, dtype=torch.half), d_bg=e(N, 3), loss=torch.zeros((), device=dev),
                 counters=torch.zeros(n_chunks, 2, dtype=torch.int32, device=dev),
                 cur_row=torch.zeros(1, dtype=torch.int32, device=dev), chunks=[])
        if shaded:
            # the step's light (direction, then the three normal draws behind it; ngp_train_light) - one for all chains -
            # and, with several chains, one event per chain's march: the orientation mean runs over the samples of all
            m["light"] = torch.zeros(6, device=dev)
            m["march_done"] = [torch.cuda.Event() for _ in range(n_chunks)] if n_chunks > 1 else []
        base = 0
        sizes = [N // n_chunks + (1 if c < N % n_chunks else 0) for c in range(n_chunks)]
        fr = os.environ.get("NGP_CHUNK_FRACTIONS")    # e.g. "0.4,0.6": unequal chains (their kernel phases then interleave)
        if fr and len(fr.split(",")) == n_chunks and N >= 256 * n_chunks:
            f = [float(v) for v in fr.split(",")]
            sizes = [max(128, int(N * v / sum(f)) // 128 * 128) for v in f]
            sizes[-1] = N - sum(sizes[:-1])
        for c in range(n_chunks):
            n_c = sizes[c]
            ws = TrainWorkspace(n_c, self.max_steps, dev, counter=m["counters"][c], shaded=shaded)
            m["chunks"].append((base, n_c, ws))
            base += n_c
        self.model._train_ws = m["chunks"][0][2]  # (what run_cuda's own fused path would allocate; kept for introspection)
        if len(self._chain) < n_chunks - 1:
            # overlap mode: the compute phase is the critical path (high priority), the next step's marching fills its gaps
            pr = -1 if self.overlap else 0
            self._chain = [torch.cuda.Stream(device=dev, priority=pr) for _ in range(n_chunks - 1)]
            self._chain_march = [torch.cuda.Stream(device=dev) for _ in range(n_chunks - 1)]
        if which is None:
            self._mws = m
        else:
            self._mws_sets[which] = m
        return m

    def _body_manual(self, rays_o, rays_d, G):
        """One `-O` train step as a fixed schedule of our kernels (no autograd):

            prologue (near/far, counters, bookkeeping) . rand . { march x3 . field fwd . ray loss (composite fwd + blend +
            both loss gradients + composite bwd) . field bwd . grid scatter } . all-reduce + Adam + GradScaler

        Shaded steps (shading != 'albedo'): light (ngp_train_light) after the prologue, the marcher also writes per-sample
        directions, and each chain runs  stencil (7 rows per sample) . field fwd (7 M rows) . shade fwd (centre density +
        colour into the per-sample rows) . ray loss . shade bwd (+ orientation term) . field bwd (7 M) . grid scatter.

        with the background net on a side stream (forward beside the marching, backward beside the field backward).
        The braces run as TWO chains over the two halves of the rays on parallel streams: the marcher and the per-ray
        loss kernel are bound by the latency of the longest ray, not by throughput, and fill the gaps of the other
        chain's field kernels.
        Same arithmetic as _body (the autograd version of the reference's train_step, nerf/utils.py:337-403,708-713):
        every kernel is either the one autograd would call or a fusion of such kernels; gradients go straight into the
        flat bucket (tests/test_gpu_train_step.py compares the two).
        The step is two phases - _manual_march (reads rays + the occupancy bitfield, no parameters) and _manual_compute
        (everything else) - run back to back here, and as separate graphs on separate streams in overlap mode."""
        with _nvtx.range("ngp.step.march"):
            m = self._manual_march(rays_o, rays_d, G.shape[0], None, bg_early=True)
        with _nvtx.range("ngp.step.compute"):
            return self._manual_compute(m, G, bg_done=True)

    def _manual_consts(self):
        model, opt = self.model, self.opt
        enc = model.encoder
        l0, l1, l2 = model.sigma_net.net
        field_params = (l0.weight, l0.bias, l1.weight, l1.bias, l2.weight, l2.bias)
        c = dict(enc=enc, L=enc.offsets.shape[0] - 1, S=float(np.log2(enc.per_level_scale)),
                 hw_field=[opt.half_view(t) for t in field_params], g_field=[opt.grad_view(t) for t in field_params],
                 table_h=opt.half_view(enc.embeddings), g_table=opt.grad_view(enc.embeddings), has_bg=model.bg_radius > 0)
        # odd-frame twin of the table gradient (ngp_grid_scatter_samples_split): indexed like g_table, 8 bytes off a 16-byte
        # boundary; folded into g_table once per step, right before the optimizer / the gradient snapshot
        c["g_table_odd"] = None
        if self.split_scatter and c["g_table"].data_ptr() % 16 == 0 and c["g_table"].numel() % 2 == 0:
            if self._g_table_odd is None or self._g_table_odd.numel() != c["g_table"].numel():
                raw = torch.zeros(c["g_table"].numel() + 4, device=self.device, dtype=torch.float32)
                self._g_table_odd = raw[2:2 + c["g_table"].numel()]
                assert self._g_table_odd.data_ptr() % 16 == 8
            c["g_table_odd"] = self._g_table_odd
        c["quads"] = None
        if self.quad_table:
            rows = c["table_h"].shape[0]
            if self._quads is None or self._quads.shape[0] != rows:
                self._quads = torch.zeros(rows, 4, dtype=torch.int32, device=self.device)
            c["quads"] = self._quads
        if c["has_bg"]:
            b0, b1 = model.bg_net.net
            bg_params = (b0.weight, b0.bias, b1.weight, b1.bias)
            c["hw_bg"] = [opt.half_view(t) for t in bg_params]
            c["g_bg"] = [opt.grad_view(t) for t in bg_params]
        return c

    def _bg_forward(self, m, c, after):
        dev, P = self.device, _cabi.ptr
        self._side_fwd.wait_stream(after)  # (the bg net reads the updated parameters / the generated ray directions)
        if c["quads"] is not None:      # the step's quad table, from the parameters this step's forward will read
            enc = c["enc"]
            with torch.cuda.stream(self._side_fwd):
                _cabi.call("ngp_grid_quad_table", dev, P(c["table_h"]), P(enc.offsets), c["L"], c["table_h"].shape[0], c["S"],
                           int(enc.base_resolution), int(enc.gridtype_id), int(bool(enc.align_corners)), P(c["quads"]))
        if not c["has_bg"]:
            return
        with torch.cuda.stream(self._side_fwd):
            _cabi.call("ngp_bg_forward", dev, P(m["rd_flat"]), m["N"], *[P(t) for t in c["hw_bg"]], 6, 64, P(m["bg"]))

    def _manual_march(self, rays_o, rays_d, B, which, bg_early):
        """Phase 1: prologue (rays from poses or given; near / far; counters; step_counter row) + per-chain ray marching."""
        model, dev = self.model, self.device
        hw = self.H * self.W
        poses = intr = None
        if self.device_rays is not None:
            # (rays_o, rays_d) carry (poses [B,4,4], intrinsics [B,4]); the rays live in the step's workspace
            poses, intr = rays_o, rays_d
            N = B * hw
            if poses.shape != (B, 4, 4) or intr.shape != (B, 4):
                raise RuntimeError("poses [B, 4, 4] and intrinsics [B, 4] expected")
            if not (poses.is_contiguous() and intr.is_contiguous() and poses.dtype == intr.dtype == torch.float32):
                raise RuntimeError("contiguous fp32 poses and intrinsics expected")
            m = self._manual_workspace(N, which)
            if "ro" not in m:
                m["ro"], m["rd"] = torch.empty(N, 3, device=dev), torch.empty(N, 3, device=dev)
            ro, rd = m["ro"], m["rd"]
        else:
            ro = rays_o.reshape(-1, 3)
            rd = rays_d.reshape(-1, 3)
            N = ro.shape[0]
            if N != B * hw:
                raise RuntimeError("rays [B, H*W, 3] expected")
            if not (ro.is_contiguous() and rd.is_contiguous() and ro.dtype == rd.dtype == torch.float32):
                raise RuntimeError("contiguous fp32 rays expected")
            m = self._manual_workspace(N, which)
        m["ro_flat"], m["rd_flat"] = ro, rd
        c = self._manual_consts()
        P = _cabi.ptr
        main = torch.cuda.current_stream(dev)
        if self.pipelined:
            self._side_opt.wait_stream(main)
            with torch.cuda.stream(self._side_opt):
                self._apply_update(deferred=True)  # the PREVIOUS step's update, beside this step's ray marching
        dev_noise = self.device_noise and not self.mirror_rng and self.fixed_noises is None
        noise_args = (P(m["noises"]), P(self._rng)) if dev_noise else (None, None)
        if poses is None:
            if (c["has_bg"] or c["quads"] is not None) and bg_early:
                self._bg_forward(m, c, self._side_opt if self.pipelined else main)
            _cabi.call("ngp_train_prologue", dev, P(ro), P(rd), P(model.aabb_train), N, 0.2, P(m["nears"]), P(m["fars"]),
                       P(m["counters"]), m["counters"].numel(), P(m["loss"]), P(model.step_counter), P(self._local_step_dev),
                       P(m["cur_row"]), *noise_args)
        else:
            h_full, row0, row_stride = self.device_rays
            _cabi.call("ngp_train_prologue_rays", dev, P(poses), P(intr), 1, B, h_full, self.W, row0, row_stride, self.H, P(ro),
                       P(rd), P(model.aabb_train), 0.2, P(m["nears"]), P(m["fars"]), P(m["counters"]), m["counters"].numel(),
                       P(m["loss"]), P(model.step_counter), P(self._local_step_dev), P(m["cur_row"]), *noise_args)
            if (c["has_bg"] or c["quads"] is not None) and bg_early:
                if self.pipelined:
                    self._side_fwd.wait_stream(self._side_opt)
                self._bg_forward(m, c, main)    # (reads the generated ray directions)
        shaded = self._shade_mode is not None
        if self.mirror_rng:
            z = torch.randn(3, device=dev)  # nerf/renderer.py:464 (light direction; unused by albedo shading)
            if shaded and self.fixed_light is None:
                from .renderer import safe_normalize
                m["light"][:3].copy_(safe_normalize(ro[0] + z))      # run_cuda's own expression
                m["light"][3:].copy_(z)
        if shaded:
            if self.fixed_light is not None:
                m["light"][:3].copy_(self.fixed_light)
            elif not self.mirror_rng:
                # after the prologue: rays_o[0] may be a generated ray; advance the counter unless the prologue did
                _cabi.call("ngp_train_light", dev, P(ro), P(self._rng), 0 if dev_noise else 1, P(m["light"]))
        if self.fixed_noises is not None:
            m["noises"].copy_(self.fixed_noises)
        elif not dev_noise:
            m["noises"].uniform_()  # the torch.rand(N) of the reference's wrapper (raymarching.py:213-216)

        chunks = m["chunks"]
        chain = self._chain if which is None else self._chain_march
        streams = [main] + chain[:len(chunks) - 1]
        for st in streams[1:]:
            st.wait_stream(main)
        for k, (st, (base, n_c, ws)) in enumerate(zip(streams, chunks)):
            with torch.cuda.stream(st):
                sl = slice(base, base + n_c)
                dirs = P(ws.dirs) if ws.dirs is not None else None     # (shaded steps: the orientation term reads them)
                if self.packed_march and self.max_steps <= 2048:
                    # one launch, no scratch: rows claimed with the reference's atomicAdd, rays land in completion order
                    _cabi.call("ngp_march_rays_train_packed", dev, P(ro[sl]), P(rd[sl]), P(model.density_bitfield),
                               float(model.bound), 0.0, int(self.max_steps), n_c, int(model.cascade), int(model.grid_size),
                               ws.cap, P(m["nears"][sl]), P(m["fars"][sl]), P(ws.xyzs), dirs, P(ws.deltas), P(ws.rays),
                               P(ws.counter), P(m["noises"][sl]))
                else:
                    _cabi.call("ngp_march_rays_train", dev, P(ro[sl]), P(rd[sl]), P(model.density_bitfield), float(model.bound),
                               0.0, int(self.max_steps), n_c, int(model.cascade), int(model.grid_size), ws.cap,
                               P(m["nears"][sl]), P(m["fars"][sl]), P(ws.xyzs), dirs, P(ws.deltas), P(ws.rays), P(ws.counter),
                               P(m["noises"][sl]), P(ws.march_ws), ws.march_ws.numel())
                if m.get("march_done"):
                    m["march_done"][k].record(st)
        if which is not None:       # a phase of its own: join the chains (in the fused step they run on into phase 2)
            for st in streams[1:]:
                main.wait_stream(st)
        return m

    def _manual_compute(self, m, G, bg_done):
        """Phase 2: background net, per chain field forward -> per-ray loss -> field backward -> grid scatter, optimizer."""
        model, opt, dev = self.model, self.opt, self.device
        N, hw = m["N"], self.H * self.W
        B = N // hw
        if G.shape != (B, 3, self.H, self.W) or not G.is_contiguous() or G.dtype != torch.float32:
            raise RuntimeError("contiguous fp32 G [B, 3, H, W] expected")
        c = self._manual_consts()
        enc, L, S, has_bg = c["enc"], c["L"], c["S"], c["has_bg"]
        hw_field, g_field, table_h, g_table = c["hw_field"], c["g_field"], c["table_h"], c["g_table"]
        g_odd = c["g_table_odd"]
        rd = m["rd_flat"]
        P = _cabi.ptr
        main = torch.cuda.current_stream(dev)
        if (has_bg or c["quads"] is not None) and not bg_done:
            self._bg_forward(m, c, main)
        chunks = m["chunks"]
        streams = [main] + self._chain[:len(chunks) - 1]
        if not bg_done:             # a phase of its own: fork the chains here (in the fused step phase 1 already did)
            for st in streams[1:]:
                st.wait_stream(main)

        shade = self._shade_mode
        ratio = float(self.ambient_ratio)

        def forward_and_loss(base, n_c, ws):
            sl = slice(base, base + n_c)
            # shaded: the field runs on the 7 stencil rows of every sample (count 7 M written on the device)
            rows = ws if shade is None else ws.stencil
            if shade is not None:
                _cabi.call("ngp_stencil_points", dev, P(ws.xyzs), ws.cap, P(ws.counter), 1e-2, float(model.bound), 1, P(rows.xyzs),
                           P(rows.counter))
            if self.pipelined:
                torch.cuda.current_stream(dev).wait_stream(self._side_opt)  # the field reads the updated parameters
            if c["quads"] is not None:
                torch.cuda.current_stream(dev).wait_stream(self._side_fwd)   # the step's quad table
                _cabi.call("ngp_field_forward_quads", dev, P(rows.xyzs), rows.cap, P(rows.counter), P(table_h), P(c["quads"]),
                           P(enc.offsets), L, 2, S, int(enc.base_resolution), int(enc.gridtype_id), int(bool(enc.align_corners)),
                           float(model.bound), *[P(t) for t in hw_field], 64, 4, P(rows.sigma), P(rows.rgb), P(rows.enc),
                           P(rows.h1), P(rows.h2))
            else:
                _cabi.call("ngp_field_forward", dev, P(rows.xyzs), rows.cap, P(rows.counter), P(table_h), P(enc.offsets), L, 2, S,
                           int(enc.base_resolution), int(enc.gridtype_id), int(bool(enc.align_corners)), float(model.bound),
                           *[P(t) for t in hw_field], 64, 4, P(rows.sigma), P(rows.rgb), P(rows.enc), P(rows.h1), P(rows.h2))
            if shade is not None:   # centre density + shaded colour into the ordinary per-sample rows
                _cabi.call("ngp_shade_forward_step", dev, P(rows.sigma), P(rows.rgb), ws.cap, P(ws.counter), P(m["light"]), ratio,
                           shade, P(ws.sigma), P(ws.rgb))
            if has_bg:
                torch.cuda.current_stream(dev).wait_stream(self._side_fwd)
            _cabi.call("ngp_train_ray_loss", dev, P(ws.sigma), P(ws.rgb), P(ws.deltas), P(ws.rays), ws.cap, n_c, 1e-4,
                       P(m["bg"][sl]) if has_bg else None, 1.0, P(G), hw, base, N, float(self.lam_local), opt.state.data_ptr(),
                       P(m["weights_sum"][sl]), P(m["depth"][sl]), P(m["image"][sl]), P(m["d_bg"][sl]) if has_bg else None,
                       P(ws.d_sigma), P(ws.d_rgb), P(m["loss"]), P(ws.counter), P(self.samples), P(model.step_counter),
                       P(m["cur_row"]))

        def backward(ws):
            rows = ws if shade is None else ws.stencil
            if shade is not None:
                for ev in m["march_done"]:      # the orientation mean needs every chain's sample count
                    torch.cuda.current_stream(dev).wait_event(ev)
                _cabi.call("ngp_shade_backward_step", dev, P(rows.sigma), P(rows.rgb), ws.cap, P(ws.counter), P(m["counters"]),
                           len(chunks), P(ws.dirs), P(m["light"]), ratio, shade, P(ws.d_sigma), P(ws.d_rgb),
                           float(self.lambda_orient) / self.world, opt.state.data_ptr(), P(rows.d_sigma), P(rows.d_rgb),
                           P(m["loss"]))
            _cabi.call("ngp_field_backward", dev, rows.cap, P(rows.counter), P(hw_field[0]), P(hw_field[2]), P(hw_field[4]), 64, 4,
                       P(rows.d_sigma), P(rows.d_rgb), P(rows.sigma), P(rows.rgb), P(rows.enc), P(rows.h1), P(rows.h2),
                       P(rows.d_enc), *[P(t) for t in g_field])
            if g_odd is None:
                _cabi.call("ngp_grid_scatter_samples", dev, P(rows.d_enc), P(rows.xyzs), float(model.bound), P(rows.counter),
                           rows.cap, P(enc.offsets), L, 2, S, int(enc.base_resolution), int(enc.gridtype_id),
                           int(bool(enc.align_corners)), P(g_table))
            else:
                _cabi.call("ngp_grid_scatter_samples_split", dev, P(rows.d_enc), P(rows.xyzs), float(model.bound), P(rows.counter),
                           rows.cap, P(enc.offsets), L, 2, S, int(enc.base_resolution), int(enc.gridtype_id),
                           int(bool(enc.align_corners)), P(g_table), P(g_odd))

        for st, (base, n_c, ws) in zip(streams, chunks):
            with torch.cuda.stream(st):
                forward_and_loss(base, n_c, ws)
        if has_bg:  # d_bg of every chunk is complete: the background net's backward, beside the field's
            for st in streams:
                self._side.wait_stream(st)
            with torch.cuda.stream(self._side):
                _cabi.call("ngp_bg_backward", dev, P(rd), P(m["d_bg"]), N, *[P(t) for t in c["hw_bg"]], 6, 64,
                           *[P(t) for t in c["g_bg"]])
        for st, (base, n_c, ws) in zip(streams, chunks):
            with torch.cuda.stream(st):
                backward(ws)
        for st in streams[1:]:
            main.wait_stream(st)
        if has_bg:
            main.wait_stream(self._side)
        if g_odd is not None and self.keep_grads:
            # (otherwise folded by _apply_update, inside the finite check or right before the NCCL all-reduce)
            _cabi.call("ngp_grid_fold_odd", dev, P(g_table), P(g_odd), g_table.numel())
        if self.keep_grads:
            if self.grad_snapshot is None:
                self.grad_snapshot = torch.empty_like(opt.flat_grads)
            self.grad_snapshot.copy_(opt.flat_grads)
        if not self.pipelined:
            self._apply_update(deferred=False)
        self._pending = True
        return m["loss"]

    def _apply_update(self, deferred):
        with _nvtx.range("ngp.step.optimizer"):
            fold = None
            if self._g_table_odd is not None and not self.keep_grads:
                fold = (self.opt.grad_view(self.model.encoder.embeddings), self._g_table_odd)
            if self.world > 1 and self.opt.peer_ptrs is None:
                # NCCL all-reduce of the bucket: the twin holds this rank's share only, so it is folded in before the reduce
                if fold is not None:
                    _cabi.call("ngp_grid_fold_odd", self.device, _cabi.ptr(fold[0]), _cabi.ptr(fold[1]), fold[0].numel())
                    fold = None
                dist.all_reduce(self.opt.flat_grads, op=dist.ReduceOp.SUM)
            self.opt.step(deferred=deferred, fold=fold)

    def fold_table_grads(self):
        """Add the odd-frame twin of the table gradient (split scatter) into the bucket now (tests that look at the bucket
        before the optimizer; the step itself folds inside the optimizer's finite check)."""
        if self._g_table_odd is not None:
            g_table = self.opt.grad_view(self.model.encoder.embeddings)
            _cabi.call("ngp_grid_fold_odd", self.device, _cabi.ptr(g_table), _cabi.ptr(self._g_table_odd), g_table.numel())

    # -- checkpoints in the reference Trainer's layout (nerf/utils.py:847-968) -------------------------------------------
    def save_checkpoint(self, path, epoch=0, full=True):
        """Collective under the fused data-parallel optimizer (its moments are sharded); write from one rank."""
        from . import checkpoint as ck
        self.flush()
        state = ck.checkpoint_dict(self.model, epoch=epoch, global_step=self.global_step, optimizer=self.opt,
                                   scaler=self.scaler, full=full)
        if not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0:
            torch.save(state, path)

    def load_checkpoint(self, path, model_only=False):
        """Reference-written and own checkpoints alike; optimizer state is restored only if it has this trainer's layout
        (a reference Adam state is reported in the returned `warnings`, as the reference itself does)."""
        from . import checkpoint as ck
        self.flush()
        info = ck.load_checkpoint(path, self.model, optimizer=self.opt if self.fused_optimizer else None,
                                  model_only=model_only, map_location=self.device)
        if not model_only:
            self.global_step = int(info["global_step"])
        if self.fused_optimizer:
            self.opt.sync_shadow_if_changed()
        return info

    def read_loss_async(self, lag=2):
        """The reference loop reads `loss.item()` after every step (nerf/utils.py:712), a device sync per step.  This is the
        same read without the stall: every call copies the latest step's loss (device scalar) into a slot of a small pinned
        ring and returns, as a Python float, the loss of `lag` calls ago - whose copy has certainly landed (its event is
        awaited, normally already complete).  None for the first `lag` calls; overlap mode already returns pinned, lagged
        losses and is passed through."""
        if self.loss is None:
            return None
        if not self.loss.is_cuda:
            return float(self.loss)
        ring = getattr(self, "_loss_ring", None)
        if ring is None or ring["lag"] != lag:
            n = lag + 2
            ring = dict(lag=lag, n=n, i=0, host=[torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(n)],
                        ev=[torch.cuda.Event() for _ in range(n)])
            self._loss_ring = ring
        k = ring["i"]
        ring["host"][k % ring["n"]].copy_(self.loss, non_blocking=True)
        ring["ev"][k % ring["n"]].record()
        ring["i"] = k + 1
        if k < lag:
            return None
        j = (k - lag) % ring["n"]
        ring["ev"][j].synchronize()
        return float(ring["host"][j])

    def flush(self):
        """Pipelined mode: apply the update that is still pending (no-op otherwise).  After it the parameters are what
        the un-pipelined step would have left."""
        if self.overlap and self._ov is not None and self._ov["pending"]:
            if self._ov["g_fused"] is not None:
                with torch.cuda.stream(self._ov["S_f"]):
                    self._ov["g_compute"][1 - self._ov["parity"]].replay()
                _cabi.LAUNCHES += self._ov["launches"][1]
                torch.cuda.current_stream(self.device).wait_stream(self._ov["S_f"])
            else:
                self._overlap_compute(1 - self._ov["parity"])     # the marched, not yet computed batch
                torch.cuda.current_stream(self.device).wait_stream(self._ov["S_c"])
            self._ov["pending"] = False
        if self.manual and self.pipelined and self._pending:
            self._apply_update(deferred=True)
            self.opt.state[6:7].zero_()  # nothing pending: the next step's leading launch only re-arms
            self._pending = False

    def _comm_error_lagged(self):
        """The fused data-parallel optimizer's sticky time-out flag WITHOUT a device sync: every call copies the flag to
        pinned host memory behind the work enqueued so far and evaluates the copy of the PREVIOUS call (one refresh interval
        earlier, long landed).  `opt.comm_error` (a blocking read) drained the launch queue at every occupancy refresh."""
        st = getattr(self, "_comm_flag", None)
        if st is None:
            st = dict(host=torch.zeros(1, dtype=torch.float32).pin_memory(), ev=torch.cuda.Event(), armed=False)
            self._comm_flag = st
        bad = False
        if st["armed"]:
            if not st["ev"].query():      # the host is more than a refresh interval ahead of the device: look next time
                return False
            bad = bool(st["host"][0] != 0)
        st["host"].copy_(self.opt.state[5:6], non_blocking=True)
        st["ev"].record()
        st["armed"] = True
        return bad

    def _bookkeeping_after(self, local_step_before):
        """Python-side effects of run_cuda that a graph replay does not re-execute."""
        model = self.model
        if not self.manual:  # (the hand-scheduled step writes step_counter and the sample total on the device)
            row = local_step_before % 16
            ws = getattr(model, "_train_ws", None)
            if ws is not None:
                model.step_counter[row].copy_(ws.counter)
        model.local_step = local_step_before + 1
        self._ls_mirror = model.local_step

    # -- inputs --------------------------------------------------------------------------------------------------
    def pack_inputs(self, rays_o, rays_d, G, pin=False):
        """One contiguous fp32 buffer [rays_o | rays_d | G] for a step: a packed batch reaches the step's static input
        buffers with ONE copy (host->device or device->device) instead of three."""
        parts = [rays_o.reshape(-1), rays_d.reshape(-1), G.reshape(-1)]
        out = torch.empty(sum(t.numel() for t in parts), dtype=torch.float32, device=rays_o.device)
        if pin and not out.is_cuda:
            out = out.pin_memory()
        torch.cat([t.float() for t in parts], out=out)
        return out

    def pack_pose_inputs(self, poses, intrinsics, G, pin=False):
        """device_rays mode: one contiguous fp32 buffer [poses (B x 16) | intrinsics (B x 4) | G] for a step."""
        return self.pack_inputs(poses, intrinsics, G, pin)

    def _batch_of(self, packed):
        per = (20 + 3 * self.H * self.W) if self.device_rays is not None else 9 * self.H * self.W
        B = packed.numel() // per
        if B * per != packed.numel():
            raise RuntimeError("packed inputs do not match H, W of this TrainStep")
        return B

    def _unpack(self, packed, B):
        if self.device_rays is not None:
            return (packed[:B * 16].view(B, 4, 4), packed[B * 16:B * 20].view(B, 4), packed[B * 20:].view(B, 3, self.H, self.W))
        n_ray = B * self.H * self.W * 3
        ro = packed[:n_ray].view(B, self.H * self.W, 3)
        rd = packed[n_ray:2 * n_ray].view(B, self.H * self.W, 3)
        G = packed[2 * n_ray:].view(B, 3, self.H, self.W)
        return ro, rd, G

    def __call__(self, rays_o, rays_d=None, G=None):
        """rays_o, rays_d [B, H*W, 3], G [B, 3, H, W] - or a single packed buffer from pack_inputs().
        device_rays mode: poses [B, 4, 4], intrinsics [B, 4], G - or a packed buffer from pack_pose_inputs()."""
        model = self.model
        if self.overlap:
            return self._call_overlap(rays_o, rays_d, G)
        packed = None
        if rays_d is None:
            packed = rays_o
            B = self._batch_of(packed)
        if self.global_step % self.update_interval == 0:
            self.flush()  # (pipelined mode) the refresh must see the parameters of the completed previous step
            if self.fused_optimizer and self.world > 1 and self.opt.peer_ptrs is not None and self.global_step > 0 \
                    and self._comm_error_lagged():
                # a cross-GPU wait inside the fused all-reduce + Adam kernel timed out: from that launch on the kernel
                # applies nothing on any rank that saw the flag (csrc/adam.cu) - stop instead of training on
                raise RuntimeError("data-parallel step: a peer did not reach the gradient exchange in time (see "
                                   "NGP_DP_TIMEOUT_MS); parameters were left untouched from that step on")
            if self.use_graph and not self.fused_optimizer:
                from . import field
                field.invalidate_half_cache()  # graph replays update the parameters without bumping ._version
            with torch.autocast("cuda", torch.float16), _nvtx.range("ngp.occupancy_refresh"):
                model.update_extra_state()
            self.n_updates += 1
        self.global_step += 1
        (self.opt.attach_grads if self.fused_optimizer else self.bucket.attach)()
        if self.fused_optimizer:
            self.opt.sync_shadow_if_changed()   # parameters edited through torch since the last step (load_state_dict ...)
        if self.manual and self._ls_mirror != model.local_step:
            self._local_step_dev.fill_(model.local_step)  # (update_extra_state restarts the 16-step window)
            self._ls_mirror = model.local_step

        if not self.use_graph:
            if packed is not None:
                if not packed.is_cuda:
                    packed = packed.to(self.device, non_blocking=True)
                rays_o, rays_d, G = self._unpack(packed, B)
            before = model.local_step
            loss = self._step_body(rays_o, rays_d, G)
            if self.manual:
                self._bookkeeping_after(before)
            else:
                self.samples.add_(model.step_counter[(model.local_step - 1) % 16, 0].long())
            self.loss = loss
            return loss

        if self._graph is None:
            if packed is not None:
                self._capture(*self._unpack(packed, B))
            else:
                self._capture(rays_o, rays_d, G)
        if packed is not None:
            self._static_packed.copy_(packed, non_blocking=True)
        else:
            ro_s, rd_s, g_s = self._static
            ro_s.copy_(rays_o, non_blocking=True)
            rd_s.copy_(rays_d, non_blocking=True)
            g_s.copy_(G, non_blocking=True)
        before = model.local_step
        if self._graph_exec:
            # bare cudaGraphLaunch: torch's replay() first enqueues two fill kernels (seed / offset of its generators),
            # ~7 us of serial device time per step; this graph holds no torch generator (device-side noise)
            with torch.cuda.device(self.device):
                _cabi.check(_cabi.load().ngp_graph_launch(self._graph_exec, _cabi.stream()), "ngp_graph_launch")
        else:
            self._graph.replay()
        self._pending = True
        _cabi.LAUNCHES += self._graph_launches  # our kernels inside the replayed graph
        self._bookkeeping_after(before)
        if not self.manual:
            self.samples.add_(model._train_ws.counter[0].long())
        return self.loss

    # -- overlap mode: march(k+1) beside compute(k) ---------------------------------------------------------------------
    _ov = None

    def _overlap_compute(self, q):
        ov = self._ov
        with torch.cuda.stream(ov["S_c"]):
            ov["S_c"].wait_event(ov["ev_march"][q])
            ov["g_compute"][q].replay()
            ov["ev_compute"][q].record(ov["S_c"])
        _cabi.LAUNCHES += ov["launches"][1]

    def _call_overlap(self, a, b=None, G=None):
        """One call = launch the MARCH half of this batch (stream S_m) and the COMPUTE half of the previous batch (stream
        S_c); the two run concurrently.  Returns the loss of the batch before the previous one as a 0-dim pinned CPU tensor
        (its compute has completed - no device sync, no stall); flush() computes the batch still pending.  Parameter
        updates happen in batch order exactly as in the sequential step; an occupancy refresh (every update_interval
        steps) first drains the pending compute, so it sees the same parameters and is seen by the same marches."""
        if not (self.manual and self.use_graph and self.fused_optimizer) or self.pipelined:
            raise RuntimeError("overlap=True needs the hand-scheduled, graphed step with the fused optimizer (and not pipelined=True)")
        model, dev = self.model, self.device
        packed = a if b is None else (self.pack_pose_inputs(a, b, G) if self.device_rays is not None else self.pack_inputs(a, b, G))
        B = self._batch_of(packed)
        cur = torch.cuda.current_stream(dev)
        if self._ov is None:
            self._capture_overlap(packed, B)
        ov = self._ov
        p = ov["parity"]
        if ov["g_fused"] is not None:
            return self._call_overlap_fused(packed, cur)
        S_m, S_c = ov["S_m"], ov["S_c"]
        ov["ev_compute"][p].synchronize()       # set p is free: compute(k-2) has finished (host-side: bounds the run-ahead)
        loss_out = ov["loss_ret"][p]
        loss_out.copy_(ov["loss_host"][p])      # its loss, before this call's graphs may overwrite the host slot
        S_m.wait_stream(cur)                    # the caller's input batch
        with torch.cuda.stream(S_m):
            ov["static"][p].copy_(packed, non_blocking=True)
            if self.global_step % self.update_interval == 0:
                if ov["pending"]:               # the refresh must see the parameters of the completed previous step
                    self._overlap_compute(1 - p)
                    ov["pending"] = False
                S_m.wait_stream(S_c)
                if self.world > 1 and self.opt.peer_ptrs is not None and self.global_step > 0 and self.opt.comm_error:
                    raise RuntimeError("data-parallel step: a peer did not reach the gradient exchange in time (see "
                                       "NGP_DP_TIMEOUT_MS); parameters were left untouched from that step on")
                with torch.autocast("cuda", torch.float16):
                    model.update_extra_state()
                self.n_updates += 1
            self.global_step += 1
            self.opt.attach_grads()
            self.opt.sync_shadow_if_changed()
            if self._ls_mirror != model.local_step:
                self._local_step_dev.fill_(model.local_step)
                self._ls_mirror = model.local_step
            ov["g_march"][p].replay()
            ov["ev_march"][p].record(S_m)
        _cabi.LAUNCHES += ov["launches"][0]
        if ov["pending"]:
            self._overlap_compute(1 - p)
        ov["pending"] = True
        ov["parity"] = 1 - p
        model.local_step += 1
        self._ls_mirror = model.local_step
        self.loss = loss_out
        return loss_out

    def _call_overlap_fused(self, packed, cur):
        """Overlap mode, one graph per call.  Call k (parity p = k % 2) puts batch k into input set p and replays, on ONE
        stream, the graph { march(set p) || compute(set 1 - p) }: batch k is marched while batch k - 1 - marched by the
        previous call - goes through field / loss / backward / scatter / optimizer.  Calls follow each other in stream order,
        so no events tie them; the host only waits for the graph of call k - 2 (the one of call k - 1 keeps the device busy
        meanwhile) and returns the loss that graph produced: the loss of batch k - 3, as a pinned CPU scalar.
        The first call, and every call that refreshes the occupancy grid (which must see the previous step's parameters and be
        seen by this step's march), run the halves as separate graphs: pending compute, refresh, march."""
        model, ov = self.model, self._ov
        p = ov["parity"]
        S_f = ov["S_f"]
        ov["ev_graph"][p].synchronize()
        loss_out = ov["loss_ret"][p]
        loss_out.copy_(ov["loss_host"][1 - p])
        S_f.wait_stream(cur)                    # the caller's input batch
        with torch.cuda.stream(S_f):
            ov["static"][p].copy_(packed, non_blocking=True)
            refresh = self.global_step % self.update_interval == 0
            split = refresh or not ov["pending"]
            if split and ov["pending"]:
                ov["g_compute"][1 - p].replay()
                _cabi.LAUNCHES += ov["launches"][1]
                ov["pending"] = False
            if refresh:
                if self.world > 1 and self.opt.peer_ptrs is not None and self.global_step > 0 and self.opt.comm_error:
                    raise RuntimeError("data-parallel step: a peer did not reach the gradient exchange in time (see "
                                       "NGP_DP_TIMEOUT_MS); parameters were left untouched from that step on")
                with torch.autocast("cuda", torch.float16):
                    model.update_extra_state()
                self.n_updates += 1
            self.global_step += 1
            self.opt.attach_grads()
            self.opt.sync_shadow_if_changed()
            if self._ls_mirror != model.local_step:
                self._local_step_dev.fill_(model.local_step)
                self._ls_mirror = model.local_step
            if split:
                ov["g_march"][p].replay()
                _cabi.LAUNCHES += ov["launches"][0]
            else:
                ov["g_fused"][p].replay()
                _cabi.LAUNCHES += ov["launches"][0] + ov["launches"][1]
            ov["ev_graph"][p].record(S_f)
        ov["pending"] = True
        ov["parity"] = 1 - p
        model.local_step += 1
        self._ls_mirror = model.local_step
        self.loss = loss_out
        return loss_out

    def _capture_overlap(self, packed, B):
        """Warm up (real steps, rolled back afterwards) and capture the four graphs: march / compute x two workspace sets."""
        model, dev = self.model, self.device
        per = packed.numel()
        S_m, S_c = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev, priority=-1)
        ov = dict(S_m=S_m, S_c=S_c, parity=0, pending=False, B=B,
                  static=[torch.empty(per, dtype=torch.float32, device=dev) for _ in range(2)],
                  ev_march=[torch.cuda.Event() for _ in range(2)], ev_compute=[torch.cuda.Event() for _ in range(2)],
                  loss_host=[torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)],
                  loss_ret=[torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)],
                  g_march=[None, None], g_compute=[None, None], launches=[0, 0])
        cur = torch.cuda.current_stream(dev)
        saved_step = model.local_step
        snap = self._snapshot_training_state()
        rng = torch.cuda.get_rng_state(dev)
        S_m.wait_stream(cur)
        with torch.cuda.stream(S_m):
            for p in (0, 1):
                ov["static"][p].copy_(packed)
        S_c.wait_stream(S_m)

        def march(p):
            ins = self._unpack(ov["static"][p], B)
            return self._manual_march(ins[0], ins[1], B, p, bg_early=False)

        def compute(p):
            m = self._mws_sets[p]
            loss = self._manual_compute(m, self._unpack(ov["static"][p], B)[2], bg_done=False)
            ov["loss_host"][p].copy_(loss, non_blocking=True)

        for p in (0, 1):
            for _ in range(2):                   # warm-up: allocations, lazy initialisation, kernel attributes
                with torch.cuda.stream(S_m):
                    march(p)
                S_c.wait_stream(S_m)
                with torch.cuda.stream(S_c):
                    compute(p)
                S_m.wait_stream(S_c)
        torch.cuda.synchronize(dev)
        self._restore_training_state(snap)
        model.local_step = saved_step
        self._local_step_dev.fill_(saved_step)
        self._ls_mirror = saved_step
        torch.cuda.synchronize(dev)
        for p in (0, 1):
            l0 = _cabi.LAUNCHES
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=S_m, capture_error_mode="thread_local"):
                march(p)
            ov["g_march"][p] = g
            l1 = _cabi.LAUNCHES
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=S_c, capture_error_mode="thread_local"):
                compute(p)
            ov["g_compute"][p] = g
            ov["launches"] = [l1 - l0, _cabi.LAUNCHES - l1]
            _cabi.LAUNCHES = l0
        ov["g_fused"] = None
        if self.overlap_fused:
            # the same two halves once more, as the two branches of ONE graph: set p marches while set 1 - p computes
            S_f = torch.cuda.Stream(device=dev)
            S_f.wait_stream(S_m)
            S_f.wait_stream(S_c)
            ov["S_f"], ov["ev_graph"], ov["g_fused"] = S_f, [torch.cuda.Event() for _ in range(2)], [None, None]
            for p in (0, 1):
                l0 = _cabi.LAUNCHES
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=S_f, capture_error_mode="thread_local"):
                    S_m.wait_stream(S_f)
                    S_c.wait_stream(S_f)
                    with torch.cuda.stream(S_c):
                        compute(1 - p)
                    with torch.cuda.stream(S_m):
                        march(p)
                    S_f.wait_stream(S_m)
                    S_f.wait_stream(S_c)
                ov["g_fused"][p] = g
                _cabi.LAUNCHES = l0
            cur.wait_stream(S_f)
        torch.cuda.set_rng_state(rng, dev)
        model.local_step = saved_step
        self._pending = False
        cur.wait_stream(S_m)
        cur.wait_stream(S_c)
        self._mws = self._mws_sets[0]
        self._ov = ov

    def _capture(self, rays_o, rays_d, G):
        model = self.model
        B = rays_o.shape[0]
        per = (20 + 3 * self.H * self.W) if self.device_rays is not None else 9 * self.H * self.W
        self._static_packed = torch.empty(B * per, dtype=torch.float32, device=self.device)
        self._static = self._unpack(self._static_packed, B)
        ro_s, rd_s, g_s = self._static
        ro_s.copy_(rays_o)
        rd_s.copy_(rays_d)
        g_s.copy_(G)
        # warm up on a side stream (allocator, lazy initialisation, cudaFuncSetAttribute) before capturing.  The warm-up
        # passes are REAL steps (they must touch every code path the capture will); everything they change - parameters,
        # fp16 shadow, Adam moments, step count / loss scale / growth tracker, step_counter rows, sample total - is
        # snapshotted first and restored afterwards, so graph=True trains exactly like graph=False.
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        saved_step = model.local_step
        snap = self._snapshot_training_state()
        with torch.cuda.stream(side):
            for _ in range(3):
                self._step_body(ro_s, rd_s, g_s)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._restore_training_state(snap)
        model.local_step = saved_step
        if self.manual:
            self._local_step_dev.fill_(saved_step)
            self._ls_mirror = saved_step
        torch.cuda.synchronize()
        self._graph = torch.cuda.CUDAGraph()
        launches0 = _cabi.LAUNCHES
        with torch.cuda.graph(self._graph, capture_error_mode="thread_local"):
            self.loss = self._step_body(ro_s, rd_s, g_s)
        self._graph_launches = _cabi.LAUNCHES - launches0
        _cabi.LAUNCHES = launches0  # capture launches nothing
        model.local_step = saved_step
        self._pending = snap["pending"]
        # a graph without torch generators (hand-scheduled step, device-side noise) is launched bare (see __call__)
        self._graph_exec = 0
        no_torch_rng = self.manual and self.device_noise and not self.mirror_rng and self.fixed_noises is None
        if no_torch_rng and os.environ.get("NGP_RAW_GRAPH_LAUNCH", "1") not in ("", "0") and hasattr(self._graph, "raw_cuda_graph_exec"):
            try:
                self._graph_exec = int(self._graph.raw_cuda_graph_exec())
            except Exception:  # noqa: BLE001 - older torch: keep replay()
                self._graph_exec = 0

    def _snapshot_training_state(self):
        """Everything a train step mutates besides its own scratch (see _capture)."""
        snap = dict(step_counter=self.model.step_counter.clone(), samples=self.samples.clone(), pending=self._pending,
                    rng=self._rng.clone())
        if self.fused_optimizer:
            o = self.opt
            snap["opt"] = [t.clone() for t in (o.flat_params, o.flat_half, o.exp_avg, o.exp_avg_sq, o.state)]
        else:
            snap["params"] = [p.detach().clone() for p in self.model.parameters()]
            snap["adam"] = {id(p): {k: (v.clone() if torch.is_tensor(v) else v) for k, v in st.items()}
                            for p, st in self.opt.state.items()}
            sc = self.scaler
            snap["scaler"] = None if sc._scale is None else (sc._scale.clone(), sc._growth_tracker.clone())
        return snap

    def _restore_training_state(self, snap):
        with torch.no_grad():
            self.model.step_counter.copy_(snap["step_counter"])
            self.samples.copy_(snap["samples"])
            self._rng.copy_(snap["rng"])
            if self.fused_optimizer:
                o = self.opt
                err = o.state[5].clone()   # a cross-GPU timeout during the warm-up must stay visible
                for dst, src in zip((o.flat_params, o.flat_half, o.exp_avg, o.exp_avg_sq, o.state), snap["opt"]):
                    dst.copy_(src)
                o.state[5].copy_(torch.maximum(err, o.state[5]))
                o.flat_grads.zero_()
                if self._g_table_odd is not None:
                    # the odd-row twin of the table gradient: pipelined mode leaves the last warm-up step's share there
                    # (its update, which folds it, is still pending) - it would land in the first real update
                    self._g_table_odd.zero_()
                # (o._sync - the cross-GPU barrier epoch - keeps counting: the peers' flags carry it)
            else:
                for p, q in zip(self.model.parameters(), snap["params"]):
                    p.copy_(q)
                for p, st in self.opt.state.items():   # in place: a capturable Adam's state tensors must keep their addresses
                    old = snap["adam"].get(id(p))
                    for k, v in st.items():
                        if torch.is_tensor(v):
                            v.copy_(old[k]) if old is not None and k in old else v.zero_()
                if snap["scaler"] is not None:
                    self.scaler._scale.copy_(snap["scaler"][0])
                    self.scaler._growth_tracker.copy_(snap["scaler"][1])
                elif self.scaler._scale is not None:
                    self.scaler._scale.fill_(self.scaler._init_scale)
                    self.scaler._growth_tracker.zero_()
                self.bucket.zero()
