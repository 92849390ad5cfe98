#!/usr/bin/env python
"""bench.py - NeRF train-step samples/s (march + hash-grid + MLP + composite, fwd + bwd) on 1..8 B200.

    python bench.py --gpus N --steps K --warmup W           # the B200-native arm (this repo)
    python bench.py --impl reference --steps K --warmup W   # the reference's CPU renderer on host cores

Workload (BASELINE.json configs[2]/[3], SURVEY.md 8d cfg3/cfg4): the `-O` train step of
nerf/network_grid.py (tiled 16x2 grid, 2^16 rows/level, 32->64->64->4 MLP, 128^3 occupancy grid,
max_steps 1024), 8 camera views of 64x64 rays per step sharded over the N ranks, fp16 autocast +
GradScaler, synthetic SDS gradient in place of the U-Net (`pred_rgb.backward(gradient=G,
retain_graph=True)`), entropy regulariser backward, flat-bucket gradient all-reduce, Adam step,
occupancy update every 16 steps (inside the timed region).  A "sample" is one marched point
actually produced (sum of step_counter[:, 0]), padding excluded.

One JSON line is printed by rank 0; see the task contract for the keys.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "single-stable-dreamfusion_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "NeRF train-step samples/s (march+hashgrid+MLP+composite fwd/bwd)"
NCU_TRAFFIC_FILE = os.path.join(ROOT, "profiles", "ncu_traffic.json")  # written by profiles/tools/ncu_traffic.py from an
#                                                                         ncu --set full capture of THIS build's kernels
UNIT = "samples/s"
VIEWS_PER_STEP = 8
H = W = 64
MAX_STEPS = 1024
LOSS_LAG = 8   # e2e leg: the host consumes step k's loss while step k + LOSS_LAG is being enqueued


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps: train steps (default 48), GridEncoder fwd / fwd+bwd "
                    "iterations of --config encoder (default 12), frames of --config infer (default --frames, the orbit is "
                    "cycled), CPU steps of --impl reference (default 12)")
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="train", choices=["train", "infer", "encoder"], help="train: the -O train step (the headline "
                    "metric, BASELINE configs[2]/[3]); infer: BASELINE configs[4], the 100-frame 800x800 test orbit through "
                    "the inference branch of run_cuda; encoder: BASELINE configs[1], the standalone GridEncoder on 2^22 points "
                    "(1 GPU; secondary lines with their own metrics)")
    ap.add_argument("--frames", type=int, default=100, help="--config infer: frames of the orbit")
    ap.add_argument("--res", type=int, default=800, help="--config infer: image side")
    ap.add_argument("--views", type=int, default=VIEWS_PER_STEP, help="camera views per step, whole job")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true", help="skip timing the reference's CUDA extensions")
    ap.add_argument("--cpu-sample-steps", type=int, default=3)
    ap.add_argument("--lr", type=float, default=1e-5)
    ap.add_argument("--no-graph", action="store_true", help="run the train step eagerly instead of as one CUDA graph")
    ap.add_argument("--autograd", action="store_true", help="autograd version of the step instead of the hand-scheduled kernels")
    ap.add_argument("--ray-order", default="rows", choices=["tiles", "rows"], help="sharding of a view's rays over the ranks "
                    "(rows: interleaved image rows, measured 9 %% faster at 8 GPUs than 8x8 blocks dealt along diagonals)")
    ap.add_argument("--pipeline", action="store_true", help="apply step k's optimizer update at the start of step k+1 "
                    "(beside the ray marching) also on ONE GPU; with more GPUs it is the default (measured at 8: -11 %% step time)")
    ap.add_argument("--no-pipeline", action="store_true", help="multi-GPU: run the fused all-reduce + Adam at the end of its own step")
    ap.add_argument("--overlap", action="store_true", help="run each step's ray marching beside the previous step's field / backward "
                    "/ optimizer half (TrainStep(overlap=True)); measured: slower at 1 GPU (both halves are issue-bound: 2.19 vs 2.11 ms) "
                    "and host-bound at 8 (0.58 vs 0.39 ms per step), kept as an option")
    ap.add_argument("--chunks", type=int, default=0, help="ray chunks run as parallel chains (0 = the default, 2)")
    ap.add_argument("--nccl", action="store_true", help="NCCL all-reduce instead of the fused peer-memory all-reduce + Adam")
    ap.add_argument("--kernel-table", default=None, help="write a torch.profiler per-kernel table of 5 steps to this file")
    ap.add_argument("--dp-sweep", action="store_true", help="multi-GPU: after the timed regions, re-time 100 steps under a few "
                    "settings of the data-parallel step (optimizer grid size, quad table, chains, optimizer placement) in the "
                    "same process group; results in the line's `dp_sweep`")
    ap.add_argument("--timeline", default=None, help="write the kernel timeline (CUPTI: name, stream, start, duration) of 3 "
                    "graphed steps to this JSON file - where the step's time goes between the kernels")
    ap.add_argument("--profile-steps", type=int, default=8, help="eager steps timed per kernel for the roofline")
    ap.add_argument("--host-rays", action="store_true", help="feed pre-generated rays (1.18 MB / step) instead of camera poses; "
                    "default: the step's input is 8 poses + intrinsics + the guidance gradient, rays are generated on the device")
    ap.add_argument("--sync-loss", action="store_true", help="e2e leg: read every step's loss with loss.item() (a device sync per "
                    "step, as the reference loop does) instead of the asynchronous pinned-memory read")
    ap.add_argument("--no-shading", action="store_true", help="skip the secondary lambertian-vs-albedo step timing")
    ap.add_argument("--ref-steps", type=int, default=200, help="timed steps of the reference CUDA-extension pipeline")
    ap.add_argument("--ref-warmup", type=int, default=50)
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="after the timed steps, write what the last timed step "
                    "returned as DIR/<name>.npy in float32 / float64, to compare two builds output for output: train: its loss "
                    "and the model state it left; infer: the last frame's rgb and depth; encoder: a fixed sample of the last "
                    "backward's table gradient; --impl reference: its loss and the model state")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 12 if (args.impl == "reference" or args.config == "encoder") else (
            args.frames if args.config == "infer" else 48)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's pure-PyTorch non-cuda-ray renderer on host cores
# ---------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, dump_dir=None):
    """BASELINE.json configs[0]: 64x64 rays x (64+32) samples, vanilla NeRF, fp32 fwd+bwd on CPU.
    Returns (samples/s, ms/step, cores, description); dump_dir: write the last step's results (dump_outputs)."""
    import torch
    from oracle import torch_renderer as TR
    # all host cores, whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1 for every rank)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    torch.manual_seed(0)
    model = TR.VanillaNeRF(bound=1.0, min_near=0.1, bg_radius=1.4)
    model.train()
    views = [TR.make_view(H, W, seed=s) for s in range(4)]
    G = torch.randn(1, H * W, 3, generator=torch.Generator().manual_seed(1))
    for i in range(warmup):
        TR.train_step(model, *views[i % 4], G)
    t0 = time.perf_counter()
    n = 0
    for i in range(steps):
        k, res = TR.train_step(model, *views[i % 4], G)
        n += k
    dt = time.perf_counter() - t0
    if dump_dir:
        dump_outputs(dump_dir, {k: v for k, v in res.items() if torch.is_tensor(v)})
    cores = torch.get_num_threads()
    desc = ("%d fwd+bwd steps of one 64x64-ray view x (64+32) samples through a port of nerf/renderer.py:run + "
            "nerf/network.py (fp32, %d torch threads of %d host cpus)" % (steps, cores, os.cpu_count() or 0))
    return n / dt, dt / max(steps, 1) * 1e3, cores, desc


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    warm = max(1, min(args.warmup, 2))
    v, ms, cores, desc = cpu_reference_run(steps, warm, dump_dir=args.dump_outputs)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "reference CPU path: nerf/network.py vanilla NeRF + NeRFRenderer.run, 64x64 rays x "
                               "(64+32) samples, fwd+bwd (BASELINE configs[0]); sample = composited sample"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
            self.f.close()
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = sorted(float(r[1]) for r in rows if len(r) >= 9)
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = max(float(r[2]) for r in rows if len(r) >= 9)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for k, nm in enumerate(names):
                    if any("Active" == r[5 + k].strip() for r in rows if len(r) >= 9):
                        out["reasons"].append(nm)
            os.remove(self.path)
        except Exception:
            pass
        return out


# ---------------------------------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------------------------------
def build_model(device):
    import torch
    from ngp_b200.network_grid import NeRFNetwork
    opt = argparse.Namespace(bound=1, cuda_ray=True, min_near=0.1, density_thresh=10, bg_radius=1.4)
    torch.manual_seed(0)
    model = NeRFNetwork(opt).to(device)
    model.train()
    return model


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: {name: tensor} as out_dir/<name>.npy; floating tensors as float32, integer ones as float64 (exact).
    Nothing is written when the whole exceeds DUMP_LIMIT_BYTES."""
    import numpy as np
    import torch
    conv = {}
    for name, t in arrays.items():
        if t is not None:
            t = torch.as_tensor(t).detach().cpu()
            conv[name] = (t.float() if t.is_floating_point() else t.double()).numpy()
    total = sum(a.nbytes for a in conv.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes, more than %d" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in conv.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure_l2_peaks(device):
    """Chip ceilings for the encoder's access shapes: random 4-byte gathers / 8-byte red.add over a 24 MB
    (L2-resident) table.  Returns (gathers/s, reds/s)."""
    import torch
    from ngp_b200 import _cabi
    words = 1 << 23  # 32 MB of u32; power of two; L2 is 126 MB
    table = torch.zeros(words, dtype=torch.int32, device=device)
    n_threads, iters = 148 * 2048 * 4, 16
    sink = torch.empty(n_threads, dtype=torch.int32, device=device)
    ftable = torch.zeros(words, dtype=torch.float32, device=device)
    res = []
    for name, args in (("ngp_bench_gather4", (_cabi.ptr(table), words, _cabi.ptr(sink), n_threads, iters, 1)),
                       ("ngp_bench_red8", (_cabi.ptr(ftable), words, n_threads, iters, 2))):
        best = 0.0
        for rep in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _cabi.call(name, device, *args)
            e1.record()
            torch.cuda.synchronize()
            ops = n_threads * iters * 8
            best = max(best, ops / (e0.elapsed_time(e1) * 1e-3))
        res.append(best)
    return res[0], res[1]


def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    from ngp_b200 import _cabi, provider
    from ngp_b200.parallel import shard_pixels, shard_rows

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "the B200 arm needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    _cabi.load()

    # Data-parallel sharding of the step's 8 x 4096 rays: every rank renders its share of EVERY view - 8x8-pixel blocks
    # dealt round-robin along the block diagonals (parallel.shard_pixels; --ray-order rows: interleaved image rows).
    # Per-rank sample counts stay balanced (whole views differ 4x in samples) and a rank's rays stay spatially coherent.
    if (H * W) % world != 0:
        raise SystemExit("--gpus must divide the ray count of a view")
    if args.ray_order == "tiles":
        pix = shard_pixels(H, W, rank, world)
    else:
        pix = [r * W + c for r in shard_rows(H, rank, world) for c in range(W)]
    pix_t = torch.tensor(pix, dtype=torch.long)
    Hl = len(pix) // W
    n_pool = 64
    device_rays = not args.host_rays and not args.autograd and args.ray_order == "rows"
    if device_rays:
        poses_all, intr_all = provider.make_training_poses(n_pool * args.views, H, W, seed=0)
        poses_all, intr_all = poses_all.view(n_pool, args.views, 4, 4), intr_all.view(n_pool, args.views, 4)
    else:
        ro_all, rd_all = provider.make_training_views(n_pool * args.views, H, W, seed=0, pin=False)
        ro_all = ro_all.view(n_pool, args.views, H * W, 3)[:, :, pix_t].contiguous()
        rd_all = rd_all.view(n_pool, args.views, H * W, 3)[:, :, pix_t].contiguous()
    # the guidance gradient of the rendered pixels, in the same ray order ([views, 3, rays of this rank])
    g_all = (torch.randn(n_pool, args.views, 3, H * W, generator=torch.Generator().manual_seed(2)) * 1e-2)[:, :, :, pix_t]
    g_all = g_all.reshape(n_pool, args.views, 3, Hl, W).contiguous()

    from ngp_b200.trainer import TrainStep
    model = build_model(device)
    # lr: the optimizer step runs in full, but a small step keeps the synthetic (random-gradient) scene at its
    # random-init occupancy so that every timed pass sees the same ~3.4 M samples per step
    step_fn = TrainStep(model, Hl, W, lr=args.lr, max_steps=MAX_STEPS, graph=not args.no_graph, world_size=world,
                        manual=False if args.autograd else None, peer_allreduce=False if args.nccl else None,
                        pipelined=(False if (args.no_pipeline or args.autograd or args.overlap) else (True if args.pipeline else None)),
                        n_chunks=args.chunks or None,
                        device_rays=(H, rank, world) if device_rays else None,
                        overlap=bool(args.overlap and not (args.no_graph or args.autograd)))
    # one packed, pinned host buffer per batch: a step's inputs are ONE copy - [poses | intrinsics | G] (the rays of this
    # rank's interleaved image rows are generated by the step's prologue kernel), or [rays_o | rays_d | G] with --host-rays
    if device_rays:
        host_pool = torch.stack([step_fn.pack_pose_inputs(poses_all[k], intr_all[k], g_all[k].contiguous())
                                 for k in range(n_pool)]).pin_memory()
    else:
        host_pool = torch.stack([step_fn.pack_inputs(ro_all[k], rd_all[k], g_all[k].contiguous()) for k in range(n_pool)]).pin_memory()

    def host_batch(i):
        return host_pool[i % n_pool]

    # inputs resident in HBM for the `value` measurement
    dev_pool = host_pool.to(device)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sample_acc = step_fn.samples

    step_events = []
    last_loss = [None]

    def run_steps(n, e2e, start_index, record=False):
        for s in range(n):
            if record:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                step_events.append(ev)
            i = start_index + s
            # graph mode copies the packed batch straight into the step's static input buffer (H2D when it is a host batch)
            loss = step_fn(host_batch(i) if e2e else dev_pool[i % n_pool])
            last_loss[0] = loss
            if e2e:
                # device -> host read of the step's result, every step: the loss is copied to pinned host memory right
                # behind the step and consumed LOSS_LAG calls later (TrainStep.read_loss_async), --sync-loss: loss.item().
                # (A lag of 2 kept the host at most two steps ahead of the device: every scheduling hiccup of one of the 4-8
                #  rank processes then stalled its GPU - and, through the gradient exchange, all of them: e2e was 13 % below
                #  `value` at 4 GPUs.)
                if args.sync_loss:
                    loss.item()
                else:
                    step_fn.read_loss_async(lag=LOSS_LAG)

    # ---- warm-up ------------------------------------------------------------------------------------
    # the clock sampler (an nvidia-smi child process) is started BEFORE the warm-up: its start-up takes driver locks that
    # stall kernel launches for 10-25 ms, which must not land inside the timed region; its samples span both timed regions
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
        time.sleep(1.0)
    run_steps(max(args.warmup, 3), False, 0)
    barrier()

    # ---- timed: inputs resident ----------------------------------------------------------------------
    sample_acc.zero_()
    updates0 = step_fn.n_updates
    launches0 = _cabi.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    host_t0 = time.perf_counter()
    run_steps(args.steps, False, 1000, record=True)
    host_ms = (time.perf_counter() - host_t0) * 1e3 / args.steps   # host time to ENQUEUE a step (the loop does not sync)
    step_fn.flush()  # pipelined optimizer: the last step's update belongs to the timed work
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    per_step_raw = [a.elapsed_time(b) for a, b in zip(step_events, step_events[1:] + [e1])]
    per_step = sorted(per_step_raw)
    launches = _cabi.LAUNCHES - launches0
    n_updates = step_fn.n_updates - updates0
    samples = int(sample_acc.item())

    # ---- timed: end to end (pinned host inputs, H2D inside, loss read back) -----------------------------
    sample_acc.zero_()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    f0.record()
    run_steps(args.steps, True, 2000)
    step_fn.flush()
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    samples_e2e = int(sample_acc.item())
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # before the untimed profiling steps below, which train the model further
        dump_outputs(args.dump_outputs, dict(model.state_dict(), loss=last_loss[0]))   # ~17 MB

    if args.kernel_table and rank == 0:
        from torch.profiler import profile, ProfilerActivity
        torch.cuda.synchronize()
        step_fn.global_step = 1
        with profile(activities=[ProfilerActivity.CUDA]) as prof_t:
            run_steps(5, False, 2500)
            torch.cuda.synchronize()
        with open(args.kernel_table, "w") as f:
            f.write("# torch.profiler (CUPTI) kernel times over 5 steps of the graphed train step; divide by 5 for per step\n")
            f.write(prof_t.key_averages().table(sort_by="cuda_time_total", row_limit=45, max_name_column_width=90))

    dp_sweep = None
    if args.dp_sweep and world > 1 and step_fn.manual and step_fn.use_graph:
        lib = _cabi.load()
        dp_sweep = []

        def variant(tag, setup, n=100):
            step_fn.flush()
            barrier()
            setup()
            step_fn._graph = None          # re-capture under the new setting
            run_steps(20, False, 4000)
            step_fn.flush()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run_steps(n, False, 5000)
            step_fn.flush()
            b.record()
            barrier()
            t = torch.tensor([a.elapsed_time(b) / n], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dp_sweep.append({"setting": tag, "ms_per_step": round(t.item(), 5)})

        def set_blocks(v):
            return lambda: _cabi.check(lib.ngp_dp_set_option(1, v), "ngp_dp_set_option")

        def set_attr(**kw):
            def f():
                for k, v in kw.items():
                    setattr(step_fn, k, v)
                if "n_chunks" in kw:
                    step_fn._mws = None
            return f

        variant("default", lambda: None)
        for v in (14, 56, 112, 148):
            variant("optimizer grid %d blocks" % v, set_blocks(v))
        variant("default again", set_blocks(0))
        variant("quad table on", set_attr(quad_table=True))
        variant("quad table off, 1 chain", set_attr(quad_table=False, n_chunks=1))
        variant("3 chains", set_attr(n_chunks=3))
        variant("2 chains, optimizer at the end of its own step", set_attr(n_chunks=2, pipelined=False))
        variant("default restored", set_attr(pipelined=True))
        if rank == 0:
            print("DP_SWEEP " + json.dumps(dp_sweep), file=sys.stderr, flush=True)

    if args.timeline and rank == 0:
        from torch.profiler import profile, ProfilerActivity
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof_t:
            run_steps(4, False, 2600)
            step_fn.flush()
            torch.cuda.synchronize()
        with tempfile.NamedTemporaryFile(suffix=".json") as tf:
            prof_t.export_chrome_trace(tf.name)
            tr = json.load(open(tf.name))
        ev = [e for e in tr.get("traceEvents", []) if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")]
        ev.sort(key=lambda e: e["ts"])
        t0 = ev[0]["ts"] if ev else 0.0
        rows = [dict(t_us=round(e["ts"] - t0, 2), dur_us=round(e["dur"], 2), stream=e.get("args", {}).get("stream"),
                     name=e["name"][:70], grid=e.get("args", {}).get("grid"), block=e.get("args", {}).get("block")) for e in ev]
        with open(args.timeline, "w") as f:
            json.dump(rows, f, indent=0)

    # ---- per-kernel durations for the roofline: a few EAGER steps with CUDA events around our entry points ----
    # (events cannot be recorded inside a graph replay; same kernels, same data shapes).  ONE serial chain on ONE stream:
    # concurrent chains inflate each other's event-to-event times, and a side-stream kernel's events would include its
    # waits - so the background-net branch is folded into the main stream for these steps and every kernel is timed alone.
    kern = {}
    prof_samples = 0
    red_lane_ops = 0
    red_samples = 0
    was_graph, was_overlap = step_fn.use_graph, step_fn.overlap
    step_fn.flush()
    torch.cuda.synchronize()
    step_fn.use_graph, step_fn.overlap = False, False
    saved_ws = (step_fn.n_chunks, step_fn._mws, step_fn._chain, getattr(model, "_train_ws", None), step_fn._side,
                step_fn._side_fwd)
    if step_fn.manual:
        step_fn.n_chunks, step_fn._mws = 1, None
        step_fn._side = step_fn._side_fwd = torch.cuda.current_stream(device)
    names = ["ngp_grid_scatter_samples", "ngp_grid_encode_backward", "ngp_field_forward", "ngp_field_forward_quads",
             "ngp_grid_quad_table", "ngp_field_backward",
             "ngp_march_rays_train", "ngp_march_rays_train_packed", "ngp_composite_rays_train_forward", "ngp_composite_rays_train_backward",
             "ngp_grid_encode_forward", "ngp_train_prologue", "ngp_train_prologue_rays", "ngp_train_ray_loss", "ngp_bg_forward", "ngp_bg_backward",
             "ngp_adam_step_fused", "ngp_grid_scatter_samples_split", "ngp_grid_fold_odd"]
    step_fn.global_step = 1  # keep the occupancy refresh out of the profiled steps
    run_steps(2, False, 3000)
    torch.cuda.synchronize()
    _cabi.PROFILE = {n: [] for n in names}
    sample_acc.zero_()
    run_steps(args.profile_steps, False, 3100)
    torch.cuda.synchronize()
    prof = _cabi.PROFILE
    _cabi.PROFILE = None
    prof_samples = int(sample_acc.item())
    for name, evs in prof.items():
        if evs:
            # (the two-buffer scatter is the same kernel as ngp_grid_scatter_samples: reported under that name)
            # (and the quad-table forward is the same kernel as ngp_field_forward)
            kern[name.replace("_samples_split", "_samples").replace("_forward_quads", "_forward")] = (
                sum(a.elapsed_time(b) for a, b in evs), len(evs))
    # post-aggregation atomic traffic of the grid scatter: the counting build of the same kernel over the same steps
    # (untimed; one counter add per lane) - the roofline divides these lane-ops by the measured red issue ceiling
    if step_fn.manual:
        import ctypes
        lib = _cabi.load()
        n_red = ctypes.c_uint64(0)
        lib.ngp_grid_red_count(ctypes.byref(n_red), 1)
        lib.ngp_grid_set_option(1, 1)
        sample_acc.zero_()
        run_steps(args.profile_steps, False, 3100)
        torch.cuda.synchronize()
        lib.ngp_grid_set_option(1, 0)
        lib.ngp_grid_red_count(ctypes.byref(n_red), 1)
        red_lane_ops = int(n_red.value)
        red_samples = int(sample_acc.item())
    step_fn.use_graph, step_fn.overlap = was_graph, was_overlap
    if step_fn.manual:
        step_fn.flush()
        torch.cuda.synchronize()
        step_fn.n_chunks, step_fn._mws, step_fn._chain, model._train_ws, step_fn._side, step_fn._side_fwd = saved_ws
    if world > 1:
        dist.barrier()

    # ---- data-parallel correctness, in the same run (N > 1): fused peer all-reduce + Adam vs NCCL all-reduce + Adam ----
    dp_result = None
    if world > 1:
        from ngp_b200 import dp_check
        try:
            dp_result = dp_check.run(device, steps=6, grad_div=1.0)
            dp_result.pop("_objects", None)
        except Exception as e:  # noqa: BLE001
            dp_result = {"ok": False, "error": repr(e)[:300]}

    # ---- reduce over ranks: time = max, samples = sum ------------------------------------------------------
    stats = torch.tensor([ms, ms_e2e, float(samples), float(samples_e2e)], dtype=torch.float64, device=device)
    if world > 1:
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, ms_e2e, samples, samples_e2e = mx[0].item(), mx[1].item(), sm[2].item(), sm[3].item()

    if rank == 0:
        value = samples / (ms * 1e-3)
        e2e_value = samples_e2e / (ms_e2e * 1e-3)
        h2d = host_batch(0).numel() * host_batch(0).element_size() * world
        gathers_s, reds_s = measure_l2_peaks(device)
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(
            os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
        hbm_peak = peaks.get("hbm_gbs") or 6650.0
        hbm_src = "MEASURED_PEAKS.json (measured)" if peaks.get("hbm_gbs") else "fallback 6.65 TB/s (B200_PROFILING.md)"
        # dominant kernel: the longest of the MAIN chain (the background net runs beside it on a side stream)
        main_chain = {k: v for k, v in kern.items() if k not in ("ngp_bg_forward", "ngp_bg_backward")}
        dom = max(main_chain, key=lambda k: main_chain[k][0])
        tot_ms, n_calls = kern[dom]
        per_launch_ms = tot_ms / max(n_calls, 1)
        launches_per_step = n_calls / max(args.profile_steps, 1)
        points_per_launch = prof_samples / max(n_calls, 1)
        sec = per_launch_ms * 1e-3
        step_kernel_ms = sum(v[0] for v in kern.values()) / max(args.profile_steps, 1)
        traffic = None
        try:
            tr = json.load(open(NCU_TRAFFIC_FILE))
            if dom in tr:
                traffic = tr[dom]   # {"dram_bytes_per_launch", "samples_per_launch", "capture"}
        except Exception:
            pass
        roofline = {"kernel": dom, "unit": "GB/s", "avg_launch_ms": per_launch_ms, "launches_per_step": launches_per_step,
                    "samples_per_launch": points_per_launch,
                    "share_of_step": (tot_ms / max(args.profile_steps, 1)) / max(step_kernel_ms, 1e-9),
                    # (the capture's bytes per launch, scaled to this run's samples per launch)
                    "traffic": (traffic["dram_bytes_per_launch"] * points_per_launch / max(traffic.get("samples_per_launch", 0.0), 1.0)
                                if traffic else None), "traffic_source": traffic,
                    "l2_gather_peak_gbs": gathers_s * 4 / 1e9, "l2_red_lane_ops_peak_per_s": reds_s,
                    "hbm_peak_gbs": hbm_peak, "hbm_peak_source": hbm_src,
                    "how": "CUDA events around each entry point over %d eager single-chain steps after the timed region, "
                           "every kernel alone on the stream" % args.profile_steps,
                    "kernels_ms_per_step": {k: v[0] / max(args.profile_steps, 1) for k, v in kern.items()},
                    "our_kernels_ms_per_step": step_kernel_ms}
        if dom in ("ngp_grid_scatter_samples", "ngp_grid_encode_backward") and red_lane_ops:
            # The scatter is bound by how fast the SMs ISSUE reds: ~1.3 cycles per active lane per SM whatever the width
            # (measured in this run by ngp_bench_red8: random 8-byte red.add over an L2-resident table).  achieved = red
            # lane-ops the kernel really issued (after warp aggregation, counted by the counting build) per second; both
            # sides are quoted at 8 bytes per lane-op.  The 512 B / sample of the un-aggregated algorithm is `naive`.
            ops_per_launch = red_lane_ops / max(n_calls, 1) * (prof_samples / max(red_samples, 1))
            achieved = ops_per_launch * 8 / sec / 1e9
            peak = reds_s * 8 / 1e9
            roofline.update({
                "bound": "l2-atomic", "achieved": achieved, "peak": peak, "frac": achieved / peak,
                "peak_source": "measured in this run: ngp_bench_red8, random red.global.add.v2.f32 over a 32 MB L2-resident "
                               "table, lane-ops/s x 8 B",
                "red_lane_ops_per_sample": red_lane_ops / max(red_samples, 1),
                "naive_red_lane_ops_per_sample": 128,
                "naive_algorithmic_gbs": 512.0 * points_per_launch / sec / 1e9,
                "note": "warp aggregation removes %.0f %% of the 128 per-sample atomics before they are issued; what is left "
                        "runs at `frac` of the chip's red issue rate" % (100.0 * (1 - red_lane_ops / max(red_samples, 1) / 128.0)),
            })
        elif dom in ("ngp_field_forward", "ngp_grid_encode_forward"):
            achieved = 512.0 * points_per_launch / sec / 1e9
            roofline.update({"bound": "l2-gather", "achieved": achieved, "peak": gathers_s * 4 / 1e9, "frac": None,
                             "note": "algorithmic gathers (512 B / sample) exceed the random-gather ceiling because "
                                     "neighbouring samples share corners in L1; see hbm / issue figures in profiles/"})
        else:
            roofline.update({"bound": "latency", "achieved": None, "peak": None, "frac": None})
        # the same kernel against HBM (the only driver-measured peak): its algorithmic stream is 76 B per sample
        roofline["hbm"] = {"algorithmic_bytes_per_sample": 76, "achieved_gbs": 76.0 * points_per_launch / sec / 1e9,
                           "peak_gbs": hbm_peak, "frac": 76.0 * points_per_launch / sec / 1e9 / hbm_peak}
        roofline["step_hbm"] = {"algorithmic_bytes_per_sample": 144, "achieved_gbs": 144.0 * samples / (ms * 1e-3) / 1e9,
                                "peak_gbs": hbm_peak, "frac": (144.0 * samples / (ms * 1e-3) / 1e9) / hbm_peak,
                                "note": "whole step, SURVEY 8d: 144 B per marched sample; the step is L2 / issue bound"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {
                "workload": "-O train step (BASELINE configs[2]/[3]): network_grid tiledgrid 16x2 @2^16 + 64-wide MLP, "
                            "128^3 occupancy grid, %d views x 64x64 rays per step over %d GPU(s), max_steps 1024, "
                            "synthetic SDS grad + entropy backward, grad all-reduce, Adam + GradScaler, occupancy "
                            "update every 16 steps" % (args.views, world),
                "views_per_step": args.views, "rays_per_step": args.views * H * W,
                "samples_per_step": samples / args.steps, "cuda_graph": not args.no_graph, "lr": args.lr,
                "hand_scheduled_step": step_fn.manual, "comm_error": bool(step_fn.fused_optimizer and step_fn.opt.comm_error),
                "sharding": ("8x8-pixel blocks of every view dealt along the block diagonals" if args.ray_order == "tiles"
                             else "image rows interleaved over ranks"),
                "pipelined_optimizer": step_fn.pipelined,
                "overlapped_steps": step_fn.overlap,
                "step_inputs": ("camera poses + intrinsics + guidance gradient; rays generated on the device (nerf/utils.py:get_rays)"
                                if device_rays else "pre-generated rays + guidance gradient"),
                "ray_chunks": len(step_fn._mws["chunks"]) if step_fn._mws else 1,
                "grad_allreduce": ("none (1 GPU)" if world == 1 else
                                   ("fused into the optimizer kernel over NVLink peer memory (%s)" % step_fn.peer.used
                                    if step_fn.opt.peer_ptrs is not None else "NCCL all_reduce (%s)" % (step_fn.peer_error or "requested"))),
                "step_ms": {"min": per_step[0], "median": per_step[len(per_step) // 2], "p90": per_step[(len(per_step) * 9) // 10],
                            "max": per_step[-1], "argmax": per_step_raw.index(per_step[-1])}, "timing": "inputs (3.5 MB/step) and the 7 MB table are "
                "smaller than L2 by nature of the workload; each step runs on a different view batch (64-batch pool), "
                "the 134+ MB/step of sample buffers exceed L2",
            },
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 * world,
                    "ms_per_step": ms_e2e / args.steps,
                    "result_read": ("loss.item() after every step" if (args.sync_loss and not step_fn.overlap) else
                                    "every step copies its loss (4 bytes) to pinned host memory behind the step; the host reads "
                                    "the value %d calls later, when that copy has landed (no per-step device sync)" % LOSS_LAG)},
            "gpu_launches": launches * world,
            "host_enqueue_ms_per_step": host_ms,
            "clocks": clk,
            "roofline": roofline,
        }
        if dp_result is not None:
            line["dp_check"] = dp_result
        if dp_sweep is not None:
            line["dp_sweep"] = dp_sweep
        if not args.no_cpu_baseline:
            try:
                v, cms, cores, desc = cpu_reference_run(args.cpu_sample_steps, 1)
                line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc,
                                        "ms_per_step": cms}
            except Exception as e:  # pragma: no cover
                line["cpu_baseline"] = {"error": repr(e)}
        if not args.no_ref_cuda:
            try:  # the reference's own CUDA extensions, in a fresh process on the same GPU (see oracle/ref_pipeline.py)
                env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[local_rank]
                           if os.environ.get("CUDA_VISIBLE_DEVICES") else str(local_rank))
                for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
                    env.pop(k, None)
                out = subprocess.run([sys.executable, "-m", "oracle.ref_pipeline", str(args.ref_steps), str(args.ref_warmup), repr(args.lr)],
                                     cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
                tag = [l for l in out.stdout.splitlines() if l.startswith("REF_PIPELINE_JSON ")]
                line["ref_cuda_ext"] = json.loads(tag[-1][len("REF_PIPELINE_JSON "):]) if tag else {
                    "unavailable": (out.stderr or out.stdout)[-300:]}
            except Exception as e:
                line["ref_cuda_ext"] = {"unavailable": repr(e)[:200]}
            if world == 1 and "value" in line.get("ref_cuda_ext", {}):
                # like for like: this repo at ONE view per step (the reference's batch, nerf/provider.py:240), same harness
                try:
                    line["one_view_per_step"] = one_view_run(device, args)
                    line["one_view_per_step"]["vs_ref_cuda_ext_median"] = (
                        line["one_view_per_step"]["value_median"] / line["ref_cuda_ext"]["value_median"])
                except Exception as e:  # noqa: BLE001
                    line["one_view_per_step"] = {"error": repr(e)[:200]}
        if world == 1 and not args.no_shading:
            try:   # secondary: the shaded step of the reference's schedule after albedo_iters (nerf/utils.py:345-356)
                line["shading"] = shading_run(device, args)
            except Exception as e:  # noqa: BLE001
                line["shading"] = {"error": repr(e)[:300]}
        emit(line)
    teardown(step_fn, world)


def shading_run(device, args, steps=12, warmup=4):
    """ONE view per step (the reference's batch) through the autograd step: albedo vs lambertian shading (7 field
    evaluations per sample for the normals + 6 for the smoothness normals, nerf/network_grid.py:90-144, nerf/renderer.py:
    485-494) with the 7-point stencil kernels (csrc/shading.cu).  Eager steps, CUDA events, median."""
    import torch
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    ro, rd = provider.make_training_views(16, H, W, seed=0, pin=False)
    ro, rd = ro.to(device), rd.to(device)
    g = (torch.randn(1, 3, H, W, generator=torch.Generator().manual_seed(2)) * 1e-2).to(device)
    out = {}
    for shading in ("albedo", "lambertian"):
        model = build_model(device)
        step_fn = TrainStep(model, H, W, lr=args.lr, max_steps=MAX_STEPS, graph=False, manual=False, shading=shading)
        for i in range(warmup):
            step_fn(ro[i % 16:i % 16 + 1], rd[i % 16:i % 16 + 1], g)
        torch.cuda.synchronize()
        step_fn.samples.zero_()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        evs[0].record()
        for i in range(steps):
            k = (warmup + i) % 16
            step_fn(ro[k:k + 1], rd[k:k + 1], g)
            evs[i + 1].record()
        torch.cuda.synchronize()
        per = sorted(a.elapsed_time(b) for a, b in zip(evs, evs[1:]))
        out[shading] = {"ms_per_step_median": per[len(per) // 2], "samples_per_step": int(step_fn.samples.item()) / steps}
        del step_fn, model
        torch.cuda.empty_cache()
    out["lambertian_over_albedo"] = out["lambertian"]["ms_per_step_median"] / out["albedo"]["ms_per_step_median"]
    out["what"] = ("autograd train step, 1 view of 64x64 rays, eager; lambertian = 13 field evaluations per sample forward (7-point "
                   "stencil + 6 smoothness normals) and 7 backward, each stencil ONE fused-field launch")
    return out


def one_view_run(device, args, steps=200, warmup=50):
    """The graphed hand-scheduled step on ONE 64x64 view per step; per-step CUDA events, median."""
    import torch
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    model = build_model(device)
    step_fn = TrainStep(model, H, W, lr=args.lr, max_steps=MAX_STEPS, graph=True)
    ro, rd = provider.make_training_views(32, H, W, seed=0, pin=False)
    g = torch.randn(1, 3, H, W, generator=torch.Generator().manual_seed(2)) * 1e-2
    pool = torch.stack([step_fn.pack_inputs(ro[k:k + 1], rd[k:k + 1], g) for k in range(32)]).to(device)
    for i in range(warmup):
        step_fn(pool[i % 32])
    torch.cuda.synchronize()
    step_fn.samples.zero_()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record()
    for i in range(steps):
        step_fn(pool[(100 + i) % 32])
        evs[i + 1].record()
    torch.cuda.synchronize()
    per = sorted(a.elapsed_time(b) for a, b in zip(evs, evs[1:]))
    total_ms = evs[0].elapsed_time(evs[-1])
    n = int(step_fn.samples.item())
    med = per[len(per) // 2]
    out = {"value": n / (total_ms * 1e-3), "value_median": (n / steps) / (med * 1e-3), "unit": UNIT, "ms_per_step": total_ms / steps,
           "ms_per_step_median": med, "views_per_step": 1, "samples_per_step": n / steps, "steps": steps, "warmup": warmup}
    step_fn._graph = None
    return out


def teardown(step_fn, world):
    """Orderly exit (the driver's exit hook records which native libraries were loaded): drop the captured graph, drain
    the device, leave the process group.  A watchdog hard-exits only if interpreter / NCCL teardown wedges AFTER the
    exit hooks have had their turn (atexit callbacks run before module teardown)."""
    import threading
    import torch
    import torch.distributed as dist
    sys.stdout.flush()
    sys.stderr.flush()
    try:
        step_fn._graph = None
        torch.cuda.synchronize()
        if world > 1 and dist.is_initialized():
            dist.barrier()
            torch.cuda.synchronize()
    except Exception:  # noqa: BLE001
        pass

    def _bail():
        os._exit(0)
    t = threading.Timer(90.0, _bail)
    t.daemon = True
    t.start()
    try:
        if world > 1 and dist.is_initialized():
            dist.destroy_process_group()
    except Exception:  # noqa: BLE001
        pass


# ---------------------------------------------------------------------------------------------------
# BASELINE configs[4]: inference render, 800x800, 100-frame 360-degree orbit
# ---------------------------------------------------------------------------------------------------
def run_infer_config(args):
    """Frames/s of the reference's --test orbit (nerf/provider.py:214-222, nerf/utils.py:435-456,507-555) through
    NeRFRenderer.run_cuda's inference branch: per frame one pose -> rays on the device -> ONE graph launch (conditional
    WHILE loop of march / fused field / composite / compaction) -> blend.  `value`: frames stay on the device;
    `e2e`: pose from pinned host memory in, the rendered RGB + depth frame read back to the host (what Trainer.test does)."""
    import torch
    from ngp_b200 import _cabi, orbit, provider
    assert torch.cuda.is_available(), "the B200 arm needs a GPU; there is no CPU fallback"
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(device)
    _cabi.load()
    R, n_frames, n_timed = args.res, args.frames, args.steps
    model = build_model(device)
    with torch.autocast("cuda", torch.float16):
        model.update_extra_state()       # the random-init scene: the density blob, ~5.6 % of the grid occupied
    model.eval()
    poses, intr = orbit.orbit_cameras(n_frames, R, R, device="cpu")
    poses_pinned = poses.pin_memory()
    poses_dev, intr_dev = poses.to(device), intr.to(device)
    rgb_host = torch.empty(R, R, 3).pin_memory()
    depth_host = torch.empty(R, R).pin_memory()

    def frame(i, e2e):
        pose = poses_pinned[i % n_frames].to(device, non_blocking=True) if e2e else poses_dev[i % n_frames]
        rgb, depth = orbit.render_frame(model, pose, intr_dev, R, R, max_steps=MAX_STEPS)
        if e2e:
            rgb_host.copy_(rgb, non_blocking=True)
            depth_host.copy_(depth, non_blocking=True)
            torch.cuda.current_stream().synchronize()      # Trainer.test converts every frame on the host
        return rgb

    clocks = ClockSampler(device.index)
    clocks.start()
    time.sleep(1.0)
    for i in range(max(args.warmup, 3)):
        frame(i, False)
    torch.cuda.synchronize()
    iters = []
    launches0 = _cabi.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n_timed):
        frame(i, False)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = _cabi.LAUNCHES - launches0
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(n_timed):
        frame(i, True)
    f1.record()
    torch.cuda.synchronize()
    ms_e2e = f0.elapsed_time(f1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"rgb": rgb_host, "depth": depth_host})   # the last timed frame, as read back
    clk = clocks.stop()
    # loop shape + samples of a few frames (diagnostics, untimed): iterations of the device loop, and the per-kernel times
    # of the same frames through the host loop (CUDA events around the entry points)
    for i in range(0, n_frames, max(1, n_frames // 5)):
        frame(i, False)
        iters.append(model.infer_loop_iterations())
    model.infer_loop = "host"
    names = ["ngp_march_rays", "ngp_field_forward", "ngp_composite_rays", "ngp_compact_alive", "ngp_get_rays", "ngp_bg_forward",
             "ngp_near_far_from_aabb", "ngp_blend_background_forward"]
    frame(0, False)
    torch.cuda.synchronize()
    _cabi.PROFILE = {n: [] for n in names}
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0.record()
    for i in range(3):
        frame(i * 7, False)
    h1.record()
    torch.cuda.synchronize()
    prof, _cabi.PROFILE = _cabi.PROFILE, None
    host_loop_ms = h0.elapsed_time(h1) / 3
    kern = {n: (sum(a.elapsed_time(b) for a, b in ev) / 3, len(ev) / 3) for n, ev in prof.items() if ev}
    model.infer_loop = "graph"
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    hbm_peak = peaks.get("hbm_gbs") or 6650.0
    gathers_s, _ = measure_l2_peaks(device)
    dom = max(kern, key=lambda k: kern[k][0]) if kern else None
    line = {
        "metric": "NeRF inference frames/s (800x800, 100-frame orbit, march_rays/composite_rays)", "value": n_timed / (ms * 1e-3),
        "unit": "frames/s", "n_gpus": 1, "steps": n_timed, "warmup": max(args.warmup, 3), "ms_per_step": ms / n_timed,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": "BASELINE configs[4]: inference render %dx%d via march_rays / composite_rays with the occupancy "
                               "grid, %d-frame 360-degree orbit (circle poses r 1.8, theta 60, fov 55), random-init scene "
                               "(density blob), max_steps 1024, T_thresh 1e-4, white background" % (R, R, n_frames),
                   "rays_per_frame": R * R, "rays_per_s": R * R * n_timed / (ms * 1e-3),
                   "inference_loop": type(model).infer_loop + " (one cudaGraphLaunch per frame, conditional WHILE node)",
                   "loop_iterations_per_frame": iters, "host_loop_ms_per_frame": host_loop_ms,
                   "timing": "every frame renders a different camera; a frame's sample / accumulator buffers (>60 MB) are "
                             "rewritten every loop iteration"},
        "e2e": {"value": n_timed / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": 64,
                "d2h_bytes_per_step": R * R * 16, "ms_per_step": ms_e2e / n_timed},
        "gpu_launches": launches, "clocks": clk,
        "roofline": {"kernel": dom, "bound": "l2-gather" if dom == "ngp_field_forward" else "latency", "unit": "GB/s",
                     "achieved": None, "peak": gathers_s * 4 / 1e9, "frac": None, "traffic": None,
                     "kernels_ms_per_frame_host_loop": {k: v[0] for k, v in kern.items()},
                     "kernel_calls_per_frame_host_loop": {k: v[1] for k, v in kern.items()}, "hbm_peak_gbs": hbm_peak,
                     "note": "per-kernel times from the host-loop variant of the same frames (events cannot be recorded inside "
                             "the graph's WHILE body); the loop is a chain of short launches bound by latency, not bandwidth"},
    }
    if not args.no_ref_cuda:
        try:
            env = dict(os.environ)
            for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
                env.pop(k, None)
            out = subprocess.run([sys.executable, "-m", "oracle.ref_pipeline", "infer", str(min(n_frames, 20)), str(R)], cwd=ROOT,
                                 env=env, capture_output=True, text=True, timeout=900)
            tag = [l for l in out.stdout.splitlines() if l.startswith("REF_PIPELINE_JSON ")]
            line["ref_cuda_ext"] = json.loads(tag[-1][len("REF_PIPELINE_JSON "):]) if tag else {"unavailable": (out.stderr or out.stdout)[-300:]}
            if "ms_per_frame_median" in line["ref_cuda_ext"]:
                line["ref_cuda_ext"]["speedup_e2e_vs_ref_median"] = line["ref_cuda_ext"]["ms_per_frame_median"] / (ms_e2e / n_timed)
        except Exception as e:  # noqa: BLE001
            line["ref_cuda_ext"] = {"unavailable": repr(e)[:200]}
    emit(line)
    sys.stdout.flush()


# ---------------------------------------------------------------------------------------------------
# BASELINE configs[1]: GridEncoder standalone, 16 levels x 2 features, hash 2^19, base 16 -> 2048, 2^22 points, fp16 fwd+bwd
# ---------------------------------------------------------------------------------------------------
def run_encoder_config(args):
    import numpy as np
    import torch
    from ngp_b200 import _cabi
    from gridencoder import GridEncoder
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(device)
    _cabi.load()
    torch.manual_seed(0)
    enc = GridEncoder(input_dim=3, num_levels=16, level_dim=2, base_resolution=16, log2_hashmap_size=19,
                      desired_resolution=2048, gridtype="hash").to(device)
    with torch.no_grad():
        enc.embeddings.uniform_(-1, 1)
    B = 1 << 22
    n_pool = 4                        # 4 x 50 MB of inputs and 4 x 134 MB of upstream gradients: more than fits beside the table in L2
    xs = [torch.rand(B, 3, device=device, generator=torch.Generator(device=device).manual_seed(1 + k)) * 2 - 1 for k in range(n_pool)]
    with torch.autocast("cuda", torch.float16):
        out = enc(xs[0], bound=1)
    gs = [torch.randn(out.shape, device=device, dtype=out.dtype, generator=torch.Generator(device=device).manual_seed(20 + k))
          for k in range(n_pool)]
    x_host = xs[0].cpu().pin_memory()

    def fwd(i):
        with torch.no_grad(), torch.autocast("cuda", torch.float16):
            return enc(xs[i % n_pool], bound=1)

    def fwd_bwd(i, x=None):
        enc.embeddings.grad = None
        with torch.autocast("cuda", torch.float16):
            o = enc(xs[i % n_pool] if x is None else x, bound=1)
        o.backward(gs[i % n_pool])

    def timed(fn, iters, warm):
        for i in range(warm):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(warm + i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    clocks = ClockSampler(device.index)
    clocks.start()
    time.sleep(1.0)
    steps, warm = args.steps, max(args.warmup, 3)
    launches0 = _cabi.LAUNCHES
    t_f = timed(fwd, steps, warm)
    t_fb = timed(fwd_bwd, steps, warm)
    launches = _cabi.LAUNCHES - launches0

    def e2e(i):
        fwd_bwd(i, x_host.to(device, non_blocking=True))
        enc.embeddings.grad.view(-1)[:1].cpu()          # a read of the step's result
    t_e2e = timed(e2e, steps, warm)
    clk = clocks.stop()
    if args.dump_outputs:
        # the table gradient of the last timed fwd + bwd (67 MB in fp32): a fixed sample of 2^20 of its rows
        rows = np.sort(np.random.default_rng(0).choice(enc.embeddings.shape[0], 1 << 20, replace=False))
        dump_outputs(args.dump_outputs, {"embeddings_grad_rows": torch.from_numpy(rows),
                                         "embeddings_grad_sample": enc.embeddings.grad[torch.from_numpy(rows).to(device)]})
    gathers_s, reds_s = measure_l2_peaks(device)
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    ach = 512.0 * B / (t_f * 1e-3) / 1e9
    line = {"metric": "GridEncoder points/s (16x2 hash 2^19, 2^22 points, fp16 fwd+bwd)", "value": B / (t_fb * 1e-3), "unit": "points/s",
            "n_gpus": 1, "steps": steps, "warmup": warm, "ms_per_step": t_fb, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": "BASELINE configs[1]: GridEncoder standalone, 16 levels x 2 feats, log2_hashmap 19, base res 16, desired "
                                   "res 2048, 2^22 uniformly random points, fp16 autocast, forward + backward (fp32-accumulated table gradient)",
                       "fwd_ms": t_f, "fwd_points_per_s": B / (t_f * 1e-3), "bwd_ms": t_fb - t_f,
                       "timing": "4 rotating input / gradient sets (736 MB) so no step finds its streams in L2; the 24.5 MB fp16 table is "
                                 "L2-resident by design"},
            "e2e": {"value": B / (t_e2e * 1e-3), "unit": "points/s", "h2d_bytes_per_step": B * 12, "d2h_bytes_per_step": 4, "ms_per_step": t_e2e},
            "gpu_launches": launches, "clocks": clk,
            "roofline": {"kernel": "ngp_grid_encode_forward", "bound": "l2-gather", "unit": "GB/s", "achieved": ach,
                         "peak": gathers_s * 4 / 1e9, "frac": ach / (gathers_s * 4 / 1e9), "traffic": None,
                         "peak_source": "measured in this run: ngp_bench_gather4, random 4-byte gathers over a 32 MB L2-resident table",
                         "backward": {"bound": "l2-atomic", "red_lane_ops_per_s": 128.0 * B / ((t_fb - t_f) * 1e-3), "peak_lane_ops_per_s": reds_s,
                                      "frac": 128.0 * B / ((t_fb - t_f) * 1e-3) / reds_s,
                                      "note": "random points share no cells: all 128 reds per point are issued (x-neighbour pairs merged "
                                              "into 16-byte reds where aligned, so the issued count is somewhat lower)"},
                         "hbm": {"algorithmic_bytes_per_point": 76, "achieved_gbs": 76.0 * B / (t_f * 1e-3) / 1e9, "peak_gbs": peaks.get("hbm_gbs")}}}
    if not args.no_ref_cuda:
        try:
            env = dict(os.environ)
            for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
                env.pop(k, None)
            out = subprocess.run([sys.executable, "-m", "oracle.ref_pipeline", "encoder"], cwd=ROOT, env=env, capture_output=True,
                                 text=True, timeout=600)
            tag = [l for l in out.stdout.splitlines() if l.startswith("REF_PIPELINE_JSON ")]
            line["ref_cuda_ext"] = json.loads(tag[-1][len("REF_PIPELINE_JSON "):]) if tag else {"unavailable": (out.stderr or out.stdout)[-300:]}
            if "fwd_bwd_ms" in line["ref_cuda_ext"]:
                line["ref_cuda_ext"]["speedup_fwd_bwd"] = line["ref_cuda_ext"]["fwd_bwd_ms"] / t_fb
        except Exception as e:  # noqa: BLE001
            line["ref_cuda_ext"] = {"unavailable": repr(e)[:200]}
    emit(line)
    sys.stdout.flush()


_REAL_STDOUT = None


def emit(line):
    """The one JSON line goes to the real stdout; everything else any library prints was diverted to stderr."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def main():
    global _REAL_STDOUT
    args = parse()
    sys.stdout.flush()  # (anything a library prints on stdout - e.g. the NCCL banner - is diverted to stderr below)
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.config == "infer":
        if int(os.environ.get("RANK", "0")) == 0:
            run_infer_config(args)
    elif args.config == "encoder":
        if int(os.environ.get("RANK", "0")) == 0:
            run_encoder_config(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
