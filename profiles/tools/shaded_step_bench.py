"""Time the shaded train step: one 64x64 view per step, bench.py's model, max_steps 1024, per-step CUDA events.

Configurations: albedo (graphed, hand-scheduled: the step bench.py times, for reference), and lambertian / textureless through
the autograd step (manual=False, what bench.py's `shading` entry times) and through the hand-scheduled step, eager and
graphed.  Writes one JSON file with, per configuration: median / p10 / p90 ms per step, samples per step and the step's
workspace bytes; plus the GPU name and power limit read in the same run.

    python profiles/tools/shaded_step_bench.py --out profiles/shaded_step_bench.json [--steps 200 --warmup 50]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for _p in (ROOT, os.path.join(ROOT, "single-stable-dreamfusion_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

CONFIGS = [  # (name, shading, manual, graph)
    ("albedo_manual_graph", "albedo", True, True),
    ("lambertian_autograd", "lambertian", False, False),
    ("textureless_autograd", "textureless", False, False),
    ("lambertian_manual_eager", "lambertian", True, False),
    ("lambertian_manual_graph", "lambertian", True, True),
    ("textureless_manual_eager", "textureless", True, False),
    ("textureless_manual_graph", "textureless", True, True),
]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [v.strip() for v in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu_query_error": repr(e)[:200]}


def run(device, shading, manual, graph, steps, warmup, lr=1e-3):
    import torch
    from bench import H, MAX_STEPS, W, build_model
    from ngp_b200 import provider
    from ngp_b200.trainer import TrainStep
    model = build_model(device)
    step_fn = TrainStep(model, H, W, lr=lr, max_steps=MAX_STEPS, graph=graph, manual=manual, shading=shading)
    assert step_fn.manual == manual
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
        step_fn(pool[(warmup + i) % 32])
        evs[i + 1].record()
    torch.cuda.synchronize()
    per = sorted(a.elapsed_time(b) for a, b in zip(evs, evs[1:]))
    pick = lambda q: per[min(len(per) - 1, int(q * len(per)))]  # noqa: E731
    ws_bytes = None
    if manual:
        ws_bytes = sum(ws.nbytes for _, _, ws in step_fn._mws["chunks"])
    loss = float(step_fn.loss.item())
    out = {"ms_per_step_median": pick(0.5), "ms_per_step_p10": pick(0.1), "ms_per_step_p90": pick(0.9),
           "samples_per_step": int(step_fn.samples.item()) / steps, "workspace_bytes": ws_bytes, "last_loss": loss,
           "n_chunks": len(step_fn._mws["chunks"]) if manual else None}
    step_fn._graph = None
    del step_fn, model
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=50)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("shaded_step_bench.py needs a CUDA device")
    device = torch.device("cuda:0")
    res = dict(what="train step, one 64x64 view (4096 rays) per step, bench.py model, max_steps 1024, ambient ratio 0.1 for "
                    "shaded steps; per-step CUDA events after warm-up; workspace_bytes = per-sample + stencil rows of the "
                    "hand-scheduled step", steps=args.steps, warmup=args.warmup, torch=torch.__version__, **gpu_info())
    res["configs"] = {}
    for name, shading, manual, graph in CONFIGS:
        res["configs"][name] = run(device, shading, manual, graph, args.steps, args.warmup)
        print(name, json.dumps(res["configs"][name]), flush=True)
    for s in ("lambertian", "textureless"):
        c = res["configs"]
        res["%s_autograd_over_manual_graph" % s] = (c["%s_autograd" % s]["ms_per_step_median"]
                                                    / c["%s_manual_graph" % s]["ms_per_step_median"])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "configs"}))


if __name__ == "__main__":
    main()
