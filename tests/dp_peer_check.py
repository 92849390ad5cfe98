#!/usr/bin/env python
"""Multi-GPU check of the fused peer-memory all-reduce + Adam kernel (csrc/adam.cu).  Run under torchrun:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
        tests/dp_peer_check.py [--n 1816256]

Every rank fills its gradient bucket with different seeded values (one step carries an inf on ONE rank), runs
FusedAdamScaler.step() over peer memory, and compares parameters / fp16 shadow / scaler state with a
single-process reference: NCCL all_reduce of the same buckets followed by the two-launch single-GPU optimizer.
Also times both variants as CUDA-graph replays.  Rank 0 prints one JSON line; exit code 1 on any mismatch.
(tests/test_gpu_dp.py launches this when the box has >= 2 GPUs.)
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "single-stable-dreamfusion_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1816256)
    ap.add_argument("--steps", type=int, default=6)
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from ngp_b200 import _cabi
    _cabi.load()

    from ngp_b200 import dp_check
    result = dp_check.run(dev, n=args.n, steps=args.steps, grad_div=float(world))
    if "error" in result:
        if rank == 0:
            print(json.dumps({"ok": False, "error": result["error"]}))
        dist.destroy_process_group()
        sys.exit(2)
    mine, ref = result.pop("_objects")
    ok = result["ok"]
    if not ok:
        print("rank %d: %r" % (rank, result.get("first_failure")), file=sys.stderr)

    # ---- data-parallel occupancy refresh: 1/world of the cells per rank + all-gather -> identical grids everywhere -----
    import argparse as _ap
    from ngp_b200.network_grid import NeRFNetwork
    torch.manual_seed(0)
    model = NeRFNetwork(_ap.Namespace(bound=1, cuda_ray=True, min_near=0.1, density_thresh=10, bg_radius=1.4)).to(dev).train()
    torch.manual_seed(100 + rank)   # different jitter streams per rank, as in training
    model.dp_shard = (rank, world)
    with torch.autocast("cuda", torch.float16):
        model.update_extra_state()
        model.update_extra_state()
    grids = [torch.empty_like(model.density_grid) for _ in range(world)]
    dist.all_gather(grids, model.density_grid)
    bits = [torch.empty_like(model.density_bitfield) for _ in range(world)]
    dist.all_gather(bits, model.density_bitfield)
    same = all(torch.equal(g, grids[0]) for g in grids) and all(torch.equal(b, bits[0]) for b in bits)
    occ = float(torch.tensor([bin(int(v)).count("1") for v in bits[0].cpu().tolist()]).sum()) / (model.density_bitfield.numel() * 8)
    result["sharded_refresh_identical"], result["sharded_refresh_occupancy"] = bool(same), occ
    ok = ok and same and 0.02 < occ < 0.15   # the random-init density blob occupies ~5.6 % of the grid (SURVEY 8)

    # ---- timing: graph replays of (fused) vs (NCCL all_reduce + check_finite + adam) -------------------------------
    def timed(fn, iters=50):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, capture_error_mode="thread_local"):
            fn()
        for _ in range(5):
            gr.replay()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            gr.replay()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / iters], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def nccl_path():
        dist.all_reduce(ref.flat_grads)
        ref.step(zero_grads=True)

    try:
        result["fused_us"] = timed(mine.step) * 1e3
        result["nccl_plus_adam_us"] = timed(nccl_path) * 1e3
        result["comm_error_after_timing"] = mine.comm_error
        ok = ok and not mine.comm_error
    except Exception as e:  # noqa: BLE001
        result["timing_error"] = repr(e)[:300]
        ok = False
    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    result["ok"] = bool(flag.item() > 0)
    if rank == 0:
        print(json.dumps(result))
    sys.stdout.flush()
    os._exit(0 if result["ok"] else 1)


if __name__ == "__main__":
    main()
