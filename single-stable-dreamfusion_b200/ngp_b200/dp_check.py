"""Self-check of the fused peer-memory all-reduce + Adam kernel (csrc/adam.cu) against NCCL all_reduce followed by the
two-launch single-GPU optimizer, on seeded synthetic gradients.  Collective: every rank of the initialised process
group must call ``run``.  Used by tests/dp_peer_check.py (torchrun script) and by bench.py, which emits the result
as ``dp_check`` in its JSON line at N > 1 so that every scaling run carries data-parallel correctness evidence.
"""
import torch
import torch.distributed as dist


def run(device, n=1816256, steps=6, grad_div=1.0):
    """Returns {"ok", "max_abs_param_diff", "skipped", "steps_taken", "backend", "multicast"[, "error"]}.
    Step 2 carries an inf on ONE rank (in the last slice): every rank must skip it."""
    from .optim import FusedAdamScaler
    from .parallel import PeerMemory
    rank, world = dist.get_rank(), dist.get_world_size()
    n_table = n - 8192
    mk = lambda: [torch.nn.Parameter(torch.randn(n_table // 2, 2, device=device) * 0.1),  # noqa: E731
                  torch.nn.Parameter(torch.randn(64, 64, device=device) * 0.1),
                  torch.nn.Parameter(torch.randn(4096, device=device) * 0.1)]
    rng_state = torch.cuda.get_rng_state(device)
    torch.manual_seed(0)   # identical initial parameters on every rank
    pa = mk()
    torch.manual_seed(0)
    pb = mk()
    torch.cuda.set_rng_state(rng_state, device)
    groups = lambda ps: [{"params": ps[:1], "lr": 1e-2}, {"params": ps[1:], "lr": 1e-3}]  # noqa: E731
    result = {"world": world, "n": n}
    try:
        peer = PeerMemory(device)
        mine = FusedAdamScaler(groups(pa), growth_interval=3, grad_div=grad_div, peer_memory=peer, lr_decay=(0.1, 10))
        result["backend"] = peer.used
        result["multicast"] = bool(mine.multicast is not None and mine.use_multicast)
    except Exception as e:  # noqa: BLE001
        result.update(ok=False, error="peer memory unavailable: %r" % (e,))
        return result
    ref = FusedAdamScaler(groups(pb), growth_interval=3, grad_div=grad_div, lr_decay=(0.1, 10))
    ok, worst = True, 0.0
    for it in range(steps):
        g = torch.Generator(device=device).manual_seed(1000 * it + rank)
        raw = torch.randn(mine.numel, device=device, generator=g) * (10.0 ** (it % 3 - 2))
        if it == 2 and rank == world - 1:
            raw[mine.numel - 5] = float("inf")
        scale = mine.get_scale()
        ok = ok and scale == ref.get_scale()
        mine.flat_grads.copy_(raw * scale)
        ref.flat_grads.copy_(raw * scale)
        torch.cuda.synchronize(device)
        dist.barrier()
        mine.step()
        dist.all_reduce(ref.flat_grads)
        ref.step(zero_grads=True)
        torch.cuda.synchronize(device)
        dist.barrier()
        d = (mine.flat_params - ref.flat_params).abs().max().item()
        worst = max(worst, d)
        same_half = torch.equal(mine.flat_half, mine.flat_params.half())
        zeroed = mine.flat_grads.abs().sum().item() == 0
        st_ok = torch.equal(mine.state[:5], ref.state[:5])
        if not (d <= 2e-6 and same_half and zeroed and st_ok and not mine.comm_error):
            ok = False
            result.setdefault("first_failure", dict(rank=rank, step=it, max_abs=d, half=same_half, zeroed=zeroed,
                                                    state=mine.state.tolist(), ref_state=ref.state.tolist()))
    result["max_abs_param_diff"] = worst
    result["steps_taken"], result["skipped"] = mine.steps_taken, int(mine.state[4].item())
    ok = ok and result["skipped"] == (1 if steps > 2 else 0)
    flag = torch.tensor([1.0 if ok else 0.0, -worst], device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    result["ok"] = bool(flag[0].item() > 0)
    result["max_abs_param_diff"] = float(-flag[1].item())
    result["_objects"] = (mine, ref)   # callers that go on to time the two variants; dropped before printing
    return result
