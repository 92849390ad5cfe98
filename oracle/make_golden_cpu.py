#!/usr/bin/env python
"""TEST INFRASTRUCTURE: pins oracle/torch_renderer.py against the REAL reference, imported from
/root/reference in this (GPU-less) container, and writes tests/golden/cpu_renderer_golden.npz.

The reference's non-cuda-ray path (nerf/renderer.py:run + nerf/network.py) is pure PyTorch except for
two CUDA-only ops, which are shimmed here ONLY to let the reference run on CPU:
``raymarching.near_far_from_aabb`` and ``FreqEncoder``.  Six absent optional dependencies that the
reference imports at module top (trimesh, mcubes, imageio, tensorboardX, matplotlib, torch_ema, ...)
are stubbed with empty modules.  Same seed + same weights + same inputs => the port must reproduce
the reference's image / depth / weights_sum and the parameter gradients.
"""
import argparse
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import torch_renderer as TR  # noqa: E402
from oracle.build_ref import REF  # noqa: E402  (the reference's source tree, NGP_REFERENCE_ROOT)


def import_reference():
    for name in ["trimesh", "mcubes", "imageio", "tensorboardX", "matplotlib", "matplotlib.pyplot", "torch_ema", "cv2",
                 "rich", "rich.console", "tqdm", "pandas"]:
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                sys.modules[name] = types.ModuleType(name)
    sys.modules["torch_ema"].ExponentialMovingAverage = object
    if not hasattr(sys.modules["rich.console"], "Console"):
        sys.modules["rich.console"].Console = object
    # CPU shims for the two CUDA-only ops on this path
    rm = types.ModuleType("raymarching")
    rm.near_far_from_aabb = lambda o, d, aabb, min_near=0.2: TR.near_far_from_aabb(o, d, aabb, min_near)
    sys.modules["raymarching"] = rm
    fe = types.ModuleType("freqencoder")
    fe.FreqEncoder = TR.FreqEncoder
    sys.modules["freqencoder"] = fe
    sys.path.insert(0, REF)
    from nerf.network import NeRFNetwork  # noqa: E402
    return NeRFNetwork


def main():
    NeRFNetwork = import_reference()
    opt = argparse.Namespace(bound=1, cuda_ray=False, min_near=0.1, density_thresh=10, bg_radius=1.4)
    torch.manual_seed(0)
    ref = NeRFNetwork(opt)
    ref.train()
    port = TR.VanillaNeRF(bound=1.0, min_near=0.1, bg_radius=1.4)
    port.train()
    # copy weights: the parameter trees have the same names
    sd = {k: v for k, v in ref.state_dict().items() if k in port.state_dict()}
    missing = set(port.state_dict()) - set(sd)
    assert not missing, missing
    port.load_state_dict(sd)

    rays_o, rays_d = TR.make_view(16, 16, seed=3)
    G = torch.randn(1, 256, 3, generator=torch.Generator().manual_seed(1))

    torch.manual_seed(123)
    out_ref = ref.render(rays_o, rays_d, staged=False, perturb=True, shading="albedo", ambient_ratio=1.0, num_steps=64,
                         upsample_steps=32)
    (out_ref["image"] * G).sum().backward()
    torch.manual_seed(123)
    out_port = port.run(rays_o, rays_d, num_steps=64, upsample_steps=32, perturb=True)
    (out_port["image"] * G).sum().backward()

    res = {}
    for k in ("image", "depth", "weights_sum"):
        a, b = out_ref[k].detach().numpy(), out_port[k].detach().numpy()
        print(k, "max abs diff ref vs port:", np.abs(a - b).max())
        assert np.allclose(a, b, rtol=1e-5, atol=1e-6), k
        res[k] = a
    gr = dict(ref.named_parameters())
    for name, p in port.named_parameters():
        a, b = gr[name].grad.numpy(), p.grad.numpy()
        assert np.allclose(a, b, rtol=1e-4, atol=1e-6), name
    res["grad_sigma_net_last_w"] = gr["sigma_net.net.4.weight"].grad.numpy()
    res["grad_bg_net_first_w"] = gr["bg_net.net.0.dense.weight"].grad.numpy()
    n_params = sum(p.numel() for p in ref.parameters())
    res["n_params"] = np.array([n_params])
    out_path = os.path.join(ROOT, "tests", "golden", "cpu_renderer_golden.npz")
    np.savez_compressed(out_path, **res)
    print("reference params:", n_params, "-> wrote", out_path)


if __name__ == "__main__":
    main()
